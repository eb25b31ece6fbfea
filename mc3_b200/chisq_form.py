"""Which chi-squared form a population of a built-in or CUDA model runs (engine.Population),
decided once on the host when the population is built.  From the most general:
  plain     the model's own kernel (k_model_chisq), or a CudaModel's
  grid      a sinusoid on a uniform, or piecewise-uniform (`seg`), abscissa grid (SineGridModel)
  fold      ... with one uncertainty for all points: mirrored point pairs (k_sinefold)
  moment    ... on sufficient statistics of those pairs (k_sinefold<MOM>, mc3b_moment_t)
  spectral  ... from a precomputed spectrum of the data (k_spectral_chisq, mc3b_spectral_t)
MC3B_NO_USIG, _GRID, _SEG, _FOLD, _MOMENT, _FUSE and _SPECTRAL=1 each turn one off.  MC3B_MOM_LAYOUT=1:
the moment sums as FP64 tensor-core products (k_sinemma), measured slower (0.127 against 0.099 ms at config 2)."""
import os
from typing import NamedTuple, Optional

import numpy as np

from . import _lib, gridseg, spectral
from .models import CudaModel, SINUSOID, SINUSOID_GRID


class Form(NamedTuple):
    model_id: Optional[int]         # the kernel's: SINUSOID_GRID for the grid forms, None for a CudaModel
    usig: bool                      # one uncertainty for all points (mc3b_chisq_opts_t.uniform_sigma)
    grid: bool
    seg: Optional[dict]             # gridseg.tile_layout of a piecewise-uniform grid, or None
    fold: bool
    nfold: int                      # points the fold covers: all, or the whole tiles of `seg`
    moment: bool
    layout: int                     # mc3b_moment_t.layout
    spectral_plan: Optional[dict]   # spectral.plan, or None


def choose_form(func, x, uncert, dtype, params, pstep, pmin, pmax):
    """Form of `func` (BuiltinModel or CudaModel) on this device's slice of `x` and `uncert` in
    dtype (_lib.F64 / _lib.F32); params, pstep, pmin, pmax bound the period (spectral.band)."""
    env = os.environ.get
    user = isinstance(func, CudaModel)
    usig = bool(uncert.size > 0 and np.all(uncert == uncert[0]) and not env('MC3B_NO_USIG'))
    grid, seg, nfold = False, None, x.size
    if not user and func.model_id == SINUSOID and dtype == _lib.F64 and x.size >= 8 and not env('MC3B_NO_GRID'):
        ideal = x[0] + np.arange(x.size)*((x[-1] - x[0])/(x.size - 1))
        if x[-1] != x[0] and np.max(np.abs(x - ideal)) <= 8*np.finfo(float).eps*np.max(np.abs(x)):
            grid = True
        elif not env('MC3B_NO_SEG'):
            seg = gridseg.tile_layout(x)
            if seg is not None:
                grid, nfold = True, 128*seg['starts'].size
    fold = grid and usig and not env('MC3B_NO_FOLD')
    moment = fold and nfold >= 256 and not env('MC3B_NO_MOMENT') and not env('MC3B_NO_FUSE')
    layout = int(env('MC3B_MOM_LAYOUT', 0)) if moment else 0
    band = spectral.band(params, pstep, pmin, pmax) if moment else None
    plan = spectral.plan(float(x.min()), float(x.max()), *band, x.size) \
        if band is not None and layout == 0 and not env('MC3B_NO_SPECTRAL') else None
    return Form(SINUSOID_GRID if grid else None if user else func.model_id, usig, grid, seg, fold, nfold,
                moment, layout, plan)
