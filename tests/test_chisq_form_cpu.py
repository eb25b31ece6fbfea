"""CPU-only: the decision table of mc3_b200.chisq_form.choose_form, the chi-squared form a
Population of a built-in or CUDA model runs, under each of the switches that turn a form off."""
import numpy as np
import pytest

from mc3_b200 import _lib, gridseg, spectral
from mc3_b200.chisq_form import choose_form
from mc3_b200.models import CudaModel, POLYNOMIAL, SINUSOID, SINUSOID_GRID, polynomial, sinusoid

SWITCHES = ('MC3B_NO_USIG', 'MC3B_NO_GRID', 'MC3B_NO_SEG', 'MC3B_NO_FOLD', 'MC3B_NO_MOMENT', 'MC3B_NO_FUSE',
            'MC3B_MOM_LAYOUT', 'MC3B_NO_SPECTRAL')
# sinusoid + line with a shared phase and a fixed slope; the period is bounded to [2.3, 2.7]
PARAMS = dict(params=np.array([1.01, 2.505, 1.01, 5.01, -0.2]), pstep=np.array([1e-2, 1e-3, -1.0, 1e-2, 0.0]),
              pmin=np.array([0.99, 2.3, -np.pi, 4.994, -1.0]), pmax=np.array([1.035, 2.7, np.pi, 5.03, 1.0]))


@pytest.fixture(autouse=True)
def no_switches(monkeypatch):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)


def gapped_x():
    """Constant cadence with three gaps: 9984 points in four runs of whole 128-point tiles."""
    idx = np.concatenate([np.arange(a, a + m) for a, m in ((0, 2560), (3000, 3840), (7500, 1280), (9100, 2304))])
    return idx*1e-3


def form(x=None, n=10000, uncert=None, func=sinusoid, dtype=_lib.F64, **kw):
    x = np.linspace(0.0, 10.0, n) if x is None else x
    uncert = np.full(x.size, 0.5) if uncert is None else uncert
    p = {k: v.copy() for k, v in PARAMS.items()}
    p.update(kw)
    return choose_form(func, x, uncert, dtype, p['params'], p['pstep'], p['pmin'], p['pmax'])


def shape(f):
    """The form's kind: the most specialised one it takes."""
    if f.spectral_plan is not None:
        return 'spectral'
    return 'moment' if f.moment else 'fold' if f.fold else 'grid' if f.grid else 'plain'


def test_uniform_grid_takes_the_spectral_form():
    f = form()
    assert (f.model_id, f.usig, f.grid, f.seg, f.fold, f.nfold, f.moment, f.layout) == \
        (SINUSOID_GRID, True, True, None, True, 10000, True, 0)
    band = spectral.band(PARAMS['params'], PARAMS['pstep'], PARAMS['pmin'], PARAMS['pmax'])
    assert f.spectral_plan == spectral.plan(0.0, 10.0, *band, 10000)


@pytest.mark.parametrize('switch, value, want', [
    ('MC3B_NO_SPECTRAL', '1', 'moment'),
    ('MC3B_MOM_LAYOUT', '1', 'moment'),
    ('MC3B_NO_MOMENT', '1', 'fold'),
    ('MC3B_NO_FUSE', '1', 'fold'),
    ('MC3B_NO_FOLD', '1', 'grid'),
    ('MC3B_NO_USIG', '1', 'grid'),
    ('MC3B_NO_GRID', '1', 'plain'),
])
def test_switches(monkeypatch, switch, value, want):
    monkeypatch.setenv(switch, value)
    f = form()
    assert shape(f) == want
    assert f.layout == (1 if switch == 'MC3B_MOM_LAYOUT' else 0)
    assert f.usig == (switch != 'MC3B_NO_USIG')
    assert f.model_id == (SINUSOID if want == 'plain' else SINUSOID_GRID) and f.seg is None


def test_per_point_sigma_keeps_the_grid_without_fold():
    f = form(uncert=np.random.RandomState(5).uniform(0.4, 0.6, 10000))
    assert shape(f) == 'grid' and not f.usig and f.model_id == SINUSOID_GRID


def test_gapped_cadence_takes_the_tile_layout():
    x = gapped_x()
    f = form(x)
    seg = gridseg.tile_layout(x)
    assert f.grid and f.model_id == SINUSOID_GRID and f.fold and f.moment
    assert f.seg['starts'].size == seg['starts'].size == 78 and np.array_equal(f.seg['perm'], seg['perm'])
    assert f.nfold == 128*78
    band = spectral.band(PARAMS['params'], PARAMS['pstep'], PARAMS['pmin'], PARAMS['pmax'])
    assert f.spectral_plan == spectral.plan(x.min(), x.max(), *band, x.size)


def test_gapped_cadence_without_the_tile_layout_is_plain(monkeypatch):
    monkeypatch.setenv('MC3B_NO_SEG', '1')
    f = form(gapped_x())
    assert shape(f) == 'plain' and f.seg is None and f.model_id == SINUSOID and f.usig


@pytest.mark.parametrize('x', [np.sort(np.random.RandomState(2).uniform(0.0, 10.0, 10000)),
                               np.linspace(0.0, 1.0, 7)], ids=['irregular', 'n7'])
def test_plain(x):
    f = form(x)
    assert shape(f) == 'plain' and f.seg is None and f.model_id == SINUSOID and f.nfold == x.size


def test_fold_without_moment_below_256_points():
    f = form(n=200)
    assert shape(f) == 'fold' and f.nfold == 200


@pytest.mark.parametrize('pmin_period', [0.0, 1e-3], ids=['band_reaches_0', 'beyond_max_nodes'])
def test_moment_without_spectral(pmin_period):
    pmin = PARAMS['pmin'].copy()
    pmin[1] = pmin_period
    # a period down to 1e-3 spans more nodes than the table holds
    assert (spectral.band(PARAMS['params'], PARAMS['pstep'], pmin, PARAMS['pmax']) is None) == (pmin_period == 0.0)
    assert shape(form(pmin=pmin)) == 'moment'


def test_f32_is_plain():
    f = form(dtype=_lib.F32)
    assert shape(f) == 'plain' and f.model_id == SINUSOID and f.usig


def test_polynomial_takes_its_own_kernel():
    f = form(func=polynomial)
    assert shape(f) == 'plain' and f.model_id == POLYNOMIAL


def test_cuda_model_takes_its_own_kernel():
    m = CudaModel('__device__ real model(real x, const real* p) { return p[0]*sin(x); }', 5)
    f = form(func=m)
    assert shape(f) == 'plain' and f.model_id is None and f.usig


def test_wavelet_likelihood_takes_the_same_form():
    """wlike=True: three wavelet parameters after the model's own."""
    ext = {k: np.concatenate([v, w]) for (k, v), w in zip(PARAMS.items(), ([1.0, 0.1, 0.0], [0.1, 0.1, 0.0],
                                                                          [0.0, 0.0, -1.0], [2.0, 2.0, 1.0]))}
    assert shape(form(**ext)) == 'spectral'
    assert form(**ext) == form()
