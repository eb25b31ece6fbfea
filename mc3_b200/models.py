"""Built-in models and the model-callable conventions of mc3_b200.

The reference's `func` is any Python callable `func(params, *indparams,
**indparams_dict) -> 1-D array` evaluated once per chain-step
(mc3/chain.py:316-319).  mc3_b200 accepts three kinds of `func`:

* a BuiltinModel (below): evaluated inside the fused CUDA model+chi-squared
  kernel for all chains at once -- the fast path;
* a TorchModel: a user torch callable evaluated ONCE per generation over the
  whole population, `fn(P[nchains, npars], *indparams) -> model[nchains, N]`
  on the device;
* a CudaModel: the user's own formula as a CUDA device function, compiled at run
  time (NVRTC, mc3_b200/jit.py) into the same fused kernel as the built-in models --
  the fast path for any model of up to MAX_INPUTS (4) per-point inputs:

      transit = CudaModel('''
          __device__ real model(real x, const real* p) {      // p[0..nparams)
              real z = fabs(x - p[1]) / p[2];                  // helpers above `model` are allowed
              return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
          }''', nparams=5, name='trapezoid')

  `real` is double (float with dtype='f32'); models.cuh is included, so fast_sin and
  fast_sincos_core are available.  nparams counts the parameters the model itself
  consumes (with wlike=True it gets params[0:-3]), at most 32.  With ninputs=k the
  model takes k reals before the parameters, `model(real t, real xc, real yc, const
  real* p)` for k = 3, and the fit passes k arrays of the data's shape as indparams,
  in the same order.  With nconst=m, the indparams after those arrays (numbers, 0-d
  or 1-D arrays) are flattened in order into m run-time constants, p[nparams:nparams+m]
  (their values are launch data, never part of the compiled module); nwork=w adds w
  slots after them for an optional `__device__ void prepare(real* p)`, run once per
  chain wherever the parameters are loaded, to hoist what depends on the chain alone
  (1/sigma, 2 pi/P).  p holds [parameters | constants | work], at most 32 slots.  The
  source compiles on first use; a compile error raises ValueError with the NVRTC log;
* a TorchModel: a user torch callable evaluated ONCE per generation over the
  whole population, `fn(P[nchains, npars], *indparams) -> model[nchains, N]`
  on the device;
* any other callable: the reference's own convention, evaluated per chain on
  the host (compatibility path; the chi-squared still runs on the GPU).

BuiltinModel and CudaModel objects are also plain callables with the reference
signature `model(params, x)`; the evaluation runs on the GPU (mc3b_model_eval,
mc3b_user_model_eval).
"""
import numpy as np

from . import _lib

POLYNOMIAL, SINUSOID, GAUSSIAN, BOX, SINUSOID_GRID = 0, 1, 2, 3, 4


class BuiltinModel:
    """A model implemented in mc3_b200/csrc/models.cuh.

    polynomial  y = sum_k p[k] x^k            (1..8 coefficients)
    sinusoid    y = p0 sin(2 pi x/p1 + p2) + p3 + p4 x
    gaussian    y = p0 exp(-0.5 ((x-p1)/p2)^2) + p3
    box         y = p3 - p0 [|x-p1| < p2/2]
    """

    def __init__(self, name, model_id, nparams):
        self.name, self.model_id, self.nparams = name, model_id, nparams

    def nmodel(self, nfunc_params):
        """Number of leading parameters the model consumes."""
        if self.nparams is None:
            if not 1 <= nfunc_params <= 8:
                raise ValueError(
                    f'{self.name} takes 1 to 8 parameters, got {nfunc_params}')
            return nfunc_params
        if nfunc_params != self.nparams:
            raise ValueError(
                f'{self.name} takes {self.nparams} parameters, got {nfunc_params}')
        return self.nparams

    def __call__(self, params, x):
        import torch
        params = np.atleast_2d(np.asarray(params, dtype=np.double))
        x = np.ascontiguousarray(x, dtype=np.double)
        nmodel = self.nmodel(params.shape[1])
        dev = torch.device('cuda')
        dp = torch.from_numpy(np.ascontiguousarray(params)).to(dev)
        dx = torch.from_numpy(x).to(dev)
        out = torch.empty((params.shape[0], x.size), dtype=torch.float64, device=dev)
        _lib.call('mc3b_model_eval', self.model_id, dp.data_ptr(), params.shape[1],
                  params.shape[0], nmodel, dx.data_ptr(), x.size, out.data_ptr(),
                  _lib.stream_ptr())
        res = out.cpu().numpy()
        return res[0] if res.shape[0] == 1 else res

    def __repr__(self):
        return f'<mc3_b200 built-in model {self.name}>'


def _eval_rows(params, xs, launch):
    """model(params, *xs) on the current GPU: [nrows, N] (or [N] for one row)."""
    import torch
    params = np.atleast_2d(np.asarray(params, dtype=np.double))
    xs = [np.ascontiguousarray(x, dtype=np.double) for x in xs]
    if any(x.shape != xs[0].shape for x in xs):
        raise ValueError('the input arrays of a model must have one shape')
    dev = torch.device('cuda')
    dp = torch.from_numpy(np.ascontiguousarray(params)).to(dev)
    dxs = [torch.from_numpy(x).to(dev) for x in xs]
    out = torch.empty((params.shape[0], xs[0].size), dtype=torch.float64, device=dev)
    launch(dp, dxs, out)
    res = out.cpu().numpy()
    return res[0] if res.shape[0] == 1 else res


class CudaModel:
    """A user model written as a CUDA device function (see the module docstring):
    `__device__ real model(real x, const real* p)` in `source`, taking `nparams`
    parameters, or with ninputs = k > 1 inputs `model(real x1, ..., real xk, const
    real* p)`.  With nconst = m, p[nparams:nparams+m] holds m run-time constants, and
    nwork more slots follow for an optional `__device__ void prepare(real* p)` to fill
    once per chain.  Compiled lazily, once per process and dtype; pickles as its source
    (one process per GPU receives it and compiles its own copy)."""

    ninputs = 1            # stored on the instance only when it is not 1
    nconst = 0             # ... only when it is not 0
    nwork = 0              # ... only when it is not 0

    def __init__(self, source, nparams, name='cuda_model', ninputs=1, nconst=0, nwork=0):
        nparams = int(nparams)
        if not 1 <= nparams <= _lib.MAX_PARS:
            raise ValueError(f'a CudaModel takes 1 to {_lib.MAX_PARS} parameters, got {nparams}')
        ninputs = int(ninputs)
        if not 1 <= ninputs <= _lib.MAX_INPUTS:
            raise ValueError(f'a CudaModel takes 1 to {_lib.MAX_INPUTS} inputs, got {ninputs}')
        nconst, nwork = int(nconst), int(nwork)
        if nconst < 0 or nwork < 0:
            raise ValueError(f'nconst and nwork must not be negative, got {nconst} and {nwork}')
        if nparams + nconst + nwork > _lib.MAX_PARS:
            raise ValueError(f'nparams + nconst + nwork = {nparams} + {nconst} + {nwork} exceeds the '
                             f'{_lib.MAX_PARS} slots of a model')
        self.source, self.nparams, self.name = str(source), nparams, str(name)
        if ninputs != 1:
            self.ninputs = ninputs
        if nconst != 0:
            self.nconst = nconst
        if nwork != 0:
            self.nwork = nwork

    def __getstate__(self):
        state = {'source': self.source, 'nparams': self.nparams, 'name': self.name}
        for key in ('ninputs', 'nconst', 'nwork'):
            if key in vars(self):
                state[key] = vars(self)[key]
        return state

    def __setstate__(self, state):
        self.__init__(state['source'], state['nparams'], state['name'], state.get('ninputs', 1),
                      state.get('nconst', 0), state.get('nwork', 0))

    def nmodel(self, nfunc_params):
        """Number of leading parameters the model consumes."""
        if nfunc_params != self.nparams:
            raise ValueError(
                f'{self.name} takes {self.nparams} parameters, got {nfunc_params}')
        return self.nparams

    def split_args(self, args):
        """(per-point arrays, constants) of the arguments after the parameters: the first
        ninputs are the arrays; with nconst or nwork set, the rest (numbers, 0-d and 1-D
        arrays) are flattened in order into the constants, which must come to nconst
        values.  A model of neither takes its arrays only (constants None)."""
        if not (self.nconst or self.nwork):
            return list(args), None
        xs, rest = list(args[:self.ninputs]), args[self.ninputs:]
        vals = [np.asarray(a, dtype=np.double) for a in rest]
        if any(v.ndim > 1 for v in vals):
            raise ValueError(f'{self.name}: constants are numbers or 1-D arrays, got shapes '
                             f'{[v.shape for v in vals]}')
        k = np.concatenate([v.ravel() for v in vals]) if vals else np.zeros(0)
        if k.size != self.nconst:
            raise ValueError(f'{self.name} takes {self.nconst} constant(s) after its {self.ninputs} input '
                             f'array(s), got {k.size}')
        return xs, k

    def cache_key(self, dtype=_lib.F64):
        from . import jit
        return jit.cache_key(self.source, self.nparams, dtype, self.ninputs, self.nconst, self.nwork)

    def handle(self, dtype=_lib.F64, stats=None):
        """mc3b_user_model_t* of this model for dtype (_lib.F64 / _lib.F32)."""
        from . import jit
        return jit.handle(self.source, self.nparams, dtype, self.name, stats, self.ninputs, self.nconst,
                          self.nwork)

    def batch_handle(self, stats=None):
        """mc3b_user_batch_t* of this model: the fp64 kernels of sample_batch, a module of
        their own (compiled on first use, not by sample())."""
        from . import jit
        return jit.handle(self.source, self.nparams, _lib.F64, self.name, stats, self.ninputs, self.nconst,
                          self.nwork, kind='batch')

    def __call__(self, params, *args):
        import torch
        xs, k = self.split_args(args)
        if len(xs) != self.ninputs:
            raise ValueError(f'{self.name} takes {self.ninputs} input array(s), got {len(xs)}')
        self.nmodel(np.shape(np.atleast_2d(params))[1])
        h = self.handle(_lib.F64)

        def launch(dp, dxs, out):
            dk = None if k is None or k.size == 0 else torch.from_numpy(k).to(out.device)
            _lib.call('mc3b_user_model_eval_consts', h, dp.data_ptr(), dp.shape[1], dp.shape[0],
                      _lib.ptrs(dxs), len(dxs), _lib.ptr(dk), self.nconst, dxs[0].numel(), out.data_ptr(),
                      _lib.stream_ptr())
        return _eval_rows(params, xs, launch)

    def __repr__(self):
        inputs = f', {self.ninputs} inputs' if self.ninputs != 1 else ''
        inputs += f', {self.nconst} constants' if self.nconst else ''
        inputs += f', {self.nwork} work slots' if self.nwork else ''
        return f'<mc3_b200 CUDA model {self.name} ({self.nparams} parameters{inputs})>'


class TorchModel:
    """Marks `fn` as batched over chains: fn(P[nchains, npars], *indparams,
    **indparams_dict) -> torch tensor [nchains, N] (float64, on P's device)."""

    def __init__(self, fn):
        self.fn = fn

    def __call__(self, params, *args, **kwargs):
        import torch
        p = torch.as_tensor(np.atleast_2d(np.asarray(params, dtype=np.double)),
                            device='cuda')
        args = [torch.as_tensor(a, device='cuda') if isinstance(a, np.ndarray) else a
                for a in args]
        out = self.fn(p, *args, **kwargs).detach().cpu().numpy()
        return out[0] if np.ndim(params) == 1 else out


polynomial = BuiltinModel('polynomial', POLYNOMIAL, None)
sinusoid = BuiltinModel('sinusoid', SINUSOID, 5)
gaussian = BuiltinModel('gaussian', GAUSSIAN, 4)
box = BuiltinModel('box', BOX, 4)
BUILTIN = {'polynomial': polynomial, 'sinusoid': sinusoid,
           'gaussian': gaussian, 'box': box}
