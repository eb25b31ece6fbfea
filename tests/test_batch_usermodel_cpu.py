"""CPU-only: sample_batch with a CudaModel rejects malformed problems before it touches a
device or compiles the model, naming the problem: the wrong number of input arrays, an
input not of the data's shape, a constant count other than nconst, a parameter count other
than nparams; and it keeps the batch's fp64 chi-squared rule."""
import numpy as np
import pytest

import mc3_b200 as mc3

HORNER = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
LINEAR2 = '__device__ real model(real x1, real x2, const real* p) { return p[0] + p[1] * x1 + p[2] * x2; }'
SCALED = '''__device__ void prepare(real* p) { p[5] = p[3] * p[4]; }
__device__ real model(real x1, real x2, const real* p) { return (p[0] + p[1] * x1 + p[2] * x2) * p[5]; }'''
N = 40
X = np.linspace(0.0, 1.0, N)


def fits(func, indparams, B=3, npars=3):
    data = [1.0 + 0.5*b + 2.0*X for b in range(B)]
    return dict(data=data, uncert=[np.full(N, 0.1)]*B, func=func,
                params=np.array([[1.0 + 0.5*b, 2.0, 0.1][:npars] + [0.0]*(npars - 3) for b in range(B)]),
                indparams=indparams, pstep=np.full(npars, 0.01), sampler='demc', nchains=8, nsamples=800)


def run(args, **kw):
    args = dict(args)
    args.update(kw)
    return mc3.sample_batch(**args)


lin2 = mc3.CudaModel(LINEAR2, 3, name='lin2', ninputs=2)
scaled = mc3.CudaModel(SCALED, 3, name='scaled', ninputs=2, nconst=2, nwork=1)
horner = mc3.CudaModel(HORNER, 3, name='horner')


@pytest.mark.parametrize('func,indparams,match', [
    (lin2, [[X, X], [X], [X, X]], r'^problem 1: lin2 takes 2 input array\(s\), got 1$'),
    (lin2, [[X, X], [X, X], [X, X, X]], r'^problem 2: lin2 takes 2 input array\(s\), got 3$'),
    (lin2, [[X, X], [X, X[:-1]], [X, X]], r'^problem 1: input 1 of lin2 has shape \(39,\), the data \(40,\)$'),
    (lin2, [[X[:, None], X], [X, X], [X, X]], r'^problem 0: input 0 of lin2 has shape \(40, 1\), the data \(40,\)$'),
    (scaled, [[X, X, 1.0, 2.0], [X, X, 1.0, 2.0], [X, X, 1.0]],
     r'^problem 2: scaled takes 2 constant\(s\) after its 2 input array\(s\), got 1$'),
    (scaled, [[X, X, 1.0, 2.0], [X, X, [1.0, 2.0, 3.0]], [X, X, 1.0, 2.0]],
     r'^problem 1: scaled takes 2 constant\(s\) after its 2 input array\(s\), got 3$'),
    (horner, [[X], [X, 1.0], [X]], r'^problem 1: horner takes 1 input array\(s\), got 2$'),
    (horner, [X, X, X], r'^problem 0: horner takes 1 input array\(s\), got 40$'),
])
def test_inputs_and_constants_are_checked_per_problem(func, indparams, match):
    with pytest.raises(ValueError, match=match):
        run(fits(func, indparams))


def test_parameter_count_is_checked():
    with pytest.raises(ValueError, match=r'^problem 0: horner takes 3 parameters, got 4$'):
        run(fits(horner, [[X]]*3, npars=4))


@pytest.mark.parametrize('kw', [dict(wlike=True), dict(dtype='f32')])
def test_fp64_chisq_only(kw):
    with pytest.raises(ValueError, match=r'fp64 chi-squared likelihood only \(no wlike, no f32\)'):
        run(fits(horner, [[X]]*3), **kw)


def test_other_models_are_refused():
    with pytest.raises(ValueError, match=r'sample_batch needs a built-in model .* or a CudaModel, got'):
        run(fits(mc3.TorchModel(lambda P, x: P), [[X]]*3))
