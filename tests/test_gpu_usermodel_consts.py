"""GPU tests of user models of run-time constants and a prepare step (CudaModel(...,
nconst=m, nwork=w)).

(1) A Gaussian whose prepare hoists 1/sigma into a work slot does the arithmetic of the
    built-in GaussModel<double>: partial rows byte-equal for every launch shape
    (LC = 1/8/32), the ragged tail, uniform and per-point sigma and the non-TMA branch,
    and whole mcmc() runs byte-equal (fused and unfused, graph and eager, three samplers).
(2) A constant is a fixed parameter: a Horner quadratic whose top coefficient is a
    constant samples exactly as the built-in polynomial with that coefficient fixed.
(3) Constant values are run-time data: two populations share one module.
(4) Chi-squared and model values against numpy: a 3-input systematics transit whose
    period is a constant, the sinusoid with prepare, a model of a 1-D constant array.
(5) sample() with the shape probe and the least-squares pre-fit, the wavelet likelihood.
(6) Error reporting.
(7) Two GPUs: the chain partition reproduces one GPU.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import models as om

GAUSS = '''__device__ void prepare(real* p) { p[4] = 1 / p[2]; }      // once per chain and launch
__device__ real model(real x, const real* p) {
    real d = (x - p[1]) * p[4];
    return fma(p[0], exp((real)(-0.5) * d * d), p[3]);
}'''
HORNER_C = '''__device__ real model(real x, const real* p) {   // p[2]: a constant
    return fma(fma(p[2], x, p[1]), x, p[0]);
}'''
# p[8] = period (a constant), p[9] = 1/period (work)
PTRANSIT = '''__device__ void prepare(real* p) { p[9] = 1 / p[8]; }
__device__ real model(real t, real xc, real yc, const real* p) {
    real dt = t - p[1];
    dt -= p[8] * rint(dt * p[9]);
    real z = fabs(dt) / p[2];
    real tr = p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
    return tr * (1 + p[5]*xc + p[6]*yc + p[7]*xc*yc);
}'''
SINE_P = '''__device__ void prepare(real* p) { p[5] = (real)6.283185307179586 / p[1]; }
__device__ real model(real x, const real* p) {
    return p[0] * sin(fma(x, p[5], p[2])) + p[3] + p[4] * x;
}'''
# p[2..4]: baseline coefficients, given as one 1-D array
LINE_ARR = '''__device__ real model(real x, const real* p) {
    return p[0] * exp(-x * x / p[1]) + (p[2] + x * (p[3] + x * p[4]));
}'''
BOX1 = '''__device__ real model(real x, const real* p) {
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''
BOXC = '''__device__ real model(real x, const real* p) {      // the baseline p[3] is a constant
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''


def np_ptransit(p, t, xc, yc, period):
    dt = t - p[1]
    dt = dt - period*np.rint(dt/period)
    z = np.abs(dt)/p[2]
    tr = p[3] - p[0]*np.where(z < 1, 1.0, np.where(z < p[4], (p[4] - z)/(p[4] - 1), 0.0))
    return tr*(1 + p[5]*xc + p[6]*yc + p[7]*xc*yc)


def np_sine(p, x):
    return p[0]*np.sin(2*np.pi*x/p[1] + p[2]) + p[3] + p[4]*x


def np_line_arr(p, x, c):
    return p[0]*np.exp(-x*x/p[1]) + (c[0] + x*(c[1] + x*c[2]))


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


# ---- (1) the Gaussian with prepare is the built-in Gaussian ---------------------------
def test_gauss_prepare_partial_rows_byte_equal_builtin(mc3):
    from mc3_b200 import _lib
    dev = torch.device('cuda')
    rs = np.random.RandomState(12)
    st = _lib.stream_ptr()
    h = mc3.CudaModel(GAUSS, 4, name='gauss', nwork=1).handle(_lib.F64)
    p0 = np.array([2.0, 0.1, 0.3, 1.0])
    for n in (100000, 100037):
        xh = np.sort(rs.uniform(-2, 2, n))
        x = torch.from_numpy(xh).to(dev)
        xbuf = torch.empty(n + 1, dtype=torch.float64, device=dev)
        xbuf[1:] = x
        x_un = xbuf[1:]                                   # 8 bytes off: the non-TMA branch
        d = torch.from_numpy(om.gaussian(p0, xh) + rs.normal(0, 0.1, n)).to(dev)
        w_var = torch.from_numpy(1.0/rs.uniform(0.05, 0.2, n)).to(dev)
        w_uni = torch.full((n,), 10.0, dtype=torch.float64, device=dev)
        for nchains in (7, 40, 4096):
            P = torch.from_numpy(p0 + 0.01*rs.normal(size=(nchains, 4))).to(dev)
            ns = ctypes.c_int(0)
            _lib.call('mc3b_model_chisq_plan', nchains, n, _lib.F64, ctypes.byref(ns))
            for usig, w in ((True, w_uni), (False, w_var)):
                o = _lib.ChisqOpts()
                o.uniform_sigma = 1 if usig else 0
                for xx in (x, x_un):
                    a = torch.full((ns.value, nchains), np.nan, dtype=torch.float64, device=dev)
                    _lib.call('mc3b_model_chisq_ex', 2, _lib.F64, P.data_ptr(), 4, nchains, 4, xx.data_ptr(),
                              d.data_ptr(), w.data_ptr(), n, a.data_ptr(), nchains, ns.value, ctypes.byref(o), st)
                    b = torch.full_like(a, np.nan)
                    _lib.call('mc3b_user_model_chisq_consts', h, P.data_ptr(), 4, nchains, _lib.ptrs([xx]), 1,
                              None, 0, d.data_ptr(), w.data_ptr(), n, b.data_ptr(), nchains, ns.value,
                              ctypes.byref(o), st)
                    c = torch.full_like(a, np.nan)             # a model of no constants: the plain entry point
                    _lib.call('mc3b_user_model_chisq_ex', h, P.data_ptr(), 4, nchains, xx.data_ptr(),
                              d.data_ptr(), w.data_ptr(), n, c.data_ptr(), nchains, ns.value, ctypes.byref(o), st)
                    torch.cuda.synchronize()
                    assert torch.isfinite(a).all()
                    assert torch.equal(a.view(torch.int64), b.view(torch.int64)), (n, nchains, usig)
                    assert torch.equal(a.view(torch.int64), c.view(torch.int64)), (n, nchains, usig)


def _gauss_problem(n=4000, seed=42):
    rs = np.random.RandomState(seed)
    x = np.linspace(-1, 1, n)
    unc = rs.uniform(0.5, 1.5, n)
    data = om.gaussian([2.0, 0.1, 0.3, 1.0], x) + rs.normal(0, 1, n)*unc
    return x, data, unc


def _mcmc(mc3, data, unc, func, p0, indparams, step, sampler, graph=True):
    from mc3_b200.mcmc_driver import mcmc
    npars = p0.size
    out = mcmc(data, unc, func, p0, indparams, {}, np.full(npars, -10.0), np.full(npars, 10.0), step,
               np.zeros(npars), np.zeros(npars), np.zeros(npars), 256, None, 256*40, sampler, False, None,
               False, 0.0, 0.5, 10, 1, 1.0, 1e-3, 4, 'normal', None, False, mc3.Log(verb=-1),
               None, None, seed=17, use_graph=graph, return_population=True)
    return out, out.pop('_population')


@pytest.mark.parametrize('sampler', ['snooker', 'demc', 'mrw'])
def test_mcmc_gauss_prepare_byte_equal_builtin(mc3, sampler, monkeypatch):
    x, data, unc = _gauss_problem()
    um = mc3.CudaModel(GAUSS, 4, name='gauss', nwork=1)
    p0 = np.array([2.0, 0.1, 0.3, 1.0])
    step = np.array([0.05, 0.01, 0.01, 0.02])
    for fuse in (True, False):
        if not fuse:
            monkeypatch.setenv('MC3B_NO_FUSE', '1')
        for graph in (True, False):
            a, pa = _mcmc(mc3, data, unc, mc3.models.gaussian, p0, [x], step, sampler, graph)
            b, pb_ = _mcmc(mc3, data, unc, um, p0, [x], step, sampler, graph)
            assert pb_.kind == 'cuda' and pb_.fused == fuse and not pb_.small
            for k in ('posterior', 'log_post', 'zchain', 'bestp', 'best_model'):
                assert np.array_equal(a[k], b[k]), (k, fuse, graph)
            assert a['acceptance_rate'] == b['acceptance_rate']
            assert np.array_equal(pa.naccept.cpu().numpy(), pb_.naccept.cpu().numpy())


# ---- (2) a constant is a fixed parameter ------------------------------------------------
@pytest.mark.parametrize('sampler', ['snooker', 'demc', 'mrw'])
def test_constant_samples_as_a_fixed_parameter(mc3, sampler):
    rs = np.random.RandomState(4)
    n = 4000
    x = np.linspace(-1, 1, n)
    unc = rs.uniform(0.5, 1.5, n)
    data = om.polynomial([1.0, -0.5, 0.25], x) + rs.normal(0, 1, n)*unc
    um = mc3.CudaModel(HORNER_C, 2, name='horner_c', nconst=1)
    a, _ = _mcmc(mc3, data, unc, mc3.models.polynomial, np.array([1.0, -0.5, 0.25]), [x],
                 np.array([0.03, 0.05, 0.0]), sampler)
    b, pb_ = _mcmc(mc3, data, unc, um, np.array([1.0, -0.5]), [x, 0.25], np.array([0.03, 0.05]), sampler)
    assert pb_.kind == 'cuda' and pb_.fused
    for k in ('posterior', 'log_post', 'zchain'):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a['bestp'][:2], b['bestp'])


# ---- (3) run-time values -------------------------------------------------------------
@pytest.mark.parametrize('dtype', ['f64', 'f32'])
def test_constant_values_share_one_module(mc3, dtype):
    from mc3_b200 import _lib
    from mc3_b200.engine import Population
    rs = np.random.RandomState(2)
    n = 20011
    x = np.sort(rs.uniform(-1, 1, n))
    unc = np.full(n, 0.05)
    um = mc3.CudaModel(HORNER_C, 2, name='horner_c_' + dtype, nconst=1)
    pops = []
    for i, c2 in enumerate((0.25, -3.5)):
        data = om.polynomial([1.0, -0.5, c2], x) + rs.normal(0, 0.05, n)
        pop = Population(data, unc, um, np.array([1.0, -0.5]), [x, c2], {}, np.full(2, 0.01), None, None, None,
                         None, None, nchains=64, sampler='demc', dtype=dtype)
        if i == 0:
            stats = {}
            um.handle(pop.dtype, stats)
            assert stats['origin'] == 'memory'
        pops.append(pop)
        P = np.array([1.0, -0.5])*(1 + 1e-3*rs.normal(size=(30, 2)))
        got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
        want = np.array([np.sum(((om.polynomial([p[0], p[1], c2], x) - data)/unc)**2) for p in P])
        np.testing.assert_allclose(got, want, rtol=1e-10 if dtype == 'f64' else 1e-5)
        np.testing.assert_allclose(um(P[0], x, c2), om.polynomial([P[0, 0], P[0, 1], c2], x), rtol=0, atol=1e-12)
    assert pops[0].jit.value == pops[1].jit.value and pops[0].jit_eval.value == pops[1].jit_eval.value


# ---- (4) against numpy -------------------------------------------------------------------
def _case(case, rs, n):
    if case == 'ptransit':
        t = np.sort(rs.uniform(-2.0, 2.0, n))
        xs = [t, rs.normal(0, 0.3, n), rs.normal(0, 0.3, n)]
        period = 0.7314
        um_args = dict(nparams=8, ninputs=3, nconst=1, nwork=1)
        p0 = np.array([0.01, 0.02, 0.05, 1.0, 1.6, 1e-3, -2e-3, 5e-4])
        return PTRANSIT, um_args, xs, [period], p0, lambda p: np_ptransit(p, *xs, period)
    if case == 'sine':
        x = np.sort(rs.uniform(-1, 1, n))
        p0 = np.array([0.7, 1.7, 0.4, 1.0, 0.2])
        return SINE_P, dict(nparams=5, nwork=1), [x], [], p0, lambda p: np_sine(p, x)
    x = np.sort(rs.uniform(-1, 1, n))
    c = np.array([1.0, 0.3, -0.2])
    p0 = np.array([2.0, 0.1])
    return LINE_ARR, dict(nparams=2, nconst=3), [x], [c], p0, lambda p: np_line_arr(p, x, c)


@pytest.mark.parametrize('case', ['ptransit', 'sine', 'array'])
@pytest.mark.parametrize('dtype', ['f64', 'f32'])
def test_chisq_and_values_vs_numpy(mc3, case, dtype):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(6)
    n = 20011
    src, kw, xs, consts, p0, npfun = _case(case, rs, n)
    um = mc3.CudaModel(src, name=case, **kw)
    unc = rs.uniform(0.5, 1.5, n)*0.02
    data = npfun(p0) + rs.normal(0, 1, n)*unc
    pop = Population(data, unc, um, p0, xs + consts, {}, np.full(p0.size, 0.01), None, None, None, None, None,
                     nchains=64, sampler='demc', dtype=dtype)
    P = p0*(1 + 3e-4*rs.normal(size=(50, p0.size)))
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    want = np.array([np.sum(((npfun(p) - data)/unc)**2) for p in P])
    np.testing.assert_allclose(got, want, rtol=1e-10 if dtype == 'f64' else 1e-5)
    vals = um(P[:3], *xs, *consts)
    for v, p in zip(vals, P[:3]):
        np.testing.assert_allclose(v, npfun(p), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(pop.model_eval(P[0]), npfun(P[0]), rtol=1e-10, atol=1e-12)


def test_gauss_prepare_f32_vs_oracle(mc3):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(7)
    n = 20011
    x = np.sort(rs.uniform(-1, 1, n))
    p0 = np.array([2.0, 0.1, 0.3, 1.0])
    unc = rs.uniform(0.5, 1.5, n)*0.02
    data = om.gaussian(p0, x) + rs.normal(0, 1, n)*unc
    pop = Population(data, unc, mc3.CudaModel(GAUSS, 4, name='gauss', nwork=1), p0, [x], {}, np.full(4, 0.01),
                     None, None, None, None, None, nchains=64, sampler='demc', dtype='f32')
    P = p0*(1 + 3e-4*rs.normal(size=(50, 4)))
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    want = np.array([np.sum(((om.gaussian(p, x) - data)/unc)**2) for p in P])
    np.testing.assert_allclose(got, want, rtol=1e-5)


# ---- (5) sample(), least squares, wavelet likelihood ---------------------------------------
def test_sample_and_leastsq_with_a_constant_period(mc3):
    import scipy.optimize as so
    rs = np.random.RandomState(9)
    n = 3000
    t = np.linspace(-1.5, 1.5, n)
    xc, yc = rs.normal(0, 0.3, n), rs.normal(0, 0.3, n)
    period = 0.7314
    ptrue = np.array([0.01, 0.002, 0.05, 1.0, 1.6, 1e-3, -2e-3, 5e-4])
    unc = np.full(n, 2e-4)
    data = np_ptransit(ptrue, t, xc, yc, period) + rs.normal(0, 1, n)*unc
    start = ptrue*(1 + 0.02*rs.normal(size=ptrue.size))
    pstep = np.array([1e-3, 1e-3, 1e-3, 1e-3, 0.0, 1e-4, 1e-4, 1e-4])     # the ramp p[4] held fixed
    um = mc3.CudaModel(PTRANSIT, 8, name='ptransit', ninputs=3, nconst=1, nwork=1)
    got = mc3.fit(data, unc, um, np.copy(start), indparams=[t, xc, yc, period], pstep=pstep, leastsq='lm')['bestp']
    free = pstep > 0

    def resid(q):
        p = np.copy(start)
        p[free] = q
        return (np_ptransit(p, t, xc, yc, period) - data)/unc
    ref = so.leastsq(resid, start[free], ftol=3e-16, xtol=3e-16, gtol=3e-16)[0]
    np.testing.assert_allclose(got[free], ref, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(np.sum(resid(got[free])**2), np.sum(resid(ref)**2), rtol=1e-9)

    out = mc3.sample(data, unc, func=um, params=np.copy(start), indparams=[t, xc, yc, period], pstep=pstep,
                     sampler='demc', nchains=256, nsamples=256*60, burnin=20, seed=5, leastsq='lm',
                     log=mc3.Log(verb=-1))
    bp = out['bestp']
    assert np.all(np.isfinite(out['posterior']))
    np.testing.assert_allclose(out['best_model'], np_ptransit(bp, t, xc, yc, period), rtol=0, atol=1e-12)
    np.testing.assert_allclose(out['best_model'], um(bp, t, xc, yc, period), rtol=0, atol=1e-12)


def test_wavelet_likelihood_constant_equals_parameter(mc3):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(3)
    n = 1 << 14
    x = np.linspace(-0.5, 0.5, n)
    params = np.array([0.0101, 0.001, 0.1003, 1.0, 1.0, 5e-4, 1e-3])
    data = om.box(params[:4], x) + rs.normal(0, 1e-3, n)
    step = np.array([2e-4, 1e-3, 1e-3, 1e-4, 0.0, 1e-4, 5e-5])
    one = mc3.CudaModel(BOX1, 4, name='box1')
    cst = mc3.CudaModel(BOXC, 3, name='boxc', nconst=1)
    keep = [0, 1, 2, 4, 5, 6]
    pa = Population(data, np.full(n, 1e-3), one, params, [x], {}, step, nchains=64, wlike=True)
    pb_ = Population(data, np.full(n, 1e-3), cst, params[keep], [x, params[3]], {}, step[keep], nchains=64,
                     wlike=True)
    P = params*(1 + 0.01*rs.normal(size=(40, 7)))
    P[:, 3] = params[3]
    a = pa.chisq(torch.as_tensor(P, device=pa.dev)).cpu().numpy()
    b = pb_.chisq(torch.as_tensor(np.ascontiguousarray(P[:, keep]), device=pb_.dev)).cpu().numpy()
    np.testing.assert_allclose(b, a, rtol=1e-12)


# ---- (6) errors --------------------------------------------------------------------------
def test_errors(mc3):
    from mc3_b200 import _lib
    from mc3_b200.engine import Population
    rs = np.random.RandomState(1)
    x = np.linspace(-1, 1, 500)
    unc = np.full(500, 0.1)
    data = om.polynomial([1.0, -0.5, 0.25], x) + rs.normal(0, 0.1, 500)
    um = mc3.CudaModel(HORNER_C, 2, name='horner_c', nconst=1)
    step = np.full(2, 0.1)
    for ind, got in (([x], 0), ([x, 1.0, 2.0], 2), ([x, [1.0, 2.0]], 2)):
        with pytest.raises(ValueError, match=f'horner_c takes 1 constant.*got {got}'):
            Population(data, unc, um, np.ones(2), ind, {}, step, nchains=16)
    with pytest.raises(ValueError, match='takes 1 constant.*got 0'):
        um(np.ones(2), x)
    with pytest.raises(ValueError, match='1-D'):
        um(np.ones(2), x, np.ones((2, 2)))

    h = um.handle(_lib.F64)
    dev = torch.device('cuda')
    dx, dd, dw = (torch.from_numpy(v).to(dev) for v in (x, data, 1.0/unc))
    dk = torch.tensor([0.25], dtype=torch.float64, device=dev)
    P = torch.ones((16, 2), dtype=torch.float64, device=dev)
    ns = ctypes.c_int(0)
    _lib.call('mc3b_model_chisq_plan', 16, x.size, _lib.F64, ctypes.byref(ns))
    part = torch.empty((ns.value, 16), dtype=torch.float64, device=dev)
    out = torch.empty((16, x.size), dtype=torch.float64, device=dev)
    st = _lib.stream_ptr()
    with pytest.raises(_lib.Mc3bError, match='mc3b_user_model_chisq_consts'):
        _lib.call('mc3b_user_model_chisq_ex', h, P.data_ptr(), 2, 16, dx.data_ptr(), dd.data_ptr(), dw.data_ptr(),
                  x.size, part.data_ptr(), 16, ns.value, None, st)
    with pytest.raises(_lib.Mc3bError, match='mc3b_user_model_chisq_consts'):
        _lib.call('mc3b_user_model_chisq_inputs', h, P.data_ptr(), 2, 16, _lib.ptrs([dx]), 1, dd.data_ptr(),
                  dw.data_ptr(), x.size, part.data_ptr(), 16, ns.value, None, st)
    with pytest.raises(_lib.Mc3bError, match='mc3b_user_model_eval_consts'):
        _lib.call('mc3b_user_model_eval', h, P.data_ptr(), 2, 16, dx.data_ptr(), x.size, out.data_ptr(), st)
    with pytest.raises(_lib.Mc3bError, match='mc3b_user_model_eval_consts'):
        _lib.call('mc3b_user_model_eval_inputs', h, P.data_ptr(), 2, 16, _lib.ptrs([dx]), 1, x.size,
                  out.data_ptr(), st)
    with pytest.raises(_lib.Mc3bError, match='takes 1 constants, got 2'):
        _lib.call('mc3b_user_model_chisq_consts', h, P.data_ptr(), 2, 16, _lib.ptrs([dx]), 1, dk.data_ptr(), 2,
                  dd.data_ptr(), dw.data_ptr(), x.size, part.data_ptr(), 16, ns.value, None, st)
    with pytest.raises(_lib.Mc3bError, match='null pointer'):
        _lib.call('mc3b_user_model_eval_consts', h, P.data_ptr(), 2, 16, _lib.ptrs([dx]), 1, None, 1, x.size,
                  out.data_ptr(), st)
    _lib.call('mc3b_user_model_eval_consts', h, P.data_ptr(), 2, 16, _lib.ptrs([dx]), 1, dk.data_ptr(), 1, x.size,
              out.data_ptr(), st)
    np.testing.assert_allclose(out[0].cpu().numpy(), om.polynomial([1.0, 1.0, 0.25], x), rtol=0, atol=1e-14)


# ---- (7) two GPUs -------------------------------------------------------------------------
NCH = 1024


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(rank, world, port, sampler, q):
    import torch.distributed as dist
    import mc3_b200 as mc3
    from mc3_b200 import workloads
    from mc3_b200.mcmc_driver import mcmc
    torch.cuda.set_device(rank)
    if world > 1:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    w = workloads.config2(n=20011)
    # the sinusoid with prepare, and its slope scaled by a constant (here 1)
    um = mc3.CudaModel('''__device__ void prepare(real* p) { p[6] = (real)6.283185307179586 / p[1]; }
    __device__ real model(real x, const real* p) {
        return p[0] * sin(fma(x, p[6], p[2])) + p[3] + p[5] * p[4] * x;
    }''', 5, name='sine_c', nconst=1, nwork=1)
    out = mcmc(w['data'], w['uncert'], um, w['params'], [w['x'], 1.0], {},
               w['pmin'], w['pmax'], w['pstep'], w['prior'], w['priorlow'], w['priorup'],
               NCH, None, NCH*24, sampler, False, None, True, 0.0, 0.5, 6, 2,
               1.0, 0.01, 4, 'normal', None, False, mc3.Log(verb=-1), None, None,
               seed=21, rank=rank, world=world, shard='chains', plan_chains=NCH, return_population=True)
    pop = out.pop('_population')
    if rank == 0:
        q.put({k: out[k] for k in ('posterior', 'zchain', 'log_post', 'bestp', 'acceptance_rate')})
        q.close()
        q.join_thread()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        pop.close()
        del pop, out
        dist.destroy_process_group()


def _launch(world, sampler):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_run, args=(r, world, port, sampler, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    res = q.get(timeout=300)
    for pr in procs:
        pr.join(120)
        assert pr.exitcode == 0, 'a rank did not shut down cleanly'
    return res


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
@pytest.mark.parametrize('sampler', ['demc', 'snooker'])
def test_two_gpus_equal_one(sampler):
    one = _launch(1, sampler)
    two = _launch(2, sampler)
    for k in ('posterior', 'zchain', 'log_post', 'bestp'):
        assert np.array_equal(one[k], two[k]), k
    assert one['acceptance_rate'] == two['acceptance_rate']
