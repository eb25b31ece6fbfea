"""GPU tests of user models of several per-point inputs (CudaModel(..., ninputs=k)).

(1) Every input slot reaches the model: a Horner quadratic in input j (the other
    inputs hold junk) gives partial rows byte-equal to the built-in polynomial for
    every launch shape (LC = 1/8/32), the ragged tail, uniform and per-point sigma,
    and the non-TMA branch (an extra input 8 bytes off alignment).
(2) Whole mcmc() runs of such a 2-input model byte-equal to the built-in model.
(3) Chi-squared and model values against numpy for a 3-input systematics transit and
    a 2-D Gaussian.
(4) sample() on a model linear in three regressors lands on the analytic posterior.
(5) The wavelet likelihood (given-model branch) and the least-squares pre-fit.
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


def horner_in(k, j):
    """A k-input model that is the quadratic p0 + p1 x + p2 x^2 (Horner) in input j."""
    args = ', '.join(f'real x{i}' for i in range(k))
    return (f'__device__ real model({args}, const real* p) '
            f'{{ return fma(fma(p[2], x{j}, p[1]), x{j}, p[0]); }}')


SYSTRANSIT = '''__device__ real trapezoid(real t, const real* p) {
    real z = fabs(t - p[1]) / p[2];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}
__device__ real model(real t, real xc, real yc, const real* p) {
    return trapezoid(t, p) * (1 + p[5]*xc + p[6]*yc + p[7]*xc*yc);
}'''
GAUSS2D = '''__device__ real model(real x, real y, const real* p) {
    real u = (x - p[1]) / p[3], v = (y - p[2]) / p[4];
    return p[0] * exp((real)-0.5 * (u*u + v*v)) + p[5];
}'''
LINEAR3 = '''__device__ real model(real a, real b, real c, const real* p) {
    return p[0] + p[1]*a + p[2]*b + p[3]*c;
}'''
BOX1 = '''__device__ real model(real x, const real* p) {
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''
BOX2 = '''__device__ real model(real x, real unused, const real* p) {
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''


def np_systransit(p, t, xc, yc):
    z = np.abs(t - p[1])/p[2]
    tr = p[3] - p[0]*np.where(z < 1, 1.0, np.where(z < p[4], (p[4] - z)/(p[4] - 1), 0.0))
    return tr*(1 + p[5]*xc + p[6]*yc + p[7]*xc*yc)


def np_gauss2d(p, x, y):
    return p[0]*np.exp(-0.5*(((x - p[1])/p[3])**2 + ((y - p[2])/p[4])**2)) + p[5]


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


# ---- (1) bit identity of every input slot -----------------------------------------
def test_every_input_slot_byte_equal_builtin_polynomial(mc3):
    from mc3_b200 import _lib
    dev = torch.device('cuda')
    rs = np.random.RandomState(12)
    st = _lib.stream_ptr()
    handles = {(k, j): mc3.CudaModel(horner_in(k, j), 3, name=f'horner{k}.{j}', ninputs=k).handle(_lib.F64)
               for k in (2, 3, 4) for j in range(k)}
    for n in (100000, 100037):
        xh = np.sort(rs.uniform(-2, 2, n))
        x = torch.from_numpy(xh).to(dev)
        xbuf = torch.empty(n + 1, dtype=torch.float64, device=dev)
        xbuf[1:] = x
        x_un = xbuf[1:]                                   # 8 bytes off: the non-TMA branch
        junk = [torch.from_numpy(rs.normal(0, 1e3, n)).to(dev) for _ in range(3)]
        jbuf = torch.empty(n + 1, dtype=torch.float64, device=dev)
        jbuf[1:] = junk[0]
        junk_un = jbuf[1:]
        d = torch.from_numpy(om.polynomial([0.3, -1.0, 0.5], xh) + rs.normal(0, 0.1, n)).to(dev)
        w_var = torch.from_numpy(1.0/rs.uniform(0.05, 0.2, n)).to(dev)
        w_uni = torch.full((n,), 10.0, dtype=torch.float64, device=dev)
        for nchains in (7, 40, 4096):
            P = torch.from_numpy(np.array([0.3, -1.0, 0.5]) + 0.01*rs.normal(size=(nchains, 3))).to(dev)
            ns = ctypes.c_int(0)
            _lib.call('mc3b_model_chisq_plan', nchains, n, _lib.F64, ctypes.byref(ns))
            for usig, w in ((True, w_uni), (False, w_var)):
                o = _lib.ChisqOpts()
                o.uniform_sigma = 1 if usig else 0
                ref = {}
                for aligned, xx in ((True, x), (False, x_un)):
                    a = torch.full((ns.value, nchains), np.nan, dtype=torch.float64, device=dev)
                    _lib.call('mc3b_model_chisq_ex', 0, _lib.F64, P.data_ptr(), 3, nchains, 3, xx.data_ptr(),
                              d.data_ptr(), w.data_ptr(), n, a.data_ptr(), nchains, ns.value, ctypes.byref(o), st)
                    ref[aligned] = a
                for (k, j), h in handles.items():
                    for aligned in (True, False):
                        others = [junk[0] if aligned else junk_un] + junk[1:]
                        xs = others[:j] + [x] + others[j:k - 1]
                        b = torch.full_like(ref[True], np.nan)
                        _lib.call('mc3b_user_model_chisq_inputs', h, P.data_ptr(), 3, nchains, _lib.ptrs(xs), k,
                                  d.data_ptr(), w.data_ptr(), n, b.data_ptr(), nchains, ns.value,
                                  ctypes.byref(o), st)
                        torch.cuda.synchronize()
                        assert torch.isfinite(ref[aligned]).all()
                        assert torch.equal(ref[aligned].view(torch.int64), b.view(torch.int64)), \
                            (n, nchains, usig, k, j, aligned)


# ---- (2) whole-run identity --------------------------------------------------------
def _linear_problem(n=4000, seed=42):
    rs = np.random.RandomState(seed)
    x = np.linspace(-1, 1, n)
    unc = rs.uniform(0.5, 1.5, n)
    data = om.polynomial([1.0, -0.5, 0.25], x) + rs.normal(0, 1, n)*unc
    return x, data, unc


@pytest.mark.parametrize('sampler', ['snooker', 'demc', 'mrw'])
def test_mcmc_two_inputs_byte_equal_builtin(mc3, sampler, monkeypatch):
    from mc3_b200.mcmc_driver import mcmc
    x, data, unc = _linear_problem()
    junk = np.random.RandomState(1).normal(0, 5, x.size)
    um = mc3.CudaModel(horner_in(2, 1), 3, name='horner2', ninputs=2)
    p0 = np.array([1.0, -0.5, 0.25])
    step = np.array([0.03, 0.05, 0.08])

    def run(func, indparams):
        out = mcmc(data, unc, func, p0, indparams, {}, np.full(3, -10.0), np.full(3, 10.0), step,
                   np.zeros(3), np.zeros(3), np.zeros(3), 256, None, 256*40, sampler, False, None,
                   False, 0.0, 0.5, 10, 1, 1.0, 1e-3, 4, 'normal', None, False, mc3.Log(verb=-1),
                   None, None, seed=17, return_population=True)
        pop = out.pop('_population')
        return out, pop
    for fuse in (True, False):
        if not fuse:
            monkeypatch.setenv('MC3B_NO_FUSE', '1')
        a, pa = run(mc3.models.polynomial, [x])
        b, pb_ = run(um, [junk, x])
        assert pb_.kind == 'cuda' and pb_.fused == fuse and not pb_.small
        for k in ('posterior', 'log_post', 'zchain', 'bestp', 'best_model'):
            assert np.array_equal(a[k], b[k]), (k, fuse)
        assert a['acceptance_rate'] == b['acceptance_rate']
        assert np.array_equal(pa.naccept.cpu().numpy(), pb_.naccept.cpu().numpy())


# ---- (3) against numpy ---------------------------------------------------------------
@pytest.mark.parametrize('case', ['systransit', 'gauss2d'])
@pytest.mark.parametrize('dtype', ['f64', 'f32'])
def test_chisq_and_values_vs_numpy(mc3, case, dtype):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(6)
    n = 20011
    if case == 'systransit':
        t = np.sort(rs.uniform(-0.2, 0.2, n))
        xs = [t, rs.normal(0, 0.3, n), rs.normal(0, 0.3, n)]
        src, npfun = SYSTRANSIT, np_systransit
        p0 = np.array([0.01, 0.02, 0.05, 1.0, 1.6, 1e-3, -2e-3, 5e-4])
    else:
        xs = [rs.uniform(-1, 1, n), rs.uniform(-1, 1, n)]
        src, npfun = GAUSS2D, np_gauss2d
        p0 = np.array([2.0, 0.1, -0.2, 0.3, 0.4, 1.0])
    um = mc3.CudaModel(src, p0.size, name=case, ninputs=len(xs))
    unc = rs.uniform(0.5, 1.5, n)*0.02
    data = npfun(p0, *xs) + rs.normal(0, 1, n)*unc
    pop = Population(data, unc, um, p0, xs, {}, np.full(p0.size, 0.01), None, None, None, None, None,
                     nchains=64, sampler='demc', dtype=dtype)
    P = p0*(1 + 3e-4*rs.normal(size=(50, p0.size)))
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    want = np.array([np.sum(((npfun(p, *xs) - data)/unc)**2) for p in P])
    np.testing.assert_allclose(got, want, rtol=1e-10 if dtype == 'f64' else 1e-5)
    vals = um(P[:3], *xs)
    for v, p in zip(vals, P[:3]):
        np.testing.assert_allclose(v, npfun(p, *xs), rtol=0, atol=1e-12)
    np.testing.assert_allclose(pop.model_eval(P[0]), npfun(P[0], *xs), rtol=0, atol=1e-12)


# ---- (4) analytic posterior ----------------------------------------------------------
def test_sample_three_regressors_analytic_posterior(mc3):
    rs = np.random.RandomState(8)
    n = 4000
    a, b = rs.normal(size=n), rs.normal(size=n)
    c = 0.5*a + rs.normal(size=n)                          # correlated with a
    unc = rs.uniform(0.5, 1.5, n)
    data = 1.0 - 0.5*a + 0.25*b + 0.75*c + rs.normal(0, 1, n)*unc
    A = np.vstack([a**0, a, b, c]).T/unc[:, None]
    cov = np.linalg.inv(A.T @ A)
    mean = cov @ (A.T @ (data/unc))
    sig = np.sqrt(np.diag(cov))
    lin = mc3.CudaModel(LINEAR3, 4, name='linear3', ninputs=3)
    out = mc3.sample(data, unc, func=lin, params=mean + sig, indparams=[a, b, c], pstep=sig, sampler='demc',
                     nchains=1024, nsamples=1024*500, burnin=200, seed=5, fepsilon=1e-3,
                     log=mc3.Log(verb=-1))
    post, _, _ = mc3.utils.burn(out)
    assert np.all(np.abs(post.mean(axis=0) - mean) <= 0.05*sig)
    np.testing.assert_allclose(post.std(axis=0), sig, rtol=0.05)
    corr = cov/np.outer(sig, sig)
    np.testing.assert_allclose(np.corrcoef(post.T), corr, rtol=0, atol=0.03)
    bp = out['bestp']
    np.testing.assert_allclose(out['best_model'], lin(bp, a, b, c), rtol=0, atol=1e-12)
    np.testing.assert_allclose(out['best_model'], bp[0] + bp[1]*a + bp[2]*b + bp[3]*c, rtol=0, atol=1e-12)


# ---- (5) wavelet likelihood, least squares ---------------------------------------------
def test_wavelet_likelihood_two_inputs_equals_one(mc3):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(3)
    n = 1 << 14
    x = np.linspace(-0.5, 0.5, n)
    params = np.array([0.0101, 0.001, 0.1003, 1.0, 1.0, 5e-4, 1e-3])
    data = om.box(params[:4], x) + rs.normal(0, 1e-3, n)
    step = np.array([2e-4, 1e-3, 1e-3, 1e-4, 0.0, 1e-4, 5e-5])
    one = mc3.CudaModel(BOX1, 4, name='box1')
    two = mc3.CudaModel(BOX2, 4, name='box2', ninputs=2)
    pa = Population(data, np.full(n, 1e-3), one, params, [x], {}, step, nchains=64, wlike=True)
    pb_ = Population(data, np.full(n, 1e-3), two, params, [x, rs.normal(size=n)], {}, step, nchains=64,
                     wlike=True)
    P = torch.as_tensor(params*(1 + 0.01*rs.normal(size=(40, 7))), device=pa.dev)
    a, b = pa.chisq(P).cpu().numpy(), pb_.chisq(P).cpu().numpy()
    np.testing.assert_allclose(b, a, rtol=1e-12)


def test_leastsq_matches_scipy(mc3):
    import scipy.optimize as so
    rs = np.random.RandomState(9)
    n = 3000
    t = np.linspace(-0.2, 0.2, n)
    xc, yc = rs.normal(0, 0.3, n), rs.normal(0, 0.3, n)
    ptrue = np.array([0.01, 0.002, 0.05, 1.0, 1.6, 1e-3, -2e-3, 5e-4])
    unc = np.full(n, 2e-4)
    data = np_systransit(ptrue, t, xc, yc) + rs.normal(0, 1, n)*unc
    start = ptrue*(1 + 0.02*rs.normal(size=ptrue.size))
    pstep = np.array([1e-3, 1e-3, 1e-3, 1e-3, 0.0, 1e-4, 1e-4, 1e-4])     # the ramp p[4] held fixed
    um = mc3.CudaModel(SYSTRANSIT, 8, name='systransit', ninputs=3)
    got = mc3.fit(data, unc, um, np.copy(start), indparams=[t, xc, yc], pstep=pstep, leastsq='lm')['bestp']
    free = pstep > 0

    def resid(q):
        p = np.copy(start)
        p[free] = q
        return (np_systransit(p, t, xc, yc) - data)/unc
    ref = so.leastsq(resid, start[free], ftol=3e-16, xtol=3e-16, gtol=3e-16)[0]
    np.testing.assert_allclose(got[free], ref, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(np.sum(resid(got[free])**2), np.sum(resid(ref)**2), rtol=1e-9)
    assert got[4] == start[4]


# ---- (6) errors ------------------------------------------------------------------------
def test_errors(mc3):
    from mc3_b200 import _lib
    from mc3_b200.engine import Population
    x, data, unc = _linear_problem(n=500)
    um = mc3.CudaModel(horner_in(2, 0), 3, name='horner2', ninputs=2)
    step = np.full(3, 0.1)
    with pytest.raises(ValueError, match="'horner2' takes 2 inputs"):
        Population(data, unc, um, np.ones(3), [x], {}, step, nchains=16)
    with pytest.raises(ValueError, match="'horner2' takes 2 inputs"):
        Population(data, unc, um, np.ones(3), [x, x, x], {}, step, nchains=16)
    with pytest.raises(ValueError, match="'horner2' takes 2 inputs"):
        Population(data, unc, um, np.ones(3), [x, x[:-1]], {}, step, nchains=16)
    with pytest.raises(ValueError, match="'horner2' takes 2 inputs"):
        Population(data, unc, um, np.ones(3), [x, np.vstack([x, x])], {}, step, nchains=16)
    with pytest.raises(ValueError, match='takes 2 input'):
        um(np.ones(3), x)
    with pytest.raises(ValueError, match="shard='data' needs a built-in model"):
        Population(data, unc, um, np.ones(3), [x, x], {}, step, nchains=16, rank=0, world=2, shard='data')

    h = um.handle(_lib.F64)
    dev = torch.device('cuda')
    dx, dd, dw = (torch.from_numpy(v).to(dev) for v in (x, data, 1.0/unc))
    P = torch.ones((16, 3), dtype=torch.float64, device=dev)
    ns = ctypes.c_int(0)
    _lib.call('mc3b_model_chisq_plan', 16, x.size, _lib.F64, ctypes.byref(ns))
    part = torch.empty((ns.value, 16), dtype=torch.float64, device=dev)
    out = torch.empty((16, x.size), dtype=torch.float64, device=dev)
    st = _lib.stream_ptr()
    with pytest.raises(_lib.Mc3bError, match='mc3b_user_model_chisq_inputs'):
        _lib.call('mc3b_user_model_chisq_ex', h, P.data_ptr(), 3, 16, dx.data_ptr(), dd.data_ptr(), dw.data_ptr(),
                  x.size, part.data_ptr(), 16, ns.value, None, st)
    with pytest.raises(_lib.Mc3bError, match='mc3b_user_model_eval_inputs'):
        _lib.call('mc3b_user_model_eval', h, P.data_ptr(), 3, 16, dx.data_ptr(), x.size, out.data_ptr(), st)
    for nx in (1, 3):
        with pytest.raises(_lib.Mc3bError, match=f'takes 2 inputs, got {nx}'):
            _lib.call('mc3b_user_model_chisq_inputs', h, P.data_ptr(), 3, 16, _lib.ptrs([dx]*nx), nx,
                      dd.data_ptr(), dw.data_ptr(), x.size, part.data_ptr(), 16, ns.value, None, st)
        with pytest.raises(_lib.Mc3bError, match=f'takes 2 inputs, got {nx}'):
            _lib.call('mc3b_user_model_eval_inputs', h, P.data_ptr(), 3, 16, _lib.ptrs([dx]*nx), nx, x.size,
                      out.data_ptr(), st)


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
    # the sinusoid with its linear term on a second input (here the abscissa itself)
    um = mc3.CudaModel('''__device__ real model(real x, real s, const real* p) {
        return p[0] * sin((real)6.283185307179586 * x / p[1] + p[2]) + p[3] + p[4] * s;
    }''', 5, name='sine2', ninputs=2)
    out = mcmc(w['data'], w['uncert'], um, w['params'], [w['x'], w['x']], {},
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
