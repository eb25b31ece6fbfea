"""GPU tests of user models compiled at run time (mc3_b200.CudaModel).

(1) A CudaModel that restates a built-in formula runs the same kernel: partial rows
    byte-equal to the built-in polynomial for every launch shape (LC = 1/8/32), the
    ragged tail, uniform and per-point sigma, the non-TMA branch.
(2) Whole mcmc() runs byte-equal to the built-in model (fused and unfused, graph
    and eager, all three samplers).
(3) Chi-squared and model values against the oracle for formulas the library has
    no kernel of its own for.
(4)-(6) sample() end to end, the wavelet likelihood, error reporting.
(7) Two GPUs: the chain partition reproduces one GPU; one handle serves both.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import kernels as ok
from oracle import models as om

HORNER3 = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
HORNER5 = '''__device__ real model(real x, const real* p) {
    real y = p[4];
    for (int k = 3; k >= 0; k--) y = fma(y, x, p[k]);
    return y;
}'''
GAUSS = '''__device__ real model(real x, const real* p) {
    real d = (x - p[1]) / p[2];
    return p[0] * exp((real)-0.5 * d * d) + p[3];
}'''
SINE = '''__device__ real model(real x, const real* p) {
    return p[0] * sin((real)6.283185307179586 * x / p[1] + p[2]) + p[3] + p[4] * x;
}'''
TRAPEZOID = '''__device__ real model(real x, const real* p) {      // p[0..nparams)
    real z = fabs(x - p[1]) / p[2];                  // helpers above `model` are allowed
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}'''
BOX = '''__device__ real model(real x, const real* p) {
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''


def np_sine(p, x):
    return p[0]*np.sin(6.283185307179586*x/p[1] + p[2]) + p[3] + p[4]*x


def np_trapezoid(p, x):
    z = np.abs(x - p[1])/p[2]
    return p[3] - p[0]*np.where(z < 1, 1.0, np.where(z < p[4], (p[4] - z)/(p[4] - 1), 0.0))


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


# ---- (1) bit identity with the built-in kernel ---------------------------------
def test_partials_byte_equal_builtin_polynomial(mc3):
    from mc3_b200 import _lib
    um = mc3.CudaModel(HORNER3, 3, name='horner')
    h = um.handle(_lib.F64)
    dev = torch.device('cuda')
    rs = np.random.RandomState(11)
    st = _lib.stream_ptr()
    for n in (100000, 100037):
        xh = np.sort(rs.uniform(-2, 2, n))
        x = torch.from_numpy(xh).to(dev)
        xbuf = torch.empty(n + 1, dtype=torch.float64, device=dev)
        xbuf[1:] = x
        x_un = xbuf[1:]                                  # 8 bytes off: the non-TMA branch
        d = torch.from_numpy(om.polynomial([0.3, -1.0, 0.5], xh) + rs.normal(0, 0.1, n)).to(dev)
        w_var = torch.from_numpy(1.0/rs.uniform(0.05, 0.2, n)).to(dev)
        w_uni = torch.full((n,), 10.0, dtype=torch.float64, device=dev)
        for nchains in (7, 40, 4096):
            P = torch.from_numpy(np.array([0.3, -1.0, 0.5]) + 0.01*rs.normal(size=(nchains, 3))).to(dev)
            ns = ctypes.c_int(0)
            _lib.call('mc3b_model_chisq_plan', nchains, n, _lib.F64, ctypes.byref(ns))
            for usig, w in ((True, w_uni), (False, w_var)):
                for xx in (x, x_un):
                    o = _lib.ChisqOpts()
                    o.uniform_sigma = 1 if usig else 0
                    a = torch.full((ns.value, nchains), np.nan, dtype=torch.float64, device=dev)
                    b = torch.full_like(a, np.nan)
                    _lib.call('mc3b_model_chisq_ex', 0, _lib.F64, P.data_ptr(), 3, nchains, 3, xx.data_ptr(),
                              d.data_ptr(), w.data_ptr(), n, a.data_ptr(), nchains, ns.value, ctypes.byref(o), st)
                    _lib.call('mc3b_user_model_chisq_ex', h, P.data_ptr(), 3, nchains, xx.data_ptr(),
                              d.data_ptr(), w.data_ptr(), n, b.data_ptr(), nchains, ns.value, ctypes.byref(o), st)
                    torch.cuda.synchronize()
                    assert torch.isfinite(a).all()
                    assert torch.equal(a.view(torch.int64), b.view(torch.int64)), (n, nchains, usig, xx is x_un)
    # options of the grid sinusoid are refused
    o = _lib.ChisqOpts()
    o.work = d.data_ptr()
    with pytest.raises(_lib.Mc3bError, match='folded, work'):
        _lib.call('mc3b_user_model_chisq_ex', h, P.data_ptr(), 3, nchains, x.data_ptr(), d.data_ptr(),
                  w_var.data_ptr(), n, a.data_ptr(), nchains, ns.value, ctypes.byref(o), st)


# ---- (2) whole-run identity ------------------------------------------------------
def _linear_problem(n=4000, seed=42):
    rs = np.random.RandomState(seed)
    x = np.linspace(-1, 1, n)
    unc = rs.uniform(0.5, 1.5, n)
    data = om.polynomial([1.0, -0.5, 0.25], x) + rs.normal(0, 1, n)*unc
    return x, data, unc


@pytest.mark.parametrize('sampler', ['snooker', 'demc', 'mrw'])
def test_mcmc_byte_equal_builtin(mc3, sampler, monkeypatch):
    from mc3_b200.mcmc_driver import mcmc
    x, data, unc = _linear_problem()
    um = mc3.CudaModel(HORNER3, 3, name='horner')
    p0 = np.array([1.0, -0.5, 0.25])
    step = np.array([0.03, 0.05, 0.08])

    def run(func, graph):
        out = mcmc(data, unc, func, p0, [x], {}, np.full(3, -10.0), np.full(3, 10.0), step,
                   np.zeros(3), np.zeros(3), np.zeros(3), 256, None, 256*40, sampler, False, None,
                   False, 0.0, 0.5, 10, 1, 1.0, 1e-3, 4, 'normal', None, False, mc3.Log(verb=-1),
                   None, None, seed=17, use_graph=graph, return_population=True)
        pop = out.pop('_population')
        return out, pop
    for fuse in (True, False):
        if not fuse:
            monkeypatch.setenv('MC3B_NO_FUSE', '1')
        for graph in (True, False):
            a, pa = run(mc3.models.polynomial, graph)
            b, pb_ = run(um, graph)
            assert pb_.kind == 'cuda' and pb_.fused == fuse and not pb_.small
            for k in ('posterior', 'log_post', 'zchain', 'bestp', 'best_model'):
                assert np.array_equal(a[k], b[k]), (k, fuse, graph)
            assert a['acceptance_rate'] == b['acceptance_rate']
            assert np.array_equal(pa.naccept.cpu().numpy(), pb_.naccept.cpu().numpy())
            assert np.array_equal(pa.outbounds.cpu().numpy(), pb_.outbounds.cpu().numpy())


# ---- (3) parity against the oracle ---------------------------------------------
@pytest.mark.parametrize('case', ['gaussian', 'sine', 'trapezoid'])
@pytest.mark.parametrize('dtype', ['f64', 'f32'])
def test_chisq_and_values_vs_oracle(mc3, case, dtype):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(5)
    n = 20011
    x = np.sort(rs.uniform(-1, 1, n))
    src, npfun, p0 = {
        'gaussian': (GAUSS, om.gaussian, np.array([2.0, 0.1, 0.3, 1.0])),
        'sine': (SINE, np_sine, np.array([0.7, 1.7, 0.4, 1.0, 0.2])),
        'trapezoid': (TRAPEZOID, np_trapezoid, np.array([0.01, 0.05, 0.1, 1.0, 1.6])),
    }[case]
    um = mc3.CudaModel(src, p0.size, name=case)
    unc = rs.uniform(0.5, 1.5, n)*0.02
    data = npfun(p0, x) + rs.normal(0, 1, n)*unc
    npar = p0.size
    pop = Population(data, unc, um, p0, [x], {}, np.full(npar, 0.01), None, None, None, None, None,
                     nchains=64, sampler='demc', dtype=dtype)
    P = p0*(1 + 3e-4*rs.normal(size=(50, npar)))
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    want = np.array([ok.chisq(npfun(p, x), data, unc) for p in P])
    np.testing.assert_allclose(got, want, rtol=1e-10 if dtype == 'f64' else 1e-5)
    vals = um(P[:3], x)
    for v, p in zip(vals, P[:3]):
        np.testing.assert_allclose(v, npfun(p, x), rtol=0, atol=1e-12)
    np.testing.assert_allclose(pop.model_eval(P[0]), npfun(P[0], x), rtol=0, atol=1e-12)


# ---- (4) sample() end to end ----------------------------------------------------
def test_sample_linear_model_analytic_posterior(mc3):
    x, data, unc = _linear_problem()
    A = np.vstack([x**0, x, x**2]).T/unc[:, None]
    cov = np.linalg.inv(A.T @ A)
    mean = cov @ (A.T @ (data/unc))
    sig = np.sqrt(np.diag(cov))
    lin = mc3.CudaModel('__device__ real model(real x, const real* p) { return p[0] + p[1]*x + p[2]*x*x; }', 3,
                        name='quadratic')
    out = mc3.sample(data, unc, func=lin, params=mean + sig, indparams=[x], pstep=sig, sampler='demc',
                     nchains=1024, nsamples=1024*500, burnin=200, seed=5, fepsilon=1e-3,
                     log=mc3.Log(verb=-1))
    post, _, _ = mc3.utils.burn(out)
    assert np.all(np.abs(post.mean(axis=0) - mean) <= 0.05*sig)
    np.testing.assert_allclose(post.std(axis=0), sig, rtol=0.05)
    np.testing.assert_allclose(out['best_model'], lin(out['bestp'], x), rtol=0, atol=1e-12)
    np.testing.assert_allclose(out['best_model'], out['bestp'][0] + out['bestp'][1]*x + out['bestp'][2]*x*x,
                               rtol=0, atol=1e-12)


def test_sample_priors_shared_fixed_and_leastsq(mc3, tmp_path):
    from oracle import problems as pb
    p = pb.mcmc_case('share')
    os.chdir(tmp_path)
    kw = dict(indparams=[p['x']], pstep=p['pstep'], pmin=p['pmin'], pmax=p['pmax'], sampler='snooker',
              nchains=128, nsamples=128*100, burnin=20, seed=1, leastsq='lm', log=mc3.Log(verb=-1),
              prior=np.array([1.0, 0, 0, 0, 0]), priorlow=np.array([0.05, 0, 0, 0, 0]),
              priorup=np.array([0.05, 0, 0, 0, 0]))
    um = mc3.CudaModel(HORNER5, 5, name='poly5')
    out = mc3.sample(p['data'], p['uncert'], func=um, params=np.copy(p['params']), **kw)
    ref = mc3.sample(p['data'], p['uncert'], func=mc3.models.polynomial, params=np.copy(p['params']), **kw)
    keys = {'pnames', 'texnames', 'pstep', 'ifree', 'burnin', 'posterior', 'zchain', 'chisq', 'log_post',
            'acceptance_rate', 'bestp', 'best_chisq', 'red_chisq', 'BIC', 'best_log_post', 'best_model',
            'stddev_residuals', 'zmask', 'medianp', 'meanp', 'stdp', 'median_low_bounds',
            'median_high_bounds', 'mode', 'hpd_low_bounds', 'hpd_high_bounds', 'CRlo', 'CRhi', 'chisq_factor'}
    assert keys <= set(out)
    assert out['bestp'][3] == out['bestp'][1]                 # shared
    assert out['bestp'][4] == p['params'][4]                  # fixed
    np.testing.assert_allclose(out['best_model'], om.polynomial(out['bestp'], p['x']), rtol=0, atol=1e-12)
    for k in ('posterior', 'log_post', 'zchain', 'bestp'):
        assert np.array_equal(out[k], ref[k]), k


# ---- (5) wavelet likelihood -------------------------------------------------------
def test_wavelet_likelihood_matches_builtin_box(mc3):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(3)
    n = 1 << 14
    x = np.linspace(-0.5, 0.5, n)
    params = np.array([0.0101, 0.001, 0.1003, 1.0, 1.0, 5e-4, 1e-3])
    data = om.box(params[:4], x) + rs.normal(0, 1e-3, n)
    args = ([x], {}, np.array([2e-4, 1e-3, 1e-3, 1e-4, 0.0, 1e-4, 5e-5]), None, None, None, None, None)
    um = mc3.CudaModel(BOX, 4, name='box')
    pa = Population(data, np.full(n, 1e-3), mc3.models.box, params, *args, nchains=64, wlike=True)
    pb_ = Population(data, np.full(n, 1e-3), um, params, *args, nchains=64, wlike=True)
    P = torch.as_tensor(params*(1 + 0.01*rs.normal(size=(40, 7))), device=pa.dev)
    a, b = pa.chisq(P).cpu().numpy(), pb_.chisq(P).cpu().numpy()
    np.testing.assert_allclose(b, a, rtol=1e-10)
    np.testing.assert_allclose(b[0], ok.dwt_chisq(om.box(P[0, :4].cpu().numpy(), x), data,
                                                  P[0].cpu().numpy()), rtol=1e-9)


# ---- (6) errors ---------------------------------------------------------------------
def test_errors(mc3):
    from mc3_b200.engine import Population
    x, data, unc = _linear_problem(n=500)
    um = mc3.CudaModel(HORNER3, 3, name='horner')
    with pytest.raises(ValueError, match='takes 3 parameters'):
        mc3.sample(data, unc, func=um, params=np.ones(4), indparams=[x], pstep=np.full(4, 0.1),
                   sampler='demc', nchains=16, nsamples=1600, log=mc3.Log(verb=-1))
    bad = mc3.CudaModel('__device__ real model(real x, const real* p) {\n  return p[0] * x +;\n}', 1, name='bad')
    with pytest.raises(ValueError, match=r'model\.cu\(2\)'):
        bad(np.ones(1), x)
    with pytest.raises(ValueError, match="shard='data' needs a built-in model"):
        Population(data, unc, um, np.ones(3), [x], {}, np.full(3, 0.1), nchains=16, rank=0, world=2,
                   shard='data')


# ---- (7) two GPUs ---------------------------------------------------------------------
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
    um = mc3.CudaModel(SINE, 5, name='sine')
    out = mcmc(w['data'], w['uncert'], um, w['params'], [w['x']], {},
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


needs2 = pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')


@needs2
@pytest.mark.parametrize('sampler', ['demc', 'snooker'])
def test_two_gpus_equal_one(sampler):
    one = _launch(1, sampler)
    two = _launch(2, sampler)
    for k in ('posterior', 'zchain', 'log_post', 'bestp'):
        assert np.array_equal(one[k], two[k]), k
    assert one['acceptance_rate'] == two['acceptance_rate']


@needs2
def test_one_handle_serves_every_device(mc3):
    um = mc3.CudaModel(SINE, 5, name='sine')
    x = np.linspace(0, 3, 1000)
    p = np.array([0.7, 0.37, 0.4, 1.0, 0.2])
    with torch.cuda.device(0):
        a = um(p, x)
    with torch.cuda.device(1):
        b = um(p, x)
    assert np.array_equal(a, b)
    np.testing.assert_allclose(a, np_sine(p, x), rtol=0, atol=1e-12)
