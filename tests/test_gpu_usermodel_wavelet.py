"""GPU tests of a CudaModel in the wavelet likelihood: the model is evaluated inside the D4
kernels of its fp64 module (mc3b_user_model_dwt_chisq), never written to memory.

n = 256, 4096 and 2^14 take the last-only, the shared-memory and the register-stage
schedules.  At 2^14 the only NVRTC-compiled kernel is k_dwt_reg_model, whose arithmetic
is explicit fma: a restated built-in model gives its bits.  At the smaller sizes NVRTC may
contract the plain sums of k_dwt_pass / k_dwt_last otherwise than nvcc did.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import kernels as ok
from oracle import models as om

BOX = '''__device__ real model(real x, const real* p) {
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''
HORNER3 = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
# three inputs, two constants and a prepare step that fills the work slot
K3 = '''__device__ void prepare(real* p) { p[6] = p[4] * p[5]; }
__device__ real model(real x, real y, real z, const real* p) {
    return fma(p[0], x, fma(p[1], y * z, p[2] * sin(p[3] * x))) * p[6];
}'''
NS = (256, 4096, 1 << 14)
WAVE = np.array([1.0, 5e-4, 1e-3])      # gamma, sigma_r, sigma_w


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def _dwt(handle_or_id, P, x, data, n, nmodel, xs=None, consts=None, nk=0):
    """Wavelet chi-squared of the rows of P: a built-in model id, or a user-model handle
    through mc3b_user_model_dwt_chisq.  The workspace is sized for x.numel() points."""
    from mc3_b200 import _lib
    nb = P.shape[0]
    ws = torch.empty(max(_lib.load().mc3b_dwt_workspace(nb, x.numel()), 8)//8, dtype=torch.float64,
                     device=P.device)
    out = torch.empty(nb, dtype=torch.float64, device=P.device)
    if isinstance(handle_or_id, int):
        _lib.call('mc3b_dwt_chisq', handle_or_id, P.data_ptr(), P.shape[1], nb, P.shape[1], nmodel,
                  x.data_ptr(), None, 0, data.data_ptr(), n, ws.data_ptr(), out.data_ptr(), _lib.stream_ptr())
    else:
        xs = [x] if xs is None else xs
        _lib.call('mc3b_user_model_dwt_chisq', handle_or_id, P.data_ptr(), P.shape[1], nb, P.shape[1],
                  _lib.ptrs(xs), len(xs), _lib.ptr(consts), nk, data.data_ptr(), n, ws.data_ptr(),
                  out.data_ptr(), _lib.stream_ptr())
    return out.cpu().numpy()


def _rows_path(h, P, xs, consts, nk, data, n):
    """The path this entry point replaces: the model's rows, then mc3b_dwt_chisq(-1)."""
    from mc3_b200 import _lib
    nb = P.shape[0]
    rows = torch.empty((nb, n), dtype=torch.float64, device=P.device)
    _lib.call('mc3b_user_model_eval_consts', h, P.data_ptr(), P.shape[1], nb, _lib.ptrs(xs), len(xs),
              _lib.ptr(consts), nk, n, rows.data_ptr(), _lib.stream_ptr())
    ws = torch.empty(max(_lib.load().mc3b_dwt_workspace(nb, n), 8)//8, dtype=torch.float64, device=P.device)
    out = torch.empty(nb, dtype=torch.float64, device=P.device)
    _lib.call('mc3b_dwt_chisq', -1, P.data_ptr(), P.shape[1], nb, P.shape[1], 0, None, rows.data_ptr(), n,
              data.data_ptr(), n, ws.data_ptr(), out.data_ptr(), _lib.stream_ptr())
    return out.cpu().numpy()


@pytest.mark.parametrize('n', NS)
@pytest.mark.parametrize('case', ['box', 'polynomial'])
def test_matches_builtin_model(mc3, case, n):
    from mc3_b200 import _lib
    rs = np.random.RandomState(n)
    dev = torch.device('cuda')
    x = np.linspace(-0.5, 0.5, n)
    if case == 'box':
        src, mid, p0, npfun = BOX, mc3.models.BOX, np.array([0.0101, 0.001, 0.1003, 1.0]), om.box
    else:
        src, mid, p0, npfun = HORNER3, mc3.models.POLYNOMIAL, np.array([1.0, -0.3, 0.7]), om.polynomial
    data = npfun(p0, x) + rs.normal(0, 1e-3, n)
    full = np.concatenate([p0, WAVE])
    P = torch.as_tensor(full*(1 + 0.01*rs.normal(size=(37, full.size))), device=dev)   # 37: ragged CTAs
    xd, dd = torch.as_tensor(x, device=dev), torch.as_tensor(data, device=dev)
    h = mc3.CudaModel(src, p0.size, name=case).handle(_lib.F64)
    want = _dwt(mid, P, xd, dd, n, p0.size)
    got = _dwt(h, P, xd, dd, n, p0.size)
    if n == 1 << 14:
        assert np.array_equal(got, want)
    else:
        np.testing.assert_allclose(got, want, rtol=1e-12)
    Ph = P.cpu().numpy()
    for i in (0, 36):
        ref = ok.dwt_chisq(npfun(Ph[i, :p0.size], x), data, Ph[i])
        np.testing.assert_allclose(got[i], ref, rtol=1e-9)
        np.testing.assert_allclose(want[i], ref, rtol=1e-9)


@pytest.mark.parametrize('n', NS)
def test_inputs_constants_and_prepare_match_the_rows_path(mc3, n):
    from mc3_b200 import _lib
    rs = np.random.RandomState(7 + n)
    dev = torch.device('cuda')
    xs = [torch.as_tensor(rs.uniform(-1, 1, n), device=dev) for _ in range(3)]
    kc = torch.as_tensor([0.5, 2.5], device=dev)
    um = mc3.CudaModel(K3, 4, name='k3', ninputs=3, nconst=2, nwork=1)
    h = um.handle(_lib.F64)
    full = np.concatenate([[0.3, -0.2, 0.1, 3.0], WAVE])
    P = torch.as_tensor(full*(1 + 0.05*rs.normal(size=(45, full.size))), device=dev)
    data = torch.as_tensor(rs.normal(0, 1e-3, n), device=dev)
    got = _dwt(h, P, xs[0], data, n, 4, xs=xs, consts=kc, nk=2)
    want = _rows_path(h, P, xs, kc, 2, data, n)
    np.testing.assert_allclose(got, want, rtol=1e-12)


@pytest.mark.parametrize('sampler', ['snooker', 'demc'])
def test_whole_runs_byte_equal_builtin_box(mc3, sampler):
    from mc3_b200.mcmc_driver import mcmc
    rs = np.random.RandomState(3)
    n = 1 << 14
    x = np.linspace(-0.5, 0.5, n)
    params = np.array([0.0101, 0.001, 0.1003, 1.0, 1.0, 5e-4, 1e-3])
    data = om.box(params[:4], x) + rs.normal(0, 1e-3, n)
    unc = np.full(n, 1e-3)
    step = np.array([2e-4, 1e-3, 1e-3, 1e-4, 0.0, 1e-4, 5e-5])
    pmin = np.array([-1, -1, 0, 0, -10, 0, 0.0])
    pmax = np.array([1, 1, 1, 2, 10, 1, 1.0])
    um = mc3.CudaModel(BOX, 4, name='box')

    def run(func, graph):
        out = mcmc(data, unc, func, np.copy(params), [x], {}, pmin, pmax, step,
                   np.zeros(7), np.zeros(7), np.zeros(7), 64, None, 64*30, sampler, True, None,
                   False, 0.0, 0.5, 5, 1, 1.0, 1e-3, 4, 'normal', None, False, mc3.Log(verb=-1),
                   None, None, seed=11, use_graph=graph, return_population=True)
        pop = out.pop('_population')
        return out, pop
    for graph in (True, False):
        a, pa = run(mc3.models.box, graph)
        b, pb_ = run(um, graph)
        assert pb_.kind == 'cuda' and pb_.wlike
        for k in ('posterior', 'log_post', 'zchain', 'bestp'):
            assert np.array_equal(a[k], b[k]), (k, graph)


def test_population_chisq_writes_no_model_rows(mc3):
    from mc3_b200 import _lib
    from mc3_b200.engine import Population
    rs = np.random.RandomState(5)
    n, nb = 1 << 16, 1024
    x = np.linspace(-0.5, 0.5, n)
    params = np.array([0.0101, 0.001, 0.1003, 1.0, 1.0, 5e-4, 1e-3])
    data = om.box(params[:4], x) + rs.normal(0, 1e-3, n)
    step = np.array([2e-4, 1e-3, 1e-3, 1e-4, 0.0, 1e-4, 5e-5])
    pop = Population(data, np.full(n, 1e-3), mc3.CudaModel(BOX, 4, name='box'), params, [x], {}, step,
                     None, None, None, None, None, nchains=64, wlike=True)
    P = torch.as_tensor(params*(1 + 0.01*rs.normal(size=(nb, 7))), device=pop.dev)
    pop.chisq(P[:8])                                # handles loaded, small workspaces made
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = pop.chisq(P).cpu().numpy()
    peak = torch.cuda.max_memory_allocated() - base
    ws = _lib.load().mc3b_dwt_workspace(nb, n)
    rows = nb*n*8                                   # 512 MB
    assert peak <= ws + (16 << 20), (peak, ws)
    assert peak < rows//4, (peak, rows)
    np.testing.assert_allclose(out[0], ok.dwt_chisq(om.box(P[0, :4].cpu().numpy(), x), data,
                                                    P[0].cpu().numpy()), rtol=1e-9)


def test_errors(mc3):
    from mc3_b200 import _lib
    dev = torch.device('cuda')
    n = 1024
    x = torch.linspace(-0.5, 0.5, n, dtype=torch.float64, device=dev)
    data = torch.zeros(n, dtype=torch.float64, device=dev)
    P = torch.as_tensor(np.tile(np.array([0.01, 0.0, 0.1, 1.0, 1.0, 5e-4, 1e-3]), (4, 1)), device=dev)
    um = mc3.CudaModel(BOX, 4, name='box')
    with pytest.raises(_lib.Mc3bError, match='fp64 module'):
        _dwt(um.handle(_lib.F32), P, x, data, n, 4)
    with pytest.raises(_lib.Mc3bError, match='takes 1 inputs, got 2'):
        _dwt(um.handle(_lib.F64), P, x, data, n, 4, xs=[x, x])
    kc = torch.ones(1, dtype=torch.float64, device=dev)
    with pytest.raises(_lib.Mc3bError, match='takes 0 constants, got 1'):
        _dwt(um.handle(_lib.F64), P, x, data, n, 4, consts=kc, nk=1)
    with pytest.raises(_lib.Mc3bError, match='n = 2.k'):
        _dwt(um.handle(_lib.F64), P, x, data, n - 24, 4)
    with pytest.raises(_lib.Mc3bError, match='npars - 3'):
        _dwt(um.handle(_lib.F64), P[:, 1:].contiguous(), x, data, n, 4)
