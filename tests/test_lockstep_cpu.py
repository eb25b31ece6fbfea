"""CPU tests of oracle/lockstep.py, the numpy restatement of a production-mode
generation that tests/test_gpu_lockstep.py checks the CUDA sampler against.

(1) Philox4x32-10 against Random123's known answers; u01 and ubelow at the ends of
    their ranges.
(2) The index rules of the draws over many generations.
(3) The anchor: fed the reference's own recorded draws (tests/golden/mcmc_*.npz,
    made from the real reference by oracle/make_golden.py) in the reference's
    sequential order, with chi-squared from oracle.kernels, the restatement's
    propose / metropolis reproduce the reference's trajectory, so that the step code
    the GPU check uses is tied to the reference and not only to the CUDA source.
"""
import os

import numpy as np
import pytest

from oracle import kernels as ok
from oracle import lockstep as ls
from oracle import models as om
from oracle import problems as pb

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _hex(words):
    return ' '.join(f'{int(w):08x}' for w in words)


@pytest.mark.parametrize('key, ctr, want', [
    ((0, 0), (0, 0, 0, 0), '6627e8d5 e169c58d bc57ac4c 9b00dbd8'),
    ((0xffffffff, 0xffffffff), (0xffffffff,)*4, '408f276d 41c83b0e a20bc7c6 6d5451fd'),
    ((0xa4093822, 0x299f31d0), (0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344),
     'd16cfe09 94fdcceb 5001e420 24126ea1'),
])
def test_philox_known_answers(key, ctr, want):
    seed = key[0] | (key[1] << 32)
    assert _hex(ls.philox(seed, *ctr)) == want
    # vectorised over counters: every element is the scalar answer
    w = ls.philox(seed, np.full(3, ctr[0]), ctr[1], ctr[2], ctr[3])
    assert all(_hex(col) == want for col in zip(*w))


def test_u01_exact_at_range_ends():
    M = 0xffffffff
    assert ls.u01(0, 0) == 0.0
    assert ls.u01(0, 64) == 2.0**-53                    # the smallest step: b>>6 = 1
    assert ls.u01(32, 0) == 2.0**-27                    # a>>5 = 1
    assert ls.u01(M, M) == 1.0 - 2.0**-53               # largest value, below 1
    assert ls.u01(0x80000000, 0) == 0.5
    a = np.array([0, 31, 32, M], dtype=np.uint64)
    b = np.array([63, 64, M, M], dtype=np.uint64)
    want = [((int(x) >> 5)*2**26 + (int(y) >> 6))/2.0**53 for x, y in zip(a, b)]
    assert np.array_equal(ls.u01(a, b), want)


def test_ubelow_exact_at_range_ends():
    M = 0xffffffff
    for n in (1, 2, 3, 7, 4096, 2**31 - 1, 2**32 + 5, 2**62 + 12345, 2**63 - 1):
        assert ls.ubelow(0, 0, n) == 0
        assert ls.ubelow(M, M, n) == n - 1             # (2^64 - 1) n >> 64
        assert ls.ubelow(0x80000000, 0, n) == n >> 1
        assert ls.ubelow(0, 1, n) == (n >> 64)          # 1 * n < 2^64: 0
    rs = np.random.RandomState(1)
    a = rs.randint(0, 2**32, 1000, dtype=np.uint64)
    b = rs.randint(0, 2**32, 1000, dtype=np.uint64)
    for n in (3, 1000, 2**40 + 1):
        got = ls.ubelow(a, b, n)
        want = [((int(x) << 32 | int(y))*n) >> 64 for x, y in zip(a, b)]
        assert np.array_equal(got, want)
        assert got.min() >= 0 and got.max() < n


@pytest.mark.parametrize('nchains', [3, 4, 7, 64, 4096])
def test_demc_partner_rules(nchains):
    c = np.arange(nchains)
    for gen in range(0, 4000*4//nchains + 1):
        d = ls.chain_draws(12345, 'demc', nchains, gen, 0)
        r1, r2 = d['a'], d['b']
        assert np.all((r1 >= 0) & (r1 < nchains) & (r2 >= 0) & (r2 < nchains))
        assert np.all(r1 != c)
        assert np.all((r2 != c) & (r2 != r1))
        assert np.all((d['u'] >= 0) & (d['u'] < 1))


@pytest.mark.parametrize('zsize', [2, 3, 70, 4096*10 + 4096*7])
def test_snooker_index_rules(zsize):
    n = 256
    hits = 0
    for gen in range(40):
        d = ls.chain_draws(777 + zsize, 'snooker', n, gen, zsize)
        i1, i2, iz = d['a'], d['b'], d['iz']
        assert np.all((i1 >= 0) & (i1 < zsize) & (i2 >= 0) & (i2 < zsize) & (iz >= 0) & (iz < zsize))
        assert np.all(i2 != i1)
        assert np.all((d['gs'] >= 1.2) & (d['gs'] < 2.2))
        hits += int(np.sum(d['usj'] < 0.1))
    assert 0.07*40*n < hits < 0.13*40*n                 # snooker jumps: 10 % of the draws


def test_draws_depend_on_chain_and_generation_only():
    """A chain's draws do not depend on which other chains are drawn with it, and the
    high word of the generation is part of the counter."""
    full = ls.chain_draws(9, 'snooker', 64, 5, 640)
    part = ls.chain_draws(9, 'snooker', 64, 5, 640, chains=[3, 40])
    for k in full:
        assert np.array_equal(full[k][[3, 40]], part[k])
    nf = ls.chain_normals(9, 64, 5, np.full(5, 0.1), np.arange(5))
    npart = ls.chain_normals(9, 64, 5, np.full(5, 0.1), np.arange(5), chains=[3, 40])
    assert np.array_equal(nf[[3, 40]], npart)
    hi = ls.chain_draws(9, 'snooker', 64, 5 + (1 << 32), 640)
    assert not np.array_equal(full['u'], hi['u'])


def _data_chisq(p, model):
    if p['wlike']:
        return lambda q: ok.dwt_chisq(model(q[:-3], p['x']), p['data'], q)
    return lambda q: ok.chisq(model(q, p['x']), p['data'], p['uncert'])


@pytest.mark.parametrize('case', pb.MCMC_CASES)
@pytest.mark.parametrize('sampler', pb.SAMPLERS)
def test_sequential_restatement_retraces_reference(case, sampler):
    """The shared step code, in the reference's sequential order (chain c sees chains
    < c already moved, as engine.Population.replay walks them), fed the reference's
    draws, reproduces the reference run exactly where it is discrete and to 1e-10
    elsewhere (the bar of test_gpu_mcmc.py::test_replay_retraces_reference)."""
    fx = np.load(os.path.join(GOLD, f'mcmc_{case}_{sampler}.npz'))
    p = pb.mcmc_case(case)
    assert pb.checksum(p['x'], p['data'], p['uncert']) == str(fx['in_checksum'])
    spec = ls.Spec(p['params'], p['pstep'], p['pmin'], p['pmax'], p['prior'], p['priorlow'],
                   p['priorup'], sampler, 1.0, p['fepsilon'])
    chi = _data_chisq(p, om.MODELS[p['model']])
    n, nfree, thin = p['nchains'], spec.nfree, p['thinning']
    M0 = 10*n
    zlen = M0 + int(np.ceil(p['nsamples']/n/thin))*n
    Z = np.zeros((zlen, nfree))
    log_post = np.zeros(zlen)
    zchain = np.full(zlen, -1)
    Z[:M0], log_post[:M0] = fx['Z0'], fx['log_post0']
    st = ls.State(Z[:n], -2.0*log_post[:n], nfree)

    d = {k[5:]: fx[k] for k in fx.files if k.startswith('draw_')}
    for g in range(int(d['ngen'])):
        nd = int(d['done'][g].sum())
        r0 = ls.zrow0(M0, n, thin, g) if nd == n else -1
        for c in range(nd):
            dr = {k: d[k][g][c:c + 1] for k in ('a', 'b', 'iz', 'usj', 'gs', 'u')}
            prop = ls.propose(spec, st.X, Z, dr, d['normal'][g][None, :], [c])
            nxt = chi(prop['nextp'][0]) if prop['inb'][0] else np.nan
            acc, _ = ls.metropolis(spec, st, [c], prop, np.array([nxt]), dr['u'], g)
            assert acc[0] == d['acc'][g][c], (g, c)
            if r0 >= 0:
                Z[r0 + c], log_post[r0 + c], zchain[r0 + c] = st.X[c], -0.5*st.cur[c], c

    nrows = fx['ref_posterior'].shape[0]
    assert np.array_equal(zchain[M0:M0 + nrows], fx['ref_zchain'])
    assert int(st.naccept.sum()) == int(fx['numaccept'])
    assert np.array_equal(st.outbounds, fx['outbounds'])
    np.testing.assert_allclose(Z[M0:M0 + nrows], fx['ref_posterior'], rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(log_post[M0:M0 + nrows], fx['ref_log_post'], rtol=1e-10)
    np.testing.assert_allclose(st.X, fx['final_freepars'], rtol=1e-10, atol=1e-13)
    # best fit: first strictly lower chi-squared in (generation, chain) order, from the
    # best of the initial population (engine.Population.counters_result)
    iz = int(np.argmax(fx['log_post0']))
    best, bestp = -2.0*fx['log_post0'][iz], np.copy(p['params'])
    bestp[spec.ifree] = fx['Z0'][iz]
    order = np.lexsort((np.arange(n), st.best_gen, st.best_chisq))
    c = order[0]
    if st.best_chisq[c] < best:
        best, bestp[spec.ifree] = st.best_chisq[c], st.best_x[c]
    for q in np.where(spec.pstep < 0)[0]:
        bestp[q] = bestp[-int(spec.pstep[q]) - 1]
    np.testing.assert_allclose(bestp, fx['ref_bestp'], rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(-0.5*best, fx['ref_best_log_post'], rtol=1e-10)
