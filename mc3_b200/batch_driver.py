"""Many independent small fits at once: sample_batch() runs B problems of the same
shape (a catalogue of light curves, one fit per star, transit or band) in one
launch, one persistent CTA per problem (csrc/batch_dev.cuh).  Problem b is

    sample(data[b], uncert[b], func, params[b], indparams[b], ...)

with the problem's own seed, and its output dictionary has the keys and meaning of
sample()'s.  What the batch shares: the model (a built-in or a CudaModel, fp64), the
sampler and its options, and the pattern of free, shared and fixed parameters.  A
CudaModel's per-point inputs and run-time constants are the problem's own: indparams[b]
is read as sample() reads it (CudaModel.split_args), and the kernels are those of the
model's batch module (CudaModel.batch_handle).  It writes no files and no log output.

With grtest, the Gelman-Rubin test runs on the device at sample()'s report points
(mcmc_driver.report_points) for every problem at once (mc3b_batch_gelman_rubin); with
grbreak, a problem that passes stops there and gives up its CTA to the problems still
running, and its output covers the thinned steps it ran.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from . import stats as ms
from .engine import column_statistics, to_host
from .models import BuiltinModel, CudaModel
from .mcmc_driver import gr_min_size, report_points
from .sampler_driver import check_sampler, read_arrays, fill_vectors

MAX_CHAINS = 256                  # SW * 32 threads of mc3b_batch_run's CTA
_VECTORS = ('pmin', 'pmax', 'pstep', 'prior', 'priorlow', 'priorup')


class _ProblemLog:
    """The `log` of sample()'s checks for problem b: errors name the problem."""

    def __init__(self, b):
        self.b = b

    def error(self, message, exception=ValueError):
        raise exception(f'problem {self.b}: {message}')


def _count(name, value):
    try:
        return len(value)
    except TypeError:
        raise ValueError(f'{name} must be a sequence with one entry per problem') from None


def _per_problem(name, value, B):
    """None, one [npars] vector shared by all problems, or [B, npars] -> list of B."""
    if value is None:
        return [None]*B
    a = np.asarray(value, dtype=float)
    if a.ndim == 2:
        if a.shape[0] != B:
            raise ValueError(f'{name} has {a.shape[0]} rows for {B} problems')
        return list(a)
    if a.ndim != 1:
        raise ValueError(f'{name} must be [npars] or [{B}, npars], got shape {a.shape}')
    return [a]*B


def sample_batch(data, uncert, func, params, indparams,
                 pmin=None, pmax=None, pstep=None, prior=None, priorlow=None, priorup=None,
                 sampler=None, nchains=7, nsamples=None, burnin=0, thinning=1,
                 grtest=False, grbreak=0.0, grnmin=0.5,
                 fgamma=1.0, fepsilon=0.0, hsize=10, kickoff='normal',
                 pnames=None, texnames=None, seed=None, device=None, wlike=False, dtype='f64',
                 _state=False):
    """Run B independent fits; returns the list of their output dictionaries.

    data, uncert  sequences of B 1-D arrays (lengths may differ between problems)
    params        [B, npars]
    indparams     sequence of B lists, as sample() takes them: [x_b] for a built-in model;
                  for a CudaModel its ninputs arrays of data[b]'s shape, then its nconst
                  constants (they may differ between problems)
    pmin, pmax, pstep, prior, priorlow, priorup
                  [npars] shared by all problems, or [B, npars]; the sign pattern of
                  pstep (free / fixed / shared) must be the same for every problem
    func          a BuiltinModel (polynomial, sinusoid, gaussian, box) or a CudaModel, fp64
    seed          int s (problem b takes s + b), B ints, or None (one drawn as sample()
                  draws it, then s + b)
    grtest, grbreak, grnmin
                  as in sample(), problem by problem: with grtest each output gains 'psrf',
                  the PSRF of the problem's last Gelman-Rubin evaluation; with grbreak > 0 a
                  problem stops at the first report where every PSRF < grbreak and its
                  history exceeds grnmin, and its outputs cover the steps it ran.  grtest is
                  off by default (sample() turns it on), since the batch prints no log.
    The other options mean what they mean in sample(); nchains <= 256.  _state=True
    returns the device state after the generations instead (for tests)."""
    check_sampler(sampler, nsamples, None, _Log0())
    if not isinstance(func, (BuiltinModel, CudaModel)):
        raise ValueError('sample_batch needs a built-in model (mc3_b200.models.polynomial, sinusoid, '
                         f'gaussian or box) or a CudaModel, got {func!r}')
    user = isinstance(func, CudaModel)
    if wlike or dtype != 'f64':
        raise ValueError('sample_batch runs the fp64 chi-squared likelihood only (no wlike, no f32)')
    nchains, thinning, hsize = int(nchains), int(thinning), int(hsize)
    if nchains > MAX_CHAINS:
        raise ValueError(f'sample_batch runs at most {MAX_CHAINS} chains per problem, got {nchains} '
                         '(sample() runs larger populations)')
    if sampler == 'demc' and nchains < 3:
        raise ValueError(f'demc needs at least 3 chains, got {nchains}')
    if grtest and nchains < 2:
        raise ValueError(f'the Gelman-Rubin test needs at least 2 chains, got {nchains}')
    if kickoff not in ('normal', 'uniform'):
        raise ValueError(f"kickoff must be 'normal' or 'uniform', got {kickoff!r}")

    # ---- one entry per problem ----
    B = _count('data', data)
    for name, v in (('uncert', uncert), ('params', params), ('indparams', indparams)):
        if _count(name, v) != B:
            raise ValueError(f'{name} has {_count(name, v)} entries for {B} problems (data has {B})')
    if B == 0:
        raise ValueError('sample_batch needs at least one problem')
    vecs = {k: _per_problem(k, v, B) for k, v in zip(_VECTORS, (pmin, pmax, pstep, prior, priorlow, priorup))}
    if seed is None:
        seed = int(np.random.randint(0, 2**31 - 1))          # as mcmc() draws it
    if np.ndim(seed) == 0:
        seeds = [int(seed) + b for b in range(B)]
    else:
        seeds = [int(s) for s in seed]
        if len(seeds) != B:
            raise ValueError(f'seed has {len(seeds)} entries for {B} problems')

    # ---- sample()'s checks, problem by problem ----
    probs = []
    for b in range(B):
        log = _ProblemLog(b)
        (p, d, u, lo, hi, st, pr, plo, pup) = read_arrays(
            params[b], data[b], uncert[b], vecs['pmin'][b], vecs['pmax'][b], vecs['pstep'][b],
            vecs['prior'][b], vecs['priorlow'][b], vecs['priorup'][b], log)
        (pn, tn, lo, hi, st, pr, plo, pup, nfree, ifree, ishare) = fill_vectors(
            p, pnames, texnames, lo, hi, st, pr, plo, pup, log)
        if user:
            xs, k = _user_inputs(func, indparams[b], d, log)
            x = xs[0]
        else:
            x = np.asarray(indparams[b][0], dtype=float) if np.iterable(indparams[b]) and len(indparams[b]) else None
            if x is None or len(indparams[b]) != 1 or x.ndim != 1:
                log.error('built-in models need indparams=[x] with the same shape as data')
            if np.shape(x) != np.shape(d):                       # a built-in model returns x's shape
                log.error(f"The size of the data array ({np.size(d)}) does not "
                          f"match the size of the func() output ({np.size(x)})")
            xs, k = [x], None
        try:
            func.nmodel(p.size)
        except ValueError as e:
            log.error(str(e))
        probs.append(dict(params=p, data=d, uncert=u, x=x, xs=xs, consts=k, pmin=lo, pmax=hi, pstep=st, prior=pr,
                          priorlow=plo, priorup=pup, pnames=pn, texnames=tn, ifree=ifree, ishare=ishare))
    npars = probs[0]['params'].size
    def pattern(q):                                 # which parameters are free, fixed, shared with which
        return q['params'].size, tuple(np.sign(q['pstep'])), tuple(q['pstep'][q['pstep'] < 0])
    for b, q in enumerate(probs):
        if pattern(q) != pattern(probs[0]):
            raise ValueError(f'problem {b}: the free/shared/fixed pattern of pstep differs from problem 0 '
                             f"({q['pstep']} against {probs[0]['pstep']}); every problem needs the same")
    ifree = probs[0]['ifree']
    nfree = ifree.size
    if nfree == 0:
        raise ValueError('sample_batch needs at least one free parameter')
    if npars > _lib.MAX_PARS:
        raise ValueError(f'at most {_lib.MAX_PARS} parameters are supported')

    nzchain = int(np.ceil(nsamples/nchains/thinning))       # mcmc_driver.py:129-134
    niter = nzchain*thinning
    burnin = int(burnin)
    if niter < burnin:
        raise ValueError(f"The number of burned-in samples ({burnin}) is greater than "
                         f"the number of iterations per chain ({niter})")
    zburn = int(burnin/thinning)
    if (nzchain - zburn)*nchains < 2:
        raise ValueError('the burned-in sample of a problem must hold at least 2 rows')
    M0 = hsize*nchains
    zlen = M0 + nzchain*nchains
    grmin = gr_min_size(grnmin, nchains, nzchain, zburn, thinning, M0, _Log0())
    reports = report_points(nzchain)

    # ---- device ----
    _lib.load()
    if not torch.cuda.is_available():
        raise _lib.Mc3bError('mc3_b200 needs a CUDA device (no CPU fallback)')
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.index is None:
        dev = torch.device('cuda', torch.cuda.current_device())
    with torch.cuda.device(dev):
        sizes = np.array([q['data'].size for q in probs], dtype=np.int64)
        need = _state_bytes(B, nchains, npars, nfree, zlen, int(sizes.sum()), len(probs[0]['xs']),
                            func.nconst if user else 0, len(reports) if grtest else 0)
        free = torch.cuda.mem_get_info(dev)[0]
        if need > free:
            raise ValueError(f'the state of {B} problems needs {need} bytes of device memory, '
                             f'{free} are free')
        run = _BatchRun(probs, seeds, sizes, dev, sampler, nchains, npars, nfree, ifree, M0, zlen,
                        thinning, fgamma, fepsilon)
        run.init(kickoff, func)
        if grtest:
            run.run_gr(func, reports, zburn, float(grbreak), grmin)
        else:
            run.run(niter, func)
        if _state:
            return run
        return run.outputs(func, zburn, nzchain, probs)


def _user_inputs(func, args, d, log):
    """(per-point arrays, constants [nconst]) of a CudaModel's indparams for data d, as
    sample() reads them (CudaModel.split_args); errors name the problem through log."""
    if not np.iterable(args) or isinstance(args, (str, bytes)):
        log.error(f'{func.name} needs indparams=[x1, ..., x{func.ninputs}, constants...] per problem')
    try:
        xs, k = func.split_args(list(args))
    except ValueError as e:
        log.error(str(e))
    if len(xs) != func.ninputs:
        log.error(f'{func.name} takes {func.ninputs} input array(s), got {len(xs)}')
    xs = [np.asarray(a, dtype=float) for a in xs]
    for j, a in enumerate(xs):
        if a.shape != np.shape(d):
            log.error(f'input {j} of {func.name} has shape {a.shape}, the data {np.shape(d)}')
    return xs, np.zeros(0) if k is None else k


class _Log0:
    """sample()'s run-option checks raise as they do there, without log output."""

    def error(self, message, exception=ValueError):
        raise exception(message)


def _state_bytes(B, nchains, npars, nfree, zlen, ntot, ninputs=1, nconst=0, nreports=0):
    """Device bytes of the batched state (history, per-chain arrays, data, a CudaModel's
    further inputs and constants, with the Gelman-Rubin test the PSRF table of nreports
    reports and the stop points) and of the post-processing copies of the history
    (chi-squared column)."""
    per = zlen*(nfree*8 + 8 + 4 + 8) + nchains*(2*nfree*8 + npars*8 + 4*8 + 2*4) + nfree*4 + 7*npars*8
    gr = B*(nreports*nfree*8 + 8) if nreports else 0
    return B*per + 3*ntot*8 + (ninputs - 1)*ntot*8 + B*nconst*8 + gr


class _BatchRun:
    """The batched state on the device and the C-ABI calls that advance it."""

    def __init__(self, probs, seeds, sizes, dev, sampler, nchains, npars, nfree, ifree, M0, zlen,
                 thinning, fgamma, fepsilon):
        B = len(probs)
        self.B, self.dev, self.nchains, self.npars, self.nfree = B, dev, nchains, npars, nfree
        self.M0, self.zlen, self.thinning = M0, zlen, thinning
        f64 = dict(dtype=torch.float64, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        n = nchains
        off = np.zeros(B + 1, dtype=np.int64)
        off[1:] = np.cumsum(sizes)
        self.off = off
        cat = lambda k: torch.from_numpy(np.concatenate([q[k] for q in probs])).to(dev)  # noqa: E731
        self.d_x, self.d_data = cat('x'), cat('data')
        # a CudaModel's inputs 2..ninputs, concatenated as x, and its constants [B, nconst]
        self.d_xs = [self.d_x] + [torch.from_numpy(np.concatenate([q['xs'][j] for q in probs])).to(dev)
                                  for j in range(1, len(probs[0]['xs']))]
        k = np.stack([q['consts'] for q in probs]) if probs[0]['consts'] is not None else None
        self.d_consts = torch.from_numpy(k).to(dev) if k is not None and k.size else None
        self.d_invsig = 1.0/cat('uncert')
        self.d_off = torch.from_numpy(off).to(dev)
        stack = lambda k: torch.from_numpy(np.stack([q[k] for q in probs])).to(dev)  # noqa: E731
        self.vec = {k: stack(k) for k in ('pstep', 'pmin', 'pmax', 'params', 'prior', 'priorlow', 'priorup')}
        self.d_ifree = torch.tensor(ifree, **i32)
        self.Z = torch.zeros((B, zlen, nfree), **f64)
        self.log_post = torch.zeros((B, zlen), **f64)
        self.zchain = torch.full((B, zlen), -1, **i32)
        self.X = torch.zeros((B, n, nfree), **f64)
        self.chisq_cur = torch.zeros((B, n), **f64)
        self.nextp = torch.zeros((B, n, npars), **f64)
        self.mrfactor = torch.ones((B, n), **f64)
        self.u = torch.zeros((B, n), **f64)
        self.inb = torch.zeros((B, n), **i32)
        self.naccept = torch.zeros((B, n), **i32)
        self.outbounds = torch.zeros((B, nfree), **i32)
        self.best_chisq = torch.full((B, n), float('inf'), **f64)
        self.best_x = torch.zeros((B, n, nfree), **f64)
        self.best_gen = torch.zeros((B, n), dtype=torch.int64, device=dev)
        self.status = torch.zeros(B, **i32)
        self.psrf = self.kstop = None               # run_gr: [B, nreports, nfree], [B]

        # one mc3b_sampler_t per problem, as engine.Population._make_struct fills it
        tab = np.zeros(B, dtype=np.dtype(_lib.SamplerStruct))
        tab['nchains'], tab['chain0'], tab['nlocal'] = n, 0, n
        tab['npars'], tab['nfree'], tab['sampler'] = npars, nfree, _lib.SAMPLERS[sampler]
        tab['ifree'] = self.d_ifree.data_ptr()
        bidx = np.arange(B, dtype=np.uint64)

        def rows(t):                                # address of problem b's slice of t
            return np.uint64(t.data_ptr()) + bidx*np.uint64(t.stride(0)*t.element_size())
        for k, field in (('pstep', 'pstep'), ('pmin', 'pmin'), ('pmax', 'pmax'), ('params', 'params0')):
            tab[field] = rows(self.vec[k])
        has_prior = np.array([np.any((q['priorlow'] > 0) & (q['priorup'] > 0)) for q in probs])
        for k in ('prior', 'priorlow', 'priorup'):
            tab[k] = np.where(has_prior, rows(self.vec[k]), np.uint64(0))
        tab['gamma'] = float(fgamma)*2.38/np.sqrt(2*nfree)  # chain.py:175
        tab['fepsilon'] = float(fepsilon)
        tab['seed'] = np.array(seeds, dtype=np.int64).astype(np.uint64)
        for field, t in (('X', self.X), ('chisq_cur', self.chisq_cur), ('Z', self.Z),
                         ('log_post', self.log_post), ('zchain', self.zchain), ('nextp', self.nextp),
                         ('mrfactor', self.mrfactor), ('u', self.u), ('inb', self.inb),
                         ('naccept', self.naccept), ('outbounds', self.outbounds),
                         ('best_chisq', self.best_chisq), ('best_x', self.best_x),
                         ('best_gen', self.best_gen)):
            tab[field] = rows(t)
        tab['zlen'], tab['M0'], tab['thinning'] = zlen, M0, thinning
        tab['world'], tab['rank'] = 1, 0
        self.table = torch.from_numpy(tab.view(np.uint8)).to(dev)
        S = _lib.BatchStruct()
        S.nproblems, S.problems, S.offsets = B, self.table.data_ptr(), self.d_off.data_ptr()
        S.x, S.data, S.invsig = self.d_x.data_ptr(), self.d_data.data_ptr(), self.d_invsig.data_ptr()
        S.status = self.status.data_ptr()
        self.S = S

    def _extra(self, func):
        """(xs, nx, consts, nk) of the mc3b_user_batch_* entry points."""
        return _lib.ptrs(self.d_xs), len(self.d_xs), _lib.ptr(self.d_consts), func.nconst

    def init(self, kickoff, func):
        """Initial population of every problem (mc3b_batch_init, mc3b_user_batch_init); the
        problems that could not be populated raise the reference's error."""
        k = {'normal': 0, 'uniform': 1}[kickoff]
        if isinstance(func, CudaModel):
            _lib.call('mc3b_user_batch_init', func.batch_handle(), ctypes.byref(self.S), *self._extra(func), k,
                      _lib.stream_ptr())
        else:
            _lib.call('mc3b_batch_init', ctypes.byref(self.S), func.model_id, func.nmodel(self.npars), k,
                      _lib.stream_ptr())
        bad = np.flatnonzero(self.status.cpu().numpy())
        if bad.size:
            who = f'problem {bad[0]}' if bad.size == 1 else 'problems ' + ', '.join(str(b) for b in bad)
            raise ValueError(
                f'{who}: Cannot populate an initial sample set of parameters, try '
                'updating the parameters initial guess to avoid sampling '
                'beyond the parameter boundaries or where the model returns '
                'non-finite values.')

    def run(self, ngen, func, gen0=0):
        if isinstance(func, CudaModel):
            _lib.call('mc3b_user_batch_run', func.batch_handle(), ctypes.byref(self.S), *self._extra(func), gen0,
                      ngen, _lib.stream_ptr())
        else:
            _lib.call('mc3b_batch_run', ctypes.byref(self.S), func.model_id, func.nmodel(self.npars),
                      gen0, ngen, _lib.stream_ptr())

    def run_gr(self, func, reports, zburn, grbreak, grmin):
        """The run with the Gelman-Rubin test (mcmc_driver.py:297-348).  grbreak > 0: report
        blocks, and the test at every report past burn-in, where the problems that pass stop
        (status 3, kstop); otherwise one run and one test at the last report.  psrf[b, i] is
        problem b's PSRF at report i (NaN where not evaluated); kstop[b] the thinned steps it
        ran.  Nothing returns to the host in between."""
        B, nf, th = self.B, self.nfree, self.thinning
        self.reports = reports
        self.psrf = torch.full((B, len(reports), nf), float('nan'), dtype=torch.float64, device=self.dev)
        self.kstop = torch.full((B,), reports[-1], dtype=torch.int64, device=self.dev)
        k0 = 0
        for i, k in enumerate(reports):
            if grbreak <= 0.0 and k < reports[-1]:
                continue
            self.run((k - k0)*th, func, gen0=k0*th)
            k0 = k
            if k > zburn:                                           # :325
                _lib.call('mc3b_batch_gelman_rubin', ctypes.byref(self.S), k, zburn, grbreak, grmin,
                          self.psrf[:, i].data_ptr(), len(reports)*nf, self.kstop.data_ptr(), _lib.stream_ptr())

    def outputs(self, func, zburn, nzchain, probs):
        """Output dictionaries (mcmc_driver.update_output + sample()'s statistics)."""
        B, n, nfree, M0, npars = self.B, self.nchains, self.nfree, self.M0, self.npars
        dev = self.dev
        ifree = self.d_ifree.long()
        pstep0 = probs[0]['pstep']

        def fill_shared(P):                         # [B, npars]: shared parameters copy their source
            for k in np.where(pstep0 < 0)[0]:
                P[:, k] = P[:, -int(pstep0[k]) - 1]
            return P
        # best of the initial population (mcmc_driver.py:273-275; first maximum)
        lp0 = self.log_post[:, :M0]
        iz = torch.argmax(lp0, dim=1)
        ar = torch.arange(B, device=dev)
        best_lp0 = lp0[ar, iz]
        bestp = self.vec['params'].clone()
        bestp[:, ifree] = self.Z[ar, iz]
        best_chi = -2.0*best_lp0
        # counters_result: lowest best chi-squared, ties to the earlier (generation, chain);
        # it replaces the initial best when strictly lower
        bc, bg = self.best_chisq, self.best_gen
        m = bc.min(dim=1, keepdim=True).values
        cand = bc == m
        gmin = torch.where(cand, bg, torch.iinfo(torch.int64).max).min(dim=1, keepdim=True).values
        ch = torch.argmax((cand & (bg == gmin)).to(torch.int32), dim=1)
        m = m[:, 0]
        better = torch.isfinite(m) & (m < best_chi)
        bestp[better.nonzero().flatten()[:, None], ifree[None, :]] = self.best_x[ar, ch][better]
        best_chi = torch.where(better, m, best_chi)
        bestp = fill_shared(bestp)
        numaccept = self.naccept.sum(dim=1)

        # best-fit model of every problem, into one flat buffer
        model = torch.empty(int(self.off[-1]), dtype=torch.float64, device=dev)
        nmodel = func.nmodel(npars)
        st = _lib.stream_ptr()
        if isinstance(func, CudaModel):                 # every problem in one launch
            _lib.call('mc3b_user_batch_eval', func.batch_handle(), ctypes.byref(self.S), *self._extra(func),
                      bestp.data_ptr(), npars, model.data_ptr(), st)
        else:
            for b in range(B):
                o, k = int(self.off[b]), int(self.off[b + 1] - self.off[b])
                _lib.call('mc3b_model_eval', func.model_id, bestp[b].data_ptr(), npars, 1, nmodel,
                          self.d_x[o:].data_ptr(), k, model[o:].data_ptr(), st)

        # thinned steps problem b ran: nzchain, or where the Gelman-Rubin test stopped it
        Ks = np.full(B, nzchain, dtype=np.int64) if self.kstop is None else to_host(self.kstop)

        # chi-squared column: -2 (log_post - log_prior) of every history row
        chisq = torch.empty((B, nzchain*n), dtype=torch.float64, device=dev)
        for b in range(B):
            _lib.call('mc3b_log_prior', self.Z[b, M0:].data_ptr(), int(Ks[b])*n, nfree, self.d_ifree.data_ptr(),
                      self.vec['prior'][b].data_ptr(), self.vec['priorlow'][b].data_ptr(),
                      self.vec['priorup'][b].data_ptr(), self.log_post[b, M0:].data_ptr(), None,
                      chisq[b].data_ptr(), st)

        # posterior statistics: the burned sample (utils.burn's lock-step closed form), at most
        # 20000 rows picked as sample() picks them -- the same rows for every problem that ran
        # the same number of steps; one pass per such group (at most one per report)
        free_stats = torch.empty((8, B, nfree), dtype=torch.float64, device=dev)
        zmasks = {}
        for K in np.unique(Ks):
            grp = np.flatnonzero(Ks == K)
            G = grp.size
            zmask = (np.arange(zburn, K)[None, :]*n + np.arange(n)[:, None]).ravel()
            pick = zmask
            if zmask.size > 20000:
                pick = zmask[np.random.default_rng(314159).choice(zmask.size, 20000, replace=False)]
            zmasks[K] = zmask
            g = torch.from_numpy(grp).to(dev)
            blk = self.Z[g[:, None], M0 + torch.from_numpy(pick).to(dev)[None, :]]     # [G, nstat, nfree]
            blk = blk.permute(1, 0, 2).reshape(blk.shape[1], G*nfree).contiguous()
            cs = column_statistics(blk, 0.683)                              # [5, G nfree]
            hpd = torch.empty((3, G*nfree), dtype=torch.float64, device=dev)
            step = 65535                                 # k_kde_grid: one grid.y per column
            ws = torch.empty(max(_lib.load().mc3b_hpd_workspace(min(step, G*nfree)), 8)//8,
                             dtype=torch.float64, device=dev)
            for c0 in range(0, G*nfree, step):
                c1 = min(c0 + step, G*nfree)
                chunk = blk[:, c0:c1].contiguous()
                o = torch.empty((3, c1 - c0), dtype=torch.float64, device=dev)
                _lib.call('mc3b_hpd', chunk.data_ptr(), chunk.shape[0], c1 - c0, 0.683, ws.data_ptr(),
                          o.data_ptr(), st)
                hpd[:, c0:c1] = o
            free_stats[:, g] = torch.cat([cs, hpd]).view(8, G, nfree)

        # to the host, one copy per array
        h = {k: to_host(v) for k, v in (
            ('Z', self.Z[:, M0:]), ('zchain', self.zchain[:, M0:]), ('log_post', self.log_post[:, M0:]),
            ('chisq', chisq), ('model', model), ('bestp', bestp), ('best_chi', best_chi),
            ('numaccept', numaccept), ('free', free_stats))}
        if self.psrf is not None:
            h['psrf'] = to_host(self.psrf)
        outs = []
        for b, q in enumerate(probs):
            o0, o1 = self.off[b], self.off[b + 1]
            K = int(Ks[b])
            rows = K*n
            nsample = rows*self.thinning
            bp = h['bestp'][b].copy()
            out = {'pnames': q['pnames'], 'texnames': q['texnames'], 'pstep': q['pstep'],
                   'ifree': q['ifree'], 'burnin': zburn,
                   'posterior': h['Z'][b, :rows], 'zchain': h['zchain'][b, :rows].astype(int),
                   'chisq': h['chisq'][b, :rows], 'log_post': h['log_post'][b, :rows],
                   'acceptance_rate': int(h['numaccept'][b])*100.0/max(nsample, 1)}
            # calc_bestfit_statistics (stats.py:855-873) from the tracked best chi-squared
            ndata = int(o1 - o0)
            best_log_post = -0.5*float(h['best_chi'][b])
            best_log_prior = ms.log_prior(bp[q['ifree']], q['prior'], q['priorlow'], q['priorup'], q['pstep'])
            best_chisq = -2*(best_log_post - best_log_prior)
            best_model = h['model'][o0:o1].copy()
            out['bestp'] = bp
            out['best_chisq'] = best_chisq
            out['red_chisq'] = best_chisq/(ndata - nfree) if ndata > nfree else np.nan
            out['BIC'] = best_chisq + nfree*np.log(ndata)
            out['best_log_post'] = best_log_post
            out['best_model'] = best_model
            out['stddev_residuals'] = np.std(best_model - q['data'])
            out['zmask'] = zmasks[K]
            st8 = ms.expand_free_stats(tuple(h['free'][:, b]), bp, q['pstep'])
            for k, v in zip(('medianp', 'meanp', 'stdp', 'median_low_bounds', 'median_high_bounds',
                             'mode', 'hpd_low_bounds', 'hpd_high_bounds'), st8):
                out[k] = v
            out['chisq_factor'] = 1.0
            out['CRlo'] = out['hpd_low_bounds'] - bp
            out['CRhi'] = out['hpd_high_bounds'] - bp
            out['CRlo'][q['pstep'] == 0] = out['CRhi'][q['pstep'] == 0] = 0.0
            if self.psrf is not None:               # the last evaluation: at K (the last report, or the stop)
                out['psrf'] = h['psrf'][b, self.reports.index(K)].copy()
            outs.append(out)
        return outs
