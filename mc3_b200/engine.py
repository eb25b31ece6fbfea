"""Device-resident chain population: the B200 replacement of the reference's
per-iteration loop (mc3/chain.py:158-299) and of the shared state that
mc3/mcmc_driver.py:143-202 allocates.

One `Population` = all chains of one device.  A generation is three kernel
launches through the C ABI (include/mc3b200.h):

    mc3b_propose      draws, jump, bounds, shared fill        chain.py:185-247
    mc3b_model_chisq  built-in model + chi-squared, all chains  chain.py:249, 302-340
                      (mc3b_user_model_chisq_consts for a CudaModel: the same kernel)
    mc3b_metropolis   partial sums + priors, accept, write    chain.py:251-289

advancing every chain in lock-step (SURVEY.md finding 6: within one generation
all chains see the population / history as it was at the start of the
generation).  The generation counter can live on the device so that the three
launches are captured once in a CUDA graph and replayed.

Replay mode (`replay`) consumes the reference's recorded random stream and
walks the chains in the reference's sequential order, to retrace its
accept/reject trajectory.

HBM layout (all fp64 unless noted; row-major):
    x, data, invsig [N]     (+ fp32 copies in dtype='f32')
    X         [nchains, nfree]   current states          (reference `freepars`)
    Z         [zlen, nfree]      history, reference row order: M0 initial rows,
                                 then row M0 + k*nchains + c for thinned step k
    log_post  [zlen], zchain [zlen] int32 (-1 = initial sample)
    nextp     [nchains, npars]   proposed full vectors
    partial   [nsplit, nchains]  per-split chi-squared partial sums
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from .models import BuiltinModel, CudaModel, TorchModel
from .chisq_form import choose_form
from .parallel import chain_slice, allgather_rows, gather_history


def to_host(t):
    """Device tensor -> numpy array backed by pinned host memory (pageable D2H
    of the 10-100 MB history costs several times the PCIe time).  The array
    owns its pinned block; torch's host allocator recycles it once the array
    is dropped, so repeated runs pay no cudaHostAlloc and no second copy."""
    if t.numel() == 0 or t.numel()*t.element_size() < (1 << 20):
        return t.cpu().numpy()
    t = t.contiguous()
    buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    buf.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return buf.numpy()


def column_statistics(blk, quantile=0.683):
    """[5, cols] device tensor: median, mean, std and central-quantile bounds of every
    column of blk [n, cols] (stats.py:764-802 'med_central'; numpy's linear percentile
    rule, population std)."""
    n = blk.shape[0]
    srt, _ = torch.sort(blk, dim=0)

    def pct(q):
        pos = q*(n - 1)
        i0 = int(np.floor(pos))
        i1 = min(i0 + 1, n - 1)
        fr = pos - i0
        return srt[i0] + (srt[i1] - srt[i0])*fr
    return torch.stack([pct(0.5), blk.mean(dim=0), blk.std(dim=0, unbiased=False),
                        pct(0.5*(1 - quantile)), pct(0.5*(1 + quantile))])


def on_device(fn):
    """Run a Population method with the population's device current: the C ABI
    launches on the current CUDA device and on its current stream."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        if torch.cuda.current_device() == self.dev.index:
            return fn(self, *args, **kwargs)
        with torch.cuda.device(self.dev):
            return fn(self, *args, **kwargs)
    return wrapped


_DT = {'f64': _lib.F64, 'f32': _lib.F32, np.float64: _lib.F64, np.float32: _lib.F32}


class GuardRecords:
    """Host side of the moment form's guard records (include/mc3b200.h mc3b_moment_t.record).
    `ring` is the int64 view of R page-locked slots the fused epilogue writes: slot g % R holds
    (g mod 2^32) << 32 | guard hits counted up to the end of generation g.  Hits counted outside
    generations (mc3b_moment_finish in chisq() and init_population) enter the next record.

    The rule (step) is a function of generation boundaries only: at the start of a run() call,
    the record of G* = the generation count at the start of the call before the previous one is
    read, G* clamped to >= gen - R + 1 so that its slot cannot have been overwritten (the device
    is never ahead of what the host has enqueued).  The form is left when the hits since the last
    record read exceed 1e-3 per chain-step.  The record has normally long arrived; until it has,
    the host polls its slot."""
    R = _lib.GUARD_RECORDS

    def __init__(self, ring):
        self.ring = ring
        # slot s only ever holds generations g = s (mod R), and R divides 2^32: stamp s + 1 is none of them
        ring[:] = ((np.arange(self.R, dtype=np.int64) + 1) % self.R) << 32
        self.starts = []        # generation counts at the start of the last calls whose record exists
        self.seen = (0, 0)      # (generation, hits) of the last record read
        self.end = None         # generation count at the end of the last recording call

    def read(self, g):
        """Hits of record g, or None while slot g % R holds another generation's stamp."""
        v = int(self.ring[g % self.R])
        return v & 0xffffffff if (v >> 32) & 0xffffffff == g & 0xffffffff else None

    def wait(self, g, idle):
        """Poll record g; idle() tells whether the stream has finished all enqueued work."""
        while True:
            h = self.read(g)
            if h is not None:
                return h
            if idle():
                h = self.read(g)
                if h is None:
                    raise _lib.Mc3bError(f'guard record of generation {g} missing with the stream idle '
                                         f'(slot holds {int(self.ring[g % self.R]):#x})')
                return h

    def step(self, gen, ngen, nlocal, recording, idle):
        """At the start of a run() call from generation count `gen` over `ngen` generations;
        recording: they run the fused moment kernel.  True: leave the moment form."""
        if not recording:
            self.starts = []        # the generations of this call leave no records
            return False
        while len(self.starts) >= 2:
            g = max(self.starts.pop(0), gen - self.R + 1)
            g0, h0 = self.seen
            if g <= g0:
                continue
            hits = self.wait(g, idle)
            if (hits - h0) & 0xffffffff > 1e-3*nlocal*(g - g0):
                return True
            self.seen = (g, hits)
        if self.end == gen:         # the record of generation `gen` exists
            self.starts.append(gen)
        self.end = gen + ngen
        return False


class Population:
    def __init__(self, data, uncert, func, params, indparams=(), indparams_dict=None,
                 pstep=None, pmin=None, pmax=None, prior=None, priorlow=None,
                 priorup=None, nchains=7, sampler='snooker', wlike=False,
                 fgamma=1.0, fepsilon=0.0, hsize=10, thinning=1, nzchain=1,
                 seed=0, dtype='f64', device=None, rank=0, world=1, group=None,
                 reflect=False, M0=None, shard='chains', plan_chains=None):
        _lib.load()
        if not torch.cuda.is_available():
            raise _lib.Mc3bError('mc3_b200 needs a CUDA device (no CPU fallback)')
        self.dev = torch.device('cuda', torch.cuda.current_device()) \
            if device is None else torch.device(device)
        if self.dev.type != 'cuda':
            raise _lib.Mc3bError('mc3_b200 needs a CUDA device (no CPU fallback)')
        if self.dev.index is None:
            self.dev = torch.device('cuda', torch.cuda.current_device())
        # every launch of this object goes to self.dev: the C ABI launches on the
        # CURRENT device, so the public methods below switch to it (on_device)
        with torch.cuda.device(self.dev):
            self._init(data, uncert, func, params, indparams, indparams_dict, pstep,
                       pmin, pmax, prior, priorlow, priorup, nchains, sampler, wlike,
                       fgamma, fepsilon, hsize, thinning, nzchain, seed, dtype, rank,
                       world, group, reflect, M0, shard, plan_chains)

    def _init(self, data, uncert, func, params, indparams, indparams_dict, pstep,
              pmin, pmax, prior, priorlow, priorup, nchains, sampler, wlike,
              fgamma, fepsilon, hsize, thinning, nzchain, seed, dtype, rank,
              world, group, reflect, M0, shard, plan_chains):
        self.rank, self.world, self.group = rank, world, group
        # shard='chains': each device owns a block of chains (population exchange
        # per generation).  shard='data': each device holds a slice of the data
        # and evaluates ALL chains on it; the per-device chi-squared sums are
        # all-gathered and added in rank order, proposals and decisions are
        # replicated bit for bit (SURVEY 8e, "large-N variant").
        self.shard = shard if world > 1 else 'chains'
        if self.shard not in ('chains', 'data'):
            raise ValueError("shard must be 'chains' or 'data'")
        self.func = func
        self.indparams = list(indparams)
        self.indparams_dict = dict(indparams_dict or {})
        self.wlike = bool(wlike)
        self.sampler = sampler
        self.dtype = _DT[dtype]
        f64 = dict(dtype=torch.float64, device=self.dev)

        params = np.array(params, dtype=np.double)
        self.npars = npars = params.size
        self.params = params
        self.pstep = np.asarray(pstep, dtype=np.double)
        self.pmin = np.full(npars, -np.inf) if pmin is None else np.asarray(pmin, np.double)
        self.pmax = np.full(npars, np.inf) if pmax is None else np.asarray(pmax, np.double)
        if prior is None or priorlow is None or priorup is None:
            prior = priorlow = priorup = np.zeros(npars)
        self.prior = np.asarray(prior, np.double)
        self.priorlow = np.asarray(priorlow, np.double)
        self.priorup = np.asarray(priorup, np.double)
        self.ifree = np.where(self.pstep > 0)[0]
        self.ishare = np.where(self.pstep < 0)[0]
        self.nfree = nfree = self.ifree.size
        if npars > _lib.MAX_PARS:
            raise ValueError(f'at most {_lib.MAX_PARS} parameters are supported')
        self.nchains = int(nchains)
        if self.shard == 'data':
            if wlike:
                raise ValueError('the wavelet likelihood cannot be sharded over data')
            self.chain0, self.nlocal = 0, self.nchains
        else:
            self.chain0, self.nlocal = chain_slice(self.nchains, rank, world)
        self.hsize, self.thinning, self.nzchain = int(hsize), int(thinning), int(nzchain)
        self.M0 = self.hsize*self.nchains if M0 is None else int(M0)
        self.zlen = self.M0 + self.nzchain*self.nchains
        self.seed = int(seed)

        # ---- data ----
        data = np.ascontiguousarray(data, dtype=np.double)
        uncert = np.ascontiguousarray(uncert, dtype=np.double)
        self.host_data = data              # whole series (best-fit residual statistics)
        self.host_uncert0 = float(uncert.flat[0]) if uncert.size else 1.0
        self.ndata_total = data.size
        lo, hi = 0, data.size
        if self.shard == 'data':
            lo, hi = rank*data.size//world, (rank + 1)*data.size//world
            data, uncert = data[lo:hi], uncert[lo:hi]
        self.data_slice = (lo, hi)
        self.ndata = data.size
        self.d_data = torch.from_numpy(data).to(self.dev)
        self.d_uncert = torch.from_numpy(uncert).to(self.dev)
        self.nfunc = npars - 3 if self.wlike else npars
        if self.shard == 'data' and not isinstance(func, BuiltinModel):
            raise ValueError("shard='data' needs a built-in model (other models run with shard='chains')")
        # the chi-squared form (chisq_form.choose_form); what does not apply stays unset
        self.usig = self.grid = self.use_moment = False
        self.chisq_model_id = self.seg = self.spectral_plan = self.d_tile_x = None
        self.d_fold = self.moment = self.spectral = self.guard_hits = None
        if isinstance(func, (BuiltinModel, CudaModel)):
            x = self._stage_model(func, lo, hi)
            form = choose_form(func, x, uncert, self.dtype, self.params, self.pstep, self.pmin, self.pmax)
            self.usig, self.grid, self.seg = form.usig, form.grid, form.seg
            self.chisq_model_id, self.spectral_plan = form.model_id, form.spectral_plan
            kx, kd, kw = self._prepare_seg(x) if form.seg is not None else (self.d_x, self.d_data, self.d_invsig)
            if form.fold:                  # the mirrored-pair copy of the data (k_sinefold)
                self.d_fold = torch.zeros_like(kd)
                _lib.call('mc3b_fold_data', kd.data_ptr(), form.nfold, self.d_fold.data_ptr(),
                          _lib.stream_ptr())
            if form.moment:
                # least-squares line through the data and the sum of squares about it, on the device (a few
                # small kernels and one read of three numbers).  Its temporaries live until the constructor
                # returns: where the later buffers land moved the generation kernel's time by 5% on a B200
                xm, dm = self.d_x.mean(), self.d_data.mean()
                xc = self.d_x - xm
                slr_t = torch.dot(xc, self.d_data - dm)/torch.dot(xc, xc)
                c0r_t = dm - slr_t*xm
                res = self.d_data - (c0r_t + slr_t*self.d_x)
                line = [float(v) for v in torch.stack([c0r_t, slr_t, torch.dot(res, res)]).cpu()]
                self._prepare_moment(x, kx, kd, form, *line)
            # what the chi-squared kernels read: the arrays of the form, or fp32 copies
            cast = (lambda t: t.float().contiguous()) if self.dtype == _lib.F32 else (lambda t: t)
            self.k_x, self.k_d, self.k_w = cast(kx), cast(kd), cast(kw)
            self.k_xs = [self.k_x] + [cast(t) for t in self.d_xs[1:]]
            self.k_xptrs = _lib.ptrs(self.k_xs)
            self.k_kc = None if self.d_kc is None else cast(self.d_kc)
        elif isinstance(func, TorchModel):
            self.kind = 'torch'
            self.t_indparams = [torch.as_tensor(a, device=self.dev)
                                if isinstance(a, np.ndarray) else a
                                for a in self.indparams]
        else:
            self.kind = 'numpy'

        # ---- small vectors ----
        self.d_ifree = torch.tensor(self.ifree, dtype=torch.int32, device=self.dev)
        self.d_pstep = torch.tensor(self.pstep, **f64)
        self.d_pmin = torch.tensor(self.pmin, **f64)
        self.d_pmax = torch.tensor(self.pmax, **f64)
        self.d_params0 = torch.tensor(params, **f64)
        self.has_prior = bool(np.any((self.priorlow > 0) & (self.priorup > 0)))
        self.d_prior = torch.tensor(self.prior, **f64)
        self.d_priorlow = torch.tensor(self.priorlow, **f64)
        self.d_priorup = torch.tensor(self.priorup, **f64)

        # ---- population state ----
        n = self.nchains
        # Multi-GPU chain partition: population (and, for snooker, history) live in
        # peer memory mapped into every process (CUDA IPC), so that the Metropolis step
        # stores every chain's next state straight into all devices over NVLink and a
        # generation flag per device orders the exchange: the next proposal kernel
        # waits on the flags -- no barrier kernel and no NCCL call per generation.
        # MC3B_P2P=0 falls back to the NCCL all-gather.
        self.p2p = None
        self._Xsym = None
        if world > 1 and self.shard == 'chains' and sampler != 'mrw' \
                and os.environ.get('MC3B_P2P', '1') != '0':
            try:
                self.p2p = self._setup_p2p(n, nfree)
            except Exception as e:                      # no peer access: NCCL path
                if rank == 0:
                    print(f'mc3_b200: peer-memory exchange unavailable ({e}); using NCCL all-gather')
                self.p2p = None
        if self.p2p is None:
            self._X = torch.zeros((n, nfree), **f64)
        self.chisq_cur = torch.zeros(n, **f64)
        if self.p2p is None or 'z' not in self.p2p:
            self.Z = torch.zeros((self.zlen, nfree), **f64)
        self.log_post = torch.zeros(self.zlen, **f64)
        self.zchain = torch.full((self.zlen,), -1, dtype=torch.int32, device=self.dev)
        self.nextp = torch.zeros((n, npars), **f64)
        self.mrfactor = torch.ones(n, **f64)
        self.u = torch.zeros(n, **f64)
        self.inb = torch.zeros(n, dtype=torch.int32, device=self.dev)
        self.naccept = torch.zeros(n, dtype=torch.int32, device=self.dev)
        self.outbounds = torch.zeros(nfree, dtype=torch.int32, device=self.dev)
        self.best_chisq = torch.full((n,), float('inf'), **f64)
        self.best_x = torch.zeros((n, nfree), **f64)
        self.best_gen = torch.zeros(n, dtype=torch.int64, device=self.dev)
        self.gen_dev = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.gen = 0                      # generations completed
        self.first_valid = self.M0        # first history row that is a chain sample
        self.resumed_rows, self.resumed_accept = None, 0     # of a resumed run (mcmc_driver._resume)
        self._gathered_k = 0              # thinned steps complete on every device (gather_history)
        self.bestp0 = np.copy(params)     # best of the initial population
        self.best_log_post0 = -np.inf

        # small populations run inside one persistent CTA (csrc/small.cu)
        self.small = (self.kind == 'builtin' and not self.wlike and world == 1
                      and self.dtype == _lib.F64 and self.nchains <= 64
                      and self.ndata <= 32768 and not os.environ.get('MC3B_NO_SMALL'))
        self._plans = {}
        self._work = {}
        self._graph = None
        self._block_graph = None
        # launch shape planned for `plan_chains` chains instead of the chains of each
        # launch: identical chi-squared bits however the population is spread over
        # launches / devices (include/mc3b200.h, mc3b_chisq_opts_t)
        self.plan_chains = int(plan_chains) if plan_chains else 0
        self._plan_rows = 0
        # Metropolis step fused into the tail of the model kernel (2 launches per
        # generation instead of 4); MC3B_NO_FUSE=1 keeps the separate kernels
        self.fused = (self.kind in ('builtin', 'cuda') and not self.wlike and self.shard == 'chains'
                      and not os.environ.get('MC3B_NO_FUSE'))
        self.fuse_done = torch.zeros(self.nlocal//8 + 8, dtype=torch.int32, device=self.dev)
        self.S = self._make_struct()
        self.set_jump_scales(fgamma, fepsilon)
        self.S.reflect = 1 if reflect else 0
        self.launches = 0                 # kernels launched by this object

    def _stage_model(self, func, lo, hi):
        """The model's inputs (d_x, d_xs), constants (d_kc) and 1/uncert on the device; returns the local x."""
        user = isinstance(func, CudaModel)
        self.kind = 'cuda' if user else 'builtin'
        self.nmodel = func.nmodel(self.nfunc)
        self.jit = func.handle(self.dtype) if user else None
        # model values are fp64 whatever the dtype, as mc3b_model_eval's
        self.jit_eval = func.handle(_lib.F64) if user else None
        nin = func.ninputs if user else 1
        # a CudaModel of run-time constants: the indparams after its inputs, flattened
        # (CudaModel.split_args); every rank builds its own copy
        xargs, kc = func.split_args(self.indparams) if user else (self.indparams, None)
        if nin > 1:
            # a CudaModel of several inputs: one 1-D array per input, in the order of
            # the arguments of its `model`
            xin = [np.ascontiguousarray(a, dtype=np.double) for a in xargs]
            if len(xin) != nin or any(a.ndim != 1 or a.size != self.ndata_total for a in xin):
                raise ValueError(f'CudaModel {func.name!r} takes {nin} inputs: it needs indparams=[x1, ..., '
                                 f'x{nin}], {nin} 1-D arrays with the same shape as data (got '
                                 f'{[np.shape(a) for a in self.indparams]} for data of {self.ndata_total})')
        x = np.ascontiguousarray(self.indparams[0], dtype=np.double)
        if x.size != self.ndata_total or x.ndim != 1:
            raise ValueError(f'{"CUDA" if user else "built-in"} models need indparams=[x] '
                             'with the same shape as data')
        x = x[lo:hi]
        self.d_x = torch.from_numpy(x).to(self.dev)
        # every input of the model on the device (d_xs[0] is d_x); their host array of
        # pointers is what mc3b_user_model_eval_consts takes
        self.d_xs = [self.d_x] + [torch.from_numpy(a[lo:hi]).to(self.dev) for a in xin[1:]] \
            if nin > 1 else [self.d_x]
        self.d_xptrs = _lib.ptrs(self.d_xs)
        # ... and its constants, fp64 (model values) and in the kernel's dtype; None: none
        self.d_kc = torch.from_numpy(kc).to(self.dev) if kc is not None and kc.size else None
        self.nconst = func.nconst if user else 0
        self.d_invsig = 1.0/self.d_uncert
        return x

    def _prepare_seg(self, x):
        """(x, data, 1/uncert) in the seg layout (include/mc3b200.h, tile_x), and the tiles' origins."""
        perm = torch.from_numpy(self.seg['perm']).to(self.dev)
        kx, kd = self.d_x[perm].contiguous(), self.d_data[perm].contiguous()
        kw = self.d_invsig if self.usig else self.d_invsig[perm].contiguous()
        self.d_tile_x = torch.from_numpy(np.ascontiguousarray(x[self.seg['starts']])).to(self.dev)
        return kx, kd, kw

    def _prepare_moment(self, x, kx, kd, form, c0r, slr, d2tot):
        """The moment form about the data's least-squares line c0r + slr x (sum of squares d2tot about
        it), which keeps the cancellation of the expansion at (signal/noise)^2: the mirrored pairs' sums,
        guard records and spectral table.  A guard in the kernel re-evaluates every chain the expansion
        is not accurate enough for; when that is not rare (_moment_policy) the pair kernel takes over."""
        self.d_mfold = torch.zeros_like(kd)
        self.d_mtiles = torch.zeros((max(form.nfold//128, 1), 4), dtype=torch.float64, device=self.dev)
        self.guard_hits = torch.zeros(1, dtype=torch.int32, device=self.dev)
        dxg = self.seg['dx'] if self.seg else float((x[-1] - x[0])/(x.size - 1))
        _lib.call('mc3b_moment_prepare', kd.data_ptr(), form.nfold//128, float(x[0]), dxg, _lib.ptr(self.d_tile_x),
                  c0r, slr, form.layout, self.d_mfold.data_ptr(), self.d_mtiles.data_ptr(), _lib.stream_ptr())
        if form.spectral_plan is not None:
            self._prepare_spectral(form.spectral_plan, kx, kd, c0r, slr)
        # the guard count of every generation, written by the fused epilogue into
        # page-locked host memory (include/mc3b200.h mc3b_moment_t.record)
        self._guard_ring = torch.empty(_lib.GUARD_RECORDS, dtype=torch.int64).pin_memory()
        dptr = ctypes.c_void_p()
        _lib.call('mc3b_host_device_pointer', self._guard_ring.data_ptr(), ctypes.byref(dptr))
        self._guard = GuardRecords(self._guard_ring.numpy())
        self.moment = _lib.MomentStruct(
            folded=self.d_mfold.data_ptr(), tiles=self.d_mtiles.data_ptr(), c0ref=c0r, slref=slr, d2tot=d2tot,
            amp_max=float(os.environ.get('MC3B_MOMENT_AMP', 4000.0)), xlo=float(x.min()), xhi=float(x.max()),
            guard_hits=self.guard_hits.data_ptr(), layout=form.layout, record=dptr.value,
            spectral=None if self.spectral is None else ctypes.pointer(self.spectral))
        self.use_moment = True

    def _prepare_spectral(self, plan, kx, kd, c0r, slr):
        """The spectral form's table: the data's spectrum on the nodes of `plan` (spectral.plan), from
        which the chi-squared of a chain takes O(1) instead of O(n)."""
        S = _lib.SpectralStruct(**{k: plan[k] for k in ('w1', 'w2', 'delta', 'xc', 'n1', 'n2', 'order')})
        size = ctypes.c_int64(0)
        _lib.call('mc3b_spectral_size', S.n1, S.n2, S.order, ctypes.byref(size))
        self.d_spectral = torch.zeros(size.value, dtype=torch.float64, device=self.dev)
        S.table = self.d_spectral.data_ptr()
        _lib.call('mc3b_spectral_prepare', kx.data_ptr(), kd.data_ptr(), self.ndata, c0r, slr,
                  ctypes.byref(S), _lib.stream_ptr())
        self.spectral = S

    # ------------------------------------------------------------------
    def _make_struct(self):
        S = _lib.SamplerStruct()
        S.nchains, S.chain0, S.nlocal = self.nchains, self.chain0, self.nlocal
        S.npars, S.nfree = self.npars, self.nfree
        S.sampler = _lib.SAMPLERS[self.sampler]
        S.reflect = 0
        S.ifree, S.pstep = self.d_ifree.data_ptr(), self.d_pstep.data_ptr()
        S.pmin, S.pmax = self.d_pmin.data_ptr(), self.d_pmax.data_ptr()
        S.params0 = self.d_params0.data_ptr()
        if self.has_prior:
            S.prior, S.priorlow = self.d_prior.data_ptr(), self.d_priorlow.data_ptr()
            S.priorup = self.d_priorup.data_ptr()
        S.gamma = 0.0
        S.fepsilon = 0.0
        S.seed = self.seed
        S.X, S.chisq_cur = self.X.data_ptr(), self.chisq_cur.data_ptr()
        S.world, S.rank = self.world, self.rank
        if self.p2p is not None:
            S.X_peers = self.p2p['x'].ptrs.data_ptr()
            S.F_peers = self.p2p['f'].ptrs.data_ptr()
            if 'z' in self.p2p:
                S.Z_peers = self.p2p['z'].ptrs.data_ptr()
        S.Z, S.log_post, S.zchain = (self.Z.data_ptr(), self.log_post.data_ptr(),
                                     self.zchain.data_ptr())
        S.zlen, S.M0 = self.zlen, self.M0
        S.nextp, S.mrfactor = self.nextp.data_ptr(), self.mrfactor.data_ptr()
        S.u, S.inb = self.u.data_ptr(), self.inb.data_ptr()
        S.naccept, S.outbounds = self.naccept.data_ptr(), self.outbounds.data_ptr()
        S.best_chisq, S.best_x = self.best_chisq.data_ptr(), self.best_x.data_ptr()
        S.best_gen = self.best_gen.data_ptr()
        S.gen_dev, S.thinning = self.gen_dev.data_ptr(), self.thinning
        return S

    @property
    def X(self):
        """Current population [nchains, nfree] (peer mode: the half of this generation)."""
        if self._Xsym is not None:
            return self._Xsym[self.gen & 1]
        return self._X

    def _setup_p2p(self, n, nfree):
        import torch.distributed as dist
        from .parallel import PeerBuffer
        grp = self.group
        args = (self, self.rank, self.world, grp, self.dev)
        out = {'x': PeerBuffer.get(2*n*nfree*8, 'x', *args),
               'f': PeerBuffer.get(max(self.world, 8)*8, 'f', *args)}
        self._Xsym = out['x'].local[:2*n*nfree].view(2, n, nfree)
        self._Xsym.zero_()
        out['f'].local.zero_()
        if self.sampler == 'snooker':
            out['z'] = PeerBuffer.get(self.zlen*nfree*8, 'z', *args)
            self.Z = out['z'].local[:self.zlen*nfree].view(self.zlen, nfree)
            self.Z.zero_()
        torch.cuda.synchronize(self.dev)
        dist.barrier(group=grp)                 # nobody stores into a peer before its buffers are zeroed
        return out

    def close(self):
        """Drop the captured graphs (they may hold NCCL kernels: destroy them before
        the process group) and release the peer buffers for reuse."""
        self._graph = None
        self._block_graph = None
        if torch.cuda.is_available():
            torch.cuda.synchronize(self.dev)

    def set_jump_scales(self, fgamma, fepsilon):
        self.S.gamma = float(fgamma)*2.38/np.sqrt(2*self.nfree)   # chain.py:175
        self.S.fepsilon = float(fepsilon)

    # ------------------------------------------------------------------
    # chi-squared of a batch of full parameter vectors
    # ------------------------------------------------------------------
    def _plan_chains(self, nb):
        """Chain count the launch shape of an nb-row launch is planned for: nb itself,
        or -- with plan_chains -- the whole population (`_plan_rows` while a larger
        batch, the initial-population trials, is evaluated in per-device blocks)."""
        if not self.plan_chains:
            return nb
        return max(self.plan_chains, self._plan_rows, nb)

    def _plan(self, nb, kind=0):
        """kind: 0 general, 1 moment form, 2 its spectral form (MC3B_PLAN_*)."""
        key = (self._plan_chains(nb), int(kind))
        if key not in self._plans:
            ns = ctypes.c_int(0)
            _lib.call('mc3b_model_chisq_plan_kind', key[1], key[0], self.ndata, self.dtype,
                      ctypes.byref(ns))
            self._plans[key] = ns.value
        return self._plans[key]

    def _workspace(self, key, shape, dtype=torch.float64):
        t = self._work.get(key)
        if t is None or tuple(t.shape) != tuple(shape):
            t = torch.empty(shape, dtype=dtype, device=self.dev)
            self._work[key] = t
        return t

    def _model_rows(self, P):
        """Model values [nb, N] on the device."""
        nb = P.shape[0]
        if self.kind in ('builtin', 'cuda'):
            rows = self._workspace(('mrows', nb), (nb, self.ndata))
            if self.kind == 'cuda':
                _lib.call('mc3b_user_model_eval_consts', self.jit_eval, P.data_ptr(), _lib.ld(P), nb,
                          self.d_xptrs, len(self.d_xs), _lib.ptr(self.d_kc), self.nconst, self.ndata,
                          rows.data_ptr(), _lib.stream_ptr())
            else:
                _lib.call('mc3b_model_eval', self.func.model_id, P.data_ptr(), _lib.ld(P), nb,
                          self.nmodel, self.d_x.data_ptr(), self.ndata, rows.data_ptr(), _lib.stream_ptr())
            self.launches += 1
            return rows
        if self.kind == 'torch':
            m = self.func.fn(P[:, :self.nfunc], *self.t_indparams, **self.indparams_dict)
            return m.to(torch.float64).contiguous()
        Ph = P.cpu().numpy()
        rows = np.empty((nb, self.ndata))
        for i in range(nb):     # the reference's per-chain host callable
            rows[i] = self.func(Ph[i, :self.nfunc], *self.indparams, **self.indparams_dict)
        return torch.from_numpy(rows).to(self.dev)

    @on_device
    def data_chisq(self, P, fuse=None, moment_ok=False):
        """(partial, ld, nsplit) holding the data chi-squared of rows of P.
        fuse = (c_off, gen, zrow0, advance): the model kernel also takes the
        Metropolis step of chains c_off .. c_off + len(P) (built-in models).
        moment_ok: the caller sums the rows with _finish() (which applies the guard
        of the sufficient-statistics form), not with mc3b_chisq_finish/mc3b_metropolis."""
        if self.shard == 'data':
            return self._data_chisq_sharded(P)
        return self._data_chisq_local(P, fuse, moment_ok)

    def _finish(self, part, ld, ns, nb, P, out, with_prior):
        """out[c] = rows of `part` added in split order (+ prior terms): mc3b_chisq_finish, or
        mc3b_moment_finish when the rows came from the unfused moment form."""
        pr = (self.d_prior.data_ptr(), self.d_priorlow.data_ptr(),
              self.d_priorup.data_ptr()) if (with_prior and self.has_prior) else (None, None, None)
        if self._part_is_moment:
            _lib.call('mc3b_moment_finish', ctypes.byref(self.moment), part.data_ptr(), ld, ns, nb,
                      P.data_ptr(), _lib.ld(P), self.npars, self.k_x.data_ptr(), self.k_d.data_ptr(),
                      self.k_w.data_ptr(), self.ndata, *pr, out.data_ptr(), _lib.stream_ptr())
        elif with_prior:
            _lib.call('mc3b_chisq_finish', part.data_ptr(), ld, ns, nb, P.data_ptr(),
                      _lib.ld(P), self.npars, *pr, out.data_ptr(), _lib.stream_ptr())
        else:
            _lib.call('mc3b_chisq_finish', part.data_ptr(), ld, ns, nb, None, 0, 0,
                      None, None, None, out.data_ptr(), _lib.stream_ptr())
        self.launches += 1

    def _data_chisq_sharded(self, P):
        """Local-slice sums, then an all-gather of one fp64 per chain and device;
        the caller adds the `world` rows in rank order (fixed order, identical
        bits on every device)."""
        import torch.distributed as dist
        nb = P.shape[0]
        part, ld, ns = self._data_chisq_local(P, None, True)
        allsum = self._workspace(('allsum', nb), (self.world, nb))
        self._finish(part, ld, ns, nb, P, allsum[self.rank], False)
        self._part_is_moment = False           # the gathered rows are plain sums
        dist.all_gather_into_tensor(allsum.view(-1), allsum[self.rank], group=self.group)
        return allsum, nb, self.world

    def _data_chisq_local(self, P, fuse=None, moment_ok=False):
        self._part_is_moment = False
        if self.wlike:
            return self._wavelet_chisq(P)
        if self.kind in ('builtin', 'cuda'):
            return self._model_chisq(P, fuse, moment_ok)
        nb, m = P.shape[0], self._model_rows(P)
        out = self._workspace(('rows', nb), (1, nb))
        _lib.call('mc3b_chisq_batch', m.data_ptr(), _lib.ld(m), nb, self.d_data.data_ptr(),
                  self.d_uncert.data_ptr(), self.ndata, out.data_ptr(), _lib.stream_ptr())
        self.launches += 1
        return out, nb, 1

    def _wavelet_chisq(self, P):
        """The wavelet likelihood (csrc/dwt.cu): one row of sums."""
        nb = P.shape[0]
        st = _lib.stream_ptr()
        out = self._workspace(('dwt', nb), (1, nb))
        ws_bytes = _lib.load().mc3b_dwt_workspace(nb, self.ndata)
        ws = self._workspace(('dwtws', nb), (max(ws_bytes, 8)//8,))
        if self.kind == 'builtin':
            _lib.call('mc3b_dwt_chisq', self.func.model_id, P.data_ptr(), _lib.ld(P), nb, self.npars, self.nmodel,
                      self.d_x.data_ptr(), None, 0, self.d_data.data_ptr(), self.ndata, ws.data_ptr(),
                      out.data_ptr(), st)
        elif self.kind == 'cuda':
            # the model is evaluated inside the D4 kernels of its fp64 module: no rows
            _lib.call('mc3b_user_model_dwt_chisq', self.jit_eval, P.data_ptr(), _lib.ld(P), nb,
                      self.npars, self.d_xptrs, len(self.d_xs), _lib.ptr(self.d_kc), self.nconst,
                      self.d_data.data_ptr(), self.ndata, ws.data_ptr(), out.data_ptr(), st)
        else:
            m = self._model_rows(P)
            _lib.call('mc3b_dwt_chisq', -1, P.data_ptr(), _lib.ld(P), nb, self.npars, 0, None, m.data_ptr(),
                      _lib.ld(m), self.d_data.data_ptr(), self.ndata, ws.data_ptr(), out.data_ptr(), st)
        self.launches += 2
        return out, nb, 1

    def _model_chisq(self, P, fuse, moment_ok):
        """The model + chi-squared kernel of a built-in or CUDA model in the population's form."""
        nb = P.shape[0]
        moment = self.use_moment and (fuse is not None or moment_ok)
        spec = moment and self.spectral is not None
        ns = self._plan(nb, 2 if spec else 1 if moment else 0)
        part = self._last_part = self._workspace(('part', nb, ns), (ns, nb))
        o = _lib.ChisqOpts()
        o.plan_chains = self._plan_chains(nb) if self.plan_chains else 0
        o.uniform_sigma = 1 if self.usig else 0
        if self.seg is not None:
            o.tile_x, o.dx, o.ntiles = self.d_tile_x.data_ptr(), self.seg['dx'], self.seg['starts'].size
        if self.d_fold is not None:
            o.folded = self.d_fold.data_ptr()
            if (not os.environ.get('MC3B_NO_FOLD_CONSTS') or moment) and not spec:
                o.work = self._workspace(('foldk', nb), (_lib.FOLD_WORK, nb)).data_ptr()
                self.launches += 1
        if moment:
            o.moment = ctypes.pointer(self.moment)
            self._part_is_moment = fuse is None
        if fuse is not None:
            o.c_off, o.gen, o.zrow0, adv = fuse
            o.advance = 1 if adv else 0
            o.fuse = ctypes.pointer(self.S)
            o.fuse_done = self.fuse_done.data_ptr()
        if self.kind == 'cuda':
            _lib.call('mc3b_user_model_chisq_consts', self.jit, P.data_ptr(), _lib.ld(P), nb, self.k_xptrs,
                      len(self.k_xs), _lib.ptr(self.k_kc), self.nconst, self.k_d.data_ptr(), self.k_w.data_ptr(),
                      self.ndata, part.data_ptr(), nb, ns, ctypes.byref(o), _lib.stream_ptr())
        else:
            _lib.call('mc3b_model_chisq_ex', self.chisq_model_id, self.dtype, P.data_ptr(), _lib.ld(P), nb,
                      self.nmodel, self.k_x.data_ptr(), self.k_d.data_ptr(), self.k_w.data_ptr(), self.ndata,
                      part.data_ptr(), nb, ns, ctypes.byref(o), _lib.stream_ptr())
        self.launches += 1
        return part, nb, ns

    @on_device
    def model_eval(self, fpar):
        """Built-in or CUDA model at one parameter vector over the (device-resident)
        abscissa, as a host array (chain.py:316-319 `func(params, *indparams)`)."""
        P = torch.as_tensor(np.atleast_2d(np.asarray(fpar, dtype=np.double)), device=self.dev)
        return to_host(self._model_rows(P)[0])

    @on_device
    def chisq(self, P):
        """chi-squared + prior terms of full parameter vectors P [nb, npars]."""
        P = P.contiguous()
        nb = P.shape[0]
        part, ld, ns = self.data_chisq(P, moment_ok=True)
        out = torch.empty(nb, dtype=torch.float64, device=self.dev)
        self._finish(part, ld, ns, nb, P, out, True)
        return out

    # ------------------------------------------------------------------
    # initial population   (mcmc_driver.py:229-278)
    # ------------------------------------------------------------------
    @on_device
    def init_population(self, kickoff='normal'):
        kick = {'normal': 0, 'uniform': 1}[kickoff]
        M0 = self.M0
        got = 0
        tried = 0
        rnd = 0
        rows, lps = [], []
        while got < M0 and tried < 100*M0:
            nt = int(min(max(M0 - got, 64)*1.25 + 64, 100*M0 - tried))
            trial = torch.empty((nt, self.npars), dtype=torch.float64, device=self.dev)
            ok = torch.empty(nt, dtype=torch.int32, device=self.dev)
            _lib.call('mc3b_init_trials', ctypes.byref(self.S), kick, nt, rnd,
                      trial.data_ptr(), ok.data_ptr(), _lib.stream_ptr())
            self.launches += 1
            # Trials are used in draw order until M0 rows are in (mcmc_driver.py:246-262):
            # evaluate the in-bounds ones up to the count still needed (+1% against
            # non-finite models), not the whole over-drawn batch.
            inb = torch.nonzero(ok != 0).flatten()
            need = M0 - got
            inb = inb[:need + max(8, need//100)]
            tried += int(inb[-1]) + 1 if inb.numel() else nt
            if inb.numel():
                cand = trial[inb]
                lp = self._trial_log_post(cand)
                idx = torch.nonzero(torch.isfinite(lp)).flatten()[:need]
                rows.append(cand[idx])
                lps.append(lp[idx])
                got += idx.numel()
            rnd += 1
        if got < M0:
            raise ValueError(
                'Cannot populate an initial sample set of parameters, try '
                'updating the parameters initial guess to avoid sampling '
                'beyond the parameter boundaries or where the model returns '
                'non-finite values.')
        full = torch.cat(rows)
        self.set_initial(full[:, self.d_ifree.long()], torch.cat(lps))

    def _trial_log_post(self, trial):
        """log-posterior of the initial-population trials.  With the chains
        partitioned over devices each device evaluates a contiguous block of the
        rows and the blocks are all-gathered (the trials themselves are Philox
        draws every device generates identically)."""
        nt = trial.shape[0]
        self._plan_rows = nt          # one launch shape for the batch, however it is split over devices
        try:
            return self._trial_log_post_blocks(trial, nt)
        finally:
            self._plan_rows = 0

    def _trial_log_post_blocks(self, trial, nt):
        if self.world == 1 or self.shard != 'chains':
            return -0.5*self.chisq(trial)
        per = -(-nt//self.world)
        buf = torch.full((self.world*per, 1), float('nan'), dtype=torch.float64,
                         device=self.dev)
        lo = min(self.rank*per, nt)
        hi = min(lo + per, nt)
        if hi > lo:
            buf[self.rank*per:self.rank*per + (hi - lo), 0] = -0.5*self.chisq(trial[lo:hi])
        allgather_rows(buf, self.rank*per, per, self.group)
        return buf[:nt, 0].contiguous()

    @on_device
    def set_initial(self, Z0, log_post0):
        """Install M0 initial history rows and start every chain from row c
        (chain.py:163-170: chain c starts at Z[c], chisq = -2 log_post[c])."""
        Z0 = torch.as_tensor(Z0, dtype=torch.float64, device=self.dev)
        lp0 = torch.as_tensor(log_post0, dtype=torch.float64, device=self.dev)
        assert Z0.shape == (self.M0, self.nfree)
        self.Z[:self.M0] = Z0
        self.log_post[:self.M0] = lp0
        if self._Xsym is not None:
            import torch.distributed as dist
            self._Xsym[0].copy_(self.Z[:self.nchains])
            self._Xsym[1].copy_(self.Z[:self.nchains])
            torch.cuda.synchronize(self.dev)    # peers may store into our halves after this barrier only
            dist.barrier(group=self.group)
        else:
            self._X.copy_(self.Z[:self.nchains])
        self.chisq_cur.copy_(-2.0*self.log_post[:self.nchains])
        iz = int(torch.argmax(lp0))                  # mcmc_driver.py:273-275
        self.best_log_post0 = float(lp0[iz])
        self.bestp0 = np.copy(self.params)
        self.bestp0[self.ifree] = Z0[iz].cpu().numpy()
        for s in self.ishare:
            self.bestp0[s] = self.bestp0[-int(self.pstep[s]) - 1]

    # ------------------------------------------------------------------
    # one lock-step generation
    # ------------------------------------------------------------------
    def _zrow0(self, gen):
        if (gen + 1) % self.thinning:
            return -1
        return self.M0 + ((gen + 1)//self.thinning - 1)*self.nchains

    def _generation(self, gen):
        """gen >= 0: host-driven; gen < 0: device-driven (graph capture)."""
        st = _lib.stream_ptr()
        c0, c1 = self.chain0, self.chain0 + self.nlocal
        zsize = self.M0 + (gen//self.thinning)*self.nchains if gen >= 0 else 0
        _lib.call('mc3b_propose', ctypes.byref(self.S), gen, zsize, c0, c1, st)
        self.launches += 1
        zrow0 = self._zrow0(gen) if gen >= 0 else -1
        # the generation counter may advance inside the fused kernel only when no
        # later launch of this generation reads it
        # peer mode: the kernel that ends the generation advances the counter and
        # publishes this device's generation flag (host-driven generations too)
        nccl = self.world > 1 and self.shard == 'chains' and self.p2p is None
        adv = (gen < 0 and not nccl) or self.p2p is not None
        if self.fused:
            self.data_chisq(self.nextp[c0:c1], fuse=(c0, gen, zrow0, adv))
        else:
            part, ld, ns = self.data_chisq(self.nextp[c0:c1])
            _lib.call('mc3b_metropolis', ctypes.byref(self.S), part.data_ptr(), ld, ns,
                      c0, gen, zrow0, c0, c1, st)
            self.launches += 1
        if nccl:
            self._exchange(gen)
        if (adv and not self.fused) or (gen < 0 and nccl):
            _lib.call('mc3b_advance', ctypes.byref(self.S), st)
            self.launches += 1

    def _exchange(self, gen):
        """Per-generation population exchange across devices (SURVEY 8e): demc
        needs every chain's current state, snooker the new history rows.  Peer
        mode: the stores were issued by k_metropolis; one signal-pad barrier
        orders them.  NCCL mode: all-gather of X (demc) / of the new rows (snooker)."""
        if self.sampler == 'demc':
            allgather_rows(self._X, self.chain0, self.nlocal, self.group)
        elif self.sampler == 'snooker':
            if gen < 0:
                raise _lib.Mc3bError('multi-GPU snooker over NCCL runs host-driven generations')
            r0 = self._zrow0(gen)
            if r0 >= 0:
                allgather_rows(self.Z[r0:r0 + self.nchains], self.chain0,
                               self.nlocal, self.group)

    def _capture(self, ngens):
        """CUDA graph of `ngens` device-driven generations.  Captured on a side
        stream with capture_begin/capture_end directly: torch.cuda.graph()'s
        gc.collect + empty_cache cost ~10 ms, a fifth of a 200-generation run."""
        g = torch.cuda.CUDAGraph()
        before = self.launches
        cur = torch.cuda.current_stream(self.dev)
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            g.capture_begin()
            try:
                for _ in range(ngens):
                    self._generation(-1)
            finally:
                g.capture_end()
        cur.wait_stream(side)
        per = self.launches - before
        self.launches = before
        return g, per

    @on_device
    def run(self, ngen, use_graph=None):
        """Advance `ngen` generations.  Built-in models replay captured CUDA
        graphs; small problems (launch-latency bound) replay graphs that hold a
        block of generations."""
        if ngen <= 0:
            return
        if use_graph is None:
            # A generation with >= ~0.3 ms of device work hides its three host
            # launches completely: skip the capture (10-15 ms) and run eagerly.
            # (single device only: an eager NCCL all-gather per generation costs the
            # host more than the generation itself, 0.69 vs 0.24 ms at 8 GPUs)
            heavy = float(self.nlocal)*self.ndata > 2e8 and not self.small and self.world == 1
            use_graph = self.kind in ('builtin', 'cuda') and not heavy and not \
                (self.world > 1 and self.shard == 'chains' and self.sampler == 'snooker'
                 and self.p2p is None)
        if self.use_moment:
            # the persistent small-population kernel never runs the moment form, and
            # unfused generations write no guard records
            self._moment_policy(ngen, self.fused and not (use_graph and self.small))
        if use_graph and self.small:
            # launch-latency-bound population: all generations inside one resident CTA
            done = 0
            while done < ngen:
                step = min(ngen - done, 200000)
                _lib.call('mc3b_run_small', ctypes.byref(self.S), self.func.model_id,
                          self.nmodel, self.d_x.data_ptr(), self.d_data.data_ptr(),
                          self.d_invsig.data_ptr(), self.ndata,
                          self.gen + done, step, _lib.stream_ptr())
                done += step
            self.launches += 1
            self.gen += ngen
            return
        if not use_graph:
            if self.p2p is not None:
                self.gen_dev.fill_(self.gen)     # the device counter advances with every generation
            for g in range(self.gen, self.gen + ngen):
                self._generation(g)
            self.gen += ngen
            self.gen_dev.fill_(self.gen)
            return
        if self._graph is None:
            self.gen_dev.fill_(self.gen)
            self._generation(self.gen)          # warm-up outside capture
            self.gen += 1
            self.gen_dev.fill_(self.gen)
            ngen -= 1
            torch.cuda.synchronize(self.dev)
            self._graph, self._graph_launches = self._capture(1)
            # generations per block graph: aim at >= ~0.3 ms of device work per replay
            work = float(self.nlocal)*self.ndata
            self._block = 1 if work > 2e8 else (8 if work > 2e7 else 32)
            self._block_graph = None
        if self._block > 1 and ngen >= self._block:
            if self._block_graph is None:
                self._block_graph, _ = self._capture(self._block)
            nb = ngen // self._block
            for _ in range(nb):
                self._block_graph.replay()
            done = nb*self._block
            self.launches += done*self._graph_launches
            self.gen += done
            ngen -= done
        for _ in range(ngen):
            self._graph.replay()
        self.launches += ngen*self._graph_launches
        self.gen += ngen

    def _moment_policy(self, ngen, recording):
        """Decide, at the start of a run() call of `ngen` generations, whether the
        generation loop keeps the sufficient-statistics kernel.  Before the first
        generation the amplification is estimated from the best chi-squared of the
        initial population; after that the guard records decide (GuardRecords.step).
        recording: this call's generations run the fused moment kernel."""
        M = self.moment
        if self.gen == 0 and np.isfinite(self.best_log_post0):
            n, w0 = self.ndata, 1.0/float(self.host_uncert0)
            mag = abs(float(self.bestp0[0]))*np.sqrt(n) + np.sqrt(M.d2tot)
            if mag*mag*w0*w0 > 0.5*M.amp_max*max(-2.0*self.best_log_post0, 1e-300):
                self._moment_off()
                return
        idle = torch.cuda.current_stream(self.dev).query
        if self._guard.step(self.gen, ngen, self.nlocal, recording, idle):
            self._moment_off()

    def _moment_off(self):
        self.use_moment = False
        self._guard.starts = []
        self._graph = None
        self._block_graph = None

    # ------------------------------------------------------------------
    # replay of the reference's recorded stream (sequential chain order)
    # ------------------------------------------------------------------
    @on_device
    def replay(self, draws, ngen=None):
        """draws: dict of arrays from oracle DrawLog.arrays() (normal, a, b, iz,
        usj, gs, u, done).  Chains are stepped one at a time for demc/snooker
        (chain j sees chains < j already moved, chain.py:190-289)."""
        G = int(draws['ngen']) if ngen is None else int(ngen)
        dv = {}
        for k in ('normal', 'usj', 'gs', 'u'):
            dv[k] = torch.as_tensor(np.ascontiguousarray(draws[k]),
                                    dtype=torch.float64, device=self.dev)
        for k in ('a', 'b', 'iz'):
            dv[k] = torch.as_tensor(np.ascontiguousarray(draws[k]),
                                    dtype=torch.int64, device=self.dev)
        done = np.asarray(draws['done'])
        st = _lib.stream_ptr()
        n = self.nchains
        D = _lib.DrawsStruct()
        for g in range(G):
            D.normal = dv['normal'][g].data_ptr()
            for k in ('a', 'b', 'iz', 'usj', 'gs', 'u'):
                setattr(D, k, dv[k][g].data_ptr())
            nd = int(done[g].sum())               # chains that ran this generation
            complete = nd == n
            zrow0 = self._zrow0(self.gen) if complete else -1
            if self.sampler == 'mrw':
                groups = [(0, nd)]
            else:
                groups = [(c, c + 1) for c in range(nd)]
            for c0, c1 in groups:
                _lib.call('mc3b_propose_replay', ctypes.byref(self.S),
                          ctypes.byref(D), c0, c1, st)
                part, ld, ns = self.data_chisq(self.nextp[c0:c1])
                _lib.call('mc3b_metropolis', ctypes.byref(self.S), part.data_ptr(),
                          ld, ns, c0, self.gen, zrow0, c0, c1, st)
                self.launches += 2
            self.gen += 1
        self.gen_dev.fill_(self.gen)

    # ------------------------------------------------------------------
    # hub-side reads
    # ------------------------------------------------------------------
    def thinned_done(self):
        return self.gen//self.thinning

    def zsize(self):
        return self.M0 + self.thinned_done()*self.nchains

    @on_device
    def gather_history(self, dst=None):
        """Make Z / log_post / zchain complete on every device, or on device `dst`
        only (no-op at world=1 and for data sharding, where the history is
        replicated).  Rows already complete (gathered earlier, or stored to every
        device as they were written) are not sent again."""
        if self.shard == 'data' or self.world == 1:
            return
        K = self.thinned_done()
        k0 = self._gathered_k
        if K <= k0:
            return
        lo = self.M0 + k0*self.nchains
        for t in (self.Z, self.log_post, self.zchain):
            if t is self.Z and self.sampler == 'snooker':
                continue                     # snooker exchanges its rows every generation
            gather_history(t, lo, K - k0, self.nchains, self.rank, self.world,
                           self.group, dst)
        if dst is None:
            self._gathered_k = K

    def counters_async(self):
        """Enqueue the report-point counters (one pack kernel, one collective at
        world > 1, one D2H into pinned memory) and return a handle; nothing blocks.
        counters_result(handle) turns it into the dictionary."""
        with torch.cuda.device(self.dev):
            n = 4 + 2*self.nfree
            gathered = self.world > 1 and self.shard == 'chains'
            rows = self.world if gathered else 1
            buf = self._workspace('pack', (rows, n))
            mine = buf[self.rank if gathered else 0]
            _lib.call('mc3b_pack_counters', ctypes.byref(self.S), mine.data_ptr(),
                      _lib.stream_ptr())
            self.launches += 1
            if gathered:
                import torch.distributed as dist
                if dist.get_backend(self.group) == 'nccl':
                    dist.all_gather_into_tensor(buf.view(-1), mine, group=self.group)
                else:
                    parts = [torch.empty_like(mine) for _ in range(self.world)]
                    dist.all_gather(parts, mine.clone(), group=self.group)
                    buf.copy_(torch.stack(parts))
            host = torch.empty((rows, n), dtype=torch.float64, pin_memory=True)
            host.copy_(buf, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            return host, ev

    def counters_result(self, handle):
        """chain.py:268-274 -- first strictly lower chi-squared in (generation,
        chain) order wins, starting from the best of the initial population."""
        host, ev = handle
        ev.synchronize()
        h = host.numpy()
        nf = self.nfree
        numaccept = int(round(h[:, 0].sum())) + self.resumed_accept
        outbounds = np.rint(h[:, 4 + nf:4 + 2*nf].sum(axis=0)).astype(int)
        best_chisq = -2.0*self.best_log_post0
        bestp = np.copy(self.bestp0)
        cand = [r for r in h if r[3] >= 0 and r[1] < best_chisq]
        if cand:
            r = min(cand, key=lambda r: (r[1], r[2], r[3]))
            best_chisq = float(r[1])
            bestp[self.ifree] = r[4:4 + nf]
            for s in self.ishare:
                bestp[s] = bestp[-int(self.pstep[s]) - 1]
        return dict(numaccept=numaccept, outbounds=outbounds, bestp=bestp,
                    best_log_post=-0.5*best_chisq)

    def counters(self):
        """Host copy of the counters (summed over devices)."""
        return self.counters_result(self.counters_async())

    @on_device
    def history_host(self, dst=None):
        """(posterior, zchain, log_post, chisq) of the valid rows as numpy arrays;
        chisq = -2 (log_post - log_prior) comes from the device (mc3b_log_prior).
        dst: only that device receives the other devices' rows and copies the
        history to its host; the others return empty arrays."""
        self.gather_history(dst)
        lo, hi = self.first_valid, self.zsize()
        if dst is not None and self.world > 1 and self.rank != dst:
            hi = lo
        if hi <= lo:
            z = np.zeros((0, self.nfree))
            return z, np.zeros(0, int), np.zeros(0), np.zeros(0)
        chisq = torch.empty(hi - lo, dtype=torch.float64, device=self.dev)
        _lib.call('mc3b_log_prior', self.Z[lo:hi].data_ptr(), hi - lo, self.nfree,
                  self.d_ifree.data_ptr(), self.d_prior.data_ptr(),
                  self.d_priorlow.data_ptr(), self.d_priorup.data_ptr(),
                  self.log_post[lo:hi].data_ptr(), None, chisq.data_ptr(),
                  _lib.stream_ptr())
        self.launches += 1
        return (to_host(self.Z[lo:hi]), to_host(self.zchain[lo:hi]).astype(int),
                to_host(self.log_post[lo:hi]), to_host(chisq))

    @on_device
    def sample_statistics(self, zburn, quantile=0.683):
        """median, mean, std and central-quantile bounds of the burned posterior,
        per free parameter, computed on the device over the lock-step block of
        rows after burn-in (stats.py:764-802 'med_central'; numpy's linear
        percentile rule) and fetched with one copy.  Sorting is torch.sort:
        post-processing, not the hot path."""
        lo, hi = self.M0 + zburn*self.nchains, self.zsize()
        return tuple(column_statistics(self.Z[lo:hi], quantile).cpu().numpy())

    def gelman_rubin_async(self, zburn):
        """PSRF per free parameter over every chain's samples after burn-in
        (gelman.py:36-92), left on the device: returns (pinned host tensor, event)
        or None when there are not enough samples.  Each device reduces ITS chains
        to mean / variance; with the chains partitioned over devices the two
        [nchains, nfree] moment blocks are all-gathered (not the history) and every
        device evaluates the same fixed-order sums over all chains."""
        with torch.cuda.device(self.dev):
            K = self.thinned_done()
            rows, ldr, burn = None, 0, zburn
            if self.first_valid == 0:        # resumed run: earlier samples count (chain.py:166-169)
                rows_t, counts = self._resumed_rows()
                niter = int(counts.min()) - zburn
                rows, ldr = rows_t.data_ptr(), rows_t.shape[1]
            else:
                niter = K - zburn
            if niter < 1:
                return None
            st = _lib.stream_ptr()
            work = self._workspace('gr', (2, self.nchains, self.nfree))
            c0, c1 = self.chain0, self.chain0 + self.nlocal
            _lib.call('mc3b_gelman_rubin_moments', self.Z.data_ptr(), self.nfree, self.nchains,
                      self.M0, rows, ldr, burn, niter, c0, c1, work.data_ptr(), st)
            if self.world > 1 and self.shard == 'chains':
                allgather_rows(work[0], self.chain0, self.nlocal, self.group)
                allgather_rows(work[1], self.chain0, self.nlocal, self.group)
            psrf = self._workspace('psrf', (self.nfree,))
            _lib.call('mc3b_gelman_rubin_psrf', work.data_ptr(), self.nfree, self.nchains,
                      niter, psrf.data_ptr(), st)
            self.launches += 2
            host = torch.empty(self.nfree, dtype=torch.float64, pin_memory=True)
            host.copy_(psrf, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            return host, ev

    def _resumed_rows(self):
        """Row table [nchains, count] of a resumed history: each chain's earlier
        samples in file order, then its new rows (lock-step layout)."""
        K = self.thinned_done()
        old = self.resumed_rows            # list of int64 arrays, one per chain
        counts = np.array([len(o) for o in old]) + K
        n = int(counts.min())
        tab = np.empty((self.nchains, n), dtype=np.int64)
        new = self.M0 + np.arange(K)[None, :]*self.nchains + np.arange(self.nchains)[:, None]
        for c in range(self.nchains):
            tab[c] = np.concatenate([old[c], new[c]])[:n]
        return torch.from_numpy(tab).to(self.dev), counts

    def chain_counts_min(self):
        """Samples per chain as the reference's `chainsize` counts them, minus hsize
        (mcmc_driver.py:178-184, 325): thinned generations done, plus on a resumed
        run the shortest chain of the file."""
        K = self.thinned_done()
        if self.first_valid == 0:
            return K + min(len(o) for o in self.resumed_rows) - self.hsize
        return K

    def gelman_rubin(self, zburn):
        """PSRF per free parameter over the thinned samples after burn-in."""
        h = self.gelman_rubin_async(zburn)
        if h is None:
            return np.zeros(self.nfree)
        h[1].synchronize()
        return h[0].numpy().copy()
