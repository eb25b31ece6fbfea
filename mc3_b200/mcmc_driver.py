"""The MCMC hub: same call signature and output dictionary as the reference's
mc3.mcmc_driver.mcmc (mc3/mcmc_driver.py:18-378), with the forked Chain
processes, shared ctypes arrays and pipes replaced by one device-resident
Population (engine.py) advanced in lock-step by CUDA kernels.

What is kept from the reference, line for line in behaviour:
  sizes          nzchain, niter, zlen, zburn, grnmin rule   mcmc_driver.py:116-198
  initial set    hsize*nchains accepted draws, best of them  :229-278
  reports        every 10%: progress, out-of-bounds, best, savefile, GR test,
                 grbreak early stop                          :297-348
  output         update_output keys                          stats.py:805-852
What differs by design: chains advance together (Jacobi order) and random
numbers come from per-chain Philox streams, so runs agree with the reference
statistically, not draw for draw (use Population.replay for the latter).
"""
import time

import numpy as np
import torch

from . import stats as ms
from . import utils as mu
from .engine import Population
from .models import BuiltinModel, TorchModel


def eval_model(pop, params, ret='model'):
    """Chain.eval_model for one parameter vector (chain.py:302-340), on the GPU."""
    P = torch.as_tensor(np.atleast_2d(np.asarray(params, float)), device=pop.dev)
    chisq = float(pop.chisq(P)[0])
    if ret == 'chisq':
        return chisq
    fpar = np.asarray(params, float)[:pop.nfunc]
    if pop.kind in ('builtin', 'cuda') and pop.shard != 'data':
        model = pop.model_eval(fpar)          # abscissa already on the device
    else:
        model = pop.func(fpar, *pop.indparams, **pop.indparams_dict)
    return (model, chisq) if ret == 'both' else model


def calc_bestfit_statistics(bestp, pop):
    """stats.py:855-873."""
    ndata = pop.ndata_total
    best_model, opt_chisq = eval_model(pop, bestp, 'both')
    best_log_post = -0.5*opt_chisq
    best_log_prior = ms.log_prior(bestp[pop.ifree], pop.prior, pop.priorlow,
                                  pop.priorup, pop.pstep)
    best_chisq = -2*(best_log_post - best_log_prior)
    bic = best_chisq + pop.nfree*np.log(ndata)
    red = best_chisq/(ndata - pop.nfree) if ndata > pop.nfree else np.nan
    data = pop.host_data
    return best_chisq, red, bic, best_log_post, best_model, np.std(best_model - data)


def update_output(output, pop, hsize, counters=None):
    """stats.py:805-852 -- fill the output dict from the device state.  The
    chi-squared column and, for a lock-step history, the burned-sample
    statistics are computed on the device; only results travel to the host."""
    zburn = output['burnin']
    root = pop.world == 1 or pop.rank == 0
    # chains partitioned over devices: only rank 0 receives the other devices'
    # rows and copies the history to its host
    dst = 0 if (pop.world > 1 and pop.shard == 'chains') else None
    Z, zchain, log_post, chisq = pop.history_host(dst)
    c = counters or pop.counters()
    nsample = (pop.zsize() - pop.first_valid)*pop.thinning
    output['posterior'] = Z
    output['zchain'] = zchain
    output['chisq'] = chisq
    output['log_post'] = log_post
    output['acceptance_rate'] = c['numaccept']*100.0/max(nsample, 1)
    bestp = c['bestp']
    best = calc_bestfit_statistics(bestp, pop)
    output['bestp'] = bestp
    (output['best_chisq'], output['red_chisq'], output['BIC'],
     output['best_log_post'], output['best_model'],
     output['stddev_residuals']) = best
    if not pop.thinned_done() > zburn:
        return None
    if not root:
        return (pop.thinned_done() - zburn)*pop.nchains
    if pop.first_valid == pop.M0:          # lock-step layout: closed-form burn mask
        K, n = pop.thinned_done(), pop.nchains
        zmask = (np.arange(zburn, K)[None, :]*n + np.arange(n)[:, None]).ravel()
        st = ms.expand_free_stats(pop.sample_statistics(zburn), bestp, pop.pstep)
        nburned = zmask.size
    else:                                  # resumed history: general host path
        posterior, _, zmask = mu.burn(Z=Z, zchain=zchain, burnin=zburn)
        st = ms.calc_sample_statistics(posterior, bestp, pop.pstep)
        nburned = len(posterior)
    output['zmask'] = zmask
    (output['medianp'], output['meanp'], output['stdp'],
     output['median_low_bounds'], output['median_high_bounds']) = st
    return nburned


def mcmc(data, uncert, func, params, indparams, indparams_dict,
         pmin, pmax, pstep, prior, priorlow, priorup, nchains, ncpu, nsamples,
         sampler, wlike, fit_output, grtest, grbreak, grnmin, burnin, thinning,
         fgamma, fepsilon, hsize, kickoff, savefile, resume, log,
         pnames, texnames, seed=None, dtype='f64', device=None, use_graph=None,
         rank=0, world=1, group=None, reflect=False, return_population=False,
         shard='chains', plan_chains=None):
    """Reference signature (mcmc_driver.py:18-26; `ncpu` is accepted and
    ignored) plus keyword-only device options."""
    pstep = np.asarray(pstep, float)
    nfree = int(np.sum(pstep > 0))
    ifree = np.where(pstep > 0)[0]
    nchains, thinning, hsize = int(nchains), int(thinning), int(hsize)

    M0 = pre_zsize = hsize*nchains
    oldrun = None
    if resume:
        oldrun = np.load(savefile)
        M0 = pre_zsize = oldrun['posterior'].shape[0]

    nzchain = int(np.ceil(nsamples/nchains/thinning))      # mcmc_driver.py:129-134
    niter = nzchain*thinning
    burnin = int(burnin)
    if not resume and niter < burnin:
        log.error(
            f"The number of burned-in samples ({burnin}) is greater than "
            f"the number of iterations per chain ({niter})")
    zburn = int(burnin/thinning)

    if grnmin >= 1:                                          # :186-198
        grnmin = int(grnmin/thinning)
    elif grnmin > 0:
        grnmin = int(grnmin*nchains*(nzchain - zburn))
    elif grnmin < 0:
        log.error(
            "Invalid 'grnmin' argument (minimum number of samples to "
            "stop the MCMC under GR convergence), must either be grnmin > 1"
            "to set the minimum number of samples, or 0 < grnmin < 1"
            "to set the fraction of samples required to evaluate.")
    grnmin += int(M0 + zburn*nchains)

    if seed is None:
        seed = int(np.random.randint(0, 2**31 - 1))
    pop = Population(
        data, uncert, func, params, indparams, indparams_dict, pstep, pmin,
        pmax, prior, priorlow, priorup, nchains=nchains, sampler=sampler,
        wlike=wlike, fgamma=fgamma, fepsilon=fepsilon, hsize=hsize,
        thinning=thinning, nzchain=nzchain, seed=seed, dtype=dtype,
        device=device, rank=rank, world=world, group=group, reflect=reflect,
        M0=M0, shard=shard, plan_chains=plan_chains)

    if resume:
        _resume(pop, oldrun)
    else:
        try:
            pop.init_population(kickoff)
        except ValueError as e:
            log.error(str(e))
        if fit_output is not None:                           # :276-278
            pop.bestp0 = np.copy(fit_output['bestp'])
            pop.best_log_post0 = float(fit_output['best_log_post'])

    output = {'pnames': pnames, 'texnames': texnames, 'pstep': pstep,
              'ifree': ifree, 'burnin': zburn}

    if rank == 0:
        print("Yippee Ki Yay Monte Carlo!")
    log.msg(f"Start MCMC chains  ({time.ctime()})")
    # Reports every tenth of the run, on whole thinned generations (:297-348).
    # A report is enqueued behind its block of generations (one pack kernel, the
    # Gelman-Rubin kernels, one D2H each into pinned memory) and printed when its
    # copies have landed: the device never waits for the host between blocks.  The
    # host only blocks where the reference's control flow needs the numbers: a
    # savefile to write, or a grbreak decision.
    step_k = max(1, int(np.ceil(nzchain/10)))
    k_done = 0
    pending = []

    def flush(block):
        """Print finished reports in order; True when one of them stops the run."""
        while pending:
            kd, hc, hg, zs = pending[0]
            if not block and not (hc[1].query() and (hg is None or hg[1].query())):
                return False
            pending.pop(0)
            if log.verb >= 2:                # (formatting the arrays costs more than the report)
                c = pop.counters_result(hc)
                log.progressbar(kd/nzchain)
                log.msg(
                    f"Out-of-bound Trials:\n{c['outbounds']}\n"
                    f"Best Parameters: (chisq={-2*c['best_log_post']:.4f})\n"
                    f"{c['bestp'][ifree]}", width=80)
            if hg is not None:
                hg[1].synchronize()
                psrf = hg[0].numpy()
                if log.verb >= 2:
                    log.msg(f"Gelman-Rubin statistics for free parameters:\n{psrf}",
                            width=80)
                    if np.all(psrf < 1.01):
                        log.msg("All parameters converged to within 1% of unity.")
                if grbreak > 0.0 and np.all(psrf < grbreak) and zs > grnmin:
                    log.msg(
                        "\nAll parameters satisfy the GR convergence "
                        f"threshold of {grbreak:g}, stopping the MCMC.")
                    pending.clear()
                    return True
        return False

    while k_done < nzchain:
        k_next = min(nzchain, k_done + step_k)
        pop.run((k_next - k_done)*thinning, use_graph=use_graph)
        k_done = k_next
        hc = pop.counters_async()
        hg = None
        if grtest and pop.chain_counts_min() > zburn:          # :325
            hg = pop.gelman_rubin_async(zburn)
        pending.append((k_done, hc, hg, pop.zsize()))
        if savefile is not None:
            # every device takes part (the history gather is collective); rank 0 writes
            flush(True)
            update_output(output, pop, hsize, pop.counters())
            if rank == 0:
                np.savez(savefile, **output)
        if flush(block=(grbreak > 0.0 and hg is not None) or k_done == nzchain):
            break

    nburned = update_output(output, pop, hsize)
    Z = output['posterior']
    nsample = len(Z)*thinning
    nzsample = 0 if nburned is None else nburned
    fmt = len(str(nsample))
    log.msg('\nMCMC Summary:\n-------------')
    log.msg(
        f"Number of evaluated samples:        {nsample:{fmt}d}\n"
        f"Number of parallel chains:          {nchains:{fmt}d}\n"
        f"Average iterations per chain:       {nsample//nchains:{fmt}d}\n"
        f"Burned-in iterations per chain:     {burnin:{fmt}d}\n"
        f"Thinning factor:                    {thinning:{fmt}d}\n"
        f"MCMC sample size (thinned, burned): {nzsample:{fmt}d}\n"
        f"Acceptance rate:   {output['acceptance_rate']:.2f}%\n", indent=2)
    if return_population:
        output['_population'] = pop
    return output


def _resume(pop, oldrun):
    """mcmc_driver.py:178-184, 223-227 + chain.py:166-169: previous samples
    become the initial history; every chain restarts from its last row."""
    zold = np.asarray(oldrun['posterior'], float)
    zc = np.asarray(oldrun['zchain']).astype(int)
    lp = np.asarray(oldrun['log_post'], float)
    M0 = zold.shape[0]
    pop.Z[:M0] = torch.as_tensor(zold, device=pop.dev)
    pop.log_post[:M0] = torch.as_tensor(lp, device=pop.dev)
    pop.zchain[:M0] = torch.as_tensor(zc, dtype=torch.int32, device=pop.dev)
    order = np.argsort(zc, kind='stable')           # each chain's rows, in file order
    zs = zc[order]
    lo = np.searchsorted(zs, np.arange(pop.nchains), side='left')
    hi = np.searchsorted(zs, np.arange(pop.nchains), side='right')
    pop.resumed_rows = [order[a:b].astype(np.int64) for a, b in zip(lo, hi)]
    last = np.array([r[-1] for r in pop.resumed_rows])
    pop.X.copy_(pop.Z[torch.as_tensor(last, device=pop.dev)])
    pop.chisq_cur.copy_(-2.0*pop.log_post[torch.as_tensor(last, device=pop.dev)])
    pop.bestp0 = np.array(oldrun['bestp'], float)
    pop.best_log_post0 = float(oldrun['best_log_post'])
    pop.resumed_accept = int(float(oldrun['acceptance_rate'])/100.0*M0)
    pop.first_valid = 0
