"""Drop-in for the reference's public entry point mc3.sample()
(mc3/sampler_driver.py:25-601): same keyword arguments and defaults, same
validation and error strings (raised as ValueError through Log.error, as the
reference's tests assert), same output-dictionary keys.  The MCMC itself runs
on the GPU (mcmc_driver.mcmc).

Extra keyword arguments (the reference's signature already ends in **kwargs):
  seed=None       Philox seed of the run (None draws one from numpy's global RNG)
  dtype='f64'     arithmetic of the fused model+chi-squared kernel ('f64'|'f32')
  device=None     CUDA device (default: current)
  use_graph=None  replay one captured CUDA graph per generation (default: auto)
  reflect=False   fold out-of-bounds proposals back inside instead of rejecting
                  them (the reference rejects; not a parity mode)

Out of scope (SURVEY.md section 8): file-name inputs, plots.
"""
import importlib
import os
import sys
from datetime import date

import numpy as np

from . import stats as ms
from . import utils as mu
from .fit_driver import fit
from .mcmc_driver import mcmc

__version__ = '0.1.0'


def _need_array(value, name, log):
    if value is None:
        log.error(f"'{name}' is a required argument")
    if isinstance(value, str) or (np.iterable(value) and len(value) > 0
                                  and isinstance(value[0], str)):
        log.error(f"{name}: file-name inputs are not supported by mc3_b200, "
                  "pass arrays")
    if not np.iterable(value):
        log.error(f'{name} must be an iterable or a file name')
    return value


def check_sampler(sampler, nsamples, leastsq, log):
    """The run options sample() checks first."""
    if sampler is None:
        log.error("'sampler' is a required argument")
    if nsamples is None and sampler in ['MRW', 'DEMC', 'snooker', 'mrw', 'demc']:
        log.error("'nsamples' is a required argument for MCMC runs")
    if leastsq not in [None, 'lm', 'trf']:
        log.error(
            f"Invalid 'leastsq' input ({leastsq}). Must select from "
            "['lm', 'trf']")
    if sampler not in ['mrw', 'demc', 'snooker']:
        log.error(f"Invalid 'sampler' input ({sampler}). Must select from "
                  "['mrw', 'demc', 'snooker']")


def read_arrays(params, data, uncert, pmin, pmax, pstep, prior, priorlow, priorup, log):
    """params (or its 2-D file form), data and uncert as float arrays; returns (params,
    data, uncert, pmin, pmax, pstep, prior, priorlow, priorup) with the vectors the 2-D
    params form carries taken from it."""
    params = _need_array(params, 'params', log)
    if np.ndim(params) > 1:                       # sampler_driver.py:284-297
        ninfo = np.shape(params)[0]
        if ninfo == 7:
            prior, priorlow, priorup = params[4], params[5], params[6]
        if ninfo >= 4:
            pstep = params[3]
        if ninfo >= 3:
            pmin, pmax = params[1], params[2]
        else:
            log.error('Invalid format/shape for params input file')
        params = params[0]
    params = np.array(params, dtype=float)

    data = _need_array(data, 'data', log)
    if np.ndim(data) > 1:
        data, uncert = data
    if uncert is None:
        log.error("'uncert' is a required argument")
    uncert = np.array(uncert, dtype=float)        # a copy: never mutate the caller's
    data = np.asarray(data, dtype=float)

    return params, data, uncert, pmin, pmax, pstep, prior, priorlow, priorup


def fill_vectors(params, pnames, texnames, pmin, pmax, pstep, prior, priorlow, priorup, log):
    """Names, default bounds, steps and priors, and the initial-guess bounds check;
    returns (pnames, texnames, pmin, pmax, pstep, prior,
    priorlow, priorup, nfree, ifree, ishare)."""
    nparams = len(params)
    if pnames is None and texnames is not None:
        pnames = texnames
    elif pnames is not None and texnames is None:
        texnames = pnames
    elif pnames is None and texnames is None:
        pnames = texnames = mu.default_parnames(nparams)
    pnames, texnames = np.asarray(pnames), np.asarray(texnames)

    pmin = np.tile(-np.inf, nparams) if pmin is None else np.asarray(pmin, float)
    pmax = np.tile(np.inf, nparams) if pmax is None else np.asarray(pmax, float)
    pstep = 0.1*np.abs(params) if pstep is None else np.asarray(pstep, float)
    if prior is None or priorup is None or priorlow is None:
        prior, priorup, priorlow = (np.zeros(nparams) for _ in range(3))
    prior = np.asarray(prior, float)
    priorlow, priorup = np.array(priorlow, float), np.array(priorup, float)
    priorlow[pstep <= 0] = 0.0                    # :370-372
    priorup[pstep <= 0] = 0.0

    if np.any(params < pmin) or np.any(params > pmax):   # :374-388
        pout = ""
        for pname, par, minp, maxp in zip(pnames, params, pmin, pmax):
            if par < minp:
                pout += f"\n{pname[:11]:11s}  {minp: 12.5e} < {par: 12.5e}"
            if par > maxp:
                pout += f"\n{pname[:11]:26s}  {par: 12.5e} > {maxp: 12.5e}"
        log.error(
            "Some initial-guess values are out of bounds:\n"
            "Param name           pmin          value           pmax\n"
            "-----------  ------------   ------------   ------------"
            f"{pout}")

    nfree = int(np.sum(pstep > 0))
    ifree = np.where(pstep > 0)[0]
    ishare = np.where(pstep < 0)[0]

    return pnames, texnames, pmin, pmax, pstep, prior, priorlow, priorup, nfree, ifree, ishare


def sample(data=None, uncert=None, func=None, params=None,
           indparams=[], indparams_dict={},
           pmin=None, pmax=None, pstep=None,
           prior=None, priorlow=None, priorup=None,
           sampler=None, ncpu=None, leastsq=None, chisqscale=False,
           nchains=7, nsamples=None, burnin=0, thinning=1,
           grtest=True, grbreak=0.0, grnmin=0.5, wlike=False,
           fgamma=1.0, fepsilon=0.0, hsize=10, kickoff='normal',
           plots=False, theme='blue', statistics='med_central',
           ioff=False, showbp=True,
           savefile=None, resume=False,
           rms=False, log=None, pnames=None, texnames=None,
           **kwargs):
    if isinstance(log, str):
        log = mu.Log(log, append=resume)
        closelog = True
    else:
        closelog = False
        if log is None:
            log = mu.Log()

    log.msg(
        f"\n{log.sep}\n"
        "  mc3_b200: B200-native Markov-chain Monte Carlo with the mc3 API.\n"
        f"  Version {__version__} ({date.today().year}).\n"
        f"{log.sep}\n\n")

    check_sampler(sampler, nsamples, leastsq, log)

    (params, data, uncert, pmin, pmax, pstep, prior, priorlow, priorup) = read_arrays(
        params, data, uncert, pmin, pmax, pstep, prior, priorlow, priorup, log)

    resume = resume and (savefile is not None)
    if resume:
        log.msg(f"\n\n{log.sep}\n{log.sep}  Resuming previous MCMC run.\n\n")

    if isinstance(func, (list, tuple, np.ndarray)):   # :320-327
        sys.path.append(func[2] if len(func) == 3 else os.getcwd())
        func = getattr(importlib.import_module(func[1]), func[0])
    elif not callable(func):
        log.error(
            "'func' must be either a callable or an iterable of strings "
            "with the model function, file, and path names")

    nparams = len(params)
    ndata = len(data)
    (pnames, texnames, pmin, pmax, pstep, prior, priorlow, priorup, nfree, ifree,
     ishare) = fill_vectors(params, pnames, texnames, pmin, pmax, pstep, prior, priorlow,
                            priorup, log)

    fpar = params[0:-3] if wlike else params
    model0 = func(fpar, *indparams, **indparams_dict)     # :394-400
    if np.shape(model0) != np.shape(data):
        log.error(
            f"The size of the data array ({np.size(data)}) does not "
            f"match the size of the func() output ({np.size(model0)})")

    if savefile is not None:
        fpath, fname = os.path.split(os.path.realpath(savefile))
        if not os.path.exists(fpath):
            log.warning(f"Output folder path: '{fpath}' does not exist. "
                        "Creating new folder.")
            os.makedirs(fpath)

    chisq_factor = 1.0
    fit_output = None
    if leastsq is not None:                        # :412-440
        fit_output = fit(data, uncert, func, np.copy(params), indparams,
                         indparams_dict, pstep, pmin, pmax, prior, priorlow,
                         priorup, leastsq, wlike=wlike)
        log.msg("Least-squares best-fitting parameters:\n"
                f"  {fit_output['bestp']}\n\n", si=2)
        if chisqscale:
            chisq_factor = np.sqrt(fit_output['best_chisq']/(ndata - nfree))
            uncert *= chisq_factor
            fit_output = fit(data, uncert, func, np.copy(params), indparams,
                             indparams_dict, pstep, pmin, pmax, prior, priorlow,
                             priorup, leastsq, wlike=wlike)
            log.msg("Least-squares best-fitting parameters (rescaled chisq):"
                    f"\n  {fit_output['bestp']}\n\n", si=2)
        params = np.copy(fit_output['bestp'])

    if resume:
        with np.load(savefile) as oldrun:
            uncert *= float(oldrun['chisq_factor'])/chisq_factor
            chisq_factor = float(oldrun['chisq_factor'])

    dev_kw = {k: kwargs[k] for k in ('seed', 'dtype', 'device', 'use_graph',
                                     'reflect', 'rank', 'world', 'group', 'shard',
                                     'plan_chains')
              if k in kwargs}
    output = mcmc(
        data, uncert, func, params, indparams, indparams_dict,
        pmin, pmax, pstep, prior, priorlow, priorup, nchains, ncpu, nsamples,
        sampler, wlike, fit_output, grtest, grbreak, grnmin, burnin, thinning,
        fgamma, fepsilon, hsize, kickoff, savefile, resume, log,
        pnames, texnames, **dev_kw)

    output['chisq_factor'] = chisq_factor
    if dev_kw.get('world', 1) > 1 and dev_kw.get('rank', 0) != 0:
        # chains partitioned over devices: rank 0 holds the gathered history,
        # computes the posterior statistics and writes the files
        if closelog:
            log.close()
        return output
    if leastsq is not None:
        dlp = output['best_log_post'] - fit_output['best_log_post']
        dpar = output['bestp'] - fit_output['bestp']
        if dlp > 5.0e-8 and np.any(dpar != 0.0):
            log.warning(
                "MCMC found a better fit than the minimizer:\n"
                "MCMC best-fitting parameters:        (chisq={:.8g})\n{}\n"
                "Minimizer best-fitting parameters:   (chisq={:.8g})\n{}".format(
                    -2*output['best_log_post'], output['bestp'],
                    -2*fit_output['best_log_post'], fit_output['bestp']))

    # Posterior statistics on the burned sample, thinned to <= 20000 rows with
    # the reference's rule (plots/posterior.py:1085-1091, seed 314159).
    posterior, zchain, zmask = mu.burn(
        Z=output['posterior'], zchain=output['zchain'], burnin=output['burnin'])
    bestp = output['bestp']
    nrows = posterior.shape[0]
    if nrows > 20000:
        pick = np.random.default_rng(314159).choice(nrows, 20000, replace=False)
        stat_post = posterior[pick]
    else:
        stat_post = np.copy(posterior)
    st = ms.calc_sample_statistics(stat_post, bestp, pstep, calc_hpd=True, device=True)
    keys = ('medianp', 'meanp', 'stdp', 'median_low_bounds', 'median_high_bounds',
            'mode', 'hpd_low_bounds', 'hpd_high_bounds')
    for k, v in zip(keys, st):
        output[k] = v
    output['CRlo'] = output['hpd_low_bounds'] - bestp
    output['CRhi'] = output['hpd_high_bounds'] - bestp
    output['CRlo'][pstep == 0] = output['CRhi'][pstep == 0] = 0.0

    median, stdp = output['medianp'], output['stdp']
    log.msg(
        "\nParameter name     best fit   median      1sigma_low   1sigma_hi        S/N"
        "\n--------------- -----------  -----------------------------------  ---------",
        width=80)
    rows = []
    for i in range(nparams):
        lo = output['median_low_bounds'][i] - median[i]
        hi = output['median_high_bounds'][i] - median[i]
        if i in ifree:
            snr = f"{np.abs(bestp[i])/stdp[i]:.1f}"
        elif i in ishare:
            snr = f"[share{-int(pstep[i]):02d}]"
        else:
            snr, lo, hi = "[fixed]", 0.0, 0.0
        rows.append(f"{pnames[i][0:15]:<15} {bestp[i]:11.4e}  {median[i]:11.4e} "
                    f"{lo:11.4e} {hi:11.4e}  {snr:>9s}")
        log.msg(rows[-1], width=160)

    fmt = len(f"{output['BIC']:.4f}")
    cs_txt = f"sqrt(reduced chi-squared) factor: {chisq_factor:.4f}\n" if chisqscale else ''
    fit_txt = (
        f"\n{cs_txt}"
        f"Best-parameter's chi-squared:       {output['best_chisq']:{fmt}.4f}\n"
        f"Best-parameter's -2*log(posterior): {-2.0*output['best_log_post']:{fmt}.4f}\n"
        f"Bayesian Information Criterion:     {output['BIC']:{fmt}.4f}\n"
        f"Reduced chi-squared:                {output['red_chisq']:{fmt}.4f}\n"
        f"Standard deviation of residuals:  {output['stddev_residuals']:.6g}\n")
    log.msg(fit_txt, indent=2)

    root = os.path.splitext(savefile)[0] if savefile is not None else 'mc3'
    stats_file = f'{root}_statistics.txt'
    ms.summary_stats(stat_post, output, filename=stats_file)      # stats.py:967-1112
    log.msg('\nFor a detailed summary with all parameter posterior statistics '
            f'see {stats_file}')
    log.msg("\nOutput sampler files:")
    log.msg(stats_file, indent=2)
    if savefile is not None:
        np.savez(savefile, **output)
        log.msg(savefile, indent=2)
    if plots:
        log.warning('plots are outside the scope of mc3_b200; pass the output '
                    'dictionary to mc3.plots')
    if closelog:
        log.msg(log.logname, indent=2)
        log.close()
    return output
