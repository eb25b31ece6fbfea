"""Least-squares pre-fit, same contract as the reference's mc3.fit
(mc3/fit_driver.py:15-206): scipy's optimiser on the host driving the GPU
residual kernel (mc3b_residuals) -- the model comes from `func` exactly as in
the sampler (built-in models evaluate on the GPU)."""
import numpy as np
import scipy.optimize as so

from . import stats as ms


def _model(func, params, indparams, indparams_dict, nfunc):
    """Built-in and CUDA models take exactly their own parameters: with the wavelet
    likelihood the three noise parameters at the end are not theirs
    (chain.py:317).  User callables get the full vector, as in the reference."""
    from .models import BuiltinModel, CudaModel
    if nfunc is not None and isinstance(func, (BuiltinModel, CudaModel)):
        return func(params[:nfunc], *indparams, **indparams_dict)
    return func(params, *indparams, **indparams_dict)


def _residuals(fitparams, params, func, data, uncert, indparams, indparams_dict,
               pstep, prior, priorlow, priorup, ifree, ishare, nfunc=None):
    params[ifree] = fitparams
    for s in ishare:
        params[s] = params[-int(pstep[s]) - 1]
    model = _model(func, params, indparams, indparams_dict, nfunc)
    return ms.residuals(model, data, uncert, params, prior, priorlow, priorup)


def fit(data, uncert, func, params, indparams=[], indparams_dict={},
        pstep=None, pmin=None, pmax=None, prior=None, priorlow=None,
        priorup=None, leastsq='lm', wlike=False):
    params = np.array(params, dtype=float)
    npars = params.size
    nfunc = npars - 3 if wlike else None
    pstep = np.ones(npars) if pstep is None else np.asarray(pstep, float)
    pmin = np.full(npars, -np.inf) if pmin is None else np.asarray(pmin, float)
    pmax = np.full(npars, np.inf) if pmax is None else np.asarray(pmax, float)
    if prior is None or priorlow is None or priorup is None:
        prior = priorlow = priorup = np.zeros(npars)
    prior, priorlow, priorup = (np.asarray(a, float) for a in (prior, priorlow, priorup))
    if np.any(params < pmin) or np.any(params > pmax):
        raise ValueError('Some initial-guess values are out of bounds')
    ifree = np.where(pstep > 0)[0]
    ishare = np.where(pstep < 0)[0]
    args = (params, func, data, uncert, indparams, indparams_dict, pstep, prior,
            priorlow, priorup, ifree, ishare, nfunc)
    tol = dict(ftol=3e-16, xtol=3e-16, gtol=3e-16)
    if leastsq == 'lm':
        res = so.leastsq(_residuals, params[ifree], args=args, full_output=True, **tol)
        params[ifree], resid = res[0], res[2]['fvec']
    elif leastsq == 'trf':
        res = so.least_squares(_residuals, params[ifree], args=args, method='trf',
                               bounds=(pmin[ifree], pmax[ifree]), **tol)
        params[ifree], resid = res['x'], res['fun']
    else:
        raise ValueError(f"Invalid 'leastsq' input ({leastsq}). Must select from ['lm', 'trf']")
    for s in ishare:
        params[s] = params[-int(pstep[s]) - 1]
    best_model = _model(func, params, indparams, indparams_dict, nfunc)
    best_log_post = -0.5*np.sum(resid**2.0)
    lpr = ms.log_prior(params[ifree], prior, priorlow, priorup, pstep)
    return {'bestp': params, 'best_log_post': best_log_post,
            'best_chisq': -2*(best_log_post - lpr), 'best_model': best_model,
            'optimizer_res': res}
