"""Spectral form of the uniform-sigma sinusoid + line chi-squared (include/mc3b200.h,
mc3b_spectral_t): node/order planning, shared by the engine and profiles/spectral_error.py,
and a numpy restatement of the table and of the per-chain formula (CPU reference).

With t = x - xc, d' = d - (c0ref + slref x), L' = a + b t and S_g(w) = sum g e^{i w x},
  sigma^2 chisq = A^2 [n/2 - Re(e^{2i ph} S_1(2w))/2] + 2A Im(e^{i ph} [a S_1 + b S_t - S_d'](w))
                + n a^2 + 2ab St + b^2 St2 - 2a Sd - 2b Std + D2.
S_g near a node w_j is a Taylor series in the offset: S_g(w_j + dw) = e^{i dw xc} sum_k (i dw)^k
T_g[j][k], T_g[j][k] = sum g t^k e^{i w_j x} / k!, truncation <= (|dw| R)^{K+1}/(K+1)! sum|g|.
"""
import math

import numpy as np

TOL = 1e-18                 # truncation bound relative to sum |g|
ORDERS = (9, 15)            # K the kernels are compiled for; 9 while the table stays small
SMALL_NODES = 4096          # ... i.e. up to this many nodes; then 15 (7x fewer nodes, 1.6x the terms)
MAX_NODES = 65536           # table cap: 64 K nodes (about 20 MB at K = 9)
MAX_NODE_POINTS = 2.5e8     # build cap: nodes x points (config 2: 5.4e7, about 0.3 ms of FP64 work on a B200)


def band(params, pstep, pmin, pmax, iperiod=1):
    """Angular-frequency band [wlo, whi] the period parameter can take: from its bounds when
    it is free, its value when it is fixed, its source's when it is shared.  None when the
    band would reach 0 or the periods are not all positive and finite."""
    i = iperiod
    for _ in range(len(pstep)):
        if pstep[i] >= 0:
            break
        i = -int(pstep[i]) - 1
    lo, hi = (pmin[i], pmax[i]) if pstep[i] > 0 else (params[i], params[i])
    if not (np.isfinite(lo) and np.isfinite(hi) and 0.0 < lo <= hi):
        return None
    return 2*np.pi/hi, 2*np.pi/lo


def plan(xlo, xhi, wlo, whi, n):
    """Nodes and order for abscissae in [xlo, xhi] and frequencies in [wlo, whi]: dict with
    order K, spacing delta, first nodes w1 (band) / w2 (doubled band), node counts n1 / n2,
    centre xc and half-width R; or None beyond the table and build caps."""
    if not (0.0 < wlo <= whi and np.isfinite(whi)) or not xhi >= xlo:
        return None
    xc = 0.5*(xlo + xhi)
    R = max(xhi - xc, xc - xlo, 1e-300)
    for K in ORDERS:
        h = (math.factorial(K + 1)*TOL)**(1.0/(K + 1))      # largest |dw| R within TOL
        delta = 2.0*h/R                                       # |dw| <= delta/2
        n1 = int(math.ceil((whi - wlo)/delta)) + 3            # one spare node below and two above
        n2 = int(math.ceil(2.0*(whi - wlo)/delta)) + 3
        if n1 + n2 <= SMALL_NODES:
            break
    if n1 + n2 > MAX_NODES or (n1 + n2)*float(n) > MAX_NODE_POINTS:
        return None
    return dict(order=K, delta=delta, w1=wlo - delta, w2=2.0*wlo - delta, n1=n1, n2=n2, xc=xc, R=R,
                bound=(0.5*delta*R)**(K + 1)/math.factorial(K + 1))


def _csum(terms, chunk=1024):
    """Sum over the last axis: pairwise within chunks, compensated (Neumaier) over chunks."""
    n = terms.shape[-1]
    s = np.zeros(terms.shape[:-1], terms.dtype)
    c = np.zeros_like(s)
    for i in range(0, n, chunk):
        v = terms[..., i:i + chunk].sum(axis=-1)
        t = s + v
        big = np.abs(s) >= np.abs(v)
        c += np.where(big, (s - t) + v, (v - t) + s)
        s = t
    return s + c


def table(x, d, c0ref, slref, p, batch=8):
    """(head, T1, Td, U): head = {n, St, St2, Sd, Std, D2}; T1 [n1, K+2], Td [n1, K+1] on the
    band's nodes, U [n2, K+1] on the doubled band's (complex, fp64, compensated sums)."""
    K, xc = p['order'], p['xc']
    t = x - xc
    dp = d - (c0ref + slref*x)
    head = np.array([x.size, *(_csum(v[None])[0] for v in (t, t*t, dp, t*dp, dp*dp))])
    fact = np.array([float(math.factorial(k)) for k in range(K + 2)])
    tk = np.stack([t**k for k in range(K + 2)])                        # [K+2, n]

    def coeffs(nodes, kmax, g):
        out = np.empty((nodes.size, kmax), complex)
        for i in range(0, nodes.size, batch):
            e = np.exp(1j*np.outer(nodes[i:i + batch], x))               # [B, n]
            if g is not None:
                e = e*g
            out[i:i + batch] = _csum(e[:, None, :]*tk[None, :kmax, :])/fact[:kmax]
        return out
    n1 = p['w1'] + p['delta']*np.arange(p['n1'])
    n2 = p['w2'] + p['delta']*np.arange(p['n2'])
    return head, coeffs(n1, K + 2, None), coeffs(n1, K + 1, dp), coeffs(n2, K + 1, None)


def chisq(tab, p, c0ref, slref, P, sigma):
    """chi-squared of sinusoid + line rows P [m, 5] from the table (NaN where w or 2w has no node)."""
    head, T1, Td, U = tab
    K, dl, xc = p['order'], p['delta'], p['xc']
    n, St, St2, Sd, Std, D2 = head
    out = np.full(len(P), np.nan)
    kk = np.arange(K + 1)
    for r, (A, per, ph, c0, sl) in enumerate(np.asarray(P, float)):
        w = 2*np.pi/per
        j1, j2 = int(np.rint((w - p['w1'])/dl)), int(np.rint((2*w - p['w2'])/dl))
        if not (0 <= j1 < p['n1'] and 0 <= j2 < p['n2']):
            continue
        d1, d2 = w - (p['w1'] + j1*dl), 2*w - (p['w2'] + j2*dl)
        b = sl - slref
        a = (c0 - c0ref) + b*xc
        coef = a*T1[j1, :K + 1] + b*(kk + 1)*T1[j1, 1:K + 2] - Td[j1]
        H = np.polyval(coef[::-1], 1j*d1)*np.exp(1j*d1*xc)
        G = np.polyval(U[j2][::-1], 1j*d2)*np.exp(1j*d2*xc)
        q = A*A*0.5*(n - (np.exp(2j*ph)*G).real) + 2*A*(np.exp(1j*ph)*H).imag \
            + n*a*a + 2*a*b*St + b*b*St2 - 2*a*Sd - 2*b*Std + D2
        out[r] = q/(sigma*sigma)
    return out
