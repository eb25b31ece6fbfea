"""numpy emulation of the spectral form of the uniform-sigma sinusoid + line chi-squared (csrc/chisq_grid.cu,
k_spectral_chisq; include/mc3b200.h mc3b_spectral_t): the data enter only through
S_g(w) = sum g e^{i w x} at the chain's frequency, evaluated from a table of Taylor coefficients at nodes
Delta apart (mc3_b200/spectral.py plans Delta and K from the half-width R of the abscissa and the band).
Like the moment form, chi-squared is what is left after terms of size (|s| + |L'| + |d'|)^2 cancel, so its
relative error is eps_eff * amp, amp = ((|A| + |L'|max) sqrt(n) + sqrt(D2))^2 / (sigma^2 chi^2) -- the bound
MomentFix tests against amp_max.  This script measures eps_eff against a long-double per-point evaluation,
over frequencies anywhere in the band (next to nodes and half-way between them), phases across [-pi, pi],
lines away from the reference line, and S/N from config 2's up to where the guard (amp_max = 4000) fires.
Runs on the CPU: python profiles/spectral_error.py"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from mc3_b200 import spectral  # noqa: E402

LD = np.longdouble


def direct(P, x, d):
    P, x, d = P.astype(LD), x.astype(LD), d.astype(LD)
    out = np.empty(len(P))
    for r, p in enumerate(P):
        m = p[0]*np.sin(2*LD(np.pi)/p[1]*x + p[2]) + p[3] + p[4]*x
        out[r] = float(((m - d)**2).sum())
    return out


def amp_bound(P, n, xlo, xhi, D2, c0r, slr, chi_sig2):
    c0, sl = P[:, 3] - c0r, P[:, 4] - slr
    lmax = np.maximum(np.abs(c0 + sl*xlo), np.abs(c0 + sl*xhi))
    return ((np.abs(P[:, 0]) + lmax)*np.sqrt(n) + np.sqrt(D2))**2/chi_sig2


def chains(rs, pt, snr, p, nc):
    """Periods across the band [1, 5] plus ones next to nodes and half-way between them; phases
    across [-pi, pi]; amplitudes and lines scattered about the truth."""
    P = np.tile(pt, (nc, 1))
    P[:, 0] *= 1 + 0.1/snr*rs.standard_normal(nc)
    P[:, 1] = rs.uniform(1.0, 5.0, nc)
    j = rs.randint(1, p['n1'] - 3, nc//2)
    w = p['w1'] + j*p['delta'] + np.where(np.arange(nc//2) % 2, 0.5 - 1e-9, 1e-9)*p['delta']
    P[:nc//2, 1] = 2*np.pi/np.clip(w, 2*np.pi/5.0, 2*np.pi/1.0)
    P[:, 2] = rs.uniform(-np.pi, np.pi, nc)
    P[:, 3] += 0.05*rs.standard_normal(nc)*np.where(np.arange(nc) % 4 == 0, 100.0, 1.0)
    P[:, 4] += 0.01*rs.standard_normal(nc)*np.where(np.arange(nc) % 4 == 1, 100.0, 1.0)
    return P


if __name__ == '__main__':
    rs = np.random.RandomState(5)
    nc = int(os.environ.get('NCHAINS', 48))
    wlo, whi = 2*np.pi/5.0, 2*np.pi/1.0
    print('      n    S/N  offset |  K  Delta    nodes  trunc | max amp | max rel err | err/amp (eps_eff)')
    worst = 0.0
    for n, snr, off in ((100_000, 2.0, 5.0), (100_000, 30.0, 5.0), (20_480, 300.0, 5e4), (20_480, 1.0, -3.0),
                        (8192, 3000.0, 1.0), (1000, 2.0, 5.0)):
        x = np.linspace(0, 10, n)
        pt = np.array([1.0, 2.5, 0.3, off, -0.2])
        sig = pt[0]/snr
        d = pt[0]*np.sin(2*np.pi*x/pt[1] + pt[2]) + pt[3] + pt[4]*x + rs.normal(0, sig, n)
        slr, c0r = np.polyfit(x, d, 1)
        p = spectral.plan(x.min(), x.max(), wlo, whi, n)
        tab = spectral.table(x, d, c0r, slr, p)
        P = chains(rs, pt, snr, p, nc)
        got = spectral.chisq(tab, p, c0r, slr, P, 1.0)
        ref = direct(P, x, d)
        amp = amp_bound(P, n, x.min(), x.max(), tab[0][5], c0r, slr, ref)
        err = np.abs(got/ref - 1)
        eff = np.max(err/amp)
        worst = max(worst, eff)
        print(f'{n:7d} {snr:6.0f} {off:7.0f} | {p["order"]:2d} {p["delta"]:.4f} {p["n1"]:4d}+{p["n2"]:4d} '
              f'{p["bound"]:.0e} | {amp.max():9.2e} | {err.max():.2e} | {eff:.2e}')
    print(f'worst eps_eff {worst:.2e} (target 3e-15); chains with amp > 4000 are re-evaluated point by point')
