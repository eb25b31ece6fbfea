"""CPU tests of the spectral form's planning and of its numpy formula (mc3_b200/spectral.py)."""
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mc3_b200 import spectral  # noqa: E402


def test_band_from_the_period_parameter():
    params = np.array([1.0, 2.5, 0.3, 5.0, -0.2])
    pmin, pmax = np.array([0.0, 1.0, -4, 0, -1]), np.array([5.0, 5.0, 4, 10, 1])
    free = np.array([0.1, 0.1, 0.1, 0.1, 0.1])
    np.testing.assert_allclose(spectral.band(params, free, pmin, pmax), (2*np.pi/5, 2*np.pi))
    fixed = free.copy()
    fixed[1] = 0.0
    np.testing.assert_allclose(spectral.band(params, fixed, pmin, pmax), (2*np.pi/2.5, 2*np.pi/2.5))
    shared = free.copy()
    shared[1] = -1.0                                  # the period copies parameter 0 (bounds [0, 5])
    assert spectral.band(params, shared, pmin, pmax) is None
    pmin2 = pmin.copy()
    pmin2[0] = 2.0
    np.testing.assert_allclose(spectral.band(params, shared, pmin2, pmax), (2*np.pi/5, 2*np.pi/2))
    lo0 = pmin.copy()
    lo0[1] = 0.0                                      # a band that reaches 0
    assert spectral.band(params, free, lo0, pmax) is None
    hi_inf = pmax.copy()
    hi_inf[1] = np.inf
    assert spectral.band(params, free, pmin, hi_inf) is None


def test_plan_meets_its_truncation_bound_and_caps():
    p = spectral.plan(0.0, 10.0, 2*np.pi/5, 2*np.pi, 100000)       # config 2
    assert p['order'] == 9 and p['R'] == 5.0 and p['xc'] == 5.0
    assert (0.5*p['delta']*p['R'])**10/math.factorial(10) <= 1.0001*spectral.TOL
    # every frequency of the band has a node within delta/2, and so has twice it
    w = np.linspace(2*np.pi/5, 2*np.pi, 10001)
    j1 = np.rint((w - p['w1'])/p['delta'])
    j2 = np.rint((2*w - p['w2'])/p['delta'])
    assert j1.min() >= 0 and j1.max() < p['n1'] and j2.min() >= 0 and j2.max() < p['n2']
    # a long baseline needs the higher order, a longer one is beyond the caps
    q = spectral.plan(0.0, 1000.0, 2*np.pi/5, 2*np.pi, 1000)
    assert q['order'] == 15
    assert spectral.plan(0.0, 1e5, 2*np.pi/5, 2*np.pi, 1000) is None
    assert spectral.plan(0.0, 10.0, 2*np.pi/5, 2*np.pi, 10**7) is None
    assert spectral.plan(0.0, 10.0, 0.0, 1.0, 1000) is None


def test_numpy_formula_matches_long_double():
    rs = np.random.RandomState(0)
    x = np.linspace(0.0, 10.0, 3000)
    truth = np.array([1.0, 2.5, 0.3, 5.0, -0.2])
    d = truth[0]*np.sin(2*np.pi*x/truth[1] + truth[2]) + truth[3] + truth[4]*x + rs.normal(0, 0.5, x.size)
    slr, c0r = np.polyfit(x, d, 1)
    p = spectral.plan(0.0, 10.0, 2*np.pi/5, 2*np.pi, x.size)
    tab = spectral.table(x, d, c0r, slr, p)
    P = truth*(1 + 0.05*rs.standard_normal((40, 5)))
    P[:, 1] = rs.uniform(1.0, 5.0, 40)
    P[0, 1] = 0.5                                      # outside the band: no node
    got = spectral.chisq(tab, p, c0r, slr, P, 0.5)
    LD = np.longdouble
    xl = x.astype(LD)
    want = np.array([float(np.sum((LD(q[0])*np.sin(2*LD(np.pi)/LD(q[1])*xl + LD(q[2])) + LD(q[3]) + LD(q[4])*xl
                                   - d.astype(LD))**2))/0.25 for q in P])
    assert np.isnan(got[0])
    np.testing.assert_allclose(got[1:], want[1:], rtol=1e-13)
