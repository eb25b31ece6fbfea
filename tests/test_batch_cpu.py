"""CPU-only: the ctypes mirror of mc3b_batch_t follows the header, and sample_batch
rejects malformed batches before it touches a device."""
import ctypes
import os
import re

import numpy as np
import pytest

import mc3_b200 as mc3
from mc3_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_batch_struct_layout_matches_header():
    text = open(os.path.join(ROOT, 'include', 'mc3b200.h')).read()
    body = text[text.index('typedef struct mc3b_batch {'):text.index('} mc3b_batch_t;')]
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    names = []
    for decl in body.split('{', 1)[1].split(';'):
        decl = decl.strip()
        if decl:
            for part in decl.split(','):
                names.append(re.findall(r'[A-Za-z_0-9]+', part)[-1])
    assert names == [f[0] for f in _lib.BatchStruct._fields_]
    assert ctypes.sizeof(_lib.BatchStruct) == 56


def line_fits(B=3, n=40):
    x = np.linspace(0.0, 1.0, n)
    data = [1.0 + 0.5*b + 2.0*x for b in range(B)]
    return dict(data=data, uncert=[np.full(n, 0.1)]*B, func=mc3.models.polynomial,
                params=np.array([[1.0 + 0.5*b, 2.0] for b in range(B)]), indparams=[[x]]*B,
                pstep=np.array([0.01, 0.01]), sampler='demc', nchains=8, nsamples=800)


def run(**kw):
    args = line_fits()
    args.update(kw)
    return mc3.sample_batch(**args)


@pytest.mark.parametrize('kw,match', [
    (dict(uncert=[np.full(40, 0.1)]*2), 'uncert has 2 entries for 3 problems'),
    (dict(params=np.ones((4, 2))), 'params has 4 entries for 3 problems'),
    (dict(indparams=[[np.linspace(0, 1, 40)]]*2), 'indparams has 2 entries for 3 problems'),
    (dict(pmin=np.zeros((2, 2))), 'pmin has 2 rows for 3 problems'),
    (dict(seed=[1, 2]), 'seed has 2 entries for 3 problems'),
    (dict(pstep=np.array([[0.01, 0.01], [0.01, 0.0], [0.01, 0.01]])),
     'problem 1: the free/shared/fixed pattern of pstep differs from problem 0'),
    (dict(func=mc3.models.polynomial.__call__), 'sample_batch needs a built-in model'),
    (dict(func=mc3.TorchModel(lambda P, x: P)), 'sample_batch needs a built-in model'),
    (dict(wlike=True), r'fp64 chi-squared likelihood only \(no wlike, no f32\)'),
    (dict(dtype='f32'), r'fp64 chi-squared likelihood only \(no wlike, no f32\)'),
    (dict(nchains=257), 'at most 256 chains per problem, got 257'),
    (dict(nchains=2), 'demc needs at least 3 chains, got 2'),
    (dict(sampler=None), "'sampler' is a required argument"),
    (dict(nsamples=None), "'nsamples' is a required argument for MCMC runs"),
    (dict(sampler='mh'), r"Invalid 'sampler' input \(mh\)"),
    (dict(pmax=np.array([1.2, 5.0])), 'problem 1: Some initial-guess values are out of bounds'),
    (dict(uncert=[np.full(40, 0.1), None, np.full(40, 0.1)]), "problem 1: 'uncert' is a required argument"),
    (dict(indparams=[[np.linspace(0, 1, 40)], [np.linspace(0, 1, 41)], [np.linspace(0, 1, 40)]]),
     r'problem 1: The size of the data array \(40\) does not match the size of the func\(\) output \(41\)'),
    (dict(params=np.ones((3, 9)), pstep=np.full(9, 0.01)), 'problem 0: polynomial takes 1 to 8 parameters, got 9'),
    (dict(burnin=1000), r'The number of burned-in samples \(1000\) is greater than'),
])
def test_errors_before_the_device(kw, match):
    with pytest.raises(ValueError, match=match):
        run(**kw)
