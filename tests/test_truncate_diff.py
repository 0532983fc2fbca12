"""`tenpy_b200.linalg.truncation.truncate` (own formulation: conditions on the number of kept values) against the
reference's `truncate` (truncation.py:146) on randomised spectra and option combinations: same number of kept values, same
norm, same truncation error.  Inputs and the reference's outputs are stored in tests/golden/truncate.npz (written by
tests/golden/make_golden_truncate.py)."""
import warnings

import numpy as np

import helpers as h

OPTION_KEYS = ('chi_max', 'chi_min', 'degeneracy_tol', 'svd_min', 'trunc_cut')
INT_OPTIONS = ('chi_max', 'chi_min')


def _trials(g):
    for i in range(len(g['n'])):
        opts = {}
        for key in OPTION_KEYS:
            if g['has_' + key][i]:
                v = g['opt_' + key][i]
                opts[key] = None if np.isnan(v) else (int(v) if key in INT_OPTIONS else float(v))
        yield g['S_pad'][i, :g['n'][i]], opts


def test_truncate_matches_reference_randomised():
    from tenpy_b200.linalg.truncation import truncate as mine
    g = h.load('truncate.npz')
    assert len(g['kept']) == 1500
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for (S, opts), k2, n2, e2 in zip(_trials(g), g['kept'], g['norm'], g['eps']):
            m1, n1, e1 = mine(S, dict(opts))
            assert m1.sum() == k2 and abs(n1 - n2) < 1e-14 and abs(e1.eps - e2) < 1e-14, (opts, S)
