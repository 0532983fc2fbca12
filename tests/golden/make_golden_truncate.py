#!/usr/bin/env python
"""Golden vectors of the UNMODIFIED reference's `truncate` (tenpy/linalg/truncation.py:146) on randomised spectra and
option combinations, for tests/test_truncate_diff.py.  Writes tests/golden/truncate.npz: the inputs of every trial (spectrum
zero-padded to ``S_pad`` with its length ``n``; per option ``has_<key>`` and ``opt_<key>``, NaN standing for None) and the
reference's outputs (number of kept values, new norm, truncation error).  The reference is taken from ``$TENPY_REFERENCE``
(a checkout of tenpy/tenpy):

    TENPY_NO_CYTHON=1 TENPY_REFERENCE=<tenpy checkout> python tests/golden/make_golden_truncate.py
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N_TRIALS = 1500
OPTION_KEYS = ('chi_max', 'chi_min', 'degeneracy_tol', 'svd_min', 'trunc_cut')


def trials():
    """(S, options) of every trial"""
    rng = np.random.default_rng(0)
    for trial in range(N_TRIALS):
        n = int(rng.integers(1, 40))
        kind = rng.integers(0, 4)
        if kind == 0:
            S = rng.random(n)
        elif kind == 1:
            S = np.exp(-rng.random(n) * 40)
        elif kind == 2:
            S = np.repeat(rng.random(max(1, n // 3)), 3)[:n]
        else:
            S = np.concatenate([rng.random(n // 2 + 1), np.zeros(n // 2)])
        S = S / np.linalg.norm(S)
        opts = {}
        if rng.random() < .8:
            opts['chi_max'] = int(rng.integers(1, 45)) if rng.random() < .9 else None
        if rng.random() < .3:
            opts['chi_min'] = int(rng.integers(1, 45))
        if rng.random() < .3:
            opts['degeneracy_tol'] = float(10 ** rng.uniform(-8, -1))
        if rng.random() < .7:
            opts['svd_min'] = float(10 ** rng.uniform(-16, -1)) if rng.random() < .9 else None
        if rng.random() < .7:
            opts['trunc_cut'] = float(10 ** rng.uniform(-16, -0.5)) if rng.random() < .9 else None
        yield S, opts


def main():
    sys.path.insert(0, os.environ['TENPY_REFERENCE'])
    from tenpy.linalg.truncation import truncate
    from tenpy.tools.params import Config
    cases = list(trials())
    kept, norm, eps = [], [], []
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for S, opts in cases:
            mask, new_norm, err = truncate(S, Config(dict(opts), 'trunc'))
            kept.append(int(mask.sum()))
            norm.append(float(new_norm))
            eps.append(float(err.eps))
    n = np.array([len(S) for S, _ in cases], np.int64)
    S_pad = np.zeros((len(cases), n.max()))
    for i, (S, _) in enumerate(cases):
        S_pad[i, :len(S)] = S
    out = dict(S_pad=S_pad, n=n, kept=np.array(kept, np.int64), norm=np.array(norm), eps=np.array(eps))
    for key in OPTION_KEYS:
        out['has_' + key] = np.array([key in opts for _, opts in cases])
        out['opt_' + key] = np.array([np.nan if opts.get(key) is None else opts[key] for _, opts in cases], np.float64)
    np.savez_compressed(os.path.join(HERE, 'truncate.npz'), **out)
    print('wrote truncate.npz:', len(kept), 'trials')


if __name__ == '__main__':
    main()
