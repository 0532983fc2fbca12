#!/usr/bin/env python
"""Goldens for BASELINE.json configs[2] / [3] at the largest size the reference finishes in the build container in a few
minutes: two-site DMRG of SpinChain (XXZ, U(1) Sz) and FermiHubbardChain (U(1) x U(1): N, Sz) with the density-matrix
mixer and a bond-dimension ramp, run by the UNMODIFIED reference (compiled Cython helper, oracle/_ref).  Writes
tests/golden/dmrg_large.json: energy, entanglement entropies, bond dimensions, centre Schmidt values, sweep times.

    python tests/golden/make_golden_large.py [xxz|hubbard ...]
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

CASES = {
    'xxz': dict(model='SpinChain', L=64, chi=256, params={'S': 0.5, 'Jx': 1., 'Jy': 1., 'Jz': 1., 'conserve': 'Sz'},
                state=['up', 'down']),
    'hubbard': dict(model='FermiHubbardChain', L=32, chi=256, params={'t': 1., 'U': 4., 'mu': 0., 'cons_N': 'N', 'cons_Sz': 'Sz'},
                    state=['up', 'down']),
}


def dmrg_options(chi):
    """shared by the reference run here and the engine runs of tests/test_large_parity.py"""
    ramp = {0: 32, 2: 64, 4: 128, 6: chi}
    return {'mixer': True, 'mixer_params': {'amplitude': 1.e-4, 'decay': 2., 'disable_after': 8}, 'chi_list': ramp,
            'combine': True, 'max_E_err': 1.e-12, 'max_S_err': 1.e-9, 'min_sweeps': 10, 'max_sweeps': 16,
            'trunc_params': {'svd_min': 1.e-12}, 'lanczos_params': {'N_min': 2, 'N_max': 20, 'P_tol': 1.e-14}}


def run_reference(name):
    from tenpy_b200 import dropin
    sys.path.insert(0, dropin.reference_path())
    import tenpy
    from tenpy.algorithms import dmrg
    from tenpy.networks.mps import MPS
    case = CASES[name]
    Model = getattr(tenpy, case['model'])
    p = dict(case['params'])
    p.update({'L': case['L'], 'bc_MPS': 'finite'})
    M = Model(p)
    L = case['L']
    psi = MPS.from_product_state(M.lat.mps_sites(), case['state'] * (L // 2), bc='finite')
    eng = dmrg.TwoSiteDMRGEngine(psi, M, dmrg_options(case['chi']))
    t0 = time.time()
    E, _ = eng.run()
    dt = time.time() - t0
    S = psi.entanglement_entropy()
    sv = psi.get_SL(L // 2)
    return {'E': float(E), 'S': [float(x) for x in S], 'chi': [int(c) for c in psi.chi],
            # Schmidt values that are determined by the physics at the convergence level of the run (weight > 1e-12); the
            # count of the smaller ones depends on rounding noise (the energy does not fix components of weight 1e-24)
            'n_schmidt_above_1e-6': [int(np.sum(np.asarray(psi.get_SL(i)) > 1.e-6)) for i in range(1, L)],
            'schmidt_above_1e-7': [[float(x) for x in np.sort(np.asarray(psi.get_SL(i)))[::-1] if x > 1.e-7] for i in range(1, L)],
            'schmidt_centre': [float(x) for x in np.sort(sv)[::-1]], 'sweeps': int(eng.sweeps), 'seconds': dt,
            'sweep_times': [float(x) for x in np.diff([0.] + list(eng.sweep_stats['time']))],
            'host_cpus': os.cpu_count(), 'L': L, 'chi_max': case['chi']}


def main():
    names = sys.argv[1:] or list(CASES)
    path = os.path.join(ROOT, 'tests', 'golden', 'dmrg_large.json')
    out = json.load(open(path)) if os.path.exists(path) else {}
    for n in names:
        out[n] = run_reference(n)
        print(n, out[n]['E'], out[n]['sweeps'], '%.1f s' % out[n]['seconds'], max(out[n]['chi']))
        with open(path, 'w') as f:
            json.dump(out, f, indent=1, sort_keys=True)


if __name__ == '__main__':
    main()
