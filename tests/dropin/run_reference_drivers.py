#!/usr/bin/env python
"""The UNMODIFIED reference drivers (tenpy.algorithms.dmrg / tebd, tenpy.networks.*, tenpy.models.*) running on the
tenpy_b200 engine (tenpy_b200.dropin).  Executed in its own process by tests/test_dropin_engine.py because the seeding has
to happen before the first ``import tenpy``.

    python tests/dropin/run_reference_drivers.py fake|cuda [case ...]

Prints one JSON line per case.  The numbers are compared with the reference running on its own NumPy engine
(tests/golden/dropin.json, written by ``--golden`` with the plain reference).
"""
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
warnings.filterwarnings('ignore')


def setup(mode):
    if mode == 'golden':             # the plain reference, to write the expected numbers
        from tenpy_b200 import dropin
        sys.path.insert(0, dropin.reference_path())
        return None
    from tenpy_b200 import backend, dropin
    if mode == 'fake':
        from fake_device import FakeDeviceLib
        backend.use_library(FakeDeviceLib())
    else:
        from tenpy_b200._lib import DeviceLib
        backend.use_library(DeviceLib())
    path = dropin.install()
    assert path is not None, 'reference not found (oracle/_ref)'
    import tenpy
    import tenpy.linalg.np_conserved as npc
    assert npc.__name__ == 'tenpy_b200.linalg.np_conserved', npc.__name__
    from tenpy.algorithms import dmrg
    assert dmrg.npc is npc
    assert os.path.realpath(dmrg.__file__).startswith(os.path.realpath(path)), dmrg.__file__
    return dropin


def _spectrum_summary(psi):
    """bond dimensions and -- robust against the rounding noise of a cut at `svd_min` -- the number of Schmidt values that are
    two orders of magnitude above it"""
    import numpy as np
    return {'chi': [int(c) for c in psi.chi],
            'n_schmidt_above_1e-8': [int(np.sum(np.asarray(psi.get_SL(i)) > 1.e-8)) for i in range(1, psi.L)]}


def case_tfi_dmrg(dropin):
    """config 0: examples/d_dmrg.py TFIChain L=20 chi=50 two-site DMRG (E = -25.1077971116238)"""
    from tenpy.models.tf_ising import TFIChain
    from tenpy.networks.mps import MPS
    from tenpy.algorithms import dmrg
    M = TFIChain({'L': 20, 'J': 1., 'g': 1., 'bc_MPS': 'finite', 'conserve': None})
    psi = MPS.from_product_state(M.lat.mps_sites(), ['up'] * 20, bc='finite')
    info = dmrg.run(psi, M, {'mixer': None, 'max_E_err': 1.e-10, 'trunc_params': {'chi_max': 50, 'svd_min': 1.e-10},
                             'combine': True})
    return dict(E=float(info['E']), S_mid=float(psi.entanglement_entropy()[9]), **_spectrum_summary(psi))


def case_xxz_dmrg_mixer(dropin):
    """SpinChain L=16 with Sz conservation, density-matrix mixer, ragged charge blocks"""
    from tenpy.models.spins import SpinChain
    from tenpy.networks.mps import MPS
    from tenpy.algorithms import dmrg
    L = 16
    M = SpinChain({'L': L, 'S': 0.5, 'Jx': 1., 'Jy': 1., 'Jz': 1., 'bc_MPS': 'finite', 'conserve': 'Sz'})
    psi = MPS.from_product_state(M.lat.mps_sites(), ['up', 'down'] * (L // 2), bc='finite')
    info = dmrg.run(psi, M, {'mixer': True, 'mixer_params': {'amplitude': 1.e-5, 'decay': 2., 'disable_after': 6},
                             'max_E_err': 1.e-11, 'max_S_err': 1.e-8, 'max_sweeps': 20, 'combine': True,
                             'trunc_params': {'chi_max': 60, 'svd_min': 1.e-10}})
    return dict(E=float(info['E']), S_mid=float(psi.entanglement_entropy()[L // 2 - 1]), **_spectrum_summary(psi))


def case_tfi_dmrg_fast_engine(dropin):
    """the reference engine with the device-optimised effective Hamiltonian plugged in at `EffectiveH`"""
    from tenpy.models.tf_ising import TFIChain
    from tenpy.networks.mps import MPS
    M = TFIChain({'L': 20, 'J': 1., 'g': 1., 'bc_MPS': 'finite', 'conserve': None})
    psi = MPS.from_product_state(M.lat.mps_sites(), ['up'] * 20, bc='finite')
    if dropin is None:
        from tenpy.algorithms.dmrg import TwoSiteDMRGEngine as Engine
    else:
        Engine = dropin.fast_two_site_engine()
        Engine.EffectiveH.SPLIT_MIN_BLOCK = 1          # force the split / identity-environment route on small blocks
    eng = Engine(psi, M, {'mixer': None, 'max_E_err': 1.e-10, 'trunc_params': {'chi_max': 50, 'svd_min': 1.e-10},
                          'combine': True})
    E, _ = eng.run()
    return dict(E=float(E), S_mid=float(psi.entanglement_entropy()[9]), **_spectrum_summary(psi))


def case_tfi_tebd_imag(dropin):
    """imaginary-time TEBD of the reference (tebd.py:446 update_bond) towards the ground state"""
    from tenpy.models.tf_ising import TFIChain
    from tenpy.networks.mps import MPS
    from tenpy.algorithms import tebd
    L = 10
    M = TFIChain({'L': L, 'J': 1., 'g': 1.5, 'bc_MPS': 'finite', 'conserve': None})
    psi = MPS.from_product_state(M.lat.mps_sites(), ['up'] * L, bc='finite')
    eng = tebd.TEBDEngine(psi, M, {'order': 2, 'delta_tau_list': [0.1, 0.01], 'N_steps': 5, 'max_error_E': 1.e-6,
                                   'trunc_params': {'chi_max': 20, 'svd_min': 1.e-10}})
    eng.run_GS()
    E = M.bond_energies(psi)
    return dict(E=float(sum(E)), S_mid=float(psi.entanglement_entropy()[L // 2 - 1]), **_spectrum_summary(psi))


def _tebd_models():
    from tenpy.models.tf_ising import TFIChain
    from tenpy.models.spins import SpinChain
    from tenpy.models.hubbard import FermiHubbardChain
    L = 10
    yield 'tfi', TFIChain(dict(L=L, J=1., g=1.2, bc_MPS='finite', conserve=None)), ['up'] * L
    yield 'tfip', TFIChain(dict(L=L, J=1., g=0.8, bc_MPS='finite', conserve='parity')), ['up'] * L
    yield 'xxz', SpinChain(dict(L=L, S=0.5, Jx=1., Jy=1., Jz=1.3, hz=0., bc_MPS='finite', conserve='Sz')), \
        ['up', 'down'] * (L // 2)
    L = 6
    yield 'hub', FermiHubbardChain(dict(L=L, t=1., U=3., mu=0., bc_MPS='finite', cons_N='N', cons_Sz='Sz')), \
        ['up', 'down'] * (L // 2)


def _tebd_record(out, tag, M, psi, eng):
    import numpy as np
    out[tag + '_Ebond'] = [float(x) for x in np.asarray(M.bond_energies(psi), dtype=np.float64)]
    out[tag + '_S'] = [float(x) for x in psi.entanglement_entropy()]
    out[tag + '_chi'] = [int(c) for c in psi.chi]
    out[tag + '_norm'] = float(psi.norm)
    out[tag + '_eps'] = float(eng.trunc_err.eps)


def case_tebd_golden(dropin):
    """the scenario of tests/golden/make_golden_tebd.py (reference TEBDEngine: imaginary-time sweeps and brick-wall evolution
    at orders 1, 2, 4; TFI, TFI with parity, XXZ with Sz, Hubbard with (N, Sz)) -> compared with tests/golden/tebd.npz"""
    from tenpy.algorithms import tebd
    from tenpy.networks.mps import MPS
    out = {}
    for name, M, state in _tebd_models():
        sites = M.lat.mps_sites()
        L = len(sites)
        out[name + '_Hbond_mid'] = M.H_bond[L // 2].to_ndarray().tolist()
        psi = MPS.from_product_state(sites, state, bc='finite')
        eng = tebd.TEBDEngine(psi, M, {'trunc_params': {'chi_max': 32, 'svd_min': 1e-8}})
        eng.calc_U(2, 0.05, type_evo='imag')
        out[name + '_U_half_mid'] = eng._U[0][L // 2].to_ndarray().tolist()
        eng.update_imag(30, call_canonical_form=False)
        _tebd_record(out, name + '_imag', M, psi, eng)
        for order in (1, 2, 4):
            psi = MPS.from_product_state(sites, state, bc='finite')
            eng = tebd.TEBDEngine(psi, M, {'trunc_params': {'chi_max': 32, 'svd_min': 1e-8}})
            eng.calc_U(order, 0.02, type_evo='imag')
            eng.evolve(6, 0.02)
            _tebd_record(out, '{0}_o{1}'.format(name, order), M, psi, eng)
    return out


def case_tebd_qr_golden(dropin):
    """tests/golden/make_golden_tebd_qr.py: the reference's QRBasedTEBDEngine (tebd.py:619; decompose_theta_qr_based,
    truncation.py:473) on the engine's npc.qr / eigh -> compared with tests/golden/tebd_qr.npz"""
    from tenpy.algorithms import tebd
    from tenpy.networks.mps import MPS
    opts = {'trunc_params': {'chi_max': 24, 'svd_min': 1e-8}, 'cbe_expand': 0.1, 'cbe_expand_0': 0.5,
            'cbe_min_block_increase': 2, 'compute_err': True}
    out = {}
    for name, M, state in _tebd_models():
        if name not in ('tfi', 'xxz'):
            continue
        sites = M.lat.mps_sites()
        psi = MPS.from_product_state(sites, state, bc='finite')
        eng = tebd.QRBasedTEBDEngine(psi, M, dict(opts))
        eng.calc_U(2, 0.05, type_evo='imag')
        eng.update_imag(20, call_canonical_form=False)
        _tebd_record(out, name + '_imag', M, psi, eng)
        psi = MPS.from_product_state(sites, state, bc='finite')
        eng = tebd.QRBasedTEBDEngine(psi, M, dict(opts))
        eng.calc_U(2, 0.02, type_evo='imag')
        eng.evolve(6, 0.02)
        _tebd_record(out, name + '_o2', M, psi, eng)
    return out


def case_qr_trunc_golden(dropin):
    """the reference's `decompose_theta_qr_based` (truncation.py:533) on engine Arrays built from the inputs of
    tests/golden/qr_trunc.npz; checked here against the stored outputs (singular values, truncation error,
    renormalisation, the reconstructed theta, isometry of the returned tensors)"""
    import numpy as np
    import helpers as h
    import tenpy.linalg.np_conserved as npc
    from tenpy.linalg.charges import LegCharge
    from tenpy.linalg.truncation import decompose_theta_qr_based
    g = h.load('qr_trunc.npz')
    worst = {'S': 0., 'approx': 0., 'iso': 0.}
    for i in range(int(g['n'])):
        key = 'q%d' % i
        move_right, eig = bool(g[key + '_move_right']), bool(g[key + '_eig'])
        theta = h.to_product(h.oarray_from(g, key + '_theta'))
        old_leg = LegCharge.from_qind(theta.chinfo, g[key + '_oldleg_slices'], g[key + '_oldleg_charges'],
                                      int(g[key + '_oldleg_qconj']))
        tp = dict(chi_max=12, svd_min=1e-10)
        T_L, S, T_R, form, err, renorm = decompose_theta_qr_based(g[key + '_qL'], g[key + '_qR'], old_leg, theta,
                                                                  move_right, 0.5, 1, eig, tp, True, True)
        assert [str(x) for x in form] == [str(x) for x in g[key + '_form']]
        assert len(S) == len(g[key + '_S'])
        dS = float(np.max(np.abs(np.sort(S) - np.sort(g[key + '_S']))))
        assert dS < (1e-7 if eig else 1e-10), (key, dS)
        assert abs(renorm - g[key + '_renorm']) < 1e-10 * g[key + '_renorm']
        assert abs(err.eps - g[key + '_eps']) < 1e-12 + 1e-6 * g[key + '_eps']
        approx = npc.tensordot(T_L, T_R, axes=['vR', 'vL']) if eig else \
            npc.tensordot(T_L.scale_axis(S, 'vR'), T_R, axes=['vR', 'vL'])
        approx.ireplace_labels(['(vL.p)', '(p.vR)'], ['(vL.p0)', '(p1.vR)'])
        h.assert_close(h.to_oracle(approx), h.oarray_from(g, key + '_approx'), 1e-9, structure=False)
        for T, lab, f in ((T_L, ['(vL*.p*)', '(vL.p)'], form[0] == 'A'), (T_R, None, form[1] == 'B')):
            if f and lab is not None:
                iso = npc.tensordot(T.conj(), T, axes=lab).to_ndarray()
                worst['iso'] = max(worst['iso'], float(np.max(np.abs(iso - np.eye(len(iso))))))
            elif f:
                iso = npc.tensordot(T, T.conj(), axes=['(p.vR)', '(p*.vR*)']).to_ndarray()
                worst['iso'] = max(worst['iso'], float(np.max(np.abs(iso - np.eye(len(iso))))))
        worst['S'] = max(worst['S'], dS if not eig else 0.)
    assert worst['iso'] < 1e-11
    return {'cases': int(g['n']), 'max_dS': worst['S'], 'max_iso_err': worst['iso']}


CASES = {'tebd_golden': case_tebd_golden, 'qr_trunc_golden': case_qr_trunc_golden, 'tebd_qr_golden': case_tebd_qr_golden, 'tfi_dmrg': case_tfi_dmrg, 'xxz_dmrg_mixer': case_xxz_dmrg_mixer, 'tfi_dmrg_fast_engine': case_tfi_dmrg_fast_engine,
         'tfi_tebd_imag': case_tfi_tebd_imag}


def main():
    mode = sys.argv[1]
    names = sys.argv[2:] or [c for c in CASES if not c.endswith('_golden')]
    dropin = setup(mode)
    out = {}
    for name in names:
        out[name] = CASES[name](dropin)
        print(json.dumps({name: out[name]}))
        sys.stdout.flush()
    if mode == 'golden':
        with open(os.path.join(ROOT, 'tests', 'golden', 'dropin.json'), 'w') as f:
            json.dump(out, f, indent=1, sort_keys=True)


if __name__ == '__main__':
    main()
