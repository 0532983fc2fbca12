"""TEBD (SURVEY.md section 8f rows 1 and 2) -- the reference's own ``tenpy/algorithms/tebd.py`` (`TEBDEngine`,
`QRBasedTEBDEngine`) and ``tenpy/linalg/truncation.py`` (`svd_theta`, `decompose_theta_qr_based`) running UNMODIFIED on the
tenpy_b200 engine (`tenpy_b200.dropin`), against golden vectors the plain reference wrote on its NumPy engine
(tests/golden/make_golden_tebd.py -> tebd.npz, make_golden_tebd_qr.py -> tebd_qr.npz).

A fixed number of imaginary-time steps (sweeps through `update_imag`, brick wall through `evolve` at orders 1, 2, 4) for TFI,
TFI with parity, XXZ with Sz and Hubbard with (N, Sz).  Tolerances: bond energies 1e-9 absolute after up to 60 sweeps of
non-unitary updates, entropies 1e-8, norms 1e-9 relative, bond dimensions exact, the H_bond / U_bond operators 1e-14."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as h

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, 'tests', 'dropin', 'run_reference_drivers.py')


def _reference_available():
    sys.path.insert(0, ROOT)
    from tenpy_b200 import dropin
    return dropin.reference_path() is not None


def _run(mode, case):
    out = subprocess.run([sys.executable, RUNNER, mode, case], capture_output=True, text=True, timeout=1500, cwd='/tmp')
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])[case]


def _compare(got, g, tags, eps_tol, tol=1e-9):
    for t in tags:
        assert np.max(np.abs(np.array(got[t + '_Ebond']) - g[t + '_Ebond'])) < tol, t
        assert np.max(np.abs(np.array(got[t + '_S']) - g[t + '_S'])) < tol * 10, t
        assert list(got[t + '_chi']) == list(g[t + '_chi']), t
        assert abs(got[t + '_norm'] - g[t + '_norm']) < 1e-9 * abs(g[t + '_norm']), t
        assert abs(got[t + '_eps'] - g[t + '_eps']) < eps_tol(g[t + '_eps']), t


def _check_tebd(mode):
    if not _reference_available():
        pytest.skip('no reference install (oracle/_ref, built from a reference checkout)')
    got, g = _run(mode, 'tebd_golden'), h.load('tebd.npz')
    for name in ('tfi', 'tfip', 'xxz', 'hub'):
        assert np.max(np.abs(np.array(got[name + '_Hbond_mid']) - g[name + '_Hbond_mid'])) < 1e-14
        assert np.max(np.abs(np.array(got[name + '_U_half_mid']) - g[name + '_U_half_mid'])) < 1e-14
        _compare(got, g, [name + '_imag'] + ['{0}_o{1}'.format(name, o) for o in (1, 2, 4)],
                 lambda e: 1e-12 + 1e-6 * abs(e))


def _check_tebd_qr(mode):
    if not _reference_available():
        pytest.skip('no reference install (oracle/_ref, built from a reference checkout)')
    got, g = _run(mode, 'tebd_qr_golden'), h.load('tebd_qr.npz')
    _compare(got, g, [n + t for n in ('tfi', 'xxz') for t in ('_imag', '_o2')], lambda e: 1e-13)


def test_reference_tebd_on_engine_host_logic():
    _check_tebd('fake')


def test_reference_tebd_qr_based_on_engine_host_logic():
    _check_tebd_qr('fake')


@pytest.mark.gpu
def test_reference_tebd_on_engine_gpu(gpu_lib):
    _check_tebd('cuda')


@pytest.mark.gpu
def test_reference_tebd_qr_based_on_engine_gpu(gpu_lib):
    _check_tebd_qr('cuda')
