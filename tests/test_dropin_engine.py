"""The reference's own drivers -- ``tenpy.algorithms.dmrg`` / ``tebd`` / ``mps_common`` / ``truncation``, ``tenpy.networks``,
``tenpy.models`` -- UNMODIFIED, running on the tenpy_b200 engine (`tenpy_b200.dropin`, boundary B1 of SURVEY.md section 8b).

Each case runs in its own process (the engine has to be seeded before the first ``import tenpy``;
tests/dropin/run_reference_drivers.py) and is compared with the numbers the plain reference gives on its NumPy engine
(tests/golden/dropin.json, written by ``run_reference_drivers.py golden``).  The reference is taken from ``$TENPY_REFERENCE``
or the install ``oracle/_ref`` that ``build()`` makes from a reference checkout; without either the tests skip."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, 'tests', 'dropin', 'run_reference_drivers.py')
CASES = ['tfi_dmrg', 'xxz_dmrg_mixer', 'tfi_dmrg_fast_engine', 'tfi_tebd_imag']


def _reference_available():
    sys.path.insert(0, ROOT)
    from tenpy_b200 import dropin
    return dropin.reference_path() is not None


def _run(mode, case):
    out = subprocess.run([sys.executable, RUNNER, mode, case], capture_output=True, text=True, timeout=900, cwd='/tmp')
    assert out.returncode == 0, out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith('{')][-1]
    return json.loads(line)[case]


def _check(case, got):
    with open(os.path.join(ROOT, 'tests', 'golden', 'dropin.json')) as f:
        ref = json.load(f)[case]
    assert abs(got['E'] - ref['E']) <= 1e-10 * abs(ref['E']), (got['E'], ref['E'])
    assert abs(got['S_mid'] - ref['S_mid']) <= 1e-8, (got['S_mid'], ref['S_mid'])
    # bond dimensions: every case cuts at svd_min = 1e-10 (chi_max is not reached), where the number of values within rounding
    # distance of the threshold is noise in either implementation; the count of values two orders above the cut is exact
    assert got['n_schmidt_above_1e-8'] == ref['n_schmidt_above_1e-8']
    assert len(got['chi']) == len(ref['chi']) and max(abs(a - b) for a, b in zip(got['chi'], ref['chi'])) <= 2, (got['chi'], ref['chi'])


@pytest.mark.parametrize('case', CASES)
def test_reference_drivers_on_engine_host_logic(case):
    """numpy test double of the device library: the engine's host logic under the reference's drivers"""
    if not _reference_available():
        pytest.skip('no reference install (oracle/_ref, built from a reference checkout)')
    _check(case, _run('fake', case))


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES)
def test_reference_drivers_on_engine_gpu(case, gpu_lib):
    """the same on the B200: every Array of the reference's DMRG / TEBD run lives in HBM, every contraction / SVD / eigh /
    block move is a kernel of libb200npc.so"""
    if not _reference_available():
        pytest.skip('no reference install (oracle/_ref, built from a reference checkout)')
    _check(case, _run('cuda', case))
