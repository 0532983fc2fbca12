"""QR based truncation (SURVEY.md 8f rank 2): the reference's own `decompose_theta_qr_based` (truncation.py:533, with
`_qr_theta_Y0` and `_eig_based_svd`) running UNMODIFIED on engine Arrays (`npc.qr`, `npc.eigh`, `svd_theta` on the device),
against the outputs the plain reference produced for the same inputs (tests/golden/qr_trunc.npz from
tests/golden/make_golden_qr_trunc.py): singular values, truncation error, renormalisation, the reconstructed (gauge
invariant) theta and the isometry of the returned tensors.  The checks run inside tests/dropin/run_reference_drivers.py
(own process: the engine is seeded before ``import tenpy``)."""
import pytest

from test_tebd import _run, _reference_available


def _check(mode):
    if not _reference_available():
        pytest.skip('no reference install (oracle/_ref, built from a reference checkout)')
    res = _run(mode, 'qr_trunc_golden')
    assert res['cases'] == 8 and res['max_iso_err'] < 1e-11


def test_reference_qr_based_truncation_on_engine_host_logic():
    _check('fake')


@pytest.mark.gpu
def test_reference_qr_based_truncation_on_engine_gpu(gpu_lib):
    _check('cuda')
