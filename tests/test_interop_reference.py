"""Checkpoint exchange with the UNMODIFIED reference (SURVEY.md section 8f rank 4): a DMRG state computed by this package
is converted with `tenpy_b200.tools.interop`, pickled, loaded by stock TeNPy (which measures the same energy and
continues the run), and a reference state comes back.  Needs the reference (``$TENPY_REFERENCE`` or the
install oracle/_ref that ``build()`` makes from a reference checkout).  Twice: on the numpy test double (host logic) and, ``-m gpu``, with
the state computed and re-imported on the B200."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tenpy_b200 import dropin  # noqa: E402

REF = dropin.reference_path() or ''

SCRIPT = r'''
import sys, pickle, warnings, io
sys.dont_write_bytecode = True
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + '/tests'); sys.path.insert(0, {ref!r})
warnings.simplefilter('ignore')
import numpy as np
from tenpy_b200 import backend
if {fake!r}:
    from fake_device import FakeDeviceLib
    backend.use_library(FakeDeviceLib())
else:
    from tenpy_b200._lib import DeviceLib
    backend.use_library(DeviceLib())
from tenpy_b200.models import SpinChain as MySpinChain
from tenpy_b200.networks.mps import MPS as MyMPS
from tenpy_b200.algorithms import dmrg as mydmrg
from tenpy_b200.tools import interop
import tenpy
from tenpy.models.spins import SpinChain
from tenpy.networks.mps import MPS
from tenpy.networks.mpo import MPOEnvironment
from tenpy.algorithms import dmrg

L = 10
mine = MySpinChain({{'L': L, 'Jx': 1., 'Jy': 1., 'Jz': 0.8, 'conserve': 'Sz'}})
ref = SpinChain(dict(L=L, S=0.5, Jx=1., Jy=1., Jz=0.8, bc_MPS='finite', conserve='Sz'))
psi = MyMPS.from_product_state(mine.lat_sites, ['up', 'down'] * (L // 2))
res = mydmrg.run(psi, mine, {{'mixer': True, 'max_E_err': 1e-11, 'trunc_params': {{'chi_max': 20, 'svd_min': 1e-10}},
                             'max_sweeps': 10}})
# device MPS -> reference MPS -> pickle -> stock TeNPy
rpsi = interop.mps_to_reference(psi, ref.lat.mps_sites())
blob = pickle.dumps(rpsi)
loaded = pickle.loads(blob)
E_ref = MPOEnvironment(loaded, ref.H_MPO, loaded).full_contraction(0)
assert abs(E_ref - res['E']) < 1e-10 * abs(res['E']), (E_ref, res['E'])
assert np.max(np.abs(loaded.entanglement_entropy() - psi.entanglement_entropy())) < 1e-10
assert np.linalg.norm(loaded.norm_test()) < 1e-9
# the reference continues the run from the checkpoint with a larger bond dimension
res2 = dmrg.run(loaded, ref, dict(mixer=True, max_E_err=1e-11, trunc_params=dict(chi_max=32, svd_min=1e-10), max_sweeps=6))
assert res2['E'] <= res['E'] + 1e-10
# ... and the refined reference state comes back to the device representation
back = interop.mps_from_reference(loaded, mine.lat_sites)
from tenpy_b200.networks.mpo import MPOEnvironment as MyEnv
E_back = MyEnv(back, mine.H_MPO, back).full_contraction(0)
assert abs(E_back - res2['E']) < 1e-10 * abs(res2['E']), (E_back, res2['E'])
# single Arrays, incl. a pipe
B = psi.get_B(L // 2).combine_legs(['vL', 'p'])
rB = interop.to_reference(B)
assert np.array_equal(rB.to_ndarray(), B.to_ndarray())
B2 = interop.from_reference(rB)
assert B2._layout.same_blocks(B._layout) and np.array_equal(B2.to_ndarray(), B.to_ndarray())
print('E_device=%.12f E_continued=%.12f' % (res['E'], res2['E']))
'''


def _roundtrip(tmp_path, fake):
    script = tmp_path / 'interop.py'
    script.write_text(SCRIPT.format(root=ROOT, ref=REF, fake=fake))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
    out = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=600, env=env, cwd='/tmp')
    assert out.returncode == 0, out.stdout + out.stderr
    assert 'E_device=' in out.stdout


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'tenpy')), reason='reference not available')
def test_checkpoint_roundtrip_with_reference(tmp_path):
    _roundtrip(tmp_path, True)


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'tenpy')), reason='reference not available (oracle/_ref)')
def test_checkpoint_roundtrip_with_reference_gpu(tmp_path, gpu_lib):
    _roundtrip(tmp_path, False)
