"""CPU test of the drop-in boundary B2 (SURVEY.md section 8b): the UNMODIFIED reference (tenpy/tenpy) runs its own
two-site DMRG with `tenpy.linalg._npc_helper` replaced by `tenpy_b200.shim._npc_helper` through the
reference's plugin switch `tools.optimization.use_cython` (doc-string check included).  Needs the reference
(`tenpy_b200.dropin.reference_path`), skipped without it; device calls go to the numpy test
double here (host logic of the shim), the kernels themselves are covered by the -m gpu tests."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tenpy_b200 import dropin  # noqa: E402

REF = dropin.reference_path() or ''

SCRIPT = r'''
import sys, warnings
sys.dont_write_bytecode = True
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + '/tests'); sys.path.insert(0, {ref!r})
from tenpy_b200 import backend
from fake_device import FakeDeviceLib
backend.use_library(FakeDeviceLib())
from tenpy_b200.shim import _npc_helper as shim
shim.install()
warnings.simplefilter('ignore')
import tenpy
from tenpy.tools import optimization
assert optimization.have_cython_functions
import tenpy.linalg.np_conserved as npc
assert npc._tensordot_worker is shim._tensordot_worker and npc._inner_worker is shim._inner_worker
from tenpy.models.spins import SpinChain
from tenpy.networks.mps import MPS
from tenpy.algorithms import dmrg
L = 10
M = SpinChain(dict(L=L, S=0.5, Jx=1., Jy=1., Jz=1., bc_MPS='finite', conserve='Sz'))
psi = MPS.from_product_state(M.lat.mps_sites(), ['up', 'down'] * (L // 2), bc='finite')
res = dmrg.run(psi, M, dict(mixer=True, max_E_err=1e-10, trunc_params=dict(chi_max=30, svd_min=1e-10), combine=True,
                            max_sweeps=8))
calls = backend.get_lib().calls
assert calls.get('tdot_plan', 0) > 100 and calls.get('dot', 0) > 10
# second run with the SVD worker replaced as well (plain assignment, INTEGRATION.md section A)
shim.install_workers()
psi2 = MPS.from_product_state(M.lat.mps_sites(), ['up', 'down'] * (L // 2), bc='finite')
res2 = dmrg.run(psi2, M, dict(mixer=None, max_E_err=1e-10, trunc_params=dict(chi_max=30, svd_min=1e-10), combine=True,
                              max_sweeps=8))
assert backend.get_lib().calls.get('block_svd', 0) > 10
assert abs(res2['E'] - res['E']) < 1e-9, (res2['E'], res['E'])
print('E=%.12f' % res['E'])
'''


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'tenpy')), reason='reference not available')
def test_reference_dmrg_runs_on_the_shim(tmp_path):
    script = tmp_path / 'dropin.py'
    script.write_text(SCRIPT.format(root=ROOT, ref=REF))
    env = {k: v for k, v in os.environ.items() if k != 'TENPY_NO_CYTHON'}
    r = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    E = float(r.stdout.strip().split('E=')[-1])
    assert abs(E - (-4.258035207282)) < 1e-9     # open Heisenberg chain L=10 (exact diagonalisation value)
