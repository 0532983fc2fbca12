"""bench.py's GPU arm executed on the numpy test double with stubbed CUDA timing (tests/dev_bench_dryrun.py): guards the
host side of the benchmark script -- JSON contract keys, probes, N=1 path -- on a box without a GPU.  The numbers of a
dry run mean nothing and are not checked."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_contract_keys_dry_run(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'dev_bench_dryrun.py'), '--L', '12', '--chi', '16',
                          '--steps', '1', '--warmup', '1', '--cpu-bonds', '1', '--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline'):
        assert key in d, key
    assert d['higher_is_better'] is False and d['dtype'] == 'f64' and 'workload' in d['config']
    for key in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert key in d['roofline'], key
    for key in ('value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'):
        assert key in d['e2e'], key
    for key in ('value', 'unit', 'cores', 'kind', 'sample'):
        assert key in d['cpu_baseline'], key
    assert 'error' not in d['matvec_orders'] and 'error' not in d['roofline_svd']['workload_theta']
    assert all('error' not in p for p in d['blocksparse_matvec'])
    assert 'E_rel_err' in d['parity'] and 'E_exact_free_fermion' in d['parity']
    # --dump-outputs: the last timed sweep's results (L = 12: 20 bond updates, 13 bonds, every tensor entry kept)
    dump = {n: np.load(os.path.join(str(tmp_path), n + '.npy')) for n in ('energy', 'trunc_err', 'schmidt_values', 'B_sample')}
    assert all(a.dtype == np.float64 for a in dump.values())
    assert dump['energy'].shape == dump['trunc_err'].shape == (20,) and dump['schmidt_values'].shape == (13, 16)
    assert abs(dump['energy'][-1] - d['result']['E'][0]) < 1e-12 * abs(dump['energy'][-1])
    dims = [min(2**i, 2**(12 - i), 16) for i in range(13)]
    assert dump['B_sample'].size == sum(dims[i] * 2 * dims[i + 1] for i in range(12))
    # the dumped right-canonical tensors are the final state: their product is normalised and has the last bond energy
    # (TFIChain J = g = 1: H = -sum X_i X_i+1 - sum Z_i)
    psi, at = np.ones(1), 0
    for i in range(12):
        n = dims[i] * 2 * dims[i + 1]
        psi = np.tensordot(psi.reshape(-1, dims[i]), dump['B_sample'][at:at + n].reshape(dims[i], 2, dims[i + 1]), axes=[1, 0])
        at += n
    psi = psi.reshape([2] * 12)
    X, Z = np.array([[0., 1.], [1., 0.]]), np.diag([1., -1.])

    def op(o, i, v):
        return np.moveaxis(np.tensordot(o, v, axes=[1, i]), 0, i)
    E = -sum(np.vdot(psi, op(X, i, op(X, i + 1, psi))) for i in range(11)) - sum(np.vdot(psi, op(Z, i, psi)) for i in range(12))
    assert abs(np.vdot(psi, psi) - 1.) < 1e-12 and abs(E - dump['energy'][-1]) < 1e-10 * abs(E), (np.vdot(psi, psi), E)


def test_bench_reference_arm():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--L', '16', '--chi', '32',
                          '--steps', '1', '--warmup', '0'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    # the unmodified reference (oracle/_ref or $TENPY_REFERENCE) when it is there, the dense numpy port otherwise
    assert d['impl'] == 'reference' and d['cpu_baseline']['kind'] in ('reference', 'port') and d['e2e']['h2d_bytes_per_step'] == 0
    assert d['value'] > 0 and d['config']['chi'] == 32 and d['extrapolated'] is True
    if d['cpu_baseline']['kind'] == 'reference':
        assert d['cpu_baseline']['thread_sweep'] and d['cpu_baseline']['cores'] >= 1
    assert abs(d['value'] - d['per_bond_s'] * d['full_chi_bonds']) < 1e-9 * d['value']


def test_bench_blocksparse_workload_dry_run():
    """`--workload xxz` (BASELINE.json configs[2] end to end: chi ramp with the mixer, timed sweeps) on the test double"""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'dev_bench_dryrun.py'), '--workload', 'xxz', '--L', '10',
                          '--chi', '16', '--steps', '1', '--warmup', '0', '--ramp', '2'], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert d['config']['chi'] == 16 and 'XXZ' in d['config']['workload'] and d['value'] > 0
    assert d['structure']['theta_blocks'] >= 2 and d['chi_reached'] <= 16 and 'gemm_by_flops' in d
