#!/usr/bin/env python
"""bench.py -- DMRG sweep wall-clock and effective-H matvec throughput, 1..N B200 vs the reference CPU path.

Workload (BASELINE.json configs[1]): TFIChain L=100, two-site DMRG at chi=1024, no charge conservation
(dense-block path).  One *step* = one full DMRG sweep = 2(L-2) = 196 two-site bond updates through
``tenpy_b200.algorithms.dmrg.TwoSiteDMRGEngine.sweep`` (Lanczos with the effective-H matvec, block SVD +
truncation, environment update), starting from a synthetic random right-canonical-on-average MPS whose inner
bonds are saturated at chi.  As in the reference's own benchmark harness
(tests/benchmark/dmrg_infinite.py:31-37) the Lanczos iteration count is fixed (N_min = N_max = 10) and
``svd_min`` is tiny so that chi stays saturated -> every step does identical work.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # CPU: oracle restatement of the reference path

N > 1 (launched by torchrun): the path shards over independent DMRG runs (a field scan, BASELINE.json
configs[4]); rank r runs the same workload at g = 1 + 0.02 r, the only collectives are an NCCL broadcast of
the model template and an all-gather of the per-run results; ``value`` = max-over-ranks sweep time / N
(seconds per sweep of the whole job, weak scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'dmrg_two_site_sweep_wall_clock'
UNIT = 's'
FP64_TENSOR_PEAK_TFLOPS = 37.0   # B200 (HGX) FP64 tensor/DFMA spec; MEASURED_PEAKS.json has no FP64 entry


def gemm_ncu_numbers():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch and tensor-pipe activity of the matvec GEMM kernel,
    taken from the committed ncu --set full summary (profiles/gemm_ncu.json, written from the capture named in it);
    ``(None, None, None)`` if no capture of the current kernel configuration is committed."""
    path = os.path.join(ROOT, 'profiles', 'gemm_ncu.json')
    if not os.path.exists(path):
        return None, None, None
    with open(path) as f:
        d = json.load(f)
    return d.get('dram_bytes_per_launch'), d.get('tensor_pipe_active_pct'), d.get('source')


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=1)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--L', type=int, default=100)
    ap.add_argument('--chi', type=int, default=1024)
    ap.add_argument('--lanczos-N', type=int, default=10)
    ap.add_argument('--cpu-bonds', type=int, default=2, help='bond updates per CPU sample')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-blocksparse', action='store_true', help='skip the configs[2]/[3] shaped matvec probes')
    ap.add_argument('--workload', default='tfi', choices=['tfi', 'xxz', 'hubbard'],
                    help='tfi = BASELINE.json configs[1] (the metric; default).  xxz / hubbard = configs[2] / [3] end to end: '
                         'SpinChain L=100 chi=1024 (U(1) Sz) / FermiHubbardChain L=64 chi=2048 (U(1)xU(1)): chi ramp with the '
                         'density-matrix mixer, then timed sweeps (own line, not the contract metric)')
    ap.add_argument('--svd-warm-start', default='default', choices=['default', 'off', 'subspace', 'full'],
                    help='--workload xxz|hubbard: engine option svd_warm_start (default: the engine default)')
    ap.add_argument('--svd-min', type=float, default=1e-10, help='--workload xxz|hubbard: truncation threshold svd_min')
    ap.add_argument('--svd-inner-sweeps', type=int, default=0,
                    help='--workload xxz|hubbard: inner sweeps of the pivot eigen-solver of the block SVD (0: library default)')
    ap.add_argument('--ramp', type=int, default=6, help='--workload xxz|hubbard: sweeps of the chi ramp (doubling from 32)')
    ap.add_argument('--driver', default='own', choices=['own', 'reference'],
                    help="'reference': the unmodified tenpy TwoSiteDMRGEngine (tenpy_b200.dropin) drives the sweep on the device "
                         "engine instead of tenpy_b200.algorithms.dmrg (short line; the default run reports it as `reference_driver`)")
    ap.add_argument('--scan', default='auto', choices=['auto', 'on', 'off'],
                    help='BASELINE.json configs[4]: chi in {256,512,1024,2048} x two fields, sharded over the ranks by LPT '
                         '(tenpy_b200.scan); auto = on for N > 1')
    ap.add_argument('--scan-chis', default='256,512,1024,2048')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed sweep computed (energies, truncation errors, Schmidt values, a seeded '
                         'sample of the MPS tensors) to DIR/<name>.npy, float64, rank 0 only; default workload only')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'b200' or args.workload != 'tfi' or args.driver != 'own'):
        ap.error('--dump-outputs applies to the default workload of the b200 arm only')
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return json.load(f), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback'


# ------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler(threading.Thread):
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in out.stdout.strip().split(',')]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.5)

    def summary(self):
        self.stop_flag = True
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = set()
        for s in self.samples:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.samples[0][1]),
                'power_w_max': max(float(s[2]) for s in self.samples), 'reasons': sorted(reasons),
                'samples': len(self.samples)}


# ------------------------------------------------------------------------------------------ CPU (oracle) arm
def _use_all_host_threads():
    """BLAS/LAPACK on every host core, also under torchrun (which exports OMP_NUM_THREADS=1 to its workers)."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([int(p.get('num_threads', 1)) for p in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count()


def cpu_bond_sample(chi, d, D, lanczos_N, n_bonds, seed=0):
    """time `n_bonds` two-site updates at the chain centre (full chi) with the dense CPU oracle, once with the
    reference's default matvec (combine=True: LHeff.theta.RHeff) and once with its combine=False contraction order
    inside Lanczos (d times fewer flops); the faster one is the CPU baseline."""
    from oracle import dmrg_dense as od
    _use_all_host_threads()
    rng = np.random.default_rng(seed)
    n = chi * d
    LP = rng.standard_normal((chi, D, chi))
    LP = LP + LP.transpose(2, 1, 0)
    RP = rng.standard_normal((chi, D, chi))
    RP = RP + RP.transpose(2, 1, 0)
    W = od.tfi_mpo(1., 1.)
    LHeff, RHeff = od.contract_LHeff(LP, W), od.contract_RHeff(RP, W)
    theta = rng.standard_normal((n, n))
    theta /= np.linalg.norm(theta)
    trunc = dict(chi_max=chi, svd_min=1e-45, trunc_cut=None)
    lan = dict(N_min=lanczos_N, N_max=lanczos_N)

    def mv_split(x):
        return od.matvec_split(LP, W, W, RP, x.reshape(chi, d, d, chi)).reshape(n, n)
    t_mv = {}
    for name, fn in (('combined', lambda x: od.matvec(LHeff, RHeff, x)), ('split', mv_split)):
        fn(theta)
        t1 = time.perf_counter()
        fn(theta)
        t_mv[name] = time.perf_counter() - t1
    best = min(t_mv, key=t_mv.get)
    t0 = time.perf_counter()
    for b in range(n_bonds):
        od.bond_update(LHeff, RHeff, theta, trunc, lan, move_right=(b % 2 == 0),
                       matvec_fn=mv_split if best == 'split' else None)
    dt = time.perf_counter() - t0
    return dt / n_bonds, t_mv, best


def cpu_sweep_estimate(args, n_bonds):
    """CPU sweep estimate = (number of full-chi bond updates per sweep) x (time of one such update)."""
    d, D = 2, 3
    full = n_full_bonds(args.L, args.chi, d)
    per_bond, t_mv, best = cpu_bond_sample(args.chi, d, D, args.lanczos_N, n_bonds)
    from oracle import dmrg_dense as od
    fl = od.matvec_flops(args.chi * d, D, args.chi * d)
    return {'sweep_s': full * per_bond, 'per_bond_s': per_bond, 'matvec_s': t_mv['combined'],
            'matvec_split_s': t_mv['split'], 'matvec_order_used': best,
            'matvec_gflops': fl / t_mv['combined'] / 1e9, 'full_chi_bonds': full}


def n_full_bonds(L, chi, d):
    """number of the 2(L-2) bond updates of a sweep whose theta has the full (chi d) x (d chi) size"""
    dims = [min(d**i, d**(L - i), chi) for i in range(L + 1)]
    i0s = list(range(0, L - 2)) + list(range(L - 2, 0, -1))
    return sum(1 for i0 in i0s if dims[i0] == chi and dims[i0 + 2] == chi)


# ------------------------------------------------------------------------------------------ the REAL reference on the CPU
def exact_tfi_energy(L, J, g):
    """exact ground-state energy of the open transverse-field Ising chain H = -J sum sx sx - g sum sz (the TFIChain of the
    benchmark) through the Jordan-Wigner free-fermion form: E0 = -sum of the singular values of (g 1 + J shift)"""
    M = g * np.eye(L) + J * np.eye(L, k=1)
    return -float(np.sum(np.linalg.svd(M, compute_uv=False)))


def synthetic_tensors_host(L, chi, d, seed):
    """the benchmark state as host arrays: B[i] of shape (chi_l, d, chi_r) right-isometric (QR of a seeded Gaussian),
    Schmidt values decaying over 7 e-folds.  Generated with torch on the GPU when there is one (the same generator and
    seeds as `synthetic_mps`, so both arms start from the identical state), else with numpy."""
    import torch
    dims = [min(d**i, d**(L - i), chi) for i in range(L + 1)]
    Bs, Ss = [], []
    cuda = torch.cuda.is_available()
    if cuda:
        dev = torch.device('cuda', torch.cuda.current_device())
        gen = torch.Generator(device=dev)
        gen.manual_seed(1234 + seed)
    else:
        rng = np.random.default_rng(1234 + seed)
    for i in range(L):
        cl, cr = dims[i], dims[i + 1]
        if cuda:
            g_ = torch.randn(d * cr, cl, dtype=torch.float64, device=dev, generator=gen)
            qm, _ = torch.linalg.qr(g_)
            B = qm.t().contiguous().cpu().numpy()
        else:
            qm, _ = np.linalg.qr(rng.standard_normal((d * cr, cl)))
            B = np.ascontiguousarray(qm.T)
        Bs.append(B.reshape(cl, d, cr))
        s_ = np.exp(-7. * np.arange(cl) / max(cl, 2))
        Ss.append(s_ / np.linalg.norm(s_))
    Ss.append(np.ones(1))
    return Bs, Ss


class ReferenceArm:
    """The unmodified reference (tenpy from ``oracle/_ref`` -- the install with the compiled Cython helper that ``build()``
    makes -- or ``$TENPY_REFERENCE``) on the host cores: its own TFIChain, MPS, MPOEnvironment and TwoSiteDMRGEngine on its own
    NumPy / BLAS / LAPACK engine, the same synthetic state and options as the GPU arm.  A full sweep at chi = 1024 takes
    10-20 minutes on the CPU, so one step is a BOUNDED SAMPLE: `n_bonds` bond updates at the chain centre through
    ``engine.sweep()`` with the schedule restricted to these bonds, scaled to the 158 full-chi bonds of a sweep
    (``extrapolated: true`` in the line)."""

    def __init__(self, args):
        from tenpy_b200 import dropin
        self.path = dropin.reference_path()
        if self.path is None:
            raise RuntimeError('no reference install (oracle/_ref) or $TENPY_REFERENCE found')
        if self.path not in sys.path:
            sys.path.insert(0, self.path)
        import tenpy
        from tenpy.algorithms import dmrg as rdmrg
        from tenpy.models.tf_ising import TFIChain
        from tenpy.networks.mps import MPS
        from tenpy.tools import optimization
        assert tenpy.linalg.np_conserved.__name__ == 'tenpy.linalg.np_conserved'     # the reference's own engine
        self.tenpy = tenpy
        self.compiled = bool(optimization.have_cython_functions)
        L, chi, d = args.L, args.chi, 2
        self.L, self.chi = L, chi
        M = TFIChain({'L': L, 'J': 1., 'g': 1., 'bc_MPS': 'finite', 'conserve': None})
        Bs, Ss = synthetic_tensors_host(L, chi, d, seed=0)
        psi = MPS.from_Bflat(M.lat.mps_sites(), [B.transpose(1, 0, 2) for B in Bs], SVs=_bond_svs(Ss, L), bc='finite',
                             form='B')
        opts = {'mixer': None, 'combine': True, 'diag_method': 'lanczos',
                'trunc_params': {'chi_max': chi, 'svd_min': 1e-45, 'trunc_cut': None},
                'lanczos_params': {'N_min': args.lanczos_N, 'N_max': args.lanczos_N}}
        c = L // 2 - 1

        class CentreBonds(rdmrg.TwoSiteDMRGEngine):
            """the reference engine; only the schedule is restricted (and environments are kept between steps)"""
            n_bonds = 1

            def get_sweep_schedule(self):
                return [(c + j, True, [True, False]) for j in range(self.n_bonds)]

            def free_no_longer_needed_envs(self):
                pass
        self.eng = CentreBonds(psi, M, opts)
        self.psi, self.M, self.centre = psi, M, c
        self.threads = None

    def choose_threads(self):
        """BLAS threads in {1, 4, 16, 64, all}: the effective-H matvec and the SVD of the centre theta, each with the best
        count (the reference's benchmark harness sweeps OMP threads the same way, tests/benchmark/benchmark.py:37)"""
        from threadpoolctl import threadpool_limits
        from tenpy.algorithms.mps_common import TwoSiteH
        import tenpy.linalg.np_conserved as npc
        ncpu = os.cpu_count() or 1
        cands = sorted(set([t for t in (1, 4, 16, 64) if t < ncpu] + [ncpu]))
        H = TwoSiteH(self.eng.env, self.centre, combine=True)
        theta = self.psi.get_theta(self.centre, 2).combine_legs([['vL', 'p0'], ['p1', 'vR']], qconj=[+1, -1])
        res = {}
        for t in cands:
            with threadpool_limits(limits=t):
                H.matvec(theta)
                t0 = time.perf_counter()
                H.matvec(theta)
                t_mv = time.perf_counter() - t0
                t0 = time.perf_counter()
                npc.svd(theta, inner_labels=['vR', 'vL'])
                t_svd = time.perf_counter() - t0
            res[t] = {'matvec_s': t_mv, 'svd_s': t_svd, 'bond_estimate_s': self.eng.lanczos_params['N_max'] * t_mv + t_svd}
        self.thread_sweep = res
        self.threads = min(res, key=lambda t: res[t]['bond_estimate_s'])
        return self.threads

    def step(self, n_bonds=1):
        """`n_bonds` centre-bond updates through the reference engine; seconds per bond"""
        from threadpoolctl import threadpool_limits
        self.eng.n_bonds = n_bonds
        with threadpool_limits(limits=self.threads or os.cpu_count()):
            t0 = time.perf_counter()
            self.eng.sweep()
            dt = time.perf_counter() - t0
        return dt / n_bonds


def reference_components_sample(args, budget_s=40.):
    """`cpu_baseline` of the GPU arm's line: the pieces of ONE centre-bond update timed on the unmodified reference's own
    engine (tenpy.linalg.np_conserved from oracle/_ref: `npc.tensordot` for the two contractions of `TwoSiteH.matvec`,
    `npc.svd` of the two-site wave function of the benchmark state), without building the 2 x 49 environments a real sweep
    needs (the `--impl reference` arm does that): bond = N_lanczos matvecs + SVD + environment update (3/4 matvec,
    SURVEY.md section 8a9).  Returns None when no reference is installed."""
    from tenpy_b200 import dropin
    path = dropin.reference_path()
    if path is None or dropin.installed():
        return None
    if path not in sys.path:
        sys.path.insert(0, path)
    import tenpy.linalg.np_conserved as npc
    from threadpoolctl import threadpool_limits
    chi, d, D, L = args.chi, 2, 3, args.L
    n = chi * d
    rng = np.random.default_rng(0)
    Bs, Ss = synthetic_tensors_host(L, chi, d, seed=0)
    c = L // 2 - 1
    th = np.tensordot(Ss[c][:, None, None] * Bs[c], Bs[c + 1], axes=[2, 0]).reshape(n, n)     # theta of the benchmark state
    del Bs
    LH = rng.standard_normal((n, D, n))
    RH = rng.standard_normal((D, n, n))
    LHeff = npc.Array.from_ndarray_trivial(LH + LH.transpose(2, 1, 0), labels=['(vR*.p0)', 'wR', '(vR.p0*)'])
    RHeff = npc.Array.from_ndarray_trivial(RH, labels=['wL', '(p1*.vL)', '(p1.vL*)'])
    theta = npc.Array.from_ndarray_trivial(th, labels=['(vL.p0)', '(p1.vR)'])
    del LH, RH

    def matvec(x):           # tenpy/algorithms/mps_common.py:1337-1339
        x = npc.tensordot(LHeff, x, axes=['(vR.p0*)', '(vL.p0)'])
        return npc.tensordot(x, RHeff, axes=[['wR', '(p1.vR)'], ['wL', '(p1*.vL)']])
    ncpu = os.cpu_count() or 1
    res, t_used = {}, time.perf_counter()
    for t in sorted(set([x for x in (8, 32) if x < ncpu] + [ncpu])):
        with threadpool_limits(limits=t):
            matvec(theta)
            t0 = time.perf_counter()
            matvec(theta)
            t_mv = time.perf_counter() - t0
            t0 = time.perf_counter()
            npc.svd(theta, inner_labels=['vR', 'vL'])
            t_svd = time.perf_counter() - t0
        res[t] = {'matvec_s': t_mv, 'svd_s': t_svd, 'bond_s': (args.lanczos_N + 0.75) * t_mv + t_svd}
        if time.perf_counter() - t_used > budget_s:
            break
    best = min(res, key=lambda t: res[t]['bond_s'])
    full = n_full_bonds(L, chi, d)
    return {'value': res[best]['bond_s'] * full, 'unit': UNIT, 'cores': best, 'kind': 'reference',
            'sample': 'unmodified tenpy engine (%s): 1 effective-H matvec (LHeff.theta.RHeff, 4 D d^3 chi^3 flop) and 1 npc.svd '
                      'of the centre two-site wave function of the benchmark state, best of BLAS threads %s; bond = %d matvecs '
                      '+ SVD + 0.75 matvec (environment update), x %d full-chi bonds per sweep'
                      % (path, sorted(res), args.lanczos_N, full),
            'per_bond_s': res[best]['bond_s'], 'matvec_s': res[best]['matvec_s'], 'svd_s': res[best]['svd_s'],
            'matvec_gflops': 4. * D * d**3 * float(chi)**3 / res[best]['matvec_s'] / 1e9, 'thread_sweep': {str(k): v for k, v in res.items()},
            'host_cpus': ncpu, 'extrapolated': True}


def _bond_svs(Ss, L):
    """singular values on the L+1 bonds for MPS.from_Bflat (form 'B': S[i] is left of site i)"""
    return [Ss[i] for i in range(L)] + [np.ones(1)]


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    try:
        arm = ReferenceArm(args)
        kind = 'reference'
    except Exception as e:      # no reference on this box: the oracle port keeps the arm alive
        arm, kind, why = None, 'port', repr(e)
    if arm is None:
        vals = []
        for it in range(args.warmup + args.steps):
            est = cpu_sweep_estimate(args, 1)
            if it >= args.warmup:
                vals.append(est)
        per_bond = float(np.mean([e['per_bond_s'] for e in vals]))
        full = vals[0]['full_chi_bonds']
        cores, extra = blas_threads(), {'fallback_reason': why, 'matvec_s': vals[0]['matvec_s']}
        sample = '1 centre-bond update per step with the dense numpy port oracle/dmrg_dense.py (reference not installed here)'
    else:
        arm.step(1)                               # builds the 2 x 49 environments up to the centre (not timed)
        threads = arm.choose_threads()
        # one bond update of this workload takes 5-50 s on the host (LAPACK on a numerically low-rank 2048 x 2048 theta):
        # W warm-up steps, then exactly K timed ones
        for _ in range(args.warmup):
            arm.step(1)
        per = [arm.step(1) for _ in range(args.steps)]
        per_bond = float(np.mean(per))
        full = n_full_bonds(args.L, args.chi, 2)
        cores = threads
        sw = arm.thread_sweep
        extra = {'reference_path': arm.path, 'cython_helper_compiled': arm.compiled, 'host_cpus': os.cpu_count(),
                 'thread_sweep': {str(k): v for k, v in sw.items()}, 'matvec_s': sw[threads]['matvec_s'],
                 'svd_s': sw[threads]['svd_s'],
                 'matvec_gflops': 4. * 3 * 8 * float(args.chi)**3 / sw[threads]['matvec_s'] / 1e9,
                 'per_bond_s_each_step': per, 'steps_measured': len(per)}
        sample = ('1 bond update at the chain centre per step through the unmodified tenpy TwoSiteDMRGEngine.sweep() '
                  '(schedule restricted to that bond; %d Lanczos matvecs LHeff.theta.RHeff + LAPACK SVD + environment '
                  'update, %d BLAS threads = best of the thread sweep), x %d full-chi bonds of a sweep'
                  % (args.lanczos_N, threads, full))
    v = per_bond * full
    line = {'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': v * 1e3, 'higher_is_better': False, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'impl': 'reference',
            'config': workload_config(args, 1), 'extrapolated': True, 'per_bond_s': per_bond, 'full_chi_bonds': full,
            'cpu_baseline': dict({'value': v, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': sample}, **extra),
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def workload_config(args, n):
    return {'workload': 'TFIChain L=%d two-site DMRG sweep (%d bond updates) at chi=%d, conserve=None (dense-block '
                        'path), d=2, MPO D=3, Lanczos N_min=N_max=%d, svd_min=1e-45' %
                        (args.L, 2 * (args.L - 2), args.chi, args.lanczos_N),
            'L': args.L, 'chi': args.chi, 'lanczos_N': args.lanczos_N,
            'matvec_order': "auto ('split' for theta blocks >= 2^20 elements: LP, W0 W1, RP applied to the split theta, "
                            "4 D d^2 chi^3 flop instead of the reference default's 4 D d^3 chi^3; same result); the "
                            "identity components LP[IdL] = RP[IdR] = 1 of the environments (checked per bond) are not "
                            "multiplied: 4 (D-1) d^2 chi^3 flop in the two large GEMMs",
            'svd': 'b200 arm: block Jacobi SVD with svd_deflation_tol=1e-10 (directions below 1e-10 |theta| are not iterated to '
                   'convergence; they get an orthonormal completion because svd_min=1e-45 keeps them, as the reference keeps '
                   "LAPACK's ~1e-17 values); reference arm: LAPACK gesdd",
            'parallelism': 'independent DMRG runs (field scan g=1+0.02*rank), %d rank(s)' % n,
            'l2': 'working set per step (100 x (LP, RP, B) ~ 7 GB) >> 126 MB L2; no explicit flush'}


# ------------------------------------------------------------------------------------------ GPU arm
def synthetic_mps(model, L, chi, d, seed):
    """random MPS with saturated inner bonds; B ~ N(0, 1/(d chi_r)) is right-isometric on average."""
    import torch
    from tenpy_b200 import backend
    from tenpy_b200.linalg import np_conserved as npc
    from tenpy_b200.linalg.charges import LegCharge
    from tenpy_b200.networks.mps import MPS
    dev = backend.get_lib().device
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + seed)
    dims = [min(d**i, d**(L - i), chi) for i in range(L + 1)]
    chinfo = model.lat_sites[0].leg.chinfo
    Bs, Ss = [], []
    for i in range(L):
        cl, cr = dims[i], dims[i + 1]
        n = cl * d * cr
        n_pad = (n + 15) // 16 * 16
        buf = torch.zeros(n_pad, dtype=torch.float64, device=dev)
        # right-canonical B: rows of the (cl x d*cr) matrix orthonormal (QR of a random matrix; data
        # generation only, outside every timed region)
        g = torch.randn(d * cr, cl, dtype=torch.float64, device=dev, generator=gen)
        qm, _ = torch.linalg.qr(g)
        buf[:n] = qm.t().contiguous().reshape(-1)
        legs = [LegCharge.from_trivial(cl, chinfo, +1), model.lat_sites[i].leg, LegCharge.from_trivial(cr, chinfo, -1)]
        Bs.append(npc.Array.from_device_buffer(legs, np.zeros((1, 3), np.int64), buf, labels=['vL', 'p', 'vR']))
        # Schmidt values decaying over ~3 decades across the bond (an entangled, well-conditioned state)
        s = np.exp(-7. * np.arange(cl) / max(cl, 2))
        Ss.append(s / np.linalg.norm(s))
    Ss.append(np.ones(1))
    return MPS(model.lat_sites, Bs, Ss, 'finite', 'B')


def psi_to_host(psi):
    """D2H of all MPS tensors (the result of a sweep)"""
    from tenpy_b200 import backend
    out, nbytes = [], 0
    for B in psi._B:
        h = backend.to_host(B._buf)
        nbytes += h.nbytes
        out.append(h)
    return out, nbytes


def psi_from_host(psi, host_bufs):
    """H2D of all MPS tensors from pinned host memory"""
    nbytes = 0
    for B, h in zip(psi._B, host_bufs):
        B._buf.copy_(h, non_blocking=True)
        nbytes += h.numel() * 8
    return nbytes


DUMP_MAX_BYTES = (64 << 20) - 4096     # all files of --dump-outputs together, .npy headers included


def _seeded_sample(a, k, rng):
    """all of `a` if it has at most `k` entries, else `k` of them chosen by `rng` (in index order)"""
    return a if a.size <= k else a[np.sort(rng.choice(a.size, k, replace=False))]


def dump_outputs(out_dir, eng, psi, L):
    """What a caller of the timed sweep receives, as float64 .npy files of at most DUMP_MAX_BYTES together: the energy and
    truncation error of each bond update of the last sweep, the Schmidt values of every bond (zero-padded to the largest
    bond dimension; a seeded sample of that array if it would take more than a quarter of the budget) and a seeded sample
    of every MPS tensor in right-canonical form, (vL, p, vR) order (all entries of a small tensor; the same entries for
    the same shapes)."""
    os.makedirs(out_dir, exist_ok=True)
    nb = 2 * (L - 2)
    energy = np.asarray([float(e) for e in eng.update_stats['E_total'][-nb:]], np.float64)
    err = np.asarray([float(getattr(e, 'eps', e)) for e in eng.update_stats['err'][-nb:]], np.float64)
    budget = DUMP_MAX_BYTES // 8 - energy.size - err.size           # float64 entries left for S and the B sample
    Ss = [np.asarray(s.detach().cpu() if hasattr(s, 'detach') else s, np.float64).ravel() for s in psi._S]
    S = np.zeros((len(Ss), max(len(s) for s in Ss)), np.float64)
    for i, s in enumerate(Ss):
        S[i, :len(s)] = s
    rng = np.random.default_rng(0)
    if S.size > budget // 4:
        S = _seeded_sample(S.ravel(), budget // 4, rng)
    per_site = (budget - S.size) // L
    samples = []
    for i in range(L):
        B = psi.get_B(i, 'B')
        dense = B.to_ndarray().transpose([B.get_leg_labels().index(l) for l in ('vL', 'p', 'vR')]).ravel()
        samples.append(_seeded_sample(dense, per_site, rng))
    for name, a in (('energy', energy), ('trunc_err', err), ('schmidt_values', S), ('B_sample', np.concatenate(samples))):
        np.save(os.path.join(out_dir, name + '.npy'), a)


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from tenpy_b200 import backend
    from tenpy_b200._lib import DeviceLib
    lib = backend.use_library(DeviceLib())
    from tenpy_b200.models import TFIChain
    from tenpy_b200.algorithms import dmrg
    d, D = 2, 3
    L, chi = args.L, args.chi

    # model: rank 0 owns the template (J, g0); NCCL broadcast, every rank patches its own field g
    tmpl = torch.tensor([1.0, 1.0], dtype=torch.float64, device=lib.device)
    if world > 1:
        dist.broadcast(tmpl, src=0)
    J, g0 = float(tmpl[0]), float(tmpl[1])
    g = g0 + 0.02 * rank
    model = TFIChain({'L': L, 'J': J, 'g': g, 'conserve': None})
    psi = synthetic_mps(model, L, chi, d, seed=rank)
    opts = {'mixer': None, 'combine': True, 'diag_method': 'lanczos',      # as tests/benchmark/dmrg_infinite.py:9,44
            'trunc_params': {'chi_max': chi, 'svd_min': 1e-45, 'trunc_cut': None, 'svd_deflation_tol': 1e-10},
            'lanczos_params': {'N_min': args.lanczos_N, 'N_max': args.lanczos_N},
            # cold-started SVD at every bond (the subspace warm start would only engage below the 1e-10 tolerance,
            # the Lanczos update of this workload changes theta by ~2e-7 per bond)
            'svd_warm_start': False}
    eng = dmrg.TwoSiteDMRGEngine(psi, model, opts)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up sweeps
    for w in range(args.warmup):
        eng.sweep()

    # ---- timed region: exactly K sweeps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    lib.kernel_launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()     # cudaProfilerStart: lets `ncu --profile-from-start off` see only the timed steps
    ev0.record()
    for _ in range(args.steps):
        eng.sweep()
    ev1.record()
    torch.cuda.profiler.stop()
    barrier()
    launches = lib.kernel_launch_count()
    ms = ev0.elapsed_time(ev1) / args.steps
    clocks = sampler.summary() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, psi, L)
    E_final = eng.update_stats['E_total'][-1]
    S_mid = eng._entropy_approx[L // 2]
    N_lan = float(np.mean(eng.update_stats['N_lanczos'][-2 * (L - 2):]))
    from tenpy_b200.linalg.np_conserved import svd_stats
    from tenpy_b200.linalg.truncation import subspace_stats as sub_stats
    jsw = svd_stats['jacobi_sweeps'][-2 * (L - 2):]

    from tenpy_b200.algorithms.mps_common import TwoSiteH as _H2
    id_stats = dict(_H2.stats)      # bonds of all sweeps so far on which the identity-environment shortcut applied

    # ---- A/B of the identity-environment shortcut of the matvec (same state, same work otherwise): one sweep without it
    ab = {}
    if rank == 0 or world == 1:
        try:
            eng.options['identity_env'] = False
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a0.record()
            eng.sweep()
            a1.record()
            torch.cuda.synchronize()
            ab['sweep_s_identity_env_off'] = a0.elapsed_time(a1) / 1e3
        except Exception as e:   # never lose the bench line
            ab['error'] = repr(e)
        finally:
            eng.options.pop('identity_env', None)

    # ---- one more sweep with per-family CUDA-event profiling (after the timed one: same, converged regime; the
    #      event pairs bracket every library call, so host gaps inside a call -- the SVD reads q doubles per Jacobi
    #      sweep -- count for that family)
    lib.profile = {}
    eng.sweep()
    prof = lib.profile_summary()
    lib.profile = None

    # ---- end-to-end: the same sweep through the public API with HOST buffers (H2D + D2H inside the timer)
    e2e = None
    if not args.no_e2e:
        host, _ = psi_to_host(psi)
        pinned = [torch.from_numpy(h).pin_memory() for h in host]
        barrier()
        t0 = time.perf_counter()
        h2d = psi_from_host(psi, pinned)
        eng.env.clear()
        eng.sweep()
        _, d2h = psi_to_host(psi)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        barrier()
        e2e = {'value': e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
               'note': 'MPS tensors from pinned host memory -> sweep (environments rebuilt) -> MPS back to host'}

    # ---- the same state with the reference's DEFAULT Lanczos settings (N_min=2, N_max=20, convergence by P_tol): a converged
    #      DMRG needs 2-3 matvecs per bond instead of the harness' fixed 10, so SVD / block moves / host latencies weigh more
    default_lanczos = {}
    try:
        opts2 = dict(opts)
        opts2['lanczos_params'] = {}
        eng2 = dmrg.TwoSiteDMRGEngine(psi, model, opts2)
        eng2.sweep()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        b0.record()
        eng2.sweep()
        b1.record()
        torch.cuda.synchronize()
        default_lanczos = {'sweep_s': b0.elapsed_time(b1) / 1e3,
                           'N_lanczos_mean': float(np.mean(eng2.update_stats['N_lanczos'][-2 * (L - 2):])),
                           'E': float(eng2.update_stats['E_total'][-1])}
        del eng2
    except Exception as e:   # never lose the bench line
        default_lanczos = {'error': repr(e)}

    # ---- kernel roofline probes at the centre-bond shapes (CUDA events on the launching stream)
    roof = kernel_probes(lib, chi, d, D)
    mv_orders = matvec_order_probe(eng, psi, L, chi, d, D)
    roof['svd']['workload_theta'] = svd_theta_probe(eng, psi, L)
    bs_probes = blocksparse_probes(small=(chi < 256)) if not args.no_blocksparse else None

    # ---- BASELINE.json configs[4]: the unequal-chi scan, sharded over the ranks (after the equal-work measurement)
    scan_res = None
    if args.scan == 'on' or (args.scan == 'auto' and world > 1):
        del eng, psi
        torch.cuda.empty_cache()
        try:
            scan_res = run_chi_scan(args, lib, world, rank)
        except Exception as e:   # never lose the bench line
            scan_res = {'error': repr(e)}

    # ---- gather over ranks
    stats = torch.tensor([ms, E_final, S_mid, e2e['value'] if e2e else 0.], dtype=torch.float64, device=lib.device)
    if world > 1:
        allst = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
        allst = torch.stack(allst).cpu().numpy()
    else:
        allst = stats.cpu().numpy()[None, :]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_max = float(allst[:, 0].max())
    value = ms_max / 1e3 / world
    # parity of the benchmark's own result: the energies of all ranks against the exact free-fermion ground-state energy
    # of the open chain (rank r runs g = g0 + 0.02 r); the line is marked failed above 1e-10 relative
    E_exact = [exact_tfi_energy(L, J, g0 + 0.02 * r) for r in range(world)]
    E_err = [abs(float(allst[r, 1]) - E_exact[r]) / abs(E_exact[r]) for r in range(world)]
    parity = {'E_exact_free_fermion': E_exact, 'E_rel_err': E_err, 'tolerance': 1e-10, 'ok': bool(max(E_err) <= 1e-10)}
    peaks, peaks_kind = measured_peaks()
    total_ms = sum(v[1] for v in prof.values()) or 1.
    shares = {k: round(v[1] / total_ms, 4) for k, v in prof.items()}
    dominant = max(shares, key=shares.get) if shares else 'gemm'
    roofline = roof['svd'] if dominant == 'svd' else roof['gemm']
    roofline = dict(roofline)
    roofline['kernel'] = 'jacobi_gram/eig/apply_kernel (block SVD)' if dominant == 'svd' else 'oz_gemm_kernel (matvec, tcgen05 kind::i8)'
    roofline['share_of_step'] = shares.get(dominant)
    if e2e:
        e2e['value'] = float(allst[:, 3].max()) / world
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_max, 'higher_is_better': False, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'impl': 'b200',
            'config': workload_config(args, world), 'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches),
            'roofline': roofline, 'roofline_gemm': roof['gemm'], 'roofline_svd': roof['svd'],
            'kernel_time_shares': shares, 'kernel_family_ms_per_sweep': {k: round(v[1], 2) for k, v in prof.items()},
            'matvec_orders': mv_orders, 'matvec_gflops': _matvec_gflops(mv_orders),
            'blocksparse_matvec': bs_probes, 'ab': ab, 'identity_env_stats': id_stats, 'peaks': peaks_kind, 'parity': parity,
            'chi_scan': scan_res, 'reference_default_lanczos': default_lanczos,
            'result': {'E': [float(x) for x in allst[:, 1]], 'S_mid': [float(x) for x in allst[:, 2]],
                       'N_lanczos_mean': N_lan, 'svd_jacobi_sweeps_mean': float(np.mean(jsw)),
                       'svd_jacobi_sweeps_max': int(np.max(jsw)), 'svd_calls': svd_stats['calls'],
                       'svd_warm_starts': svd_stats.get('guess_used', 0),
                       'svd_null_space_completions': svd_stats.get('completions', 0),
                       'svd_subspace_tried': sub_stats['tried'], 'svd_subspace_used': sub_stats['used'],
                       'svd_subspace_residual_median': float(np.median(sub_stats['residuals'][-2 * (L - 2):]))
                       if sub_stats['residuals'] else None}}
    if not args.no_cpu:
        cb = None
        try:
            cb = reference_components_sample(args)
        except Exception as e:      # never lose the bench line
            cb = None
            line['cpu_baseline_reference_error'] = repr(e)
        if cb is None:
            est = cpu_sweep_estimate(args, args.cpu_bonds)
            cb = {'value': est['sweep_s'], 'unit': UNIT, 'cores': blas_threads(), 'kind': 'port',
                  'sample': '%d centre-bond updates (oracle/dmrg_dense.py, numpy/OpenBLAS/LAPACK gesdd; Lanczos matvec in '
                            'the faster of the two reference contraction orders: %s) x %d full-chi bonds per sweep'
                            % (args.cpu_bonds, est['matvec_order_used'], est['full_chi_bonds']),
                  'per_bond_s': est['per_bond_s'], 'matvec_gflops': est['matvec_gflops'],
                  'matvec_s': est['matvec_s'], 'matvec_split_s': est['matvec_split_s']}
        line['cpu_baseline'] = cb
    if world == 1 and not args.no_e2e:
        # the same sweep driven by the unmodified reference's engine class (own process)
        try:
            del eng, psi
        except NameError:
            pass
        torch.cuda.empty_cache()
        line['reference_driver'] = reference_driver_line(args)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if not parity['ok']:
        sys.stderr.write('bench.py: energy parity FAILED: rel. err %r > 1e-10\n' % (E_err,))
        sys.exit(3)


def run_chi_scan(args, lib, world, rank):
    """BASELINE.json configs[4]: 8 independent DMRG runs, chi in {256, 512, 1024, 2048} x g in {0.9, 1.1}, sharded over the
    ranks with `tenpy_b200.scan` (largest estimated cost chi^3 first; every rank pulls its next run when it becomes free).  Each run = the
    benchmark's workload at its own chi: synthetic state, one warm-up sweep, one timed sweep (CUDA events).  Returns on
    rank 0 the per-run table, the per-rank busy times and the load-balance efficiency (mean / max rank time)."""
    import torch
    from tenpy_b200 import scan
    from tenpy_b200.models import TFIChain
    from tenpy_b200.algorithms import dmrg
    chis = [int(x) for x in args.scan_chis.split(',')]
    configs = [{'chi': c, 'g': g} for c in chis for g in (0.9, 1.1)]

    def run(cfg):
        model = TFIChain({'L': args.L, 'J': 1., 'g': cfg['g'], 'conserve': None})
        psi = synthetic_mps(model, args.L, cfg['chi'], 2, seed=cfg['chi'])
        opts = {'mixer': None, 'combine': True, 'diag_method': 'lanczos', 'svd_warm_start': False,
                'trunc_params': {'chi_max': cfg['chi'], 'svd_min': 1e-45, 'trunc_cut': None, 'svd_deflation_tol': 1e-10},
                'lanczos_params': {'N_min': args.lanczos_N, 'N_max': args.lanczos_N}}
        eng = dmrg.TwoSiteDMRGEngine(psi, model, opts)
        eng.sweep()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        eng.sweep()
        ev1.record()
        torch.cuda.synchronize()
        E = float(eng.update_stats['E_total'][-1])
        del eng, psi
        torch.cuda.empty_cache()
        return [cfg['chi'], cfg['g'], ev0.elapsed_time(ev1) / 1e3, E, rank]
    table = scan.run_scan(configs, run, cost_fn=lambda c: float(c['chi'])**3)
    if rank != 0:
        return None
    per_rank = [float(np.sum(table[table[:, 5] == r, 3])) for r in range(world)]
    return {'runs': [{'chi': int(r[1]), 'g': float(r[2]), 'sweep_s': float(r[3]), 'E': float(r[4]), 'rank': int(r[5])}
                     for r in table],
            'rank_busy_s': per_rank, 'makespan_s': max(per_rank),
            'load_balance_efficiency': float(np.mean(per_rank) / max(per_rank)) if max(per_rank) > 0 else None,
            'assignment': 'runs ordered by chi^3, pulled by the ranks from a shared counter as they become free (tenpy_b200.scan.run_scan, '
                          "schedule='dynamic'; static LPT on chi^3 if the ranks share no store)", 'sweeps_per_run': '1 warm-up + 1 timed'}


def _matvec_gflops(mv_orders):
    """effective-H matvec rate of the order the sweep uses, in the reference's flop count 4 D d^3 chi^3 (BASELINE
    metric ii) -- the executed flops of the 'split' order are d times fewer, see `matvec_orders`"""
    sel = mv_orders.get(mv_orders.get('auto_selects', ''), None)
    return None if sel is None else sel['reference_equivalent_tflops'] * 1e3


def matvec_order_probe(eng, psi, L, chi, d, D, reps=5):
    """TwoSiteH.matvec at the centre bond of the benchmark state in both contraction orders (the sweep uses
    matvec_order='auto' = 'split' at this size): ms per matvec (CUDA events) and the reference-equivalent rate
    4 D d^3 chi^3 / t.  Executed flops: combined 4 D d^3 chi^3, split 4 D d^2 chi^3 + O(chi^2)."""
    import torch
    from tenpy_b200.algorithms.mps_common import TwoSiteH
    out = {}
    try:
        i0 = L // 2 - 1
        for order in ('combined', 'split'):
            H = TwoSiteH(eng.env, i0, combine=True, matvec_order=order)
            H.identity_env = False          # plain contraction orders; the sweep's route is timed by the sweep itself
            theta = H.combine_theta(psi.get_theta(i0, 2))
            for _ in range(3):
                H.matvec(theta)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                H.matvec(theta)
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / reps
            executed = 4. * D * d**3 * chi**3 if order == 'combined' else 4. * D * d**2 * chi**3
            out[order] = {'ms_per_matvec': ms, 'executed_flop': executed, 'executed_tflops': executed / ms / 1e9,
                          'reference_equivalent_tflops': 4. * D * d**3 * chi**3 / ms / 1e9,
                          # the probe's environments are contracted from the chain end through inverse Schmidt values and
                          # are not canonical, so the identity-component shortcut of the sweep is normally off here
                          'identity_env_used': bool(getattr(H, '_id_env', False))}
            del H, theta
        out['auto_selects'] = 'split' if TwoSiteH(eng.env, i0, combine=True)._use_split(
            TwoSiteH(eng.env, i0, combine=True).combine_theta(psi.get_theta(i0, 2))) else 'combined'
    except Exception as e:  # a probe must never lose the bench line
        out['error'] = repr(e)
    return out


def svd_theta_probe(eng, psi, L, reps=3):
    """block SVD (npc.svd with the sweep's deflation tolerance) of the two-site wave function at the centre bond of the
    benchmark state -- the matrix the sweep actually decomposes (numerically low rank once DMRG has converged), next
    to the generic full-rank block of `roofline_svd`."""
    import torch
    from tenpy_b200.algorithms.mps_common import TwoSiteH
    from tenpy_b200.linalg import np_conserved as npc
    try:
        i0 = L // 2 - 1
        H = TwoSiteH(eng.env, i0, combine=True)
        theta = H.combine_theta(psi.get_theta(i0, 2))
        tol = eng.trunc_params.get('svd_deflation_tol', 1.e-10)
        chi_max = eng.trunc_params.get('chi_max', None)
        U, S, VH = npc.svd(theta, inner_labels=['vR', 'vL'], deflation_tol=tol, n_keep=chi_max)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        n0 = len(npc.svd_stats['jacobi_sweeps'])
        ev0.record()
        for _ in range(reps):
            npc.svd(theta, inner_labels=['vR', 'vL'], deflation_tol=tol, n_keep=chi_max)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / reps
        m, n = theta.shape
        by = 8. * (m * n + m * min(m, n) + min(m, n) + min(m, n) * n)
        return {'shape': [int(m), int(n)], 'ms_per_svd': ms, 'GB/s_algorithmic': by / ms / 1e6,
                'jacobi_sweeps': npc.svd_stats['jacobi_sweeps'][n0:],
                'rank_above_1e-10': int(np.sum(S > 1e-10 * S.max())), 'rank_above_1e-8': int(np.sum(S > 1e-8 * S.max()))}
    except Exception as e:  # a probe must never lose the bench line
        return {'error': repr(e)}


def blocksparse_probes(small=False):
    """effective-H matvec (LHeff . theta . RHeff) on synthetic random-charge Arrays of the BASELINE.json configs[2] / [3]
    shapes (SURVEY.md section 8d; generator modelled on the reference's tests/benchmark/tensordot_npc.py:36-51):
    U(1) chi=1024 d=2 D=5 (XXZ-like) and U(1)xU(1) chi=2048 d=4 D=6 (Hubbard-like).  Reports GEMMs per matvec, executed
    flops (sum 2 m k n over the block products) and ms per matvec (CUDA events).  These shapes are launch / latency bound
    (two grouped launches per matvec), not flop bound."""
    import torch
    from tenpy_b200.linalg import np_conserved as npc
    from tenpy_b200.linalg.charges import ChargeInfo, LegCharge
    out = []
    cases = [('xxz_like', 1024, 12), ('hubbard_like', 2048, 40)] if not small else [('xxz_like', 32, 4), ('hubbard_like', 32, 6)]
    for kind, chi, nsec in cases:
        try:
            rng = np.random.default_rng(0)
            if kind == 'xxz_like':
                ci = ChargeInfo([1], ['2*Sz'])
                p = LegCharge.from_qflat(ci, [[-1], [1]], +1)
                wq, spread = np.array([[0], [2], [-2], [0], [0]]), 16
            else:
                ci = ChargeInfo([1, 1], ['N', '2*Sz'])
                p = LegCharge.from_qflat(ci, [[0, 0], [1, -1], [1, 1], [2, 0]], +1)
                wq, spread = np.array([[0, 0], [1, 1], [-1, -1], [1, -1], [-1, 1], [0, 0]]), 8

            def sector_leg(qconj):
                cuts = np.sort(rng.choice(np.arange(1, chi), size=nsec - 1, replace=False))
                charges = set()
                while len(charges) < nsec:
                    charges.add(tuple(int(x) for x in rng.integers(-spread, spread + 1, size=ci.qnumber)))
                charges = np.array(sorted(charges))
                charges = charges[np.lexsort(charges.T)]
                return LegCharge.from_qind(ci, np.concatenate(([0], cuts, [chi])), charges, qconj)
            D = len(wq)
            vL, vR = sector_leg(+1), sector_leg(-1)
            w = LegCharge.from_qind(ci, np.arange(D + 1), wq, -1)
            gen = rng.standard_normal
            L4 = npc.Array.from_func(gen, [vL, p, w, vL.conj(), p.conj()], labels=['vR*', 'p0', 'wR', 'vR', 'p0*'])
            LHeff = L4.combine_legs([['vR*', 'p0'], ['vR', 'p0*']], qconj=[+1, -1], new_axes=[0, 2])
            R4 = npc.Array.from_func(gen, [w.conj(), p.conj(), vR.conj(), p, vR], labels=['wL', 'p1*', 'vL', 'p1', 'vL*'])
            RHeff = R4.combine_legs([['p1', 'vL*'], ['p1*', 'vL']], qconj=[-1, +1], new_axes=[2, 1])
            del L4, R4
            theta = npc.Array.from_func(gen, [LHeff.get_leg('(vR.p0*)').conj(), RHeff.get_leg('(p1*.vL)').conj()],
                                        labels=['(vL.p0)', '(p1.vR)'])

            def mv(th):
                t = npc.tensordot(LHeff, th, axes=['(vR.p0*)', '(vL.p0)'])
                return npc.tensordot(t, RHeff, axes=[['wR', '(p1.vR)'], ['wL', '(p1*.vL)']])
            n_plans0 = set(npc._PLAN_CACHE.keys())
            for _ in range(3):
                mv(theta)
            new = [v for k, v in npc._PLAN_CACHE.items() if k not in n_plans0]
            flops = float(sum(v[2].flops for v in new))
            ngemm = int(sum(v[2].n_pairs for v in new))
            reps = 20
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                mv(theta)
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / reps
            out.append({'case': kind, 'chi': chi, 'd': int(p.ind_len), 'D': D, 'n_sectors': nsec,
                        'blocks': {'LHeff': LHeff.stored_blocks, 'theta': theta.stored_blocks, 'RHeff': RHeff.stored_blocks},
                        'gemms_per_matvec': ngemm, 'flop_per_matvec': flops,
                        'dense_equivalent_flop': 4. * D * p.ind_len**3 * float(chi)**3, 'ms_per_matvec': ms,
                        'gflops': flops / ms / 1e6 if ms > 0 else None})
            del LHeff, RHeff, theta
        except Exception as e:  # a probe must never lose the bench line
            out.append({'case': kind, 'error': repr(e)})
    return out


def kernel_probes(lib, chi, d, D):
    """time the two dominant kernels alone on centre-bond shapes (after warm-up, CUDA events)"""
    import torch
    from tenpy_b200 import backend
    from tenpy_b200.linalg import np_conserved as npc
    peaks, kind = measured_peaks()
    n = chi * d
    dev = lib.device

    def rnd(legs):
        t = torch.randn(int(np.prod([l.ind_len for l in legs])), dtype=torch.float64, device=dev)
        return npc.Array.from_device_buffer(legs, np.zeros((1, len(legs)), np.int64), t)
    ci = npc.ChargeInfo()
    lL, lR, lW = (npc.LegCharge.from_trivial(n, ci, +1), npc.LegCharge.from_trivial(n, ci, -1),
                  npc.LegCharge.from_trivial(D, ci, -1))
    vL, vR, lp = (npc.LegCharge.from_trivial(chi, ci, +1), npc.LegCharge.from_trivial(chi, ci, -1),
                  npc.LegCharge.from_trivial(d, ci, +1))
    theta = rnd([lL, lR])
    # the two large products of the matvec as the sweep runs them (identity-environment route): the D - 1 non-identity
    # components of LP onto theta and the W0 W1 . theta intermediate onto those of RP, on the int8 tensor path with 7 digit
    # planes (csrc/ozaki.cu); the digit planes of LP / RP are cached per bond, those of theta / the intermediate are
    # produced by the split kernels once per matvec (timed separately: `split_ms_per_operand`)
    from tenpy_b200.linalg.np_conserved import OZAKI
    s7 = int(OZAKI['slices_matvec'])
    Dr = max(D - 1, 1)
    shapes = [(chi * Dr, d * d * chi, chi), (chi * d * d, chi, chi * Dr)]      # (m, n, k)
    ops, ms_mm, ms_split = [], [], []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    for (m_, n_, k_) in shapes:
        A = torch.randn(m_ * k_, dtype=torch.float64, device=dev)
        B = torch.randn(k_ * n_, dtype=torch.float64, device=dev)
        C = torch.empty(m_ * n_, dtype=torch.float64, device=dev)
        a_s = lib.ozaki_split(m_, k_, A, k_, 1, s7)
        b_s = lib.ozaki_split(n_, k_, B, 1, n_, s7)
        for _ in range(3):
            lib.ozaki_mm(m_, n_, k_, s7, a_s, b_s, C, n_)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            lib.ozaki_mm(m_, n_, k_, s7, a_s, b_s, C, n_)
        ev1.record()
        torch.cuda.synchronize()
        ms_mm.append(ev0.elapsed_time(ev1) / reps)
        ev0.record()
        for _ in range(reps):
            lib.ozaki_split(n_, k_, B, 1, n_, s7)
        ev1.record()
        torch.cuda.synchronize()
        ms_split.append(ev0.elapsed_time(ev1) / reps)
        ops.append((A, B, C))
    lib.ozaki_check_abort()
    # parity of the timed kernel at the timed size (size-independent property: linearity in a random probe vector,
    # (A B) x = A (B x) evaluated in FP64 on the device)
    m_, n_, k_ = shapes[-1]
    A, B, C = ops[-1]
    x = torch.randn(n_, dtype=torch.float64, device=dev)
    lhs = C.view(m_, n_) @ x
    rhs = A.view(m_, k_) @ (B.view(k_, n_) @ x)
    scale = A.view(m_, k_).abs() @ (B.view(k_, n_).abs() @ x.abs())
    oz_err = float(((lhs - rhs).abs() / scale).max())
    del ops
    ms = float(np.mean(ms_mm))
    flops = 2. * Dr * d**2 * chi**3                  # per launch (FP64-equivalent)
    n_prod = s7 * (s7 + 1) // 2                      # exact int8 slice products per FP64 product
    tf = flops / (ms * 1e-3) / 1e12
    traffic, pipe_pct, ncu_src = gemm_ncu_numbers() if (chi, d, D) == (1024, 2, 3) else (None, None, None)
    int8_peak = 2. * peaks.get('bf16_tflops', 0.)    # tcgen05 kind::i8 runs at twice the bf16 rate
    peak_equiv = int8_peak / n_prod
    gemm = {'bound': 'tensor', 'achieved': tf, 'peak': peak_equiv, 'unit': 'TFLOP/s', 'frac': tf / peak_equiv if peak_equiv else None,
            'traffic': traffic, 'ms_per_launch': ms, 'ms_per_launch_by_shape': {'%dx%dx%d' % sh: t for sh, t in zip(shapes, ms_mm)},
            'int8_tops_achieved': tf * n_prod, 'int8_tops_peak': int8_peak, 'frac_of_nominal_int8_4500': tf * n_prod / 4500., 'digit_planes': s7, 'int8_products_per_fp64_product': n_prod,
            'split_ms_per_operand': float(np.mean(ms_split)),
            'fp64_dmma_peak_tflops': FP64_TENSOR_PEAK_TFLOPS, 'frac_of_fp64_dmma_peak': tf / FP64_TENSOR_PEAK_TFLOPS,
            'algorithmic_bytes_per_launch': float(s7 * (shapes[0][0] * shapes[0][2] + shapes[0][1] * shapes[0][2]) + 8 * shapes[0][0] * shapes[0][1]),
            'tensor_pipe_active_pct_ncu': pipe_pct, 'ncu_source': ncu_src, 'rel_err_vs_fp64_probe': oz_err,
            'peak_note': 'achieved = FP64-equivalent flops (2 m n k) per launch / CUDA-event time of oz_gemm_kernel alone, operands pre-split '
                         'as in the sweep; peak = int8 tensor peak / %d slice products, int8 peak = 2 x bf16_tflops of MEASURED_PEAKS.json '
                         '(%.0f TFLOP/s %s, burst) = %.0f Top/s (nominal 4500; MMA-only ceiling of this tile shape measured by '
                         'profiles/tc_i8_probe.cu: 4000-4540); the FP64 tensor (DMMA) pipe the round-1 kernel ran on peaks at %.0f TFLOP/s'
                         % (n_prod, peaks.get('bf16_tflops', 0.), kind, int8_peak, FP64_TENSOR_PEAK_TFLOPS),
            'algorithmic': '2 (D-1) d^2 chi^3 = %.3e FP64-equivalent flop per launch = %.3e int8 op: (chi (D-1) x chi).(chi x d^2 chi) and '
                           '(chi d^2 x chi (D-1)).(chi (D-1) x chi), the two large products of one matvec' % (flops, flops * n_prod)}
    # SVD of the centre theta: bytes = 8 (mn + mk + k + kn)
    from tenpy_b200.linalg.np_conserved import svd
    svd(theta)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(2):
        svd(theta)
    ev1.record()
    torch.cuda.synchronize()
    ms_svd = ev0.elapsed_time(ev1) / 2
    by = 8. * (n * n + n * n + n + n * n)
    gbs = by / (ms_svd * 1e-3) / 1e9
    svdr = {'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'],
            'traffic': None, 'ms_per_svd': ms_svd,
            'algorithmic': '8 (mn + mk + k + kn) = %.3e bytes per %dx%d block (read A once, write U, S, VH once); '
                           'the Jacobi iteration itself is compute/latency bound for a block this large' % (by, n, n),
            'peak_note': 'hbm_gbs %s' % kind}
    return {'gemm': gemm, 'svd': svdr}


def run_b200_reference_driver(args):
    """The benchmark sweep driven by the UNMODIFIED reference: ``tenpy.algorithms.dmrg.TwoSiteDMRGEngine.sweep`` (its
    `Sweep` loop, `update_local`, `mixed_svd` -> `svd_theta` / `truncate`, `LanczosGroundState`, `MPOEnvironment`, `MPS`,
    `TFIChain`) on the device engine through `tenpy_b200.dropin`; the effective Hamiltonian is the engine's device-optimised
    `TwoSiteH` plugged in at the reference's `EffectiveH` hook.  Same synthetic state and options as the default arm."""
    import torch
    from tenpy_b200 import backend, dropin
    from tenpy_b200._lib import DeviceLib
    torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
    lib = backend.use_library(DeviceLib())
    path = dropin.install()
    if path is None:
        print(json.dumps({'driver': 'reference', 'unavailable': 'no reference install (oracle/_ref)'}))
        return
    import tenpy
    from tenpy.models.tf_ising import TFIChain
    from tenpy.networks.mps import MPS
    import tenpy.linalg.np_conserved as npc
    L, chi, d = args.L, args.chi, 2
    M = TFIChain({'L': L, 'J': 1., 'g': 1., 'bc_MPS': 'finite', 'conserve': None})
    sites = M.lat.mps_sites()

    class _Shim:                      # synthetic_mps only needs the site legs
        lat_sites = sites
    own = synthetic_mps(_Shim, L, chi, d, seed=0)
    psi = MPS(sites, [B for B in own._B], [np.asarray(s_) for s_ in own._S], bc='finite', form='B')
    opts = {'mixer': None, 'combine': True, 'diag_method': 'lanczos',
            'trunc_params': {'chi_max': chi, 'svd_min': 1e-45, 'trunc_cut': None, 'svd_deflation_tol': 1e-10},
            'lanczos_params': {'N_min': args.lanczos_N, 'N_max': args.lanczos_N}}
    opts['trunc_params'].pop('svd_deflation_tol')        # not an option of the reference's svd_theta ...
    npc.SVD_DEFAULTS['deflation_tol'] = 1e-10             # ... the engine's npc.svd takes it as its default instead
    Engine = dropin.fast_two_site_engine()
    eng = Engine(psi, M, opts)
    for _ in range(args.warmup):
        eng.sweep()
    torch.cuda.synchronize()
    lib.kernel_launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        eng.sweep()
    ev1.record()
    torch.cuda.synchronize()
    E = float(eng.update_stats['E_total'][-1])
    E_exact = exact_tfi_energy(L, 1., 1.)
    print(json.dumps({'driver': 'reference', 'impl': 'b200', 'metric': METRIC, 'unit': UNIT,
                      'value': ev0.elapsed_time(ev1) / 1e3 / args.steps, 'steps': args.steps, 'warmup': args.warmup,
                      'gpu_launches': int(lib.kernel_launch_count()), 'E': E, 'E_rel_err': abs(E - E_exact) / abs(E_exact),
                      'engine_module': npc.__name__, 'dmrg_file': tenpy.algorithms.dmrg.__file__,
                      'int8_products': npc.OZAKI['calls']}))


def reference_driver_line(args):
    """run `--driver reference` in its own process (the engine has to be seeded before `import tenpy`) and return its line"""
    cmd = [sys.executable, os.path.abspath(__file__), '--driver', 'reference', '--steps', '1', '--warmup', '2', '--L', str(args.L),
           '--chi', str(args.chi), '--lanczos-N', str(args.lanczos_N)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, WORLD_SIZE='1', RANK='0'))
        lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
        return json.loads(lines[-1]) if lines else {'error': out.stderr[-500:]}
    except Exception as e:
        return {'error': repr(e)}


def run_blocksparse(args):
    """BASELINE.json configs[2] / [3] end to end on one GPU: two-site DMRG with charge conservation from a product state,
    bond dimension ramped up (mixer on), then `--steps` timed sweeps at the final chi (mixer off, the reference's default
    adaptive Lanczos).  One JSON line: seconds per sweep, kernel-family times, the contraction-size histogram (where the
    GEMM time goes), sector / block structure, E, S.  Parity of this path: tests/test_large_parity.py (same models at
    L=64 / L=32, chi=256 against the unmodified reference)."""
    import torch
    from tenpy_b200 import backend
    from tenpy_b200._lib import DeviceLib
    from tenpy_b200.models import SpinChain, FermiHubbardChain
    from tenpy_b200.networks.mps import MPS
    from tenpy_b200.algorithms import dmrg
    from tenpy_b200.algorithms.mps_common import TwoSiteH
    from tenpy_b200.linalg import np_conserved as npc
    torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
    lib = backend.use_library(DeviceLib())
    if args.svd_inner_sweeps:
        lib.svd_set_eig_inner_sweeps(args.svd_inner_sweeps)
    xxz = args.workload == 'xxz'
    L = args.L if args.L != 100 or xxz else 64
    chi = args.chi if args.chi != 1024 or xxz else 2048
    M = SpinChain({'L': L, 'Jx': 1., 'Jy': 1., 'Jz': 1., 'conserve': 'Sz'}) if xxz else \
        FermiHubbardChain({'L': L, 't': 1., 'U': 4., 'mu': 0.})
    psi = MPS.from_product_state(M.lat_sites, ['up', 'down'] * (L // 2))
    chis = [min(chi, 32 * 2**k) for k in range(args.ramp)]
    chis[-1] = chi
    opts = {'mixer': True, 'mixer_params': {'amplitude': 1e-4, 'decay': 2., 'disable_after': args.ramp},
            'combine': True, 'trunc_params': {'chi_max': chis[0], 'svd_min': args.svd_min}}
    if args.svd_warm_start != 'default':
        opts['svd_warm_start'] = False if args.svd_warm_start == 'off' else args.svd_warm_start
    eng = dmrg.TwoSiteDMRGEngine(psi, M, opts)
    t_ramp = []
    for c in chis:
        eng.trunc_params['chi_max'] = c
        t0 = time.perf_counter()
        eng.sweep()
        lib.synchronize()
        t_ramp.append(round(time.perf_counter() - t0, 3))
    eng.mixer_deactivate()
    for _ in range(args.warmup):
        eng.sweep()
    sampler = ClockSampler(0)
    sampler.start()
    torch.cuda.synchronize()
    lib.kernel_launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        eng.sweep()
    ev1.record()
    torch.cuda.synchronize()
    launches = lib.kernel_launch_count()
    sweep_s = ev0.elapsed_time(ev1) / 1e3 / args.steps
    clocks = sampler.summary()
    # one more sweep with per-call profiling
    lib.profile = {}
    plans0 = len(npc._PLAN_CACHE)
    t0 = time.perf_counter()
    eng.sweep()
    lib.synchronize()
    wall = time.perf_counter() - t0
    fam = {k: round(v[1], 1) for k, v in lib.profile_summary().items()}
    det = lib.profile_detail()
    lib.profile = None
    g = [(ms, info) for ms, info in det.get('gemm', []) if info]
    hist = []
    for lo, hi in ((0, 1e6), (1e6, 1e7), (1e7, 1e8), (1e8, 1e9), (1e9, 1e10), (1e10, 1e13)):
        sel = [(ms, i) for ms, i in g if lo <= i[0] < hi]
        if sel:
            tms, tfl = sum(x[0] for x in sel), sum(x[1][0] for x in sel)
            hist.append({'flop_range': [lo, hi], 'calls': len(sel), 'ms': round(tms, 2), 'gflop': round(tfl / 1e9, 2),
                         'tflops': round(tfl / tms / 1e9, 3) if tms else None})
    i0 = L // 2 - 1
    H = TwoSiteH(eng.env, i0, combine=True)
    theta = H.combine_theta(psi.get_theta(i0, 2))
    nb = 2 * (L - 2)
    peaks, peaks_kind = measured_peaks()
    total_flop = float(sum(i[0] for _, i in g))
    line = {'metric': METRIC, 'value': sweep_s, 'unit': UNIT, 'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': sweep_s * 1e3, 'higher_is_better': False, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
            'data': 'product state -> DMRG (no synthetic tensors)', 'impl': 'b200',
            'config': {'workload': ('SpinChain XXZ L=%d chi=%d, U(1) Sz' if xxz else 'FermiHubbardChain L=%d chi=%d, U(1)xU(1) (N, Sz)')
                       % (L, chi) + ', two-site DMRG sweep after a chi ramp %r with the density-matrix mixer; timed sweeps: mixer '
                       'off, adaptive Lanczos (reference defaults), svd_min=%g, svd_warm_start=%s' % (chis, args.svd_min, args.svd_warm_start),
                       'L': L, 'chi': chi, 'svd_inner_sweeps': args.svd_inner_sweeps or 'library default',
                       'l2': 'working set (environments + MPS) >> 126 MB L2'},
            'clocks': clocks, 'gpu_launches': int(launches), 'ramp_sweep_s': t_ramp, 'chi_reached': int(max(psi.chi)),
            'result': {'E': float(eng.update_stats['E_total'][-1]), 'S_mid': float(psi.entanglement_entropy()[L // 2 - 1]),
                       'N_lanczos_mean': float(np.mean(eng.update_stats['N_lanczos'][-nb:])),
                       'trunc_err_max': float(max(getattr(e, 'eps', e) for e in eng.update_stats['err'][-nb:])),
                       'svd_jacobi_sweeps_mean': float(np.mean(npc.svd_stats['jacobi_sweeps'][-nb:])),
                       'svd_guess_used': npc.svd_stats.get('guess_used', 0)},
            'structure': {'theta_blocks': int(theta.stored_blocks), 'theta_shape': list(theta.shape),
                          'theta_largest_block': [int(x) for x in theta._layout.shapes[np.argmax(theta._layout.sizes)]],
                          'bond_sectors': int(psi.get_B(L // 2).get_leg('vL').block_number)},
            'kernel_family_ms_per_sweep': fam, 'host_wall_s_profiled_sweep': wall,
            'gemm_by_flops': hist, 'plans_built_profiled_sweep': len(npc._PLAN_CACHE) - plans0,
            'contraction_flop_per_sweep': total_flop,
            'roofline': {'bound': 'tensor', 'achieved': total_flop / max(fam.get('gemm', 0.), 1e-9) / 1e9, 'peak': FP64_TENSOR_PEAK_TFLOPS,
                         'unit': 'TFLOP/s', 'frac': total_flop / max(fam.get('gemm', 0.), 1e-9) / 1e9 / FP64_TENSOR_PEAK_TFLOPS,
                         'traffic': None, 'kernel': 'grouped_gemm_kernel / thin_n / thin_m / oz_gemm_kernel (all contractions of a sweep)',
                         'note': 'ragged charge blocks: launch / latency bound, see gemm_by_flops'},
            'peaks': peaks_kind}
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.workload != 'tfi' and args.impl != 'reference':
        return run_blocksparse(args)
    if args.impl == 'reference':
        run_reference(args)
    elif args.driver == 'reference':
        run_b200_reference_driver(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
