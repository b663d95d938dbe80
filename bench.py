#!/usr/bin/env python
"""bench.py - AO-ADMM outer iterations/s on B200 (metric of BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            our engine (CUDA, C ABI of include/aoadmm.h)
  python bench.py --impl reference --gpus N --steps K ...  the reference's algorithm on the host cores
                                                           (NumPy/OpenBLAS oracle port: MATLAB cannot run offline)
  --dump-outputs DIR   after the timed steps, write what the timed run returned as DIR/<name>.npy (float64), so that
                       two builds can be compared output for output (the inputs are the same from run to run)

A "step" is one outer AO-ADMM iteration (one sweep over all modes: 3 tensor MTTKRPs + 2 matrix products + every
inner ADMM loop with all tolerances 0, i.e. MaxInnerIters=5 inner iterations per mode group) of the workload below.

Workload (same for every N so that the 1->8 curve is a strong-scaling curve): the C3 family of SURVEY.md 8d,
a 4096 x 4096 x K3 nonneg CP tensor (R=64) coupled in mode 1 with a 4096 x 8192 matrix, K3 = 1024 so that the
FP64 tensor (137.4 GB) fits ONE B200; the tensor is generated on device (it cannot exist in host memory at that
size) and sharded along mode 3 across the N ranks.  BENCH_WORKLOAD=c2 selects configs[1] (1000^3, R=32, 1000x5000).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if '--impl' in sys.argv and 'reference' in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 for nproc > 1, which would halve the CPU arm against its own N=1 run:
    # the reference arm always gets every host core (set before NumPy / OpenBLAS load)
    try:
        _cores = len(os.sched_getaffinity(0))
    except Exception:
        _cores = os.cpu_count() or 1
    for _k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_k] = str(_cores)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, 'matlab-code_b200'))

WORKLOADS = {
    # name: (I, J, K, M, R, cpu_sample_dims)
    'c3k1024': dict(I=4096, J=4096, K=1024, M=8192, R=64, sample=dict(I=1024, J=1024, K=256, M=2048)),
    # BASELINE configs[2] at its own size: 274.9 GB in FP64, needs >= 2 GPUs (137.4 GB per GPU at N=2)
    'c3': dict(I=4096, J=4096, K=2048, M=8192, R=64, sample=dict(I=1024, J=1024, K=512, M=2048), min_gpus=2),
    'c2': dict(I=1000, J=1000, K=1000, M=5000, R=32, sample=dict(I=1000, J=1000, K=1000, M=5000)),
    'tiny': dict(I=64, J=48, K=40, M=80, R=8, sample=dict(I=64, J=48, K=40, M=80)),
}
FP64_DMMA_PEAK_TFLOPS = 37.1   # measured on this pool: profiles/r01_fp64_probe.log (DMMA.8x8x4 issue-rate probe)
FP64_NOMINAL_TFLOPS = 40.0     # NVIDIA's B200 FP64 / FP64-tensor figure (HGX B200 sheet: 296 per 8 GPUs = 37; DGX B200: 40)


# `value` is measured on the reference's own work per step: three independent MTTKRP passes (options.dimtree = 0).
# The dimension-tree sweep (2 tensor passes per step, results equal to rounding) is reported beside it as `dimtree`.
DIMTREE = int(os.environ.get('BENCH_DIMTREE', '0'))


# --dump-outputs: what a caller of the timed run receives, the state G (cmtf_fun_AOADMM.m:1) and the per-iteration arrays
# of `out`.  Left out: time_at_it (wall-clock stamps) and func_rel_missing (all NaN without a missing-data mask).
DUMP_STATE_KEYS = ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_fac', 'coupling_dual_fac')
DUMP_OUT_KEYS = ('func_val_conv', 'func_coupl_conv', 'func_constr_conv', 'func_PAR2_coupl', 'innerIters')
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, G, out):
    """G[key][m] -> <path>/<key>_<m>.npy, out[key] -> <path>/<key>.npy, all float64."""
    arrays = {}
    for key in DUMP_STATE_KEYS:
        for m, a in enumerate(G.get(key) or []):
            if a is not None:
                arrays['%s_%d' % (key, m)] = np.asarray(a, dtype=np.float64)
    for key in DUMP_OUT_KEYS:
        arrays[key] = np.asarray(out[key], dtype=np.float64)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, 'outputs of %d bytes exceed the %d-byte dump limit' % (total, DUMP_MAX_BYTES)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def zero_tol_options(iters):
    return dict(MaxOuterIters=iters, MaxInnerIters=5, AbsFuncTol=0.0, OuterRelTol=0.0, innerRelPrTol_coupl=0.0,
                innerRelPrTol_constr=0.0, innerRelDualTol_coupl=0.0, innerRelDualTol_constr=0.0, bsum=0, dimtree=DIMTREE)


def make_problem(I, J, K, M, R, seed=0, with_tensor=False):
    """C2/C3 construction of SURVEY.md 8d: X = [[A,B,C]] + noise (level 0.2), Y = A V' + noise, all nonneg, w=[1/2 1/2].
    Factors are host-side (small); the tensor itself is only built on the host when with_tensor=True."""
    rng = np.random.RandomState(seed)
    rng32 = np.random.default_rng(seed + 1)
    A, B, C, V = rng.rand(I, R), rng.rand(J, R), rng.rand(K, R), rng.rand(M, R)
    Y = A @ V.T
    N = rng.standard_normal((I, M))
    Y = Y + 0.2 * np.linalg.norm(Y) / np.linalg.norm(N) * N
    Y = np.asfortranarray(Y / np.linalg.norm(Y))
    X = None
    if with_tensor:
        X = np.empty((I, J, K), order='F')
        nrm2_x = 0.0
        nrm2_n = 0.0
        noise = np.empty((I, J, K), order='F', dtype=np.float32)
        for k in range(K):   # slab-wise to bound temporaries
            slab = (A * C[k, :]) @ B.T
            X[:, :, k] = slab
            nrm2_x += float(np.sum(slab * slab))
            nz = rng32.standard_normal((I, J), dtype=np.float32)
            noise[:, :, k] = nz
            nrm2_n += float(np.sum(nz.astype(np.float64) ** 2))
        sigma = 0.2 * np.sqrt(nrm2_x) / np.sqrt(nrm2_n)
        for k in range(K):
            X[:, :, k] += sigma * noise[:, :, k]
        del noise
        X /= np.sqrt(float(np.sum(X * X)))
    nn = ('non-negativity',)
    sz = [I, J, K, I, M]
    Z = {'loss_function': ['Frobenius'] * 2, 'model': ['CP', 'CP'], 'modes': [[1, 2, 3], [4, 5]], 'size': sz,
         'coupling': {'lin_coupled_modes': [1, 0, 0, 1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 5},
         'constrained_modes': [1] * 5, 'constraints': [nn] * 5, 'weights': [0.5, 0.5], 'object': [X, Y], 'rank': [R, R]}

    def normc(F):
        return F / np.linalg.norm(F, axis=0)
    G = {'fac': [normc(rng.rand(s, R)) for s in sz], 'constraint_fac': [rng.rand(s, R) for s in sz],
         'constraint_dual_fac': [rng.rand(s, R) for s in sz],
         'coupling_dual_fac': [rng.rand(I, R), None, None, rng.rand(I, R), None], 'coupling_fac': [rng.rand(I, R)],
         'P': [None, None], 'DeltaB': [None, None], 'mu_DeltaB': [None, None]}
    return Z, G, (A, B, C)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (profiling recipe)."""

    def __init__(self, device):
        self.rows = []
        self.proc = None
        self.device = device

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.device), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            p = [x.strip() for x in r.split(',')]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx = float(p[1])
            except ValueError:
                continue
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], p[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        busy = [x for x in sm if mx and x > 0.5 * mx] or sm
        return {'sm_mhz': float(np.median(busy)) if busy else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


def cpu_baseline_run(wl, steps, warmup, keep=False):
    """The oracle (NumPy restatement of cmtf_fun_AOADMM.m, Tensor-Toolbox-style MTTKRP = unfold + Khatri-Rao + DGEMM)
    on the host cores, on a bounded sample of the workload; flop-proportional extrapolation to the full size.
    keep=True also returns the sample problem and the oracle's result (for the parity check of the bench itself)."""
    sys.path.insert(0, ROOT)
    from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
    sm = wl['sample']
    Z, G, _ = make_problem(sm['I'], sm['J'], sm['K'], sm['M'], wl['R'], seed=0, with_tensor=True)
    zn = [float(np.sum(Z['object'][0] ** 2)), float(np.sum(Z['object'][1] ** 2))]
    if warmup > 0:
        oracle_solve(Z, zn, G, options=zero_tol_options(warmup))
    t = time.perf_counter()
    Go, out = oracle_solve(Z, zn, G, options=zero_tol_options(steps))
    dt = time.perf_counter() - t
    per_iter = (out['time_at_it'][-1] - out['time_at_it'][0]) / steps   # excludes the iteration-0 objective
    scale = (wl['I'] * wl['J'] * wl['K']) / float(sm['I'] * sm['J'] * sm['K'])
    full = (scale == 1.0)
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count()
    sample = '%d outer iterations of %dx%dx%d R=%d + %dx%d matrix (%s)' % (
        steps, sm['I'], sm['J'], sm['K'], wl['R'], sm['I'], sm['M'],
        'full workload' if full else 'tensor sample, it/s scaled by 1/%g ~ flops' % scale)
    cb = {'value': 1.0 / (per_iter * scale), 'unit': 'outer_iters/s', 'cores': cores, 'kind': 'port',
          'sample': sample, 'sample_s_per_iter': per_iter, 'wall_s': dt,
          'blas_threads': os.environ.get('OMP_NUM_THREADS', 'default (all cores)')}
    if keep:
        return cb, (Z, G, zn, Go, out)
    return cb


def workload_config(name, wl, world, launch):
    I, J, K, M, R = wl['I'], wl['J'], wl['K'], wl['M'], wl['R']
    fits = 'K=%d so the FP64 tensor fits one GPU' % K if name == 'c3k1024' else \
        ('BASELINE configs[2] at its own size, 274.9 GB: needs >= 2 GPUs' if name == 'c3' else 'BASELINE configs[1]')
    return {'workload': 'CP %dx%dx%d R=%d nonneg + coupled %dx%d matrix (SURVEY 8d C3 family, %s), MaxInnerIters=5, '
                        'all tolerances 0' % (I, J, K, R, I, M, fits),
            'name': name, 'sharding': 'mode-3 slabs over %d GPU(s)' % world, 'launch': launch,
            'l2_policy': 'inputs (%.1f GB tensor) far larger than the 126 MB L2' % (8.0 * I * J * K / 1e9),
            'tensor_passes_per_step': 2 if DIMTREE else 3,
            'dimtree': ('on: the mode-2 MTTKRP also emits T = X x_1 A (J x K x R), mode 3 is a pass over T; 2 tensor passes '
                        'and 2/3 of the reference flops per step, results equal to rounding' if DIMTREE else
                        'off: three independent MTTKRP passes (the reference flop/byte count)')}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=os.environ.get('BENCH_WORKLOAD', 'c3k1024'))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-c3-full', action='store_true', help='skip the extra 4096x4096x2048 run of the N >= 2 lines')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    # `--gpus N` without a launcher: ONE process drives the N GPUs through aoadmm_create_multi (the form a MATLAB
    # session uses); under torchrun (the driver's launch for N > 1) it is one process per GPU
    single_process = (world == 1 and args.gpus > 1)
    n_gpus = args.gpus if single_process else world
    launch = ('one process, %d worker threads (aoadmm_create_multi)' % n_gpus) if single_process else \
        ('one process per GPU (aoadmm_create + aoadmm_dist)' if world > 1 else 'one process, one GPU')
    if wl.get('min_gpus', 1) > n_gpus:
        raise SystemExit('bench.py: workload %s (%.1f GB) needs at least %d GPUs' %
                         (args.workload, 8.0 * wl['I'] * wl['J'] * wl['K'] / 1e9, wl['min_gpus']))
    config = workload_config(args.workload, wl, n_gpus, launch)

    if args.impl == 'reference':
        if rank != 0:
            return 0
        # exactly `steps` timed steps after `warmup` untimed ones; a step of this arm is one outer iteration on the bounded
        # sample of the workload (cpu_baseline.sample), so ms_per_step is the measured time of such a step and `value`
        # is the whole-workload rate it extrapolates to (flop-proportional, factor in `sample_scale`)
        steps = args.steps
        cb, (_, _, _, Go, oo) = cpu_baseline_run(wl, steps, args.warmup, keep=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, Go, oo)
        sm = wl['sample']
        scale = (wl['I'] * wl['J'] * wl['K']) / float(sm['I'] * sm['J'] * sm['K'])
        line = {'impl': 'reference', 'metric': 'ao_admm_outer_iters_per_s', 'value': cb['value'], 'unit': 'outer_iters/s',
                'n_gpus': args.gpus, 'steps': steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * cb['sample_s_per_iter'],
                'sample_scale': scale, 'full_workload_ms_per_step': 1e3 / cb['value'],
                'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': config, 'cpu_baseline': cb,
                'e2e': {'value': cb['value'], 'unit': 'outer_iters/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'note': 'MATLAB/Octave + Tensor Toolbox are not available offline: this is the NumPy/OpenBLAS port of '
                        'cmtf_fun_AOADMM.m (oracle/), timed on the host cores with every core (OMP_NUM_THREADS is set '
                        'explicitly so that a torchrun launch does not pin BLAS to one thread)'}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    import aoadmm_b200 as ab

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the engine has no CPU fallback)')
    torch.cuda.set_device(local_rank)
    uid = None
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        # ONE unique id for the whole process: the engine caches the communicator per id, so every handle of this run
        # (device-resident leg, end-to-end leg, C3-full leg) shares one NCCL bootstrap
        t = torch.zeros(128, dtype=torch.uint8, device='cuda')
        if rank == 0:
            t.copy_(torch.tensor(list(ab.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(t, 0)
        uid = bytes(t.cpu().tolist())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def make_solver(Zx, zn, K):
        if single_process:
            return ab.Solver(Zx, zn, n_gpus=n_gpus), (0, K)
        lo, hi = ab.shard_range(K, rank, world)
        return ab.Solver(Zx, zn, rank=rank, world_size=world, device=local_rank, unique_id=uid, shard=[(lo, hi), None]), (lo, hi)

    warm_out = [None]   # `out` of the most recent warm-up run (the trajectory from G)

    def timed_run(solver, G, opts_fn, steps, whole_ms=None):
        """W warm-up steps, then exactly `steps` outer iterations timed with CUDA events on the engine's stream(s)."""
        solver.set_state(G)
        warm_out[0] = solver.run(opts_fn(max(args.warmup, 3)))
        barrier()
        l0 = solver.launch_count()
        ph0 = solver.phase_ms().copy()
        barrier()
        t0 = time.perf_counter()
        out = solver.run(opts_fn(steps))
        ms = solver.last_loop_ms()
        if whole_ms is not None:
            whole_ms[0] = solver.last_run_ms()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        assert out['OuterIterations'] == steps and np.isfinite(out['f_tensors'])
        return max_over_ranks(ms), wall, solver.launch_count() - l0, solver.phase_ms() - ph0, out

    I, J, K, M, R = wl['I'], wl['J'], wl['K'], wl['M'], wl['R']
    Z, G, facs = make_problem(I, J, K, M, R, seed=0, with_tensor=False)
    zn = [1.0, float(np.sum(Z['object'][1] ** 2))]
    solver, (lo, hi) = make_solver(Z, zn, K)
    Kloc = (hi - lo) if not single_process else K // n_gpus   # per-GPU slab (roofline is per kernel launch = per GPU)
    solver.generate_cp_data(1, facs, 0.2, 20261018)
    solver.set_state(G)

    # ---- device-resident throughput (`value`) ----
    whole_ms = [0.0]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dev_ms, wall_ms, launches, ph, out = timed_run(solver, G, zero_tol_options, args.steps, whole_ms)
    traj = np.array(warm_out[0]['func_val_conv'])   # objective of the first W iterations from G (device-resident data)
    call_ms = whole_ms[0]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        G_out = solver.get_state()   # collective: every rank takes part, rank 0 writes
        if rank == 0:
            dump_outputs(args.dump_outputs, G_out, out)
        del G_out
    if world == 1 and (clocks is None or not clocks.get('samples')):
        # the timed region was shorter than the nvidia-smi sampling period: sample the clocks over a repeat of the same
        # steps (not used for timing) so that the record still shows the clocks under this load
        sampler = ClockSampler(local_rank)
        sampler.start()
        t_end = time.perf_counter() + 1.0
        while time.perf_counter() < t_end:
            solver.run(zero_tol_options(args.steps))
        clocks = sampler.stop()
        clocks['note'] = 'sampled over a 1 s repeat of the timed steps (timed region shorter than the sampling period)'
    # the other sweep variant, for transparency: dimension tree when `value` is three-pass and vice versa
    n3 = max(3, args.steps // 2)
    other_ms = timed_run(solver, G, lambda it: dict(zero_tol_options(it), dimtree=0 if DIMTREE else 1), n3)[0] / n3

    # ---- per-mode MTTKRP kernel times (CUDA events on the engine's stream) for the roofline ----
    flops_mode = 2.0 * I * J * Kloc * R
    bytes_mode = 8.0 * I * J * Kloc
    solver.run(zero_tol_options(1))    # leaves the FP64 precision selected for time_mttkrp
    mode_ms = [solver.time_mttkrp(1, pos, 3) for pos in (1, 2, 3)]
    tsum = sum(mode_ms)
    # the opt-in reduced-precision MTTKRPs (options.mttkrp_precision: 1 = TF32 and 2 = BF16 on tcgen05 / TMEM, 3 = TF32 on
    # the mma.sync variant of the FP64 kernels); reported beside the FP64 number, never as `value`
    n32 = max(3, args.steps // 2)
    reduced = {}
    for prec, key, what in ((1, 'tf32_opt_in', 'TF32 operands, tcgen05.mma.kind::tf32, FP32 accumulation in TMEM per slab, FP64 across slabs'),
                            (2, 'bf16_opt_in', 'BF16 operands, tcgen05.mma.kind::f16, FP32 accumulation in TMEM per slab, FP64 across slabs'),
                            (3, 'tf32_mma_sync', 'TF32 operands on HMMA.1688.F32.TF32 (mma.sync variant of the FP64 kernels), kept for comparison')):
        ms_lo, _, _, _, out_lo = timed_run(solver, G, lambda it, p=prec: dict(zero_tol_options(it), mttkrp_precision=p), n32)
        ms_lo /= n32
        mode_lo = [solver.time_mttkrp(1, pos, 3) for pos in (1, 2, 3)]
        reduced[key] = {'value': 1e3 / ms_lo, 'ms_per_step': ms_lo, 'mttkrp_ms_per_mode': mode_lo,
                        'mttkrp_gbs': [bytes_mode / (t * 1e-3) / 1e9 for t in mode_lo],
                        'hbm_frac': [bytes_mode / (t * 1e-3) / 1e9 / 6557.1 for t in mode_lo],
                        'final_f_tensors': out_lo['f_tensors'],
                        'note': 'options.mttkrp_precision=%d (opt-in, not the parity mode): %s; the tensor stays FP64 in HBM, so '
                                'the pass is bound by the 8-byte read' % (prec, what)}
    achieved = 3 * flops_mode / (tsum * 1e-3) / 1e12
    hbm_peak = 6557.1
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            hbm_peak = float(json.load(f)['hbm_gbs'])
    except Exception:
        pass
    # dram bytes per launch from the ncu --set full captures: 1.004x the algorithmic bytes at R=32 (the C2 launch itself,
    # profiles/r01_ncu_mttkrp_summary.md), 1.008x at R=64 (round-2 LEAD kernel on a K=64 slab of the same 4096x4096 tile
    # shape, profiles/r02_ncu_mttkrp_summary.md: 8.646 GB read + 15.8 MB written for 8.590 GB)
    traffic_ratio = {'c2': 1.004, 'c3k1024': 1.008, 'c3': 1.008}.get(args.workload)
    passes = 2 if DIMTREE else 3
    roofline = {'bound': 'tensor', 'achieved': achieved, 'peak': FP64_DMMA_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                'frac': achieved / FP64_DMMA_PEAK_TFLOPS,
                'peak_nominal': FP64_NOMINAL_TFLOPS, 'frac_nominal': achieved / FP64_NOMINAL_TFLOPS,
                'traffic': bytes_mode * traffic_ratio if traffic_ratio else None,
                'traffic_note': 'dram__bytes_read+write per launch = %.3f x algorithmic bytes (ncu --set full, '
                                'profiles/r02_ncu_mttkrp_summary.md)' % traffic_ratio if traffic_ratio else None,
                'kernel': 'mttkrp_lead_kernel / mttkrp_inner_kernel (FP64 DMMA.8x8x4 + TMA), 3 modes',
                'per_mode_ms': mode_ms, 'per_mode_tflops': [flops_mode / (m * 1e-3) / 1e12 for m in mode_ms],
                'per_mode_hbm_gbs': [bytes_mode / (m * 1e-3) / 1e9 for m in mode_ms], 'hbm_peak_gbs_measured': hbm_peak,
                'hbm_frac': (3 * bytes_mode / (tsum * 1e-3) / 1e9) / hbm_peak,
                'in_step_tflops': passes * flops_mode / (dev_ms / args.steps * 1e-3) / 1e12,
                'peak_source': 'measured: FP64 tensor peak from a DMMA.8x8x4 issue-rate probe on this pool '
                               '(profiles/r01_fp64_probe.log; MEASURED_PEAKS.json has no FP64 entry; cuBLAS DGEMM '
                               'reaches 34.2-35.8 TFLOP/s on the same box); peak_nominal is the data-sheet figure',
                'algorithmic_flops_per_launch': flops_mode, 'algorithmic_bytes_per_launch': bytes_mode,
                'mttkrp_share_of_step': float(ph[0] / call_ms) if call_ms > 0 else None}

    # ---- end-to-end through the C ABI with HOST buffers ----
    e2e = None
    if not args.no_e2e:
        # The tensor slab of this rank (the whole tensor in the one-process form) is brought to the host once, outside
        # the timed region, so that the timed call starts, like the reference's cmtf_fun_AOADMM call, from data in host
        # memory: create copies the tensor and the coupled matrix host->device, set_state the 16 state matrices, run does
        # `steps` outer iterations, get_state brings the state back.
        Khost = K if single_process else (hi - lo)
        n_loc = I * J * Khost
        host, how, tpin = None, None, None
        if _host_memory_ok(8.0 * I * J * K):
            try:
                tpin = torch.empty(n_loc, dtype=torch.float64, pin_memory=True)
                host, how = tpin.numpy().reshape((I, J, Khost), order='F'), 'pinned'
            except Exception:
                try:
                    host, how = np.empty((I, J, Khost), order='F'), 'pageable'
                except MemoryError:
                    host = None
        if host is not None:
            solver.get_object_data(1, host)
        solver.close()   # the resident tensor must go before the end-to-end leg allocates its own
        Zh = dict(Z, object=[host, Z['object'][1]])

        def e2e_call(dimtree):
            barrier()
            t0 = time.perf_counter()
            s2, _ = make_solver(Zh, zn, K)
            if host is None:
                s2.generate_cp_data(1, facs, 0.2, 20261018)
            t1 = time.perf_counter()
            s2.set_state(G)
            t2 = time.perf_counter()
            o2 = s2.run(dict(zero_tol_options(args.steps), dimtree=dimtree))
            t3 = time.perf_counter()
            s2.get_state()
            barrier()
            secs = time.perf_counter() - t0
            parts = {'create_s': t1 - t0, 'set_state_s': t2 - t1, 'run_s': t3 - t2, 'get_state_s': t0 + secs - t3}
            dev = s2.last_run_ms()
            s2.close()
            assert o2['OuterIterations'] == args.steps and np.isfinite(o2['f_tensors'])
            return max_over_ranks(secs), parts, dev, o2

        # the call a user makes: the gateway's defaults (aoadmm_mex.cpp: options.b200_dimtree defaults to 1)
        e2e_s, e2e_parts, e2e_run_dev_ms, o2 = e2e_call(1)
        e2e3_s, e2e3_parts, _, o3 = e2e_call(0)
        # the end-to-end call starts from the same data and state as the device-resident leg's warm-up run: the same
        # objective trajectory over the iterations both have made
        nt = min(len(traj), len(o2['func_val_conv']))
        assert np.max(np.abs(o2['func_val_conv'][:nt] - traj[:nt]) / np.maximum(1.0, np.abs(traj[:nt]))) < 1e-10, \
            (o2['func_val_conv'][:nt], traj[:nt])
        assert np.max(np.abs(o3['func_val_conv'] - o2['func_val_conv']) / np.maximum(1.0, np.abs(o2['func_val_conv']))) < 1e-10
        state_bytes = sum(a.nbytes for k in ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac')
                          for a in G[k] if a is not None)
        h2d = state_bytes + Z['object'][1].nbytes + (8.0 * n_loc if host is not None else sum(f.nbytes for f in facs))
        e2e = {'value': args.steps / e2e_s, 'unit': 'outer_iters/s', 'h2d_bytes_per_step': h2d / args.steps,
               'd2h_bytes_per_step': state_bytes / args.steps, 'seconds': e2e_s, 'host_tensor': how or 'none',
               'parts_rank0': e2e_parts, 'run_device_ms': e2e_run_dev_ms,
               'options': 'gateway defaults (options.b200_dimtree = 1: two tensor passes per step, results equal to rounding)',
               'three_pass': {'value': args.steps / e2e3_s, 'seconds': e2e3_s, 'parts_rank0': e2e3_parts,
                              'note': 'the same call with options.b200_dimtree = 0 (three tensor passes per step, the '
                                      "reference's flop count - what `value` is measured on)"},
               'note': ('one cmtf_fun_AOADMM call of %d outer iterations through the C ABI, host wall clock, max over ranks: '
                        'create (tensor %.1f GB per process + matrix host->device from %s host memory) + set_state + run + '
                        'get_state + destroy; the solver is iterative, so the data cross PCIe once per call, not once per step; '
                        'the NCCL communicator is the cached one of this process'
                        % (args.steps, 8.0 * n_loc / 1e9, how)) if host is not None else
                       ('host memory cannot hold the %.1f GB tensor on this box: the tensor is re-generated on device inside '
                        'the timed region instead of copied' % (8.0 * n_loc / 1e9))}
        del host, tpin, Zh
    else:
        solver.close()

    # ---- BASELINE configs[2] at its own size (4096 x 4096 x 2048, 274.9 GB): extra key of the N >= 2 lines ----
    c3_full = None
    if n_gpus >= 2 and args.workload == 'c3k1024' and not args.no_c3_full:
        w3 = WORKLOADS['c3']
        Z3, G3, facs3 = make_problem(w3['I'], w3['J'], w3['K'], w3['M'], w3['R'], seed=0, with_tensor=False)
        zn3 = [1.0, float(np.sum(Z3['object'][1] ** 2))]
        barrier()
        t0 = time.perf_counter()
        s3, (lo3, hi3) = make_solver(Z3, zn3, w3['K'])
        s3.generate_cp_data(1, facs3, 0.2, 20261018)
        gen_s = time.perf_counter() - t0
        steps3 = max(3, min(args.steps, 10))
        ms3, _, l3, ph3, out3 = timed_run(s3, G3, zero_tol_options, steps3)
        ms3t = timed_run(s3, G3, lambda it: dict(zero_tol_options(it), dimtree=1), steps3)[0]
        s3.run(zero_tol_options(1))
        mode3_ms = [s3.time_mttkrp(1, pos, 2) for pos in (1, 2, 3)]
        s3.close()
        K3loc = w3['K'] // n_gpus
        fl3 = 2.0 * w3['I'] * w3['J'] * K3loc * w3['R']
        c3_full = {'config': workload_config('c3', w3, n_gpus, launch), 'value': steps3 / (ms3 * 1e-3), 'unit': 'outer_iters/s',
                   'ms_per_step': ms3 / steps3, 'steps': steps3, 'gpu_launches': int(l3),
                   'dimtree_value': steps3 / (ms3t * 1e-3), 'final_f_tensors': out3['f_tensors'],
                   'f_tensors_start': float(out3['func_val_conv'][0]),
                   'per_mode_ms': mode3_ms, 'per_mode_tflops': [fl3 / (m * 1e-3) / 1e12 for m in mode3_ms],
                   'roofline_frac': (3 * fl3 / (sum(mode3_ms) * 1e-3) / 1e12) / FP64_DMMA_PEAK_TFLOPS,
                   'create_and_generate_s': gen_s, 'tensor_gb_per_gpu': 8.0 * w3['I'] * w3['J'] * K3loc / 1e9}
        assert out3['f_tensors'] < out3['func_val_conv'][0]

    cb = None
    parity = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        cb, (Zs, Gs, zns, Go, oo) = cpu_baseline_run(wl, 3, 1, keep=True)
        # the bench checks itself: the engine on the CPU arm's own sample (host buffers, same options) must reproduce the
        # oracle's factors (1e-8) and objective history (1e-10) - north_star's tolerances
        Gd, od = ab.cmtf_fun_AOADMM(Zs, zns, Gs, None, None, None, None, zero_tol_options(3))
        ferr = max(float(np.linalg.norm(Gd['fac'][m] - Go['fac'][m]) / np.linalg.norm(Go['fac'][m])) for m in range(5))
        oerr = float(np.max(np.abs(od['func_val_conv'] - oo['func_val_conv'])))
        parity = {'sample': cb['sample'], 'max_factor_rel_err': ferr, 'max_objective_abs_err': oerr,
                  'final_f_tensors_engine': od['f_tensors'], 'final_f_tensors_oracle': oo['f_tensors'], 'dimtree': DIMTREE}
        assert ferr < 1e-8 and oerr < 1e-10, parity

    if rank == 0:
        line = {'metric': 'ao_admm_outer_iters_per_s', 'value': args.steps / (dev_ms * 1e-3), 'unit': 'outer_iters/s',
                'n_gpus': n_gpus, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': dev_ms / args.steps,
                'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': config, 'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches), 'roofline': roofline,
                'cpu_baseline': cb, 'parity_check': parity, 'wall_ms_per_step': wall_ms / args.steps,
                ('three_pass' if DIMTREE else 'dimtree'): {
                    'value': 1e3 / other_ms, 'ms_per_step': other_ms,
                    'note': ('same step with options.dimtree=0: three independent tensor passes, the reference\'s flop and '
                             'byte count') if DIMTREE else
                            ('same step with options.dimtree=1 (engine knob, not the default of this line): the mode-2 pass '
                             'also emits T = X x_1 A and mode 3 is a pass over T - 2 tensor passes per step, results equal '
                             'to rounding (parity-tested)')},
                'tf32_opt_in': reduced['tf32_opt_in'], 'bf16_opt_in': reduced['bf16_opt_in'], 'tf32_mma_sync': reduced['tf32_mma_sync'],
                'c3_full': c3_full,
                'final_f_tensors': out['f_tensors'],
                'call_ms': call_ms,
                'timing': 'CUDA events on the engine stream around exactly `steps` outer iterations (cmtf_fun_AOADMM.m:87-476), '
                          'max over ranks; call_ms is the same run including the one-off iteration-0 objective of '
                          'cmtf_fun_AOADMM.m:32 (one extra MTTKRP per tensor, rank 0)'}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def _host_memory_ok(need_bytes):
    """True when the box (and the cgroup, if limited) can hold `need_bytes` more host memory with 15 % headroom."""
    try:
        avail = None
        for line in open('/proc/meminfo'):
            if line.startswith('MemAvailable:'):
                avail = int(line.split()[1]) * 1024
        for path in ('/sys/fs/cgroup/memory.max', '/sys/fs/cgroup/memory/memory.limit_in_bytes'):
            if os.path.exists(path):
                txt = open(path).read().strip()
                if txt.isdigit():
                    used = 0
                    for up in ('/sys/fs/cgroup/memory.current', '/sys/fs/cgroup/memory/memory.usage_in_bytes'):
                        if os.path.exists(up):
                            used = int(open(up).read().strip())
                    avail = min(avail, int(txt) - used) if avail is not None else int(txt) - used
        return avail is not None and need_bytes * 1.15 < avail
    except Exception:
        return False


if __name__ == '__main__':
    sys.exit(main())
