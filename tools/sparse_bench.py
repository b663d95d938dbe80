"""Sparse CP objects on the device: one JSON line per workload (engine through the ctypes binding, one GPU).

  s1-<density>  1000^3 CP tensor, R = 32, nonneg, coupled in mode 1 to a dense 1000 x 5000 matrix (the C2 structure),
                seeded uniform subscripts at the given density, both objects normalised to unit Frobenius norm as in the
                reference's example scripts (so the objective tolerance is absolute and relative alike); the dense engine
                on full(X) runs in the same call
                (the two handles alternate) and both are run from the same initial state to compare their outputs.
  s2            2^20 x 2^20 x 2^14 CP tensor, R = 32, ~2e8 power-law nonzeros (i = floor(I u^3)), coupled in mode 1 to a
                sparse 2^20 x 2^16 matrix with ~2e7 nonzeros: a problem whose dense form (2^54 = 1.8e16 entries) cannot exist.
                CPU baseline: NumPy COO MTTKRP on the host cores on a 1 % nonzero sample, extrapolated in proportion to nnz.

  m1            131072 x 32768 rating matrix with ~2.5e7 observed entries (power-law rows and columns, rank 32 + noise)
                and a sparse mask of exactly those entries, coupled in mode 2 to a dense 32768 x 1024 side matrix, R = 32,
                nonneg: the sparse-mask engine against the dense EM engine on full(S) + the dense mask (34 GB + 4.3 GB
                on the host and the device; that arm is skipped, with the reason, when the host cannot hold it), both
                from the same state; outer it/s, the per-iteration phase split (torch.profiler kernel times), compare,
                and the held-out RMSE on 1 % of the entries withheld from both, over every iteration, from the device
                held-out history (aoadmm_set_heldout), with the outer it/s with and without the held-out set, the
                held-out pass time next to the imputation pass, and the time of the host NumPy evaluation it replaces.
  m2            2^20 x 2^16 x 2^10 with 1e8 observed power-law entries and their mask, R = 32, nonneg (no dense form):
                it/s, the phase split, the create time, and the overhead against the same object without the mask;
                the same held-out measurements as m1 with 1e7 unobserved power-law entries held out.
                CPU baseline as in s2: NumPy imputed pass (model at the entries + residual MTTKRP per mode) on a 1 %
                sample, extrapolated in proportion to nnz.
  m1, m2        also an early-stopping leg (set_heldout_stopping, patience 3, at most --stop-iters iterations): the
                snapshot kernel time and bytes, the restore time with the re-imputation, outer it/s with stopping on
                and off (alternating), k*, n and the held-out RMSE at k* and after n.
  c1_em         the same leg on a launch-bound dense EM problem: the C1 structure (example_script6 sizes) fitted at
                three times its rank with 70 % of the first tensor missing.

Every line carries the card name and power limit (nvidia-smi, read in the same call), the create time (upload + sorts),
the per-mode sparse MTTKRP time (CUDA events, aoadmm_time_mttkrp), outer iterations/s, and the algorithmic bytes per mode
computed from the shapes: stream = nnz (8 + 4 (N-1)) + row pointers + output, gathered upper bound = nnz (N-1) 8 R, and
the stream rate against the 6557 GB/s measured copy peak.  nnz is the number of nonzeros handed to the engine (before
duplicates are merged).

usage: python tools/sparse_bench.py [--workloads s1,s2,m1,m2,c1_em] [--densities 0.001,0.01,0.1] [--s2-scale 1.0]
                                    [--m-scale 1.0] [--iters 5] [--stop-iters 30]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'matlab-code_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

import aoadmm_b200 as ab  # noqa: E402

COPY_PEAK_GBS = 6557.0
ZERO_TOL = dict(AbsFuncTol=0.0, OuterRelTol=0.0, innerRelPrTol_coupl=0.0, innerRelPrTol_constr=0.0,
                innerRelDualTol_coupl=0.0, innerRelDualTol_constr=0.0)


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True, check=True).stdout.strip().split('\n')
    first = out[0].split(', ')
    return {'name': first[0], 'power_limit': first[1], 'visible_gpus': len(out),
            'power_limits': sorted(set(l.split(', ')[1] for l in out))}


def options(iters, **kw):
    o = dict(MaxOuterIters=iters, MaxInnerIters=5, bsum=0, **ZERO_TOL)
    o.update(kw)
    return o


def problem(objects, sizes, R, coupling_modes):
    n = len(sizes)
    return {'loss_function': ['Frobenius'] * len(objects), 'model': ['CP'] * len(objects),
            'modes': [[1, 2, 3], [4, 5]], 'size': list(sizes),
            'coupling': {'lin_coupled_modes': coupling_modes, 'coupling_type': [0], 'coupl_trafo_matrices': [None] * n},
            'constrained_modes': [1] * n, 'constraints': [('non-negativity',)] * n, 'weights': [0.5, 0.5],
            'object': objects, 'rank': [R, R]}


def init_state(Z, R, seed):
    rng = np.random.RandomState(seed)
    io = {'lambdas_init': [[1.0] * R] * 2, 'nvecs': 0, 'normalize': 1,
          'distr': [lambda a, b: rng.rand(a, b)] * len(Z['size'])}
    return ab.init_coupled_AOADMM_CMTF(Z, io, rng=rng)


def mode_bytes(nnz, shape, n, R):
    N = len(shape)
    stream = nnz * (8 + 4 * (N - 1)) + (shape[n] + 1) * 8 + shape[n] * R * 8
    return stream, nnz * (N - 1) * 8 * R


def sparse_modes(s, shape, nnz, R, reps):
    out = []
    for n in range(len(shape)):
        ms = s.time_mttkrp(1, n + 1, reps)
        stream, gath = mode_bytes(nnz, shape, n, R)
        out.append({'mode': n + 1, 'ms': ms, 'stream_bytes': stream, 'gather_bytes_upper': gath,
                    'stream_GBs': stream / ms / 1e6, 'stream_share_of_copy_peak': stream / ms / 1e6 / COPY_PEAK_GBS})
    return out


def timed_create(Z, zn):
    t0 = time.perf_counter()
    s = ab.Solver(Z, zn)
    return s, time.perf_counter() - t0


def iters_per_s(s, G, iters, **kw):
    s.set_state(G)
    s.run(options(iters, **kw))
    return iters / (s.last_loop_ms() / 1e3)


def s1(density, iters, reps, seed=0, R=32, I=1000, M=5000):
    rng = np.random.RandomState(seed)
    shape = (I, I, I)
    A, B, C, D = (rng.rand(n, R) for n in (I, I, I, M))
    lin = np.unique(rng.randint(0, I ** 3, size=int(density * I ** 3)))    # uniform, without repeats
    i, j, k = lin % I, (lin // I) % I, lin // (I * I)
    vals = np.empty(lin.size)
    for a in range(0, lin.size, 1 << 22):                                  # CP values at the nonzeros + 10 % noise
        sl = slice(a, a + (1 << 22))
        v = np.einsum('er,er,er->e', A[i[sl]], B[j[sl]], C[k[sl]])
        vals[sl] = v * (1.0 + 0.1 * rng.randn(v.size))
    vals /= np.linalg.norm(vals)                                           # ||X||_F = 1 (example_script6...m:101-102)
    Xs = ab.sptensor(np.stack([i, j, k], axis=1), vals, shape)
    Xd = np.zeros(I ** 3)
    Xd[lin] = vals                                                         # column-major linear index
    Xd = Xd.reshape(shape, order='F')
    Y = A @ D.T + 0.1 * rng.randn(I, M)
    Y /= np.linalg.norm(Y)
    sizes = [I, I, I, I, M]
    Zs = problem([Xs, Y], sizes, R, [1, 0, 0, 1, 0])
    Zd = problem([Xd, Y], sizes, R, [1, 0, 0, 1, 0])
    zY = float(np.sum(Y * Y))
    G = init_state(Zd, R, seed + 1)
    sp, t_sp = timed_create(Zs, [float('nan'), zY])
    de, t_de = timed_create(Zd, [float('nan'), zY])
    # outputs from the same initial state
    sp.set_state(G)
    o_sp = sp.run(options(iters))
    G_sp = sp.get_state()
    de.set_state(G)
    o_de = de.run(options(iters))
    G_de = de.get_state()
    fac_rel = max(float(np.linalg.norm(a - b) / np.linalg.norm(b)) for a, b in zip(G_sp['fac'], G_de['fac']))
    obj_abs = float(np.max(np.abs(o_sp['func_val_conv'] - o_de['func_val_conv'])))
    # timings, alternating the two handles
    rounds = []
    for _ in range(3):
        rounds.append(('sparse', [sp.time_mttkrp(1, n, reps) for n in (1, 2, 3)], iters_per_s(sp, G, iters)))
        rounds.append(('dense', [de.time_mttkrp(1, n, reps) for n in (1, 2, 3)], iters_per_s(de, G, iters)))
    med = {}
    for arm in ('sparse', 'dense'):
        rs = [r for r in rounds if r[0] == arm]
        med[arm] = ([float(np.median([r[1][n] for r in rs])) for n in range(3)], float(np.median([r[2] for r in rs])))
    modes = sparse_modes(sp, shape, Xs.nnz, R, reps)
    for n, m in enumerate(modes):
        m['ms'] = med['sparse'][0][n]
        m['stream_GBs'] = m['stream_bytes'] / m['ms'] / 1e6
        m['stream_share_of_copy_peak'] = m['stream_GBs'] / COPY_PEAK_GBS
        m['dense_ms'] = med['dense'][0][n]
        m['sparse_over_dense'] = m['ms'] / m['dense_ms']
    line = {'workload': 's1', 'density': density, 'shape': list(shape), 'R': R, 'nnz': int(Xs.nnz),
            'create_s': {'sparse': t_sp, 'dense': t_de}, 'modes': modes,
            'outer_iters_per_s': {'sparse': med['sparse'][1], 'dense': med['dense'][1]}, 'iters': iters,
            'compare': {'factors_max_rel': fac_rel, 'objective_max_abs': obj_abs,
                        'ok': bool(fac_rel <= 1e-8 and obj_abs <= 1e-10)},
            'f_tensors': {'sparse': o_sp['f_tensors'], 'dense': o_de['f_tensors']}}
    sp.close()
    de.close()
    return line


def powerlaw(rng, n, extent):
    return np.minimum((extent * rng.rand(n) ** 3).astype(np.int64), extent - 1)


def s2_problem(rng, scale, R):
    I, J, K, M = 1 << 20, 1 << 20, 1 << 14, 1 << 16
    shape = (I, J, K)
    nnz = int(2e8 * scale)
    subs = np.stack([powerlaw(rng, nnz, I), powerlaw(rng, nnz, J), powerlaw(rng, nnz, K)], axis=1)
    vals = rng.rand(nnz)
    ny = int(2e7 * scale)
    ysubs = np.stack([powerlaw(rng, ny, I), rng.randint(0, M, size=ny)], axis=1)
    yvals = rng.rand(ny)
    Zs = problem([ab.sptensor(subs, vals, shape), ab.sptensor(ysubs, yvals, (I, M))], [I, J, K, I, M], R, [1, 0, 0, 1, 0])
    return Zs, shape, nnz, subs, vals, ny, (I, M)


def s2(scale, iters, reps, seed=0, R=32):
    rng = np.random.RandomState(seed)
    Zs, shape, nnz, subs, vals, ny, (I, M) = s2_problem(rng, scale, R)
    sp, t_create = timed_create(Zs, [float('nan'), float('nan')])
    G = init_state(Zs, R, seed + 1)
    sp.set_state(G)
    ips = iters_per_s(sp, G, iters)
    modes = sparse_modes(sp, shape, nnz, R, reps)
    matrix_ms = [sp.time_mttkrp(2, n, reps) for n in (1, 2)]
    sp.close()
    # CPU baseline: NumPy COO MTTKRP on a 1 % sample, extrapolated in proportion to nnz
    frac = 0.01
    pick = rng.rand(nnz) < frac
    ss, sv = subs[pick], vals[pick]
    U = [np.random.RandomState(n).rand(s, R) for n, s in enumerate(shape)]
    t0 = time.perf_counter()
    for n in range(3):
        contrib = sv[:, None] * np.ones((1, R))
        for m in range(3):
            if m != n:
                contrib *= U[m][ss[:, m]]
        out = np.zeros((shape[n], R))
        np.add.at(out, ss[:, n], contrib)
    cpu_ms = (time.perf_counter() - t0) / 3 * 1e3 * nnz / max(int(pick.sum()), 1)
    return {'workload': 's2', 'shape': list(shape), 'R': R, 'nnz': nnz, 'matrix_shape': [I, M], 'matrix_nnz': ny,
            'create_s': t_create, 'modes': modes, 'matrix_modes_ms': matrix_ms, 'outer_iters_per_s': ips,
            'iters': iters, 'cpu_baseline': {'kind': 'numpy COO MTTKRP on the host cores, 1 % nonzero sample, '
                                                      'extrapolated in proportion to nnz',
                                             'cores': os.cpu_count(), 'ms_per_mode': cpu_ms}}


# ---- m1 / m2: sparse objects with a sparse Z.miss mask ------------------------------------------------------------
def mem_available_bytes():
    try:
        with open('/proc/meminfo') as f:
            for line in f:
                if line.startswith('MemAvailable:'):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def phase_split(solver, G, iters, order):
    """Per-iteration device time of the masked-sparse phases from one profiled run (graph off so that every kernel is
    listed): the imputation pass, each mode's sparse MTTKRP (unit pass + fix-up), the low-rank terms, the EM norms
    (stacked Grams + telescoped reduction) and everything else, in ms."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    solver.set_state(G)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        solver.run(options(iters, graph=-1))
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda e: e.time_range.start)
    out = {'impute_pass': 0.0, 'heldout_pass': 0.0, 'lowrank': 0.0, 'em_norms': 0.0, 'factor_transposes': 0.0,
           'other': 0.0}
    for n in range(order):
        out['mttkrp_mode%d' % (n + 1)] = 0.0
    k_sp = k_fix = 0
    follow = None      # category of the GEMM launched right after a hadamard / stack kernel
    for e in ev:
        nm, us = e.name, e.time_range.elapsed_us() / 1e3
        if 'sp_model_kernel' in nm:
            cat = 'impute_pass'
        elif 'heldout_kernel' in nm or 'sum_partials_kernel' in nm:   # its factor transposes: factor_transposes
            cat = 'heldout_pass'
        elif 'sp_mttkrp_kernel' in nm:
            cat = 'mttkrp_mode%d' % (k_sp % order + 1)
            k_sp += 1
        elif 'sp_fixup_kernel' in nm:
            cat = 'mttkrp_mode%d' % (k_fix % order + 1)
            k_fix += 1
        elif 'hadamard_others' in nm:
            cat, follow = 'lowrank', 'lowrank'
        elif 'stack3' in nm or 'tele_partials' in nm or 'em_final' in nm or 'cg_from_g3' in nm:
            cat, follow = 'em_norms', 'em_norms'
        elif 'dgemm' in nm and follow is not None:
            cat = follow
            if 'reduce' in nm or follow == 'lowrank':
                follow = None
        elif 'transpose_scale' in nm:
            cat = 'factor_transposes'
        else:
            cat = 'other'
            follow = None
        out[cat] += us
    return {k: v / iters for k, v in out.items()}


def rating_data(rng, I, J, n_obs, n_test, R, noise=0.1):
    """~n_obs + n_test distinct power-law (i, j) with values (A B')_ij (1 + noise N(0,1)), A, B ~ U(0,1)."""
    want = n_obs + n_test
    lin = np.empty(0, dtype=np.int64)
    while lin.size < want:
        m = int(1.3 * (want - lin.size)) + 1000
        lin = np.unique(np.r_[lin, powerlaw(rng, m, I) * J + np.minimum((J * rng.rand(m) ** 2).astype(np.int64), J - 1)])
    lin = lin[rng.permutation(lin.size)[:want]]
    i, j = lin // J, lin % J
    A, B = rng.rand(I, R), rng.rand(J, R)
    vals = np.empty(want)
    for a in range(0, want, 1 << 22):
        sl = slice(a, a + (1 << 22))
        v = np.einsum('er,er->e', A[i[sl]], B[j[sl]])
        vals[sl] = v * (1.0 + noise * rng.randn(v.size))
    return i, j, vals, B


def heldout_first_run(sp, G, iters, H, host_model):
    """A run of `sp` with the held-out set H attached: the held-out RMSE curve over all iterations from the device history,
    and what that replaces: the factors read back and the model evaluated at the held-out entries in NumPy
    (host_model(fac) -> predictions).  Returns (fields, out, state); the set stays attached."""
    sp.set_heldout(1, H)
    sp.set_state(G)
    out = sp.run(options(iters))
    sse, count = sp.heldout_history(1)
    t0 = time.perf_counter()
    Gh = sp.get_state()
    pred = host_model(Gh['fac'])
    host_sse = float(np.sum((H.vals - pred) ** 2))
    host_ms = (time.perf_counter() - t0) * 1e3
    return {'heldout_entries': count, 'held_out_rmse_curve': [float(x) for x in np.sqrt(sse / count)],
            'held_out_rmse': float(np.sqrt(sse[-1] / count)), 'held_out_rmse_host': float(np.sqrt(host_sse / count)),
            'host_eval_ms': host_ms}, out, Gh


def heldout_legs(sp, G, iters, H, order):
    """Outer it/s without and with the held-out set H attached (alternating) and the per-iteration held-out pass and
    imputation pass times (profiled run).  Leaves the set detached."""
    ips = {'no_heldout': [], 'heldout': []}
    for _ in range(2):
        sp.set_heldout(1, None)
        ips['no_heldout'].append(iters_per_s(sp, G, iters))
        sp.set_heldout(1, H)
        ips['heldout'].append(iters_per_s(sp, G, iters))
    med = {k: float(np.median(v)) for k, v in ips.items()}
    ph = phase_split(sp, G, iters, order)
    sp.set_heldout(1, None)
    return {'heldout_outer_iters_per_s': med, 'heldout_it_s_change': med['heldout'] / med['no_heldout'] - 1.0,
            'heldout_pass_ms_per_iter': ph['heldout_pass'], 'impute_pass_ms_per_iter': ph['impute_pass']}


def state_bytes(G):
    """Bytes of the snapshot list of early stopping: every array of G (factors, constraint and coupling duals, coupling
    factors, PARAFAC2 P / DeltaB / mu_DeltaB)."""
    tot = 0
    for v in G.values():
        for a in v:
            for x in (a if isinstance(a, list) else [a]):
                tot += 0 if x is None else np.asarray(x).nbytes
    return tot


def stopping_leg(sp, G, H, iters, patience=3, rounds=2):
    """Early stopping on the held-out error (set_heldout_stopping) with the held-out set H on object 1:
      - one profiled run (graph off) with the given patience and at most `iters` iterations: the kernel time of each
        snapshot (state_copy_kernel<0>) and the bytes it moves (read + write of the snapshot list), and the restore
        time (state_copy_kernel<1> and the re-imputation: from its start to the end of the run's last kernel);
      - outer it/s of the same run with stopping off and on (patience > iters, so both run `iters` iterations and the
        second snapshots after every improving iteration), alternating rounds;
      - k*, n and the held-out RMSE at k* against the RMSE after n.
    Leaves the set detached and stopping off."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    sp.set_heldout(1, H)
    sp.set_heldout_stopping(patience)
    sp.set_state(G)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = sp.run(options(iters, graph=-1))
        torch.cuda.synchronize()
    k_best, _ = sp.heldout_best()
    n = out['OuterIterations']
    sse, count = sp.heldout_history(1)
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda e: e.time_range.start)
    snaps = [e.time_range.elapsed_us() / 1e3 for e in ev if 'state_copy_kernel<0>' in e.name]
    rst = [e for e in ev if 'state_copy_kernel<1>' in e.name]
    restore_ms = None
    if rst:
        t0 = rst[0].time_range.start
        restore_ms = (max(e.time_range.end for e in ev if e.time_range.start >= t0) - t0) / 1e3
    ips = {'stopping_off': [], 'stopping_on': []}
    for _ in range(rounds):
        sp.set_heldout_stopping(0)
        ips['stopping_off'].append(iters_per_s(sp, G, iters))
        sp.set_heldout_stopping(iters + 1)
        ips['stopping_on'].append(iters_per_s(sp, G, iters))
    sp.set_heldout_stopping(0)
    sp.set_heldout(1, None)
    med = {k: float(np.median(v)) for k, v in ips.items()}
    nbytes = 2 * state_bytes(G)
    snap_ms = float(np.median(snaps)) if snaps else None
    return {'patience': patience, 'max_iters': iters, 'best_iter': k_best, 'iters_run': n,
            'exit_flag': out['exit_flag'] if isinstance(out['exit_flag'], str) else 'tolerance',
            'held_out_rmse_at_best': float(np.sqrt(sse[k_best] / count)),
            'held_out_rmse_at_end': float(np.sqrt(sse[n] / count)),
            'snapshots': len(snaps), 'snapshot_kernel_ms': snap_ms, 'snapshot_bytes': nbytes,
            'snapshot_GBs': nbytes / snap_ms / 1e6 if snap_ms else None,
            'restore_ms': restore_ms if restore_ms is not None else 'not triggered (k* = n)',
            'outer_iters_per_s': med, 'it_s_change': med['stopping_on'] / med['stopping_off'] - 1.0,
            'outer_iters_per_s_rounds': ips}


def c1_em(iters, seed=0):
    """Early stopping on a launch-bound problem: the C1 structure (example_script6 sizes, three coupled nonneg objects,
    R = 3 fitted at R = 9) with 70 % of the first tensor missing and half of the missing entries held out."""
    from oracle import problem_gen as pg
    Z, _, _ = pg.config_script6(seed=seed)
    rng = np.random.RandomState(seed + 1)
    io = {'lambdas_init': [[1.0] * 9] * 3, 'nvecs': 0, 'normalize': 1, 'distr': [pg.d_rand] * len(Z['size'])}
    G = pg.init_coupled_AOADMM_CMTF(Z, io, rng)
    Zm = pg.add_missing(Z, 0.7, seed=seed, objects=[0])
    X, W = Z['object'][0], Zm['miss'][0]
    hs = np.argwhere(~W)
    hs = hs[np.random.RandomState(seed).rand(len(hs)) < 0.5]
    H = ab.sptensor(hs, X[tuple(hs.T)], X.shape)
    with ab.Solver(ab._with_rank(Zm, G), pg.znorm_const(Zm)) as s:
        leg = stopping_leg(s, G, H, iters)
    return {'workload': 'c1_em', 'sizes': [int(x) for x in Z['size']], 'R': 9, 'missing': 0.7,
            'held_out': int(len(hs)), 'early_stopping': leg}


def m1(scale, iters, stop_iters, seed=0, R=32):
    rng = np.random.RandomState(seed)
    I, J, L = 131072, 32768, 1024
    n_obs = int(2.5e7 * scale)
    n_test = n_obs // 100
    i, j, vals, B = rating_data(rng, I, J, n_obs, n_test, R)
    nrm = np.linalg.norm(vals[:n_obs])
    vals /= nrm                                                            # observed part at unit norm
    subs = np.stack([i[:n_obs], j[:n_obs]], axis=1)
    S = ab.sptensor(subs, vals[:n_obs], (I, J))
    Wm = ab.sptensor(subs, np.ones(n_obs), (I, J))
    Y = B @ rng.rand(L, R).T
    Y = np.asfortranarray(Y * (1.0 + 0.1 * rng.randn(J, L)))
    Y /= np.linalg.norm(Y)
    zY = float(np.sum(Y * Y))
    n = 4

    def Zof(obj, miss):
        return {'loss_function': ['Frobenius'] * 2, 'model': ['CP'] * 2, 'modes': [[1, 2], [3, 4]],
                'size': [I, J, J, L],
                'coupling': {'lin_coupled_modes': [0, 1, 1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * n},
                'constrained_modes': [1] * n, 'constraints': [('non-negativity',)] * n, 'weights': [0.5, 0.5],
                'object': [obj, Y], 'miss': [miss, None], 'rank': [R, R]}

    Zs = Zof(S, Wm)
    G = init_state(Zs, R, seed + 1)
    sp, t_sp = timed_create(Zs, [float('nan'), zY])
    line = {'workload': 'm1', 'shape': [I, J], 'side_shape': [J, L], 'R': R, 'observed': n_obs, 'held_out': n_test,
            'iters': iters, 'create_s': {'sparse_mask': t_sp}}
    H = ab.sptensor(np.stack([i[n_obs:], j[n_obs:]], axis=1), vals[n_obs:], (I, J))
    # the first run carries the held-out set (it does not change the solve): RMSE curve on the device, host evaluation
    held, o_sp, G_sp = heldout_first_run(sp, G, iters, H, lambda F: np.einsum('er,er->e', F[0][i[n_obs:]], F[1][j[n_obs:]]))
    sp.set_heldout(1, None)
    line.update(held)
    dense_bytes = I * J * 9
    avail = mem_available_bytes()
    de = None
    if avail < 2.5 * dense_bytes:
        line['dense_arm'] = 'skipped: the host has %.1f GB available, the dense arm needs about %.1f GB' % (
            avail / 1e9, 2.5 * dense_bytes / 1e9)
    else:
        Xd = np.zeros((I, J), order='F')
        Xd[subs[:, 0], subs[:, 1]] = vals[:n_obs]
        Md = np.zeros((I, J), dtype=np.uint8, order='F')
        Md[subs[:, 0], subs[:, 1]] = 1
        de, t_de = timed_create(Zof(Xd, Md), [float('nan'), zY])
        del Xd, Md
        line['create_s']['dense_em'] = t_de
        de.set_state(G)
        o_de = de.run(options(iters))
        G_de = de.get_state()
        line['compare'] = {
            'factors_max_rel': max(float(np.linalg.norm(a - b) / np.linalg.norm(b)) for a, b in zip(G_sp['fac'], G_de['fac'])),
            'objective_max_abs': float(np.max(np.abs(o_sp['func_val_conv'] - o_de['func_val_conv']))),
            'f_rel_missing_max_abs': float(np.max(np.abs(o_sp['func_rel_missing'][1:] - o_de['func_rel_missing'][1:])))}
    ips = {'sparse_mask': [], 'dense_em': []}
    for _ in range(2):
        ips['sparse_mask'].append(iters_per_s(sp, G, iters))
        if de is not None:
            ips['dense_em'].append(iters_per_s(de, G, iters))
    line['outer_iters_per_s'] = {k: float(np.median(v)) for k, v in ips.items() if v}
    line.update(heldout_legs(sp, G, iters, H, 2))
    line['early_stopping'] = stopping_leg(sp, G, H, stop_iters)
    line['phase_ms_per_iter'] = {'sparse_mask': phase_split(sp, G, iters, 2)}
    line['held_out_rms_value'] = float(np.sqrt(np.mean(vals[n_obs:] ** 2)))
    line['f_rel_missing_last'] = float(o_sp['f_rel_missing'])
    sp.close()
    if de is not None:
        de.close()
    return line


def m2_problem(rng, scale, R):
    shape = (1 << 20, 1 << 16, 1 << 10)
    nnz = int(1e8 * scale)
    subs = np.stack([powerlaw(rng, nnz, shape[0]), powerlaw(rng, nnz, shape[1]), powerlaw(rng, nnz, shape[2])], axis=1)
    vals = rng.rand(nnz)
    n = 3
    Z = {'loss_function': ['Frobenius'], 'model': ['CP'], 'modes': [[1, 2, 3]], 'size': list(shape),
         'coupling': {'lin_coupled_modes': [0] * n, 'coupling_type': [], 'coupl_trafo_matrices': [None] * n},
         'constrained_modes': [1] * n, 'constraints': [('non-negativity',)] * n, 'weights': [1.0],
         'object': [ab.sptensor(subs, vals, shape)], 'rank': [R]}
    Zm = dict(Z, miss=[ab.sptensor(subs, np.ones(nnz), shape)])
    return Z, Zm, shape, nnz, subs, vals


def m2(scale, iters, stop_iters, seed=0, R=32):
    rng = np.random.RandomState(seed)
    Z, Zm, shape, nnz, subs, vals = m2_problem(rng, scale, R)
    G = init_state(Zm, R, seed + 1)
    sp, t_sp = timed_create(Zm, [float('nan')])
    un, t_un = timed_create(Z, [float('nan')])
    # 1e7 held-out entries: power-law subscripts that are not observed, random true values
    n_held = int(1e7 * scale)
    key = lambda a: (a[:, 0] * shape[1] + a[:, 1]) * shape[2] + a[:, 2]
    hs = np.empty((0, 3), dtype=np.int64)
    obs = np.sort(key(subs))
    while hs.shape[0] < n_held:
        c = np.stack([powerlaw(rng, 2 * n_held, s) for s in shape], axis=1)
        k = key(c)
        pos = np.searchsorted(obs, k).clip(max=obs.size - 1)
        c = c[obs[pos] != k]
        hs = np.unique(np.vstack([hs, c]), axis=0)
    hs = hs[rng.permutation(hs.shape[0])[:n_held]]
    H = ab.sptensor(hs, rng.rand(n_held), shape)

    def host_model(F):
        m = np.ones((n_held, R))
        for d in range(3):
            m *= F[d][hs[:, d]]
        return m.sum(axis=1)

    held, _, _ = heldout_first_run(sp, G, iters, H, host_model)
    sp.set_heldout(1, None)
    ips = {'sparse_mask': [], 'no_mask': []}
    for _ in range(2):
        ips['sparse_mask'].append(iters_per_s(sp, G, iters))
        ips['no_mask'].append(iters_per_s(un, G, iters))
    med = {k: float(np.median(v)) for k, v in ips.items()}
    phases = {'sparse_mask': phase_split(sp, G, iters, 3), 'no_mask': phase_split(un, G, iters, 3)}
    held.update(heldout_legs(sp, G, iters, H, 3))
    held['early_stopping'] = stopping_leg(sp, G, H, stop_iters)
    sp.close()
    un.close()
    # CPU baseline: the imputed pass in NumPy on a 1 % sample, extrapolated in proportion to nnz
    pick = rng.rand(nnz) < 0.01
    ss, sv = subs[pick], vals[pick]
    U = [np.random.RandomState(k).rand(s, R) for k, s in enumerate(shape)]
    t0 = time.perf_counter()
    m = np.ones((ss.shape[0], R))
    for d in range(3):
        m *= U[d][ss[:, d]]
    r = sv - m.sum(axis=1)
    for k in range(3):
        contrib = r[:, None] * np.ones((1, R))
        for d in range(3):
            if d != k:
                contrib *= U[d][ss[:, d]]
        out = np.zeros((shape[k], R))
        np.add.at(out, ss[:, k], contrib)
    cpu_ms = (time.perf_counter() - t0) * 1e3 * nnz / max(int(pick.sum()), 1)
    return {'workload': 'm2', 'shape': list(shape), 'R': R, 'nnz': nnz, 'iters': iters,
            'create_s': {'sparse_mask': t_sp, 'no_mask': t_un}, 'outer_iters_per_s': med,
            'mask_overhead': med['no_mask'] / med['sparse_mask'] - 1.0, 'phase_ms_per_iter': phases,
            'heldout': held,
            'cpu_baseline': {'kind': 'numpy imputed pass (model at the entries + residual MTTKRP of every mode) on the '
                                     'host cores, 1 % nonzero sample, extrapolated in proportion to nnz',
                             'cores': os.cpu_count(), 'ms_per_iteration': cpu_ms}}


# ---- s2 / m2 on several GPUs (aoadmm_create_sparse_multi) --------------------------------------------------------
def per_gpu_ms(fn, names, div):
    """Device time per GPU (ms / div) of the kernels whose name contains one of `names`, from one profiled call."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and any(k in e.name for k in names):
            per[e.device_index] = per.get(e.device_index, 0.0) + e.time_range.elapsed_us() / 1e3
    return per


def multi(name, counts, scale, iters, reps, seed=0, R=32):
    """s2 or m2 with Solver(..., n_gpus=N, shard_sparse=True) for every N in counts: the nonzero share of every GPU,
    create time, outer it/s (median of rounds that alternate the GPU counts), the local sparse pass per mode (max and
    min over the GPUs, torch.profiler kernel times of aoadmm_time_mttkrp), the NCCL all-reduce time per outer iteration
    (torch.profiler, a separate run with graph replay off) and agreement with the one-GPU run."""
    rng = np.random.RandomState(seed)
    if name == 's2':
        Z, shape, nnz, subs, _, _, _ = s2_problem(rng, scale, R)
        zn = [float('nan'), float('nan')]
    else:
        _, Z, shape, nnz, subs, _ = m2_problem(rng, scale, R)
        zn = [float('nan')]
    G = init_state(Z, R, seed + 1)
    last = np.sort(subs[:, -1])
    sol, lines = {}, {}
    for n in counts:
        t0 = time.perf_counter()
        sol[n] = ab.Solver(Z, zn, n_gpus=n, shard_sparse=True)
        b = ab.sparse_shard_bounds(Z['object'][0], n)
        lines[n] = {'workload': name + '_multi', 'n_gpus': n, 'shape': list(shape), 'R': R, 'nnz': nnz, 'iters': iters,
                    'create_s': time.perf_counter() - t0, 'bounds': b.tolist(),
                    'nnz_share': (np.diff(np.searchsorted(last, b)) / nnz).tolist()}
    ref = None
    for n in counts:
        s = sol[n]
        s.set_state(G)
        o = s.run(options(iters))
        Gn = s.get_state()
        if ref is None:
            ref = (n, o, Gn)
        lines[n]['compare_to_gpus'] = ref[0]
        lines[n]['factors_max_rel'] = max(float(np.linalg.norm(a - c) / np.linalg.norm(c))
                                          for a, c in zip(Gn['fac'], ref[2]['fac']))
        lines[n]['objective_max_rel'] = float(np.max(np.abs(o['func_val_conv'] - ref[1]['func_val_conv']) /
                                                     np.abs(ref[1]['func_val_conv'])))
    ips = {n: [] for n in counts}
    for _ in range(3):
        for n in counts:
            ips[n].append(iters_per_s(sol[n], G, iters))
    kern = ('sp_mttkrp_kernel', 'sp_fixup_kernel', 'transpose_scale')
    for n in counts:
        s = sol[n]
        lines[n]['outer_iters_per_s'] = float(np.median(ips[n]))
        lines[n]['outer_iters_per_s_rounds'] = ips[n]
        modes = []
        for pos in range(1, len(shape) + 1):
            per = per_gpu_ms(lambda: s.time_mttkrp(1, pos, reps), kern, reps + 1)
            modes.append({'mode': pos, 'local_pass_ms_max': max(per.values()), 'local_pass_ms_min': min(per.values()),
                          'time_mttkrp_ms': s.time_mttkrp(1, pos, reps)})
        lines[n]['modes'] = modes
        s.set_state(G)
        per = per_gpu_ms(lambda: s.run(options(iters, graph=-1)), ('nccl',), iters)
        lines[n]['allreduce_ms_per_iter'] = {'max': max(per.values()) if per else 0.0,
                                             'min': min(per.values()) if per else 0.0}
        s.close()
    return [lines[n] for n in counts]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--workloads', default='s1,s2')
    ap.add_argument('--densities', default='0.001,0.01,0.1')
    ap.add_argument('--s2-scale', type=float, default=1.0, help='fraction of the s2 nonzero counts (1.0 = 2e8 / 2e7)')
    ap.add_argument('--m-scale', type=float, default=1.0, help='fraction of the m1 / m2 observed-entry counts')
    ap.add_argument('--iters', type=int, default=5)
    ap.add_argument('--stop-iters', type=int, default=30,
                    help='the most outer iterations of the early-stopping legs (m1, m2, c1_em)')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--gpus', default=None,
                    help='comma-separated GPU counts, e.g. 1,2,8: run s2 / m2 (from --workloads) with shard_sparse=True '
                         'on each count instead of the one-GPU workloads')
    a = ap.parse_args()
    if ab.device_count() < 1:
        raise SystemExit('sparse_bench: no CUDA device (the engine has no CPU path)')
    c = card()
    wl = a.workloads.split(',')
    if a.gpus is not None:
        for w in ('s2', 'm2'):
            if w in wl:
                scale = a.s2_scale if w == 's2' else a.m_scale
                for line in multi(w, [int(x) for x in a.gpus.split(',')], scale, a.iters, a.reps):
                    print(json.dumps(dict(line, card=c)), flush=True)
        return
    if 's1' in wl:
        for d in (float(x) for x in a.densities.split(',')):
            print(json.dumps(dict(s1(d, a.iters, a.reps), card=c)), flush=True)
    if 's2' in wl:
        print(json.dumps(dict(s2(a.s2_scale, a.iters, a.reps), card=c)), flush=True)
    if 'm1' in wl:
        print(json.dumps(dict(m1(a.m_scale, a.iters, a.stop_iters), card=c)), flush=True)
    if 'm2' in wl:
        print(json.dumps(dict(m2(a.m_scale, a.iters, a.stop_iters), card=c)), flush=True)
    if 'c1_em' in wl:
        print(json.dumps(dict(c1_em(a.stop_iters), card=c)), flush=True)


if __name__ == '__main__':
    main()
