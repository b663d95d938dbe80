"""Sparse CP objects on the device: one JSON line per workload (engine through the ctypes binding, one GPU).

  s1-<density>  1000^3 CP tensor, R = 32, nonneg, coupled in mode 1 to a dense 1000 x 5000 matrix (the C2 structure),
                seeded uniform subscripts at the given density, both objects normalised to unit Frobenius norm as in the
                reference's example scripts (so the objective tolerance is absolute and relative alike); the dense engine
                on full(X) runs in the same call
                (the two handles alternate) and both are run from the same initial state to compare their outputs.
  s2            2^20 x 2^20 x 2^14 CP tensor, R = 32, ~2e8 power-law nonzeros (i = floor(I u^3)), coupled in mode 1 to a
                sparse 2^20 x 2^16 matrix with ~2e7 nonzeros: a problem whose dense form (2^54 = 1.8e16 entries) cannot exist.
                CPU baseline: NumPy COO MTTKRP on the host cores on a 1 % nonzero sample, extrapolated in proportion to nnz.

Every line carries the card name and power limit (nvidia-smi, read in the same call), the create time (upload + sorts),
the per-mode sparse MTTKRP time (CUDA events, aoadmm_time_mttkrp), outer iterations/s, and the algorithmic bytes per mode
computed from the shapes: stream = nnz (8 + 4 (N-1)) + row pointers + output, gathered upper bound = nnz (N-1) 8 R, and
the stream rate against the 6557 GB/s measured copy peak.  nnz is the number of nonzeros handed to the engine (before
duplicates are merged).

usage: python tools/sparse_bench.py [--workloads s1,s2] [--densities 0.001,0.01,0.1] [--s2-scale 1.0] [--iters 5]
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
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True, check=True).stdout.strip().split(', ')
    return {'name': out[0], 'power_limit': out[1]}


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


def s2(scale, iters, reps, seed=0, R=32):
    rng = np.random.RandomState(seed)
    I, J, K, M = 1 << 20, 1 << 20, 1 << 14, 1 << 16
    shape = (I, J, K)
    nnz = int(2e8 * scale)
    subs = np.stack([powerlaw(rng, nnz, I), powerlaw(rng, nnz, J), powerlaw(rng, nnz, K)], axis=1)
    vals = rng.rand(nnz)
    ny = int(2e7 * scale)
    ysubs = np.stack([powerlaw(rng, ny, I), rng.randint(0, M, size=ny)], axis=1)
    yvals = rng.rand(ny)
    Zs = problem([ab.sptensor(subs, vals, shape), ab.sptensor(ysubs, yvals, (I, M))], [I, J, K, I, M], R, [1, 0, 0, 1, 0])
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--workloads', default='s1,s2')
    ap.add_argument('--densities', default='0.001,0.01,0.1')
    ap.add_argument('--s2-scale', type=float, default=1.0, help='fraction of the s2 nonzero counts (1.0 = 2e8 / 2e7)')
    ap.add_argument('--iters', type=int, default=5)
    ap.add_argument('--reps', type=int, default=5)
    a = ap.parse_args()
    if ab.device_count() < 1:
        raise SystemExit('sparse_bench: no CUDA device (the engine has no CPU path)')
    c = card()
    wl = a.workloads.split(',')
    if 's1' in wl:
        for d in (float(x) for x in a.densities.split(',')):
            print(json.dumps(dict(s1(d, a.iters, a.reps), card=c)), flush=True)
    if 's2' in wl:
        print(json.dumps(dict(s2(a.s2_scale, a.iters, a.reps), card=c)), flush=True)


if __name__ == '__main__':
    main()
