"""nvecs of sparse modes (aoadmm_nvecs_sparse) on the device: one JSON line per mode.

  n1   both modes of m1's 131072 x 32768 rating matrix (tools/sparse_bench.py rating_data: ~2.5e7 power-law entries,
       rank 32 + noise), r = 32.  Host baseline: SciPy eigsh on a LinearOperator v -> A (A' v) over the CSR unfolding
       (full size), its time and the largest principal angle between its subspace and the device's.
  n2   all three modes of m2's 2^20 x 2^16 x 2^10 tensor (1e8 power-law entries, uniform values), r = 32.

Per mode: nnz, nfib (distinct fibers, counted on the host), the column chunks per application (from the trace) and the
chunk width they imply, iterations and residual, the whole call (host clock around the synchronising call), the build
(first device activity of the call to the first pass-A kernel), the median pass A and pass B (unit kernel + fix-up of
one column chunk), the rest of an iteration (iteration window minus the pass kernels, over the iterations: the dense
Rayleigh-Ritz work, the layout transposes and the host synchronisations) and the peak extra device memory (free memory
sampled every 2 ms during the call).  The timed call and the profiled call are separate runs.  Every line carries the
card name and power limit, read in the same call.

usage: python tools/nvecs_sparse_bench.py [--workloads n1,n2] [--scale 1.0] [--r 32] [--out FILE] [--no-eigsh]
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import sparse_bench as sb  # noqa: E402  (puts the package on sys.path)

ab = sb.ab


def single_Z(S):
    N = len(S.shape)
    return {'loss_function': ['Frobenius'], 'model': ['CP'], 'modes': [list(range(1, N + 1))], 'size': list(S.shape),
            'coupling': {'lin_coupled_modes': [0] * N, 'coupling_type': [], 'coupl_trafo_matrices': [None] * N},
            'constrained_modes': [0] * N, 'constraints': [None] * N, 'weights': [1.0], 'object': [S]}


def nfib(subs, shape, n):
    others = [d for d in range(len(shape)) if d != n]
    lin = np.ravel_multi_index(tuple(subs[:, d] for d in others), tuple(shape[d] for d in others))
    return int(np.unique(lin).size)


def timed_call(s, n, r):
    import torch
    free0 = torch.cuda.mem_get_info(0)[0]
    low = [free0]
    done = threading.Event()

    def poll():
        while not done.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info(0)[0])
            time.sleep(0.002)

    th = threading.Thread(target=poll)
    th.start()
    t0 = time.perf_counter()
    U, info = s.nvecs_sparse(n, r, return_info=True)
    ms = (time.perf_counter() - t0) * 1e3
    done.set()
    th.join()
    return U, info, ms, free0 - low[0]


def profiled_call(s, n, r):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, info = s.nvecs_sparse(n, r, return_info=True)
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda e: e.time_range.start)
    a_pass = [e for e in ev if 'nvecs_fiber_pass_kernel' in e.name]
    a_fix = [e for e in ev if 'nvecs_fiber_fixup_kernel' in e.name]
    b_pass = [e for e in ev if 'nvecs_row_pass_kernel' in e.name]
    b_fix = [e for e in ev if 'nvecs_row_fixup_kernel' in e.name]
    us = lambda e: e.time_range.elapsed_us()  # noqa: E731
    A = [us(p) + us(f) for p, f in zip(a_pass, a_fix)]
    B = [us(p) + us(f) for p, f in zip(b_pass, b_fix)]
    t_first, t_iter0, t_end = ev[0].time_range.start, a_pass[0].time_range.start, ev[-1].time_range.end
    its = info['iterations']
    return {'build_ms': (t_iter0 - t_first) / 1e3,
            'pass_a_median_ms': float(np.median(A)) / 1e3, 'pass_b_median_ms': float(np.median(B)) / 1e3,
            'chunks_per_apply': len(a_pass) / its,
            'rest_of_iteration_ms': ((t_end - t_iter0) - sum(A) - sum(B)) / 1e3 / its,
            'passes_per_iteration_ms': (sum(A) + sum(B)) / 1e3 / its}


def eigsh_baseline(subs, vals, shape, n, r, U):
    import scipy.sparse as sps
    import scipy.sparse.linalg as sla
    m = 1 - n
    A = sps.csr_matrix((vals, (subs[:, n], subs[:, m])), shape=(shape[n], shape[m]))
    op = sla.LinearOperator((shape[n],) * 2, matvec=lambda v: A @ (A.T @ v), dtype=np.float64)
    t0 = time.perf_counter()
    th, V = sla.eigsh(op, k=r, which='LM', tol=0, v0=np.ones(shape[n]))
    sec = time.perf_counter() - t0
    sv = np.linalg.svd(V.T @ U, compute_uv=False)
    angle = float(np.arccos(np.clip(sv.min(), -1.0, 1.0)))
    return {'eigsh_s': sec, 'eigsh_max_angle_rad': angle, 'host_cores': os.cpu_count()}


def warm_up():
    rng = np.random.RandomState(0)
    subs = np.stack([rng.randint(0, s, 5000) for s in (300, 200, 100)], axis=1)
    with ab.Solver(dict(single_Z(ab.sptensor(subs, rng.randn(5000), (300, 200, 100))), rank=[32]), [float('nan')]) as s:
        for n in (1, 2, 3):
            s.nvecs_sparse(n, 32)


def run_modes(name, S, subs, vals, shape, r, eigsh, card, out):
    Z = dict(single_Z(S), rank=[r])
    with ab.Solver(Z, [float('nan')]) as s:
        for n in range(len(shape)):
            U, info, ms, peak = timed_call(s, n + 1, r)
            line = {'workload': name, 'mode': n + 1, 'shape': list(shape), 'nnz': int(len(vals)), 'r': r,
                    'nfib': nfib(subs, shape, n), 'iterations': info['iterations'], 'residual': info['residual'],
                    'call_ms': ms, 'peak_extra_device_bytes': int(peak)}
            line.update(profiled_call(s, n + 1, r))
            rb = r + max(8, r // 4) if shape[n] > 128 else shape[n]
            line['chunk_columns'] = int(np.ceil(rb / round(line['chunks_per_apply'])))
            if eigsh and len(shape) == 2:
                line.update(eigsh_baseline(subs, vals, shape, n, r, U))
            line.update({'card': card['name'], 'power_limit': card['power_limit']})
            print(json.dumps(line), flush=True)
            out.write(json.dumps(line) + '\n')
            out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='n1,n2')
    ap.add_argument('--scale', type=float, default=1.0)
    ap.add_argument('--r', type=int, default=32)
    ap.add_argument('--out', default=os.path.join('profiles', 'nvecs_sparse_bench.jsonl'))
    ap.add_argument('--no-eigsh', action='store_true')
    a = ap.parse_args()
    if ab.device_count() < 1:
        raise SystemExit('nvecs_sparse_bench: no CUDA device')
    card = sb.card()
    warm_up()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'a') as out:
        for w in a.workloads.split(','):
            rng = np.random.RandomState(0)
            if w == 'n1':
                I, J = 131072, 32768
                i, j, vals, _ = sb.rating_data(rng, I, J, int(2.5e7 * a.scale), 0, 32)
                subs = np.stack([i, j], axis=1)
                shape = (I, J)
            elif w == 'n2':
                _, _, shape, _, subs, vals = sb.m2_problem(rng, a.scale, 32)
            else:
                raise SystemExit('unknown workload ' + w)
            run_modes(w, ab.sptensor(subs, vals, shape), subs, vals, shape, a.r, not a.no_eigsh, card, out)


if __name__ == '__main__':
    main()
