"""Sparse objects with a sparse Z.miss mask: EM imputation of the unstored (unobserved) entries without densifying.

A sparse object whose mask marks exactly its stored entries must give what the dense EM path gives on full(S) with the
dense mask W of that pattern.  CPU tests restate the algorithm of aoadmm_create_sparse_masked in NumPy (imputed MTTKRP
as a residual pass plus a low-rank term, the telescoped ||M' - M||^2, the f_rel_missing terms) and check it against the
dense quantities, plus the ctypes checks and Python refusals that happen before any device call.  GPU tests (-m gpu)
compare whole solves with the dense oracle on full(S) + W (north-star tolerances), with the dense engine, and check
bit-reproducibility and a large known-answer completion."""
import ctypes

import numpy as np
import pytest

from oracle import problem_gen as pg
from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
from oracle.tensor_ops import mttkrp as dense_mttkrp
from _cases import FIT_TOL, ZERO_TOL, assert_state_close

INVALID, NO_DEVICE = 1, 8


def full_cp(U):
    """[[U_1, ..., U_N]] as a dense array."""
    X = U[0]
    for F in U[1:]:
        X = np.einsum('...r,jr->...jr', X, F)
    return X.sum(axis=-1)


def model_at(subs, U):
    """m(e) = [[U]](subs[e]) for every row of subs."""
    p = np.ones((subs.shape[0], U[0].shape[1]))
    for d, F in enumerate(U):
        p = p * F[subs[:, d], :]
    return p.sum(axis=1)


def coo_mttkrp(subs, vals, shape, U, n):
    out = np.zeros((shape[n], U[0].shape[1]))
    contrib = np.repeat(vals[:, None], U[0].shape[1], axis=1)
    for m in range(len(shape)):
        if m != n:
            contrib = contrib * U[m][subs[:, m], :]
    np.add.at(out, subs[:, n], contrib)
    return out


def imputed_mttkrp(subs, vals, shape, B, F, n):
    """Step 1: MTTKRP of S + (1-W).*[[B]] = (S - W.*[[B]]) + [[B]]: the sparse pass on r = s - m plus B_n * H_n."""
    r = vals - model_at(subs, B)
    H = np.ones((F[0].shape[1],) * 2)
    for k in range(len(shape)):
        if k != n:
            H = H * (B[k].T @ F[k])
    return coo_mttkrp(subs, r, shape, F, n) + B[n] @ H


def telescoped_diff2(A, B):
    """Step 3: ||[[A]] - [[B]]||^2 = sum_{k,l} <T_k, T_l>, T_k = [[A_1..A_{k-1}, A_k - B_k, B_{k+1}..B_N]], from the
    cross-Grams of [A_j | B_j | A_j - B_j] (never two model norms subtracted)."""
    N = len(A)
    X = [[A[d], B[d], A[d] - B[d]] for d in range(N)]
    typ = lambda k, d: 0 if d < k else (2 if d == k else 1)
    tot = 0.0
    for k in range(N):
        for l in range(N):
            h = np.ones((A[0].shape[1],) * 2)
            for d in range(N):
                h = h * (X[d][typ(k, d)].T @ X[d][typ(l, d)])
            tot += h.sum()
    return tot


def model_norm2(B):
    h = np.ones((B[0].shape[1],) * 2)
    for F in B:
        h = h * (F.T @ F)
    return h.sum()


def random_pattern(shape, frac, rng):
    W = rng.rand(*shape) < frac
    subs = np.argwhere(W).astype(np.int64)
    return subs, rng.randn(subs.shape[0]), W


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('shape', [(9, 7), (7, 6, 5), (6, 5, 4, 3)])
def test_imputed_mttkrp_restatement_equals_dense(shape):
    rng = np.random.RandomState(len(shape))
    R = 3
    subs, vals, W = random_pattern(shape, 0.3, rng)
    S = np.zeros(shape)
    S[tuple(subs.T)] = vals
    B = [rng.randn(s, R) for s in shape]
    F = [rng.randn(s, R) for s in shape]
    Ximp = np.where(W, S, full_cp(B))       # the dense EM data after an imputation with the factors B
    for n in range(len(shape)):
        ref = dense_mttkrp(Ximp, F, n)
        got = imputed_mttkrp(subs, vals, shape, B, F, n)
        assert np.max(np.abs(got - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref))), n
    # before the first imputation B = 0: the imputed tensor is full(S) itself
    Z0 = [np.zeros_like(b) for b in B]
    for n in range(len(shape)):
        assert np.allclose(imputed_mttkrp(subs, vals, shape, Z0, F, n), dense_mttkrp(S, F, n), rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize('shape', [(9, 7), (7, 6, 5), (6, 5, 4, 3)])
def test_telescoped_norm_and_f_rel_missing_terms(shape):
    rng = np.random.RandomState(10 + len(shape))
    R = 4
    subs, vals, W = random_pattern(shape, 0.4, rng)
    B = [rng.randn(s, R) for s in shape]
    A = [rng.randn(s, R) for s in shape]
    MA, MB = full_cp(A), full_cp(B)
    assert abs(telescoped_diff2(A, B) - np.sum((MA - MB) ** 2)) <= 1e-11 * np.sum((MA - MB) ** 2)
    assert abs(model_norm2(B) - np.sum(MB ** 2)) <= 1e-12 * np.sum(MB ** 2)
    # f_rel_missing terms of the dense path (em.cuh: [0] sum_missing (m'-x)^2, [1] sum_missing x^2 with x = m there)
    m_new, m_old = model_at(subs, A), model_at(subs, B)
    num = telescoped_diff2(A, B) - np.sum((m_new - m_old) ** 2)
    den = model_norm2(B) - np.sum(m_old ** 2)
    assert abs(num - np.sum(((MA - MB) ** 2)[~W])) <= 1e-10 * np.sum((MA - MB) ** 2)
    assert abs(den - np.sum((MB ** 2)[~W])) <= 1e-10 * np.sum(MB ** 2)
    # near convergence: ||M' - M||^2 ~ 1e-18 ||M||^2; the telescoped form keeps its relative accuracy where the
    # difference of two model norms has none left
    A2 = [b + 1e-9 * rng.randn(*b.shape) for b in B]
    direct = np.sum((full_cp(A2) - MB) ** 2)
    tele = telescoped_diff2(A2, B)
    assert abs(tele - direct) <= 1e-6 * direct, (tele, direct)
    naive = model_norm2(A2) - 2 * np.sum(full_cp(A2) * MB) + model_norm2(B)
    assert abs(naive - direct) > 1e-3 * direct   # what the telescoped form avoids


class _Problem:
    """One-object problem (2-way CP, 4 x 3, rank 2) flattened by hand into the C structs."""

    def __init__(self, c, miss=False, sparse=True):
        self.rows = np.asarray([4, 3], dtype=np.int64)
        self.rank = np.full(2, 2, dtype=np.int32)
        self.modes = np.arange(1, 3, dtype=np.int32)
        self.zero32 = np.zeros(2, dtype=np.int32)
        self.cons = (c.Constraint * 2)()
        self.mask = np.ones(12, dtype=np.uint8)
        self.dense = np.zeros(12)
        obj = c.Object()
        obj.model, obj.order, obj.weight, obj.znorm_const = 0, 2, 1.0, float('nan')
        obj.modes = self.modes.ctypes.data_as(c.c_int32_p)
        obj.shard_offset, obj.shard_extent = 0, 3
        obj.data = None if sparse else self.dense.ctypes.data_as(c.c_double_p)
        obj.miss = self.mask.ctypes.data_as(c.c_uint8_p) if miss else None
        self.objs = (c.Object * 1)(obj)
        pb = c.Problem()
        pb.nb_modes, pb.n_objects, pb.n_couplings = 2, 1, 0
        pb.mode_rows = self.rows.ctypes.data_as(c.c_int64_p)
        pb.mode_rank = self.rank.ctypes.data_as(c.c_int32_p)
        pb.n_slices = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.objects = self.objs
        pb.lin_coupled_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constrained_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constraints = self.cons
        self.pb = pb
        self.sparse = sparse

    def _so(self, c, nnz, subs, vals):
        subs = None if subs is None else np.asfortranarray(np.asarray(subs, dtype=np.int64))
        vals = None if vals is None else np.asarray(vals, dtype=np.float64)
        so = c.SparseObject()
        so.nnz = nnz
        so.subs = None if subs is None else subs.ctypes.data_as(c.c_int64_p)
        so.vals = None if vals is None else vals.ctypes.data_as(c.c_double_p)
        self._keep = getattr(self, '_keep', []) + [subs, vals, so]
        return so

    def create(self, c, subs, vals, mnnz, msubs, mvals):
        so = self._so(c, len(vals), subs, vals)
        mo = self._so(c, mnnz, msubs, mvals)
        sp = (ctypes.POINTER(c.SparseObject) * 1)(ctypes.pointer(so) if self.sparse else None)
        mk = (ctypes.POINTER(c.SparseObject) * 1)(ctypes.pointer(mo))
        dist = c.Dist()
        dist.rank, dist.world_size, dist.device = 0, 1, 0
        h = c.HandleP()
        rc = c.lib.aoadmm_create_sparse_masked(ctypes.byref(self.pb), sp, mk, ctypes.byref(dist), ctypes.byref(h))
        if h.value:
            c.lib.aoadmm_destroy(h)
        return rc


def test_create_sparse_masked_validates_before_touching_a_device(ab):
    c = ab._capi
    subs = np.array([[0, 0], [3, 2], [1, 1]])
    vals = np.array([1.0, 2.0, 0.0])          # an explicit zero is a stored (observed) entry
    ones = np.ones(3)
    assert c.lib.aoadmm_create_sparse_masked(None, None, None, None, None) == INVALID
    cases = [
        (dict(), -1, subs, ones, INVALID, 'negative'),
        (dict(), 3, None, ones, INVALID, 'NULL'),
        (dict(), 3, subs, None, INVALID, 'NULL'),
        (dict(), 3, [[0, 0], [4, 2], [1, 1]], ones, INVALID, 'out of range'),
        (dict(), 3, [[0, 0], [3, 3], [1, 1]], ones, INVALID, 'out of range'),
        (dict(sparse=False), 3, subs, ones, INVALID, 'dense'),
        (dict(miss=True), 3, subs, ones, INVALID, 'Z.miss'),
    ]
    for kw, mnnz, msubs, mvals, want, msg in cases:
        pr = _Problem(c, **kw)
        assert pr.create(c, subs, vals, mnnz, msubs, mvals) == want, (kw, mnnz, msubs)
        err = c.lib.aoadmm_last_error(None).decode()
        assert msg in err and 'mask' in err, (msg, err)
    if ab.device_count() == 0:   # well-formed descriptors get as far as the device
        assert _Problem(c).create(c, subs, vals, 3, subs, ones) == NO_DEVICE
        assert _Problem(c).create(c, subs, vals, 0, None, None) == NO_DEVICE   # the pattern is checked on the device


def _matrix_pair(I=30, J=25, M=20, R=3, seed=0, constraints=None, noise=0.1):
    """A matrix I x J coupled in its rows to a side matrix I x M (the CMTF structure of example_script6)."""
    rng = np.random.RandomState(seed)
    constraints = constraints or [None] * 4
    coupling = {'lin_coupled_modes': [1, 0, 1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 4}
    return pg._finish(['CP', 'CP'], [I, J, I, M], [[1, 2], [3, 4]], [[1.0] * R] * 2, [noise] * 2, coupling,
                      [pg.d_rand] * 4, [1 if c else 0 for c in constraints], constraints, [0.5, 0.5], rng)


def _mask_object(ab, X, frac, rng):
    """Observe a random fraction of X: (sptensor S, sparse mask, full(S), dense mask)."""
    W = rng.rand(*X.shape) < frac
    subs = np.argwhere(W).astype(np.int64)
    S = ab.sptensor(subs, X[W], X.shape)
    return S, ab.sptensor(subs, np.ones(subs.shape[0]), X.shape), np.asfortranarray(np.where(W, X, 0.0)), \
        np.asfortranarray(W)


def _masked_pair(ab, Z, objects, frac, seed):
    """Z with the chosen objects observed on a random pattern: (sparse form, dense form on full(S) + W)."""
    rng = np.random.RandomState(seed)
    P = len(Z['object'])
    os_, od, ms, md = list(Z['object']), list(Z['object']), [None] * P, [None] * P
    for p in objects:
        os_[p], ms[p], od[p], md[p] = _mask_object(ab, Z['object'][p], frac, rng)
    return dict(Z, object=os_, miss=ms), dict(Z, object=od, miss=md)


def test_python_refusals_happen_before_any_device_call(ab):
    Z, G, _ = _matrix_pair()
    Zs, Zd = _masked_pair(ab, Z, [0], 0.3, 0)
    zn = [float('nan'), pg.znorm_const(Z)[1]]
    opts = pg.default_options(MaxOuterIters=2)
    # a sparse mask on a dense object
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(dict(Zd, miss=[Zs['miss'][0], None]), pg.znorm_const(Zd), G, None, None, None, None, opts)
    assert e.value.status_name == 'INVALID_ARG' and 'dense' in str(e.value)
    # a dense mask on a sparse object keeps its refusal
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(dict(Zs, miss=[Zd['miss'][0], None]), zn, G, None, None, None, None, opts)
    assert e.value.status_name == 'UNSUPPORTED' and 'Z.miss' in str(e.value)
    # a sparse mask of the wrong shape
    bad = ab.sptensor(Zs['miss'][0].subs, Zs['miss'][0].vals, (30, 26))
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(dict(Zs, miss=[bad, None]), zn, G, None, None, None, None, opts)
    assert e.value.status_name == 'INVALID_ARG' and 'shape' in str(e.value)
    # several GPUs stay refused for sparse objects
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(Zs, zn, G, None, None, None, None, opts, n_gpus=2)
    assert e.value.status_name == 'UNSUPPORTED' and 'one GPU' in str(e.value)


# ---------------------------------------------------------------------------------------------- GPU
def _need_gpu(ab):
    assert ab.device_count() >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'


def _assert_missing_close(od, oo):
    n = oo['OuterIterations'] + 1
    a, b = od['func_rel_missing'][1:n], oo['func_rel_missing'][1:n]
    assert np.isnan(od['func_rel_missing'][0]) and np.max(np.abs(a - b)) < FIT_TOL
    assert abs(od['f_rel_missing'] - oo['f_rel_missing']) < FIT_TOL


def _zn(ab, Zs, Zd):
    zd = pg.znorm_const(Zd)
    return [float('nan') if ab.as_sparse(x) is not None else z for x, z in zip(Zs['object'], zd)], zd


def _check_against_oracle(ab, Zs, Zd, G, opts):
    zs, zd = _zn(ab, Zs, Zd)
    Go, oo = oracle_solve(Zd, zd, G, options=opts)
    Gd, od = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts)
    assert od['OuterIterations'] == oo['OuterIterations']
    assert od['exit_flag'] == oo['exit_flag']
    n = oo['OuterIterations'] + 1
    for key in ('func_val_conv', 'func_coupl_conv', 'func_constr_conv'):
        assert np.max(np.abs(od[key][:n] - oo[key][:n])) < FIT_TOL, key
    assert np.array_equal(od['innerIters'], oo['innerIters'])
    _assert_missing_close(od, oo)
    assert_state_close(Gd, Go)
    return od


def _assert_bitwise(Ga, Gb):
    for key in ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac'):
        for a, b in zip(Ga[key], Gb[key]):
            assert (a is None and b is None) or np.array_equal(a, b), key


@pytest.mark.gpu
@pytest.mark.parametrize('R', [1, 7, 32, 200])
def test_sparse_matrix_with_mask_coupled_to_dense_side_matrix(ab, R):
    _need_gpu(ab)
    nn = ('non-negativity',)
    Z, G, _ = _matrix_pair(I=260, J=220, M=230, R=R, seed=R, constraints=[nn, None, nn, None])
    Zs, Zd = _masked_pair(ab, Z, [0], 0.3, R)
    _check_against_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=12, **ZERO_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('sz,R', [((30, 25, 20), 7), ((30, 25, 20), 64), ((12, 10, 9, 8), 32)])
def test_sparse_tensor_with_mask_nonneg(ab, sz, R):
    _need_gpu(ab)
    Z, G, _ = pg.config_single_cp(sz=sz, R=R, seed=R, noise=0.1, constraints=[('non-negativity',)] * len(sz))
    Zs, Zd = _masked_pair(ab, Z, [0], 0.25, len(sz))
    _check_against_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=10, **ZERO_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('mode1', [('TV regularization',), ('simplex column-wise', 1.0)])
def test_column_wise_prox_on_a_masked_sparse_tensor(ab, mode1):
    _need_gpu(ab)
    Z, G, _ = pg.config_cp_tv(I=40, J=30, K=26, R=3, seed=4, mode1=mode1, eta=1e-3 if len(mode1) == 1 else 1.0)
    Zs, Zd = _masked_pair(ab, Z, [0], 0.3, 2)
    _check_against_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=15, **ZERO_TOL))


@pytest.mark.gpu
def test_default_tolerances_stop_on_f_rel_missing(ab):
    """Default tolerances on exact low-rank data: the objective falls below AbsFuncTol early, and the run goes on until
    the extra stopping condition f_rel_missing < OuterRelTol (:457-459) holds, in the same iteration as the oracle."""
    _need_gpu(ab)
    Z, G, _ = pg.config_single_cp(sz=(25, 20, 18), R=2, seed=2, noise=0.0, constraints=[('non-negativity',)] * 3)
    Zs, Zd = _masked_pair(ab, Z, [0], 0.7, 5)
    opts = pg.default_options(MaxOuterIters=1500)
    od = _check_against_oracle(ab, Zs, Zd, G, opts)
    n = od['OuterIterations']
    assert od['exit_flag'] != 0 and n < 1500
    assert od['f_rel_missing'] < opts['OuterRelTol'] <= od['func_rel_missing'][n - 1]
    assert np.min(od['func_val_conv'][:n]) < opts['AbsFuncTol']   # the objective alone would have stopped earlier


@pytest.mark.gpu
def test_dense_mask_and_sparse_mask_in_one_problem(ab):
    """A dense tensor with a dense Z.miss coupled to a sparse matrix with a sparse mask: the two kinds of missing-entry
    sums add up to one f_rel_missing."""
    _need_gpu(ab)
    Z, G, _ = pg.config_cp_matrix(40, 30, 20, 60, 5, seed=3)
    Zm = pg.add_missing(Z, 0.3, seed=1, objects=[0])
    Zs, Zd = _masked_pair(ab, Zm, [1], 0.2, 9)
    Zs['miss'][0] = Zm['miss'][0]
    Zd['miss'][0] = Zm['miss'][0]
    _check_against_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=15, **ZERO_TOL))


@pytest.mark.gpu
def test_dense_engine_agrees_over_two_consecutive_runs(ab):
    """A second run continues from the last imputation in both engines."""
    _need_gpu(ab)
    Z, G, _ = _matrix_pair(I=200, J=150, M=120, R=5, seed=1, constraints=[('non-negativity',)] * 4)
    Zs, Zd = _masked_pair(ab, Z, [0], 0.2, 3)
    zs, zd = _zn(ab, Zs, Zd)
    opts = pg.default_options(MaxOuterIters=8, **ZERO_TOL)
    outs = []
    for Zx, zx in ((Zs, zs), (Zd, zd)):
        with ab.Solver(dict(Zx, rank=[5, 5]), zx) as s:
            s.set_state(G)
            o1 = s.run(opts)
            o2 = s.run(opts)
            outs.append((o1, o2, s.get_state()))
    for a, b in zip(outs[0][:2], outs[1][:2]):
        assert np.max(np.abs(a['func_val_conv'] - b['func_val_conv'])) < FIT_TOL
        assert np.max(np.abs(a['func_rel_missing'][1:] - b['func_rel_missing'][1:])) < FIT_TOL
    assert outs[0][1]['func_rel_missing'][1] < outs[0][0]['func_rel_missing'][1]   # continued, not restarted
    assert_state_close(outs[0][2], outs[1][2])


@pytest.mark.gpu
def test_bit_identical_under_graph_replay_and_permutations(ab):
    _need_gpu(ab)
    Z, G, _ = pg.config_single_cp(sz=(40, 30, 25), R=6, seed=3, noise=0.1, constraints=[('non-negativity',)] * 3)
    Zs, _ = _masked_pair(ab, Z, [0], 0.2, 4)
    X, Mk = Zs['object'][0], Zs['miss'][0]
    zs = [float('nan')]
    opts = pg.default_options(MaxOuterIters=12, **ZERO_TOL)
    runs = [ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, dict(opts, graph=g)) for g in (1, -1, 1)]
    rng = np.random.RandomState(0)
    p1, p2 = rng.permutation(X.nnz), rng.permutation(Mk.nnz)
    Zp = dict(Zs, object=[ab.sptensor(X.subs[p1], X.vals[p1], X.shape)])
    Zq = dict(Zs, miss=[ab.sptensor(Mk.subs[p2], Mk.vals[p2], Mk.shape)])
    runs += [ab.cmtf_fun_AOADMM(Zx, zs, G, None, None, None, None, opts) for Zx in (Zp, Zq)]
    for Gx, ox in runs[1:]:
        _assert_bitwise(runs[0][0], Gx)
        assert np.array_equal(runs[0][1]['func_val_conv'], ox['func_val_conv'])
        assert np.array_equal(runs[0][1]['func_rel_missing'], ox['func_rel_missing'], equal_nan=True)


@pytest.mark.gpu
def test_pattern_mismatch_is_refused_by_create(ab):
    _need_gpu(ab)
    Z, G, _ = _matrix_pair()
    Zs, _ = _masked_pair(ab, dict(Z, rank=[3, 3]), [0], 0.3, 0)
    X, Mk = Zs['object'][0], Zs['miss'][0]
    zn = [float('nan'), pg.znorm_const(Z)[1]]
    variants = [ab.sptensor(Mk.subs[1:], Mk.vals[1:], Mk.shape),                        # one stored entry unobserved
                ab.sptensor(Mk.subs, np.r_[0.0, Mk.vals[1:]], Mk.shape),                # ... as an explicit zero
                ab.sptensor(np.vstack([Mk.subs, [[0, 0]] if not np.any(np.all(X.subs == 0, axis=1)) else [[1, 0]]]),
                            np.r_[Mk.vals, 1.0], Mk.shape)]                             # an unstored entry observed
    for bad in variants:
        with pytest.raises(ab.AoadmmError) as e:
            ab.Solver(dict(Zs, miss=[bad, None]), zn)
        assert e.value.status_name == 'UNSUPPORTED' and 'object 1' in str(e.value)
    # duplicates that merge to a nonzero are one observed entry
    dup = ab.sptensor(np.vstack([Mk.subs, Mk.subs[:5]]), np.r_[Mk.vals, np.ones(5)], Mk.shape)
    with ab.Solver(dict(Zs, miss=[dup, None]), zn) as s:
        s.set_state(G)
        assert s.run(pg.default_options(MaxOuterIters=2))['OuterIterations'] == 2


@pytest.mark.gpu
def test_large_low_rank_completion_known_answer(ab):
    """20000 x 15000, rank 8, 5 % observed, low noise: far beyond the dense oracle (3e8 entries).  EM imputation
    (cmtf_fun_AOADMM.m:408-441) recovers the held-out entries with correlation > 0.99 and f_rel_missing decreases."""
    _need_gpu(ab)
    rng = np.random.RandomState(7)
    I, J, R = 20000, 15000, 8
    A, B = rng.randn(I, R), rng.randn(J, R)
    n_obs, n_test = int(0.05 * I * J), 200000
    flat = np.unique(rng.randint(0, I * J, size=int(1.2 * (n_obs + n_test))))   # ~3 % of the draws collide
    flat = flat[rng.permutation(flat.size)[:n_obs + n_test]]
    assert flat.size == n_obs + n_test
    ii, jj = flat // J, flat % J
    vals = np.einsum('er,er->e', A[ii], B[jj])
    vals_noisy = vals + 1e-3 * np.std(vals) * rng.randn(vals.size)
    subs = np.stack([ii[:n_obs], jj[:n_obs]], axis=1).astype(np.int64)
    X = ab.sptensor(subs, vals_noisy[:n_obs], (I, J))
    Mk = ab.sptensor(subs, np.ones(n_obs), (I, J))
    Z = {'loss_function': ['Frobenius'], 'model': ['CP'], 'modes': [[1, 2]], 'size': [I, J],
         'coupling': {'lin_coupled_modes': [0, 0], 'coupling_type': [], 'coupl_trafo_matrices': [None] * 2},
         'constrained_modes': [0, 0], 'constraints': [None, None], 'weights': [1.0], 'object': [X], 'miss': [Mk],
         'rank': [R]}
    G = {'fac': [rng.randn(I, R), rng.randn(J, R)], 'constraint_fac': [None, None], 'constraint_dual_fac': [None, None],
         'coupling_dual_fac': [None, None], 'coupling_fac': []}
    Gd, od = ab.cmtf_fun_AOADMM(Z, [float('nan')], G, None, None, None, None,
                                pg.default_options(MaxOuterIters=200, **ZERO_TOL))
    pred = np.einsum('er,er->e', Gd['fac'][0][ii[n_obs:]], Gd['fac'][1][jj[n_obs:]])
    corr = np.corrcoef(pred, vals[n_obs:])[0, 1]
    assert corr > 0.99, corr
    frm = od['func_rel_missing']
    assert np.all(np.isfinite(frm[1:])) and frm[-1] < 0.1 * frm[1], frm[[1, 2, -1]]
