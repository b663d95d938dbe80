"""Sparse (COO) CP objects: aoadmm_create_sparse, the deterministic sparse MTTKRP and full solves.

CPU tests check a COO restatement of the sptensor mttkrp against the dense oracle, the ctypes mirror and every refusal
that happens before a device is touched; GPU tests (-m gpu) check the device MTTKRP against that restatement and whole
solves against the dense oracle on full(X) (north-star tolerances: factors 1e-8 relative Frobenius, objective 1e-10)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import problem_gen as pg
from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
from oracle.tensor_ops import mttkrp as dense_mttkrp
from _cases import FIT_TOL, ZERO_TOL, assert_state_close, rel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sparse_mttkrp(subs, vals, shape, U, n):
    """Reference for the device: the Tensor Toolbox sptensor `mttkrp(X,U,n)` restated in COO form (0-based n).  Every
    nonzero adds val * prod_{m != n} U[m][i_m, :] to row i_n; duplicate subscripts add up, as in the sptensor
    constructor.  `subs` is nnz x N (0-based), `vals` nnz values.  Checked against the dense oracle below."""
    subs = np.asarray(subs, dtype=np.int64).reshape(-1, len(shape))
    vals = np.asarray(vals, dtype=np.float64).reshape(-1)
    contrib = np.repeat(vals[:, None], U[0].shape[1], axis=1)
    for m in range(len(shape)):
        if m != n:
            contrib = contrib * np.asarray(U[m])[subs[:, m], :]
    out = np.zeros((shape[n], U[0].shape[1]))
    np.add.at(out, subs[:, n], contrib)
    return out


def random_coo(shape, nnz, rng, dup=0, empty=()):
    """nnz uniform nonzeros (plus `dup` repeated subscripts); modes listed in `empty` keep index 0 free."""
    subs = np.stack([rng.randint(1 if d in empty else 0, s, size=nnz) for d, s in enumerate(shape)], axis=1)
    if dup:
        subs = np.vstack([subs, subs[rng.randint(0, nnz, size=dup)]])
    return subs.astype(np.int64), rng.randn(subs.shape[0])


def sparsify(X, frac, rng):
    """Keep a random fraction of the entries of a dense array: (sptensor, dense array with the others zeroed)."""
    import aoadmm_b200 as ab
    mask = rng.rand(*X.shape) < frac
    return ab.sptensor(np.argwhere(mask), X[mask], X.shape), np.asfortranarray(X * mask)


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('shape', [(7, 5), (6, 5, 4), (5, 4, 3, 6)])
def test_coo_reference_mttkrp_equals_dense_oracle(ab, shape):
    rng = np.random.RandomState(len(shape))
    subs, vals = random_coo(shape, 40, rng, dup=10, empty=(0,))   # duplicates (summed) and an empty first row / slice
    X = ab.sptensor(subs, vals, shape).full()
    assert np.all(X[0] == 0)
    U = [rng.randn(s, 3) for s in shape]
    for n in range(len(shape)):
        ref = dense_mttkrp(X, U, n)
        got = sparse_mttkrp(subs, vals, shape, U, n)
        assert np.max(np.abs(got - ref)) <= 1e-13 * max(1.0, np.max(np.abs(ref))), n


def test_sparse_object_struct_layout_matches_header(ab, tmp_path):
    cls = ab._capi.SparseObject
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "aoadmm.h"', 'int main(void){',
             'printf("size %zu\\n", sizeof(aoadmm_sparse_object));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(aoadmm_sparse_object, %s));' % (fname, fname))
    lines.append('return 0;}')
    src = tmp_path / 'sp.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'sp'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got['size']) == ctypes.sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(got[fname]) == getattr(cls, fname).offset, fname


class _Problem:
    """A one-object problem (3-way CP, 4 x 3 x 2, rank 2) flattened by hand into the C structs."""

    def __init__(self, c, model=0, miss=False, data=False, rows=(4, 3, 2)):
        self.rows = np.asarray(rows, dtype=np.int64)
        self.rank = np.full(3, 2, dtype=np.int32)
        self.modes = np.arange(1, 4, dtype=np.int32)
        self.zero32 = np.zeros(3, dtype=np.int32)
        self.cons = (c.Constraint * 3)()
        self.mask = np.ones(int(np.prod(rows[:3])) if max(rows) < 1 << 20 else 1, dtype=np.uint8)
        self.dense = np.zeros(self.mask.size)
        obj = c.Object()
        obj.model, obj.order, obj.weight, obj.znorm_const = model, 3, 1.0, float('nan')
        obj.modes = self.modes.ctypes.data_as(c.c_int32_p)
        obj.shard_offset, obj.shard_extent = 0, int(rows[2])
        obj.data = self.dense.ctypes.data_as(c.c_double_p) if data else None
        obj.miss = self.mask.ctypes.data_as(c.c_uint8_p) if miss else None
        self.objs = (c.Object * 1)(obj)
        pb = c.Problem()
        pb.nb_modes, pb.n_objects, pb.n_couplings = 3, 1, 0
        pb.mode_rows = self.rows.ctypes.data_as(c.c_int64_p)
        pb.mode_rank = self.rank.ctypes.data_as(c.c_int32_p)
        pb.n_slices = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.objects = self.objs
        pb.lin_coupled_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constrained_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constraints = self.cons
        self.pb = pb

    def create(self, c, nnz, subs, vals, world_size=1):
        self.subs = None if subs is None else np.asfortranarray(np.asarray(subs, dtype=np.int64))
        self.vals = None if vals is None else np.asarray(vals, dtype=np.float64)
        so = c.SparseObject()
        so.nnz = nnz
        so.subs = None if self.subs is None else self.subs.ctypes.data_as(c.c_int64_p)
        so.vals = None if self.vals is None else self.vals.ctypes.data_as(c.c_double_p)
        self.so = so
        arr = (ctypes.POINTER(c.SparseObject) * 1)(ctypes.pointer(so))
        dist = c.Dist()
        dist.rank, dist.world_size, dist.device = 0, world_size, 0
        h = c.HandleP()
        rc = c.lib.aoadmm_create_sparse(ctypes.byref(self.pb), arr, ctypes.byref(dist), ctypes.byref(h))
        if h.value:
            c.lib.aoadmm_destroy(h)
        return rc


def test_create_sparse_validates_before_touching_a_device(ab):
    c = ab._capi
    ok_subs = np.array([[0, 0, 0], [3, 2, 1], [1, 1, 1]])
    ok_vals = np.array([1.0, 2.0, 3.0])
    INVALID, UNSUPPORTED, NO_DEVICE = 1, 2, 8
    assert c.lib.aoadmm_create_sparse(None, None, None, None) == INVALID
    h = c.HandleP()
    assert c.lib.aoadmm_create_sparse(None, None, None, ctypes.byref(h)) == INVALID and not h.value
    cases = [
        (dict(), -1, ok_subs, ok_vals, 1, INVALID, 'negative'),
        (dict(), 3, None, ok_vals, 1, INVALID, 'NULL'),
        (dict(), 3, ok_subs, None, 1, INVALID, 'NULL'),
        (dict(), 3, [[0, 0, 0], [4, 2, 1], [1, 1, 1]], ok_vals, 1, INVALID, 'out of range'),
        (dict(), 3, [[0, 0, 0], [3, 2, 1], [1, -1, 1]], ok_vals, 1, INVALID, 'out of range'),
        (dict(), 3, [[0, 0, 0], [3, 2, 2], [1, 1, 1]], ok_vals, 1, INVALID, 'out of range'),
        (dict(data=True), 3, ok_subs, ok_vals, 1, INVALID, 'both'),
        (dict(rows=(1 << 31, 3, 2)), 3, ok_subs, ok_vals, 1, INVALID, '2^31'),
        (dict(miss=True), 3, ok_subs, ok_vals, 1, UNSUPPORTED, 'Z.miss'),
        (dict(model=1), 3, ok_subs, ok_vals, 1, UNSUPPORTED, 'PARAFAC2'),
        (dict(), 3, ok_subs, ok_vals, 2, UNSUPPORTED, 'one GPU'),
    ]
    for kw, nnz, subs, vals, world, want, msg in cases:
        pr = _Problem(c, **kw)
        assert pr.create(c, nnz, subs, vals, world) == want, (kw, nnz, subs, world)
        assert msg in c.lib.aoadmm_last_error(None).decode(), (msg, c.lib.aoadmm_last_error(None))
    if ab.device_count() == 0:   # a well-formed descriptor gets as far as the device
        assert _Problem(c).create(c, 3, ok_subs, ok_vals) == NO_DEVICE
        assert _Problem(c).create(c, 0, None, None) == NO_DEVICE


def _sparse_script6(ab, frac=0.3, seed=0, sz=(20, 18, 16, 20, 22, 18, 24)):
    Z, G, _ = pg.config_script6(seed=seed, sz=sz)
    Xs, Xd = sparsify(Z['object'][0], frac, np.random.RandomState(seed + 100))
    return dict(Z, object=[Xs] + Z['object'][1:]), dict(Z, object=[Xd] + Z['object'][1:]), G


def test_solver_refuses_unsupported_sparse_combinations_before_any_device_call(ab):
    Zs, Zd, G = _sparse_script6(ab)
    zn = [float('nan')] + pg.znorm_const(Zd)[1:]
    opts = pg.default_options(MaxOuterIters=2)
    for dist, msg in ((dict(n_gpus=2), 'one GPU'), (dict(world_size=2, rank=0), 'one GPU')):
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_fun_AOADMM(Zs, zn, G, None, None, None, None, opts, **dist)
        assert e.value.status_name == 'UNSUPPORTED' and msg in str(e.value)
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(dict(Zs, miss=[np.ones(Zd['object'][0].shape), None, None]), zn, G, None, None, None, None, opts)
    assert e.value.status_name == 'UNSUPPORTED' and 'Z.miss' in str(e.value)
    Zp, Gp, _ = pg.config_single_par2(I=6, Jk=(5, 4), R=2, seed=0)
    sl = [sparsify(x, 0.5, np.random.RandomState(k))[0] for k, x in enumerate(Zp['object'][0])]
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(dict(Zp, object=[sl]), [float('nan')], Gp, None, None, None, None, opts)
    assert e.value.status_name == 'UNSUPPORTED' and 'PARAFAC2' in str(e.value)
    bad = ab.sptensor(Zs['object'][0].subs, Zs['object'][0].vals, (20, 18, 17))
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(dict(Zs, object=[bad] + Zs['object'][1:]), zn, G, None, None, None, None, opts)
    assert e.value.status_name == 'INVALID_ARG'
    # nvecs needs a dense unfolding (cmtf_nvecs.m refuses sparse input too)
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_nvecs(Zs, 2, 3)
    assert e.value.status_name == 'UNSUPPORTED'
    io = {'lambdas_init': [[1.0] * 3] * 3, 'nvecs': 1, 'distr': [pg.d_rand] * 7, 'normalize': 1}
    with pytest.raises(ab.AoadmmError) as e:
        ab.init_coupled_AOADMM_CMTF(Zs, io)
    assert e.value.status_name == 'UNSUPPORTED'


def test_scipy_sparse_matrix_is_recognised_by_duck_typing(ab):
    sps = pytest.importorskip('scipy.sparse')
    Y = sps.random(9, 7, density=0.3, format='csr', random_state=1)
    s = ab.as_sparse(Y)
    assert s.shape == (9, 7) and s.nnz == Y.nnz
    assert np.array_equal(s.full(), Y.toarray())
    assert ab.as_sparse(np.zeros((3, 3))) is None and ab.as_sparse([[1.0]]) is None


# ---------------------------------------------------------------------------------------------- GPU
def _need_gpu(ab):
    assert ab.device_count() >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'


def _single_object_Z(X, R):
    N = X.ndim
    return {'loss_function': ['Frobenius'], 'model': ['CP'], 'modes': [list(range(1, N + 1))], 'size': list(X.shape),
            'coupling': {'lin_coupled_modes': [0] * N, 'coupling_type': [], 'coupl_trafo_matrices': [None] * N},
            'constrained_modes': [0] * N, 'constraints': [None] * N, 'weights': [1.0], 'object': [X], 'rank': [R]}


def _device_mttkrps(ab, X, U, precision=0):
    with ab.Solver(_single_object_Z(X, U[0].shape[1]), [float('nan')]) as s:
        s.set_state({'fac': U})
        return [s.object_mttkrp(1, n + 1, precision) for n in range(X.ndim)]


def _coo_case(kind, shape, rng):
    if kind == 'uniform':
        return random_coo(shape, 3000, rng, dup=50)
    if kind == 'skewed':    # one row of mode 1 holds half of the nonzeros (the row spans many units of work)
        subs, vals = random_coo(shape, 6000, rng)
        subs[::2, 0] = 1
        return subs, vals
    if kind == 'empty':     # empty rows in every mode and an empty last slice
        subs, vals = random_coo(shape, 500, rng, empty=tuple(range(len(shape))))
        subs[:, -1] = np.minimum(subs[:, -1], shape[-1] - 2)
        return subs, vals
    return np.zeros((0, len(shape)), dtype=np.int64), np.zeros(0)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(300, 200), (40, 30, 20), (12, 10, 9, 8)])
@pytest.mark.parametrize('R', [1, 7, 32, 64, 200])
@pytest.mark.parametrize('kind', ['uniform', 'skewed', 'empty', 'nnz0'])
def test_sparse_mttkrp_matches_oracle(ab, shape, R, kind):
    _need_gpu(ab)
    rng = np.random.RandomState(sum(shape) + R)
    subs, vals = _coo_case(kind, shape, rng)
    U = [rng.randn(s, R) for s in shape]
    got = _device_mttkrps(ab, ab.sptensor(subs, vals, shape), U)
    for n in range(len(shape)):
        ref = sparse_mttkrp(subs, vals, shape, U, n)
        if kind == 'nnz0':
            assert np.all(got[n] == 0), n
        else:
            assert rel(got[n], ref) <= 1e-12, (n, rel(got[n], ref))


@pytest.mark.gpu
def test_sparse_mttkrp_large_skewed_row_and_permutation_invariance(ab):
    """A row with half of 200k nonzeros spans hundreds of units; a permutation of the input gives identical bits."""
    _need_gpu(ab)
    rng = np.random.RandomState(5)
    shape, R = (500, 400, 300), 32
    subs, vals = random_coo(shape, 200000, rng)
    subs[::2, 1] = 7
    subs, idx = np.unique(subs, axis=0, return_index=True)
    vals = vals[idx]
    U = [rng.rand(s, R) for s in shape]
    a = _device_mttkrps(ab, ab.sptensor(subs, vals, shape), U)
    perm = rng.permutation(vals.size)
    b = _device_mttkrps(ab, ab.sptensor(subs[perm], vals[perm], shape), U)
    for n in range(3):
        assert rel(a[n], sparse_mttkrp(subs, vals, shape, U, n)) <= 1e-12
        assert np.array_equal(a[n], b[n]), n


def _solve_pair(ab, Zs, Zd, G, opts):
    """device on the sparse objects (Znorm_const of a sparse object computed on the device) vs oracle on full(X)"""
    zn = pg.znorm_const(Zd)
    zs = [float('nan') if ab.as_sparse(x) is not None else z for x, z in zip(Zs['object'], zn)]
    Go, oo = oracle_solve(Zd, zn, G, options=opts)
    Gd, od = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts)
    return Go, oo, Gd, od


def _assert_close(Go, oo, Gd, od):
    assert od['OuterIterations'] == oo['OuterIterations']
    n = oo['OuterIterations'] + 1
    for key in ('func_val_conv', 'func_coupl_conv', 'func_constr_conv'):
        assert np.max(np.abs(od[key][:n] - oo[key][:n])) < FIT_TOL, key
    assert np.array_equal(od['innerIters'], oo['innerIters'])
    assert_state_close(Gd, Go)


def _assert_bitwise(Ga, Gb):
    for key in ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac'):
        for a, b in zip(Ga[key], Gb[key]):
            assert (a is None and b is None) or np.array_equal(a, b), key


@pytest.mark.gpu
def test_sparse_example_script6_structure(ab):
    _need_gpu(ab)
    Zs, Zd, G = _sparse_script6(ab, frac=0.2, sz=(50, 60, 40, 50, 70, 60, 80))
    _assert_close(*_solve_pair(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=40)))


@pytest.mark.gpu
def test_dense_tensor_coupled_to_sparse_matrix(ab):
    _need_gpu(ab)
    sps = pytest.importorskip('scipy.sparse')
    Z, G, _ = pg.config_cp_matrix(40, 30, 20, 60, 5, seed=3)
    _, Yd = sparsify(Z['object'][1], 0.1, np.random.RandomState(7))
    Zs = dict(Z, object=[Z['object'][0], sps.csr_matrix(Yd)])
    Zd = dict(Z, object=[Z['object'][0], Yd])
    _assert_close(*_solve_pair(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=25, **ZERO_TOL)))


@pytest.mark.gpu
def test_four_way_sparse_cp(ab):
    _need_gpu(ab)
    Z, G, _ = pg.config_single_cp(sz=(14, 12, 10, 9), R=4, seed=9, noise=0.1, constraints=[('non-negativity',)] * 4)
    Xs, Xd = sparsify(Z['object'][0], 0.25, np.random.RandomState(1))
    _assert_close(*_solve_pair(ab, dict(Z, object=[Xs]), dict(Z, object=[Xd]), G,
                               pg.default_options(MaxOuterIters=20, **ZERO_TOL)))


@pytest.mark.gpu
@pytest.mark.parametrize('mode1', [('TV regularization',), ('simplex column-wise', 1.0)])
def test_non_elementwise_prox_on_a_sparse_object(ab, mode1):
    _need_gpu(ab)
    Z, G, _ = pg.config_cp_tv(I=40, J=30, K=26, R=3, seed=4, mode1=mode1, eta=1e-3 if len(mode1) == 1 else 1.0)
    Xs, Xd = sparsify(Z['object'][0], 0.3, np.random.RandomState(2))
    _assert_close(*_solve_pair(ab, dict(Z, object=[Xs]), dict(Z, object=[Xd]), G,
                               pg.default_options(MaxOuterIters=20, **ZERO_TOL)))


@pytest.mark.gpu
def test_type4_linear_coupling_with_a_sparse_tensor(ab):
    _need_gpu(ab)
    Z, G, _ = pg.config_linear_coupling(4, seed=4)
    Xs, Xd = sparsify(Z['object'][0], 0.3, np.random.RandomState(3))
    _assert_close(*_solve_pair(ab, dict(Z, object=[Xs] + Z['object'][1:]), dict(Z, object=[Xd] + Z['object'][1:]), G,
                               pg.default_options(MaxOuterIters=20, **ZERO_TOL)))


@pytest.mark.gpu
def test_graph_replay_and_repeated_runs_are_bit_identical(ab):
    _need_gpu(ab)
    Zs, Zd, G = _sparse_script6(ab, frac=0.2)
    zs = [float('nan')] + pg.znorm_const(Zd)[1:]
    opts = pg.default_options(MaxOuterIters=12, **ZERO_TOL)
    runs = [ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, dict(opts, graph=g)) for g in (1, -1, 1)]
    for Gx, ox in runs[1:]:
        _assert_bitwise(runs[0][0], Gx)
        assert np.array_equal(runs[0][1]['func_val_conv'], ox['func_val_conv'])


@pytest.mark.gpu
def test_permuted_nonzeros_give_bit_identical_factors_and_dense_engine_agrees(ab):
    _need_gpu(ab)
    Zs, Zd, G = _sparse_script6(ab, frac=0.2, seed=3)
    X = Zs['object'][0]
    perm = np.random.RandomState(0).permutation(X.nnz)
    Zp = dict(Zs, object=[ab.sptensor(X.subs[perm], X.vals[perm], X.shape)] + Zs['object'][1:])
    zn = pg.znorm_const(Zd)
    zs = [float('nan')] + zn[1:]
    opts = pg.default_options(MaxOuterIters=15, **ZERO_TOL)
    Ga, oa = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts)
    Gb, ob = ab.cmtf_fun_AOADMM(Zp, zs, G, None, None, None, None, opts)
    _assert_bitwise(Ga, Gb)
    assert np.array_equal(oa['func_val_conv'], ob['func_val_conv'])
    Gd, od = ab.cmtf_fun_AOADMM(Zd, zn, G, None, None, None, None, opts)   # the dense engine on full(X)
    assert np.max(np.abs(oa['func_val_conv'] - od['func_val_conv'])) < FIT_TOL
    assert_state_close(Ga, Gd)


@pytest.mark.gpu
def test_reduced_precision_option_leaves_sparse_objects_in_fp64(ab):
    """A problem mixing a sparse tensor and a dense matrix run with mttkrp_precision = 1: the dense objects take the
    option, the sparse object's MTTKRP stays FP64 (bit-identical to precision 0)."""
    _need_gpu(ab)
    Z, G, _ = pg.config_cp_matrix(40, 30, 20, 60, 5, seed=3)
    Xs, Xd = sparsify(Z['object'][0], 0.3, np.random.RandomState(4))
    Zs = dict(Z, object=[Xs, Z['object'][1]], rank=[5, 5])
    zs = [float('nan'), pg.znorm_const(Z)[1]]
    with ab.Solver(Zs, zs) as s:
        s.set_state(G)
        out = s.run(pg.default_options(MaxOuterIters=5, mttkrp_precision=1))
        assert out['OuterIterations'] == 5 and np.all(np.isfinite(out['func_val_conv']))
        for pos in (1, 2, 3):
            assert np.array_equal(s.object_mttkrp(1, pos, 1), s.object_mttkrp(1, pos, 0)), pos
        Gs = s.get_state()
        U = [Gs['fac'][m - 1] for m in Zs['modes'][0]]
        assert rel(s.object_mttkrp(1, 1, 0), sparse_mttkrp(Xs.subs, Xs.vals, Xs.shape, U, 0)) <= 1e-12
        assert s.time_mttkrp(1, 1, 2) > 0 and s.launch_count() > 0 and s.last_run_ms() > 0
        assert s.phase_ms()[0] > 0
        for call in (lambda: s.nvecs(1, 2), lambda: s.get_object_data(1, np.zeros(Xd.shape, order='F')),
                     lambda: s.generate_cp_data(1, U, 0.1, 1)):
            with pytest.raises(ab.AoadmmError) as e:
                call()
            assert e.value.status_name == 'UNSUPPORTED' and 'sparse' in str(e.value)
