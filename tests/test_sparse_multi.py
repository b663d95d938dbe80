"""Sparse objects on several GPUs from one caller: aoadmm_sparse_shard_bounds and aoadmm_create_sparse_multi.

CPU tests check the slab rule against a NumPy restatement, every status returned before a device is touched, the Python
refusals, the header / ctypes signatures and a NumPy model of how the masked EM sums are assembled from slabs.  GPU
tests (-m gpu) need two or more GPUs for the sharded runs (they skip otherwise) and compare against the oracle on
full(X) and against the one-GPU sparse engine; the n_gpus = 1 identity needs one GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import problem_gen as pg
from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
from _cases import FAC_TOL, FIT_TOL, ZERO_TOL, assert_state_close, rel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID, UNSUPPORTED, NO_DEVICE = 1, 2, 8


# ---------------------------------------------------------------------------------------------- the slab rule
def np_bounds(last, ext, n):
    """The rule of aoadmm_sparse_shard_bounds restated: c[k] entries with last subscript k, C[k] = sum_{j<k} c[j],
    b_r = the smallest k with C[k] * n >= r * nnz, clamped to [b_{r-1} + 1, ext - (n - r)]; nnz = 0: ext * r // n."""
    last = np.asarray(last, dtype=np.int64)
    nnz = last.size
    b = [0]
    C = np.concatenate([[0], np.cumsum(np.bincount(last, minlength=ext))]).astype(np.int64)
    for r in range(1, n):
        k = ext * r // n if nnz == 0 else int(np.argmax(C * n >= r * nnz))
        b.append(min(max(k, b[-1] + 1), ext - (n - r)))
    return np.array(b + [ext], dtype=np.int64)


def c_bounds(ab, subs, ext, n):
    c = ab._capi
    subs = np.asfortranarray(np.asarray(subs, dtype=np.int64))
    so = c.SparseObject()
    so.nnz, so.subs, so.vals = subs.shape[0], subs.ctypes.data_as(c.c_int64_p), None
    b = np.zeros(n + 1, dtype=np.int64)
    rc = c.lib.aoadmm_sparse_shard_bounds(ctypes.byref(so), subs.shape[1], ext, n, b.ctypes.data_as(c.c_int64_p))
    return rc, b


def _subs(kind, shape, nnz, rng):
    subs = np.stack([rng.randint(0, s, size=nnz) for s in shape], axis=1).astype(np.int64)
    ext = shape[-1]
    if kind == 'powerlaw':     # the generator of tools/sparse_bench.py: extent * u^3
        subs[:, -1] = np.minimum((ext * rng.rand(nnz) ** 3).astype(np.int64), ext - 1)
    elif kind == 'one_index':
        subs[:, -1] = ext // 3
    elif kind == 'skew40':     # one index with 40 % of the entries
        subs[rng.rand(nnz) < 0.4, -1] = 1
    return subs


@pytest.mark.parametrize('kind', ['uniform', 'powerlaw', 'one_index', 'skew40'])
@pytest.mark.parametrize('n', [1, 2, 3, 8])
def test_shard_bounds_match_numpy(ab, kind, n):
    rng = np.random.RandomState(n)
    for shape, nnz in (((30, 20, 64), 5000), ((40, 17), 999), ((5, 4, 3, 9), 200)):
        if shape[-1] < n:
            continue
        subs = _subs(kind, shape, nnz, rng)
        rc, b = c_bounds(ab, subs, shape[-1], n)
        assert rc == 0 and np.array_equal(b, np_bounds(subs[:, -1], shape[-1], n)), (kind, shape, b)
        assert np.all(np.diff(b) >= 1)
        perm = rng.permutation(nnz)      # the bounds depend on the multiset of subscripts only
        assert np.array_equal(c_bounds(ab, subs[perm], shape[-1], n)[1], b)
        S = ab.sptensor(subs, np.ones(nnz), shape)
        assert np.array_equal(ab.sparse_shard_bounds(S, n), b)


def test_shard_bounds_edge_cases(ab):
    rng = np.random.RandomState(0)
    empty = np.zeros((0, 3), dtype=np.int64)
    for ext, n in ((10, 3), (7, 7), (5, 1)):
        rc, b = c_bounds(ab, empty, ext, n)
        assert rc == 0 and np.array_equal(b, [ext * r // n for r in range(n + 1)])
    subs = _subs('uniform', (6, 5, 9), 300, rng)
    rc, b = c_bounds(ab, subs, 9, 9)                # N = ext: one index per GPU
    assert rc == 0 and np.array_equal(b, np.arange(10))
    rc, b = c_bounds(ab, subs, 9, 1)
    assert rc == 0 and np.array_equal(b, [0, 9])
    subs[:, -1] = 0                                   # everything at index 0: the other GPUs get one index each
    rc, b = c_bounds(ab, subs, 9, 4)
    assert rc == 0 and np.array_equal(b, np_bounds(subs[:, -1], 9, 4)) and np.array_equal(b, [0, 1, 2, 3, 9])
    # s2's last mode: the first 1/8 of the indices holds half of the nonzeros under uniform slabs
    big = _subs('powerlaw', (4, 4, 1 << 14), 200000, rng)
    b = c_bounds(ab, big, 1 << 14, 8)[1]
    share = np.diff(np.searchsorted(np.sort(big[:, -1]), b))
    assert share.max() < 0.14 * big.shape[0] and np.sum(big[:, -1] < (1 << 11)) > 0.45 * big.shape[0]
    rc, _ = c_bounds(ab, subs, 3, 4)
    assert rc == INVALID and 'fewer indices' in ab._capi.lib.aoadmm_last_error(None).decode()
    bad = subs.copy()
    bad[5, -1] = 9
    assert c_bounds(ab, bad, 9, 2)[0] == INVALID
    assert c_bounds(ab, subs, 9, 0)[0] == INVALID
    c = ab._capi
    assert c.lib.aoadmm_sparse_shard_bounds(None, 3, 9, 2, None) == INVALID
    with pytest.raises(ab.AoadmmError) as e:
        ab.sparse_shard_bounds(ab.sptensor(subs, np.ones(300), (6, 5, 3)), 4)
    assert e.value.status_name == 'INVALID_ARG'


# ---------------------------------------------------------------------------------------------- ABI
def test_header_and_ctypes_signatures(ab):
    c = ab._capi
    hdr = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    SO = ctypes.POINTER(c.SparseObject)
    want = {
        'aoadmm_sparse_shard_bounds': (
            r'int aoadmm_sparse_shard_bounds\(const aoadmm_sparse_object \*so, int32_t order, int64_t extent, '
            r'int32_t n_gpus,\s+int64_t \*bounds\);', [SO, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, c.c_int64_p]),
        'aoadmm_create_sparse_multi': (
            r'int aoadmm_create_sparse_multi\(const aoadmm_problem \*problem, const aoadmm_sparse_object \*const \*sparse,'
            r'\s+const aoadmm_sparse_object \*const \*masks, int32_t n_gpus, const int32_t \*devices,\s+'
            r'aoadmm_handle \*\*out\);', [ctypes.POINTER(c.Problem), ctypes.POINTER(SO), ctypes.POINTER(SO),
                                          ctypes.c_int32, c.c_int32_p, ctypes.POINTER(c.HandleP)]),
    }
    for name, (proto, argtypes) in want.items():
        assert re.search(proto, hdr), name
        assert name in c.EXPORTS
        assert list(getattr(c.lib, name).argtypes) == argtypes, name


class _Problem:
    """A 3-way CP object (6 x 5 x 4, rank 2), sparse unless dense=True, plus an optional dense 6 x 3 matrix."""

    def __init__(self, c, model=0, dense=False, miss=False, with_matrix=False, rows=(6, 5, 4)):
        self.rows = np.asarray(list(rows) + [3], dtype=np.int64)
        self.rank = np.full(4, 2, dtype=np.int32)
        self.m1, self.m2 = np.arange(1, 4, dtype=np.int32), np.asarray([1, 4], dtype=np.int32)
        self.zero32 = np.zeros(4, dtype=np.int32)
        self.lin = np.asarray([1, 0, 0, 1] if with_matrix else [0] * 4, dtype=np.int32)
        self.ctype = np.zeros(1, dtype=np.int32)
        self.cons = (c.Constraint * 4)()
        self.dense = np.zeros(int(np.prod(rows)))
        self.mask = np.ones(self.dense.size, dtype=np.uint8)
        self.mat = np.zeros(rows[0] * 3)
        objs = (c.Object * 2)()
        o = objs[0]
        o.model, o.order, o.weight, o.znorm_const = model, 3, 1.0, float('nan')
        o.modes = self.m1.ctypes.data_as(c.c_int32_p)
        o.shard_offset, o.shard_extent = 0, int(rows[2])
        o.data = self.dense.ctypes.data_as(c.c_double_p) if dense else None
        o.miss = self.mask.ctypes.data_as(c.c_uint8_p) if miss else None
        m = objs[1]
        m.model, m.order, m.weight, m.znorm_const = 0, 2, 1.0, 0.0
        m.modes = self.m2.ctypes.data_as(c.c_int32_p)
        m.shard_offset, m.shard_extent = 0, 3
        m.data = self.mat.ctypes.data_as(c.c_double_p)
        self.objs = objs
        pb = c.Problem()
        pb.nb_modes, pb.n_objects = 4 if with_matrix else 3, 2 if with_matrix else 1
        pb.n_couplings = 1 if with_matrix else 0
        pb.mode_rows = self.rows.ctypes.data_as(c.c_int64_p)
        pb.mode_rank = self.rank.ctypes.data_as(c.c_int32_p)
        pb.n_slices = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.objects = objs
        pb.lin_coupled_modes = self.lin.ctypes.data_as(c.c_int32_p)
        pb.coupling_type = self.ctype.ctypes.data_as(c.c_int32_p)
        pb.constrained_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constraints = self.cons
        self.pb = pb
        self._keep = []

    def _so(self, c, nnz, subs, vals):
        subs = None if subs is None else np.asfortranarray(np.asarray(subs, dtype=np.int64))
        vals = None if vals is None else np.asarray(vals, dtype=np.float64)
        so = c.SparseObject()
        so.nnz = nnz
        so.subs = None if subs is None else subs.ctypes.data_as(c.c_int64_p)
        so.vals = None if vals is None else vals.ctypes.data_as(c.c_double_p)
        self._keep += [subs, vals, so]
        return ctypes.pointer(so)

    def create(self, c, sp=None, mk=None, n_gpus=2, devices=None):
        """sp / mk: None or (nnz, subs, vals) of object 1"""
        P = self.pb.n_objects
        sa = (ctypes.POINTER(c.SparseObject) * P)()
        ma = (ctypes.POINTER(c.SparseObject) * P)()
        if sp is not None:
            sa[0] = self._so(c, *sp)
        if mk is not None:
            ma[0] = self._so(c, *mk)
        dv = None if devices is None else np.asarray(devices, dtype=np.int32)
        h = c.HandleP()
        rc = c.lib.aoadmm_create_sparse_multi(ctypes.byref(self.pb), sa, ma if mk is not None else None, n_gpus,
                                              None if dv is None else dv.ctypes.data_as(c.c_int32_p), ctypes.byref(h))
        if h.value:
            c.lib.aoadmm_destroy(h)
        return rc


def test_create_sparse_multi_validates_before_touching_a_device(ab):
    c = ab._capi
    subs = np.array([[0, 0, 0], [5, 4, 3], [1, 1, 1], [2, 3, 2]])
    vals = np.array([1.0, 2.0, 3.0, 4.0])
    ok = (4, subs, vals)
    assert c.lib.aoadmm_create_sparse_multi(None, None, None, 2, None, None) == INVALID
    h = c.HandleP()
    assert c.lib.aoadmm_create_sparse_multi(None, None, None, 2, None, ctypes.byref(h)) == INVALID and not h.value
    cases = [
        (dict(), dict(sp=(-1, subs, vals)), INVALID, 'negative'),
        (dict(), dict(sp=(4, None, vals)), INVALID, 'NULL'),
        (dict(), dict(sp=(4, [[0, 0, 0], [6, 4, 3], [1, 1, 1], [2, 3, 2]], vals)), INVALID, 'out of range'),
        (dict(), dict(sp=(4, [[0, 0, 0], [5, 4, 4], [1, 1, 1], [2, 3, 2]], vals)), INVALID, 'out of range'),
        (dict(dense=True), dict(sp=ok), INVALID, 'both'),
        (dict(dense=True), dict(mk=ok), INVALID, 'dense objects take Z.miss'),        # a mask on a dense object
        (dict(), dict(sp=ok, mk=(4, [[0, 0, 0], [5, 4, 3], [1, 1, 9], [2, 3, 2]], vals)), INVALID, 'mask'),  # malformed
        (dict(), dict(sp=ok, mk=(-2, subs, vals)), INVALID, 'mask'),
        (dict(miss=True), dict(sp=ok), UNSUPPORTED, 'Z.miss'),
        (dict(model=1), dict(sp=ok), UNSUPPORTED, 'PARAFAC2'),
        (dict(), dict(sp=ok, n_gpus=0), INVALID, 'n_gpus'),
        (dict(), dict(sp=ok, devices=[0, 0]), INVALID, 'twice'),
        (dict(), dict(sp=ok, n_gpus=5), INVALID, 'fewer indices'),                    # 4 last-mode indices
        (dict(dense=True, with_matrix=True), dict(n_gpus=5), INVALID, 'fewer indices'),   # dense tensors too
    ]
    for kw, ckw, want, msg in cases:
        pr = _Problem(c, **kw)
        assert pr.create(c, **ckw) == want, (kw, ckw)
        err = c.lib.aoadmm_last_error(None).decode()
        assert msg in err, (msg, err)
    if ab.device_count() == 0:   # well-formed descriptors get as far as the device
        assert _Problem(c, with_matrix=True).create(c, sp=ok, mk=(4, subs, np.ones(4))) == NO_DEVICE
        assert _Problem(c).create(c, sp=(0, None, None), n_gpus=4) == NO_DEVICE
        assert _Problem(c).create(c, sp=ok, n_gpus=1) == NO_DEVICE


def _sparse_script6(ab, frac=0.3, seed=0, sz=(20, 18, 16, 20, 22, 18, 24), R=3):
    Z, G, _ = pg.config_script6(seed=seed, sz=sz, R=R)
    rng = np.random.RandomState(seed + 100)
    X = Z['object'][0]
    W = rng.rand(*X.shape) < frac
    Xs = ab.sptensor(np.argwhere(W), X[W], X.shape)
    return dict(Z, object=[Xs] + Z['object'][1:]), dict(Z, object=[np.asfortranarray(X * W)] + Z['object'][1:]), G


def test_python_refusals_happen_before_any_device_call(ab):
    Zs, Zd, G = _sparse_script6(ab)
    zn = [float('nan')] + pg.znorm_const(Zd)[1:]
    opts = pg.default_options(MaxOuterIters=2)
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(Zs, zn, G, None, None, None, None, opts, world_size=2, rank=0, shard_sparse=True)
    assert e.value.status_name == 'UNSUPPORTED' and 'shard_sparse' in str(e.value)
    with pytest.raises(ab.AoadmmError) as e:   # without the keyword nothing changes
        ab.cmtf_fun_AOADMM(Zs, zn, G, None, None, None, None, opts, n_gpus=2)
    assert e.value.status_name == 'UNSUPPORTED' and 'sparse objects run on one GPU' in str(e.value)
    with pytest.raises(ab.AoadmmError) as e:   # the slab rule is checked on the host too
        ab.Solver(ab._with_rank(Zs, G), zn, n_gpus=17, shard_sparse=True)
    assert e.value.status_name == 'INVALID_ARG' and 'fewer indices' in str(e.value)


# ---------------------------------------------------------------------------------------------- masked EM sums
def test_sharded_masked_em_sums_model(ab):
    """sparse_em_nonzeros / sparse_em_finish: per-slab nonzero-side sums, all-reduced, then assembled once with the
    replicated telescoped terms, equal the whole-object sums; all-reducing the finished sums would count the
    telescoped terms once per GPU."""
    rng = np.random.RandomState(3)
    shape, R, n = (9, 8, 10), 3, 3
    F = [rng.randn(s, R) for s in shape]
    B = [rng.randn(s, R) for s in shape]
    full = lambda U: np.einsum('ir,jr,kr->ijk', *U)
    W = rng.rand(*shape) < 0.3
    S = rng.randn(*shape) * W
    MF, MB = full(F), full(B)
    tele, mm = np.sum((MF - MB) ** 2), np.sum(MB ** 2)          # replicated (factor side)

    def nz(sl):
        w, s, mp, m = W[..., sl], S[..., sl], MF[..., sl], MB[..., sl]
        return np.array([np.sum(s * mp * w), np.sum(mp * mp * w), np.sum((mp - m) ** 2 * w), np.sum(m * m * w)])

    def assemble(a):
        return np.array([max(tele - a[2], 0.0), max(mm - a[3], 0.0), a[0], a[1], 0.0])

    last = np.nonzero(W)[2]
    b = np_bounds(last, shape[2], n)
    parts = [nz(slice(b[r], b[r + 1])) for r in range(n)]
    whole = assemble(nz(slice(None)))
    assert np.allclose(assemble(np.sum(parts, axis=0)), whole, rtol=1e-12, atol=1e-12)
    # the reference quantities: the missing-entry numerator / denominator of f_rel_missing
    assert np.isclose(whole[0], np.sum((MF - MB) ** 2 * ~W), rtol=1e-10) and np.isclose(whole[1], np.sum(MB ** 2 * ~W), rtol=1e-10)
    wrong = np.sum([assemble(p) for p in parts], axis=0)
    assert abs(wrong[0] - whole[0]) > 0.5 * tele


# ---------------------------------------------------------------------------------------------- GPU
def _gpus(ab):
    n = ab.device_count()
    assert n >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'
    return n


@pytest.fixture(params=['2', '4', 'all'])
def N(request, ab):
    n = _gpus(ab)
    want = n if request.param == 'all' else int(request.param)
    if n < 2 or want > n or (request.param == 'all' and n in (2, 4)):
        pytest.skip('needs %s GPUs (%d visible)' % (request.param, n))
    return want


def _zn(ab, Zs, Zd):
    zd = pg.znorm_const(Zd)
    return [float('nan') if ab.as_sparse(x) is not None else z for x, z in zip(Zs['object'], zd)], zd


def _run(ab, Z, zn, G, opts, **dist):
    return ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, **dist)


def _check_oracle(ab, Zs, Zd, G, opts, N):
    zs, zd = _zn(ab, Zs, Zd)
    Go, oo = oracle_solve(Zd, zd, G, options=opts)
    Gd, od = _run(ab, Zs, zs, G, opts, n_gpus=N, shard_sparse=True)
    assert od['OuterIterations'] == oo['OuterIterations']
    n = oo['OuterIterations'] + 1
    for key in ('func_val_conv', 'func_coupl_conv', 'func_constr_conv'):
        assert np.max(np.abs(od[key][:n] - oo[key][:n])) < FIT_TOL, key
    if Zd.get('miss') and any(m is not None for m in Zd['miss']):
        a, b = od['func_rel_missing'][1:n], oo['func_rel_missing'][1:n]
        assert np.max(np.abs(a - b)) < FIT_TOL and abs(od['f_rel_missing'] - oo['f_rel_missing']) < FIT_TOL
    assert np.array_equal(od['innerIters'], oo['innerIters'])
    assert_state_close(Gd, Go, tol=FAC_TOL)
    return Gd, od


def _check_one_gpu(ab, Zs, zs, G, opts, N, tol=1e-12):
    G1, o1 = _run(ab, Zs, zs, G, opts)
    GN, oN = _run(ab, Zs, zs, G, opts, n_gpus=N, shard_sparse=True)
    assert oN['OuterIterations'] == o1['OuterIterations']
    for a, b in zip(GN['fac'], G1['fac']):
        assert rel(a, b) <= tol
    return (G1, o1), (GN, oN)


def _masked(ab, Z, p, frac, seed):
    rng = np.random.RandomState(seed)
    X = Z['object'][p]
    W = rng.rand(*X.shape) < frac
    subs = np.argwhere(W).astype(np.int64)
    os_, od, ms, md = list(Z['object']), list(Z['object']), [None] * len(Z['object']), [None] * len(Z['object'])
    os_[p], ms[p] = ab.sptensor(subs, X[W], X.shape), ab.sptensor(subs, np.ones(len(subs)), X.shape)
    od[p], md[p] = np.asfortranarray(np.where(W, X, 0.0)), np.asfortranarray(W)
    return dict(Z, object=os_, miss=ms), dict(Z, object=od, miss=md)


def _matrix_pair(I, J, M, R, seed, constraints=None, noise=0.1):
    rng = np.random.RandomState(seed)
    constraints = constraints or [None] * 4
    coupling = {'lin_coupled_modes': [1, 0, 1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 4}
    return pg._finish(['CP', 'CP'], [I, J, I, M], [[1, 2], [3, 4]], [[1.0] * R] * 2, [noise] * 2, coupling,
                      [pg.d_rand] * 4, [1 if c else 0 for c in constraints], constraints, [0.5, 0.5], rng)


def _bitwise(Ga, Gb):
    for key in ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac'):
        for a, b in zip(Ga[key], Gb[key]):
            assert (a is None and b is None) or np.array_equal(a, b), key


@pytest.mark.gpu
@pytest.mark.parametrize('R', [1, 32])
def test_script6_structure_against_oracle(ab, N, R):
    Zs, Zd, G = _sparse_script6(ab, frac=0.2, sz=(40, 36, 32, 40, 44, 36, 48), R=R, seed=R)
    _check_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=15, **ZERO_TOL), N)


@pytest.mark.gpu
def test_four_way_against_oracle_and_one_gpu(ab, N):
    Z, G, _ = pg.config_single_cp(sz=(14, 12, 10, 16), R=7, seed=9, noise=0.1, constraints=[('non-negativity',)] * 4)
    X = Z['object'][0]
    W = np.random.RandomState(1).rand(*X.shape) < 0.25
    Zs, Zd = dict(Z, object=[ab.sptensor(np.argwhere(W), X[W], X.shape)]), dict(Z, object=[np.asfortranarray(X * W)])
    opts = pg.default_options(MaxOuterIters=12, **ZERO_TOL)
    _check_oracle(ab, Zs, Zd, G, opts, N)
    _check_one_gpu(ab, Zs, [float('nan')], G, opts, N)


@pytest.mark.gpu
@pytest.mark.parametrize('R', [64, 200])
def test_sparse_matrix_coupled_to_dense_side_matrix(ab, N, R):
    nn = ('non-negativity',)
    Z, G, _ = _matrix_pair(I=120, J=90, M=80, R=R, seed=R, constraints=[nn, None, nn, None])
    X = Z['object'][0]
    W = np.random.RandomState(R).rand(*X.shape) < 0.3
    Zs = dict(Z, object=[ab.sptensor(np.argwhere(W), X[W], X.shape), Z['object'][1]])
    Zd = dict(Z, object=[np.asfortranarray(X * W), Z['object'][1]])
    opts = pg.default_options(MaxOuterIters=8, **ZERO_TOL)
    _check_oracle(ab, Zs, Zd, G, opts, N)
    _check_one_gpu(ab, Zs, [float('nan'), pg.znorm_const(Z)[1]], G, opts, N)


@pytest.mark.gpu
@pytest.mark.parametrize('mode1', [('TV regularization',), ('simplex column-wise', 1.0)])
def test_non_elementwise_prox(ab, N, mode1):
    Z, G, _ = pg.config_cp_tv(I=40, J=30, K=26, R=3, seed=4, mode1=mode1, eta=1e-3 if len(mode1) == 1 else 1.0)
    X = Z['object'][0]
    W = np.random.RandomState(2).rand(*X.shape) < 0.3
    Zs, Zd = dict(Z, object=[ab.sptensor(np.argwhere(W), X[W], X.shape)]), dict(Z, object=[np.asfortranarray(X * W)])
    _check_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=15, **ZERO_TOL), N)


@pytest.mark.gpu
def test_sharded_sparse_tensor_with_sharded_dense_tensor(ab, N):
    """A sparse 3-way tensor coupled in mode 1 to a dense 3-way tensor: both are cut along their last mode, the dense
    one uniformly, the sparse one by its nonzeros."""
    rng = np.random.RandomState(5)
    coupling = {'lin_coupled_modes': [1, 0, 0, 1, 0, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 6}
    Z, G, _ = pg._finish(['CP', 'CP'], [30, 24, 28, 30, 20, 22], [[1, 2, 3], [4, 5, 6]], [[1.0] * 4] * 2, [0.1] * 2,
                         coupling, [pg.d_rand] * 6, [1] * 6, [('non-negativity',)] * 6, [0.5, 0.5], rng)
    X = Z['object'][0]
    W = rng.rand(*X.shape) < 0.2
    W[..., :3] |= rng.rand(*X.shape[:2], 3) < 0.6          # skewed towards the first indices
    Zs = dict(Z, object=[ab.sptensor(np.argwhere(W), X[W], X.shape), Z['object'][1]])
    Zd = dict(Z, object=[np.asfortranarray(X * W), Z['object'][1]])
    opts = pg.default_options(MaxOuterIters=12, **ZERO_TOL)
    _check_oracle(ab, Zs, Zd, G, opts, N)
    with ab.Solver(ab._with_rank(Zs, G), _zn(ab, Zs, Zd)[0], n_gpus=N, shard_sparse=True) as s:
        b = ab.sparse_shard_bounds(Zs['object'][0], N)
        assert s.shards[0] == [(int(b[r]), int(b[r + 1])) for r in range(N)]


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['skew40', 'empty_slab', 'nnz0'])
def test_skewed_and_empty_shards(ab, N, kind):
    rng = np.random.RandomState(11)
    Z, G, _ = pg.config_single_cp(sz=(30, 25, 20), R=5, seed=3, noise=0.1, constraints=[('non-negativity',)] * 3)
    X = Z['object'][0]
    subs = np.argwhere(rng.rand(*X.shape) < 0.15)
    if kind == 'skew40':
        subs[rng.rand(len(subs)) < 0.4, 2] = 7
    elif kind == 'empty_slab':      # every nonzero at last index 0: the other GPUs own no nonzero
        subs[:, 2] = 0
    else:
        subs = subs[:0]
    subs = np.unique(subs, axis=0)
    vals = X[tuple(subs.T)]
    S = ab.sptensor(subs, vals, X.shape)
    b = ab.sparse_shard_bounds(S, N)
    if kind == 'empty_slab':
        assert b[1] == 1
    opts = pg.default_options(MaxOuterIters=8, **ZERO_TOL)
    _check_oracle(ab, dict(Z, object=[S]), dict(Z, object=[S.full()]), G, opts, N)


@pytest.mark.gpu
def test_bit_reproducible_and_order_independent(ab, N):
    Z, G, _ = pg.config_single_cp(sz=(40, 30, 25), R=6, seed=3, noise=0.1, constraints=[('non-negativity',)] * 3)
    Zs, _ = _masked(ab, Z, 0, 0.2, 4)
    X, Mk = Zs['object'][0], Zs['miss'][0]
    opts = pg.default_options(MaxOuterIters=10, **ZERO_TOL)
    rng = np.random.RandomState(0)
    p1, p2 = rng.permutation(X.nnz), rng.permutation(Mk.nnz)
    variants = [Zs, Zs, dict(Zs, object=[ab.sptensor(X.subs[p1], X.vals[p1], X.shape)]),
                dict(Zs, miss=[ab.sptensor(Mk.subs[p2], Mk.vals[p2], Mk.shape)])]
    runs = [_run(ab, Zx, [float('nan')], G, opts, n_gpus=N, shard_sparse=True) for Zx in variants]
    for Gx, ox in runs[1:]:
        _bitwise(runs[0][0], Gx)
        assert np.array_equal(runs[0][1]['func_val_conv'], ox['func_val_conv'])
        assert np.array_equal(runs[0][1]['func_rel_missing'], ox['func_rel_missing'], equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize('R', [7, 64])
def test_masked_against_oracle(ab, N, R):
    nn = ('non-negativity',)
    Z, G, _ = _matrix_pair(I=150, J=120, M=100, R=R, seed=R, constraints=[nn, None, nn, None])
    Zs, Zd = _masked(ab, Z, 0, 0.3, R)
    _check_oracle(ab, Zs, Zd, G, pg.default_options(MaxOuterIters=10, **ZERO_TOL), N)
    Z3, G3, _ = pg.config_single_cp(sz=(30, 25, 22), R=R, seed=R, noise=0.1, constraints=[nn] * 3)
    Zs3, Zd3 = _masked(ab, Z3, 0, 0.25, 3)
    _check_oracle(ab, Zs3, Zd3, G3, pg.default_options(MaxOuterIters=8, **ZERO_TOL), N)


@pytest.mark.gpu
def test_masked_default_tolerances_stop_with_one_gpu(ab, N):
    Z, G, _ = pg.config_single_cp(sz=(25, 20, 18), R=2, seed=2, noise=0.0, constraints=[('non-negativity',)] * 3)
    Zs, _ = _masked(ab, Z, 0, 0.7, 5)
    opts = pg.default_options(MaxOuterIters=1500)
    (G1, o1), (GN, oN) = _check_one_gpu(ab, Zs, [float('nan')], G, opts, N, tol=1e-9)
    assert o1['exit_flag'] != 0 and oN['exit_flag'] == o1['exit_flag']
    assert oN['f_rel_missing'] < opts['OuterRelTol']


@pytest.mark.gpu
def test_heldout_history_and_refusal(ab, N):
    Z, G, _ = _matrix_pair(I=80, J=64, M=50, R=5, seed=1)
    X = Z['object'][0]
    rng = np.random.RandomState(1)
    u = rng.rand(*X.shape)
    W, H = u < 0.4, (u >= 0.4) & (u < 0.7)
    subs, hsubs = np.argwhere(W), np.argwhere(H)
    Zs = dict(Z, object=[ab.sptensor(subs, X[W], X.shape), Z['object'][1]],
              miss=[ab.sptensor(subs, np.ones(len(subs)), X.shape), None])
    held = ab.sptensor(hsubs, X[H], X.shape)
    zs = [float('nan'), pg.znorm_const(Z)[1]]
    opts = pg.default_options(MaxOuterIters=10, **ZERO_TOL)
    _, o1 = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts, heldout=[held, None])
    _, oN = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts, heldout=[held, None], n_gpus=N,
                               shard_sparse=True)
    assert oN['heldout_count'] == o1['heldout_count']
    assert rel(oN['heldout_sse'][0], o1['heldout_sse'][0]) <= 1e-12
    # an entry stored in the last GPU's slab
    b = ab.sparse_shard_bounds(Zs['object'][0], N)
    e = subs[subs[:, 1] >= b[N - 1]][0]
    bad = ab.sptensor(np.vstack([hsubs, e]), np.r_[X[H], 1.0], X.shape)
    with ab.Solver(ab._with_rank(Zs, G), zs, n_gpus=N, shard_sparse=True) as s:
        s.set_state(G)
        with pytest.raises(ab.AoadmmError) as err:
            s.set_heldout(1, bad)
        assert err.value.status_name == 'INVALID_ARG' and '(%d, %d)' % tuple(e) in str(err.value)


def _free_bytes():
    cudart = ctypes.CDLL('libcudart.so')
    f, t = ctypes.c_size_t(), ctypes.c_size_t()
    assert cudart.cudaMemGetInfo(ctypes.byref(f), ctypes.byref(t)) == 0
    return f.value


def _free_all(n):
    cudart = ctypes.CDLL('libcudart.so')
    out = []
    for d in range(n):
        assert cudart.cudaSetDevice(d) == 0
        out.append(_free_bytes())
    assert cudart.cudaSetDevice(0) == 0
    return out


@pytest.mark.gpu
def test_mask_mismatch_in_last_slab_fails_and_releases(ab, N):
    Z, G, _ = _matrix_pair(I=60, J=48, M=40, R=3, seed=2)
    Zs, _ = _masked(ab, dict(Z, rank=[3, 3]), 0, 0.3, 0)
    X, Mk = Zs['object'][0], Zs['miss'][0]
    zn = [float('nan'), pg.znorm_const(Z)[1]]
    with ab.Solver(Zs, zn, n_gpus=N, shard_sparse=True):   # communicators and contexts exist before we measure
        pass
    b = ab.sparse_shard_bounds(X, N)
    drop = np.nonzero(Mk.subs[:, 1] >= b[N - 1])[0][0]     # one stored entry of the last slab unobserved
    keep = np.ones(Mk.nnz, dtype=bool)
    keep[drop] = False
    bad = ab.sptensor(Mk.subs[keep], Mk.vals[keep], Mk.shape)
    before = _free_all(N)
    with pytest.raises(ab.AoadmmError) as e:
        ab.Solver(dict(Zs, miss=[bad, None]), zn, n_gpus=N, shard_sparse=True)
    assert e.value.status_name == 'UNSUPPORTED' and 'object 1' in str(e.value)
    after = _free_all(N)
    assert all(b0 - a < (8 << 20) for a, b0 in zip(after, before)), (before, after)


@pytest.mark.gpu
def test_one_gpu_through_the_new_entry_point_is_bit_identical(ab):
    _gpus(ab)
    Zs, Zd, G = _sparse_script6(ab, frac=0.2, seed=2)
    zs = [float('nan')] + pg.znorm_const(Zd)[1:]
    opts = pg.default_options(MaxOuterIters=10, **ZERO_TOL)
    Ga, oa = _run(ab, Zs, zs, G, opts)
    Gb, ob = _run(ab, Zs, zs, G, opts, n_gpus=1, shard_sparse=True)
    _bitwise(Ga, Gb)
    assert np.array_equal(oa['func_val_conv'], ob['func_val_conv'])
    Z, G2, _ = _matrix_pair(I=60, J=48, M=40, R=4, seed=3)
    Zm, _ = _masked(ab, Z, 0, 0.3, 1)
    zm = [float('nan'), pg.znorm_const(Z)[1]]
    Ga, oa = _run(ab, Zm, zm, G2, opts)
    Gb, ob = _run(ab, Zm, zm, G2, opts, n_gpus=1, shard_sparse=True)
    _bitwise(Ga, Gb)
    assert np.array_equal(oa['func_rel_missing'], ob['func_rel_missing'], equal_nan=True)
