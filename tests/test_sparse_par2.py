"""PARAFAC2 objects with sparse slices: aoadmm_create_sparse_slices, Solver(..., sparse_slices=True) and full solves.

The K slices of such an object are stacked side by side into one I x Jtot COO object; the two products of the PARAFAC2
block are the deterministic sparse MTTKRP of that object and the explicit residual is one pass over its stored
entries.  CPU tests check every refusal that happens before a device is touched and the host stacking; GPU tests (-m gpu)
compare whole solves on sparse slices against the oracle and the dense engine on the dense slices (north-star
tolerances: factors 1e-8 relative Frobenius, objective 1e-10), and check bit reproducibility."""
import ctypes

import numpy as np
import pytest

from oracle import problem_gen as pg
from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
from _cases import FIT_TOL, ZERO_TOL, assert_state_close

INVALID, UNSUPPORTED, NO_DEVICE = 1, 2, 8


def sparsify_slices(ab, slices, frac, rng):
    """Keep a random fraction of the entries of every dense slice: (sparse slices, dense slices with the others zeroed)."""
    sp, dn = [], []
    for X in slices:
        mask = rng.rand(*X.shape) < frac
        sp.append(ab.sptensor(np.argwhere(mask), X[mask], X.shape))
        dn.append(np.asfortranarray(X * mask))
    return sp, dn


# ---------------------------------------------------------------------------------------------- CPU
class _Par2Problem:
    """A one-object problem flattened by hand into the C structs: PARAFAC2 with I = 4, J_k = (3, 2) and rank 2
    (model=0: a 3-way CP object 4 x 3 x 2 instead)."""

    def __init__(self, c, model=1, I=4, Jk=(3, 2), slice_sizes=True, dense=False, miss=False):
        self.rows = np.asarray([I, 0 if model == 1 else 3, len(Jk) if model == 1 else 2], dtype=np.int64)
        self.rank = np.full(3, 2, dtype=np.int32)
        self.modes = np.arange(1, 4, dtype=np.int32)
        self.zero32 = np.zeros(3, dtype=np.int32)
        self.nsl = np.asarray([0, len(Jk) if model == 1 else 0, 0], dtype=np.int32)
        self.jk = np.asarray(Jk, dtype=np.int64)
        self.slice_rows = (c.c_int64_p * 3)()
        if model == 1 and slice_sizes:
            self.slice_rows[1] = self.jk.ctypes.data_as(c.c_int64_p)
        self.cons = (c.Constraint * 3)()
        self.dense = [np.zeros(4 * 3), np.zeros(4 * 2)]
        self.dense_p = (c.c_double_p * 2)(*[d.ctypes.data_as(c.c_double_p) for d in self.dense])
        self.masks = [np.ones(12, dtype=np.uint8), np.ones(8, dtype=np.uint8)]
        self.masks_p = (c.c_uint8_p * 2)(*[m.ctypes.data_as(c.c_uint8_p) for m in self.masks])
        obj = c.Object()
        obj.model, obj.order, obj.weight, obj.znorm_const = model, 3, 1.0, float('nan')
        obj.modes = self.modes.ctypes.data_as(c.c_int32_p)
        obj.n_slices = len(Jk) if model == 1 else 0
        obj.shard_offset, obj.shard_extent = 0, int(self.rows[2])
        obj.slices = self.dense_p if dense else None
        obj.miss_slices = self.masks_p if miss else None
        self.objs = (c.Object * 1)(obj)
        pb = c.Problem()
        pb.nb_modes, pb.n_objects, pb.n_couplings = 3, 1, 0
        pb.mode_rows = self.rows.ctypes.data_as(c.c_int64_p)
        pb.mode_rank = self.rank.ctypes.data_as(c.c_int32_p)
        pb.slice_rows = self.slice_rows
        pb.n_slices = self.nsl.ctypes.data_as(c.c_int32_p)
        pb.objects = self.objs
        pb.lin_coupled_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constrained_modes = self.zero32.ctypes.data_as(c.c_int32_p)
        pb.constraints = self.cons
        self.pb = pb

    def create(self, c, nnz, subs, vals, world_size=1, as_cp=False):
        """slices[0] = the descriptor (as_cp: passed as sparse[0] instead)"""
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
        rc = c.lib.aoadmm_create_sparse_slices(ctypes.byref(self.pb), arr if as_cp else None, None if as_cp else arr,
                                               ctypes.byref(dist), ctypes.byref(h))
        if h.value:
            c.lib.aoadmm_destroy(h)
        return rc


def test_create_sparse_slices_validates_before_touching_a_device(ab):
    c = ab._capi
    # rows 0..3, stacked columns 0..4 (slice 1: columns 0..2, slice 2: columns 3..4)
    ok_subs = np.array([[0, 0], [3, 4], [1, 2]])
    ok_vals = np.array([1.0, 2.0, 3.0])
    assert c.lib.aoadmm_create_sparse_slices(None, None, None, None, None) == INVALID
    h = c.HandleP()
    assert c.lib.aoadmm_create_sparse_slices(None, None, None, None, ctypes.byref(h)) == INVALID and not h.value
    big = 2 ** 31 - 257
    cases = [
        (dict(), {}, -1, ok_subs, ok_vals, INVALID, 'negative'),
        (dict(), {}, 3, None, ok_vals, INVALID, 'NULL'),
        (dict(), {}, 3, ok_subs, None, INVALID, 'NULL'),
        (dict(), {}, 3, [[0, 0], [4, 4], [1, 2]], ok_vals, INVALID, 'row subscript 4'),
        (dict(), {}, 3, [[0, 0], [3, 5], [1, 2]], ok_vals, INVALID, 'column subscript 5'),
        (dict(), {}, 3, [[0, 0], [3, 4], [1, -1]], ok_vals, INVALID, 'out of range'),
        (dict(dense=True), {}, 3, ok_subs, ok_vals, INVALID, 'both'),
        (dict(slice_sizes=False), {}, 3, ok_subs, ok_vals, INVALID, 'missing slice sizes'),
        (dict(I=2 ** 31), {}, 3, ok_subs, ok_vals, INVALID, '2^31 - 1'),
        (dict(Jk=(2 ** 31 - 2, 2)), {}, 3, ok_subs, ok_vals, INVALID, '2^31 - 1'),
        (dict(), {}, big, ok_subs, ok_vals, INVALID, '2^31 - 257'),
        (dict(model=0), {}, 3, ok_subs, ok_vals, INVALID, 'CP object'),
        (dict(), dict(as_cp=True), 3, ok_subs, ok_vals, INVALID, 'PARAFAC2 object'),
        (dict(), dict(world_size=2), 3, ok_subs, ok_vals, UNSUPPORTED, 'one GPU'),
        (dict(miss=True), {}, 3, ok_subs, ok_vals, UNSUPPORTED, 'Z.miss'),
    ]
    for kw, ckw, nnz, subs, vals, want, msg in cases:
        pr = _Par2Problem(c, **kw)
        assert pr.create(c, nnz, subs, vals, **ckw) == want, (kw, ckw, nnz)
        assert msg in c.lib.aoadmm_last_error(None).decode(), (msg, c.lib.aoadmm_last_error(None))
    if ab.device_count() == 0:   # a well-formed descriptor gets as far as the device
        assert _Par2Problem(c).create(c, 3, ok_subs, ok_vals) == NO_DEVICE
        assert _Par2Problem(c).create(c, 0, None, None) == NO_DEVICE


def _small_sparse_par2(ab, frac=0.5, seed=0):
    Z, G, _ = pg.config_single_par2(I=6, Jk=(5, 4, 3), R=2, seed=seed)
    sl, dn = sparsify_slices(ab, Z['object'][0], frac, np.random.RandomState(seed))
    return dict(Z, object=[sl]), dict(Z, object=[dn]), G


def test_solver_refuses_sparse_slices_before_any_device_call(ab):
    Zs, Zd, G = _small_sparse_par2(ab)
    opts = pg.default_options(MaxOuterIters=2)
    nan = [float('nan')]

    def refused(Z, **dist):
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_fun_AOADMM(Z, nan, G, None, None, None, None, opts, **dist)
        return e.value

    e = refused(Zs)   # no keyword: today's refusal
    assert e.status_name == 'UNSUPPORTED' and 'PARAFAC2 objects with sparse slices are not supported' in str(e)
    mixed = [Zs['object'][0][0], Zd['object'][0][1], Zs['object'][0][2]]
    e = refused(dict(Zs, object=[mixed]), sparse_slices=True)
    assert e.status_name == 'INVALID_ARG' and 'object 1' in str(e) and 'slice 2' in str(e)
    X1 = Zs['object'][0][1]
    wrong = [Zs['object'][0][0], ab.sptensor(X1.subs, X1.vals, (6, 5)), Zs['object'][0][2]]
    e = refused(dict(Zs, object=[wrong]), sparse_slices=True)
    assert e.status_name == 'INVALID_ARG' and 'object 1' in str(e) and 'slice 2' in str(e)
    # subscripts outside their own slice: a column >= J_k would become an entry of slice k + 1 once stacked, a negative
    # column in slice k > 0 one of slice k - 1, a row >= I one of no slice
    for k, bad_entry in ((0, (2, 5)), (1, (0, -1)), (2, (6, 0))):
        X = Zs['object'][0][k]
        bad = ab.sptensor(np.vstack([X.subs, bad_entry]), np.r_[X.vals, 1.0], X.shape)
        sl = list(Zs['object'][0])
        sl[k] = bad
        e = refused(dict(Zs, object=[sl]), sparse_slices=True)
        assert e.status_name == 'INVALID_ARG' and 'object 1' in str(e) and 'slice %d' % (k + 1) in str(e), str(e)
        assert 'out of range' in str(e)
        with pytest.raises(ab.AoadmmError) as eh:
            ab.stack_sparse_slices(sl)
        assert eh.value.status_name == 'INVALID_ARG' and 'slice %d' % (k + 1) in str(eh.value)
    miss = [[np.ones(x.shape) for x in Zd['object'][0]]]
    e = refused(dict(Zs, miss=miss), sparse_slices=True)
    assert e.status_name == 'UNSUPPORTED' and 'Z.miss' in str(e)
    e = refused(Zs, sparse_slices=True, n_gpus=2)
    assert e.status_name == 'UNSUPPORTED' and 'one GPU' in str(e)
    e = refused(Zs, sparse_slices=True, world_size=2, rank=0)
    assert e.status_name == 'UNSUPPORTED' and 'one GPU' in str(e)


def test_stacked_slices_equal_the_dense_slices_side_by_side(ab):
    rng = np.random.RandomState(3)
    I, Jk = 7, (4, 3, 5, 2)
    dense = [np.zeros((I, j)) for j in Jk]
    slices = []
    for k, j in enumerate(Jk):
        if k == 2:    # an empty slice
            slices.append(ab.sptensor(np.zeros((0, 2)), np.zeros(0), (I, j)))
            continue
        subs = np.stack([rng.randint(0, I, 6), rng.randint(0, j, 6)], axis=1)
        subs = np.vstack([subs, subs[:2]])          # duplicates: summed by full()
        vals = rng.randn(subs.shape[0])
        np.add.at(dense[k], tuple(subs.T), vals)
        slices.append(ab.sptensor(subs, vals, (I, j)))
    S, joff = ab.stack_sparse_slices(slices)
    assert S.shape == (I, sum(Jk)) and S.nnz == sum(x.nnz for x in slices)
    assert list(joff) == [0, 4, 7, 12, 14]
    assert np.array_equal(S.full(), np.hstack(dense))
    sps = pytest.importorskip('scipy.sparse')   # SciPy sparse slices are accepted as well
    S2, _ = ab.stack_sparse_slices([sps.csr_matrix(d) for d in dense])
    assert np.array_equal(S2.full(), np.hstack(dense))


# ---------------------------------------------------------------------------------------------- GPU
def _need_gpu(ab):
    assert ab.device_count() >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'


def _zn(ab, Zs, Zd):
    """Znorm_const: NaN (on the device) for every object with sparse data, the host value for the others"""
    zn = pg.znorm_const(Zd)
    sparse = [any(ab.as_sparse(x) is not None for x in o) if m == 'PAR2' else ab.as_sparse(o) is not None
              for m, o in zip(Zs['model'], Zs['object'])]
    return [float('nan') if s else z for s, z in zip(sparse, zn)], zn


def _assert_close(Go, oo, Gd, od):
    assert od['OuterIterations'] == oo['OuterIterations']
    n = oo['OuterIterations'] + 1
    for key in ('func_val_conv', 'func_coupl_conv', 'func_constr_conv'):
        assert np.max(np.abs(od[key][:n] - oo[key][:n])) < FIT_TOL, key
    assert np.array_equal(od['innerIters'], oo['innerIters'])
    assert_state_close(Gd, Go)


def _solve_three(ab, Zs, Zd, G, opts):
    """oracle and dense engine on the dense slices, the device on the sparse slices: all three agree"""
    zs, zn = _zn(ab, Zs, Zd)
    Go, oo = oracle_solve(Zd, zn, G, options=opts)
    Gs, os_ = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts, sparse_slices=True)
    Gd, od = ab.cmtf_fun_AOADMM(Zd, zn, G, None, None, None, None, opts)
    _assert_close(Go, oo, Gs, os_)
    _assert_close(Gd, od, Gs, os_)
    return Gs, os_


def _assert_bitwise(Ga, oa, Gb, ob):
    for key in ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac'):
        for a, b in zip(Ga[key], Gb[key]):
            if isinstance(a, list):
                assert all(np.array_equal(x, y) for x, y in zip(a, b)), key
            else:
                assert (a is None and b is None) or np.array_equal(a, b), key
    assert np.array_equal(oa['func_val_conv'], ob['func_val_conv'])


@pytest.mark.gpu
@pytest.mark.parametrize('frac', [0.05, 0.2, 0.5])
def test_irregular_slices_nonneg_A_and_C(ab, frac):
    """example_script4 / 8 structure: irregular J_k, non-negative A and C; mode C is updated last, so the residual
    pass over the stored entries runs in every iteration"""
    _need_gpu(ab)
    Z, G, _ = pg.config_single_par2(I=40, Jk=(12, 30, 9, 25, 17, 40, 11, 22), R=3, seed=2)
    sl, dn = sparsify_slices(ab, Z['object'][0], frac, np.random.RandomState(int(frac * 100)))
    _solve_three(ab, dict(Z, object=[sl]), dict(Z, object=[dn]), G, pg.default_options(MaxOuterIters=20, **ZERO_TOL))


@pytest.mark.gpu
def test_unimodal_B_k_non_elementwise_prox(ab):
    _need_gpu(ab)
    nn = ('non-negativity',)
    Z, G, _ = pg.config_single_par2(I=30, Jk=(14, 11, 16, 12, 13, 15), R=3, seed=8, constrained=(0, 1, 1),
                                    constraints=[None, ('unimodality', True), nn])
    sl, dn = sparsify_slices(ab, Z['object'][0], 0.3, np.random.RandomState(9))
    _solve_three(ab, dict(Z, object=[sl]), dict(Z, object=[dn]), G, pg.default_options(MaxOuterIters=12, **ZERO_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('cp_sparse', [False, True])
def test_cp_coupled_to_sparse_par2_in_mode_A(ab, cp_sparse):
    """script 1 / C4: CP coupled with the PARAFAC2 mode A, which is then updated last (shortcut objective from the
    sparse product); with cp_sparse the CP tensor is sparse too, so both sparse paths run in one problem"""
    _need_gpu(ab)
    Z, G, _ = pg.config_cp_par2(I=24, J=20, K=18, Jk=16, Kp=10, R=3, seed=3, noise=0.1)
    rng = np.random.RandomState(4)
    sl, dn = sparsify_slices(ab, Z['object'][1], 0.3, rng)
    X0 = Z['object'][0]
    if cp_sparse:
        mask = rng.rand(*X0.shape) < 0.3
        Xs, Xd = ab.sptensor(np.argwhere(mask), X0[mask], X0.shape), np.asfortranarray(X0 * mask)
    else:
        Xs = Xd = X0
    Gs, os_ = _solve_three(ab, dict(Z, object=[Xs, sl]), dict(Z, object=[Xd, dn]), G,
                           pg.default_options(MaxOuterIters=15, **ZERO_TOL))
    # Znorm_const = NaN of the sparse slices, read back: mode A is updated last, so from iteration 1 on the object's
    # term is w * (znorm - 2 f2 + f3).  The same run with znorm = 0 follows bit-identical iterates (znorm enters the
    # objective only), so the difference of the two histories is w * the device norm up to a few roundings of the terms
    zs, zn = _zn(ab, dict(Z, object=[Xs, sl]), dict(Z, object=[Xd, dn]))
    opts = pg.default_options(MaxOuterIters=15, **ZERO_TOL)
    G0, o0 = ab.cmtf_fun_AOADMM(dict(Z, object=[Xs, sl]), [zs[0], 0.0], G, None, None, None, None, opts,
                                sparse_slices=True)
    for a, b in zip(Gs['fac'], G0['fac']):
        assert all(np.array_equal(x, y) for x, y in zip(a, b)) if isinstance(a, list) else np.array_equal(a, b)
    host = sum(float(np.sum(x.full() ** 2)) for x in sl)   # the merged stored values
    assert abs(host - zn[1]) <= 1e-14 * zn[1]
    dev = (np.asarray(os_['func_val_conv'])[1:16] - np.asarray(o0['func_val_conv'])[1:16]) / Z['weights'][1]
    assert np.max(np.abs(dev - host)) <= 1e-14 * host, (dev, host)


@pytest.mark.gpu
def test_script14_coupling_type1_on_mode_C(ab):
    """coupling type 1 on the PARAFAC2 mode C: mode A is not updated last, the residual pass runs every iteration"""
    _need_gpu(ab)
    Z, G, _ = pg.config_script14(seed=2)
    sl, dn = sparsify_slices(ab, Z['object'][1], 0.4, np.random.RandomState(5))
    _solve_three(ab, dict(Z, object=[Z['object'][0], sl]), dict(Z, object=[Z['object'][0], dn]), G,
                 pg.default_options(MaxOuterIters=12, **ZERO_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('R', [2, 16, 17, 65])
def test_ranks_across_the_dispatch_groups(ab, R):
    """R = 2 / 16 / 17 / 65: lanes per entry 2, 16, 32 and two columns per lane; register and CTA polar factors; the
    R > 64 workspace of the per-slice systems"""
    _need_gpu(ab)
    J = max(R + 3, 12)
    Z, G, _ = pg.config_single_par2(I=R + 20, Jk=(J, J + 5, J + 1, J + 9), R=R, seed=R)
    sl, dn = sparsify_slices(ab, Z['object'][0], 0.4, np.random.RandomState(R))
    _solve_three(ab, dict(Z, object=[sl]), dict(Z, object=[dn]), G, pg.default_options(MaxOuterIters=6, **ZERO_TOL))


def _edge_slices(ab, Z, rng):
    """an empty slice, row 0 of A without entries in any slice, duplicates split in two (summed), explicit zeros (kept)"""
    sl, dn = [], []
    for k, X in enumerate(Z['object'][0]):
        mask = rng.rand(*X.shape) < 0.4
        mask[0, :] = False
        if k == 2:
            mask[:] = False
        subs, vals = np.argwhere(mask), X[mask]
        half = vals / 2
        zs = np.argwhere(~mask)[:3]
        subs = np.vstack([subs, subs, zs])
        vals = np.concatenate([half, vals - half, np.zeros(len(zs))])
        sl.append(ab.sptensor(subs, vals, X.shape))
        dn.append(np.asfortranarray(X * mask))
    return sl, dn


@pytest.mark.gpu
def test_empty_slice_empty_row_duplicates_and_explicit_zeros(ab):
    _need_gpu(ab)
    Z, G, _ = pg.config_single_par2(I=20, Jk=(10, 12, 9, 11, 8), R=3, seed=6)
    sl, dn = _edge_slices(ab, Z, np.random.RandomState(6))
    assert sl[2].full().any() == False and all(x.full()[0].any() == False for x in sl)
    _solve_three(ab, dict(Z, object=[sl]), dict(Z, object=[dn]), G, pg.default_options(MaxOuterIters=10, **ZERO_TOL))


@pytest.mark.gpu
def test_permuted_entries_graph_replay_and_repeated_runs_are_bit_identical(ab, monkeypatch):
    _need_gpu(ab)
    Z, G, _ = pg.config_cp_par2(I=24, J=20, K=18, Jk=16, Kp=10, R=3, seed=5, noise=0.1)
    sl, dn = sparsify_slices(ab, Z['object'][1], 0.3, np.random.RandomState(1))
    Zs = dict(Z, object=[Z['object'][0], sl])
    zs, _ = _zn(ab, Zs, dict(Z, object=[Z['object'][0], dn]))
    opts = pg.default_options(MaxOuterIters=12, **ZERO_TOL)
    runs = [ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, dict(opts, graph=g), sparse_slices=True)
            for g in (1, -1, 1)]
    for Gx, ox in runs[1:]:
        _assert_bitwise(runs[0][0], runs[0][1], Gx, ox)
    rng = np.random.RandomState(2)
    within = []
    for x in sl:   # every slice's entries permuted
        p = rng.permutation(x.nnz)
        within.append(ab.sptensor(x.subs[p], x.vals[p], x.shape))
    Gw, ow = ab.cmtf_fun_AOADMM(dict(Z, object=[Z['object'][0], within]), zs, G, None, None, None, None, opts,
                                sparse_slices=True)
    _assert_bitwise(runs[0][0], runs[0][1], Gw, ow)
    stack = ab.stack_sparse_slices

    def shuffled(slices):   # the stacked entries permuted across slices
        S, joff = stack(slices)
        p = np.random.RandomState(3).permutation(S.nnz)
        return ab.sptensor(S.subs[p], S.vals[p], S.shape), joff

    monkeypatch.setattr(ab, 'stack_sparse_slices', shuffled)
    Ga, oa = ab.cmtf_fun_AOADMM(Zs, zs, G, None, None, None, None, opts, sparse_slices=True)
    _assert_bitwise(runs[0][0], runs[0][1], Ga, oa)


@pytest.mark.gpu
def test_sparse_slice_handle_refuses_nvecs_and_model_at(ab):
    _need_gpu(ab)
    Zs, Zd, G = _small_sparse_par2(ab)
    with ab.Solver(dict(Zs, rank=[2]), [float('nan')], sparse_slices=True) as s:
        for mode, sl in ((1, 0), (2, 1)):
            with pytest.raises(ab.AoadmmError) as e:
                s.nvecs(mode, 2, slice=sl)
            assert e.value.status_name == 'UNSUPPORTED' and 'sparse slices' in str(e.value)
        with pytest.raises(ab.AoadmmError) as e:
            s.nvecs_sparse(1, 2)
        assert 'PARAFAC2' in str(e.value)
        with pytest.raises(ab.AoadmmError) as e:
            s.model_at(1, np.zeros((1, 3), dtype=np.int64))
        assert 'PARAFAC2' in str(e.value)


@pytest.mark.gpu
def test_problem_without_a_dense_form(ab):
    """I = 2^15, K = 2000, J_k = 1024: the dense slices would take 512 GB.  About 10^6 stored entries, R = 4."""
    _need_gpu(ab)
    torch = pytest.importorskip('torch')
    I, K, J, R, per = 1 << 15, 2000, 1024, 4, 500
    rng = np.random.RandomState(0)
    sl = [ab.sptensor(np.stack([rng.randint(0, I, per), rng.randint(0, J, per)], axis=1), rng.rand(per), (I, J))
          for _ in range(K)]
    nn = ('non-negativity',)
    Z = {'loss_function': ['Frobenius'], 'model': ['PAR2'], 'modes': [[1, 2, 3]], 'size': [I, [J] * K, K],
         'coupling': {'lin_coupled_modes': [0, 0, 0], 'coupling_type': [], 'coupl_trafo_matrices': [None] * 3},
         'constrained_modes': [1, 0, 1], 'constraints': [nn, None, nn], 'weights': [1.0], 'object': [sl]}
    io = {'lambdas_init': [[1.0] * R], 'nvecs': 0, 'distr': [pg.d_rand, pg.d_rand, pg.d_rand01], 'normalize': 1}
    G = pg.init_coupled_AOADMM_CMTF(Z, io, np.random.RandomState(1))
    torch.cuda.init()
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info(0)
    with ab.Solver(dict(Z, rank=[R]), [float('nan')], sparse_slices=True) as s:
        free1, _ = torch.cuda.mem_get_info(0)
        assert free0 - free1 < 10 * 2 ** 30, (free0 - free1) / 2 ** 30
        s.set_state(G)
        out = s.run(pg.default_options(MaxOuterIters=3, **ZERO_TOL))
    f = np.asarray(out['func_val_conv'])[:4]
    assert out['OuterIterations'] == 3 and np.all(np.isfinite(f)), f
