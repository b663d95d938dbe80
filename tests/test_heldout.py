"""Held-out entries: the model at given subscripts (aoadmm_model_at) and the validation error per outer iteration
(aoadmm_set_heldout / aoadmm_heldout_history).

CPU tests restate the kernel's evaluation order in NumPy, check the refusals that happen before any device call and the
signatures of the three entry points.  GPU tests (-m gpu) compare the model with NumPy, the held-out SSE history with the
oracle run for k = 0..n iterations, and check that attaching a held-out set leaves the solve bit-identical."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import problem_gen as pg
from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
from _cases import ZERO_TOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 1


def model_at(subs, U):
    """[[U]](subs[e]) for every row of subs, by direct indexing."""
    p = np.ones((subs.shape[0], U[0].shape[1]))
    for d, F in enumerate(U):
        p = p * F[subs[:, d], :]
    return p.sum(axis=1)


def lanes(R):
    """(G, CPL) of the rank dispatch of sparse.cuh."""
    for lim, g, c in ((1, 1, 1), (2, 2, 1), (4, 4, 1), (8, 8, 1), (16, 16, 1), (32, 32, 1), (64, 32, 2), (128, 32, 4)):
        if R <= lim:
            return g, c
    return 32, 8


def model_at_lanes(subs, U):
    """The kernel's order: lane j of G sums its columns j, j+G, ... in ascending order (each a product over the positions
    in ascending order), then the lanes are summed by an xor butterfly with offsets G/2, G/4, ..., 1."""
    R = U[0].shape[1]
    G, CPL = lanes(R)
    P = np.ones((subs.shape[0], G * CPL))
    P[:, R:] = 0.0
    for d, F in enumerate(U):
        P[:, :R] = P[:, :R] * F[subs[:, d], :]
    t = np.zeros((subs.shape[0], G))
    for q in range(CPL):
        t = t + P[:, q * G:(q + 1) * G]
    off = G // 2
    while off > 0:
        t = t + t[:, np.arange(G) ^ off]
        off //= 2
    return t[:, 0]


def full_cp(U):
    X = U[0]
    for F in U[1:]:
        X = np.einsum('...r,jr->...jr', X, F)
    return X.sum(axis=-1)


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('shape,R', [((9, 7), 1), ((7, 6, 5), 7), ((6, 5, 4, 3), 32), ((8, 6, 5), 64), ((5, 4), 200)])
def test_model_at_restatement_equals_full_ktensor(shape, R):
    rng = np.random.RandomState(R)
    U = [rng.rand(s, R) for s in shape]
    X = full_cp(U)
    subs = np.argwhere(rng.rand(*shape) < 0.5)
    ref = X[tuple(subs.T)]
    for got in (model_at(subs, U), model_at_lanes(subs, U)):
        assert np.max(np.abs(got - ref) / np.abs(ref)) < 1e-13


def _matrix_pair(I=30, J=25, M=20, R=3, seed=0, noise=0.1):
    rng = np.random.RandomState(seed)
    coupling = {'lin_coupled_modes': [1, 0, 1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 4}
    return pg._finish(['CP', 'CP'], [I, J, I, M], [[1, 2], [3, 4]], [[1.0] * R] * 2, [noise] * 2, coupling,
                      [pg.d_rand] * 4, [0] * 4, [None] * 4, [0.5, 0.5], rng)


def _split(ab, X, frac_train, frac_held, rng):
    """Observe frac_train of the matrix / tensor X and hold out frac_held of the rest: (S, sparse mask, held-out set)."""
    u = rng.rand(*X.shape)
    W, H = u < frac_train, (u >= frac_train) & (u < frac_train + frac_held)
    ts, hs = np.argwhere(W), np.argwhere(H)
    return (ab.sptensor(ts, X[W], X.shape), ab.sptensor(ts, np.ones(len(ts)), X.shape), ab.sptensor(hs, X[H], X.shape))


def test_python_refusals_happen_before_any_device_call(ab):
    Z, G, _ = _matrix_pair()
    opts = pg.default_options(MaxOuterIters=2)
    zn = pg.znorm_const(Z)
    S, Mk, H = _split(ab, Z['object'][0], 0.5, 0.2, np.random.RandomState(0))
    cases = [
        (dict(), [H, None], 'no missing data'),                                       # object without Z.miss
        (dict(miss=[Mk, None]), [None, H], 'no missing data'),
        (dict(miss=[Mk, None]), [ab.sptensor(H.subs, H.vals, (30, 26)), None], 'shape'),
        (dict(miss=[Mk, None]), [np.zeros((30, 25)), None], 'sptensor'),              # a dense array is not a set
        (dict(miss=[Mk, None]), [H], 'one entry per object'),
    ]
    for kw, heldout, msg in cases:
        Zx = dict(Z, object=[S, Z['object'][1]], **kw) if kw else Z
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_fun_AOADMM(Zx, zn, G, None, None, None, None, opts, heldout=heldout)
        assert e.value.status_name == 'INVALID_ARG' and msg in str(e.value), (msg, str(e.value))
    Zp, _, _ = pg.config_single_par2()
    Zp = dict(Zp, miss=[[np.ones(x.shape) for x in Zp['object'][0]]])
    with pytest.raises(ab.AoadmmError) as e:
        ab._check_heldout(Zp, 0, H)
    assert e.value.status_name == 'INVALID_ARG' and 'PARAFAC2' in str(e.value)


def test_header_and_ctypes_signatures(ab):
    c = ab._capi
    hdr = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    want = {
        'aoadmm_model_at': (r'int aoadmm_model_at\(aoadmm_handle \*h, int32_t object, const aoadmm_sparse_object \*entries, '
                            r'double \*out\);', [c.HandleP, ctypes.c_int32, ctypes.POINTER(c.SparseObject), c.c_double_p]),
        'aoadmm_set_heldout': (r'int aoadmm_set_heldout\(aoadmm_handle \*h, int32_t object, '
                               r'const aoadmm_sparse_object \*entries\);',
                               [c.HandleP, ctypes.c_int32, ctypes.POINTER(c.SparseObject)]),
        'aoadmm_heldout_history': (r'int aoadmm_heldout_history\(const aoadmm_handle \*h, int32_t object, double \*sse, '
                                   r'int64_t n, int64_t \*count\);',
                                   [c.HandleP, ctypes.c_int32, c.c_double_p, ctypes.c_int64, c.c_int64_p]),
    }
    for name, (proto, argtypes) in want.items():
        assert re.search(proto, hdr), name
        assert name in c.EXPORTS
        assert list(getattr(c.lib, name).argtypes) == argtypes, name
    # NULL handles and bad sizes are refused without a device
    so = c.SparseObject()
    out = np.zeros(1)
    assert c.lib.aoadmm_model_at(None, 1, ctypes.byref(so), out.ctypes.data_as(c.c_double_p)) == INVALID
    assert c.lib.aoadmm_set_heldout(None, 1, None) == INVALID
    assert c.lib.aoadmm_heldout_history(None, 1, None, 0, None) == INVALID


# ---------------------------------------------------------------------------------------------- GPU
def _need_gpu(ab):
    assert ab.device_count() >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'


def _single(sz, R, seed):
    Z, G, _ = pg.config_single_cp(sz=sz, R=R, seed=seed, noise=0.1)
    return Z, G


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['dense', 'sparse', 'masked'])
@pytest.mark.parametrize('R,sz', [(1, (40, 30)), (7, (20, 15, 12)), (32, (12, 10, 9, 8)), (64, (25, 20)),
                                  (200, (14, 12, 10))])
def test_model_at_matches_numpy(ab, kind, R, sz):
    _need_gpu(ab)
    rng = np.random.RandomState(R)
    Z, G = _single(sz, R, R)
    X = Z['object'][0]
    if kind == 'sparse':
        subs = np.argwhere(rng.rand(*sz) < 0.3)
        Z = dict(Z, object=[ab.sptensor(subs, X[tuple(subs.T)], sz)])
    elif kind == 'masked':
        Z = pg.add_missing(Z, 0.3, seed=R)
    U = [rng.rand(s, R) for s in sz]
    G = dict(G, fac=U)
    n = 5000
    skew = np.stack([np.minimum((rng.pareto(1.5, n) * 0.5).astype(np.int64), s - 1) for s in sz], axis=1)  # hot rows
    unif = np.stack([rng.randint(0, s, n) for s in sz], axis=1)
    zn = [float('nan')] if kind == 'sparse' else pg.znorm_const(Z)
    with ab.Solver(ab._with_rank(Z, G), zn) as s:
        s.set_state(G)
        for subs in (skew, unif, unif[:0], unif[:1]):
            got = s.model_at(1, subs)
            ref = model_at(subs, U)
            assert got.shape == ref.shape
            if subs.shape[0]:
                assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-13
        # the caller's order is kept, and each value does not depend on it
        p = rng.permutation(n)
        assert np.array_equal(s.model_at(1, unif[p]), s.model_at(1, unif)[p])


def _dense_em_case(ab, seed=3):
    """example_script12's CP part: a 3-way tensor with missing entries coupled to a matrix; a held-out set of 40 % of
    the missing entries with their true values."""
    Z, G, _ = pg.config_cp_matrix(30, 25, 20, 40, 4, seed=seed)
    Zm = pg.add_missing(Z, 0.3, seed=seed, objects=[0])
    X, W = Z['object'][0], Zm['miss'][0]
    hs = np.argwhere(~W)
    hs = hs[np.random.RandomState(seed).rand(len(hs)) < 0.4]
    return Zm, G, [ab.sptensor(hs, X[tuple(hs.T)], X.shape), None]


def _sparse_em_case(ab, seed=1):
    """A masked sparse matrix coupled to a dense side matrix; a held-out set of unobserved entries."""
    Z, G, _ = _matrix_pair(I=60, J=50, M=40, R=5, seed=seed)
    S, Mk, H = _split(ab, Z['object'][0], 0.4, 0.3, np.random.RandomState(seed))
    return dict(Z, object=[S, Z['object'][1]], miss=[Mk, None]), G, [H, None]


def _dense_twin(Z):
    """The dense EM problem equal to a masked sparse one (full(S) + dense mask) for the oracle."""
    obj, miss = list(Z['object']), list(Z['miss'])
    for p, (x, m) in enumerate(zip(obj, miss)):
        if hasattr(x, 'full'):
            obj[p], miss[p] = x.full(), np.asfortranarray(m.full() != 0)
    return dict(Z, object=obj, miss=miss)


def _zn(ab, Z):
    zd = pg.znorm_const(_dense_twin(Z))
    return [float('nan') if ab.as_sparse(x) is not None else z for x, z in zip(Z['object'], zd)]


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['dense_em', 'sparse_em'])
def test_heldout_history_matches_oracle(ab, case):
    _need_gpu(ab)
    Z, G, held = (_dense_em_case if case == 'dense_em' else _sparse_em_case)(ab)
    n = 6
    opts = pg.default_options(MaxOuterIters=n, **ZERO_TOL)
    Gd, od = ab.cmtf_fun_AOADMM(Z, _zn(ab, Z), G, None, None, None, None, opts, heldout=held)
    H = held[0]
    assert od['heldout_sse'][1] is None and od['heldout_count'] == [len(np.unique(H.subs, axis=0)), None]
    hist = od['heldout_sse'][0]
    assert hist.shape == (n + 1,)
    Zd = _dense_twin(Z)
    zd = pg.znorm_const(Zd)
    modes = Z['modes'][0]
    ref = []
    for k in range(n + 1):
        fac = G['fac'] if k == 0 else oracle_solve(Zd, zd, G, options=dict(opts, MaxOuterIters=k))[0]['fac']
        m = model_at(H.subs, [fac[i - 1] for i in modes])
        ref.append(np.sum((H.vals - m) ** 2))
    ref = np.asarray(ref)
    assert np.max(np.abs(hist - ref) / ref) <= 1e-10, (hist, ref)
    # the device history is the error of the returned factors
    last = np.sum((H.vals - model_at(H.subs, [Gd['fac'][i - 1] for i in modes])) ** 2)
    assert abs(hist[-1] - last) <= 1e-12 * last


def _bitwise(Ga, Gb):
    for key in ('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac'):
        for a, b in zip(Ga[key], Gb[key]):
            assert (a is None and b is None) or np.array_equal(a, b), key


def _same_out(oa, ob):
    assert set(oa) == set(ob)
    for k, v in oa.items():
        if k == 'time_at_it':
            continue
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, ob[k], equal_nan=True), k
        elif isinstance(v, float) and np.isnan(v):
            assert np.isnan(ob[k]), k
        else:
            assert v == ob[k], k


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['dense_em', 'sparse_em'])
def test_heldout_set_leaves_the_solve_bit_identical(ab, case):
    _need_gpu(ab)
    Z, G, held = (_dense_em_case if case == 'dense_em' else _sparse_em_case)(ab)
    zn = _zn(ab, Z)
    opts = pg.default_options(MaxOuterIters=10, **ZERO_TOL)
    base = {}
    for g in (1, -1):
        Gp, op = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, dict(opts, graph=g))
        Gh, oh = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, dict(opts, graph=g), heldout=held)
        _bitwise(Gp, Gh)
        hist = oh.pop('heldout_sse')
        oh.pop('heldout_count')
        _same_out(op, oh)
        base[g] = (Gp, op, hist[0])
    _bitwise(base[1][0], base[-1][0])
    assert np.array_equal(base[1][2], base[-1][2])
    # the order of the held-out entries does not change a bit of the history
    H = held[0]
    p = np.random.RandomState(0).permutation(H.nnz)
    _, oq = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts,
                               heldout=[ab.sptensor(H.subs[p], H.vals[p], H.shape), None])
    assert np.array_equal(oq['heldout_sse'][0], base[1][2])
    # duplicates are summed: every value split into two exact halves gives the same set
    dup = ab.sptensor(np.vstack([H.subs, H.subs]), np.r_[0.5 * H.vals, 0.5 * H.vals], H.shape)
    _, od = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, heldout=[dup, None])
    assert od['heldout_count'][0] == oq['heldout_count'][0] == H.nnz
    assert np.array_equal(od['heldout_sse'][0], base[1][2])


def _raw_set(ab, s, obj, subs, vals):
    c = ab._capi
    so, keep = ab._coo(np.asarray(subs, dtype=np.int64), np.asarray(vals, dtype=np.float64))
    rc = c.lib.aoadmm_set_heldout(s._h, obj, ctypes.byref(so))
    return rc, c.lib.aoadmm_last_error(s._h).decode()


@pytest.mark.gpu
def test_invalid_heldout_sets(ab):
    _need_gpu(ab)
    # dense mask: a held-out entry whose mask byte is set
    Z, G, held = _dense_em_case(ab)
    W = Z['miss'][0]
    obs = np.argwhere(W)[7]
    with ab.Solver(ab._with_rank(Z, G), pg.znorm_const(Z)) as s:
        s.set_state(G)
        H = held[0]
        rc, err = _raw_set(ab, s, 1, np.vstack([H.subs, obs]), np.r_[H.vals, 1.0])
        assert rc == INVALID and 'object 1' in err and 'observed' in err and '(%d, %d, %d)' % tuple(obs) in err, err
        rc, err = _raw_set(ab, s, 1, np.vstack([H.subs, [30, 0, 0]]), np.r_[H.vals, 1.0])   # out of range
        assert rc == INVALID and 'out of range' in err, err
        rc, err = _raw_set(ab, s, 2, [[0, 0]], [1.0])                                          # no Z.miss
        assert rc == INVALID and 'no missing data' in err, err
        rc, err = _raw_set(ab, s, 3, [[0, 0]], [1.0])
        assert rc == INVALID and 'out of range' in err, err
        s.set_heldout(1, H)     # a valid set after the refusals
        s.run(pg.default_options(MaxOuterIters=2))
        sse, count = s.heldout_history(1)
        assert sse.shape == (3,) and count == H.nnz and np.all(np.isfinite(sse))
        s.set_heldout(1, None)
        with pytest.raises(ab.AoadmmError):
            s.heldout_history(1)
    # sparse object: a held-out entry that is stored
    Z, G, held = _sparse_em_case(ab)
    with ab.Solver(ab._with_rank(Z, G), _zn(ab, Z)) as s:
        s.set_state(G)
        H, stored = held[0], Z['object'][0].subs[3]
        rc, err = _raw_set(ab, s, 1, np.vstack([H.subs, stored]), np.r_[H.vals, 1.0])
        assert rc == INVALID and 'object 1' in err and '(%d, %d)' % tuple(stored) in err, err
        # model_at works on every object, held-out set or not
        assert s.model_at(2, [[0, 0], [1, 2]]).shape == (2,)


@pytest.mark.gpu
def test_multi_gpu_history_equals_one_gpu(ab):
    if ab.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    Z, G, held = _dense_em_case(ab, seed=5)
    zn = pg.znorm_const(Z)
    opts = pg.default_options(MaxOuterIters=6, **ZERO_TOL)
    _, o1 = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, heldout=held)
    _, o2 = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, heldout=held, n_gpus=2)
    a, b = o1['heldout_sse'][0], o2['heldout_sse'][0]
    assert np.max(np.abs(a - b) / a) <= 1e-12
