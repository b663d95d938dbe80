"""Early stopping on the held-out error (aoadmm_set_heldout_stopping / aoadmm_heldout_best).

CPU tests restate the rule in NumPy on crafted histories, check every refusal that happens before a device is touched
and the signatures of the two entry points.  GPU tests (-m gpu) take problems whose held-out error provably rises (rank
three times the true rank, 70 % missing, noise 0.5), check that the rule fired, and compare the early-stopped handle bit
for bit with a handle run from the same G with MaxOuterIters = k*: the state, the f_* values, the histories up to k* and
a further run of both."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import problem_gen as pg
from _cases import ZERO_TOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 1
NAN = float('nan')


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('s,P,want', [
    ([9, 8, 7, 6, 5, 4], 1, (5, None)),            # monotone decrease: the last iteration, the rule never fires
    ([9, 3, 4, 5, 6, 7], 2, (1, 3)),               # an immediate rise: k* = 1
    ([9, 3, 4, 5, 6, 7], 1, (1, 2)),
    ([9, 5, 4, 4, 4, 3], 2, (2, 4)),               # ties are no new best
    ([9, 5, 4, 4, 3, 3], 3, (4, None)),
    ([9, NAN, 5, NAN, NAN, 6], 2, (2, 4)),         # NaN is never a new best
    ([9, NAN, NAN, 5, 4, 6], 1, (4, 5)),
    ([9, NAN, NAN, NAN], 1, (3, None)),            # no number at all: k* = n, nothing fires
    ([9, 1, 2, 3], 10, (1, None)),                 # patience longer than the run
    ([9], 1, (0, None)),                           # n = 0
    ([1, 2, 3, 4], 2, (1, 3)),                     # iteration 0 is not a candidate
])
def test_rule_on_crafted_histories(ab, s, P, want):
    assert ab.heldout_stopping_rule(s, P) == want


def test_rule_is_the_first_smallest_value_before_the_stop(ab):
    rng = np.random.RandomState(0)
    for _ in range(200):
        n = rng.randint(0, 30)
        s = rng.randint(0, 6, n + 1).astype(float)
        s[rng.rand(n + 1) < 0.2] = NAN
        P = rng.randint(1, 6)
        k, stop = ab.heldout_stopping_rule(s, P)
        end = n if stop is None else stop
        body = s[1:end + 1]
        if np.all(np.isnan(body)):
            assert k == n and stop is None
            continue
        assert k == 1 + int(np.nanargmin(body)) and s[k] == np.nanmin(body)
        if stop is not None:
            assert stop - k == P
        else:
            assert n - k < P or n == 0


def test_heldout_sum_adds_in_object_order(ab):
    a, b, c = np.array([1e16, 1.0]), np.array([1.0, 1e16]), np.array([-1e16, -1e16])
    got = ab._heldout_sum([a, b, c])
    assert got[0] == (1e16 + 1.0) + -1e16 and got[1] == (1.0 + 1e16) + -1e16


def _matrix_pair(I=40, J=30, M=25, R=2, seed=4, noise=0.5):
    rng = np.random.RandomState(seed)
    coupling = {'lin_coupled_modes': [1, 0, 1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 4}
    return pg._finish(['CP', 'CP'], [I, J, I, M], [[1, 2], [3, 4]], [[1.0] * R] * 2, [noise] * 2, coupling,
                      [pg.d_rand] * 4, [0] * 4, [None] * 4, [0.5, 0.5], rng)


def _overrank(Z, R, seed):
    """A random initial G of rank R for the objects of Z."""
    rng = np.random.RandomState(seed + 100)
    init = {'lambdas_init': [[1.0] * R] * len(Z['modes']), 'nvecs': 0, 'distr': [pg.d_rand] * len(Z['size']),
            'normalize': 1}
    return pg.init_coupled_AOADMM_CMTF(Z, init, rng)


def _held(ab, Z, Zm, seed):
    """Half of the missing entries of object 1 with their true values."""
    X, W = Z['object'][0], Zm['miss'][0]
    hs = np.argwhere(~W)
    hs = hs[np.random.RandomState(seed).rand(len(hs)) < 0.5]
    return [ab.sptensor(hs, X[tuple(hs.T)], X.shape)] + [None] * (len(Z['modes']) - 1)


def _sparse(ab, Zm, p=0):
    """Object p of a dense EM problem as a masked sparse object: the observed entries and their pattern."""
    X, W = Zm['object'][p], Zm['miss'][p]
    ts = np.argwhere(W)
    obj, miss = list(Zm['object']), list(Zm['miss'])
    obj[p] = ab.sptensor(ts, X[W], X.shape)
    miss[p] = ab.sptensor(ts, np.ones(len(ts)), X.shape)
    return dict(Zm, object=obj, miss=miss)


def _zn(ab, Z, Zdense):
    zd = pg.znorm_const(Zdense)
    return [NAN if ab.as_sparse(x) is not None else z for x, z in zip(Z['object'], zd)]


def case(ab, name):
    """(Z, Znorm_const, G, heldout) of a problem whose held-out error rises after about ten outer iterations."""
    if name == 'par2':                       # example_script12: CP + PARAFAC2, both with missing entries
        Z, _, _ = pg.config_cp_par2(I=16, J=14, K=12, Jk=10, Kp=8, R=3, seed=5, noise=0.5)
        G = _overrank(Z, 9, 5)
        Zm = pg.add_missing(Z, 0.7, seed=5, objects=[0, 1])
        return Zm, pg.znorm_const(Zm), G, _held(ab, Z, Zm, 5)
    if name == 'sparse_matrix':              # a masked sparse matrix coupled to a dense side matrix
        Z, _, _ = _matrix_pair()
        G = _overrank(Z, 6, 4)
        Zm = pg.add_missing(Z, 0.7, seed=4, objects=[0])
        Zs = _sparse(ab, Zm)
        return Zs, _zn(ab, Zs, Zm), G, _held(ab, Z, Zm, 4)
    Z, _, _ = pg.config_cp_matrix(16, 14, 12, 20, 3, seed=2, noise=0.5)
    G = _overrank(Z, 9, 2)
    Zm = pg.add_missing(Z, 0.7, seed=2, objects=[0])
    held = _held(ab, Z, Zm, 2)
    if name == 'dense':                      # a dense 3-way EM tensor coupled to a matrix
        return Zm, pg.znorm_const(Zm), G, held
    Zt = {k: (v[:1] if isinstance(v, list) and len(v) == 2 else v) for k, v in Zm.items()}   # the tensor alone
    Zt.update(size=Zm['size'][:3], coupling={'lin_coupled_modes': [0, 0, 0], 'coupling_type': [],
                                             'coupl_trafo_matrices': [None] * 3},
              constrained_modes=Zm['constrained_modes'][:3], constraints=Zm['constraints'][:3], weights=[1.0])
    Gt = {k: (v[:3] if k in ('fac', 'constraint_fac', 'constraint_dual_fac') else [None] * 3 if k == 'coupling_dual_fac'
              else [] if k == 'coupling_fac' else v[:1]) for k, v in G.items()}
    Zs = _sparse(ab, Zt)                     # a 3-way masked sparse tensor
    return Zs, _zn(ab, Zs, Zt), Gt, held[:1]


def test_python_refusals_happen_before_any_device_call(ab, monkeypatch):
    Z, zn, G, held = case(ab, 'dense')
    opts = pg.default_options(MaxOuterIters=2)

    def no_device(*a, **k):
        raise AssertionError('a device call was made')
    monkeypatch.setattr(ab, 'Solver', no_device)
    for kw, msg in [(dict(heldout_patience=2), 'needs a held-out set'),
                    (dict(heldout=[None, None], heldout_patience=2), 'needs a held-out set'),
                    (dict(heldout=held, heldout_patience=-1), '>= 0')]:
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, **kw)
        assert e.value.status_name == 'INVALID_ARG' and msg in str(e.value), str(e.value)


def test_header_and_ctypes_signatures(ab):
    c = ab._capi
    hdr = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    want = {
        'aoadmm_set_heldout_stopping': (r'int aoadmm_set_heldout_stopping\(aoadmm_handle \*h, int32_t patience\);',
                                        [c.HandleP, ctypes.c_int32]),
        'aoadmm_heldout_best': (r'int aoadmm_heldout_best\(const aoadmm_handle \*h, int32_t \*iteration, double \*sse\);',
                                [c.HandleP, c.c_int32_p, c.c_double_p]),
    }
    for name, (proto, argtypes) in want.items():
        assert re.search(proto, hdr), name
        assert name in c.EXPORTS
        assert list(getattr(c.lib, name).argtypes) == argtypes, name
    k, s = ctypes.c_int32(), ctypes.c_double()
    assert c.lib.aoadmm_set_heldout_stopping(None, 1) == INVALID
    assert c.lib.aoadmm_set_heldout_stopping(None, 0) == INVALID
    assert c.lib.aoadmm_heldout_best(None, ctypes.byref(k), ctypes.byref(s)) == INVALID
    assert '1 << 9' in hdr and 'heldoutStop' in open(os.path.join(ROOT, 'matlab-code_b200', 'matlab',
                                                                    'aoadmm_mex.cpp')).read()


# ---------------------------------------------------------------------------------------------- GPU
def _need_gpu(ab):
    assert ab.device_count() >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'


def _same_state(Ga, Gb):
    assert set(Ga) == set(Gb)
    for key in Ga:
        for a, b in zip(Ga[key], Gb[key]):
            if isinstance(a, list):
                assert all(np.array_equal(x, y) for x, y in zip(a, b)), key
            else:
                assert (a is None and b is None) or np.array_equal(a, b), key


def _same_out(oa, ob, drop=('time_at_it',)):
    assert set(oa) - set(drop) == set(ob) - set(drop)
    for k, v in oa.items():
        if k in drop:
            continue
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, ob[k], equal_nan=True), k
        elif isinstance(v, float) and np.isnan(v):
            assert np.isnan(ob[k]), k
        else:
            assert v == ob[k], k


F_FIELDS = ('f_tensors', 'f_couplings', 'f_constraints', 'f_PAR2_couplings', 'f_rel_missing')
HISTORIES = ('func_val_conv', 'func_coupl_conv', 'func_constr_conv', 'func_PAR2_coupl', 'func_rel_missing')


def _solve(ab, Z, zn, G, held, opts, patience=None, more=3, **dist):
    """A run (with stopping when patience is set), its state, k* / s_k*, then `more` iterations with stopping off."""
    with ab.Solver(ab._with_rank(Z, G), zn, **dist) as s:
        s.set_state(G)
        for p, X in enumerate(held):
            if X is not None:
                s.set_heldout(p + 1, X)
        if patience:
            s.set_heldout_stopping(patience)
        o1 = s.run(opts)
        best = s.heldout_best() if patience else None
        G1 = s.get_state()
        s.set_heldout_stopping(0)
        o2 = s.run(dict(opts, MaxOuterIters=more))
        G2 = s.get_state()
    return o1, G1, best, o2, G2


def _check_against_truncated(ab, Z, zn, G, held, opts, patience, expect_flag, **dist):
    oa, Ga, (k, sk), oa2, Ga2 = _solve(ab, Z, zn, G, held, opts, patience, **dist)
    n = oa['OuterIterations']
    assert k < n, (k, n)
    assert oa['exit_flag'] == expect_flag
    hs = oa['func_val_conv']   # the histories describe the n iterations run
    assert len(hs) == n + 1
    ob, Gb, _, ob2, Gb2 = _solve(ab, Z, zn, G, held, dict(opts, MaxOuterIters=k), **dist)
    assert ob['OuterIterations'] == k
    _same_state(Ga, Gb)
    for f in F_FIELDS:
        assert np.array_equal(oa[f], ob[f], equal_nan=True), f
        assert np.array_equal(oa[f], oa[HISTORIES[F_FIELDS.index(f)]][k], equal_nan=True), f
    for h in HISTORIES:
        assert np.array_equal(oa[h][:k + 1], ob[h], equal_nan=True), h
    assert np.array_equal(oa['innerIters'][:, :k], ob['innerIters'])
    # the imputation state and every carried buffer were restored: a further run stays bit-identical
    _same_state(Ga2, Gb2)
    _same_out(oa2, ob2)
    return k, n, sk


GPU_CASES = [('dense', {}), ('dense', dict(dimtree=1)), ('dense', dict(bsum=1, bsum_weight=0.1)),
             ('sparse_matrix', {}), ('sparse_tensor', {}), ('par2', {})]


@pytest.mark.gpu
@pytest.mark.parametrize('graph', [1, -1])
@pytest.mark.parametrize('name,extra', GPU_CASES, ids=['dense', 'dense-dimtree', 'dense-bsum', 'sparse_matrix',
                                                       'sparse_tensor', 'par2'])
def test_early_stopped_state_equals_the_truncated_run(ab, name, extra, graph):
    _need_gpu(ab)
    Z, zn, G, held = case(ab, name)
    opts = pg.default_options(MaxOuterIters=40, graph=graph, **ZERO_TOL, **extra)
    k, n, sk = _check_against_truncated(ab, Z, zn, G, held, opts, 3, 'heldoutStop')
    assert n == k + 3
    # the Python front end reports the same iteration and flag
    _, o = ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, heldout=held, heldout_patience=3)
    assert o['heldout_best_iter'] == k and o['exit_flag'] == 'heldoutStop' and o['OuterIterations'] == n
    total = ab._heldout_sum([h for h in o['heldout_sse'] if h is not None])
    assert total[k] == sk and ab.heldout_stopping_rule(total, 3) == (k, n)


@pytest.mark.gpu
def test_run_ended_by_max_iterations_is_restored(ab):
    _need_gpu(ab)
    Z, zn, G, held = case(ab, 'dense')
    opts = pg.default_options(MaxOuterIters=18, **ZERO_TOL)
    k, n, _ = _check_against_truncated(ab, Z, zn, G, held, opts, 1000, 'maxIterations')
    assert n == 18
    # k* = n: nothing is restored and the run equals the plain run bit for bit
    oa, Ga, best, oa2, Ga2 = _solve(ab, Z, zn, G, held, dict(opts, MaxOuterIters=k), 1000)
    ob, Gb, _, ob2, Gb2 = _solve(ab, Z, zn, G, held, dict(opts, MaxOuterIters=k))
    assert best[0] == k
    _same_state(Ga, Gb)
    _same_out(oa, ob)
    _same_state(Ga2, Gb2)
    _same_out(oa2, ob2)


@pytest.mark.gpu
def test_stopping_turned_off_again_changes_nothing(ab):
    _need_gpu(ab)
    Z, zn, G, held = case(ab, 'sparse_matrix')
    opts = pg.default_options(MaxOuterIters=25, **ZERO_TOL)
    ob, Gb, _, ob2, Gb2 = _solve(ab, Z, zn, G, held, opts)
    with ab.Solver(ab._with_rank(Z, G), zn) as s:
        s.set_state(G)
        s.set_heldout(1, held[0])
        s.set_heldout_stopping(3)
        s.set_heldout_stopping(None)
        oa = s.run(opts)
        with pytest.raises(ab.AoadmmError) as e:
            s.heldout_best()
        assert e.value.status_name == 'INVALID_ARG'
        _same_state(s.get_state(), Gb)
        _same_out(oa, ob)
        # stopping on, then every held-out set detached: the run is refused before any device work
        s.set_heldout_stopping(2)
        s.set_heldout(1, None)
        with pytest.raises(ab.AoadmmError) as e:
            s.run(opts)
        assert e.value.status_name == 'INVALID_ARG'
        _same_state(s.get_state(), Gb)
        # refusals of the entry point itself
        with pytest.raises(ab.AoadmmError) as e:
            s.set_heldout_stopping(1)                      # no held-out set attached
        assert e.value.status_name == 'INVALID_ARG'
        with pytest.raises(ab.AoadmmError) as e:
            s.set_heldout_stopping(-1)
        assert e.value.status_name == 'INVALID_ARG'
    # n = 0: k* = 0 and s_0
    with ab.Solver(ab._with_rank(Z, G), zn) as s:
        s.set_state(G)
        s.set_heldout(1, held[0])
        s.set_heldout_stopping(1)
        s.run(dict(opts, MaxOuterIters=0))
        k, s0 = s.heldout_best()
        assert k == 0 and s0 == s.heldout_history(1)[0][0]


def _free_bytes():
    cudart = ctypes.CDLL('libcudart.so')
    f, t = ctypes.c_size_t(), ctypes.c_size_t()
    assert cudart.cudaMemGetInfo(ctypes.byref(f), ctypes.byref(t)) == 0
    return f.value


@pytest.mark.gpu
def test_destroy_frees_the_snapshot(ab):
    _need_gpu(ab)
    Z, zn, G, held = case(ab, 'dense')
    opts = pg.default_options(MaxOuterIters=20, **ZERO_TOL)
    ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, heldout=held, heldout_patience=3)   # warm-up
    before = _free_bytes()
    ab.cmtf_fun_AOADMM(Z, zn, G, None, None, None, None, opts, heldout=held, heldout_patience=3)
    assert _free_bytes() == before


@pytest.mark.gpu
@pytest.mark.parametrize('name,kw', [('dense', {}), ('sparse_matrix', dict(shard_sparse=True))])
def test_two_gpus_early_stopped_state_equals_the_truncated_run(ab, name, kw):
    if ab.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    Z, zn, G, held = case(ab, name)
    opts = pg.default_options(MaxOuterIters=40, **ZERO_TOL)
    _check_against_truncated(ab, Z, zn, G, held, opts, 3, 'heldoutStop', n_gpus=2, **kw)
