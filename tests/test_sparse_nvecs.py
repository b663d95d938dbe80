"""nvecs of sparse modes (aoadmm_nvecs_sparse, Solver.nvecs_sparse, cmtf_nvecs_sparse, init_options['nvecs_sparse']):
the leading eigenvectors of X_(n) X_(n)' from the fiber-compressed unfolding, against the oracle's cmtf_nvecs on
full(S), the dense engine on full(S) and, where no dense form is possible, SciPy eigsh on the CSR unfolding."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import problem_gen as pg
from _cases import ZERO_TOL, assert_state_close
from test_gpu_parity import _nvecs_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _Z(X):
    N = len(X.shape)
    return {'loss_function': ['Frobenius'], 'model': ['CP'], 'modes': [list(range(1, N + 1))], 'size': list(X.shape),
            'coupling': {'lin_coupled_modes': [0] * N, 'coupling_type': [], 'coupl_trafo_matrices': [None] * N},
            'constrained_modes': [0] * N, 'constraints': [None] * N, 'weights': [1.0], 'object': [X]}


def _coo(shape, density, rng):
    """distinct uniform subscripts at the given density, standard normal values"""
    total = int(np.prod(shape))
    lin = rng.choice(total, size=max(1, int(density * total)), replace=False)
    subs = np.stack(np.unravel_index(lin, shape, order='F'), axis=1).astype(np.int64)
    return subs, rng.randn(len(lin))


def _pair(ab, subs, vals, shape):
    S = ab.sptensor(subs, vals, shape)
    return _Z(S), _Z(np.asfortranarray(S.full()))


# ---------------------------------------------------------------------------------------------- CPU
def test_refusals_before_any_device_call(ab):
    Zd = _Z(np.ones((4, 3, 2), order='F'))
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_nvecs_sparse(Zd, 1, 2)
    assert e.value.status_name == 'INVALID_ARG' and 'nvecs' in str(e.value)
    Zp, _, _ = pg.config_single_par2(I=6, Jk=(5, 4), R=2, seed=0)
    for n in (1, 2, 3):
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_nvecs_sparse(Zp, n, 1)
        assert e.value.status_name == 'INVALID_ARG'
    Zs = _Z(ab.sptensor(np.array([[0, 1, 1]]), np.array([2.0]), (4, 3, 2)))
    for n, r in ((1, 0), (1, 5), (3, 3), (0, 1), (4, 1)):
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_nvecs_sparse(Zs, n, r)
        assert e.value.status_name == 'INVALID_ARG', (n, r)
    # the method runs the same checks before it reaches the handle (none exists here)
    s = object.__new__(ab.Solver)
    s.Z, s._h = Zd, None
    with pytest.raises(ab.AoadmmError) as e:
        s.nvecs_sparse(1, 1)
    assert e.value.status_name == 'INVALID_ARG'


def test_nvecs_sparse_option_is_ignored_without_nvecs(ab):
    rng = np.random.RandomState(0)
    subs, vals = _coo((6, 5, 4), 0.3, rng)
    Z = dict(_Z(ab.sptensor(subs, vals, (6, 5, 4))), rank=[2])
    ra, rb = np.random.RandomState(3), np.random.RandomState(3)
    io = {'lambdas_init': [[1.0] * 2], 'normalize': 1}
    Ga = ab.init_coupled_AOADMM_CMTF(Z, dict(io, nvecs=0, distr=[lambda a, b: ra.rand(a, b)] * 3), rng=ra)
    Gb = ab.init_coupled_AOADMM_CMTF(Z, dict(io, nvecs=0, nvecs_sparse=1, distr=[lambda a, b: rb.rand(a, b)] * 3), rng=rb)
    for a, b in zip(Ga['fac'], Gb['fac']):
        assert np.array_equal(a, b)


def test_mex_gateway_and_shim_sources():
    header = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    declared = set(re.findall(r'\b(aoadmm_[a-z_0-9]+)\s*\(', header))
    src = os.path.join(ROOT, 'matlab-code_b200', 'matlab', 'aoadmm_nvecs_sparse_mex.cpp')
    subprocess.check_call(['g++', '-std=c++17', '-fsyntax-only', '-Wall', '-I', os.path.join(ROOT, 'tests', 'stubs'),
                           '-I', os.path.join(ROOT, 'include'), src])
    used = set(re.findall(r'\b(aoadmm_[a-z_0-9]+)\s*\(', open(src).read())) - {'aoadmm_nvecs_sparse_mex'}
    assert 'aoadmm_nvecs_sparse' in used and 'aoadmm_create_sparse' in used and used <= declared, used - declared
    m = open(os.path.join(ROOT, 'matlab-code_b200', 'matlab', 'cmtf_nvecs_sparse.m')).read()
    assert m.startswith('function U = cmtf_nvecs_sparse(Z,n,r)')


# ---------------------------------------------------------------------------------------------- GPU
SHAPES = [((30, 20), 0.3), ((12, 10, 9), 0.2), ((9, 8, 7, 6), 0.1), ((7, 6, 5, 4, 3), 0.05), ((5, 4, 3, 3, 2, 2), 0.3),
          ((4, 3, 3, 2, 2, 2, 2), 0.3), ((3, 3, 2, 2, 2, 2, 2, 2), 0.3)]


@pytest.mark.gpu
@pytest.mark.parametrize('shape,density', SHAPES)
def test_parity_every_mode_position(ab, shape, density):
    """every mode position of 2..8-way sparse objects against the oracle and the dense engine on full(S)"""
    subs, vals = _coo(shape, density, np.random.RandomState(len(shape)))
    Zs, Zd = _pair(ab, subs, vals, shape)
    with ab.Solver(dict(Zs, rank=[3]), [float('nan')]) as s, ab.Solver(dict(Zd, rank=[3]), [float('nan')]) as d:
        for n in range(1, len(shape) + 1):
            r = min(3, shape[n - 1])
            U, info = s.nvecs_sparse(n, r, return_info=True)
            _nvecs_close(U, pg.cmtf_nvecs(Zd, n, r), Zd, n)
            _nvecs_close(U, d.nvecs(n, r), Zd, n)
            assert info['residual'] < 1e-12, (n, info)


@pytest.mark.gpu
def test_column_chunks_whole_space_block_and_r_equal_n(ab):
    """r = 200 on a 300-row mode (block of 250 columns: four column chunks), a 40-row mode (whole-space path) with r = n"""
    shape = (300, 40, 9)
    subs, vals = _coo(shape, 0.2, np.random.RandomState(5))
    Zs, Zd = _pair(ab, subs, vals, shape)
    with ab.Solver(dict(Zs, rank=[200]), [float('nan')]) as s:
        for n, r in ((1, 200), (2, 40), (3, 9)):
            U, info = s.nvecs_sparse(n, r, return_info=True)
            _nvecs_close(U, pg.cmtf_nvecs(Zd, n, r), Zd, n)
            assert info['residual'] < 1e-12, (n, info)


def _structure_case(kind, rng):
    shape = (20, 15, 12)
    if kind == 'duplicates':     # duplicates are summed
        subs, vals = _coo(shape, 0.15, rng)
        pick = rng.randint(0, len(vals), 200)
        return np.vstack([subs, subs[pick]]), np.r_[vals, rng.randn(200)], shape
    if kind == 'explicit_zeros':
        subs, vals = _coo(shape, 0.15, rng)
        vals[::5] = 0.0
        return subs, vals, shape
    if kind == 'empty_rows':     # rows 0, 7 and the last of every mode are empty
        subs, vals = _coo(shape, 0.2, rng)
        keep = np.all([(subs[:, d] != 0) & (subs[:, d] != 7) & (subs[:, d] != shape[d] - 1) for d in range(3)], axis=0)
        return subs[keep], vals[keep], shape
    # single_fibers: every fiber of mode 1 holds one nonzero (distinct (j, k) per entry)
    jk = rng.choice(15 * 12, size=120, replace=False)
    subs = np.stack([rng.randint(0, 20, 120), jk % 15, jk // 15], axis=1).astype(np.int64)
    return subs, rng.randn(120), shape


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['duplicates', 'explicit_zeros', 'empty_rows', 'single_fibers'])
def test_structure(ab, kind):
    subs, vals, shape = _structure_case(kind, np.random.RandomState(7))
    Zs, Zd = _pair(ab, subs, vals, shape)
    with ab.Solver(dict(Zs, rank=[4]), [float('nan')]) as s:
        for n in (1, 2, 3):
            U, info = s.nvecs_sparse(n, 4, return_info=True)
            _nvecs_close(U, pg.cmtf_nvecs(Zd, n, 4), Zd, n)
            assert info['residual'] < 1e-12, (n, info)


@pytest.mark.gpu
def test_no_nonzeros_gives_orthonormal_columns(ab):
    Zs = _Z(ab.sptensor(np.zeros((0, 3), dtype=np.int64), np.zeros(0), (30, 20, 10)))
    with ab.Solver(dict(Zs, rank=[3]), [float('nan')]) as s:
        for n in (1, 2, 3):
            U = s.nvecs_sparse(n, 3)
            assert U.shape == (Zs['size'][n - 1], 3)
            assert np.linalg.norm(U.T @ U - np.eye(3)) < 1e-12


@pytest.mark.gpu
def test_rank_deficient_data_spans_the_true_factors(ab):
    """noise-free rank-3 data with sparse factor supports: Y has 3 nonzero eigenvalues, the block is rank deficient"""
    rng = np.random.RandomState(11)
    F = [rng.rand(s, 3) * (rng.rand(s, 3) < 0.4) for s in (90, 40, 50)]
    X = np.einsum('ir,jr,kr->ijk', *F)
    subs = np.argwhere(X != 0)
    Zs, Zd = _pair(ab, subs, X[X != 0], X.shape)
    for n in (1, 2, 3):
        U = ab.cmtf_nvecs_sparse(Zs, n, 3)
        _nvecs_close(U, pg.cmtf_nvecs(Zd, n, 3))
        assert np.linalg.norm(F[n - 1] - U @ (U.T @ F[n - 1])) < 1e-10 * np.linalg.norm(F[n - 1])


@pytest.mark.gpu
def test_invariance_and_untouched_handle_state(ab):
    """permuted and split-duplicate nonzeros give the same bits; two calls give the same bits; a solve after the call is
    bit-identical to one without it; the device memory free after the call equals the memory free before it"""
    import torch
    shape = (60, 50, 40)
    rng = np.random.RandomState(9)
    subs, vals = _coo(shape, 0.05, rng)
    vals = np.round(vals * 1024) / 1024            # dyadic values: a split into two halves sums back exactly
    perm = rng.permutation(len(vals))
    half = rng.rand(len(vals)) < 0.3
    subs2 = np.vstack([subs[perm], subs[half]])
    vals2 = np.r_[np.where(half, vals / 2, vals)[perm], vals[half] / 2]
    Za, _ = _pair(ab, subs, vals, shape)
    Zb, _ = _pair(ab, subs2, vals2, shape)
    R = 4
    io = {'lambdas_init': [[1.0] * R], 'nvecs': 0, 'normalize': 1,
          'distr': [lambda a, b: np.random.RandomState(a * 7 + b).rand(a, b)] * 3}
    G = ab.init_coupled_AOADMM_CMTF(dict(Za, rank=[R]), io, rng=np.random.RandomState(2))
    opts = pg.default_options(MaxOuterIters=4, **ZERO_TOL)
    with ab.Solver(dict(Za, rank=[R]), [float('nan')]) as a, ab.Solver(dict(Zb, rank=[R]), [float('nan')]) as b:
        for n in (1, 2, 3):
            Ua = a.nvecs_sparse(n, 5)
            assert np.array_equal(Ua, b.nvecs_sparse(n, 5)), n
            free0 = torch.cuda.mem_get_info(0)[0]
            assert np.array_equal(Ua, a.nvecs_sparse(n, 5)), n
            assert torch.cuda.mem_get_info(0)[0] == free0
        a.set_state(G)
        a.run(opts)
        Fa = a.get_state()
    with ab.Solver(dict(Za, rank=[R]), [float('nan')]) as c:
        c.set_state(G)
        c.run(opts)
        Fc = c.get_state()
    for x, y in zip(Fa['fac'], Fc['fac']):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_masked_object_uses_the_observed_values_before_and_after_a_run(ab):
    shape = (25, 20, 15)
    subs, vals = _coo(shape, 0.2, np.random.RandomState(4))
    Zs, Zd = _pair(ab, subs, vals, shape)
    Zm = dict(Zs, miss=[ab.sptensor(subs, np.ones(len(vals)), shape)], rank=[3])
    rr = np.random.RandomState(1)
    io = {'lambdas_init': [[1.0] * 3], 'nvecs': 0, 'normalize': 1, 'distr': [lambda a, b: rr.rand(a, b)] * 3}
    G = ab.init_coupled_AOADMM_CMTF(Zm, io, rng=rr)
    with ab.Solver(Zm, [float('nan')]) as s:
        before = [s.nvecs_sparse(n, 3) for n in (1, 2, 3)]
        s.set_state(G)
        s.run(pg.default_options(MaxOuterIters=3, **ZERO_TOL))
        for n in (1, 2, 3):
            _nvecs_close(before[n - 1], pg.cmtf_nvecs(Zd, n, 3), Zd, n)
            assert np.array_equal(before[n - 1], s.nvecs_sparse(n, 3)), n


@pytest.mark.gpu
def test_no_dense_reference_possible_against_eigsh(ab):
    """2^17 x 2^12 x 2^8 with about 2e6 nonzeros (its dense form would need 1 PB): modes 1 and 3 against SciPy eigsh on
    the CSR unfolding; host-computed residuals"""
    sps = pytest.importorskip('scipy.sparse')
    sla = pytest.importorskip('scipy.sparse.linalg')
    rng = np.random.RandomState(12)
    shape = (1 << 17, 1 << 12, 1 << 8)
    nnz = 2_000_000
    subs = np.stack([rng.randint(0, s, nnz) for s in shape], axis=1).astype(np.int64)
    F = [rng.rand(s, 4) for s in shape]
    w = np.array([8.0, 4.0, 2.0, 1.0])             # planted rank-4 part with separated weights, plus noise
    vals = np.einsum('er,er,er,r->e', F[0][subs[:, 0]], F[1][subs[:, 1]], F[2][subs[:, 2]], w) + 0.1 * rng.randn(nnz)
    Zs = _Z(ab.sptensor(subs, vals, shape))
    r = 4
    with ab.Solver(dict(Zs, rank=[r]), [float('nan')]) as s:
        for n in (1, 3):
            U, info = s.nvecs_sparse(n, r, return_info=True)
            others = [d for d in range(3) if d != n - 1]
            col = np.ravel_multi_index(tuple(subs[:, d] for d in others), tuple(shape[d] for d in others), order='F')
            _, col = np.unique(col, return_inverse=True)       # columns of the fibers that occur (the others are 0)
            A = sps.csr_matrix((vals, (subs[:, n - 1], col)), shape=(shape[n - 1], int(col.max()) + 1))
            AAt = sla.LinearOperator((shape[n - 1],) * 2, matvec=lambda v: A @ (A.T @ v), dtype=np.float64)
            th, V = sla.eigsh(AAt, k=r + 1, which='LM', tol=0, v0=np.ones(shape[n - 1]))
            order = np.argsort(th)[::-1]
            th, V = th[order], V[:, order]
            for c in range(r):
                v = V[:, c] * np.sign(V[np.argmax(np.abs(V[:, c])), c])
                gap = min(abs(th[c] - th[d]) for d in range(r + 1) if d != c)
                assert np.linalg.norm(U[:, c] - v) < 1e-8 + 2e-13 * th[0] / gap, (n, c)
                u = U[:, c]
                Au = A @ (A.T @ u)
                assert np.linalg.norm(Au - (u @ Au) * u) / th[0] <= 1e-12, (n, c)
            assert info['residual'] < 1e-12, (n, info)


@pytest.mark.gpu
def test_front_end_sparse_tensor_coupled_to_dense_matrix(ab):
    """init_coupled_AOADMM_CMTF with nvecs + nvecs_sparse against the oracle's on the densified Z, then a run from it"""
    Z, _, _ = pg.config_cp_matrix(40, 30, 20, 25, 3, seed=6)
    X = np.asarray(Z['object'][0])
    mask = np.random.RandomState(3).rand(*X.shape) < 0.25
    S = ab.sptensor(np.argwhere(mask), X[mask], X.shape)
    Zs = dict(Z, object=[S] + Z['object'][1:])
    Zd = dict(Z, object=[np.asfortranarray(X * mask)] + Z['object'][1:])
    R = 3
    r1, r2 = np.random.RandomState(21), np.random.RandomState(21)
    io = {'lambdas_init': [[1.0] * R] * 2, 'nvecs': 1, 'normalize': 1}
    Gd = ab.init_coupled_AOADMM_CMTF(Zs, dict(io, nvecs_sparse=1, distr=[lambda a, b: r1.rand(a, b)] * 5), rng=r1)
    Go = pg.init_coupled_AOADMM_CMTF(Zd, dict(io, distr=[pg.d_rand] * 5), r2)
    assert_state_close(Gd, Go, keys=('fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac', 'coupling_fac'))
    _, Fd, _, od = ab.cmtf_AOADMM(Zs, Gd, pg.default_options(MaxOuterIters=5, **ZERO_TOL))
    assert np.isfinite(od['f_tensors']) and all(np.all(np.isfinite(f)) for f in Fd['fac'])


@pytest.mark.gpu
def test_several_gpus(ab):
    if ab.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    shape = (40, 30, 50)
    subs, vals = _coo(shape, 0.1, np.random.RandomState(8))
    Zs, Zd = _pair(ab, subs, vals, shape)
    Zr = dict(Zs, rank=[3])
    with ab.Solver(Zr, [float('nan')]) as one, ab.Solver(Zr, [float('nan')], n_gpus=2, shard_sparse=True) as two:
        for n in (1, 2):
            _nvecs_close(two.nvecs_sparse(n, 3), one.nvecs_sparse(n, 3), Zd, n)
        with pytest.raises(ab.AoadmmError) as e:
            two.nvecs_sparse(3, 3)
        assert e.value.status_name == 'UNSUPPORTED' and 'sharded last mode' in str(e.value)
