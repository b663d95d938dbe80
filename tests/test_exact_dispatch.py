"""Every rank-dispatch branch and tensor orders 2..8 against exact integer references.

With small-integer tensors and factors (entries in [-2, 2]) every path of the engine computes the exact result: the
FP64 kernels while every partial sum stays below 2^53, and the reduced-precision MTTKRPs as well, because TF32 holds
integers up to 2^11 and BF16 up to 2^8 exactly and their FP32 accumulators (one slab of one tile on tcgen05, 128 terms on
mma.sync) stay below 2^24.  The reference is then plain int64 arithmetic and the device must match it bit for bit,
element by element, at every precision, rank and order; the summation order does not matter, so this holds on several
GPUs too.  A tolerance relative to sum |X||F||F| cannot see a dropped or duplicated term of a sum of thousands; an exact
comparison can.

CPU tests check that premise for every GPU case of this file (a bound on the largest partial sum of each path, and each
int64 reference against the same quantity computed in another order) and read the kernels' dispatch thresholds from
the sources, so that the rank lists below keep a rank on both sides of every threshold when a kernel is retuned.
GPU tests (-m gpu) compare the dense, reduced-precision and sparse MTTKRPs, the model at given subscripts and the
held-out SSE with those references, and whole solves at the new edges with the FP64 oracle."""
import functools
import os
import re

import numpy as np
import pytest

from oracle import problem_gen as pg
from oracle.cmtf_fun_aoadmm import cmtf_fun_AOADMM as oracle_solve
from _cases import FIT_TOL, ZERO_TOL, assert_state_close
from test_gpu_parity import _nvecs_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'matlab-code_b200', 'csrc')
FP64_EXACT = 2.0 ** 53
FP32_EXACT = 2.0 ** 24
MMA_SYNC_SPAN = 128          # FP32 terms per accumulator of the TF32 mma.sync variant (mttkrp_precision = 3)
PRECISIONS = {1: 'TF32 tcgen05', 2: 'BF16 tcgen05', 3: 'TF32 mma.sync'}
OPERAND_EXACT = {1: 2 ** 11, 2: 2 ** 8, 3: 2 ** 11}   # largest integer magnitude every smaller one of which is exact

# ---------------------------------------------------------------------------------------------- the cases
# Dense MTTKRP (ab.mttkrp and Solver.object_mttkrp, every mode position): orders 2..8, odd leading extents, partial
# tiles, extent-1 modes, and every chunk width of the FP64 kernels (8 / 16 / 32 / 64 columns, several 64-column chunks).
DENSE_CASES = [
    ((7, 1), 1), ((131, 45), 129), ((45, 1), 256),
    ((33, 17, 5), 8), ((65, 1, 9), 9), ((131, 7, 3), 16), ((17, 9, 13), 256),
    ((9, 130, 1, 5), 17), ((5, 4, 1, 3, 7), 32),
    ((5, 2, 3, 1, 2, 3), 1), ((3, 5, 2, 1, 3, 5), 33),
    ((3, 2, 3, 1, 3, 2, 5), 64), ((3, 1, 2, 3, 2, 3, 2), 129),
    ((3,) * 8, 65), ((3, 3, 1, 3, 3, 2, 3, 3), 128), ((5, 3, 2, 3, 1, 3, 2, 3), 256),
]
# Reduced-precision MTTKRP of 3-way objects: partial 128-row tiles, reduction extents that are not multiples of 32,
# K = 1, and the multi-wave / slab-split tensor of test_reduced_precision_multi_wave_tensor.
TC_RANKS = [1, 63, 64, 65, 129, 256]
MULTI_WAVE = (640, 520, 96)
TC_CASES = [(s, R) for s in ((130, 90, 70), (257, 33, 45), (200, 45, 1)) for R in TC_RANKS] + \
           [(MULTI_WAVE, R) for R in (65, 256)]
# Sparse MTTKRP, model_at and held-out SSE: every (lanes per nonzero, columns per lane) bucket of rank_dispatch.
SPARSE_RANKS = [1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128, 129, 256]
SPARSE_KINDS = {'units': (2, 3, 4, 5, 6, 7, 8), 'nnz1': (8, 2), 'nnz255': (2, 6), 'nnz256': (5, 3), 'nnz257': (7, 4),
                'one_row': (3, 6), 'dups': (4, 8)}
MODEL_KINDS = ['dense', 'masked', 'sparse', 'sparse_masked']
MODEL_SHAPES = [(37, 29), (17, 1, 13), (9, 7, 1, 5), (7, 3, 5, 1, 4), (5, 3, 1, 4, 3, 2), (5, 1, 3, 2, 3, 2, 3),
                (3, 2, 3, 1, 3, 2, 3, 3)]
# several GPUs: 8-way objects whose last mode (11 indices) is cut into uneven slabs
MULTI_DENSE = (5, 3, 1, 3, 2, 3, 2, 11)
MULTI_SPARSE = (13, 3, 3, 3, 3, 3, 3, 11)
MULTI_RANKS = (17, 129)
# solves against the FP64 oracle
EM_RANKS = [32, 33, 64, 65, 128, 129, 200]
EM_SHAPE = (41, 37, 12)                 # K = 12 >= 8 slabs
NWAY_EM_SHAPES = [(6, 5, 4, 3, 3, 2), (6, 5, 4, 3, 1, 3, 2), (5, 4, 3, 3, 3, 2, 3, 4),
                  (9, 7, 1, 2, 1, 3)]   # the last: trailing extents with a product of 6 < 8
SPARSE_EM_RANKS = [2, 4, 16, 100]
SPARSE_EM_SHAPES = [(6, 5, 4, 3, 3, 4), (5, 4, 3, 3, 3, 2, 3, 4)]
NVECS_SHAPES = [(3, 300, 2, 3, 2, 2), (4, 3, 260, 2, 2, 1, 3), (3, 2, 2, 270, 2, 1, 2, 3)]


# ---------------------------------------------------------------------------------------------- references
def _seed(*xs):
    return int(sum((i + 1) * 7919 * int(x) for i, x in enumerate(xs)) % (2 ** 31 - 1))


def ints(rng, shape, nonzero=False):
    """Integers drawn uniformly from [-2, 2] (from {-2, -1, 1, 2} with nonzero=True), int64."""
    if nonzero:
        return rng.choice(np.array([-2, -1, 1, 2], dtype=np.int64), size=shape)
    return rng.randint(-2, 3, size=shape).astype(np.int64)


def khatri_rao(mats):
    """Khatri-Rao product, first matrix varying fastest (the column order of the mode-n unfolding)."""
    K = mats[0]
    for M in mats[1:]:
        K = (M[:, None, :] * K[None, :, :]).reshape(-1, K.shape[1])
    return K


def unfold(X, n):
    return np.moveaxis(X, n, 0).reshape(X.shape[n], -1, order='F')


def fp64_bound(X, U, n):
    """max |x| * prod_{m != n} max |U_m| * terms: a bound on every partial sum of an output of the FP64 MTTKRP."""
    terms = int(np.prod([s for m, s in enumerate(X.shape) if m != n]))
    return float(np.max(np.abs(X), initial=0)) * float(np.prod([np.max(np.abs(U[m])) for m in range(len(U)) if m != n])) \
        * terms


def exact_mttkrp(X, U, n):
    """int64 mode-n MTTKRP of integer X and U.  The product runs in FP64 BLAS, which is exact because every partial sum
    is an integer below 2^53 (asserted); test_dense_references_are_exact checks it against int64 einsum."""
    assert fp64_bound(X, U, n) < FP64_EXACT
    M = unfold(X.astype(np.float64), n) @ khatri_rao([U[m] for m in range(len(U)) if m != n]).astype(np.float64)
    return np.rint(M).astype(np.int64)


def einsum_mttkrp(X, U, n):
    """The same quantity in int64 throughout, in einsum's contraction order."""
    N = X.ndim
    idx = ''.join(chr(97 + d) for d in range(N))
    ops = [X] + [U[m] for m in range(N) if m != n]
    spec = idx + ',' + ','.join(idx[m] + 'z' for m in range(N) if m != n) + '->' + idx[n] + 'z'
    return np.einsum(spec, *ops, optimize=True)


def coo_mttkrp(subs, vals, shape, U, n):
    """int64 COO restatement: every nonzero adds v * prod_{m != n} U_m(i_m, :) to row i_n (duplicates add up)."""
    contrib = np.repeat(vals[:, None], U[0].shape[1], axis=1)
    for m in range(len(shape)):
        if m != n:
            contrib = contrib * U[m][subs[:, m], :]
    out = np.zeros((shape[n], U[0].shape[1]), dtype=np.int64)
    np.add.at(out, subs[:, n], contrib)
    return out


def coo_full(subs, vals, shape):
    X = np.zeros(shape, dtype=np.int64)
    np.add.at(X, tuple(subs.T), vals)
    return X


def model_int(subs, U):
    p = np.ones((subs.shape[0], U[0].shape[1]), dtype=np.int64)
    for d, F in enumerate(U):
        p = p * F[subs[:, d], :]
    return p.sum(axis=1)


def full_cp_int(U):
    X = U[0]
    for F in U[1:]:
        X = (X[..., None, :] * F.reshape((1,) * (X.ndim - 1) + F.shape))
    return X.sum(axis=-1)


def cp_bound(U, terms):
    """max |model value| bound: R * prod max |U_d|, times the number of terms summed."""
    return U[0].shape[1] * float(np.prod([np.max(np.abs(F)) for F in U])) * terms


# ---------------------------------------------------------------------------------------------- case data
@functools.lru_cache(maxsize=None)
def dense_data(shape, R):
    rng = np.random.RandomState(_seed(R, *shape))
    return ints(rng, shape), [ints(rng, (s, R)) for s in shape]


@functools.lru_cache(maxsize=None)
def dense_refs(shape, R):
    X, U = dense_data(shape, R)
    return [exact_mttkrp(X, U, n) for n in range(len(shape))]


def _sparse_shape(order):
    """First mode 61 (odd) with room for rows of more than 2048 distinct nonzeros in every order."""
    return {2: (61, 2400), 3: (61, 50, 49), 4: (61, 13, 14, 13), 5: (61, 7, 7, 7, 7), 6: (61, 5, 5, 5, 4, 5),
            7: (61, 4, 4, 3, 4, 3, 4), 8: (61, 3, 3, 3, 3, 3, 3, 4)}[order]


def _row_entries(rng, shape, row, count):
    """`count` distinct nonzeros in row `row` of mode 1."""
    others = shape[1:]
    flat = rng.choice(int(np.prod(others)), size=count, replace=False)
    rest = np.stack(np.unravel_index(flat, others, order='F'), axis=1)
    return np.hstack([np.full((count, 1), row), rest])


def unit_rows():
    """Row lengths of mode 1, in row order (None: an empty row), laid out against units of kSparseChunk = 256 merged
    nonzeros: a row of exactly 256 that starts on a unit boundary, a row that ends exactly on a unit end, and rows
    starting mid-unit that span 2..9 units (4k+1, 4k+2 and 4k+3 of them: every remainder of the four-way fix-up loop)."""
    rows = [256, 100, 156, None, 256]          # [0,256) [256,356) [356,512) empty [512,768)
    pos = 768
    for span in range(2, 10):
        rows.append(10)                        # the next row starts 10 entries into a unit
        pos += 10
        length = (span - 1) * 256 + 20         # ... and ends 30 entries into its span-th unit
        rows += [length, None]
        pos += length
        fill = (-pos) % 256 or 256             # back to a unit boundary
        rows.append(fill)
        pos += fill
    return rows


@functools.lru_cache(maxsize=None)
def sparse_case(order, kind):
    """(shape, subs, vals) of one sparse test object: integer values in {-2, -1, 1, 2} (stored values are never zero), at
    least one nonzero with last-mode index = extent - 1."""
    shape = _sparse_shape(order)
    rng = np.random.RandomState(_seed(order, len(kind), ord(kind[-1])))
    if kind == 'units':
        blocks = [_row_entries(rng, shape, r, n) for r, n in enumerate(unit_rows()) if n is not None]
        blocks.append(_row_entries(rng, shape, shape[0] - 1, 3))   # the last row of mode 1
        subs = np.vstack(blocks)
    elif kind == 'one_row':                                        # every nonzero in one row (several units)
        subs = _row_entries(rng, shape, 29, 1000)
    else:
        n = {'nnz1': 1, 'nnz255': 255, 'nnz256': 256, 'nnz257': 257, 'dups': 600}[kind]
        flat = rng.choice(int(np.prod(shape)), size=n, replace=False)
        subs = np.stack(np.unravel_index(flat, shape, order='F'), axis=1)
    subs = _touch_last_index(subs.astype(np.int64), shape[-1])
    if kind == 'dups':                                             # repeated subscripts are summed
        subs = np.vstack([subs, subs[rng.randint(0, len(subs), size=200)]])
    return shape, subs, ints(rng, subs.shape[0], nonzero=True)


def _touch_last_index(subs, ext):
    """Move the last-mode subscript of one entry to ext - 1 unless one is there already, keeping the entries distinct
    and every other subscript (so the row lengths of mode 1 stay as laid out)."""
    if np.any(subs[:, -1] == ext - 1):
        return subs
    seen = {tuple(s) for s in subs}
    for e in range(len(subs) - 1, -1, -1):
        if tuple(subs[e, :-1]) + (ext - 1,) not in seen:
            subs[e, -1] = ext - 1
            return subs
    raise AssertionError('no entry can take last-mode index %d' % (ext - 1))


@functools.lru_cache(maxsize=None)
def sparse_factors(order, R):
    rng = np.random.RandomState(_seed(order, R, 3))
    return [ints(rng, (s, R)) for s in _sparse_shape(order)]


def model_case(shape, R, kind):
    """Integer factors, an integer tensor, an observation pattern (about 60 %) and up to 300 unobserved entries held out
    with their true values."""
    rng = np.random.RandomState(_seed(R, len(kind), *shape))
    U = [ints(rng, (s, R)) for s in shape]
    X = ints(rng, shape, nonzero=kind.startswith('sparse'))
    W = rng.rand(*shape) < 0.6
    W.flat[0] = W.flat[-1] = True
    hs = np.argwhere(~W)
    hs = hs[rng.permutation(len(hs))[:300]]
    probe = np.vstack([np.stack([rng.randint(0, s, 400) for s in shape], axis=1),
                       np.zeros((1, len(shape)), dtype=np.int64), np.asarray(shape)[None, :] - 1])
    return U, X, W, hs, probe


# ---------------------------------------------------------------------------------------------- CPU: the premise
def test_unit_layout_hits_every_boundary():
    lengths = [n or 0 for n in unit_rows()]
    ends = np.cumsum(lengths)
    starts = ends - np.asarray(lengths)
    assert 0 in starts and 256 in ends and 512 in ends            # a whole unit from a boundary; a row ending on one
    spans = {int((e - 1) // 256 - s // 256 + 1) for s, e, n in zip(starts, ends, lengths) if n > 256}
    assert {2, 3, 4, 5, 6, 7, 8, 9} <= spans and {s % 4 for s in spans} == {0, 1, 2, 3}
    for order in SPARSE_KINDS['units']:
        shape, subs, vals = sparse_case(order, 'units')
        assert max(lengths) <= np.prod(shape[1:])
        assert len(np.unique(subs, axis=0)) == len(subs) and np.all(vals != 0)
        assert np.array_equal(np.bincount(subs[:, 0], minlength=shape[0])[:len(lengths)], lengths)
    for order, kind in [(o, k) for k, os_ in SPARSE_KINDS.items() for o in os_]:
        shape, subs, vals = sparse_case(order, kind)
        assert np.any(subs[:, -1] == shape[-1] - 1) and np.all(subs < np.asarray(shape)) and np.all(subs >= 0)
    assert [len(sparse_case(o, k)[1]) for o, k in ((8, 'nnz1'), (2, 'nnz255'), (5, 'nnz256'), (7, 'nnz257'))] == \
        [1, 255, 256, 257]


@pytest.mark.parametrize('shape,R', DENSE_CASES)
def test_dense_references_are_exact(shape, R):
    """FP64: every partial sum below 2^53; mma.sync (order >= 3): 128 products of the TF32 operands below 2^24; the
    operands themselves (the Khatri-Rao rows of up to N - 2 factors) exact in TF32.  The reference equals int64 einsum."""
    X, U = dense_data(shape, R)
    N = len(shape)
    amax = float(np.max(np.abs(X)))
    fmax = [float(np.max(np.abs(F))) for F in U]
    for n in range(N):
        assert fp64_bound(X, U, n) < FP64_EXACT
        if N >= 3:
            prod_all = amax * float(np.prod([fmax[m] for m in range(N) if m != n]))
            assert prod_all * MMA_SYNC_SPAN < FP32_EXACT
            assert float(np.prod([fmax[m] for m in range(N) if m != n])) <= OPERAND_EXACT[3]
        assert np.array_equal(exact_mttkrp(X, U, n), einsum_mttkrp(X, U, n)), n


@pytest.mark.parametrize('shape,R', TC_CASES)
def test_reduced_precision_references_are_exact(shape, R):
    """tcgen05 (TF32 / BF16): operands exact, the FP32 sum over the reduction extent of one slab of one tile below 2^24,
    also for the partial contraction T of the dimension tree; FP64 across slabs below 2^53.  The reference equals int64
    einsum (on 7 rows of every mode for the multi-wave tensor)."""
    X, U = dense_data(shape, R)
    amax, fmax = float(np.max(np.abs(X))), [float(np.max(np.abs(F))) for F in U]
    assert amax <= OPERAND_EXACT[2] and max(fmax) <= OPERAND_EXACT[2]
    I, J, K = shape
    for n, red in ((0, J), (1, I), (2, I)):                      # the FP32-accumulated (contracted) extent per mode
        assert amax * fmax[1 if n == 0 else 0] * red < FP32_EXACT
        assert amax * float(np.prod([fmax[m] for m in range(3) if m != n])) * MMA_SYNC_SPAN < FP32_EXACT
        assert fp64_bound(X, U, n) < FP64_EXACT
    for n in range(3):
        rows = np.unique(np.r_[0, 1, shape[n] // 2, shape[n] - 2, shape[n] - 1, 3 % shape[n], 5 % shape[n]]) \
            if shape == MULTI_WAVE else np.arange(shape[n])
        Xs = np.take(X, rows, axis=n)
        got = unfold(Xs.astype(float), n) @ khatri_rao([U[m] for m in range(3) if m != n]).astype(float)
        assert np.array_equal(np.rint(got).astype(np.int64), einsum_mttkrp(Xs, U, n)), n


@pytest.mark.parametrize('kind', list(SPARSE_KINDS))
def test_sparse_references_are_exact(kind):
    """Every partial row sum of the sparse kernels below 2^53 at every rank, and the COO restatement (np.add.at over
    the nonzeros) equal to the int64 product of the dense unfolding with the Khatri-Rao product, at the smallest and
    the largest rank (the restatement does not depend on R otherwise)."""
    for order in SPARSE_KINDS[kind]:
        shape, subs, vals = sparse_case(order, kind)
        merged = np.abs(coo_full(subs, vals, shape)).max()
        for R in SPARSE_RANKS:
            U = sparse_factors(order, R)
            assert merged * float(np.prod([np.abs(F).max() for F in U])) * len(vals) < FP64_EXACT
        Xf = coo_full(subs, vals, shape)
        for R in (SPARSE_RANKS[0], SPARSE_RANKS[-1]):
            U = sparse_factors(order, R)
            for n in range(order):
                alt = unfold(Xf, n) @ khatri_rao([U[m] for m in range(order) if m != n])
                assert np.array_equal(coo_mttkrp(subs, vals, shape, U, n), alt), (order, R, n)


def test_model_and_heldout_references_are_exact():
    """The model at a subscript and the held-out SSE below 2^53 at every rank and order; the model by direct indexing
    equal to the full int64 ktensor at the same subscripts."""
    for shape in MODEL_SHAPES:
        for kind in MODEL_KINDS:
            for R in SPARSE_RANKS:
                U, X, W, hs, probe = model_case(shape, R, kind)
                assert (np.abs(X).max() + cp_bound(U, 1)) ** 2 * max(len(hs), 1) < FP64_EXACT
                if R in (SPARSE_RANKS[0], SPARSE_RANKS[-1]):
                    full = full_cp_int(U)
                    assert np.array_equal(model_int(probe, U), full[tuple(probe.T)])
                    assert np.array_equal(model_int(hs, U), full[tuple(hs.T)])


def test_multi_gpu_references_are_exact():
    shape, subs, vals = multi_sparse_case()
    for R in MULTI_RANKS:
        X, U = dense_data(MULTI_DENSE, R)
        for n in range(len(MULTI_DENSE)):
            assert np.array_equal(dense_refs(MULTI_DENSE, R)[n], einsum_mttkrp(X, U, n))
        Us = multi_sparse_factors(R)
        Xf = coo_full(subs, vals, shape)
        for n in range(len(shape)):
            assert np.abs(Xf).max() * float(np.prod([np.abs(Us[m]).max() for m in range(8) if m != n])) * len(vals) \
                < FP64_EXACT
            assert np.array_equal(coo_mttkrp(subs, vals, shape, Us, n),
                                  unfold(Xf, n) @ khatri_rao([Us[m] for m in range(len(shape)) if m != n]))


def multi_sparse_factors(R):
    return [ints(np.random.RandomState(_seed(R, d, 5)), (s, R)) for d, s in enumerate(MULTI_SPARSE)]


def multi_sparse_case():
    """8-way sparse object for several GPUs: 20 % of the nonzeros at last-mode index 0, the rest at index 10, so that the
    nonzero-balanced slabs are uneven and, from three GPUs on, some hold no nonzero."""
    rng = np.random.RandomState(17)
    shape = MULTI_SPARSE
    flat = rng.choice(int(np.prod(shape[:-1])), size=3000, replace=False)
    subs = np.stack(np.unravel_index(flat, shape[:-1], order='F'), axis=1)
    last = np.where(rng.rand(3000) < 0.2, 0, shape[-1] - 1)
    subs = np.hstack([subs, last[:, None]]).astype(np.int64)
    return shape, subs, ints(rng, 3000, nonzero=True)


def test_multi_gpu_slabs_are_uneven_and_one_is_empty(ab):
    shape, subs, vals = multi_sparse_case()
    X = ab.sptensor(subs, vals, shape)
    for n in (2, 3, 8):
        b = ab.sparse_shard_bounds(X, n)
        counts = [int(np.sum((subs[:, -1] >= b[r]) & (subs[:, -1] < b[r + 1]))) for r in range(n)]
        assert len(set(np.diff(b))) > 1 and len(set(counts)) > 1, (n, b, counts)
        if n >= 3:
            assert 0 in counts, (n, b, counts)
    assert len({hi - lo for lo, hi in (ab.shard_range(shape[-1], r, 2) for r in range(2))}) > 1


# ---------------------------------------------------------------------------------------------- CPU: dispatch guard
def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _changed(name, what, pattern):
    pytest.fail('%s: the pattern %r no longer matches %s.  The dispatch was changed: read its new thresholds there and '
                'update the rank lists of tests/test_exact_dispatch.py so that each has a rank on both sides of every '
                'threshold, then this pattern.' % (what, pattern, name))


def _match(name, pattern, what, flags=0):
    found = re.findall(pattern, _source(name), flags)
    if not found:
        _changed(name, what, pattern)
    return found


def _both_sides(ranks, t, what):
    assert t in ranks and t + 1 in ranks, ('%s: the threshold R <= %d is not straddled by the ranks %s; add %d and %d'
                                           % (what, t, sorted(ranks), t, t + 1))


def test_rank_lists_straddle_every_dispatch_threshold():
    body = _match('sparse.cuh', r'void rank_dispatch\(int R, Fn&& f\) \{(.*?)\n\}', 'rank_dispatch', re.S)[0]
    bucket_re = r'if \(R <= (\d+)\) f\(integral_constant<int, (\d+)>\{\}, integral_constant<int, (\d+)>\{\}\)'
    buckets = re.findall(bucket_re, body)
    if len(buckets) < 2 or 'else f(' not in body:
        _changed('sparse.cuh', 'rank_dispatch', bucket_re)
    for t, _, _ in buckets:
        _both_sides(SPARSE_RANKS, int(t), 'rank_dispatch (sparse MTTKRP, fix-up, model and held-out kernels)')
    assert max(SPARSE_RANKS) > max(int(t) for t, _, _ in buckets)
    # the masked sparse solves reach the buckets with 2, 4 and 16 lanes per nonzero and 4 columns per lane
    def bucket(R):
        return next(((g, c) for t, g, c in buckets if R <= int(t)), 'last')
    assert len({bucket(R) for R in SPARSE_EM_RANKS}) == len(SPARSE_EM_RANKS)

    expr = _match('mttkrp.cuh', r'inline int mttkrp_chunk_cols\(int R\) \{ return (.*?); \}', 'mttkrp_chunk_cols')[0]
    cols = [int(t) for t in re.findall(r'R <= (\d+)', expr)]
    widest = re.findall(r': (\d+)\)*$', expr)
    if not cols or not widest:
        _changed('mttkrp.cuh', 'mttkrp_chunk_cols', r'R <= (\d+) ... : (\d+)')
    widest = int(widest[0])
    dense_ranks = [R for _, R in DENSE_CASES]
    for t in cols + [widest, 2 * widest]:
        _both_sides(dense_ranks, t, 'mttkrp_chunk_cols (FP64 DMMA MTTKRP)')
    assert max(dense_ranks) >= 4 * widest

    nc = int(_match('mttkrp_tc.cu', r'constexpr int kNCols = (\d+);', 'kNCols')[0])
    _both_sides(TC_RANKS, nc, 'kNCols (tcgen05 MTTKRP rank chunks)')
    assert any(2 * nc < R <= 3 * nc for R in TC_RANKS) and max(TC_RANKS) == 4 * nc, 'three and four rank chunks'

    maxr = int(_match('em.cu', r'constexpr int kPMaxR = (\d+);', 'kPMaxR')[0])
    regks = int(_match('em.cu', r'constexpr int kPRegKs = (\d+);', 'kPRegKs')[0])
    regmul = int(_match('em.cu', r'if \(L\.Rp <= (\d+) \* kPRegKs\)', 'register-fragment switch of em_pass')[0])
    kmin = int(_match('em.cu', r'a\.K >= (\d+) && a\.R <= kPMaxR', 'K test of em_use_pipe')[0])
    _both_sides(EM_RANKS, maxr, 'kPMaxR (pipelined EM kernel / em_kernel fallback)')
    # the switch compares the rank padded to a multiple of 4, so regmul * regks + 1 is the first rank above it
    _both_sides(EM_RANKS, regmul * regks, 'kPRegKs (register / shared-memory GEMM operands of the pipelined EM kernel)')
    assert EM_SHAPE[2] >= kmin
    trailing = [int(np.prod(s[2:])) for s in NWAY_EM_SHAPES]
    assert any(k >= kmin for k in trailing) and any(k < kmin for k in trailing), (trailing, kmin)

    prep = _match('smallops.cu', r'int prep_system\(const PrepArgs& a, cudaStream_t st, const int\* skip\) \{\s*'
                                 r'const size_t smem = \(a\.R <= (\d+)\)', 'prep_system shared-memory switch')
    row = _match('smallops.cu', r'c\.BT = \(R <= (\d+)\) \? 128 : \(\(R <= (\d+)\) \? 64 : 32\);', 'row_launch_cfg')
    for t in [int(prep[0])] + [int(x) for x in row[0]]:
        _both_sides(EM_RANKS, t, 'prep_system / row_launch_cfg (small systems of the solves)')


# ---------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture
def gpu(ab):
    assert ab.device_count() >= 1, 'GPU tests need a CUDA device (the engine has no CPU fallback)'
    return ab


def _Z(obj, shape, R, miss=None):
    N = len(shape)
    Z = {'loss_function': ['Frobenius'], 'model': ['CP'], 'modes': [list(range(1, N + 1))], 'size': list(shape),
         'coupling': {'lin_coupled_modes': [0] * N, 'coupling_type': [], 'coupl_trafo_matrices': [None] * N},
         'constrained_modes': [0] * N, 'constraints': [None] * N, 'weights': [1.0], 'object': [obj], 'rank': [R]}
    if miss is not None:
        Z['miss'] = [miss]
    return Z


def _f(a):
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


def _exact(got, ref, what):
    ref = np.asarray(ref)
    if not np.array_equal(got, ref.astype(np.float64)):
        bad = np.argwhere(got != ref)
        i = tuple(bad[0])
        pytest.fail('%s: %d of %d elements differ; first at %s: device %r, int64 %r'
                    % (what, len(bad), ref.size, i, got[i], int(ref[i])))


# ---------------------------------------------------------------------------------------------- GPU: dense MTTKRP
@pytest.mark.gpu
@pytest.mark.parametrize('shape,R', DENSE_CASES)
def test_dense_mttkrp_exact_every_mode(gpu, shape, R):
    """ab.mttkrp and Solver.object_mttkrp of every mode position.  Orders >= 3 with mttkrp_precision = 3 (TF32 mma.sync,
    also on N-way objects) are exact too; matrices and N-way objects with precision 1 or 2 (and matrices with 3) fall
    back to FP64 and return its bits, also with non-integer factors."""
    ab = gpu
    X, U = dense_data(shape, R)
    refs = dense_refs(shape, R)
    N = len(shape)
    Uf = [_f(F) for F in U]
    for n in range(N):
        _exact(ab.mttkrp(_f(X), Uf, n + 1), refs[n], 'ab.mttkrp mode %d' % (n + 1))
    fallback = [1, 2, 3] if N == 2 else ([1, 2] if N >= 4 else [])
    with ab.Solver(_Z(_f(X), shape, R), [float('nan')]) as s:
        s.set_state({'fac': Uf})
        for pos in range(1, N + 1):
            _exact(s.object_mttkrp(1, pos, 0), refs[pos - 1], 'object_mttkrp pos %d' % pos)
            if N >= 3:
                _exact(s.object_mttkrp(1, pos, 3), refs[pos - 1], 'object_mttkrp pos %d, TF32 mma.sync' % pos)
            for prec in fallback:
                _exact(s.object_mttkrp(1, pos, prec), refs[pos - 1], 'object_mttkrp pos %d, precision %d' % (pos, prec))
        rng = np.random.RandomState(1)
        s.set_state({'fac': [_f(rng.randn(*F.shape)) for F in U]})
        for pos in range(1, N + 1):
            m64 = s.object_mttkrp(1, pos, 0)
            for prec in fallback:
                assert np.array_equal(s.object_mttkrp(1, pos, prec), m64), (pos, prec)


# ---------------------------------------------------------------------------------------------- GPU: reduced precision
@pytest.mark.gpu
@pytest.mark.parametrize('prec', sorted(PRECISIONS))
@pytest.mark.parametrize('shape,R', TC_CASES)
def test_reduced_precision_mttkrp_exact(gpu, shape, R, prec):
    """Every mode of a 3-way object in TF32 / BF16 on tcgen05 and TF32 on mma.sync, and the partial contraction T that a
    dimtree = 1 mode-2 pass emits, checked through the mode-3 result computed from it.  object_mttkrp uses the options
    of the last run: one run with dimtree = 1 and no iteration, then the integer factors; position 3 before position 2
    is a full pass (the factors changed since T), position 3 after position 2 reads T."""
    ab = gpu
    X, U = dense_data(shape, R)
    refs = dense_refs(shape, R)
    with ab.Solver(_Z(_f(X), shape, R), [float('nan')]) as s:
        s.set_state({'fac': [_f(F) for F in U]})
        s.run(pg.default_options(MaxOuterIters=0, dimtree=1, **ZERO_TOL))
        s.set_state({'fac': [_f(F) for F in U]})
        for pos in (1, 3, 2):
            _exact(s.object_mttkrp(1, pos, prec), refs[pos - 1], '%s pos %d' % (PRECISIONS[prec], pos))
        _exact(s.object_mttkrp(1, 3, prec), refs[2], '%s pos 3 from the dimension-tree T' % PRECISIONS[prec])


# ---------------------------------------------------------------------------------------------- GPU: sparse MTTKRP
@pytest.mark.gpu
@pytest.mark.parametrize('kind', list(SPARSE_KINDS))
@pytest.mark.parametrize('R', SPARSE_RANKS)
def test_sparse_mttkrp_exact_every_bucket(gpu, R, kind):
    """Every mode position of sparse objects of the listed orders, laid out against the 256-nonzero units of the kernel
    (see unit_rows), at every rank_dispatch bucket; a permutation of the nonzeros gives the same bits."""
    ab = gpu
    for order in SPARSE_KINDS[kind]:
        shape, subs, vals = sparse_case(order, kind)
        U = sparse_factors(order, R)
        Uf = [_f(F) for F in U]
        perm = np.random.RandomState(order).permutation(len(vals))
        got = []
        for sb, vl in ((subs, vals), (subs[perm], vals[perm])):
            with ab.Solver(_Z(ab.sptensor(sb, vl.astype(np.float64), shape), shape, R), [float('nan')]) as s:
                s.set_state({'fac': Uf})
                got.append([s.object_mttkrp(1, pos, 0) for pos in range(1, order + 1)])
        for n in range(order):
            _exact(got[0][n], coo_mttkrp(subs, vals, shape, U, n), 'order %d pos %d' % (order, n + 1))
            assert np.array_equal(got[0][n], got[1][n]), ('permuted nonzeros', order, n + 1)


# ---------------------------------------------------------------------------------------------- GPU: model and held-out SSE
@pytest.mark.gpu
@pytest.mark.parametrize('kind', MODEL_KINDS)
@pytest.mark.parametrize('R', SPARSE_RANKS)
def test_model_at_and_heldout_sse_exact(gpu, R, kind):
    """Solver.model_at on dense, masked dense, sparse and masked sparse objects of orders 2..8, and for the objects
    with missing data the held-out SSE of the integer initial factors (heldout_history entry 0) against int64."""
    ab = gpu
    for shape in MODEL_SHAPES:
        U, X, W, hs, probe = model_case(shape, R, kind)
        Uf = [_f(F) for F in U]
        if kind == 'dense':
            Z, zn = _Z(_f(X), shape, R), [float('nan')]
        elif kind == 'masked':
            Z = _Z(_f(np.where(W, X, 0)), shape, R, miss=np.asfortranarray(W))
            zn = [float(np.sum(np.where(W, X, 0) ** 2))]
        else:
            ts = np.argwhere(W)
            S = ab.sptensor(ts, X[W].astype(np.float64), shape)
            Z = _Z(S, shape, R, miss=ab.sptensor(ts, np.ones(len(ts)), shape) if kind == 'sparse_masked' else None)
            zn = [float('nan')]
        with ab.Solver(Z, zn) as s:
            s.set_state({'fac': Uf})
            _exact(s.model_at(1, probe), model_int(probe, U), 'model_at order %d' % len(shape))
            if kind in ('masked', 'sparse_masked'):
                H = ab.sptensor(hs, X[tuple(hs.T)].astype(np.float64), shape)
                s.set_heldout(1, H)
                s.run(pg.default_options(MaxOuterIters=0, **ZERO_TOL))
                sse, count = s.heldout_history(1)
                ref = int(np.sum((X[tuple(hs.T)] - model_int(hs, U)) ** 2))
                assert count == len(hs) and sse[0] == float(ref), (len(shape), sse[0], ref)


# ---------------------------------------------------------------------------------------------- GPU: several GPUs
@pytest.mark.gpu
@pytest.mark.parametrize('n', [2, 'all'])
def test_multi_gpu_eight_way_exact(ab, n):
    """An 8-way dense object through n_gpus = N and an 8-way sparse object through shard_sparse=True, with uneven
    last-mode slabs (an empty one from three GPUs on): object_mttkrp of every position and model_at."""
    count = ab.device_count()
    if count < 2:
        pytest.skip('needs 2 GPUs')
    N = count if n == 'all' else n
    rng = np.random.RandomState(23)
    for R in MULTI_RANKS:
        X, U = dense_data(MULTI_DENSE, R)
        probe = np.stack([rng.randint(0, s, 500) for s in MULTI_DENSE], axis=1)
        with ab.Solver(_Z(_f(X), MULTI_DENSE, R), [float('nan')], n_gpus=N) as s:
            s.set_state({'fac': [_f(F) for F in U]})
            for pos in range(1, 9):
                _exact(s.object_mttkrp(1, pos, 0), dense_refs(MULTI_DENSE, R)[pos - 1], 'dense, %d GPUs, pos %d' % (N, pos))
            _exact(s.model_at(1, probe), model_int(probe, U), 'dense model_at, %d GPUs' % N)
        shape, subs, vals = multi_sparse_case()
        Us = multi_sparse_factors(R)
        probe = np.stack([rng.randint(0, s, 500) for s in shape], axis=1)
        with ab.Solver(_Z(ab.sptensor(subs, vals.astype(np.float64), shape), shape, R), [float('nan')], n_gpus=N,
                       shard_sparse=True) as s:
            s.set_state({'fac': [_f(F) for F in Us]})
            for pos in range(1, 9):
                _exact(s.object_mttkrp(1, pos, 0), coo_mttkrp(subs, vals, shape, Us, pos - 1),
                       'sparse, %d GPUs, pos %d' % (N, pos))
            _exact(s.model_at(1, probe), model_int(probe, Us), 'sparse model_at, %d GPUs' % N)


# ---------------------------------------------------------------------------------------------- GPU: solves at the new edges
def _solve_and_compare(ab, Zd, G, opts, Zdev=None):
    """Oracle on the dense problem Zd, device on Zdev (default Zd): north-star tolerances."""
    zd = pg.znorm_const(Zd)
    Zdev = Zdev or Zd
    zs = [float('nan') if ab.as_sparse(x) is not None else z for x, z in zip(Zdev['object'], zd)]
    Go, oo = oracle_solve(Zd, zd, G, options=opts)
    Gd, od = ab.cmtf_fun_AOADMM(Zdev, zs, G, None, None, None, None, opts)
    assert od['OuterIterations'] == oo['OuterIterations']
    n = oo['OuterIterations'] + 1
    for key in ('func_val_conv', 'func_coupl_conv', 'func_constr_conv'):
        assert np.max(np.abs(od[key][:n] - oo[key][:n])) < FIT_TOL, key
    assert np.array_equal(od['innerIters'], oo['innerIters'])
    a, b = od['func_rel_missing'][1:n], oo['func_rel_missing'][1:n]
    assert np.max(np.abs(a - b)) < FIT_TOL and abs(od['f_rel_missing'] - oo['f_rel_missing']) < FIT_TOL
    assert_state_close(Gd, Go)


@pytest.mark.gpu
@pytest.mark.parametrize('sz', NWAY_EM_SHAPES)
def test_masked_dense_six_to_eight_way_solves(gpu, sz):
    """Z.miss on 6-, 7- and 8-way tensors: the EM third factor is the Khatri-Rao product of four to six trailing modes
    (the pipelined EM kernel for a product >= 8, the other one below)."""
    nn = ('non-negativity',)
    Z, G, _ = pg.config_single_cp(sz=sz, R=4, seed=len(sz), noise=0.1, constraints=[nn] * len(sz))
    _solve_and_compare(gpu, pg.add_missing(Z, 0.3, seed=2), G, pg.default_options(MaxOuterIters=5, **ZERO_TOL))


@pytest.mark.gpu
def test_masked_eight_way_tensor_coupled_to_a_matrix(gpu):
    sz = [5, 4, 3, 3, 1, 2, 3, 4, 5, 7]
    nn = ('non-negativity',)
    coupling = {'lin_coupled_modes': [1] + [0] * 7 + [1, 0], 'coupling_type': [0], 'coupl_trafo_matrices': [None] * 10}
    Z, G, _ = pg._finish(['CP', 'CP'], sz, [list(range(1, 9)), [9, 10]], [[1.0] * 3] * 2, [0.1] * 2, coupling,
                         [pg.d_rand] * 10, [1] * 10, [nn] * 10, [0.5, 0.5], np.random.RandomState(8))
    _solve_and_compare(gpu, pg.add_missing(Z, 0.3, seed=3), G, pg.default_options(MaxOuterIters=5, **ZERO_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('R', EM_RANKS)
def test_masked_dense_three_way_em_kernels_and_small_systems(gpu, R):
    """K >= 8 slabs: the pipelined EM kernel with register (R <= 32) and shared-memory operands, the em_kernel fallback
    above R = 128, and both prep_system edges (R = 32 / 33, 64 / 65).  Non-negativity on every mode keeps every system
    shifted, so R above an extent is well posed."""
    nn = ('non-negativity',)
    Z, G, _ = pg.config_single_cp(sz=EM_SHAPE, R=R, seed=R, noise=0.1, constraints=[nn] * 3)
    _solve_and_compare(gpu, pg.add_missing(Z, 0.3, seed=R), G, pg.default_options(MaxOuterIters=3, **ZERO_TOL))


@pytest.mark.gpu
@pytest.mark.parametrize('R', SPARSE_EM_RANKS)
@pytest.mark.parametrize('sz', SPARSE_EM_SHAPES)
def test_masked_sparse_six_and_eight_way_solves(gpu, sz, R):
    """Masked sparse objects at the rank buckets with 2, 4 and 16 lanes per nonzero and 4 columns per lane: the model
    pass, the telescoped norms and the imputed MTTKRP, against the dense oracle on full(S) with the mask."""
    ab = gpu
    nn = ('non-negativity',)
    Z, G, _ = pg.config_single_cp(sz=sz, R=R, seed=R + len(sz), noise=0.1, constraints=[nn] * len(sz))
    X = Z['object'][0]
    W = np.random.RandomState(R).rand(*X.shape) < 0.3
    ts = np.argwhere(W)
    Zs = dict(Z, object=[ab.sptensor(ts, X[W], X.shape)], miss=[ab.sptensor(ts, np.ones(len(ts)), X.shape)])
    Zd = dict(Z, object=[np.asfortranarray(np.where(W, X, 0.0))], miss=[np.asfortranarray(W)])
    _solve_and_compare(ab, Zd, G, pg.default_options(MaxOuterIters=4, **ZERO_TOL), Zdev=Zs)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', NVECS_SHAPES)
def test_nvecs_every_mode_of_six_to_eight_way_tensors(gpu, shape):
    """Leading eigenvectors of X_(n) X_(n)' of every mode of 6-, 7- and 8-way tensors, a long mode (more than 256 rows)
    in a middle position."""
    ab = gpu
    rng = np.random.RandomState(len(shape))
    N, R = len(shape), 3
    facs = [rng.rand(s, R) * (1.0 + np.arange(R))[None, :] for s in shape]
    X = np.einsum(','.join(chr(97 + d) + 'z' for d in range(N)) + '->' + ''.join(chr(97 + d) for d in range(N)), *facs)
    X = X + 0.2 * np.linalg.norm(X) / np.sqrt(X.size) * rng.randn(*shape)
    Z = _Z(X, shape, R)
    with ab.Solver(Z, [float('nan')]) as s:
        for n in range(1, N + 1):
            r = min(R, shape[n - 1])
            Ud, info = s.nvecs(n, r, return_info=True)
            _nvecs_close(Ud, pg.cmtf_nvecs(Z, n, r), Z, n)
            assert info['residual'] < 1e-12 and info['iterations'] < 1000, info
