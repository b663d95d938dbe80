"""aoadmm_b200 - host-side mirror of the reference interface for the AO-ADMM hot path.

`cmtf_fun_AOADMM(Z, Znorm_const, G, fh, gh, lscalar, uscalar, options)` has the signature, argument meaning
and error behaviour of functions/cmtf_fun_AOADMM.m:1 and is what `cmtf_AOADMM` (functions/cmtf_AOADMM.m:193)
calls; everything numerical happens in libaoadmm_b200.so (CUDA, sm_100a) behind the C ABI of include/aoadmm.h.
There is no CPU path: importing this package fails when the library is missing, and every call fails with
AoadmmError(NO_DEVICE) when no GPU is present.

Struct conventions (dicts mirroring the MATLAB structs, 1-based labels where they are data):
  Z : 'object' (dense arrays; a CP object may also be a sparse `sptensor` or, 2-way, any SciPy sparse matrix), 'model',
      'modes', 'size', 'coupling' {'lin_coupled_modes','coupling_type',
      'coupl_trafo_matrices'[,'coupl_trafo_matrices2']}, 'constrained_modes', 'constraints', 'weights',
      'loss_function', optional 'ridge', optional 'miss' (Z.miss: dense 0/1 arrays; for a sparse object a sparse mask
      whose nonzeros are exactly its stored entries, the unstored entries being unobserved)
  G : 'fac', 'constraint_fac', 'constraint_dual_fac', 'coupling_dual_fac' (per mode), 'coupling_fac' (per coupling)
  options : fields of example_script6...m:120-132
"""
import ctypes as C

import numpy as np

from . import _capi
from ._capi import AoadmmError, lib

__all__ = ['cmtf_fun_AOADMM', 'cmtf_AOADMM', 'cmtf_nvecs', 'cmtf_nvecs_sparse', 'init_coupled_AOADMM_CMTF', 'Solver', 'AoadmmError', 'sptensor', 'mttkrp',
           'prox', 'chol_solve', 'gram',
           'shard_range', 'sparse_shard_bounds', 'device_count', 'nccl_unique_id']


def _dp(a):
    return a.ctypes.data_as(_capi.c_double_p)


def _f64(a):
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


class sptensor:
    """A sparse tensor in coordinate form, the Tensor Toolbox sptensor(subs, vals, sz) with 0-based subscripts: `subs` is
    nnz x N, `vals` nnz values, `shape` the N extents.  Duplicate subscripts are summed when the object is used."""

    def __init__(self, subs, vals, shape):
        self.shape = tuple(int(s) for s in shape)
        self.subs = np.asarray(subs, dtype=np.int64).reshape(-1, len(self.shape))
        self.vals = np.asarray(vals, dtype=np.float64).reshape(-1)
        if self.subs.shape[0] != self.vals.size:
            raise ValueError('sptensor: subs has %d rows but there are %d values' % (self.subs.shape[0], self.vals.size))

    @property
    def ndim(self):
        return len(self.shape)

    @property
    def nnz(self):
        return self.vals.size

    def full(self):
        """The dense array (column-major), duplicates summed."""
        X = np.zeros(self.shape, order='F')
        np.add.at(X, tuple(self.subs.T), self.vals)
        return X


def as_sparse(X):
    """`X` as an sptensor when it is sparse (an sptensor, or anything with `tocoo()` such as a SciPy sparse matrix),
    else None.  Duck typing keeps SciPy an optional dependency."""
    if isinstance(X, sptensor):
        return X
    if hasattr(X, 'tocoo') and not isinstance(X, np.ndarray):
        c = X.tocoo()
        return sptensor(np.stack([np.asarray(c.row), np.asarray(c.col)], axis=1), c.data, c.shape)
    return None


def _check_heldout(Z, p, X):
    """A held-out set `X` (sptensor or SciPy sparse) of object p (0-based) as an sptensor, checked on the host: a CP object
    with missing data (Z.miss) and the shape of the object."""
    P = len(Z['modes'])
    if not 0 <= p < P:
        raise AoadmmError(1, 'held-out set: object %d is out of range (1..%d)' % (p + 1, P))
    if Z['model'][p] != 'CP':
        raise AoadmmError(1, 'held-out set: object %d is a PARAFAC2 object (CP objects only)' % (p + 1))
    S = as_sparse(X)
    if S is None:
        raise AoadmmError(1, 'held-out set of object %d must be an sptensor or a SciPy sparse matrix' % (p + 1))
    miss = Z.get('miss') or [None] * P
    if miss[p] is None:
        raise AoadmmError(1, 'held-out set: object %d has no missing data (Z.miss); a held-out set is validated '
                             'against what training did not observe' % (p + 1))
    want = tuple(int(Z['size'][m - 1]) for m in Z['modes'][p])
    if S.shape != want:
        raise AoadmmError(1, 'held-out set: shape %s does not match object %d %s' % (S.shape, p + 1, want))
    return S


def heldout_stopping_rule(s, patience):
    """The rule of early stopping on the held-out error (aoadmm_set_heldout_stopping) on a history s_0..s_n of summed
    held-out SSEs: (k_best, k_stop).  k_best is the first k >= 1 with the smallest s_k (a new best must be strictly
    smaller, a NaN is never one); n when no s_k (k >= 1) is a number, which includes n = 0.  k_stop is the first k with
    k - k_best >= patience, or None when the rule does not fire within the history."""
    s = [float(v) for v in s]
    best, stop = -1, None
    for k in range(1, len(s)):
        if (not np.isnan(s[k])) if best < 0 else s[k] < s[best]:
            best = k
        elif best > 0 and k - best >= patience:
            stop = k
            break
    return (len(s) - 1 if best < 0 else best), stop


def _heldout_sum(hists):
    """s_k = the sum of the per-object held-out SSEs in object order, added as the engine adds them."""
    n = max(len(h) for h in hists)
    out = np.zeros(n)
    for k in range(n):
        t = 0.0
        for h in hists:
            t += h[k]
        out[k] = t
    return out


def _coo(subs, vals):
    """aoadmm_sparse_object over column-major copies of subs (nnz x N) and vals; returns it with the arrays to keep."""
    subs = np.asfortranarray(np.asarray(subs, dtype=np.int64))
    vals = None if vals is None else np.ascontiguousarray(vals, dtype=np.float64)
    so = _capi.SparseObject()
    so.nnz = subs.shape[0]
    so.subs = subs.ctypes.data_as(_capi.c_int64_p)
    so.vals = None if vals is None else _dp(vals)
    return so, (subs, vals)


def device_count():
    n = C.c_int(0)
    _capi.check(lib.aoadmm_device_count(C.byref(n)))
    return n.value


def nccl_unique_id():
    buf = (C.c_uint8 * 128)()
    _capi.check(lib.aoadmm_nccl_unique_id(buf))
    return bytes(buf)


def shard_range(extent, rank, world_size):
    """Contiguous slab [lo, hi) of the last tensor mode owned by `rank` (SURVEY.md 8e: mode-3 slabs)."""
    lo = (extent * rank) // world_size
    hi = (extent * (rank + 1)) // world_size
    return lo, hi


def sparse_shard_bounds(X, n_gpus):
    """The n_gpus + 1 bounds of the last-mode slabs into which Solver(..., n_gpus=N, shard_sparse=True) cuts the sparse
    object X (sptensor or SciPy sparse matrix): GPU r owns last-mode indices bounds[r] .. bounds[r+1]-1.  The slabs
    balance the nonzeros (the rule is stated with aoadmm_sparse_shard_bounds in include/aoadmm.h)."""
    S = as_sparse(X)
    if S is None:
        raise AoadmmError(1, 'sparse_shard_bounds: X must be an sptensor or a SciPy sparse matrix')
    so, keep = _coo(S.subs, S.vals)
    b = np.zeros(max(int(n_gpus), 0) + 1, dtype=np.int64)
    _capi.check(lib.aoadmm_sparse_shard_bounds(C.byref(so), S.ndim, S.shape[-1], int(n_gpus),
                                               b.ctypes.data_as(_capi.c_int64_p)))
    return b


def constraint_spec(c):
    """Z.constraints{m} (name, params...) -> aoadmm_constraint (constraints_to_prox.m:13-91)."""
    spec = _capi.Constraint()
    spec.kind, spec.p0, spec.p1, spec.matrix, spec.matrix_n = 0, 0.0, 0.0, None, 0
    keep = None
    if c is None or len(c) == 0:
        return spec, keep
    name = c[0]
    if name not in _capi.CONSTRAINT_KINDS:
        raise ValueError('unknown constraint %r' % (name,))
    spec.kind = _capi.CONSTRAINT_KINDS[name]
    if name == 'box':
        spec.p0, spec.p1 = float(c[1]), float(c[2])
    elif name == 'unimodality':
        spec.p0 = 1.0 if c[1] else 0.0
    elif name == 'quadratic regularization':
        spec.p0 = float(c[1])
        keep = _f64(c[2])
        spec.matrix = _dp(keep)
        spec.matrix_n = keep.shape[0]
    elif name in ('non-negativity', 'non-decreasing', 'non-increasing', 'orthonormal', 'custom'):
        pass
    elif len(c) > 1 and np.isscalar(c[1]):
        spec.p0 = float(c[1])
    return spec, keep


class Solver:
    """Handle lifecycle around the C ABI: create (tensors to HBM once) -> set_state -> run -> get_state."""

    def __init__(self, Z, Znorm_const, rank=0, world_size=1, device=0, unique_id=None, shard=None, n_gpus=1,
                 devices=None, shard_sparse=False):
        """One GPU: defaults.  Several GPUs from THIS process (one caller, like a MATLAB session): n_gpus=N [, devices=[..]]
        with the whole objects in Z (aoadmm_create_multi cuts the slabs).  One process per GPU (torchrun): rank,
        world_size, device, unique_id [, shard] with this rank's slab or the whole object in Z.
        shard_sparse=True (with n_gpus): sparse objects are cut into nonzero-balanced slabs of their last mode
        (aoadmm_create_sparse_multi); `shards[p]` then lists the (lo, hi) slab of every GPU.  Without it sparse objects
        run on one GPU only."""
        if n_gpus > 1 and world_size > 1:
            raise ValueError('n_gpus > 1 (one process drives all GPUs) and world_size > 1 (one process per GPU) exclude each other')
        if shard_sparse and world_size > 1:
            raise AoadmmError(2, 'shard_sparse: sparse objects are sharded by one caller driving n_gpus GPUs, not with one '
                                 'process per GPU (world_size must be 1)')
        self.shard_sparse = bool(shard_sparse)
        self.n_gpus = int(n_gpus)
        self._keep = []
        self._h = _capi.HandleP()
        self.Z = Z
        nb_modes = len(Z['size'])
        modes = [list(m) for m in Z['modes']]
        P = len(modes)
        self.nb_modes, self.P = nb_modes, P
        which_p = {}
        for p in range(P):
            for m in modes[p]:
                which_p[m] = p
        model = list(Z['model'])
        for p in range(P):
            if Z['loss_function'][p] != 'Frobenius':
                raise AoadmmError(2, "loss function %r is not supported (Frobenius only)" % (Z['loss_function'][p],))
        miss = Z.get('miss') or [None] * P
        # sparse objects (aoadmm_create_sparse): the refused combinations raise here, before any device call
        sparse = [as_sparse(Z['object'][p]) if model[p] == 'CP' else None for p in range(P)]
        # sparse Z.miss masks (aoadmm_create_sparse_masked): only on sparse objects
        smask = [as_sparse(miss[p]) if model[p] == 'CP' and miss[p] is not None else None for p in range(P)]
        for p in range(P):
            if smask[p] is not None and sparse[p] is None:
                raise AoadmmError(1, 'Z.miss{%d} is sparse but Z.object{%d} is dense (a dense object takes a dense mask)'
                                  % (p + 1, p + 1))
        for p in range(P):
            if model[p] != 'CP' and any(as_sparse(x) is not None for x in Z['object'][p]):
                raise AoadmmError(2, 'object %d: PARAFAC2 objects with sparse slices are not supported' % (p + 1))
            if sparse[p] is None:
                continue
            if (n_gpus > 1 and not shard_sparse) or world_size > 1:
                raise AoadmmError(2, 'object %d is sparse: sparse objects run on one GPU (or on n_gpus GPUs with '
                                     'shard_sparse=True)' % (p + 1))
            if miss[p] is not None and smask[p] is None:
                raise AoadmmError(2, 'object %d is sparse: a dense Z.miss needs a dense object (a sparse object takes a '
                                     'sparse mask of its stored entries)' % (p + 1))
            want = tuple(int(Z['size'][m - 1]) for m in modes[p])
            if sparse[p].shape != want:
                raise AoadmmError(1, 'object %d: sparse shape %s does not match Z.size %s' % (p + 1, sparse[p].shape, want))
            if smask[p] is not None and smask[p].shape != want:
                raise AoadmmError(1, 'Z.miss{%d}: sparse mask shape %s does not match Z.object{%d} %s'
                                  % (p + 1, smask[p].shape, p + 1, want))
        sp_objs = (C.POINTER(_capi.SparseObject) * P)()
        sp_masks = (C.POINTER(_capi.SparseObject) * P)()
        ranks = self._infer_ranks(Z)
        rows = np.zeros(nb_modes, dtype=np.int64)
        nsl = np.zeros(nb_modes, dtype=np.int32)
        slice_rows = (_capi.c_int64_p * nb_modes)()
        for m in range(nb_modes):
            s = Z['size'][m]
            if isinstance(s, (list, tuple, np.ndarray)):
                arr = np.asarray(s, dtype=np.int64)
                self._keep.append(arr)
                slice_rows[m] = arr.ctypes.data_as(_capi.c_int64_p)
                nsl[m] = arr.size
                rows[m] = 0
            else:
                rows[m] = int(s)
        objs = (_capi.Object * P)()
        self.shards = []
        for p in range(P):
            o = objs[p]
            o.model = _capi.MODEL_CP if model[p] == 'CP' else _capi.MODEL_PAR2
            o.order = len(modes[p])
            marr = np.asarray(modes[p], dtype=np.int32)
            self._keep.append(marr)
            o.modes = marr.ctypes.data_as(_capi.c_int32_p)
            o.weight = float(Z['weights'][p])
            o.znorm_const = float(Znorm_const[p])
            if model[p] == 'CP' and sparse[p] is not None:
                full_last = int(Z['size'][modes[p][-1] - 1])
                if shard_sparse:
                    b = sparse_shard_bounds(sparse[p], self.n_gpus)
                    self.shards.append([(int(b[r]), int(b[r + 1])) for r in range(self.n_gpus)])
                else:
                    self.shards.append((0, full_last))
                subs = np.asfortranarray(sparse[p].subs)    # column-major: subs[d*nnz + e]
                vals = np.ascontiguousarray(sparse[p].vals)
                so = _capi.SparseObject()
                so.nnz = vals.size
                so.subs = subs.ctypes.data_as(_capi.c_int64_p)
                so.vals = _dp(vals)
                self._keep += [subs, vals, so]
                sp_objs[p] = C.pointer(so)
                if smask[p] is not None:
                    msubs = np.asfortranarray(smask[p].subs)
                    mvals = np.ascontiguousarray(smask[p].vals)
                    mo = _capi.SparseObject()
                    mo.nnz = mvals.size
                    mo.subs = msubs.ctypes.data_as(_capi.c_int64_p)
                    mo.vals = _dp(mvals)
                    self._keep += [msubs, mvals, mo]
                    sp_masks[p] = C.pointer(mo)
                o.data = None
                o.shard_offset, o.shard_extent = 0, full_last
                o.slices, o.n_slices = None, 0
                o.miss, o.miss_slices = None, None
            elif model[p] == 'CP':
                X = Z['object'][p]
                full_last = int(Z['size'][modes[p][-1] - 1])
                if shard is not None and shard[p] is not None:
                    lo, hi = shard[p]
                elif world_size > 1 and o.order >= 3 and X is not None and X.shape[-1] == full_last:
                    lo, hi = shard_range(full_last, rank, world_size)
                    X = X[..., lo:hi]
                else:
                    lo, hi = 0, full_last
                self.shards.append((lo, hi))
                if X is not None:
                    Xf = _f64(X)
                    self._keep.append(Xf)
                    o.data = _dp(Xf)
                else:
                    o.data = None
                o.shard_offset, o.shard_extent = lo, hi - lo
                o.slices, o.n_slices = None, 0
                o.miss, o.miss_slices = None, None
                if miss[p] is not None:   # Z.miss{p}: true = observed (example_script12_CP_PAR2_EM.m:118-124)
                    Mk = np.asarray(miss[p])
                    if Mk.shape[-1] == full_last and (hi - lo) != full_last:
                        Mk = Mk[..., lo:hi]
                    Mk = np.asfortranarray(Mk != 0, dtype=np.uint8)
                    if X is None or Mk.shape != np.shape(X):
                        raise AoadmmError(1, 'Z.miss{%d} size does not match Z.object{%d}.' % (p + 1, p + 1))
                    self._keep.append(Mk)
                    o.miss = Mk.ctypes.data_as(_capi.c_uint8_p)
            else:
                self.shards.append(None)
                sl = [_f64(x) for x in Z['object'][p]]
                self._keep.append(sl)
                arr = (_capi.c_double_p * len(sl))(*[_dp(x) for x in sl])
                self._keep.append(arr)
                o.data = None
                o.slices = arr
                o.n_slices = len(sl)
                o.miss, o.miss_slices = None, None
                if miss[p] is not None:
                    if not isinstance(miss[p], (list, tuple)) or len(miss[p]) != len(sl):
                        raise AoadmmError(1, 'Z.miss{%d} must be a cell array of length %d for PAR2.' % (p + 1, len(sl)))
                    for k, m in enumerate(miss[p]):          # cmtf_AOADMM.m:107-114
                        ma = np.asarray(m)
                        if ma.dtype != np.bool_ and not (np.issubdtype(ma.dtype, np.number) and np.all((ma == 0) | (ma == 1))):
                            raise AoadmmError(1, 'Z.miss{%d}{%d} must be a logical or binary (0/1) array.' % (p + 1, k + 1))
                    mk = [np.asfortranarray(np.asarray(m) != 0, dtype=np.uint8) for m in miss[p]]
                    for k, (m, x) in enumerate(zip(mk, sl)):
                        if m.shape != x.shape:
                            raise AoadmmError(1, 'Z.miss{%d}{%d} size does not match Z.object{%d}{%d}.' % (p + 1, k + 1, p + 1, k + 1))
                    marr = (_capi.c_uint8_p * len(mk))(*[m.ctypes.data_as(_capi.c_uint8_p) for m in mk])
                    self._keep += [mk, marr]
                    o.miss_slices = marr
        lin = np.asarray(Z['coupling']['lin_coupled_modes'], dtype=np.int32)
        ctype = np.asarray(Z['coupling'].get('coupling_type', []), dtype=np.int32)
        ncoup = int(lin.max()) if lin.size else 0
        trafo = Z['coupling'].get('coupl_trafo_matrices') or [None] * nb_modes
        trafo2 = Z['coupling'].get('coupl_trafo_matrices2') or [None] * nb_modes

        def mats(lst):
            ptrs = (_capi.c_double_p * nb_modes)()
            r = np.zeros(nb_modes, dtype=np.int64)
            c = np.zeros(nb_modes, dtype=np.int64)
            for m in range(nb_modes):
                H = lst[m] if m < len(lst) else None
                if H is not None and np.size(H) > 0:
                    Hf = _f64(H)
                    self._keep.append(Hf)
                    ptrs[m] = _dp(Hf)
                    r[m], c[m] = Hf.shape
            self._keep += [r, c]
            return ptrs, r, c

        tp, tr, tc = mats(trafo)
        tp2, tr2, tc2 = mats(trafo2)
        self.coupling_shapes = self._coupling_shapes(Z, ranks, ncoup, trafo, trafo2)
        crow = np.asarray([s[0] for s in self.coupling_shapes], dtype=np.int64)
        ccol = np.asarray([s[1] for s in self.coupling_shapes], dtype=np.int64)
        constrained = np.asarray(Z['constrained_modes'], dtype=np.int32)
        cons = (_capi.Constraint * nb_modes)()
        for m in range(nb_modes):
            c = Z['constraints'][m] if constrained[m] else None
            spec, keep = constraint_spec(c)
            cons[m] = spec
            if keep is not None:
                self._keep.append(keep)
        ridge = None
        if Z.get('ridge') is not None:
            ridge = np.asarray(Z['ridge'], dtype=np.float64)
        rk = np.asarray(ranks, dtype=np.int32)
        self.ranks = ranks
        pb = _capi.Problem()
        pb.nb_modes = nb_modes
        pb.mode_rows = rows.ctypes.data_as(_capi.c_int64_p)
        pb.mode_rank = rk.ctypes.data_as(_capi.c_int32_p)
        pb.slice_rows = slice_rows
        pb.n_slices = nsl.ctypes.data_as(_capi.c_int32_p)
        pb.n_objects = P
        pb.objects = objs
        pb.lin_coupled_modes = lin.ctypes.data_as(_capi.c_int32_p)
        pb.n_couplings = ncoup
        pb.coupling_type = ctype.ctypes.data_as(_capi.c_int32_p)
        pb.trafo, pb.trafo_rows, pb.trafo_cols = tp, tr.ctypes.data_as(_capi.c_int64_p), tc.ctypes.data_as(_capi.c_int64_p)
        pb.trafo2, pb.trafo2_rows, pb.trafo2_cols = tp2, tr2.ctypes.data_as(_capi.c_int64_p), tc2.ctypes.data_as(_capi.c_int64_p)
        pb.coupling_rows = crow.ctypes.data_as(_capi.c_int64_p)
        pb.coupling_cols = ccol.ctypes.data_as(_capi.c_int64_p)
        pb.constrained_modes = constrained.ctypes.data_as(_capi.c_int32_p)
        pb.constraints = cons
        pb.ridge = _dp(ridge) if ridge is not None else None
        self._keep += [rows, nsl, slice_rows, objs, lin, ctype, constrained, cons, ridge, rk, crow, ccol, tp, tp2]
        dist = _capi.Dist()
        dist.rank, dist.world_size, dist.device = rank, world_size, device
        if unique_id is not None:
            C.memmove(dist.nccl_unique_id, unique_id, 128)
        elif world_size > 1:
            raise ValueError('world_size > 1 needs the NCCL unique id of rank 0')
        self.rank, self.world_size = rank, world_size
        self.rows = rows
        self.nsl = nsl
        if self.n_gpus > 1 or shard_sparse:
            devs = None
            if devices is not None:
                devs = np.asarray(list(devices), dtype=np.int32)
                if devs.size != self.n_gpus:
                    raise ValueError('devices must list n_gpus ordinals')
                self._keep.append(devs)
            dp = devs.ctypes.data_as(_capi.c_int32_p) if devs is not None else None
            if shard_sparse:
                self._keep += [sp_objs, sp_masks]
                _capi.check(lib.aoadmm_create_sparse_multi(C.byref(pb), sp_objs,
                                                           sp_masks if any(m is not None for m in smask) else None,
                                                           self.n_gpus, dp, C.byref(self._h)))
            else:
                _capi.check(lib.aoadmm_create_multi(C.byref(pb), self.n_gpus, dp, C.byref(self._h)))
        else:
            if devices is not None:
                dist.device = int(list(devices)[0])
            if any(m is not None for m in smask):
                self._keep += [sp_objs, sp_masks]
                _capi.check(lib.aoadmm_create_sparse_masked(C.byref(pb), sp_objs, sp_masks, C.byref(dist),
                                                            C.byref(self._h)))
            elif any(sp is not None for sp in sparse):
                self._keep.append(sp_objs)
                _capi.check(lib.aoadmm_create_sparse(C.byref(pb), sp_objs, C.byref(dist), C.byref(self._h)))
            else:
                _capi.check(lib.aoadmm_create(C.byref(pb), C.byref(dist), C.byref(self._h)))
        self._keep_problem = pb

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _infer_ranks(Z):
        """columns of fac{m}: from Z['rank'] if present, else must be supplied with the state."""
        if 'rank' in Z:
            out = []
            for m in range(len(Z['size'])):
                p = [q for q in range(len(Z['modes'])) if (m + 1) in Z['modes'][q]][0]
                out.append(int(Z['rank'][p]))
            return out
        raise ValueError("Z['rank'] (components per object) is required")

    @staticmethod
    def _coupling_shapes(Z, ranks, ncoup, trafo, trafo2):
        lin = Z['coupling']['lin_coupled_modes']
        ctype = Z['coupling'].get('coupling_type', [])
        shapes = []
        for n in range(1, ncoup + 1):
            m1 = [m for m in range(1, len(lin) + 1) if lin[m - 1] == n][0]
            s = Z['size'][m1 - 1]
            r1 = int(s) if not isinstance(s, (list, tuple, np.ndarray)) else len(s)
            R1 = ranks[m1 - 1]
            H = trafo[m1 - 1] if m1 - 1 < len(trafo) else None
            ct = ctype[n - 1]
            if ct == 0:
                shapes.append((r1, R1))
            elif ct == 1:
                shapes.append((H.shape[0], R1))
            elif ct == 2:
                shapes.append((r1, H.shape[1]))
            elif ct == 3:
                shapes.append((H.shape[1], R1))
            elif ct == 4:
                shapes.append((r1, H.shape[0]))
            else:
                H2 = trafo2[m1 - 1]
                shapes.append((H.shape[0], H2.shape[0]))
        return shapes

    def close(self):
        if self._h:
            lib.aoadmm_destroy(self._h)
            self._h = _capi.HandleP()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------------------------------
    def _set(self, field, index, slice_, arr):
        a = _f64(arr)
        if a.ndim == 1:
            a = a.reshape(-1, 1)
        _capi.check(lib.aoadmm_set_state(self._h, field, index, slice_, _dp(a), a.shape[0], a.shape[1]), self._h)

    def _get(self, field, index, slice_, shape):
        a = np.zeros(shape, dtype=np.float64, order='F')
        _capi.check(lib.aoadmm_get_state(self._h, field, index, slice_, _dp(a), shape[0], shape[1]), self._h)
        return a

    def set_state(self, G):
        """Upload the state struct G (init_coupled_AOADMM_CMTF.m:41-45, :133-169)."""
        self._shapes = {}
        for m in range(1, self.nb_modes + 1):
            for field, key in ((_capi.FIELD_FAC, 'fac'), (_capi.FIELD_CONSTRAINT_FAC, 'constraint_fac'),
                               (_capi.FIELD_CONSTRAINT_DUAL, 'constraint_dual_fac'),
                               (_capi.FIELD_COUPLING_DUAL, 'coupling_dual_fac')):
                v = G.get(key, [None] * self.nb_modes)[m - 1]
                if v is None or (isinstance(v, (list, np.ndarray)) and len(v) == 0):
                    continue
                if isinstance(v, list):
                    for k, vk in enumerate(v):
                        self._set(field, m, k, vk)
                    self._shapes[(key, m)] = [np.shape(vk) for vk in v]
                else:
                    self._set(field, m, 0, v)
                    self._shapes[(key, m)] = np.shape(v)
        for n, D in enumerate(G.get('coupling_fac', []) or []):
            if D is not None:
                self._set(_capi.FIELD_COUPLING_FAC, n + 1, 0, D)
                self._shapes[('coupling_fac', n + 1)] = np.shape(D)
        for p in range(self.P):
            if self.Z['model'][p] != 'PAR2':
                continue
            for k, Pk in enumerate(G['P'][p]):
                self._set(_capi.FIELD_PAR2_P, p + 1, k, Pk)
            self._shapes[('P', p + 1)] = [np.shape(x) for x in G['P'][p]]
            self._set(_capi.FIELD_PAR2_DELTAB, p + 1, 0, G['DeltaB'][p])
            self._shapes[('DeltaB', p + 1)] = np.shape(G['DeltaB'][p])
            for k, mk in enumerate(G['mu_DeltaB'][p]):
                self._set(_capi.FIELD_PAR2_MU_DELTAB, p + 1, k, mk)
            self._shapes[('mu_DeltaB', p + 1)] = [np.shape(x) for x in G['mu_DeltaB'][p]]

    def get_state(self):
        """Download the full state in the layout of the reference's output G (cmtf_fun_AOADMM.m:1)."""
        nb = self.nb_modes
        G = {'fac': [None] * nb, 'constraint_fac': [None] * nb, 'constraint_dual_fac': [None] * nb,
             'coupling_dual_fac': [None] * nb, 'coupling_fac': [], 'P': [None] * self.P, 'DeltaB': [None] * self.P,
             'mu_DeltaB': [None] * self.P}
        fields = {'fac': _capi.FIELD_FAC, 'constraint_fac': _capi.FIELD_CONSTRAINT_FAC,
                  'constraint_dual_fac': _capi.FIELD_CONSTRAINT_DUAL, 'coupling_dual_fac': _capi.FIELD_COUPLING_DUAL}
        for (key, idx), shp in self._shapes.items():
            if key in fields:
                if isinstance(shp, list):
                    G[key][idx - 1] = [self._get(fields[key], idx, k, s) for k, s in enumerate(shp)]
                else:
                    G[key][idx - 1] = self._get(fields[key], idx, 0, shp)
        ncoup = len(self.coupling_shapes)
        G['coupling_fac'] = [None] * ncoup
        for n in range(1, ncoup + 1):
            if ('coupling_fac', n) in self._shapes:
                G['coupling_fac'][n - 1] = self._get(_capi.FIELD_COUPLING_FAC, n, 0, self._shapes[('coupling_fac', n)])
        for p in range(1, self.P + 1):
            if ('P', p) in self._shapes:
                G['P'][p - 1] = [self._get(_capi.FIELD_PAR2_P, p, k, s) for k, s in enumerate(self._shapes[('P', p)])]
                G['DeltaB'][p - 1] = self._get(_capi.FIELD_PAR2_DELTAB, p, 0, self._shapes[('DeltaB', p)])
                G['mu_DeltaB'][p - 1] = [self._get(_capi.FIELD_PAR2_MU_DELTAB, p, k, s)
                                         for k, s in enumerate(self._shapes[('mu_DeltaB', p)])]
        return G

    def run(self, options):
        """The body of cmtf_fun_AOADMM.m:32-506 on device; returns the `out` struct (:480-494)."""
        o = _capi.Options()
        o.MaxOuterIters = int(options['MaxOuterIters'])
        o.MaxInnerIters = int(options['MaxInnerIters'])
        o.AbsFuncTol = float(options['AbsFuncTol'])
        o.OuterRelTol = float(options['OuterRelTol'])
        o.innerRelPrTol_coupl = float(options['innerRelPrTol_coupl'])
        o.innerRelPrTol_constr = float(options['innerRelPrTol_constr'])
        o.innerRelDualTol_coupl = float(options['innerRelDualTol_coupl'])
        o.innerRelDualTol_constr = float(options['innerRelDualTol_constr'])
        o.bsum = int(bool(options.get('bsum', 0)))
        o.bsum_weight = float(options.get('bsum_weight', 0.0))
        o.iter_start_PAR2Bkconstraint = int(options.get('iter_start_PAR2Bkconstraint', 0))
        o.has_increase_factor_rhoBk = int('increase_factor_rhoBk' in options)
        o.increase_factor_rhoBk = float(options.get('increase_factor_rhoBk', 1.0))
        o.mttkrp_precision = int(options.get('mttkrp_precision', 0))
        o.dimtree = int(options.get('dimtree', 0))
        o.graph = int(options.get('graph', 0))
        o.fuse_inner = int(options.get('fuse_inner', 0))
        n = o.MaxOuterIters + 1
        hist = [np.zeros(n) for _ in range(5)]
        hmiss = np.full(n, np.nan)
        inner = np.zeros((self.nb_modes, max(o.MaxOuterIters, 1)), dtype=np.int32, order='F')
        out = _capi.Out()
        out.func_val_conv, out.func_coupl_conv, out.func_constr_conv, out.func_PAR2_coupl, out.time_at_it = \
            [_dp(h) for h in hist]
        out.inner_iters = inner.ctypes.data_as(_capi.c_int32_p)
        out.func_rel_missing = _dp(hmiss)
        _capi.check(lib.aoadmm_run(self._h, C.byref(o), C.byref(out)), self._h)
        it = out.OuterIterations
        self._last_iters = it
        if out.exit_flag == 0:
            flag = 'maxIterations'                                        # make_exit_flag.m:4-5
        elif out.exit_flag == 1 << 9:
            flag = 'heldoutStop'                                          # set_heldout_stopping
        else:
            names = ['f_tensors', 'f_couplings', 'f_constraints', 'f_PAR2_couplings']
            flag = {nm: ('AbsFuncTol' if (out.exit_flag >> q) & 1 else 'RelFuncTol') for q, nm in enumerate(names)}
        return {'f_tensors': out.f_tensors, 'f_couplings': out.f_couplings, 'f_constraints': out.f_constraints,
                'f_PAR2_couplings': out.f_PAR2_couplings, 'f_rel_missing': out.f_rel_missing,
                'func_rel_missing': hmiss[:it + 1].copy(), 'exit_flag': flag,
                'OuterIterations': it, 'func_val_conv': hist[0][:it + 1].copy(),
                'func_coupl_conv': hist[1][:it + 1].copy(), 'func_constr_conv': hist[2][:it + 1].copy(),
                'func_PAR2_coupl': hist[3][:it + 1].copy(), 'time_at_it': hist[4][:it + 1].copy(),
                'innerIters': inner[:, :it].astype(np.float64), 'non_finite_mode': int(out.non_finite_mode)}

    # ---- held-out entries ---------------------------------------------------------------------
    def model_at(self, obj, subs):
        """The current model of CP object `obj` (1-based) at the 0-based subscripts `subs` (nnz x N), in their order."""
        N = len(self.Z['modes'][obj - 1]) if 1 <= obj <= self.P else 1
        subs = np.asarray(subs, dtype=np.int64).reshape(-1, N)
        so, keep = _coo(subs, None)
        out = np.zeros(subs.shape[0])
        _capi.check(lib.aoadmm_model_at(self._h, int(obj), C.byref(so), _dp(out)), self._h)
        return out

    def set_heldout(self, obj, X):
        """Attach the held-out set `X` (an sptensor or SciPy sparse matrix of entries withheld from training, with their
        true values) to CP object `obj` (1-based), which must have missing data; X = None detaches it.  Every run then
        records the held-out SSE after each outer iteration (heldout_history)."""
        if X is None:
            _capi.check(lib.aoadmm_set_heldout(self._h, int(obj), None), self._h)
            return
        S = _check_heldout(self.Z, obj - 1, X)
        so, keep = _coo(S.subs, S.vals)
        _capi.check(lib.aoadmm_set_heldout(self._h, int(obj), C.byref(so)), self._h)

    def heldout_history(self, obj):
        """(sse, count): the held-out SSE after outer iterations 0..OuterIterations of the last run, and the number of
        held-out entries after merging duplicates."""
        n = getattr(self, '_last_iters', -1) + 1
        sse = np.full(max(n, 1), np.nan)
        count = C.c_int64(0)
        _capi.check(lib.aoadmm_heldout_history(self._h, int(obj), _dp(sse), n, C.byref(count)), self._h)
        return sse[:n], count.value

    def set_heldout_stopping(self, patience):
        """Early stopping on the held-out error: patience P >= 1 ends a run once P outer iterations have passed without
        a new smallest sum of the held-out SSEs, and leaves the solver in the state of the best iteration k* (factors,
        duals and the imputation of missing entries); the f_* values of `out` are then those at k*.  None or 0 turns it
        off.  Needs an attached held-out set (see include/aoadmm.h for the whole rule)."""
        _capi.check(lib.aoadmm_set_heldout_stopping(self._h, 0 if patience is None else int(patience)), self._h)

    def heldout_best(self):
        """(k*, s_k*) of the last run, which must have had early stopping on."""
        k, sse = C.c_int32(0), C.c_double(0)
        _capi.check(lib.aoadmm_heldout_best(self._h, C.byref(k), C.byref(sse)), self._h)
        return k.value, sse.value

    # ---- benchmark helpers --------------------------------------------------------------------
    def generate_cp_data(self, obj, factors, noise, seed):
        fs = [_f64(f) for f in factors]
        arr = (_capi.c_double_p * len(fs))(*[_dp(f) for f in fs])
        _capi.check(lib.aoadmm_generate_cp_data(self._h, obj, arr, float(noise), int(seed)), self._h)

    def get_object_data(self, obj, out):
        """This rank's slab of CP object `obj` (1-based) - the whole object for an n_gpus handle - into the F-contiguous
        float64 array `out`."""
        assert out.dtype == np.float64 and out.flags['F_CONTIGUOUS']
        _capi.check(lib.aoadmm_get_object_data(self._h, obj, _dp(out), out.size), self._h)
        return out

    def nvecs(self, mode, r, slice=0, return_info=False):
        """cmtf_nvecs(Z,n,r) (cmtf_nvecs.m:33-58) on the resident data: r leading eigenvectors of X_(n) X_(n)'.
        `mode` is the 1-based global mode id; `slice` (1-based) selects B_k of a PARAFAC2 object."""
        if not 1 <= mode <= len(self.Z['size']):
            raise AoadmmError(1, 'nvecs: mode out of range')
        s = self.Z['size'][mode - 1]
        if isinstance(s, (list, tuple, np.ndarray)):
            if not 1 <= slice <= len(s):
                raise AoadmmError(1, 'nvecs: a PARAFAC2 B_k mode needs slice = 1..K')
            rows = int(s[slice - 1])
        else:
            rows = int(s)
        out = np.zeros((rows, int(r)), order='F')
        info = np.zeros(2)
        _capi.check(lib.aoadmm_nvecs(self._h, int(mode), int(slice), int(r), _dp(out), rows, _dp(info)), self._h)
        return (out, {'iterations': int(info[0]), 'residual': float(info[1])}) if return_info else out

    def nvecs_sparse(self, mode, r, return_info=False):
        """nvecs of a mode whose first object is a sparse CP object (aoadmm_nvecs_sparse): the r leading eigenvectors of
        X_(n) X_(n)' with the unstored entries counted as zero, without forming X_(n) X_(n)'.  Same column order, signs
        and info as `nvecs`.  A mode of a dense or PARAFAC2 object is refused (use `nvecs`)."""
        rows = _check_nvecs_sparse(self.Z, mode, r)
        out = np.zeros((rows, int(r)), order='F')
        info = np.zeros(2)
        _capi.check(lib.aoadmm_nvecs_sparse(self._h, int(mode), int(r), _dp(out), rows, _dp(info)), self._h)
        return (out, {'iterations': int(info[0]), 'residual': float(info[1])}) if return_info else out

    def object_mttkrp(self, obj, pos, precision=0):
        """MTTKRP of resident CP object `obj` (1-based) in mode position `pos` with the current factors."""
        m = self.Z['modes'][obj - 1][pos - 1]
        out = np.zeros((int(self.Z['size'][m - 1]), int(self._infer_ranks(self.Z)[m - 1])), order='F')
        _capi.check(lib.aoadmm_object_mttkrp(self._h, obj, pos, int(precision), _dp(out)), self._h)
        return out

    def time_mttkrp(self, obj, pos, reps=3):
        ms = C.c_float(0)
        _capi.check(lib.aoadmm_time_mttkrp(self._h, obj, pos, reps, C.byref(ms)), self._h)
        return ms.value

    def launch_count(self):
        n = C.c_int64(0)
        _capi.check(lib.aoadmm_launch_count(self._h, C.byref(n)), self._h)
        return n.value

    def last_run_ms(self):
        v = C.c_double(0)
        _capi.check(lib.aoadmm_last_run_ms(self._h, C.byref(v)), self._h)
        return v.value

    def last_loop_ms(self):
        v = C.c_double(0)
        _capi.check(lib.aoadmm_last_loop_ms(self._h, C.byref(v)), self._h)
        return v.value

    def phase_ms(self):
        a = np.zeros(3)
        _capi.check(lib.aoadmm_phase_ms(self._h, _dp(a)), self._h)
        return a


def _with_rank(Z, G):
    """Z['rank'] is not a field of the reference struct: the rank is the column count of G.fac (cmtf_AOADMM.m:57)."""
    if 'rank' in Z:
        return Z
    Z = dict(Z)
    ranks = []
    for p, ms in enumerate(Z['modes']):
        f = G['fac'][ms[0] - 1]
        ranks.append(int((f[0] if isinstance(f, list) else f).shape[1]))
    Z['rank'] = ranks
    return Z


def cmtf_fun_AOADMM(Z, Znorm_const, G, fh=None, gh=None, lscalar=None, uscalar=None, options=None, heldout=None,
                    heldout_patience=None, **dist):
    """[G,out] = cmtf_fun_AOADMM(Z,Znorm_const,G,fh,gh,lscalar,uscalar,options)  (cmtf_fun_AOADMM.m:1).

    fh/gh/lscalar/uscalar are [] for the Frobenius loss (cmtf_AOADMM.m:158-161) and are ignored.
    `heldout`: one entry per object, None or a held-out set (sptensor / SciPy sparse) of an object with Z.miss; adds
    out['heldout_sse'] (per object: the SSE after outer iterations 0..OuterIterations, or None) and out['heldout_count'].
    `heldout_patience` (needs `heldout`): early stopping on the summed held-out SSE (Solver.set_heldout_stopping); G and
    the f_* values are those of the best iteration, out['heldout_best_iter'] is that iteration, and out['exit_flag'] is
    'heldoutStop' when the held-out rule ended the run.
    `dist` (rank, world_size, device, unique_id, or n_gpus [, devices, shard_sparse]) selects the multi-GPU layout;
    default one GPU."""
    if heldout is not None:
        if len(heldout) != len(Z['modes']):
            raise AoadmmError(1, 'heldout needs one entry per object (None where an object has no held-out set)')
        for p, X in enumerate(heldout):
            if X is not None:
                _check_heldout(Z, p, X)
    if heldout_patience is not None:
        if int(heldout_patience) < 0:
            raise AoadmmError(1, 'heldout_patience must be >= 0 (0: no early stopping)')
        if heldout_patience and not any(X is not None for X in (heldout or [])):
            raise AoadmmError(1, 'heldout_patience needs a held-out set (heldout=[...])')
    with Solver(_with_rank(Z, G), Znorm_const, **dist) as s:
        s.set_state(G)
        for p, X in enumerate(heldout or []):
            if X is not None:
                s.set_heldout(p + 1, X)
        if heldout_patience:
            s.set_heldout_stopping(int(heldout_patience))
        out = s.run(options)
        if heldout is not None:
            hist = [s.heldout_history(p + 1) if X is not None else (None, None) for p, X in enumerate(heldout)]
            out['heldout_sse'] = [h[0] for h in hist]
            out['heldout_count'] = [h[1] for h in hist]
        if heldout_patience:
            k_best, _ = s.heldout_best()
            want, k_stop = heldout_stopping_rule(_heldout_sum([h[0] for h in hist if h[0] is not None]),
                                                 int(heldout_patience))
            if k_best != want or (out['exit_flag'] == 'heldoutStop' and k_stop != out['OuterIterations']):
                raise AoadmmError(5, 'early stopping: the engine kept iteration %d, the rule gives %d' % (k_best, want))
            out['heldout_best_iter'] = k_best
        Gout = s.get_state()
    return Gout, out


def cmtf_AOADMM(Z, init, alg_options, init_options=None, **dist):
    """[Zhat,Fac,G,out] = cmtf_AOADMM(Z,'init',G,'alg_options',options)  (cmtf_AOADMM.m:1-207), Frobenius loss.
    init: the state struct G, or 'random' together with init_options (:44-53).

    The front end only computes Znorm_const (:124-156) and packs Zhat (:197-206); constraints stay named specs
    because the device cannot call MATLAB/Python function handles ('custom' -> AoadmmError UNSUPPORTED)."""
    P = len(Z['object'])
    for m, con in enumerate(Z['constraints']):                             # :33-39
        if Z['constrained_modes'][m] and con and con[0] == 'tPARAFAC2':
            p = [q for q in range(P) if (m + 1) in Z['modes'][q]][0]
            if Z['model'][p] != 'PAR2' or list(Z['modes'][p]).index(m + 1) != 1:
                raise ValueError('The tPARAFAC2 constraint can only be imposed on the second mode of a PARAFAC2 model')
    if isinstance(init, str):                                              # :44-53
        if init.lower() != 'random':
            raise ValueError('Initialization type not supported')
        if not init_options:
            raise ValueError('init_options are missing as input in cmtf_AOADMM.')
        init = init_coupled_AOADMM_CMTF(Z, init_options, **dist)
    for p in range(P):                                                     # :55-65 PARAFAC2 rank check
        if Z['model'][p] == 'PAR2':
            R = init['fac'][Z['modes'][p][0] - 1].shape[1]
            for k, jk in enumerate(Z['size'][Z['modes'][p][1] - 1]):
                if jk < R:
                    raise ValueError('Number of components for PARAFAC2 is larger than size of slice %d of data '
                                     'tensor %d.' % (k + 1, p + 1))
    zn = []
    miss = Z.get('miss') or [None] * P
    for p in range(P):                                                     # :124-156 (with Z.miss: observed entries only)
        if Z['model'][p] == 'CP' and as_sparse(Z['object'][p]) is not None:
            zn.append(float('nan'))                                        # computed on the device from the nonzeros
        elif Z['model'][p] == 'CP':
            X = np.asarray(Z['object'][p])
            if miss[p] is not None:
                X = X * (np.asarray(miss[p]) != 0)
            zn.append(float(np.linalg.norm(X.ravel()) ** 2))
        else:
            zn.append(float(sum(np.linalg.norm(Xk if miss[p] is None else Xk * (np.asarray(miss[p][k]) != 0), 'fro') ** 2
                                for k, Xk in enumerate(Z['object'][p]))))
    Fac, out = cmtf_fun_AOADMM(Z, zn, init, None, None, None, None, alg_options, **dist)
    Zhat = []
    for p in range(P):
        ms = Z['modes'][p]
        if Z['model'][p] == 'CP':
            Zhat.append([Fac['fac'][m - 1] for m in ms])
        else:
            Zhat.append({'A': Fac['fac'][ms[0] - 1], 'Bk': Fac['fac'][ms[1] - 1], 'C': Fac['fac'][ms[2] - 1]})
    return Zhat, Fac, init, out


# ---- operator-level entry points (tests / profiling) --------------------------------------------
def mttkrp(X, U, n, device=0):
    """Tensor Toolbox mttkrp(X,U,n) as called at cmtf_fun_AOADMM.m:97; n is 1-based."""
    Xf = _f64(X)
    Uf = [_f64(u) for u in U]
    dims = np.asarray(Xf.shape, dtype=np.int64)
    R = Uf[0].shape[1]
    out = np.zeros((Xf.shape[n - 1], R), order='F')
    arr = (_capi.c_double_p * len(Uf))(*[_dp(u) for u in Uf])
    _capi.check(lib.aoadmm_mttkrp(_dp(Xf), Xf.ndim, dims.ctypes.data_as(_capi.c_int64_p), arr, R, n, _dp(out), device))
    return out


def prox(constraint, X, rho=1.0, device=0):
    """feval(Z.prox_operators{m}, X, rho) for a named constraint spec (cmtf_fun_AOADMM.m:1424-1426)."""
    spec, keep = constraint_spec(constraint)
    Xf = _f64(X)
    out = np.zeros_like(Xf, order='F')
    _capi.check(lib.aoadmm_prox(C.byref(spec), _dp(Xf), Xf.shape[0], Xf.shape[1], float(rho), _dp(out), device))
    return out


def chol_solve(B, A, device=0):
    """(A/L')/L with L = chol(B','lower')  (cmtf_fun_AOADMM.m:142, :609)."""
    Bf, Af = _f64(B), _f64(A)
    out = np.zeros_like(Af, order='F')
    _capi.check(lib.aoadmm_chol_solve(_dp(Bf), Bf.shape[0], _dp(Af), Af.shape[0], _dp(out), device))
    return out


def gram(F, device=0):
    """F'*F (cmtf_fun_AOADMM.m:66)."""
    Ff = _f64(F)
    out = np.zeros((Ff.shape[1], Ff.shape[1]), order='F')
    _capi.check(lib.aoadmm_gram(_dp(Ff), Ff.shape[0], Ff.shape[1], _dp(out), device))
    return out


# ---- initialisation front end (the caller side of the boundary, SURVEY 8f-4) -------------------
def _refuse_sparse_nvecs(Z, mode_ids):
    """nvecs (cmtf_nvecs.m:6,13 refuses sparse input too) needs a dense unfolding of the first object holding the mode."""
    for n in mode_ids:
        p = [q for q in range(len(Z['modes'])) if n in list(Z['modes'][q])][0]
        if Z['model'][p] == 'CP' and as_sparse(Z['object'][p]) is not None:
            raise AoadmmError(2, 'nvecs: mode %d belongs to sparse object %d (initialise it from a distribution)' % (n, p + 1))


def _first_object(Z, n):
    return [q for q in range(len(Z['modes'])) if n in list(Z['modes'][q])][0]


def _is_sparse_mode(Z, n):
    p = _first_object(Z, n)
    return Z['model'][p] == 'CP' and as_sparse(Z['object'][p]) is not None


def _check_nvecs_sparse(Z, n, r):
    """host-side checks of nvecs_sparse (before any device call); returns the rows of mode n"""
    if not 1 <= n <= len(Z['size']):
        raise AoadmmError(1, 'nvecs_sparse: mode out of range')
    if not _is_sparse_mode(Z, n):
        raise AoadmmError(1, 'nvecs_sparse: mode %d belongs to a dense or PARAFAC2 object (use nvecs)' % n)
    rows = int(Z['size'][n - 1])
    if not 1 <= int(r) <= rows:
        raise AoadmmError(1, 'nvecs_sparse: the number of vectors must be between 1 and the mode size')
    return rows


def cmtf_nvecs(Z, n, r, solver=None, **dist):
    """U = cmtf_nvecs(Z,n,r)  (cmtf_nvecs.m:33-58): r leading eigenvectors of X_(n) X_(n)', computed on the device from
    the tensor resident in `solver` (or in a temporary handle), so a large tensor never has to be unfolded on the host."""
    _refuse_sparse_nvecs(Z, [n])
    if solver is not None:
        return solver.nvecs(n, r)
    P = len(Z['object'])
    with Solver(dict(Z, rank=[int(r)] * P), [float('nan')] * P, **dist) as s:
        return s.nvecs(n, r)


def cmtf_nvecs_sparse(Z, n, r, solver=None, **dist):
    """U = cmtf_nvecs(Z,n,r) for a mode whose first object is a sparse CP object (cmtf_nvecs refuses those): the r leading
    eigenvectors of X_(n) X_(n)' with the unstored entries counted as zero, on the device, without forming the n x n
    matrix.  A mode of a dense or PARAFAC2 object is refused before any device call (use cmtf_nvecs)."""
    _check_nvecs_sparse(Z, n, r)
    if solver is not None:
        return solver.nvecs_sparse(n, r)
    P = len(Z['object'])
    with Solver(dict(Z, rank=[int(r)] * P), [float('nan')] * P, **dist) as s:
        return s.nvecs_sparse(n, r)


def init_coupled_AOADMM_CMTF(Z, init_options, rng=None, Delta=None, **dist):
    """G = init_coupled_AOADMM_CMTF(Z,'init_options',init_options)  (init_coupled_AOADMM_CMTF.m:37-169).

    init_options: 'lambdas_init' (per object, its length is the rank), 'distr' (per mode, callable (rows, cols) ->
    array, the @(x,y) rand(x,y) handles of the example scripts), 'normalize', 'nvecs', 'nvecs_sparse'.  With nvecs the
    factors are the leading eigenvectors of X_(n) X_(n)' (:50-69), computed on the device; a mode of a sparse object is
    refused unless 'nvecs_sparse' is 1 as well, which computes it with nvecs_sparse (it has no effect without 'nvecs');
    constraint factors go through the device
    prox (:99-124); duals and coupling factors are uniform random (:126-169) from `rng` (numpy RandomState)."""
    rng = rng if rng is not None else np.random.RandomState()
    sz, modes, model = Z['size'], Z['modes'], Z['model']
    lambdas, distr = init_options['lambdas_init'], init_options['distr']
    normalize, use_nvecs = bool(init_options.get('normalize', 0)), bool(init_options.get('nvecs', 0))
    use_nvecs_sparse = use_nvecs and bool(init_options.get('nvecs_sparse', 0))
    lin = list(Z['coupling']['lin_coupled_modes'])
    ctype = list(Z['coupling'].get('coupling_type', []))
    trafo = Z['coupling'].get('coupl_trafo_matrices') or [None] * len(sz)
    constrained, constraints = Z['constrained_modes'], Z['constraints']
    P, nb_modes = len(modes), len(sz)
    if max(max(m) for m in modes) != nb_modes:
        raise ValueError('Mismatch between size and modes inputs')                       # :33-35
    nb_c = max(lin) if lin else 0
    G = {'fac': [None] * nb_modes, 'coupling_fac': [None] * nb_c, 'constraint_fac': [None] * nb_modes,
         'coupling_dual_fac': [None] * nb_modes, 'constraint_dual_fac': [None] * nb_modes,
         'P': [None] * P, 'DeltaB': [None] * P, 'mu_DeltaB': [None] * P}

    def normcols(M):
        return M / np.sqrt(np.sum(M * M, axis=0))[None, :]

    def rows_of(n):
        return int(sz[n - 1])

    solver = None
    if use_nvecs and not use_nvecs_sparse:
        _refuse_sparse_nvecs(Z, [n for p in range(P) for n in modes[p]])
    try:
        if use_nvecs:
            solver = Solver(dict(Z, rank=[len(l) for l in lambdas]), [float('nan')] * P, **dist)
        for p in range(P):
            R = len(lambdas[p])
            for n in modes[p]:
                pos = list(modes[p]).index(n)
                par2_b = model[p] == 'PAR2' and pos == 1
                if par2_b:
                    K = len(sz[n - 1])
                    G['DeltaB'][p] = rng.rand(R, R)
                    G['P'][p] = [np.eye(int(sz[n - 1][k]), R) for k in range(K)]
                    facs, mus = [], []
                    for k in range(K):
                        jk = int(sz[n - 1][k])
                        if use_nvecs:
                            Fk = solver.nvecs(n, R, slice=k + 1)                        # :61-66
                        else:
                            Fk = np.asarray(distr[n - 1](jk, R), dtype=np.float64)
                            if normalize:
                                Fk = normcols(Fk)
                        mus.append(rng.rand(jk, R))
                        facs.append(Fk)
                    G['fac'][n - 1], G['mu_DeltaB'][p] = facs, mus
                elif use_nvecs:
                    if model[p] == 'PAR2' and pos == 2:
                        G['fac'][n - 1] = np.ones((rows_of(n), R))                       # :68
                    elif use_nvecs_sparse and _is_sparse_mode(Z, n):
                        G['fac'][n - 1] = solver.nvecs_sparse(n, R)
                    else:
                        G['fac'][n - 1] = solver.nvecs(n, R)                             # :52, :55-60
                else:
                    F = np.asarray(distr[n - 1](rows_of(n), R), dtype=np.float64)
                    G['fac'][n - 1] = normcols(F) if normalize else F
    finally:
        if solver is not None:
            solver.close()
    for p in range(P):                                                                    # :99-124
        for n in modes[p]:
            if not constrained[n - 1]:
                continue
            if not constraints[n - 1]:
                raise ValueError('No constraint provided for mode %d.' % n)
            name = constraints[n - 1][0]
            if model[p] == 'PAR2' and list(modes[p]).index(n) == 1:
                zs, ds = [], []
                for Fk in G['fac'][n - 1]:
                    Zk = np.asarray(distr[n - 1](*Fk.shape), dtype=np.float64)
                    if name != 'tPARAFAC2':
                        Zk = prox(constraints[n - 1], Zk, 1.0, device=dist.get('device', 0))
                    zs.append(Zk)
                    ds.append(rng.rand(*Fk.shape))
                G['constraint_fac'][n - 1], G['constraint_dual_fac'][n - 1] = zs, ds
            else:
                if name == 'tPARAFAC2':
                    raise ValueError('The tPARAFAC2 constraint can only be imposed on the second mode of a PARAFAC2 model')
                F = G['fac'][n - 1]
                Zc = np.asarray(distr[n - 1](*F.shape), dtype=np.float64)
                G['constraint_fac'][n - 1] = prox(constraints[n - 1], Zc, 1.0, device=dist.get('device', 0))
                G['constraint_dual_fac'][n - 1] = rng.rand(*F.shape)
    for c in range(1, nb_c + 1):                                                          # :126-169
        cmodes = [m for m in range(1, nb_modes + 1) if lin[m - 1] == c]
        F1, H1 = G['fac'][cmodes[0] - 1], trafo[cmodes[0] - 1]
        ct = ctype[c - 1]
        if ct == 0:
            shape = F1.shape
        elif ct == 1:
            shape = (np.shape(H1)[0], F1.shape[1])
        elif ct == 2:
            shape = (F1.shape[0], np.shape(H1)[1])
        elif ct == 3:
            shape = (np.shape(H1)[1], F1.shape[1])
        elif ct == 4:
            shape = (F1.shape[0], np.shape(H1)[0])
        elif ct == 5:
            shape = np.shape(Delta[c - 1])
        else:
            raise ValueError('coupling type %r' % (ct,))
        G['coupling_fac'][c - 1] = rng.rand(*shape)
        for m in cmodes:
            if ct in (0, 1, 2):
                G['coupling_dual_fac'][m - 1] = rng.rand(*shape)
            elif ct in (3, 4):
                G['coupling_dual_fac'][m - 1] = rng.rand(*G['fac'][m - 1].shape)
            else:
                G['coupling_dual_fac'][m - 1] = rng.rand(shape[0], G['fac'][m - 1].shape[1])
    return G
