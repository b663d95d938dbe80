/*
 * aoadmm.h - C ABI of the B200-native AO-ADMM engine.
 *
 * Drop-in boundary: this library replaces the single call
 *     [Fac,out] = cmtf_fun_AOADMM(Z,Znorm_const,G,fh,gh,lscalar,uscalar,options)
 * made at functions/cmtf_AOADMM.m:193 of the reference (signature: functions/cmtf_fun_AOADMM.m:1).
 * The caller (MATLAB via the MEX gateway in matlab-code_b200/matlab/, or Python via ctypes)
 * still builds Z / options / G exactly as before (init_coupled_AOADMM_CMTF.m, constraints_to_prox.m);
 * the gateway flattens those structs into the plain-C structs below.
 *
 * Conventions
 *  - every matrix / tensor is IEEE double, column-major (MATLAB layout), dense;
 *  - mode ids, coupling ids are 1-based exactly as in Z.modes / Z.coupling.lin_coupled_modes;
 *  - the caller owns every host buffer; the library owns all device memory;
 *  - every entry point returns an aoadmm_status (0 = ok); no C++ exception crosses the ABI;
 *  - a handle is not thread-safe; one host thread drives one handle.  Multi-GPU comes in two forms:
 *      aoadmm_create_multi : ONE caller process / thread (a MATLAB session) hands over the whole problem and the
 *                            library drives n_gpus devices itself (the form the MEX gateway uses);
 *      aoadmm_create + aoadmm_dist : one process per GPU (torchrun / MPI launchers), each passing its own slab.
 */
#ifndef AOADMM_H_
#define AOADMM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 1: first release; 2: Z.miss masks, device Znorm_const, engine options (dimtree, fuse_inner, graph,
 * mttkrp_precision), out.f_rel_missing; 3: aoadmm_nvecs, aoadmm_object_mttkrp (no struct changed since 2);
 * 4: aoadmm_create_multi / aoadmm_gpu_count / aoadmm_comm_release, communicators cached per process,
 *    aoadmm_out.non_finite_mode appended (a non-finite inner residual no longer aborts the run);
 *    later additions that leave every v4 struct and entry point unchanged: aoadmm_sparse_object / aoadmm_create_sparse
 *    (sparse CP objects), aoadmm_create_sparse_masked (sparse Z.miss masks on sparse objects), aoadmm_model_at /
 *    aoadmm_set_heldout / aoadmm_heldout_history (held-out entries), aoadmm_sparse_shard_bounds /
 *    aoadmm_create_sparse_multi (sparse objects on several GPUs from one caller), aoadmm_set_heldout_stopping /
 *    aoadmm_heldout_best and bit 9 of aoadmm_out.exit_flag (early stopping on the held-out error), aoadmm_nvecs_sparse
 *    (nvecs of a sparse mode), aoadmm_create_sparse_slices (PARAFAC2 objects with sparse slices). */
#define AOADMM_ABI_VERSION 4

typedef struct aoadmm_handle aoadmm_handle;

/* Error convention: replaces MATLAB error() (cmtf_AOADMM.m:37,:48,:61; chol failure; the
 * 'MATLAB:nearlySingularMatrix' warning-as-error at cmtf_fun_AOADMM.m:83). */
typedef enum {
  AOADMM_OK = 0,
  AOADMM_ERR_INVALID_ARG = 1,
  AOADMM_ERR_UNSUPPORTED = 2,          /* 'custom' constraint, non-Frobenius loss, ... */
  AOADMM_ERR_NOT_POSITIVE_DEFINITE = 3, /* chol() would have thrown (cmtf_fun_AOADMM.m:142 ...) */
  AOADMM_ERR_NON_FINITE = 4,            /* kept for ABI stability; no entry point returns it since version 4 */
  AOADMM_ERR_CUDA = 5,
  AOADMM_ERR_NCCL = 6,
  AOADMM_ERR_OOM = 7,
  AOADMM_ERR_NO_DEVICE = 8
} aoadmm_status;

/* Z.model{p} */
typedef enum { AOADMM_MODEL_CP = 0, AOADMM_MODEL_PAR2 = 1 } aoadmm_model;

/* Z.constraints{m}{1}: the named specs of functions/constraints_to_prox.m:13-91
 * ("List of constraints and regularizations.txt" 1-21). */
typedef enum {
  AOADMM_CON_NONE = 0,
  AOADMM_CON_NONNEG = 1,            /* 'non-negativity'                      :13 */
  AOADMM_CON_BOX = 2,               /* 'box', l=p0, u=p1                     :15 */
  AOADMM_CON_SIMPLEX_COL = 3,       /* 'simplex column-wise', eta=p0         :19 */
  AOADMM_CON_SIMPLEX_ROW = 4,       /* 'simplex row-wise', eta=p0            :22 */
  AOADMM_CON_NONDECREASING = 5,     /* 'non-decreasing'                      :25 */
  AOADMM_CON_NONINCREASING = 6,     /* 'non-increasing'                      :27 */
  AOADMM_CON_UNIMODAL = 7,          /* 'unimodality', nonneg flag=p0         :29 */
  AOADMM_CON_L1_BALL = 8,           /* 'l1-ball', eta=p0                     :32 */
  AOADMM_CON_L2_BALL = 9,           /* 'l2-ball', eta=p0                     :35 */
  AOADMM_CON_NONNEG_L2_BALL = 10,   /* 'non-negative l2-ball', eta=p0        :38 */
  AOADMM_CON_NONNEG_L2_SPHERE = 11, /* 'non-negative l2-sphere'              :41 */
  AOADMM_CON_ORTHONORMAL = 12,      /* 'orthonormal'                         :44 */
  AOADMM_CON_L1_REG = 13,           /* 'l1 regularization', eta=p0           :46 */
  AOADMM_CON_L0_REG = 14,           /* 'l0 regularization', eta=p0           :50 */
  AOADMM_CON_L2_REG = 15,           /* 'l2 regularization', eta=p0           :54 */
  AOADMM_CON_RIDGE = 16,            /* 'ridge', eta=p0                       :58 */
  AOADMM_CON_QUADRATIC = 17,        /* 'quadratic regularization', eta=p0, L=matrix :62 */
  AOADMM_CON_GL_SMOOTH = 18,        /* 'GL smoothness', eta=p0               :68 */
  AOADMM_CON_TV = 19,               /* 'TV regularization', eta=p0           :78 */
  AOADMM_CON_TPARAFAC2 = 20,        /* 'tPARAFAC2', eta=p0                   :82 */
  AOADMM_CON_CUSTOM = 21            /* 'custom' (function handles) -> AOADMM_ERR_UNSUPPORTED :86 */
} aoadmm_constraint_kind;

typedef struct {
  int32_t kind;          /* aoadmm_constraint_kind */
  double p0, p1;         /* numeric parameters, see above */
  const double *matrix;  /* QUADRATIC: n x n col-major L; else NULL */
  int64_t matrix_n;
} aoadmm_constraint;

/* One entry of Z.object / Z.model / Z.modes / Z.weights + Znorm_const{p} (cmtf_AOADMM.m:124-156). */
typedef struct {
  int32_t model;          /* aoadmm_model */
  int32_t order;          /* number of modes of this object: 2 (matrix), >=3 (tensor); PAR2: 3 */
  const int32_t *modes;   /* `order` global 1-based mode ids (Z.modes{p}) */
  double weight;          /* Z.weights(p) */
  double znorm_const;     /* Znorm_const{p} = ||X_p||_F^2 (observed entries only with Z.miss); NaN = compute it on
                             the device from the data (cmtf_AOADMM.m:124-156) */
  /* CP: dense column-major data of THIS RANK's slab: extents size(modes[0..order-2]) x shard_extent.
   * With one GPU shard_offset = 0 and shard_extent = size of the last mode. */
  const double *data;
  int64_t shard_offset;   /* first index (0-based) of the last mode held by this rank */
  int64_t shard_extent;   /* number of last-mode indices held by this rank */
  /* PAR2: K slices X_k (I x J_k col-major); every rank passes all slices (small objects) */
  const double *const *slices;
  int32_t n_slices;
  /* Z.miss{p} (cmtf_AOADMM.m:68-121): NULL = no missing data; else one byte per element with the layout of
   * `data` (CP, this rank's slab) / of each slice (PAR2): 1 = observed, 0 = missing.  Missing entries are
   * re-imputed from the model after every outer iteration (cmtf_fun_AOADMM.m:408-441). */
  const uint8_t *miss;
  const uint8_t *const *miss_slices;
} aoadmm_object;

/* The problem struct Z (example_script6_matrix_matrix_CP_nonneg.m:84-92) flattened. */
typedef struct {
  int32_t nb_modes;
  const int64_t *mode_rows;          /* rows of fac{m}; for the PAR2 B_k mode: 0 (see slice_rows) */
  const int32_t *mode_rank;          /* columns of fac{m} */
  const int64_t *const *slice_rows;  /* per mode: NULL, or K values J_k for the PAR2 B_k mode (Z.size{m}) */
  const int32_t *n_slices;           /* per mode: 0, or K */
  int32_t n_objects;
  const aoadmm_object *objects;
  const int32_t *lin_coupled_modes;  /* nb_modes entries: 0 = uncoupled, else coupling id (1-based) */
  int32_t n_couplings;
  const int32_t *coupling_type;      /* per coupling id: 0 exact,1 HC=D,2 CH=D,3 C=HD,4 C=DH,5 H1C=DH2 */
  const double *const *trafo;        /* per mode: Z.coupling.coupl_trafo_matrices{m} or NULL */
  const int64_t *trafo_rows, *trafo_cols;
  const double *const *trafo2;       /* per mode: coupl_trafo_matrices2{m} or NULL (type 5) */
  const int64_t *trafo2_rows, *trafo2_cols;
  const int64_t *coupling_rows, *coupling_cols; /* per coupling id: shape of G.coupling_fac{c} (Delta) */
  const int32_t *constrained_modes;  /* Z.constrained_modes */
  const aoadmm_constraint *constraints; /* nb_modes entries (kind NONE where unconstrained) */
  const double *ridge;               /* Z.ridge (nb_modes) or NULL */
} aoadmm_problem;

/* Multi-GPU: one process per GPU.  The tensor objects are sharded along their LAST mode
 * (contiguous slabs in column-major order); rank r passes its slab (aoadmm_object.data,
 * shard_offset, shard_extent).  `nccl_unique_id` is the 128-byte ncclUniqueId created by rank 0
 * with aoadmm_nccl_unique_id() and distributed by the host (MPI / torch.distributed / files). */
typedef struct {
  int32_t rank, world_size;
  int32_t device;                 /* CUDA device ordinal for this process */
  uint8_t nccl_unique_id[128];
} aoadmm_dist;

/* options struct (example_script6...m:120-132, cmtf_fun_AOADMM.m:7-9, :196-198) */
typedef struct {
  int32_t MaxOuterIters, MaxInnerIters;
  double AbsFuncTol, OuterRelTol;
  double innerRelPrTol_coupl, innerRelPrTol_constr, innerRelDualTol_coupl, innerRelDualTol_constr;
  int32_t bsum;
  double bsum_weight;
  int32_t iter_start_PAR2Bkconstraint;
  int32_t has_increase_factor_rhoBk;
  double increase_factor_rhoBk;
  /* engine-only knobs (0 = default) */
  int32_t mttkrp_precision;   /* 0: FP64 DMMA (default, the parity mode).  Opt-in reduced precision for the MTTKRPs of
                                 3-way tensors (the tensor stays FP64 in HBM, the pass becomes HBM bound; everything else
                                 stays FP64): 1 = TF32 operands, 2 = BF16 operands, both on the 5th-generation tensor cores
                                 (tcgen05.mma, FP32 accumulation in TMEM per slab, FP64 across slabs; operand rounding
                                 2^-11 / 2^-8); 3 = TF32 on the mma.sync variant of the FP64 kernels (kept for comparison) */
  int32_t dimtree;            /* 0: three independent MTTKRP passes (reference flop/byte count) */
  int32_t fuse_inner;         /* 0 (default): run the whole inner ADMM loop of a group in one cooperative launch when
                                 possible; -1: one launch per inner iteration; results are identical */
  int32_t graph;              /* CUDA-graph replay of the outer iteration: 0 auto (launch-bound problems on one GPU),
                                 1 on, -1 off; results are identical */
} aoadmm_options;

/* out struct (cmtf_fun_AOADMM.m:480-494).  History arrays are caller-allocated with
 * MaxOuterIters+1 entries; inner_iters is nb_modes x MaxOuterIters column-major (out.innerIters). */
typedef struct {
  double f_tensors, f_couplings, f_constraints, f_PAR2_couplings;
  int32_t OuterIterations;
  int32_t exit_flag;          /* 0 'maxIterations'; else bit mask of the make_exit_flag.m:9-28 struct:
                                 bit0 f_tensors<AbsFuncTol, bit1 f_couplings, bit2 f_constraints,
                                 bit3 f_PAR2 (bit set = "AbsFuncTol", clear = "RelFuncTol"), bit8 = stopped;
                                 exactly 1 << 9: the held-out rule of aoadmm_set_heldout_stopping ended the run */
  double *func_val_conv, *func_coupl_conv, *func_constr_conv, *func_PAR2_coupl, *time_at_it;
  int32_t *inner_iters;
  int32_t error_mode;         /* mode id that raised NOT_POSITIVE_DEFINITE / NON_FINITE (0 if none) */
  double f_rel_missing;       /* out.f_rel_missing (NaN without Z.miss), cmtf_fun_AOADMM.m:436-440 */
  double *func_rel_missing;   /* out.func_rel_missing, MaxOuterIters+1 entries, or NULL */
  int32_t non_finite_mode;    /* 0, or the id of the first mode whose inner ADMM loop saw a NaN/Inf residual ratio
                                 (||fac|| = 0 or ||mu_DeltaB|| = 0, cmtf_fun_AOADMM.m:584, :1086-1112).  Like the
                                 reference the run goes on (NaN > tol is false, Inf > tol is true); this is a warning. */
} aoadmm_out;

/* State fields of G (init_coupled_AOADMM_CMTF.m:41-45, :62-80, :133-169) */
typedef enum {
  AOADMM_FIELD_FAC = 0,             /* G.fac{m}               index=m, slice=k (PAR2 B_k) or 0 */
  AOADMM_FIELD_CONSTRAINT_FAC = 1,  /* G.constraint_fac{m}                                      */
  AOADMM_FIELD_CONSTRAINT_DUAL = 2, /* G.constraint_dual_fac{m}                                 */
  AOADMM_FIELD_COUPLING_FAC = 3,    /* G.coupling_fac{c}      index=c (coupling id)             */
  AOADMM_FIELD_COUPLING_DUAL = 4,   /* G.coupling_dual_fac{m}                                   */
  AOADMM_FIELD_PAR2_P = 5,          /* G.P{p}{k}              index=p (1-based object), slice=k */
  AOADMM_FIELD_PAR2_DELTAB = 6,     /* G.DeltaB{p}                                              */
  AOADMM_FIELD_PAR2_MU_DELTAB = 7   /* G.mu_DeltaB{p}{k}                                        */
} aoadmm_field;

/* ---- lifecycle ---------------------------------------------------------------------------- */
int aoadmm_abi_version(void);
int aoadmm_device_count(int *count);
/* rank 0 fills the 128-byte id; replaces nothing in the reference (no distributed layer exists) */
int aoadmm_nccl_unique_id(uint8_t id[128]);
/* copies / partitions the data to HBM once.  dist may be NULL (single GPU, device 0).  With dist->world_size > 1 the
 * NCCL communicator of (nccl_unique_id, rank, world_size) is created on first use and cached for the life of the
 * process: passing the same id again (every rank alike) reuses it, so repeated solves pay the bootstrap once. */
int aoadmm_create(const aoadmm_problem *problem, const aoadmm_dist *dist, aoadmm_handle **out);
/* Multi-GPU from ONE caller (functions/cmtf_AOADMM.m:193 is one MATLAB process): `problem` describes the WHOLE
 * objects (shard_offset = 0, shard_extent = size of the last mode, `data` / `miss` = the full arrays).  The library
 * cuts every tensor of order >= 3 into n_gpus contiguous slabs of its last mode (slab r = indices
 * [extent*r/n, extent*(r+1)/n)), uploads slab r to devices[r] (NULL = devices 0..n_gpus-1) from its own worker
 * thread, creates the communicators with ncclCommInitAll (cached per device list) and returns ONE handle.  Every
 * entry point below then acts on all devices: set_state replicates, run drives one worker thread per GPU,
 * get_state / out come from device 0 (all replicas are bit-identical), aoadmm_get_object_data gathers the slabs.
 * n_gpus = 1 is the same as aoadmm_create(problem, {0,1,devices[0]}). */
int aoadmm_create_multi(const aoadmm_problem *problem, int32_t n_gpus, const int32_t *devices, aoadmm_handle **out);
/* number of GPUs driven by this handle (1 for aoadmm_create) */
int aoadmm_gpu_count(const aoadmm_handle *h, int32_t *n_gpus);
/* destroys every cached NCCL communicator of this process (no handle may be alive) */
int aoadmm_comm_release(void);
int aoadmm_destroy(aoadmm_handle *h);
const char *aoadmm_last_error(const aoadmm_handle *h); /* h may be NULL: last creation error */

/* One sparse CP object (Tensor Toolbox sptensor / MATLAB sparse): COO, 0-based. */
typedef struct {
  int64_t nnz;
  const int64_t *subs;   /* nnz x order, column-major: subs[d*nnz + e] = index of nonzero e in mode position d */
  const double *vals;    /* nnz values */
} aoadmm_sparse_object;

/* aoadmm_create with per-object sparse data: sparse[p] (n_objects entries) is NULL for a dense object, else the COO
 * data of CP object p (problem->objects[p].data must then be NULL).  dist: NULL or world_size 1.
 * Duplicate subscripts are summed (as the sptensor(subs,vals) constructor does); explicit zeros are kept.  The data is
 * sorted once on the device (one copy per mode); results do not depend on the order of the nonzeros.  A sparse object
 * always runs the FP64 sparse MTTKRP (options.mttkrp_precision and options.dimtree act on dense objects only);
 * Znorm_const = NaN is the sum of the squared (merged) values.
 * Checked before any device is touched: AOADMM_ERR_INVALID_ARG for nnz < 0, nnz > 0 with NULL subs / vals, a subscript
 * out of range, data and sparse[p] both set, a sparse object with a mode of more than 2^31 - 1 rows;
 * AOADMM_ERR_UNSUPPORTED for a sparse object with Z.miss, a sparse PARAFAC2 object, world_size > 1.
 * aoadmm_generate_cp_data, aoadmm_get_object_data and aoadmm_nvecs on a mode of a sparse object return
 * AOADMM_ERR_UNSUPPORTED; every other entry point works on such a handle. */
int aoadmm_create_sparse(const aoadmm_problem *problem, const aoadmm_sparse_object *const *sparse,
                         const aoadmm_dist *dist, aoadmm_handle **out);

/* aoadmm_create_sparse with sparse missing-data masks (Z.miss{p} given as an sptensor / MATLAB sparse matrix): masks is
 * NULL (= aoadmm_create_sparse) or n_objects entries; masks[p] may only be set where sparse[p] is.  A mask entry is
 * observed when its merged value (duplicates summed) is nonzero, and the observed entries must be exactly the stored
 * entries of the object (explicit zeros included): unstored entries are unobserved, not zero.  The run then equals the
 * dense EM path (cmtf_fun_AOADMM.m:408-441) on full(X) with the dense mask of that pattern: the unobserved entries start
 * at 0, the masked objective and f_rel_missing / func_rel_missing and its stopping rule (:457-459) are the same, and
 * nothing of size prod(size) is formed (memory grows by about 24 + 4*(order-1) bytes per nonzero plus a few
 * factor-sized buffers).  A second aoadmm_run continues from the last imputation.  aoadmm_object_mttkrp and
 * aoadmm_time_mttkrp act on the stored values, not on the imputed tensor.
 * Checked before any device is touched: AOADMM_ERR_INVALID_ARG for a malformed mask (as for sparse[p]), a mask on a
 * dense object, a mask together with a dense objects[p].miss.  After the device sort: AOADMM_ERR_UNSUPPORTED when the
 * observed pattern differs from the stored one (the message names the object). */
int aoadmm_create_sparse_masked(const aoadmm_problem *problem, const aoadmm_sparse_object *const *sparse,
                                const aoadmm_sparse_object *const *masks, const aoadmm_dist *dist, aoadmm_handle **out);

/* aoadmm_create_sparse with PARAFAC2 objects whose slices are sparse.  sparse: NULL or n_objects entries, set only for
 * CP objects, with the meaning and checks of aoadmm_create_sparse (no masks).  slices: NULL or n_objects entries, set
 * only for PARAFAC2 objects: slices[p] holds the K slices side by side as one order-2 COO object over I x Jtot
 * (Jtot = J_1 + ... + J_K from problem->slice_rows of the B_k mode): subs[e] = row i (0..I-1), subs[nnz + e] =
 * joff[k] + j with joff[k] = J_1 + ... + J_{k-1}; objects[p].slices must then be NULL.  Duplicates are summed, explicit
 * zeros are kept; results do not depend on the order of the entries.  Such an object never forms an I x Jtot array:
 * the products Xall W and Xall' A of the PARAFAC2 block are the deterministic sparse MTTKRP of the stacked object, the
 * explicit residual is one pass over the stored entries plus ||model||^2 from the Grams, it always runs FP64, and
 * Znorm_const = NaN is the sum of the squared merged values (about 2 * (12 + 4) bytes per stored entry on the device).
 * Checked before any device is touched: AOADMM_ERR_INVALID_ARG for NULL pointers, nnz < 0, a row or column subscript
 * out of range, dense and sparse slices both set, missing slice sizes, I or Jtot above 2^31 - 1, 2^31 - 257 entries
 * or more, slices[p] on a CP object or sparse[p] on a PARAFAC2 object; AOADMM_ERR_UNSUPPORTED for world_size > 1 and
 * objects[p].miss_slices on an object with sparse slices.  aoadmm_nvecs on the A or B_k mode of such an object returns
 * AOADMM_ERR_UNSUPPORTED; the other entry points refuse or accept it as they do a dense PARAFAC2 object. */
int aoadmm_create_sparse_slices(const aoadmm_problem *problem, const aoadmm_sparse_object *const *sparse,
                                const aoadmm_sparse_object *const *slices, const aoadmm_dist *dist,
                                aoadmm_handle **out);

/* ---- sparse objects on several GPUs from one caller ---------------------------------------------
 * aoadmm_sparse_shard_bounds: bounds[0..n_gpus] of the slabs of the last mode (extent indices) into which
 *     aoadmm_create_sparse_multi cuts a sparse object of `order` modes; GPU r owns indices bounds[r] .. bounds[r+1]-1.
 *     The slabs balance the number of nonzeros: with c[k] = the number of entries whose last subscript is k (duplicates
 *     counted before merging), C[k] = c[0] + ... + c[k-1] and nnz = so->nnz, bounds[0] = 0, bounds[n] = extent and for
 *     r = 1..n-1 bounds[r] = the smallest k with C[k] * n >= r * nnz, clamped to [bounds[r-1] + 1, extent - (n - r)] so
 *     that every GPU owns at least one index.  nnz = 0: the uniform slabs of dense objects (extent * r / n).  The bounds
 *     depend on the multiset of subscripts only, never on their order.  Host only; touches no device.
 *     AOADMM_ERR_INVALID_ARG for NULL pointers, order outside 2..8, n_gpus < 1, nnz < 0, a last subscript outside
 *     0..extent-1, and extent < n_gpus (fewer indices than there are GPUs).
 * aoadmm_create_sparse_multi: aoadmm_create_multi for a problem with sparse objects (sparse[p], masks[p] as in
 *     aoadmm_create_sparse_masked; masks may be NULL).  Takes whole objects.  Dense objects are cut as
 *     aoadmm_create_multi cuts them; every sparse CP object (order 2..8, matrices included) is cut into the slabs of
 *     aoadmm_sparse_shard_bounds, and its mask with the object's bounds.  The caller's entries are copied once into
 *     slab order on the host (8 * order + 8 bytes per nonzero of an object or mask, plus 4 bytes per nonzero while the
 *     bounds are computed); each GPU's worker thread then uploads and sorts only its own entries, so a GPU holds about
 *     1/n_gpus of the nonzeros and the limit of 2^31 - 257 nonzeros applies per GPU.  The factors stay replicated and
 *     full-size; per outer iteration every MTTKRP of a sparse object is all-reduced once (its last position as the
 *     zero-padded gather of the slabs), and a masked object all-reduces 4 more numbers in its EM step.  The results
 *     equal those of one GPU up to the summation order of the all-reduces; at a fixed n_gpus they are bit-reproducible
 *     and do not depend on the order of the nonzeros.  n_gpus = 1 gives the handle of aoadmm_create_sparse{,_masked}
 *     on devices[0].  Every check of aoadmm_create_sparse_masked and of aoadmm_sparse_shard_bounds on the descriptors
 *     happens before any device is touched; then the device checks of aoadmm_create_multi.  A mask whose observed
 *     pattern differs from the stored one inside one GPU's slab fails the whole create with AOADMM_ERR_UNSUPPORTED
 *     naming the object, and every device is released.  aoadmm_object_mttkrp returns the summed product,
 *     aoadmm_time_mttkrp times the slowest GPU's local pass; aoadmm_create_sparse{,_masked} with world_size > 1 stay
 *     AOADMM_ERR_UNSUPPORTED (one process per GPU is not offered for sparse objects). */
int aoadmm_sparse_shard_bounds(const aoadmm_sparse_object *so, int32_t order, int64_t extent, int32_t n_gpus,
                               int64_t *bounds);
int aoadmm_create_sparse_multi(const aoadmm_problem *problem, const aoadmm_sparse_object *const *sparse,
                               const aoadmm_sparse_object *const *masks, int32_t n_gpus, const int32_t *devices,
                               aoadmm_handle **out);

/* ---- held-out entries: how well the model predicts entries it was not trained on ----------------
 * aoadmm_model_at:   out[e] = the current model [[F_1, ..., F_N]] of CP object `object` (1-based) at the 0-based
 *                    subscripts entries->subs (entries->vals is ignored), in the caller's order.  Any CP object (dense,
 *                    sparse, with or without missing data) on any handle; with several GPUs device 0 evaluates (the
 *                    factors are replicated).
 * aoadmm_set_heldout: attaches a held-out set (entries withheld from training, with their true values) to a CP object
 *                    with missing data (a dense Z.miss, or a sparse mask of aoadmm_create_sparse_masked); entries = NULL
 *                    detaches it.  Duplicates are summed; the set is sorted once on the device, so results and their
 *                    bits do not depend on the order of the entries.  Everything is uploaded and allocated here: every
 *                    aoadmm_run then also computes the held-out SSE = sum (v - m)^2 after each outer iteration, inside
 *                    the CUDA graph when replay is on, with no extra synchronisation.  Attaching a set does not change
 *                    the solve (factors, duals and every out field are bit-identical).  With several GPUs the set is
 *                    replicated and every rank computes the same SSE without communication.  A failed call leaves the
 *                    object without a held-out set.
 * aoadmm_heldout_history: sse[i] (i < n) = the held-out SSE after outer iteration i of the last aoadmm_run, for
 *                    i = 0..OuterIterations (0 = the initial state, evaluated with the iteration-0 objective); NaN
 *                    beyond it.  *count (may be NULL) = the number of held-out entries after merging duplicates.
 * Checked before any device is touched: AOADMM_ERR_INVALID_ARG for NULL pointers, nnz < 0, an object index out of range,
 * a PARAFAC2 object, a subscript out of range, a held-out set on an object without missing data.  After the device sort,
 * aoadmm_set_heldout returns AOADMM_ERR_INVALID_ARG when a held-out entry was observed in training (a nonzero byte of a
 * dense mask, a stored entry of a sparse object); the message names the object and one such subscript. */
int aoadmm_model_at(aoadmm_handle *h, int32_t object, const aoadmm_sparse_object *entries, double *out);
int aoadmm_set_heldout(aoadmm_handle *h, int32_t object, const aoadmm_sparse_object *entries);
int aoadmm_heldout_history(const aoadmm_handle *h, int32_t object, double *sse, int64_t n, int64_t *count);

/* ---- early stopping on the held-out error: keep the best iterate and return it ------------------
 * Let s_k be the sum, over the objects with a held-out set (in object order), of the held-out SSE after outer iteration
 * k.  k* is the first k in 1..n with the smallest s_k: a new best must be strictly smaller, a NaN is never one, and the
 * initial state (k = 0) is not a candidate.  With patience P >= 1 the run ends after iteration k once k - k* >= P.
 * MaxOuterIters and the tolerance rule (evaluate_stopping_conditions.m:44, cmtf_fun_AOADMM.m:457-459) still apply; the
 * held-out rule ends the run only at an iteration where neither of them does.  However the run ends, the handle is
 * then left in the state after iteration k*: G, the PARAFAC2 state, the imputation of every object with missing data
 * and everything else a next aoadmm_run reads, so that run continues exactly as if this one had been made with
 * MaxOuterIters = k*.  When no s_k (k >= 1) is a number, or n = 0, k* = n and nothing is restored.
 * out: the history arrays and OuterIterations describe the n iterations run; f_tensors, f_couplings, f_constraints,
 * f_PAR2_couplings and f_rel_missing are the values at k* (the history entries at k*); exit_flag is exactly 1 << 9 when
 * the held-out rule ended the run, and what it would be without stopping otherwise.  With stopping off (the default)
 * nothing changes.
 * aoadmm_set_heldout_stopping: patience >= 1 turns stopping on, 0 turns it off.  The snapshot buffers are allocated here
 *     (one copy of the buffers above: about the size of G, the factor-side state, again) and freed when it is turned
 *     off, so aoadmm_run stays allocation-free.  A snapshot is one kernel launch after an iteration that sets a new best,
 *     outside the CUDA graph; the restore is one launch plus the EM pass of the objects with missing data.
 *     AOADMM_ERR_INVALID_ARG for a NULL handle, a negative patience, or (patience >= 1) no attached held-out set;
 *     AOADMM_ERR_OOM when the snapshot cannot be allocated, leaving stopping off.  aoadmm_run returns
 *     AOADMM_ERR_INVALID_ARG before any device work when stopping is on but every held-out set has been detached.
 *     With several GPUs every rank sees the same SSE bits and makes the same decisions without communication; each
 *     snapshots and restores what it holds.
 * aoadmm_heldout_best: k* and s_{k*} of the last run (n = 0: 0 and s_0).  AOADMM_ERR_INVALID_ARG when the last run had
 *     stopping off, or when there was no run. */
int aoadmm_set_heldout_stopping(aoadmm_handle *h, int32_t patience);
int aoadmm_heldout_best(const aoadmm_handle *h, int32_t *iteration, double *sse);

/* ---- state in / out (G is both input and output of cmtf_fun_AOADMM.m:1) ------------------- */
int aoadmm_set_state(aoadmm_handle *h, int32_t field, int32_t index, int32_t slice,
                     const double *data, int64_t rows, int64_t cols);
int aoadmm_get_state(aoadmm_handle *h, int32_t field, int32_t index, int32_t slice,
                     double *data, int64_t rows, int64_t cols);

/* ---- the solver: the body of cmtf_fun_AOADMM.m:32-506 ------------------------------------- */
int aoadmm_run(aoadmm_handle *h, const aoadmm_options *options, aoadmm_out *out);

/* ---- operator-level entry points (the reference's L0/L1 calls, for tests / profiling) ------
 * aoadmm_mttkrp:   Tensor Toolbox mttkrp(X,U,n) as called at cmtf_fun_AOADMM.m:97 (n 1-based).
 *                  X: dims[0..order-1] col-major host buffer, factors[k]: dims[k] x R host buffers,
 *                  out: dims[n-1] x R host buffer.
 * aoadmm_prox:     feval(Z.prox_operators{m}, X, rho) (cmtf_fun_AOADMM.m:1424-1426) for a named spec.
 * aoadmm_chol_solve: X = (A / L') / L with L = chol(B','lower') (cmtf_fun_AOADMM.m:142, :609).
 * aoadmm_gram:     G = F'*F (cmtf_fun_AOADMM.m:66, :148).
 */
int aoadmm_mttkrp(const double *X, int32_t order, const int64_t *dims, const double *const *factors,
                  int32_t R, int32_t n, double *out, int32_t device);
int aoadmm_prox(const aoadmm_constraint *spec, const double *X, int64_t rows, int64_t cols, double rho,
                double *out, int32_t device);
int aoadmm_chol_solve(const double *B, int32_t R, const double *A, int64_t rows, double *X, int32_t device);
int aoadmm_gram(const double *F, int64_t rows, int32_t R, double *G, int32_t device);

/* ---- device-resident benchmark helpers ----------------------------------------------------
 * Replace the data of CP object `object` (1-based) by a synthetic tensor generated ON DEVICE:
 * X = [[lambda; U_1..U_N]] + sigma*N(0,1) with sigma = noise*||X0||/||N|| (create_coupled_data.m:158-162),
 * then normalised to ||X||_F = 1 (example_script6...m:101-102).  factors[k] are host buffers of the
 * full (unsharded) factor matrices.  Needed for configs whose tensor does not fit host memory
 * (SURVEY.md 8d C3).  Writes the new Znorm_const (=1) into the handle. */
int aoadmm_generate_cp_data(aoadmm_handle *h, int32_t object, const double *const *factors,
                            double noise, uint64_t seed);
/* Copy this rank's slab of CP object `object` (1-based) back to a caller buffer with the layout aoadmm_create
 * takes (dims of the leading modes x shard_extent, column-major, no padding).  bench.py uses it to obtain the
 * device-generated tensor as a HOST buffer for the end-to-end leg. */
int aoadmm_get_object_data(aoadmm_handle *h, int32_t object, double *out, int64_t n_elements);
/* Leading eigenvectors for the 'nvecs' initialisation (cmtf_nvecs.m:33-58; init_coupled_AOADMM_CMTF.m:50-69):
 * out (rows x r, column-major host buffer) = eigs(Y, r, 'LM') with Y = X_(mode) X_(mode)' of the first object that
 * contains global mode id `mode` (1-based), computed from the data resident in the handle.  PARAFAC2 objects: mode A uses
 * the slices side by side, a B_k mode needs `slice` (1-based; Y = X_k' X_k), mode C is ones in the reference and is
 * refused.  slice = 0 otherwise.  Columns come in descending eigenvalue order, each signed so that its entry of
 * largest magnitude is positive (eigs leaves the sign open).  info (may be NULL): [0] subspace iterations,
 * [1] max ||Y u - theta u|| / theta_1 over the returned pairs.  With more than one GPU every rank must make the call
 * (collective): partial Gram matrices of the slabs are all-reduced; for the sharded (last) mode the slabs are exchanged
 * chunk by chunk with NCCL point-to-point transfers. */
int aoadmm_nvecs(aoadmm_handle *h, int32_t mode, int32_t slice, int32_t r, double *out, int64_t rows, double *info);
/* aoadmm_nvecs for a mode whose first object is a sparse CP object (aoadmm_nvecs refuses those): the r leading
 * eigenvectors of Y = X_(mode) X_(mode)' with the unstored entries counted as zero (a masked object: its stored, observed
 * values; the imputation state never enters).  Y is never formed: Y V = U (U' V) on the unfolding U with its columns
 * compressed to the fibers that occur, two deterministic passes over the nonzeros per iteration; results do not depend
 * on the order of the nonzeros or on the memory free at the call.  Same column order, sign rule and info as aoadmm_nvecs.
 * The call allocates its own temporaries and frees them; the handle's state is unchanged.
 * AOADMM_ERR_INVALID_ARG for a mode whose first object is dense or PARAFAC2 (use aoadmm_nvecs), r outside 1..rows,
 * rows not the mode size; AOADMM_ERR_UNSUPPORTED for the last mode of a sparse object on several GPUs (its fibers cross
 * GPUs); AOADMM_ERR_OOM when not even one column of the operator fits in half of the free device memory.  With more
 * than one GPU every rank must make the call (collective). */
int aoadmm_nvecs_sparse(aoadmm_handle *h, int32_t mode, int32_t r, double *out, int64_t rows, double *info);
/* MTTKRP of the resident CP object `object` in mode position `pos` (1-based) with the factors currently in the handle
 * (cmtf_fun_AOADMM.m:97), at `precision` (0 FP64, 1/2/3 reduced precision: see aoadmm_options.mttkrp_precision), summed over
 * ranks; out: rows(mode) x R host buffer. */
int aoadmm_object_mttkrp(aoadmm_handle *h, int32_t object, int32_t pos, int32_t precision, double *out);
/* one timed MTTKRP of object `object` in mode position `pos` (1-based position inside the object)
 * using the factors currently resident in the handle; returns device milliseconds (CUDA events). */
int aoadmm_time_mttkrp(aoadmm_handle *h, int32_t object, int32_t pos, int32_t reps, float *ms_out);
/* number of kernels launched by this handle so far, summed over its GPUs (bench.py "gpu_launches"). */
int aoadmm_launch_count(const aoadmm_handle *h, int64_t *count);
/* per-phase device time accumulated by aoadmm_run since creation, milliseconds:
 * [0] MTTKRP (tensor), [1] matrix-block products, [2] everything else */
int aoadmm_phase_ms(const aoadmm_handle *h, double ms[3]);
/* device time (CUDA events on the engine's stream, first to last kernel) of the last aoadmm_run, ms */
int aoadmm_last_run_ms(const aoadmm_handle *h, double *ms);
/* same, but only the outer iterations (cmtf_fun_AOADMM.m:87-476), i.e. without the one-off iteration-0 objective
 * of cmtf_fun_AOADMM.m:32 (one extra MTTKRP per tensor) */
int aoadmm_last_loop_ms(const aoadmm_handle *h, double *ms);

#ifdef __cplusplus
}
#endif
#endif /* AOADMM_H_ */
