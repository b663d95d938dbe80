// sparse.cuh - sparse (COO) CP objects: device layout, preprocessing and the deterministic sparse MTTKRP (sm_100a).
//
// Replaces the Tensor Toolbox sptensor mttkrp / norm (and Y*F for a MATLAB sparse matrix) behind
// cmtf_fun_AOADMM.m:97.  The engine only calls sparse_build / sparse_mttkrp / sparse_norm2 / sparse_free; the layout
// below is private to sparse.cu.
//
// Layout: for every mode position n a mode-n-sorted copy of the merged nonzeros (duplicates summed): lexicographic
// order with i_n as the major key and the other modes in ascending position, FP64 values, the other modes' indices as
// int32 (column-major, one array per other mode) and an int64 row pointer over i_n.
//
// MTTKRP: the nonzeros are cut into units of kSparseChunk consecutive entries (compile-time constant, so the summation
// order never depends on the launch configuration).  A group of lanes (columns across lanes) walks one unit; a row that
// starts and ends inside the unit is written directly, the partial rows at the unit's ends go to carry buffers, and a
// fix-up pass adds the carries of a split row in unit order.  No floating-point atomics: every output is bit-reproducible.
//
// Several GPUs (aoadmm_create_sparse_multi): each GPU holds the nonzeros of one contiguous slab of the last mode,
// shard_offset .. shard_offset + shard_extent - 1.  The nonzero side (the sorted copies, the imputation state m / r) is
// local, with the last subscript shifted into the slab on the device; the factors and the factor side of the EM state
// (B, the cross-Grams, the stacks and their Grams) keep the full extents and are replicated.  The caller all-reduces the
// partial products (sparse_mttkrp) and the nonzero-side EM sums (sparse_em_nonzeros), then adds the replicated terms.
#pragma once
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace aoadmm {

constexpr int kSparseChunk = 256;   // nonzeros per unit of work

// lanes per nonzero (G) and columns per lane (CPL) for rank R: f(integral_constant<G>, integral_constant<CPL>)
template <typename Fn>
void rank_dispatch(int R, Fn&& f) {
  using std::integral_constant;
  if (R <= 1) f(integral_constant<int, 1>{}, integral_constant<int, 1>{});
  else if (R <= 2) f(integral_constant<int, 2>{}, integral_constant<int, 1>{});
  else if (R <= 4) f(integral_constant<int, 4>{}, integral_constant<int, 1>{});
  else if (R <= 8) f(integral_constant<int, 8>{}, integral_constant<int, 1>{});
  else if (R <= 16) f(integral_constant<int, 16>{}, integral_constant<int, 1>{});
  else if (R <= 32) f(integral_constant<int, 32>{}, integral_constant<int, 1>{});
  else if (R <= 64) f(integral_constant<int, 32>{}, integral_constant<int, 2>{});
  else if (R <= 128) f(integral_constant<int, 32>{}, integral_constant<int, 4>{});
  else f(integral_constant<int, 32>{}, integral_constant<int, 8>{});
}

// CTAs of a pass in which one group of G lanes walks each unit of kSparseChunk entries
long long model_blocks(long long n, int R);

// m(e) = sum_c prod_d F_d(i_d, c) for entry e of a COO list: position-1 subscripts row0[e], positions 2..no+1 at
// idx[(d-1) * stride + e]; F row-major.  Lane gl of a group of G owns columns gl, gl + G, ... (ascending), the group
// sums its lanes with a fixed xor tree, so the bits depend on R and the data only.  Every lane of the warp must call it
// (ok = false: the lane has no entry and contributes 0).
template <int G, int CPL>
__device__ __forceinline__ double model_at_entry(const double* const (&F)[8], const int* row0, const int* idx,
                                                 long long stride, int no, int R, long long e, int gl, bool ok) {
  double t = 0.0;
  if (ok) {
    double p[CPL];
    const double* f0 = F[0] + (long long)__ldg(row0 + e) * R;
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
      const int c = gl + G * q;
      p[q] = c < R ? __ldg(f0 + c) : 0.0;
    }
    for (int m = 0; m < no; ++m) {
      const double* f = F[m + 1] + (long long)__ldg(idx + m * stride + e) * R;
#pragma unroll
      for (int q = 0; q < CPL; ++q) {
        const int c = gl + G * q;
        if (c < R) p[q] *= __ldg(f + c);
      }
    }
#pragma unroll
    for (int q = 0; q < CPL; ++q) t += p[q];
  }
#pragma unroll
  for (int off = G / 2; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
  return t;
}

// out(j + ldo*i) = scale * in(i + ldi*j), i < rows, j < cols (the row-major factor copies).  Returns the launches.
int transpose_scale(const double* in, long long rows, long long cols, long long ldi, double* out, long long ldo, double scale,
                    cudaStream_t st);

// Uploads n > 0 COO entries (subs n x order column-major, 0-based, validated by the caller), sorts them on the device
// into full lexicographic order (mode 0 major) and sums duplicates.  *subs_out (order x nm int32, column-major) and
// *vals_out (nm) are new device allocations owned by the caller.  Synchronous on `st`; returns nm.
long long coo_sort_merge(int order, const long long* dims, long long n, const long long* subs, const double* vals,
                         cudaStream_t st, int** subs_out, double** vals_out);

struct SparseMode {
  long long* rowptr = nullptr;      // rows + 1
  int* chunk_row = nullptr;         // row of the first nonzero of every unit
  int* head_row = nullptr;          // per unit: its first row when that row began in an earlier unit, else -1
  int* tail_row = nullptr;          // per unit: its last row when that row goes on in a later unit, else -1
  double* vals = nullptr;           // nnz
  int* idx = nullptr;               // (order-1) x nnz: indices of the other modes in ascending position
  int* perm = nullptr;              // masked objects, positions >= 1: canonical index of every nonzero of this copy
};

struct SparseTensor {
  int order = 0, R = 0;
  long long nnz = 0;                // after merging duplicates (this GPU's slab)
  long long dims[8] = {0};          // extents of the nonzero side: the last one is the slab extent
  long long fdims[8] = {0};         // full extents (factor side)
  long long shift = 0;              // first last-mode index of the slab
  std::vector<SparseMode> modes;
  double* factT[8] = {nullptr};     // row-major (rows x R) copies of the factors, refreshed per MTTKRP
  double* outT = nullptr;           // row-major product, max rows x R
  double* head = nullptr;           // units x R: partial sums of the head rows
  double* tail = nullptr;           // units x R: partial sums of the tail rows
  double* norm_partials = nullptr;  // deterministic two-level reduction
  double* norm_out = nullptr;
  // Z.miss on a sparse object (aoadmm_create_sparse_masked): EM imputation state, allocated for masked objects only.
  // Canonical order = the order of the position-1 copy.
  bool masked = false;
  int* row0 = nullptr;              // nnz: position-1 subscript of every nonzero (canonical order)
  double* mvals = nullptr;          // nnz: model [[B]] at the nonzeros (canonical order)
  double* rvals = nullptr;          // nnz: residual s - m (canonical order); the imputed MTTKRP streams these
  double* B[8] = {nullptr};         // dims[d] x R column-major: factors at the last imputation (all zero before it)
  double* cg = nullptr;             // order x R x R: cross-Grams B_d' F_d with the current factors F_d
  double* H = nullptr;              // R x R: Hadamard product of the cross-Grams of the other positions
  double* stack = nullptr;          // max rows x 3R: [F_d | B_d | F_d - B_d]
  double* g3 = nullptr;             // order x (3R)^2: Grams of the stacks
  double* gemm_ws = nullptr;        // split-K partial tiles of the Gram products
  double* em_partials = nullptr;    // per-CTA sums of the model pass (4 per CTA) and of the telescoped norms (2 per CTA)
  double* em_nz = nullptr;          // 4: nonzero-side sums of the model pass (sparse_em_nonzeros)
};

// Uploads and preprocesses one COO object: subs is nnz x order column-major (0-based, validated by the caller), vals nnz
// values.  Duplicates are summed.  Allocates every scratch buffer the MTTKRP needs.  Synchronous on `st`.
// full_dims: the object's extents; the entries all lie in the slab [shard_offset, shard_offset + shard_extent) of the
// last mode (whole object: 0, full_dims[order - 1]).
// masked: the object has a sparse Z.miss mask (mask_nnz entries, same layout as subs / vals).  An entry is observed when its merged value
// is nonzero; the observed set must equal the stored set of the object (else CudaError UNSUPPORTED).  Allocates the EM
// state (sparse.cuh above) with m = 0, r = s, B = 0.
// model_pass: keep row0 and the per-CTA partials of one model pass (sparse_par2_residual) without the EM state.
void sparse_build(SparseTensor& s, int order, const long long* full_dims, long long shard_offset, long long shard_extent,
                  int R, long long nnz, const long long* subs, const double* vals, cudaStream_t st, bool masked = false,
                  long long mask_nnz = 0, const long long* mask_subs = nullptr, const double* mask_vals = nullptr,
                  bool model_pass = false);
void sparse_free(SparseTensor& s);
// ||X||_F^2 = sum of the squared merged values (fixed-order reduction); the result lands in s.norm_out (device).  A slab
// gives its partial sum.
int sparse_norm2(const SparseTensor& s, cudaStream_t st);
// out (rows(n) x R, column-major, leading dimension ldout) = scale * MTTKRP of mode position n over this GPU's nonzeros,
// from the full column-major factors fac[d] (leading dimension ld[d]) of all mode positions.  For the last position only
// the slab's rows (at their global position) are written.  Returns the number of kernel launches.
// imputed (masked objects): the sparse pass over the residuals r, the first part of the MTTKRP of the imputed tensor
// S + (1-W).*[[B]] = (S - W.*[[B]]) + [[B]]; sparse_lowrank_add adds the second; else the MTTKRP of the stored values.
int sparse_mttkrp(SparseTensor& s, int n, const double* const* fac, const long long* ld, double scale, double* out,
                  long long ldout, cudaStream_t st, bool imputed = false);
// masked objects: out (full rows(n) x R) += scale * B_n * (Hadamard of cg_k, k != n), the low-rank term of the imputed
// MTTKRP.  It only reads replicated state: with several GPUs it is added once, after the all-reduce of the sparse part.
int sparse_lowrank_add(SparseTensor& s, int n, double scale, double* out, long long ldout, cudaStream_t st);
// masked objects: cg_n = B_n' * F (F: dims[n] x R, leading dimension ld), after every update of position n
int sparse_cross_gram(SparseTensor& s, int n, const double* F, long long ld, cudaStream_t st);
// masked objects: the EM step of cmtf_fun_AOADMM.m:408-441 without a dense tensor, in two parts (graph-capturable).
// sparse_em_nonzeros: one pass over this GPU's nonzeros computes m' = [[F]] there and the nonzero-side sums s.em_nz =
// [sum s m', sum m'^2, sum_W (m' - m)^2, sum_W m^2]; impute: afterwards m = m', r = s - m'.  With several GPUs the
// caller all-reduces the 4 values of s.em_nz.
// sparse_em_finish: the replicated factor side, then sums[2] = sum s m', sums[3] = sum m'^2 (masked objective),
// sums[0] / sums[1] = the missing-entry numerator / denominator of f_rel_missing from the telescoped ||[[F]] - [[B]]||^2
// and ||[[B]]||^2 minus the nonzero-side terms, sums[4] = 0; impute: B = F and the cross-Grams are refreshed.
int sparse_em_nonzeros(SparseTensor& s, const double* const* fac, const long long* ld, bool impute, cudaStream_t st);
int sparse_em_finish(SparseTensor& s, const double* const* fac, const long long* ld, bool impute, double* sums,
                     cudaStream_t st);

// PARAFAC2 object with sparse slices (an I x Jtot order-2 object built with model_pass = true): one pass over the
// stored entries gives sum (x - m)^2 and sum m^2 with m = A(i,:) . W(j,:) (the model at the entry, the lane layout of
// sp_model_kernel), then *res = sum (x - m)^2 + max(0, sum(GA .* GC) - sum m^2), GA = A'A and GC = sum_k
// diag(c_k) B_k'B_k diag(c_k) (R x R, so that sum(GA .* GC) = ||A diag(c_k) B_k'||^2 summed over k).  Allocation-free, fixed
// summation order.
int sparse_par2_residual(SparseTensor& s, const double* A, long long ldA, const double* W, long long ldW, const double* GA,
                         const double* GC, double* res, cudaStream_t st);

// nvecs of a sparse mode (aoadmm_nvecs_sparse): U = X_(n) of mode position n with its columns compressed to the distinct
// fibers (the other-mode subscripts that occur), so that Y V = X_(n) X_(n)' V = U (U' V) without forming Y.  Built per
// call from the resident mode-n copy (stable LSD radix passes over the other modes put the nonzeros in fiber order) and
// freed by the destructor; the object's MTTKRP scratch is never touched.  The build depends only on the multiset of
// entries.  With several GPUs, every fiber of a position before the last lies on one GPU: apply() gives this GPU's
// share of W, the caller sums the shares.
class FiberUnfolding {
 public:
  FiberUnfolding(const SparseTensor& s, int n, cudaStream_t st);
  ~FiberUnfolding();
  FiberUnfolding(const FiberUnfolding&) = delete;
  FiberUnfolding& operator=(const FiberUnfolding&) = delete;
  long long fibers() const { return nfib_; }
  // widest column chunk c = min(cols, 64), halved until T (fibers x c), the carries (2 units x c) and the row-major
  // V / W chunk (rows x c) fit in `budget` bytes; 0 when one column does not fit
  int chunk_columns(int cols, size_t budget) const;
  // allocates the buffers of c-column chunks
  void reserve(int c);
  // W (rows x cols, column-major, ld = rows) = U U' V (V likewise) over this GPU's nonzeros, c columns at a time: pass A
  // T = U' V in fiber order, pass B W = U T in the mode-n copy, both the deterministic unit / carry sums of the MTTKRP
  // with one gathered operand.  Every column of W is one lane's fixed-order sum plus a fixed-order fix-up, so its bits
  // do not depend on c.  Returns the launches.
  int apply(const double* V, double* W, int cols, cudaStream_t st);

 private:
  template <typename T>
  T* alloc(size_t count);
  const SparseTensor& s_;
  int n_ = 0, c_ = 0;
  long long rows_ = 0, nnz_ = 0, nfib_ = 0, units_ = 0;
  std::vector<void*> bufs_;
  int* in_ = nullptr;           // fiber order: i_n of every nonzero
  double* vals_ = nullptr;      // fiber order: value of every nonzero
  long long* fptr_ = nullptr;   // fibers + 1: first nonzero of every fiber
  int *fchunk_ = nullptr, *fhead_ = nullptr, *ftail_ = nullptr;   // unit metadata of the fiber order
  int* fib_ = nullptr;          // mode-n order: fiber id of every nonzero
  double *T_ = nullptr, *head_ = nullptr, *tail_ = nullptr, *X_ = nullptr;   // chunk buffers (reserve)
};

}  // namespace aoadmm
