// sparse.cu - sparse (COO) CP objects: preprocessing (CUB radix sorts, duplicate merge), deterministic sparse MTTKRP
// and ||X||_F^2.  Layout and scheme: sparse.cuh.
#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <type_traits>
#include <utility>

#include "linalg.cuh"
#include "sparse.cuh"

namespace aoadmm {
namespace {

constexpr int kNormBlocks = 512;
constexpr int kTeleBlocks = 64;         // CTAs of the telescoped-norm reduction at most (2 partial sums each)

inline unsigned grid_for(long long n, int threads = 256) {
  return (unsigned)std::max<long long>(1, std::min<long long>(ceil_div(n, threads), 148LL * 32));
}

inline int key_bits(long long extent) {
  int b = 1;
  while (b < 32 && (1LL << b) < extent) ++b;
  return b;
}

__global__ void iota_kernel(int* p, long long n) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) p[e] = (int)e;
}

// shift: first index of this GPU's slab when src holds last-mode subscripts of a sharded object, else 0
__global__ void gather_keys_kernel(const int* __restrict__ src, const int* __restrict__ perm, unsigned* __restrict__ keys,
                                   long long n, int shift) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    keys[e] = (unsigned)(src[perm[e]] - shift);
}

// sorted copy of the caller's nonzeros: ss(d, e) = raw(d, perm[e]) (last mode: minus shift), sv(e) = rv(perm[e])
__global__ void gather_coo_kernel(const int* __restrict__ raw, const double* __restrict__ rv, const int* __restrict__ perm,
                                  long long n, int order, int shift, int* __restrict__ ss, double* __restrict__ sv) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const long long src = perm[e];
    for (int d = 0; d < order; ++d) ss[d * n + e] = raw[d * n + src] - (d == order - 1 ? shift : 0);
    sv[e] = rv[src];
  }
}

// flags[e] = 1 where nonzero e starts a run of equal subscripts (the input is fully sorted)
__global__ void head_flags_kernel(const int* __restrict__ ss, int order, long long n, int* __restrict__ flags) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    int f = (e == 0);
    for (int d = 0; d < order && !f; ++d) f = ss[d * n + e] != ss[d * n + e - 1];
    flags[e] = f;
  }
}

// duplicates summed in the (stable) sorted order
__global__ void merge_kernel(const int* __restrict__ ss, const double* __restrict__ sv, const int* __restrict__ flags,
                             const int* __restrict__ pos, long long n, int order, int* __restrict__ ms,
                             double* __restrict__ mv, long long nm) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    if (!flags[e]) continue;
    const long long t = pos[e] - 1;
    for (int d = 0; d < order; ++d) ms[d * nm + t] = ss[d * n + e];
    double v = sv[e];
    for (long long f = e + 1; f < n && !flags[f]; ++f) v += sv[f];
    mv[t] = v;
  }
}

// mode-n copy: values and the other modes' indices in the order given by perm (nullptr = identity)
__global__ void mode_copy_kernel(const int* __restrict__ ms, const double* __restrict__ mv, const int* __restrict__ perm,
                                 long long nm, int order, int n, double* __restrict__ vals, int* __restrict__ idx) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nm; e += (long long)gridDim.x * blockDim.x) {
    const long long src = perm ? perm[e] : e;
    vals[e] = mv[src];
    int q = 0;
    for (int d = 0; d < order; ++d) {
      if (d == n) continue;
      idx[q * nm + e] = ms[d * nm + src];
      ++q;
    }
  }
}

// rowptr[r] = first nonzero whose row is >= r (keys sorted ascending), r = 0..rows
__global__ void rowptr_kernel(const unsigned* __restrict__ keys, long long nm, long long rows, long long* __restrict__ rowptr) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r <= rows; r += (long long)gridDim.x * blockDim.x) {
    long long lo = 0, hi = nm;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if ((long long)keys[mid] < r) lo = mid + 1;
      else hi = mid;
    }
    rowptr[r] = lo;
  }
}

// per unit: row of its first nonzero; the row whose partial sum goes to the head / tail carry (-1: none)
__global__ void unit_rows_kernel(const unsigned* __restrict__ keys, const long long* __restrict__ rowptr, long long nm,
                                 long long units, int* __restrict__ chunk_row, int* __restrict__ head_row,
                                 int* __restrict__ tail_row) {
  for (long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x; u < units; u += (long long)gridDim.x * blockDim.x) {
    const long long s = u * kSparseChunk, e1 = (s + kSparseChunk < nm) ? s + kSparseChunk : nm;
    const int r0 = (int)keys[s], r1 = (int)keys[e1 - 1];
    chunk_row[u] = r0;
    const int h = rowptr[r0] < s ? r0 : -1;
    head_row[u] = h;
    tail_row[u] = (rowptr[r1 + 1] > e1 && h != r1) ? r1 : -1;
  }
}

// out(j + ldo*i) = scale * in(i + ldi*j), i < rows, j < cols; 32 x 32 tiles, grid-stride over tiles
__global__ void __launch_bounds__(256) transpose_scale_kernel(const double* __restrict__ in, long long rows, long long cols,
                                                              long long ldi, double* __restrict__ out, long long ldo,
                                                              double scale) {
  __shared__ double tile[32][33];
  const long long tr = (rows + 31) / 32, tc = (cols + 31) / 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (long long t = blockIdx.x; t < tr * tc; t += gridDim.x) {
    const long long i0 = (t % tr) * 32, j0 = (t / tr) * 32;
    for (int q = ty; q < 32; q += 8) {
      const long long i = i0 + tx, j = j0 + q;
      tile[q][tx] = (i < rows && j < cols) ? in[i + ldi * j] : 0.0;
    }
    __syncthreads();
    for (int q = ty; q < 32; q += 8) {
      const long long j = j0 + tx, i = i0 + q;
      if (i < rows && j < cols) out[j + ldo * i] = scale * tile[tx][q];
    }
    __syncthreads();
  }
}

}  // namespace

int transpose_scale(const double* in, long long rows, long long cols, long long ldi, double* out, long long ldo, double scale,
                    cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return 0;
  const long long tiles = ceil_div(rows, 32) * ceil_div(cols, 32);
  transpose_scale_kernel<<<(unsigned)std::min<long long>(tiles, 148LL * 16), 256, 0, st>>>(in, rows, cols, ldi, out, ldo, scale);
  AO_CHECK_LAUNCH();
  return 1;
}

namespace {

struct SpArgs {
  const long long* rowptr;
  const int* chunk_row;
  const int* head_row;
  const int* tail_row;
  const double* vals;
  const int* idx;
  long long nnz, units;
  int no, R;
  const double* F[7];   // row-major factors of the other modes, ascending position
  double* outT;
  double* head;
  double* tail;
  const int* perm;      // PERM instantiation: vals is read through perm (copy position -> canonical index)
};

// One group of G lanes per unit; lane j of a group owns columns j, j+G, ... (CPL of them).  The row sums run in the
// sorted nonzero order, so every value depends on the data and kSparseChunk only.
// PERM (imputed MTTKRP of a masked object, positions >= 2): the value of nonzero e is vals[perm[e]]; the unmasked
// instantiation (PERM = false) is the original kernel.
template <int G, int CPL, bool PERM>
__device__ __forceinline__ void sp_unit_rows(const SpArgs& a) {
  const long long unit = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
  const int gl = threadIdx.x % G;
  if (unit >= a.units) return;
  const long long s = unit * kSparseChunk, e_end = (s + kSparseChunk < a.nnz) ? s + kSparseChunk : a.nnz;
  const int R = a.R;
  long long r = a.chunk_row[unit];
  long long e = s;
  while (e < e_end) {
    const long long rb = a.rowptr[r], re = a.rowptr[r + 1];
    const long long stop = re < e_end ? re : e_end;
    double acc[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) acc[q] = 0.0;
#pragma unroll 2
    for (; e < stop; ++e) {
      const double v = PERM ? __ldg(a.vals + __ldg(a.perm + e)) : __ldg(a.vals + e);
      double p[CPL];
#pragma unroll
      for (int q = 0; q < CPL; ++q) p[q] = v;
      for (int m = 0; m < a.no; ++m) {
        const double* f = a.F[m] + (long long)__ldg(a.idx + m * a.nnz + e) * R;
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
          const int c = gl + G * q;
          if (c < R) p[q] *= __ldg(f + c);
        }
      }
#pragma unroll
      for (int q = 0; q < CPL; ++q) acc[q] += p[q];
    }
    double* dst = rb < s ? a.head + unit * R : (re > e_end ? a.tail + unit * R : a.outT + r * R);
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
      const int c = gl + G * q;
      if (c < R) dst[c] = acc[q];
    }
    ++r;
    while (e < e_end && a.rowptr[r + 1] <= e) ++r;   // skip empty rows
  }
}

template <int G, int CPL, bool PERM>
__global__ void __launch_bounds__(256) sp_mttkrp_kernel(const SpArgs a) {
  sp_unit_rows<G, CPL, PERM>(a);
}

// rows split over units: tail carry of the unit where the row starts + head carries of the following units, in a fixed
// order (four interleaved partial sums, combined pairwise)
template <int G, int CPL>
__device__ __forceinline__ void sp_fixup_rows(const SpArgs& a) {
  const long long unit = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G;
  const int gl = threadIdx.x % G;
  if (unit >= a.units) return;
  const int r = a.tail_row[unit];
  if (r < 0) return;
  const int R = a.R;
  const long long c1 = (a.rowptr[r + 1] - 1) / kSparseChunk;
#pragma unroll
  for (int q = 0; q < CPL; ++q) {
    const int col = gl + G * q;
    if (col >= R) continue;
    double s0 = a.tail[unit * R + col], s1 = 0.0, s2 = 0.0, s3 = 0.0;
    long long c = unit + 1;
    for (; c + 3 <= c1; c += 4) {
      s0 += a.head[c * R + col];
      s1 += a.head[(c + 1) * R + col];
      s2 += a.head[(c + 2) * R + col];
      s3 += a.head[(c + 3) * R + col];
    }
    for (; c <= c1; ++c) s0 += a.head[c * R + col];
    a.outT[(long long)r * R + col] = (s0 + s1) + (s2 + s3);
  }
}

template <int G, int CPL>
__global__ void __launch_bounds__(256) sp_fixup_kernel(const SpArgs a) {
  sp_fixup_rows<G, CPL>(a);
}

template <int G, int CPL, bool PERM>
void launch_sp(const SpArgs& a, cudaStream_t st) {
  const long long threads = a.units * G;
  const unsigned blocks = (unsigned)ceil_div(threads, 256);
  sp_mttkrp_kernel<G, CPL, PERM><<<blocks, 256, 0, st>>>(a);
  AO_CHECK_LAUNCH();
  sp_fixup_kernel<G, CPL><<<blocks, 256, 0, st>>>(a);
  AO_CHECK_LAUNCH();
}

// ---- EM imputation of masked sparse objects ----
struct ModelArgs {
  long long nnz;
  int no, R, impute;
  const int* row0;      // canonical order: position-1 subscripts
  const int* idx;       // canonical order: (order-1) x nnz subscripts of positions 2..order
  const double* vals;   // s
  const double* F[8];   // row-major factors of every position
  double* m;            // model at the last imputation (in), m' (out, impute)
  double* r;            // s - m' (out, impute)
  double* part;         // 4 per CTA
};

// m'(e) = sum_c prod_d F_d(i_d, c): a group of G lanes walks one unit of kSparseChunk consecutive nonzeros (columns
// across lanes, a fixed xor tree across them; consecutive nonzeros share rows and index sectors, as in the MTTKRP).
// Every group runs kSparseChunk steps so that each shuffle has the whole warp.  Per CTA, in a fixed order:
// [0] sum s m', [1] sum m'^2, [2] sum (m' - m)^2, [3] sum m^2.
template <int G, int CPL>
__global__ void __launch_bounds__(256) sp_model_kernel(const ModelArgs a) {
  __shared__ double scratch[32];
  const int gl = threadIdx.x % G;
  const long long e0 = (((long long)blockIdx.x * blockDim.x + threadIdx.x) / G) * kSparseChunk;
  const int R = a.R;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int q0 = 0; q0 < kSparseChunk; ++q0) {
    const long long e = e0 + q0;
    const bool ok = e < a.nnz;
    const double t = model_at_entry<G, CPL>(a.F, a.row0, a.idx, a.nnz, a.no, R, e, gl, ok);
    if (ok && gl == 0) {
      const double s = __ldg(a.vals + e), mo = a.m[e], d = t - mo;
      s0 = fma(s, t, s0);
      s1 = fma(t, t, s1);
      s2 = fma(d, d, s2);
      s3 = fma(mo, mo, s3);
      if (a.impute) {
        a.m[e] = t;
        a.r[e] = s - t;
      }
    }
  }
  s0 = block_sum(s0, scratch);
  s1 = block_sum(s1, scratch);
  s2 = block_sum(s2, scratch);
  s3 = block_sum(s3, scratch);
  if (threadIdx.x == 0) {
    double* o = a.part + 4 * (long long)blockIdx.x;
    o[0] = s0;
    o[1] = s1;
    o[2] = s2;
    o[3] = s3;
  }
}

}  // namespace

long long model_blocks(long long nnz, int R) {
  long long b = 0;
  rank_dispatch(R, [&](auto g, auto) { b = ceil_div(ceil_div(nnz, kSparseChunk) * decltype(g)::value, 256); });
  return b;
}

namespace {

// S = [F | B | F - B] (rows x 3R, ld = rows); impute: B = F afterwards
__global__ void stack3_kernel(const double* __restrict__ F, long long ldf, double* __restrict__ B, long long rows, int R,
                              double* __restrict__ S, int impute) {
  const long long n = rows * R;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i % rows, c = i / rows;
    const double f = F[r + ldf * c], b = B[i];
    S[i] = f;
    S[i + n] = b;
    S[i + 2 * n] = f - b;
    if (impute) B[i] = f;
  }
}

// With G_d = [F_d | B_d | D_d]' [F_d | B_d | D_d], D_d = F_d - B_d (3R x 3R, blocks 0 = F, 1 = B, 2 = D):
//   ||[[F]] - [[B]]||^2 = sum_{k,l} <T_k, T_l>,  T_k = [[F_1..F_{k-1}, D_k, B_{k+1}..B_N]]  (telescoped difference)
//   ||[[B]]||^2 = sum(Hadamard of the B'B blocks)
// so that near convergence the difference is never formed from two nearly equal model norms.  Per CTA: [0], [1].
__global__ void __launch_bounds__(256) tele_partials_kernel(const double* __restrict__ g3, int order, int R,
                                                            double* __restrict__ part) {
  __shared__ double scratch[32];
  const int R3 = 3 * R, G9 = R3 * R3;   // (3 * 256)^2 * 8 < 2^31
  double acc = 0.0, mm = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < R * R; i += gridDim.x * blockDim.x) {
    const int r = i % R, c = i / R;
    double sk = 0.0;
#pragma unroll 1
    for (int k = 0; k < order; ++k)
#pragma unroll 1
      for (int l = 0; l < order; ++l) {
        double p = 1.0;
        const double* g = g3 + r + R3 * c;
#pragma unroll 1
        for (int d = 0; d < order; ++d, g += G9) {
          const int tk = d < k ? 0 : (d == k ? 2 : 1), tl = d < l ? 0 : (d == l ? 2 : 1);
          p *= __ldg(g + tk * R + R3 * tl * R);
        }
        sk += p;
      }
    acc += sk;
    double q = 1.0;
    for (int d = 0; d < order; ++d) q *= __ldg(g3 + d * G9 + (R + r) + R3 * (R + c));
    mm += q;
  }
  acc = block_sum(acc, scratch);
  mm = block_sum(mm, scratch);
  if (threadIdx.x == 0) {
    part[2 * blockIdx.x] = acc;
    part[2 * blockIdx.x + 1] = mm;
  }
}

// nonzero-side sums of this GPU's entries, from the per-CTA partials of sp_model_kernel (fixed order):
// nz[0] sum s m', [1] sum m'^2, [2] sum_W (m' - m)^2, [3] sum_W m^2
__global__ void em_nz_kernel(const double* __restrict__ mpart, unsigned nm, double* __restrict__ nz) {
  const double a0 = warp_sum_partials(mpart, nm, 4), a1 = warp_sum_partials(mpart + 1, nm, 4);
  const double a2 = warp_sum_partials(mpart + 2, nm, 4), a3 = warp_sum_partials(mpart + 3, nm, 4);
  if (threadIdx.x == 0) {
    nz[0] = a0;
    nz[1] = a1;
    nz[2] = a2;
    nz[3] = a3;
  }
}

// em_sums slots of the object: [0] ||M'-M||^2 - sum_W (m'-m)^2, [1] ||M||^2 - sum_W m^2 (both clamped at 0: they are
// sums of squares over the unobserved entries, a negative value is rounding), [2] sum s m', [3] sum m'^2, [4] 0.
// nz: the nonzero-side sums of the whole object (em_nz_kernel, summed over the GPUs); tpart: the telescoped terms.
__global__ void em_final_kernel(const double* __restrict__ nz, const double* __restrict__ tpart, unsigned nt,
                                double* __restrict__ sums) {
  const double t = warp_sum_partials(tpart, nt, 2), mm = warp_sum_partials(tpart + 1, nt, 2);
  if (threadIdx.x == 0) {
    const double num = t - nz[2], den = mm - nz[3];
    sums[0] = num > 0.0 ? num : 0.0;
    sums[1] = den > 0.0 ? den : 0.0;
    sums[2] = nz[0];
    sums[3] = nz[1];
    sums[4] = 0.0;
  }
}

// cg_d = leading R x R block of g3_d (= F_d' F_d = B_d' F_d right after B = F)
__global__ void cg_from_g3_kernel(const double* __restrict__ g3, int order, int R, double* __restrict__ cg) {
  const long long R3 = 3LL * R, RR = (long long)R * R, n = order * RR;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long d = i / RR, j = i % RR, r = j % R, c = j / R;
    cg[i] = g3[d * R3 * R3 + r + R3 * c];
  }
}

// H = Hadamard product of cg_k over k != n (ascending k)
__global__ void hadamard_others_kernel(const double* __restrict__ cg, int order, int n, int R, double* __restrict__ H) {
  const long long RR = (long long)R * R;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < RR; i += (long long)gridDim.x * blockDim.x) {
    double h = 1.0;
    for (int k = 0; k < order; ++k)
      if (k != n) h *= cg[k * RR + i];
    H[i] = h;
  }
}

__global__ void nonzero_flags_kernel(const double* __restrict__ v, long long n, int* __restrict__ flags) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    flags[e] = v[e] != 0.0;
}

// observed entries of the merged mask, in the same (full lexicographic) order
__global__ void compact_kernel(const int* __restrict__ ms, const int* __restrict__ flags, const int* __restrict__ pos,
                               long long n, int order, int* __restrict__ out, long long nout) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    if (!flags[e]) continue;
    const long long t = pos[e] - 1;
    for (int d = 0; d < order; ++d) out[d * nout + t] = ms[d * n + e];
  }
}

__global__ void differ_kernel(const int* __restrict__ a, const int* __restrict__ b, long long n, int* __restrict__ bad) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    if (a[e] != b[e]) atomicOr(bad, 1);
}

__global__ void __launch_bounds__(256) sq_partials_kernel(const double* __restrict__ v, long long n, double* __restrict__ part) {
  __shared__ double scratch[32];
  double s = 0.0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    s += v[e] * v[e];
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

__global__ void sq_final_kernel(const double* __restrict__ part, unsigned n, double* __restrict__ out) {
  const double s = warp_sum_partials(part, n, 1);
  if (threadIdx.x == 0) *out = s;
}

template <typename T>
T* dalloc(size_t count) {
  T* p = nullptr;
  AO_CUDA(cudaMalloc(&p, std::max<size_t>(count * sizeof(T), 256)));
  return p;
}

struct Temps {
  std::vector<void*> p;
  ~Temps() {
    for (void* q : p) cudaFree(q);
  }
  template <typename T>
  T* get(size_t count) {
    T* q = dalloc<T>(count);
    p.push_back(q);
    return q;
  }
};

// radix-sort scratch shared by the merge and the per-mode sorts of one COO set
struct SortWs {
  unsigned *k0 = nullptr, *k1 = nullptr;
  int *p0 = nullptr, *p1 = nullptr;
  void* tmp = nullptr;
  size_t bytes = 0;
};

// uploads n > 0 COO entries, sorts them into full lexicographic order (mode 0 major) and sums duplicates (the Tensor
// Toolbox sptensor(subs,vals) constructor sums them): ms (order x nm, column-major), mv (nm).  Returns nm.
// shift: subtracted from the last-mode subscripts on the device (first index of this GPU's slab; 0 = whole object)
long long sort_merge(Temps& tmp, SortWs& w, int order, const long long* dims, long long n, const long long* subs,
                     const double* vals, cudaStream_t st, int*& ms, double*& mv, int shift = 0) {
  std::vector<int> h((size_t)order * n);
  for (size_t i = 0; i < h.size(); ++i) h[i] = (int)subs[i];
  int* raw = tmp.get<int>((size_t)order * n);
  double* rv = tmp.get<double>(n);
  AO_CUDA(cudaMemcpyAsync(raw, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  AO_CUDA(cudaMemcpyAsync(rv, vals, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
  AO_CUDA(cudaStreamSynchronize(st));
  w.k0 = tmp.get<unsigned>(n);
  w.k1 = tmp.get<unsigned>(n);
  w.p0 = tmp.get<int>(n);
  w.p1 = tmp.get<int>(n);
  AO_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, w.bytes, w.k0, w.k1, w.p0, w.p1, (int)n, 0, 32, st));
  size_t scan_bytes = 0;
  AO_CUDA(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (int*)w.k0, (int*)w.k1, (int)n, st));
  w.bytes = std::max(w.bytes, scan_bytes);
  w.tmp = tmp.get<char>(w.bytes);
  // full lexicographic order (mode 0 major): stable LSD passes from the last mode to the first
  iota_kernel<<<grid_for(n), 256, 0, st>>>(w.p0, n);
  AO_CHECK_LAUNCH();
  for (int d = order - 1; d >= 0; --d) {
    gather_keys_kernel<<<grid_for(n), 256, 0, st>>>(raw + (size_t)d * n, w.p0, w.k0, n, d == order - 1 ? shift : 0);
    AO_CHECK_LAUNCH();
    size_t b = w.bytes;
    AO_CUDA(cub::DeviceRadixSort::SortPairs(w.tmp, b, w.k0, w.k1, w.p0, w.p1, (int)n, 0, key_bits(dims[d]), st));
    std::swap(w.p0, w.p1);
  }
  int* ss = tmp.get<int>((size_t)order * n);
  double* sv = tmp.get<double>(n);
  gather_coo_kernel<<<grid_for(n), 256, 0, st>>>(raw, rv, w.p0, n, order, shift, ss, sv);
  AO_CHECK_LAUNCH();
  int* flags = (int*)w.k0;
  int* pos = (int*)w.k1;
  head_flags_kernel<<<grid_for(n), 256, 0, st>>>(ss, order, n, flags);
  AO_CHECK_LAUNCH();
  size_t b = w.bytes;
  AO_CUDA(cub::DeviceScan::InclusiveSum(w.tmp, b, flags, pos, (int)n, st));
  int last = 0;
  AO_CUDA(cudaMemcpyAsync(&last, pos + n - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
  AO_CUDA(cudaStreamSynchronize(st));
  const long long nm = last;
  ms = tmp.get<int>((size_t)order * nm);
  mv = tmp.get<double>(nm);
  merge_kernel<<<grid_for(n), 256, 0, st>>>(ss, sv, flags, pos, n, order, ms, mv, nm);
  AO_CHECK_LAUNCH();
  return nm;
}

// true when the observed entries of the mask (merged value != 0) are exactly the merged subscripts ms (order x nm)
bool mask_matches(Temps& tmp, int order, const long long* dims, long long nm, const int* ms, long long mask_nnz,
                  const long long* mask_subs, const double* mask_vals, int shift, cudaStream_t st) {
  long long nobs = 0;
  int* obs = nullptr;
  if (mask_nnz > 0) {
    SortWs w;
    int* mms = nullptr;
    double* mmv = nullptr;
    const long long mm = sort_merge(tmp, w, order, dims, mask_nnz, mask_subs, mask_vals, st, mms, mmv, shift);
    int* flags = (int*)w.k0;
    int* pos = (int*)w.k1;
    nonzero_flags_kernel<<<grid_for(mm), 256, 0, st>>>(mmv, mm, flags);
    AO_CHECK_LAUNCH();
    size_t b = w.bytes;
    AO_CUDA(cub::DeviceScan::InclusiveSum(w.tmp, b, flags, pos, (int)mm, st));
    int last = 0;
    AO_CUDA(cudaMemcpyAsync(&last, pos + mm - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    AO_CUDA(cudaStreamSynchronize(st));
    nobs = last;
    obs = tmp.get<int>((size_t)order * nobs);
    compact_kernel<<<grid_for(mm), 256, 0, st>>>(mms, flags, pos, mm, order, obs, nobs);
    AO_CHECK_LAUNCH();
  }
  if (nobs != nm) return false;
  if (nm == 0) return true;
  int* bad = tmp.get<int>(1);
  AO_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), st));
  differ_kernel<<<grid_for((long long)order * nm), 256, 0, st>>>(ms, obs, (long long)order * nm, bad);
  AO_CHECK_LAUNCH();
  int hb = 0;
  AO_CUDA(cudaMemcpyAsync(&hb, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
  AO_CUDA(cudaStreamSynchronize(st));
  return hb == 0;
}

}  // namespace

void sparse_build(SparseTensor& s, int order, const long long* full_dims, long long shard_offset, long long shard_extent,
                  int R, long long nnz, const long long* subs, const double* vals, cudaStream_t st, bool masked,
                  long long mask_nnz, const long long* mask_subs, const double* mask_vals) {
  if (order < 2 || order > 8) throw CudaError(1, "sparse object: order must be in 2..8");
  if (nnz < 0) throw CudaError(1, "sparse object: negative nnz");
  if (nnz > 0x7fffffffLL - kSparseChunk) throw CudaError(2, "sparse object: more than 2^31 - 257 nonzeros on one GPU");
  if (masked && (mask_nnz < 0 || mask_nnz > 0x7fffffffLL - kSparseChunk))
    throw CudaError(1, "sparse object: mask nnz out of range");
  s.order = order;
  s.R = R;
  for (int d = 0; d < order; ++d) {
    if (full_dims[d] < 0 || full_dims[d] > 0x7fffffffLL) throw CudaError(1, "sparse object: a mode exceeds 2^31 - 1 rows");
    s.fdims[d] = full_dims[d];
    s.dims[d] = full_dims[d];
  }
  if (shard_offset < 0 || shard_extent < 0 || shard_offset + shard_extent > full_dims[order - 1])
    throw CudaError(1, "sparse object: invalid shard range");
  s.shift = shard_offset;
  s.dims[order - 1] = shard_extent;
  const long long* dims = s.dims;   // nonzero side: local extents
  Temps tmp;   // temporaries of the preprocessing: released on every exit path
  long long nm = 0;
  int* ms = nullptr;
  double* mv = nullptr;
  SortWs w;
  if (nnz > 0) nm = sort_merge(tmp, w, order, dims, nnz, subs, vals, st, ms, mv, (int)shard_offset);
  if (masked && !mask_matches(tmp, order, dims, nm, ms, mask_nnz, mask_subs, mask_vals, (int)shard_offset, st))
    throw CudaError(2, "the observed entries of the sparse mask (Z.miss) differ from the stored entries of the object "
                       "(a sparse mask must mark exactly the stored entries)");
  s.nnz = nm;
  const long long units = ceil_div(nm, kSparseChunk);
  long long max_rows = 1;
  s.modes.resize(order);
  for (int m = 0; m < order; ++m) {
    SparseMode& sm = s.modes[m];
    const long long rows = dims[m];
    max_rows = std::max(max_rows, rows);
    sm.rowptr = dalloc<long long>(rows + 1);
    sm.chunk_row = dalloc<int>(units);
    sm.head_row = dalloc<int>(units);
    sm.tail_row = dalloc<int>(units);
    sm.vals = dalloc<double>(nm);
    sm.idx = dalloc<int>((size_t)(order - 1) * nm);
    if (masked && m > 0) sm.perm = dalloc<int>(nm);
    if (nm == 0) {
      AO_CUDA(cudaMemsetAsync(sm.rowptr, 0, (rows + 1) * sizeof(long long), st));
      continue;
    }
    // the merged set is in full order with mode 0 major; a stable sort on i_m alone gives the order with i_m major and
    // the other modes ascending
    const unsigned* keys = (const unsigned*)(ms + (size_t)m * nm);
    const int* perm = nullptr;
    if (m > 0) {
      iota_kernel<<<grid_for(nm), 256, 0, st>>>(w.p0, nm);
      AO_CHECK_LAUNCH();
      size_t b = w.bytes;
      AO_CUDA(cub::DeviceRadixSort::SortPairs(w.tmp, b, keys, w.k1, w.p0, w.p1, (int)nm, 0, key_bits(rows), st));
      keys = w.k1;
      perm = w.p1;
      if (masked) AO_CUDA(cudaMemcpyAsync(sm.perm, perm, (size_t)nm * sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    mode_copy_kernel<<<grid_for(nm), 256, 0, st>>>(ms, mv, perm, nm, order, m, sm.vals, sm.idx);
    AO_CHECK_LAUNCH();
    rowptr_kernel<<<grid_for(rows + 1), 256, 0, st>>>(keys, nm, rows, sm.rowptr);
    AO_CHECK_LAUNCH();
    unit_rows_kernel<<<grid_for(units), 256, 0, st>>>(keys, sm.rowptr, nm, units, sm.chunk_row, sm.head_row, sm.tail_row);
    AO_CHECK_LAUNCH();
    AO_CUDA(cudaStreamSynchronize(st));   // k1 / p0 / p1 are reused by the next mode
  }
  for (int d = 0; d < order; ++d) s.factT[d] = dalloc<double>((size_t)dims[d] * R);
  s.outT = dalloc<double>((size_t)max_rows * R);
  s.head = dalloc<double>((size_t)units * R);
  s.tail = dalloc<double>((size_t)units * R);
  s.norm_partials = dalloc<double>(kNormBlocks);
  s.norm_out = dalloc<double>(1);
  if (masked) {
    // the factor side (B, cross-Grams, stacks and their Grams) has the full extents and is replicated on every GPU
    // EM state: m = 0, r = s, B = 0 ("the unobserved entries start at 0"), every buffer of sparse_em / the imputed MTTKRP
    s.masked = true;
    s.row0 = dalloc<int>(nm);
    s.mvals = dalloc<double>(nm);
    s.rvals = dalloc<double>(nm);
    if (nm > 0) {
      AO_CUDA(cudaMemcpyAsync(s.row0, ms, (size_t)nm * sizeof(int), cudaMemcpyDeviceToDevice, st));
      AO_CUDA(cudaMemsetAsync(s.mvals, 0, (size_t)nm * sizeof(double), st));
      AO_CUDA(cudaMemcpyAsync(s.rvals, s.modes[0].vals, (size_t)nm * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    const long long RR = (long long)R * R, R3 = 3LL * R;
    size_t ws = 1;
    long long max_full = 1;
    for (int d = 0; d < order; ++d) {
      const long long rows = full_dims[d];
      max_full = std::max(max_full, rows);
      s.B[d] = dalloc<double>((size_t)rows * R);
      AO_CUDA(cudaMemsetAsync(s.B[d], 0, (size_t)rows * R * sizeof(double), st));
      ws = std::max<size_t>(ws, (size_t)dgemm_splitk_count(R, R, rows) * RR);
      ws = std::max<size_t>(ws, (size_t)dgemm_splitk_count(R3, R3, rows) * R3 * R3);
    }
    s.cg = dalloc<double>((size_t)order * RR);
    AO_CUDA(cudaMemsetAsync(s.cg, 0, (size_t)order * RR * sizeof(double), st));
    s.H = dalloc<double>(RR);
    s.stack = dalloc<double>((size_t)max_full * R3);
    s.g3 = dalloc<double>((size_t)order * R3 * R3);
    s.gemm_ws = dalloc<double>(ws);
    s.em_partials = dalloc<double>(2 * kTeleBlocks + 4 * (size_t)model_blocks(nm, R));
    s.em_nz = dalloc<double>(4);
  }
  AO_CUDA(cudaStreamSynchronize(st));
}

long long coo_sort_merge(int order, const long long* dims, long long n, const long long* subs, const double* vals,
                         cudaStream_t st, int** subs_out, double** vals_out) {
  Temps tmp;
  SortWs w;
  int* ms = nullptr;
  double* mv = nullptr;
  const long long nm = sort_merge(tmp, w, order, dims, n, subs, vals, st, ms, mv);
  int* so = dalloc<int>((size_t)order * nm);
  double* vo = nullptr;
  try {
    vo = dalloc<double>(nm);
    AO_CUDA(cudaMemcpyAsync(so, ms, (size_t)order * nm * sizeof(int), cudaMemcpyDeviceToDevice, st));
    AO_CUDA(cudaMemcpyAsync(vo, mv, (size_t)nm * sizeof(double), cudaMemcpyDeviceToDevice, st));
    AO_CUDA(cudaStreamSynchronize(st));
  } catch (...) {
    cudaFree(so);
    if (vo) cudaFree(vo);
    throw;
  }
  *subs_out = so;
  *vals_out = vo;
  return nm;
}

void sparse_free(SparseTensor& s) {
  auto f = [](auto*& p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  for (auto& m : s.modes) {
    f(m.rowptr);
    f(m.chunk_row);
    f(m.head_row);
    f(m.tail_row);
    f(m.vals);
    f(m.idx);
    f(m.perm);
  }
  s.modes.clear();
  for (auto& p : s.factT) f(p);
  f(s.outT);
  f(s.head);
  f(s.tail);
  f(s.norm_partials);
  f(s.norm_out);
  f(s.row0);
  f(s.mvals);
  f(s.rvals);
  for (auto& p : s.B) f(p);
  f(s.cg);
  f(s.H);
  f(s.stack);
  f(s.g3);
  f(s.gemm_ws);
  f(s.em_partials);
  f(s.em_nz);
}

int sparse_norm2(const SparseTensor& s, cudaStream_t st) {
  const double* v = s.order > 0 ? s.modes[0].vals : nullptr;
  sq_partials_kernel<<<kNormBlocks, 256, 0, st>>>(v, s.nnz, s.norm_partials);
  AO_CHECK_LAUNCH();
  sq_final_kernel<<<1, 32, 0, st>>>(s.norm_partials, kNormBlocks, s.norm_out);
  AO_CHECK_LAUNCH();
  return 2;
}

int sparse_mttkrp(SparseTensor& s, int n, const double* const* fac, const long long* ld, double scale, double* out,
                  long long ldout, cudaStream_t st, bool imputed) {
  const int last = s.order - 1;
  const long long rows = s.dims[n];
  const int R = s.R;
  const SparseMode& sm = s.modes[n];
  const bool imp = imputed && s.masked;
  int launches = 0;
  AO_CUDA(cudaMemsetAsync(s.outT, 0, (size_t)std::max<long long>(rows, 1) * R * sizeof(double), st));
  SpArgs a{};
  a.rowptr = sm.rowptr;
  a.chunk_row = sm.chunk_row;
  a.head_row = sm.head_row;
  a.tail_row = sm.tail_row;
  a.vals = imp ? s.rvals : sm.vals;   // imputed: the residual values, read through the copy -> canonical permutation
  a.perm = imp ? sm.perm : nullptr;   // (position 1 is the canonical order itself: perm == nullptr)
  a.idx = sm.idx;
  a.nnz = s.nnz;
  a.units = ceil_div(s.nnz, kSparseChunk);
  a.no = s.order - 1;
  a.R = R;
  a.outT = s.outT;
  a.head = s.head;
  a.tail = s.tail;
  if (a.units > 0) {
    int q = 0;
    for (int d = 0; d < s.order; ++d) {
      if (d == n) continue;
      launches += transpose_scale(fac[d] + (d == last ? s.shift : 0), s.dims[d], R, ld[d], s.factT[d], R, 1.0, st);
      a.F[q++] = s.factT[d];
    }
    rank_dispatch(R, [&](auto g, auto c) {
      if (a.perm != nullptr) launch_sp<decltype(g)::value, decltype(c)::value, true>(a, st);
      else launch_sp<decltype(g)::value, decltype(c)::value, false>(a, st);
    });
    launches += 2;
  }
  // out(i, c) = scale * outT(c + R*i), this GPU's rows of the last mode at their global position
  launches += transpose_scale(s.outT, R, rows, R, out + (n == last ? s.shift : 0), ldout, scale, st);
  return launches;
}

int sparse_lowrank_add(SparseTensor& s, int n, double scale, double* out, long long ldout, cudaStream_t st) {
  const long long rows = s.fdims[n];
  const int R = s.R;
  if (!s.masked || rows == 0) return 0;
  // low-rank term of the imputed tensor: out += scale * B_n * (Hadamard of B_k' F_k, k != n)
  const long long RR = (long long)R * R;
  hadamard_others_kernel<<<grid_for(RR), 256, 0, st>>>(s.cg, s.order, n, R, s.H);
  AO_CHECK_LAUNCH();
  return 1 + dgemm_small(0, 0, rows, R, R, scale, nullptr, s.B[n], rows, s.H, R, 1.0, out, ldout, st, nullptr);
}

int sparse_cross_gram(SparseTensor& s, int n, const double* F, long long ld, cudaStream_t st) {
  if (!s.masked || s.fdims[n] == 0) return 0;
  const int R = s.R;
  return dgemm_small_splitk(1, 0, R, R, s.fdims[n], 1.0, s.B[n], s.fdims[n], F, ld, 0.0, s.cg + (size_t)n * R * R, R,
                            s.gemm_ws, st, nullptr);
}

int sparse_em_nonzeros(SparseTensor& s, const double* const* fac, const long long* ld, bool impute, cudaStream_t st) {
  const int R = s.R;
  int launches = 0;
  // model at the nonzeros (canonical order), four fixed-order sums; impute: m = m', r = s - m'
  unsigned nbm = 0;
  if (s.nnz > 0) {
    ModelArgs a{};
    a.nnz = s.nnz;
    a.no = s.order - 1;
    a.R = R;
    a.impute = impute ? 1 : 0;
    a.row0 = s.row0;
    a.idx = s.modes[0].idx;
    a.vals = s.modes[0].vals;
    for (int d = 0; d < s.order; ++d) {
      launches += transpose_scale(fac[d] + (d == s.order - 1 ? s.shift : 0), s.dims[d], R, ld[d], s.factT[d], R, 1.0, st);
      a.F[d] = s.factT[d];
    }
    a.m = s.mvals;
    a.r = s.rvals;
    a.part = s.em_partials + 2 * kTeleBlocks;
    nbm = (unsigned)model_blocks(s.nnz, R);
    rank_dispatch(R, [&](auto g, auto c) { sp_model_kernel<decltype(g)::value, decltype(c)::value><<<nbm, 256, 0, st>>>(a); });
    AO_CHECK_LAUNCH();
    ++launches;
  }
  em_nz_kernel<<<1, 32, 0, st>>>(s.em_partials + 2 * kTeleBlocks, nbm, s.em_nz);
  AO_CHECK_LAUNCH();
  return launches + 1;
}

int sparse_em_finish(SparseTensor& s, const double* const* fac, const long long* ld, bool impute, double* sums,
                     cudaStream_t st) {
  const int R = s.R;
  int launches = 0;
  // Grams of [F_d | B_d | F_d - B_d] (impute: B_d = F_d afterwards), telescoped ||M' - M||^2 and ||M||^2
  const long long R3 = 3LL * R;
  for (int d = 0; d < s.order; ++d) {
    const long long rows = s.fdims[d];
    double* g = s.g3 + (size_t)d * R3 * R3;
    if (rows == 0) {
      AO_CUDA(cudaMemsetAsync(g, 0, (size_t)R3 * R3 * sizeof(double), st));
      continue;
    }
    stack3_kernel<<<grid_for(rows * R), 256, 0, st>>>(fac[d], ld[d], s.B[d], rows, R, s.stack, impute ? 1 : 0);
    AO_CHECK_LAUNCH();
    launches += 1 + dgemm_small_splitk(1, 0, R3, R3, rows, 1.0, s.stack, rows, s.stack, rows, 0.0, g, R3, s.gemm_ws, st, nullptr);
  }
  const unsigned nbt = (unsigned)std::min<long long>(ceil_div((long long)R * R, 256), kTeleBlocks);
  double* tpart = s.em_partials;
  tele_partials_kernel<<<nbt, 256, 0, st>>>(s.g3, s.order, R, tpart);
  AO_CHECK_LAUNCH();
  em_final_kernel<<<1, 32, 0, st>>>(s.em_nz, tpart, nbt, sums);
  AO_CHECK_LAUNCH();
  launches += 2;
  if (impute) {   // B = F: the cross-Grams B_d' F_d are the F_d' F_d blocks just computed
    cg_from_g3_kernel<<<grid_for((long long)s.order * R * R), 256, 0, st>>>(s.g3, s.order, R, s.cg);
    AO_CHECK_LAUNCH();
    ++launches;
  }
  return launches;
}


// ---- nvecs of a sparse mode: fiber-compressed unfolding and its two passes ----
namespace {

// row of nonzero e of a mode copy: the last r with rowptr[r] <= e
__device__ __forceinline__ int row_of(const long long* __restrict__ rowptr, long long rows, long long e) {
  long long lo = 0, hi = rows;   // rowptr[lo] <= e < rowptr[hi]
  while (hi - lo > 1) {
    const long long mid = (lo + hi) >> 1;
    if (rowptr[mid] <= e) lo = mid;
    else hi = mid;
  }
  return (int)lo;
}

// flags[k] = 1 where the k-th nonzero in fiber order starts a fiber (its other-mode subscripts differ from the previous)
__global__ void fiber_flags_kernel(const int* __restrict__ idx, int no, long long nnz, const int* __restrict__ perm,
                                   int* __restrict__ flags) {
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < nnz; k += (long long)gridDim.x * blockDim.x) {
    int f = (k == 0);
    if (!f) {
      const long long a = perm[k], b = perm[k - 1];
      for (int q = 0; q < no && !f; ++q) f = idx[q * nnz + a] != idx[q * nnz + b];
    }
    flags[k] = f;
  }
}

// fiber order: key (fiber id), i_n and value of every nonzero; mode-n order: its fiber id.  pos = inclusive scan of the
// fiber flags.
__global__ void fiber_scatter_kernel(const int* __restrict__ pos, const int* __restrict__ perm,
                                     const long long* __restrict__ rowptr, long long rows, const double* __restrict__ vals,
                                     long long nnz, unsigned* __restrict__ fkey, int* __restrict__ in,
                                     double* __restrict__ fvals, int* __restrict__ fib) {
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < nnz; k += (long long)gridDim.x * blockDim.x) {
    const int f = pos[k] - 1;
    const long long e = perm[k];
    fkey[k] = (unsigned)f;
    in[k] = row_of(rowptr, rows, e);
    fvals[k] = vals[e];
    fib[e] = f;
  }
}

// pass A (fiber order) and pass B (mode-n copy) of the nvecs operator: the MTTKRP unit / carry sums with one gathered
// operand, under names of their own
template <int G, int CPL>
__global__ void __launch_bounds__(256) nvecs_fiber_pass_kernel(const SpArgs a) {
  sp_unit_rows<G, CPL, false>(a);
}
template <int G, int CPL>
__global__ void __launch_bounds__(256) nvecs_fiber_fixup_kernel(const SpArgs a) {
  sp_fixup_rows<G, CPL>(a);
}
template <int G, int CPL>
__global__ void __launch_bounds__(256) nvecs_row_pass_kernel(const SpArgs a) {
  sp_unit_rows<G, CPL, false>(a);
}
template <int G, int CPL>
__global__ void __launch_bounds__(256) nvecs_row_fixup_kernel(const SpArgs a) {
  sp_fixup_rows<G, CPL>(a);
}

}  // namespace

template <typename T>
T* FiberUnfolding::alloc(size_t count) {
  T* p = dalloc<T>(count);
  bufs_.push_back(p);
  return p;
}

FiberUnfolding::FiberUnfolding(const SparseTensor& s, int n, cudaStream_t st) : s_(s), n_(n) {
  rows_ = s.dims[n];
  nnz_ = s.nnz;
  units_ = ceil_div(nnz_, kSparseChunk);
  if (nnz_ == 0) return;
  try {
    const SparseMode& sm = s.modes[n];
    const int no = s.order - 1;
    in_ = alloc<int>(nnz_);
    vals_ = alloc<double>(nnz_);
    fib_ = alloc<int>(nnz_);
    fchunk_ = alloc<int>(units_);
    fhead_ = alloc<int>(units_);
    ftail_ = alloc<int>(units_);
    Temps tmp;
    SortWs w;
    w.k0 = tmp.get<unsigned>(nnz_);
    w.k1 = tmp.get<unsigned>(nnz_);
    w.p0 = tmp.get<int>(nnz_);
    w.p1 = tmp.get<int>(nnz_);
    const int nm = (int)nnz_;
    AO_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, w.bytes, w.k0, w.k1, w.p0, w.p1, nm, 0, 32, st));
    size_t scan_bytes = 0;
    AO_CUDA(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (int*)w.k0, (int*)w.k1, nm, st));
    w.bytes = std::max(w.bytes, scan_bytes);
    w.tmp = tmp.get<char>(w.bytes);
    // fiber order: stable LSD passes from the last other mode to the first, starting from the mode-n order (so i_n
    // ascends inside a fiber)
    iota_kernel<<<grid_for(nnz_), 256, 0, st>>>(w.p0, nnz_);
    AO_CHECK_LAUNCH();
    for (int q = no - 1; q >= 0; --q) {
      const int d = q < n ? q : q + 1;
      gather_keys_kernel<<<grid_for(nnz_), 256, 0, st>>>(sm.idx + (size_t)q * nnz_, w.p0, w.k0, nnz_, 0);
      AO_CHECK_LAUNCH();
      size_t b = w.bytes;
      AO_CUDA(cub::DeviceRadixSort::SortPairs(w.tmp, b, w.k0, w.k1, w.p0, w.p1, nm, 0, key_bits(s.dims[d]), st));
      std::swap(w.p0, w.p1);
    }
    int* flags = (int*)w.k0;
    int* pos = (int*)w.k1;
    fiber_flags_kernel<<<grid_for(nnz_), 256, 0, st>>>(sm.idx, no, nnz_, w.p0, flags);
    AO_CHECK_LAUNCH();
    size_t b = w.bytes;
    AO_CUDA(cub::DeviceScan::InclusiveSum(w.tmp, b, flags, pos, nm, st));
    int last = 0;
    AO_CUDA(cudaMemcpyAsync(&last, pos + nnz_ - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    AO_CUDA(cudaStreamSynchronize(st));
    nfib_ = last;
    fptr_ = alloc<long long>(nfib_ + 1);
    unsigned* fkey = w.k0;   // the flags are consumed by the scan
    fiber_scatter_kernel<<<grid_for(nnz_), 256, 0, st>>>(pos, w.p0, sm.rowptr, rows_, sm.vals, nnz_, fkey, in_, vals_, fib_);
    AO_CHECK_LAUNCH();
    rowptr_kernel<<<grid_for(nfib_ + 1), 256, 0, st>>>(fkey, nnz_, nfib_, fptr_);
    AO_CHECK_LAUNCH();
    unit_rows_kernel<<<grid_for(units_), 256, 0, st>>>(fkey, fptr_, nnz_, units_, fchunk_, fhead_, ftail_);
    AO_CHECK_LAUNCH();
    AO_CUDA(cudaStreamSynchronize(st));   // the sort scratch is released on return
  } catch (...) {
    for (void* p : bufs_) cudaFree(p);
    throw;
  }
}

FiberUnfolding::~FiberUnfolding() {
  for (void* p : bufs_) cudaFree(p);
}

int FiberUnfolding::chunk_columns(int cols, size_t budget) const {
  for (int c = std::min(cols, 64); c >= 1; c /= 2) {
    const double bytes = 8.0 * c * ((double)nfib_ + 2.0 * (double)units_ + (double)rows_);
    if (bytes <= (double)budget) return c;
  }
  return 0;
}

void FiberUnfolding::reserve(int c) {
  c_ = c;
  T_ = alloc<double>((size_t)nfib_ * c);
  head_ = alloc<double>((size_t)units_ * c);
  tail_ = alloc<double>((size_t)units_ * c);
  X_ = alloc<double>((size_t)rows_ * c);
}

int FiberUnfolding::apply(const double* V, double* W, int cols, cudaStream_t st) {
  if (nnz_ == 0 || rows_ == 0) {
    if (rows_ > 0) AO_CUDA(cudaMemsetAsync(W, 0, (size_t)rows_ * cols * sizeof(double), st));
    return 0;
  }
  const SparseMode& sm = s_.modes[n_];
  SpArgs fa{};   // pass A: T(f, :) = sum over the nonzeros e of fiber f of x_e V(i_n(e), :)
  fa.rowptr = fptr_;
  fa.chunk_row = fchunk_;
  fa.head_row = fhead_;
  fa.tail_row = ftail_;
  fa.vals = vals_;
  fa.idx = in_;
  fa.nnz = nnz_;
  fa.units = units_;
  fa.no = 1;
  fa.F[0] = X_;
  fa.outT = T_;
  fa.head = head_;
  fa.tail = tail_;
  SpArgs ra = fa;   // pass B: W(i, :) = sum over the nonzeros e of row i of x_e T(fib(e), :)
  ra.rowptr = sm.rowptr;
  ra.chunk_row = sm.chunk_row;
  ra.head_row = sm.head_row;
  ra.tail_row = sm.tail_row;
  ra.vals = sm.vals;
  ra.idx = fib_;
  ra.F[0] = T_;
  ra.outT = X_;
  int launches = 0;
  for (int j0 = 0; j0 < cols; j0 += c_) {
    const int c = std::min(c_, cols - j0);
    fa.R = ra.R = c;
    launches += transpose_scale(V + (size_t)j0 * rows_, rows_, c, rows_, X_, c, 1.0, st);   // X = V chunk, row-major
    rank_dispatch(c, [&](auto g, auto cpl) {
      constexpr int G = decltype(g)::value, CPL = decltype(cpl)::value;
      const unsigned blocks = (unsigned)ceil_div(units_ * G, 256);
      nvecs_fiber_pass_kernel<G, CPL><<<blocks, 256, 0, st>>>(fa);
      AO_CHECK_LAUNCH();
      nvecs_fiber_fixup_kernel<G, CPL><<<blocks, 256, 0, st>>>(fa);
      AO_CHECK_LAUNCH();
      AO_CUDA(cudaMemsetAsync(X_, 0, (size_t)rows_ * c * sizeof(double), st));   // rows without nonzeros stay zero
      nvecs_row_pass_kernel<G, CPL><<<blocks, 256, 0, st>>>(ra);
      AO_CHECK_LAUNCH();
      nvecs_row_fixup_kernel<G, CPL><<<blocks, 256, 0, st>>>(ra);
      AO_CHECK_LAUNCH();
    });
    launches += 4;
    launches += transpose_scale(X_, c, rows_, c, W + (size_t)j0 * rows_, rows_, 1.0, st);   // W chunk, column-major
  }
  return launches;
}

}  // namespace aoadmm
