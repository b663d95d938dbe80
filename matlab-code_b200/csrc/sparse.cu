// sparse.cu - sparse (COO) CP objects: preprocessing (CUB radix sorts, duplicate merge), deterministic sparse MTTKRP
// and ||X||_F^2.  Layout and scheme: sparse.cuh.
#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <utility>

#include "sparse.cuh"

namespace aoadmm {
namespace {

constexpr int kNormBlocks = 512;

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

__global__ void gather_keys_kernel(const int* __restrict__ src, const int* __restrict__ perm, unsigned* __restrict__ keys,
                                   long long n) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    keys[e] = (unsigned)src[perm[e]];
}

// sorted copy of the caller's nonzeros: ss(d, e) = raw(d, perm[e]), sv(e) = rv(perm[e])
__global__ void gather_coo_kernel(const int* __restrict__ raw, const double* __restrict__ rv, const int* __restrict__ perm,
                                  long long n, int order, int* __restrict__ ss, double* __restrict__ sv) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const long long src = perm[e];
    for (int d = 0; d < order; ++d) ss[d * n + e] = raw[d * n + src];
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

int transpose_scale(const double* in, long long rows, long long cols, long long ldi, double* out, long long ldo, double scale,
                    cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return 0;
  const long long tiles = ceil_div(rows, 32) * ceil_div(cols, 32);
  transpose_scale_kernel<<<(unsigned)std::min<long long>(tiles, 148LL * 16), 256, 0, st>>>(in, rows, cols, ldi, out, ldo, scale);
  AO_CHECK_LAUNCH();
  return 1;
}

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
};

// One group of G lanes per unit; lane j of a group owns columns j, j+G, ... (CPL of them).  The row sums run in the
// sorted nonzero order, so every value depends on the data and kSparseChunk only.
template <int G, int CPL>
__global__ void __launch_bounds__(256) sp_mttkrp_kernel(const SpArgs a) {
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
      const double v = __ldg(a.vals + e);
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

// rows split over units: tail carry of the unit where the row starts + head carries of the following units, in a fixed
// order (four interleaved partial sums, combined pairwise)
template <int G, int CPL>
__global__ void __launch_bounds__(256) sp_fixup_kernel(const SpArgs a) {
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
void launch_sp(const SpArgs& a, cudaStream_t st) {
  const long long threads = a.units * G;
  const unsigned blocks = (unsigned)ceil_div(threads, 256);
  sp_mttkrp_kernel<G, CPL><<<blocks, 256, 0, st>>>(a);
  AO_CHECK_LAUNCH();
  sp_fixup_kernel<G, CPL><<<blocks, 256, 0, st>>>(a);
  AO_CHECK_LAUNCH();
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

}  // namespace

void sparse_build(SparseTensor& s, int order, const long long* dims, int R, long long nnz, const long long* subs,
                  const double* vals, cudaStream_t st) {
  if (order < 2 || order > 8) throw CudaError(1, "sparse object: order must be in 2..8");
  if (nnz < 0) throw CudaError(1, "sparse object: negative nnz");
  if (nnz > 0x7fffffffLL - kSparseChunk) throw CudaError(2, "sparse object: more than 2^31 - 257 nonzeros");
  s.order = order;
  s.R = R;
  for (int d = 0; d < order; ++d) {
    if (dims[d] < 0 || dims[d] > 0x7fffffffLL) throw CudaError(1, "sparse object: a mode exceeds 2^31 - 1 rows");
    s.dims[d] = dims[d];
  }
  Temps tmp;   // temporaries of the preprocessing: released on every exit path
  const long long n = nnz;
  long long nm = 0;
  int* ms = nullptr;
  double* mv = nullptr;
  unsigned *k0 = nullptr, *k1 = nullptr;
  int *p0 = nullptr, *p1 = nullptr;
  void* sort_tmp = nullptr;
  size_t sort_bytes = 0;
  if (n > 0) {
    std::vector<int> h((size_t)order * n);
    for (size_t i = 0; i < h.size(); ++i) h[i] = (int)subs[i];
    int* raw = tmp.get<int>((size_t)order * n);
    double* rv = tmp.get<double>(n);
    AO_CUDA(cudaMemcpyAsync(raw, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    AO_CUDA(cudaMemcpyAsync(rv, vals, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
    AO_CUDA(cudaStreamSynchronize(st));
    k0 = tmp.get<unsigned>(n);
    k1 = tmp.get<unsigned>(n);
    p0 = tmp.get<int>(n);
    p1 = tmp.get<int>(n);
    AO_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, k0, k1, p0, p1, (int)n, 0, 32, st));
    size_t scan_bytes = 0;
    AO_CUDA(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (int*)k0, (int*)k1, (int)n, st));
    sort_bytes = std::max(sort_bytes, scan_bytes);
    sort_tmp = tmp.get<char>(sort_bytes);
    // full lexicographic order (mode 0 major): stable LSD passes from the last mode to the first
    iota_kernel<<<grid_for(n), 256, 0, st>>>(p0, n);
    AO_CHECK_LAUNCH();
    for (int d = order - 1; d >= 0; --d) {
      gather_keys_kernel<<<grid_for(n), 256, 0, st>>>(raw + (size_t)d * n, p0, k0, n);
      AO_CHECK_LAUNCH();
      size_t b = sort_bytes;
      AO_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp, b, k0, k1, p0, p1, (int)n, 0, key_bits(dims[d]), st));
      std::swap(p0, p1);
    }
    int* ss = tmp.get<int>((size_t)order * n);
    double* sv = tmp.get<double>(n);
    gather_coo_kernel<<<grid_for(n), 256, 0, st>>>(raw, rv, p0, n, order, ss, sv);
    AO_CHECK_LAUNCH();
    // merge duplicates (the Tensor Toolbox sptensor(subs,vals) constructor sums them)
    int* flags = (int*)k0;
    int* pos = (int*)k1;
    head_flags_kernel<<<grid_for(n), 256, 0, st>>>(ss, order, n, flags);
    AO_CHECK_LAUNCH();
    size_t b = sort_bytes;
    AO_CUDA(cub::DeviceScan::InclusiveSum(sort_tmp, b, flags, pos, (int)n, st));
    int last = 0;
    AO_CUDA(cudaMemcpyAsync(&last, pos + n - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    AO_CUDA(cudaStreamSynchronize(st));
    nm = last;
    ms = tmp.get<int>((size_t)order * nm);
    mv = tmp.get<double>(nm);
    merge_kernel<<<grid_for(n), 256, 0, st>>>(ss, sv, flags, pos, n, order, ms, mv, nm);
    AO_CHECK_LAUNCH();
  }
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
    if (nm == 0) {
      AO_CUDA(cudaMemsetAsync(sm.rowptr, 0, (rows + 1) * sizeof(long long), st));
      continue;
    }
    // the merged set is in full order with mode 0 major; a stable sort on i_m alone gives the order with i_m major and
    // the other modes ascending
    const unsigned* keys = (const unsigned*)(ms + (size_t)m * nm);
    const int* perm = nullptr;
    if (m > 0) {
      iota_kernel<<<grid_for(nm), 256, 0, st>>>(p0, nm);
      AO_CHECK_LAUNCH();
      size_t b = sort_bytes;
      AO_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp, b, keys, k1, p0, p1, (int)nm, 0, key_bits(rows), st));
      keys = k1;
      perm = p1;
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
  AO_CUDA(cudaStreamSynchronize(st));
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
  }
  s.modes.clear();
  for (auto& p : s.factT) f(p);
  f(s.outT);
  f(s.head);
  f(s.tail);
  f(s.norm_partials);
  f(s.norm_out);
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
                  long long ldout, cudaStream_t st) {
  const long long rows = s.dims[n];
  const int R = s.R;
  const SparseMode& sm = s.modes[n];
  int launches = 0;
  AO_CUDA(cudaMemsetAsync(s.outT, 0, (size_t)std::max<long long>(rows, 1) * R * sizeof(double), st));
  SpArgs a{};
  a.rowptr = sm.rowptr;
  a.chunk_row = sm.chunk_row;
  a.head_row = sm.head_row;
  a.tail_row = sm.tail_row;
  a.vals = sm.vals;
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
      launches += transpose_scale(fac[d], s.dims[d], R, ld[d], s.factT[d], R, 1.0, st);
      a.F[q++] = s.factT[d];
    }
    if (R <= 1) launch_sp<1, 1>(a, st);
    else if (R <= 2) launch_sp<2, 1>(a, st);
    else if (R <= 4) launch_sp<4, 1>(a, st);
    else if (R <= 8) launch_sp<8, 1>(a, st);
    else if (R <= 16) launch_sp<16, 1>(a, st);
    else if (R <= 32) launch_sp<32, 1>(a, st);
    else if (R <= 64) launch_sp<32, 2>(a, st);
    else if (R <= 128) launch_sp<32, 4>(a, st);
    else launch_sp<32, 8>(a, st);
    launches += 2;
  }
  // out(i, c) = scale * outT(c + R*i)
  launches += transpose_scale(s.outT, R, rows, R, out, ldout, scale, st);
  return launches;
}

}  // namespace aoadmm
