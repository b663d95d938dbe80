// heldout.cu - the model at given subscripts and the held-out error pass of a CP object.  Layout: heldout.cuh.
#include <algorithm>
#include <vector>

#include "heldout.cuh"

namespace aoadmm {
namespace {

inline unsigned grid_for(long long n) {
  return (unsigned)std::max<long long>(1, std::min<long long>(ceil_div(n, 256), 148LL * 32));
}

struct EntryArgs {
  long long n;
  int no, R;            // no = order - 1
  const int* subs;      // order x n, column-major
  const double* vals;   // error pass: the true values; nullptr: write the model to out
  const double* F[8];   // row-major factors of every position
  double* out;
  double* part;         // error pass: one partial sum per CTA
};

// A group of G lanes walks one unit of kSparseChunk consecutive entries (every group runs all kSparseChunk steps so
// that each shuffle has the whole warp).  Model mode: out[e] = m(e).  Error mode: lane 0 of the group accumulates
// (v - m)^2 in entry order, then one fixed-order block sum per CTA.
template <int G, int CPL>
__global__ void __launch_bounds__(256) heldout_kernel(const __grid_constant__ EntryArgs a) {
  __shared__ double scratch[32];
  const int gl = threadIdx.x % G;
  const long long e0 = (((long long)blockIdx.x * blockDim.x + threadIdx.x) / G) * kSparseChunk;
  double s = 0.0;
  for (int q0 = 0; q0 < kSparseChunk; ++q0) {
    const long long e = e0 + q0;
    const bool ok = e < a.n;
    const double t = model_at_entry<G, CPL>(a.F, a.subs, a.subs + a.n, a.n, a.no, a.R, e, gl, ok);
    if (ok && gl == 0) {
      if (a.vals != nullptr) {
        const double d = __ldg(a.vals + e) - t;
        s = fma(d, d, s);
      } else {
        a.out[e] = t;
      }
    }
  }
  if (a.vals == nullptr) return;   // uniform over the grid
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) a.part[blockIdx.x] = s;
}

__global__ void sum_partials_kernel(const double* __restrict__ part, unsigned n, double* __restrict__ out) {
  const double s = warp_sum_partials(part, n, 1);
  if (threadIdx.x == 0) *out = s;
}

void launch_entries(const EntryArgs& a, cudaStream_t st) {
  const unsigned nb = (unsigned)model_blocks(a.n, a.R);
  rank_dispatch(a.R, [&](auto g, auto c) { heldout_kernel<decltype(g)::value, decltype(c)::value><<<nb, 256, 0, st>>>(a); });
  AO_CHECK_LAUNCH();
}

// key of row i_1 = subs[e] in the mode-1 copy: lower bound of (i_2..i_N) among its stored entries.  The copy holds the
// slab [shift, shift + ext) of the last mode with local subscripts: only the entries of the slab are looked up.
__global__ void stored_kernel(const int* __restrict__ subs, long long n, int order, const long long* __restrict__ rowptr,
                              const int* __restrict__ idx, long long nnz, int shift, int ext,
                              unsigned long long* __restrict__ count, long long* __restrict__ first) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const int il = subs[(order - 1) * n + e] - shift;
    if (il < 0 || il >= ext) continue;
    const int i0 = subs[e];
    const long long end = rowptr[i0 + 1];
    long long lo = rowptr[i0], hi = end;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      int cmp = 0;
      for (int d = 1; d < order && cmp == 0; ++d) {
        const int a = idx[(d - 1) * nnz + mid], b = d == order - 1 ? il : subs[d * n + e];
        cmp = a < b ? -1 : (a > b ? 1 : 0);
      }
      if (cmp < 0) lo = mid + 1;
      else hi = mid;
    }
    bool eq = lo < end;
    for (int d = 1; d < order && eq; ++d) eq = idx[(d - 1) * nnz + lo] == (d == order - 1 ? il : subs[d * n + e]);
    if (eq) {
      atomicAdd(count, 1ULL);
      atomicMin(first, e);
    }
  }
}

struct DenseIdx {
  long long ld0, shard_offset;
  long long dims[8];   // local extents (the last one = this slab)
};

__global__ void masked_kernel(const int* __restrict__ subs, long long n, int order, const uint8_t* __restrict__ mask,
                              const __grid_constant__ DenseIdx di, unsigned long long* __restrict__ count,
                              long long* __restrict__ first) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    long long off = subs[e], stride = di.ld0;
    bool mine = true;
    for (int d = 1; d < order; ++d) {
      long long i = subs[d * n + e];
      if (d == order - 1) {
        i -= di.shard_offset;
        mine = i >= 0 && i < di.dims[d];
      }
      off += i * stride;
      stride *= di.dims[d];
    }
    if (mine && mask[off] != 0) {
      atomicAdd(count, 1ULL);
      atomicMin(first, e);
    }
  }
}

// count / first of a check kernel: res = {count, first} (device), launched by `launch`
template <typename F>
long long run_check(long long* first, cudaStream_t st, F&& launch) {
  void* res = nullptr;
  AO_CUDA(cudaMalloc(&res, 2 * sizeof(long long)));
  long long h[2] = {0, 0x7fffffffffffffffLL};
  try {
    AO_CUDA(cudaMemcpyAsync(res, h, sizeof(h), cudaMemcpyHostToDevice, st));
    launch((unsigned long long*)res, (long long*)res + 1);
    AO_CUDA(cudaMemcpyAsync(h, res, sizeof(h), cudaMemcpyDeviceToHost, st));
    AO_CUDA(cudaStreamSynchronize(st));
  } catch (...) {
    cudaFree(res);
    throw;
  }
  cudaFree(res);
  *first = h[0] > 0 ? h[1] : -1;
  return h[0];
}

// device buffers of one call, released on every exit path
struct DevTemps {
  std::vector<void*> p;
  ~DevTemps() {
    for (void* q : p) cudaFree(q);
  }
  template <typename T>
  T* get(size_t count) {
    void* q = nullptr;
    AO_CUDA(cudaMalloc(&q, std::max<size_t>(count * sizeof(T), 256)));
    p.push_back(q);
    return (T*)q;
  }
};

}  // namespace

void heldout_build(HeldOut& h, int order, const long long* dims, int R, long long n, const long long* subs,
                   const double* vals, cudaStream_t st) {
  h.order = order;
  h.R = R;
  for (int d = 0; d < order; ++d) h.dims[d] = dims[d];
  if (n > 0) h.n = coo_sort_merge(order, dims, n, subs, vals, st, &h.subs, &h.vals);
  for (int d = 0; d < order; ++d) AO_CUDA(cudaMalloc(&h.factT[d], std::max<size_t>((size_t)dims[d] * R * sizeof(double), 256)));
  AO_CUDA(cudaMalloc(&h.partials, std::max<size_t>((size_t)model_blocks(h.n, R) * sizeof(double), 256)));
}

void heldout_free(HeldOut& h) {
  auto f = [](auto*& p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  f(h.subs);
  f(h.vals);
  for (auto& p : h.factT) f(p);
  f(h.partials);
  h.n = 0;
}

int heldout_sse(HeldOut& h, const double* const* fac, const long long* ld, double* sse, cudaStream_t st) {
  int launches = 0;
  unsigned nb = 0;
  if (h.n > 0) {
    EntryArgs a{};
    a.n = h.n;
    a.no = h.order - 1;
    a.R = h.R;
    a.subs = h.subs;
    a.vals = h.vals;
    for (int d = 0; d < h.order; ++d) {
      launches += transpose_scale(fac[d], h.dims[d], h.R, ld[d], h.factT[d], h.R, 1.0, st);
      a.F[d] = h.factT[d];
    }
    a.part = h.partials;
    nb = (unsigned)model_blocks(h.n, h.R);
    launch_entries(a, st);
    ++launches;
  }
  sum_partials_kernel<<<1, 32, 0, st>>>(h.partials, nb, sse);
  AO_CHECK_LAUNCH();
  return launches + 1;
}

long long heldout_stored(const HeldOut& h, const SparseTensor& s, long long* first, cudaStream_t st) {
  *first = -1;
  if (h.n == 0 || s.nnz == 0) return 0;
  const SparseMode& m1 = s.modes[0];
  return run_check(first, st, [&](unsigned long long* count, long long* fst) {
    stored_kernel<<<grid_for(h.n), 256, 0, st>>>(h.subs, h.n, h.order, m1.rowptr, m1.idx, s.nnz, (int)s.shift,
                                                 (int)s.dims[h.order - 1], count, fst);
    AO_CHECK_LAUNCH();
  });
}

long long heldout_masked(const HeldOut& h, const uint8_t* mask, long long ld0, const long long* ldims,
                         long long shard_offset, long long* first, cudaStream_t st) {
  *first = -1;
  if (h.n == 0) return 0;
  DenseIdx di{};
  di.ld0 = ld0;
  di.shard_offset = shard_offset;
  for (int d = 0; d < h.order; ++d) di.dims[d] = ldims[d];
  return run_check(first, st, [&](unsigned long long* count, long long* fst) {
    masked_kernel<<<grid_for(h.n), 256, 0, st>>>(h.subs, h.n, h.order, mask, di, count, fst);
    AO_CHECK_LAUNCH();
  });
}

void heldout_subscript(const HeldOut& h, long long e, long long* out, cudaStream_t st) {
  for (int d = 0; d < h.order; ++d) {
    int v = 0;
    AO_CUDA(cudaMemcpyAsync(&v, h.subs + (size_t)d * h.n + e, sizeof(int), cudaMemcpyDeviceToHost, st));
    AO_CUDA(cudaStreamSynchronize(st));
    out[d] = v;
  }
}

void model_at_host(int order, int R, const double* const* fac, const long long* rows, long long n, const long long* subs,
                   double* out, cudaStream_t st) {
  if (n == 0) return;
  DevTemps tmp;
  std::vector<int> hs((size_t)order * n);
  for (size_t i = 0; i < hs.size(); ++i) hs[i] = (int)subs[i];
  EntryArgs a{};
  a.n = n;
  a.no = order - 1;
  a.R = R;
  int* ds = tmp.get<int>(hs.size());
  AO_CUDA(cudaMemcpyAsync(ds, hs.data(), hs.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  a.subs = ds;
  a.vals = nullptr;
  for (int d = 0; d < order; ++d) {
    double* f = tmp.get<double>((size_t)rows[d] * R);
    transpose_scale(fac[d], rows[d], R, rows[d], f, R, 1.0, st);
    a.F[d] = f;
  }
  a.out = tmp.get<double>(n);
  launch_entries(a, st);
  AO_CUDA(cudaMemcpyAsync(out, a.out, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
  AO_CUDA(cudaStreamSynchronize(st));
}

}  // namespace aoadmm
