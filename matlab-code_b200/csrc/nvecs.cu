// nvecs.cu - see nvecs.cuh
#include "nvecs.cuh"
#include "mttkrp.cuh"

#include <algorithm>
#include <cmath>
#include <numeric>
#include <vector>

namespace aoadmm {

namespace {

constexpr int kBK = 32;      // reduction depth of one pipeline stage
constexpr int kStages = 3;

// 16-byte asynchronous copy of two doubles; only the first `bytes` (0, 8 or 16) are read, the rest is zero-filled
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

struct GramArgs {
  UnfoldSpec s;
  long long nchunks, cps;   // reduction chunks in total / per split
  long long cpi;            // layout 1: chunks per batch entry = ceil(I / kBK)
  double* P;                // splits x n x n partial results (upper-triangle tiles only)
};

// shared-memory image of one operand tile:  layout 0: T[kk][a] (pitch BMT+4),  layout 1: T[a][kk] (pitch kBK+4).
// Both pitches are = 4 (mod 16) doubles, which makes the 64-bit DMMA fragment reads (8 rows x 4 k) conflict-free.
template <int L, int BMT>
struct TileGeom {
  static constexpr int pitch = (L == 0) ? BMT + 4 : kBK + 4;
  static constexpr int doubles = (L == 0) ? kBK * pitch : BMT * pitch;
};

template <int L, int BMT>
__device__ __forceinline__ void load_tile(const GramArgs& g, uint32_t dst, long long a0, long long chunk, int tid) {
  using G = TileGeom<L, BMT>;
  const UnfoldSpec& s = g.s;
  if (L == 0) {
    const long long c0 = chunk * kBK;
#pragma unroll 4
    for (int p = tid; p < (BMT / 2) * kBK; p += 256) {
      const int kk = p / (BMT / 2), a = 2 * (p % (BMT / 2));
      const long long left = s.n - (a0 + a);
      const int bytes = (c0 + kk < s.ncols && left > 0) ? (left > 1 ? 16 : 8) : 0;
      const double* src = bytes ? s.X + (a0 + a) + s.ld * (c0 + kk) : s.X;
      cp_async16(dst + (uint32_t)(kk * G::pitch + a) * 8u, src, bytes);
    }
  } else {
    const long long b = chunk / g.cpi, i0 = (chunk % g.cpi) * kBK;
#pragma unroll 4
    for (int p = tid; p < BMT * (kBK / 2); p += 256) {
      const int a = p / (kBK / 2), kk = 2 * (p % (kBK / 2));
      const long long left = s.I - (i0 + kk);
      const int bytes = (a0 + a < s.n && left > 0) ? (left > 1 ? 16 : 8) : 0;
      const double* src = bytes ? s.X + (i0 + kk) + s.cs * (a0 + a) + s.bs * b : s.X;
      cp_async16(dst + (uint32_t)(a * G::pitch + kk) * 8u, src, bytes);
    }
  }
}

// One CTA: the BMT x BMT tile (ta, tb), tb >= ta, of Y over the reduction chunks of split blockIdx.z.
// 8 warps as 2 (rows) x 4 (columns); warp tile (BMT/2) x (BMT/4) = MI x NI DMMA 8x8 blocks.
template <int L, int BMT>
__global__ void __launch_bounds__(256) unfold_gram_kernel(GramArgs g) {
  using G = TileGeom<L, BMT>;
  constexpr int MI = BMT / 16, NI = BMT / 32;
  const int ta = blockIdx.x, tb = blockIdx.y;
  if (tb < ta) return;
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wm = warp & 1, wn = warp >> 1;
  const bool diag = (ta == tb);
  const long long a0 = (long long)ta * BMT, b0 = (long long)tb * BMT;
  const long long c_begin = (long long)blockIdx.z * g.cps, c_end = min(g.nchunks, c_begin + g.cps);
  const uint32_t sbase = smem_u32(smem);
  auto stageA = [&](int st) { return sbase + (uint32_t)(st * 2 * G::doubles) * 8u; };
  auto stageB = [&](int st) { return sbase + (uint32_t)(st * 2 * G::doubles + (diag ? 0 : G::doubles)) * 8u; };

  double acc[MI][NI][2];
#pragma unroll
  for (int mi = 0; mi < MI; ++mi)
#pragma unroll
    for (int ni = 0; ni < NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

#pragma unroll
  for (int st = 0; st < kStages - 1; ++st) {
    if (c_begin + st < c_end) {
      load_tile<L, BMT>(g, stageA(st), a0, c_begin + st, tid);
      if (!diag) load_tile<L, BMT>(g, stageB(st), b0, c_begin + st, tid);
    }
    cp_async_commit();
  }
  const int gid = lane >> 2, tig = lane & 3;
  for (long long c = c_begin; c < c_end; ++c) {
    cp_async_wait<kStages - 2>();
    __syncthreads();
    {
      const long long cn = c + kStages - 1;
      if (cn < c_end) {
        const int st = (int)((cn - c_begin) % kStages);
        load_tile<L, BMT>(g, stageA(st), a0, cn, tid);
        if (!diag) load_tile<L, BMT>(g, stageB(st), b0, cn, tid);
      }
      cp_async_commit();
    }
    const int st = (int)((c - c_begin) % kStages);
    const uint32_t As = stageA(st), Bs = stageB(st);
#pragma unroll
    for (int k4 = 0; k4 < kBK / 4; ++k4) {
      double a[MI], b[NI];
#pragma unroll
      for (int mi = 0; mi < MI; ++mi) {
        const int row = wm * (BMT / 2) + mi * 8 + gid, k = k4 * 4 + tig;
        a[mi] = lds_f64(As + (uint32_t)(L == 0 ? k * G::pitch + row : row * G::pitch + k) * 8u);
      }
#pragma unroll
      for (int ni = 0; ni < NI; ++ni) {
        const int col = wn * (BMT / 4) + ni * 8 + gid, k = k4 * 4 + tig;
        b[ni] = lds_f64(Bs + (uint32_t)(L == 0 ? k * G::pitch + col : col * G::pitch + k) * 8u);
      }
#pragma unroll
      for (int mi = 0; mi < MI; ++mi)
#pragma unroll
        for (int ni = 0; ni < NI; ++ni) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
    }
  }
  cp_async_wait<0>();
  double* P = g.P + (long long)blockIdx.z * g.s.n * g.s.n;
#pragma unroll
  for (int mi = 0; mi < MI; ++mi)
#pragma unroll
    for (int ni = 0; ni < NI; ++ni) {
      const long long row = a0 + wm * (BMT / 2) + mi * 8 + gid;
      const long long col = b0 + wn * (BMT / 4) + ni * 8 + 2 * tig;
      if (row < g.s.n) {
        if (col < g.s.n) P[row + g.s.n * col] = acc[mi][ni][0];
        if (col + 1 < g.s.n) P[row + g.s.n * (col + 1)] = acc[mi][ni][1];
      }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Long modes (n > 256): the same 128 x 128 tiles, fed by TMA.  A producer warp (one elected lane) streams the two
// operand tiles of every 32-deep reduction chunk into a 3-stage ring of 128-byte-swizzled shared-memory tiles
// (cp.async.bulk.tensor, zero fill outside the object, completion on an mbarrier); the eight consumer warps (2 x 4,
// warp tile 64 x 32 = 8 x 4 DMMA blocks) never issue a copy or a CTA barrier - they wait on the stage's `full`
// barrier, read fragments and release the stage through its `empty` barrier, as the MTTKRP kernels do.
//   layout 0 (mode contiguous):   tile = 8 boxes of [32 reduction rows][16 a]  (box 16 x 32 of the n x ncols view)
//   layout 1 (reduction contiguous): tile = 2 boxes of [128 a][16 i]            (box 16 x 128 x 1 or 16 x 1 x 128)
// Fragment index maps (which 8 of a box's indices form one DMMA block) are those of mttkrp.cu: every 64-bit
// fragment load of a half-warp covers 16 distinct 8-byte slots of the swizzled rows.
// ---------------------------------------------------------------------------------------------------------
constexpr int kGT = 128;                         // tile edge
constexpr int kGStages = 3;
constexpr int kGTileBytes = kGT * kBK * 8;       // 32 KB per operand tile
constexpr int kGConsumers = 8;
constexpr int kGThreads = (kGConsumers + 1) * 32;
constexpr int kGSmem = kGStages * 2 * kGTileBytes + 2 * kGStages * 8 + 1024;

struct GramTmaArgs {
  long long n, nchunks, cps, cpi;
  int a_dim;      // layout 1: which map dimension (1 or 2) carries the mode index a
  double* P;
};

template <int L>
__global__ void __launch_bounds__(kGThreads, 1) unfold_gram_tma_kernel(const __grid_constant__ CUtensorMap tmap, GramTmaArgs g) {
  const int ta = blockIdx.x, tb = blockIdx.y;
  if (tb < ta) return;
  extern __shared__ uint8_t gsm_raw[];
  const uint32_t sbase = (smem_u32(gsm_raw) + 1023u) & ~1023u;
  const uint32_t sBar = sbase + kGStages * 2 * kGTileBytes;   // full[kGStages], empty[kGStages]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool diag = (ta == tb);
  const int a0 = ta * kGT, b0 = tb * kGT;
  const long long c_begin = (long long)blockIdx.z * g.cps, c_end = min(g.nchunks, c_begin + g.cps);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kGStages; ++s) {
      mbar_init(sBar + s * 8, 1);
      mbar_init(sBar + (kGStages + s) * 8, kGConsumers);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (warp == kGConsumers) {
    if (lane == 0) {
      prefetch_tensormap(&tmap);
      for (long long c = c_begin; c < c_end; ++c) {
        const long long cl = c - c_begin;
        const int s = (int)(cl % kGStages);
        const uint32_t ph = (uint32_t)((cl / kGStages) & 1);
        mbar_wait(sBar + (kGStages + s) * 8, ph ^ 1u);
        const uint32_t full = sBar + s * 8;
        const uint32_t sA = sbase + s * 2 * kGTileBytes, sB = sA + kGTileBytes;
        mbar_expect_tx(full, diag ? kGTileBytes : 2 * kGTileBytes);
        if (L == 0) {
          const int c0 = (int)(c * kBK);
#pragma unroll
          for (int b = 0; b < 8; ++b) tma_load_3d(sA + b * 4096, &tmap, a0 + 16 * b, c0, 0, full);
          if (!diag) {
#pragma unroll
            for (int b = 0; b < 8; ++b) tma_load_3d(sB + b * 4096, &tmap, b0 + 16 * b, c0, 0, full);
          }
        } else {
          const int bidx = (int)(c / g.cpi), i0 = (int)((c % g.cpi) * kBK);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (g.a_dim == 1) tma_load_3d(sA + h * 16384, &tmap, i0 + 16 * h, a0, bidx, full);
            else tma_load_3d(sA + h * 16384, &tmap, i0 + 16 * h, bidx, a0, full);
          }
          if (!diag) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              if (g.a_dim == 1) tma_load_3d(sB + h * 16384, &tmap, i0 + 16 * h, b0, bidx, full);
              else tma_load_3d(sB + h * 16384, &tmap, i0 + 16 * h, bidx, b0, full);
            }
          }
        }
      }
    }
    return;
  }

  // ===== consumers: 2 (rows) x 4 (columns) warps =====
  const int wm = warp & 1, wn = warp >> 1;
  const int m = lane >> 2, kk = lane & 3;
  double acc[8][4][2];
#pragma unroll
  for (int mi = 0; mi < 8; ++mi)
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

  // per-fragment byte offsets inside an operand tile (without the k4-step part)
  uint32_t aoff[8], axr[8], boff[4], bxr[4];
  if (L == 0) {
    const int cbase = ((m >> 1) & 1) * 4 + (m >> 2), off = m & 1;
#pragma unroll
    for (int mi = 0; mi < 8; ++mi) {
      aoff[mi] = (uint32_t)((4 * wm + (mi >> 1)) * 4096 + kk * 128 + off * 8);
      axr[mi] = (uint32_t)(((cbase + 2 * (mi & 1)) ^ kk) << 4);
    }
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) {
      boff[ni] = (uint32_t)((2 * wn + (ni >> 1)) * 4096 + kk * 128 + off * 8);
      bxr[ni] = (uint32_t)(((cbase + 2 * (ni & 1)) ^ kk) << 4);
    }
  } else {
#pragma unroll
    for (int mi = 0; mi < 8; ++mi) {
      const int row = 16 * (4 * wm + (mi >> 1)) + 2 * m + (mi & 1);
      aoff[mi] = (uint32_t)(row * 128 + (kk & 1) * 8);
      axr[mi] = (uint32_t)(row & 7);
    }
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) {
      const int row = 16 * (2 * wn + (ni >> 1)) + 2 * m + (ni & 1);
      boff[ni] = (uint32_t)(row * 128 + (kk & 1) * 8);
      bxr[ni] = (uint32_t)(row & 7);
    }
  }

  for (long long c = c_begin; c < c_end; ++c) {
    const long long cl = c - c_begin;
    const int s = (int)(cl % kGStages);
    const uint32_t ph = (uint32_t)((cl / kGStages) & 1);
    mbar_wait(sBar + s * 8, ph);
    const uint32_t sA = sbase + s * 2 * kGTileBytes, sB = diag ? sA : sA + kGTileBytes;
#pragma unroll
    for (int t = 0; t < kBK / 4; ++t) {
      double a[8], b[4];
      if (L == 0) {
        const uint32_t rowoff = (uint32_t)(t * 512), flip = (uint32_t)((t & 1) << 6);
#pragma unroll
        for (int mi = 0; mi < 8; ++mi) a[mi] = lds_f64(sA + aoff[mi] + rowoff + (axr[mi] ^ flip));
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = lds_f64(sB + boff[ni] + rowoff + (bxr[ni] ^ flip));
      } else {
        const uint32_t hoff = (uint32_t)((t >> 2) * 16384);
        const uint32_t chunk = (uint32_t)((t & 3) * 2 + (kk >> 1));
#pragma unroll
        for (int mi = 0; mi < 8; ++mi) a[mi] = lds_f64(sA + hoff + aoff[mi] + ((chunk ^ axr[mi]) << 4));
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = lds_f64(sB + hoff + boff[ni] + ((chunk ^ bxr[ni]) << 4));
      }
#pragma unroll
      for (int mi = 0; mi < 8; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) dmma884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(sBar + (kGStages + s) * 8);
  }

  double* P = g.P + (long long)blockIdx.z * g.n * g.n;
#pragma unroll
  for (int mi = 0; mi < 8; ++mi) {
    long long row;
    if (L == 0) {
      const int cbase = ((m >> 1) & 1) * 4 + (m >> 2);
      row = a0 + 16 * (4 * wm + (mi >> 1)) + 2 * (cbase + 2 * (mi & 1)) + (m & 1);
    } else {
      row = a0 + 16 * (4 * wm + (mi >> 1)) + 2 * m + (mi & 1);
    }
    if (row >= g.n) continue;
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int nn = 2 * kk + e;   // column index inside the DMMA block
        long long col;
        if (L == 0) {
          const int cb = ((nn >> 1) & 1) * 4 + (nn >> 2);
          col = b0 + 16 * (2 * wn + (ni >> 1)) + 2 * (cb + 2 * (ni & 1)) + (nn & 1);
        } else {
          col = b0 + 16 * (2 * wn + (ni >> 1)) + 2 * nn + (ni & 1);
        }
        if (col < g.n) P[row + g.n * col] = acc[mi][ni][e];
      }
  }
}

// Y(a,b) = Y(b,a) = sum over splits (fixed order) of the upper-triangle partials
__global__ void gram_reduce_mirror_kernel(const double* __restrict__ P, int splits, long long n, double* __restrict__ Y,
                                          int accumulate) {
  const long long nn = n * n;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < nn; idx += (long long)gridDim.x * blockDim.x) {
    const long long a = idx % n, b = idx / n;
    if (a > b) continue;
    double s = 0.0;
    for (int z = 0; z < splits; ++z) s += P[(long long)z * nn + idx];
    if (accumulate) s += Y[idx];   // Y stays exactly symmetric: both triangles receive the same sum
    Y[idx] = s;
    Y[b + n * a] = s;
  }
}

struct GramPlan {
  int bmt;
  long long T, nchunks, cpi, cps;
  int splits;
};

GramPlan plan_gram(const UnfoldSpec& s) {
  GramPlan p{};
  p.bmt = (s.n > 256) ? 128 : (s.n > 32 ? 64 : 32);
  p.T = ceil_div(s.n, p.bmt);
  if (s.layout == 0) {
    p.cpi = 0;
    p.nchunks = ceil_div(s.ncols, kBK);
  } else {
    p.cpi = ceil_div(s.I, kBK);
    p.nchunks = p.cpi * s.nb;
  }
  p.nchunks = std::max<long long>(p.nchunks, 1);
  const long long active = p.T * (p.T + 1) / 2;
  long long splits = std::max<long long>(1, ceil_div(2 * 148, active));
  const long long cap = std::max<long long>(1, (1LL << 28) / std::max<long long>(s.n * s.n, 1));  // <= 2 GB of partials
  if (p.bmt == 128) {
    // TMA kernel: one CTA per SM, so the pass lasts ceil(active * splits / 148) / splits tile-times.  Take the smallest
    // split count whose last wave is (nearly) as full as the best one's (n = 4096: 528 tiles -> 3.57 waves rounded up
    // to 4 with one split, 17.8 -> 18 with five).
    const long long smax = std::max<long long>(1, std::min<long long>({p.nchunks / 8, cap, 64LL}));
    double best = 0.0;
    for (long long q = 1; q <= smax; ++q) {
      const double w = (double)(active * q) / 148.0;
      best = std::max(best, w / std::ceil(w));
    }
    for (long long q = 1; q <= smax; ++q) {
      const double w = (double)(active * q) / 148.0;
      if (w / std::ceil(w) >= best - 0.01) {
        splits = q;
        break;
      }
    }
  }
  splits = std::min(splits, std::max<long long>(1, p.nchunks / 8));         // at least 8 chunks per split
  splits = std::min({splits, cap, (long long)65535});
  p.cps = ceil_div(p.nchunks, splits);
  p.splits = (int)ceil_div(p.nchunks, p.cps);
  return p;
}

template <int L, int BMT>
void launch_gram(const GramArgs& g, const GramPlan& p, cudaStream_t st) {
  const size_t smem = (size_t)kStages * 2 * TileGeom<L, BMT>::doubles * sizeof(double);
  ensure_dynamic_smem(reinterpret_cast<const void*>(unfold_gram_kernel<L, BMT>), smem, 0);
  dim3 grid((unsigned)p.T, (unsigned)p.T, (unsigned)p.splits);
  unfold_gram_kernel<L, BMT><<<grid, 256, smem, st>>>(g);
  AO_CHECK_LAUNCH();
}

// ---- small helpers of the eigen-solver ---------------------------------------------------------------------------
__global__ void fill_hash_kernel(double* __restrict__ V, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    unsigned long long z = (unsigned long long)i * 0x9E3779B97F4A7C15ull + 0x2545F4914F6CDD1Dull;   // splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    V[i] = (double)(z >> 11) * (1.0 / 9007199254740992.0) - 0.5;
  }
}

__global__ void symmetrize_kernel(double* __restrict__ H, int n) {
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n * n; idx += gridDim.x * blockDim.x) {
    const int a = idx % n, b = idx / n;
    if (a < b) {
      const double v = 0.5 * (H[a + n * b] + H[b + n * a]);
      H[a + n * b] = v;
      H[b + n * a] = v;
    }
  }
}

// V(:,j) = T(:,j) / sqrt(ev[j])   (0 when ev[j] is not a positive number: a direction outside the range of the block)
__global__ void scale_cols_rsqrt_kernel(double* __restrict__ V, const double* __restrict__ T, long long rows, int cols,
                                        const double* __restrict__ ev) {
  const long long n = rows * cols;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
    const double e = ev[idx / rows];
    V[idx] = (e > 0.0) ? T[idx] * rsqrt(e) : 0.0;
  }
}

// res[j] = || Z(:,j) - theta[j] * U(:,j) ||_2      (one CTA per column)
__global__ void __launch_bounds__(256) ritz_residual_kernel(const double* __restrict__ Z, const double* __restrict__ U,
                                                            const double* __restrict__ theta, long long rows,
                                                            double* __restrict__ res) {
  __shared__ double red[32];
  const int j = blockIdx.x;
  const double th = theta[j];
  double s = 0.0;
  for (long long i = threadIdx.x; i < rows; i += blockDim.x) {
    const double d = Z[i + rows * j] - th * U[i + rows * j];
    s = fma(d, d, s);
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) res[j] = sqrt(s);
}

// out(:,c) = sign * U(:, order[c]) with sign chosen so that the entry of largest magnitude (first one on ties) is positive
__global__ void __launch_bounds__(256) gather_signed_kernel(const double* __restrict__ U, long long rows,
                                                            const int* __restrict__ order, double* __restrict__ out) {
  __shared__ double bestv[256];
  __shared__ long long besti[256];
  const int c = blockIdx.x;
  const double* u = U + rows * order[c];
  double bv = -1.0;
  long long bi = 0;
  for (long long i = threadIdx.x; i < rows; i += blockDim.x) {
    const double a = fabs(u[i]);
    if (a > bv) {
      bv = a;
      bi = i;
    }
  }
  bestv[threadIdx.x] = bv;
  besti[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double v2 = bestv[threadIdx.x + o];
      const long long i2 = besti[threadIdx.x + o];
      if (v2 > bestv[threadIdx.x] || (v2 == bestv[threadIdx.x] && i2 < besti[threadIdx.x])) {
        bestv[threadIdx.x] = v2;
        besti[threadIdx.x] = i2;
      }
    }
    __syncthreads();
  }
  const double sg = (u[besti[0]] < 0.0) ? -1.0 : 1.0;
  for (long long i = threadIdx.x; i < rows; i += blockDim.x) out[i + rows * c] = sg * u[i];
}

inline unsigned blocks_for(long long n) { return (unsigned)std::min<long long>(std::max<long long>(ceil_div(n, 256), 1), 148 * 8); }

}  // namespace

size_t unfold_gram_workspace(const UnfoldSpec& s) {
  const GramPlan p = plan_gram(s);
  return (size_t)p.splits * (size_t)s.n * (size_t)s.n;
}

int unfold_gram(const UnfoldSpec& s, double* Y, double* work, cudaStream_t st, bool accumulate) {
  if (s.n <= 0) return 0;
  // the operand tiles are fetched in 16-byte pieces: base and all strides must keep pairs of doubles aligned
  if ((reinterpret_cast<uintptr_t>(s.X) & 15) != 0 || (s.layout == 0 ? (s.ld & 1) : ((s.cs | s.bs) & 1)) != 0)
    throw CudaError(1, "nvecs: object storage must be 16-byte aligned with an even leading dimension");
  const GramPlan p = plan_gram(s);
  GramArgs g{};
  g.s = s;
  g.nchunks = p.nchunks;
  g.cps = p.cps;
  g.cpi = std::max<long long>(p.cpi, 1);
  g.P = work;
  if (p.T > 65535) throw CudaError(2, "nvecs: mode too long for an explicit Gram matrix");
  if (p.bmt == 128) {
    // TMA-fed kernel: tensor map of the unfolding view
    CUtensorMap map;
    GramTmaArgs ga{};
    ga.n = s.n;
    ga.nchunks = p.nchunks;
    ga.cps = p.cps;
    ga.cpi = std::max<long long>(p.cpi, 1);
    ga.P = work;
    ga.a_dim = 1;
    dim3 grid((unsigned)p.T, (unsigned)p.T, (unsigned)p.splits);
    if (s.layout == 0) {
      const uint64_t dims[3] = {(uint64_t)s.n, (uint64_t)s.ncols, 1};
      const uint64_t str[2] = {(uint64_t)s.ld * 8, (uint64_t)s.ld * 8 * (uint64_t)s.ncols};
      const uint32_t box[3] = {16, 32, 1};
      encode_map3(&map, s.X, dims, str, box);
      ensure_dynamic_smem(reinterpret_cast<const void*>(unfold_gram_tma_kernel<0>), kGSmem, 0);
      unfold_gram_tma_kernel<0><<<grid, kGThreads, kGSmem, st>>>(map, ga);
    } else {
      // dimensions in storage order: the smaller stride first
      const bool a_first = (s.nb <= 1) || (s.cs <= s.bs);
      ga.a_dim = a_first ? 1 : 2;
      const uint64_t dims[3] = {(uint64_t)s.I, (uint64_t)(a_first ? s.n : s.nb), (uint64_t)(a_first ? std::max<long long>(s.nb, 1) : s.n)};
      const uint64_t str[2] = {(uint64_t)(a_first ? s.cs : s.bs) * 8, (uint64_t)(a_first ? std::max<long long>(s.bs, s.cs * s.n) : s.cs) * 8};
      const uint32_t box[3] = {16, a_first ? 128u : 1u, a_first ? 1u : 128u};
      encode_map3(&map, s.X, dims, str, box);
      ensure_dynamic_smem(reinterpret_cast<const void*>(unfold_gram_tma_kernel<1>), kGSmem, 0);
      unfold_gram_tma_kernel<1><<<grid, kGThreads, kGSmem, st>>>(map, ga);
    }
    AO_CHECK_LAUNCH();
  } else if (s.layout == 0) {
    if (p.bmt == 128) launch_gram<0, 128>(g, p, st);
    else if (p.bmt == 64) launch_gram<0, 64>(g, p, st);
    else launch_gram<0, 32>(g, p, st);
  } else {
    if (p.bmt == 128) launch_gram<1, 128>(g, p, st);
    else if (p.bmt == 64) launch_gram<1, 64>(g, p, st);
    else launch_gram<1, 32>(g, p, st);
  }
  gram_reduce_mirror_kernel<<<blocks_for(s.n * s.n), 256, 0, st>>>(work, p.splits, s.n, Y, accumulate ? 1 : 0);
  AO_CHECK_LAUNCH();
  return 2;
}

int eig_block(long long n, int r) {
  // short modes: the block is the whole space, one Rayleigh-Ritz step (a Jacobi eigen-decomposition of Y) is exact
  return (n <= 128) ? (int)n : (int)std::min<long long>(n, (long long)r + std::max(8, r / 4));
}

EigInfo top_eigvecs(const double* Y, long long n, int r, double* U, double* theta, cudaStream_t st) {
  const EigOperator apply = [&](const double* V, double* W, int Rb) {
    return dgemm_small(0, 0, n, Rb, n, 1.0, nullptr, Y, n, V, n, 0.0, W, n, st, nullptr);
  };
  return top_eigvecs(apply, n, r, U, theta, st);
}

EigInfo top_eigvecs(const EigOperator& apply, long long n, int r, double* U, double* theta, cudaStream_t st) {
  EigInfo info;
  if (r < 1 || r > n) throw CudaError(1, "nvecs: the number of vectors must be between 1 and the mode size");
  const int Rb = eig_block(n, r);
  const size_t nb = (size_t)n * Rb, bb = (size_t)Rb * Rb;
  double* buf = nullptr;
  int* order_dev = nullptr;
  const size_t wsd = (size_t)dgemm_splitk_count(Rb, Rb, n) * bb;   // split-K partials of the block x block products
  AO_CUDA(cudaMalloc(&buf, (4 * nb + 3 * bb + 3 * (size_t)Rb + wsd) * sizeof(double)));
  AO_CUDA(cudaMalloc(&order_dev, sizeof(int) * (size_t)r));
  double *V = buf, *W = V + nb, *Z = W + nb, *Ur = Z + nb, *H = Ur + nb, *Q = H + bb, *G = Q + bb, *sig = G + bb,
         *ev = sig + Rb, *res = ev + Rb, *ws = res + Rb;
  std::vector<double> h_sig(Rb), h_res(Rb);
  std::vector<int> order(Rb);
  int L = 0;
  try {
    // orthonormalise the columns of `src` (n x Rb) into V: Gram matrix, Jacobi eigen-decomposition, rotate, scale.
    // Done twice: the first pass may leave rounding-noise directions when the block is rank deficient.
    auto orthonormalise = [&](double* src) {
      for (int pass = 0; pass < 2; ++pass) {
        const double* in = (pass == 0) ? src : V;
        L += dgemm_small_splitk(1, 0, Rb, Rb, n, 1.0, in, n, in, n, 0.0, G, Rb, ws, st, nullptr);
        symmetrize_kernel<<<blocks_for((long long)bb), 256, 0, st>>>(G, Rb);
        L += 1 + jacobi_onesided(G, Rb, Rb, Q, ev, st);
        L += dgemm_small(0, 0, n, Rb, Rb, 1.0, nullptr, in, n, Q, Rb, 0.0, W, n, st, nullptr);
        scale_cols_rsqrt_kernel<<<blocks_for((long long)nb), 256, 0, st>>>(V, W, n, Rb, ev);
        AO_CHECK_LAUNCH();
        ++L;
      }
    };
    fill_hash_kernel<<<blocks_for((long long)nb), 256, 0, st>>>(Z, (long long)nb);
    AO_CHECK_LAUNCH();
    ++L;
    orthonormalise(Z);
    // Eigenvector error = residual / gap, so the iteration runs down to the rounding floor of the residual (about
    // eps*sqrt(n)*theta_1), detected as "no new minimum (by 5 %) within the last 6 iterations".
    const double tol = 4.0 * 2.220446049250313e-16;
    double best = 1e300;
    int since_best = 0;
    const int maxit = 3000;
    for (int it = 1; it <= maxit; ++it) {
      info.iterations = it;
      L += apply(V, W, Rb);                                                                       // W = Y V
      L += dgemm_small_splitk(1, 0, Rb, Rb, n, 1.0, V, n, W, n, 0.0, H, Rb, ws, st, nullptr);    // H = V' Y V
      symmetrize_kernel<<<blocks_for((long long)bb), 256, 0, st>>>(H, Rb);
      L += 1 + jacobi_onesided(H, Rb, Rb, Q, sig, st);                                           // H = Q diag(sig) Q'
      L += dgemm_small(0, 0, n, Rb, Rb, 1.0, nullptr, W, n, Q, Rb, 0.0, Z, n, st, nullptr);      // Z = Y (V Q)
      L += dgemm_small(0, 0, n, Rb, Rb, 1.0, nullptr, V, n, Q, Rb, 0.0, Ur, n, st, nullptr);     // Ritz vectors
      ritz_residual_kernel<<<Rb, 256, 0, st>>>(Z, Ur, sig, n, res);
      AO_CHECK_LAUNCH();
      ++L;
      AO_CUDA(cudaMemcpyAsync(h_sig.data(), sig, sizeof(double) * Rb, cudaMemcpyDeviceToHost, st));
      AO_CUDA(cudaMemcpyAsync(h_res.data(), res, sizeof(double) * Rb, cudaMemcpyDeviceToHost, st));
      AO_CUDA(cudaStreamSynchronize(st));
      std::iota(order.begin(), order.end(), 0);
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h_sig[a] > h_sig[b]; });
      const double top = h_sig[order[0]];
      double worst = 0.0;
      for (int i = 0; i < r; ++i) {
        if (!std::isfinite(h_sig[order[i]]) || !std::isfinite(h_res[order[i]])) throw CudaError(4, "nvecs: non-finite data");
        worst = std::max(worst, h_res[order[i]]);
      }
      info.residual = (top > 0.0) ? worst / top : 0.0;
      if (info.residual <= tol || Rb == n) break;
      if (info.residual < 0.95 * best) {
        best = info.residual;
        since_best = 0;
      } else if (++since_best >= 6 && best < 1e-10) {
        break;
      }
      orthonormalise(Z);
    }
    for (int i = 0; i < r; ++i) theta[i] = h_sig[order[i]];
    AO_CUDA(cudaMemcpyAsync(order_dev, order.data(), sizeof(int) * (size_t)r, cudaMemcpyHostToDevice, st));
    gather_signed_kernel<<<r, 256, 0, st>>>(Ur, n, order_dev, U);
    AO_CHECK_LAUNCH();
    ++L;
    AO_CUDA(cudaStreamSynchronize(st));
  } catch (...) {
    cudaFree(buf);
    cudaFree(order_dev);
    throw;
  }
  cudaFree(buf);
  cudaFree(order_dev);
  info.launches = L;
  return info;
}

}  // namespace aoadmm
