// smallops.cu - Gram / system preparation / fused ADMM iteration / reductions (sm_100a).
//
// Reference lines replaced (functions/cmtf_fun_AOADMM.m):
//   gram                 :66, :148, :190, :396           G_transp_G{m} = fac'*fac
//   prep_system          :98-103, :115-119, :124-127, :141-142, :257-276 (Hadamard, rho, B, chol)
//   admm_iteration       :591-623 (ADMM_constrained_only), :625-695 (ADMM_coupled_case0),
//                        :1420-1429 (update_constraint), :1079-1115 (eval_res_*), element-wise prox of
//                        functions/constraints_to_prox.m:13-18,:46-61
//   ls_solve             :134  fac = A/B
//   reduce_jobs          :1235-1241, :1272-1300, :1311, :1341 (objective reductions)
#include "smallops.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <map>

namespace aoadmm {

namespace {

// =====================================================================================================
// Gram
// =====================================================================================================
constexpr int kGramChunk = 64;   // rows per CTA: a 4096-row factor gives 64 x (R/32)^2 CTAs instead of 16 (the kernel is latency bound)

__global__ void gram_partial_kernel(const double* __restrict__ F, long long rows, long long ld, int R,
                                    double* __restrict__ ws, const int* __restrict__ skip) {
  if (skip != nullptr && *skip != 0) return;
  __shared__ double As[32][33];
  __shared__ double Bs[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * 16 + tx;
  const int bi = blockIdx.y, bj = blockIdx.z;
  const long long r0 = (long long)blockIdx.x * kGramChunk;
  const long long r1 = min(rows, r0 + (long long)kGramChunk);
  double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
  for (long long rb = r0; rb < r1; rb += 32) {
    for (int e = tid; e < 1024; e += 256) {
      const int rr = e & 31, c = e >> 5;
      const long long row = rb + rr;
      const int ca = bi * 32 + c, cb = bj * 32 + c;
      As[rr][c] = (row < r1 && ca < R) ? F[(long long)ca * ld + row] : 0.0;
      Bs[rr][c] = (row < r1 && cb < R) ? F[(long long)cb * ld + row] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr) {
      const double a0 = As[rr][2 * ty], a1 = As[rr][2 * ty + 1];
      const double b0 = Bs[rr][2 * tx], b1 = Bs[rr][2 * tx + 1];
      acc[0][0] = fma(a0, b0, acc[0][0]);
      acc[0][1] = fma(a0, b1, acc[0][1]);
      acc[1][0] = fma(a1, b0, acc[1][0]);
      acc[1][1] = fma(a1, b1, acc[1][1]);
    }
    __syncthreads();
  }
  double* out = ws + (long long)blockIdx.x * R * R;
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const int ia = bi * 32 + 2 * ty + a, ib = bj * 32 + 2 * tx + b;
      if (ia < R && ib < R) out[(long long)ib * R + ia] = acc[a][b];
    }
}

__global__ void gram_reduce_kernel(const double* __restrict__ ws, int nchunks, int RR, double* __restrict__ G,
                                   const int* __restrict__ skip) {
  if (skip != nullptr && *skip != 0) return;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= RR) return;
  double v = 0.0;
  for (int c = 0; c < nchunks; ++c) v += ws[(long long)c * RR + e];
  G[e] = v;
}

// =====================================================================================================
// prep_system: C = prod(had), rho = trace(C)/R, B = w*C + shifts, L = chol(B)
// =====================================================================================================
__global__ void __launch_bounds__(256, 1) prep_system_kernel(PrepArgs a, const int* __restrict__ skip) {
  if (skip != nullptr && *skip != 0) return;
  extern __shared__ double S[];  // R*R + R*(R+1) when R <= 64, else unused (factorisation runs in global memory)
  __shared__ double red[32];
  __shared__ double s_rho;
  __shared__ int s_err;
  const int R = a.R, RR = R * R, tid = threadIdx.x, nt = blockDim.x;
  const bool use_smem = (R <= 64);
  double* W = use_smem ? S : a.L;
  if (tid == 0) s_err = 0;
  // Hadamard product and trace
  double tr = 0.0;
  for (int e = tid; e < RR; e += nt) {
    double c = a.had[0][e];
    for (int h = 1; h < a.nhad; ++h) c *= a.had[h][e];
    a.C[e] = c;
    if (e % (R + 1) == 0) tr += c;
  }
  tr = block_sum(tr, red);
  if (tid == 0) {
    s_rho = tr / (double)R * a.rho_scale;
    *a.rho = s_rho;
  }
  __syncthreads();
  const double half = s_rho / 2.0;
  for (int e = tid; e < RR; e += nt) {
    double b = a.weight * a.C[e];
    if (e % (R + 1) == 0) {
      if (a.ridge != 0.0) b += a.ridge;
      if (a.bsum_half != 0.0) b += a.bsum_half;
      for (int q = 0; q < a.n_rho_terms; ++q) b += half;
    }
    if (a.HHt != nullptr) b += half * a.HHt[e];
    a.B[e] = b;
    W[e] = b;
  }
  __syncthreads();
  if (a.do_chol) {
    // Right-looking Cholesky on the lower triangle of W (column-major, ld = R).  The kernel is one CTA walking R
    // dependent steps, so a step is kept to ONE barrier and no division or square root: 1/sqrt(d) comes from rsqrt
    // (every thread computes it from the pivot it reads), the trailing update multiplies the still unscaled column by
    // it on the fly, and the column itself is scaled after the barrier - nothing reads column j again before the
    // substitution below.  L(i,j) = W(i,j) * rsqrt(d) in both places, so the factor is consistent to the bit.
    for (int j = 0; j < R; ++j) {
      const double d = W[j * R + j];
      if (!(d > 0.0) || !isfinite(d)) {
        if (tid == 0) s_err = 3;
        break;  // uniform: every thread read the same d
      }
      const double is = rsqrt(d);
      const int n = R - j - 1;
      const double* col = W + j * R + j + 1;
      // trailing block: 64 rows x (nt / 64) columns per pass (shifts and masks only - an integer division per entry
      // was most of a step)
      // The entries of a thread are loaded in batches of eight before any is stored: the compiler cannot move a
      // load above a possibly aliasing store, and one dependent shared-memory round trip per entry was the step time.
      const int cstep = nt >> 6;
      for (int ri = tid & 63; ri < n; ri += 64) {
        const double lr = col[ri] * is;
        double* wrow = W + (j + 1) * R + (j + 1 + ri);
        for (int c0 = tid >> 6; c0 <= ri; c0 += 8 * cstep) {
          double w8[8], l8[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int ci = c0 + u * cstep;
            const bool ok = ci <= ri;
            w8[u] = ok ? wrow[ci * R] : 0.0;
            l8[u] = ok ? col[ci] : 0.0;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int ci = c0 + u * cstep;
            if (ci <= ri) wrow[ci * R] = w8[u] - lr * (l8[u] * is);
          }
        }
      }
      __syncthreads();
      for (int i = j + 1 + tid; i < R; i += nt) W[j * R + i] *= is;
      if (tid == 0) W[j * R + j] = d * is;
    }
    __syncthreads();
    for (int e = tid; e < RR; e += nt) {
      const int ci = e / R, ri = e % R;
      const double v = (ri >= ci) ? W[e] : 0.0;
      a.L[e] = v;
      if (ri == ci) a.invdiag[ri] = 1.0 / v;
    }
    if (a.Binv != nullptr && s_err == 0) {
      // inv(L) by forward substitution on all columns at once: V = I; for every pivot j, row j is divided by L(j,j) and
      // L(i,j) * row j is subtracted from the rows below - again one barrier per step: the rows below use the scaled
      // row j on the fly (V(j,c) * 1/L(j,j)), row j is scaled in place after the barrier (zeros above the diagonal).
      // In shared memory V is stored transposed with an odd pitch, V(i,c) at V[c*(R+1) + i]: the substitution runs
      // with lanes over the rows i, the product below with lanes over the columns - both conflict-free.
      double* V = use_smem ? (S + RR) : a.Binv;
      const int vi = use_smem ? 1 : R, vc = use_smem ? R + 1 : 1;   // strides of the row / column index
      __syncthreads();
      for (int e = tid; e < RR; e += nt) V[(e / R) * vi + (e % R) * vc] = (e / R == e % R) ? 1.0 : 0.0;
      __syncthreads();
      for (int j = 0; j < R; ++j) {
        const double id = a.invdiag[j];   // 1 / L(j,j), stored above (visible after the barrier): no division on the chain
        const int cstep = nt >> 6;
        for (int i2 = j + 1 + (tid & 63); i2 < R; i2 += 64) {
          const double lij = -W[j * R + i2];
          for (int c0 = tid >> 6; c0 <= j; c0 += 8 * cstep) {   // batches of eight loads before the stores (see above)
            double v8[8], r8[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int c = c0 + u * cstep;
              const bool ok = c <= j;
              v8[u] = ok ? V[i2 * vi + c * vc] : 0.0;
              r8[u] = ok ? V[j * vi + c * vc] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int c = c0 + u * cstep;
              if (c <= j) V[i2 * vi + c * vc] = fma(lij, r8[u] * id, v8[u]);
            }
          }
        }
        __syncthreads();
        for (int c = tid; c <= j; c += nt) V[j * vi + c * vc] *= id;
      }
      __syncthreads();
      // inv(B) = inv(L)' * inv(L)
      if (use_smem) {
        for (int e = tid; e < RR; e += nt) {
          const int ca = e / R, cb = e % R;
          const int lo = ca > cb ? ca : cb;
          const double* va = V + ca * vc;
          const double* vb = V + cb * vc;
          double acc = 0.0;
          for (int i2 = lo; i2 < R; ++i2) acc = fma(va[i2], vb[i2], acc);
          a.Binv[e] = acc;
        }
      } else {
        // large R: V aliases a.Binv, so form the product into the scratch matrix first
        double* T = a.Btmp;
        for (int e = tid; e < RR; e += nt) {
          const int ca = e / R, cb = e % R;
          const int lo = ca > cb ? ca : cb;
          double acc = 0.0;
          for (int i2 = lo; i2 < R; ++i2) acc = fma(V[i2 * R + ca], V[i2 * R + cb], acc);
          T[e] = acc;
        }
        __syncthreads();
        for (int e = tid; e < RR; e += nt) a.Binv[e] = T[e];
      }
    }
  }
  if (tid == 0 && a.ctl != nullptr) {
    a.ctl->done = 0;
    a.ctl->iters = 0;
    if (s_err != 0) a.ctl->err = s_err;
    a.ctl->res[0] = a.ctl->res[1] = a.ctl->res[2] = a.ctl->res[3] = 0.0;
  }
}

// =====================================================================================================
// fused ADMM iteration (row-parallel)
// =====================================================================================================
struct FinInfo {
  int nmodes;
  int coupled;
  int constrained[kMaxGroup];
};

__device__ void finalize_ctl(const double* sums, const FinInfo& fin, const InnerTol& tol, InnerCtl* ctl) {
  double rpk = 0.0, rdk = 0.0, rpc = 0.0, rdc = 0.0;
  int nc = 0;
  const double dd = sqrt(sums[6 * fin.nmodes]);
  for (int mi = 0; mi < fin.nmodes; ++mi) {
    const double* s = sums + 6 * mi;
    const double nF = sqrt(s[0]);
    if (fin.coupled) {
      rpk += sqrt(s[1]) / nF;
      const double sc = sqrt(s[2]);
      rdk += (sc > 0.0) ? dd / sc : dd;
    }
    if (fin.constrained[mi]) {
      ++nc;
      rpc += sqrt(s[3]) / nF;
      const double sc = sqrt(s[5]);
      const double zz = sqrt(s[4]);
      rdc += (sc > 0.0) ? zz / sc : zz;
    }
  }
  if (fin.coupled) {
    rpk /= (double)fin.nmodes;
    rdk /= (double)fin.nmodes;
  }
  if (nc > 0) {
    rpc /= (double)nc;
    rdc /= (double)nc;
  }
  ctl->res[0] = rpk;
  ctl->res[1] = rdk;
  ctl->res[2] = rpc;
  ctl->res[3] = rdc;
  ctl->iters += 1;
  const bool cont = (rpk > tol.pr_coupl) || (rpc > tol.pr_constr) || (rdk > tol.du_coupl) || (rdc > tol.du_constr);
  if (!cont) ctl->done = 1;
  // a NaN ratio (0/0 of a factor driven to zero) makes its comparison false and an Inf keeps the loop going, exactly
  // as in the reference's while-test (:600, :633, :519); the run goes on and the event is only recorded
  if (!isfinite(rpk + rdk + rpc + rdc)) ctl->warn = 4;
}

// Solves x * (L L') = a in place for one row held in shared memory (element e at row_s[e*BT]).
__device__ __forceinline__ void solve_row(double* row_s, int BT, int R, const double* __restrict__ L,
                                          const double* __restrict__ invd) {
  for (int j = 0; j < R; ++j) {
    const double yj = row_s[j * BT] * invd[j];
    row_s[j * BT] = yj;
    const double* Lj = L + (long long)j * R;
    for (int e = j + 1; e < R; ++e) row_s[e * BT] = fma(-yj, Lj[e], row_s[e * BT]);
  }
  for (int j = R - 1; j >= 0; --j) {
    const double xj = row_s[j * BT] * invd[j];
    row_s[j * BT] = xj;
    for (int e = 0; e < j; ++e) row_s[e * BT] = fma(-xj, L[(long long)e * R + j], row_s[e * BT]);
  }
}

// One inner ADMM iteration for a tile of 32 rows (lanes) x all R columns (warp w owns columns 8w..8w+7):
//   per mode:  A_inner = A + rho/2 (Delta - muD) + rho/2 (Z - muZ)            (:608, :647-650)
//              F = A_inner * inv(B)                                           (:609, :651  (A_inner/L')/L)
//   Delta = sum_m rho_m (F_m + muD_m) / sum_m rho_m                            (:661-675)
//   muD_m += F_m - Delta ; Z_m = prox(F_m + muZ_m) ; muZ_m += F_m - Z_m        (:679-682, :1420-1429)
//   residual norms (:1079-1115) reduced deterministically; the last CTA evaluates the while-condition.
// inv(B) is formed once per outer iteration by prep_system (B = w*C + n*rho/2*I has cond(B) <= 1 + 2wR/n, so the
// explicit inverse is as accurate as the two triangular solves it replaces and turns the solve into a GEMM tile).
template <bool BSMEM>
__global__ void __launch_bounds__(BSMEM ? 256 : 1024) admm_tile_kernel(AdmmGroup g, FinInfo fin, InnerTol tol, InnerCtl* ctl, double* sums, double* partials,
                                 unsigned* counter, int finalize, int max_iters) {
  // max_iters > 1 (cooperative launch, every CTA resident): the whole inner ADMM loop of :600 / :633 runs inside one
  // launch, with a grid-wide barrier after every iteration so that all CTAs see the exit test of the last CTA.
  extern __shared__ double sm[];
  __shared__ double redm[32 * (6 * kMaxGroup + 1)];   // per-warp values of the NS running sums
  __shared__ bool s_last;
  const int R = g.R, tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nthreads = blockDim.x;
  // max_iters > 1: the grid-wide barrier between inner iterations is the "last CTA has evaluated the exit test" event
  // itself - counter[1] is a generation number the last CTA bumps after finalize_ctl, everybody else spins on it (all
  // CTAs are resident: cooperative launch).  One global round trip per inner iteration instead of the arrival counter
  // plus a separate grid.sync(); these loops are pure latency (107 us for 5 iterations on 4 CTAs as on 256).
  unsigned gen = (max_iters > 1) ? *reinterpret_cast<volatile unsigned*>(counter + 1) : 0u;
  double* a_s = sm;                      // [R][32]
  double* Binv_s = sm + (size_t)R * 32;  // [R*R] when BSMEM
  const long long i = (long long)blockIdx.x * 32 + lane;
  const bool active = i < g.rows;
  const int e0 = w * 8;
  const int NS = 6 * g.nmodes + 1;
  const bool coupled = g.Delta != nullptr;
  const bool binv_once = BSMEM && g.nmodes == 1;
  for (int inner = 0; inner < max_iters; ++inner) {
  if (*reinterpret_cast<volatile int*>(&ctl->done) != 0) return;  // uniform over the grid
  double lsum[6 * kMaxGroup + 1];
  for (int s = 0; s < NS; ++s) lsum[s] = 0.0;
  double dsum[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) dsum[c] = 0.0;
  double sum_rho = 0.0;

  for (int mi = 0; mi < g.nmodes; ++mi) {
    const AdmmMode& md = g.m[mi];
    // PARAFAC2 mode C: every row k has its own rho_k and its own R x R system (cmtf_fun_AOADMM.m:602-606, :638-645)
    const bool rowsys = md.Binv_rows != nullptr;
    const double rho = (md.rho_rows != nullptr) ? (active ? md.rho_rows[i] : 0.0) : *md.rho;
    const double half = rho / 2.0;
    sum_rho += rho;
    __syncthreads();  // previous mode's GEMM has finished reading a_s / Binv_s
    if (BSMEM && !rowsys && !(binv_once && inner > 0))   // a single-mode group stages its inverse once for the whole loop
      for (int e = tid; e < R * R; e += nthreads) Binv_s[e] = md.Binv[e];
    if (active) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int e = e0 + c;
        if (e < R) {
          const long long idx = (long long)e * g.rows + i;
          double a = md.A[(long long)e * md.ldA + i];
          if (coupled) a += half * (g.Delta[idx] - md.muD[idx]);
          if (md.constrained) a += half * (md.Z[idx] - md.muZ[idx]);
          a_s[e * 32 + lane] = a;
        }
      }
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (e0 + c < R) a_s[(e0 + c) * 32 + lane] = 0.0;
    }
    __syncthreads();
    double x[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) x[c] = 0.0;
    if (rowsys) {
      if (active) {
        const double* Br = md.Binv_rows + (size_t)i * R * R;
        for (int j = 0; j < R; ++j) {
          const double aj = a_s[j * 32 + lane];
#pragma unroll
          for (int c = 0; c < 8; ++c)
            if (e0 + c < R) x[c] = fma(aj, Br[(size_t)j * R + e0 + c], x[c]);
        }
      }
    } else if (BSMEM && e0 + 8 <= R) {
      const double* bp = Binv_s + e0;
#pragma unroll 4
      for (int j = 0; j < R; ++j) {
        const double aj = a_s[j * 32 + lane];
        const double* br = bp + (size_t)j * R;
#pragma unroll
        for (int c = 0; c < 8; ++c) x[c] = fma(aj, br[c], x[c]);
      }
    } else {
      const double* B0 = BSMEM ? Binv_s : md.Binv;
      for (int j = 0; j < R; ++j) {
        const double aj = a_s[j * 32 + lane];
#pragma unroll
        for (int c = 0; c < 8; ++c)
          if (e0 + c < R) x[c] = fma(aj, B0[(size_t)j * R + e0 + c], x[c]);
      }
    }
    if (active) {
      double sF2 = 0.0;
      // loads first, stores last: the compiler cannot move a global load above a possibly aliasing global store, so
      // interleaving them would serialise one memory round trip per column
      double mud[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) mud[c] = (coupled && e0 + c < R) ? md.muD[(long long)(e0 + c) * g.rows + i] : 0.0;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int e = e0 + c;
        if (e < R) {
          md.F[(long long)e * md.ldF + i] = x[c];
          sF2 = fma(x[c], x[c], sF2);
          if (coupled) dsum[c] += rho * (x[c] + mud[c]);
        }
      }
      lsum[6 * mi + 0] = sF2;
    }
  }

  if (active) {
    if (coupled) {
      const double inv = 1.0 / sum_rho;
      double sDD = 0.0;
      double dold[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) dold[c] = (e0 + c < R) ? g.Delta[(long long)(e0 + c) * g.rows + i] : 0.0;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int e = e0 + c;
        if (e < R) {
          const long long idx = (long long)e * g.rows + i;
          const double dn = inv * dsum[c];
          const double df = dn - dold[c];
          g.Delta[idx] = dn;
          dsum[c] = dn;
          sDD = fma(df, df, sDD);
        }
      }
      lsum[6 * g.nmodes] = sDD;
    }
    for (int mi = 0; mi < g.nmodes; ++mi) {
      const AdmmMode& md = g.m[mi];
      const double rho = *md.rho;  // for a vector rho the prox uses max(rho) (update_constraint, :1423-1424)
      double sFD = 0.0, sMuD = 0.0, sFZ = 0.0, sZZ = 0.0, sMuZ = 0.0;
      const bool do_con = md.constrained && prox_is_elementwise(md.prox_kind);
      double xf[8], vmd[8], vmz[8], vz[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) {  // all loads of this mode first (see above)
        const int e = e0 + c;
        const bool ok = e < R;
        const long long idx = (long long)e * g.rows + i;
        xf[c] = ok ? md.F[(long long)e * md.ldF + i] : 0.0;
        vmd[c] = (ok && coupled) ? md.muD[idx] : 0.0;
        vmz[c] = (ok && do_con) ? md.muZ[idx] : 0.0;
        vz[c] = (ok && do_con) ? md.Z[idx] : 0.0;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int e = e0 + c;
        if (e >= R) continue;
        const long long idx = (long long)e * g.rows + i;
        const double x = xf[c];
        if (coupled) {
          const double dn = dsum[c];
          const double mu = vmd[c] + x - dn;
          md.muD[idx] = mu;
          const double fd = x - dn;
          sFD = fma(fd, fd, sFD);
          sMuD = fma(mu, mu, sMuD);
        }
        if (do_con) {
          const double muz = vmz[c];
          const double zold = vz[c];
          const double z = prox_elem(md.prox_kind, x + muz, md.p0, md.p1, rho);
          const double munew = muz + x - z;
          md.Z[idx] = z;
          md.muZ[idx] = munew;
          const double fz = x - z, zz = z - zold;
          sFZ = fma(fz, fz, sFZ);
          sZZ = fma(zz, zz, sZZ);
          sMuZ = fma(munew, munew, sMuZ);
        }
      }
      lsum[6 * mi + 1] = sFD;
      lsum[6 * mi + 2] = sMuD;
      lsum[6 * mi + 3] = sFZ;
      lsum[6 * mi + 4] = sZZ;
      lsum[6 * mi + 5] = sMuZ;
    }
  }

  // deterministic two-level reduction: per-CTA partials (all NS sums at once: shuffles, one barrier, the warps' values
  // added in warp order), then the last CTA sums the partials in a fixed order
  for (int s = 0; s < NS; ++s) {
    const double v = warp_sum(lsum[s]);
    if (lane == 0) redm[w * (6 * kMaxGroup + 1) + s] = v;
  }
  __syncthreads();
  if (tid < NS) {
    double v = 0.0;
    for (int ww = 0; ww < (nthreads >> 5); ++ww) v += redm[ww * (6 * kMaxGroup + 1) + tid];
    partials[(long long)blockIdx.x * NS + tid] = v;
    __threadfence();
  }
  __syncthreads();
  if (tid == 0) {
    const unsigned t = atomicAdd(counter, 1u);
    s_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    for (int s = w; s < NS; s += (nthreads >> 5)) {   // one warp per sum
      const int mi = s / 6, ww = s % 6;
      // sums owned by a deferred (non element-wise) constraint update are left untouched
      const bool deferred = (s < 6 * g.nmodes) && (ww >= 3) && g.m[mi].constrained &&
                            !prox_is_elementwise(g.m[mi].prox_kind);
      if (deferred) continue;
      const double v = warp_sum_partials(partials + s, gridDim.x, (unsigned)NS);
      if (lane == 0) sums[s] = v;
    }
    __syncthreads();
    if (tid == 0) {
      *counter = 0u;
      if (finalize) finalize_ctl(sums, fin, tol, ctl);
      __threadfence();
      if (max_iters > 1) atomicAdd(counter + 1, 1u);   // releases the other CTAs into the next inner iteration
    }
  }
  if (max_iters > 1 && inner + 1 < max_iters) {
    if (tid == 0) {
      while (*reinterpret_cast<volatile unsigned*>(counter + 1) == gen) {
      }
      __threadfence();
    }
    gen += 1u;
    __syncthreads();
  }
  }  // inner iterations
}

// deferred constraint update for a mode whose prox is not element-wise
__global__ void admm_constraint_update_kernel(AdmmGroup g, int which, const double* __restrict__ Znew, FinInfo fin,
                                              InnerTol tol, InnerCtl* ctl, double* sums, double* partials,
                                              unsigned* counter, int finalize) {
  if (ctl->done != 0) return;
  __shared__ double red[32];
  __shared__ bool s_last;
  const AdmmMode& md = g.m[which];
  const long long n = g.rows * g.R;
  double sFZ = 0.0, sZZ = 0.0, sMuZ = 0.0;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long e = idx / g.rows, i = idx % g.rows;
    const double x = md.F[e * md.ldF + i];
    const double z = Znew[idx];
    const double zold = md.Z[idx];
    const double munew = md.muZ[idx] + x - z;
    md.Z[idx] = z;
    md.muZ[idx] = munew;
    const double fz = x - z, zz = z - zold;
    sFZ = fma(fz, fz, sFZ);
    sZZ = fma(zz, zz, sZZ);
    sMuZ = fma(munew, munew, sMuZ);
  }
  double v;
  v = block_sum(sFZ, red);
  if (threadIdx.x == 0) partials[blockIdx.x * 3 + 0] = v;
  v = block_sum(sZZ, red);
  if (threadIdx.x == 0) partials[blockIdx.x * 3 + 1] = v;
  v = block_sum(sMuZ, red);
  if (threadIdx.x == 0) partials[blockIdx.x * 3 + 2] = v;
  __threadfence();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(counter, 1u);
    s_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    if ((threadIdx.x >> 5) < 3) {   // one warp per sum
      const int q = threadIdx.x >> 5;
      const double t = warp_sum_partials(partials + q, gridDim.x, 3u);
      if ((threadIdx.x & 31) == 0) sums[6 * which + 3 + q] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      *counter = 0u;
      if (finalize) finalize_ctl(sums, fin, tol, ctl);
    }
  }
}

__global__ void admm_form_prox_input_kernel(AdmmGroup g, int which, double* __restrict__ V, const InnerCtl* ctl) {
  if (ctl != nullptr && ctl->done != 0) return;
  const AdmmMode& md = g.m[which];
  const long long n = g.rows * g.R;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long e = idx / g.rows, i = idx % g.rows;
    V[idx] = md.F[e * md.ldF + i] + md.muZ[idx];
  }
}

template <bool LSMEM>
__global__ void ls_solve_kernel(const double* __restrict__ A, long long ldA, const double* __restrict__ Lg,
                                const double* __restrict__ invdg, double* __restrict__ F, long long ldF,
                                long long rows, int R, const int* __restrict__ skip) {
  if (skip != nullptr && *skip != 0) return;
  extern __shared__ double sm[];
  const int BT = blockDim.x, tid = threadIdx.x;
  double* row_s = sm + tid;
  double* Ls = sm + (size_t)R * BT;
  double* invd_s = Ls + (LSMEM ? R * R : 0);
  const double* L = Lg;
  const double* invd = invdg;
  if (LSMEM) {
    for (int e = tid; e < R * R; e += BT) Ls[e] = Lg[e];
    for (int e = tid; e < R; e += BT) invd_s[e] = invdg[e];
    __syncthreads();
    L = Ls;
    invd = invd_s;
  }
  const long long i = (long long)blockIdx.x * BT + tid;
  if (i >= rows) return;
  for (int e = 0; e < R; ++e) row_s[e * BT] = A[(long long)e * ldA + i];
  solve_row(row_s, BT, R, L, invd);
  for (int e = 0; e < R; ++e) F[(long long)e * ldF + i] = row_s[e * BT];
}

// =====================================================================================================
// reductions: one CTA per job
// =====================================================================================================
constexpr int kRedSplit = 8;

// one job = sum over columns of a per-column quantity; CTA (job, y) handles columns y, y+kRedSplit, ...;
// the last CTA adds the kRedSplit partials of every job in fixed order (deterministic).
__global__ void reduce_jobs_kernel(const RedJob* __restrict__ jobs, double* __restrict__ results,
                                   double* __restrict__ partials, unsigned* counter, const int* __restrict__ skip) {
  if (skip != nullptr && *skip != 0) return;
  __shared__ double red[32];
  __shared__ bool s_last;
  const RedJob jb = jobs[blockIdx.x];
  const int tid = threadIdx.x, nt = blockDim.x;
  double total = 0.0;  // valid in thread 0
  double carry = 0.0;  // per-thread running sum over the columns of this CTA
  for (int c = blockIdx.y; c < jb.cols; c += kRedSplit) {
    const double* a = jb.a + (long long)c * jb.lda;
    const double* b = (jb.b != nullptr) ? jb.b + (long long)c * jb.ldb : nullptr;
    double acc = 0.0;
    long long i = tid;
    if (jb.kind == RED_DOT || jb.kind == RED_NORM2 || jb.kind == RED_COLNORM || jb.kind == RED_DIFF2) {
      // the three hot kinds: four independent load streams per thread (latency hiding at one CTA per SM)
      double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
      for (; i + 3LL * nt < jb.rows; i += 4LL * nt) {
        const double v0 = a[i], v1 = a[i + nt], v2 = a[i + 2LL * nt], v3 = a[i + 3LL * nt];
        if (jb.kind == RED_DOT) {
          c0 = fma(v0, b[i], c0);
          c1 = fma(v1, b[i + nt], c1);
          c2 = fma(v2, b[i + 2LL * nt], c2);
          c3 = fma(v3, b[i + 3LL * nt], c3);
        } else if (jb.kind == RED_DIFF2) {
          const double d0 = v0 - b[i], d1 = v1 - b[i + nt], d2 = v2 - b[i + 2LL * nt], d3 = v3 - b[i + 3LL * nt];
          c0 = fma(d0, d0, c0);
          c1 = fma(d1, d1, c1);
          c2 = fma(d2, d2, c2);
          c3 = fma(d3, d3, c3);
        } else {
          c0 = fma(v0, v0, c0);
          c1 = fma(v1, v1, c1);
          c2 = fma(v2, v2, c2);
          c3 = fma(v3, v3, c3);
        }
      }
      acc = (c0 + c1) + (c2 + c3);
    }
    for (; i < jb.rows; i += nt) {
      const double v = a[i];
      switch (jb.kind) {
        case RED_DOT: acc = fma(v, b[i], acc); break;
        case RED_NORM2:
        case RED_COLNORM: acc = fma(v, v, acc); break;
        case RED_DIFF2: {
          const double d = v - b[i];
          acc = fma(d, d, acc);
          break;
        }
        case RED_L1: acc += fabs(v); break;
        case RED_SUM: acc += v; break;
        case RED_NNZ: acc += (v != 0.0) ? 1.0 : 0.0; break;
        case RED_TVSUM:
          if (i + 1 < jb.rows) acc += a[i + 1] - v;
          break;
        case RED_GLQUAD: {
          // (L x)_i with L = tridiag(-1, 2, -1), corners 1
          double lx = v;  // rows == 1: L = [1]
          if (jb.rows > 1) {
            if (i == 0) lx = v - a[1];
            else if (i == jb.rows - 1) lx = v - a[i - 1];
            else lx = 2.0 * v - a[i - 1] - a[i + 1];
          }
          acc = fma(v, lx, acc);
          break;
        }
        default: break;
      }
    }
    if (jb.kind == RED_COLNORM) {   // needs the square root of every column's sum
      acc = block_sum(acc, red);
      if (tid == 0) total += sqrt(acc);
    } else {
      carry += acc;                 // one block reduction for all columns of this CTA (two barriers per column were most
    }                               // of the kernel on factor-sized jobs)
  }
  if (jb.kind != RED_COLNORM) {
    carry = block_sum(carry, red);
    if (tid == 0) total = carry;
  }
  if (tid == 0) partials[blockIdx.x * kRedSplit + blockIdx.y] = total;
  __threadfence();
  if (tid == 0) {
    const unsigned t = atomicAdd(counter, 1u);
    s_last = (t == gridDim.x * gridDim.y - 1);
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    for (int j = tid; j < (int)gridDim.x; j += nt) {
      double v = 0.0;
      for (int y = 0; y < kRedSplit; ++y) v += partials[j * kRedSplit + y];
      results[j] = v;
    }
    if (tid == 0) *counter = 0u;
  }
}

}  // namespace

// =====================================================================================================
// host wrappers
// =====================================================================================================
size_t gram_ws_doubles(int64_t rows, int R) { return (size_t)ceil_div(std::max<int64_t>(rows, 1), kGramChunk) * R * R; }

int gram(const double* F, int64_t rows, int64_t ld, int R, double* G, double* ws, cudaStream_t st, const int* skip) {
  const int nchunks = (int)ceil_div(std::max<int64_t>(rows, 1), kGramChunk);
  const int nb = (int)ceil_div(R, 32);
  dim3 grid(nchunks, nb, nb), block(16, 16);
  gram_partial_kernel<<<grid, block, 0, st>>>(F, rows, ld, R, ws, skip);
  AO_CHECK_LAUNCH();
  gram_reduce_kernel<<<(unsigned)ceil_div(R * R, 256), 256, 0, st>>>(ws, nchunks, R * R, G, skip);
  AO_CHECK_LAUNCH();
  return 2;
}

int prep_system(const PrepArgs& a, cudaStream_t st, const int* skip) {
  const size_t smem = (a.R <= 64) ? ((size_t)2 * a.R * a.R + a.R) * sizeof(double) : 0;
  if (smem > 40 * 1024) ensure_dynamic_smem(reinterpret_cast<const void*>(prep_system_kernel), (2 * 64 * 64 + 64) * 8, 40 * 1024);
  if (a.Binv != nullptr && a.R > 64 && a.Btmp == nullptr) throw CudaError(1, "prep_system: Btmp scratch required for R > 64");
  prep_system_kernel<<<1, 256, smem, st>>>(a, skip);
  AO_CHECK_LAUNCH();
  return 1;
}

namespace {
struct RowLaunch {
  int BT;
  bool lsmem;
  size_t smem;
};
RowLaunch row_launch_cfg(int R, int nrowbuf) {
  RowLaunch c;
  c.BT = (R <= 32) ? 128 : ((R <= 64) ? 64 : 32);
  c.lsmem = (R <= 64);
  c.smem = ((size_t)nrowbuf * R * c.BT + (c.lsmem ? (size_t)R * R + R : 0)) * sizeof(double);
  return c;
}
FinInfo make_fin(const AdmmGroup& g) {
  FinInfo f;
  f.nmodes = g.nmodes;
  f.coupled = g.Delta != nullptr;
  for (int i = 0; i < kMaxGroup; ++i) f.constrained[i] = (i < g.nmodes) ? g.m[i].constrained : 0;
  return f;
}
template <typename K>
void set_smem(K kern, size_t smem) {
  // once per device, kernel and size: no attribute calls on the steady-state path (not allowed inside graph capture)
  ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem, 40 * 1024);
}
}  // namespace

size_t admm_ws_doubles(long long rows, int R, int nmodes) {
  (void)R;
  const size_t ctas_row = (size_t)ceil_div(std::max<long long>(rows, 1), 32);
  return std::max<size_t>(ctas_row * (6 * nmodes + 1), (size_t)148 * 8 * 3) + 16;
}

int admm_iteration(const AdmmGroup& g, const InnerTol& tol, InnerCtl* ctl, double* sums, double* partials,
                   unsigned* counter, int finalize, cudaStream_t st, int max_iters) {
  const int nw = (int)ceil_div(g.R, 8);
  const unsigned ctas = (unsigned)ceil_div(std::max<long long>(g.rows, 1), 32);
  const bool bsmem = g.R <= 64;
  const size_t smem = ((size_t)g.R * 32 + (bsmem ? (size_t)g.R * g.R : 0)) * sizeof(double);
  const FinInfo fin = make_fin(g);
  if (bsmem) set_smem(admm_tile_kernel<true>, smem);
  else set_smem(admm_tile_kernel<false>, smem);
  if (max_iters > 1) {
    AdmmGroup gg = g;
    FinInfo ff = fin;
    InnerTol tt = tol;
    void* args[] = {&gg, &ff, &tt, &ctl, &sums, &partials, &counter, &finalize, &max_iters};
    const void* fn = bsmem ? reinterpret_cast<const void*>(admm_tile_kernel<true>)
                           : reinterpret_cast<const void*>(admm_tile_kernel<false>);
    AO_CUDA(cudaLaunchCooperativeKernel(fn, dim3(ctas), dim3(nw * 32), args, smem, st));
    return 1;
  }
  if (bsmem)
    admm_tile_kernel<true><<<ctas, nw * 32, smem, st>>>(g, fin, tol, ctl, sums, partials, counter, finalize, 1);
  else
    admm_tile_kernel<false><<<ctas, nw * 32, smem, st>>>(g, fin, tol, ctl, sums, partials, counter, finalize, 1);
  AO_CHECK_LAUNCH();
  return 1;
}

// true when all CTAs of the ADMM tile kernel for this group can be resident at once (cooperative launch possible)
bool admm_can_fuse_inner(const AdmmGroup& g) {
  const int nw = (int)ceil_div(g.R, 8);
  const long long ctas = ceil_div(std::max<long long>(g.rows, 1), 32);
  const bool bsmem = g.R <= 64;
  const size_t smem = ((size_t)g.R * 32 + (bsmem ? (size_t)g.R * g.R : 0)) * sizeof(double);
  if (bsmem) set_smem(admm_tile_kernel<true>, smem);
  else set_smem(admm_tile_kernel<false>, smem);
  int per_sm = 0, dev = 0, sms = 0, coop = 0;
  AO_CUDA(cudaGetDevice(&dev));
  AO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  AO_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
  if (!coop) return false;
  if (bsmem)
    AO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, admm_tile_kernel<true>, nw * 32, smem));
  else
    AO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, admm_tile_kernel<false>, nw * 32, smem));
  return ctas <= (long long)per_sm * sms;
}

int admm_constraint_update(const AdmmGroup& g, int which, const double* Znew, const InnerTol& tol, InnerCtl* ctl,
                           double* sums, double* partials, unsigned* counter, int finalize, cudaStream_t st) {
  const long long n = g.rows * g.R;
  const unsigned ctas = (unsigned)std::min<long long>(ceil_div(std::max<long long>(n, 1), 256), 148 * 8);
  admm_constraint_update_kernel<<<ctas, 256, 0, st>>>(g, which, Znew, make_fin(g), tol, ctl, sums, partials, counter,
                                                      finalize);
  AO_CHECK_LAUNCH();
  return 1;
}

int admm_form_prox_input(const AdmmGroup& g, int which, double* V, const InnerCtl* ctl, cudaStream_t st) {
  const long long n = g.rows * g.R;
  const unsigned ctas = (unsigned)std::min<long long>(ceil_div(std::max<long long>(n, 1), 256), 148 * 8);
  admm_form_prox_input_kernel<<<ctas, 256, 0, st>>>(g, which, V, ctl);
  AO_CHECK_LAUNCH();
  return 1;
}

int ls_solve(const double* A, long long ldA, const double* L, const double* invdiag, double* F, long long ldF,
             long long rows, int R, InnerCtl* ctl, cudaStream_t st, const int* skip) {
  (void)ctl;
  const RowLaunch c = row_launch_cfg(R, 1);
  const unsigned ctas = (unsigned)ceil_div(std::max<long long>(rows, 1), c.BT);
  if (c.lsmem) {
    set_smem(ls_solve_kernel<true>, c.smem);
    ls_solve_kernel<true><<<ctas, c.BT, c.smem, st>>>(A, ldA, L, invdiag, F, ldF, rows, R, skip);
  } else {
    set_smem(ls_solve_kernel<false>, c.smem);
    ls_solve_kernel<false><<<ctas, c.BT, c.smem, st>>>(A, ldA, L, invdiag, F, ldF, rows, R, skip);
  }
  AO_CHECK_LAUNCH();
  return 1;
}

size_t reduce_ws_doubles(int njobs) { return (size_t)njobs * kRedSplit; }

int reduce_jobs(const RedJob* jobs_dev, int njobs, double* results_dev, double* partials, unsigned* counter,
                cudaStream_t st, const int* skip) {
  if (njobs <= 0) return 0;
  dim3 grid(njobs, kRedSplit);
  reduce_jobs_kernel<<<grid, 256, 0, st>>>(jobs_dev, results_dev, partials, counter, skip);
  AO_CHECK_LAUNCH();
  return 1;
}

namespace {
// every pair of the table in one launch: each thread walks all pairs, grid-striding over the elements of each; 16-byte
// accesses where both ends allow them (the buffers are separate cudaMalloc allocations or 256-byte aligned offsets)
template <int kDir>
__global__ void __launch_bounds__(256) state_copy_kernel(const CopyDesc* __restrict__ table, int n_desc) {
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nt = (long long)gridDim.x * blockDim.x;
  for (int q = 0; q < n_desc; ++q) {
    const CopyDesc c = table[q];
    const double* __restrict__ src = kDir == 0 ? c.state : c.snap;
    double* __restrict__ dst = kDir == 0 ? c.snap : c.state;
    long long done = 0;
    if ((((uintptr_t)src | (uintptr_t)dst) & 15) == 0) {
      const long long n2 = c.n >> 1;
      const double2* s2 = reinterpret_cast<const double2*>(src);
      double2* d2 = reinterpret_cast<double2*>(dst);
      for (long long e = tid; e < n2; e += nt) d2[e] = s2[e];
      done = n2 << 1;
    }
    for (long long e = done + tid; e < c.n; e += nt) dst[e] = src[e];
  }
}
}  // namespace

int state_copy(const CopyDesc* table_dev, int n_desc, long long max_n, int direction, cudaStream_t st) {
  if (n_desc <= 0 || max_n <= 0) return 0;
  const unsigned ctas = (unsigned)std::min<long long>(ceil_div((max_n + 1) / 2, 256), 148 * 8);
  if (direction == 0) state_copy_kernel<0><<<ctas, 256, 0, st>>>(table_dev, n_desc);
  else state_copy_kernel<1><<<ctas, 256, 0, st>>>(table_dev, n_desc);
  AO_CHECK_LAUNCH();
  return 1;
}

}  // namespace aoadmm
