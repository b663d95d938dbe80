// smallops.cuh - the O((I+J+K) R^2) part of the AO-ADMM sweep: Grams, Hadamard-of-Grams + rho + system
// matrix + Cholesky, the fused ADMM row kernel (solve / Delta / duals / elementwise prox / residual sums),
// stand-alone prox kernels and the objective reductions.
#pragma once
#include "common.cuh"

namespace aoadmm {

enum ProxKind : int {
  PROX_NONE = 0, PROX_NONNEG = 1, PROX_BOX = 2, PROX_SIMPLEX_COL = 3, PROX_SIMPLEX_ROW = 4,
  PROX_NONDECREASING = 5, PROX_NONINCREASING = 6, PROX_UNIMODAL = 7, PROX_L1_BALL = 8, PROX_L2_BALL = 9,
  PROX_NONNEG_L2_BALL = 10, PROX_NONNEG_L2_SPHERE = 11, PROX_ORTHONORMAL = 12, PROX_L1_REG = 13,
  PROX_L0_REG = 14, PROX_L2_REG = 15, PROX_RIDGE = 16, PROX_QUADRATIC = 17, PROX_GL_SMOOTH = 18, PROX_TV = 19,
  PROX_TPARAFAC2 = 20, PROX_CUSTOM = 21
};

#ifdef __CUDACC__
__host__ __device__
#endif
inline bool prox_is_elementwise(int k) {
  return k == PROX_NONNEG || k == PROX_BOX || k == PROX_L1_REG || k == PROX_L0_REG || k == PROX_RIDGE;
}

#ifdef __CUDACC__
// element-wise prox operators (constraints_to_prox.m:13-18, :46-61)
__device__ __forceinline__ double prox_elem(int kind, double v, double p0, double p1, double rho) {
  switch (kind) {
    case PROX_NONNEG: return fmax(v, 0.0);
    case PROX_BOX: return fmin(fmax(v, p0), p1);
    case PROX_L1_REG: {
      const double g = p0 / rho;
      const double mag = fmax(fabs(v) - g, 0.0);
      return (v > 0.0) ? mag : ((v < 0.0) ? -mag : 0.0);
    }
    case PROX_L0_REG: {
      const double g = p0 / rho;
      return (fabs(v) > sqrt(2.0 * g)) ? v : 0.0;
    }
    case PROX_RIDGE: return 1.0 / (2.0 * (p0 / rho) + 1.0) * v;
    default: return v;
  }
}
#endif

// ---- inner-loop control block (device resident) ---------------------------------------------------
struct InnerCtl {
  int done;        // 1: the data-dependent exit test of the ADMM while-loop has fired
  int iters;       // inner iterations executed so far (the reference's inner_iter-1)
  int err;         // 0 ok, 3 not positive definite
  int warn;        // 4: a residual ratio of this loop was NaN/Inf at least once during the run (not an error)
  double res[4];   // rel_primal_coupling, rel_dual_coupling, rel_primal_constr, rel_dual_constr
};

struct InnerTol {
  double pr_coupl, du_coupl, pr_constr, du_constr;
};

// ---- Gram ----------------------------------------------------------------------------------------
// G (R x R col-major) = F' * F, F rows x R (ld).  ws: >= gram_ws_doubles(rows,R) doubles.
size_t gram_ws_doubles(int64_t rows, int R);
int gram(const double* F, int64_t rows, int64_t ld, int R, double* G, double* ws, cudaStream_t st, const int* skip);

// ---- system preparation ----------------------------------------------------------------------------
struct PrepArgs {
  const double* had[8];   // Gram matrices multiplied element-wise (C = prod had[i]); nhad >= 1
  int nhad;
  int R;
  double weight;          // Z.weights(p)
  double ridge;           // Z.ridge(m) or 0
  double bsum_half;       // options.bsum_weight/2 or 0
  int n_rho_terms;        // how many rho/2*I terms are added (constraint / coupling)
  double rho_scale;       // increase_factor_rhoBk or 1
  const double* HHt;      // optional R x R matrix added as rho/2 * HHt (coupling type 2), else nullptr
  int do_chol;            // 0: leave B unfactored (unconstrained least squares uses LU-free Cholesky too)
  double* C;              // out: Hadamard product (last_had)
  double* B;              // out: system matrix
  double* L;              // out: lower Cholesky factor of B (col-major), strictly upper part zeroed
  double* invdiag;        // out: 1 / diag(L)
  double* Binv;           // out (optional): inv(B) = inv(L)'*inv(L), used by the ADMM tile kernel
  double* Btmp;           // scratch R x R, needed with Binv when R > 64
  double* rho;            // out: trace(C)/R * rho_scale
  InnerCtl* ctl;          // reset (done = 0, iters = 0); err set on failure
};
int prep_system(const PrepArgs& a, cudaStream_t st, const int* skip);

// Cholesky-based solve  X = A * inv(B)  for a general (symmetric positive definite) B: used for the
// unconstrained least-squares update fac = A/B (cmtf_fun_AOADMM.m:134).
// ---- fused ADMM iteration ---------------------------------------------------------------------------
constexpr int kMaxGroup = 8;

struct AdmmMode {
  const double* A;        // right-hand side (weighted MTTKRP [+ bsum term]) rows x R
  const double* Binv;     // inv(B), R x R (symmetric)
  const double* rho;      // device scalar (PARAFAC2 mode C: max_k rho_k, used by the prox)
  const double* rho_rows; // optional: per-row rho (PARAFAC2 mode C), else nullptr
  const double* Binv_rows;// optional: per-row inv(B_k), rows x R x R (PARAFAC2 mode C), else nullptr
  double* F;              // factor matrix
  double* Z;              // constraint_fac or nullptr
  double* muZ;            // constraint_dual_fac or nullptr
  double* muD;            // coupling_dual_fac or nullptr
  long long ldA, ldF;
  int constrained;        // Z.constrained_modes(m)
  int prox_kind;          // ProxKind
  double p0, p1;
};

struct AdmmGroup {
  int nmodes;
  AdmmMode m[kMaxGroup];
  double* Delta;          // coupling_fac (nullptr when the mode is not coupled)
  long long rows;
  int R;
};

size_t admm_ws_doubles(long long rows, int R, int nmodes);
// one inner iteration: returns launches.  `partials` (>= admm_ws_doubles) and `counter` (one uint, zeroed once)
// are scratch; `ctl` is updated by the last CTA (residuals, exit test, iteration count).
// `sums` (6*nmodes+1 doubles, device) holds the reduced norms of the current inner iteration; `finalize` != 0
// makes the kernel evaluate the exit test (set it on the LAST kernel of the inner iteration).
// max_iters > 1: ONE cooperative launch runs up to max_iters inner iterations (grid barrier between them); only valid
// when admm_can_fuse_inner(g) and every constrained mode of the group has an element-wise prox.
int admm_iteration(const AdmmGroup& g, const InnerTol& tol, InnerCtl* ctl, double* sums, double* partials,
                   unsigned* counter, int finalize, cudaStream_t st, int max_iters = 1);
bool admm_can_fuse_inner(const AdmmGroup& g);
// the deferred constraint part for modes whose prox is not element-wise:  Z = prox(F+muZ) computed by
// prox_apply into Znew, then this kernel forms muZ, the residual sums and copies Znew -> Z.
// `finalize` recomputes ctl from the partial sums (same test as admm_iteration).
int admm_constraint_update(const AdmmGroup& g, int which, const double* Znew, const InnerTol& tol, InnerCtl* ctl,
                           double* sums, double* partials, unsigned* counter, int finalize, cudaStream_t st);

// V = F + muZ for mode `which` of the group (input of a non-elementwise prox)
int admm_form_prox_input(const AdmmGroup& g, int which, double* V, const InnerCtl* ctl, cudaStream_t st);

// unconstrained least squares:  F = A * inv(B) using L (cmtf_fun_AOADMM.m:134)
int ls_solve(const double* A, long long ldA, const double* L, const double* invdiag, double* F, long long ldF,
             long long rows, int R, InnerCtl* ctl, cudaStream_t st, const int* skip);

// ---- stand-alone prox -------------------------------------------------------------------------------
// out = prox_kind(X, rho)   (X, out: rows x cols col-major with leading dimensions ldx, ldo; may alias).
// rho is read from device memory (rho_dev) when non-null, else rho_host is used.
size_t prox_scratch_bytes(int kind, long long rows, int cols);
int prox_apply(int kind, double p0, double p1, const double* X, long long ldx, double* out, long long ldo,
               long long rows, int cols, const double* rho_dev, double rho_host, void* scratch, cudaStream_t st,
               const int* skip);

// The same operator applied to K row segments of a stacked matrix in ONE launch (PARAFAC2 B_k mode, :567-568: the prox of
// every slice with its own rho_k): segment k = rows seg_off_dev[k] .. seg_off_dev[k+1]-1 of every column, rho of segment
// k = rho_dev_per_seg[k].  Only kinds with prox_supports_segments(); scratch >= prox_segments_scratch_bytes().
bool prox_supports_segments(int kind);
size_t prox_segments_scratch_bytes(int kind, long long max_rows, int cols, int nseg);
int prox_apply_segments(int kind, double p0, double p1, const double* X, long long ldx, double* out, long long ldo,
                        const long long* seg_off_dev, int nseg, long long max_rows, long long total_rows, int cols,
                        const double* rho_dev_per_seg, void* scratch, cudaStream_t st, const int* skip);

// 'quadratic regularization' (constraints_to_prox.m:62-67): prox(x,rho) = (2*eta/rho*L + I) \ x for a SYMMETRIC L,
// applied in the eigen-basis L = Q diag(lam) Q' (computed once): out = Q * ((Q'x) ./ (2*eta/rho*lam + 1)).
struct QuadProx {
  double* L = nullptr;    // n x n (kept for the regulariser value eta*trace(x'Lx))
  double* Q = nullptr;    // n x n eigenvectors
  double* lam = nullptr;  // n eigenvalues
  double* tmp = nullptr;  // n x maxcols scratch
  long long n = 0;
  int maxcols = 0;
  double eta = 0.0;
};
void quad_prox_setup(QuadProx& q, const double* L_host, long long n, double eta, int maxcols, cudaStream_t st);
void quad_prox_free(QuadProx& q);
int quad_prox_apply(const QuadProx& q, const double* X, long long ldx, double* out, long long ldo, int cols,
                    const double* rho_dev, double rho_host, cudaStream_t st, const int* skip);

// ---- reductions ---------------------------------------------------------------------------------------
enum RedKind : int {
  RED_DOT = 0,         // sum a.*b
  RED_NORM2 = 1,       // sum a.^2
  RED_DIFF2 = 2,       // sum (a-b).^2
  RED_L1 = 3,          // sum |a|
  RED_NNZ = 4,         // count(a != 0)
  RED_COLNORM = 5,     // sum_r ||a(:,r)||_2
  RED_TVSUM = 6,       // sum_r sum_i a(i+1,r)-a(i,r)      (constraints_to_prox.m:81, no abs)
  RED_GLQUAD = 7,      // trace(a' * Lgl * a) with the graph-Laplacian of constraints_to_prox.m:71-73
  RED_SUM = 8          // sum a
};
struct RedJob {
  int kind;
  int cols;
  long long rows, lda, ldb;
  const double* a;
  const double* b;
};
// results[j] for each job; jobs resident in device memory (uploaded once)
// `partials` (>= reduce_ws_doubles(njobs)) and `counter` (one zeroed uint) are scratch.
size_t reduce_ws_doubles(int njobs);
int reduce_jobs(const RedJob* jobs_dev, int njobs, double* results_dev, double* partials, unsigned* counter,
                cudaStream_t st, const int* skip);

// ---- state snapshot (early stopping on the held-out error) ------------------------------------------
// one buffer of the snapshot list: n doubles of device state and their copy in the snapshot
struct CopyDesc {
  double* state;
  double* snap;
  long long n;
};
// direction 0: snap = state (snapshot), 1: state = snap (restore), for all n_desc pairs of the device-resident table in
// ONE launch sized for the largest pair (max_n doubles).  Returns the launches.
int state_copy(const CopyDesc* table_dev, int n_desc, long long max_n, int direction, cudaStream_t st);

}  // namespace aoadmm
