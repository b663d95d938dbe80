// nvecs.cuh - device-side "nvecs" initialisation: the leading eigenvectors of X_(n) X_(n)'.
//
// Reference: functions/cmtf_nvecs.m:33-58 (A = unfolding of the object that contains mode n; Y = A*A';
// [U,~] = eigs(Y, r, 'LM')) and functions/init_coupled_AOADMM_CMTF.m:50-69 (PARAFAC2: mode A from the slices side by
// side, B_k from X_k'X_k, C = ones).
//
// Two steps, both on the device:
//   1. unfold_gram: Y = X_(n) X_(n)' straight from the resident tensor (no unfolding is materialised), FP64 tensor
//      cores (DMMA.8x8x4), 128 x 128 output tiles of the upper triangle, cp.async 3-stage pipeline, split over the
//      reduction range with a fixed-order reduction that also mirrors the triangle (Y exactly symmetric).
//   2. top_eigvecs: block subspace iteration with Rayleigh-Ritz on Y (oversampled block, one-sided Jacobi for the
//      small eigenproblems), until the residuals ||Y u - theta u|| of the r leading pairs are at rounding level.
#pragma once
#include <functional>

#include "linalg.cuh"

namespace aoadmm {

// Which elements form the unfolding.  layout 0 ("NT"): A(a, c) = X[a + ld*c], a < n, c < ncols (mode is the
// contiguous one).  layout 1 ("TN"): A(a, (i,b)) = X[i + cs*a + bs*b], i < I, b < nb (reduction over the contiguous
// index i and a batch index b).
// X must be 16-byte aligned and ld / cs / bs even (the engine pads every leading dimension to an even length).
struct UnfoldSpec {
  const double* X = nullptr;
  int layout = 0;
  long long n = 0;              // rows/cols of Y
  long long ld = 0, ncols = 0;  // layout 0
  long long I = 0, cs = 0, bs = 0, nb = 0;  // layout 1
};

// doubles of workspace needed by unfold_gram for this spec
size_t unfold_gram_workspace(const UnfoldSpec& s);
// Y (n x n, ld = n) = A A'  (accumulate: Y += A A').  Returns the number of launches.
int unfold_gram(const UnfoldSpec& s, double* Y, double* work, cudaStream_t st, bool accumulate = false);

struct EigInfo {
  int iterations = 0;
  double residual = 0.0;   // max_i ||Y u_i - theta_i u_i|| / theta_1 over the r returned pairs
  int launches = 0;
};
// U (n x r, ld = n, device) = eigenvectors of the symmetric positive semi-definite Y (n x n, ld = n, device) for its r
// largest eigenvalues, in descending order (eigs(Y,r,'LM')); theta (host, r entries).  Every column is signed so that its
// entry of largest magnitude is positive.  Synchronises the stream.
EigInfo top_eigvecs(const double* Y, long long n, int r, double* U, double* theta, cudaStream_t st);

// Operator form: apply(V, W, cols) sets W = Y V for V, W n x cols (column-major, ld = n, device, on `st`) and returns its
// launches.  Everything else (block size, start vectors, stopping rule, sign rule) is the dense iteration's; the dense
// overload is this one with the dgemm W = Y V, so its results are unchanged bit for bit.
using EigOperator = std::function<int(const double* V, double* W, int cols)>;
EigInfo top_eigvecs(const EigOperator& apply, long long n, int r, double* U, double* theta, cudaStream_t st);
// columns of the iteration block for r vectors of an n-row mode (the operator is applied to n x eig_block(n, r))
int eig_block(long long n, int r);

}  // namespace aoadmm
