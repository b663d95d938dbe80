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
#pragma once
#include <vector>

#include "common.cuh"

namespace aoadmm {

constexpr int kSparseChunk = 256;   // nonzeros per unit of work

struct SparseMode {
  long long* rowptr = nullptr;      // rows + 1
  int* chunk_row = nullptr;         // row of the first nonzero of every unit
  int* head_row = nullptr;          // per unit: its first row when that row began in an earlier unit, else -1
  int* tail_row = nullptr;          // per unit: its last row when that row goes on in a later unit, else -1
  double* vals = nullptr;           // nnz
  int* idx = nullptr;               // (order-1) x nnz: indices of the other modes in ascending position
};

struct SparseTensor {
  int order = 0, R = 0;
  long long nnz = 0;                // after merging duplicates
  long long dims[8] = {0};
  std::vector<SparseMode> modes;
  double* factT[8] = {nullptr};     // row-major (rows x R) copies of the factors, refreshed per MTTKRP
  double* outT = nullptr;           // row-major product, max rows x R
  double* head = nullptr;           // units x R: partial sums of the head rows
  double* tail = nullptr;           // units x R: partial sums of the tail rows
  double* norm_partials = nullptr;  // deterministic two-level reduction
  double* norm_out = nullptr;
};

// Uploads and preprocesses one COO object: subs is nnz x order column-major (0-based, validated by the caller), vals nnz
// values.  Duplicates are summed.  Allocates every scratch buffer the MTTKRP needs.  Synchronous on `st`.
void sparse_build(SparseTensor& s, int order, const long long* dims, int R, long long nnz, const long long* subs,
                  const double* vals, cudaStream_t st);
void sparse_free(SparseTensor& s);
// ||X||_F^2 = sum of the squared merged values (fixed-order reduction); the result lands in s.norm_out (device)
int sparse_norm2(const SparseTensor& s, cudaStream_t st);
// out (rows(n) x R, column-major, leading dimension ldout) = scale * MTTKRP of mode position n, from the column-major
// factors fac[d] (leading dimension ld[d]) of all mode positions.  Returns the number of kernel launches.
int sparse_mttkrp(SparseTensor& s, int n, const double* const* fac, const long long* ld, double scale, double* out,
                  long long ldout, cudaStream_t st);

}  // namespace aoadmm
