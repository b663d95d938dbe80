// heldout.cuh - held-out entries of a CP object (sm_100a, FP64): the model at given subscripts and, once per outer
// iteration, the squared error of the model on a held-out set that was withheld from training.
//
// Both passes use the lane layout of the sparse path (sparse.cuh): a group of lanes walks a unit of kSparseChunk
// consecutive entries, the rank dispatch and the row-major factor copies are those of sparse.cu, and the sum over the
// rank runs in a fixed order (model_at_entry).  The held-out error reduces per-CTA partials and then one fixed-order
// sum: no floating-point atomics, so every result is bit-reproducible.  A held-out set is sorted once on the device by
// its full subscript key (duplicates summed), so results do not depend on the order in which the caller listed it.
#pragma once
#include <cstdint>

#include "sparse.cuh"

namespace aoadmm {

struct HeldOut {
  int order = 0, R = 0;
  long long n = 0;                  // entries after merging duplicates
  long long dims[8] = {0};          // full mode sizes
  int* subs = nullptr;              // order x n, column-major, full lexicographic order (mode 1 major)
  double* vals = nullptr;           // n true values
  double* factT[8] = {nullptr};     // row-major copies of the factors, refreshed per pass
  double* partials = nullptr;       // per-CTA partial sums of the error pass
};

// Uploads n >= 0 entries (subs n x order column-major, 0-based, validated by the caller), sorts and merges them on the
// device and allocates every buffer of heldout_sse.  Synchronous on `st`.
void heldout_build(HeldOut& h, int order, const long long* dims, int R, long long n, const long long* subs,
                   const double* vals, cudaStream_t st);
void heldout_free(HeldOut& h);
// *sse (device) = sum_e (v_e - m_e)^2 with m = [[F]] at the held-out entries, from the column-major factors fac[d]
// (leading dimension ld[d]).  Allocation-free and graph-capturable.  Returns the number of kernel launches.
int heldout_sse(HeldOut& h, const double* const* fac, const long long* ld, double* sse, cudaStream_t st);
// Held-out entries that were observed in training.  Sparse masked object `s`: the entry is stored (looked up in the
// mode-1 copy; a slab of a sharded object checks only the entries of its slab).  Dense mask (ld0 bytes per leading column, local extents ldims, the last mode starting at
// shard_offset): its mask byte is nonzero; only the entries of this slab are checked.  Returns the count and the
// position (in h's sorted order) of the first such entry in *first (-1: none).  Synchronous on `st`.
long long heldout_stored(const HeldOut& h, const SparseTensor& s, long long* first, cudaStream_t st);
long long heldout_masked(const HeldOut& h, const uint8_t* mask, long long ld0, const long long* ldims,
                         long long shard_offset, long long* first, cudaStream_t st);
// subscripts of sorted entry e of h (host copy; for messages)
void heldout_subscript(const HeldOut& h, long long e, long long* out, cudaStream_t st);
// out[e] (host) = [[F]] at subs[e, :] (host, n x order column-major, validated by the caller) for column-major
// factors fac[d] (device, rows[d] x R, leading dimension rows[d]), in the caller's order.  Synchronous on `st`.
void model_at_host(int order, int R, const double* const* fac, const long long* rows, long long n, const long long* subs,
                   double* out, cudaStream_t st);

}  // namespace aoadmm
