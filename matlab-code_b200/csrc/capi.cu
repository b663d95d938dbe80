// capi.cu - extern "C" boundary (include/aoadmm.h).  No C++ exception crosses the ABI: every entry point
// converts failures into an aoadmm_status and records a message retrievable with aoadmm_last_error().
#include <algorithm>
#include <cstring>
#include <exception>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "engine.h"

struct aoadmm_handle {
  std::vector<aoadmm::Engine*> eng;   // one per GPU driven by this handle (rank order)
  std::string err;
  ~aoadmm_handle() {
    for (auto* e : eng) delete e;
  }
};

namespace aoadmm {
void nccl_unique_id(uint8_t id[128]);
}

namespace {
std::string g_create_error;
std::mutex g_mu;

template <typename F>
int guard(aoadmm_handle* h, F&& fn) {
  try {
    fn();
    return AOADMM_OK;
  } catch (const aoadmm::CudaError& e) {
    if (h) h->err = e.what(); else { std::lock_guard<std::mutex> l(g_mu); g_create_error = e.what(); }
    cudaGetLastError();
    return e.code;
  } catch (const std::bad_alloc&) {
    if (h) h->err = "host allocation failed"; else { std::lock_guard<std::mutex> l(g_mu); g_create_error = "host allocation failed"; }
    return AOADMM_ERR_OOM;
  } catch (const std::exception& e) {
    if (h) h->err = e.what(); else { std::lock_guard<std::mutex> l(g_mu); g_create_error = e.what(); }
    return AOADMM_ERR_INVALID_ARG;
  }
}

// fn(rank) for rank = 0..n-1: inline for one GPU, else one worker thread per GPU (the engine methods are host-blocking:
// they synchronise their stream once per outer iteration).  Every worker runs to completion; the first failure (in
// rank order) is rethrown on the caller's thread.  Replicated state makes data-dependent failures identical on all ranks.
template <typename F>
void for_each_rank(int n, F&& fn) {
  if (n == 1) {
    fn(0);
    return;
  }
  std::vector<std::exception_ptr> errs(n);
  std::vector<std::thread> th;
  th.reserve(n);
  for (int r = 0; r < n; ++r)
    th.emplace_back([&, r] {
      try {
        fn(r);
      } catch (...) {
        errs[r] = std::current_exception();
      }
    });
  for (auto& t : th) t.join();
  for (int r = 0; r < n; ++r)
    if (errs[r]) std::rethrow_exception(errs[r]);
}

struct DevBuf {
  double* p = nullptr;
  explicit DevBuf(size_t n) { AO_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(double))); }
  ~DevBuf() { if (p) cudaFree(p); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

void select_device(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) throw aoadmm::CudaError(AOADMM_ERR_NO_DEVICE, "no CUDA device available");
  if (device < 0 || device >= n) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "device ordinal out of range");
  AO_CUDA(cudaSetDevice(device));
}
}  // namespace

extern "C" {

int aoadmm_abi_version(void) { return AOADMM_ABI_VERSION; }

int aoadmm_device_count(int* count) {
  if (!count) return AOADMM_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  *count = n;
  return AOADMM_OK;
}

int aoadmm_nccl_unique_id(uint8_t id[128]) {
  if (!id) return AOADMM_ERR_INVALID_ARG;
  return guard(nullptr, [&] { aoadmm::nccl_unique_id(id); });
}

int aoadmm_comm_release(void) {
  return guard(nullptr, [&] { aoadmm::comm_release_all(); });
}

int aoadmm_create(const aoadmm_problem* problem, const aoadmm_dist* dist, aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    h = new aoadmm_handle();
    h->eng.push_back(nullptr);
    h->eng[0] = new aoadmm::Engine(problem, dist);   // a throwing constructor has released everything it acquired
    h->eng[0]->reduce_norms();
  });
  if (rc != AOADMM_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return AOADMM_OK;
}

namespace {

// subscripts of one COO descriptor against the mode sizes of CP object `ob`
void check_coo(const aoadmm_problem* problem, const aoadmm_object& ob, const aoadmm_sparse_object* so,
               const std::string& who) {
  using aoadmm::CudaError;
  if (so->nnz < 0) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "nnz is negative");
  if (so->nnz > 0 && (so->subs == nullptr || so->vals == nullptr))
    throw CudaError(AOADMM_ERR_INVALID_ARG, who + "subs / vals is NULL");
  if (ob.order < 2 || ob.order > 8 || ob.modes == nullptr || problem->mode_rows == nullptr)
    throw CudaError(AOADMM_ERR_INVALID_ARG, who + "order must be in 2..8 with its modes given");
  for (int d = 0; d < ob.order; ++d) {
    const int mid = ob.modes[d];
    if (mid < 1 || mid > problem->nb_modes) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "mode id out of range");
    const int64_t rows = problem->mode_rows[mid - 1];
    if (rows > 0x7fffffffLL) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "a mode has more than 2^31 - 1 rows");
    const int64_t* sd = so->subs + (size_t)d * (size_t)so->nnz;
    for (int64_t e = 0; e < so->nnz; ++e)
      if (sd[e] < 0 || sd[e] >= rows)
        throw CudaError(AOADMM_ERR_INVALID_ARG, who + "subscript " + std::to_string(sd[e]) + " of nonzero " + std::to_string(e) +
                                                    " is out of range for mode position " + std::to_string(d + 1));
  }
}

// every check create_sparse / aoadmm_create_sparse_multi make on the sparse descriptors and masks; touches no device
void check_sparse(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                  const aoadmm_sparse_object* const* masks, const aoadmm_dist* dist) {
  using aoadmm::CudaError;
  if (problem == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "problem is NULL");
  if (problem->n_objects > 0 && problem->objects == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "objects is NULL");
  for (int p = 0; masks != nullptr && p < problem->n_objects; ++p) {
    if (masks[p] == nullptr) continue;
    const std::string who = "sparse mask " + std::to_string(p + 1) + ": ";
    if (sparse == nullptr || sparse[p] == nullptr)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "a sparse mask needs a sparse object (dense objects take Z.miss)");
    if (problem->objects[p].miss != nullptr)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "both a dense Z.miss and a sparse mask are set");
    if (problem->objects[p].model == AOADMM_MODEL_CP) check_coo(problem, problem->objects[p], masks[p], who);
  }
  for (int p = 0; sparse != nullptr && p < problem->n_objects; ++p) {
    const aoadmm_sparse_object* so = sparse[p];
    if (so == nullptr) continue;
    const aoadmm_object& ob = problem->objects[p];
    const std::string who = "sparse object " + std::to_string(p + 1) + ": ";
    if (dist != nullptr && dist->world_size > 1)
      throw CudaError(AOADMM_ERR_UNSUPPORTED, who + "sparse objects run on one GPU (world_size must be 1)");
    if (ob.model != AOADMM_MODEL_CP) throw CudaError(AOADMM_ERR_UNSUPPORTED, who + "PARAFAC2 objects must be dense");
    if (ob.miss != nullptr) throw CudaError(AOADMM_ERR_UNSUPPORTED, who + "missing-data masks (Z.miss) need a dense object");
    if (ob.data != nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "both dense data and sparse data are set");
    check_coo(problem, ob, so, who);
  }
}

int create_sparse(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                  const aoadmm_sparse_object* const* masks, const aoadmm_dist* dist, aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    check_sparse(problem, sparse, masks, dist);   // every check on the descriptors happens before a device is touched
    h = new aoadmm_handle();
    h->eng.push_back(nullptr);
    h->eng[0] = new aoadmm::Engine(problem, dist, nullptr, sparse, masks);
  });
  if (rc != AOADMM_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return AOADMM_OK;
}

// every check aoadmm_create_sparse_slices makes on the descriptors; touches no device.  slices[p]: the K slices of
// PARAFAC2 object p side by side as one order-2 COO object over I x Jtot (column joff[k] + j of slice k).
void check_sparse_slices(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                         const aoadmm_sparse_object* const* slices, const aoadmm_dist* dist) {
  using aoadmm::CudaError;
  if (problem == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "problem is NULL");
  if (problem->n_objects > 0 && problem->objects == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "objects is NULL");
  for (int p = 0; sparse != nullptr && p < problem->n_objects; ++p)
    if (sparse[p] != nullptr && problem->objects[p].model != AOADMM_MODEL_CP)
      throw CudaError(AOADMM_ERR_INVALID_ARG, "sparse object " + std::to_string(p + 1) +
                                                  ": a PARAFAC2 object takes its sparse data through `slices`");
  check_sparse(problem, sparse, nullptr, dist);
  for (int p = 0; slices != nullptr && p < problem->n_objects; ++p) {
    const aoadmm_sparse_object* so = slices[p];
    if (so == nullptr) continue;
    const aoadmm_object& ob = problem->objects[p];
    const std::string who = "sparse slices of object " + std::to_string(p + 1) + ": ";
    if (ob.model != AOADMM_MODEL_PAR2)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "a CP object takes its sparse data through `sparse`");
    if (dist != nullptr && dist->world_size > 1)
      throw CudaError(AOADMM_ERR_UNSUPPORTED, who + "sparse slices run on one GPU (world_size must be 1)");
    if (ob.miss_slices != nullptr)
      throw CudaError(AOADMM_ERR_UNSUPPORTED, who + "missing-data masks (Z.miss) need dense slices");
    if (ob.slices != nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "both dense slices and sparse slices are set");
    if (so->nnz < 0) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "nnz is negative");
    if (so->nnz >= 0x7fffffffLL - aoadmm::kSparseChunk)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "2^31 - 257 entries or more");
    if (so->nnz > 0 && (so->subs == nullptr || so->vals == nullptr))
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "subs / vals is NULL");
    if (ob.order != 3 || ob.modes == nullptr || problem->mode_rows == nullptr)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "a PARAFAC2 object has three modes (A, B_k, C)");
    for (int d = 0; d < 3; ++d)
      if (ob.modes[d] < 1 || ob.modes[d] > problem->nb_modes) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "mode id out of range");
    const int mb = ob.modes[1] - 1;
    const int K = problem->n_slices != nullptr ? problem->n_slices[mb] : 0;
    const int64_t* jk = problem->slice_rows != nullptr ? problem->slice_rows[mb] : nullptr;
    if (K <= 0 || jk == nullptr)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "missing slice sizes (Z.size of the second mode)");
    const int64_t I = problem->mode_rows[ob.modes[0] - 1];
    int64_t Jtot = 0;
    for (int k = 0; k < K; ++k) {
      if (jk[k] < 0) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "slice " + std::to_string(k + 1) + " has a negative size");
      Jtot += jk[k];
      if (Jtot > 0x7fffffffLL) break;
    }
    if (I < 0 || I > 0x7fffffffLL) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "I must be in 0..2^31 - 1");
    if (Jtot > 0x7fffffffLL) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "the slices have more than 2^31 - 1 columns in all");
    const int64_t ext[2] = {I, Jtot};
    for (int d = 0; d < 2; ++d) {
      const int64_t* sd = so->subs + (size_t)d * (size_t)so->nnz;
      for (int64_t e = 0; e < so->nnz; ++e)
        if (sd[e] < 0 || sd[e] >= ext[d])
          throw CudaError(AOADMM_ERR_INVALID_ARG, who + (d == 0 ? "row" : "column") + " subscript " + std::to_string(sd[e]) +
                                                      " of entry " + std::to_string(e) + " is out of range");
    }
  }
}

// b[0..n]: the nonzero-balanced slab bounds of the last mode (include/aoadmm.h, aoadmm_sparse_shard_bounds).  With the
// last subscripts sorted (s_0 <= s_1 <= ...), C[k] >= t holds exactly for k > s_{t-1}: the smallest k with
// C[k] * n >= r * nnz is s_{t-1} + 1 for t = ceil(r * nnz / n) >= 1 (0 for t = 0).  The order statistics come from
// nth_element on one int32 copy of the last subscripts (4 bytes per nonzero, O(nnz log n) time).
void shard_bounds(const aoadmm_sparse_object* so, int order, int64_t ext, int n, int64_t* b, const std::string& who) {
  using aoadmm::CudaError;
  if (so == nullptr || b == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "NULL descriptor / bounds");
  if (order < 2 || order > 8) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "order must be in 2..8");
  if (n < 1) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "n_gpus must be >= 1");
  if (ext < 0 || ext > 0x7fffffffLL) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "the last mode must have 0..2^31 - 1 indices");
  if (so->nnz < 0) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "nnz is negative");
  if (so->nnz > 0 && so->subs == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, who + "subs is NULL");
  if (ext < n)
    throw CudaError(AOADMM_ERR_INVALID_ARG, who + "the last mode has fewer indices (" + std::to_string(ext) +
                                                ") than there are GPUs");
  const int64_t nnz = so->nnz;
  const int64_t* last = so->subs + (size_t)(order - 1) * (size_t)nnz;
  std::vector<int32_t> v((size_t)nnz);
  for (int64_t e = 0; e < nnz; ++e) {
    if (last[e] < 0 || last[e] >= ext)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "last-mode subscript " + std::to_string(last[e]) + " of nonzero " +
                                                  std::to_string(e) + " is out of range");
    v[e] = (int32_t)last[e];
  }
  b[0] = 0;
  b[n] = ext;
  size_t lo = 0;
  for (int r = 1; r < n; ++r) {
    int64_t k;
    if (nnz == 0) {
      k = ext * r / n;   // the uniform rule of dense slabs
    } else {
      const int64_t t = (r * nnz + n - 1) / n;
      if (t == 0) {
        k = 0;
      } else {
        const size_t at = (size_t)(t - 1);
        if (at >= lo) {
          std::nth_element(v.begin() + lo, v.begin() + at, v.end());
          lo = at;
        }
        k = (int64_t)v[at] + 1;
      }
    }
    b[r] = std::min<int64_t>(std::max<int64_t>(k, b[r - 1] + 1), ext - (n - r));
  }
}

// The slabs of aoadmm_create_multi / aoadmm_create_sparse_multi.  objs[r]: the objects of rank r; a dense CP object
// of order >= 3 is cut into the uniform slabs of its last mode.  sparse != nullptr: a sparse object (any order) is cut
// by shard_bounds and sp[r][p] / mk[r][p] describe rank r's entries of it and of its mask, in a permuted copy of the
// caller's entries (one slab after the other; n == 1 keeps the caller's descriptors).
struct Slabs {
  std::vector<std::vector<aoadmm_object>> objs;
  std::vector<std::vector<aoadmm_sparse_object>> sp, mk;
  std::vector<std::vector<const aoadmm_sparse_object*>> sp_ptr, mk_ptr;
  std::vector<std::vector<int64_t>> subs;   // the permuted copies
  std::vector<std::vector<double>> vals;
};

// rank r's entries of `so` (bounds b of its object's last mode) into out[r]; the copy is kept in sl.subs / sl.vals
void split_entries(Slabs& sl, const aoadmm_sparse_object& so, int order, const std::vector<int64_t>& b, int n,
                   std::vector<aoadmm_sparse_object>& out) {
  const int64_t nnz = so.nnz;
  const int64_t* last = so.subs + (size_t)(order - 1) * (size_t)nnz;
  auto slab_of = [&](int64_t i) { return (int)(std::upper_bound(b.begin() + 1, b.begin() + n, i) - (b.begin() + 1)); };
  std::vector<int64_t> cnt(n, 0), base(n + 1, 0);
  for (int64_t e = 0; e < nnz; ++e) ++cnt[slab_of(last[e])];
  for (int r = 0; r < n; ++r) base[r + 1] = base[r] + cnt[r];
  sl.subs.emplace_back((size_t)nnz * order);
  sl.vals.emplace_back((size_t)nnz);
  int64_t* ps = sl.subs.back().data();
  double* pv = sl.vals.back().data();
  std::vector<int64_t> fill(n, 0);
  for (int64_t e = 0; e < nnz; ++e) {
    const int r = slab_of(last[e]);
    const int64_t j = fill[r]++;
    for (int d = 0; d < order; ++d) ps[base[r] * order + d * cnt[r] + j] = so.subs[(size_t)d * nnz + e];
    pv[base[r] + j] = so.vals[e];
  }
  for (int r = 0; r < n; ++r) {
    out[r].nnz = cnt[r];
    out[r].subs = ps + base[r] * order;
    out[r].vals = pv + base[r];
  }
}

void cut_slabs(const aoadmm_problem* problem, int n_gpus, const aoadmm_sparse_object* const* sparse,
               const aoadmm_sparse_object* const* masks, Slabs& sl) {
  using aoadmm::CudaError;
  if (problem->nb_modes <= 0 || problem->n_objects <= 0 || problem->objects == nullptr || problem->mode_rows == nullptr)
    throw CudaError(AOADMM_ERR_INVALID_ARG, "empty problem");
  const int P = problem->n_objects;
  sl.objs.assign(n_gpus, std::vector<aoadmm_object>(problem->objects, problem->objects + P));
  sl.sp.assign(n_gpus, std::vector<aoadmm_sparse_object>(P));
  sl.mk.assign(n_gpus, std::vector<aoadmm_sparse_object>(P));
  sl.sp_ptr.assign(n_gpus, std::vector<const aoadmm_sparse_object*>(P, nullptr));
  sl.mk_ptr.assign(n_gpus, std::vector<const aoadmm_sparse_object*>(P, nullptr));
  for (int p = 0; p < P; ++p) {
    const aoadmm_object& src = problem->objects[p];
    const bool is_sparse = sparse != nullptr && sparse[p] != nullptr;
    const aoadmm_sparse_object* mask = (is_sparse && masks != nullptr) ? masks[p] : nullptr;
    if (is_sparse && n_gpus == 1) {
      sl.sp_ptr[0][p] = sparse[p];
      sl.mk_ptr[0][p] = mask;
      continue;
    }
    // slabs of the last mode of every >= 3-way dense CP object and every sparse one (column-major: a dense slab is one
    // contiguous range)
    if (src.model != AOADMM_MODEL_CP || (src.order < 3 && !is_sparse) || n_gpus == 1) continue;
    if (src.modes == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "object without modes");
    int64_t lead = 1;
    for (int d = 0; d < src.order; ++d) {
      if (src.modes[d] < 1 || src.modes[d] > problem->nb_modes) throw CudaError(AOADMM_ERR_INVALID_ARG, "mode id out of range");
      if (d + 1 < src.order) lead *= problem->mode_rows[src.modes[d] - 1];
    }
    const int64_t ext = problem->mode_rows[src.modes[src.order - 1] - 1];
    if (src.shard_offset != 0 || (src.shard_extent != ext && src.shard_extent != 0))
      throw CudaError(AOADMM_ERR_INVALID_ARG, "aoadmm_create_multi takes whole objects (shard_offset = 0, shard_extent = size of the last mode)");
    const std::string who = "object " + std::to_string(p + 1) + ": ";
    if (ext < n_gpus)
      throw CudaError(AOADMM_ERR_INVALID_ARG, who + "the last mode has fewer indices (" + std::to_string(ext) +
                                                  ") than there are GPUs");
    std::vector<int64_t> b(n_gpus + 1);
    if (is_sparse) {
      shard_bounds(sparse[p], src.order, ext, n_gpus, b.data(), who);
      std::vector<aoadmm_sparse_object> parts(n_gpus);
      split_entries(sl, *sparse[p], src.order, b, n_gpus, parts);
      for (int r = 0; r < n_gpus; ++r) {
        sl.sp[r][p] = parts[r];
        sl.sp_ptr[r][p] = &sl.sp[r][p];
      }
      if (mask != nullptr) {   // a mask is cut with the object's bounds
        split_entries(sl, *mask, src.order, b, n_gpus, parts);
        for (int r = 0; r < n_gpus; ++r) {
          sl.mk[r][p] = parts[r];
          sl.mk_ptr[r][p] = &sl.mk[r][p];
        }
      }
    } else {
      for (int r = 0; r <= n_gpus; ++r) b[r] = ext * r / n_gpus;
    }
    for (int r = 0; r < n_gpus; ++r) {
      aoadmm_object& o = sl.objs[r][p];
      o.shard_offset = b[r];
      o.shard_extent = b[r + 1] - b[r];
      if (src.data != nullptr) o.data = src.data + lead * b[r];
      if (src.miss != nullptr) o.miss = src.miss + lead * b[r];
    }
  }
}

// devices[r] (NULL: r) of n_gpus GPUs: distinct ordinals of visible devices
std::vector<int> device_list(int32_t n_gpus, const int32_t* devices) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw aoadmm::CudaError(AOADMM_ERR_NO_DEVICE, "no CUDA device available");
  if (n_gpus < 1 || n_gpus > ndev)
    throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "n_gpus must be between 1 and the number of visible devices (" + std::to_string(ndev) + ")");
  std::vector<int> devs(n_gpus);
  for (int r = 0; r < n_gpus; ++r) {
    devs[r] = devices ? devices[r] : r;
    if (devs[r] < 0 || devs[r] >= ndev) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "device ordinal out of range");
    for (int q = 0; q < r; ++q)
      if (devs[q] == devs[r]) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "a device is listed twice");
  }
  return devs;
}

// one engine per GPU, each from its own worker thread; the norms are summed once every constructor has returned
void build_engines(aoadmm_handle* h, const aoadmm_problem* problem, const std::vector<int>& devs, Slabs& sl, bool sparse,
                   bool masked) {
  const int n_gpus = (int)devs.size();
  std::vector<void*> comms(n_gpus, nullptr);
  if (n_gpus > 1) comms = aoadmm::comms_for_devices(devs);
  h->eng.assign(n_gpus, nullptr);
  for_each_rank(n_gpus, [&](int r) {
    aoadmm_problem pr = *problem;
    pr.objects = sl.objs[r].data();
    aoadmm_dist d{};
    d.rank = r;
    d.world_size = n_gpus;
    d.device = devs[r];
    h->eng[r] = new aoadmm::Engine(&pr, &d, comms[r], sparse ? sl.sp_ptr[r].data() : nullptr,
                                   masked ? sl.mk_ptr[r].data() : nullptr);
  });
  for_each_rank(n_gpus, [&](int r) { h->eng[r]->reduce_norms(); });
}

}  // namespace

int aoadmm_create_sparse(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse, const aoadmm_dist* dist,
                         aoadmm_handle** out) {
  return create_sparse(problem, sparse, nullptr, dist, out);
}

int aoadmm_create_sparse_masked(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                                const aoadmm_sparse_object* const* masks, const aoadmm_dist* dist, aoadmm_handle** out) {
  return create_sparse(problem, sparse, masks, dist, out);
}

int aoadmm_create_sparse_slices(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                                const aoadmm_sparse_object* const* slices, const aoadmm_dist* dist, aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    check_sparse_slices(problem, sparse, slices, dist);   // every check on the descriptors happens before a device is touched
    h = new aoadmm_handle();
    h->eng.push_back(nullptr);
    h->eng[0] = new aoadmm::Engine(problem, dist, nullptr, sparse, nullptr, slices);
  });
  if (rc != AOADMM_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return AOADMM_OK;
}

int aoadmm_create_multi(const aoadmm_problem* problem, int32_t n_gpus, const int32_t* devices, aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    if (problem == nullptr) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "problem is NULL");
    const std::vector<int> devs = device_list(n_gpus, devices);
    Slabs sl;
    cut_slabs(problem, n_gpus, nullptr, nullptr, sl);
    h = new aoadmm_handle();
    build_engines(h, problem, devs, sl, false, false);
  });
  if (rc != AOADMM_OK) {
    delete h;   // engines that were built on the other devices go with it
    return rc;
  }
  *out = h;
  return AOADMM_OK;
}

int aoadmm_sparse_shard_bounds(const aoadmm_sparse_object* so, int32_t order, int64_t extent, int32_t n_gpus,
                               int64_t* bounds) {
  return guard(nullptr, [&] { shard_bounds(so, order, extent, n_gpus, bounds, ""); });
}

int aoadmm_create_sparse_multi(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                               const aoadmm_sparse_object* const* masks, int32_t n_gpus, const int32_t* devices,
                               aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    // every check on the arguments that needs no device first, the slabs included
    check_sparse(problem, sparse, masks, nullptr);
    if (n_gpus < 1) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "n_gpus must be >= 1");
    if (devices != nullptr)
      for (int r = 0; r < n_gpus; ++r)
        for (int q = 0; q < r; ++q)
          if (devices[q] == devices[r]) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "a device is listed twice");
    Slabs sl;
    cut_slabs(problem, n_gpus, sparse, masks, sl);
    const std::vector<int> devs = device_list(n_gpus, devices);
    h = new aoadmm_handle();
    build_engines(h, problem, devs, sl, sparse != nullptr, masks != nullptr);
  });
  if (rc != AOADMM_OK) {
    delete h;   // engines that were built on the other devices go with it
    return rc;
  }
  *out = h;
  return AOADMM_OK;
}

int aoadmm_gpu_count(const aoadmm_handle* h, int32_t* n_gpus) {
  if (!h || !n_gpus) return AOADMM_ERR_INVALID_ARG;
  *n_gpus = (int32_t)h->eng.size();
  return AOADMM_OK;
}

int aoadmm_destroy(aoadmm_handle* h) {
  if (!h) return AOADMM_OK;
  delete h;
  return AOADMM_OK;
}

const char* aoadmm_last_error(const aoadmm_handle* h) {
  if (h) return h->err.c_str();
  std::lock_guard<std::mutex> l(g_mu);
  static thread_local std::string copy;
  copy = g_create_error;
  return copy.c_str();
}

int aoadmm_set_state(aoadmm_handle* h, int32_t field, int32_t index, int32_t slice, const double* data, int64_t rows,
                     int64_t cols) {
  if (!h) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    for_each_rank((int)h->eng.size(), [&](int r) { h->eng[r]->set_state(field, index, slice, data, rows, cols); });
  });
}

int aoadmm_get_state(aoadmm_handle* h, int32_t field, int32_t index, int32_t slice, double* data, int64_t rows,
                     int64_t cols) {
  if (!h) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    for_each_rank((int)h->eng.size(), [&](int r) { h->eng[r]->prepare_state_read(); });   // collective (no-op unless stale)
    h->eng[0]->get_state(field, index, slice, data, rows, cols);                            // replicas are identical
  });
}

int aoadmm_run(aoadmm_handle* h, const aoadmm_options* options, aoadmm_out* out) {
  if (!h) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    if (out == nullptr) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "run: NULL options/out");
    const int n = (int)h->eng.size();
    std::vector<aoadmm_out> others(n);   // ranks > 0: scalars only, no history arrays
    for (auto& o : others) std::memset(&o, 0, sizeof(o));
    for_each_rank(n, [&](int r) { h->eng[r]->run(options, r == 0 ? out : &others[r]); });
  });
}

int aoadmm_generate_cp_data(aoadmm_handle* h, int32_t object, const double* const* factors, double noise, uint64_t seed) {
  if (!h || !factors) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    for_each_rank((int)h->eng.size(), [&](int r) { h->eng[r]->generate_cp_data(object, factors, noise, seed); });
  });
}

int aoadmm_get_object_data(aoadmm_handle* h, int32_t object, double* out, int64_t n_elements) {
  if (!h || !out) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    const int n = (int)h->eng.size();
    if (n == 1) {
      h->eng[0]->object_to_host(object, out, n_elements);
      return;
    }
    int64_t total = 0;
    std::vector<int64_t> off(n), cnt(n);
    for (int r = 0; r < n; ++r) {
      h->eng[r]->object_slab(object, &off[r], &cnt[r]);
      total += cnt[r];
    }
    if (total != n_elements) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "get_object_data: size mismatch");
    for_each_rank(n, [&](int r) { h->eng[r]->object_to_host(object, out + off[r], cnt[r]); });
  });
}

int aoadmm_nvecs(aoadmm_handle* h, int32_t mode, int32_t slice, int32_t r, double* out, int64_t rows, double* info) {
  if (!h || !out || r < 1 || rows < 1) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    const int n = (int)h->eng.size();
    std::vector<std::vector<double>> tmp(n);
    for (int q = 1; q < n; ++q) tmp[q].resize((size_t)rows * r);
    for_each_rank(n, [&](int q) { h->eng[q]->nvecs_to_host(mode, slice, r, q == 0 ? out : tmp[q].data(), rows, q == 0 ? info : nullptr); });
  });
}

int aoadmm_nvecs_sparse(aoadmm_handle* h, int32_t mode, int32_t r, double* out, int64_t rows, double* info) {
  if (!h || !out || r < 1 || rows < 1) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    const int n = (int)h->eng.size();
    std::vector<std::vector<double>> tmp(n);
    for (int q = 1; q < n; ++q) tmp[q].resize((size_t)rows * r);
    for_each_rank(n, [&](int q) { h->eng[q]->nvecs_sparse_to_host(mode, r, q == 0 ? out : tmp[q].data(), rows, q == 0 ? info : nullptr); });
  });
}

int aoadmm_object_mttkrp(aoadmm_handle* h, int32_t object, int32_t pos, int32_t precision, double* out) {
  if (!h || !out || precision < 0 || precision > 3) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    const int n = (int)h->eng.size();
    std::vector<std::vector<double>> tmp(n);
    if (n > 1) {
      const int m = h->eng[0]->object_mode(object, pos);
      if (m < 0) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "mttkrp: object / position out of range");
      for (int q = 1; q < n; ++q) tmp[q].resize((size_t)h->eng[0]->mode_rows(m) * h->eng[0]->mode_rank(m));
    }
    for_each_rank(n, [&](int q) { h->eng[q]->mttkrp_to_host(object, pos, q == 0 ? out : tmp[q].data(), precision); });
  });
}

int aoadmm_time_mttkrp(aoadmm_handle* h, int32_t object, int32_t pos, int32_t reps, float* ms_out) {
  if (!h || !ms_out) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    const int n = (int)h->eng.size();
    std::vector<float> ms(n, 0.f);
    for_each_rank(n, [&](int q) { ms[q] = h->eng[q]->time_mttkrp(object, pos, reps); });
    *ms_out = *std::max_element(ms.begin(), ms.end());
  });
}

int aoadmm_model_at(aoadmm_handle* h, int32_t object, const aoadmm_sparse_object* entries, double* out) {
  if (!h) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    if (entries == nullptr || (entries->nnz > 0 && out == nullptr))
      throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "model_at: NULL entries / out");
    h->eng[0]->check_entries(object, entries, false);
    h->eng[0]->model_at(object, entries, out);   // the factors are replicated: device 0 evaluates
  });
}

int aoadmm_set_heldout(aoadmm_handle* h, int32_t object, const aoadmm_sparse_object* entries) {
  if (!h) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    h->eng[0]->check_entries(object, entries, true);   // every rank holds the same objects and modes
    for_each_rank((int)h->eng.size(), [&](int r) { h->eng[r]->set_heldout(object, entries); });
  });
}

int aoadmm_heldout_history(const aoadmm_handle* h, int32_t object, double* sse, int64_t n, int64_t* count) {
  if (!h || n < 0 || (n > 0 && !sse)) return AOADMM_ERR_INVALID_ARG;
  return guard(const_cast<aoadmm_handle*>(h), [&] { h->eng[0]->heldout_history(object, sse, n, count); });
}

int aoadmm_set_heldout_stopping(aoadmm_handle* h, int32_t patience) {
  if (!h || patience < 0) return AOADMM_ERR_INVALID_ARG;
  return guard(h, [&] {
    if (patience > 0 && h->eng[0]->heldout_sets() == 0)
      throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "set_heldout_stopping: no object has a held-out set");
    const int n = (int)h->eng.size();
    try {
      for_each_rank(n, [&](int r) { h->eng[r]->set_heldout_stopping(patience); });
    } catch (...) {   // e.g. OOM on one GPU: stopping stays off everywhere
      for_each_rank(n, [&](int r) { h->eng[r]->set_heldout_stopping(0); });
      throw;
    }
  });
}

int aoadmm_heldout_best(const aoadmm_handle* h, int32_t* iteration, double* sse) {
  if (!h || !iteration || !sse) return AOADMM_ERR_INVALID_ARG;
  return guard(const_cast<aoadmm_handle*>(h), [&] {
    int k = 0;
    h->eng[0]->heldout_best(&k, sse);
    *iteration = k;
  });
}

int aoadmm_launch_count(const aoadmm_handle* h, int64_t* count) {
  if (!h || !count) return AOADMM_ERR_INVALID_ARG;
  int64_t total = 0;
  for (auto* e : h->eng) total += e->launches();
  *count = total;
  return AOADMM_OK;
}

int aoadmm_phase_ms(const aoadmm_handle* h, double ms[3]) {
  if (!h || !ms) return AOADMM_ERR_INVALID_ARG;
  ms[0] = ms[1] = ms[2] = 0.0;
  for (auto* e : h->eng) {   // slowest GPU per phase
    double v[3];
    e->phase_ms(v);
    for (int q = 0; q < 3; ++q) ms[q] = std::max(ms[q], v[q]);
  }
  return AOADMM_OK;
}

int aoadmm_last_run_ms(const aoadmm_handle* h, double* ms) {
  if (!h || !ms) return AOADMM_ERR_INVALID_ARG;
  *ms = 0.0;
  for (auto* e : h->eng) *ms = std::max(*ms, e->last_run_ms());
  return AOADMM_OK;
}

int aoadmm_last_loop_ms(const aoadmm_handle* h, double* ms) {
  if (!h || !ms) return AOADMM_ERR_INVALID_ARG;
  *ms = 0.0;
  for (auto* e : h->eng) *ms = std::max(*ms, e->last_loop_ms());
  return AOADMM_OK;
}

// ---- operator-level entry points ---------------------------------------------------------------
int aoadmm_mttkrp(const double* X, int32_t order, const int64_t* dims, const double* const* factors, int32_t R,
                  int32_t n, double* out, int32_t device) {
  if (!X || !dims || !factors || !out || order < 2 || order > 8 || n < 1 || n > order || R < 1 || R > 256)
    return AOADMM_ERR_INVALID_ARG;
  return guard(nullptr, [&] {
    // a one-object problem driven through the engine so that exactly the production kernels run
    std::vector<int64_t> rows(dims, dims + order);
    std::vector<int32_t> rank(order, R), modes(order), lin(order, 0), constrained(order, 0);
    std::vector<aoadmm_constraint> cons(order);
    std::memset(cons.data(), 0, sizeof(aoadmm_constraint) * order);
    for (int d = 0; d < order; ++d) modes[d] = d + 1;
    aoadmm_object obj{};
    obj.model = AOADMM_MODEL_CP;
    obj.order = order;
    obj.modes = modes.data();
    obj.weight = 1.0;
    obj.znorm_const = 0.0;
    obj.data = X;
    obj.shard_offset = 0;
    obj.shard_extent = dims[order - 1];
    aoadmm_problem pb{};
    pb.nb_modes = order;
    pb.mode_rows = rows.data();
    pb.mode_rank = rank.data();
    pb.n_objects = 1;
    pb.objects = &obj;
    pb.lin_coupled_modes = lin.data();
    pb.n_couplings = 0;
    pb.constrained_modes = constrained.data();
    pb.constraints = cons.data();
    aoadmm_dist dist{};
    dist.rank = 0;
    dist.world_size = 1;
    dist.device = device;
    aoadmm::Engine eng(&pb, &dist);
    for (int d = 0; d < order; ++d) eng.set_state(AOADMM_FIELD_FAC, d + 1, 0, factors[d], dims[d], R);
    eng.mttkrp_to_host(1, n, out);
  });
}

int aoadmm_prox(const aoadmm_constraint* spec, const double* X, int64_t rows, int64_t cols, double rho, double* out,
                int32_t device) {
  if (!spec || !X || !out || rows < 0 || cols < 0 || cols > (1 << 20)) return AOADMM_ERR_INVALID_ARG;
  return guard(nullptr, [&] {
    select_device(device);
    const size_t n = (size_t)rows * cols;
    DevBuf dx(n), dout(n);
    const size_t sb = aoadmm::prox_scratch_bytes(spec->kind, rows, (int)cols);
    DevBuf scratch(sb / sizeof(double) + 1);
    AO_CUDA(cudaMemcpy(dx.p, X, n * sizeof(double), cudaMemcpyHostToDevice));
    if (spec->kind == AOADMM_CON_QUADRATIC) {
      if (spec->matrix_n != rows) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "quadratic regularization: L must be rows x rows");
      aoadmm::QuadProx q;
      aoadmm::quad_prox_setup(q, spec->matrix, rows, spec->p0, (int)cols, 0);
      aoadmm::quad_prox_apply(q, dx.p, rows, dout.p, rows, (int)cols, nullptr, rho, 0, nullptr);
      AO_CUDA(cudaDeviceSynchronize());
      aoadmm::quad_prox_free(q);
      AO_CUDA(cudaMemcpy(out, dout.p, n * sizeof(double), cudaMemcpyDeviceToHost));
      return;
    }
    if (spec->kind == AOADMM_CON_TPARAFAC2)
      throw aoadmm::CudaError(AOADMM_ERR_UNSUPPORTED, "tPARAFAC2 acts on all PARAFAC2 slices at once: use the solver");
    aoadmm::prox_apply(spec->kind, spec->p0, spec->p1, dx.p, rows, dout.p, rows, rows, (int)cols, nullptr, rho,
                       sb ? scratch.p : nullptr, 0, nullptr);
    AO_CUDA(cudaDeviceSynchronize());
    AO_CUDA(cudaMemcpy(out, dout.p, n * sizeof(double), cudaMemcpyDeviceToHost));
  });
}

int aoadmm_chol_solve(const double* B, int32_t R, const double* A, int64_t rows, double* X, int32_t device) {
  if (!B || !A || !X || R < 1 || R > 256 || rows < 0) return AOADMM_ERR_INVALID_ARG;
  return guard(nullptr, [&] {
    select_device(device);
    const size_t RR = (size_t)R * R, n = (size_t)rows * R;
    DevBuf dB(RR), dC(RR), dBo(RR), dL(RR), dinv(R), drho(1), dA(n), dX(n);
    DevBuf ones(RR);
    aoadmm::InnerCtl* ctl = nullptr;
    AO_CUDA(cudaMalloc(&ctl, sizeof(aoadmm::InnerCtl)));
    AO_CUDA(cudaMemset(ctl, 0, sizeof(aoadmm::InnerCtl)));
    AO_CUDA(cudaMemcpy(dB.p, B, RR * sizeof(double), cudaMemcpyHostToDevice));
    AO_CUDA(cudaMemcpy(dA.p, A, n * sizeof(double), cudaMemcpyHostToDevice));
    aoadmm::PrepArgs a{};
    a.had[0] = dB.p;
    a.nhad = 1;
    a.R = R;
    a.weight = 1.0;
    a.rho_scale = 1.0;
    a.do_chol = 1;
    a.C = dC.p;
    a.B = dBo.p;
    a.L = dL.p;
    a.invdiag = dinv.p;
    a.rho = drho.p;
    a.ctl = ctl;
    aoadmm::prep_system(a, 0, nullptr);
    aoadmm::ls_solve(dA.p, rows, dL.p, dinv.p, dX.p, rows, rows, R, ctl, 0, nullptr);
    AO_CUDA(cudaDeviceSynchronize());
    aoadmm::InnerCtl hc;
    AO_CUDA(cudaMemcpy(&hc, ctl, sizeof(hc), cudaMemcpyDeviceToHost));
    cudaFree(ctl);
    if (hc.err != 0) throw aoadmm::CudaError(AOADMM_ERR_NOT_POSITIVE_DEFINITE, "matrix is not positive definite");
    AO_CUDA(cudaMemcpy(X, dX.p, n * sizeof(double), cudaMemcpyDeviceToHost));
  });
}

int aoadmm_gram(const double* F, int64_t rows, int32_t R, double* G, int32_t device) {
  if (!F || !G || R < 1 || R > 256 || rows < 0) return AOADMM_ERR_INVALID_ARG;
  return guard(nullptr, [&] {
    select_device(device);
    const size_t n = (size_t)rows * R;
    DevBuf dF(n), dG((size_t)R * R), ws(aoadmm::gram_ws_doubles(rows, R));
    AO_CUDA(cudaMemcpy(dF.p, F, n * sizeof(double), cudaMemcpyHostToDevice));
    aoadmm::gram(dF.p, rows, rows, R, dG.p, ws.p, 0, nullptr);
    AO_CUDA(cudaDeviceSynchronize());
    AO_CUDA(cudaMemcpy(G, dG.p, (size_t)R * R * sizeof(double), cudaMemcpyDeviceToHost));
  });
}

}  // extern "C"
