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

int create_sparse(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                  const aoadmm_sparse_object* const* masks, const aoadmm_dist* dist, aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    using aoadmm::CudaError;
    if (problem == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "problem is NULL");
    if (problem->n_objects > 0 && problem->objects == nullptr) throw CudaError(AOADMM_ERR_INVALID_ARG, "objects is NULL");
    // every check on the sparse descriptors and masks happens here, before a device is touched
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

}  // namespace

int aoadmm_create_sparse(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse, const aoadmm_dist* dist,
                         aoadmm_handle** out) {
  return create_sparse(problem, sparse, nullptr, dist, out);
}

int aoadmm_create_sparse_masked(const aoadmm_problem* problem, const aoadmm_sparse_object* const* sparse,
                                const aoadmm_sparse_object* const* masks, const aoadmm_dist* dist, aoadmm_handle** out) {
  return create_sparse(problem, sparse, masks, dist, out);
}

int aoadmm_create_multi(const aoadmm_problem* problem, int32_t n_gpus, const int32_t* devices, aoadmm_handle** out) {
  if (!out) return AOADMM_ERR_INVALID_ARG;
  *out = nullptr;
  aoadmm_handle* h = nullptr;
  int rc = guard(nullptr, [&] {
    if (problem == nullptr) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "problem is NULL");
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
    if (problem->nb_modes <= 0 || problem->n_objects <= 0 || problem->objects == nullptr || problem->mode_rows == nullptr)
      throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "empty problem");
    // slabs of the last mode of every >= 3-way CP object (column-major: a slab is one contiguous range)
    std::vector<std::vector<aoadmm_object>> objs(n_gpus, std::vector<aoadmm_object>(problem->objects, problem->objects + problem->n_objects));
    for (int p = 0; p < problem->n_objects; ++p) {
      const aoadmm_object& src = problem->objects[p];
      if (src.model != AOADMM_MODEL_CP || src.order < 3 || n_gpus == 1) continue;
      if (src.modes == nullptr) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "object without modes");
      int64_t lead = 1;
      for (int d = 0; d < src.order; ++d) {
        if (src.modes[d] < 1 || src.modes[d] > problem->nb_modes) throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "mode id out of range");
        if (d + 1 < src.order) lead *= problem->mode_rows[src.modes[d] - 1];
      }
      const int64_t ext = problem->mode_rows[src.modes[src.order - 1] - 1];
      if (src.shard_offset != 0 || (src.shard_extent != ext && src.shard_extent != 0))
        throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "aoadmm_create_multi takes whole objects (shard_offset = 0, shard_extent = size of the last mode)");
      if (ext < n_gpus)
        throw aoadmm::CudaError(AOADMM_ERR_INVALID_ARG, "object " + std::to_string(p + 1) + ": the last mode has fewer indices (" +
                                                           std::to_string(ext) + ") than there are GPUs");
      for (int r = 0; r < n_gpus; ++r) {
        const int64_t lo = ext * r / n_gpus, hi = ext * (r + 1) / n_gpus;
        aoadmm_object& o = objs[r][p];
        o.shard_offset = lo;
        o.shard_extent = hi - lo;
        if (src.data != nullptr) o.data = src.data + lead * lo;
        if (src.miss != nullptr) o.miss = src.miss + lead * lo;
      }
    }
    std::vector<void*> comms(n_gpus, nullptr);
    if (n_gpus > 1) comms = aoadmm::comms_for_devices(devs);
    h = new aoadmm_handle();
    h->eng.assign(n_gpus, nullptr);
    for_each_rank(n_gpus, [&](int r) {
      aoadmm_problem pr = *problem;
      pr.objects = objs[r].data();
      aoadmm_dist d{};
      d.rank = r;
      d.world_size = n_gpus;
      d.device = devs[r];
      h->eng[r] = new aoadmm::Engine(&pr, &d, comms[r]);
    });
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
