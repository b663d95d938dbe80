// engine.cu - the AO-ADMM outer loop on device-resident state.
//
// Control flow mirrors functions/cmtf_fun_AOADMM.m:
//   :10        couplings = unique(lin_coupled_modes)  (0 = uncoupled modes first)
//   :62-81     initial Grams
//   :87-476    outer loop: per coupling id -> per object -> per mode precompute (MTTKRP, Hadamard, rho, B, chol),
//              uncoupled modes updated immediately (LS :134 or ADMM_constrained_only :144), coupled groups
//              updated jointly after all their precomputes (ADMM_coupled_case0 :277)
//   :447-456   objective (shortcut :1235-1241) + evaluate_stopping_conditions.m:8-44
//   :478       make_exit_flag.m:4-29
// All numerics run in the kernels of mttkrp.cu / smallops.cu / prox.cu; this file only sequences launches and
// does the scalar bookkeeping the reference does in MATLAB scalars.
#include "engine.h"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <thread>

namespace aoadmm {

// ---------------------------------------------------------------------------------------------------
// NCCL through dlopen (only needed when world_size > 1)
// ---------------------------------------------------------------------------------------------------
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  // point-to-point exchange of tensor slabs (nvecs of the sharded mode)
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
};

NcclApi* load_nccl() {
  static NcclApi api;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (api.lib != nullptr) return &api;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  if (!api.lib) throw CudaError(6, std::string("cannot dlopen libnccl.so.2: ") + dlerror());
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.lib, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.lib, "ncclCommInitRank"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(api.lib, "ncclAllReduce"));
  api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(dlsym(api.lib, "ncclCommInitAll"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.lib, "ncclCommDestroy"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.lib, "ncclGetErrorString"));
  api.Send = reinterpret_cast<decltype(api.Send)>(dlsym(api.lib, "ncclSend"));
  api.Recv = reinterpret_cast<decltype(api.Recv)>(dlsym(api.lib, "ncclRecv"));
  api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(dlsym(api.lib, "ncclGroupStart"));
  api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(dlsym(api.lib, "ncclGroupEnd"));
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy)
    throw CudaError(6, "libnccl.so.2 lacks required symbols");
  return &api;
}

void nccl_unique_id(uint8_t id[128]) {
  NcclApi* api = load_nccl();
  ncclUniqueId uid;
  ncclResult_t r = api->GetUniqueId(&uid);
  if (r != ncclSuccess) throw CudaError(6, "ncclGetUniqueId failed");
  std::memcpy(id, uid.internal, 128);
}

// ---------------------------------------------------------------------------------------------------
// Process-wide communicator cache.  Creating a communicator costs seconds at 8 ranks (bootstrap + the connection set-up
// of the first collective), far more than a solve of a resident problem, so communicators outlive the handles:
//   * one process per GPU (aoadmm_dist): the 128-byte unique id is the key - a handle created with an id that was
//     used before in this process gets the same communicator (every rank must then reuse it, which holds when all
//     ranks pass the same id again);
//   * one process driving several GPUs (aoadmm_create_multi): the device list is the key (ncclCommInitAll).
// A fresh communicator runs one small all-reduce so that the first timed collective does not pay the lazy set-up.
// Released by aoadmm_comm_release() or at process exit.
// ---------------------------------------------------------------------------------------------------
namespace {
struct CommCache {
  std::mutex mu;
  std::map<std::string, ncclComm_t> by_uid;                       // key: 128-byte id + rank + world
  std::map<std::vector<int>, std::vector<ncclComm_t>> by_devices;
};
CommCache& comm_cache() {
  static CommCache c;
  return c;
}
void warm_up_comm(NcclApi* api, ncclComm_t comm, cudaStream_t st) {
  double* buf = nullptr;
  AO_CUDA(cudaMalloc(&buf, 256 * sizeof(double)));
  AO_CUDA(cudaMemsetAsync(buf, 0, 256 * sizeof(double), st));
  const ncclResult_t r = api->AllReduce(buf, buf, 256, ncclDouble, ncclSum, comm, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(buf);
  if (r != ncclSuccess) throw CudaError(6, std::string("NCCL warm-up all-reduce: ") + (api->GetErrorString ? api->GetErrorString(r) : "error"));
  AO_CUDA(e);
}
}  // namespace

// communicator of (unique id, rank, world) - created on first use, cached afterwards
void* comm_for_unique_id(const uint8_t id[128], int rank, int world, cudaStream_t st) {
  NcclApi* api = load_nccl();
  std::string key(reinterpret_cast<const char*>(id), 128);
  key += "/" + std::to_string(rank) + "/" + std::to_string(world);
  CommCache& c = comm_cache();
  {
    std::lock_guard<std::mutex> lock(c.mu);
    auto it = c.by_uid.find(key);
    if (it != c.by_uid.end()) return it->second;
  }
  ncclUniqueId uid;
  std::memcpy(uid.internal, id, 128);
  ncclComm_t comm = nullptr;
  const ncclResult_t r = api->CommInitRank(&comm, world, uid, rank);
  if (r != ncclSuccess) throw CudaError(6, std::string("ncclCommInitRank: ") + (api->GetErrorString ? api->GetErrorString(r) : "error"));
  warm_up_comm(api, comm, st);
  std::lock_guard<std::mutex> lock(c.mu);
  c.by_uid[key] = comm;
  return comm;
}

// communicators of a single-process device group (one per device, in the order of `devices`)
std::vector<void*> comms_for_devices(const std::vector<int>& devices) {
  NcclApi* api = load_nccl();
  if (!api->CommInitAll) throw CudaError(6, "libnccl.so.2 lacks ncclCommInitAll");
  CommCache& c = comm_cache();
  std::lock_guard<std::mutex> lock(c.mu);
  auto it = c.by_devices.find(devices);
  if (it == c.by_devices.end()) {
    std::vector<ncclComm_t> comms(devices.size(), nullptr);
    const ncclResult_t r = api->CommInitAll(comms.data(), (int)devices.size(), devices.data());
    if (r != ncclSuccess) throw CudaError(6, std::string("ncclCommInitAll: ") + (api->GetErrorString ? api->GetErrorString(r) : "error"));
    // warm-up: every rank must enter the collective, so issue them as one group from this thread
    std::vector<double*> bufs(devices.size(), nullptr);
    std::vector<cudaStream_t> sts(devices.size(), nullptr);
    int prev = 0;
    cudaGetDevice(&prev);
    bool ok = true;
    for (size_t i = 0; i < devices.size() && ok; ++i) {
      ok = cudaSetDevice(devices[i]) == cudaSuccess && cudaStreamCreateWithFlags(&sts[i], cudaStreamNonBlocking) == cudaSuccess &&
           cudaMalloc(&bufs[i], 256 * sizeof(double)) == cudaSuccess &&
           cudaMemsetAsync(bufs[i], 0, 256 * sizeof(double), sts[i]) == cudaSuccess;
    }
    if (ok && api->GroupStart && api->GroupEnd) {
      api->GroupStart();
      for (size_t i = 0; i < devices.size(); ++i)
        ok = ok && api->AllReduce(bufs[i], bufs[i], 256, ncclDouble, ncclSum, comms[i], sts[i]) == ncclSuccess;
      ok = (api->GroupEnd() == ncclSuccess) && ok;
    }
    for (size_t i = 0; i < devices.size(); ++i) {
      cudaSetDevice(devices[i]);
      if (sts[i]) {
        ok = (cudaStreamSynchronize(sts[i]) == cudaSuccess) && ok;
        cudaStreamDestroy(sts[i]);
      }
      if (bufs[i]) cudaFree(bufs[i]);
    }
    cudaSetDevice(prev);
    if (!ok) {
      for (auto cm : comms)
        if (cm) api->CommDestroy(cm);
      cudaGetLastError();
      throw CudaError(6, "NCCL warm-up all-reduce over the device group failed");
    }
    it = c.by_devices.emplace(devices, comms).first;
  }
  return std::vector<void*>(it->second.begin(), it->second.end());
}

void comm_release_all() {
  CommCache& c = comm_cache();
  std::lock_guard<std::mutex> lock(c.mu);
  NcclApi* api = nullptr;
  try {
    api = load_nccl();
  } catch (...) {
    return;
  }
  for (auto& kv : c.by_uid) api->CommDestroy(kv.second);
  for (auto& kv : c.by_devices)
    for (auto cm : kv.second) api->CommDestroy(cm);
  c.by_uid.clear();
  c.by_devices.clear();
}

#define AO_NCCL(expr)                                                                                 \
  do {                                                                                                \
    ncclResult_t _r = (expr);                                                                         \
    if (_r != ncclSuccess)                                                                            \
      throw CudaError(6, std::string(#expr) + ": " +                                                 \
                             (nccl_->GetErrorString ? nccl_->GetErrorString(_r) : "nccl error"));     \
  } while (0)

// ---------------------------------------------------------------------------------------------------
// small utility kernels
// ---------------------------------------------------------------------------------------------------
namespace {

__global__ void axpy_kernel(double* __restrict__ y, const double* __restrict__ x, double alpha, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = y[i] + alpha * x[i];
}

// dense Khatri-Rao: out(a + rows_a*b, r) = Fa(a,r) * Fb(b,r); rows a >= valid_a are zero
__global__ void kr_dense_kernel(double* __restrict__ out, const double* __restrict__ Fa, long long rows_a,
                                long long valid_a, long long lda, const double* __restrict__ Fb, long long rows_b,
                                long long ldb, int R) {
  const long long rows = rows_a * rows_b, n = rows * R;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx / rows, row = idx % rows;
    const long long a = row % rows_a, b = row / rows_a;
    out[idx] = (a < valid_a) ? Fa[r * lda + a] * Fb[r * ldb + b] : 0.0;
  }
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// counter-based N(0,1): hash(seed, global element index) -> Box-Muller
__device__ __forceinline__ double normal_at(uint64_t seed, uint64_t idx) {
  const uint64_t h1 = splitmix64(seed ^ (idx * 0xD1342543DE82EF95ull));
  const uint64_t h2 = splitmix64(h1 ^ 0xA5A5A5A5A5A5A5A5ull);
  const double u1 = ((double)(h1 >> 11) + 1.0) * (1.0 / 9007199254740993.0);
  const double u2 = (double)(h2 >> 11) * (1.0 / 9007199254740992.0);
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

struct GenArgs {
  int order, R;
  long long dims[8];        // local dims
  long long full_last;      // unsharded extent of the last mode
  long long shard_offset;
  long long ld0;
  const double* fac[8];     // device factor matrices (full rows), leading dimension = rows
  long long fld[8];
};

// mode 0: sums[0] += x0^2, sums[1] += n^2 ; mode 1: x = x0 + sigma*n, sums[2] += x^2 ; mode 2: x *= scale
__global__ void gen_cp_kernel(GenArgs g, double* __restrict__ X, uint64_t seed, int pass, double sigma, double scale,
                              double* __restrict__ sums) {
  __shared__ double red[32];
  long long n = 1;
  for (int d = 0; d < g.order; ++d) n *= g.dims[d];
  double s0 = 0.0, s1 = 0.0;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
       idx += (long long)gridDim.x * blockDim.x) {
    long long rem = idx, sub[8];
    for (int d = 0; d < g.order; ++d) {
      sub[d] = rem % g.dims[d];
      rem /= g.dims[d];
    }
    long long addr = sub[0], mult = g.ld0, gidx = sub[0], gmult = g.dims[0];
    for (int d = 1; d < g.order; ++d) {
      addr += sub[d] * mult;
      mult *= g.dims[d];
      const long long gs = (d == g.order - 1) ? sub[d] + g.shard_offset : sub[d];
      gidx += gs * gmult;
      gmult *= (d == g.order - 1) ? g.full_last : g.dims[d];
    }
    if (pass == 2) {
      X[addr] *= scale;
      continue;
    }
    double x0 = 0.0;
    for (int r = 0; r < g.R; ++r) {
      double t = 1.0;
      for (int d = 0; d < g.order; ++d) {
        const long long row = (d == g.order - 1) ? sub[d] + g.shard_offset : sub[d];
        t *= g.fac[d][(long long)r * g.fld[d] + row];
      }
      x0 += t;
    }
    const double nz = normal_at(seed, (uint64_t)gidx);
    if (pass == 0) {
      s0 = fma(x0, x0, s0);
      s1 = fma(nz, nz, s1);
    } else {
      const double x = x0 + sigma * nz;
      X[addr] = x;
      s0 = fma(x, x, s0);
    }
  }
  if (pass == 2) return;
  s0 = block_sum(s0, red);
  s1 = block_sum(s1, red);
  // per-CTA partials, summed in CTA order by gen_sum_kernel: the generated tensor is bit-reproducible
  if (threadIdx.x == 0) {
    sums[4 + 2 * blockIdx.x] = s0;
    sums[4 + 2 * blockIdx.x + 1] = s1;
  }
}

// sums[dst0] (and sums[dst0 + 1] when two) = fixed-order sums of the per-CTA partials stored behind sums[4]
__global__ void gen_sum_kernel(double* __restrict__ sums, int ctas, int dst0, int two) {
  __shared__ double red[32];
  double a = 0.0, b = 0.0;
  for (int c = threadIdx.x; c < ctas; c += blockDim.x) {
    a += sums[4 + 2 * c];
    b += sums[4 + 2 * c + 1];
  }
  a = block_sum(a, red);
  b = block_sum(b, red);
  if (threadIdx.x == 0) {
    sums[dst0] = a;
    if (two) sums[dst0 + 1] = b;
  }
}

// Host -> device copy of a large contiguous buffer.  Page-locked sources go down in one DMA (about 55 GB/s on this
// pool); pageable sources (MATLAB arrays, plain malloc) would be staged by the driver at about 11 GB/s, so they are
// staged here instead: a few worker threads copy interleaved 8 MB chunks into their own pinned buffers and issue the
// DMA of each chunk on their own stream while the next chunk is being copied (profiles/r01_h2d_probe.log).
void h2d_copy_large(void* dst, const void* src, size_t bytes, int device) {
  constexpr size_t kChunk = 8u << 20;
  cudaPointerAttributes attr{};
  const bool pinned = (cudaPointerGetAttributes(&attr, src) == cudaSuccess) &&
                      (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
  cudaGetLastError();  // an unregistered host pointer may leave cudaErrorInvalidValue behind on old drivers
  if (pinned || bytes < 8 * kChunk) {
    AO_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return;
  }
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const int T = (int)std::min<size_t>(std::min<unsigned>(8u, std::max(2u, hw / 2)), bytes / kChunk);
  const size_t nchunks = (bytes + kChunk - 1) / kChunk;
  std::vector<cudaError_t> status(T, cudaSuccess);
  char* staging = nullptr;  // one page-locked block: two chunks per worker
  if (cudaHostAlloc(reinterpret_cast<void**>(&staging), (size_t)T * 2 * kChunk, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();   // no page-locked memory to spare: let the driver stage the copy
    AO_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return;
  }
  auto worker = [&](int t) {
    cudaError_t e = cudaSetDevice(device);
    void* buf[2] = {staging + ((size_t)t * 2) * kChunk, staging + ((size_t)t * 2 + 1) * kChunk};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    cudaStream_t st = nullptr;
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    for (int b = 0; b < 2 && e == cudaSuccess; ++b) e = cudaEventCreateWithFlags(&ev[b], cudaEventDisableTiming);
    int use = 0;
    for (size_t c = t; c < nchunks && e == cudaSuccess; c += T, use ^= 1) {
      const size_t off = c * kChunk, n = std::min(kChunk, bytes - off);
      e = cudaEventSynchronize(ev[use]);  // the DMA that last read this staging buffer has finished
      if (e != cudaSuccess) break;
      std::memcpy(buf[use], static_cast<const char*>(src) + off, n);
      e = cudaMemcpyAsync(static_cast<char*>(dst) + off, buf[use], n, cudaMemcpyHostToDevice, st);
      if (e == cudaSuccess) e = cudaEventRecord(ev[use], st);
    }
    if (st != nullptr) {
      const cudaError_t e2 = cudaStreamSynchronize(st);
      if (e == cudaSuccess) e = e2;
    }
    for (int b = 0; b < 2; ++b)
      if (ev[b]) cudaEventDestroy(ev[b]);
    if (st) cudaStreamDestroy(st);
    status[t] = e;
  };
  std::vector<std::thread> th;
  for (int t = 0; t < T; ++t) th.emplace_back(worker, t);
  for (auto& x : th) x.join();
  cudaFreeHost(staging);
  for (int t = 0; t < T; ++t)
    if (status[t] != cudaSuccess)
      throw CudaError(status[t] == cudaErrorMemoryAllocation ? 7 : 5,
                      std::string("host->device copy of the tensor: ") + cudaGetErrorString(status[t]));
}

double now_s() {
  using namespace std::chrono;
  return duration_cast<duration<double>>(steady_clock::now().time_since_epoch()).count();
}

bool constraint_supported(int kind) {
  switch (kind) {
    case AOADMM_CON_NONE:
    case AOADMM_CON_NONNEG:
    case AOADMM_CON_BOX:
    case AOADMM_CON_SIMPLEX_COL:
    case AOADMM_CON_SIMPLEX_ROW:
    case AOADMM_CON_NONDECREASING:
    case AOADMM_CON_NONINCREASING:
    case AOADMM_CON_UNIMODAL:
    case AOADMM_CON_L1_BALL:
    case AOADMM_CON_L2_BALL:
    case AOADMM_CON_NONNEG_L2_BALL:
    case AOADMM_CON_NONNEG_L2_SPHERE:
    case AOADMM_CON_L1_REG:
    case AOADMM_CON_L0_REG:
    case AOADMM_CON_L2_REG:
    case AOADMM_CON_RIDGE:
    case AOADMM_CON_GL_SMOOTH:
    case AOADMM_CON_TV:
    case AOADMM_CON_ORTHONORMAL:
    case AOADMM_CON_QUADRATIC:
    case AOADMM_CON_TPARAFAC2: return true;
    default: return false;
  }
}

}  // namespace

void dev_alloc(DevMat& m, int64_t rows, int64_t cols) {
  m.rows = rows;
  m.cols = cols;
  if (rows * cols > 0) {
    AO_CUDA(cudaMalloc(&m.p, m.bytes()));
    AO_CUDA(cudaMemset(m.p, 0, m.bytes()));
    // the engine stream is non-blocking: legacy-stream memsets must have landed before it touches the buffer
    AO_CUDA(cudaStreamSynchronize(0));
  }
}
void dev_free(DevMat& m) {
  if (m.p) cudaFree(m.p);
  m.p = nullptr;
}

// reg_func of constraints_to_prox.m:49,:53,:57,:61,:77,:81 as a reduction kind (-1: the constraint has no regulariser value)
static int reg_red_kind(int con_kind) {
  switch (con_kind) {
    case AOADMM_CON_L1_REG: return RED_L1;
    case AOADMM_CON_L0_REG: return RED_NNZ;
    case AOADMM_CON_L2_REG: return RED_COLNORM;
    case AOADMM_CON_RIDGE: return RED_NORM2;
    case AOADMM_CON_GL_SMOOTH: return RED_GLQUAD;
    case AOADMM_CON_TV: return RED_TVSUM;
    case AOADMM_CON_TPARAFAC2: return RED_TSMOOTH;   // t_smoothness_penalty.m:5-9 (only through par2_seg_norms)
    default: return -1;
  }
}

struct Engine::ObjTerms {
  struct PerObject {
    int idx_dot = -1, idx_had = -1;
  };
  struct PerMode {
    int idx_norm2 = -1, idx_diffZ = -1, idx_diffD = -1, idx_reg = -1, idx_normG = -1;
  };
  std::vector<PerObject> obj;
  std::vector<PerMode> mode;
};

// ---------------------------------------------------------------------------------------------------
// construction
// ---------------------------------------------------------------------------------------------------
Engine::Engine(const aoadmm_problem* prob, const aoadmm_dist* dist, void* shared_comm,
               const aoadmm_sparse_object* const* sparse, const aoadmm_sparse_object* const* masks) {
  // A constructor that throws never runs the destructor: everything acquired so far (up to the whole tensor in HBM,
  // streams, events, pinned buffers) is released here before the error leaves.
  try {
    construct(prob, dist, shared_comm, sparse, masks);
  } catch (...) {
    release();
    throw;
  }
}

void Engine::construct(const aoadmm_problem* prob, const aoadmm_dist* dist, void* shared_comm,
                       const aoadmm_sparse_object* const* sparse, const aoadmm_sparse_object* const* masks) {
  if (prob == nullptr) throw CudaError(1, "problem is NULL");
  if (dist != nullptr) {
    rank_ = dist->rank;
    world_ = dist->world_size;
    device_ = dist->device;
    if (world_ < 1 || rank_ < 0 || rank_ >= world_) throw CudaError(1, "invalid rank/world_size");
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw CudaError(8, "no CUDA device available");
  if (device_ >= ndev) throw CudaError(1, "device ordinal out of range");
  AO_CUDA(cudaSetDevice(device_));
  AO_CUDA(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
  AO_CUDA(cudaStreamCreateWithFlags(&st2_, cudaStreamNonBlocking));
  AO_CUDA(cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming));
  AO_CUDA(cudaEventCreateWithFlags(&ev_join_, cudaEventDisableTiming));
  if (world_ > 1) {
    // the communicator first: a problem that is rejected below is rejected on every rank alike (the problem struct is
    // the same everywhere), so no rank is left waiting inside ncclCommInitRank for a peer that already gave up
    nccl_ = load_nccl();
    comm_ = shared_comm != nullptr ? shared_comm : comm_for_unique_id(dist->nccl_unique_id, rank_, world_, st_);
  }

  nb_modes_ = prob->nb_modes;
  n_objects_ = prob->n_objects;
  n_couplings_ = prob->n_couplings;
  if (nb_modes_ <= 0 || n_objects_ <= 0) throw CudaError(1, "empty problem");
  has_ridge_ = prob->ridge != nullptr;
  coupling_type_.assign(prob->coupling_type, prob->coupling_type + n_couplings_);
  lin_groups_.resize(n_couplings_);

  modes_.resize(nb_modes_);
  for (int i = 0; i < nb_modes_; ++i) {
    ModeState& m = modes_[i];
    m.id = i + 1;
    m.rows = prob->mode_rows[i];
    m.R = prob->mode_rank[i];
    m.coupling = prob->lin_coupled_modes[i];
    m.constrained = prob->constrained_modes[i] != 0;
    m.con = prob->constraints[i];
    if (!m.constrained) m.con.kind = AOADMM_CON_NONE;
    m.ridge = has_ridge_ ? prob->ridge[i] : 0.0;
    if (m.coupling < 0 || m.coupling > n_couplings_) throw CudaError(1, "lin_coupled_modes out of range");
    if (m.constrained && !constraint_supported(m.con.kind))
      throw CudaError(2, "constraint kind " + std::to_string(m.con.kind) + " of mode " + std::to_string(m.id) +
                             " is not supported on device");
    if (m.R <= 0 || m.R > 256) throw CudaError(1, "rank must be in 1..256");
  }

  objects_.resize(n_objects_);
  for (int p = 0; p < n_objects_; ++p) {
    const aoadmm_object& src = prob->objects[p];
    ObjectState& o = objects_[p];
    o.model = src.model;
    o.order = src.order;
    if (o.model != AOADMM_MODEL_CP && o.model != AOADMM_MODEL_PAR2) throw CudaError(1, "unknown object model");
    if (o.order < 2 || o.order > 8) throw CudaError(1, "object order must be in 2..8");
    o.modes.assign(src.modes, src.modes + o.order);
    o.weight = src.weight;
    o.znorm = src.znorm_const;
    if (o.model == AOADMM_MODEL_PAR2) {
      setup_par2(prob, p);
      continue;
    }
    int R = 0;
    for (int d = 0; d < o.order; ++d) {
      const int mid = o.modes[d];
      if (mid < 1 || mid > nb_modes_) throw CudaError(1, "mode id out of range");
      ModeState& m = mode(mid);
      if (m.p != -1) throw CudaError(1, "mode " + std::to_string(mid) + " belongs to two objects");
      m.p = p;
      m.pos = d;
      if (d == 0) R = m.R;
      if (m.R != R) throw CudaError(1, "all modes of a CP object need the same rank");
      o.dims.push_back(m.rows);
    }
    o.last_full = o.dims.back();
    const bool is_sparse = sparse != nullptr && sparse[p] != nullptr;
    // dense matrices are replicated; tensors and sparse objects of any order hold one slab of their last mode
    o.sharded = (world_ > 1 && (o.order >= 3 || is_sparse));
    if (o.sharded) {
      o.shard_offset = src.shard_offset;
      o.shard_extent = src.shard_extent;
      if (o.shard_offset < 0 || o.shard_extent < 0 || o.shard_offset + o.shard_extent > o.last_full)
        throw CudaError(1, "invalid shard range");
    } else {
      o.shard_offset = 0;
      o.shard_extent = o.last_full;
    }
    o.dims.back() = o.shard_extent;
    if (is_sparse) {
      // sparse CP object (aoadmm_create_sparse, or this GPU's slab from aoadmm_create_sparse_multi): no dense mask;
      // sorted device copies instead of a dense array.  A sparse mask (aoadmm_create_sparse_masked) must mark exactly
      // the stored entries; EM state in o.sp.
      if (src.miss != nullptr || src.data != nullptr) throw CudaError(2, "sparse object: unsupported combination");
      const aoadmm_sparse_object& so = *sparse[p];
      const aoadmm_sparse_object* mk = masks != nullptr ? masks[p] : nullptr;
      std::vector<long long> dl(o.dims.begin(), o.dims.end());
      dl.back() = o.last_full;
      o.sp = new SparseTensor();
      try {
        sparse_build(*o.sp, o.order, dl.data(), o.shard_offset, o.shard_extent, R, so.nnz,
                     reinterpret_cast<const long long*>(so.subs), so.vals, st_, mk != nullptr, mk ? mk->nnz : 0,
                     mk ? reinterpret_cast<const long long*>(mk->subs) : nullptr, mk ? mk->vals : nullptr);
      } catch (const CudaError& e) {
        throw CudaError(e.code, "sparse object " + std::to_string(p + 1) + ": " + e.what());
      }
      if (mk != nullptr) has_missing_ = true;
      continue;
    }
    o.ld0 = round_up(o.dims[0], 2);
    size_t slab = 1;
    for (int d = 1; d < o.order; ++d) slab *= (size_t)o.dims[d];
    const size_t bytes = std::max<size_t>((size_t)o.ld0 * slab * sizeof(double), 256);
    AO_CUDA(cudaMalloc(&o.data, bytes));
    if (o.ld0 != o.dims[0] || src.data == nullptr) AO_CUDA(cudaMemset(o.data, 0, bytes));
    if (src.data != nullptr && slab > 0) {
      // no padding: one linear copy (a pitched copy of narrow rows runs at ~2/3 of the PCIe rate, profiles/r01_h2d_probe.log)
      if (o.ld0 == o.dims[0])
        h2d_copy_large(o.data, src.data, (size_t)o.dims[0] * slab * 8, device_);
      else
        AO_CUDA(cudaMemcpy2D(o.data, (size_t)o.ld0 * 8, src.data, (size_t)o.dims[0] * 8, (size_t)o.dims[0] * 8, slab,
                             cudaMemcpyHostToDevice));
    }
    if (src.miss != nullptr) {  // Z.miss{p} (cmtf_AOADMM.m:68-121)
      if (o.order > 8) throw CudaError(2, "missing data is supported for objects with up to 8 modes");
      if (src.data == nullptr) throw CudaError(1, "Z.miss without data");
      const size_t mbytes = std::max<size_t>((size_t)o.ld0 * slab, 256);
      AO_CUDA(cudaMalloc(&o.mask, mbytes));
      AO_CUDA(cudaMemset(o.mask, 0, mbytes));
      if (slab > 0)
        AO_CUDA(cudaMemcpy2D(o.mask, (size_t)o.ld0, src.miss, (size_t)o.dims[0], (size_t)o.dims[0], slab,
                             cudaMemcpyHostToDevice));
      has_missing_ = true;
    }
    if (o.order == 2 && o.mask == nullptr && o.dims[0] >= 1 && o.dims[1] >= 1 &&
        ceil_div(o.dims[1], 32) <= 65535 &&   // grid.y of the transpose
        (size_t)o.dims[0] * (size_t)o.dims[1] * 8 <= ((size_t)2 << 30)) {
      // second copy of a (small) matrix, transposed; a failed allocation just keeps the single-copy path
      o.ldT = round_up(o.dims[1], 2);
      if (cudaMalloc(&o.dataT, (size_t)o.ldT * (size_t)o.dims[0] * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        o.dataT = nullptr;
      } else {
        AO_CUDA(cudaDeviceSynchronize());   // the upload above (null stream) before the kernel on the engine's stream
        AO_CUDA(cudaMemsetAsync(o.dataT, 0, (size_t)o.ldT * (size_t)o.dims[0] * sizeof(double), st_));
        refresh_transposed(o);
      }
    }
    AO_CUDA(cudaDeviceSynchronize());  // pageable H2D copies return before the DMA has finished
  }
  for (auto& m : modes_) {
    if (m.p < 0) throw CudaError(1, "mode " + std::to_string(m.id) + " belongs to no object");
    if (!m.constrained) continue;
    if (m.con.kind == AOADMM_CON_TPARAFAC2) {  // cmtf_AOADMM.m:33-41
      if (m.par2_role != 2)
        throw CudaError(1, "The tPARAFAC2 constraint can only be imposed on the second mode of a PARAFAC2 model");
      const Par2State& s = par2_[m.par2];
      for (int k = 0; k < s.K; ++k)
        if (s.joff[k + 1] - s.joff[k] != s.Jmax) throw CudaError(1, "tPARAFAC2 needs slices of equal size");
    }
    if (m.con.kind == AOADMM_CON_QUADRATIC) {
      int64_t nq = m.rows;
      if (m.par2_role == 2) {
        // one L for every slice (constraints_to_prox.m:60-66 applied to G.fac{m}{k}, :567-568): regular slices only
        const Par2State& s = par2_[m.par2];
        nq = s.joff[1] - s.joff[0];
        for (int k = 0; k < s.K; ++k)
          if (s.joff[k + 1] - s.joff[k] != nq)
            throw CudaError(1, "quadratic regularization on the second PARAFAC2 mode needs slices of equal size");
      }
      if (m.con.matrix_n != nq) throw CudaError(1, "quadratic regularization: L must be rows x rows");
      quad_prox_setup(m.quad, m.con.matrix, nq, m.con.p0, m.R, st_);
      m.con.matrix = nullptr;  // the host buffer belongs to the caller
    }
  }

  // couplings: exact coupling needs identical shapes
  delta_.resize(n_couplings_);
  for (int c = 1; c <= n_couplings_; ++c) {
    if (coupling_type_[c - 1] != 0) {
      setup_linear_coupling(prob, c);
      continue;
    }
    int first = -1;
    for (auto& m : modes_)
      if (m.coupling == c) {
        if (first < 0) first = m.id;
        if (m.par2_role == 2) throw CudaError(1, "the second PARAFAC2 mode cannot be coupled (cmtf_fun_AOADMM.m:191)");
        if (m.rows != mode(first).rows || m.R != mode(first).R)
          throw CudaError(1, "exactly coupled modes need identical factor shapes");
      }
    if (first < 0) throw CudaError(1, "coupling id without modes");
    dev_alloc(delta_[c - 1], mode(first).rows, mode(first).R);
  }

  // per-mode buffers
  size_t gram_ws = 0, admm_ws = 0, prox_bytes = 0;
  for (auto& m : modes_) {
    dev_alloc(m.fac, m.rows, m.R);
    if (m.constrained) {
      dev_alloc(m.Z, m.rows, m.R);
      dev_alloc(m.muZ, m.rows, m.R);
      if (!prox_is_elementwise(m.con.kind)) {
        dev_alloc(m.Znew, m.rows, m.R);
        dev_alloc(m.V, m.rows, m.R);
        prox_bytes = std::max(prox_bytes, prox_scratch_bytes(m.con.kind, m.rows, m.R));
        if (m.par2_role == 2 && prox_supports_segments(m.con.kind)) {
          const Par2State& s = par2_[m.par2];
          prox_bytes = std::max(prox_bytes, prox_segments_scratch_bytes(m.con.kind, s.Jmax, m.R, s.K));
        }
      }
    }
    if (m.coupling != 0 && m.lin < 0) dev_alloc(m.muD, m.rows, m.R);  // linear couplings: allocated with their own shape
    dev_alloc(m.A, m.rows, m.R);
    dev_alloc(m.Alast, m.rows, m.R);
    dev_alloc(m.C, m.R, m.R);
    dev_alloc(m.B, m.R, m.R);
    dev_alloc(m.L, m.R, m.R);
    dev_alloc(m.Binv, m.R, m.R);
    dev_alloc(m.Btmp, m.R, m.R);
    dev_alloc(m.GtG, m.R, m.R);
    AO_CUDA(cudaMalloc(&m.invdiag, sizeof(double) * m.R));
    AO_CUDA(cudaMalloc(&m.rho, sizeof(double)));
    AO_CUDA(cudaMemset(m.rho, 0, sizeof(double)));
    gram_ws = std::max(gram_ws, gram_ws_doubles(m.rows, m.R));
    admm_ws = std::max(admm_ws, admm_ws_doubles(m.rows, m.R, kMaxGroup));
  }
  for (int c = 1; c <= n_couplings_; ++c)
    if (coupling_type_[c - 1] != 0) lin_build_jobs(c);
  AO_CUDA(cudaMalloc(&gram_ws_, gram_ws * sizeof(double)));
  AO_CUDA(cudaMalloc(&admm_partials_, admm_ws * sizeof(double)));
  AO_CUDA(cudaMalloc(&admm_sums_, (6 * kMaxGroup + 1) * sizeof(double)));
  AO_CUDA(cudaMemset(admm_sums_, 0, (6 * kMaxGroup + 1) * sizeof(double)));
  AO_CUDA(cudaMalloc(&admm_counter_, 2 * sizeof(unsigned)));   // [0] arrival counter, [1] generation of the inner-loop barrier
  AO_CUDA(cudaMemset(admm_counter_, 0, 2 * sizeof(unsigned)));
  if (prox_bytes > 0) AO_CUDA(cudaMalloc(&prox_scratch_, prox_bytes));

  // control blocks: one per mode (a coupled group uses the block of its first mode)
  n_ctl_ = nb_modes_;
  AO_CUDA(cudaMalloc(&ctl_dev_, sizeof(InnerCtl) * n_ctl_));
  AO_CUDA(cudaMemset(ctl_dev_, 0, sizeof(InnerCtl) * n_ctl_));
  AO_CUDA(cudaMallocHost(&ctl_host_, sizeof(InnerCtl) * n_ctl_));
  std::memset(ctl_host_, 0, sizeof(InnerCtl) * n_ctl_);
  for (auto& m : modes_) {
    int owner = m.id;
    if (m.coupling != 0)
      for (auto& q : modes_)
        if (q.coupling == m.coupling) {
          owner = q.id;
          break;
        }
    m.ctl_index = owner - 1;
    m.ctl = ctl_dev_ + m.ctl_index;
  }

  // views + workspaces
  size_t ws_bytes = 0, kr_doubles = 0;
  size_t cp0 = 0;
  for (auto& s : par2_) ws_bytes = std::max(ws_bytes, mttkrp_workspace_bytes(s.view, s.R));
  for (auto& o : objects_) {
    if (o.model == AOADMM_MODEL_PAR2) continue;
    cp0 = std::max(cp0, (size_t)mode(o.modes[0]).rows * mode(o.modes[0]).R);
    if (o.sp != nullptr) continue;   // sparse objects own their scratch (sparse_build)
    build_views(o);
    for (auto& v : o.views) {
      ws_bytes = std::max(ws_bytes, mttkrp_workspace_bytes(v.t, mode(o.modes[0]).R));
      if (v.f0_modes.size() >= 2) kr_doubles = std::max(kr_doubles, (size_t)v.f0_rows * mode(o.modes[0]).R);
      if (v.f1_modes.size() >= 2) kr_doubles = std::max(kr_doubles, (size_t)v.f1_rows * mode(o.modes[0]).R);
    }
  }
  mws_.ws_bytes = ws_bytes;
  AO_CUDA(cudaMalloc(&mws_.ws, ws_bytes));
  if (kr_doubles > 0) {
    krtmp_doubles_ = kr_doubles;
    AO_CUDA(cudaMalloc(&krtmp_[0], kr_doubles * sizeof(double)));
    AO_CUDA(cudaMalloc(&krtmp_[1], kr_doubles * sizeof(double)));
  }
  AO_CUDA(cudaMalloc(&cp0_tmp_, (cp0 + 4 * 256 * 256 + 512 + 148 * 8 + 8) * sizeof(double)));
  // Znorm_const on device where the caller passed NaN (cmtf_AOADMM.m:124-156)
  for (int p = 0; p < n_objects_; ++p) {
    ObjectState& o = objects_[p];
    if (!std::isnan(o.znorm)) continue;
    double* part = cp0_tmp_;
    double* res = cp0_tmp_ + 148 * 8;
    if (o.model == AOADMM_MODEL_PAR2) {
      Par2State& s = par2_[mode(o.modes[0]).par2];
      launches_ += object_norm2(s.X_alloc, s.mask_alloc, s.I, s.ldX, s.jhi - s.jlo, part, res, st_);
    } else if (o.sp != nullptr) {
      launches_ += sparse_norm2(*o.sp, st_);
      res = o.sp->norm_out;
    } else {
      size_t slab = 1;
      for (int d = 1; d < o.order; ++d) slab *= (size_t)o.dims[d];
      if (o.data == nullptr) throw CudaError(1, "Znorm_const = NaN needs the object data");
      launches_ += object_norm2(o.data, o.mask, o.dims[0], o.ld0, (long long)slab, part, res, st_);
    }
    AO_CUDA(cudaMemcpyAsync(&o.znorm, res, sizeof(double), cudaMemcpyDeviceToHost, st_));
    AO_CUDA(cudaStreamSynchronize(st_));
    // partial norm of this rank's slab / slices: summed by reduce_norms
    o.znorm_pending_allreduce = o.model == AOADMM_MODEL_PAR2 ? par2_[mode(o.modes[0]).par2].sharded : o.sharded;
  }
  AO_CUDA(cudaDeviceSynchronize());

  // static sweep order -> last updated mode of every object (cmtf_fun_AOADMM.m:121-123)
  {
    std::set<int> cset;
    for (auto& m : modes_) cset.insert(m.coupling);
    for (int cid : cset) {
      std::set<int> ps;
      for (auto& m : modes_)
        if (m.coupling == cid) ps.insert(m.p);
      for (int p : ps)
        for (auto& m : modes_)
          if (m.coupling == cid && m.p == p) objects_[p].last_m = m.id;
    }
  }
  build_objective_jobs();
  if (has_missing_) {
    AO_CUDA(cudaMalloc(&em_sums_, sizeof(double) * 5 * n_objects_));
    AO_CUDA(cudaMemset(em_sums_, 0, sizeof(double) * 5 * n_objects_));
    AO_CUDA(cudaMallocHost(&em_sums_host_, sizeof(double) * 5 * n_objects_));
    size_t need = 0;
    for (int p = 0; p < n_objects_; ++p) {
      ObjectState& o = objects_[p];
      EmArgs a{};
      a.R = mode(o.modes[0]).R;
      if (o.model == AOADMM_MODEL_PAR2) {
        const Par2State& s = par2_[mode(o.modes[0]).par2];
        if (s.mask == nullptr) continue;
        a.I = s.I;
        a.J = s.Jtot;
        a.K = 1;
      } else {
        if (o.mask == nullptr) continue;
        a.I = o.dims[0];
        a.J = o.dims[1];
        long long kk = 1;
        for (int d = 2; d < o.order; ++d) kk *= o.dims[d];
        if (kk > 0x7fffffffLL) throw CudaError(2, "missing data: trailing extent too large");
        a.K = (int)kk;
        if (o.order > 3) AO_CUDA(cudaMalloc(&o.em_kr, std::max<size_t>((size_t)kk * a.R * sizeof(double), 256)));
        if (o.order >= 3) AO_CUDA(cudaMalloc(&o.em_fkT, std::max<size_t>(em_fkT_doubles(kk, a.R) * sizeof(double), 256)));
      }
      need = std::max(need, em_partials_doubles(a));
    }
    AO_CUDA(cudaMalloc(&em_partials_, std::max<size_t>(need, 8) * sizeof(double)));
  }
  AO_CUDA(cudaDeviceSynchronize());
}

// The only collective of creation.  It runs after every rank's constructor has returned, so a rank whose slab fails
// to build (a sparse mask that does not match inside it) never leaves the others waiting in an all-reduce.
void Engine::reduce_norms() {
  if (world_ <= 1) return;
  AO_CUDA(cudaSetDevice(device_));
  for (auto& o : objects_)
    if (o.znorm_pending_allreduce) {  // partial norms of the slabs -> norm of the whole tensor
      AO_CUDA(cudaMemcpyAsync(cp0_tmp_, &o.znorm, sizeof(double), cudaMemcpyHostToDevice, st_));
      allreduce(cp0_tmp_, 1);
      AO_CUDA(cudaMemcpyAsync(&o.znorm, cp0_tmp_, sizeof(double), cudaMemcpyDeviceToHost, st_));
      AO_CUDA(cudaStreamSynchronize(st_));
      o.znorm_pending_allreduce = false;
    }
}

Engine::~Engine() { release(); }

// frees every device / pinned resource; safe on a partially constructed engine and idempotent
void Engine::release() {
  cudaSetDevice(device_);
  if (st_) cudaStreamSynchronize(st_);
  if (st2_) cudaStreamSynchronize(st2_);
  cudaGetLastError();
  comm_ = nullptr;   // communicators belong to the process-wide cache (comm_for_unique_id / comms_for_devices)
  free_snapshot();
  auto dfree = [](auto*& p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  auto hfree = [](auto*& p) {
    if (p) cudaFreeHost(p);
    p = nullptr;
  };
  for (auto& m : modes_) {
    for (DevMat* d : {&m.fac, &m.Z, &m.muZ, &m.muD, &m.A, &m.Alast, &m.C, &m.B, &m.L, &m.Binv, &m.Btmp, &m.GtG, &m.Znew, &m.V}) dev_free(*d);
    dfree(m.invdiag);
    dfree(m.rho);
    quad_prox_free(m.quad);
  }
  modes_.clear();
  for (auto& o : objects_) {
    if (o.ho != nullptr) {
      heldout_free(*o.ho);
      delete o.ho;
      o.ho = nullptr;
    }
    if (o.sp != nullptr) {
      sparse_free(*o.sp);
      delete o.sp;
      o.sp = nullptr;
    }
    dfree(o.data);
    dfree(o.dataT);
    dfree(o.Tbuf);
    dfree(o.mask);
    dfree(o.em_kr);
    dfree(o.em_fkT);
    for (auto& v : o.views) {
      if (v.f0_own) packed_factor_free(v.f0);
      if (v.f1_own) packed_factor_free(v.f1);
    }
  }
  objects_.clear();
  for (auto& d : delta_) dev_free(d);
  delta_.clear();
  free_linear_coupling();
  lin_modes_.clear();
  lin_groups_.clear();
  for (auto& s : par2_) {
    for (DevMat* d : {&s.W, &s.T, &s.P, &s.muDB, &s.DeltaB, &s.PDold, &s.gM, &s.gS}) dev_free(*d);
    for (void* q : {(void*)s.joff_dev, (void*)s.seg_dev, (void*)s.X_alloc, (void*)s.mask_alloc, (void*)s.redbuf, (void*)s.G2, (void*)s.Binv2, (void*)s.Binv3,
                    (void*)s.rho2, (void*)s.rho3, (void*)s.tdiag, (void*)s.contrib, (void*)s.Vprev, (void*)s.sysws, (void*)s.norms, (void*)s.Csum, (void*)s.segn,
                    (void*)s.res_partials})
      if (q) cudaFree(q);
    if (s.segn_host) cudaFreeHost(s.segn_host);
    packed_factor_free(s.fW);
    packed_factor_free(s.fA);
    packed_factor_free(s.ones);
  }
  par2_.clear();
  dfree(mws_.ws);
  tc_operand_free(tc_op_);
  dfree(gram_ws_);
  dfree(admm_partials_);
  dfree(admm_sums_);
  dfree(admm_counter_);
  dfree(prox_scratch_);
  dfree(krtmp_[0]);
  dfree(krtmp_[1]);
  dfree(ctl_dev_);
  dfree(jobs_dev_);
  dfree(red_dev_);
  dfree(red_partials_);
  dfree(cp0_tmp_);
  dfree(em_sums_);
  dfree(em_partials_);
  hfree(em_sums_host_);
  dfree(ho_sse_);
  hfree(ho_sse_host_);
  hfree(ctl_host_);
  hfree(red_host_);
  for (auto& e : run_ev_) {
    if (e) cudaEventDestroy(e);
    e = nullptr;
  }
  for (auto& e : ev_pool_) {
    cudaEventDestroy(e.first);
    cudaEventDestroy(e.second);
  }
  ev_pool_.clear();
  if (ev_fork_) cudaEventDestroy(ev_fork_);
  if (ev_join_) cudaEventDestroy(ev_join_);
  ev_fork_ = ev_join_ = nullptr;
  if (st2_) cudaStreamDestroy(st2_);
  if (st_) cudaStreamDestroy(st_);
  st_ = st2_ = nullptr;
  cudaGetLastError();
}

namespace {
// out (cols x rows, leading dimension ldo) = in' (in: rows x cols, leading dimension ldi); 32 x 32 tiles through shared memory
__global__ void __launch_bounds__(256) transpose_ld_kernel(const double* __restrict__ in, long long rows, long long cols,
                                                            long long ldi, double* __restrict__ out, long long ldo) {
  __shared__ double tile[32][33];
  const long long r0 = (long long)blockIdx.x * 32, c0 = (long long)blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int q = ty; q < 32; q += 8) {
    const long long r = r0 + tx, c = c0 + q;
    tile[q][tx] = (r < rows && c < cols) ? in[r + ldi * c] : 0.0;
  }
  __syncthreads();
  for (int q = ty; q < 32; q += 8) {
    const long long c = c0 + tx, r = r0 + q;
    if (r < rows && c < cols) out[c + ldo * r] = tile[tx][q];
  }
}
}  // namespace

// (re)build the transposed copy of a matrix object after its data changed
void Engine::refresh_transposed(ObjectState& o) {
  if (o.dataT == nullptr) return;
  dim3 grid((unsigned)ceil_div(o.dims[0], 32), (unsigned)ceil_div(o.dims[1], 32));
  transpose_ld_kernel<<<grid, 256, 0, st_>>>(o.data, o.dims[0], o.dims[1], o.ld0, o.dataT, o.ldT);
  AO_CHECK_LAUNCH();
  ++launches_;
}

void Engine::build_views(ObjectState& o) {
  const int N = o.order;
  const int R = mode(o.modes[0]).R;
  o.views.resize(N);
  auto prod = [&](int a, int b) {  // product of local dims[a..b]
    int64_t v = 1;
    for (int d = a; d <= b; ++d) v *= o.dims[d];
    return v;
  };
  for (int n = 0; n < N; ++n) {
    View3& v = o.views[n];
    int64_t I, J, K, ldI;
    const double* base = o.data;
    if (N == 2 && n == 1 && o.dataT != nullptr) {
      // mode 2 of a matrix from its transposed copy: out(j,:) = sum_i Yt(j,i) F1(i,:) - the contiguous-mode (LEAD) form
      base = o.dataT;
      I = o.dims[1];
      J = o.dims[0];
      K = 1;
      ldI = o.ldT;
      v.kernel_pos = 0;
      v.f0_modes = {o.modes[0]};
      v.f1_modes = {};
    } else if (N == 2) {
      I = o.dims[0];
      J = o.dims[1];
      K = 1;
      ldI = o.ld0;
      v.kernel_pos = (n == 0) ? 0 : 1;
      v.f0_modes = {o.modes[n == 0 ? 1 : 0]};
      v.f1_modes = {};
    } else if (n == 0 || n == N - 1) {
      I = o.dims[0];
      J = prod(1, N - 2);
      K = o.dims[N - 1];
      ldI = o.ld0;
      v.kernel_pos = (n == 0) ? 0 : 2;
      std::vector<int> mid(o.modes.begin() + 1, o.modes.begin() + N - 1);
      if (n == 0) {
        v.f0_modes = mid;
        v.f1_modes = {o.modes[N - 1]};
      } else {
        v.f0_modes = {o.modes[0]};
        v.f1_modes = mid;
      }
    } else {
      I = (n == 1) ? o.dims[0] : o.ld0 * prod(1, n - 1);
      ldI = (n == 1) ? o.ld0 : I;
      J = o.dims[n];
      K = prod(n + 1, N - 1);
      v.kernel_pos = 1;
      v.f0_modes.assign(o.modes.begin(), o.modes.begin() + n);
      v.f1_modes.assign(o.modes.begin() + n + 1, o.modes.end());
    }
    make_tensor3(v.t, base, I, J, K, ldI);
    auto rows_of = [&](const std::vector<int>& ms, bool padded_first) {
      int64_t r = 1;
      for (size_t q = 0; q < ms.size(); ++q) {
        const ModeState& mm = mode(ms[q]);
        int64_t rr = o.dims[mm.pos];
        if (q == 0 && padded_first && mm.pos == 0 && ms.size() > 1) rr = o.ld0;
        r *= rr;
      }
      return r;
    };
    v.f0_rows = rows_of(v.f0_modes, true);
    v.f1_rows = rows_of(v.f1_modes, false);
    packed_factor_alloc(v.f0, v.f0_rows, R);
    v.f0_own = true;
    packed_factor_alloc(v.f1, v.f1_rows, R);
    v.f1_own = true;
    if (v.f1_modes.empty()) {
      packed_factor_pack(v.f1, nullptr, 1, st_, nullptr);  // ones row (matrices: K = 1)
      ++launches_;
    }
    const bool last = (N >= 3 && n == N - 1);
    v.out_rows = last ? o.shard_extent : mode(o.modes[n]).rows;
    v.out_offset = last ? o.shard_offset : 0;
    v.needs_allreduce = o.sharded;
  }
}

// pack operand `which` (0/1) of a view from the current factor matrices
void Engine::pack_operand(View3& v, int which) {
  const std::vector<int>& ms = which == 0 ? v.f0_modes : v.f1_modes;
  PackedFactor& pf = which == 0 ? v.f0 : v.f1;
  if (ms.empty()) return;  // ones, packed once
  ObjectState& o = objects_[mode(ms[0]).p];
  auto fac_ptr = [&](const ModeState& mm) {  // local slice of the (possibly sharded) last mode
    return (mm.pos == o.order - 1) ? mm.fac.p + o.shard_offset : mm.fac.p;
  };
  auto local_rows = [&](const ModeState& mm) { return o.dims[mm.pos]; };
  if (ms.size() == 1) {
    const ModeState& mm = mode(ms[0]);
    packed_factor_pack(pf, fac_ptr(mm), mm.rows, st_, nullptr);
    ++launches_;
    return;
  }
  // Khatri-Rao chain, first listed mode varies fastest
  const ModeState& m0 = mode(ms[0]);
  const bool pad0 = (which == 0 && m0.pos == 0);
  int64_t rows_a = pad0 ? o.ld0 : local_rows(m0);
  int64_t valid_a = local_rows(m0);
  const double* Fa = fac_ptr(m0);
  int64_t lda = m0.rows;
  const int R = m0.R;
  for (size_t q = 1; q < ms.size(); ++q) {
    const ModeState& mb = mode(ms[q]);
    const bool final_step = (q + 1 == ms.size());
    if (final_step && q == 1 && !pad0) {
      packed_factor_pack_kr(pf, Fa, rows_a, lda, fac_ptr(mb), local_rows(mb), mb.rows, st_, nullptr);
      ++launches_;
      return;
    }
    double* dst = krtmp_[(q - 1) & 1];
    const int64_t rows_b = local_rows(mb);
    const long long n = rows_a * rows_b * R;
    const unsigned ctas = (unsigned)std::min<long long>(ceil_div(n, 256), 148 * 8);
    kr_dense_kernel<<<ctas, 256, 0, st_>>>(dst, Fa, rows_a, valid_a, lda, fac_ptr(mb), rows_b, mb.rows, R);
    AO_CHECK_LAUNCH();
    ++launches_;
    Fa = dst;
    rows_a = rows_a * rows_b;
    valid_a = rows_a;
    lda = rows_a;
  }
  packed_factor_pack(pf, Fa, lda, st_, nullptr);
  ++launches_;
}

void Engine::allreduce(double* buf, size_t count) {
  if (world_ <= 1) return;
  AO_NCCL(nccl_->AllReduce(buf, buf, count, ncclDouble, ncclSum, static_cast<ncclComm_t>(comm_), st_));
}

// sparse objects: always FP64, no dimension tree (options.mttkrp_precision / dimtree apply to dense objects only); the
// pass over this GPU's nonzeros
int Engine::sparse_mttkrp_of(ObjectState& o, int pos, double scale, double* out, int64_t ldout, bool imputed) {
  const double* fac[8];
  long long ld[8];
  for (int d = 0; d < o.order; ++d) {
    const ModeState& mm = mode(o.modes[d]);
    fac[d] = mm.fac.p;
    ld[d] = mm.rows;
  }
  return sparse_mttkrp(*o.sp, pos, fac, ld, scale, out, ldout, st_, imputed);
}

void Engine::compute_mttkrp(ObjectState& o, int pos, double scale, double* out, int64_t ldout, bool imputed) {
  if (o.sp != nullptr) {
    phase_begin(o.order >= 3 ? 0 : 1);
    const int R = o.sp->R;
    // a slab writes the rows of its last-mode indices only: the others must be zero for the all-reduce
    if (o.sharded && pos == o.order - 1) AO_CUDA(cudaMemsetAsync(out, 0, (size_t)ldout * R * sizeof(double), st_));
    launches_ += sparse_mttkrp_of(o, pos, scale, out, ldout, imputed);
    if (o.sharded) allreduce(out, (size_t)ldout * R);
    // the low-rank term reads replicated state only: added once, after the all-reduce
    if (imputed && sparse_masked(o)) launches_ += sparse_lowrank_add(*o.sp, pos, scale, out, ldout, st_);
    phase_end();
    return;
  }
  View3& v = o.views[pos];
  const int R = mode(o.modes[0]).R;
  const bool last_sharded = o.sharded && o.order >= 3 && pos == o.order - 1;
  // dimension tree (3-way CP objects): the mode-2 pass also emits T = X x_1 F1; while F1 is unchanged the mode-3
  // MTTKRP is a cheap pass over T instead of a third pass over the tensor.
  const bool tree = opt_.dimtree != 0 && o.order == 3;
  const uint64_t v1 = mode(o.modes[0]).version;
  if (tree && pos == 2 && o.Tbuf != nullptr && o.T_version == v1) {
    phase_begin(0);
    if (last_sharded) AO_CUDA(cudaMemsetAsync(out, 0, (size_t)ldout * R * sizeof(double), st_));
    const ModeState& mj = mode(o.modes[1]);
    launches_ += mttkrp3_from_T(v.t, o.Tbuf, R, mj.fac.p, mj.rows, scale, out + v.out_offset, ldout, st_, nullptr);
    if (v.needs_allreduce) allreduce(out, (size_t)ldout * R);
    phase_end();
    return;
  }
  double* emit = nullptr;
  if (tree && pos == 1) {
    if (o.Tbuf == nullptr) AO_CUDA(cudaMalloc(&o.Tbuf, mttkrp_T_bytes(v.t, R)));
    emit = o.Tbuf;
    o.T_version = v1;
  }
  const int prec = opt_.mttkrp_precision;
  if ((prec == 1 || prec == 2) && o.order == 3) {
    // opt-in reduced precision (3-way tensors): tcgen05 / TMEM kernels straight from the column-major factors
    phase_begin(0);
    if (last_sharded) AO_CUDA(cudaMemsetAsync(out, 0, (size_t)ldout * R * sizeof(double), st_));
    launches_ += tc_mttkrp(o, pos, scale, out + v.out_offset, ldout, emit, prec);
    if (v.needs_allreduce) allreduce(out, (size_t)ldout * R);
    phase_end();
    return;
  }
  const int legacy = (prec == 3 && o.order >= 3) ? 1 : 0;   // 3: the TF32 mma.sync variant of the DMMA kernels
  pack_operand(v, 0);
  pack_operand(v, 1);
  if (legacy) {
    packed_factor_to_tf32(v.f0, st_, nullptr);
    ++launches_;
  }
  phase_begin(o.order >= 3 ? 0 : 1);
  if (last_sharded) AO_CUDA(cudaMemsetAsync(out, 0, (size_t)ldout * R * sizeof(double), st_));
  launches_ += mttkrp3(v.t, v.kernel_pos, v.f0, v.f1, R, scale, out + v.out_offset, ldout, mws_, st_, nullptr, emit, legacy);
  if (v.needs_allreduce) allreduce(out, (size_t)ldout * R);
  phase_end();
}

// reduced-precision MTTKRP of a 3-way object (mttkrp_tc.cu): the contracted factor F0 and the epilogue factor Fe per mode
int Engine::tc_mttkrp(ObjectState& o, int pos, double scale, double* out, int64_t ldout, double* emit, int prec) {
  View3& v = o.views[pos];
  const ModeState &mi = mode(o.modes[0]), &mj = mode(o.modes[1]), &mk = mode(o.modes[2]);
  const int R = mi.R;
  if (tc_op_.data == nullptr) {
    int64_t mx = 1;
    for (auto& ob : objects_)
      if (ob.model == AOADMM_MODEL_CP && ob.order == 3) mx = std::max<int64_t>(mx, std::max(ob.dims[0], ob.dims[1]));
    int Rmax = 1;
    for (auto& m : modes_) Rmax = std::max(Rmax, m.R);
    tc_operand_alloc(tc_op_, mx, Rmax);
  }
  const double* Fk = mk.fac.p + o.shard_offset;   // this rank's rows of the (possibly sharded) last mode
  const double *F0, *Fe;
  int64_t ld0, ldfe;
  if (pos == 0) {
    F0 = mj.fac.p, ld0 = mj.rows, Fe = Fk, ldfe = mk.rows;
  } else if (pos == 1) {
    F0 = mi.fac.p, ld0 = mi.rows, Fe = Fk, ldfe = mk.rows;
  } else {
    F0 = mi.fac.p, ld0 = mi.rows, Fe = mj.fac.p, ldfe = mj.rows;
  }
  return mttkrp3_tc(v.t, pos, tc_op_, F0, ld0, Fe, ldfe, R, scale, out, ldout, mws_, st_, nullptr, emit, prec);
}

void Engine::refresh_gram(ModeState& m) {
  launches_ += gram(m.fac.p, m.rows, m.rows, m.R, m.GtG.p, gram_ws_, st_, nullptr);
  if (m.p >= 0 && sparse_masked(objects_[m.p]))   // B_pos' F_pos for the low-rank term of the imputed MTTKRP
    launches_ += sparse_cross_gram(*objects_[m.p].sp, m.pos, m.fac.p, m.rows, st_);
}

void Engine::precompute_mode(ModeState& m, int n_rho_terms, bool do_chol) {
  ObjectState& o = objects_[m.p];
  PrepArgs a{};
  a.nhad = 0;
  for (int d = 0; d < o.order; ++d)
    if (o.modes[d] != m.id) a.had[a.nhad++] = mode(o.modes[d]).GtG.p;  // :98-103, :109, :112
  fill_prep(m, a, n_rho_terms, do_chol);
  // the system preparation depends only on the Grams of the other modes: run it on the side stream while the
  // MTTKRP of this mode streams the tensor on the main stream
  AO_CUDA(cudaEventRecord(ev_fork_, st_));
  AO_CUDA(cudaStreamWaitEvent(st2_, ev_fork_, 0));
  launches_ += prep_system(a, st2_, nullptr);
  AO_CUDA(cudaEventRecord(ev_join_, st2_));
  compute_mttkrp(o, m.pos, o.weight, m.A.p, m.rows, true);  // A{m} = w * mttkrp (:97, :108, :111)
  AO_CUDA(cudaStreamWaitEvent(st_, ev_join_, 0));
  apply_bsum(m);
}

// ---------------------------------------------------------------------------------------------------
// PARAFAC2 block
// ---------------------------------------------------------------------------------------------------
void Engine::setup_par2(const aoadmm_problem* prob, int p) {
  const aoadmm_object& src = prob->objects[p];
  ObjectState& o = objects_[p];
  if (o.order != 3) throw CudaError(1, "a PARAFAC2 object has exactly three modes (A, B_k, C)");
  par2_.emplace_back();
  Par2State& s = par2_.back();
  const int idx = (int)par2_.size() - 1;
  s.p = p;
  s.m1 = o.modes[0];
  s.m2 = o.modes[1];
  s.m3 = o.modes[2];
  for (int d = 0; d < 3; ++d) {
    const int mid = o.modes[d];
    if (mid < 1 || mid > nb_modes_) throw CudaError(1, "mode id out of range");
    ModeState& m = mode(mid);
    if (m.p != -1) throw CudaError(1, "mode " + std::to_string(mid) + " belongs to two objects");
    m.p = p;
    m.pos = d;
    m.par2_role = d + 1;
    m.par2 = idx;
  }
  ModeState &ma = mode(s.m1), &mb = mode(s.m2), &mc = mode(s.m3);
  s.R = ma.R;
  if (mb.R != s.R || mc.R != s.R) throw CudaError(1, "all modes of a PARAFAC2 object need the same rank");
  if (s.R > 128) throw CudaError(2, "PARAFAC2 objects support at most 128 components on device");
  s.K = (prob->n_slices != nullptr) ? prob->n_slices[s.m2 - 1] : 0;
  const int64_t* jk = (prob->slice_rows != nullptr) ? prob->slice_rows[s.m2 - 1] : nullptr;
  if (s.K <= 0 || jk == nullptr || src.n_slices != s.K || src.slices == nullptr)
    throw CudaError(1, "PARAFAC2 object: slice sizes (Z.size of the second mode) and K data slices are required");
  if (mc.rows != s.K) throw CudaError(1, "PARAFAC2 object: the third mode must have K rows");
  s.I = ma.rows;
  s.joff.assign(s.K + 1, 0);
  for (int k = 0; k < s.K; ++k) {
    if (jk[k] < s.R)  // cmtf_AOADMM.m:55-65
      throw CudaError(1, "Number of components for PARAFAC2 is larger than size of slice " + std::to_string(k + 1));
    s.joff[k + 1] = s.joff[k] + jk[k];
    s.Jmax = std::max<int64_t>(s.Jmax, jk[k]);
  }
  s.Jtot = s.joff[s.K];
  mb.rows = s.Jtot;
  o.dims = {s.I, s.Jtot, (int64_t)s.K};
  o.last_full = s.K;
  o.shard_extent = s.K;
  s.ldX = round_up(s.I, 2);
  // Slices sharded over the GPUs (SURVEY 8e) unless a path needs every slice on every rank: a linear coupling on one of
  // the object's modes (the (K*R)^2 / row-wise systems of :283-355 are assembled from all slices), the tPARAFAC2 prox
  // (a solve ACROSS the slices), quadratic regularisation on B_k, or fewer slices than ranks.
  s.k0 = 0;
  s.k1 = s.K;
  if (world_ > 1 && s.K >= world_) {
    bool ok = true;
    for (int d = 0; d < 3; ++d) {
      const ModeState& m = mode(o.modes[d]);
      if (m.coupling != 0 && coupling_type_[m.coupling - 1] != 0) ok = false;
    }
    if (mb.constrained && (mb.con.kind == AOADMM_CON_TPARAFAC2 || mb.con.kind == AOADMM_CON_QUADRATIC ||
                           mb.con.kind == AOADMM_CON_ORTHONORMAL))
      ok = false;
    if (ok) {
      s.sharded = true;
      s.k0 = (int)((int64_t)s.K * rank_ / world_);
      s.k1 = (int)((int64_t)s.K * (rank_ + 1) / world_);
    }
  }
  s.jlo = s.joff[s.k0];
  s.jhi = s.joff[s.k1];
  const int64_t Jloc = s.jhi - s.jlo;
  const size_t xbytes = std::max<size_t>((size_t)s.ldX * Jloc * sizeof(double), 256);
  AO_CUDA(cudaMalloc(&s.X_alloc, xbytes));
  if (s.ldX != s.I) AO_CUDA(cudaMemset(s.X_alloc, 0, xbytes));
  s.X = s.X_alloc - (size_t)s.jlo * s.ldX;      // global column indexing (only columns jlo..jhi-1 are ever touched)
  std::vector<int> seg((size_t)s.Jtot);
  for (int k = 0; k < s.K; ++k) {
    for (int64_t j = s.joff[k]; j < s.joff[k + 1]; ++j) seg[(size_t)j] = k;
    if (k < s.k0 || k >= s.k1) continue;          // another rank's slice (its pointer may be NULL)
    if (src.slices[k] == nullptr) throw CudaError(1, "PARAFAC2 object: NULL slice");
    AO_CUDA(cudaMemcpy2D(s.X + (size_t)s.joff[k] * s.ldX, (size_t)s.ldX * 8, src.slices[k], (size_t)s.I * 8,
                         (size_t)s.I * 8, (size_t)jk[k], cudaMemcpyHostToDevice));
  }
  if (src.miss_slices != nullptr) {
    const size_t mbytes = std::max<size_t>((size_t)s.ldX * Jloc, 256);
    AO_CUDA(cudaMalloc(&s.mask_alloc, mbytes));
    AO_CUDA(cudaMemset(s.mask_alloc, 0, mbytes));
    s.mask = s.mask_alloc - (size_t)s.jlo * s.ldX;
    for (int k = s.k0; k < s.k1; ++k) {
      if (src.miss_slices[k] == nullptr) throw CudaError(1, "Z.miss{p}{k} must be given for every PARAFAC2 slice");
      AO_CUDA(cudaMemcpy2D(s.mask + (size_t)s.joff[k] * s.ldX, (size_t)s.ldX, src.miss_slices[k], (size_t)s.I, (size_t)s.I,
                           (size_t)jk[k], cudaMemcpyHostToDevice));
    }
    has_missing_ = true;
  }
  AO_CUDA(cudaMalloc(&s.joff_dev, sizeof(long long) * (s.K + 1)));
  {
    std::vector<long long> tmp(s.joff.begin(), s.joff.end());
    AO_CUDA(cudaMemcpy(s.joff_dev, tmp.data(), sizeof(long long) * (s.K + 1), cudaMemcpyHostToDevice));
  }
  AO_CUDA(cudaMalloc(&s.seg_dev, sizeof(int) * (size_t)s.Jtot));
  AO_CUDA(cudaMemcpy(s.seg_dev, seg.data(), sizeof(int) * (size_t)s.Jtot, cudaMemcpyHostToDevice));
  s.lay.K = s.K;
  s.lay.R = s.R;
  s.lay.Jtot = s.Jtot;
  s.lay.Jmax = s.Jmax;
  s.lay.joff = s.joff_dev;
  s.lay.seg = s.seg_dev;
  s.lay.k0 = s.k0;
  s.lay.k1 = s.k1;
  s.lay.jlo = s.jlo;
  s.lay.jhi = s.jhi;
  make_tensor3(s.view, s.X_alloc, s.I, Jloc, 1, s.ldX);   // this rank's columns as an I x Jloc x 1 tensor
  packed_factor_alloc(s.fW, Jloc, s.R);
  AO_CUDA(cudaMalloc(&s.redbuf, sizeof(double) * ((size_t)s.R * s.R + 8)));
  packed_factor_alloc(s.fA, s.I, s.R);
  packed_factor_alloc(s.ones, 1, s.R);
  packed_factor_pack(s.ones, nullptr, 1, st_, nullptr);
  ++launches_;
  for (DevMat* d : {&s.W, &s.T, &s.P, &s.muDB, &s.PDold, &s.gM, &s.gS}) dev_alloc(*d, s.Jtot, s.R);
  dev_alloc(s.DeltaB, s.R, s.R);
  const size_t KRR = (size_t)s.K * s.R * s.R;
  AO_CUDA(cudaMalloc(&s.G2, KRR * sizeof(double)));
  AO_CUDA(cudaMalloc(&s.Binv2, KRR * sizeof(double)));
  AO_CUDA(cudaMalloc(&s.Binv3, KRR * sizeof(double)));
  AO_CUDA(cudaMalloc(&s.contrib, KRR * sizeof(double)));
  AO_CUDA(cudaMalloc(&s.Vprev, KRR * sizeof(double)));
  if (s.R > 64) AO_CUDA(cudaMalloc(&s.sysws, 2 * KRR * sizeof(double)));
  AO_CUDA(cudaMalloc(&s.rho2, sizeof(double) * s.K));
  AO_CUDA(cudaMalloc(&s.rho3, sizeof(double) * s.K));
  AO_CUDA(cudaMalloc(&s.tdiag, sizeof(double) * s.K));
  AO_CUDA(cudaMalloc(&s.norms, sizeof(double) * s.K * 8));
  AO_CUDA(cudaMemset(s.norms, 0, sizeof(double) * s.K * 8));
  AO_CUDA(cudaMalloc(&s.Csum, sizeof(double) * s.R * s.R));
  AO_CUDA(cudaMalloc(&s.segn, sizeof(double) * (s.K * 4 + 8)));
  AO_CUDA(cudaMemset(s.segn, 0, sizeof(double) * (s.K * 4 + 8)));
  AO_CUDA(cudaMalloc(&s.res_partials, sizeof(double) * 148 * 8));
  AO_CUDA(cudaMallocHost(&s.segn_host, sizeof(double) * (s.K * 4 + 8)));
  s.res = s.segn + (size_t)s.K * 4;
  mc.rho_rows = s.rho3;
  mc.Binv_rows = s.Binv3;
  AO_CUDA(cudaDeviceSynchronize());
}

void Engine::par2_refresh_gram(Par2State& s) {  // :71-73, :216-218
  launches_ += par2_batched_gram(s.lay, mode(s.m2).fac.p, s.G2, st_);
}

// T = Xall' * A (Jtot x R): shared by the mode-B right-hand sides (:193) and the mode-C ones (:221)
void Engine::par2_update_T(Par2State& s) {
  ModeState& a = mode(s.m1);
  if (s.T_version == a.version) return;
  phase_begin(1);
  packed_factor_pack(s.fA, a.fac.p, a.rows, st_, nullptr);
  ++launches_;
  launches_ += mttkrp3(s.view, 1, s.fA, s.ones, s.R, 1.0, s.T.p + s.jlo, s.Jtot, mws_, st_, nullptr);   // local rows of T
  phase_end();
  s.T_version = a.version;
}

void Engine::fill_prep(ModeState& m, PrepArgs& a, int n_rho_terms, bool do_chol) {
  ObjectState& o = objects_[m.p];
  a.R = m.R;
  a.weight = o.weight;
  a.ridge = m.ridge;
  a.bsum_half = opt_.bsum ? opt_.bsum_weight / 2.0 : 0.0;
  a.n_rho_terms = n_rho_terms;
  a.rho_scale = 1.0;
  a.HHt = (m.lin >= 0 && lin_modes_[m.lin].ctype == 2) ? lin_modes_[m.lin].HHt.p : nullptr;  // :314
  a.do_chol = do_chol ? 1 : 0;
  a.C = m.C.p;
  a.B = m.B.p;
  a.L = m.L.p;
  a.invdiag = m.invdiag;
  a.Binv = m.Binv.p;
  a.Btmp = m.Btmp.p;
  a.rho = m.rho;
  a.ctl = m.ctl;
}

void Engine::apply_bsum(ModeState& m) {
  if (!opt_.bsum) return;  // :124-127 (last_mttkrp keeps the value before the BSUM term, :121)
  AO_CUDA(cudaMemcpyAsync(m.Alast.p, m.A.p, m.A.bytes(), cudaMemcpyDeviceToDevice, st_));
  const long long n = m.rows * m.R;
  axpy_kernel<<<(unsigned)std::min<long long>(ceil_div(n, 256), 148 * 8), 256, 0, st_>>>(m.A.p, m.fac.p,
                                                                                         opt_.bsum_weight / 2.0, n);
  AO_CHECK_LAUNCH();
  ++launches_;
}

// first PARAFAC2 mode (:159-178): A = w * sum_k X_k B_k diag(c_k),  C = sum_k diag(c_k) B_k'B_k diag(c_k)
void Engine::par2_precompute_A(ModeState& m, int n_rho_terms, bool do_chol) {
  Par2State& s = par2_[m.par2];
  ObjectState& o = objects_[m.p];
  ModeState &mb = mode(s.m2), &mc = mode(s.m3);
  phase_begin(1);
  launches_ += par2_scale_rows(s.lay, s.W.p, mb.fac.p, mc.fac.p, mc.rows, 1.0, nullptr, 0.0, st_);
  packed_factor_pack(s.fW, s.W.p + s.jlo, s.Jtot, st_, nullptr);
  ++launches_;
  launches_ += mttkrp3(s.view, 0, s.fW, s.ones, s.R, o.weight, m.A.p, m.rows, mws_, st_, nullptr);
  if (s.sharded) allreduce(m.A.p, (size_t)m.rows * m.R);    // sum over the ranks' slices (:159-163)
  phase_end();
  launches_ += par2_modeA_had(s.lay, s.G2, mc.fac.p, mc.rows, s.Csum, st_);
  if (s.sharded) allreduce(s.Csum, (size_t)s.R * s.R);      // :164
  PrepArgs a{};
  a.nhad = 1;
  a.had[0] = s.Csum;
  fill_prep(m, a, n_rho_terms, do_chol);
  launches_ += prep_system(a, st_, nullptr);
  apply_bsum(m);
}

// second PARAFAC2 mode: per-slice systems (:192-213) and ADMM_B_Parafac2 (:509-589)
void Engine::par2_update_B(ModeState& m, int outer_iter) {
  Par2State& s = par2_[m.par2];
  ObjectState& o = objects_[m.p];
  ModeState &ma = mode(s.m1), &mc = mode(s.m3);
  par2_update_T(s);
  const bool bs = opt_.bsum != 0;
  launches_ += par2_scale_rows(s.lay, m.A.p, s.T.p, mc.fac.p, mc.rows, o.weight, bs ? m.fac.p : nullptr,
                               bs ? opt_.bsum_weight / 2.0 : 0.0, st_);
  const bool con_active = m.constrained && outer_iter >= opt_.iter_start_PAR2Bkconstraint;
  Par2SysArgs sa{};
  sa.mode = 2;
  sa.G1 = ma.GtG.p;
  sa.C = mc.fac.p;
  sa.ldc = mc.rows;
  sa.weight = o.weight;
  sa.ridge = m.ridge;
  sa.bsum_half = bs ? opt_.bsum_weight / 2.0 : 0.0;
  sa.rho_scale = opt_.has_increase_factor_rhoBk ? opt_.increase_factor_rhoBk : 1.0;
  sa.n_rho_terms = 1 + (con_active ? 1 : 0);
  sa.rho_k = s.rho2;
  sa.Binv = s.Binv2;
  sa.ctl = m.ctl;
  sa.gws = s.sysws;
  launches_ += par2_sys_prep(s.lay, sa, st_);
  const bool deferred = con_active && !prox_is_elementwise(m.con.kind);
  Par2BArgs b{};
  b.A = m.A.p;
  b.Binv = s.Binv2;
  b.rho_k = s.rho2;
  b.B = m.fac.p;
  b.P = s.P.p;
  b.mu = s.muDB.p;
  b.DeltaB = s.DeltaB.p;
  b.Z = m.Z.p;
  b.muZ = m.muZ.p;
  b.con_active = con_active ? 1 : 0;
  b.prox_kind = m.con.kind;
  b.p0 = m.con.p0;
  b.p1 = m.con.p1;
  b.PDold = s.PDold.p;
  b.contrib = s.contrib;
  b.gM = s.gM.p;
  b.gS = s.gS.p;
  b.norms = s.norms;
  b.Znew = deferred ? m.Znew.p : nullptr;
  b.Vprev = s.Vprev;
  InnerTol tol{opt_.innerRelPrTol_coupl, opt_.innerRelDualTol_coupl, opt_.innerRelPrTol_constr,
               opt_.innerRelDualTol_constr};
  for (int it = 0; it < opt_.MaxInnerIters; ++it) {
    launches_ += par2_B_step1(s.lay, b, m.ctl, it > 0 ? 1 : 0, st_);  // cold start once per outer iteration
    if (s.sharded) {   // DeltaB = sum_k rho_k P_k'(B_k + mu_k) / sum_k rho_k over ALL slices (:541-544)
      launches_ += par2_B_deltaB(s.lay, b, m.ctl, st_, s.redbuf);
      allreduce(s.redbuf, (size_t)s.R * s.R + 1);
      launches_ += par2_B_deltaB_finish(s.lay, b, s.redbuf, m.ctl, st_);
    } else {
      launches_ += par2_B_deltaB(s.lay, b, m.ctl, st_);
    }
    launches_ += par2_B_step2a(s.lay, b, m.ctl, st_);
    if (deferred) {
      launches_ += par2_B_form_prox_input(s.lay, b, m.V.p, m.ctl, st_);
      if (m.con.kind == AOADMM_CON_TPARAFAC2) {  // :553-554: all slices at once with the vector rho
        launches_ += par2_tsmooth_prox(s.lay, m.V.p, s.rho2, m.con.p0, s.tdiag, m.Znew.p, m.ctl, st_);
      } else if (prox_supports_segments(m.con.kind)) {
        // :567-568: prox of every slice with its own rho_k - all K slices and R columns in ONE launch
        if (m.con.kind == AOADMM_CON_SIMPLEX_ROW)   // independent rows: this rank's stacked rows as one matrix
          launches_ += apply_prox(m, m.V.p + s.jlo, s.Jtot, m.Znew.p + s.jlo, s.Jtot, s.jhi - s.jlo, s.R, s.rho2, &m.ctl->done);
        else
          launches_ += prox_apply_segments(m.con.kind, m.con.p0, m.con.p1, m.V.p, s.Jtot, m.Znew.p, s.Jtot, s.joff_dev + s.k0,
                                           s.k1 - s.k0, s.Jmax, s.Jtot, s.R, s.rho2 + s.k0, prox_scratch_, st_, &m.ctl->done);
      } else {
        for (int k = 0; k < s.K; ++k)  // whole-matrix operators ('orthonormal', 'quadratic regularization'): per slice
          launches_ += apply_prox(m, m.V.p + s.joff[k], s.Jtot, m.Znew.p + s.joff[k], s.Jtot, s.joff[k + 1] - s.joff[k], s.R,
                                  s.rho2 + k, &m.ctl->done);
      }
    }
    if (s.sharded) {   // residual ratios averaged over ALL slices (:558-585): same exit test on every rank
      launches_ += par2_B_step2b(s.lay, b, tol, m.ctl, admm_counter_, st_, s.redbuf);
      allreduce(s.redbuf, 4);
      launches_ += par2_B_finalize(s.lay, s.redbuf, tol, m.ctl, st_);
    } else {
      launches_ += par2_B_step2b(s.lay, b, tol, m.ctl, admm_counter_, st_);
    }
  }
  par2_refresh_gram(s);
  s.state_stale = s.sharded;
  ++m.version;
}

// third PARAFAC2 mode (:220-243): per-row right-hand sides and systems
void Engine::par2_precompute_C(ModeState& m, int n_rho_terms, bool ls_direct, double* Bsys_out, const double* HHt) {
  Par2State& s = par2_[m.par2];
  ObjectState& o = objects_[m.p];
  ModeState &ma = mode(s.m1), &mb = mode(s.m2);
  par2_update_T(s);
  Par2SysArgs sa{};
  sa.mode = 3;
  sa.G1 = ma.GtG.p;
  sa.G2 = s.G2;
  sa.C = m.fac.p;
  sa.ldc = m.rows;
  sa.weight = o.weight;
  sa.ridge = m.ridge;
  sa.bsum_half = opt_.bsum ? opt_.bsum_weight / 2.0 : 0.0;
  sa.rho_scale = 1.0;
  sa.n_rho_terms = n_rho_terms;
  sa.T = s.T.p;
  sa.Bst = mb.fac.p;
  sa.rhs = m.A.p;
  sa.ls_direct = ls_direct ? 1 : 0;
  sa.fac_out = m.fac.p;
  sa.rho_k = s.rho3;
  sa.Binv = s.Binv3;
  sa.Bsys = Bsys_out;
  sa.no_factor = (Bsys_out != nullptr) ? 1 : 0;
  sa.HHt = HHt;
  sa.ctl = m.ctl;
  sa.gws = s.sysws;
  launches_ += par2_sys_prep(s.lay, sa, st_);
  if (s.sharded) {
    // the third mode is updated on every rank (its K rows are few): gather the rows each rank prepared -
    // right-hand sides, rho_k, inv(B_k) (or the directly solved rows of C, :236)
    const size_t RR = (size_t)s.R * s.R;
    launches_ += zero_rows_outside(ls_direct ? m.fac.p : m.A.p, s.K, s.R, s.k0, s.k1, st_);
    allreduce(ls_direct ? m.fac.p : m.A.p, (size_t)s.K * s.R);
    launches_ += zero_rows_outside(s.rho3, s.K, 1, s.k0, s.k1, st_);
    allreduce(s.rho3, (size_t)s.K);
    if (!ls_direct) {
      launches_ += zero_rows_outside(s.Binv3, (long long)(s.K * RR), 1, (long long)(s.k0 * RR), (long long)(s.k1 * RR), st_);
      allreduce(s.Binv3, (size_t)s.K * RR);
    }
  }
  launches_ += par2_rho_max(s.rho3, s.K, m.rho, st_);
}

int Engine::apply_prox(ModeState& m, const double* X, long long ldx, double* out, long long ldo, long long rows, int cols,
                       const double* rho_dev, const int* skip) {
  if (m.con.kind == AOADMM_CON_QUADRATIC) return quad_prox_apply(m.quad, X, ldx, out, ldo, cols, rho_dev, 0.0, st_, skip);
  return prox_apply(m.con.kind, m.con.p0, m.con.p1, X, ldx, out, ldo, rows, cols, rho_dev, 0.0, prox_scratch_, st_, skip);
}

void Engine::run_admm(std::vector<ModeState*>& group, double* Delta, const aoadmm_options& opt) {
  if ((int)group.size() > kMaxGroup) throw CudaError(2, "more than 8 modes in one coupling group");
  AdmmGroup g{};
  g.nmodes = (int)group.size();
  g.Delta = Delta;
  g.rows = group[0]->rows;
  g.R = group[0]->R;
  std::vector<int> deferred;
  for (int i = 0; i < g.nmodes; ++i) {
    ModeState& m = *group[i];
    AdmmMode& am = g.m[i];
    am.A = m.A.p;
    am.Binv = m.Binv.p;
    am.rho = m.rho;
    am.rho_rows = m.rho_rows;
    am.Binv_rows = m.Binv_rows;
    am.F = m.fac.p;
    am.Z = m.Z.p;
    am.muZ = m.muZ.p;
    am.muD = m.muD.p;
    am.ldA = m.rows;
    am.ldF = m.rows;
    am.constrained = m.constrained ? 1 : 0;
    am.prox_kind = m.con.kind;
    am.p0 = m.con.p0;
    am.p1 = m.con.p1;
    if (m.constrained && !prox_is_elementwise(m.con.kind)) deferred.push_back(i);
  }
  for (ModeState* mp : group) ++mp->version;
  InnerCtl* ctl = group[0]->ctl;
  InnerTol tol{opt.innerRelPrTol_coupl, opt.innerRelDualTol_coupl, opt.innerRelPrTol_constr, opt.innerRelDualTol_constr};
  if (deferred.empty() && opt.MaxInnerIters > 1 && opt_.fuse_inner >= 0 && admm_can_fuse_inner(g)) {
    // every prox of the group is element-wise and all CTAs fit on the GPU at once: the whole inner loop is one
    // cooperative launch (grid barrier + device-side exit test between the iterations)
    launches_ += admm_iteration(g, tol, ctl, admm_sums_, admm_partials_, admm_counter_, 1, st_, opt.MaxInnerIters);
    return;
  }
  for (int it = 0; it < opt.MaxInnerIters; ++it) {
    launches_ += admm_iteration(g, tol, ctl, admm_sums_, admm_partials_, admm_counter_, deferred.empty() ? 1 : 0, st_);
    for (size_t d = 0; d < deferred.size(); ++d) {
      ModeState& m = *group[deferred[d]];
      launches_ += admm_form_prox_input(g, deferred[d], m.V.p, ctl, st_);
      launches_ += apply_prox(m, m.V.p, m.rows, m.Znew.p, m.rows, m.rows, m.R, m.rho, &ctl->done);
      launches_ += admm_constraint_update(g, deferred[d], m.Znew.p, tol, ctl, admm_sums_, admm_partials_, admm_counter_,
                                          (d + 1 == deferred.size()) ? 1 : 0, st_);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// objective (cmtf_fun_AOADMM.m:1213-1363)
// ---------------------------------------------------------------------------------------------------
void Engine::build_objective_jobs() {
  terms_.reset(new ObjTerms());
  terms_->obj.resize(n_objects_);
  terms_->mode.resize(nb_modes_);
  jobs_host_.clear();
  auto add = [&](int kind, const double* a, const double* b, int64_t rows, int cols) {
    RedJob j{};
    j.kind = kind;
    j.cols = cols;
    j.rows = rows;
    j.lda = rows;
    j.ldb = rows;
    j.a = a;
    j.b = b;
    jobs_host_.push_back(j);
    return (int)jobs_host_.size() - 1;
  };
  for (int p = 0; p < n_objects_; ++p) {
    ModeState& lm = mode(objects_[p].last_m);
    if (objects_[p].model == AOADMM_MODEL_PAR2 && lm.par2_role != 1) {
      // :1254 - the shortcut only exists when the first PARAFAC2 mode is the one updated last
      par2_[lm.par2].explicit_residual = true;
      continue;
    }
    // Alast holds last_mttkrp when BSUM is on; decided at run time by swapping the pointer (see eval_objective)
    terms_->obj[p].idx_dot = add(RED_DOT, lm.A.p, lm.fac.p, lm.rows, lm.R);
    terms_->obj[p].idx_had = add(RED_DOT, lm.C.p, lm.GtG.p, lm.R, lm.R);
  }
  for (int i = 0; i < nb_modes_; ++i) {
    ModeState& m = modes_[i];
    auto& t = terms_->mode[i];
    if (m.par2_role == 2) {          // per-slice terms come from par2_seg_norms ...
      if (m.constrained && m.con.kind == AOADMM_CON_QUADRATIC)   // ... except sum_k eta*trace(B_k' L B_k): L*B_k in m.V
        t.idx_reg = add(RED_DOT, m.fac.p, m.V.p, m.rows, m.R);
      continue;
    }
    t.idx_norm2 = add(RED_NORM2, m.fac.p, nullptr, m.rows, m.R);
    if (m.constrained) t.idx_diffZ = add(RED_DIFF2, m.fac.p, m.Z.p, m.rows, m.R);
    if (m.coupling != 0 && m.lin < 0) t.idx_diffD = add(RED_DIFF2, m.fac.p, delta_[m.coupling - 1].p, m.rows, m.R);
    if (m.lin >= 0) {  // :1313-1321: ||G(F) - D(Delta)|| over ||G(F)|| (types 1,2,5) or ||F|| (types 3,4)
      LinMode& lm = lin_modes_[m.lin];
      t.idx_diffD = add(RED_DIFF2, lm.S1.p, lm.S2.p, lm.S1.rows, (int)lm.S1.cols);
      if (lm.ctype == 1 || lm.ctype == 2 || lm.ctype == 5) t.idx_normG = add(RED_NORM2, lm.S1.p, nullptr, lm.S1.rows, (int)lm.S1.cols);
    }
    if (m.constrained && reg_red_kind(m.con.kind) >= 0)
      t.idx_reg = add(reg_red_kind(m.con.kind), m.fac.p, nullptr, m.rows, m.R);
    if (m.constrained && m.con.kind == AOADMM_CON_QUADRATIC)   // constraints_to_prox.m:67: eta*trace(x'*L*x), L*x in m.V
      t.idx_reg = add(RED_DOT, m.fac.p, m.V.p, m.rows, m.R);
  }
  const size_t nj = jobs_host_.size();
  AO_CUDA(cudaMalloc(&jobs_dev_, sizeof(RedJob) * (nj + 8)));
  AO_CUDA(cudaMemcpy(jobs_dev_, jobs_host_.data(), sizeof(RedJob) * nj, cudaMemcpyHostToDevice));
  AO_CUDA(cudaMalloc(&red_dev_, sizeof(double) * (nj + 8)));
  AO_CUDA(cudaMallocHost(&red_host_, sizeof(double) * (nj + 8)));
  AO_CUDA(cudaMalloc(&red_partials_, sizeof(double) * reduce_ws_doubles((int)nj + 8)));
}

void Engine::em_step(bool impute) {
  if (!has_missing_) return;
  for (int p = 0; p < n_objects_; ++p) {
    ObjectState& o = objects_[p];
    EmArgs a{};
    a.R = mode(o.modes[0]).R;
    a.impute = impute ? 1 : 0;
    a.partials = em_partials_;
    if (o.model == AOADMM_MODEL_PAR2) {
      Par2State& s = par2_[mode(o.modes[0]).par2];
      if (s.mask == nullptr) continue;
      ModeState &ma = mode(s.m1), &mb = mode(s.m2), &mc = mode(s.m3);
      // model of slice k: A diag(c_k) B_k' (:426)  =  A * W' on the stacked layout, W(j,:) = B(j,:) .* C(seg(j),:)
      launches_ += par2_scale_rows(s.lay, s.W.p, mb.fac.p, mc.fac.p, mc.rows, 1.0, nullptr, 0.0, st_);
      a.X = s.X_alloc;              // this rank's slices (all of them on one GPU)
      a.mask = s.mask_alloc;
      a.ldI = s.ldX;
      a.I = s.I;
      a.J = s.jhi - s.jlo;
      a.K = 1;
      a.Fi = ma.fac.p;
      a.ldFi = ma.rows;
      a.Fj = s.W.p + s.jlo;
      a.ldFj = s.Jtot;
      a.Fk = nullptr;
      launches_ += em_pass(a, em_sums_ + 5 * p, st_);
      if (s.sharded) allreduce(em_sums_ + 5 * p, 5);
      if (impute) s.T_version = 0;
    } else if (sparse_masked(o)) {
      // model at the stored entries + telescoped norms of the unobserved part, nothing dense (sparse.cuh)
      phase_begin(2);
      const double* fac[8];
      long long ld[8];
      for (int d = 0; d < o.order; ++d) {
        const ModeState& md = mode(o.modes[d]);
        fac[d] = md.fac.p;
        ld[d] = md.rows;
      }
      launches_ += sparse_em_nonzeros(*o.sp, fac, ld, impute, st_);
      // only the nonzero-side sums are partial: the telescoped terms are replicated and must be counted once
      if (o.sharded) allreduce(o.sp->em_nz, 4);
      launches_ += sparse_em_finish(*o.sp, fac, ld, impute, em_sums_ + 5 * p, st_);
      phase_end();
    } else {
      if (o.mask == nullptr) continue;
      ModeState &m0 = mode(o.modes[0]), &m1 = mode(o.modes[1]);
      a.X = o.data;
      a.mask = o.mask;
      a.ldI = o.ld0;
      a.I = o.dims[0];
      a.J = o.dims[1];
      a.Fi = m0.fac.p;
      a.ldFi = m0.rows;
      a.Fj = m1.fac.p;
      a.ldFj = m1.rows;
      if (o.order > 3) {
        // trailing modes merged: K = prod dims[2..], third factor = their Khatri-Rao product (memory order)
        KrArgs kr{};
        kr.n = o.order - 2;
        long long kk = 1;
        for (int d = 2; d < o.order; ++d) {
          ModeState& md = mode(o.modes[d]);
          kr.F[d - 2] = md.fac.p + (d == o.order - 1 ? o.shard_offset : 0);
          kr.ld[d - 2] = md.rows;
          kr.d[d - 2] = o.dims[d];
          kk *= o.dims[d];
        }
        launches_ += em_khatri_rao(kr, o.em_kr, kk, a.R, st_);
        a.K = (int)kk;
        a.Fk = o.em_kr;
        a.ldFk = kk;
      } else if (o.order == 3) {
        ModeState& m2 = mode(o.modes[2]);
        a.K = (int)o.dims[2];
        a.Fk = m2.fac.p + o.shard_offset;  // this rank's rows of the (possibly sharded) last mode
        a.ldFk = m2.rows;
      } else {
        a.K = 1;
        a.Fk = nullptr;
      }
      a.fkT = o.em_fkT;
      launches_ += em_pass(a, em_sums_ + 5 * p, st_);
      if (o.sharded) allreduce(em_sums_ + 5 * p, 5);
      if (impute) o.T_version = 0;
    }
  }
}

void Engine::eval_objective(bool first, double f[4]) {
  enqueue_objective(first);
  finish_objective(first, f);
}

// device part of CMTF_AOADMM_func_eval: every reduction kernel + the device->host copies of their results
void Engine::enqueue_objective(bool first) {
  const int nj = (int)jobs_host_.size();
  std::vector<double>& f_obj = f_obj_;
  f_obj.assign(n_objects_, 0.0);
  if (first) {
    // cp_func.m:47-56 / pca_func.m:29-40: f = w*(||X||^2 - 2*sum(A1 .* mttkrp(X,A,1)) + sum(prod of all Grams))
    for (int p = 0; p < n_objects_; ++p) {
      ObjectState& o = objects_[p];
      if (o.model == AOADMM_MODEL_PAR2) continue;  // explicit residual below (:1262-1264)
      if (o.mask != nullptr || sparse_masked(o)) continue;   // masked objective from the EM sums (:1224-1226)
      ModeState& m0 = mode(o.modes[0]);
      double* M = cp0_tmp_;
      double* scr = cp0_tmp_ + (size_t)m0.rows * m0.R;  // C | B | L | invdiag | rho
      const size_t RR = (size_t)256 * 256;
      compute_mttkrp(o, 0, 1.0, M, m0.rows);
      PrepArgs a{};
      a.nhad = 0;
      for (int d = 0; d < o.order; ++d) a.had[a.nhad++] = mode(o.modes[d]).GtG.p;
      a.R = m0.R;
      a.weight = 1.0;
      a.rho_scale = 1.0;
      a.do_chol = 0;
      a.C = scr;
      a.B = scr + RR;
      a.L = scr + 2 * RR;
      a.invdiag = scr + 3 * RR;
      a.rho = scr + 3 * RR + 256;
      a.ctl = nullptr;
      launches_ += prep_system(a, st_, nullptr);
      RedJob jb[2]{};
      jb[0].kind = RED_DOT;
      jb[0].cols = m0.R;
      jb[0].rows = jb[0].lda = jb[0].ldb = m0.rows;
      jb[0].a = M;
      jb[0].b = m0.fac.p;
      jb[1].kind = RED_SUM;  // f_3 = sum(W(:)) (cp_func.m:52)
      jb[1].cols = 1;
      jb[1].rows = jb[1].lda = jb[1].ldb = (long long)m0.R * m0.R;
      jb[1].a = scr;
      jb[1].b = nullptr;
      AO_CUDA(cudaMemcpyAsync(jobs_dev_ + nj, jb, sizeof(jb), cudaMemcpyHostToDevice, st_));
      launches_ += reduce_jobs(jobs_dev_ + nj, 2, red_dev_ + nj, red_partials_, admm_counter_, st_, nullptr);
      double r2[2];
      AO_CUDA(cudaMemcpyAsync(r2, red_dev_ + nj, sizeof(r2), cudaMemcpyDeviceToHost, st_));
      AO_CUDA(cudaStreamSynchronize(st_));
      f_obj[p] = o.weight * (o.znorm - 2.0 * r2[0] + r2[1]);
    }
  }
  for (auto& m : modes_)
    if (m.constrained && m.con.kind == AOADMM_CON_QUADRATIC) {
      if (m.par2_role == 2) {   // the same L on every (regular) slice of the stacked B
        const Par2State& s = par2_[m.par2];
        const long long J = m.quad.n;
        for (int k = 0; k < s.K; ++k)
          launches_ += dgemm_small(0, 0, J, m.R, J, 1.0, nullptr, m.quad.L, J, m.fac.p + s.joff[k], m.rows, 0.0,
                                   m.V.p + s.joff[k], m.rows, st_, nullptr);
      } else {
        launches_ += dgemm_small(0, 0, m.rows, m.R, m.rows, 1.0, nullptr, m.quad.L, m.rows, m.fac.p, m.rows, 0.0, m.V.p, m.rows, st_, nullptr);
      }
    }
  for (auto& m : modes_)
    if (m.lin >= 0) {
      LinMode& lm = lin_modes_[m.lin];
      lin_G(lm, m, m.fac.p, lm.S1.p, nullptr);
      lin_D(lm, m, delta_[m.coupling - 1].p, delta_[m.coupling - 1], lm.S2.p, nullptr);
    }
  for (auto& s : par2_) {
    ModeState& mb = mode(s.m2);
    launches_ += par2_seg_norms(s.lay, mb.fac.p, mb.constrained ? mb.Z.p : nullptr, s.P.p, s.DeltaB.p,
                                mb.constrained ? reg_red_kind(mb.con.kind) : -1, s.segn, st_);
    if (first || s.explicit_residual)
      launches_ += par2_residual(s.lay, s.X, s.ldX, s.I, mode(s.m1).fac.p, mode(s.m1).rows, mb.fac.p, mode(s.m3).fac.p,
                                 mode(s.m3).rows, s.res_partials, admm_counter_, s.res, st_);
    if (s.sharded) {
      // per-slice terms of the other ranks' slices (zero here) and the partial residuals: one all-reduce gathers / sums
      launches_ += zero_rows_outside(s.segn, (long long)s.K * 4, 1, (long long)s.k0 * 4, (long long)s.k1 * 4, st_);
      allreduce(s.segn, (size_t)s.K * 4 + 1);
    }
    AO_CUDA(cudaMemcpyAsync(s.segn_host, s.segn, sizeof(double) * (s.K * 4 + 1), cudaMemcpyDeviceToHost, st_));
  }
  if (has_missing_)
    AO_CUDA(cudaMemcpyAsync(em_sums_host_, em_sums_, sizeof(double) * 5 * n_objects_, cudaMemcpyDeviceToHost, st_));
  launches_ += reduce_jobs(jobs_dev_, nj, red_dev_, red_partials_, admm_counter_, st_, nullptr);
  AO_CUDA(cudaMemcpyAsync(red_host_, red_dev_, sizeof(double) * nj, cudaMemcpyDeviceToHost, st_));
  AO_CUDA(cudaMemcpyAsync(ctl_host_, ctl_dev_, sizeof(InnerCtl) * n_ctl_, cudaMemcpyDeviceToHost, st_));
  if (n_heldout_ > 0) heldout_pass();
}

// held-out SSE of every object with a held-out set, from the factors after this iteration's sweep and EM step.  It
// only reads the factors, so the solve is the same with and without held-out sets.  The factors are replicated on
// every rank, so every rank computes the same value without communication.
void Engine::heldout_pass() {
  phase_begin(2);
  for (int p = 0; p < n_objects_; ++p) {
    ObjectState& o = objects_[p];
    if (o.ho == nullptr) continue;
    const double* fac[8];
    long long ld[8];
    for (int d = 0; d < o.order; ++d) {
      const ModeState& md = mode(o.modes[d]);
      fac[d] = md.fac.p;
      ld[d] = md.rows;
    }
    launches_ += heldout_sse(*o.ho, fac, ld, ho_sse_ + p, st_);
  }
  phase_end();
  AO_CUDA(cudaMemcpyAsync(ho_sse_host_, ho_sse_, sizeof(double) * n_objects_, cudaMemcpyDeviceToHost, st_));
}

void Engine::record_heldout() {
  for (int p = 0; p < n_objects_; ++p)
    if (objects_[p].ho != nullptr) objects_[p].ho_hist.push_back(ho_sse_host_[p]);
}

// host part: the scalar arithmetic of :1213-1363 on the reduced values
void Engine::finish_objective(bool first, double f[4]) {
  std::vector<double>& f_obj = f_obj_;
  AO_CUDA(cudaStreamSynchronize(st_));
  phase_collect();
  const double* r = red_host_;
  double f_tensors = 0.0;
  // per-slice terms of the PARAFAC2 second modes (host side: K ratios each)
  struct SliceTerms {
    double con = 0.0, par2 = 0.0, reg = 0.0, n2 = 0.0;
  };
  std::vector<SliceTerms> st2(par2_.size());
  for (size_t q = 0; q < par2_.size(); ++q) {
    const Par2State& s = par2_[q];
    for (int k = 0; k < s.K; ++k) {
      const double* h = s.segn_host + (size_t)k * 4;
      const double nB = std::sqrt(h[0]);
      st2[q].con += std::sqrt(h[1]) / nB;    // :1337
      st2[q].par2 += std::sqrt(h[2]) / nB;   // :1355
      st2[q].reg += h[3];                    // :1279-1281
      st2[q].n2 += h[0];                     // :1293-1295
    }
  }
  if (has_missing_) {  // :436-440
    double num = 0.0, den = 0.0;
    for (int p = 0; p < n_objects_; ++p) {
      num += em_sums_host_[5 * p + 0];
      den += em_sums_host_[5 * p + 1];
    }
    f_rel_missing_ = (den > 0.0) ? std::sqrt(num / den) : std::sqrt(num);
  }
  for (int p = 0; p < n_objects_; ++p) {
    ObjectState& o = objects_[p];
    const bool masked = has_missing_ && ((o.model == AOADMM_MODEL_PAR2) ? par2_[mode(o.modes[0]).par2].mask != nullptr
                                                                        : (o.mask != nullptr || sparse_masked(o)));
    if (masked) {
      const double* e = em_sums_host_ + 5 * p;
      f_obj[p] = (o.model == AOADMM_MODEL_PAR2) ? o.weight * e[4]                               // :1249-1252, :1267
                                                : o.weight * (o.znorm - 2.0 * e[2] + e[3]);     // :1224-1226
    } else if (o.model == AOADMM_MODEL_PAR2 && (first || terms_->obj[p].idx_dot < 0)) {
      const Par2State& s = par2_[mode(o.modes[0]).par2];
      f_obj[p] = o.weight * s.segn_host[(size_t)s.K * 4];   // :1262-1267
    } else if (!first) {
      // f_2 = sum(last_mttkrp .* fac) with last_mttkrp = A/w (:121, :1236-1237, :1256)
      const double f2 = r[terms_->obj[p].idx_dot] / o.weight;
      const double f3 = r[terms_->obj[p].idx_had];
      f_obj[p] = o.weight * (o.znorm - 2.0 * f2 + f3);
    }
    f_tensors += f_obj[p];
  }
  for (int i = 0; i < nb_modes_; ++i) {  // :1272-1288 regularisers
    const ModeState& m = modes_[i];
    if (m.par2_role == 2) {
      if (m.constrained && reg_red_kind(m.con.kind) >= 0) f_tensors += m.con.p0 * st2[m.par2].reg;
      if (terms_->mode[i].idx_reg >= 0) f_tensors += m.con.p0 * r[terms_->mode[i].idx_reg];   // quadratic regularization
      continue;
    }
    const int ir = terms_->mode[i].idx_reg;
    if (ir >= 0) f_tensors += m.con.p0 * r[ir];
  }
  if (has_ridge_)  // :1290-1300 (second PARAFAC2 mode: the loop runs over length(G.constraint_fac{n}), :1293)
    for (int i = 0; i < nb_modes_; ++i) {
      if (modes_[i].par2_role == 2) {
        if (modes_[i].constrained) f_tensors += modes_[i].ridge * st2[modes_[i].par2].n2;
      } else {
        f_tensors += modes_[i].ridge * r[terms_->mode[i].idx_norm2];
      }
    }
  double f_coupl = 0.0;
  int nz = 0;
  for (int c = 1; c <= n_couplings_; ++c) {  // :1303-1329
    double cp = 0.0;
    for (int i = 0; i < nb_modes_; ++i)
      if (modes_[i].coupling == c) {
        const int iden = terms_->mode[i].idx_normG >= 0 ? terms_->mode[i].idx_normG : terms_->mode[i].idx_norm2;
        cp += std::sqrt(r[terms_->mode[i].idx_diffD]) / std::sqrt(r[iden]);
      }
    f_coupl += cp;
    if (cp != 0.0) ++nz;
  }
  if (f_coupl > 0.0) f_coupl /= (double)nz;
  double f_con = 0.0;
  nz = 0;
  for (int i = 0; i < nb_modes_; ++i) {  // :1332-1348
    if (!modes_[i].constrained) continue;
    const double v = (modes_[i].par2_role == 2)
                         ? st2[modes_[i].par2].con / (double)par2_[modes_[i].par2].K   // :1336-1339
                         : std::sqrt(r[terms_->mode[i].idx_diffZ]) / std::sqrt(r[terms_->mode[i].idx_norm2]);
    f_con += v;
    if (v != 0.0) ++nz;
  }
  if (f_con > 0.0) f_con /= (double)nz;
  double f_par2 = 0.0;                    // :1351-1362
  for (size_t q = 0; q < par2_.size(); ++q) f_par2 += st2[q].par2;
  if (f_par2 > 0.0) {
    // the divisor is length(Z.size{Z.modes{pp}(2)}) with pp left at P by the loop (:1361)
    const ObjectState& ol = objects_[n_objects_ - 1];
    const double div = (ol.model == AOADMM_MODEL_PAR2) ? (double)par2_[mode(ol.modes[0]).par2].K : 1.0;
    f_par2 /= div;
  }
  f[0] = f_tensors;
  f[1] = f_coupl;
  f[2] = f_con;
  f[3] = f_par2;
}

// ---------------------------------------------------------------------------------------------------
// state exchange
// ---------------------------------------------------------------------------------------------------
// Resolves a state field to its device matrix and, for the per-slice fields of a PARAFAC2 object, the row range of
// slice `slice` inside the stacked Jtot x R storage.
DevMat* Engine::par2_field(int field, int index, int slice, int64_t* row_off, int64_t* nrows) {
  *row_off = 0;
  *nrows = -1;
  auto slice_range = [&](const Par2State& s) {
    if (slice < 0 || slice >= s.K) throw CudaError(1, "state: slice index out of range");
    *row_off = s.joff[slice];
    *nrows = s.joff[slice + 1] - s.joff[slice];
  };
  switch (field) {
    case AOADMM_FIELD_FAC:
    case AOADMM_FIELD_CONSTRAINT_FAC:
    case AOADMM_FIELD_CONSTRAINT_DUAL:
    case AOADMM_FIELD_COUPLING_DUAL: {
      if (index < 1 || index > nb_modes_) throw CudaError(1, "state: mode index out of range");
      ModeState& m = modes_[index - 1];
      if (m.par2_role == 2) slice_range(par2_[m.par2]);
      if (field == AOADMM_FIELD_FAC) return &m.fac;
      if (field == AOADMM_FIELD_CONSTRAINT_FAC) return &m.Z;
      if (field == AOADMM_FIELD_CONSTRAINT_DUAL) return &m.muZ;
      return &m.muD;
    }
    case AOADMM_FIELD_COUPLING_FAC:
      if (index < 1 || index > n_couplings_) throw CudaError(1, "state: coupling index out of range");
      return &delta_[index - 1];
    case AOADMM_FIELD_PAR2_P:
    case AOADMM_FIELD_PAR2_DELTAB:
    case AOADMM_FIELD_PAR2_MU_DELTAB: {
      for (auto& s : par2_)
        if (s.p == index - 1) {
          if (field == AOADMM_FIELD_PAR2_DELTAB) return &s.DeltaB;
          slice_range(s);
          return field == AOADMM_FIELD_PAR2_P ? &s.P : &s.muDB;
        }
      throw CudaError(1, "state: object " + std::to_string(index) + " is not a PARAFAC2 object");
    }
    default: return nullptr;
  }
}

void Engine::set_state(int field, int index, int slice, const double* data, int64_t rows, int64_t cols) {
  AO_CUDA(cudaSetDevice(device_));
  if (data == nullptr) throw CudaError(1, "set_state: NULL data");
  int64_t off = 0, nr = -1;
  DevMat* d = par2_field(field, index, slice, &off, &nr);
  if (d == nullptr) throw CudaError(2, "set_state: field not supported by this build");
  if (d->p == nullptr) throw CudaError(1, "set_state: field " + std::to_string(field) + " does not exist for index " + std::to_string(index));
  const int64_t want_rows = nr >= 0 ? nr : d->rows;
  if (want_rows != rows || d->cols != cols)
    throw CudaError(1, "set_state: shape mismatch for field " + std::to_string(field) + " index " +
                           std::to_string(index) + ": expected " + std::to_string(want_rows) + "x" +
                           std::to_string(d->cols));
  if (nr >= 0)
    AO_CUDA(cudaMemcpy2DAsync(d->p + off, (size_t)d->rows * 8, data, (size_t)rows * 8, (size_t)rows * 8, (size_t)cols,
                              cudaMemcpyHostToDevice, st_));
  else
    AO_CUDA(cudaMemcpyAsync(d->p, data, d->bytes(), cudaMemcpyHostToDevice, st_));
  AO_CUDA(cudaStreamSynchronize(st_));
  if (field == AOADMM_FIELD_FAC) ++modes_[index - 1].version;
}

// Sharded PARAFAC2 slices: during the solve every rank keeps only ITS rows of the stacked per-slice state (B_k, Z_k,
// mu_Z_k, P_k, mu_DeltaB_k) up to date.  Before the state is read back the owners' rows are gathered (zero the foreign
// rows, all-reduce).  Collective: every rank reads the state after a run (the bindings do).
void Engine::par2_gather_state(Par2State& s) {
  if (!s.sharded || !s.state_stale) return;
  ModeState& mb = mode(s.m2);
  for (DevMat* d : {&mb.fac, &mb.Z, &mb.muZ, &s.P, &s.muDB}) {
    if (d->p == nullptr) continue;
    launches_ += zero_rows_outside(d->p, d->rows, (int)d->cols, s.jlo, s.jhi, st_);
    allreduce(d->p, (size_t)d->rows * d->cols);
  }
  AO_CUDA(cudaStreamSynchronize(st_));
  s.state_stale = false;
}

void Engine::prepare_state_read() {
  AO_CUDA(cudaSetDevice(device_));
  for (auto& ps : par2_) par2_gather_state(ps);
}

void Engine::get_state(int field, int index, int slice, double* data, int64_t rows, int64_t cols) {
  AO_CUDA(cudaSetDevice(device_));
  if (data == nullptr) throw CudaError(1, "get_state: NULL data");
  int64_t off = 0, nr = -1;
  DevMat* d = par2_field(field, index, slice, &off, &nr);
  if (d == nullptr) throw CudaError(2, "get_state: field not supported by this build");
  if (d->p == nullptr) throw CudaError(1, "get_state: field does not exist for this index");
  const int64_t want_rows = nr >= 0 ? nr : d->rows;
  if (want_rows != rows || d->cols != cols) throw CudaError(1, "get_state: shape mismatch");
  if (nr >= 0)
    AO_CUDA(cudaMemcpy2DAsync(data, (size_t)rows * 8, d->p + off, (size_t)d->rows * 8, (size_t)rows * 8, (size_t)cols,
                              cudaMemcpyDeviceToHost, st_));
  else
    AO_CUDA(cudaMemcpyAsync(data, d->p, d->bytes(), cudaMemcpyDeviceToHost, st_));
  AO_CUDA(cudaStreamSynchronize(st_));
}

// ---------------------------------------------------------------------------------------------------
// timing helpers
// ---------------------------------------------------------------------------------------------------
void Engine::phase_begin(int phase) {
  if (capturing_) return;  // timing events cannot be queried from inside a CUDA graph
  if (ev_used_ == ev_pool_.size()) {
    cudaEvent_t a, b;
    AO_CUDA(cudaEventCreate(&a));
    AO_CUDA(cudaEventCreate(&b));
    ev_pool_.push_back({a, b});
    ev_phase_.push_back(0);
  }
  ev_phase_[ev_used_] = phase;
  AO_CUDA(cudaEventRecord(ev_pool_[ev_used_].first, st_));
}
void Engine::phase_end() {
  if (capturing_) return;
  AO_CUDA(cudaEventRecord(ev_pool_[ev_used_].second, st_));
  ++ev_used_;
}
void Engine::phase_collect() {  // call only after a stream synchronisation
  for (size_t i = 0; i < ev_used_; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev_pool_[i].first, ev_pool_[i].second) == cudaSuccess) phase_ms_[ev_phase_[i]] += ms;
  }
  ev_used_ = 0;
}
void Engine::phase_ms(double ms[3]) {
  ms[0] = phase_ms_[0];
  ms[1] = phase_ms_[1];
  ms[2] = phase_ms_[2];
}

void Engine::check_errors(aoadmm_out* out) {
  for (int i = 0; i < n_ctl_; ++i) {
    if (ctl_host_[i].err != 0) {
      if (out) out->error_mode = i + 1;
      const int code = ctl_host_[i].err;
      throw CudaError(code, "system matrix of mode " + std::to_string(i + 1) +
                                " is not positive definite (chol would fail, cmtf_fun_AOADMM.m:142)");
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// the solver
// ---------------------------------------------------------------------------------------------------
static bool stop_one(double f, double f_old, double abs_tol, double rel_tol) {  // evaluate_stopping_conditions.m:8-15
  const double rel = (f_old > 0.0) ? std::fabs(f_old - f) / f_old : std::fabs(f_old - f);
  return (f < abs_tol) || (rel < rel_tol);
}

// One sweep over all modes (cmtf_fun_AOADMM.m:89-406): uncoupled modes first (coupl_id 0), then every coupling group.
void Engine::sweep(int iter, std::vector<int>& inner_fixed) {
  std::set<int> cset;
  for (auto& m : modes_) cset.insert(m.coupling);
  std::fill(inner_fixed.begin(), inner_fixed.end(), 0);
  for (int coupl_id : cset) {                                      // :89
    std::vector<ModeState*> cm;
    std::set<int> ps;
    for (auto& m : modes_)
      if (m.coupling == coupl_id) {
        cm.push_back(&m);
        ps.insert(m.p);
      }
    for (int p : ps) {                                             // :91
      for (ModeState* mp : cm) {                                   // :93
        ModeState& m = *mp;
        if (m.p != p) continue;
        if (m.par2_role != 0) {                                    // :157-250
          const int nterms = (coupl_id == 0) ? (m.constrained ? 1 : 0) : 1 + (m.constrained ? 1 : 0);
          if (m.par2_role == 1) {
            // :159-178, then the generic (non-third-mode) branches of the coupled precompute (:269-273, :288-294,
            // :314-318, :336-340, :358-362, :377-383): the first PARAFAC2 mode behaves like a CP mode there
            const int ct = (coupl_id == 0) ? 0 : coupling_type_[coupl_id - 1];
            const int con = m.constrained ? 1 : 0;
            if (coupl_id == 0 || ct == 0 || ct == 3 || ct == 4) par2_precompute_A(m, nterms, true);
            else if (ct == 2) par2_precompute_A(m, con, true);
            else par2_precompute_A(m, 0, false);
            if (coupl_id == 0) {
              if (!m.constrained) {
                launches_ += ls_solve(m.A.p, m.rows, m.L.p, m.invdiag, m.fac.p, m.rows, m.rows, m.R, m.ctl, st_, nullptr);  // :181
                inner_fixed[m.id - 1] = 1;
                ++m.version;
              } else {
                std::vector<ModeState*> g1{&m};
                run_admm(g1, nullptr, opt_);                       // :186
              }
              refresh_gram(m);                                     // :190
            }
          } else if (m.par2_role == 2) {
            par2_update_B(m, iter);                                // :192-218
          } else {
            const bool ls = (coupl_id == 0 && !m.constrained);
            if (m.lin >= 0 && lin_modes_[m.lin].par2c) {
              // coupling type 1: B{m}{k} stay w*C_k, the coupled system is assembled later (:283-297)
              par2_precompute_C(m, 0, false, lin_modes_[m.lin].Bsys3);
            } else if (m.lin >= 0) {
              // coupling types 2, 3, 4: per-slice systems like the exact coupling (:305-311, :327-333, :349-355);
              // type 2 replaces the coupling shift rho_k/2*I by rho_k/2*H*H'
              const LinMode& lm = lin_modes_[m.lin];
              const int con = m.constrained ? 1 : 0;
              if (lm.ctype == 2) par2_precompute_C(m, con, false, nullptr, lm.HHt.p);
              else par2_precompute_C(m, 1 + con, false);
            } else
              par2_precompute_C(m, nterms, ls);                    // :220-243
            if (ls) {
              inner_fixed[m.id - 1] = 1;
              ++m.version;
            } else if (coupl_id == 0) {
              std::vector<ModeState*> g1{&m};
              run_admm(g1, nullptr, opt_);                         // :245
            }
          }
          continue;
        }
        if (coupl_id == 0) {
          if (!m.constrained) {
            precompute_mode(m, 0, true);
            launches_ += ls_solve(m.A.p, m.rows, m.L.p, m.invdiag, m.fac.p, m.rows, m.rows, m.R, m.ctl, st_, nullptr);  // :134
            inner_fixed[m.id - 1] = 1;
            ++m.version;
          } else {
            precompute_mode(m, 1, true);                           // :141-142
            std::vector<ModeState*> g1{&m};
            run_admm(g1, nullptr, opt_);                           // :144
          }
          refresh_gram(m);                                         // :148
        } else {
          const int ct = coupling_type_[coupl_id - 1];
          const int con = m.constrained ? 1 : 0;
          if (ct == 0 || ct == 3 || ct == 4) precompute_mode(m, 1 + con, true);   // :269-273, :336-340, :358-362
          else if (ct == 2) precompute_mode(m, con, true);                         // :314-318 (rho/2*H*H' + constraint)
          else precompute_mode(m, 0, false);                                       // :288-294, :377-383: B stays w*C
        }
      }
    }
    if (coupl_id != 0) {                                           // :253
      if (coupling_type_[coupl_id - 1] == 0) {
        run_admm(cm, delta_[coupl_id - 1].p, opt_);                // :277
      } else {
        lin_prepare_group(coupl_id);
        run_admm_linear(coupl_id, cm, opt_);                       // :300, :322, :344, :366, :389
      }
      for (ModeState* mp : cm) refresh_gram(*mp);                  // :393-403
    }
  }
}

void Engine::run(const aoadmm_options* opt, aoadmm_out* out) {
  if (opt == nullptr || out == nullptr) throw CudaError(1, "run: NULL options/out");
  if (ho_patience_ > 0 && n_heldout_ == 0)
    throw CudaError(1, "run: early stopping on the held-out error is on, but no object has a held-out set any more");
  ho_best_iter_ = -1;
  AO_CUDA(cudaSetDevice(device_));
  opt_ = *opt;
  if (opt_.MaxInnerIters < 1) throw CudaError(1, "MaxInnerIters must be >= 1");
  if (opt_.mttkrp_precision < 0 || opt_.mttkrp_precision > 3)
    throw CudaError(2, "mttkrp_precision: 0 (FP64), 1 (TF32, tcgen05), 2 (BF16, tcgen05) or 3 (TF32, mma.sync)");
  out->error_mode = 0;
  out->non_finite_mode = 0;
  if (run_ev_[0] == nullptr) {
    AO_CUDA(cudaEventCreate(&run_ev_[0]));
    AO_CUDA(cudaEventCreate(&run_ev_[1]));
    AO_CUDA(cudaEventCreate(&run_ev_[2]));
  }
  AO_CUDA(cudaEventRecord(run_ev_[0], st_));
  AO_CUDA(cudaMemsetAsync(ctl_dev_, 0, sizeof(InnerCtl) * n_ctl_, st_));
  const double t_start = now_s();

  // BSUM: the objective dot product uses last_mttkrp = A before the BSUM term (:121)
  {
    bool changed = false;
    for (int p = 0; p < n_objects_; ++p) {
      ModeState& lm = mode(objects_[p].last_m);
      if (terms_->obj[p].idx_dot < 0) continue;
      const double* want = opt_.bsum ? lm.Alast.p : lm.A.p;
      RedJob& j = jobs_host_[terms_->obj[p].idx_dot];
      if (j.a != want) {
        j.a = want;
        changed = true;
      }
    }
    if (changed)
      AO_CUDA(cudaMemcpyAsync(jobs_dev_, jobs_host_.data(), sizeof(RedJob) * jobs_host_.size(), cudaMemcpyHostToDevice, st_));
  }

  for (auto& m : modes_)                    // :62-81
    if (m.par2_role != 2) refresh_gram(m);
  for (auto& s : par2_) {
    par2_refresh_gram(s);
    s.T_version = 0;
  }
  double f[4];
  em_step(false);                           // masked iteration-0 objective needs the model at the observed entries
  for (auto& o : objects_) o.ho_hist.clear();
  eval_objective(true, f);                  // :32
  record_heldout();
  f_rel_missing_ = std::nan("");
  if (out->func_rel_missing) out->func_rel_missing[0] = f_rel_missing_;
  if (out->func_val_conv) out->func_val_conv[0] = f[0];
  if (out->func_coupl_conv) out->func_coupl_conv[0] = f[1];
  if (out->func_constr_conv) out->func_constr_conv[0] = f[2];
  if (out->func_PAR2_coupl) out->func_PAR2_coupl[0] = f[3];
  if (out->time_at_it) out->time_at_it[0] = 0.0;

  std::vector<int> inner_fixed(nb_modes_, 0), fixed_captured;
  AO_CUDA(cudaEventRecord(run_ev_[2], st_));  // the outer loop starts here (iteration-0 objective done)

  // CUDA graph replay for launch-bound problems (engine knob options.graph: 0 auto, 1 on, -1 off)
  bool graph_ok = false;
  if (world_ == 1 && opt_.graph >= 0 && opt_.MaxOuterIters >= 6) {
    double elems = 0.0;
    for (auto& o : objects_) {
      double e = 1.0;
      for (auto d : o.dims) e *= (double)d;
      elems += o.sp != nullptr ? (double)o.sp->nnz : e;   // sparse objects: the work scales with nnz
    }
    graph_ok = (opt_.graph > 0) || elems <= 33554432.0;
  }
  struct GraphGuard {
    cudaGraphExec_t& g;
    ~GraphGuard() {
      if (g) cudaGraphExecDestroy(g);
      g = nullptr;
    }
  };
  cudaGraphExec_t gexec = nullptr;
  GraphGuard guard{gexec};
  int64_t graph_launches = 0;

  // early stopping on the held-out error: s_k = the sum of the held-out SSEs after iteration k (object order); k* = the
  // first k >= 1 with the smallest s_k (strictly smaller to replace, NaN never); stop once k - k* >= patience
  auto heldout_sum = [&]() {
    double t = 0.0;
    for (int p = 0; p < n_objects_; ++p)
      if (objects_[p].ho != nullptr) t += ho_sse_host_[p];
    return t;
  };
  int best_k = -1;
  double best_s = 0.0, best_f[4] = {0, 0, 0, 0}, best_rel = 0.0;
  bool ho_stop = false;

  int iter = 1;
  bool stop = false;
  while (iter <= opt_.MaxOuterIters && !stop && !ho_stop) {
    const double f_old[4] = {f[0], f[1], f[2], f[3]};
    if (gexec != nullptr) {
      // steady state of a launch-bound problem: the whole outer iteration is one CUDA-graph launch
      AO_CUDA(cudaGraphLaunch(gexec, st_));
      launches_ += graph_launches;
      inner_fixed = fixed_captured;
    } else if (graph_ok && iter >= 2 && iter > opt_.iter_start_PAR2Bkconstraint + 1 && iter < opt_.MaxOuterIters) {
      // capture this iteration (every lazy allocation / attribute call happened in iteration 1) and replay it from now on:
      // the launch sequence of an outer iteration is static because the inner-loop exit test lives on the device
      const int64_t l0 = launches_;
      cudaGraph_t graph = nullptr;
      capturing_ = true;
      AO_CUDA(cudaStreamBeginCapture(st_, cudaStreamCaptureModeRelaxed));
      try {
        sweep(iter, inner_fixed);
        em_step(true);
        enqueue_objective(false);
      } catch (...) {
        cudaStreamEndCapture(st_, &graph);
        if (graph) cudaGraphDestroy(graph);
        capturing_ = false;
        throw;
      }
      capturing_ = false;
      AO_CUDA(cudaStreamEndCapture(st_, &graph));
      const cudaError_t ie = cudaGraphInstantiate(&gexec, graph, 0);
      cudaGraphDestroy(graph);
      if (ie != cudaSuccess) {
        gexec = nullptr;
        throw CudaError(5, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ie));
      }
      graph_launches = launches_ - l0;
      fixed_captured = inner_fixed;
      AO_CUDA(cudaGraphLaunch(gexec, st_));
    } else {
      sweep(iter, inner_fixed);
      em_step(true);                                                 // :408-441
      enqueue_objective(false);                                      // :447
    }
    finish_objective(false, f);                                      // synchronises
    record_heldout();
    check_errors(out);
    if (out->func_val_conv) out->func_val_conv[iter] = f[0];
    if (out->func_coupl_conv) out->func_coupl_conv[iter] = f[1];
    if (out->func_constr_conv) out->func_constr_conv[iter] = f[2];
    if (out->func_PAR2_coupl) out->func_PAR2_coupl[iter] = f[3];
    if (out->time_at_it) out->time_at_it[iter] = now_s() - t_start;
    if (out->func_rel_missing) out->func_rel_missing[iter] = f_rel_missing_;
    if (out->inner_iters)
      for (int i = 0; i < nb_modes_; ++i)
        out->inner_iters[(size_t)(iter - 1) * nb_modes_ + i] =
            inner_fixed[i] ? inner_fixed[i] : ctl_host_[modes_[i].ctl_index].iters;
    stop = stop_one(f[0], f_old[0], opt_.AbsFuncTol, opt_.OuterRelTol) &&
           stop_one(f[1], f_old[1], opt_.AbsFuncTol, opt_.OuterRelTol) &&
           stop_one(f[2], f_old[2], opt_.AbsFuncTol, opt_.OuterRelTol) &&
           stop_one(f[3], f_old[3], opt_.AbsFuncTol, opt_.OuterRelTol);   // evaluate_stopping_conditions.m:44
    if (has_missing_) stop = stop && (f_rel_missing_ < opt_.OuterRelTol);  // :457-459
    if (ho_patience_ > 0) {
      const double sk = heldout_sum();
      if (best_k < 0 ? !std::isnan(sk) : sk < best_s) {
        best_k = iter;
        best_s = sk;
        std::copy(f, f + 4, best_f);
        best_rel = f_rel_missing_;
        // a later restore needs this state only when the run goes on (every rank decides alike: the SSE is replicated)
        if (!stop && iter < opt_.MaxOuterIters) snapshot_state();
      } else if (best_k > 0 && iter - best_k >= ho_patience_ && !stop && iter < opt_.MaxOuterIters) {
        ho_stop = true;   // the held-out rule ends the run only where the other rules would not
      }
    }
    ++iter;
  }
  const int n_run = iter - 1;
  int exit_flag = 0;
  if (ho_stop) {
    exit_flag = 1 << 9;
  } else if (iter <= opt_.MaxOuterIters) {                           // make_exit_flag.m:4-5
    exit_flag = 1 << 8;
    for (int q = 0; q < 4; ++q)
      if (f[q] < opt_.AbsFuncTol) exit_flag |= (1 << q);
  }
  if (ho_patience_ > 0) {
    if (best_k < 0) {   // no iteration (n = 0) or only NaN sums: the last state is kept
      best_k = n_run;
      best_s = heldout_sum();
    } else if (best_k < n_run) {
      restore_state();
      std::copy(best_f, best_f + 4, f);
      f_rel_missing_ = best_rel;
    }
    ho_best_iter_ = best_k;
    ho_best_sse_ = best_s;
  }
  AO_CUDA(cudaEventRecord(run_ev_[1], st_));
  AO_CUDA(cudaEventSynchronize(run_ev_[1]));
  {
    float ms = 0.f;
    AO_CUDA(cudaEventElapsedTime(&ms, run_ev_[0], run_ev_[1]));
    last_run_ms_ = ms;
    AO_CUDA(cudaEventElapsedTime(&ms, run_ev_[2], run_ev_[1]));
    last_loop_ms_ = ms;
  }
  out->f_tensors = f[0];
  out->f_couplings = f[1];
  out->f_constraints = f[2];
  out->f_PAR2_couplings = f[3];
  out->f_rel_missing = has_missing_ ? f_rel_missing_ : std::nan("");
  out->OuterIterations = n_run;
  for (int i = n_ctl_ - 1; i >= 0; --i)
    if (ctl_host_[i].warn != 0) out->non_finite_mode = i + 1;
  out->exit_flag = exit_flag;
}

// ---------------------------------------------------------------------------------------------------
// benchmark helpers
// ---------------------------------------------------------------------------------------------------
void Engine::generate_cp_data(int object, const double* const* factors, double noise, uint64_t seed) {
  AO_CUDA(cudaSetDevice(device_));
  if (object < 1 || object > n_objects_) throw CudaError(1, "generate_cp_data: object out of range");
  ObjectState& o = objects_[object - 1];
  if (o.model != AOADMM_MODEL_CP) throw CudaError(1, "generate_cp_data: not a CP object");
  if (o.sp != nullptr) throw CudaError(2, "generate_cp_data: object " + std::to_string(object) + " is sparse (dense objects only)");
  const int R = mode(o.modes[0]).R;
  GenArgs g{};
  g.order = o.order;
  g.R = R;
  std::vector<double*> tmp(o.order, nullptr);
  for (int d = 0; d < o.order; ++d) {
    const ModeState& mm = mode(o.modes[d]);
    g.dims[d] = o.dims[d];
    AO_CUDA(cudaMalloc(&tmp[d], (size_t)mm.rows * R * sizeof(double)));
    AO_CUDA(cudaMemcpyAsync(tmp[d], factors[d], (size_t)mm.rows * R * sizeof(double), cudaMemcpyHostToDevice, st_));
    g.fac[d] = tmp[d];
    g.fld[d] = mm.rows;
  }
  g.full_last = o.last_full;
  g.shard_offset = o.shard_offset;
  g.ld0 = o.ld0;
  double* sums = nullptr;
  const int ctas = 148 * 8;
  AO_CUDA(cudaMalloc(&sums, (4 + 2 * ctas) * sizeof(double)));
  AO_CUDA(cudaMemsetAsync(sums, 0, (4 + 2 * ctas) * sizeof(double), st_));
  double h[4];
  gen_cp_kernel<<<ctas, 256, 0, st_>>>(g, o.data, seed, 0, 0.0, 1.0, sums);
  AO_CHECK_LAUNCH();
  gen_sum_kernel<<<1, 256, 0, st_>>>(sums, ctas, 0, 1);
  AO_CHECK_LAUNCH();
  if (o.sharded) allreduce(sums, 2);
  AO_CUDA(cudaMemcpyAsync(h, sums, sizeof(h), cudaMemcpyDeviceToHost, st_));
  AO_CUDA(cudaStreamSynchronize(st_));
  const double sigma = (noise > 0.0) ? noise * std::sqrt(h[0]) / std::sqrt(h[1]) : 0.0;  // create_coupled_data.m:161
  gen_cp_kernel<<<ctas, 256, 0, st_>>>(g, o.data, seed, 1, sigma, 1.0, sums);
  AO_CHECK_LAUNCH();
  gen_sum_kernel<<<1, 256, 0, st_>>>(sums, ctas, 2, 0);
  AO_CHECK_LAUNCH();
  if (o.sharded) allreduce(sums + 2, 1);
  AO_CUDA(cudaMemcpyAsync(h, sums, sizeof(h), cudaMemcpyDeviceToHost, st_));
  AO_CUDA(cudaStreamSynchronize(st_));
  gen_cp_kernel<<<ctas, 256, 0, st_>>>(g, o.data, seed, 2, 0.0, 1.0 / std::sqrt(h[2]), sums);  // script6 :101-102
  AO_CHECK_LAUNCH();
  AO_CUDA(cudaStreamSynchronize(st_));
  launches_ += 5;
  o.znorm = 1.0;
  o.T_version = 0;  // cached partial contractions refer to the old data
  refresh_transposed(o);
  for (auto p : tmp) cudaFree(p);
  cudaFree(sums);
}

// position of this rank's slab of CP object `object` inside the whole object (elements, column-major)
void Engine::object_slab(int object, int64_t* offset_elems, int64_t* n_elems) const {
  if (object < 1 || object > n_objects_) throw CudaError(1, "object out of range");
  const ObjectState& o = objects_[object - 1];
  if (o.model != AOADMM_MODEL_CP) throw CudaError(1, "not a CP object");
  if (o.sp != nullptr) throw CudaError(2, "get_object_data: object " + std::to_string(object) + " is sparse (dense objects only)");
  int64_t lead = 1;
  for (int d = 0; d + 1 < o.order; ++d) lead *= o.dims[d];
  *offset_elems = lead * o.shard_offset;
  *n_elems = lead * o.dims[o.order - 1];
}

void Engine::object_to_host(int object, double* out, int64_t n_elements) {
  AO_CUDA(cudaSetDevice(device_));
  if (object < 1 || object > n_objects_) throw CudaError(1, "get_object_data: object out of range");
  ObjectState& o = objects_[object - 1];
  if (o.model != AOADMM_MODEL_CP) throw CudaError(1, "get_object_data: not a CP object");
  if (o.sp != nullptr) throw CudaError(2, "get_object_data: object " + std::to_string(object) + " is sparse (dense objects only)");
  size_t slab = 1;
  for (int d = 1; d < o.order; ++d) slab *= (size_t)o.dims[d];
  if ((int64_t)((size_t)o.dims[0] * slab) != n_elements) throw CudaError(1, "get_object_data: size mismatch");
  AO_CUDA(cudaStreamSynchronize(st_));
  AO_CUDA(cudaMemcpy2D(out, (size_t)o.dims[0] * 8, o.data, (size_t)o.ld0 * 8, (size_t)o.dims[0] * 8, slab,
                       cudaMemcpyDeviceToHost));
}

void Engine::nvecs_to_host(int mode_id, int slice, int r, double* out, int64_t rows, double* info) {
  AO_CUDA(cudaSetDevice(device_));
  if (mode_id < 1 || mode_id > nb_modes_) throw CudaError(1, "nvecs: mode out of range");
  // the first object that contains the mode (cmtf_nvecs.m:36-51)
  int p = -1, pos = -1;
  for (int q = 0; q < n_objects_ && p < 0; ++q)
    for (int d = 0; d < objects_[q].order; ++d)
      if (objects_[q].modes[d] == mode_id) {
        p = q;
        pos = d;
        break;
      }
  if (p < 0) throw CudaError(1, "nvecs: no object contains this mode");
  ObjectState& o = objects_[p];
  UnfoldSpec s;
  bool reduce_over_ranks = false, skip_local_gram = false;
  if (o.sp != nullptr)
    throw CudaError(2, "nvecs: mode " + std::to_string(mode_id) + " belongs to a sparse object (initialise it from a distribution)");
  if (o.model == AOADMM_MODEL_CP) {
    if (slice != 0) throw CudaError(1, "nvecs: slice given for a CP mode");
    if (o.sharded && pos == o.order - 1) {
      nvecs_sharded_mode(o, r, out, rows, info);
      return;
    }
    const View3& v = o.views[pos];
    const Tensor3& t = v.t;
    s.X = t.X;
    if (v.kernel_pos == 0) {
      s.layout = 0;
      s.n = t.I;
      s.ld = t.ldI;
      s.ncols = t.J * t.K;
    } else if (v.kernel_pos == 1) {
      s.layout = 1;
      s.n = t.J;
      s.I = t.I;
      s.cs = t.ldI;
      s.bs = t.ldI * t.J;
      s.nb = t.K;
    } else {
      s.layout = 1;
      s.n = t.K;
      s.I = t.I;
      s.cs = t.ldI * t.J;
      s.bs = t.ldI;
      s.nb = t.J;
    }
    reduce_over_ranks = o.sharded;
  } else {
    Par2State* ps = nullptr;
    for (auto& c : par2_)
      if (c.p == p) ps = &c;
    if (ps == nullptr) throw CudaError(1, "nvecs: PARAFAC2 state missing");
    if (pos == 0) {          // init_coupled_AOADMM_CMTF.m:55-60: slices side by side
      if (slice != 0) throw CudaError(1, "nvecs: slice given for PARAFAC2 mode A");
      s.X = ps->X_alloc;     // this rank's slices; the partial Gram matrices are summed over the ranks
      s.layout = 0;
      s.n = ps->I;
      s.ld = ps->ldX;
      s.ncols = ps->jhi - ps->jlo;
      reduce_over_ranks = ps->sharded;
    } else if (pos == 1) {   // :61-66: X_k' X_k
      if (slice < 1 || slice > ps->K) throw CudaError(1, "nvecs: PARAFAC2 slice out of range");
      if (ps->sharded) {     // only the owner of the slice holds it: the others contribute a zero matrix to the sum
        reduce_over_ranks = true;
        skip_local_gram = (slice - 1 < ps->k0 || slice - 1 >= ps->k1);
      }
      s.X = skip_local_gram ? ps->X_alloc : ps->X + ps->joff[slice - 1] * ps->ldX;
      s.layout = 1;
      s.n = ps->joff[slice] - ps->joff[slice - 1];
      s.I = ps->I;
      s.cs = ps->ldX;
      s.bs = 0;
      s.nb = 1;
    } else {
      throw CudaError(1, "nvecs: PARAFAC2 mode C is initialised with ones (init_coupled_AOADMM_CMTF.m:68)");
    }
  }
  if (rows != s.n) throw CudaError(1, "nvecs: output rows do not match the mode size");
  if (r < 1 || r > s.n) throw CudaError(1, "nvecs: the number of vectors must be between 1 and the mode size");
  double *Y = nullptr, *work = nullptr, *U = nullptr;
  const size_t nn = (size_t)s.n * (size_t)s.n;
  try {
    AO_CUDA(cudaMalloc(&Y, std::max<size_t>(nn * sizeof(double), 256)));
    AO_CUDA(cudaMalloc(&work, std::max<size_t>(unfold_gram_workspace(s) * sizeof(double), 256)));
    AO_CUDA(cudaMalloc(&U, std::max<size_t>((size_t)s.n * r * sizeof(double), 256)));
    if (skip_local_gram) AO_CUDA(cudaMemsetAsync(Y, 0, nn * sizeof(double), st_));
    else launches_ += unfold_gram(s, Y, work, st_);
    if (reduce_over_ranks) allreduce(Y, nn);
    std::vector<double> theta(r);
    const EigInfo ei = top_eigvecs(Y, s.n, r, U, theta.data(), st_);
    launches_ += ei.launches;
    if (info != nullptr) {
      info[0] = ei.iterations;
      info[1] = ei.residual;
    }
    AO_CUDA(cudaMemcpyAsync(out, U, (size_t)s.n * r * sizeof(double), cudaMemcpyDeviceToHost, st_));
    AO_CUDA(cudaStreamSynchronize(st_));
  } catch (...) {
    cudaFree(Y);
    cudaFree(work);
    cudaFree(U);
    throw;
  }
  cudaFree(Y);
  cudaFree(work);
  cudaFree(U);
}

// nvecs of the mode the tensor is sharded along (the last one): Y(k,k') = <X(:,:,k), X(:,:,k')> needs pairs of slices
// that live on different GPUs.  The middle extent J is cut into chunks; chunk c is gathered on rank c mod P with NCCL
// point-to-point transfers over NVLink (every rank sends its k-range of the chunk, packed, straight into the owner's
// buffer at its place in the global k order), the owner adds the chunk's K x K Gram matrix with the same DMMA kernel, and
// one all-reduce at the end sums the owners' partial matrices.  Each slab crosses NVLink once.
void Engine::nvecs_sharded_mode(ObjectState& o, int r, double* out, int64_t rows, double* info) {
  if (!nccl_->Send || !nccl_->Recv || !nccl_->GroupStart || !nccl_->GroupEnd)
    throw CudaError(6, "libnccl.so.2 lacks ncclSend/ncclRecv (needed for nvecs of the sharded mode)");
  const Tensor3& t = o.views[o.order - 1].t;   // I x J x Kloc, leading dimension ldI
  const long long Kt = o.last_full, Kloc = t.K, J = t.J, ld = t.ldI;
  if (rows != Kt) throw CudaError(1, "nvecs: output rows do not match the mode size");
  if (r < 1 || r > Kt) throw CudaError(1, "nvecs: the number of vectors must be between 1 and the mode size");
  // slab ranges of all ranks (the caller chooses them): one all-reduce of a zero-padded table
  std::vector<double> tab(2 * (size_t)world_, 0.0);
  tab[2 * rank_] = (double)o.shard_offset;
  tab[2 * rank_ + 1] = (double)Kloc;
  double* tab_dev = nullptr;
  AO_CUDA(cudaMalloc(&tab_dev, tab.size() * sizeof(double)));
  AO_CUDA(cudaMemcpyAsync(tab_dev, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st_));
  allreduce(tab_dev, tab.size());
  AO_CUDA(cudaMemcpyAsync(tab.data(), tab_dev, tab.size() * sizeof(double), cudaMemcpyDeviceToHost, st_));
  AO_CUDA(cudaStreamSynchronize(st_));
  cudaFree(tab_dev);
  long long Kmax = 0;
  for (int q = 0; q < world_; ++q) Kmax = std::max<long long>(Kmax, (long long)tab[2 * q + 1]);
  // chunk width: gathered chunk <= 256 MB, at least one chunk per rank when J allows
  long long cj = std::max<long long>(1, (256LL << 20) / std::max<long long>(ld * Kt * 8, 1));
  cj = std::min(cj, std::max<long long>(1, ceil_div(J, world_)));
  const long long nchunks = ceil_div(J, cj), ngroups = ceil_div(nchunks, world_);
  const size_t nn = (size_t)Kt * (size_t)Kt;
  UnfoldSpec s;
  s.layout = 1;
  s.n = Kt;
  s.I = t.I;
  s.bs = ld;
  double *gathered = nullptr, *send = nullptr, *Y = nullptr, *work = nullptr, *U = nullptr;
  try {
    AO_CUDA(cudaMalloc(&gathered, std::max<size_t>((size_t)ld * cj * Kt * 8, 256)));
    AO_CUDA(cudaMalloc(&send, std::max<size_t>((size_t)ld * cj * std::max<long long>(Kloc, 1) * 8 * world_, 256)));
    AO_CUDA(cudaMalloc(&Y, std::max<size_t>(nn * 8, 256)));
    AO_CUDA(cudaMalloc(&U, std::max<size_t>((size_t)Kt * r * 8, 256)));
    AO_CUDA(cudaMemsetAsync(Y, 0, nn * 8, st_));
    s.X = gathered;
    s.cs = ld * cj;   // upper bound for the workspace query
    s.nb = cj;
    AO_CUDA(cudaMalloc(&work, std::max<size_t>(unfold_gram_workspace(s) * 8, 256)));
    const size_t part = (size_t)ld * cj * std::max<long long>(Kloc, 1);
    for (long long g = 0; g < ngroups; ++g) {
      // pack this rank's k-range of the P chunks of the group (chunk g*P + p goes to rank p)
      for (int p = 0; p < world_; ++p) {
        const long long j0 = (g * world_ + p) * cj, w = std::min(cj, J - j0);
        if (w <= 0 || Kloc <= 0) continue;
        AO_CUDA(cudaMemcpy2DAsync(send + part * p, (size_t)w * ld * 8, t.X + j0 * ld, (size_t)J * ld * 8, (size_t)w * ld * 8,
                                  (size_t)Kloc, cudaMemcpyDeviceToDevice, st_));
      }
      const long long myj0 = (g * world_ + rank_) * cj, myw = std::min(cj, J - myj0);
      AO_NCCL(nccl_->GroupStart());
      for (int p = 0; p < world_; ++p) {
        const long long j0 = (g * world_ + p) * cj, w = std::min(cj, J - j0);
        if (w <= 0) continue;
        if (p != rank_) {
          if (Kloc > 0)
            AO_NCCL(nccl_->Send(send + part * p, (size_t)(w * ld * Kloc), ncclDouble, p, static_cast<ncclComm_t>(comm_), st_));
        } else {
          for (int q = 0; q < world_; ++q) {
            const long long off = (long long)tab[2 * q], kq = (long long)tab[2 * q + 1];
            if (q == rank_ || kq <= 0) continue;
            AO_NCCL(nccl_->Recv(gathered + (size_t)off * w * ld, (size_t)(w * ld * kq), ncclDouble, q,
                                static_cast<ncclComm_t>(comm_), st_));
          }
        }
      }
      AO_NCCL(nccl_->GroupEnd());
      if (myw > 0) {
        if (Kloc > 0)
          AO_CUDA(cudaMemcpyAsync(gathered + (size_t)o.shard_offset * myw * ld, send + part * rank_,
                                  (size_t)myw * ld * Kloc * 8, cudaMemcpyDeviceToDevice, st_));
        s.cs = ld * myw;   // element (i, jj, k) of the gathered chunk at i + ld*(jj + myw*k)
        s.nb = myw;
        launches_ += unfold_gram(s, Y, work, st_, true);
      }
    }
    allreduce(Y, nn);
    std::vector<double> theta(r);
    const EigInfo ei = top_eigvecs(Y, Kt, r, U, theta.data(), st_);
    launches_ += ei.launches;
    if (info != nullptr) {
      info[0] = ei.iterations;
      info[1] = ei.residual;
    }
    AO_CUDA(cudaMemcpyAsync(out, U, (size_t)Kt * r * sizeof(double), cudaMemcpyDeviceToHost, st_));
    AO_CUDA(cudaStreamSynchronize(st_));
  } catch (...) {
    cudaFree(gathered);
    cudaFree(send);
    cudaFree(Y);
    cudaFree(work);
    cudaFree(U);
    throw;
  }
  cudaFree(gathered);
  cudaFree(send);
  cudaFree(Y);
  cudaFree(work);
  cudaFree(U);
}

void Engine::nvecs_sparse_to_host(int mode_id, int r, double* out, int64_t rows, double* info) {
  AO_CUDA(cudaSetDevice(device_));
  if (mode_id < 1 || mode_id > nb_modes_) throw CudaError(1, "nvecs_sparse: mode out of range");
  int p = -1, pos = -1;   // the first object that contains the mode, as for nvecs
  for (int q = 0; q < n_objects_ && p < 0; ++q)
    for (int d = 0; d < objects_[q].order; ++d)
      if (objects_[q].modes[d] == mode_id) {
        p = q;
        pos = d;
        break;
      }
  if (p < 0) throw CudaError(1, "nvecs_sparse: no object contains this mode");
  ObjectState& o = objects_[p];
  if (o.sp == nullptr)
    throw CudaError(1, "nvecs_sparse: mode " + std::to_string(mode_id) +
                           " belongs to a dense or PARAFAC2 object (use aoadmm_nvecs)");
  const SparseTensor& sp = *o.sp;
  if (o.sharded && pos == o.order - 1)
    throw CudaError(2, "nvecs_sparse: mode " + std::to_string(mode_id) +
                           " is the sharded last mode of a sparse object (its fibers cross GPUs)");
  const long long n = sp.dims[pos];
  if (rows != n) throw CudaError(1, "nvecs_sparse: output rows do not match the mode size");
  if (r < 1 || r > n) throw CudaError(1, "nvecs_sparse: the number of vectors must be between 1 and the mode size");
  // build and chunk buffers (the chunk width c may differ between ranks: the bits of W do not depend on it).  A failure
  // on one rank must not leave the others in a collective, so every rank learns whether all succeeded (c > 0 on every
  // rank) before the iteration.
  std::unique_ptr<FiberUnfolding> fu;
  std::exception_ptr err;
  int c = 0;
  try {
    fu.reset(new FiberUnfolding(sp, pos, st_));
    size_t free_b = 0, total_b = 0;
    AO_CUDA(cudaMemGetInfo(&free_b, &total_b));
    c = fu->chunk_columns(eig_block(n, r), free_b / 2);
    if (c > 0) fu->reserve(c);
  } catch (...) {
    err = std::current_exception();
    c = 0;
  }
  if (world_ > 1) {
    std::vector<double> tab((size_t)world_, 0.0);
    tab[rank_] = (double)c;
    double* tab_dev = nullptr;
    AO_CUDA(cudaMalloc(&tab_dev, tab.size() * sizeof(double)));
    AO_CUDA(cudaMemcpyAsync(tab_dev, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st_));
    allreduce(tab_dev, tab.size());
    AO_CUDA(cudaMemcpyAsync(tab.data(), tab_dev, tab.size() * sizeof(double), cudaMemcpyDeviceToHost, st_));
    AO_CUDA(cudaStreamSynchronize(st_));
    cudaFree(tab_dev);
    for (double v : tab) c = std::min(c, (int)v);
  }
  if (err) std::rethrow_exception(err);
  if (c == 0) throw CudaError(7, "nvecs_sparse: not even one column of the sparse operator fits in half of the free device memory");
  double* U = nullptr;
  try {
    AO_CUDA(cudaMalloc(&U, std::max<size_t>((size_t)n * r * sizeof(double), 256)));
    // W = Y V; with several GPUs each rank's fibers give its share, summed by one all-reduce per application
    const EigOperator apply = [&](const double* V, double* W, int cols) {
      const int L = fu->apply(V, W, cols, st_);
      allreduce(W, (size_t)n * cols);
      return L;
    };
    std::vector<double> theta(r);
    const EigInfo ei = top_eigvecs(apply, n, r, U, theta.data(), st_);
    launches_ += ei.launches;
    if (info != nullptr) {
      info[0] = ei.iterations;
      info[1] = ei.residual;
    }
    AO_CUDA(cudaMemcpyAsync(out, U, (size_t)n * r * sizeof(double), cudaMemcpyDeviceToHost, st_));
    AO_CUDA(cudaStreamSynchronize(st_));
  } catch (...) {
    cudaFree(U);
    throw;
  }
  cudaFree(U);
}

void Engine::mttkrp_to_host(int object, int pos, double* out, int precision) {
  AO_CUDA(cudaSetDevice(device_));
  if (object < 1 || object > n_objects_) throw CudaError(1, "mttkrp: object out of range");
  ObjectState& o = objects_[object - 1];
  if (o.model != AOADMM_MODEL_CP) throw CudaError(1, "mttkrp: not a CP object");
  if (pos < 1 || pos > o.order) throw CudaError(1, "mttkrp: position out of range");
  ModeState& m = mode(o.modes[pos - 1]);
  const int saved = opt_.mttkrp_precision;
  if (precision >= 0) opt_.mttkrp_precision = precision;
  try {
    compute_mttkrp(o, pos - 1, 1.0, m.A.p, m.rows);
  } catch (...) {
    opt_.mttkrp_precision = saved;
    throw;
  }
  opt_.mttkrp_precision = saved;
  AO_CUDA(cudaMemcpyAsync(out, m.A.p, m.A.bytes(), cudaMemcpyDeviceToHost, st_));
  AO_CUDA(cudaStreamSynchronize(st_));
  phase_collect();
}

float Engine::time_mttkrp(int object, int pos, int reps) {
  AO_CUDA(cudaSetDevice(device_));
  if (object < 1 || object > n_objects_) throw CudaError(1, "time_mttkrp: object out of range");
  ObjectState& o = objects_[object - 1];
  if (o.model != AOADMM_MODEL_CP) throw CudaError(1, "time_mttkrp: not a CP object");
  if (pos < 1 || pos > o.order) throw CudaError(1, "time_mttkrp: position out of range");
  ModeState& m = mode(o.modes[pos - 1]);
  cudaEvent_t a, b;
  if (o.sp != nullptr) {   // the whole sparse MTTKRP: factor transposes, unit pass, fix-up, output transpose
    AO_CUDA(cudaEventCreate(&a));
    AO_CUDA(cudaEventCreate(&b));
    launches_ += sparse_mttkrp_of(o, pos - 1, 1.0, m.Alast.p, m.rows);  // warm-up
    AO_CUDA(cudaEventRecord(a, st_));
    for (int r = 0; r < reps; ++r) launches_ += sparse_mttkrp_of(o, pos - 1, 1.0, m.Alast.p, m.rows);
    AO_CUDA(cudaEventRecord(b, st_));
    AO_CUDA(cudaEventSynchronize(b));
    float ms = 0.f;
    AO_CUDA(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return ms / (float)std::max(reps, 1);
  }
  View3& v = o.views[pos - 1];
  pack_operand(v, 0);
  pack_operand(v, 1);
  AO_CUDA(cudaEventCreate(&a));
  AO_CUDA(cudaEventCreate(&b));
  const int R = m.R;
  const int prec = opt_.mttkrp_precision;  // precision of the last aoadmm_run (0 before any run)
  const bool tc = (prec == 1 || prec == 2) && o.order == 3;
  const int legacy = (prec == 3 && o.order >= 3) ? 1 : 0;
  if (legacy) {
    packed_factor_to_tf32(v.f0, st_, nullptr);
    ++launches_;
  }
  auto one = [&]() {
    if (tc) return tc_mttkrp(o, pos - 1, 1.0, m.Alast.p + v.out_offset, m.rows, nullptr, prec);
    return mttkrp3(v.t, v.kernel_pos, v.f0, v.f1, R, 1.0, m.Alast.p + v.out_offset, m.rows, mws_, st_, nullptr, nullptr, legacy);
  };
  launches_ += one();  // warm-up
  AO_CUDA(cudaEventRecord(a, st_));
  for (int r = 0; r < reps; ++r) launches_ += one();
  AO_CUDA(cudaEventRecord(b, st_));
  AO_CUDA(cudaEventSynchronize(b));
  float ms = 0.f;
  AO_CUDA(cudaEventElapsedTime(&ms, a, b));
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  return ms / (float)std::max(reps, 1);
}

// ---------------------------------------------------------------------------------------------------
// held-out entries (aoadmm_model_at, aoadmm_set_heldout, aoadmm_heldout_history)
// ---------------------------------------------------------------------------------------------------
void Engine::check_entries(int object, const aoadmm_sparse_object* entries, bool heldout) const {
  const std::string who = std::string(heldout ? "set_heldout" : "model_at") + ": object " + std::to_string(object);
  if (object < 1 || object > n_objects_) throw CudaError(1, who + " is out of range");
  const ObjectState& o = objects_[object - 1];
  if (o.model != AOADMM_MODEL_CP) throw CudaError(1, who + " is a PARAFAC2 object (CP objects only)");
  if (entries == nullptr) return;
  if (entries->nnz < 0) throw CudaError(1, who + ": nnz is negative");
  if (entries->nnz > 0x7fffffffLL - kSparseChunk) throw CudaError(1, who + ": more than 2^31 - 257 entries");
  if (entries->nnz > 0 && (entries->subs == nullptr || (heldout && entries->vals == nullptr)))
    throw CudaError(1, who + ": subs / vals is NULL");
  if (heldout && o.mask == nullptr && !sparse_masked(o))
    throw CudaError(1, who + " has no missing data (a held-out set needs a dense Z.miss or a sparse mask)");
  for (int d = 0; d < o.order; ++d) {
    const int64_t rows = modes_[o.modes[d] - 1].rows;
    const int64_t* sd = entries->subs + (size_t)d * (size_t)entries->nnz;
    for (int64_t e = 0; e < entries->nnz; ++e)
      if (sd[e] < 0 || sd[e] >= rows)
        throw CudaError(1, who + ": subscript " + std::to_string(sd[e]) + " of entry " + std::to_string(e) +
                               " is out of range for mode position " + std::to_string(d + 1));
  }
}

void Engine::model_at(int object, const aoadmm_sparse_object* entries, double* out) {
  AO_CUDA(cudaSetDevice(device_));
  const ObjectState& o = objects_[object - 1];
  const double* fac[8];
  long long rows[8];
  for (int d = 0; d < o.order; ++d) {
    const ModeState& md = modes_[o.modes[d] - 1];
    fac[d] = md.fac.p;
    rows[d] = md.rows;
  }
  model_at_host(o.order, modes_[o.modes[0] - 1].R, fac, rows, entries->nnz,
                reinterpret_cast<const long long*>(entries->subs), out, st_);
}

void Engine::set_heldout(int object, const aoadmm_sparse_object* entries) {
  AO_CUDA(cudaSetDevice(device_));
  ObjectState& o = objects_[object - 1];
  if (o.ho != nullptr) {
    AO_CUDA(cudaStreamSynchronize(st_));
    heldout_free(*o.ho);
    delete o.ho;
    o.ho = nullptr;
    o.ho_hist.clear();
    --n_heldout_;
  }
  if (entries == nullptr) return;
  if (ho_sse_ == nullptr) {
    AO_CUDA(cudaMalloc(&ho_sse_, sizeof(double) * n_objects_));
    AO_CUDA(cudaMemset(ho_sse_, 0, sizeof(double) * n_objects_));
    AO_CUDA(cudaMallocHost(&ho_sse_host_, sizeof(double) * n_objects_));
  }
  std::unique_ptr<HeldOut> h(new HeldOut());
  long long dims[8];
  for (int d = 0; d < o.order; ++d) dims[d] = modes_[o.modes[d] - 1].rows;
  try {
    heldout_build(*h, o.order, dims, modes_[o.modes[0] - 1].R, entries->nnz,
                  reinterpret_cast<const long long*>(entries->subs), entries->vals, st_);
    // a held-out entry that was observed in training would make the validation error meaningless
    long long first = -1, count = 0;
    if (o.sp != nullptr) {
      count = heldout_stored(*h, *o.sp, &first, st_);
    } else {
      std::vector<long long> ld(o.dims.begin(), o.dims.end());
      count = heldout_masked(*h, o.mask, o.ld0, ld.data(), o.shard_offset, &first, st_);
    }
    if (o.sharded) {   // each rank checked the entries of its slab: one all-reduce of the counts and first positions
      std::vector<double> hb(world_ + 1, 0.0);
      hb[0] = (double)count;
      hb[1 + rank_] = (double)(first + 1);
      double* db = nullptr;
      AO_CUDA(cudaMalloc(&db, hb.size() * sizeof(double)));
      try {
        AO_CUDA(cudaMemcpyAsync(db, hb.data(), hb.size() * sizeof(double), cudaMemcpyHostToDevice, st_));
        allreduce(db, hb.size());
        AO_CUDA(cudaMemcpyAsync(hb.data(), db, hb.size() * sizeof(double), cudaMemcpyDeviceToHost, st_));
        AO_CUDA(cudaStreamSynchronize(st_));
      } catch (...) {
        cudaFree(db);
        throw;
      }
      cudaFree(db);
      count = (long long)hb[0];
      first = -1;
      for (int r = 0; r < world_ && first < 0; ++r)
        if (hb[1 + r] > 0.0) first = (long long)hb[1 + r] - 1;
    }
    if (count > 0) {
      long long sub[8];
      heldout_subscript(*h, first, sub, st_);
      std::string s = "(";
      for (int d = 0; d < o.order; ++d) s += (d ? ", " : "") + std::to_string(sub[d]);
      throw CudaError(1, "set_heldout: object " + std::to_string(object) + ": " + std::to_string(count) +
                             " held-out entries are observed in training, e.g. the entry at 0-based subscript " + s + ")");
    }
  } catch (...) {
    heldout_free(*h);
    throw;
  }
  o.ho = h.release();
  ++n_heldout_;
}

void Engine::heldout_history(int object, double* sse, int64_t n, int64_t* count) const {
  if (object < 1 || object > n_objects_) throw CudaError(1, "heldout_history: object out of range");
  const ObjectState& o = objects_[object - 1];
  if (o.ho == nullptr) throw CudaError(1, "heldout_history: object " + std::to_string(object) + " has no held-out set");
  for (int64_t i = 0; i < n; ++i) sse[i] = i < (int64_t)o.ho_hist.size() ? o.ho_hist[i] : std::nan("");
  if (count != nullptr) *count = o.ho->n;
}

// ---------------------------------------------------------------------------------------------------
// early stopping on the held-out error (aoadmm_set_heldout_stopping, aoadmm_heldout_best)
// ---------------------------------------------------------------------------------------------------
// The snapshot list is every device buffer whose value after an outer iteration a later run reads before rewriting it:
// G (fac, constraint_fac, constraint_dual_fac, coupling_dual_fac of every mode, coupling_fac of every coupling) and the
// PARAFAC2 P, DeltaB, mu_DeltaB.  Everything else carried over is a function of these and is rebuilt at restore: the
// imputation of missing entries (the EM pass), the dimension-tree contraction and the version stamps; the Grams and the
// packed operands are recomputed by every run and every MTTKRP.  The sweep's other buffers (A, Alast under BSUM, the
// linear-coupling Dold / Zold, the PARAFAC2 PDold / Vprev / per-slice systems) are written in every outer iteration
// before they are read.  With sharded PARAFAC2 slices or sparse slabs each rank copies what it holds.
void Engine::free_snapshot() {
  if (snap_ != nullptr) cudaFree(snap_);
  if (snap_table_ != nullptr) cudaFree(snap_table_);
  snap_ = nullptr;
  snap_table_ = nullptr;
  snap_n_ = 0;
  snap_max_ = 0;
  ho_patience_ = 0;
}

void Engine::set_heldout_stopping(int patience) {
  AO_CUDA(cudaSetDevice(device_));
  AO_CUDA(cudaStreamSynchronize(st_));
  free_snapshot();
  if (patience <= 0) return;
  std::vector<CopyDesc> list;
  auto add = [&](DevMat& d) {
    if (d.p != nullptr && d.rows * d.cols > 0) list.push_back({d.p, nullptr, (long long)(d.rows * d.cols)});
  };
  for (auto& m : modes_)
    for (DevMat* d : {&m.fac, &m.Z, &m.muZ, &m.muD}) add(*d);
  for (auto& d : delta_) add(d);
  for (auto& ps : par2_)
    for (DevMat* d : {&ps.P, &ps.DeltaB, &ps.muDB}) add(*d);
  size_t total = 0;
  for (const auto& c : list) total += (size_t)round_up(c.n, 32);   // 256-byte aligned offsets
  try {
    AO_CUDA(cudaMalloc(&snap_, std::max<size_t>(total, 1) * sizeof(double)));
    AO_CUDA(cudaMalloc(&snap_table_, std::max<size_t>(list.size(), 1) * sizeof(CopyDesc)));
    size_t off = 0;
    for (auto& c : list) {
      c.snap = snap_ + off;
      off += (size_t)round_up(c.n, 32);
      snap_max_ = std::max(snap_max_, c.n);
    }
    AO_CUDA(cudaMemcpy(snap_table_, list.data(), list.size() * sizeof(CopyDesc), cudaMemcpyHostToDevice));
  } catch (...) {
    free_snapshot();
    throw;
  }
  snap_n_ = (int)list.size();
  snap_tree_.assign(n_objects_, 0);
  ho_patience_ = patience;
}

// after the synchronisation of a new best iteration, before the next outer iteration (graph launch) is enqueued
void Engine::snapshot_state() {
  launches_ += state_copy(snap_table_, snap_n_, snap_max_, 0, st_);
  for (int p = 0; p < n_objects_; ++p) {
    const ObjectState& o = objects_[p];
    snap_tree_[p] = o.Tbuf != nullptr && o.T_version == mode(o.modes[0]).version;
  }
}

// back to the state after iteration k*: the copy, new version stamps, then the same deterministic kernels that ran at
// k* rebuild what depends on the factors, so the state is bit-identical to the one iteration k* left
void Engine::restore_state() {
  launches_ += state_copy(snap_table_, snap_n_, snap_max_, 1, st_);
  for (auto& m : modes_) ++m.version;
  for (auto& ps : par2_) ps.T_version = 0;
  // a dimension-tree contraction that was current at k* may be used by the next run without recomputation: emit it
  // again from the restored mode-1 factor (by the mode-2 MTTKRP, into scratch the next sweep overwrites)
  for (int p = 0; p < n_objects_; ++p) {
    ObjectState& o = objects_[p];
    if (!snap_tree_[p]) continue;
    ModeState& m2 = mode(o.modes[1]);
    compute_mttkrp(o, 1, o.weight, m2.A.p, m2.rows);
  }
  em_step(true);   // the imputation from the restored factors (its sums are recomputed by the next run)
}

void Engine::heldout_best(int* iteration, double* sse) const {
  if (ho_best_iter_ < 0) throw CudaError(1, "heldout_best: the last run had early stopping off (or there was no run)");
  *iteration = ho_best_iter_;
  *sse = ho_best_sse_;
}

}  // namespace aoadmm
