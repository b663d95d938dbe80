// engine.h - host-side driver of the AO-ADMM sweep: owns all device state, mirrors the control flow of
// functions/cmtf_fun_AOADMM.m:87-476 and launches the sm_100a kernels.
#pragma once
#include <chrono>
#include <memory>
#include <string>
#include <vector>

#include "../../include/aoadmm.h"
#include "em.cuh"
#include "heldout.cuh"
#include "linalg.cuh"
#include "mttkrp.cuh"
#include "nvecs.cuh"
#include "par2.cuh"
#include "smallops.cuh"
#include "sparse.cuh"

namespace aoadmm {

struct DevMat {
  double* p = nullptr;
  int64_t rows = 0, cols = 0;
  size_t bytes() const { return (size_t)rows * cols * sizeof(double); }
};

void dev_alloc(DevMat& m, int64_t rows, int64_t cols);  // zero-initialised device matrix
void dev_free(DevMat& m);

struct NcclApi;  // dlopen'ed NCCL entry points (multi-GPU only)
// process-wide communicator cache (engine.cu)
void* comm_for_unique_id(const uint8_t id[128], int rank, int world, cudaStream_t st);
std::vector<void*> comms_for_devices(const std::vector<int>& devices);
void comm_release_all();

struct ModeState {
  int id = 0;                 // 1-based global mode id
  int p = -1;                 // owning object
  int pos = 0;                // 0-based position inside the object
  int64_t rows = 0;
  int R = 0;
  int coupling = 0;           // lin_coupled_modes(m)
  bool constrained = false;
  aoadmm_constraint con{};
  double ridge = 0.0;
  DevMat fac, Z, muZ, muD;    // G.fac, G.constraint_fac, G.constraint_dual_fac, G.coupling_dual_fac
  DevMat A, Alast, C, B, L, Binv, Btmp, GtG, Znew, V;
  double* invdiag = nullptr;
  double* rho = nullptr;      // device scalar
  PackedFactor packed;        // transposed copy used as DMMA B operand
  InnerCtl* ctl = nullptr;    // device; for coupled modes all modes of the group share the group's block
  int ctl_index = -1;
  uint64_t version = 1;       // bumped whenever fac changes (validity stamp for cached partial contractions)
  QuadProx quad;              // 'quadratic regularization': eigen-basis of L
  int lin = -1;               // index into Engine::lin_modes_ when the mode is linearly coupled (type 1..5)
  // PARAFAC2 objects: role 1 = A (first mode), 2 = stacked B_k, 3 = C; par2 = index into Engine::par2_
  int par2_role = 0, par2 = -1;
  const double* rho_rows = nullptr;   // role 3: per-row rho_k
  const double* Binv_rows = nullptr;  // role 3: per-row inv(B_k)
};

// Linear coupling (coupling types 1..5, cmtf_fun_AOADMM.m:278-389, :698-1075): per-mode operands.
// The coupling constraint of mode m is  G_m(F_m) = D_m(Delta)  in the "coupling space" S_m where mu_Delta_m lives:
//   type 1: H F = Delta        type 2: F H = Delta       type 3: F = H Delta       type 4: F = Delta H
//   type 5: H F = Delta H2
struct LinMode {
  int ctype = 0;
  DevMat H, H2;                 // Z.coupling.coupl_trafo_matrices{m}, ...matrices2{m}
  DevMat HHt;                   // type 2: H*H' (R x R), added to the system matrix as rho/2*HHt (:314)
  DevMat tmpF, tmpF2;           // factor-shaped scratch
  DevMat S1, S2, S3;            // coupling-space scratch: G_m(F), D_m(Delta), D_m(Delta - Delta_old)
  DevMat Zold;                  // constrained modes: Z before the update
  // types 1 and 5: sylvester(B2,B,A_inner) in the eigen-bases of H'H (computed once) and of B (per outer iteration)
  DevMat U, VB, Bwork;
  double* lam = nullptr;        // eigenvalues of H'H (rows of F)
  double* muB = nullptr;        // eigenvalues of B (R)
  // type 1 with a PARAFAC2 third mode (:283-297, :710-722): one (K*R) x (K*R) system instead of a Sylvester equation
  bool par2c = false;
  DevMat HtH, B2, B2L, B2B, B2C;
  double* B2invdiag = nullptr;
  double* Bsys3 = nullptr;      // K x R x R: the per-row matrices B{m}{k}
  double* rho_stats = nullptr;  // [0] mean(rho), [1] sum(rho)
  const double* rho_A = nullptr;  // scalar rho used in A_inner  (m.rho, or mean(rho) for par2c)
  const double* rho_D = nullptr;  // scalar weight in the Delta update (m.rho, or sum(rho) for par2c)
  // types 2, 3, 4 with a PARAFAC2 third mode (:305-311, :327-333, :349-355): row-wise rho_k and systems B{m}{k}
  bool par2row = false;
  DevMat Hs;                    // type 3: diag(rho) * H
  DevMat AAA;                   // type 4: H * H'
};

struct LinGroup {
  int ctype = 0;
  std::vector<int> modes;       // global ids, ascending
  DevMat Dold, Ddiff, AA, AAL, AAB, AAC, BB, Dt;
  double* AAinvdiag = nullptr;
  int par2row = -1;             // position (in `modes`) of a third PARAFAC2 mode with row-wise rho, or -1
  double* wsum = nullptr;       // type 2 with par2row: per-row sum of the weights (:813)
  double* Minv = nullptr;       // type 4 with par2row: inv(AA + rho_k*AAA) per row (:957-960)
  double* scal = nullptr;       // device scalars: [0] sum rho, [1] 1/sum rho, [2] scratch rho of prep_system
  RedJob* jobs_dev = nullptr;
  int njobs = 0;
  double* red = nullptr;        // reduction results (njobs)
  double* red_partials = nullptr;
  LinFin fin{};                 // which reduction feeds which residual
};

// Device state of one PARAFAC2 object (layout in par2.cuh)
struct Par2State {
  int p = -1, K = 0, R = 0;
  int64_t I = 0, Jtot = 0, Jmax = 0, ldX = 0;
  int m1 = 0, m2 = 0, m3 = 0;            // global mode ids of A, B_k, C
  std::vector<int64_t> joff;             // K+1 host copy of the slice offsets
  Par2Layout lay;
  long long* joff_dev = nullptr;
  int* seg_dev = nullptr;
  double* X = nullptr;                   // I x Jtot (leading dimension ldX), addressed with GLOBAL column indices: with
                                         // sharded slices only columns jlo..jhi-1 exist (X = X_alloc - jlo*ldX)
  uint8_t* mask = nullptr;               // Z.miss{p}{k} side by side like X (nullptr: complete data), same addressing
  double* X_alloc = nullptr;             // the allocations behind X / mask (this rank's columns)
  uint8_t* mask_alloc = nullptr;
  // multi-GPU (SURVEY 8e): the K slices are sharded over the ranks in contiguous ranges k0..k1-1 (= stacked rows /
  // columns jlo..jhi-1); per-slice work runs on the owner only, sums over k are all-reduced, the rows of the third mode
  // are gathered.  sharded == false: every rank holds and updates all slices (one GPU, or objects the sharding does not
  // cover: linear couplings on a PARAFAC2 mode, tPARAFAC2 / quadratic regularisation, fewer slices than ranks).
  bool sharded = false;
  int k0 = 0, k1 = 0;
  int64_t jlo = 0, jhi = 0;
  double* redbuf = nullptr;              // R*R + 8 doubles: local sums on their way through an all-reduce
  bool state_stale = false;              // sharded: the non-local rows of the stacked state are not up to date
  Tensor3 view;                          // X as an I x Jtot x 1 tensor for the DMMA product kernels
  PackedFactor fW, fA, ones;
  DevMat W, T;                           // Jtot x R: scaled operand of the mode-A product; T = Xall' * A
  uint64_t T_version = 0;                // version of A that T was computed from
  DevMat P, muDB, DeltaB, PDold, gM, gS;
  double *G2 = nullptr, *Binv2 = nullptr, *Binv3 = nullptr, *rho2 = nullptr, *rho3 = nullptr, *contrib = nullptr,
         *norms = nullptr, *Csum = nullptr, *segn = nullptr, *res = nullptr, *res_partials = nullptr, *tdiag = nullptr, *Vprev = nullptr,
         *sysws = nullptr;   // R > 64: factorisation workspace of the per-slice systems (2 R^2 per slice)
  double* segn_host = nullptr;           // pinned: K x 4 per-slice objective terms + 1 residual
  bool explicit_residual = false;        // objective needs ||X_k - A D_k B_k'||^2 (mode A is not updated last)
  // sparse slices (aoadmm_create_sparse_slices): Xall as an order-2 COO object over I x Jtot.  X, mask, view, fW, fA and
  // ones stay empty; the two products are mode positions 0 / 1 of the sparse MTTKRP with the factors {A, W}.
  SparseTensor* sp = nullptr;
  double* mgram = nullptr;               // sparse slices: 2 R^2 scratch of the residual (A'A, sum_k diag(c_k) B_k'B_k diag(c_k))
};

struct View3 {                // how mode position n of an object is computed
  Tensor3 t;
  int kernel_pos = 0;         // 0 lead, 1 inner/epilogue0, 2 inner/epilogue1
  std::vector<int> f0_modes, f1_modes;  // global mode ids whose Khatri-Rao product forms operand 0 / 1 (empty = ones)
  int64_t f0_rows = 0, f1_rows = 0;
  PackedFactor f0, f1;        // packed operands (allocated when a KR product or ones are needed)
  bool f0_own = false, f1_own = false;
  int64_t out_rows = 0;       // rows produced by this rank (== rows of the factor unless sharded last mode)
  int64_t out_offset = 0;
  bool needs_allreduce = false;
};

struct ObjectState {
  int model = 0, order = 0;
  std::vector<int> modes;     // global mode ids (1-based)
  std::vector<int64_t> dims;  // local dims (last one = shard extent)
  double weight = 1.0, znorm = 0.0;
  bool znorm_pending_allreduce = false;
  double* data = nullptr;     // device, leading dimension ld0
  int64_t ld0 = 0;
  double* dataT = nullptr;    // matrices without a mask: transposed copy (dims[1] x dims[0], leading dimension ldT) so that
  int64_t ldT = 0;            // the mode-2 product is a LEAD launch too (the K = 1 INNER launch cannot split inside its one slab)
  int64_t shard_offset = 0, shard_extent = 0, last_full = 0;
  bool sharded = false;
  std::vector<View3> views;   // one per mode position
  int last_m = 0;             // global id of the mode updated last in a sweep (static)
  uint8_t* mask = nullptr;    // Z.miss{p}: 1 = observed, 0 = missing, same indexing as data (nullptr: complete data)
  double* em_kr = nullptr;    // masked objects of order > 3: Khatri-Rao product of the factors of modes 3..N
  double* em_fkT = nullptr;   // masked objects of order >= 3: transposed third factor for the pipelined EM kernel
  double* Tbuf = nullptr;     // dimension tree: T(j,k,r) = sum_i X(i,j,k) F1(i,r), emitted by the mode-2 MTTKRP
  uint64_t T_version = 0;     // version of the mode-1 factor T was computed from (0 = invalid)
  SparseTensor* sp = nullptr; // sparse (COO) object: sorted device copies of this rank's slab (sparse.cuh); data, views stay empty
  HeldOut* ho = nullptr;      // held-out set (aoadmm_set_heldout), replicated on every rank
  std::vector<double> ho_hist;  // held-out SSE after outer iteration 0, 1, ... of the last run
};

class Engine {
 public:
  // shared_comm: communicator of this rank created by the caller (single-process device group), else nullptr and the
  // communicator of dist->nccl_unique_id is taken from the process-wide cache.  sparse: nullptr, or n_objects entries
  // (nullptr for a dense object) with the COO data of sparse CP objects (aoadmm_create_sparse, validated by the caller);
  // masks: nullptr, or n_objects entries with the sparse Z.miss masks of sparse objects (aoadmm_create_sparse_masked);
  // slices: nullptr, or n_objects entries with the stacked I x Jtot COO slices of PARAFAC2 objects
  // (aoadmm_create_sparse_slices, validated by the caller)
  Engine(const aoadmm_problem* prob, const aoadmm_dist* dist, void* shared_comm = nullptr,
         const aoadmm_sparse_object* const* sparse = nullptr, const aoadmm_sparse_object* const* masks = nullptr,
         const aoadmm_sparse_object* const* slices = nullptr);
  ~Engine();
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;
  void set_state(int field, int index, int slice, const double* data, int64_t rows, int64_t cols);
  void get_state(int field, int index, int slice, double* data, int64_t rows, int64_t cols);
  // collective over the ranks: makes the replicated copy of the state complete on every rank (gathers the rows of sharded
  // PARAFAC2 slices from their owners).  Call on EVERY rank before get_state; a no-op when nothing is stale.
  void prepare_state_read();
  void run(const aoadmm_options* opt, aoadmm_out* out);
  void generate_cp_data(int object, const double* const* factors, double noise, uint64_t seed);
  float time_mttkrp(int object, int pos, int reps);
  void object_to_host(int object, double* out, int64_t n_elements);
  void object_slab(int object, int64_t* offset_elems, int64_t* n_elems) const;
  int device() const { return device_; }
  int64_t mode_rows(int mode_id) const { return (mode_id >= 1 && mode_id <= nb_modes_) ? modes_[mode_id - 1].rows : -1; }
  int mode_rank(int mode_id) const { return (mode_id >= 1 && mode_id <= nb_modes_) ? modes_[mode_id - 1].R : -1; }
  int object_mode(int object, int pos) const {   // global mode id at 1-based position `pos` of 1-based object, or -1
    if (object < 1 || object > n_objects_) return -1;
    const ObjectState& o = objects_[object - 1];
    return (pos >= 1 && pos <= o.order) ? o.modes[pos - 1] : -1;
  }
  // cmtf_nvecs.m / init_coupled_AOADMM_CMTF.m:50-69: r leading eigenvectors of X_(n) X_(n)' for global mode id `mode`
  // (slice: 1-based slice of a PARAFAC2 B_k mode, else 0); out: rows x r host buffer; info: [iterations, residual]
  void nvecs_to_host(int mode_id, int slice, int r, double* out, int64_t rows, double* info);
  void nvecs_sharded_mode(ObjectState& o, int r, double* out, int64_t rows, double* info);
  // aoadmm_nvecs_sparse: the same for a mode whose first object is a sparse CP object, with Y V applied as U (U' V) on the
  // fiber-compressed unfolding U (sparse.cuh, FiberUnfolding); collective over the ranks
  void nvecs_sparse_to_host(int mode_id, int r, double* out, int64_t rows, double* info);
  void mttkrp_to_host(int object, int pos, double* out, int precision = -1);  // unweighted MTTKRP of the resident factors (-1: precision of the last run)
  // held-out entries (aoadmm_model_at / aoadmm_set_heldout): host-only checks of object and subscripts, then the work
  void check_entries(int object, const aoadmm_sparse_object* entries, bool heldout) const;
  void model_at(int object, const aoadmm_sparse_object* entries, double* out);   // on this engine's device
  void set_heldout(int object, const aoadmm_sparse_object* entries);             // collective over the ranks
  // collective over the ranks, once after every rank's constructor returned: sums the partial Znorm_const = NaN norms
  // of sharded objects (a no-op on one GPU)
  void reduce_norms();
  void heldout_history(int object, double* sse, int64_t n, int64_t* count) const;
  // early stopping on the held-out error (aoadmm_set_heldout_stopping): patience 0 frees the snapshot, >= 1 allocates it
  void set_heldout_stopping(int patience);
  int heldout_sets() const { return n_heldout_; }
  void heldout_best(int* iteration, double* sse) const;   // k* and its SSE sum of the last run (CudaError if none)
  int64_t launches() const { return launches_; }
  void phase_ms(double ms[3]);
  double last_run_ms() const { return last_run_ms_; }
  double last_loop_ms() const { return last_loop_ms_; }
  std::string last_error;

 private:
  // setup
  void construct(const aoadmm_problem* prob, const aoadmm_dist* dist, void* shared_comm,
                 const aoadmm_sparse_object* const* sparse, const aoadmm_sparse_object* const* masks,
                 const aoadmm_sparse_object* const* slices);
  // imputed: the MTTKRP of the EM-imputed tensor of a masked sparse object (the sweep); else of the stored values
  int sparse_mttkrp_of(ObjectState& o, int pos, double scale, double* out, int64_t ldout, bool imputed = false);
  static bool sparse_masked(const ObjectState& o) { return o.sp != nullptr && o.sp->masked; }
  void release();
  void build_views(ObjectState& o);
  void refresh_transposed(ObjectState& o);
  void build_objective_jobs();
  // sweep pieces
  void refresh_gram(ModeState& m);
  void compute_mttkrp(ObjectState& o, int pos, double scale, double* out, int64_t ldout, bool imputed = false);
  int tc_mttkrp(ObjectState& o, int pos, double scale, double* out, int64_t ldout, double* emit, int prec);
  void pack_operand(View3& v, int which);
  void precompute_mode(ModeState& m, int n_rho_terms, bool do_chol);
  void fill_prep(ModeState& m, PrepArgs& a, int n_rho_terms, bool do_chol);
  // Z.prox_operators{m}(X, rho) for the constraint of mode m on a rows x cols block (cmtf_fun_AOADMM.m:1424-1426)
  int apply_prox(ModeState& m, const double* X, long long ldx, double* out, long long ldo, long long rows, int cols,
                 const double* rho_dev, const int* skip);
  void apply_bsum(ModeState& m);
  void run_admm(std::vector<ModeState*>& group, double* Delta, const aoadmm_options& opt);
  void eval_objective(bool first, double f[4]);
  void enqueue_objective(bool first);
  void finish_objective(bool first, double f[4]);
  void sweep(int iter, std::vector<int>& inner_fixed);
  void check_errors(aoadmm_out* out);
  void allreduce(double* buf, size_t count);
  // EM imputation of missing entries + masked objective sums (cmtf_fun_AOADMM.m:408-441, :1224-1226, :1249-1252)
  void em_step(bool impute);
  // linear couplings (cmtf_fun_AOADMM.m:278-389, :698-1075)
  void setup_linear_coupling(const aoadmm_problem* prob, int coupl_id);
  void lin_G(const LinMode& lm, const ModeState& m, const double* F, double* out, const int* skip);
  void lin_D(const LinMode& lm, const ModeState& m, const double* Delta, const DevMat& Dshape, double* out, const int* skip);
  void lin_Gt(const LinMode& lm, const ModeState& m, const double* Y, double* out, const int* skip);
  void lin_build_jobs(int coupl_id);
  void free_linear_coupling();
  void lin_prepare_group(int coupl_id);
  void run_admm_linear(int coupl_id, std::vector<ModeState*>& group, const aoadmm_options& opt);
  // PARAFAC2 block (cmtf_fun_AOADMM.m:157-250, :509-589)
  void setup_par2(const aoadmm_problem* prob, int p, const aoadmm_sparse_object* slices);
  void par2_sparse_residual(Par2State& s);
  void par2_update_T(Par2State& s);
  void par2_precompute_A(ModeState& m, int n_rho_terms, bool do_chol = true);
  void par2_update_B(ModeState& m, int outer_iter);
  void par2_precompute_C(ModeState& m, int n_rho_terms, bool ls_direct, double* Bsys_out = nullptr,
                         const double* HHt = nullptr);
  void par2_refresh_gram(Par2State& s);
  void par2_gather_state(Par2State& s);   // sharded slices: bring every rank's stacked rows up to date (get_state)
  DevMat* par2_field(int field, int index, int slice, int64_t* row_off, int64_t* nrows);

  ModeState& mode(int id) { return modes_[id - 1]; }

  int nb_modes_ = 0, n_objects_ = 0, n_couplings_ = 0;
  std::vector<ModeState> modes_;
  std::vector<ObjectState> objects_;
  std::vector<int> coupling_type_;
  std::vector<DevMat> delta_;  // coupling_fac per coupling id
  std::vector<Par2State> par2_;
  std::vector<LinMode> lin_modes_;
  std::vector<LinGroup> lin_groups_;   // indexed by coupling id - 1 (ctype 0 groups stay empty)
  bool has_ridge_ = false;

  // distributed
  int rank_ = 0, world_ = 1, device_ = 0;
  NcclApi* nccl_ = nullptr;
  void* comm_ = nullptr;

  // scratch
  cudaStream_t st_ = nullptr;
  cudaStream_t st2_ = nullptr;   // side stream: system preparation overlaps the MTTKRP of the same mode
  cudaEvent_t ev_fork_ = nullptr, ev_join_ = nullptr;
  MttkrpWorkspace mws_;
  TcOperand tc_op_;              // low-precision operand scratch of the opt-in tcgen05 MTTKRP (allocated on first use)
  double* gram_ws_ = nullptr;
  double* admm_partials_ = nullptr;
  double* admm_sums_ = nullptr;
  unsigned* admm_counter_ = nullptr;
  void* prox_scratch_ = nullptr;
  double* krtmp_[2] = {nullptr, nullptr};
  size_t krtmp_doubles_ = 0;
  InnerCtl* ctl_dev_ = nullptr;
  InnerCtl* ctl_host_ = nullptr;  // pinned
  int n_ctl_ = 0;
  // objective
  std::vector<RedJob> jobs_host_;
  RedJob* jobs_dev_ = nullptr;
  double* red_dev_ = nullptr;
  double* red_partials_ = nullptr;
  double* red_host_ = nullptr;  // pinned
  struct ObjTerms;
  std::unique_ptr<ObjTerms> terms_;
  double* cp0_tmp_ = nullptr;     // iteration-0 MTTKRP / Hadamard scratch
  std::vector<double> f_obj_;     // per-object objective terms between enqueue_objective and finish_objective
  bool capturing_ = false;        // inside cudaStreamBeginCapture / EndCapture
  bool has_missing_ = false;      // any object with a Z.miss mask
  double* em_sums_ = nullptr;     // device, 5 per object (see em.cuh)
  double* em_sums_host_ = nullptr;  // pinned
  double* em_partials_ = nullptr;
  double f_rel_missing_ = 0.0;
  int n_heldout_ = 0;             // objects with a held-out set
  double* ho_sse_ = nullptr;      // device, one per object: held-out SSE of the current iteration
  double* ho_sse_host_ = nullptr; // pinned
  void heldout_pass();            // enqueued with the objective; the result rides on its device-to-host copies
  void record_heldout();
  // early stopping: the snapshot list (one allocation `snap_`, descriptor table on the device) holds every buffer a
  // later run reads before rewriting it; see set_heldout_stopping
  int ho_patience_ = 0;
  double* snap_ = nullptr;
  CopyDesc* snap_table_ = nullptr;
  int snap_n_ = 0;
  long long snap_max_ = 0;        // doubles of the largest buffer of the list
  std::vector<char> snap_tree_;   // per object: the dimension-tree contraction was current at the snapshot
  int ho_best_iter_ = -1;         // k* of the last run with stopping on, -1 after a run with stopping off
  double ho_best_sse_ = 0.0;
  void free_snapshot();
  void snapshot_state();
  void restore_state();
  int64_t launches_ = 0;
  // timing
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool_;
  std::vector<int> ev_phase_;
  size_t ev_used_ = 0;
  double phase_ms_[3] = {0, 0, 0};
  void phase_begin(int phase);
  void phase_end();
  void phase_collect();
  aoadmm_options opt_{};
  cudaEvent_t run_ev_[3] = {nullptr, nullptr, nullptr};
  double last_run_ms_ = 0.0, last_loop_ms_ = 0.0;
};

}  // namespace aoadmm
