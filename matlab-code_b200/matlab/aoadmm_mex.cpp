// aoadmm_mex.cpp - MATLAB MEX gateway in front of the C ABI of include/aoadmm.h.
//
//   [G, out] = aoadmm_mex(Z, Znorm_const, G, options)
//
// replaces the body of functions/cmtf_fun_AOADMM.m (called at functions/cmtf_AOADMM.m:193).  Z, Znorm_const, G and
// options are exactly the variables cmtf_AOADMM.m holds at that line: Z built by the user script
// (example_script6_matrix_matrix_CP_nonneg.m:84-92) plus Z.prox_operators / Z.reg_func (ignored here: the device
// cannot call MATLAB function handles, the named specs in Z.constraints are used instead), Znorm_const from
// cmtf_AOADMM.m:124-156, G from init_coupled_AOADMM_CMTF.m or the caller, options from the script (:120-132).
//
// Engine knobs read from options (all optional): b200_gpus (number of B200s this MATLAB session drives through
// aoadmm_create_multi, default 1), b200_shard_sparse (with b200_gpus > 1: sparse objects too, through
// aoadmm_create_sparse_multi), b200_dimtree, b200_mttkrp_precision, b200_fuse_inner, b200_graph.
//
// Sparse CP objects arrive as struct('subs',S,'vals',V,'size',sz) (cmtf_fun_AOADMM.m unwrap_data: sptensor or a MATLAB
// sparse matrix through find); the 1-based double subscripts become 0-based int64 and the handle is created with
// aoadmm_create_sparse (one GPU, CP only: anything else raises aoadmm:unsupported).  Z.miss{p} of a sparse object must
// be sparse too (the same struct); its nonzeros mark the observed entries (aoadmm_create_sparse_masked).
//
// Error handling: mexErrMsgIdAndTxt leaves mexFunction with a longjmp that runs no C++ destructor, so nothing in
// here calls it directly - failures travel as a C++ exception (MexError) to the bottom of mexFunction, where every
// local (mask byte vectors, the engine handle, property copies) has already been destroyed.
//
// Build (on a machine with MATLAB; not possible in the offline build container, see INTEGRATION.md):
//   mex -R2018a -I<repo>/include aoadmm_mex.cpp -L<repo>/matlab-code_b200/aoadmm_b200 -laoadmm_b200
// tests/test_capi_host.py compiles this file against a stub mex.h so that it at least stays syntactically valid.
#include <cstring>
#include <string>
#include <vector>

#include "mex.h"

#include "aoadmm.h"

namespace {

struct MexError {
  std::string id, msg;
};
[[noreturn]] void fail(const char* id, const std::string& msg) { throw MexError{id, msg}; }

// mxGetProperty returns a deep COPY that the caller owns (a second host copy of a whole tensor): the copies made during
// one call are collected here and destroyed when the call ends.  cmtf_fun_AOADMM.m passes Z.object{p}.data (shared
// data, no copy), so this path only serves callers that hand a Tensor Toolbox object to aoadmm_mex directly.
struct PropertyCopies {
  std::vector<mxArray*> owned;
  ~PropertyCopies() {
    for (mxArray* a : owned) mxDestroyArray(a);
  }
};

// engine handle owned for the duration of the call
struct HandleGuard {
  aoadmm_handle* h = nullptr;
  ~HandleGuard() {
    if (h != nullptr) aoadmm_destroy(h);
  }
};

const mxArray* field(const mxArray* s, const char* name, bool required = true) {
  const mxArray* f = mxIsStruct(s) ? mxGetField(s, 0, name) : nullptr;
  if (f == nullptr && required) fail("aoadmm:invalidArg", std::string("missing field '") + name + "'");
  return f;
}

double scalar_of(const mxArray* a, const char* what) {
  if (a == nullptr || !mxIsNumeric(a) || mxGetNumberOfElements(a) < 1) fail("aoadmm:invalidArg", std::string(what) + " must be numeric");
  return mxGetScalar(a);
}

double opt_scalar(const mxArray* s, const char* name, double dflt) {
  const mxArray* f = field(s, name, false);
  return (f != nullptr && !mxIsEmpty(f)) ? mxGetScalar(f) : dflt;
}

std::string string_of(const mxArray* a) {
  if (a == nullptr || !mxIsChar(a)) return std::string();
  char* c = mxArrayToString(a);
  std::string s(c ? c : "");
  mxFree(c);
  return s;
}

// numeric data of a Tensor Toolbox `tensor` object (property .data) or of a plain double array
const mxArray* dense_data(const mxArray* obj, PropertyCopies& pc) {
  if (std::strcmp(mxGetClassName(obj), "tensor") == 0) {
    mxArray* d = mxGetProperty(obj, 0, "data");
    if (d == nullptr) fail("aoadmm:invalidArg", "tensor object without .data");
    pc.owned.push_back(d);
    return d;
  }
  if (!mxIsDouble(obj) || mxIsComplex(obj) || mxIsSparse(obj))
    fail("aoadmm:unsupported", "data objects must be dense real double arrays or Tensor Toolbox tensors");
  return obj;
}

// Z.miss{p} (cmtf_AOADMM.m:68-121): logical / numeric array, Tensor Toolbox tensor, or sptensor (converted with
// full()) -> one byte per element, 1 = observed
std::vector<uint8_t> mask_bytes(const mxArray* m, size_t expected, int p, PropertyCopies& pc) {
  if (std::strcmp(mxGetClassName(m), "sptensor") == 0) {
    mxArray* in = const_cast<mxArray*>(m);
    mxArray* conv = nullptr;
    if (mexCallMATLAB(1, &conv, 1, &in, "full") != 0 || conv == nullptr)
      fail("cmtf:missingData:maskTypeError", "Z.miss{" + std::to_string(p + 1) + "} cannot be converted with full()");
    pc.owned.push_back(conv);
    m = conv;
  }
  if (std::strcmp(mxGetClassName(m), "tensor") == 0) {
    mxArray* d = mxGetProperty(m, 0, "data");
    if (d != nullptr) pc.owned.push_back(d);
    m = d;
  }
  if (m == nullptr || mxGetNumberOfElements(m) != expected)
    fail("cmtf:missingData:maskSizeMismatch", "Z.miss{" + std::to_string(p + 1) + "} size does not match Z.object{" + std::to_string(p + 1) + "}.");
  std::vector<uint8_t> out(expected);
  if (mxIsLogical(m)) {
    const mxLogical* v = mxGetLogicals(m);
    for (size_t i = 0; i < expected; ++i) out[i] = v[i] ? 1 : 0;
  } else if (mxIsDouble(m)) {
    const double* v = mxGetPr(m);
    for (size_t i = 0; i < expected; ++i) out[i] = (v[i] != 0.0) ? 1 : 0;
  } else {
    fail("cmtf:missingData:maskTypeError", "Z.miss{" + std::to_string(p + 1) + "} must be logical, double, tensor or sptensor");
  }
  return out;
}

// a sparse object as cmtf_fun_AOADMM.m's unwrap_data hands it over: struct('subs',S,'vals',V,'size',sz) with S the
// nnz x N matrix of 1-based subscripts (Tensor Toolbox sptensor .subs, or [i j] from find() for a MATLAB sparse matrix)
bool is_coo_struct(const mxArray* a) {
  return a != nullptr && mxIsStruct(a) && mxGetField(a, 0, "subs") != nullptr && mxGetField(a, 0, "vals") != nullptr;
}

// subs (1-based doubles, nnz x order) -> 0-based int64, column-major, with an integer and range check per entry
void coo_subs(const mxArray* a, int p, int order, const std::vector<int64_t>& rows, std::vector<int64_t>& subs, int64_t* nnz) {
  const mxArray* S = mxGetField(a, 0, "subs");
  const mxArray* V = mxGetField(a, 0, "vals");
  const std::string who = "Z.object{" + std::to_string(p + 1) + "} (sparse): ";
  if (!mxIsDouble(S) || !mxIsDouble(V)) fail("aoadmm:invalidArg", who + "subs and vals must be double");
  const size_t n = mxGetNumberOfElements(V);
  if (n > 0 && (mxGetM(S) != n || (int)mxGetN(S) != order))
    fail("aoadmm:invalidArg", who + "subs must be nnz x " + std::to_string(order) + " with one row per value");
  const double* s = n > 0 ? mxGetPr(S) : nullptr;
  subs.resize(n * (size_t)order);
  for (int d = 0; d < order; ++d)
    for (size_t e = 0; e < n; ++e) {
      const double v = s[(size_t)d * n + e];
      if (!(v >= 1.0 && v <= (double)rows[d]) || v != (double)(int64_t)v)
        fail("aoadmm:invalidArg", who + "subscript " + std::to_string(v) + " in column " + std::to_string(d + 1) +
                                      " is not an integer in 1.." + std::to_string(rows[d]));
      subs[(size_t)d * n + e] = (int64_t)v - 1;
    }
  *nnz = (int64_t)n;
}

int constraint_kind(const std::string& n) {  // constraints_to_prox.m:13-91
  static const struct { const char* name; int kind; } table[] = {
      {"non-negativity", AOADMM_CON_NONNEG}, {"box", AOADMM_CON_BOX}, {"simplex column-wise", AOADMM_CON_SIMPLEX_COL},
      {"simplex row-wise", AOADMM_CON_SIMPLEX_ROW}, {"non-decreasing", AOADMM_CON_NONDECREASING},
      {"non-increasing", AOADMM_CON_NONINCREASING}, {"unimodality", AOADMM_CON_UNIMODAL}, {"l1-ball", AOADMM_CON_L1_BALL},
      {"l2-ball", AOADMM_CON_L2_BALL}, {"non-negative l2-ball", AOADMM_CON_NONNEG_L2_BALL},
      {"non-negative l2-sphere", AOADMM_CON_NONNEG_L2_SPHERE}, {"orthonormal", AOADMM_CON_ORTHONORMAL},
      {"l1 regularization", AOADMM_CON_L1_REG}, {"l0 regularization", AOADMM_CON_L0_REG},
      {"l2 regularization", AOADMM_CON_L2_REG}, {"ridge", AOADMM_CON_RIDGE},
      {"quadratic regularization", AOADMM_CON_QUADRATIC}, {"GL smoothness", AOADMM_CON_GL_SMOOTH},
      {"TV regularization", AOADMM_CON_TV}, {"tPARAFAC2", AOADMM_CON_TPARAFAC2}, {"custom", AOADMM_CON_CUSTOM}};
  for (const auto& t : table)
    if (n == t.name) return t.kind;
  fail("aoadmm:invalidArg", "unknown constraint '" + n + "'");
}

void check(int status, aoadmm_handle* h) {
  if (status == AOADMM_OK) return;
  const std::string msg = aoadmm_last_error(h);   // copied before the HandleGuard of the caller destroys its owner
  switch (status) {
    case AOADMM_ERR_UNSUPPORTED: fail("aoadmm:unsupported", msg);
    case AOADMM_ERR_NOT_POSITIVE_DEFINITE: fail("aoadmm:notPositiveDefinite", msg);  // chol() would have thrown
    case AOADMM_ERR_NON_FINITE: fail("aoadmm:nonFinite", msg);
    case AOADMM_ERR_NO_DEVICE: fail("aoadmm:noDevice", msg);
    case AOADMM_ERR_OOM: fail("aoadmm:outOfMemory", msg);
    case AOADMM_ERR_CUDA: fail("aoadmm:cuda", msg);
    case AOADMM_ERR_NCCL: fail("aoadmm:nccl", msg);
    default: fail("aoadmm:invalidArg", msg);
  }
}

struct StateField {
  const char* name;
  int field;
};
const StateField kModeFields[] = {{"fac", AOADMM_FIELD_FAC},
                                  {"constraint_fac", AOADMM_FIELD_CONSTRAINT_FAC},
                                  {"constraint_dual_fac", AOADMM_FIELD_CONSTRAINT_DUAL},
                                  {"coupling_dual_fac", AOADMM_FIELD_COUPLING_DUAL}};

}  // namespace

namespace {
void solve(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  PropertyCopies pc;
  if (nrhs != 4) fail("aoadmm:invalidArg", "usage: [G,out] = aoadmm_mex(Z, Znorm_const, G, options)");
  if (nlhs > 2) fail("aoadmm:invalidArg", "too many outputs");
  const mxArray *Z = prhs[0], *Zn = prhs[1], *G = prhs[2], *opt = prhs[3];
  if (!mxIsStruct(Z) || !mxIsCell(Zn) || !mxIsStruct(G) || !mxIsStruct(opt)) fail("aoadmm:invalidArg", "Z, G, options must be structs, Znorm_const a cell");

  // ---- Z -------------------------------------------------------------------------------------
  const mxArray* objects = field(Z, "object");
  const mxArray* modes_c = field(Z, "modes");
  const mxArray* size_c = field(Z, "size");
  const mxArray* model_c = field(Z, "model");
  const mxArray* loss_c = field(Z, "loss_function");
  const mxArray* coupling = field(Z, "coupling");
  const int P = (int)mxGetNumberOfElements(objects);
  const int nb_modes = (int)mxGetNumberOfElements(size_c);
  const mxArray* miss = field(Z, "miss", false);
  std::vector<std::vector<uint8_t>> miss_cp(P);
  std::vector<std::vector<int64_t>> sp_subs(P);
  std::vector<aoadmm_sparse_object> sp_obj(P);
  std::vector<const aoadmm_sparse_object*> sp_ptr(P, nullptr);
  bool any_sparse = false, any_mask = false;
  std::vector<std::vector<int64_t>> mk_subs(P);
  std::vector<aoadmm_sparse_object> mk_obj(P);
  std::vector<const aoadmm_sparse_object*> mk_ptr(P, nullptr);
  std::vector<std::vector<std::vector<uint8_t>>> miss_par2(P);
  std::vector<std::vector<const uint8_t*>> miss_par2_ptr(P);
  for (int p = 0; p < P; ++p)
    if (string_of(mxGetCell(loss_c, p)) != "Frobenius")
      fail("aoadmm:unsupported", "only the Frobenius loss runs on the B200 engine");

  std::vector<int64_t> mode_rows(nb_modes, 0);
  std::vector<std::vector<int64_t>> slice_rows(nb_modes);
  std::vector<const int64_t*> slice_ptr(nb_modes, nullptr);
  std::vector<int32_t> n_slices(nb_modes, 0), mode_rank(nb_modes, 0);
  for (int m = 0; m < nb_modes; ++m) {
    const mxArray* s = mxIsCell(size_c) ? mxGetCell(size_c, m) : nullptr;
    const size_t n = s ? mxGetNumberOfElements(s) : 1;
    if (s != nullptr && n > 1) {  // second PARAFAC2 mode: vector of J_k
      const double* v = mxGetPr(s);
      slice_rows[m].assign(n, 0);
      for (size_t k = 0; k < n; ++k) slice_rows[m][k] = (int64_t)v[k];
      n_slices[m] = (int32_t)n;
    } else {
      mode_rows[m] = (int64_t)(s ? mxGetScalar(s) : mxGetPr(size_c)[m]);
    }
  }
  for (int m = 0; m < nb_modes; ++m) slice_ptr[m] = slice_rows[m].empty() ? nullptr : slice_rows[m].data();

  const mxArray* Gfac = field(G, "fac");
  std::vector<std::vector<int32_t>> obj_modes(P);
  std::vector<std::vector<const double*>> obj_slices(P);
  std::vector<aoadmm_object> objs(P);
  const double* weights = mxGetPr(field(Z, "weights"));
  for (int p = 0; p < P; ++p) {
    const mxArray* mv = mxGetCell(modes_c, p);
    const double* md = mxGetPr(mv);
    const int order = (int)mxGetNumberOfElements(mv);
    obj_modes[p].resize(order);
    for (int d = 0; d < order; ++d) obj_modes[p][d] = (int32_t)md[d];
    // rank = columns of G.fac{modes{p}(1)} (cmtf_AOADMM.m:57)
    const mxArray* f1 = mxGetCell(Gfac, obj_modes[p][0] - 1);
    const int R = (int)mxGetN(f1);
    for (int d = 0; d < order; ++d) mode_rank[obj_modes[p][d] - 1] = R;
    aoadmm_object& o = objs[p];
    std::memset(&o, 0, sizeof(o));
    const bool par2 = string_of(mxGetCell(model_c, p)) == "PAR2";
    o.model = par2 ? AOADMM_MODEL_PAR2 : AOADMM_MODEL_CP;
    o.order = order;
    o.modes = obj_modes[p].data();
    o.weight = weights[p];
    o.znorm_const = scalar_of(mxGetCell(Zn, p), "Znorm_const{p}");
    const mxArray* obj = mxGetCell(objects, p);
    if (par2) {
      const int K = (int)mxGetNumberOfElements(obj);
      obj_slices[p].resize(K);
      for (int k = 0; k < K; ++k) {
        if (is_coo_struct(mxGetCell(obj, k))) fail("aoadmm:unsupported", "PARAFAC2 objects with sparse slices are not supported");
        obj_slices[p][k] = mxGetPr(dense_data(mxGetCell(obj, k), pc));
      }
      o.slices = obj_slices[p].data();
      o.n_slices = K;
    } else if (is_coo_struct(obj)) {   // sparse object -> aoadmm_create_sparse
      std::vector<int64_t> rows(order);
      for (int d = 0; d < order; ++d) rows[d] = mode_rows[obj_modes[p][d] - 1];
      coo_subs(obj, p, order, rows, sp_subs[p], &sp_obj[p].nnz);
      sp_obj[p].subs = sp_subs[p].data();
      sp_obj[p].vals = sp_obj[p].nnz > 0 ? mxGetPr(mxGetField(obj, 0, "vals")) : nullptr;
      sp_ptr[p] = &sp_obj[p];
      any_sparse = true;
      o.data = nullptr;
      o.shard_offset = 0;
      o.shard_extent = rows[order - 1];
    } else {
      const mxArray* dd = dense_data(obj, pc);
      size_t expect = 1;
      for (int d = 0; d < order; ++d) expect *= (size_t)mode_rows[obj_modes[p][d] - 1];
      if (mxGetNumberOfElements(dd) != expect) fail("aoadmm:invalidArg", "Z.object{" + std::to_string(p + 1) + "} does not have the size Z.size prescribes");
      o.data = mxGetPr(dd);
      o.shard_offset = 0;
      o.shard_extent = mode_rows[obj_modes[p][order - 1] - 1];
    }
    const mxArray* mp = (miss != nullptr && mxIsCell(miss) && p < (int)mxGetNumberOfElements(miss)) ? mxGetCell(miss, p) : nullptr;
    if (mp != nullptr && is_coo_struct(mp)) {   // sparse mask (unwrap_data of an sptensor / sparse Z.miss{p})
      if (sp_ptr[p] == nullptr)
        fail("aoadmm:invalidArg", "Z.miss{" + std::to_string(p + 1) + "} is sparse but Z.object{" + std::to_string(p + 1) + "} is dense");
      std::vector<int64_t> rows(order);
      for (int d = 0; d < order; ++d) rows[d] = mode_rows[obj_modes[p][d] - 1];
      coo_subs(mp, p, order, rows, mk_subs[p], &mk_obj[p].nnz);
      mk_obj[p].subs = mk_subs[p].data();
      mk_obj[p].vals = mk_obj[p].nnz > 0 ? mxGetPr(mxGetField(mp, 0, "vals")) : nullptr;
      mk_ptr[p] = &mk_obj[p];
      any_mask = true;
      continue;
    }
    if (mp != nullptr && !mxIsEmpty(mp) && sp_ptr[p] != nullptr)
      fail("aoadmm:unsupported", "Z.miss{" + std::to_string(p + 1) + "} on a sparse object: a sparse object needs a sparse mask");
    if (mp != nullptr && !mxIsEmpty(mp)) {  // EM imputation of the entries with Z.miss == 0 (cmtf_fun_AOADMM.m:408-441)
      if (par2) {
        const int K = o.n_slices;
        if (!mxIsCell(mp) || (int)mxGetNumberOfElements(mp) != K)
          fail("cmtf:missingData:PAR2maskNotCell", "Z.miss{p} must be a cell array with one mask per PARAFAC2 slice");
        miss_par2[p].resize(K);
        miss_par2_ptr[p].resize(K);
        for (int k = 0; k < K; ++k) {
          miss_par2[p][k] = mask_bytes(mxGetCell(mp, k), (size_t)mode_rows[obj_modes[p][0] - 1] * (size_t)slice_rows[obj_modes[p][1] - 1][k], p, pc);
          miss_par2_ptr[p][k] = miss_par2[p][k].data();
        }
        o.miss_slices = miss_par2_ptr[p].data();
      } else {
        size_t expect = 1;
        for (int d = 0; d < order; ++d) expect *= (size_t)mode_rows[obj_modes[p][d] - 1];
        miss_cp[p] = mask_bytes(mp, expect, p, pc);
        o.miss = miss_cp[p].data();
      }
    }
  }

  // couplings
  const mxArray* lin = field(coupling, "lin_coupled_modes");
  std::vector<int32_t> lin_v(nb_modes, 0);
  int n_couplings = 0;
  for (int m = 0; m < nb_modes; ++m) {
    lin_v[m] = (int32_t)mxGetPr(lin)[m];
    if (lin_v[m] > n_couplings) n_couplings = lin_v[m];
  }
  std::vector<int32_t> ctype(n_couplings > 0 ? n_couplings : 1, 0);
  if (const mxArray* ct = field(coupling, "coupling_type", n_couplings > 0))
    for (int c = 0; c < n_couplings && c < (int)mxGetNumberOfElements(ct); ++c) ctype[c] = (int32_t)mxGetPr(ct)[c];
  std::vector<const double*> trafo(nb_modes, nullptr), trafo2(nb_modes, nullptr);
  std::vector<int64_t> tr(nb_modes, 0), tc(nb_modes, 0), tr2(nb_modes, 0), tc2(nb_modes, 0);
  auto read_trafo = [&](const char* name, std::vector<const double*>& ptr, std::vector<int64_t>& r, std::vector<int64_t>& c) {
    const mxArray* t = field(coupling, name, false);
    if (t == nullptr || !mxIsCell(t)) return;
    for (int m = 0; m < nb_modes && m < (int)mxGetNumberOfElements(t); ++m) {
      const mxArray* H = mxGetCell(t, m);
      if (H == nullptr || mxIsEmpty(H)) continue;
      if (mxIsSparse(H)) fail("aoadmm:unsupported", "sparse transformation matrices: pass full(H)");
      ptr[m] = mxGetPr(H);
      r[m] = (int64_t)mxGetM(H);
      c[m] = (int64_t)mxGetN(H);
    }
  };
  read_trafo("coupl_trafo_matrices", trafo, tr, tc);
  read_trafo("coupl_trafo_matrices2", trafo2, tr2, tc2);
  const mxArray* Gcf = field(G, "coupling_fac", n_couplings > 0);
  std::vector<int64_t> crow(n_couplings > 0 ? n_couplings : 1, 0), ccol(n_couplings > 0 ? n_couplings : 1, 0);
  for (int c = 0; c < n_couplings; ++c) {
    const mxArray* D = mxGetCell(Gcf, c);
    crow[c] = (int64_t)mxGetM(D);
    ccol[c] = (int64_t)mxGetN(D);
  }

  // constraints: the named specs (Z.constraints), not the function handles
  const double* cm = mxGetPr(field(Z, "constrained_modes"));
  const mxArray* cons_c = field(Z, "constraints");
  std::vector<int32_t> constrained(nb_modes, 0);
  std::vector<aoadmm_constraint> cons(nb_modes);
  for (int m = 0; m < nb_modes; ++m) {
    std::memset(&cons[m], 0, sizeof(aoadmm_constraint));
    constrained[m] = cm[m] != 0.0;
    if (!constrained[m]) continue;
    const mxArray* c = mxGetCell(cons_c, m);
    if (c == nullptr || !mxIsCell(c) || mxGetNumberOfElements(c) < 1) fail("aoadmm:invalidArg", "Z.constraints{m} must be a cell {name, params...}");
    const std::string name = string_of(mxGetCell(c, 0));
    cons[m].kind = constraint_kind(name);
    const size_t np = mxGetNumberOfElements(c);
    if (cons[m].kind == AOADMM_CON_CUSTOM) fail("aoadmm:unsupported", "'custom' constraints (function handles) cannot run on the device");
    if (cons[m].kind == AOADMM_CON_BOX) {
      cons[m].p0 = scalar_of(mxGetCell(c, 1), "box lower bound");
      cons[m].p1 = scalar_of(mxGetCell(c, 2), "box upper bound");
    } else if (cons[m].kind == AOADMM_CON_UNIMODAL) {
      const mxArray* nn = np > 1 ? mxGetCell(c, 1) : nullptr;
      cons[m].p0 = (nn != nullptr && ((mxIsLogical(nn) && mxIsLogicalScalarTrue(nn)) || (mxIsNumeric(nn) && mxGetScalar(nn) != 0.0))) ? 1.0 : 0.0;
    } else if (cons[m].kind == AOADMM_CON_QUADRATIC) {
      cons[m].p0 = scalar_of(mxGetCell(c, 1), "eta");
      const mxArray* Lm = mxGetCell(c, 2);
      if (mxIsSparse(Lm)) fail("aoadmm:unsupported", "quadratic regularization: pass full(L)");
      cons[m].matrix = mxGetPr(Lm);
      cons[m].matrix_n = (int64_t)mxGetM(Lm);
    } else if (np > 1 && mxIsNumeric(mxGetCell(c, 1))) {
      cons[m].p0 = mxGetScalar(mxGetCell(c, 1));
    }
  }
  const mxArray* ridge = field(Z, "ridge", false);

  aoadmm_problem pb;
  std::memset(&pb, 0, sizeof(pb));
  pb.nb_modes = nb_modes;
  pb.mode_rows = mode_rows.data();
  pb.mode_rank = mode_rank.data();
  pb.slice_rows = slice_ptr.data();
  pb.n_slices = n_slices.data();
  pb.n_objects = P;
  pb.objects = objs.data();
  pb.lin_coupled_modes = lin_v.data();
  pb.n_couplings = n_couplings;
  pb.coupling_type = ctype.data();
  pb.trafo = trafo.data();
  pb.trafo_rows = tr.data();
  pb.trafo_cols = tc.data();
  pb.trafo2 = trafo2.data();
  pb.trafo2_rows = tr2.data();
  pb.trafo2_cols = tc2.data();
  pb.coupling_rows = crow.data();
  pb.coupling_cols = ccol.data();
  pb.constrained_modes = constrained.data();
  pb.constraints = cons.data();
  pb.ridge = (ridge != nullptr && !mxIsEmpty(ridge)) ? mxGetPr(ridge) : nullptr;

  // one MATLAB session drives options.b200_gpus devices (default 1): the library cuts the mode-3 slabs itself.
  // options.b200_shard_sparse = true also cuts sparse objects, into nonzero-balanced slabs of their last mode.
  const int n_gpus = (int)opt_scalar(opt, "b200_gpus", 1.0);
  const bool shard_sparse = opt_scalar(opt, "b200_shard_sparse", 0.0) != 0.0;
  if (n_gpus < 1) fail("aoadmm:invalidArg", "options.b200_gpus must be >= 1");
  if (any_sparse && n_gpus > 1 && !shard_sparse)
    fail("aoadmm:unsupported", "sparse objects run on one GPU (options.b200_gpus must be 1, or set options.b200_shard_sparse)");
  HandleGuard guard;
  if (any_sparse && n_gpus > 1)
    check(aoadmm_create_sparse_multi(&pb, sp_ptr.data(), any_mask ? mk_ptr.data() : nullptr, n_gpus, nullptr, &guard.h),
          nullptr);
  else if (any_mask)
    check(aoadmm_create_sparse_masked(&pb, sp_ptr.data(), mk_ptr.data(), nullptr, &guard.h), nullptr);
  else if (any_sparse)
    check(aoadmm_create_sparse(&pb, sp_ptr.data(), nullptr, &guard.h), nullptr);
  else
    check(n_gpus > 1 ? aoadmm_create_multi(&pb, n_gpus, nullptr, &guard.h) : aoadmm_create(&pb, nullptr, &guard.h), nullptr);
  aoadmm_handle* h = guard.h;

  // ---- state in ------------------------------------------------------------------------------
  auto put = [&](int fld, int index, int slice, const mxArray* a) {
    if (a == nullptr || mxIsEmpty(a)) return;
    check(aoadmm_set_state(h, fld, index, slice, mxGetPr(a), (int64_t)mxGetM(a), (int64_t)mxGetN(a)), h);
  };
  for (const StateField& sf : kModeFields) {
    const mxArray* c = field(G, sf.name, false);
    if (c == nullptr) continue;
    for (int m = 0; m < nb_modes && m < (int)mxGetNumberOfElements(c); ++m) {
      const mxArray* v = mxGetCell(c, m);
      if (v == nullptr || mxIsEmpty(v)) continue;
      if (mxIsCell(v))
        for (int k = 0; k < (int)mxGetNumberOfElements(v); ++k) put(sf.field, m + 1, k, mxGetCell(v, k));
      else
        put(sf.field, m + 1, 0, v);
    }
  }
  for (int c = 0; c < n_couplings; ++c) put(AOADMM_FIELD_COUPLING_FAC, c + 1, 0, mxGetCell(Gcf, c));
  const mxArray *GP = field(G, "P", false), *GD = field(G, "DeltaB", false), *GM = field(G, "mu_DeltaB", false);
  for (int p = 0; p < P; ++p) {
    if (objs[p].model != AOADMM_MODEL_PAR2) continue;
    const mxArray *Pp = mxGetCell(GP, p), *Mp = mxGetCell(GM, p);
    for (int k = 0; k < objs[p].n_slices; ++k) {
      put(AOADMM_FIELD_PAR2_P, p + 1, k, mxGetCell(Pp, k));
      put(AOADMM_FIELD_PAR2_MU_DELTAB, p + 1, k, mxGetCell(Mp, k));
    }
    put(AOADMM_FIELD_PAR2_DELTAB, p + 1, 0, mxGetCell(GD, p));
  }

  // ---- options + run -------------------------------------------------------------------------
  aoadmm_options o;
  std::memset(&o, 0, sizeof(o));
  o.MaxOuterIters = (int32_t)scalar_of(field(opt, "MaxOuterIters"), "MaxOuterIters");
  o.MaxInnerIters = (int32_t)scalar_of(field(opt, "MaxInnerIters"), "MaxInnerIters");
  o.AbsFuncTol = scalar_of(field(opt, "AbsFuncTol"), "AbsFuncTol");
  o.OuterRelTol = scalar_of(field(opt, "OuterRelTol"), "OuterRelTol");
  o.innerRelPrTol_coupl = scalar_of(field(opt, "innerRelPrTol_coupl"), "innerRelPrTol_coupl");
  o.innerRelPrTol_constr = scalar_of(field(opt, "innerRelPrTol_constr"), "innerRelPrTol_constr");
  o.innerRelDualTol_coupl = scalar_of(field(opt, "innerRelDualTol_coupl"), "innerRelDualTol_coupl");
  o.innerRelDualTol_constr = scalar_of(field(opt, "innerRelDualTol_constr"), "innerRelDualTol_constr");
  o.bsum = opt_scalar(opt, "bsum", 0.0) != 0.0;
  o.bsum_weight = opt_scalar(opt, "bsum_weight", 0.0);
  o.iter_start_PAR2Bkconstraint = (int32_t)opt_scalar(opt, "iter_start_PAR2Bkconstraint", 0.0);  // cmtf_fun_AOADMM.m:7-9
  o.has_increase_factor_rhoBk = field(opt, "increase_factor_rhoBk", false) != nullptr;            // :196-198
  o.increase_factor_rhoBk = opt_scalar(opt, "increase_factor_rhoBk", 1.0);
  o.dimtree = (int32_t)opt_scalar(opt, "b200_dimtree", 1.0);  // engine knob, results equal to rounding
  o.mttkrp_precision = (int32_t)opt_scalar(opt, "b200_mttkrp_precision", 0.0);  // opt-in: 1 TF32, 2 BF16 (tcgen05), 3 TF32 (mma.sync)
  o.fuse_inner = (int32_t)opt_scalar(opt, "b200_fuse_inner", 0.0);
  o.graph = (int32_t)opt_scalar(opt, "b200_graph", 0.0);      // engine knob: 0 auto, 1 on, -1 off

  // options.b200_heldout{p}: held-out set of object p (unwrap_data struct of an sptensor / sparse matrix), empty = none
  const mxArray* hcell = field(opt, "b200_heldout", false);
  std::vector<bool> has_ho(P, false);
  if (hcell != nullptr && mxIsCell(hcell)) {
    for (int p = 0; p < P && p < (int)mxGetNumberOfElements(hcell); ++p) {
      const mxArray* hp = mxGetCell(hcell, p);
      if (hp == nullptr || mxIsEmpty(hp)) continue;
      if (!is_coo_struct(hp) || objs[p].model != AOADMM_MODEL_CP)
        fail("aoadmm:invalidArg", "options.b200_heldout{" + std::to_string(p + 1) + "} must be an sptensor or a sparse matrix of a CP object");
      const int order = objs[p].order;
      std::vector<int64_t> rows(order), hs;
      for (int d = 0; d < order; ++d) rows[d] = mode_rows[obj_modes[p][d] - 1];
      aoadmm_sparse_object ho{};
      coo_subs(hp, p, order, rows, hs, &ho.nnz);
      ho.subs = hs.data();
      ho.vals = ho.nnz > 0 ? mxGetPr(mxGetField(hp, 0, "vals")) : nullptr;
      check(aoadmm_set_heldout(h, p + 1, &ho), h);
      has_ho[p] = true;
    }
  }
  // options.b200_heldout_patience = P (needs options.b200_heldout): early stopping on the held-out error; G and the f_*
  // values are those of the best iteration (out.heldout_best_iter)
  const double patience = opt_scalar(opt, "b200_heldout_patience", 0.0);
  if (patience < 0.0) fail("aoadmm:invalidArg", "options.b200_heldout_patience must be >= 0");
  if (patience > 0.0) check(aoadmm_set_heldout_stopping(h, (int32_t)patience), h);

  const int n_hist = o.MaxOuterIters + 1;
  mxArray* hist[6];
  for (auto& a : hist) a = mxCreateDoubleMatrix(1, n_hist, mxREAL);
  std::vector<int32_t> inner((size_t)nb_modes * (o.MaxOuterIters > 0 ? o.MaxOuterIters : 1), 0);
  aoadmm_out ro;
  std::memset(&ro, 0, sizeof(ro));
  ro.func_val_conv = mxGetPr(hist[0]);
  ro.func_coupl_conv = mxGetPr(hist[1]);
  ro.func_constr_conv = mxGetPr(hist[2]);
  ro.func_PAR2_coupl = mxGetPr(hist[3]);
  ro.time_at_it = mxGetPr(hist[4]);
  ro.func_rel_missing = mxGetPr(hist[5]);
  ro.inner_iters = inner.data();
  check(aoadmm_run(h, &o, &ro), h);

  // ---- state out: same struct, same shapes (cmtf_fun_AOADMM.m:1) ------------------------------------
  mxArray* Gout = mxDuplicateArray(G);
  auto get = [&](int fld, int index, int slice, mxArray* a) {
    if (a == nullptr || mxIsEmpty(a)) return;
    check(aoadmm_get_state(h, fld, index, slice, mxGetPr(a), (int64_t)mxGetM(a), (int64_t)mxGetN(a)), h);
  };
  for (const StateField& sf : kModeFields) {
    mxArray* c = mxGetField(Gout, 0, sf.name);
    if (c == nullptr) continue;
    for (int m = 0; m < nb_modes && m < (int)mxGetNumberOfElements(c); ++m) {
      mxArray* v = mxGetCell(c, m);
      if (v == nullptr || mxIsEmpty(v)) continue;
      if (mxIsCell(v))
        for (int k = 0; k < (int)mxGetNumberOfElements(v); ++k) get(sf.field, m + 1, k, mxGetCell(v, k));
      else
        get(sf.field, m + 1, 0, v);
    }
  }
  if (n_couplings > 0) {
    mxArray* c = mxGetField(Gout, 0, "coupling_fac");
    for (int q = 0; q < n_couplings; ++q) get(AOADMM_FIELD_COUPLING_FAC, q + 1, 0, mxGetCell(c, q));
  }
  for (int p = 0; p < P; ++p) {
    if (objs[p].model != AOADMM_MODEL_PAR2) continue;
    mxArray *Pp = mxGetCell(mxGetField(Gout, 0, "P"), p), *Mp = mxGetCell(mxGetField(Gout, 0, "mu_DeltaB"), p);
    for (int k = 0; k < objs[p].n_slices; ++k) {
      get(AOADMM_FIELD_PAR2_P, p + 1, k, mxGetCell(Pp, k));
      get(AOADMM_FIELD_PAR2_MU_DELTAB, p + 1, k, mxGetCell(Mp, k));
    }
    get(AOADMM_FIELD_PAR2_DELTAB, p + 1, 0, mxGetCell(mxGetField(Gout, 0, "DeltaB"), p));
  }
  plhs[0] = Gout;

  // ---- out struct (cmtf_fun_AOADMM.m:480-494) --------------------------------------------------
  if (nlhs > 1) {
    const char* names[] = {"f_tensors", "f_couplings", "f_constraints", "f_PAR2_couplings", "f_rel_missing", "exit_flag",
                           "OuterIterations", "func_val_conv", "func_coupl_conv", "func_constr_conv", "func_PAR2_coupl",
                           "time_at_it", "innerIters", "func_rel_missing", "non_finite_mode", "heldout_sse",
                           "heldout_best_iter"};
    mxArray* out = mxCreateStructMatrix(1, 1, 17, names);
    mxSetField(out, 0, "non_finite_mode", mxCreateDoubleScalar((double)ro.non_finite_mode));
    mxSetField(out, 0, "f_tensors", mxCreateDoubleScalar(ro.f_tensors));
    mxSetField(out, 0, "f_couplings", mxCreateDoubleScalar(ro.f_couplings));
    mxSetField(out, 0, "f_constraints", mxCreateDoubleScalar(ro.f_constraints));
    mxSetField(out, 0, "f_PAR2_couplings", mxCreateDoubleScalar(ro.f_PAR2_couplings));
    mxSetField(out, 0, "f_rel_missing", mxCreateDoubleScalar(ro.f_rel_missing));
    if (ro.exit_flag == 0) {  // make_exit_flag.m:4-5
      mxSetField(out, 0, "exit_flag", mxCreateString("maxIterations"));
    } else if (ro.exit_flag == (1 << 9)) {   // the held-out rule of aoadmm_set_heldout_stopping ended the run
      mxSetField(out, 0, "exit_flag", mxCreateString("heldoutStop"));
    } else {                   // make_exit_flag.m:9-28
      const char* fn[] = {"f_tensors", "f_couplings", "f_constraints", "f_PAR2_couplings"};
      mxArray* ef = mxCreateStructMatrix(1, 1, 4, fn);
      for (int q = 0; q < 4; ++q) mxSetField(ef, 0, fn[q], mxCreateString(((ro.exit_flag >> q) & 1) ? "AbsFuncTol" : "RelFuncTol"));
      mxSetField(out, 0, "exit_flag", ef);
    }
    const int it = ro.OuterIterations;
    mxSetField(out, 0, "OuterIterations", mxCreateDoubleScalar((double)it));
    const char* hn[] = {"func_val_conv", "func_coupl_conv", "func_constr_conv", "func_PAR2_coupl", "time_at_it",
                        "func_rel_missing"};
    for (int q = 0; q < 6; ++q) {
      mxSetN(hist[q], it + 1);  // histories hold it+1 entries (:450-455)
      mxSetField(out, 0, hn[q], hist[q]);
    }
    mxArray* ii = mxCreateDoubleMatrix(nb_modes, it, mxREAL);
    for (int c = 0; c < it; ++c)
      for (int m = 0; m < nb_modes; ++m) mxGetPr(ii)[(size_t)c * nb_modes + m] = (double)inner[(size_t)c * nb_modes + m];
    mxSetField(out, 0, "innerIters", ii);
    // (it+1) x P held-out SSE histories, NaN columns for objects without a held-out set (cmtf_fun_AOADMM.m makes the cell)
    mxArray* hs = mxCreateDoubleMatrix(it + 1, P, mxREAL);
    for (int p = 0; p < P; ++p) {
      double* col = mxGetPr(hs) + (size_t)p * (it + 1);
      if (has_ho[p]) check(aoadmm_heldout_history(h, p + 1, col, it + 1, nullptr), h);
      else for (int i = 0; i <= it; ++i) col[i] = mxGetNaN();
    }
    mxSetField(out, 0, "heldout_sse", hs);
    if (patience > 0.0) {
      int32_t best = 0;
      double best_sse = 0.0;
      check(aoadmm_heldout_best(h, &best, &best_sse), h);
      mxSetField(out, 0, "heldout_best_iter", mxCreateDoubleScalar((double)best));
    }
    plhs[1] = out;
  } else {
    for (auto& a : hist) mxDestroyArray(a);
  }
}
}  // namespace

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  std::string id, msg;
  try {
    solve(nlhs, plhs, nrhs, prhs);
    return;
  } catch (const MexError& e) {
    id = e.id;
    msg = e.msg;
  } catch (const std::exception& e) {
    id = "aoadmm:internal";
    msg = e.what();
  }
  // MATLAB copies the formatted message before the longjmp; the two strings above are the only live C++ objects
  static char idbuf[128], msgbuf[2048];
  std::strncpy(idbuf, id.c_str(), sizeof(idbuf) - 1);
  std::strncpy(msgbuf, msg.c_str(), sizeof(msgbuf) - 1);
  id.clear();
  id.shrink_to_fit();
  msg.clear();
  msg.shrink_to_fit();
  mexErrMsgIdAndTxt(idbuf, "%s", msgbuf);
}
