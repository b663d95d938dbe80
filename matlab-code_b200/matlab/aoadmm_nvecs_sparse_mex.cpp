// aoadmm_nvecs_sparse_mex.cpp - MEX gateway of the device-side nvecs initialisation of a sparse mode.
//
//   U = aoadmm_nvecs_sparse_mex(S, i, r)
//     S : struct('subs',subs,'vals',vals,'size',sz) of the sparse tensor (or matrix) that contains the mode, as
//         cmtf_fun_AOADMM.m's unwrap_data hands a sptensor / MATLAB sparse matrix over: subs nnz x N 1-based double
//         subscripts (2 <= N <= 8), vals nnz doubles, sz the N extents
//     i : position of the mode inside S (1-based)
//     r : number of vectors
// the leading eigenvectors of Y = X_(i) X_(i)' with the unstored entries counted as zero, computed on the device without
// forming Y (include/aoadmm.h: aoadmm_nvecs_sparse).  Build:
//   mex -R2018a -I<repo>/include aoadmm_nvecs_sparse_mex.cpp -L<repo>/matlab-code_b200/aoadmm_b200 -laoadmm_b200
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "aoadmm.h"
#include "mex.h"

namespace {

// subs (1-based doubles, nnz x order) -> 0-based int64, column-major, with an integer and range check per entry
void coo_subs(const mxArray* a, int order, const std::vector<int64_t>& rows, std::vector<int64_t>& subs, int64_t* nnz) {
  const mxArray* S = mxGetField(a, 0, "subs");
  const mxArray* V = mxGetField(a, 0, "vals");
  if (!mxIsDouble(S) || !mxIsDouble(V)) mexErrMsgIdAndTxt("aoadmm:invalidArg", "S: subs and vals must be double");
  const size_t n = mxGetNumberOfElements(V);
  if (n > 0 && (mxGetM(S) != n || (int)mxGetN(S) != order))
    mexErrMsgIdAndTxt("aoadmm:invalidArg", "S: subs must be nnz x %d with one row per value", order);
  const double* s = n > 0 ? mxGetPr(S) : nullptr;
  subs.resize(n * (size_t)order);
  for (int d = 0; d < order; ++d)
    for (size_t e = 0; e < n; ++e) {
      const double v = s[(size_t)d * n + e];
      if (!(v >= 1.0 && v <= (double)rows[d]) || v != (double)(int64_t)v)
        mexErrMsgIdAndTxt("aoadmm:invalidArg", "S: subscript %g in column %d is not an integer in 1..%lld", v, d + 1,
                          (long long)rows[d]);
      subs[(size_t)d * n + e] = (int64_t)v - 1;
    }
  *nnz = (int64_t)n;
}

}  // namespace

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs != 3 || nlhs > 1) mexErrMsgIdAndTxt("aoadmm:invalidArg", "usage: U = aoadmm_nvecs_sparse_mex(S, i, r)");
  const mxArray* S = prhs[0];
  if (!mxIsStruct(S) || mxGetField(S, 0, "subs") == nullptr || mxGetField(S, 0, "vals") == nullptr ||
      mxGetField(S, 0, "size") == nullptr)
    mexErrMsgIdAndTxt("aoadmm:invalidArg", "S must be struct('subs',subs,'vals',vals,'size',sz)");
  const mxArray* sz = mxGetField(S, 0, "size");
  if (!mxIsDouble(sz)) mexErrMsgIdAndTxt("aoadmm:invalidArg", "S.size must be double");
  const int order = (int)mxGetNumberOfElements(sz);
  const int pos = (int)mxGetScalar(prhs[1]), r = (int)mxGetScalar(prhs[2]);
  if (order < 2 || order > 8 || pos < 1 || pos > order) mexErrMsgIdAndTxt("aoadmm:invalidArg", "mode position out of range");

  std::vector<int64_t> rows(order);
  std::vector<int32_t> rank(order, r), modes(order), lin(order, 0), constrained(order, 0);
  std::vector<aoadmm_constraint> cons(order);
  std::memset(cons.data(), 0, sizeof(aoadmm_constraint) * order);
  for (int d = 0; d < order; ++d) {
    const double v = mxGetPr(sz)[d];
    if (!(v >= 1.0) || v != (double)(int64_t)v) mexErrMsgIdAndTxt("aoadmm:invalidArg", "S.size must hold positive integers");
    rows[d] = (int64_t)v;
    modes[d] = d + 1;
  }
  if (r < 1 || r > rows[pos - 1]) mexErrMsgIdAndTxt("aoadmm:invalidArg", "r must be between 1 and the mode size");
  std::vector<int64_t> subs;
  aoadmm_sparse_object sp;
  std::memset(&sp, 0, sizeof(sp));
  coo_subs(S, order, rows, subs, &sp.nnz);
  sp.subs = subs.data();
  sp.vals = sp.nnz > 0 ? mxGetPr(mxGetField(S, 0, "vals")) : nullptr;
  const aoadmm_sparse_object* sp_ptr = &sp;
  aoadmm_object obj;
  std::memset(&obj, 0, sizeof(obj));
  obj.model = AOADMM_MODEL_CP;
  obj.order = order;
  obj.modes = modes.data();
  obj.weight = 1.0;
  obj.znorm_const = 0.0;
  obj.data = nullptr;
  obj.shard_offset = 0;
  obj.shard_extent = rows[order - 1];
  aoadmm_problem pb;
  std::memset(&pb, 0, sizeof(pb));
  pb.nb_modes = order;
  pb.mode_rows = rows.data();
  pb.mode_rank = rank.data();
  pb.n_objects = 1;
  pb.objects = &obj;
  pb.lin_coupled_modes = lin.data();
  pb.n_couplings = 0;
  pb.constrained_modes = constrained.data();
  pb.constraints = cons.data();
  aoadmm_dist dist;
  std::memset(&dist, 0, sizeof(dist));
  dist.world_size = 1;

  aoadmm_handle* h = nullptr;
  int st = aoadmm_create_sparse(&pb, &sp_ptr, &dist, &h);
  if (st != AOADMM_OK) mexErrMsgIdAndTxt("aoadmm:create", "%s", aoadmm_last_error(h));
  plhs[0] = mxCreateDoubleMatrix((mwSize)rows[pos - 1], (mwSize)r, mxREAL);
  st = aoadmm_nvecs_sparse(h, pos, r, mxGetPr(plhs[0]), rows[pos - 1], nullptr);
  if (st != AOADMM_OK) {
    // copy the message before the handle (its owner) goes away
    char msg[512];
    std::strncpy(msg, aoadmm_last_error(h), sizeof(msg) - 1);
    msg[sizeof(msg) - 1] = 0;
    aoadmm_destroy(h);
    mexErrMsgIdAndTxt(st == AOADMM_ERR_UNSUPPORTED ? "aoadmm:unsupported" : "aoadmm:nvecs", "%s", msg);
  }
  aoadmm_destroy(h);
}
