// Device-resident TT containers and the TT-level operations built from the kernels (internal).
#pragma once
#include "ttn_internal.h"

namespace ttn {

// TTvector (src/tt_tools.jl:23-29) resident in HBM.  Core k is the dense column-major array
// (n_k, r_k, r_{k+1}, batch): `batch` independent TTs of identical shape share one allocation per site so
// that every kernel can address them through a batch stride (cfg5: 4096 QTT vectors).
template <class T>
struct TT {
  int d = 0;
  int batch = 1;
  std::vector<int64_t> dims, rks, ot;
  std::vector<DevBuf> cores;
  int64_t core_elems(int k) const { return dims[k] * rks[k] * rks[k + 1]; }
  T* core(int k) const { return cores[k].as<T>(); }
  void alloc_core(int k) { cores[k].alloc(sizeof(T) * (size_t)core_elems(k) * batch); }
};

// TToperator (src/tt_tools.jl:48-54): core k is (n_k, n_k, R_k, R_{k+1}); never batched.
template <class T>
struct TTO {
  int d = 0;
  std::vector<int64_t> dims, rks;
  std::vector<DevBuf> cores;
  T* core(int k) const { return cores[k].as<T>(); }
};

template <class T> void tt_copy(const TT<T>& x, TT<T>& y);
template <class T> void tt_apply(const TTO<T>& A, const TT<T>& x, TT<T>& y);
template <class T> void tt_dot(const TT<T>& a, const TT<T>& b, std::vector<T>& out);
template <class T> void tt_add(const TT<T>& x, const TT<T>& y, TT<T>& z);
template <class T> void tt_scale(const TT<T>& x, T a, TT<T>& y);
template <class T> void tt_orthogonalize(const TT<T>& x, int center /*1-based*/, TT<T>& y);
// tail-norm rank rule of src/tt_cross_interpolation.jl:149-166
int rank_tailnorm(const double* s, int len, int64_t max_bond, double truncerr);
// returns the buffers of the two cores it replaced (k and k+1); dropping them releases them
template <class T>
std::pair<DevBuf, DevBuf> tt_bond_truncate(TT<T>& x, int k /*1-based*/, int64_t max_bond, double truncerr, double* sigma_out,
                                           int64_t sigma_cap);
template <class T>
void tt_compress(TT<T>& x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride);

// y = tt_compress!(A * x, ...) with the product cores folded into the two-site merges (tt.cu)
template <class T>
void tt_apply_compress(const TTO<T>& A, const TT<T>& x, TT<T>& y, int64_t max_bond, double truncerr, int sweeps, double* sigma_out,
                       int64_t sigma_stride);

// site surgery (sites.cu): adjacent-site swap, diagonal merge, site split.  mode 0: relative threshold `tol` on sigma_j/sigma_1
// (qtt_tools.jl:680-685);  mode 1: `_svdtrunc` tail-norm rule with `max_bond` cap (tt_cross_interpolation.jl:149-166)
template <class T> void tt_swap_sites(TT<T>& x, int k /*1-based*/, int mode, int64_t max_bond, double tol);
template <class T> void tt_merge_diag(TT<T>& x, int k /*1-based*/);
template <class T> void tt_split_site(TT<T>& x, int k /*1-based*/, int64_t coarse, int mode, int64_t max_bond, double tol);

// Truncated split of a strided p x q matrix Theta (batch 1):  Theta ~ U * (S Vt),  U (p x r) orthonormal columns
// (column-major, ld p) and SVt = U^H Theta (r x q, column-major, ld r).  `rule(sigma, k)` returns the rank.
template <class T, class Rule>
int split_left(const T* Theta, int p, int q, int64_t rs, int64_t cs, bool conj, Rule rule, DevBuf& U, DevBuf& SVt,
               std::vector<double>* sigma_host = nullptr) {
  SvdLeft sv;
  svd_left<T>(Theta, p, q, rs, cs, conj, sv, 1, 0);
  int r = rule(sv.sigma.data(), sv.k);
  if (r < 1) r = 1;
  if (r > sv.k) r = sv.k;
  std::vector<double> sc(r);
  for (int j = 0; j < r; ++j) sc[j] = sv.sigma[j] > 1e-290 ? 1.0 / sv.sigma[j] : 0.0;
  DevBuf dperm(sizeof(int) * r), dsc(sizeof(double) * r);
  TTN_CUDA(cudaMemcpyAsync(dperm.p, sv.perm.data(), sizeof(int) * r, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(dsc.p, sc.data(), sizeof(double) * r, cudaMemcpyHostToDevice, ctx().stream));
  U.alloc(sizeof(T) * (size_t)p * r);
  gather_cols<T>(sv.X.as<T>(), p, p, dperm.as<int>(), dsc.as<double>(), r, U.as<T>(), 1, p);
  SVt.alloc(sizeof(T) * (size_t)r * q);
  GemmArgs g;
  g.M = r; g.N = q; g.K = p;
  g.A = U.p; g.sAm = p; g.sAk = 1; g.conjA = true;
  g.B = Theta; g.sBk = rs; g.sBn = cs; g.conjB = conj;
  g.C = SVt.p; g.sCm = 1; g.sCn = r;
  gemm<T>(g);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));  // sc / perm host staging must outlive the copies
  if (sigma_host) sigma_host->assign(sv.sigma.begin(), sv.sigma.begin() + sv.k);
  return r;
}

}  // namespace ttn

// opaque handle types of the C ABI
struct ttn_ttv_s {
  int dtype = 0;
  ttn::TT<double> r;
  ttn::TT<ttn::zc> c;
  // asynchronous host <-> device traffic on the library's copy stream (ttn_ttv_upload_async / ttn_ttv_download_async):
  cudaEvent_t ready = nullptr;   // recorded after the H2D copies: the compute stream must wait for it before the first use
  cudaEvent_t busy = nullptr;    // recorded after the D2H copies: the cores must not be released before it
  // A handle freed while its D2H copies are still in flight parks its cores on the calling thread's deferred list (api.cu) and
  // they go back to the block cache once the event has completed, so the compute stream never waits for the copy engine.
  ~ttn_ttv_s();
};
namespace ttn {
/// returns the cores of freed handles whose asynchronous downloads have completed to the block cache (`block`: wait for all)
void drain_deferred_releases(bool block);
}
struct ttn_tto_s {
  int dtype = 0;
  ttn::TTO<double> r;
  ttn::TTO<ttn::zc> c;
};
