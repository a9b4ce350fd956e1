// TT-level operations on device-resident trains: apply, dot, +, scalar *, orthogonalize, tt_compress!.
// Each function cites the reference lines it reproduces; the arithmetic is carried by the kernels in
// gemm.cu / apply.cu / qr.cu / jacobi.cu / elementwise.cu, the host code here only sequences launches.
#include <functional>
#include "tt.h"

namespace ttn {

template <class T>
void tt_copy(const TT<T>& x, TT<T>& y) {
  y.d = x.d; y.batch = x.batch; y.dims = x.dims; y.rks = x.rks; y.ot = x.ot;
  y.cores.clear();
  y.cores.resize(x.d);
  for (int k = 0; k < x.d; ++k) {
    y.alloc_core(k);
    TTN_CUDA(cudaMemcpyAsync(y.cores[k].p, x.cores[k].p, y.cores[k].bytes, cudaMemcpyDeviceToDevice, ctx().stream));
  }
}

// shape of y = A * x (ranks A.rks * x.rks), no core allocated yet
template <class T>
static void product_shape(const TTO<T>& A, const TT<T>& x, TT<T>& y) {
  y.d = x.d; y.batch = x.batch; y.dims = x.dims;
  y.rks.resize(x.d + 1);
  for (int k = 0; k <= x.d; ++k) y.rks[k] = A.rks[k] * x.rks[k];
  y.ot.assign(x.d, 0);
  y.cores.clear();
  y.cores.resize(x.d);
}

// core k of y = A * x   (src/tt_operations.jl:105-108)
template <class T>
static void apply_site(const TTO<T>& A, const TT<T>& x, TT<T>& y, int k) {
  y.alloc_core(k);
  apply_core<T>(A.core(k), x.core(k), y.core(k), (int)A.dims[k], (int)A.dims[k], (int)A.rks[k], (int)A.rks[k + 1], (int)x.rks[k],
                (int)x.rks[k + 1], x.batch, x.core_elems(k), y.core_elems(k));
}

// src/tt_operations.jl:101-111
template <class T>
void tt_apply(const TTO<T>& A, const TT<T>& x, TT<T>& y) {
  ttn_assert(A.d == x.d && A.dims == x.dims, 1, "Incompatible dimensions");
  product_shape(A, x, y);
  for (int k = 0; k < x.d; ++k) apply_site(A, x, y, k);
}

// src/tt_operations.jl:239-250:  M <- A_k^H (B_k M), conj on the first argument
template <class T>
void tt_dot(const TT<T>& A, const TT<T>& B, std::vector<T>& out) {
  ttn_assert(A.d == B.d && A.dims == B.dims && A.batch == B.batch, 1, "TT dimensions are not compatible");
  const int batch = A.batch;
  DevBuf M(sizeof(T) * (size_t)A.rks[0] * B.rks[0] * batch);
  ttn_assert(A.rks[0] == 1 && B.rks[0] == 1, 1, "dot: boundary ranks must be 1");
  fill<T>(M.as<T>(), batch, t_one<T>());
  for (int k = 0; k < A.d; ++k) {
    const int n = (int)A.dims[k];
    const int ral = (int)A.rks[k], rar = (int)A.rks[k + 1], rbl = (int)B.rks[k], rbr = (int)B.rks[k + 1];
    DevBuf Tb(sizeof(T) * (size_t)n * ral * rbr * batch);
    GemmArgs g;  // T[z,alpha,b] = sum_beta M[alpha,beta] B[z,beta,b]
    g.M = ral; g.N = rbr; g.K = rbl;
    g.A = M.p; g.sAm = 1; g.sAk = ral; g.bA1 = 0; g.bA2 = (int64_t)ral * rbl;
    g.B = B.cores[k].p; g.sBk = n; g.sBn = (int64_t)n * rbl; g.bB1 = 1; g.bB2 = B.core_elems(k);
    g.C = Tb.p; g.sCm = n; g.sCn = (int64_t)n * ral; g.bC1 = 1; g.bC2 = (int64_t)n * ral * rbr;
    g.batch1 = n; g.batch2 = batch;
    gemm<T>(g);
    DevBuf Mn(sizeof(T) * (size_t)rar * rbr * batch);
    GemmArgs h;  // M'[a,b] = sum_(z,alpha) conj(A[(z,alpha),a]) T[(z,alpha),b]
    h.M = rar; h.N = rbr; h.K = n * ral;
    h.A = A.cores[k].p; h.sAm = (int64_t)n * ral; h.sAk = 1; h.conjA = true; h.bA2 = A.core_elems(k);
    h.B = Tb.p; h.sBk = 1; h.sBn = (int64_t)n * ral; h.bB2 = (int64_t)n * ral * rbr;
    h.C = Mn.p; h.sCm = 1; h.sCn = rar; h.bC2 = (int64_t)rar * rbr;
    h.batch1 = 1; h.batch2 = batch;
    gemm<T>(h);
    M = std::move(Mn);
  }
  ttn_assert(A.rks[A.d] == 1 && B.rks[B.d] == 1, 1, "dot: boundary ranks must be 1");
  out.resize(batch);
  read_back(out.data(), M.p, sizeof(T) * batch);
}

// src/tt_operations.jl:10-35 (block-diagonal concatenation)
template <class T>
void tt_add(const TT<T>& x, const TT<T>& y, TT<T>& z) {
  ttn_assert(x.d == y.d && x.dims == y.dims && x.batch == y.batch, 1, "Incompatible dimensions");
  const int d = x.d, batch = x.batch;
  z.d = d; z.batch = batch; z.dims = x.dims; z.ot.assign(d, 0);
  z.rks.resize(d + 1);
  for (int k = 0; k <= d; ++k) z.rks[k] = x.rks[k] + y.rks[k];
  z.rks[0] = 1; z.rks[d] = 1;
  z.cores.clear();
  z.cores.resize(d);
  for (int k = 0; k < d; ++k) {
    z.alloc_core(k);
    const int64_t n = x.dims[k], zl = z.rks[k], zr = z.rks[k + 1];
    if (d == 1) {
      TTN_CUDA(cudaMemcpyAsync(z.cores[k].p, x.cores[k].p, z.cores[k].bytes, cudaMemcpyDeviceToDevice, ctx().stream));
      axpy<T>(z.core_elems(k) * batch, t_one<T>(), y.core(k), z.core(k));
      continue;
    }
    fill<T>(z.core(k), z.core_elems(k) * batch, t_zero<T>());
    for (int which = 0; which < 2; ++which) {
      const TT<T>& s = which == 0 ? x : y;
      const int64_t sl = s.rks[k], sr = s.rks[k + 1];
      const int64_t offl = (which == 1 && k > 0) ? x.rks[k] : 0;
      const int64_t offr = (which == 1 && k < d - 1) ? x.rks[k + 1] : 0;
      Copy4 c;
      c.n0 = n * sl; c.n1 = sr; c.n2 = batch;                 // (s,alpha) fused is contiguous in the source
      c.s0 = 1; c.s1 = n * sl; c.s2 = s.core_elems(k);
      c.d0 = 1; c.d1 = n * zl; c.d2 = z.core_elems(k);
      // destination offset: rows start at alpha = offl, columns at beta = offr; the fused (s,alpha) index is only
      // contiguous when zl == sl, so copy per physical index otherwise
      if (zl == sl) {
        copy4<T>(s.core(k), z.core(k) + n * offl + n * zl * offr, c);
      } else {
        Copy4 e;
        e.n0 = n; e.n1 = sl; e.n2 = sr; e.n3 = batch;
        e.s0 = 1; e.s1 = n; e.s2 = n * sl; e.s3 = s.core_elems(k);
        e.d0 = 1; e.d1 = n; e.d2 = n * zl; e.d3 = z.core_elems(k);
        copy4<T>(s.core(k), z.core(k) + n * offl + n * zl * offr, e);
      }
    }
    (void)zr;
  }
}

// src/tt_operations.jl:256-266: scales the first core whose ot flag is 0 (core 1 if there is none)
template <class T>
void tt_scale(const TT<T>& x, T a, TT<T>& y) {
  tt_copy(x, y);
  if (t_abs2(a) == 0.0) {
    for (int k = 0; k < y.d; ++k) fill<T>(y.core(k), y.core_elems(k) * y.batch, t_zero<T>());
    y.ot.assign(y.d, 0);
    return;
  }
  int i = 0;
  for (int k = 0; k < x.d; ++k)
    if (x.ot[k] == 0) { i = k; break; }
  scal<T>(y.core_elems(i) * y.batch, a, y.core(i));
}

// src/tt_tools.jl:511-543
template <class T>
void tt_orthogonalize(const TT<T>& x, int center, TT<T>& y) {
  const int d = x.d, batch = x.batch;
  ttn_assert(1 <= center && center <= d, 3, "Impossible orthogonalization");
  ttn_assert(x.rks[0] == 1 && x.rks[d] == 1, 1, "orthogonalize: boundary ranks must be 1");
  y.d = d; y.batch = batch; y.dims = x.dims; y.rks = x.rks; y.ot.assign(d, 0);
  y.cores.clear();
  y.cores.resize(d);
  const int ci = center - 1;

  // left sweep: QR of (r_{j-1} n) x r_j with row index alpha + r_{j-1} s   (tt_tools.jl:518-525)
  DevBuf FR(sizeof(T) * batch);
  fill<T>(FR.as<T>(), batch, t_one<T>());
  int fr_rows = 1;  // FR is (fr_rows x x.rks[j]) per batch element, ld = fr_rows
  for (int j = 0; j < ci; ++j) {
    const int n = (int)x.dims[j], xl = (int)x.rks[j], xr = (int)x.rks[j + 1], yl = fr_rows;
    const int m = yl * n, k = std::min(m, xr);
    DevBuf W(sizeof(T) * (size_t)m * xr * batch), tau(sizeof(T) * (size_t)k * batch);
    GemmArgs g;  // W[(alpha,s), gamma] = sum_beta FR[alpha,beta] x[s,beta,gamma]
    g.M = yl; g.N = xr; g.K = xl;
    g.A = FR.p; g.sAm = 1; g.sAk = yl; g.bA1 = 0; g.bA2 = (int64_t)yl * xl;
    g.B = x.cores[j].p; g.sBk = n; g.sBn = (int64_t)n * xl; g.bB1 = 1; g.bB2 = x.core_elems(j);
    g.C = W.p; g.sCm = 1; g.sCn = m; g.bC1 = yl; g.bC2 = (int64_t)m * xr;
    g.batch1 = n; g.batch2 = batch;
    gemm<T>(g);
    qr_factor<T>(W.as<T>(), m, xr, m, tau.as<T>(), batch, (int64_t)m * xr, k);
    DevBuf Q(sizeof(T) * (size_t)m * k * batch);
    qr_form_q<T>(W.as<T>(), m, k, m, tau.as<T>(), Q.as<T>(), m, batch, (int64_t)m * xr, k, (int64_t)m * k);
    y.rks[j] = yl; y.rks[j + 1] = k; y.ot[j] = 1;
    y.alloc_core(j);
    Copy4 c;  // y[s,alpha,kappa] = Q[alpha + yl*s, kappa]
    c.n0 = yl; c.n1 = n; c.n2 = k; c.n3 = batch;
    c.s0 = 1; c.s1 = yl; c.s2 = m; c.s3 = (int64_t)m * k;
    c.d0 = n; c.d1 = 1; c.d2 = (int64_t)n * yl; c.d3 = y.core_elems(j);
    copy4<T>(Q.as<T>(), y.core(j), c);
    DevBuf FRn(sizeof(T) * (size_t)k * xr * batch);
    Copy4 t;  // FR = R[1:k, :]
    t.n0 = k; t.n1 = xr; t.n2 = batch; t.s0 = 1; t.s1 = m; t.s2 = (int64_t)m * xr; t.d0 = 1; t.d1 = k; t.d2 = (int64_t)k * xr;
    t.tri = 1;
    copy4<T>(W.as<T>(), FRn.as<T>(), t);
    FR = std::move(FRn);
    fr_rows = k;
  }

  // right sweep: LQ of r_{j-1} x (r_j n) with column index beta + r_j s  (tt_tools.jl:528-536), done as the QR of
  // the conjugate transpose
  DevBuf FL(sizeof(T) * batch);
  fill<T>(FL.as<T>(), batch, t_one<T>());
  int fl_cols = 1;  // FL is (x.rks[j+1] x fl_cols) per batch element, ld = x.rks[j+1]
  for (int j = d - 1; j > ci; --j) {
    const int n = (int)x.dims[j], xl = (int)x.rks[j], xr = (int)x.rks[j + 1], yr = fl_cols;
    const int m = yr * n, k = std::min(m, xl);
    DevBuf W(sizeof(T) * (size_t)m * xl * batch), tau(sizeof(T) * (size_t)k * batch);
    GemmArgs g;  // W[(beta,s), alpha] = conj( sum_gamma x[s,alpha,gamma] FL[gamma,beta] )
    g.M = yr; g.N = xl; g.K = xr;
    g.A = FL.p; g.sAm = xr; g.sAk = 1; g.conjA = true; g.bA1 = 0; g.bA2 = (int64_t)xr * yr;
    g.B = x.cores[j].p; g.sBk = (int64_t)n * xl; g.sBn = n; g.conjB = true; g.bB1 = 1; g.bB2 = x.core_elems(j);
    g.C = W.p; g.sCm = 1; g.sCn = m; g.bC1 = yr; g.bC2 = (int64_t)m * xl;
    g.batch1 = n; g.batch2 = batch;
    gemm<T>(g);
    qr_factor<T>(W.as<T>(), m, xl, m, tau.as<T>(), batch, (int64_t)m * xl, k);
    DevBuf Q(sizeof(T) * (size_t)m * k * batch);
    qr_form_q<T>(W.as<T>(), m, k, m, tau.as<T>(), Q.as<T>(), m, batch, (int64_t)m * xl, k, (int64_t)m * k);
    y.rks[j] = k; y.rks[j + 1] = yr; y.ot[j] = -1;
    y.alloc_core(j);
    Copy4 c;  // y[s,kappa,beta] = conj(Q[beta + yr*s, kappa])
    c.n0 = yr; c.n1 = n; c.n2 = k; c.n3 = batch;
    c.s0 = 1; c.s1 = yr; c.s2 = m; c.s3 = (int64_t)m * k;
    c.d0 = (int64_t)n * k; c.d1 = 1; c.d2 = n; c.d3 = y.core_elems(j);
    c.conj = true;
    copy4<T>(Q.as<T>(), y.core(j), c);
    DevBuf FLn(sizeof(T) * (size_t)xl * k * batch);
    Copy4 t;  // FL[alpha,kappa] = conj(R[kappa,alpha]), kappa <= alpha
    t.n0 = k; t.n1 = xl; t.n2 = batch; t.s0 = 1; t.s1 = m; t.s2 = (int64_t)m * xl; t.d0 = xl; t.d1 = 1; t.d2 = (int64_t)xl * k;
    t.tri = 1; t.conj = true;
    copy4<T>(W.as<T>(), FLn.as<T>(), t);
    FL = std::move(FLn);
    fl_cols = k;
  }

  // centre core: y[s,:,:] = FR x[s,:,:] FL  (tt_tools.jl:538-541)
  {
    const int n = (int)x.dims[ci], xl = (int)x.rks[ci], xr = (int)x.rks[ci + 1], yl = fr_rows, yr = fl_cols;
    DevBuf Tmp(sizeof(T) * (size_t)n * yl * xr * batch);
    GemmArgs g;  // Tmp[s,alpha,gamma] = sum_beta FR[alpha,beta] x[s,beta,gamma]
    g.M = yl; g.N = xr; g.K = xl;
    g.A = FR.p; g.sAm = 1; g.sAk = yl; g.bA2 = (int64_t)yl * xl;
    g.B = x.cores[ci].p; g.sBk = n; g.sBn = (int64_t)n * xl; g.bB1 = 1; g.bB2 = x.core_elems(ci);
    g.C = Tmp.p; g.sCm = n; g.sCn = (int64_t)n * yl; g.bC1 = 1; g.bC2 = (int64_t)n * yl * xr;
    g.batch1 = n; g.batch2 = batch;
    gemm<T>(g);
    y.rks[ci] = yl; y.rks[ci + 1] = yr; y.ot[ci] = 0;
    y.alloc_core(ci);
    GemmArgs h;  // y[(s,alpha), beta'] = sum_gamma Tmp[(s,alpha),gamma] FL[gamma,beta']
    h.M = n * yl; h.N = yr; h.K = xr;
    h.A = Tmp.p; h.sAm = 1; h.sAk = (int64_t)n * yl; h.bA2 = (int64_t)n * yl * xr;
    h.B = FL.p; h.sBk = 1; h.sBn = xr; h.bB2 = (int64_t)xr * yr;
    h.C = y.cores[ci].p; h.sCm = 1; h.sCn = (int64_t)n * yl; h.bC2 = y.core_elems(ci);
    h.batch1 = 1; h.batch2 = batch;
    gemm<T>(h);
  }
}

int rank_tailnorm(const double* s, int len, int64_t max_bond, double truncerr) {
  int r = len;
  if (truncerr > 0) {
    double n2 = 0.0;
    for (int i = 0; i < len; ++i) n2 += s[i] * s[i];
    const double nrm = std::sqrt(n2);
    double cum = 0.0;
    for (int i = len; i >= 1; --i) {
      cum += s[i - 1] * s[i - 1];
      if (std::sqrt(cum) > truncerr * nrm) { r = i; break; }
    }
  }
  if ((int64_t)r > max_bond) r = (int)max_bond;
  return r;
}

// Theta[(s1,alpha),(s2,beta)] = sum_gamma A[s1,alpha,gamma] B[s2,gamma,beta] of bond (k, k+1)     (tt_tools.jl:749)
template <class T>
static void two_site_merge(const TT<T>& x, int k, DevBuf& Th) {
  const int n2 = (int)x.dims[k + 1], p = (int)x.dims[k] * (int)x.rks[k], r = (int)x.rks[k + 1], rr = (int)x.rks[k + 2];
  GemmArgs g;
  g.M = p; g.N = rr; g.K = r;
  g.A = x.cores[k].p; g.sAm = 1; g.sAk = p; g.bA1 = 0; g.bA2 = x.core_elems(k);
  g.B = x.cores[k + 1].p; g.sBk = n2; g.sBn = (int64_t)n2 * r; g.bB1 = 1; g.bB2 = x.core_elems(k + 1);
  g.C = Th.p; g.sCm = 1; g.sCn = (int64_t)p * n2; g.bC1 = p; g.bC2 = (int64_t)p * n2 * rr;
  g.batch1 = n2; g.batch2 = x.batch;
  gemm<T>(g);
}

// newB[s2,kappa,beta] = sum_row conj(G2[row,kappa]) Th[row,(s2,beta)] for the rc computed of rn rows: core k+1 of a split bond
template <class T>
static void project(const DevBuf& G2, const DevBuf& Th, int pe, int rc, int rn, int n2, int rr, int batch, DevBuf& newB) {
  GemmArgs g;
  g.M = rc; g.N = rr; g.K = pe;
  g.A = G2.p; g.sAm = pe; g.sAk = 1; g.conjA = true; g.bA1 = 0; g.bA2 = (int64_t)pe * rc;
  g.B = Th.p; g.sBk = 1; g.sBn = (int64_t)pe * n2; g.bB1 = pe; g.bB2 = (int64_t)pe * n2 * rr;
  g.C = newB.p; g.sCm = n2; g.sCn = (int64_t)n2 * rn; g.bC1 = 1; g.bC2 = (int64_t)n2 * rn * rr;
  g.batch1 = n2; g.batch2 = batch;
  gemm<T>(g);
}

// the cores that replace k and k+1 of a truncated bond, A (p x rn) and B (n2 x rn x rr) per train, and the squared column norms w
// (rn per train) of a core k = U sqrt(S)
struct NewBond { DevBuf A, B, w; };

// allocates a NewBond (w only when asked) and zero-fills it when only `computed` < rn columns will be written
template <class T>
static NewBond new_bond(int p, int n2, int rn, int rr, int batch, int computed, bool with_w) {
  NewBond nb;
  nb.A.alloc(sizeof(T) * (size_t)p * rn * batch);
  nb.B.alloc(sizeof(T) * (size_t)n2 * rn * rr * batch);
  if (with_w) nb.w.alloc(sizeof(double) * (size_t)rn * batch);
  if (computed < rn) {
    fill<T>(nb.A.as<T>(), (int64_t)p * rn * batch, t_zero<T>());
    fill<T>(nb.B.as<T>(), (int64_t)n2 * rn * rr * batch, t_zero<T>());
    if (with_w) TTN_CUDA(cudaMemsetAsync(nb.w.p, 0, nb.w.bytes, ctx().stream));
  }
  return nb;
}

// src/tt_tools.jl:743-768 (without the discarded orthogonalize of :769)
template <class T>
std::pair<DevBuf, DevBuf> tt_bond_truncate(TT<T>& x, int k1, int64_t max_bond, double truncerr, double* sigma_out, int64_t sigma_cap) {
  ttn_assert(1 <= k1 && k1 < x.d, 2, "k must be in 1:(N-1)");
  ttn_assert(max_bond >= 1, 2, "max_bond must be >= 1");
  const int k = k1 - 1, batch = x.batch;
  ttn_assert(batch == 1 || truncerr == 0.0, 2, "batched tt_compress needs truncerr == 0 (uniform ranks)");
  const int n1 = (int)x.dims[k], n2 = (int)x.dims[k + 1];
  const int rl = (int)x.rks[k], r = (int)x.rks[k + 1], rr = (int)x.rks[k + 2];
  const int p = n1 * rl, q = n2 * rr;
  // Rank-deficient bond (inner dimension r well below min(p,q): every R->L step of tt_compress!, and the first sweep after
  // A*x): Theta = A B has rank <= r, so the SVD is taken of the r x q matrix Theta' = R_A B with A = Q_A R_A (Householder):
  // same singular values, U = Q_A U'.  The Jacobi problem shrinks from min(p,q) to r columns, and it is full rank
  // (one-sided Jacobi needs 2-3x more sweeps on a matrix whose trailing singular values are rounding noise).
  const int kmin = std::min(p, q);
  const bool factored = (int64_t)r * 4 <= (int64_t)kmin * 3;
  const int pe = factored ? r : p;                   // rows of the matrix that is actually decomposed
  DevBuf Theta(sizeof(T) * (size_t)pe * q * batch), QA;
  if (!factored) {
    two_site_merge(x, k, Theta);
  } else {
    const int64_t bA = (int64_t)p * r;
    DevBuf RA(sizeof(T) * (size_t)r * r * batch);
    QA.alloc(sizeof(T) * (size_t)bA * batch);
    if (!cholqr2<T>(x.core(k), p, r, p, bA, RA.as<T>(), QA.as<T>(), p, bA, batch)) {
      DevBuf W(sizeof(T) * (size_t)bA * batch), tau(sizeof(T) * (size_t)r * batch);
      TTN_CUDA(cudaMemcpyAsync(W.p, x.cores[k].p, W.bytes, cudaMemcpyDeviceToDevice, ctx().stream));
      qr_factor<T>(W.as<T>(), p, r, p, tau.as<T>(), batch, bA, r);
      qr_form_q<T>(W.as<T>(), p, r, p, tau.as<T>(), QA.as<T>(), p, batch, bA, r, bA);
      Copy4 t; t.n0 = r; t.n1 = r; t.n2 = batch; t.s0 = 1; t.s1 = p; t.s2 = bA; t.d0 = 1; t.d1 = r; t.d2 = (int64_t)r * r; t.tri = 1;
      copy4<T>(W.as<T>(), RA.as<T>(), t);
    }
    GemmArgs g;  // Theta'[gamma',(s2,beta)] = sum_gamma R_A[gamma',gamma] B[s2,gamma,beta]
    g.M = r; g.N = rr; g.K = r;
    g.A = RA.p; g.sAm = 1; g.sAk = r; g.bA1 = 0; g.bA2 = (int64_t)r * r;
    g.B = x.cores[k + 1].p; g.sBk = n2; g.sBn = (int64_t)n2 * r; g.bB1 = 1; g.bB2 = x.core_elems(k + 1);
    g.C = Theta.p; g.sCm = 1; g.sCn = (int64_t)r * n2; g.bC1 = r; g.bC2 = (int64_t)r * q;
    g.batch1 = n2; g.batch2 = batch;
    gemm<T>(g);
  }
  SvdLeft sv;
  svd_left<T>(Theta.as<T>(), pe, q, 1, pe, false, sv, batch, (int64_t)pe * q);
  const int kk = sv.k;
  // rank rule on the min(p,q) singular values of Theta (the kmin - kk values the factored form does not compute are zero)
  int rn;
  if (batch == 1) {
    std::vector<double> sig(sv.sigma.begin(), sv.sigma.begin() + kk);
    sig.resize(kmin, 0.0);
    rn = rank_tailnorm(sig.data(), kmin, max_bond, truncerr);
  } else {
    rn = (int)std::min<int64_t>(kmin, max_bond);
  }
  if (rn < 1) rn = 1;
  const int rc = std::min(rn, kk);                   // columns that are actually computed; the rest (sigma = 0) stay zero
  if (sigma_out) {
    for (int64_t j = 0; j < sigma_cap; ++j) sigma_out[j] = j < rc ? sv.sigma[j] : 0.0;
  }
  // scales: core k <- U sqrt(S) = X_j sigma_j^{-1/2};  projection basis G2 = X_j sigma_j^{-3/2}  so that
  // core k+1 <- sqrt(S) Vt = S^{-1/2} U^H Theta = G2^H Theta                                   (tt_tools.jl:754-757)
  std::vector<double> s1((size_t)rc * batch), s2((size_t)rc * batch);
  std::vector<int> perm((size_t)rc * batch);
  for (int b = 0; b < batch; ++b) {
    const double smax = sv.sigma[(size_t)b * kk];
    for (int j = 0; j < rc; ++j) {
      const double s = sv.sigma[(size_t)b * kk + j];
      // X_j = u_j sigma_j: core k <- X_j sigma^{-1/2}, G2 <- X_j sigma^{-3/2}; formed as (1/sigma)(1/sqrt(sigma)) so that
      // sigma^{3/2} cannot underflow on small-norm trains, and gated on a finite result
      const double is = 1.0 / std::sqrt(s), s2v = (1.0 / s) * is;
      const bool ok = s > 1e-290 && s > smax * 1e-140 && std::isfinite(is) && std::isfinite(s2v);
      s1[(size_t)b * rc + j] = ok ? is : 0.0;
      s2[(size_t)b * rc + j] = ok ? s2v : 0.0;
      perm[(size_t)b * rc + j] = sv.perm[(size_t)b * kk + j];
    }
  }
  DevBuf dperm(sizeof(int) * perm.size()), ds1(sizeof(double) * s1.size()), ds2(sizeof(double) * s2.size());
  TTN_CUDA(cudaMemcpyAsync(dperm.p, perm.data(), dperm.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(ds1.p, s1.data(), ds1.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(ds2.p, s2.data(), ds2.bytes, cudaMemcpyHostToDevice, ctx().stream));

  NewBond nb = new_bond<T>(p, n2, rn, rr, batch, rc, false);
  DevBuf G2(sizeof(T) * (size_t)pe * rc * batch);
  if (!factored) {
    gather_cols<T>(sv.X.as<T>(), p, p, dperm.as<int>(), ds1.as<double>(), rc, nb.A.as<T>(), 1, p, batch, (int64_t)p * kk, rc,
                   (int64_t)p * rn);
  } else {
    DevBuf Us(sizeof(T) * (size_t)pe * rc * batch);   // U' sqrt(S)^{-1}-scaled columns of the small problem
    gather_cols<T>(sv.X.as<T>(), pe, pe, dperm.as<int>(), ds1.as<double>(), rc, Us.as<T>(), 1, pe, batch, (int64_t)pe * kk, rc,
                   (int64_t)pe * rc);
    GemmArgs g;  // core k <- Q_A (U' S^{-1/2} scaled)
    g.M = p; g.N = rc; g.K = pe;
    g.A = QA.p; g.sAm = 1; g.sAk = p; g.bA1 = (int64_t)p * r;
    g.B = Us.p; g.sBk = 1; g.sBn = pe; g.bB1 = (int64_t)pe * rc;
    g.C = nb.A.p; g.sCm = 1; g.sCn = p; g.bC1 = (int64_t)p * rn;
    g.batch1 = batch;
    gemm<T>(g);
  }
  gather_cols<T>(sv.X.as<T>(), pe, pe, dperm.as<int>(), ds2.as<double>(), rc, G2.as<T>(), 1, pe, batch, (int64_t)pe * kk, rc,
                 (int64_t)pe * rc);
  project<T>(G2, Theta, pe, rc, rn, n2, rr, batch, nb.B);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  std::swap(x.cores[k], nb.A);
  std::swap(x.cores[k + 1], nb.B);
  x.rks[k + 1] = rn;
  return {std::move(nb.A), std::move(nb.B)};
}

// ---------------------------------------------------------------------------------------------------------------------
// Gram path of tt_compress! for a pure rank cap (truncerr == 0): no host round trip inside the sweep.
//   L->R bond:  Theta = A B,  G = Theta Theta^H (split-K partials, summed by the eigensolver's loader),  G = U S^2 U^H
//               (heig.cu: tridiagonalisation + multisection + twisted factorisation),  core k <- U sqrt(S),
//               core k+1 <- S^{-1/2} U^H Theta.
//   R->L bond:  core k = U_k sqrt(S_k) was produced by the L->R step of the same bond and has orthogonal columns with known
//               squared norms w = S_k, so its QR factor is diag(sqrt(w)):  Theta' = sqrt(w) B (r x q),  G' = Theta' Theta'^H
//               = W S'^2 W^H,  core k <- A w^{-1/2} W sqrt(S'),  core k+1 <- S'^{-1/2} W^H Theta'.
// Every eigen-decomposition raises a per-train flag when the fast path cannot vouch for it (clustered or non-positive kept
// spectrum, sigma_r < 1e-5 sigma_1); the flags are read ONCE at the end of the call and a flagged call is redone from the
// preserved input cores by the QR + one-sided-Jacobi path.  Bonds the eigensolver does not serve (more than 128 / 176
// rows, tall Theta) take the classic step inside the same sweep.
// ---------------------------------------------------------------------------------------------------------------------
// Theta[row, i + n2 (b + Wr mu)] = sum_{a,j} A[i,j,a,b] Z[row, a + Wl j, mu]: the MPO core of site k+1 applied to
// Z = P x_{k+1} (the apply of src/tt_operations.jl:105-108 folded into the two-site merge of tt_tools.jl:749): the product
// core y_{k+1} (n2, Wl r, Wr r') is never written to HBM.  One CTA per (mu, train), one thread per row; A in shared memory.
template <class T>
__global__ void __launch_bounds__(256) kron_mix_kernel(const T* __restrict__ Z, const T* __restrict__ A, T* __restrict__ Th, int p,
                                                       int n2, int Wl, int Wr, int rp, int64_t bZ, int64_t bTh) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* As = reinterpret_cast<T*>(smem_raw);   // [ (i,b) ][ (a,j) ]
  const int KA = Wl * n2, KB = n2 * Wr;
  for (int t = threadIdx.x; t < KA * KB; t += blockDim.x) {
    const int aj = t % KA, ib = t / KA;
    const int a = aj % Wl, j = aj / Wl, i = ib % n2, b = ib / n2;
    As[t] = A[i + n2 * (j + n2 * (a + Wl * b))];
  }
  __syncthreads();
  const int mu = blockIdx.x;
  const T* Zb = Z + blockIdx.y * bZ + (int64_t)p * KA * mu;
  T* Tb = Th + blockIdx.y * bTh + (int64_t)p * KB * mu;
  for (int row = threadIdx.x; row < p; row += blockDim.x) {
    for (int ib = 0; ib < KB; ++ib) {
      T acc = t_zero<T>();
      const T* ar = As + ib * KA;
      for (int aj = 0; aj < KA; ++aj) t_fma(acc, ar[aj], Zb[row + (int64_t)p * aj]);
      Tb[row + (int64_t)p * ib] = acc;
    }
  }
  (void)rp;
}

// y = A * x not yet materialised beyond its first core: the L->R pass of the Gram sweep consumes (A_{k+1}, x_{k+1}) directly
template <class T>
struct LazyProd {
  const TTO<T>* A = nullptr;
  const TT<T>* x = nullptr;
  std::vector<char> virt;     // virt[k] != 0: core k of y is still the un-materialised product A_k (x) x_k
};

template <class T>
struct GramSweep {
  LazyProd<T>* lazy = nullptr;
  TT<T>& x;
  int64_t max_bond;
  DevBuf flags;                       // int per train, sticky
  std::vector<DevBuf> colw;           // colw[k]: squared column norms of core k (batch x r) while it is U sqrt(S) of bond k
  std::vector<DevBuf> orig;           // input cores (the first buffer replaced per site), alive until the flags are read
  std::vector<char> have_orig;
  DevBuf sigdev;                      // steps x stride singular values of train 0
  std::vector<int> gram_steps;
  int64_t sigma_stride = 0;

  GramSweep(TT<T>& x_, int64_t mb) : x(x_), max_bond(mb), colw(x_.d), orig(x_.d), have_orig(x_.d, 0) {
    flags.alloc(sizeof(int) * (size_t)x.batch);
    TTN_CUDA(cudaMemsetAsync(flags.p, 0, flags.bytes, ctx().stream));
  }
  // a buffer that has left site k: the first one is the input core and is kept for the rollback, later ones are released
  void retire(int k, DevBuf old) {
    if (!have_orig[k]) { orig[k] = std::move(old); have_orig[k] = 1; }
  }
  // the truncated bond replaces cores k and k+1 (no longer a pending product); nb.w, possibly empty, becomes colw[k]
  void install(int k, NewBond&& nb, int rn) {
    colw[k] = std::move(nb.w);
    std::swap(x.cores[k], nb.A);
    std::swap(x.cores[k + 1], nb.B);
    retire(k, std::move(nb.A));
    retire(k + 1, std::move(nb.B));
    if (lazy) lazy->virt[k + 1] = 0;
    x.rks[k + 1] = rn;
  }
  // split-K Gram matrix of Th (pe x q, ld pe, batch stride pe*q): partials [nsplit][batch][pe x pe]
  int gram(const T* Th, int pe, int q, DevBuf& Gp) {
    const int batch = x.batch;
    int nsplit = 1;
    if (batch * 4 < ctx().sm_count)
      while (nsplit < 16 && q % (nsplit * 2) == 0 && q / (nsplit * 2) >= 64 && batch * nsplit * 4 < ctx().sm_count) nsplit *= 2;
    const int kc = q / nsplit;
    Gp.alloc(sizeof(T) * (size_t)pe * pe * batch * nsplit);
    GemmArgs g;
    g.M = pe; g.N = pe; g.K = kc;
    g.A = Th; g.sAm = 1; g.sAk = pe; g.bA1 = (int64_t)pe * kc; g.bA2 = (int64_t)pe * q;
    g.B = Th; g.sBk = pe; g.sBn = 1; g.conjB = true; g.bB1 = (int64_t)pe * kc; g.bB2 = (int64_t)pe * q;
    g.C = Gp.p; g.sCm = 1; g.sCn = pe; g.bC1 = (int64_t)batch * pe * pe; g.bC2 = (int64_t)pe * pe;
    g.batch1 = nsplit; g.batch2 = batch;
    gemm<T>(g);
    return nsplit;
  }
  // G = V diag(lam) V^H of order n (the sum of nsplit partials sG apart): its top nev eigenpairs, then heig_finalize into out1 /
  // out2 (and the kept weights into w) with the sweep's flags and this step's sig0.  False when the shape is not served.
  bool eig_split(const DevBuf& G, int n, int nsplit, int64_t sG, int nev, const double* w_in, T* out1, int64_t ld1, int64_t b1,
                 T* out2, int64_t ld2, int64_t b2, double* w, int64_t bw, double* sig0) {
    const int batch = x.batch;
    DevBuf lam(sizeof(double) * (size_t)nev * batch), V(sizeof(T) * (size_t)n * nev * batch);
    if (!heig_top<T>(G.as<T>(), n, n, (int64_t)n * n, nsplit, sG, nev, batch, lam.as<double>(), V.as<T>(), flags.as<int>()))
      return false;
    heig_finalize<T>(V.as<T>(), n, nev, batch, lam.as<double>(), w_in, out1, ld1, b1, out2, ld2, b2, w, bw, sig0, flags.as<int>());
    return true;
  }
  void materialize(int k) {
    if (!lazy || !lazy->virt[k]) return;
    apply_site(*lazy->A, *lazy->x, x, k);
    lazy->virt[k] = 0;
  }
  // Theta (p x q) of bond (k, k+1) when core k+1 is still A_{k+1} (x) x_{k+1}:  Z = P x_{k+1} (GEMMs), then the MPO mix
  void theta_lazy(int k, DevBuf& Th) {
    const TTO<T>& A = *lazy->A;
    const TT<T>& v = *lazy->x;
    const int batch = x.batch;
    const int n1 = (int)x.dims[k], n2 = (int)x.dims[k + 1];
    const int p = n1 * (int)x.rks[k];
    const int Wl = (int)A.rks[k + 1], Wr = (int)A.rks[k + 2], r = (int)v.rks[k + 1], rp = (int)v.rks[k + 2];
    const int KA = Wl * n2, KB = n2 * Wr;
    DevBuf Z(sizeof(T) * (size_t)p * KA * rp * batch);
    for (int j = 0; j < n2; ++j) {
      // Z[(row,a), j, mu] = sum_nu P[(row,a), nu] x[j, nu, mu]: the fused left bond (a + Wl nu) of P makes (row, a) one
      // contiguous M index of length p*Wl, so the Wl products of a site are ONE GEMM (larger tiles than Wl small ones)
      GemmArgs g;
      g.M = p * Wl; g.N = rp; g.K = r;
      g.A = x.cores[k].p; g.sAm = 1; g.sAk = (int64_t)Wl * p; g.bA2 = x.core_elems(k);
      g.B = v.core(k + 1) + j; g.sBk = n2; g.sBn = (int64_t)n2 * r; g.bB2 = v.core_elems(k + 1);
      g.C = Z.as<T>() + (int64_t)p * Wl * j; g.sCm = 1; g.sCn = (int64_t)p * KA; g.bC2 = (int64_t)p * KA * rp;
      g.batch1 = 1; g.batch2 = batch;
      gemm<T>(g);
    }
    const int nt = std::min(256, ((p + 31) / 32) * 32);
    ProfScope prof_scope_(KF_APPLY);
    for (int b0 = 0; b0 < batch; b0 += 65535) {
      const int nb = std::min(65535, batch - b0);
      kron_mix_kernel<T><<<dim3(rp, nb), nt, sizeof(T) * (size_t)KA * KB, ctx().stream>>>(
          Z.as<T>() + (int64_t)b0 * p * KA * rp, A.core(k + 1), Th.as<T>() + (int64_t)b0 * p * KB * rp, p, n2, Wl, Wr, rp,
          (int64_t)p * KA * rp, (int64_t)p * KB * rp);
      TTN_CHECK_LAUNCH();
      ctx().launches++;
    }
  }
  // Theta (p x q) of bond (k, k+1), materialised or folded product
  void theta(int k, DevBuf& Th) {
    const int n2 = (int)x.dims[k + 1];
    if (lazy && lazy->virt[k + 1] && (size_t)lazy->A->rks[k + 1] * n2 * n2 * lazy->A->rks[k + 2] * sizeof(T) <= 40 * 1024) {
      theta_lazy(k, Th);           // core k+1 stays virtual until the truncated core replaces it
    } else {
      materialize(k + 1);
      two_site_merge(x, k, Th);
    }
  }
  // one bond step; returns false when the shape is not served (caller takes the classic step)
  bool step(int k, bool left_to_right, int64_t step_idx) {
    const int batch = x.batch;
    materialize(k);
    const int n1 = (int)x.dims[k], n2 = (int)x.dims[k + 1];
    const int rl = (int)x.rks[k], r = (int)x.rks[k + 1], rr = (int)x.rks[k + 2];
    const int p = n1 * rl, q = n2 * rr;
    const int rn = (int)std::min<int64_t>(std::min(p, q), max_bond), nev = std::min(rn, r);
    double* sig0 = sigdev.p ? sigdev.as<double>() + step_idx * sigma_stride : nullptr;
    if (rn < 1 || ((int64_t)nev > sigma_stride && sig0)) return false;
    if (!left_to_right && colw[k].p != nullptr && colw[k].bytes == sizeof(double) * (size_t)r * batch) {
      // R->L: G' = Theta' Theta'^H of Theta' = sqrt(w) B (r x q), the weights w of core k taken from its L->R step
      if (r > heig_max_n<T>() || r > q) return false;
      materialize(k + 1);
      DevBuf Th(sizeof(T) * (size_t)r * q * batch);
      Copy4 c;   // Th[gamma, s2 + n2*beta] = B[s2, gamma, beta]
      c.n0 = r; c.s0 = n2; c.d0 = 1;
      c.n1 = n2; c.s1 = 1; c.d1 = r;
      c.n2 = rr; c.s2 = (int64_t)n2 * r; c.d2 = (int64_t)r * n2;
      c.n3 = batch; c.s3 = x.core_elems(k + 1); c.d3 = (int64_t)r * q;
      copy4<T>(x.core(k + 1), Th.as<T>(), c);
      diag_scale<T>(Th.as<T>(), r, q, 1, r, colw[k].as<double>(), 1, 0, batch, (int64_t)r * q, r);
      DevBuf Gp;
      const int nsplit = gram(Th.as<T>(), r, q, Gp);
      DevBuf M1(sizeof(T) * (size_t)r * nev * batch), G2(sizeof(T) * (size_t)r * nev * batch);
      if (!eig_split(Gp, r, nsplit, (int64_t)batch * r * r, nev, colw[k].as<double>(), M1.as<T>(), r, (int64_t)r * nev, G2.as<T>(), r,
                     (int64_t)r * nev, nullptr, 0, sig0))
        return false;
      NewBond nb = new_bond<T>(p, n2, rn, rr, batch, nev, false);
      GemmArgs g;   // core k <- A M1
      g.M = p; g.N = nev; g.K = r;
      g.A = x.cores[k].p; g.sAm = 1; g.sAk = p; g.bA1 = x.core_elems(k);
      g.B = M1.p; g.sBk = 1; g.sBn = r; g.bB1 = (int64_t)r * nev;
      g.C = nb.A.p; g.sCm = 1; g.sCn = p; g.bC1 = (int64_t)p * rn;
      g.batch1 = batch;
      gemm<T>(g);
      project<T>(G2, Th, r, nev, rn, n2, rr, batch, nb.B);
      install(k, std::move(nb), rn);
      return true;
    }
    // L->R: Theta = A B and its Gram matrix of order min(p, q), Theta Theta^H (wide) or Theta^H Theta (tall)
    if (!left_to_right || std::min(p, q) > heig_max_n<T>()) return false;
    DevBuf Th(sizeof(T) * (size_t)p * q * batch);
    theta(k, Th);
    NewBond nb;
    if (p <= q) {
      DevBuf Gp;
      const int nsplit = gram(Th.as<T>(), p, q, Gp);
      nb = new_bond<T>(p, n2, rn, rr, batch, nev, true);
      DevBuf G2(sizeof(T) * (size_t)p * nev * batch);
      if (!eig_split(Gp, p, nsplit, (int64_t)batch * p * p, nev, nullptr, nb.A.as<T>(), p, (int64_t)p * rn, G2.as<T>(), p,
                     (int64_t)p * nev, nb.w.as<double>(), rn, sig0))
        return false;
      project<T>(G2, Th, p, nev, rn, n2, rr, batch, nb.B);
    } else {
      // a TALL bond (the last sites of a train): G = Theta^H Theta = V S^2 V^H (q x q), core k+1 <- sqrt(S) V^H,
      // core k <- Theta V S^{-1/2} = U sqrt(S)
      DevBuf Gp(sizeof(T) * (size_t)q * q * batch);
      {
        GemmArgs g;   // G[c, c'] = sum_row conj(Theta[row, c]) Theta[row, c']
        g.M = q; g.N = q; g.K = p;
        g.A = Th.p; g.sAm = p; g.sAk = 1; g.conjA = true; g.bA1 = (int64_t)p * q;
        g.B = Th.p; g.sBk = 1; g.sBn = p; g.bB1 = (int64_t)p * q;
        g.C = Gp.p; g.sCm = 1; g.sCn = q; g.bC1 = (int64_t)q * q;
        g.batch1 = batch;
        gemm<T>(g);
      }
      nb = new_bond<T>(p, n2, rn, rr, batch, nev, true);
      DevBuf Vs(sizeof(T) * (size_t)q * nev * batch), Vi(sizeof(T) * (size_t)q * nev * batch);
      if (!eig_split(Gp, q, 1, 0, nev, nullptr, Vs.as<T>(), q, (int64_t)q * nev, Vi.as<T>(), q, (int64_t)q * nev, nb.w.as<double>(), rn,
                     sig0))
        return false;
      Copy4 c;   // newB[s2, kappa, beta] = conj(Vs[(s2, beta), kappa])
      c.n0 = n2; c.s0 = 1; c.d0 = 1;
      c.n1 = nev; c.s1 = q; c.d1 = n2;
      c.n2 = rr; c.s2 = n2; c.d2 = (int64_t)n2 * rn;
      c.n3 = batch; c.s3 = (int64_t)q * nev; c.d3 = (int64_t)n2 * rn * rr;
      c.conj = true;
      copy4<T>(Vs.as<T>(), nb.B.as<T>(), c);
      GemmArgs g;   // core k <- Theta (V S^{-1/2})
      g.M = p; g.N = nev; g.K = q;
      g.A = Th.p; g.sAm = 1; g.sAk = p; g.bA1 = (int64_t)p * q;
      g.B = Vi.p; g.sBk = 1; g.sBn = q; g.bB1 = (int64_t)q * nev;
      g.C = nb.A.p; g.sCm = 1; g.sCn = p; g.bC1 = (int64_t)p * rn;
      g.batch1 = batch;
      gemm<T>(g);
    }
    install(k, std::move(nb), rn);
    return true;
  }
};

// calls step(k, left_to_right, i) for every bond step of `sweeps` sweeps, each bonds k = 1..d-1 (1-based) L->R and then R->L;
// i numbers the steps from 0 (the row of sigma_out)
static void for_each_bond_step(int d, int sweeps, const std::function<void(int, bool, int64_t)>& step) {
  int64_t i = 0;
  for (int sw = 0; sw < sweeps; ++sw) {
    for (int k = 1; k <= d - 1; ++k) step(k, true, i++);
    for (int k = d - 1; k >= 1; --k) step(k, false, i++);
  }
}

// the Gram path serves a pure rank cap (truncerr == 0) of a train with at least one bond
static bool gram_path_applies(int d, int64_t max_bond, double truncerr) {
  return ctx().gram_compress && truncerr == 0.0 && d >= 2 && max_bond >= 1;
}

// returns false (x restored to its input) when some eigen-decomposition declined; true when the sweep stands
template <class T>
bool tt_compress_gram(TT<T>& x, int64_t max_bond, int sweeps, double* sigma_out, int64_t sigma_stride, LazyProd<T>* lazy = nullptr) {
  const std::vector<int64_t> rks0 = x.rks;
  GramSweep<T> gs(x, max_bond);
  gs.lazy = lazy;
  const int64_t nsteps = (int64_t)sweeps * 2 * (x.d - 1);
  gs.sigma_stride = sigma_stride;
  if (sigma_out && sigma_stride > 0) {
    gs.sigdev.alloc(sizeof(double) * (size_t)nsteps * sigma_stride);
    TTN_CUDA(cudaMemsetAsync(gs.sigdev.p, 0, gs.sigdev.bytes, ctx().stream));
  }
  int ngram = 0;
  bool threw = false;   // a classic step that is fed the output of a declined Gram step may meet non-finite data
  const bool dbg = debug_svd();
  int dbg_prev = 0;
  for_each_bond_step(x.d, sweeps, [&](int k1, bool l2r, int64_t step) {
    if (threw) return;
    if (gs.step(k1 - 1, l2r, step)) {
      gs.gram_steps.push_back((int)step); ++ngram;
      if (dbg) {   // debugging only: a flag read per step shows which bond declined
        std::vector<int> f(x.batch);
        read_back(f.data(), gs.flags.p, gs.flags.bytes);
        int a = 0;
        for (int v : f) a |= v;
        if (a != dbg_prev) {
          fprintf(stderr, "[ttn] gram step %lld bond %d %s ranks (%lld,%lld,%lld): flags 0x%x\n", (long long)step, k1, l2r ? "L->R" : "R->L",
                  (long long)x.rks[k1 - 1], (long long)x.rks[k1], (long long)x.rks[k1 + 1], a);
          dbg_prev = a;
        }
      }
    }
    else {
      gs.colw[k1 - 1].release();
      gs.materialize(k1 - 1);
      gs.materialize(k1);
      try {
        auto old = tt_bond_truncate<T>(x, k1, max_bond, 0.0, sigma_out ? sigma_out + step * sigma_stride : nullptr, sigma_stride);
        gs.retire(k1 - 1, std::move(old.first));
        gs.retire(k1, std::move(old.second));
      } catch (const Error&) {
        if (ngram == 0) throw;        // no Gram step before it: the error is the input's
        threw = true;
      }
    }
  });
  if (ngram == 0) return true;    // every bond took the classic step: nothing to verify
  ctx().gram_calls++;
  std::vector<int> hf(x.batch);
  std::vector<double> hs;
  {   // one read per call, through the context's pinned staging area (a pageable destination serialises in the driver)
    const size_t fb = (gs.flags.bytes + 15) & ~(size_t)15;
    const size_t sb = gs.sigdev.p ? gs.sigdev.bytes : 0;
    char* st = (char*)host_stage(fb + sb);
    TTN_CUDA(cudaMemcpyAsync(st, gs.flags.p, gs.flags.bytes, cudaMemcpyDeviceToHost, ctx().stream));
    if (sb) TTN_CUDA(cudaMemcpyAsync(st + fb, gs.sigdev.p, sb, cudaMemcpyDeviceToHost, ctx().stream));
    TTN_CUDA(cudaStreamSynchronize(ctx().stream));
    memcpy(hf.data(), st, sizeof(int) * hf.size());
    if (sb) {
      hs.resize((size_t)nsteps * sigma_stride);
      memcpy(hs.data(), st + fb, sb);
    }
  }
  int any = threw ? 32 : 0;
  for (int f : hf) any |= f;
  ctx().gram_last_flags = any;
  if (any) {
    ctx().gram_fallbacks++;
    if (debug_svd()) fprintf(stderr, "[ttn] tt_compress: Gram path declined (flags 0x%x), redoing with the Jacobi path\n", any);
    for (int k = 0; k < x.d; ++k)
      if (gs.have_orig[k]) x.cores[k] = std::move(gs.orig[k]);
    x.rks = rks0;
    return false;
  }
  if (sigma_out)
    for (int st : gs.gram_steps)
      std::memcpy(sigma_out + (int64_t)st * sigma_stride, hs.data() + (size_t)st * sigma_stride, sizeof(double) * sigma_stride);
  return true;
}

// the plain sweeps of tt_compress!: one Jacobi-SVD bond truncation per step
template <class T>
void tt_compress_classic(TT<T>& x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride) {
  for_each_bond_step(x.d, sweeps, [&](int k, bool, int64_t step) {
    tt_bond_truncate<T>(x, k, max_bond, truncerr, sigma_out ? sigma_out + step * sigma_stride : nullptr, sigma_stride);
  });
}

// src/tt_tools.jl:772-789
template <class T>
void tt_compress(TT<T>& x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride) {
  ttn_assert(sweeps >= 1, 2, "sweeps must be >= 1");
  if (gram_path_applies(x.d, max_bond, truncerr) && tt_compress_gram<T>(x, max_bond, sweeps, sigma_out, sigma_stride)) return;
  tt_compress_classic<T>(x, max_bond, truncerr, sweeps, sigma_out, sigma_stride);
}

// y = tt_compress!(A * x, max_bond; truncerr, sweeps)  (src/tt_operations.jl:101-111 followed by tt_tools.jl:772-789).
// With truncerr == 0 the product cores are consumed by the L->R pass of the Gram sweep without ever being written to HBM
// (cfg5: 40.5 MB per vector); otherwise, or when the fast path declines, it is tt_apply followed by the plain sweeps.
template <class T>
void tt_apply_compress(const TTO<T>& A, const TT<T>& x, TT<T>& y, int64_t max_bond, double truncerr, int sweeps, double* sigma_out,
                       int64_t sigma_stride) {
  ttn_assert(A.d == x.d && A.dims == x.dims, 1, "Incompatible dimensions");
  ttn_assert(sweeps >= 1, 2, "sweeps must be >= 1");
  if (gram_path_applies(x.d, max_bond, truncerr)) {
    product_shape(A, x, y);
    LazyProd<T> lazy;
    lazy.A = &A; lazy.x = &x;
    lazy.virt.assign(x.d, 1);
    if (tt_compress_gram<T>(y, max_bond, sweeps, sigma_out, sigma_stride, &lazy)) {
      bool left = false;
      for (char v : lazy.virt) left |= (v != 0);
      ttn_assert(!left, 7, "apply_compress: a product core was never materialised");
      return;
    }
  }
  tt_apply<T>(A, x, y);
  tt_compress_classic<T>(y, max_bond, truncerr, sweeps, sigma_out, sigma_stride);   // the Gram path has declined or does not apply
}

#define INST(T)                                                                                   \
  template void tt_apply_compress<T>(const TTO<T>&, const TT<T>&, TT<T>&, int64_t, double, int, double*, int64_t); \
  template void tt_copy<T>(const TT<T>&, TT<T>&);                                                 \
  template void tt_apply<T>(const TTO<T>&, const TT<T>&, TT<T>&);                                 \
  template void tt_dot<T>(const TT<T>&, const TT<T>&, std::vector<T>&);                           \
  template void tt_add<T>(const TT<T>&, const TT<T>&, TT<T>&);                                    \
  template void tt_scale<T>(const TT<T>&, T, TT<T>&);                                             \
  template void tt_orthogonalize<T>(const TT<T>&, int, TT<T>&);                                   \
  template std::pair<DevBuf, DevBuf> tt_bond_truncate<T>(TT<T>&, int, int64_t, double, double*, int64_t);   \
  template void tt_compress<T>(TT<T>&, int64_t, double, int, double*, int64_t);
INST(double)
INST(zc)
#undef INST

}  // namespace ttn
