// Effective operator of a window, environment updates and MPO fusion (kernel families F1/F2/F7).
//
// Reference compute sites replaced here:
//   matvec      src/solvers/dmrg.jl:239-244 (K_matfree), :99-168 (the scalar-loop matvec of Ksolve!),
//               als.jl:78, mals.jl:193-198, tdvp.jl:29-35,205-208 (_applyH1_lsr/_applyH0/_applyH2_lsr)
//   env updates src/solvers/dmrg.jl:27-35,73-81; als.jl:23-55; mals.jl:10-13,60-66; tdvp.jl:37-43
//   MPO fusion  src/solvers/dmrg.jl:38-46 (Amid)
// The contraction order is the optimal three-GEMM chain T1 = L·V, T2 = W·T1, Y = T2·R (SURVEY.md §8(d):
// 4·w·n²·chi³ + 2·w²·n⁴·chi² flops for the two-site window); all three run on the DMMA GEMM of gemm.cu and the
// intermediates T1/T2 stay in HBM/L2 between them.  The dense assemblies K_full of the reference
// (als.jl:58-63, mals.jl:148-157, dmrg.jl:49-54) are never formed.
#include <memory>
#include "solvers.h"

namespace ttn {

template <class T>
void LocalOp<T>::setup(const T* Lenv, int chil, int wl, const T* Renv, int chir, int wr, const T* Wfused, int nn_, bool sym) {
  chi_l = chil; w_l = wl; chi_r = chir; w_r = wr; nn = nn_;
  zero_site = (Wfused == nullptr);
  symmetrize = sym;
  L = Lenv;
  if (zero_site) ttn_assert(wl == wr && nn_ == 1, 7, "zero-site operator needs matching MPO bonds");
  Rm.alloc(sizeof(T) * (size_t)w_r * chi_r * chi_r);
  {
    Copy4 c;  // Rm[(z,f),c] = R[c,z,f]
    c.n0 = chi_r; c.s0 = 1; c.d0 = (int64_t)w_r * chi_r;
    c.n1 = w_r; c.s1 = chi_r; c.d1 = 1;
    c.n2 = chi_r; c.s2 = (int64_t)chi_r * w_r; c.d2 = w_r;
    copy4<T>(Renv, Rm.as<T>(), c);
  }
  if (!zero_site) {
    Wp.alloc(sizeof(T) * (size_t)w_l * nn * nn * w_r);
    Copy4 c;  // Wp[(y,e),(b,z)] = W[y,b,e,z]
    c.n0 = w_l; c.s0 = 1; c.d0 = 1;
    c.n1 = nn; c.s1 = w_l; c.d1 = (int64_t)w_l * nn;
    c.n2 = nn; c.s2 = (int64_t)w_l * nn; c.d2 = w_l;
    c.n3 = w_r; c.s3 = (int64_t)w_l * nn * nn; c.d3 = (int64_t)w_l * nn * nn;
    copy4<T>(Wfused, Wp.as<T>(), c);
  }
  if (symmetrize) {
    Lt.alloc(sizeof(T) * (size_t)chi_l * w_l * chi_l);
    {
      Copy4 c;  // Lt[a,y,d] = L[d,y,a]
      c.n0 = chi_l; c.s0 = (int64_t)chi_l * w_l; c.d0 = 1;
      c.n1 = w_l; c.s1 = chi_l; c.d1 = chi_l;
      c.n2 = chi_l; c.s2 = 1; c.d2 = (int64_t)chi_l * w_l;
      copy4<T>(Lenv, Lt.as<T>(), c);
    }
    Rmt.alloc(sizeof(T) * (size_t)w_r * chi_r * chi_r);
    {
      Copy4 c;  // Rmt[(z,f),c] = R[f,z,c]
      c.n0 = w_r; c.s0 = chi_r; c.d0 = 1;
      c.n1 = chi_r; c.s1 = 1; c.d1 = w_r;
      c.n2 = chi_r; c.s2 = (int64_t)chi_r * w_r; c.d2 = (int64_t)w_r * chi_r;
      copy4<T>(Renv, Rmt.as<T>(), c);
    }
    if (!zero_site) {
      Wpt.alloc(sizeof(T) * (size_t)w_l * nn * nn * w_r);
      Copy4 c;  // Wpt[(y,e),(b,z)] = W[y,e,b,z]
      c.n0 = w_l; c.s0 = 1; c.d0 = 1;
      c.n1 = nn; c.s1 = (int64_t)w_l * nn; c.d1 = (int64_t)w_l * nn;
      c.n2 = nn; c.s2 = w_l; c.d2 = w_l;
      c.n3 = w_r; c.s3 = (int64_t)w_l * nn * nn; c.d3 = (int64_t)w_l * nn * nn;
      copy4<T>(Wfused, Wpt.as<T>(), c);
    }
  }
  T1.alloc(sizeof(T) * (size_t)chi_l * w_l * nn * chi_r);
  if (!zero_site) T2.alloc(sizeof(T) * (size_t)chi_l * nn * w_r * chi_r);
}

// One pass of the three-GEMM chain on `nvec` window vectors stored back to back (V, Y: (chi_l, nn, chi_r, nvec)).
template <class T>
static void localop_pass(LocalOp<T>& op, const T* Lx, const T* Wx, const T* Rx, const T* V, T* Y, double alpha, double beta,
                         int nvec, T* T1, T* T2) {
  const int cl = op.chi_l, cr = op.chi_r, wl = op.w_l, wr = op.w_r, nn = op.nn;
  {
    GemmArgs g;  // T1[(a,y),(e,f,j)] = L[(a,y),d] V[d,(e,f,j)]
    g.M = cl * wl; g.N = nn * cr * nvec; g.K = cl;
    g.A = Lx; g.sAm = 1; g.sAk = (int64_t)cl * wl;
    g.B = V; g.sBk = 1; g.sBn = cl;
    g.C = T1; g.sCm = 1; g.sCn = (int64_t)cl * wl;
    gemm<T>(g);
  }
  if (op.zero_site) {
    GemmArgs g;  // Y[a,c,j] = T1[a,(y,f),j] R[(y,f),c]
    g.M = cl; g.N = cr; g.K = wr * cr;
    g.A = T1; g.sAm = 1; g.sAk = cl; g.bA1 = (int64_t)cl * wl * cr;
    g.B = Rx; g.sBk = 1; g.sBn = (int64_t)wr * cr;
    g.C = Y; g.sCm = 1; g.sCn = cl; g.bC1 = (int64_t)cl * cr; g.alpha = alpha; g.beta = beta;
    g.batch1 = nvec;
    gemm<T>(g);
    return;
  }
  {
    GemmArgs g;  // T2[a,(b,z),(f,j)] = T1[a,(y,e),(f,j)] W'[(y,e),(b,z)]   (batch over (f,j))
    g.M = cl; g.N = nn * wr; g.K = wl * nn;
    g.A = T1; g.sAm = 1; g.sAk = cl; g.bA1 = (int64_t)cl * wl * nn;
    g.B = Wx; g.sBk = 1; g.sBn = (int64_t)wl * nn; g.bB1 = 0;
    g.C = T2; g.sCm = 1; g.sCn = cl; g.bC1 = (int64_t)cl * nn * wr;
    const int64_t nb = (int64_t)cr * nvec;
    if (nb <= 65535) { g.batch1 = (int)nb; }
    else { g.batch1 = cr; g.batch2 = nvec; g.bA2 = g.bA1 * cr; g.bC2 = g.bC1 * cr; }
    gemm<T>(g);
  }
  {
    GemmArgs g;  // Y[(a,b),c,j] = T2[(a,b),(z,f),j] R[(z,f),c]
    g.M = cl * nn; g.N = cr; g.K = wr * cr;
    g.A = T2; g.sAm = 1; g.sAk = (int64_t)cl * nn; g.bA1 = (int64_t)cl * nn * wr * cr;
    g.B = Rx; g.sBk = 1; g.sBn = (int64_t)wr * cr;
    g.C = Y; g.sCm = 1; g.sCn = (int64_t)cl * nn; g.bC1 = (int64_t)cl * nn * cr; g.alpha = alpha; g.beta = beta;
    g.batch1 = nvec;
    gemm<T>(g);
  }
}

template <class T>
void LocalOp<T>::apply(const T* V, T* Y) {
  if (ext_apply) { ext_apply(V, Y); return; }
  apply_batch(V, Y, 1);
}

template <class T>
void LocalOp<T>::apply_batch(const T* V, T* Y, int nvec) {
  ttn_assert(!ext_apply, 7, "apply_batch: not available for an external operator");
  DevBuf B1, B2;
  T* t1 = T1.as<T>();
  T* t2 = T2.as<T>();
  if (nvec > 1) {   // the resident workspaces hold one vector
    B1.alloc(sizeof(T) * (size_t)chi_l * w_l * nn * chi_r * nvec);
    if (!zero_site) B2.alloc(sizeof(T) * (size_t)chi_l * nn * w_r * chi_r * nvec);
    t1 = B1.as<T>(); t2 = B2.as<T>();
  }
  if (symmetrize) {
    localop_pass<T>(*this, L, Wp.as<T>(), Rm.as<T>(), V, Y, 0.5, 0.0, nvec, t1, t2);
    localop_pass<T>(*this, Lt.as<T>(), Wpt.as<T>(), Rmt.as<T>(), V, Y, 0.5, 1.0, nvec, t1, t2);
  } else {
    localop_pass<T>(*this, L, Wp.as<T>(), Rm.as<T>(), V, Y, 1.0, 0.0, nvec, t1, t2);
  }
}

template <class T>
double LocalOp<T>::flops() const {
  const double c = is_cplx<T>::value ? 4.0 : 1.0;
  double f = 2.0 * chi_l * w_l * (double)chi_l * nn * chi_r;
  if (zero_site) f += 2.0 * chi_l * (double)w_r * chi_r * chi_r;
  else f += 2.0 * chi_l * (double)(w_l * nn) * (nn * w_r) * chi_r + 2.0 * chi_l * nn * (double)w_r * chi_r * chi_r;
  return c * f * (symmetrize ? 2.0 : 1.0);
}

template <class T>
void env_update(bool left, const T* Ein, int chi_in, int w_in, const T* x, int n, int rl, int rr, const T* A, int Rl, int Rr,
                DevBuf& Eout) {
  const int chi_out = left ? rr : rl, w_out = left ? Rr : Rl;
  ttn_assert(chi_in == (left ? rl : rr) && w_in == (left ? Rl : Rr), 7, "env_update: shape mismatch");
  const int64_t si = left ? n : (int64_t)n * rl, so = left ? (int64_t)n * rl : n;
  DevBuf W2(sizeof(T) * (size_t)w_in * n * n * w_out);
  {
    Copy4 c;  // left: W2[(y,k),(j,z)] = A[j,k,y,z];  right: W2[(z,k),(j,y)] = A[j,k,y,z]
    c.n0 = n; c.s0 = 1; c.d0 = (int64_t)w_in * n;                                  // j
    c.n1 = n; c.s1 = n; c.d1 = w_in;                                               // k
    c.n2 = Rl; c.s2 = (int64_t)n * n; c.d2 = left ? 1 : (int64_t)w_in * n * n;     // y
    c.n3 = Rr; c.s3 = (int64_t)n * n * Rl; c.d3 = left ? (int64_t)w_in * n * n : 1;  // z
    copy4<T>(A, W2.as<T>(), c);
  }
  DevBuf T1(sizeof(T) * (size_t)chi_in * w_in * n * chi_out), T2(sizeof(T) * (size_t)chi_in * n * w_out * chi_out);
  {
    GemmArgs g;  // T1[(a,y),k,d'] = E[(a,y),d] x[k,d,d']   (batch over k)
    g.M = chi_in * w_in; g.N = chi_out; g.K = chi_in;
    g.A = Ein; g.sAm = 1; g.sAk = (int64_t)chi_in * w_in;
    g.B = x; g.sBk = si; g.sBn = so; g.bB1 = 1;
    g.C = T1.p; g.sCm = 1; g.sCn = (int64_t)chi_in * w_in * n; g.bC1 = (int64_t)chi_in * w_in;
    g.batch1 = n;
    gemm<T>(g);
  }
  {
    GemmArgs g;  // T2[a,(j,z),d'] = T1[a,(y,k),d'] W2[(y,k),(j,z)]   (batch over d')
    g.M = chi_in; g.N = n * w_out; g.K = w_in * n;
    g.A = T1.p; g.sAm = 1; g.sAk = chi_in; g.bA1 = (int64_t)chi_in * w_in * n;
    g.B = W2.p; g.sBk = 1; g.sBn = (int64_t)w_in * n;
    g.C = T2.p; g.sCm = 1; g.sCn = chi_in; g.bC1 = (int64_t)chi_in * n * w_out;
    g.batch1 = chi_out;
    gemm<T>(g);
  }
  Eout.alloc(sizeof(T) * (size_t)chi_out * w_out * chi_out);
  for (int j = 0; j < n; ++j) {
    GemmArgs g;  // E'[a',(z,d')] += conj(x[j,a,a'])^T T2[a,j,(z,d')]
    g.M = chi_out; g.N = w_out * chi_out; g.K = chi_in;
    g.A = x + j; g.sAm = so; g.sAk = si; g.conjA = true;
    g.B = T2.as<T>() + (int64_t)chi_in * j; g.sBk = 1; g.sBn = (int64_t)chi_in * n;
    g.C = Eout.p; g.sCm = 1; g.sCn = chi_out; g.beta = j > 0 ? 1.0 : 0.0;
    gemm<T>(g);
  }
}

template <class T>
void envb_update(bool left, const T* Bin, int chi_in, int rb_in, const T* x, int n, int rl, int rr, const T* b, int bl, int br,
                 DevBuf& Bout) {
  const int chi_out = left ? rr : rl, rb_out = left ? br : bl;
  ttn_assert(chi_in == (left ? rl : rr) && rb_in == (left ? bl : br), 7, "envb_update: shape mismatch");
  const int64_t si = left ? n : (int64_t)n * rl, so = left ? (int64_t)n * rl : n;
  const int64_t sib = left ? n : (int64_t)n * bl, sob = left ? (int64_t)n * bl : n;
  DevBuf T1(sizeof(T) * (size_t)chi_in * n * rb_out);
  {
    GemmArgs g;  // T1[a,j,beta'] = Bin[a,beta] b[j,beta,beta']   (batch over j)
    g.M = chi_in; g.N = rb_out; g.K = rb_in;
    g.A = Bin; g.sAm = 1; g.sAk = chi_in;
    g.B = b; g.sBk = sib; g.sBn = sob; g.bB1 = 1;
    g.C = T1.p; g.sCm = 1; g.sCn = (int64_t)chi_in * n; g.bC1 = chi_in;
    g.batch1 = n;
    gemm<T>(g);
  }
  Bout.alloc(sizeof(T) * (size_t)chi_out * rb_out);
  for (int j = 0; j < n; ++j) {
    GemmArgs g;
    g.M = chi_out; g.N = rb_out; g.K = chi_in;
    g.A = x + j; g.sAm = so; g.sAk = si; g.conjA = true;
    g.B = T1.as<T>() + (int64_t)chi_in * j; g.sBk = 1; g.sBn = (int64_t)chi_in * n;
    g.C = Bout.p; g.sCm = 1; g.sCn = chi_out; g.beta = j > 0 ? 1.0 : 0.0;
    gemm<T>(g);
  }
}

template <class T>
void fuse_mpo(const TTO<T>& A, int i, int N, DevBuf& W, int& nn) {
  ttn_assert(N == 1 || N == 2, 2, "window size N must be 1 or 2");
  const int n1 = (int)A.dims[i], Rl = (int)A.rks[i], Rm = (int)A.rks[i + 1];
  if (N == 1) {
    nn = n1;
    W.alloc(sizeof(T) * (size_t)Rl * n1 * n1 * Rm);
    Copy4 c;  // W[y,b,e,z] = A[b,e,y,z]
    c.n0 = Rl; c.s0 = (int64_t)n1 * n1; c.d0 = 1;
    c.n1 = n1; c.s1 = 1; c.d1 = Rl;
    c.n2 = n1; c.s2 = n1; c.d2 = (int64_t)Rl * n1;
    c.n3 = Rm; c.s3 = (int64_t)n1 * n1 * Rl; c.d3 = (int64_t)Rl * n1 * n1;
    copy4<T>(A.core(i), W.as<T>(), c);
    return;
  }
  const int n2 = (int)A.dims[i + 1], Rr = (int)A.rks[i + 2];
  nn = n1 * n2;
  // Wt[(b1,e1,y),(b2,e2),z] = sum_xi A_i[(b1,e1,y),xi] A_{i+1}[(b2,e2),xi,z]   (batch over z)
  const int64_t rows = (int64_t)n1 * n1 * Rl, cols = (int64_t)n2 * n2;
  DevBuf Wt(sizeof(T) * (size_t)rows * cols * Rr);
  GemmArgs g;
  g.M = (int)rows; g.N = (int)cols; g.K = Rm;
  g.A = A.core(i); g.sAm = 1; g.sAk = rows;
  g.B = A.core(i + 1); g.sBk = cols; g.sBn = 1; g.bB1 = cols * Rm;
  g.C = Wt.p; g.sCm = 1; g.sCn = rows; g.bC1 = rows * cols;
  g.batch1 = Rr;
  gemm<T>(g);
  W.alloc(sizeof(T) * (size_t)Rl * nn * nn * Rr);
  // W[y,b1,b2,e1,e2,z]  <-  Wt[b1,e1,y,b2,e2,z]; one 4-d copy per b2
  for (int b2 = 0; b2 < n2; ++b2) {
    Copy4 c;
    c.n0 = n1; c.s0 = 1; c.d0 = Rl;                                                   // b1
    c.n1 = n1; c.s1 = n1; c.d1 = (int64_t)Rl * n1 * n2;                                // e1
    c.n2 = Rl; c.s2 = (int64_t)n1 * n1; c.d2 = 1;                                      // y
    c.n3 = (int64_t)n2 * Rr; c.s3 = rows * n2; c.d3 = (int64_t)Rl * n1 * n2 * n1;      // (e2,z)
    copy4<T>(Wt.as<T>() + rows * b2, W.as<T>() + (int64_t)Rl * n1 * b2, c);
  }
}

// reference layout [mpo, bra, ket] <-> canonical [bra, mpo, ket]
template <class T>
static void env_ref_to_canon(const T* src, T* dst, int w, int chi, bool inverse) {
  Copy4 c;
  c.n0 = w; c.n1 = chi; c.n2 = chi;
  if (!inverse) { c.s0 = 1; c.s1 = w; c.s2 = (int64_t)w * chi; c.d0 = chi; c.d1 = 1; c.d2 = (int64_t)w * chi; }
  else { c.s0 = chi; c.s1 = 1; c.s2 = (int64_t)w * chi; c.d0 = 1; c.d1 = w; c.d2 = (int64_t)w * chi; }
  copy4<T>(src, dst, c);
}

template <class T>
static void setup_from_host(LocalOp<T>& op, DevBuf& L, DevBuf& R, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G,
                            const void* Amid, const void* H, bool symmetrize) {
  const size_t nl = (size_t)w_l * chi_l * chi_l, nr = (size_t)w_r * chi_r * chi_r, nw = (size_t)w_l * nn * nn * w_r;
  DevBuf Gd(sizeof(T) * nl), Hd(sizeof(T) * nr), Wd(sizeof(T) * nw);
  TTN_CUDA(cudaMemcpyAsync(Gd.p, G, Gd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(Hd.p, H, Hd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(Wd.p, Amid, Wd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  L.alloc(sizeof(T) * nl);
  R.alloc(sizeof(T) * nr);
  env_ref_to_canon<T>(Gd.as<T>(), L.as<T>(), w_l, chi_l, false);
  env_ref_to_canon<T>(Hd.as<T>(), R.as<T>(), w_r, chi_r, false);
  op.setup(L.as<T>(), chi_l, w_l, R.as<T>(), chi_r, w_r, Wd.as<T>(), nn, symmetrize);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}

template <class T>
void matvec2_host(int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid, const void* H, const void* V,
                  void* Y, bool symmetrize) {
  LocalOp<T> op;
  DevBuf L, R;
  setup_from_host<T>(op, L, R, w_l, w_r, chi_l, chi_r, nn, G, Amid, H, symmetrize);
  DevBuf Vd(sizeof(T) * (size_t)op.size()), Yd(sizeof(T) * (size_t)op.size());
  TTN_CUDA(cudaMemcpyAsync(Vd.p, V, Vd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  op.apply(Vd.as<T>(), Yd.as<T>());
  read_back(Y, Yd.p, Yd.bytes);
}

template <class T>
void env_host(bool left, int n, int w_l, int w_r, int r_l, int r_r, const void* E, const void* x, const void* A, void* Eout) {
  const int chi_in = left ? r_l : r_r, w_in = left ? w_l : w_r, chi_out = left ? r_r : r_l, w_out = left ? w_r : w_l;
  DevBuf Ed(sizeof(T) * (size_t)w_in * chi_in * chi_in), Ec(sizeof(T) * (size_t)w_in * chi_in * chi_in);
  DevBuf xd(sizeof(T) * (size_t)n * r_l * r_r), Ad(sizeof(T) * (size_t)n * n * w_l * w_r);
  TTN_CUDA(cudaMemcpyAsync(Ed.p, E, Ed.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(xd.p, x, xd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(Ad.p, A, Ad.bytes, cudaMemcpyHostToDevice, ctx().stream));
  env_ref_to_canon<T>(Ed.as<T>(), Ec.as<T>(), w_in, chi_in, false);
  DevBuf Eo;
  env_update<T>(left, Ec.as<T>(), chi_in, w_in, xd.as<T>(), n, r_l, r_r, Ad.as<T>(), w_l, w_r, Eo);
  DevBuf Er(sizeof(T) * (size_t)w_out * chi_out * chi_out);
  env_ref_to_canon<T>(Eo.as<T>(), Er.as<T>(), w_out, chi_out, true);
  read_back(Eout, Er.p, Er.bytes);
}

ttn_matvec matvec2_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                          const void* H) {
  auto mv = std::make_unique<ttn_matvec_s>();
  mv->dtype = dtype;
  mv->visit([&](auto& op) { setup_from_host(op, mv->L, mv->R, w_l, w_r, chi_l, chi_r, nn, G, Amid, H, false); });
  return mv.release();
}
void matvec2_apply(ttn_matvec mv, const void* V, void* Y) {
  ttn_assert(mv != nullptr, 2, "null matvec handle");
  with_dtype(mv->dtype, [&](auto t) {
    using T = decltype(t);
    mv->as<T>().apply((const T*)V, (T*)Y);
  });
}

#define INST(T)                                                                                                          \
  template struct LocalOp<T>;                                                                                            \
  template void env_update<T>(bool, const T*, int, int, const T*, int, int, int, const T*, int, int, DevBuf&);           \
  template void envb_update<T>(bool, const T*, int, int, const T*, int, int, int, const T*, int, int, DevBuf&);          \
  template void fuse_mpo<T>(const TTO<T>&, int, int, DevBuf&, int&);                                                     \
  template void matvec2_host<T>(int, int, int, int, int, const void*, const void*, const void*, const void*, void*, bool); \
  template void env_host<T>(bool, int, int, int, int, int, const void*, const void*, const void*, void*);
INST(double)
INST(zc)
#undef INST

}  // namespace ttn
