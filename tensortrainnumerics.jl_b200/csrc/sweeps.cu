// ALS / MALS / DMRG / TDVP sweep drivers on device-resident trains.
//
// One engine serves the four solver families of the reference: the train `x`, canonical-layout left/right
// environments per bond (LocalOp docs in solvers.h), optional right-hand-side environments, and matrix-free
// local solves.  The reference's pre-contracted environments (ALS `G` already multiplied by A_i,
// als.jl:47-50; MALS 5-index `H` containing A_{i+1}, mals.jl:10-13) describe the same local operator
// K = L·W_i(·W_{i+1})·R, so the local problems — and hence the sweep results — are the same; the dense
// assemblies + LU (als.jl:58-70, mals.jl:148-169) are replaced by Krylov solves on the matvec.
#include <memory>
#include "solvers.h"

namespace ttn {

// ---------------------------------------------------------------------------------------------------------
// small host helpers
// ---------------------------------------------------------------------------------------------------------
static int64_t prod_wrap(const std::vector<int64_t>& v, int lo, int hi) {  // Julia Int64 prod with wraparound
  uint64_t p = 1;
  for (int i = lo; i < hi; ++i) p *= (uint64_t)v[i];
  return (int64_t)p;
}
// src/tt_tools.jl:407-425
std::vector<int64_t> r_and_d_to_rks(const std::vector<int64_t>& rks, const std::vector<int64_t>& dims, int64_t rmax) {
  std::vector<int64_t> out(rks.size(), 1);
  const int d = (int)dims.size();
  for (int i = 0; i < d; ++i) {
    const int64_t left = prod_wrap(dims, 0, i), right = prod_wrap(dims, i, d);
    int64_t v = std::min(rks[i], rmax);
    if (right > 0) v = std::min(v, right);
    if (left > 0) v = std::min(v, left);
    out[i] = v;
  }
  return out;
}
// src/solvers/mals.jl:42-56 (returns the number of retained singular values)
int sv_trunc_count(const double* s, int len, double tol) {
  if (tol == 0.0) return len;
  int i = 0;
  double weight = 0.0, norm2 = 0.0;
  for (int j = 0; j < len; ++j) norm2 += s[j] * s[j];
  while (i < len && weight < tol * norm2) { weight += s[len - i - 1] * s[len - i - 1]; ++i; }
  return len - i + 1;
}
// src/solvers/dmrg.jl:179-185
int cut_off_index(const double* s, int len, double tol) {
  double n2 = 0.0;
  for (int j = 0; j < len; ++j) n2 += s[j] * s[j];
  const double thr = std::sqrt(n2) * tol;
  int k = 0;
  for (int j = 0; j < len; ++j) if (s[j] > thr) ++k;
  const double dt = 1e-10;
  while (k >= 1 && k < len && std::fabs(s[k - 1] - s[k]) <= std::max(dt, dt * std::max(std::fabs(s[k - 1]), std::fabs(s[k])))) ++k;
  return k;
}

void tt_to_complex(const TT<double>& x, TT<zc>& y) {
  y.d = x.d; y.batch = x.batch; y.dims = x.dims; y.rks = x.rks; y.ot = x.ot;
  y.cores.clear();
  y.cores.resize(x.d);
  for (int k = 0; k < x.d; ++k) {
    y.alloc_core(k);
    real_to_cplx(x.core(k), y.core(k), x.core_elems(k) * x.batch);
  }
}
template <class T>
void tto_copy(const TTO<T>& a, TTO<T>& b) {
  b.d = a.d; b.dims = a.dims; b.rks = a.rks;
  b.cores.clear();
  b.cores.resize(a.d);
  for (int k = 0; k < a.d; ++k) {
    b.cores[k].alloc(a.cores[k].bytes);
    TTN_CUDA(cudaMemcpyAsync(b.cores[k].p, a.cores[k].p, a.cores[k].bytes, cudaMemcpyDeviceToDevice, ctx().stream));
  }
}
void tto_to_complex(const TTO<double>& a, TTO<zc>& b) {
  b.d = a.d; b.dims = a.dims; b.rks = a.rks;
  b.cores.clear();
  b.cores.resize(a.d);
  for (int k = 0; k < a.d; ++k) {
    const int64_t n = (int64_t)(a.cores[k].bytes / sizeof(double));
    b.cores[k].alloc(sizeof(zc) * (size_t)n);
    real_to_cplx(a.core(k), b.core(k), n);
  }
}

// src/tt_tools.jl:443-489 with noise = 0 (exact zero padding)
template <class T>
static void increase_ranks(TT<T>& x, int64_t max_bond) {
  const int d = x.d;
  int64_t cur = 0;
  for (auto r : x.rks) cur = std::max(cur, r);
  ttn_assert(max_bond > cur, 2, "New bond dimension too low");
  std::vector<int64_t> tgt(d + 1, max_bond);
  tgt[0] = 1; tgt[d] = 1;
  tgt = r_and_d_to_rks(tgt, x.dims, max_bond);
  for (int k = 0; k < d; ++k) {
    const int64_t n = x.dims[k], ol = x.rks[k], orr = x.rks[k + 1], nl = tgt[k], nr = tgt[k + 1];
    ttn_assert(nl >= ol && nr >= orr, 2, "increase_ranks: target ranks below current ranks");
    DevBuf nb(sizeof(T) * (size_t)(n * nl * nr));
    fill<T>(nb.as<T>(), n * nl * nr, t_zero<T>());
    Copy4 c;
    c.n0 = n; c.n1 = ol; c.n2 = orr;
    c.s0 = 1; c.s1 = n; c.s2 = n * ol;
    c.d0 = 1; c.d1 = n; c.d2 = n * nl;
    copy4<T>(x.core(k), nb.as<T>(), c);
    x.cores[k] = std::move(nb);
  }
  x.rks = tgt;
  x.ot.assign(d, 0);
}

template <class T>
static void orthogonalize_in_place(TT<T>& x) {  // tt_orthogonalize(x, 1) written back into x
  TT<T> y;
  tt_orthogonalize(x, 1, y);
  x.cores = std::move(y.cores); x.rks = y.rks; x.ot = y.ot;
}

// The reference's sweep schedule: stage i ends when the sweep count reaches sweep_schedule[i] and the next stage starts with
// that sweep; the solve ends with the last stage.
struct SweepSchedule {
  const ttn_solver_params& p;
  int nsweeps = 0, stage = 0;
  bool new_stage = false;  // the sweep started by the last next() opened a stage
  explicit SweepSchedule(const ttn_solver_params& p_) : p(p_) {
    ttn_assert(p.n_sweep_schedule >= 1 && p.n_sweep_schedule == p.n_rmax_schedule && p.sweep_schedule && p.rmax_schedule, 4,
               "Sweep schedule error");
  }
  bool next() {  // starts a sweep; false once the last stage has ended
    new_stage = (++nsweeps == p.sweep_schedule[stage]);
    if (new_stage) ++stage;
    return stage < p.n_sweep_schedule;
  }
  int64_t rmax() const { return p.rmax_schedule[stage]; }
};

// ---------------------------------------------------------------------------------------------------------
// sweep state
// ---------------------------------------------------------------------------------------------------------
template <class T>
struct Sweeper {
  const TTO<T>& A;
  const TT<T>* b;
  TT<T>& x;
  int d;
  std::vector<DevBuf> L, R, bL, bR;  // per bond 0..d, canonical layouts

  Sweeper(const TTO<T>& A_, const TT<T>* b_, TT<T>& x_) : A(A_), b(b_), x(x_), d(x_.d) {
    ttn_assert(A.d == d && A.dims == x.dims, 1, "Incompatible dimensions");
    if (b) ttn_assert(b->d == d && b->dims == x.dims, 1, "Incompatible dimensions");
    ttn_assert(x.batch == 1 && (!b || b->batch == 1), 2, "solvers operate on a single TT (batch == 1)");
    ttn_assert(A.rks[0] == 1 && A.rks[d] == 1 && x.rks[0] == 1 && x.rks[d] == 1, 1, "boundary ranks must be 1");
    L.resize(d + 1); R.resize(d + 1);
    if (b) { bL.resize(d + 1); bR.resize(d + 1); }
    L[0].alloc(sizeof(T)); R[d].alloc(sizeof(T));
    fill<T>(L[0].as<T>(), 1, t_one<T>());
    fill<T>(R[d].as<T>(), 1, t_one<T>());
    if (b) {
      bL[0].alloc(sizeof(T)); bR[d].alloc(sizeof(T));
      fill<T>(bL[0].as<T>(), 1, t_one<T>());
      fill<T>(bR[d].as<T>(), 1, t_one<T>());
    }
  }
  int chi(int bond) const { return (int)x.rks[bond]; }
  int w(int bond) const { return (int)A.rks[bond]; }
  int n(int site) const { return (int)x.dims[site]; }

  void update_left(int k) {   // L[k+1] from L[k] and site k
    env_update<T>(true, L[k].as<T>(), chi(k), w(k), x.core(k), n(k), chi(k), chi(k + 1), A.core(k), w(k), w(k + 1), L[k + 1]);
    if (b) envb_update<T>(true, bL[k].as<T>(), chi(k), (int)b->rks[k], x.core(k), n(k), chi(k), chi(k + 1), b->core(k),
                          (int)b->rks[k], (int)b->rks[k + 1], bL[k + 1]);
  }
  void update_right(int k) {  // R[k] from R[k+1] and site k
    env_update<T>(false, R[k + 1].as<T>(), chi(k + 1), w(k + 1), x.core(k), n(k), chi(k), chi(k + 1), A.core(k), w(k), w(k + 1),
                  R[k]);
    if (b) envb_update<T>(false, bR[k + 1].as<T>(), chi(k + 1), (int)b->rks[k + 1], x.core(k), n(k), chi(k), chi(k + 1),
                          b->core(k), (int)b->rks[k], (int)b->rks[k + 1], bR[k]);
  }
  void init_right(int down_to) {  // R[d-1] ... R[down_to]
    for (int k = d - 1; k >= down_to; --k) update_right(k);
  }

  void setup_op(LocalOp<T>& op, DevBuf& W, int k, int N, bool sym) {
    int nn;
    fuse_mpo<T>(A, k, N, W, nn);
    op.setup(L[k].as<T>(), chi(k), w(k), R[k + N].as<T>(), chi(k + N), w(k + N), W.as<T>(), nn, sym);
  }

  // current window tensor in the V layout (chi_l, n^N, chi_r)
  void window(int k, int N, DevBuf& V) {
    const int cl = chi(k), cr = chi(k + N);
    if (N == 1) {
      V.alloc(sizeof(T) * (size_t)cl * n(k) * cr);
      Copy4 c;  // V[a,s,c] = x[s,a,c]
      c.n0 = n(k); c.s0 = 1; c.d0 = cl;
      c.n1 = cl; c.s1 = n(k); c.d1 = 1;
      c.n2 = cr; c.s2 = (int64_t)n(k) * cl; c.d2 = (int64_t)cl * n(k);
      copy4<T>(x.core(k), V.as<T>(), c);
      return;
    }
    const int n1 = n(k), n2 = n(k + 1), cm = chi(k + 1);
    V.alloc(sizeof(T) * (size_t)cl * n1 * n2 * cr);
    GemmArgs g;  // V[a,s1,s2,c] = sum_g x_k[s1,a,g] x_{k+1}[s2,g,c]
    g.M = cl; g.N = cr; g.K = cm;
    g.A = x.core(k); g.sAm = n1; g.sAk = (int64_t)n1 * cl; g.bA1 = 1; g.bA2 = 0;
    g.B = x.core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * cm; g.bB1 = 0; g.bB2 = 1;
    g.C = V.p; g.sCm = 1; g.sCn = (int64_t)cl * n1 * n2; g.bC1 = cl; g.bC2 = (int64_t)cl * n1;
    g.batch1 = n1; g.batch2 = n2;
    gemm<T>(g);
  }

  // projected right-hand side Pb (chi_l, n^N, chi_r)   (als.jl:68, mals.jl:165, dmrg.jl:94)
  void local_rhs(int k, int N, DevBuf& Pb) {
    const int cl = chi(k), cr = chi(k + N);
    const int n1 = n(k), bl = (int)b->rks[k], bm = (int)b->rks[k + 1];
    DevBuf T1(sizeof(T) * (size_t)cl * n1 * bm);
    {
      GemmArgs g;  // T1[a,s,gamma] = bL[a,beta] b_k[s,beta,gamma]
      g.M = cl; g.N = bm; g.K = bl;
      g.A = bL[k].p; g.sAm = 1; g.sAk = cl;
      g.B = b->core(k); g.sBk = n1; g.sBn = (int64_t)n1 * bl; g.bB1 = 1;
      g.C = T1.p; g.sCm = 1; g.sCn = (int64_t)cl * n1; g.bC1 = cl;
      g.batch1 = n1;
      gemm<T>(g);
    }
    int64_t rows = (int64_t)cl * n1;
    int bk = bm;
    DevBuf T2;
    const T* last = T1.as<T>();
    if (N == 2) {
      const int n2 = n(k + 1), br = (int)b->rks[k + 2];
      T2.alloc(sizeof(T) * (size_t)rows * n2 * br);
      GemmArgs g;  // T2[(a,s1),s2,gamma2] = T1[(a,s1),gamma1] b_{k+1}[s2,gamma1,gamma2]
      g.M = (int)rows; g.N = br; g.K = bm;
      g.A = T1.p; g.sAm = 1; g.sAk = rows;
      g.B = b->core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * bm; g.bB1 = 1;
      g.C = T2.p; g.sCm = 1; g.sCn = rows * n2; g.bC1 = rows;
      g.batch1 = n2;
      gemm<T>(g);
      rows *= n2;
      bk = br;
      last = T2.as<T>();
    }
    Pb.alloc(sizeof(T) * (size_t)rows * cr);
    GemmArgs g;  // Pb[(a,s..),c] = T[(a,s..),gamma] bR[c,gamma]
    g.M = (int)rows; g.N = cr; g.K = bk;
    g.A = last; g.sAm = 1; g.sAk = rows;
    g.B = bR[k + N].p; g.sBk = cr; g.sBn = 1;
    g.C = Pb.p; g.sCm = 1; g.sCn = rows;
    gemm<T>(g);
  }

  // x_k[s,a,kappa] = U[a + chi_l*s, kappa]
  void store_core_from_rows(int k, const T* U, int cl, int r) {
    const int nk = n(k);
    DevBuf nc(sizeof(T) * (size_t)nk * cl * r);
    Copy4 c;
    c.n0 = cl; c.s0 = 1; c.d0 = nk;
    c.n1 = nk; c.s1 = cl; c.d1 = 1;
    c.n2 = r; c.s2 = (int64_t)cl * nk; c.d2 = (int64_t)nk * cl;
    copy4<T>(U, nc.as<T>(), c);
    x.cores[k] = std::move(nc);
  }
  // x_k[s,kappa,c] = M[kappa + r*(s + n*c)]  (optionally conjugated source laid out as [(s,c), kappa])
  void store_core_from_SVt(int k, const T* SVt, int r, int cr) {
    const int nk = n(k);
    DevBuf nc(sizeof(T) * (size_t)nk * r * cr);
    Copy4 c;
    c.n0 = r; c.s0 = 1; c.d0 = nk;
    c.n1 = nk; c.s1 = r; c.d1 = 1;
    c.n2 = cr; c.s2 = (int64_t)r * nk; c.d2 = (int64_t)nk * r;
    copy4<T>(SVt, nc.as<T>(), c);
    x.cores[k] = std::move(nc);
  }
  // x_k[s,kappa,c] = conj(Vq[(s + n*c), kappa])
  void store_core_from_Vq(int k, const T* Vq, int q, int r, int cr) {
    const int nk = n(k);
    DevBuf nc(sizeof(T) * (size_t)nk * r * cr);
    Copy4 c;
    c.n0 = nk; c.s0 = 1; c.d0 = 1;
    c.n1 = cr; c.s1 = nk; c.d1 = (int64_t)nk * r;
    c.n2 = r; c.s2 = q; c.d2 = nk;
    c.conj = true;
    copy4<T>(Vq, nc.as<T>(), c);
    x.cores[k] = std::move(nc);
  }

  double residual() {  // ||A x - b|| / max(||b||, eps)     (als.jl:224, mals.jl:308, dmrg.jl:441,472)
    TT<T> y, mb, z;
    tt_apply(A, x, y);
    tt_scale(*b, t_from<T>(-1.0, 0.0), mb);
    tt_add(mb, y, z);
    std::vector<T> zz, bb;
    tt_dot(z, z, zz);
    tt_dot(*b, *b, bb);
    const double nz = std::sqrt(std::max(0.0, t_real(zz[0]))), nb = std::sqrt(std::max(0.0, t_real(bb[0])));
    return nz / std::max(nb, 2.220446049250313e-16);
  }
};

// ---------------------------------------------------------------------------------------------------------
// QR right move shared by ALS (als.jl:104-136) and TDVP (tdvp.jl:83): the window V of site k, viewed as (chi_l n_k) x chi_r,
// is factored V = Q R with r = min(chi_l n_k, chi_r); core k <- Q, bond k+1 <- r, R (r x chi_r) returned for the caller to absorb.
// ---------------------------------------------------------------------------------------------------------
template <class T>
static int qr_right_move(Sweeper<T>& S, int k, DevBuf& V, DevBuf& R) {
  const int cl = S.chi(k), cr = S.chi(k + 1), m = cl * S.n(k), r = std::min(m, cr);
  DevBuf tau(sizeof(T) * (size_t)r), Q(sizeof(T) * (size_t)m * r);
  R.alloc(sizeof(T) * (size_t)r * cr);
  qr_factor<T>(V.as<T>(), m, cr, m, tau.as<T>());
  qr_form_q<T>(V.as<T>(), m, r, m, tau.as<T>(), Q.as<T>(), m);
  Copy4 t; t.n0 = r; t.n1 = cr; t.s0 = 1; t.s1 = m; t.d0 = 1; t.d1 = r; t.tri = 1;
  copy4<T>(V.as<T>(), R.as<T>(), t);
  S.store_core_from_rows(k, Q.as<T>(), cl, r);
  S.x.rks[k + 1] = r;
  return r;
}

// ---------------------------------------------------------------------------------------------------------
// ALS core moves (src/solvers/als.jl:104-136): QR of the local solution, R absorbed into the neighbour
// ---------------------------------------------------------------------------------------------------------
template <class T>
static void als_right_move(Sweeper<T>& S, int k, DevBuf& V) {
  const int cr = S.chi(k + 1);
  ttn_assert(S.chi(k) * S.n(k) >= cr, 1, "ALS: TT ranks exceed the local unfolding (over-full ranks)");
  DevBuf Rb;
  qr_right_move(S, k, V, Rb);
  S.x.ot[k] = -1;
  // x_{k+1}[s,kappa,c'] = sum_z R[kappa,z] x_{k+1}[s,z,c']
  const int n2 = S.n(k + 1), c2 = S.chi(k + 2);
  DevBuf nc(sizeof(T) * (size_t)n2 * cr * c2);
  GemmArgs g;
  g.M = cr; g.N = c2; g.K = cr;
  g.A = Rb.p; g.sAm = 1; g.sAk = cr;
  g.B = S.x.core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * cr; g.bB1 = 1;
  g.C = nc.p; g.sCm = n2; g.sCn = (int64_t)n2 * cr; g.bC1 = 1;
  g.batch1 = n2;
  gemm<T>(g);
  S.x.cores[k + 1] = std::move(nc);
  S.x.ot[k + 1] = 0;
}

template <class T>
static void als_left_move(Sweeper<T>& S, int k, DevBuf& V) {
  const int cl = S.chi(k), cr = S.chi(k + 1), nk = S.n(k), m = nk * cr;
  ttn_assert(m >= cl, 1, "ALS: TT ranks exceed the local unfolding (over-full ranks)");
  DevBuf W(sizeof(T) * (size_t)m * cl), tau(sizeof(T) * (size_t)cl), Q(sizeof(T) * (size_t)m * cl), Rb(sizeof(T) * (size_t)cl * cl);
  Copy4 c;  // W[(s,c), a] = V[a,s,c]
  c.n0 = m; c.s0 = cl; c.d0 = 1;
  c.n1 = cl; c.s1 = 1; c.d1 = m;
  copy4<T>(V.as<T>(), W.as<T>(), c);
  qr_factor<T>(W.as<T>(), m, cl, m, tau.as<T>());
  qr_form_q<T>(W.as<T>(), m, cl, m, tau.as<T>(), Q.as<T>(), m);
  Copy4 t; t.n0 = cl; t.n1 = cl; t.s0 = 1; t.s1 = m; t.d0 = 1; t.d1 = cl; t.tri = 1;
  copy4<T>(W.as<T>(), Rb.as<T>(), t);
  {
    DevBuf nc(sizeof(T) * (size_t)nk * cl * cr);
    Copy4 e;  // x_k[s,kappa,c] = Q[s + n*c, kappa]
    e.n0 = nk; e.s0 = 1; e.d0 = 1;
    e.n1 = cr; e.s1 = nk; e.d1 = (int64_t)nk * cl;
    e.n2 = cl; e.s2 = m; e.d2 = nk;
    copy4<T>(Q.as<T>(), nc.as<T>(), e);
    S.x.cores[k] = std::move(nc);
    S.x.ot[k] = 1;
  }
  // x_{k-1}[(s,b),kappa] = sum_z x_{k-1}[(s,b),z] R[kappa,z]
  const int n0 = S.n(k - 1), c0 = S.chi(k - 1);
  DevBuf nc(sizeof(T) * (size_t)n0 * c0 * cl);
  GemmArgs g;
  g.M = n0 * c0; g.N = cl; g.K = cl;
  g.A = S.x.core(k - 1); g.sAm = 1; g.sAk = (int64_t)n0 * c0;
  g.B = Rb.p; g.sBk = cl; g.sBn = 1;
  g.C = nc.p; g.sCm = 1; g.sCn = (int64_t)n0 * c0;
  gemm<T>(g);
  S.x.cores[k - 1] = std::move(nc);
  S.x.ot[k - 1] = 0;
}

// ---------------------------------------------------------------------------------------------------------
// SVD core moves shared by MALS (mals.jl:94-146), DMRG (dmrg.jl:187-232) and TDVP2 (tdvp.jl:250,278).
// Theta = V viewed as (chi_l n_k) x (rest).  `rule` maps the sorted singular values to the retained rank.
// right move: core k <- U, returns S·Vt (r x q);   left move: core `site` <- Vt, returns U·S (p x r)
// ---------------------------------------------------------------------------------------------------------
template <class T, class Rule>
static int svd_right_move(Sweeper<T>& S, int k, const T* V, int p, int q, Rule rule, DevBuf& SVt) {
  DevBuf U;
  const int r = split_left<T>(V, p, q, 1, p, false, rule, U, SVt);
  S.store_core_from_rows(k, U.as<T>(), S.chi(k), r);
  S.x.rks[k + 1] = r;
  return r;
}
template <class T, class Rule>
static int svd_left_move(Sweeper<T>& S, int site, const T* V, int p, int q, Rule rule, DevBuf& US) {
  DevBuf Vq, SVtp;  // Theta^H = Vq * (S U^H)
  const int r = split_left<T>(V, q, p, p, 1, true, rule, Vq, SVtp);
  S.store_core_from_Vq(site, Vq.as<T>(), q, r, S.chi(site + 1));
  S.x.rks[site] = r;
  US.alloc(sizeof(T) * (size_t)p * r);
  Copy4 c;  // US[i,kappa] = conj(SVtp[kappa,i])
  c.n0 = p; c.s0 = r; c.d0 = 1;
  c.n1 = r; c.s1 = 1; c.d1 = p;
  c.conj = true;
  copy4<T>(SVtp.as<T>(), US.as<T>(), c);
  return r;
}

// ---------------------------------------------------------------------------------------------------------
// als_linsolve (src/solvers/als.jl:161-225)
// ---------------------------------------------------------------------------------------------------------
template <class T>
void als_linsolve(const TTO<T>& A, const TT<T>& b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, double* residual) {
  tt_orthogonalize(x0, 1, x);
  ttn_assert(x.rks == x0.rks, 1, "ALS: tt_start has over-full ranks (orthogonalize changed them)");
  Sweeper<T> S(A, &b, x);
  const int d = S.d;
  S.init_right(1);
  const double tol = 1e-14;
  const int kd = std::max(p.krylovdim, 2), maxit = std::max(p.linsolv_maxiter, 1);
  auto solve_site = [&](int k, DevBuf& V) {
    LocalOp<T> op; DevBuf W, Pb;
    S.setup_op(op, W, k, 1, false);
    S.local_rhs(k, 1, Pb);
    S.window(k, 1, V);
    local_linsolve<T>(op, Pb.as<T>(), V.as<T>(), kd, maxit, tol, p);
  };
  int nsweeps = 0;
  while (nsweeps < p.sweep_count) {
    ++nsweeps;
    for (int k = 0; k < d - 1; ++k) {
      DevBuf V;
      solve_site(k, V);
      als_right_move(S, k, V);
      S.update_left(k);
    }
    if (nsweeps == p.sweep_count) break;
    ++nsweeps;
    for (int k = d - 1; k >= 1; --k) {
      DevBuf V;
      solve_site(k, V);
      als_left_move(S, k, V);
      S.update_right(k);
    }
  }
  if (residual) *residual = S.residual();
}

// ---------------------------------------------------------------------------------------------------------
// als_eigsolve (src/solvers/als.jl:251-321), noise_schedule = 0
// ---------------------------------------------------------------------------------------------------------
// stage change: ranks raised to the stage's rmax by zero padding, then the train is left-orthogonalised again
template <class T>
static void als_next_stage(TT<T>& x, int64_t rmax) {
  increase_ranks(x, rmax);
  orthogonalize_in_place(x);
}

template <class T>
void als_eigsolve(const TTO<T>& A, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, std::vector<double>& E) {
  SweepSchedule sched(p);
  tt_orthogonalize(x0, 1, x);
  E.clear();
  const int kd = std::max(p.krylovdim, 2), maxit = std::max(p.linsolv_maxiter, 1);
  std::unique_ptr<Sweeper<T>> S(new Sweeper<T>(A, nullptr, x));
  const int d = x.d;
  S->init_right(1);
  auto eig_site = [&](int k, DevBuf& V) {
    LocalOp<T> op; DevBuf W;
    S->setup_op(op, W, k, 1, false);
    S->window(k, 1, V);
    return lanczos_lowest<T>(op, V.as<T>(), kd, maxit, p.linsolv_tol, nullptr);
  };
  while (sched.next()) {
    if (sched.new_stage) {
      als_next_stage(x, sched.rmax());
      S.reset(new Sweeper<T>(A, nullptr, x));
      S->init_right(1);
    }
    for (int k = 0; k < d - 1; ++k) {
      DevBuf V;
      E.push_back(eig_site(k, V));
      als_right_move(*S, k, V);
      S->update_left(k);
    }
    for (int k = d - 1; k >= 1; --k) {
      DevBuf V;
      E.push_back(eig_site(k, V));
      als_left_move(*S, k, V);
      S->update_right(k);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// als_gen_eigsolv (src/solvers/als.jl:344-440): A x = lambda S x.  Two sets of environments over the same train
// (G/H for A, K/L for S in the reference); the local pencil is solved densely like `K_eiggenmin` (als.jl:89-102).
// ---------------------------------------------------------------------------------------------------------
template <class T>
void als_gen_eigsolve(const TTO<T>& A, const TTO<T>& Sop, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x,
                      std::vector<double>& E) {
  SweepSchedule sched(p);
  tt_orthogonalize(x0, 1, x);
  E.clear();
  const int kd = std::max(p.krylovdim, 2), maxit = std::max(p.linsolv_maxiter, 1);
  std::unique_ptr<Sweeper<T>> SA(new Sweeper<T>(A, nullptr, x)), SS(new Sweeper<T>(Sop, nullptr, x));
  const int d = x.d;
  SA->init_right(1);
  SS->init_right(1);
  auto eig_site = [&](int k, DevBuf& V) {
    LocalOp<T> opK, opM; DevBuf WK, WM;
    SA->setup_op(opK, WK, k, 1, false);
    SS->setup_op(opM, WM, k, 1, false);
    SA->window(k, 1, V);
    const double lam = gen_eig_lowest<T>(opK, opM, V.as<T>(), kd, maxit, p.linsolv_tol);
    if (std::is_same<T, zc>::value) {
      // `K_eiggenmin` contracts `Gi[d,e,a,b,z] * Hi[z,f,c]` (als.jl:91-92), the TRANSPOSE of `K_full`'s matrix (als.jl:60); for a
      // Hermitian pencil that is the complex-conjugate problem, whose eigenvector is conj(v).  Reproduced as is.
      DevBuf Vc(V.bytes);
      Copy4 c; c.n0 = (int64_t)opK.size(); c.conj = true;
      copy4<T>(V.as<T>(), Vc.as<T>(), c);
      V = std::move(Vc);
    }
    return lam;
  };
  while (sched.next()) {
    if (sched.new_stage) {
      als_next_stage(x, sched.rmax());
      SA.reset(new Sweeper<T>(A, nullptr, x));
      SS.reset(new Sweeper<T>(Sop, nullptr, x));
      SA->init_right(1);
      SS->init_right(1);
    }
    for (int k = 0; k < d - 1; ++k) {
      DevBuf V;
      E.push_back(eig_site(k, V));
      als_right_move(*SA, k, V);
      SA->update_left(k);
      SS->update_left(k);
    }
    for (int k = d - 1; k >= 1; --k) {
      DevBuf V;
      E.push_back(eig_site(k, V));
      als_left_move(*SA, k, V);
      SA->update_right(k);
      SS->update_right(k);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// MALS (src/solvers/mals.jl:240-309, :335-425)
// ---------------------------------------------------------------------------------------------------------
template <class T>
static void mals_right(Sweeper<T>& S, int k, DevBuf& V, double tol, int64_t rmax) {
  const int p_ = S.chi(k) * S.n(k), q_ = S.n(k + 1) * S.chi(k + 2);
  DevBuf SVt;
  auto rule = [&](const double* s, int len) { return (int)std::min<int64_t>(sv_trunc_count(s, len, tol), rmax); };
  const int r = svd_right_move<T>(S, k, V.as<T>(), p_, q_, rule, SVt);
  S.x.ot[k] = -1;
  S.store_core_from_SVt(k + 1, SVt.as<T>(), r, S.chi(k + 2));
  S.x.ot[k + 1] = 0;
}
template <class T>
static void mals_left(Sweeper<T>& S, int k, DevBuf& V, double tol, int64_t rmax) {
  const int cl = S.chi(k), p_ = cl * S.n(k), q_ = S.n(k + 1) * S.chi(k + 2);
  DevBuf US;
  auto rule = [&](const double* s, int len) { return (int)std::min<int64_t>(sv_trunc_count(s, len, tol), rmax); };
  const int r = svd_left_move<T>(S, k + 1, V.as<T>(), p_, q_, rule, US);
  S.x.ot[k + 1] = 1;
  S.store_core_from_rows(k, US.as<T>(), cl, r);
  S.x.ot[k] = 0;
}

template <class T>
void mals_linsolve(const TTO<T>& A, const TT<T>& b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, double* residual) {
  tt_orthogonalize(x0, 1, x);
  Sweeper<T> S(A, &b, x);
  const int d = S.d;
  ttn_assert(d >= 2, 2, "MALS needs at least two sites");
  int64_t rmax = p.rmax;
  if (rmax <= 0) {
    double pr = 1.0;
    for (auto v : x.dims) pr *= (double)v;
    rmax = (int64_t)std::llround(std::sqrt(pr));
  }
  S.init_right(2);
  const double tol = 1e-14;
  const int kd = std::max(p.krylovdim, 2), maxit = std::max(p.linsolv_maxiter, 1);
  auto solve_win = [&](int k, DevBuf& V) {
    LocalOp<T> op; DevBuf W, Pb;
    S.setup_op(op, W, k, 2, false);
    S.local_rhs(k, 2, Pb);
    S.window(k, 2, V);
    local_linsolve<T>(op, Pb.as<T>(), V.as<T>(), kd, maxit, tol, p);
  };
  for (int k = 0; k < d - 1; ++k) {
    DevBuf V;
    solve_win(k, V);
    mals_right(S, k, V, p.tol, rmax);
    S.update_left(k);
  }
  for (int k = d - 2; k >= 0; --k) {
    DevBuf V;
    solve_win(k, V);
    mals_left(S, k, V, p.tol, rmax);
    if (k > 0) S.update_right(k + 1);
  }
  if (residual) *residual = S.residual();
}

template <class T>
void mals_eigsolve(const TTO<T>& A, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, std::vector<double>& E,
                   std::vector<int64_t>& r_hist) {
  SweepSchedule sched(p);
  tt_orthogonalize(x0, 1, x);
  Sweeper<T> S(A, nullptr, x);
  const int d = S.d;
  ttn_assert(d >= 2, 2, "MALS needs at least two sites");
  E.clear(); r_hist.clear();
  S.init_right(2);
  const int kd = std::max(p.krylovdim, 2), maxit = std::max(p.linsolv_maxiter, 1);
  auto eig_win = [&](int k, DevBuf& V) {
    LocalOp<T> op; DevBuf W;
    S.setup_op(op, W, k, 2, false);
    S.window(k, 2, V);
    return lanczos_lowest<T>(op, V.as<T>(), kd, maxit, p.linsolv_tol, nullptr);
  };
  auto maxrank = [&]() { int64_t m = 0; for (auto r : x.rks) m = std::max(m, r); return m; };
  while (sched.next()) {
    const int64_t rmax = sched.rmax();
    for (int k = 0; k < d - 1; ++k) {
      DevBuf V;
      E.push_back(eig_win(k, V));
      mals_right(S, k, V, p.tol, rmax);
      r_hist.push_back(maxrank());
      S.update_left(k);
    }
    for (int k = d - 2; k >= 0; --k) {
      DevBuf V;
      E.push_back(eig_win(k, V));
      mals_left(S, k, V, p.tol, rmax);
      r_hist.push_back(maxrank());
      if (k > 0) S.update_right(k + 1);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// DMRG (src/solvers/dmrg.jl:385-473, :501-578), N in {1, 2}
// ---------------------------------------------------------------------------------------------------------
template <class T>
struct DmrgLocal {
  const ttn_solver_params& p;
  bool lin;
  ShardCtxT<T>* shard;
  int kd, maxit;
  DmrgLocal(const ttn_solver_params& p_, bool lin_, ShardCtxT<T>* shard_)
      : p(p_), lin(lin_), shard(shard_), kd(std::max(p.krylovdim, 2)), maxit(std::max(p.linsolv_maxiter, 1)) {}
  // solves the local problem at window k in place on V (holding the initial guess); returns lambda for eig
  double solve(Sweeper<T>& S, int k, int N, DevBuf& V) {
    LocalOp<T> op; DevBuf W;
    S.setup_op(op, W, k, N, p.symmetrize != 0);
    // multi-GPU: the matvec of this window sharded over the ranks (shard.cu); windows too small to shard stay local
    if (!lin && shard != nullptr)
      shard_install<T>(*shard, op, S.L[k].template as<T>(), S.R[k + N].template as<T>(), W.as<T>());
    if (lin) {
      DevBuf Pb;
      S.local_rhs(k, N, Pb);
      local_linsolve<T>(op, Pb.as<T>(), V.as<T>(), kd, maxit, p.linsolv_tol, p);
      return 0.0;
    }
    return lanczos_lowest<T>(op, V.as<T>(), kd, maxit, p.linsolv_tol, nullptr);
  }
};

// right move + next guess (dmrg.jl:312-326); V is (chi_l, n^N, chi_r) for window k
template <class T>
static void dmrg_right(Sweeper<T>& S, int k, int N, DevBuf& V, double tol, int64_t rmax, DevBuf& Vnext) {
  const int cl = S.chi(k), nk = S.n(k);
  const int p_ = cl * nk;
  const int q_ = (N == 2 ? S.n(k + 1) : 1) * S.chi(k + N);
  DevBuf SVt;
  auto rule = [&](const double* s, int len) { return (int)std::min<int64_t>(cut_off_index(s, len, tol), rmax); };
  const int r = svd_right_move<T>(S, k, V.as<T>(), p_, q_, rule, SVt);
  S.x.ot[k] = 1;
  S.x.ot[k + 1] = 0;
  // next guess V0[kappa, (J, s'), c'] = sum_c SVt[kappa, (J, c)] x_{k+N}[s', c, c']
  const int J = (N == 2 ? S.n(k + 1) : 1), cr = S.chi(k + N);
  if (k + N < S.d) {
    const int n3 = S.n(k + N), c3 = S.chi(k + N + 1);
    Vnext.alloc(sizeof(T) * (size_t)r * J * n3 * c3);
    GemmArgs g;
    g.M = r; g.N = c3; g.K = cr;
    g.A = SVt.p; g.sAm = 1; g.sAk = (int64_t)r * J; g.bA1 = r; g.bA2 = 0;
    g.B = S.x.core(k + N); g.sBk = n3; g.sBn = (int64_t)n3 * cr; g.bB1 = 0; g.bB2 = 1;
    g.C = Vnext.p; g.sCm = 1; g.sCn = (int64_t)r * J * n3; g.bC1 = r; g.bC2 = (int64_t)r * J;
    g.batch1 = J; g.batch2 = n3;
    gemm<T>(g);
  } else {
    Vnext = std::move(SVt);
  }
}

// left move + next guess (dmrg.jl:328-342); the guess uses the window's natural index order
template <class T>
static void dmrg_left(Sweeper<T>& S, int k, int N, DevBuf& V, double tol, int64_t rmax, DevBuf& Vnext) {
  const int site = k + N - 1;
  const int cl = S.chi(k);
  const int p_ = cl * (N == 2 ? S.n(k) : 1);
  const int q_ = S.n(site) * S.chi(site + 1);
  DevBuf US;
  auto rule = [&](const double* s, int len) { return (int)std::min<int64_t>(cut_off_index(s, len, tol), rmax); };
  const int r = svd_left_move<T>(S, site, V.as<T>(), p_, q_, rule, US);
  S.x.ot[site] = -1;
  if (site >= 1) S.x.ot[site - 1] = 0;
  const int J = (N == 2 ? S.n(k) : 1);
  if (k >= 1) {
    // V0[a', (s0, J), kappa] = sum_a x_{k-1}[s0, a', a] US[(a, J), kappa]
    const int n0 = S.n(k - 1), c0 = S.chi(k - 1);
    Vnext.alloc(sizeof(T) * (size_t)c0 * n0 * J * r);
    GemmArgs g;
    g.M = c0; g.N = r; g.K = cl;
    g.A = S.x.core(k - 1); g.sAm = n0; g.sAk = (int64_t)n0 * c0; g.bA1 = 1; g.bA2 = 0;
    g.B = US.p; g.sBk = 1; g.sBn = p_; g.bB1 = 0; g.bB2 = cl;
    g.C = Vnext.p; g.sCm = 1; g.sCn = (int64_t)c0 * n0 * J; g.bC1 = c0; g.bC2 = (int64_t)c0 * n0;
    g.batch1 = n0; g.batch2 = J;
    gemm<T>(g);
  } else {
    Vnext = std::move(US);
  }
}

template <class T>
static void dmrg_final_split(Sweeper<T>& S, int N, DevBuf& V, double tol, int64_t rmax) {
  if (N == 1) {
    // core 1 <- V  (dmrg.jl:451,540): x_0[s,0,c] = V[0,s,c]; with chi_0 = 1 the layouts coincide
    S.x.cores[0] = std::move(V);
  } else {
    DevBuf Vn;
    dmrg_left(S, 0, 2, V, tol, rmax, Vn);   // core 2 <- Vt, Vn = U·S (n_1 x r)
    S.x.cores[0] = std::move(Vn);
  }
  S.x.ot[0] = 0;
}

template <class T>
static void dmrg_run(const TTO<T>& A, const TT<T>* b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x,
                     std::vector<double>* E, std::vector<int64_t>* r_hist, double* residual, ShardCtxT<T>* shard) {
  SweepSchedule sched(p);
  const int N = p.N;
  ttn_assert(N == 1 || N == 2, 2, "dmrg: window size N must be 1 or 2");
  const bool lin = (b != nullptr);
  int64_t rmax_all = 0;
  for (int i = 0; i < p.n_rmax_schedule; ++i) rmax_all = std::max(rmax_all, p.rmax_schedule[i]);
  if (lin && N == 1) {
    TT<T> tmp;
    tt_copy(x0, tmp);
    int64_t cur = 0;
    for (auto r : tmp.rks) cur = std::max(cur, r);
    if (rmax_all > cur) increase_ranks(tmp, rmax_all);   // dmrg.jl:401-403
    tt_orthogonalize(tmp, 1, x);
  } else {
    tt_orthogonalize(x0, 1, x);
  }
  Sweeper<T> S(A, b, x);
  const int d = S.d;
  ttn_assert(d >= N + 0 && d >= 2, 2, "dmrg: too few sites");
  if (E) E->clear();
  if (r_hist) r_hist->clear();
  S.init_right(N);
  DmrgLocal<T> loc(p, lin, shard);
  DevBuf V;
  S.window(0, N, V);   // V0 = b_mid(tt_opt, 1, N)   (dmrg.jl:275-276)
  auto maxrank = [&]() { int64_t m = 0; for (auto r : x.rks) m = std::max(m, r); return m; };
  while (sched.next()) {
    const int64_t rmax = sched.rmax();
    for (int k = 0; k <= d - N - 1; ++k) {
      const double lam = loc.solve(S, k, N, V);
      if (E) E->push_back(lam);
      DevBuf Vn;
      dmrg_right(S, k, N, V, p.tol, rmax, Vn);
      S.update_left(k);
      V = std::move(Vn);
      if (r_hist) r_hist->push_back(maxrank());
    }
    for (int k = d - N; k >= 1; --k) {
      const double lam = loc.solve(S, k, N, V);
      if (E) E->push_back(lam);
      DevBuf Vn;
      dmrg_left(S, k, N, V, p.tol, rmax, Vn);
      S.update_right(k + N - 1);
      V = std::move(Vn);
      if (r_hist) r_hist->push_back(maxrank());
    }
  }
  const double lam = loc.solve(S, 0, N, V);
  if (E) E->push_back(lam);
  if (r_hist) r_hist->push_back(maxrank());
  dmrg_final_split(S, N, V, p.tol, p.rmax_schedule[p.n_rmax_schedule - 1]);
  if (residual) *residual = S.residual();
}

template <class T>
void dmrg_linsolve(const TTO<T>& A, const TT<T>& b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, double* residual) {
  dmrg_run<T>(A, &b, x0, p, x, nullptr, nullptr, residual, nullptr);
}
template <class T>
void dmrg_eigsolve(const TTO<T>& A, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, std::vector<double>& E,
                   std::vector<int64_t>& r_hist, ShardCtxT<T>* shard) {
  dmrg_run<T>(A, nullptr, x0, p, x, &E, &r_hist, nullptr, shard);
}

// ---------------------------------------------------------------------------------------------------------
// TDVP / TDVP2 (src/solvers/tdvp.jl:45-357).  The one-, two- and zero-site effective operators of tdvp.jl:29-35,205-208 are
// LocalOps of this engine (the (l,s,r) / (a,s_out,b,s_in) layouts of tdvp.jl:54-55 coincide with the window layout), the
// environment recursions of tdvp.jl:37-43 are update_left / update_right, `exponentiate` is lanczos_expm, and the truncations
// (tdvp.jl:250,278) are the SVD moves with the tail-norm rule.  A sweep carries the window AC of the orthogonality centre from
// site 0 to the last site and back to site 0.
// ---------------------------------------------------------------------------------------------------------
// V <- exp(t K) V with t = (tre, tim) (KrylovKit.exponentiate, tdvp.jl:75); the Krylov settings are clamped once per solve
struct Expm {
  int kd, maxit;
  double tol;
  explicit Expm(const ttn_tdvp_params& p) : kd(std::max(p.krylovdim, 2)), maxit(std::max(p.krylov_maxiter, 1)), tol(p.krylov_tol) {}
  template <class T>
  void operator()(LocalOp<T>& op, DevBuf& V, double tre, double tim) const {
    lanczos_expm<T>(op, V.as<T>(), tre, tim, kd, maxit, tol, nullptr);
  }
};
// the same on the one- or two-site window at k
template <class T>
static void evolve(Sweeper<T>& S, const Expm& ex, int k, int N, DevBuf& V, double tre, double tim) {
  LocalOp<T> op; DevBuf W;
  S.setup_op(op, W, k, N, false);
  ex(op, V, tre, tim);
}

// one-site sweep (tdvp.jl:45-152): each site forward by t1, each bond between two sites backward by t0
template <class T>
static void tdvp_sweep1(Sweeper<T>& S, const Expm& ex, DevBuf& AC, double t1re, double t1im, double t0re, double t0im) {
  TT<T>& x = S.x;
  const int d = S.d;
  for (int k = 0; k < d - 1; ++k) {
    evolve(S, ex, k, 1, AC, t1re, t1im);
    const int cr = S.chi(k + 1);
    DevBuf C;
    const int r = qr_right_move(S, k, AC, C);
    S.update_left(k);
    {
      LocalOp<T> op;   // bond k+1: L[k+1] has the new bond r, R[k+1] still the old bond cr; C is r x cr
      op.setup(S.L[k + 1].template as<T>(), r, S.w(k + 1), S.R[k + 1].template as<T>(), cr, S.w(k + 1), nullptr, 1, false);
      ex(op, C, t0re, t0im);
    }
    // AC[a,s,c] = sum_g C[a,g] x_{k+1}[s,g,c]
    const int n2 = S.n(k + 1), c2 = S.chi(k + 2);
    DevBuf ACn(sizeof(T) * (size_t)r * n2 * c2);
    GemmArgs g;
    g.M = r; g.N = c2; g.K = cr;
    g.A = C.p; g.sAm = 1; g.sAk = r;
    g.B = x.core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * cr; g.bB1 = 1;
    g.C = ACn.p; g.sCm = 1; g.sCn = (int64_t)r * n2; g.bC1 = r;
    g.batch1 = n2;
    gemm<T>(g);
    AC = std::move(ACn);
  }
  evolve(S, ex, d - 1, 1, AC, t1re, t1im);
  for (int k = d - 2; k >= 0; --k) {
    // AC belongs to site k+1: (cl, n, cr);  LQ of cl x (n cr) via QR of the conjugate transpose.  Unlike als_left_move, which
    // keeps R as factored and absorbs it transposed into the core on its left, the factor is taken as L = R^H: the bond
    // matrix C that the zero-site step evolves.
    const int cl = S.chi(k + 1), cr = S.chi(k + 2), nk = S.n(k + 1), m = nk * cr, r = std::min(cl, m);
    DevBuf W(sizeof(T) * (size_t)m * cl), tau(sizeof(T) * (size_t)r), Q(sizeof(T) * (size_t)m * r), C(sizeof(T) * (size_t)cl * r);
    Copy4 c;  // W[(s,c), a] = conj(AC[a,s,c])
    c.n0 = m; c.s0 = cl; c.d0 = 1;
    c.n1 = cl; c.s1 = 1; c.d1 = m;
    c.conj = true;
    copy4<T>(AC.as<T>(), W.as<T>(), c);
    qr_factor<T>(W.as<T>(), m, cl, m, tau.as<T>());
    qr_form_q<T>(W.as<T>(), m, r, m, tau.as<T>(), Q.as<T>(), m);
    Copy4 t;  // C = L = R^H : C[a,kappa] = conj(R[kappa,a])
    t.n0 = r; t.n1 = cl; t.s0 = 1; t.s1 = m; t.d0 = cl; t.d1 = 1; t.tri = 1; t.conj = true;
    copy4<T>(W.as<T>(), C.as<T>(), t);
    S.store_core_from_Vq(k + 1, Q.as<T>(), m, r, cr);   // x_{k+1}[s,kappa,c] = conj(Q[s + n c, kappa])
    x.rks[k + 1] = r;
    S.update_right(k + 1);
    {
      LocalOp<T> op;   // bond k+1: L[k+1] has the old bond cl, R[k+1] the new bond r; C is cl x r
      op.setup(S.L[k + 1].template as<T>(), cl, S.w(k + 1), S.R[k + 1].template as<T>(), r, S.w(k + 1), nullptr, 1, false);
      ex(op, C, t0re, t0im);
    }
    // AC[(a,s), g'] = sum_g x_k[(s,a), g] C[g,g']  -> window layout [a,s,g']
    const int c0 = S.chi(k), n0 = S.n(k);
    DevBuf ACn(sizeof(T) * (size_t)c0 * n0 * r);
    GemmArgs g;
    g.M = c0; g.N = r; g.K = cl;
    g.A = x.core(k); g.sAm = n0; g.sAk = (int64_t)n0 * c0; g.bA1 = 1;
    g.B = C.p; g.sBk = 1; g.sBn = cl; g.bB1 = 0;
    g.C = ACn.p; g.sCm = 1; g.sCn = (int64_t)c0 * n0; g.bC1 = c0;
    g.batch1 = n0;
    gemm<T>(g);
    AC = std::move(ACn);
    evolve(S, ex, k, 1, AC, t1re, t1im);
  }
}

// two-site sweep (tdvp.jl:210-301): each pair of sites forward by t2, each site between two pairs backward by t1
template <class T, class Rule>
static void tdvp_sweep2(Sweeper<T>& S, const Expm& ex, Rule rule, DevBuf& AC, double t2re, double t2im, double t1re,
                        double t1im) {
  const int d = S.d;
  for (int k = 0; k < d - 1; ++k) {
    const int cl = S.chi(k), cm = S.chi(k + 1), n1 = S.n(k), n2 = S.n(k + 1), cr = S.chi(k + 2);
    DevBuf AAC(sizeof(T) * (size_t)cl * n1 * n2 * cr);
    GemmArgs g;  // AAC[(a,s1),s2,c] = sum_g AC[(a,s1),g] x_{k+1}[s2,g,c]
    g.M = cl * n1; g.N = cr; g.K = cm;
    g.A = AC.p; g.sAm = 1; g.sAk = (int64_t)cl * n1;
    g.B = S.x.core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * cm; g.bB1 = 1;
    g.C = AAC.p; g.sCm = 1; g.sCn = (int64_t)cl * n1 * n2; g.bC1 = (int64_t)cl * n1;
    g.batch1 = n2;
    gemm<T>(g);
    evolve(S, ex, k, 2, AAC, t2re, t2im);
    DevBuf SVt;
    svd_right_move<T>(S, k, AAC.as<T>(), cl * n1, n2 * cr, rule, SVt);
    S.update_left(k);
    AC = std::move(SVt);   // (r, n2, cr) window of site k+1, whose core is not stored
    if (k < d - 2) evolve(S, ex, k + 1, 1, AC, t1re, t1im);
  }
  for (int k = d - 2; k >= 0; --k) {
    // AC is the window of site k+1: (cm, n2, cr)
    const int cl = S.chi(k), cm = S.chi(k + 1), n1 = S.n(k), n2 = S.n(k + 1), cr = S.chi(k + 2);
    DevBuf AAC(sizeof(T) * (size_t)cl * n1 * n2 * cr);
    GemmArgs g;  // AAC[a,s1,(s2,c)] = sum_g x_k[s1,a,g] AC[g,(s2,c)]
    g.M = cl; g.N = n2 * cr; g.K = cm;
    g.A = S.x.core(k); g.sAm = n1; g.sAk = (int64_t)n1 * cl; g.bA1 = 1;
    g.B = AC.p; g.sBk = 1; g.sBn = cm; g.bB1 = 0;
    g.C = AAC.p; g.sCm = 1; g.sCn = (int64_t)cl * n1; g.bC1 = cl;
    g.batch1 = n1;
    gemm<T>(g);
    evolve(S, ex, k, 2, AAC, t2re, t2im);
    DevBuf US;
    svd_left_move<T>(S, k + 1, AAC.as<T>(), cl * n1, n2 * cr, rule, US);
    S.update_right(k + 1);
    AC = std::move(US);   // (cl, n1, r) window of site k
    if (k > 0) evolve(S, ex, k, 1, AC, t1re, t1im);
  }
}

template <class T>
void tdvp_run(const TTO<T>& H, const TT<T>& u0, const ttn_tdvp_params& p, TT<T>& psi) {
  ttn_assert(p.n_steps >= 0 && (p.n_steps == 0 || p.steps), 2, "tdvp: bad steps");
  ttn_assert(is_cplx<T>::value || p.imaginary_time, 2, "tdvp: real-time evolution needs a complex state");
  const Expm ex(p);
  auto rule = [&](const double* s, int len) { return rank_tailnorm(s, len, p.max_bond, p.truncerr); };
  tt_orthogonalize(u0, 1, psi);
  for (int is = 0; is < p.n_steps; ++is) {
    const double h = p.steps[is];
    // dt_eff = +i h (imaginary time) or h (real time);  t1 = -i dt_eff,  t0 = +i dt_eff   (tdvp.jl:74,94,179)
    double t1re, t1im;
    if (p.imaginary_time) { t1re = h; t1im = 0.0; } else { t1re = 0.0; t1im = -h; }
    for (int s = 0; s < std::max(1, p.sweeps); ++s) {
      Sweeper<T> S(H, nullptr, psi);
      S.init_right(1);
      DevBuf AC;
      S.window(0, 1, AC);
      if (p.two_site) tdvp_sweep2(S, ex, rule, AC, 0.5 * t1re, 0.5 * t1im, -0.5 * t1re, -0.5 * t1im);
      else tdvp_sweep1(S, ex, AC, t1re, t1im, -t1re, -t1im);
      S.store_core_from_rows(0, AC.as<T>(), S.chi(0), S.chi(1));
      psi.ot.assign(psi.d, 0);
    }
    if (p.normalize) {
      std::vector<T> nn;
      tt_dot(psi, psi, nn);
      const double nrm = std::sqrt(std::max(0.0, t_real(nn[0])));
      ttn_assert(nrm > 0.0, 5, "tdvp: state norm vanished");
      scal<T>(psi.core_elems(0), t_from<T>(1.0 / nrm, 0.0), psi.core(0));
    }
    orthogonalize_in_place(psi);
  }
}

#define INST(T)                                                                                                           \
  template void tto_copy<T>(const TTO<T>&, TTO<T>&);                                                                      \
  template void als_linsolve<T>(const TTO<T>&, const TT<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&, double*);     \
  template void als_eigsolve<T>(const TTO<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&, std::vector<double>&);      \
  template void als_gen_eigsolve<T>(const TTO<T>&, const TTO<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&,          \
                                    std::vector<double>&);                                                                \
  template void mals_linsolve<T>(const TTO<T>&, const TT<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&, double*);    \
  template void mals_eigsolve<T>(const TTO<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&, std::vector<double>&,      \
                                 std::vector<int64_t>&);                                                                   \
  template void dmrg_linsolve<T>(const TTO<T>&, const TT<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&, double*);    \
  template void dmrg_eigsolve<T>(const TTO<T>&, const TT<T>&, const ttn_solver_params&, TT<T>&, std::vector<double>&,      \
                                 std::vector<int64_t>&, ShardCtxT<T>*);                                                    \
  template void tdvp_run<T>(const TTO<T>&, const TT<T>&, const ttn_tdvp_params&, TT<T>&);
INST(double)
INST(zc)
#undef INST

}  // namespace ttn
