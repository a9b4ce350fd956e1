// TDVP / TDVP2 sweeps on device-resident trains (src/solvers/tdvp.jl:45-357).
//
// The one-, two- and zero-site effective operators of tdvp.jl:29-35,205-208 are the LocalOp of localop.cu
// (the (l,s,r) / (a,s_out,b,s_in) layouts of tdvp.jl:54-55 coincide with the window layout used there), the
// environment recursions of tdvp.jl:37-43 are env_update, `exponentiate` is lanczos_expm, the QR steps
// (tdvp.jl:83,116) run on qr.cu and the truncations (tdvp.jl:250,278) on the Jacobi SVD with the tail-norm rule.
#include <memory>
#include "solvers.h"

namespace ttn {
namespace {

template <class T>
struct Tdvp {
  const TTO<T>& H;
  TT<T>& x;
  const ttn_tdvp_params& p;
  int d;
  std::vector<DevBuf> L, R;   // canonical environments per bond
  Tdvp(const TTO<T>& H_, TT<T>& x_, const ttn_tdvp_params& p_) : H(H_), x(x_), p(p_), d(x_.d) {
    ttn_assert(H.d == d && H.dims == x.dims, 1, "Incompatible dimensions");
    ttn_assert(x.batch == 1, 2, "tdvp operates on a single TT");
    L.resize(d + 1); R.resize(d + 1);
    L[0].alloc(sizeof(T)); R[d].alloc(sizeof(T));
    fill<T>(L[0].as<T>(), 1, t_one<T>());
    fill<T>(R[d].as<T>(), 1, t_one<T>());
  }
  int chi(int b) const { return (int)x.rks[b]; }
  int w(int b) const { return (int)H.rks[b]; }
  int n(int s) const { return (int)x.dims[s]; }
  void up_left(int k) {
    env_update<T>(true, L[k].as<T>(), chi(k), w(k), x.core(k), n(k), chi(k), chi(k + 1), H.core(k), w(k), w(k + 1), L[k + 1]);
  }
  void up_right(int k) {
    env_update<T>(false, R[k + 1].as<T>(), chi(k + 1), w(k + 1), x.core(k), n(k), chi(k), chi(k + 1), H.core(k), w(k), w(k + 1),
                  R[k]);
  }
  // exp(t K) on a window tensor; nsite = 1, 2 (window starting at k) or 0 (bond k: L[k], R[k])
  void evolve(int k, int nsite, DevBuf& V, double tre, double tim) {
    LocalOp<T> op; DevBuf W;
    if (nsite == 0) {
      op.setup(L[k].as<T>(), chi(k), w(k), R[k].as<T>(), chi(k), w(k), nullptr, 1, false);
    } else {
      int nn;
      fuse_mpo<T>(H, k, nsite, W, nn);
      op.setup(L[k].as<T>(), chi(k), w(k), R[k + nsite].as<T>(), chi(k + nsite), w(k + nsite), W.as<T>(), nn, false);
    }
    lanczos_expm<T>(op, V.as<T>(), tre, tim, std::max(p.krylovdim, 2), std::max(p.krylov_maxiter, 1), p.krylov_tol, nullptr);
  }
  void core_to_window(int k, DevBuf& V) {  // V[a,s,c] = x_k[s,a,c]
    const int cl = chi(k), cr = chi(k + 1), nk = n(k);
    V.alloc(sizeof(T) * (size_t)cl * nk * cr);
    Copy4 c;
    c.n0 = nk; c.s0 = 1; c.d0 = cl;
    c.n1 = cl; c.s1 = nk; c.d1 = 1;
    c.n2 = cr; c.s2 = (int64_t)nk * cl; c.d2 = (int64_t)cl * nk;
    copy4<T>(x.core(k), V.as<T>(), c);
  }
  void window_to_core(int k, const T* V, int cl, int cr) {  // x_k[s,a,c] = V[a,s,c]
    const int nk = n(k);
    DevBuf nc(sizeof(T) * (size_t)nk * cl * cr);
    Copy4 c;
    c.n0 = cl; c.s0 = 1; c.d0 = nk;
    c.n1 = nk; c.s1 = cl; c.d1 = 1;
    c.n2 = cr; c.s2 = (int64_t)cl * nk; c.d2 = (int64_t)nk * cl;
    copy4<T>(V, nc.as<T>(), c);
    x.cores[k] = std::move(nc);
    x.rks[k] = cl; x.rks[k + 1] = cr;
  }

  // ---- one-site sweep (tdvp.jl:45-152) -------------------------------------------------------------------
  void sweep1(double t1re, double t1im, double t0re, double t0im) {
    for (int k = d - 1; k >= 1; --k) up_right(k);
    DevBuf AC;
    core_to_window(0, AC);
    for (int k = 0; k < d - 1; ++k) {
      evolve(k, 1, AC, t1re, t1im);
      const int cl = chi(k), cr = chi(k + 1), nk = n(k), m = cl * nk, r = std::min(m, cr);
      DevBuf tau(sizeof(T) * (size_t)r), Q(sizeof(T) * (size_t)m * r), C(sizeof(T) * (size_t)r * cr);
      qr_factor<T>(AC.as<T>(), m, cr, m, tau.as<T>());
      qr_form_q<T>(AC.as<T>(), m, r, m, tau.as<T>(), Q.as<T>(), m);
      Copy4 t; t.n0 = r; t.n1 = cr; t.s0 = 1; t.s1 = m; t.d0 = 1; t.d1 = r; t.tri = 1;
      copy4<T>(AC.as<T>(), C.as<T>(), t);
      window_to_core(k, Q.as<T>(), cl, r);
      up_left(k);
      // bond evolution with L[k+1] (new bond r) and R[k+1] (old bond cr): C is r x cr
      {
        LocalOp<T> op;
        op.chi_l = r; op.chi_r = cr;
        op.setup(L[k + 1].as<T>(), r, w(k + 1), R[k + 1].as<T>(), cr, w(k + 1), nullptr, 1, false);
        lanczos_expm<T>(op, C.as<T>(), t0re, t0im, std::max(p.krylovdim, 2), std::max(p.krylov_maxiter, 1), p.krylov_tol,
                        nullptr);
      }
      // AC[a,s,c] = sum_g C[a,g] x_{k+1}[s,g,c]
      const int n2 = n(k + 1), c2 = chi(k + 2);
      DevBuf ACn(sizeof(T) * (size_t)r * n2 * c2);
      GemmArgs g;
      g.M = r; g.N = c2; g.K = cr;
      g.A = C.p; g.sAm = 1; g.sAk = r;
      g.B = x.core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * cr; g.bB1 = 1;
      g.C = ACn.p; g.sCm = 1; g.sCn = (int64_t)r * n2; g.bC1 = r;
      g.batch1 = n2;
      gemm<T>(g);
      AC = std::move(ACn);
      x.rks[k + 1] = r;   // bond k+1 now has dimension r on both sides of the centre
    }
    evolve(d - 1, 1, AC, t1re, t1im);
    for (int k = d - 2; k >= 0; --k) {
      // AC belongs to site k+1: (cl, n, cr);  LQ of cl x (n cr) via QR of the conjugate transpose
      const int cl = chi(k + 1), cr = chi(k + 2), nk = n(k + 1), m = nk * cr, r = std::min(cl, m);
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
      {
        DevBuf nc(sizeof(T) * (size_t)nk * r * cr);
        Copy4 e;  // x_{k+1}[s,kappa,c] = conj(Q[s + n c, kappa])
        e.n0 = nk; e.s0 = 1; e.d0 = 1;
        e.n1 = cr; e.s1 = nk; e.d1 = (int64_t)nk * r;
        e.n2 = r; e.s2 = m; e.d2 = nk;
        e.conj = true;
        copy4<T>(Q.as<T>(), nc.as<T>(), e);
        x.cores[k + 1] = std::move(nc);
      }
      const int old_bond = cl;
      x.rks[k + 1] = r;
      up_right(k + 1);
      {
        LocalOp<T> op;   // bond k+1: L[k+1] has the old bond dimension, R[k+1] the new one; C is old x r
        op.setup(L[k + 1].as<T>(), old_bond, w(k + 1), R[k + 1].as<T>(), r, w(k + 1), nullptr, 1, false);
        lanczos_expm<T>(op, C.as<T>(), t0re, t0im, std::max(p.krylovdim, 2), std::max(p.krylov_maxiter, 1), p.krylov_tol,
                        nullptr);
      }
      // AC[(a,s), g'] = sum_g x_k[(s,a), g] C[g,g']  -> window layout [a,s,g']
      const int c0 = chi(k), n0 = n(k);
      DevBuf ACn(sizeof(T) * (size_t)c0 * n0 * r);
      GemmArgs g;
      g.M = c0; g.N = r; g.K = old_bond;
      g.A = x.core(k); g.sAm = n0; g.sAk = (int64_t)n0 * c0; g.bA1 = 1;
      g.B = C.p; g.sBk = 1; g.sBn = old_bond; g.bB1 = 0;
      g.C = ACn.p; g.sCm = 1; g.sCn = (int64_t)c0 * n0; g.bC1 = c0;
      g.batch1 = n0;
      gemm<T>(g);
      AC = std::move(ACn);
      evolve(k, 1, AC, t1re, t1im);
    }
    window_to_core(0, AC.as<T>(), chi(0), chi(1));
    x.ot.assign(d, 0);
  }

  // ---- two-site sweep (tdvp.jl:210-301) ------------------------------------------------------------------
  void sweep2(double t2re, double t2im, double t1re, double t1im) {
    for (int k = d - 1; k >= 1; --k) up_right(k);
    DevBuf AC;
    core_to_window(0, AC);
    auto rule = [&](const double* s, int len) { return rank_tailnorm(s, len, p.max_bond, p.truncerr); };
    for (int k = 0; k < d - 1; ++k) {
      const int cl = chi(k), cm = chi(k + 1), n1 = n(k), n2 = n(k + 1), cr = chi(k + 2);
      DevBuf AAC(sizeof(T) * (size_t)cl * n1 * n2 * cr);
      GemmArgs g;  // AAC[(a,s1),s2,c] = sum_g AC[(a,s1),g] x_{k+1}[s2,g,c]
      g.M = cl * n1; g.N = cr; g.K = cm;
      g.A = AC.p; g.sAm = 1; g.sAk = (int64_t)cl * n1;
      g.B = x.core(k + 1); g.sBk = n2; g.sBn = (int64_t)n2 * cm; g.bB1 = 1;
      g.C = AAC.p; g.sCm = 1; g.sCn = (int64_t)cl * n1 * n2; g.bC1 = (int64_t)cl * n1;
      g.batch1 = n2;
      gemm<T>(g);
      evolve(k, 2, AAC, t2re, t2im);
      DevBuf U, SVt;
      const int pp = cl * n1, qq = n2 * cr;
      const int r = split_left<T>(AAC.as<T>(), pp, qq, 1, pp, false, rule, U, SVt);
      window_to_core(k, U.as<T>(), cl, r);
      up_left(k);
      AC = std::move(SVt);   // (r, n2, cr) window of site k+1
      x.rks[k + 1] = r;
      if (k < d - 2) {
        // the core of site k+1 is not stored yet; evolve AC with L[k+1], R[k+2]
        LocalOp<T> op; DevBuf W; int nn;
        fuse_mpo<T>(H, k + 1, 1, W, nn);
        op.setup(L[k + 1].as<T>(), r, w(k + 1), R[k + 2].as<T>(), cr, w(k + 2), W.as<T>(), nn, false);
        lanczos_expm<T>(op, AC.as<T>(), t1re, t1im, std::max(p.krylovdim, 2), std::max(p.krylov_maxiter, 1), p.krylov_tol,
                        nullptr);
      }
    }
    for (int k = d - 2; k >= 0; --k) {
      // AC is the window of site k+1: (cm, n2, cr)
      const int cl = chi(k), cm = chi(k + 1), n1 = n(k), n2 = n(k + 1), cr = chi(k + 2);
      DevBuf AAC(sizeof(T) * (size_t)cl * n1 * n2 * cr);
      GemmArgs g;  // AAC[a,s1,(s2,c)] = sum_g x_k[s1,a,g] AC[g,(s2,c)]
      g.M = cl; g.N = n2 * cr; g.K = cm;
      g.A = x.core(k); g.sAm = n1; g.sAk = (int64_t)n1 * cl; g.bA1 = 1;
      g.B = AC.p; g.sBk = 1; g.sBn = cm; g.bB1 = 0;
      g.C = AAC.p; g.sCm = 1; g.sCn = (int64_t)cl * n1; g.bC1 = cl;
      g.batch1 = n1;
      gemm<T>(g);
      evolve(k, 2, AAC, t2re, t2im);
      const int pp = cl * n1, qq = n2 * cr;
      DevBuf Vq, SVtp;
      const int r = split_left<T>(AAC.as<T>(), qq, pp, pp, 1, true, rule, Vq, SVtp);
      {
        DevBuf nc(sizeof(T) * (size_t)n2 * r * cr);
        Copy4 e;  // x_{k+1}[s,kappa,c] = conj(Vq[s + n2 c, kappa])
        e.n0 = n2; e.s0 = 1; e.d0 = 1;
        e.n1 = cr; e.s1 = n2; e.d1 = (int64_t)n2 * r;
        e.n2 = r; e.s2 = qq; e.d2 = n2;
        e.conj = true;
        copy4<T>(Vq.as<T>(), nc.as<T>(), e);
        x.cores[k + 1] = std::move(nc);
      }
      x.rks[k + 1] = r;
      up_right(k + 1);
      DevBuf ACn(sizeof(T) * (size_t)pp * r);
      Copy4 c;  // AC[(a,s1),kappa] = conj(SVtp[kappa,(a,s1)])
      c.n0 = pp; c.s0 = r; c.d0 = 1;
      c.n1 = r; c.s1 = 1; c.d1 = pp;
      c.conj = true;
      copy4<T>(SVtp.as<T>(), ACn.as<T>(), c);
      AC = std::move(ACn);
      if (k > 0) {
        LocalOp<T> op; DevBuf W; int nn;
        fuse_mpo<T>(H, k, 1, W, nn);
        op.setup(L[k].as<T>(), cl, w(k), R[k + 1].as<T>(), r, w(k + 1), W.as<T>(), nn, false);
        lanczos_expm<T>(op, AC.as<T>(), t1re, t1im, std::max(p.krylovdim, 2), std::max(p.krylov_maxiter, 1), p.krylov_tol,
                        nullptr);
      }
    }
    window_to_core(0, AC.as<T>(), chi(0), chi(1));
    x.ot.assign(d, 0);
  }
};

}  // namespace

template <class T>
void tdvp_run(const TTO<T>& H, const TT<T>& u0, const ttn_tdvp_params& p, TT<T>& psi) {
  ttn_assert(p.n_steps >= 0 && (p.n_steps == 0 || p.steps), 2, "tdvp: bad steps");
  ttn_assert(is_cplx<T>::value || p.imaginary_time, 2, "tdvp: real-time evolution needs a complex state");
  tt_orthogonalize(u0, 1, psi);
  for (int is = 0; is < p.n_steps; ++is) {
    const double h = p.steps[is];
    // dt_eff = +i h (imaginary time) or h (real time);  t1 = -i dt_eff,  t0 = +i dt_eff   (tdvp.jl:74,94,179)
    double t1re, t1im;
    if (p.imaginary_time) { t1re = h; t1im = 0.0; } else { t1re = 0.0; t1im = -h; }
    for (int s = 0; s < std::max(1, p.sweeps); ++s) {
      Tdvp<T> sw(H, psi, p);
      if (p.two_site) sw.sweep2(0.5 * t1re, 0.5 * t1im, -0.5 * t1re, -0.5 * t1im);
      else sw.sweep1(t1re, t1im, -t1re, -t1im);
    }
    if (p.normalize) {
      std::vector<T> nn;
      tt_dot(psi, psi, nn);
      const double nrm = std::sqrt(std::max(0.0, t_real(nn[0])));
      ttn_assert(nrm > 0.0, 5, "tdvp: state norm vanished");
      scal<T>(psi.core_elems(0), t_from<T>(1.0 / nrm, 0.0), psi.core(0));
    }
    TT<T> y;
    tt_orthogonalize(psi, 1, y);
    psi.cores = std::move(y.cores); psi.rks = y.rks; psi.ot = y.ot;
  }
}

template void tdvp_run<double>(const TTO<double>&, const TT<double>&, const ttn_tdvp_params&, TT<double>&);
template void tdvp_run<zc>(const TTO<zc>&, const TT<zc>&, const ttn_tdvp_params&, TT<zc>&);

}  // namespace ttn
