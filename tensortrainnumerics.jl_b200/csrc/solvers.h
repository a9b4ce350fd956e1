// Alternating solvers (ALS / MALS / DMRG / TDVP) on device-resident trains (internal).
#pragma once
#include "../../include/ttn_b200.h"
#include "tt.h"
#include <functional>

namespace ttn {

template <class T> void tto_copy(const TTO<T>& a, TTO<T>& b);
void tto_to_complex(const TTO<double>& a, TTO<zc>& b);
void tt_to_complex(const TT<double>& x, TT<zc>& y);

// ---------------------------------------------------------------------------------------------------------
// Effective operator of an N-site window:  Y[a,b,c] = sum L[a,y,d] W[y,b,e,z] V[d,e,f] R[c,z,f]
// Environments are kept in one canonical layout E[bra, mpo, ket] (column-major, bra fastest):
//   reference G[y,a,d] (dmrg.jl:32-35)  <-> L[a,y,d];   reference H[z,c,f] (dmrg.jl:27-30) <-> R[c,z,f].
// V / Y use the reference's (chi_l, n^N, chi_r) layout with the first site's physical index fastest (dmrg.jl:38-46).
// ---------------------------------------------------------------------------------------------------------
template <class T>
struct LocalOp {
  int chi_l = 1, chi_r = 1, w_l = 1, w_r = 1, nn = 1;
  bool zero_site = false;          // TDVP bond operator (tdvp.jl:33-35): no MPO core in the window
  bool symmetrize = false;         // 0.5 (K + K^T) as in dmrg.jl:241
  const T* L = nullptr;            // (chi_l, w_l, chi_l)
  DevBuf Rm;                       // R permuted to [(z,f), c]
  DevBuf Wp;                       // W'[(y,e),(b,z)]
  DevBuf Lt, Rmt, Wpt;             // transposed operator pieces (symmetrize only)
  DevBuf T1, T2;                   // workspaces
  std::function<void(const T*, T*)> ext_apply;   // sharded operator (shard.cu): replaces the local three-GEMM chain
  int64_t size() const { return (int64_t)chi_l * nn * chi_r; }
  // Wfused: (w_l, nn, nn, w_r) in the reference Amid layout [y, b, e, z]; nullptr for zero_site
  void setup(const T* Lenv, int chil, int wl, const T* Renv, int chir, int wr, const T* Wfused, int nn_, bool sym);
  void apply(const T* V, T* Y);
  void apply_batch(const T* V, T* Y, int nvec);   // nvec window vectors stored back to back
  double flops() const;
};

// canonical-layout environment update (left: in-bond = left bond of x; right: in-bond = right bond of x)
//   Eout[a', z, d'] = sum conj(x[j,a,a']) Ein[a,y,d] x[k,d,d'] A[j,k,(y,z) or (z,y)]
template <class T>
void env_update(bool left, const T* Ein, int chi_in, int w_in, const T* x, int n, int rl, int rr, const T* A, int Rl, int Rr,
                DevBuf& Eout);
// RHS environment update: Bout[a', beta'] = sum conj(x[j,a,a']) Bin[a,beta] b[j,beta,beta']
template <class T>
void envb_update(bool left, const T* Bin, int chi_in, int rb_in, const T* x, int n, int rl, int rr, const T* b, int bl, int br,
                 DevBuf& Bout);
// fused MPO of sites i..i+N-1 in the reference Amid layout (dmrg.jl:38-46), N in {1,2}
template <class T> void fuse_mpo(const TTO<T>& A, int i, int N, DevBuf& W, int& nn);

// ---------------------------------------------------------------------------------------------------------
// Krylov drivers around LocalOp (kernel family F8)
// ---------------------------------------------------------------------------------------------------------
struct KrylovInfo { int matvecs = 0; int restarts = 0; double resid = 0.0; bool converged = false; };
// lowest eigenpair (KrylovKit.eigsolve(..., :SR) stand-in, dmrg.jl:245): x holds the start vector on entry
template <class T> double lanczos_lowest(LocalOp<T>& op, T* x, int krylovdim, int maxiter, double tol, KrylovInfo* info);
// K x = rhs (GMRES(m); stands in for `\` als.jl:69 / mals.jl:167 and KrylovKit.linsolve dmrg.jl:170)
template <class T> void gmres_solve(LocalOp<T>& op, const T* rhs, T* x, int krylovdim, int maxiter, double tol, KrylovInfo* info);
// dense direct solve K x = rhs for small windows (`K_full` + `\\`: als.jl:58-70, mals.jl:148-169, dmrg.jl:49-54,173-174):
// K assembled by applying the operator to the identity (one batched three-GEMM pass), Householder QR, back substitution
template <class T> void dense_solve(LocalOp<T>& op, const T* rhs, T* x);
// lowest eigenpair of the Hermitian-definite pencil (K, M), dense (`K_eiggenmin`, als.jl:89-102); v: start vector in, eigenvector out
template <class T> double gen_eig_lowest(LocalOp<T>& opK, LocalOp<T>& opM, T* v, int krylovdim, int maxiter, double tol);
// dense when the window has at most max(itslv_thresh, 2048) unknowns and it_solver is off, GMRES otherwise
template <class T>
void local_linsolve(LocalOp<T>& op, const T* rhs, T* x, int krylovdim, int maxiter, double tol, const ttn_solver_params& p);
// x <- exp(t K) x  for Hermitian K (KrylovKit.exponentiate stand-in, tdvp.jl:75); t = (tre, tim)
template <class T>
void lanczos_expm(LocalOp<T>& op, T* x, double tre, double tim, int krylovdim, int maxiter, double tol, KrylovInfo* info);

// rank rules of the core moves (host): `sv_trunc` (mals.jl:42-56, number of retained values) and `cut_off_index`
// (dmrg.jl:179-185); the `_svdtrunc` tail-norm rule is rank_tailnorm (tt.h)
int sv_trunc_count(const double* s, int len, double tol);
int cut_off_index(const double* s, int len, double tol);
// src/tt_tools.jl:407-425, including the overflow-tolerant `prod(...) > 0` tests (Int64 products wrap around)
std::vector<int64_t> r_and_d_to_rks(const std::vector<int64_t>& rks, const std::vector<int64_t>& dims, int64_t rmax);

// ---------------------------------------------------------------------------------------------------------
// sweep drivers
// ---------------------------------------------------------------------------------------------------------
template <class T>
void als_linsolve(const TTO<T>& A, const TT<T>& b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, double* residual);
template <class T>
void als_eigsolve(const TTO<T>& A, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, std::vector<double>& E);
// als_gen_eigsolv(A, S, x0): A x = lambda S x                                   (src/solvers/als.jl:344-440)
template <class T>
void als_gen_eigsolve(const TTO<T>& A, const TTO<T>& Sop, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x,
                      std::vector<double>& E);
template <class T>
void mals_linsolve(const TTO<T>& A, const TT<T>& b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, double* residual);
template <class T>
void mals_eigsolve(const TTO<T>& A, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, std::vector<double>& E,
                   std::vector<int64_t>& r_hist);
template <class T>
void dmrg_linsolve(const TTO<T>& A, const TT<T>& b, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, double* residual);
template <class T> struct ShardCtxT;
// shard: multi-GPU context whose ranks run the same sweep with the Lanczos matvec sharded over them (nullptr: one GPU)
template <class T>
void dmrg_eigsolve(const TTO<T>& A, const TT<T>& x0, const ttn_solver_params& p, TT<T>& x, std::vector<double>& E,
                   std::vector<int64_t>& r_hist, ShardCtxT<T>* shard = nullptr);
// tdvp.jl:45-357 on a state of the operator's element type (real-time evolution needs ComplexF64)
template <class T>
void tdvp_run(const TTO<T>& H, const TT<T>& u0, const ttn_tdvp_params& p, TT<T>& psi);

// kernel-level test / benchmark entry points
template <class T>
void matvec2_host(int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid, const void* H, const void* V,
                  void* Y, bool symmetrize);
template <class T>
void env_host(bool left, int n, int w_l, int w_r, int r_l, int r_r, const void* E, const void* x, const void* A, void* Eout);

}  // namespace ttn

struct ttn_matvec_s : ttn::ByDtype<ttn::LocalOp> {
  ttn::DevBuf L, R;
};
namespace ttn {
// Effective-operator matvec sharded over the GPUs of one node (shard.cu): rank `rank` owns the bra slice [c0, c0 + cp) of
// the right environment, and the last GEMM's epilogue stores every finished tile to all peers as well.
template <class T>
struct ShardOp {
  int chi_l = 1, chi_r = 1, w_l = 1, w_r = 1, nn = 1, rank = 0, nranks = 1, c0 = 0, cp = 1;
  DevBuf L, Rs, Wq, T1, T2, err;
  const void* Lp = nullptr;                // L2[a,(y,d)] used by the last GEMM: L.p, or the sweep's environment itself (no copy)
  void* Ybuf[2] = {nullptr, nullptr};      // cudaMalloc (IPC-exportable), full (chi_l, nn, chi_r) vectors
  unsigned* flags = nullptr;               // cudaMalloc, [2][nranks] epoch counters (one row per buffer parity is not needed)
  void* Ypeer[2][8] = {};
  unsigned* flag_peer_h[8] = {};
  DevBuf flag_peer_d;
  std::vector<void*> opened;
  bool bound = false;
  unsigned epoch = 0;
  int64_t size() const { return (int64_t)chi_l * nn * chi_r; }
  ~ShardOp() {
    for (void* p : opened) cudaIpcCloseMemHandle(p);
    if (Ybuf[0]) cudaFree(Ybuf[0]);
    if (Ybuf[1]) cudaFree(Ybuf[1]);
    if (flags) cudaFree(flags);
  }
};
// The sharded operator inside a DMRG sweep: exchange buffers allocated once per solve at the largest window size; op[1] is
// the transposed operator of the symmetrised pair 0.5 (K + K^T) of dmrg.jl:241.
template <class T>
struct ShardCtxT {
  ShardOp<T> op[2];
  int rank = 0, nranks = 1;
  int64_t max_elems = 0;
};
}  // namespace ttn
struct ttn_shard_matvec_s : ttn::ByDtype<ttn::ShardOp> {};
struct ttn_shard_ctx_s : ttn::ByDtype<ttn::ShardCtxT> {};
typedef struct ttn_shard_matvec_s* ttn_shard_matvec;
typedef struct ttn_shard_ctx_s* ttn_shard_ctx;
namespace ttn {
// sharded matvec inside a sweep (shard.cu): persistent exchange buffers + per-window re-binding
ttn_shard_ctx shard_ctx_create(int dtype, int64_t max_elems, int rank, int nranks);
void shard_ctx_handles(ttn_shard_ctx c, void* out384);
void shard_ctx_bind(ttn_shard_ctx c, const void* all);
int shard_ctx_error(ttn_shard_ctx c);
// installs the sharded matvec on `lop` for the current window; false: the window is not sharded (too small), lop unchanged
template <class T> bool shard_install(ShardCtxT<T>& sc, LocalOp<T>& lop, const T* Lc, const T* Rc, const T* Wf);
// sharded effective operator (shard.cu)
void shard_range(int chi, int rank, int nranks, int* c0, int* cp);
ttn_shard_matvec shard_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                              const void* H, int rank, int nranks);
void shard_handles(ttn_shard_matvec mv, void* out192);
void shard_bind_handles(ttn_shard_matvec mv, const void* all);
void* shard_apply_any(ttn_shard_matvec mv, const void* V);
double shard_eigsolve(ttn_shard_matvec mv, void* x, int krylovdim, int maxiter, double tol, int* matvecs);
int shard_error(ttn_shard_matvec mv);
void shard_slice(ttn_shard_matvec mv, int* c0, int* cp);
ttn_matvec matvec2_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                          const void* H);
void matvec2_apply(ttn_matvec mv, const void* V, void* Y);
}  // namespace ttn
