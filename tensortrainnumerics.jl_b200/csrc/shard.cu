// Effective-operator matvec sharded over the GPUs of one NVLink/NVSwitch node (SURVEY.md §8(e), cfg4 large-chi row).
//
//   Y[a,b,c] = sum L[a,y,d] W[y,b,e,z] V[d,e,f] R[c,z,f]          (src/solvers/dmrg.jl:239-244, one application)
//
// Partition: the *spectator* bra index c of the right environment is cut into `nranks` contiguous slices; rank p keeps
// R[c_p, :, :], the full L and the full vector V.  Run from the right, all three contractions are local and
// reduction-free, and the slice Y[:, :, c_p] is one contiguous chunk of the column-major result:
//   T1[(d,e),(z,c_p)] = V[(d,e),f] * Rs[f,(z,c_p)]                    DMMA GEMM  (2 w n^2 chi^3 / nranks flop)
//   T2[(y,d),b,c_p]   = sum_(e,z) W[y,b,e,z] T1[d,(e,z),c_p]          small-K contraction (w^2 n^4 chi^2 / nranks), HBM-bound
//   Y[a,(b,c_p)]      = L[a,(y,d)] * T2[(y,d),(b,c_p)]                DMMA GEMM  (2 w n^2 chi^3 / nranks flop)
// The exchange step (the next Krylov vector must be complete on every rank) is fused into the last GEMM: its epilogue
// stores every finished tile to the own buffer AND to the mapped buffers of all peers (P2P stores over NVLink), so the
// all-gather overlaps the tensor-pipe work tile by tile and no separate collective is launched.  Completion is a
// per-rank epoch flag written to every peer after the GEMM and awaited before the result is consumed; the result
// buffers are double-buffered by epoch parity so that a rank running one matvec ahead never overwrites a vector a
// slower peer is still reading.  All Krylov vector algebra stays replicated (bit-identical on every rank), so no
// scalar all-reduce is needed.
#include <memory>
#include "solvers.h"

namespace ttn {

namespace {

// T2[y + w_l*(d + chi_l*(b + nn*c))] = sum_{e,z} Wq[(e + nn*z) + nn*w_r*(y + w_l*b)] * T1[d + chi_l*(e + nn*(z + w_r*c))]
template <class T, int KMAX>
__global__ void __launch_bounds__(128) mid_contract_kernel(const T* __restrict__ T1, const T* __restrict__ Wq, T* __restrict__ T2,
                                                           int chi_l, int nn, int w_l, int w_r, int cp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* ws = reinterpret_cast<T*>(smem_raw);
  const int kin = nn * w_r, kout = w_l * nn;
  for (int i = threadIdx.x; i < kin * kout; i += blockDim.x) ws[i] = Wq[i];
  __syncthreads();
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y;
  if (d >= chi_l) return;
  T in[KMAX];
  const T* src = T1 + d + (int64_t)chi_l * kin * c;
#pragma unroll
  for (int k = 0; k < KMAX; ++k)
    if (k < kin) in[k] = src[(int64_t)chi_l * k];
  T* dst = T2 + (int64_t)w_l * d + (int64_t)w_l * chi_l * nn * c;
  for (int b = 0; b < nn; ++b)
    for (int y = 0; y < w_l; ++y) {
      const T* wrow = ws + (size_t)kin * (y + w_l * b);
      T acc = t_zero<T>();
#pragma unroll
      for (int k = 0; k < KMAX; ++k)
        if (k < kin) t_fma(acc, wrow[k], in[k]);
      dst[y + (int64_t)w_l * chi_l * b] = acc;
    }
}

// epoch flag to every rank (system scope), issued after the GEMM whose epilogue carried the data
__global__ void shard_signal_kernel(unsigned* const* flag_peer, int nranks, int rank, unsigned epoch) {
  const int i = threadIdx.x;
  if (i >= nranks) return;
  __threadfence_system();
  volatile unsigned* f = flag_peer[i] + rank;
  *f = epoch;
  __threadfence_system();
}

// waits until every rank has published `epoch` in this rank's flag array; bounded spin (`timeout_ns` of the global timer,
// default 60 s, TTN_SHARD_TIMEOUT_S overrides) -> sticky error flag.  Once the flag is set the gathered vector is invalid:
// shard_eigsolve throws, and callers of ttn_shard_matvec_apply must poll ttn_shard_matvec_error before using Y.
__global__ void shard_wait_kernel(volatile unsigned* flags, int nranks, unsigned epoch, int* err, unsigned long long timeout_ns) {
  const int i = threadIdx.x;
  if (i >= nranks) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while ((int)(flags[i] - epoch) < 0) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > timeout_ns) { *err = 1; break; }
    __nanosleep(200);
  }
  __threadfence_system();
}

unsigned long long shard_timeout_ns() {
  static const unsigned long long v = [] {
    const char* e = getenv("TTN_SHARD_TIMEOUT_S");
    const double s = e ? atof(e) : 60.0;
    return (unsigned long long)((s > 0.001 ? s : 60.0) * 1e9);
  }();
  return v;
}

}  // namespace

// contiguous slice [c0, c0 + cp) of `chi` owned by `rank` (first chi % nranks ranks get one extra element)
void shard_range(int chi, int rank, int nranks, int* c0, int* cp) {
  const int base = chi / nranks, rem = chi % nranks;
  *cp = base + (rank < rem ? 1 : 0);
  *c0 = rank * base + std::min(rank, rem);
}

template <class T>
static void shard_setup(ShardOp<T>& op, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                        const void* H, int rank, int nranks) {
  ttn_assert(nranks >= 1 && nranks <= 8 && rank >= 0 && rank < nranks, 2, "shard: bad rank / nranks");
  ttn_assert(nn * w_r <= 32, 2, "shard: window too large for the mid contraction (n^N * w_r <= 32)");
  op.chi_l = chi_l; op.chi_r = chi_r; op.w_l = w_l; op.w_r = w_r; op.nn = nn; op.rank = rank; op.nranks = nranks;
  shard_range(chi_r, rank, nranks, &op.c0, &op.cp);
  ttn_assert(op.cp >= 1, 2, "shard: more ranks than bond indices");
  const size_t nl = (size_t)w_l * chi_l * chi_l, nr = (size_t)w_r * chi_r * chi_r, nw = (size_t)w_l * nn * nn * w_r;
  DevBuf Gd(sizeof(T) * nl), Hd(sizeof(T) * nr), Wd(sizeof(T) * nw);
  TTN_CUDA(cudaMemcpyAsync(Gd.p, G, Gd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(Hd.p, H, Hd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(Wd.p, Amid, Wd.bytes, cudaMemcpyHostToDevice, ctx().stream));
  // L2[a, (y,d)] = G[y,a,d]   (reference layout [mpo, bra, ket], dmrg.jl:32-35)
  op.L.alloc(sizeof(T) * nl);
  {
    Copy4 c;
    c.n0 = w_l; c.s0 = 1; c.d0 = chi_l;
    c.n1 = chi_l; c.s1 = w_l; c.d1 = 1;
    c.n2 = chi_l; c.s2 = (int64_t)w_l * chi_l; c.d2 = (int64_t)chi_l * w_l;
    copy4<T>(Gd.as<T>(), op.L.template as<T>(), c);
  }
  op.Lp = op.L.p;
  // Rs[f, z, c_loc] = H[z, c0 + c_loc, f]   (reference layout [mpo, bra, ket], dmrg.jl:27-30)
  op.Rs.alloc(sizeof(T) * (size_t)chi_r * w_r * op.cp);
  {
    Copy4 c;
    c.n0 = w_r; c.s0 = 1; c.d0 = chi_r;
    c.n1 = op.cp; c.s1 = w_r; c.d1 = (int64_t)chi_r * w_r;
    c.n2 = chi_r; c.s2 = (int64_t)w_r * chi_r; c.d2 = 1;
    copy4<T>(Hd.as<T>() + (int64_t)w_r * op.c0, op.Rs.template as<T>(), c);
  }
  // Wq[(e,z),(y,b)] = Amid[y,b,e,z]
  op.Wq.alloc(sizeof(T) * nw);
  {
    Copy4 c;
    c.n0 = w_l; c.s0 = 1; c.d0 = (int64_t)nn * w_r;
    c.n1 = nn; c.s1 = w_l; c.d1 = (int64_t)nn * w_r * w_l;
    c.n2 = nn; c.s2 = (int64_t)w_l * nn; c.d2 = 1;
    c.n3 = w_r; c.s3 = (int64_t)w_l * nn * nn; c.d3 = nn;
    copy4<T>(Wd.as<T>(), op.Wq.template as<T>(), c);
  }
  op.T1.alloc(sizeof(T) * (size_t)chi_l * nn * w_r * op.cp);
  op.T2.alloc(sizeof(T) * (size_t)w_l * chi_l * nn * op.cp);
  op.err.alloc(sizeof(int));
  TTN_CUDA(cudaMemsetAsync(op.err.p, 0, sizeof(int), ctx().stream));
  for (int i = 0; i < 2; ++i) {
    TTN_CUDA(cudaMalloc(&op.Ybuf[i], sizeof(T) * (size_t)op.size()));
    TTN_CUDA(cudaMemsetAsync(op.Ybuf[i], 0, sizeof(T) * (size_t)op.size(), ctx().stream));
  }
  TTN_CUDA(cudaMalloc((void**)&op.flags, sizeof(unsigned) * 8));
  TTN_CUDA(cudaMemsetAsync(op.flags, 0, sizeof(unsigned) * 8, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}

// Y slice of this rank; with peers bound the last GEMM also stores to every peer and the call returns after the
// epoch handshake has been queued (the wait is stream-ordered: later work on the stream sees the complete vector)
template <class T>
static T* shard_apply(ShardOp<T>& op, const T* V) {
  const int cl = op.chi_l, cr = op.chi_r, wl = op.w_l, wr = op.w_r, nn = op.nn, cp = op.cp;
  op.epoch++;
  const int par = op.epoch & 1;
  T* Y = reinterpret_cast<T*>(op.Ybuf[par]);
  {
    GemmArgs g;  // T1[(d,e),(z,c)] = V[(d,e),f] Rs[f,(z,c)]
    g.M = cl * nn; g.N = wr * cp; g.K = cr;
    g.A = V; g.sAm = 1; g.sAk = (int64_t)cl * nn;
    g.B = op.Rs.p; g.sBk = 1; g.sBn = cr;
    g.C = op.T1.p; g.sCm = 1; g.sCn = (int64_t)cl * nn;
    gemm<T>(g);
  }
  {
    ProfScope prof_scope_(KF_APPLY);
    dim3 grid((cl + 127) / 128, cp);
    const size_t smem = sizeof(T) * (size_t)nn * wr * wl * nn;
    mid_contract_kernel<T, 32><<<grid, 128, smem, ctx().stream>>>(op.T1.template as<T>(), op.Wq.template as<T>(), op.T2.template as<T>(), cl, nn, wl, wr, cp);
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
  {
    GemmArgs g;  // Y[a,(b,c)] = L[a,(y,d)] T2[(y,d),(b,c)]   (+ fused all-gather: peers get the same tiles)
    g.M = cl; g.N = nn * cp; g.K = wl * cl;
    g.A = op.Lp; g.sAm = 1; g.sAk = cl;
    g.B = op.T2.p; g.sBk = 1; g.sBn = (int64_t)wl * cl;
    g.C = Y + (int64_t)cl * nn * op.c0; g.sCm = 1; g.sCn = cl;
    if (op.bound) {
      for (int q = 0; q < op.nranks; ++q)
        if (q != op.rank) g.Cpeer[g.npeer++] = reinterpret_cast<T*>(op.Ypeer[par][q]) + (int64_t)cl * nn * op.c0;
    }
    gemm<T>(g);
  }
  if (op.bound && op.nranks > 1) {
    shard_signal_kernel<<<1, 32, 0, ctx().stream>>>(op.flag_peer_d.template as<unsigned*>(), op.nranks, op.rank, op.epoch);
    TTN_CHECK_LAUNCH();
    shard_wait_kernel<<<1, 32, 0, ctx().stream>>>(op.flags, op.nranks, op.epoch, op.err.template as<int>(), shard_timeout_ns());
    TTN_CHECK_LAUNCH();
    ctx().launches += 2;
  }
  return Y;
}

struct ShardHandles { cudaIpcMemHandle_t y[2]; cudaIpcMemHandle_t flags; };

template <class T>
static void shard_bind(ShardOp<T>& op, const ShardHandles* all, int stride = 1) {
  std::vector<unsigned*> fp(8, nullptr);
  for (int q = 0; q < op.nranks; ++q) {
    if (q == op.rank) {
      op.Ypeer[0][q] = op.Ybuf[0]; op.Ypeer[1][q] = op.Ybuf[1]; fp[q] = op.flags;
      continue;
    }
    for (int i = 0; i < 2; ++i) {
      void* p = nullptr;
      TTN_CUDA(cudaIpcOpenMemHandle(&p, all[q * stride].y[i], cudaIpcMemLazyEnablePeerAccess));
      op.opened.push_back(p);
      op.Ypeer[i][q] = p;
    }
    void* f = nullptr;
    TTN_CUDA(cudaIpcOpenMemHandle(&f, all[q * stride].flags, cudaIpcMemLazyEnablePeerAccess));
    op.opened.push_back(f);
    fp[q] = reinterpret_cast<unsigned*>(f);
  }
  op.flag_peer_d.alloc(sizeof(unsigned*) * 8);
  TTN_CUDA(cudaMemcpyAsync(op.flag_peer_d.p, fp.data(), sizeof(unsigned*) * 8, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  op.bound = true;
}

}  // namespace ttn

namespace ttn {

// ---------------------------------------------------------------------------------------------------------------------
// The sharded operator INSIDE a DMRG sweep (SURVEY.md section 8(e), cfg4): every rank runs the same sweep on identical data
// (environment updates and the two-site SVD are replicated); the Lanczos matvec of every bond step is sharded on the bra
// index of the right environment and exchanged through the fused all-gather epilogue.  The exchange buffers are allocated
// ONCE per solve at the largest window size and exported as CUDA IPC handles; per bond step the operator is re-bound to the
// sweep's device-resident environments (canonical layout E[bra, mpo, ket]): the left environment is used in place, the owned
// slice of the right environment and the fused MPO are re-laid out by two strided copies.  op[1] is the transposed operator
// of the symmetrised pair 0.5 (K + K^T) of dmrg.jl:241.
// ---------------------------------------------------------------------------------------------------------------------
template <class T>
static void shard_ctx_alloc(ShardCtxT<T>& c, int64_t max_elems, int rank, int nranks) {
  ttn_assert(nranks >= 1 && nranks <= 8 && rank >= 0 && rank < nranks && max_elems >= 1, 2, "shard ctx: bad arguments");
  c.rank = rank; c.nranks = nranks; c.max_elems = max_elems;
  for (int t = 0; t < 2; ++t) {
    ShardOp<T>& op = c.op[t];
    op.rank = rank; op.nranks = nranks;
    op.err.alloc(sizeof(int));
    TTN_CUDA(cudaMemsetAsync(op.err.p, 0, sizeof(int), ctx().stream));
    for (int i = 0; i < 2; ++i) {
      TTN_CUDA(cudaMalloc(&op.Ybuf[i], sizeof(T) * (size_t)max_elems));
      TTN_CUDA(cudaMemsetAsync(op.Ybuf[i], 0, sizeof(T) * (size_t)max_elems, ctx().stream));
    }
    TTN_CUDA(cudaMalloc((void**)&op.flags, sizeof(unsigned) * 8));
    TTN_CUDA(cudaMemsetAsync(op.flags, 0, sizeof(unsigned) * 8, ctx().stream));
  }
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}

// Re-binds op to the window (Lc: chi_l x w_l x chi_l, Rc: chi_r x w_r x chi_r, canonical layout; Wf: fused MPO in the
// reference Amid layout [y, b, e, z]).  transposed: the pieces of K^T.  false when the window cannot be sharded.
template <class T>
static bool shard_rebind(ShardOp<T>& op, int64_t max_elems, const T* Lc, int chi_l, int w_l, const T* Rc, int chi_r, int w_r,
                         const T* Wf, int nn, bool transposed) {
  if (chi_r < op.nranks || nn * w_r > 32 || (int64_t)chi_l * nn * chi_r > max_elems) return false;
  op.chi_l = chi_l; op.chi_r = chi_r; op.w_l = w_l; op.w_r = w_r; op.nn = nn;
  shard_range(chi_r, op.rank, op.nranks, &op.c0, &op.cp);
  if (!transposed) {
    op.Lp = Lc;                                   // L2[a,(y,d)] is the canonical layout itself
  } else {
    op.L.alloc(sizeof(T) * (size_t)chi_l * w_l * chi_l);
    Copy4 c;   // Lt[a,y,d] = L[d,y,a]
    c.n0 = chi_l; c.s0 = (int64_t)chi_l * w_l; c.d0 = 1;
    c.n1 = w_l; c.s1 = chi_l; c.d1 = chi_l;
    c.n2 = chi_l; c.s2 = 1; c.d2 = (int64_t)chi_l * w_l;
    copy4<T>(Lc, op.L.template as<T>(), c);
    op.Lp = op.L.p;
  }
  // Rs[f, z, c_loc] = R[c0 + c_loc, z, f]   (transposed: R[f, z, c0 + c_loc])
  op.Rs.alloc(sizeof(T) * (size_t)chi_r * w_r * op.cp);
  {
    Copy4 c;
    c.n0 = chi_r; c.d0 = 1;
    c.n1 = w_r; c.s1 = chi_r; c.d1 = chi_r;
    c.n2 = op.cp; c.d2 = (int64_t)chi_r * w_r;
    if (!transposed) { c.s0 = (int64_t)chi_r * w_r; c.s2 = 1; copy4<T>(Rc + op.c0, op.Rs.template as<T>(), c); }
    else { c.s0 = 1; c.s2 = (int64_t)chi_r * w_r; copy4<T>(Rc + (int64_t)op.c0 * chi_r * w_r, op.Rs.template as<T>(), c); }
  }
  // Wq[(e,z),(y,b)] = Amid[y,b,e,z]   (transposed: Amid[y,e,b,z])
  op.Wq.alloc(sizeof(T) * (size_t)w_l * nn * nn * w_r);
  {
    Copy4 c;
    c.n0 = w_l; c.s0 = 1; c.d0 = (int64_t)nn * w_r;                                   // y
    c.n1 = nn; c.s1 = transposed ? (int64_t)w_l * nn : w_l; c.d1 = (int64_t)nn * w_r * w_l;   // b
    c.n2 = nn; c.s2 = transposed ? w_l : (int64_t)w_l * nn; c.d2 = 1;                          // e
    c.n3 = w_r; c.s3 = (int64_t)w_l * nn * nn; c.d3 = nn;                                     // z
    copy4<T>(Wf, op.Wq.template as<T>(), c);
  }
  op.T1.alloc(sizeof(T) * (size_t)chi_l * nn * w_r * op.cp);
  op.T2.alloc(sizeof(T) * (size_t)w_l * chi_l * nn * op.cp);
  return true;
}

ttn_shard_matvec shard_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                              const void* H, int rank, int nranks) {
  auto mv = std::make_unique<ttn_shard_matvec_s>();
  mv->dtype = dtype;
  mv->visit([&](auto& op) { shard_setup(op, w_l, w_r, chi_l, chi_r, nn, G, Amid, H, rank, nranks); });
  return mv.release();
}

static void export_handles(void* const* yb, unsigned* fl, void* out) {
  ShardHandles h;
  TTN_CUDA(cudaIpcGetMemHandle(&h.y[0], yb[0]));
  TTN_CUDA(cudaIpcGetMemHandle(&h.y[1], yb[1]));
  TTN_CUDA(cudaIpcGetMemHandle(&h.flags, fl));
  memcpy(out, &h, sizeof(h));
}

void shard_handles(ttn_shard_matvec mv, void* out192) {
  ttn_assert(mv != nullptr && out192 != nullptr, 2, "null argument");
  static_assert(sizeof(ShardHandles) == 192, "three 64-byte IPC handles");
  mv->visit([&](auto& op) { export_handles(op.Ybuf, op.flags, out192); });
}

void shard_bind_handles(ttn_shard_matvec mv, const void* all) {
  ttn_assert(mv != nullptr && all != nullptr, 2, "null argument");
  mv->visit([&](auto& op) { shard_bind(op, reinterpret_cast<const ShardHandles*>(all)); });
}

void* shard_apply_any(ttn_shard_matvec mv, const void* V) {
  ttn_assert(mv != nullptr && V != nullptr, 2, "null argument");
  return with_dtype(mv->dtype, [&](auto t) -> void* {
    using T = decltype(t);
    return shard_apply<T>(mv->as<T>(), (const T*)V);
  });
}

template <class T>
static double shard_eig_t(ShardOp<T>& op, T* x, int krylovdim, int maxiter, double tol, int* matvecs) {
  LocalOp<T> lop;   // carrier of the vector shape; the three-GEMM chain is replaced by the sharded one
  lop.chi_l = op.chi_l; lop.chi_r = op.chi_r; lop.w_l = op.w_l; lop.w_r = op.w_r; lop.nn = op.nn;
  lop.ext_apply = [&op](const T* V, T* Y) {
    const T* Yp = shard_apply<T>(op, V);
    TTN_CUDA(cudaMemcpyAsync(Y, Yp, sizeof(T) * (size_t)op.size(), cudaMemcpyDeviceToDevice, ctx().stream));
  };
  KrylovInfo info;
  const double th = lanczos_lowest<T>(lop, x, krylovdim, maxiter, tol, &info);
  if (matvecs) *matvecs = info.matvecs;
  if (op.bound && op.nranks > 1) {
    int e = 0;
    read_back(&e, op.err.p, sizeof(int));
    if (e) throw Error(6, "sharded matvec: a peer did not publish its slice within the epoch timeout (TTN_SHARD_TIMEOUT_S); "
                          "the gathered vector and the eigenpair are invalid");
  }
  return th;
}

// lowest eigenpair of the sharded operator (KrylovKit.eigsolve stand-in of dmrg.jl:245); every rank runs the same
// replicated Lanczos recurrence on bit-identical vectors, only the matvec is distributed
double shard_eigsolve(ttn_shard_matvec mv, void* x, int krylovdim, int maxiter, double tol, int* matvecs) {
  ttn_assert(mv != nullptr && x != nullptr, 2, "null argument");
  return with_dtype(mv->dtype, [&](auto t) {
    using T = decltype(t);
    return shard_eig_t<T>(mv->as<T>(), (T*)x, krylovdim, maxiter, tol, matvecs);
  });
}

static int read_err(const DevBuf& err) {
  int e = 0;
  read_back(&e, err.p, sizeof(int));
  return e;
}

int shard_error(ttn_shard_matvec mv) {
  return mv->visit([](auto& op) { return read_err(op.err); });
}

void shard_slice(ttn_shard_matvec mv, int* c0, int* cp) {
  mv->visit([&](auto& op) { *c0 = op.c0; *cp = op.cp; });
}

ttn_shard_ctx shard_ctx_create(int dtype, int64_t max_elems, int rank, int nranks) {
  auto c = std::make_unique<ttn_shard_ctx_s>();
  c->dtype = dtype;
  c->visit([&](auto& sc) { shard_ctx_alloc(sc, max_elems, rank, nranks); });
  return c.release();
}
// 2 x 192 bytes: the IPC handles of the two operators' exchange buffers
void shard_ctx_handles(ttn_shard_ctx c, void* out384) {
  ttn_assert(c != nullptr && out384 != nullptr, 2, "null argument");
  c->visit([&](auto& sc) {
    for (int t = 0; t < 2; ++t) export_handles(sc.op[t].Ybuf, sc.op[t].flags, reinterpret_cast<char*>(out384) + t * sizeof(ShardHandles));
  });
}
void shard_ctx_bind(ttn_shard_ctx c, const void* all) {
  ttn_assert(c != nullptr && all != nullptr, 2, "null argument");
  const ShardHandles* hs = reinterpret_cast<const ShardHandles*>(all);
  c->visit([&](auto& sc) { for (int t = 0; t < 2; ++t) shard_bind(sc.op[t], hs + t, 2); });
}
int shard_ctx_error(ttn_shard_ctx c) {
  return c->visit([](auto& sc) { return read_err(sc.op[0].err) | read_err(sc.op[1].err); });
}

// installs the sharded matvec on `lop` for the current window; false: the window is not sharded (too small), lop unchanged
template <class T>
bool shard_install(ShardCtxT<T>& sc, LocalOp<T>& lop, const T* Lc, const T* Rc, const T* Wf) {
  if (sc.nranks <= 1 || !sc.op[0].bound || lop.zero_site) return false;
  if (!shard_rebind<T>(sc.op[0], sc.max_elems, Lc, lop.chi_l, lop.w_l, Rc, lop.chi_r, lop.w_r, Wf, lop.nn, false)) return false;
  const bool sym = lop.symmetrize;
  if (sym && !shard_rebind<T>(sc.op[1], sc.max_elems, Lc, lop.chi_l, lop.w_l, Rc, lop.chi_r, lop.w_r, Wf, lop.nn, true)) return false;
  const int64_t nel = lop.size();
  lop.ext_apply = [&sc, sym, nel](const T* V, T* Y) {
    const T* Y1 = shard_apply<T>(sc.op[0], V);
    TTN_CUDA(cudaMemcpyAsync(Y, Y1, sizeof(T) * (size_t)nel, cudaMemcpyDeviceToDevice, ctx().stream));
    if (sym) {
      const T* Y2 = shard_apply<T>(sc.op[1], V);
      axpy<T>(nel, t_one<T>(), Y2, Y);
      scal<T>(nel, t_from<T>(0.5, 0.0), Y);
    }
  };
  return true;
}
template bool shard_install<double>(ShardCtxT<double>&, LocalOp<double>&, const double*, const double*, const double*);
template bool shard_install<zc>(ShardCtxT<zc>&, LocalOp<zc>&, const zc*, const zc*, const zc*);

}  // namespace ttn
