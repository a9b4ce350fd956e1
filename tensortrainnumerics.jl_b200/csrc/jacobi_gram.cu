// Gram-block one-sided Jacobi SVD on the FP64 tensor pipe, for bond matrices too large for one SM / one cluster
// (DMRG and MALS core moves at chi >= 256: svd of (r_l n) x (n r_r), src/solvers/dmrg.jl:189,213, mals.jl:99,126;
// tdvp2 tdvp.jl:250,278).  Same contract as jacobi_kernel (jacobi.cu): X <- X V, columns orthogonal on exit.
//
// The n columns are cut into blocks of 32; a sweep is a round-robin tournament of the blocks (circle method), and one
// step treats n/64 disjoint block pairs concurrently with three kernels:
//   1. gram_pairs_kernel  : G_k = P_k^H P_k for every 64-column panel P_k = [X_i X_j]   — DMMA, split over the rows;
//   2. gram_eig_kernel    : one two-sided Jacobi pass over the cross pairs of the 64 x 64 Hermitian G_k in shared memory, rotations
//                           accumulated in V_k (the plane rotations are the ones the scalar method would apply to the
//                           columns, but each costs 64-vectors instead of m-vectors);
//   3. update_pairs_kernel: P_k <- P_k V_k in place                                      — DMMA.
// The O(m n^2) work per sweep runs as GEMM tiles (8 m n^2 flop per sweep at ~70 % of the DMMA peak) instead of scalar
// rotations bound by shared-memory bandwidth and shuffle latency (jacobi_cross_kernel: FP64 pipe 22 % busy, profiles/ncu_dmrg_svd_r01.txt).
// Entries of G are inner products of the actual columns, i.e. accurate relative to ||x_p|| ||x_q||, and two-sided Jacobi
// on a positive definite matrix is relatively accurate (Demmel-Veselic), so the rotation threshold stays the relative
// one, |x_p^H x_q| <= tol ||x_p|| ||x_q||, evaluated on a freshly computed Gram matrix at every step.
#include "ttn_internal.h"
#include "dmma.h"

namespace ttn {
namespace {

constexpr int GB = 32;        // block width
constexpr int PW = 2 * GB;    // panel width (columns of a block pair)
constexpr int GT = 256;       // threads per CTA
constexpr int GK = 32;        // rows per staged slab in the Gram kernel
constexpr int UM = 128;       // rows per CTA tile in the update kernel
constexpr int GE = 1024;      // threads of the inner eigen-sweep kernel (one 2 x 2 block of G per thread)

// column j of panel (blkA, blkB): pointer to its first row, or nullptr beyond the matrix
template <class T>
__device__ __forceinline__ T* panel_col(T* X, int64_t ldx, int n, int blkA, int blkB, int j) {
  if (j >= GB && blkB < 0) return nullptr;           // single-block panel (intra-block step)
  const int c = (j < GB ? blkA * GB + j : blkB * GB + (j - GB));
  return c < n ? X + (int64_t)c * ldx : nullptr;
}

// ---------------------------------------------------------------------------------------------------------------------
// 1. Gram matrices of all panels of a step.  grid (npairs, nsplit); CTA (k, z) accumulates rows [z*mc, (z+1)*mc).
// ---------------------------------------------------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(GT) gram_pairs_kernel(const T* __restrict__ X, int m, int n, int64_t ldx,
                                                        const int* __restrict__ pairA, const int* __restrict__ pairB,
                                                        int mc, T* __restrict__ Gp) {
  constexpr int PITCH = GK + 4;                       // == 4 mod 16: conflict-free m8n8k4 fragment loads
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* S = reinterpret_cast<T*>(smem_raw);              // [2][PW][PITCH]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g8 = lane >> 2, t4 = lane & 3;
  const int blkA = pairA[blockIdx.x], blkB = pairB[blockIdx.x];
  const int r0 = blockIdx.y * mc, r1 = min(m, r0 + mc);
  const int wm0 = (warp & 1) * 32, wn0 = (warp >> 1) * 16;
  const int lk = tid & 31, lc0 = tid >> 5;            // loader: row lk of the slab, columns lc0 + 8 i

  const T* colp[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) colp[i] = panel_col<T>(const_cast<T*>(X), ldx, n, blkA, blkB, lc0 + 8 * i);

  Acc<T> acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) acc[i][j].zero();

  T stage[8];
  auto load_slab = [&](int k0) {
    const int row = k0 + lk;
#pragma unroll
    for (int i = 0; i < 8; ++i) stage[i] = (colp[i] != nullptr && row < r1) ? colp[i][row] : t_zero<T>();
  };
  auto store_slab = [&](int buf) {
    T* s = S + (size_t)buf * PW * PITCH;
#pragma unroll
    for (int i = 0; i < 8; ++i) s[(lc0 + 8 * i) * PITCH + lk] = stage[i];
  };
  const int nslab = (r1 - r0 + GK - 1) / GK;
  if (nslab > 0) { load_slab(r0); store_slab(0); }
  __syncthreads();
  for (int sl = 0; sl < nslab; ++sl) {
    const int buf = sl & 1;
    if (sl + 1 < nslab) load_slab(r0 + (sl + 1) * GK);
    const T* s = S + (size_t)buf * PW * PITCH;
#pragma unroll
    for (int kk = 0; kk < GK; kk += 4) {
      T af[4], bf[2];
#pragma unroll
      for (int i = 0; i < 4; ++i) af[i] = t_conj(s[(wm0 + 8 * i + g8) * PITCH + kk + t4]);
#pragma unroll
      for (int j = 0; j < 2; ++j) bf[j] = s[(wn0 + 8 * j + g8) * PITCH + kk + t4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) acc[i][j].mma(af[i], bf[j]);
    }
    if (sl + 1 < nslab) store_slab(buf ^ 1);
    __syncthreads();
  }
  T* out = Gp + ((size_t)blockIdx.x * gridDim.y + blockIdx.y) * PW * PW;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int row = wm0 + 8 * i + g8, col = wn0 + 8 * j + 2 * t4 + e;
        out[(size_t)col * PW + row] = acc[i][j].get(e);
      }
}

// ---------------------------------------------------------------------------------------------------------------------
// 2. Two-sided Jacobi on the 64 x 64 Gram matrix of every panel; V accumulates the rotations.  grid (npairs).
// ---------------------------------------------------------------------------------------------------------------------
// cross_only: the panel is [A | B] and only the 32 x 32 pairs (p in A, q in B) are rotated, 32 steps of 32 disjoint pairs
// (p, 32 + (p + s) mod 32) — every column pair of the matrix is then rotated exactly once per sweep; otherwise a full
// round-robin over the 64 panel columns (used for the intra-block step, where B is empty).
template <class T, int ET>
__global__ void __launch_bounds__(ET) gram_eig_kernel(const T* __restrict__ Gp, int nsplit, int cross_only, double tol,
                                                      T* __restrict__ Vg, int* __restrict__ skip, unsigned int* __restrict__ d_rotated) {
  constexpr int P = PW + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* G = reinterpret_cast<T*>(smem_raw);      // [PW][P]
  T* V = G + PW * P;                          // [PW][P]
  __shared__ double s_cs[GB];
  __shared__ T s_sn[GB];
  __shared__ int s_p[GB], s_q[GB];
  __shared__ int s_any, s_big, s_step[2];
  const int tid = threadIdx.x;
  const double tol2 = tol * tol;
  const T* gp = Gp + (size_t)blockIdx.x * nsplit * PW * PW;
  for (int idx = tid; idx < PW * PW; idx += ET) {
    T a = t_zero<T>();
    T v[4];
    for (int z0 = 0; z0 < nsplit; z0 += 4) {           // four partial loads in flight
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = (z0 + u < nsplit) ? gp[(size_t)(z0 + u) * PW * PW + idx] : t_zero<T>();
#pragma unroll
      for (int u = 0; u < 4; ++u) a = t_add(a, v[u]);
    }
    const int i = idx % PW, j = idx / PW;
    G[i * P + j] = a;
    V[i * P + j] = i == j ? t_one<T>() : t_zero<T>();
  }
  if (tid == 0) { s_any = 0; s_big = 0; s_step[0] = 0; s_step[1] = 0; }
  __syncthreads();

  int gs = 0;   // global step counter: its parity selects the rotation flag slot
  {
    const int nsteps = cross_only ? GB : PW - 1;
    for (int r = 0; r < nsteps; ++r, ++gs) {
      if (tid < GB) {
        int p, q;
        if (cross_only) { p = tid; q = GB + ((tid + r) & (GB - 1)); }
        else if (tid == 0) { p = PW - 1; q = r; }
        else { p = r + tid; if (p >= PW - 1) p -= PW - 1; q = r - tid; if (q < 0) q += PW - 1; }
        if (p > q) { const int t_ = p; p = q; q = t_; }
        const double a = t_real(G[p * P + p]), b = t_real(G[q * P + q]);
        const T c = G[p * P + q];
        const double cr = t_real(c), ci = t_imag(c);
        const double cc = cr * cr + ci * ci;
        double cs = 1.0;
        T sn = t_zero<T>();
        if (cc > tol2 * fmax(a, 0.0) * fmax(b, 0.0) && a > 0.0 && b > 0.0 && cc > 1e-290) {
          const double tau = 0.5 * (b - a);
          const double z = tau * tau + cc;
          const double h = z * rsqrt(z);
          const double d = tau + (tau >= 0.0 ? h : -h);
          const double rinv = rsqrt(d * d + cc);
          cs = fabs(d) * rinv;
          const double f = (d >= 0.0 ? 1.0 : -1.0) * rinv;      // sn * phase = sign(d) c / sqrt(d^2 + |c|^2)
          sn = t_from<T>(cr * f, ci * f);
          s_step[gs & 1] = 1;
          // "big" rotation: not yet second order (see rotate_pair in jacobi_cluster.cu) -> a further sweep is needed
          if (cc > 1e-18 * a * b || cc * f * f > 1e-10) s_big = 1;
        }
        s_cs[tid] = cs; s_sn[tid] = sn; s_p[tid] = p; s_q[tid] = q;
      }
      __syncthreads();
      const int stepped = s_step[gs & 1];
      if (tid == 0) { s_step[(gs + 1) & 1] = 0; if (stepped) s_any = 1; }   // the other slot is idle during this phase
      if (stepped && cross_only && ET == GB * GB) {
        // cross ordering: pair i is (i, 32 + (i + r) mod 32), so the column indices need no shared-memory reads; one
        // 2 x 2 block of G and two rows of V per thread (the kernel is bound by shared-memory instruction issue)
        const int k = tid >> 5, l = tid & (GB - 1);
        const int pk = k, qk = GB + ((k + r) & (GB - 1)), pl = l, ql = GB + ((l + r) & (GB - 1));
        const double ck = s_cs[k], cl = s_cs[l];
        const T sk = s_sn[k], sl = s_sn[l];
        const T b00 = G[pk * P + pl], b01 = G[pk * P + ql], b10 = G[qk * P + pl], b11 = G[qk * P + ql];
        const T slc = t_conj(sl), skc = t_conj(sk);
        const T t00 = t_sub(t_scale(b00, cl), t_mul(b01, slc)), t01 = t_add(t_mul(b00, sl), t_scale(b01, cl));
        const T t10 = t_sub(t_scale(b10, cl), t_mul(b11, slc)), t11 = t_add(t_mul(b10, sl), t_scale(b11, cl));
        G[pk * P + pl] = t_sub(t_scale(t00, ck), t_mul(sk, t10));
        G[pk * P + ql] = t_sub(t_scale(t01, ck), t_mul(sk, t11));
        G[qk * P + pl] = t_add(t_mul(skc, t00), t_scale(t10, ck));
        G[qk * P + ql] = t_add(t_mul(skc, t01), t_scale(t11, ck));
        // V <- V J: rows i = k and i = k + 32 of column pair l (same l: its rotation is already in registers)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int i = k + h * GB;
          const T vp = V[i * P + pl], vq = V[i * P + ql];
          V[i * P + pl] = t_sub(t_scale(vp, cl), t_mul(vq, slc));
          V[i * P + ql] = t_add(t_mul(vp, sl), t_scale(vq, cl));
        }
      } else if (stepped) {
        // G <- J^H G J on the 32 x 32 grid of 2 x 2 blocks (rows of pair k, columns of pair l); J = [[cs, s], [-conj(s), cs]]
#pragma unroll
        for (int it = 0; it < (GB * GB) / ET; ++it) {
          const int bidx = tid + it * ET;
          const int k = bidx / GB, l = bidx % GB;
          const int pk = s_p[k], qk = s_q[k], pl = s_p[l], ql = s_q[l];
          const double ck = s_cs[k], cl = s_cs[l];
          const T sk = s_sn[k], sl = s_sn[l];
          const T b00 = G[pk * P + pl], b01 = G[pk * P + ql], b10 = G[qk * P + pl], b11 = G[qk * P + ql];
          const T slc = t_conj(sl);
          const T t00 = t_sub(t_scale(b00, cl), t_mul(b01, slc)), t01 = t_add(t_mul(b00, sl), t_scale(b01, cl));
          const T t10 = t_sub(t_scale(b10, cl), t_mul(b11, slc)), t11 = t_add(t_mul(b10, sl), t_scale(b11, cl));
          const T skc = t_conj(sk);
          G[pk * P + pl] = t_sub(t_scale(t00, ck), t_mul(sk, t10));
          G[pk * P + ql] = t_sub(t_scale(t01, ck), t_mul(sk, t11));
          G[qk * P + pl] = t_add(t_mul(skc, t00), t_scale(t10, ck));
          G[qk * P + ql] = t_add(t_mul(skc, t01), t_scale(t11, ck));
        }
        // V <- V J
#pragma unroll
        for (int it = 0; it < (PW * GB) / ET; ++it) {
          const int vidx = tid + it * ET;
          const int i = vidx % PW, l = vidx / PW;
          const int pl = s_p[l], ql = s_q[l];
          const double cl = s_cs[l];
          const T sl = s_sn[l];
          const T vp = V[i * P + pl], vq = V[i * P + ql];
          V[i * P + pl] = t_sub(t_scale(vp, cl), t_mul(vq, t_conj(sl)));
          V[i * P + ql] = t_add(t_mul(vp, sl), t_scale(vq, cl));
        }
      }
      __syncthreads();
    }
  }
  const int any = s_any;
  T* vout = Vg + (size_t)blockIdx.x * PW * PW;
  if (any)
    for (int idx = tid; idx < PW * PW; idx += ET) vout[idx] = V[(idx % PW) * P + idx / PW];   // column-major V[k + 64 n]
  if (tid == 0) {
    skip[blockIdx.x] = any ? 0 : 1;
    if (any) atomicOr(d_rotated, s_big ? 3u : 1u);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// 3. P_k <- P_k V_k in place.  grid (npairs, ceil(m / UM)).
// ---------------------------------------------------------------------------------------------------------------------
// The UM = 128 rows of a CTA tile are processed as two halves of 64: both halves (and V) are requested with cp.async up
// front, the DMMA work on the first half and its write-back overlap the arrival of the second.
template <class T>
__global__ void __launch_bounds__(GT) update_pairs_kernel(T* __restrict__ X, int m, int n, int64_t ldx,
                                                          const int* __restrict__ pairA, const int* __restrict__ pairB,
                                                          const T* __restrict__ Vg, const int* __restrict__ skip) {
  if (skip[blockIdx.x]) return;
  constexpr int UH = UM / 2;                 // rows per half tile
  constexpr int PA = UH + 4, PB = PW + 4;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* As = reinterpret_cast<T*>(smem_raw);   // [2][PW][PA]  As[h][k][row]
  T* Bs = As + 2 * PW * PA;                 // [PW][PB]     Bs[k][ncol]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g8 = lane >> 2, t4 = lane & 3;
  const int blkA = pairA[blockIdx.x], blkB = pairB[blockIdx.x];
  const int row0 = blockIdx.y * UM;
  {
    const T* vg = Vg + (size_t)blockIdx.x * PW * PW;
    const int k = tid & (PW - 1), n0 = tid / PW;             // 4 column phases
#pragma unroll 4
    for (int i = 0; i < PW / 4; ++i) {
      const int nc = n0 + 4 * i;
      cp_async_elem<T>(Bs + k * PB + nc, vg + (size_t)nc * PW + k, true);
    }
    const int row = tid & (UH - 1), c0 = tid / UH;           // 4 column phases of 64 rows
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const bool rok = row0 + h * UH + row < m;
#pragma unroll 4
      for (int i = 0; i < PW / 4; ++i) {
        const int c = c0 + 4 * i;
        const T* cp = panel_col<T>(X, ldx, n, blkA, blkB, c);
        const bool ok = cp != nullptr && rok;
        cp_async_elem<T>(As + (size_t)h * PW * PA + c * PA + row, ok ? cp + row0 + h * UH + row : X, ok);
      }
      cp_async_commit();                                      // group 0: V + half 0, group 1: half 1
    }
  }
  const int wm0 = (warp & 1) * 32, wn0 = (warp >> 1) * 16;    // 2 x 4 warps over the 64 x 64 half tile
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (h == 0) cp_async_wait<1>(); else cp_async_wait<0>();
    __syncthreads();
    const T* as = As + (size_t)h * PW * PA;
    Acc<T> acc[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) acc[i][j].zero();
#pragma unroll 4
    for (int kk = 0; kk < PW; kk += 4) {
      T af[4], bf[2];
#pragma unroll
      for (int i = 0; i < 4; ++i) af[i] = as[(kk + t4) * PA + wm0 + 8 * i + g8];
#pragma unroll
      for (int j = 0; j < 2; ++j) bf[j] = Bs[(kk + t4) * PB + wn0 + 8 * j + g8];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) acc[i][j].mma(af[i], bf[j]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = wn0 + 8 * j + 2 * t4 + e;
        T* cp = panel_col<T>(X, ldx, n, blkA, blkB, col);
        if (cp == nullptr) continue;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = row0 + h * UH + wm0 + 8 * i + g8;
          if (row < m) cp[row] = acc[i][j].get(e);
        }
      }
  }
}

}  // namespace

// Orthogonalises the n columns of X (m x n, one matrix); returns the number of sweeps, or -1 if the shape is not served.
template <class T>
int jacobi_gram(T* X, int m, int n, int64_t ldx, double tol, int max_sweeps) {
  if (n < 2 * PW || m < PW) return -1;
  const int nblk = (n + GB - 1) / GB;
  const int ne = nblk + (nblk & 1);
  // pair lists of every tournament step (circle method), uploaded once
  std::vector<int> hA, hB, off(ne, 0);
  for (int r = 0; r < ne - 1; ++r) {
    for (int i = 0; i < ne / 2; ++i) {
      int p, q;
      if (i == 0) { p = ne - 1; q = r; }
      else { p = (r + i) % (ne - 1); q = (r - i + (ne - 1)) % (ne - 1); }
      if (p < nblk && q < nblk) { hA.push_back(std::min(p, q)); hB.push_back(std::max(p, q)); }
    }
    off[r + 1] = (int)hA.size();
  }
  // intra-block step: every block alone (B = -1), full round-robin inside the kernel
  const int off_diag = (int)hA.size();
  for (int i = 0; i < nblk; ++i) { hA.push_back(i); hB.push_back(-1); }
  const int maxpairs = std::max(ne / 2, nblk);
  // Two pair groups per step on two streams: while the (few, latency-bound) inner eigen-sweep CTAs of one group run, the
  // DMMA Gram / update tiles of the other fill the remaining SMs.  Each group has its own Gram / V / skip buffers
  // and its own split of the rows sized for ~2 CTAs per SM.
  constexpr int NG = 2;
  static cudaStream_t strm[NG] = {nullptr, nullptr};   // strm[0] is the library stream
  static cudaEvent_t ev_grp[NG], ev_join = nullptr;
  static int strm_dev = -1;   // streams and events belong to a device: rebuild them when ttn_init re-binds the library
  if (ev_join != nullptr && strm_dev != ctx().device) {
    for (int g = 1; g < NG; ++g) { cudaStreamDestroy(strm[g]); strm[g] = nullptr; }
    for (int g = 0; g < NG; ++g) cudaEventDestroy(ev_grp[g]);
    cudaEventDestroy(ev_join);
    ev_join = nullptr;
  }
  if (ev_join == nullptr) {
    strm_dev = ctx().device;
    for (int g = 1; g < NG; ++g) TTN_CUDA(cudaStreamCreateWithFlags(&strm[g], cudaStreamNonBlocking));
    for (int g = 0; g < NG; ++g) TTN_CUDA(cudaEventCreateWithFlags(&ev_grp[g], cudaEventDisableTiming));
    TTN_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
  }
  strm[0] = ctx().stream;
  const int grpmax = (maxpairs + NG - 1) / NG;
  auto split_for = [&](int cnt, int& ns, int& mcs) {
    ns = std::max(1, std::min((2 * ctx().sm_count + cnt - 1) / std::max(cnt, 1), m / (2 * GK)));
    ns = std::min(ns, 16);
    mcs = (m + ns - 1) / ns;
    mcs = (mcs + GK - 1) / GK * GK;
    ns = (m + mcs - 1) / mcs;
  };
  const size_t gp_elems = (size_t)grpmax * 16 * PW * PW;          // <= 16 row splits
  DevBuf gA(sizeof(int) * hA.size()), gB(sizeof(int) * hB.size());
  DevBuf Gp[NG], Vg[NG], skip[NG], rot(sizeof(unsigned int));
  for (int g = 0; g < NG; ++g) {
    Gp[g].alloc(sizeof(T) * gp_elems);
    Vg[g].alloc(sizeof(T) * (size_t)grpmax * PW * PW);
    skip[g].alloc(sizeof(int) * grpmax);
  }
  TTN_CUDA(cudaMemcpyAsync(gA.p, hA.data(), sizeof(int) * hA.size(), cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(gB.p, hB.data(), sizeof(int) * hB.size(), cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));   // host staging vectors must outlive the copies
  const size_t smem_g = sizeof(T) * 2 * PW * (GK + 4);
  const size_t smem_u = sizeof(T) * ((size_t)2 * PW * (UM / 2 + 4) + (size_t)PW * (PW + 4));
  const size_t smem_e = sizeof(T) * 2 * PW * (PW + 1);
  static int attr_dev = -1;   // function attributes are per device (ttn_init may re-bind)
  if (attr_dev != ctx().device) {
    TTN_CUDA(cudaFuncSetAttribute(gram_eig_kernel<T, GE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_e));
    TTN_CUDA(cudaFuncSetAttribute(gram_pairs_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g));
    TTN_CUDA(cudaFuncSetAttribute(update_pairs_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_u));
    attr_dev = ctx().device;
  }
  int sweeps = 0;
  auto group = [&](int g, const int* pa, const int* pb, int cnt, int cross) {
    if (cnt <= 0) return;
    cudaStream_t st = strm[g];
    int ns, mcs;
    split_for(cnt, ns, mcs);
    gram_pairs_kernel<T><<<dim3(cnt, ns), GT, smem_g, st>>>(X, m, n, ldx, pa, pb, mcs, Gp[g].as<T>());
    TTN_CHECK_LAUNCH();
    gram_eig_kernel<T, GE><<<cnt, GE, smem_e, st>>>(Gp[g].as<T>(), ns, cross, tol, Vg[g].as<T>(), skip[g].as<int>(), rot.as<unsigned int>());
    TTN_CHECK_LAUNCH();
    update_pairs_kernel<T><<<dim3(cnt, (m + UM - 1) / UM), GT, smem_u, st>>>(X, m, n, ldx, pa, pb, Vg[g].as<T>(), skip[g].as<int>());
    TTN_CHECK_LAUNCH();
    ctx().launches += 3;
  };
  // join: the library stream waits for every group, then every group stream waits for the library stream
  auto join = [&]() {
    for (int g = 1; g < NG; ++g) {
      TTN_CUDA(cudaEventRecord(ev_grp[g], strm[g]));
      TTN_CUDA(cudaStreamWaitEvent(strm[0], ev_grp[g], 0));
    }
    TTN_CUDA(cudaEventRecord(ev_join, strm[0]));
    for (int g = 1; g < NG; ++g) TTN_CUDA(cudaStreamWaitEvent(strm[g], ev_join, 0));
  };
  // one tournament step: the pairs are dealt to the groups in contiguous chunks, all groups run concurrently
  auto step = [&](const int* pa, const int* pb, int cnt, int cross) {
    const int per = (cnt + NG - 1) / NG;
    for (int g = 0; g < NG; ++g) {
      const int lo = g * per, c = std::min(per, cnt - lo);
      group(g, pa + lo, pb + lo, c, cross);
    }
    join();
  };
  ProfScope prof_scope_(KF_JACOBI);                  // (per-kernel families are not separable across the streams)
  for (int sw = 0; sw < max_sweeps; ++sw) {
    TTN_CUDA(cudaMemsetAsync(rot.p, 0, sizeof(unsigned int), ctx().stream));
    join();                                           // group streams start after everything queued so far
    step(gA.as<int>() + off_diag, gB.as<int>() + off_diag, nblk, 0);          // pairs inside each block
    for (int st = 0; st < ne - 1; ++st) {                                      // cross pairs of the block tournament
      const int cnt = off[st + 1] - off[st];
      if (cnt > 0) step(gA.as<int>() + off[st], gB.as<int>() + off[st], cnt, 1);
    }
    unsigned int rotated = 0;
    read_back(&rotated, rot.p, sizeof(rotated));
    sweeps = sw + 1;
    // bit 1 = some rotation of this sweep was not yet of second order; without one, what is left after the sweep is below the
    // tolerance and the confirming sweep (6 ms at 2048^2) is skipped, as in the cluster kernel
    if (!(rotated & 2u)) break;
  }
  return sweeps;
}

template int jacobi_gram<double>(double*, int, int, int64_t, double, int);
template int jacobi_gram<zc>(zc*, int, int, int64_t, double, int);

}  // namespace ttn
