// One-sided Jacobi SVD of ONE bond-sized matrix spread over a thread-block cluster (8 SMs, distributed shared memory).
//
// Same contract as jacobi_kernel (jacobi.cu): X <- X V with orthogonal columns, used behind `_svdtrunc`
// (src/tt_cross_interpolation.jl:150) / `svd` in the MALS, DMRG and TDVP core moves (mals.jl:99,126, dmrg.jl:189,213,
// tdvp.jl:250,278) when there is a single matrix (or a handful) to factor: a TT-rounding sweep (tt_tools.jl:743-789)
// is a chain of such SVDs, so its speed is the latency of one SVD, and one SM cannot go below ~1.5 ms for 128 columns
// (profiles/ncu_jacobi_r01.txt: FP64 pipe 33 % busy, the rest is dependent-issue latency over 64 pairs per step).
//
// Layout.  The n columns are cut into 2*CL blocks of W columns (CL = 8 CTAs of the cluster); every CTA owns two blocks
// ("top", "bottom") in its shared memory.  A sweep is a round-robin tournament of the 2*CL blocks (2*CL-1 block steps):
//   block step 0      : all pairs among the 2W local columns (intra-block + cross), 2W-1 local steps of W disjoint pairs;
//   block steps 1..   : the W*W cross pairs between the two resident blocks, W local steps of W disjoint pairs;
// after each block step every column is written straight into the shared memory of the CTA that owns it next
// (st.shared::cluster through DSMEM; circle method: top_0 fixed, the other 2*CL-1 block slots rotate), followed by one
// cluster barrier.  One lane group (GL lanes) owns a pair: RPL rows of both columns per lane in registers, the inner
// product reduced by shuffles, maintained squared norms travelling with the columns, division-free rotations.
// 127 local steps per sweep at n = 128 as in any parallel ordering, but each step is 8 pairs per SM instead of 64.
#include "ttn_internal.h"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace ttn {
namespace {

constexpr int JC_MAX_SWEEPS = 40;

// destination (cta, slot) of block slot (c, top?) after one block step of the circle method
template <int CL>
__device__ __forceinline__ void next_slot(int c, bool top, int& dc, bool& dtop) {
  if (top) {
    if (c == 0) { dc = 0; dtop = true; }
    else if (c == CL - 1) { dc = CL - 1; dtop = false; }
    else { dc = c + 1; dtop = true; }
  } else {
    if (c == 0) { dc = 1; dtop = true; }
    else { dc = c - 1; dtop = false; }
  }
}


// One plane rotation of the column pair held in registers (rp, rq: RPL rows per lane of a GL-lane group) with maintained
// squared norms an, bn.  Returns 0 (skipped), 1 (rotated, |x_p^H x_q|^2 <= 1e-18 a b and sin^2 <= 1e-10) or 2 (rotated).
template <class T, int GL, int RPL>
__device__ __forceinline__ int rotate_pair(T (&rp)[RPL], T (&rq)[RPL], double& an, double& bn, double tol2) {
  T c2v[2] = {t_zero<T>(), t_zero<T>()};
#pragma unroll
  for (int k = 0; k < RPL; ++k) t_fma(c2v[k & 1], t_conj(rp[k]), rq[k]);
  const T c = t_add(c2v[0], c2v[1]);
  double cr = t_real(c), ci = t_imag(c);
#pragma unroll
  for (int o = GL / 2; o > 0; o >>= 1) {
    cr += __shfl_xor_sync(0xffffffffu, cr, o);
    if (is_cplx<T>::value) ci += __shfl_xor_sync(0xffffffffu, ci, o);
  }
  const double cc = cr * cr + ci * ci;
  const double ab = an * bn;
  if (!(cc > tol2 * ab) || !(an > 0.0) || !(bn > 0.0)) return 0;   // group-uniform; zero columns, NaNs
  double absc, phr, phi;
  if (is_cplx<T>::value) {
    const double inv = rsqrt(cc);
    absc = cc * inv; phr = cr * inv; phi = ci * inv;
  } else {
    absc = fabs(cr); phr = cr >= 0.0 ? 1.0 : -1.0; phi = 0.0;
  }
  // tau = (b-a)/2, h = sqrt(tau^2+|c|^2), d = tau + sign(tau) h: cs = |d|/sqrt(d^2+|c|^2), sn = sign(d)|c|/sqrt(d^2+|c|^2)
  const double tau = 0.5 * (bn - an);
  const double z = tau * tau + cc;
  const double h = z * rsqrt(z);
  const double d = tau + (tau >= 0.0 ? h : -h);
  const double rinv = rsqrt(d * d + cc);
  const double cs = fabs(d) * rinv;
  const double sn = (d >= 0.0 ? absc : -absc) * rinv;
  const double x2 = 2.0 * cs * sn * absc;
  const double an_new = fmax(cs * cs * an - x2 + sn * sn * bn, 0.0);
  bn = fmax(sn * sn * an + x2 + cs * cs * bn, 0.0);
  an = an_new;
  const T ph = t_from<T>(sn * phr, sn * phi);
  const T phc = t_from<T>(sn * phr, -sn * phi);
#pragma unroll
  for (int k = 0; k < RPL; ++k) {
    const T pv = rp[k], qv = rq[k];
    rp[k] = t_sub(t_scale(pv, cs), t_mul(phc, qv));
    rq[k] = t_add(t_mul(ph, pv), t_scale(qv, cs));
  }
  // level 1 = "second-order" rotation: the pair was orthogonal to ~1e-9 AND the angle is small.  A large angle (clustered or
  // degenerate singular values: tan 2θ = 2|c|/(b-a)) re-fills already-zeroed inner products (p,k) with sn * (q,k), which stays
  // below the tolerance m*eps/2 only when |sn| <~ 1e-5 — so such a rotation still asks for a confirming sweep.
  return (cc > 1e-18 * ab || sn * sn > 1e-10) ? 2 : 1;
}

// writes local column j (registers) into the shared memory of the CTA that owns it in the next block step
template <class T, int CL, int GL, int RPL>
__device__ __forceinline__ void send_column(cg::cluster_group& cluster, T* cols, double* nrm, int crank, int j, int W, int nxt,
                                            int ncl, int pitch, int gl, const T (&rc)[RPL], double nv) {
  int dc; bool dtop;
  next_slot<CL>(crank, j < W, dc, dtop);
  const int dj = (dtop ? 0 : W) + (j < W ? j : j - W);
  T* dst = cluster.map_shared_rank(cols, dc) + ((size_t)nxt * ncl + dj) * pitch + gl;
#pragma unroll
  for (int k = 0; k < RPL; ++k) dst[k * GL] = rc[k];
  if (gl == 0) *(cluster.map_shared_rank(nrm, dc) + nxt * ncl + dj) = nv;
}

// DB: double-buffered column storage (one cluster barrier per block step; remote stores land in the other buffer) —
// the latency-optimal form for a single matrix.  !DB: single buffer, an extra cluster barrier separates the last reads
// of a block step from the remote stores — half the shared memory, used to pack a batch of matrices onto the SMs.
template <class T, int CL, int GL, int RPL, bool DB>
__global__ void __launch_bounds__(512) jacobi_cluster_kernel(T* __restrict__ X, int m, int n, int64_t ldx, int64_t bX, int W,
                                                              double tol, int* __restrict__ d_sweeps) {
  cg::cluster_group cluster = cg::this_cluster();
  const int crank = (int)cluster.block_rank();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int ncl = 2 * W;                                 // local columns
  const int pitch = GL * RPL;                            // rows padded to the register tile
  constexpr int NBUF = DB ? 2 : 1;
  T* cols = reinterpret_cast<T*>(smem_raw);              // [NBUF][ncl][pitch]
  double* nrm = reinterpret_cast<double*>(cols + (size_t)NBUF * ncl * pitch);   // [NBUF][ncl]
  int* flags = reinterpret_cast<int*>(nrm + NBUF * ncl);    // [CL]
  __shared__ int s_rot;

  const int tid = threadIdx.x;
  const int grp = tid / GL, gl = tid % GL;               // grp < W
  const double tol2 = tol * tol;
  T* Xb = X + (int64_t)(blockIdx.x / CL) * bX;           // grid.x = CL * batch
  const int col0 = crank * ncl;

  // load the two home blocks (zero columns beyond n, zero rows beyond m)
  for (int idx = tid; idx < ncl * pitch; idx += blockDim.x) {
    const int j = idx / pitch, i = idx - j * pitch;
    const int gc = col0 + j;
    cols[idx] = (gc < n && i < m) ? Xb[(int64_t)gc * ldx + i] : t_zero<T>();
  }
  if (tid == 0) s_rot = 0;
  int cur = 0;
  __syncthreads();
  cluster.sync();   // every CTA of the cluster is resident before the first remote store

  int sw = 0;
  for (; sw < JC_MAX_SWEEPS; ++sw) {
    // exact squared norms once per sweep
    for (int j = grp; j < ncl; j += W) {
      const T* x = cols + ((size_t)cur * ncl + j) * pitch;
      double a = 0.0;
#pragma unroll
      for (int k = 0; k < RPL; ++k) a += t_abs2(x[gl + k * GL]);
#pragma unroll
      for (int o = GL / 2; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if (gl == 0) nrm[cur * ncl + j] = a;
    }
    __syncthreads();
    int lvl = 0;   // 0: no rotation this sweep, 1: only rotations of already tiny inner products, 2: a significant rotation
    for (int bs = 0; bs < 2 * CL - 1; ++bs) {
      T* cb = cols + (size_t)cur * ncl * pitch;
      double* nb = nrm + cur * ncl;
      const int nxt = DB ? cur ^ 1 : cur;
      if (bs == 0) {
        // all pairs among the 2W resident columns: both columns of a pair go through shared memory every step
        const int M1 = ncl - 1;
        for (int r = 0; r < M1; ++r) {
          int p, q;
          if (grp == 0) { p = M1; q = r; }
          else { p = r + grp; if (p >= M1) p -= M1; q = r - grp; if (q < 0) q += M1; }
          T* xp = cb + (size_t)p * pitch + gl;
          T* xq = cb + (size_t)q * pitch + gl;
          T rp[RPL], rq[RPL];
#pragma unroll
          for (int k = 0; k < RPL; ++k) { rp[k] = xp[k * GL]; rq[k] = xq[k * GL]; }
          double an = nb[p], bn = nb[q];
          lvl = max(lvl, rotate_pair<T, GL, RPL>(rp, rq, an, bn, tol2));
          if (r + 1 < M1) {
#pragma unroll
            for (int k = 0; k < RPL; ++k) { xp[k * GL] = rp[k]; xq[k * GL] = rq[k]; }
            if (gl == 0) { nb[p] = an; nb[q] = bn; }
            __syncthreads();
          } else {
            if (!DB) cluster.sync();   // every CTA has finished reading its columns before any remote store lands
            send_column<T, CL, GL, RPL>(cluster, cols, nrm, crank, p, W, nxt, ncl, pitch, gl, rp, an);
            send_column<T, CL, GL, RPL>(cluster, cols, nrm, crank, q, W, nxt, ncl, pitch, gl, rq, bn);
          }
        }
      } else {
        // cross pairs top x bottom: the top column of a lane group is stationary in registers for the whole block step
        T rp[RPL];
        {
          const T* xp = cb + (size_t)grp * pitch + gl;
#pragma unroll
          for (int k = 0; k < RPL; ++k) rp[k] = xp[k * GL];
        }
        double an = nb[grp];
        int qi = grp;
        for (int r = 0; r < W; ++r) {
          const int q = W + qi;
          T* xq = cb + (size_t)q * pitch + gl;
          T rq[RPL];
#pragma unroll
          for (int k = 0; k < RPL; ++k) rq[k] = xq[k * GL];
          double bn = nb[q];
          lvl = max(lvl, rotate_pair<T, GL, RPL>(rp, rq, an, bn, tol2));
          if (r + 1 < W) {
#pragma unroll
            for (int k = 0; k < RPL; ++k) xq[k * GL] = rq[k];
            if (gl == 0) nb[q] = bn;
            __syncthreads();
          } else {
            if (!DB) cluster.sync();
            send_column<T, CL, GL, RPL>(cluster, cols, nrm, crank, q, W, nxt, ncl, pitch, gl, rq, bn);
          }
          if (++qi == W) qi = 0;
        }
        send_column<T, CL, GL, RPL>(cluster, cols, nrm, crank, grp, W, nxt, ncl, pitch, gl, rp, an);
      }
      if (bs == 2 * CL - 2) {
        // end of sweep: publish this CTA's rotation level to every CTA of the cluster
        if (lvl) atomicMax(&s_rot, lvl);
        __syncthreads();
        if (tid < CL) *(cluster.map_shared_rank(flags, tid) + crank) = s_rot;
      }
      cluster.sync();
      if (DB) cur ^= 1;
    }
    int any = 0;
#pragma unroll
    for (int c = 0; c < CL; ++c) any = max(any, flags[c]);
    __syncthreads();
    if (tid == 0) s_rot = 0;
    // level 1: every inner product was already below ~1e-9 relative before its rotation, so what is left is of second
    // order (< tol) and the confirming sweep is skipped
    if (any <= 1) { ++sw; break; }
  }

  // after whole sweeps every block is back in its home CTA
  __syncthreads();
  for (int idx = tid; idx < ncl * pitch; idx += blockDim.x) {
    const int j = idx / pitch, i = idx - j * pitch;
    const int gc = col0 + j;
    if (gc < n && i < m) Xb[(int64_t)gc * ldx + i] = cols[(size_t)cur * ncl * pitch + idx];
  }
  if (tid == 0 && crank == 0 && d_sweeps) d_sweeps[blockIdx.x / CL] = sw;
  cluster.sync();   // no CTA may exit while a peer can still address its shared memory
}

template <class T, int CL, int GL, int RPL, bool DB>
bool launch_cluster(T* X, int m, int n, int64_t ldx, int batch, int64_t bX, double tol, int* d_sweeps) {
  const int W = (n + 2 * CL - 1) / (2 * CL);
  const int threads = W * GL;
  if (threads > 512 || threads < 32 || (threads & 31)) return false;
  const size_t smem = sizeof(T) * (size_t)(DB ? 2 : 1) * 2 * W * GL * RPL + sizeof(double) * (DB ? 2 : 1) * 2 * W + sizeof(int) * CL;
  if (smem > 224 * 1024) return false;
  auto kern = jacobi_cluster_kernel<T, CL, GL, RPL, DB>;
  static int attr_dev = -1;   // function attributes are per device (ttn_init may re-bind)
  if (attr_dev != ctx().device) {
    TTN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
    attr_dev = ctx().device;
  }
  for (int b0 = 0; b0 < batch; b0 += 8192) {
    const int nb = std::min(8192, batch - b0);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(CL * nb, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx().stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    ProfScope prof_scope_(KF_JACOBI);
    TTN_CUDA(cudaLaunchKernelEx(&cfg, kern, X + (int64_t)b0 * bX, m, n, ldx, bX, W, tol, d_sweeps + b0));
    ctx().launches++;
  }
  return true;
}

}  // namespace

// Returns false when the shape is not served by the cluster kernel (caller falls back to the single-SM / block paths).
//   few matrices  : 8 CTAs per matrix, double-buffered (latency of the single SVD is what matters: TT-rounding chain);
//   large batches : the smallest cluster whose shared memory holds the matrix (2 or 4 CTAs, single buffer), so that
//                   sm_count/CL matrices are in flight at once (cfg5: ComplexF64 128 x 128 does not fit in one SM).
template <class T>
bool jacobi_cluster(T* X, int m, int n, int64_t ldx, int batch, int64_t bX, double tol, int* d_sweeps) {
  if (n < 32) return false;                       // tiny problems: one SM is enough
  const bool few = batch * 8 <= ctx().sm_count;
  if (few) {
    if (m <= 128) return launch_cluster<T, 8, 32, 4, true>(X, m, n, ldx, batch, bX, tol, d_sweeps);
    if (m <= 256) return launch_cluster<T, 8, 32, 8, true>(X, m, n, ldx, batch, bX, tol, d_sweeps);
    return false;
  }
  const size_t one_sm = (sizeof(T) * (size_t)(m + 4) + 8) * n;   // footprint of the single-SM kernel (jacobi.cu)
  if (one_sm <= 216 * 1024) return false;         // fits in one SM: one matrix per SM is the throughput-optimal layout
  if (m <= 128) {
    // 4 CTAs x 64 KB (two clusters' CTAs co-resident per SM) measured 5 % faster than 2 CTAs x 128 KB on cfg5
    if (n <= 256 && launch_cluster<T, 4, 16, 8, false>(X, m, n, ldx, batch, bX, tol, d_sweeps)) return true;
    if (n <= 128 && launch_cluster<T, 2, 16, 8, false>(X, m, n, ldx, batch, bX, tol, d_sweeps)) return true;
    return launch_cluster<T, 8, 32, 4, false>(X, m, n, ldx, batch, bX, tol, d_sweeps);
  }
  if (m <= 256) {
    if (launch_cluster<T, 4, 32, 8, false>(X, m, n, ldx, batch, bX, tol, d_sweeps)) return true;
    return launch_cluster<T, 8, 32, 8, false>(X, m, n, ldx, batch, bX, tol, d_sweeps);
  }
  return false;
}

template bool jacobi_cluster<double>(double*, int, int, int64_t, int, int64_t, double, int*);
template bool jacobi_cluster<zc>(zc*, int, int, int64_t, int, int64_t, double, int*);

}  // namespace ttn
