// One-sided (Hestenes) Jacobi SVD (kernel family F5, SURVEY.md §2.1).
//
// Replaces the LAPACK gesdd calls behind the reference's truncations: `_svdtrunc`
// (src/tt_cross_interpolation.jl:150, used by tt_compress! src/tt_tools.jl:752 and tdvp2
// src/solvers/tdvp.jl:250,278), the MALS core moves (src/solvers/mals.jl:99,126) and the DMRG core moves
// (src/solvers/dmrg.jl:189,213).  The bond-sized matrix is first reduced to a square triangular factor by
// the Householder QR of qr.cu (svd.cu), then its columns are orthogonalised in place by plane rotations:
//       X <- X V,   X^H X diagonal,   sigma_j = ||x_j||,   u_j = x_j / sigma_j.
// One-sided Jacobi delivers small singular values with high *relative* accuracy, which the reference's
// tolerance-driven rank rules (mals.jl:42-56 `sv_trunc`, dmrg.jl:179-185 `cut_off_index`) depend on.
//
// Kernel: a CTA stages a group of columns in shared memory (conflict-free: lanes walk down a column),
// one warp per column pair and round (round-robin tournament, all pairs of a round are disjoint), three
// dot products by warp shuffles, rotation applied in place.  If all n columns fit in one SM's shared
// memory the CTA iterates sweeps to convergence without leaving the kernel; otherwise the host walks a
// block round-robin (one launch per step, CTAs = independent block pairs, data stays in L2).
#include "ttn_internal.h"

namespace ttn {
namespace {

constexpr int JAC_MAX_SWEEPS = 40;

__device__ __forceinline__ double wsumd(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Plane rotation that orthogonalises two columns with squared norms a, b and inner product c = x_p^H x_q
// (|c| = absc, phase ph = c/|c|):  x_p' = cs x_p - sn conj(ph) x_q,  x_q' = sn ph x_p + cs x_q.
// With tau = (b-a)/2, h = sqrt(tau^2 + |c|^2), d = tau + sign(tau) h the smaller root is t = |c|/d and
// cs = |d|/sqrt(d^2+|c|^2), sn = sign(d)|c|/sqrt(d^2+|c|^2): one sqrt and one rsqrt, no division.
__device__ __forceinline__ void rot_params(double a, double b, double absc, double& cs, double& sn) {
  const double tau = 0.5 * (b - a);
  const double h = sqrt(tau * tau + absc * absc);
  const double d = tau + (tau >= 0.0 ? h : -h);
  const double rinv = rsqrt(d * d + absc * absc);
  cs = fabs(d) * rinv;
  sn = (d >= 0.0 ? absc : -absc) * rinv;
}

constexpr int JAC_T = 256;   // threads per CTA (measured: 256 thr x 4 lanes per pair beats 512 x 8 and 1024 x 16 on B200)

// One-sided Jacobi on a group of columns staged in shared memory (column pitch m+PADC keeps the strided row
// accesses of neighbouring lane groups on distinct banks).
//
// Ordering.  A sweep over nc columns is organised as log2(npad) *levels* of a recursive halving (npad = nc rounded up
// to a power of two): at the level with half-size h the columns are split into blocks of 2h, and within each block
// every column a of the first half meets every column q of the second half, h rounds of npad/2 disjoint pairs
// (a = block + j, q = block + h + (j + r) mod h).  Summed over the levels h = npad/2, ..., 1 this is npad-1 rounds and
// every pair exactly once — the same count as a round-robin tournament — but the a-column of a lane group is
// *stationary* for a whole level: it is loaded into registers once per level and only the moving q-column goes
// through shared memory, which halves the shared-memory traffic that bounds this kernel.
// mode 1 (block Jacobi across CTAs): a single level of cross pairs between column groups A (stationary) and B.
//
// A group of GL lanes owns a pair: RPL rows of both columns per lane in registers (RPL == 0: generic length, rows
// re-read from shared memory), inner product reduced with GL-wide shuffles, plane rotation by rot_params (no
// division), squared column norms maintained by the rotation identities and recomputed exactly once per sweep.
// With GL = 4 a warp carries 8 pairs, so the scalar rotation set-up is amortised over 8 pairs per warp instruction.
// full != 0: iterate sweeps until a whole sweep applies no rotation (single-CTA problem), else run `sweeps` sweeps.
template <class T, int GL, int RPL, bool FULLM>
__global__ void __launch_bounds__(JAC_T) jacobi_kernel(T* __restrict__ X, int m, int64_t ldx, int64_t bX,
                                                       const int* __restrict__ grpA, const int* __restrict__ grpB, int bsz,
                                                       int n, int mode, int full, int sweeps, double tol,
                                                       unsigned int* __restrict__ d_rotated, int* __restrict__ d_sweeps) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_rot;
  constexpr int PADC = is_cplx<T>::value ? 0 : 4;
  constexpr int NR = RPL > 0 ? RPL : 1;
  T* Xb = X + blockIdx.y * bX;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int grp = tid / GL, ngrp = blockDim.x / GL, gl = tid % GL;
  const double tol2 = tol * tol;
  const int pitch = m + PADC;

  const int a0 = grpA[blockIdx.x] * bsz;
  const int na = min(bsz, n - a0);
  const int gb = grpB[blockIdx.x];
  const int b0 = gb >= 0 ? gb * bsz : 0;
  const int nb = gb >= 0 ? min(bsz, n - b0) : 0;
  const int nc = na + nb;
  int npad = 2;
  while (npad < nc) npad <<= 1;
  const int bm = max(na, nb);

  T* Xs = reinterpret_cast<T*>(smem_raw);                            // [nc][pitch]
  double* nrm2 = reinterpret_cast<double*>(Xs + (size_t)nc * pitch);   // [nc]

  for (int c = warp; c < nc; c += nwarps) {
    const T* src = Xb + (int64_t)(c < na ? a0 + c : b0 + (c - na)) * ldx;
    T* dst = Xs + (size_t)c * pitch;
    for (int i = lane; i < m; i += 32) dst[i] = src[i];
  }
  if (tid == 0) s_rot = 0;
  __syncthreads();

  int sw = 0;
  const int max_sw = full ? JAC_MAX_SWEEPS : sweeps;
  bool any_rot = false;
  for (; sw < max_sw; ++sw) {
    for (int c = warp; c < nc; c += nwarps) {       // exact squared norms once per sweep
      const T* x = Xs + (size_t)c * pitch;
      double a = 0.0;
      for (int i = lane; i < m; i += 32) a += t_abs2(x[i]);
      a = wsumd(a);
      if (lane == 0) nrm2[c] = a;
    }
    __syncthreads();
    bool myrot = false;
    // levels: mode 0 -> h = npad/2, npad/4, ..., 1 ; mode 1 -> the single cross level h = bm
    for (int h = (mode == 0 ? npad / 2 : bm); h >= 1; h = (mode == 0 ? h >> 1 : 0)) {
      const int nslots = (mode == 0) ? npad / 2 : bm;
      for (int i0 = 0; i0 < nslots; i0 += ngrp) {   // passes; warp-uniform trip counts (shuffles + barriers inside)
        const int i = i0 + grp;
        int a, j, qbase;
        if (mode == 0) { j = i & (h - 1); a = ((i - j) << 1) + j; qbase = a - j + h; }
        else { j = i; a = i; qbase = na; }
        const bool actA = i < nslots && a < (mode == 0 ? nc : na);
        T* xa = Xs + (actA ? a : 0) * pitch;
        T ra[NR];
        double an = actA ? nrm2[a] : 0.0;
        if (RPL > 0) {
#pragma unroll
          for (int k = 0; k < RPL; ++k) {
            const int row = gl + k * GL;
            ra[k] = (FULLM || row < m) ? xa[row] : t_zero<T>();
          }
        }
        for (int r = 0; r < h; ++r) {
          int jq = j + r;
          if (jq >= h) jq -= h;
          const int q = qbase + jq;
          const bool act = actA && q < (mode == 0 ? nc : na + nb);
          T* xq = Xs + (act ? q : 0) * pitch;
          T rq[NR];
          T c = t_zero<T>();
          if (RPL > 0) {
            // (inactive groups read column 0: harmless, the result is discarded; keeps the loads unpredicated)
#pragma unroll
            for (int k = 0; k < RPL; ++k) {
              const int row = gl + k * GL;
              rq[k] = (FULLM || row < m) ? xq[row] : t_zero<T>();
            }
            T c4[4] = {t_zero<T>(), t_zero<T>(), t_zero<T>(), t_zero<T>()};   // independent accumulation chains
#pragma unroll
            for (int k = 0; k < RPL; ++k) t_fma(c4[k & 3], t_conj(ra[k]), rq[k]);
            c = t_add(t_add(c4[0], c4[1]), t_add(c4[2], c4[3]));
          } else if (act) {
            for (int row = gl; row < m; row += GL) t_fma(c, t_conj(xa[row]), xq[row]);
          }
          double cr = t_real(c), ci = t_imag(c);
#pragma unroll
          for (int o = GL / 2; o > 0; o >>= 1) {
            cr += __shfl_xor_sync(0xffffffffu, cr, o);
            if (is_cplx<T>::value) ci += __shfl_xor_sync(0xffffffffu, ci, o);
          }
          if (act) {
            const double b = nrm2[q];
            const double c2 = cr * cr + ci * ci;
            if (c2 > tol2 * an * b && an > 0.0 && b > 0.0) {   // false for zero columns and NaNs
              double cs, sn, absc, phr, phi;
              if (is_cplx<T>::value) {
                const double inv = rsqrt(c2);
                absc = c2 * inv; phr = cr * inv; phi = ci * inv;
              } else {
                absc = fabs(cr); phr = cr >= 0.0 ? 1.0 : -1.0; phi = 0.0;
              }
              rot_params(an, b, absc, cs, sn);
              const double x = 2.0 * cs * sn * absc;
              const double an_new = fmax(cs * cs * an - x + sn * sn * b, 0.0);
              if (gl == 0) nrm2[q] = fmax(sn * sn * an + x + cs * cs * b, 0.0);
              an = an_new;
              myrot = true;
              const T ph = t_from<T>(sn * phr, sn * phi);      // sn * phase
              const T phc = t_from<T>(sn * phr, -sn * phi);    // sn * conj(phase)
              if (RPL > 0) {
#pragma unroll
                for (int k = 0; k < RPL; ++k) {
                  const int row = gl + k * GL;
                  const T pv = ra[k], qv = rq[k];
                  ra[k] = t_sub(t_scale(pv, cs), t_mul(phc, qv));
                  if (FULLM || row < m) xq[row] = t_add(t_mul(ph, pv), t_scale(qv, cs));
                }
              } else {
                for (int row = gl; row < m; row += GL) {
                  const T pv = xa[row], qv = xq[row];
                  xa[row] = t_sub(t_scale(pv, cs), t_mul(phc, qv));
                  xq[row] = t_add(t_mul(ph, pv), t_scale(qv, cs));
                }
              }
            }
          }
          __syncthreads();
        }
        if (actA) {
          if (RPL > 0) {
#pragma unroll
            for (int k = 0; k < RPL; ++k) {
              const int row = gl + k * GL;
              if (FULLM || row < m) xa[row] = ra[k];
            }
          }
          if (gl == 0) nrm2[a] = an;
        }
        __syncthreads();
      }
    }
    if (myrot) s_rot = 1;       // benign race: every writer stores the same value
    __syncthreads();
    const int rot = s_rot;
    __syncthreads();
    if (tid == 0) s_rot = 0;
    any_rot |= (rot != 0);
    if (full && !rot) { ++sw; break; }
  }

  __syncthreads();
  for (int c = warp; c < nc; c += nwarps) {
    T* dst = Xb + (int64_t)(c < na ? a0 + c : b0 + (c - na)) * ldx;
    const T* src = Xs + (size_t)c * pitch;
    for (int i = lane; i < m; i += 32) dst[i] = src[i];
  }
  if (tid == 0) {
    if (d_rotated && any_rot) atomicOr(d_rotated, 1u);
    if (d_sweeps && full) d_sweeps[blockIdx.y] = sw;
  }
}

// Block Jacobi across CTAs for matrices that do not fit in one SM's shared memory (DMRG / MALS bond matrices of
// order 512 ... 4096).  One CTA = one pair of column blocks (A, B) and all na*nb cross pairs between them:
//   - the B block is staged in shared memory together with its maintained squared norms;
//   - the A block is processed in passes of one column per warp: the warp keeps its whole A column in registers
//     (RPLA rows per lane, m <= 32*RPLA), so a rotation streams the B column twice (inner product, update) and the A
//     column never leaves the register file until the pass ends;
//   - at round r warp w meets B column (w + r) mod R with R = max(nb, #warps): all warps touch distinct columns,
//     one block barrier per round.
// Squared norms of both blocks are recomputed exactly when the blocks are loaded.
template <class T, int RPLA>
__global__ void __launch_bounds__(JAC_T) jacobi_cross_kernel(T* __restrict__ X, int m, int64_t ldx, int64_t bX,
                                                             const int* __restrict__ grpA, const int* __restrict__ grpB,
                                                             int bsz, int n, double tol, unsigned int* __restrict__ d_rotated) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Xb = X + blockIdx.y * bX;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = JAC_T / 32;
  const double tol2 = tol * tol;
  const int a0 = grpA[blockIdx.x] * bsz, na = min(bsz, n - a0);
  const int b0 = grpB[blockIdx.x] * bsz, nb = min(bsz, n - b0);
  const int pitch = m + (is_cplx<T>::value ? 0 : 4);
  T* Bs = reinterpret_cast<T*>(smem_raw);                             // [nb][pitch]
  double* nrmB = reinterpret_cast<double*>(Bs + (size_t)nb * pitch);    // [nb]

  for (int c = warp; c < nb; c += NW) {
    const T* src = Xb + (int64_t)(b0 + c) * ldx;
    T* dst = Bs + (size_t)c * pitch;
    double s = 0.0;
    for (int i = lane; i < m; i += 32) { const T v = src[i]; dst[i] = v; s += t_abs2(v); }
    s = wsumd(s);
    if (lane == 0) nrmB[c] = s;
  }
  __syncthreads();

  bool myrot = false;
  const int R = max(nb, NW);
  for (int ap = 0; ap < na; ap += NW) {
    const int a = ap + warp;
    const bool actA = a < na;
    T* ga = Xb + (int64_t)(a0 + (actA ? a : 0)) * ldx;
    T ra[RPLA];
    double an = 0.0;
#pragma unroll
    for (int k = 0; k < RPLA; ++k) {
      const int row = lane + 32 * k;
      ra[k] = (actA && row < m) ? ga[row] : t_zero<T>();
      an += t_abs2(ra[k]);
    }
    an = wsumd(an);
    for (int r = 0; r < R; ++r) {
      int bq = warp + r;
      if (bq >= R) bq -= R;
      const bool act = actA && bq < nb;
      T* xq = Bs + (size_t)(act ? bq : 0) * pitch;
      T c4[4] = {t_zero<T>(), t_zero<T>(), t_zero<T>(), t_zero<T>()};
      if (act) {
#pragma unroll
        for (int k = 0; k < RPLA; ++k) {
          const int row = lane + 32 * k;
          if (row < m) t_fma(c4[k & 3], t_conj(ra[k]), xq[row]);
        }
      }
      const T c = t_add(t_add(c4[0], c4[1]), t_add(c4[2], c4[3]));
      const double cr = wsumd(t_real(c));
      const double ci = is_cplx<T>::value ? wsumd(t_imag(c)) : 0.0;
      if (act) {
        const double b = nrmB[bq];
        const double c2 = cr * cr + ci * ci;
        if (c2 > tol2 * an * b && an > 0.0 && b > 0.0) {
          double cs, sn, absc, phr, phi;
          if (is_cplx<T>::value) {
            const double inv = rsqrt(c2);
            absc = c2 * inv; phr = cr * inv; phi = ci * inv;
          } else {
            absc = fabs(cr); phr = cr >= 0.0 ? 1.0 : -1.0; phi = 0.0;
          }
          rot_params(an, b, absc, cs, sn);
          const double x = 2.0 * cs * sn * absc;
          if (lane == 0) nrmB[bq] = fmax(sn * sn * an + x + cs * cs * b, 0.0);
          an = fmax(cs * cs * an - x + sn * sn * b, 0.0);
          myrot = true;
          const T ph = t_from<T>(sn * phr, sn * phi);
          const T phc = t_from<T>(sn * phr, -sn * phi);
#pragma unroll
          for (int k = 0; k < RPLA; ++k) {
            const int row = lane + 32 * k;
            if (row < m) {
              const T pv = ra[k], qv = xq[row];
              ra[k] = t_sub(t_scale(pv, cs), t_mul(phc, qv));
              xq[row] = t_add(t_mul(ph, pv), t_scale(qv, cs));
            }
          }
        }
      }
      __syncthreads();
    }
    if (actA) {
#pragma unroll
      for (int k = 0; k < RPLA; ++k) {
        const int row = lane + 32 * k;
        if (row < m) ga[row] = ra[k];
      }
    }
  }
  __syncthreads();
  for (int c = warp; c < nb; c += NW) {
    T* dst = Xb + (int64_t)(b0 + c) * ldx;
    const T* src = Bs + (size_t)c * pitch;
    for (int i = lane; i < m; i += 32) dst[i] = src[i];
  }
  if (myrot && lane == 0 && d_rotated) atomicOr(d_rotated, 1u);
}

template <class T> struct JacCfg;
template <> struct JacCfg<double> { static constexpr int GL = 4, RPL = 32, GLG = 8; };
template <> struct JacCfg<zc> { static constexpr int GL = 8, RPL = 16, GLG = 8; };

template <class T>
__global__ void colnorm_kernel(const T* __restrict__ X, int m, int n, int64_t ldx, int64_t bX, double* __restrict__ norms,
                               int64_t bnorms) {
  // one warp per column
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const T* x = X + blockIdx.y * bX + (int64_t)warp * ldx;
  double a = 0.0;
  for (int i = lane; i < m; i += 32) a += t_abs2(x[i]);
  a = wsumd(a);
  if (lane == 0) norms[blockIdx.y * bnorms + warp] = sqrt(a);
}

template <class T>
__global__ void gather_kernel(const T* __restrict__ X, int m, int64_t ldx, const int* __restrict__ perm,
                              const double* __restrict__ scale, int r, T* __restrict__ dst, int64_t rs, int64_t cs,
                              int64_t bX, int64_t bperm, int64_t bdst) {
  const int64_t total = (int64_t)m * r;
  const T* Xb = X + blockIdx.y * bX;
  const int* pb = perm + blockIdx.y * bperm;
  const double* sb = scale + blockIdx.y * bperm;
  T* db = dst + blockIdx.y * bdst;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx % m), j = (int)(idx / m);
    db[i * rs + j * cs] = t_scale(Xb[i + (int64_t)pb[j] * ldx], sb[j]);
  }
}

}  // namespace

template <class T>
int jacobi_orth(T* X, int m, int n, int64_t ldx, double* norms, int batch, int64_t bX, int64_t bnorms) {
  if (n <= 0 || m <= 0 || batch <= 0) return 0;
  // rotation threshold |x_p^H x_q| <= tol ||x_p|| ||x_q||: m·eps is the rounding level of the computed inner product
  const double tol = (double)std::max(m, 8) * 1.1102230246251565e-16;
  const size_t budget = 216 * 1024;
  typedef JacCfg<T> Cfg;
  // rows-per-lane specialisation: columns of up to GL*RPL = 128 rows live in registers during a rotation
  const bool regs = m <= Cfg::GL * Cfg::RPL;
  const bool fullm = m == Cfg::GL * Cfg::RPL;
  auto kern = regs ? (fullm ? jacobi_kernel<T, Cfg::GL, Cfg::RPL, true> : jacobi_kernel<T, Cfg::GL, Cfg::RPL, false>)
                   : jacobi_kernel<T, Cfg::GLG, 0, false>;
  static int attr_dev = -1;   // function attributes are per device (ttn_init may re-bind)
  if (attr_dev != ctx().device) {
    const int mx = 224 * 1024;
    TTN_CUDA(cudaFuncSetAttribute(jacobi_kernel<T, Cfg::GL, Cfg::RPL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
    TTN_CUDA(cudaFuncSetAttribute(jacobi_kernel<T, Cfg::GL, Cfg::RPL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
    TTN_CUDA(cudaFuncSetAttribute(jacobi_kernel<T, Cfg::GLG, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
    attr_dev = ctx().device;
  }
  const size_t col_bytes = sizeof(T) * (size_t)(m + (is_cplx<T>::value ? 0 : 4)) + sizeof(double);   // column + its norm
  const int threads = JAC_T;
  int sweeps_used = 0;
  ttn_assert(2 * col_bytes <= budget, 2, "jacobi: a column pair does not fit in shared memory");
  DevBuf dsw_cl(sizeof(int) * batch);
  if (jacobi_cluster<T>(X, m, n, ldx, batch, bX, tol, dsw_cl.as<int>())) {
    int hsw = 0;
    read_back(&hsw, dsw_cl.p, sizeof(int));
    sweeps_used = hsw;
  } else if ((size_t)n * col_bytes <= budget) {
    // whole matrix in one SM: iterate to convergence inside the kernel
    int h_grp[2] = {0, -1};
    DevBuf grp(sizeof(int) * 2), dsw(sizeof(int) * batch);
    TTN_CUDA(cudaMemcpyAsync(grp.p, h_grp, sizeof(h_grp), cudaMemcpyHostToDevice, ctx().stream));
    for (int b0 = 0; b0 < batch; b0 += 65535) {
      const int nb = std::min(65535, batch - b0);
      dim3 grid(1, nb);
      ProfScope prof_scope_(KF_JACOBI);
      kern<<<grid, threads, (size_t)n * col_bytes, ctx().stream>>>(X + (int64_t)b0 * bX, m, ldx, bX, grp.as<int>(),
                                                                 grp.as<int>() + 1, n, n, 0, 1, 0, tol, nullptr,
                                                                 dsw.as<int>() + b0);
      TTN_CHECK_LAUNCH();
      ctx().launches++;
    }
    int hsw = 0;   // sweeps of batch element 0 (diagnostics; one 4-byte D2H, overlapped with the norms read-back sync)
    read_back(&hsw, dsw.p, sizeof(int));
    sweeps_used = hsw;
  } else if (n >= 128 && m >= 64 && std::min(m, n) >= ctx().gram_jacobi_min) {
    // large matrices: Gram-block Jacobi, O(m n^2) work on the FP64 tensor pipe (jacobi_gram.cu)
    for (int b = 0; b < batch; ++b) {
      const int sw = jacobi_gram<T>(X + (int64_t)b * bX, m, n, ldx, tol, JAC_MAX_SWEEPS);
      ttn_assert(sw >= 0, 7, "jacobi_gram: shape not served");
      if (b == 0) sweeps_used = sw;
    }
  } else {
    // block Jacobi across CTAs.  Fast path (m <= 32*RPLA): blocks of #warps columns, cross steps on
    // jacobi_cross_kernel (A block in registers, B block in shared memory); generic path: two blocks per CTA in
    // shared memory on jacobi_kernel.
    constexpr int RPLA_S = is_cplx<T>::value ? 16 : 32, RPLA_L = is_cplx<T>::value ? 32 : 64;
    const bool fast = m <= 32 * RPLA_L;
    const bool small_rows = m <= 32 * RPLA_S;
    int bsz = fast ? JAC_T / 32 : (int)(budget / (2 * col_bytes));
    if (bsz > 32) bsz = 32;
    ttn_assert(bsz >= 1, 2, "jacobi: a column pair does not fit in shared memory");
    if (fast) {
      static bool cattr = false;
      if (!cattr) {
        const int mx = 224 * 1024;
        TTN_CUDA(cudaFuncSetAttribute(jacobi_cross_kernel<T, RPLA_S>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        TTN_CUDA(cudaFuncSetAttribute(jacobi_cross_kernel<T, RPLA_L>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        cattr = true;
      }
      ttn_assert((size_t)bsz * col_bytes <= budget, 2, "jacobi: block does not fit in shared memory");
    }
    const int nblk = (n + bsz - 1) / bsz;
    const int ne = nblk + (nblk & 1);
    DevBuf dmax(sizeof(unsigned int));
    // pair lists of every round-robin step, uploaded once: step 0 = pairs inside each block,
    // steps 1..ne-1 = block tournament (cross pairs only)
    std::vector<int> hA, hB, off(ne + 1, 0);
    for (int i = 0; i < nblk; ++i) { hA.push_back(i); hB.push_back(-1); }
    off[1] = nblk;
    for (int r = 0; r < ne - 1; ++r) {
      for (int i = 0; i < ne / 2; ++i) {
        int p, q;
        if (i == 0) { p = ne - 1; q = r; }
        else { p = (r + i) % (ne - 1); q = (r - i + (ne - 1)) % (ne - 1); }
        if (p < nblk && q < nblk) { hA.push_back(std::min(p, q)); hB.push_back(std::max(p, q)); }
      }
      off[r + 2] = (int)hA.size();
    }
    DevBuf gA(sizeof(int) * hA.size()), gB(sizeof(int) * hB.size());
    TTN_CUDA(cudaMemcpyAsync(gA.p, hA.data(), sizeof(int) * hA.size(), cudaMemcpyHostToDevice, ctx().stream));
    TTN_CUDA(cudaMemcpyAsync(gB.p, hB.data(), sizeof(int) * hB.size(), cudaMemcpyHostToDevice, ctx().stream));
    TTN_CUDA(cudaStreamSynchronize(ctx().stream));
    ttn_assert(batch <= 65535, 2, "jacobi: batch too large for the block path");
    auto gen = jacobi_kernel<T, Cfg::GLG, 0, false>;
    for (int sw = 0; sw < JAC_MAX_SWEEPS; ++sw) {
      TTN_CUDA(cudaMemsetAsync(dmax.p, 0, sizeof(unsigned int), ctx().stream));
      for (int st = 0; st < ne; ++st) {
        const int cnt = off[st + 1] - off[st];
        if (cnt <= 0) continue;
        dim3 grid(cnt, batch);
        ProfScope prof_scope_(KF_JACOBI);
        if (st == 0 || !fast) {
          const size_t smem = (size_t)(st == 0 ? 1 : 2) * bsz * col_bytes;
          gen<<<grid, threads, smem, ctx().stream>>>(X, m, ldx, bX, gA.as<int>() + off[st], gB.as<int>() + off[st], bsz, n,
                                                    st == 0 ? 0 : 1, 0, 1, tol, dmax.as<unsigned int>(), nullptr);
        } else if (small_rows) {
          jacobi_cross_kernel<T, RPLA_S><<<grid, threads, (size_t)bsz * col_bytes, ctx().stream>>>(
              X, m, ldx, bX, gA.as<int>() + off[st], gB.as<int>() + off[st], bsz, n, tol, dmax.as<unsigned int>());
        } else {
          jacobi_cross_kernel<T, RPLA_L><<<grid, threads, (size_t)bsz * col_bytes, ctx().stream>>>(
              X, m, ldx, bX, gA.as<int>() + off[st], gB.as<int>() + off[st], bsz, n, tol, dmax.as<unsigned int>());
        }
        TTN_CHECK_LAUNCH();
        ctx().launches++;
      }
      unsigned int rotated = 0;
      read_back(&rotated, dmax.p, sizeof(rotated));
      sweeps_used = sw + 1;
      if (!rotated) break;
    }
  }
  {
    const int wpb = 8;
    for (int b0 = 0; b0 < batch; b0 += 65535) {
      const int nb = std::min(65535, batch - b0);
      dim3 grid((n + wpb - 1) / wpb, nb);
      ProfScope prof_scope_(KF_GATHER);
      colnorm_kernel<T><<<grid, wpb * 32, 0, ctx().stream>>>(X + (int64_t)b0 * bX, m, n, ldx, bX, norms + (int64_t)b0 * bnorms,
                                                            bnorms);
      TTN_CHECK_LAUNCH();
      ctx().launches++;
    }
  }
  ctx().last_jacobi_sweeps = sweeps_used;
  return sweeps_used;
}

template <class T>
void gather_cols(const T* X, int m, int64_t ldx, const int* perm, const double* scale, int r, T* dst, int64_t rs, int64_t cs,
                 int batch, int64_t bX, int64_t bperm, int64_t bdst) {
  if (r <= 0 || m <= 0 || batch <= 0) return;
  const int64_t total = (int64_t)m * r;
  int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)ctx().sm_count * 4);
  for (int b0 = 0; b0 < batch; b0 += 65535) {
    const int nb = std::min(65535, batch - b0);
    dim3 grid(blocks, nb);
    ProfScope prof_scope_(KF_GATHER);
    gather_kernel<T><<<grid, 256, 0, ctx().stream>>>(X + (int64_t)b0 * bX, m, ldx, perm + (int64_t)b0 * bperm,
                                                    scale + (int64_t)b0 * bperm, r, dst + (int64_t)b0 * bdst, rs, cs, bX, bperm,
                                                    bdst);
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
}

#define INST(T)                                                                                   \
  template int jacobi_orth<T>(T*, int, int, int64_t, double*, int, int64_t, int64_t);              \
  template void gather_cols<T>(const T*, int, int64_t, const int*, const double*, int, T*, int64_t, int64_t, int, int64_t, \
                               int64_t, int64_t);
INST(double)
INST(zc)
#undef INST

}  // namespace ttn
