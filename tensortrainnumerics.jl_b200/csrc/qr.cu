// Batched Householder QR (kernel family F4, SURVEY.md §2.1).
//
// Replaces the LAPACK geqrf/orgqr (+ `Matrix(F.Q)`) calls of the reference's QR/LQ sweeps and core moves:
// orthogonalize (src/tt_tools.jl:521,532), ALS core moves (src/solvers/als.jl:109,125), TDVP
// (src/solvers/tdvp.jl:83,116), and serves as the preconditioner of the Jacobi SVD (svd.cu).
// Conventions follow LAPACK: H_j = I - tau_j v_j v_j^H with v_j(j) = 1 stored below the diagonal,
// A = Q R with Q = H_0 H_1 ... H_{k-1}; the factorization applies H_j^H from the left.
//
// Layout: column-major, leading dimension lda, `batch` independent matrices (grid.y / grid.x).
// Two kernels:
//   qr_panel_kernel — one CTA per matrix factors NB columns in place (fixed row ownership per thread,
//                     block reductions through warp shuffles), so reflector generation never leaves the SM;
//   qr_apply_kernel — applies a range of reflectors to a slab of CC target columns held in shared memory;
//                     slabs are independent, so the trailing update / Q formation spreads over the grid.
// The trailing update is a BLAS-2 style sweep over L2-resident data (the matrices on this path are at most
// a few MB), which keeps the factorization in two kernels per panel with no host synchronisation.
#include "ttn_internal.h"

namespace ttn {
namespace {

constexpr int PANEL_T = 512;
constexpr int PANEL_NB = 16;
constexpr int APPLY_T = 256;
constexpr int APPLY_CC = 8;

__device__ __forceinline__ double wsum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ zc wsum(zc v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
    v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
  }
  return v;
}

// Householder generation (LAPACK xLARFG without the safmin rescaling loop)
__device__ __forceinline__ void larfg(double alpha, double xn2, double& beta, double& tau, double& scal) {
  if (xn2 == 0.0) { beta = alpha; tau = 0.0; scal = 0.0; return; }
  beta = -copysign(sqrt(alpha * alpha + xn2), alpha);
  tau = (beta - alpha) / beta;
  scal = 1.0 / (alpha - beta);
}
__device__ __forceinline__ void larfg(zc alpha, double xn2, zc& beta, zc& tau, zc& scal) {
  if (xn2 == 0.0 && alpha.y == 0.0) { beta = alpha; tau = make_cuDoubleComplex(0, 0); scal = make_cuDoubleComplex(0, 0); return; }
  const double b = -copysign(sqrt(alpha.x * alpha.x + alpha.y * alpha.y + xn2), alpha.x);
  beta = make_cuDoubleComplex(b, 0.0);
  tau = make_cuDoubleComplex((b - alpha.x) / b, -alpha.y / b);
  const double dr = alpha.x - b, di = alpha.y;
  const double den = dr * dr + di * di;
  scal = make_cuDoubleComplex(dr / den, -di / den);
}

template <class T, int NB>
__global__ void __launch_bounds__(PANEL_T) qr_panel_kernel(T* __restrict__ A, int m, int n, int64_t lda, T* __restrict__ tau,
                                                           int j0, int64_t bA, int64_t btau) {
  T* Ab = A + blockIdx.x * bA;
  T* taub = tau + blockIdx.x * btau;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = PANEL_T / 32;
  const int kmax = m < n ? m : n;
  const int jend = (j0 + NB < n) ? j0 + NB : n;
  const int cend = (j0 + NB < kmax) ? j0 + NB : kmax;
  __shared__ double s_red[NW];
  __shared__ T s_part[NW][NB];
  __shared__ T s_w[NB];
  __shared__ T s_scal, s_tau;

  for (int c = j0; c < cend; ++c) {
    T* col = Ab + (int64_t)c * lda;
    // rows above the diagonal are never touched: every row loop starts in the 512-row slab that holds row c (the row
    // ownership i mod PANEL_T is unchanged), which halves the L2 traffic of a square factorisation
    const int ibase = (c / PANEL_T) * PANEL_T + tid;
    double p = 0.0;
    for (int i = ibase; i < m; i += PANEL_T)
      if (i > c) p += t_abs2(col[i]);
    p = wsum(p);
    if (lane == 0) s_red[warp] = p;
    __syncthreads();
    if (tid == 0) {
      double xn2 = 0.0;
      for (int w = 0; w < NW; ++w) xn2 += s_red[w];
      T beta, tv, sc;
      larfg(col[c], xn2, beta, tv, sc);
      taub[c] = tv;
      s_tau = tv;
      s_scal = sc;
      col[c] = beta;
    }
    __syncthreads();
    const T scal = s_scal;
    const T tauc = t_conj(s_tau);
    const int nrem = jend - (c + 1);
    T acc[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) acc[q] = t_zero<T>();
    for (int i = ibase; i < m; i += PANEL_T) {
      if (i < c) continue;
      T vi;
      if (i == c) vi = t_one<T>();
      else { vi = t_mul(col[i], scal); col[i] = vi; }
      const T vc = t_conj(vi);
#pragma unroll
      for (int q = 0; q < NB; ++q)
        if (q < nrem) t_fma(acc[q], vc, Ab[i + (int64_t)(c + 1 + q) * lda]);
    }
    if (nrem > 0) {
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        if (q < nrem) {
          const T s = wsum(acc[q]);
          if (lane == 0) s_part[warp][q] = s;
        }
      }
      __syncthreads();
      if (tid < nrem) {
        T s = s_part[0][tid];
        for (int w = 1; w < NW; ++w) s = t_add(s, s_part[w][tid]);
        s_w[tid] = t_mul(tauc, s);
      }
      __syncthreads();
      for (int i = ibase; i < m; i += PANEL_T) {
        if (i < c) continue;
        const T vi = (i == c) ? t_one<T>() : col[i];
#pragma unroll
        for (int q = 0; q < NB; ++q)
          if (q < nrem) {
            T* p2 = Ab + i + (int64_t)(c + 1 + q) * lda;
            *p2 = t_sub(*p2, t_mul(s_w[q], vi));
          }
      }
    }
    __syncthreads();
  }
}

// Tall panels (one matrix, m - j0 >= 512): the same NB-column panel factorisation with the working set in shared memory.
// The unblocked kernel above streams the (m - j0) x NB panel through one SM three times per column (~8.8 us per column at
// m = 2048: single-SM L2 bandwidth); here the panel is processed in sub-panels of SW columns that fit in shared memory
// (SW * (m - j0) elements): a sub-panel is loaded once, receives the reflectors of the earlier sub-panels of this panel
// (read from global memory, where they were written back), is factored column by column entirely in shared memory, and is
// written back once.  Requires the whole panel inside min(m, n) (the host checks).
constexpr int PSW_MAX = 8;
template <class T, int NB>
__global__ void __launch_bounds__(PANEL_T) qr_panel_smem_kernel(T* __restrict__ A, int m, int64_t lda, T* __restrict__ tau,
                                                                int j0, int SW, int64_t bA, int64_t btau) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Ab = A + blockIdx.x * bA;
  T* taub = tau + blockIdx.x * btau;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = PANEL_T / 32;
  const int L = m - j0;                          // local row i' = i - j0
  T* Ps = reinterpret_cast<T*>(smem_raw);        // [SW][L]
  __shared__ double s_red[NW];
  __shared__ T s_part[NW][PSW_MAX];
  __shared__ T s_w[PSW_MAX];
  __shared__ T s_scal, s_tau;

  for (int c0 = j0; c0 < j0 + NB; c0 += SW) {
    const int sw = (c0 + SW <= j0 + NB) ? SW : j0 + NB - c0;
    for (int q = 0; q < sw; ++q)
      for (int il = tid; il < L; il += PANEL_T) Ps[(size_t)q * L + il] = Ab[(j0 + il) + (int64_t)(c0 + q) * lda];
    __syncthreads();
    // reflectors of the earlier sub-panels: Ps <- H_r^H Ps,  r = j0 .. c0-1
    for (int r = j0; r < c0; ++r) {
      const T* vcol = Ab + (int64_t)r * lda;
      const T tc = t_conj(taub[r]);
      T acc[PSW_MAX];
#pragma unroll
      for (int q = 0; q < PSW_MAX; ++q) acc[q] = t_zero<T>();
      for (int il = tid; il < L; il += PANEL_T) {
        const int gi = j0 + il;
        if (gi < r) continue;
        const T vc = (gi == r) ? t_one<T>() : t_conj(vcol[gi]);
#pragma unroll
        for (int q = 0; q < PSW_MAX; ++q)
          if (q < sw) t_fma(acc[q], vc, Ps[(size_t)q * L + il]);
      }
#pragma unroll
      for (int q = 0; q < PSW_MAX; ++q)
        if (q < sw) {
          const T sm = wsum(acc[q]);
          if (lane == 0) s_part[warp][q] = sm;
        }
      __syncthreads();
      if (tid < sw) {
        T sm = s_part[0][tid];
        for (int w = 1; w < NW; ++w) sm = t_add(sm, s_part[w][tid]);
        s_w[tid] = t_mul(tc, sm);
      }
      __syncthreads();
      for (int il = tid; il < L; il += PANEL_T) {
        const int gi = j0 + il;
        if (gi < r) continue;
        const T vi = (gi == r) ? t_one<T>() : vcol[gi];
#pragma unroll
        for (int q = 0; q < PSW_MAX; ++q)
          if (q < sw) {
            T* p2 = Ps + (size_t)q * L + il;
            *p2 = t_sub(*p2, t_mul(s_w[q], vi));
          }
      }
      // s_part / s_w of the next reflector are rewritten only after the two barriers of its own reduction
    }
    __syncthreads();
    // factor the sub-panel in shared memory
    for (int qc = 0; qc < sw; ++qc) {
      const int c = c0 + qc, cl = c - j0;        // global column / local diagonal row
      T* col = Ps + (size_t)qc * L;
      double p = 0.0;
      for (int il = cl + 1 + tid; il < L; il += PANEL_T) p += t_abs2(col[il]);
      p = wsum(p);
      if (lane == 0) s_red[warp] = p;
      __syncthreads();
      if (tid == 0) {
        double xn2 = 0.0;
        for (int w = 0; w < NW; ++w) xn2 += s_red[w];
        T beta, tv, sc;
        larfg(col[cl], xn2, beta, tv, sc);
        taub[c] = tv;
        s_tau = tv;
        s_scal = sc;
        col[cl] = beta;
      }
      __syncthreads();
      const T scal = s_scal;
      const T tauc = t_conj(s_tau);
      const int nrem = sw - 1 - qc;
      T acc[PSW_MAX];
#pragma unroll
      for (int q = 0; q < PSW_MAX; ++q) acc[q] = t_zero<T>();
      for (int il = cl + tid; il < L; il += PANEL_T) {
        T vi;
        if (il == cl) vi = t_one<T>();
        else { vi = t_mul(col[il], scal); col[il] = vi; }
        const T vc = t_conj(vi);
#pragma unroll
        for (int q = 0; q < PSW_MAX; ++q)
          if (q < nrem) t_fma(acc[q], vc, Ps[(size_t)(qc + 1 + q) * L + il]);
      }
      if (nrem > 0) {
#pragma unroll
        for (int q = 0; q < PSW_MAX; ++q)
          if (q < nrem) {
            const T sm = wsum(acc[q]);
            if (lane == 0) s_part[warp][q] = sm;
          }
        __syncthreads();
        if (tid < nrem) {
          T sm = s_part[0][tid];
          for (int w = 1; w < NW; ++w) sm = t_add(sm, s_part[w][tid]);
          s_w[tid] = t_mul(tauc, sm);
        }
        __syncthreads();
        for (int il = cl + tid; il < L; il += PANEL_T) {
          const T vi = (il == cl) ? t_one<T>() : col[il];
#pragma unroll
          for (int q = 0; q < PSW_MAX; ++q)
            if (q < nrem) {
              T* p2 = Ps + (size_t)(qc + 1 + q) * L + il;
              *p2 = t_sub(*p2, t_mul(s_w[q], vi));
            }
        }
      }
      __syncthreads();
    }
    for (int q = 0; q < sw; ++q)
      for (int il = tid; il < L; il += PANEL_T) Ab[(j0 + il) + (int64_t)(c0 + q) * lda] = Ps[(size_t)q * L + il];
    __syncthreads();                             // the next sub-panel reads these reflectors back from global memory
  }
}

// Applies reflectors j in [jlo, jhi) of (A, tau) to columns [c0, c0+nc) of C, rows >= jlo.
//   trans = true : C <- H_{jhi-1}^H ... H_{jlo}^H C   (forward order, conj(tau))   -> Q^H C
//   trans = false: C <- H_{jlo} ... H_{jhi-1} C        (backward order, tau)        -> Q C
template <class T>
__global__ void __launch_bounds__(APPLY_T) qr_apply_kernel(const T* __restrict__ A, int m, int64_t lda,
                                                           const T* __restrict__ tau, int jlo, int jhi, T* __restrict__ C,
                                                           int c0, int nc, int64_t ldc, int cc_per_cta, bool trans,
                                                           int64_t bA, int64_t btau, int64_t bC) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int L = m - jlo;  // rows jlo..m-1
  T* Cs = reinterpret_cast<T*>(smem_raw);            // [cc][L]
  T* vs = Cs + (size_t)cc_per_cta * L;               // [L]
  constexpr int NW = APPLY_T / 32;
  __shared__ T s_part[NW][APPLY_CC];
  __shared__ T s_w[APPLY_CC];
  const T* Ab = A + blockIdx.y * bA;
  const T* taub = tau + blockIdx.y * btau;
  T* Cb = C + blockIdx.y * bC;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int col0 = c0 + blockIdx.x * cc_per_cta;
  int ncc = c0 + nc - col0;
  if (ncc > cc_per_cta) ncc = cc_per_cta;
  if (ncc <= 0) return;

  for (int cc = 0; cc < ncc; ++cc)
    for (int i = tid; i < L; i += APPLY_T) Cs[(size_t)cc * L + i] = Cb[(jlo + i) + (int64_t)(col0 + cc) * ldc];
  __syncthreads();

  const int nref = jhi - jlo;
  for (int s = 0; s < nref; ++s) {
    const int j = trans ? (jlo + s) : (jhi - 1 - s);
    const T tj = trans ? t_conj(taub[j]) : taub[j];
    const T* vcol = Ab + (int64_t)j * lda;
    T acc[APPLY_CC];
#pragma unroll
    for (int q = 0; q < APPLY_CC; ++q) acc[q] = t_zero<T>();
    for (int i = tid; i < L; i += APPLY_T) {
      const int gi = jlo + i;
      if (gi < j) continue;
      const T vi = (gi == j) ? t_one<T>() : vcol[gi];
      vs[i] = vi;
      const T vc = t_conj(vi);
#pragma unroll
      for (int q = 0; q < APPLY_CC; ++q)
        if (q < ncc) t_fma(acc[q], vc, Cs[(size_t)q * L + i]);
    }
#pragma unroll
    for (int q = 0; q < APPLY_CC; ++q) {
      if (q < ncc) {
        const T r = wsum(acc[q]);
        if (lane == 0) s_part[warp][q] = r;
      }
    }
    __syncthreads();
    if (tid < ncc) {
      T r = s_part[0][tid];
      for (int w = 1; w < NW; ++w) r = t_add(r, s_part[w][tid]);
      s_w[tid] = t_mul(tj, r);
    }
    __syncthreads();
    for (int i = tid; i < L; i += APPLY_T) {
      const int gi = jlo + i;
      if (gi < j) continue;
      const T vi = vs[i];
#pragma unroll
      for (int q = 0; q < APPLY_CC; ++q)
        if (q < ncc) {
          T* p = Cs + (size_t)q * L + i;
          *p = t_sub(*p, t_mul(s_w[q], vi));
        }
    }
    // fixed row ownership: the next reflector's first pass touches the same rows from the same thread;
    // s_part / s_w reuse is ordered by the two barriers above.
  }
  __syncthreads();
  for (int cc = 0; cc < ncc; ++cc)
    for (int i = tid; i < L; i += APPLY_T) Cb[(jlo + i) + (int64_t)(col0 + cc) * ldc] = Cs[(size_t)cc * L + i];
}

template <class T>
void launch_apply(const T* A, int m, int64_t lda, const T* tau, int jlo, int jhi, T* C, int c0, int nc, int64_t ldc,
                  bool trans, int batch, int64_t bA, int64_t btau, int64_t bC) {
  if (nc <= 0 || jhi <= jlo || batch <= 0) return;
  ProfScope prof_scope_(KF_QR_APPLY);
  const int L = m - jlo;
  const size_t budget = 200 * 1024;
  const size_t fit = budget / (sizeof(T) * (size_t)L);
  ttn_assert(fit >= 2, 2, "qr_apply: column does not fit in shared memory");
  int cc = (int)std::min<size_t>(APPLY_CC, fit - 1);
  // spread over the SMs when there are few columns
  const int want = (nc * batch + ctx().sm_count - 1) / ctx().sm_count;
  if (cc > want) cc = std::max(1, want);
  const size_t smem = sizeof(T) * (size_t)(cc + 1) * L;
  auto kern = qr_apply_kernel<T>;
  static size_t attr = 0;
  if (smem > attr) {
    TTN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
    attr = smem;
  }
  for (int b0 = 0; b0 < batch; b0 += 65535) {
    const int nb = std::min(65535, batch - b0);
    dim3 grid((nc + cc - 1) / cc, nb);
    kern<<<grid, APPLY_T, smem, ctx().stream>>>(A + (int64_t)b0 * bA, m, lda, tau + (int64_t)b0 * btau, jlo, jhi,
                                               C + (int64_t)b0 * bC, c0, nc, ldc, cc, trans, bA, btau, bC);
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
}

}  // namespace

template <class T>
void qr_factor(T* A, int m, int n, int64_t lda, T* tau, int batch, int64_t bA, int64_t btau) {
  const int k = std::min(m, n);
  if (k <= 0 || batch <= 0) return;
  static int attr_dev = -1;   // function attributes are per device (ttn_init may re-bind)
  for (int j0 = 0; j0 < k; j0 += PANEL_NB) {
    // tall single matrix, whole panel inside min(m, n): shared-memory sub-panel kernel
    int SW = 0;
    if (batch == 1 && m - j0 >= 512 && j0 + PANEL_NB <= k)
      for (int c : {8, 4, 2})
        if (sizeof(T) * (size_t)c * (m - j0) <= 200 * 1024) { SW = c; break; }
    if (SW > 0) {
      if (attr_dev != ctx().device) {
        TTN_CUDA(cudaFuncSetAttribute(qr_panel_smem_kernel<T, PANEL_NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_dev = ctx().device;
      }
      ProfScope prof_scope_(KF_QR_PANEL);
      qr_panel_smem_kernel<T, PANEL_NB><<<1, PANEL_T, sizeof(T) * (size_t)SW * (m - j0), ctx().stream>>>(A, m, lda, tau, j0, SW, bA,
                                                                                                       btau);
      TTN_CHECK_LAUNCH();
      ctx().launches++;
    } else
    for (int b0 = 0; b0 < batch; b0 += 65535) {
      const int nb = std::min(65535, batch - b0);
      ProfScope prof_scope_(KF_QR_PANEL);
      qr_panel_kernel<T, PANEL_NB><<<nb, PANEL_T, 0, ctx().stream>>>(A + (int64_t)b0 * bA, m, n, lda, tau + (int64_t)b0 * btau,
                                                                     j0, bA, btau);
      TTN_CHECK_LAUNCH();
      ctx().launches++;
    }
    const int jhi = std::min(j0 + PANEL_NB, k);
    const int c0 = j0 + PANEL_NB;
    if (c0 < n) launch_apply<T>(A, m, lda, tau, j0, jhi, A, c0, n - c0, lda, true, batch, bA, btau, bA);
  }
}

template <class T>
void qr_apply(const T* A, int m, int k, int64_t lda, const T* tau, T* C, int nc, int64_t ldc, bool trans, int batch,
              int64_t bA, int64_t btau, int64_t bC) {
  launch_apply<T>(A, m, lda, tau, 0, k, C, 0, nc, ldc, trans, batch, bA, btau, bC);
}

template <class T>
void qr_form_q(const T* A, int m, int k, int64_t lda, const T* tau, T* Q, int64_t ldq, int batch, int64_t bA, int64_t btau,
               int64_t bQ) {
  for (int b = 0; b < batch; ++b) set_identity<T>(Q + (int64_t)b * bQ, m, k, ldq);
  launch_apply<T>(A, m, lda, tau, 0, k, Q, 0, k, ldq, false, batch, bA, btau, bQ);
}

#define INST(T)                                                                                                        \
  template void qr_factor<T>(T*, int, int, int64_t, T*, int, int64_t, int64_t);                                        \
  template void qr_apply<T>(const T*, int, int, int64_t, const T*, T*, int, int64_t, bool, int, int64_t, int64_t, int64_t); \
  template void qr_form_q<T>(const T*, int, int, int64_t, const T*, T*, int64_t, int, int64_t, int64_t, int64_t);
INST(double)
INST(zc)
#undef INST

}  // namespace ttn
