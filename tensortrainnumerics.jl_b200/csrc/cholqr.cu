// CholeskyQR2 of tall-skinny bond matrices on the FP64 tensor pipe.
//
// Serves the same call sites as the Householder QR of qr.cu where the matrix is tall and skinny (m >= 2k, k <= ~160)
// and well conditioned: the R-only preconditioner of the Jacobi SVD (`svd` behind `_svdtrunc`,
// src/tt_cross_interpolation.jl:150, called from tt_tools.jl:752) and the thin QR of a TT core in the factored bond
// split (tt.cu).  Householder QR of a 1024 x 128 panel is a chain of 128 reflector generations (BLAS-2, ~0.7 ms on
// B200); here the O(m k^2) work is three DMMA GEMMs and the sequential part is a k x k Cholesky in one SM:
//     G1 = A^H A,  R1 = chol(G1),  Q1 = A R1^-1,  G2 = Q1^H Q1,  R2 = chol(G2),  Q = Q1 R2^-1,  R = R2 R1.
// The second pass restores orthogonality to O(eps) as long as eps*cond(A)^2 << 1.  The first Cholesky reports
// min/max of diag(R1) (an upper bound of 1/cond(A)): below 1e-4 (or with a non-positive pivot) the caller falls back to
// Householder; above 0.3 (cond(A) of a few units) the first pass alone is accurate to a few tens of eps and the second one
// is skipped.  Because the diagonal only bounds the conditioning from one side, the second pass verifies itself: diag(R2)
// must be 1 within 10 % (Q1 orthonormal to O(eps cond^2)), otherwise the factorisation is rejected as well, so
// ill-conditioned and rank-deficient inputs never leave this path with a result.
#include "ttn_internal.h"

namespace ttn {

namespace {

constexpr int CQ_T = 256;
constexpr int CQ_B = 16;     // block size of the triangular inverse
constexpr int CQ_KEEP = 16;

__device__ __forceinline__ double shfl_t(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ zc shfl_t(zc v, int src) {
  return make_cuDoubleComplex(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src));
}
  // >= number of 16 x 16 blocks on a block super-diagonal (kp <= 256)

// One CTA per matrix: sums the Gram partials, factors G = R^H R (R upper), optionally inverts R (X = R^-1, upper),
// optionally multiplies R <- R * Rprev.  Shared memory: one kp x (kp+1) array; R lives in the upper triangle (diagonal
// included), X strictly-upper entries are stored transposed in the strictly lower triangle, diag(X) = 1/diag(R).
template <class T>
__global__ void __launch_bounds__(CQ_T) chol_inv_kernel(const T* __restrict__ Gp, int nsplit, int k, const T* __restrict__ Rprev,
                                                        T* __restrict__ Rout, T* __restrict__ Xout, double* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int kp = (k + CQ_B - 1) / CQ_B * CQ_B;
  const int P = kp + 1;
  T* S = reinterpret_cast<T*>(smem_raw);          // [kp][P], S[i*P + j] = element (i, j)
  double* dinv = reinterpret_cast<double*>(S + (size_t)kp * P);   // [kp] 1 / R_ii
  __shared__ double s_dmin, s_dmax;
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  const T* gp = Gp + (size_t)blockIdx.x * nsplit * k * k;
  // the partial Gram matrices are summed with all loads of a 4-element group in flight (nsplit <= 8)
  for (int idx0 = tid; idx0 < kp * kp; idx0 += 4 * CQ_T) {
    T v[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = idx0 + u * CQ_T;
      const int i = idx % kp, j = idx / kp;
      const bool in = idx < kp * kp && i < k && j < k;
#pragma unroll
      for (int z = 0; z < 8; ++z) v[u][z] = (in && z < nsplit) ? gp[(size_t)z * k * k + (size_t)j * k + i] : t_zero<T>();
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = idx0 + u * CQ_T;
      if (idx >= kp * kp) continue;
      const int i = idx % kp, j = idx / kp;
      T a = t_zero<T>();
#pragma unroll
      for (int z = 0; z < 8; ++z) a = t_add(a, v[u][z]);
      if (!(i < k && j < k)) a = (i == j) ? t_one<T>() : t_zero<T>();     // identity padding beyond k
      S[i * P + j] = a;
    }
  }
  if (tid == 0) { s_dmin = 1e300; s_dmax = 0.0; s_bad = 0; }
  __syncthreads();

  // blocked right-looking Cholesky on the upper triangle, blocks of CQ_B = 16 (nb block steps, 3 barriers each):
  //   (a) warp 0 factors the diagonal block (thread l owns column l; 16 scalar steps with warp barriers),
  //   (b) one thread per trailing column solves R11^H R12 = G12 by forward substitution,
  //   (c) rank-16 update of the trailing upper triangle, one entry per thread and 16 x 16 tile.
  const int nbk = kp / CQ_B;
  for (int jb = 0; jb < nbk; ++jb) {
    const int b0 = jb * CQ_B;
    if (tid < 32) {
      // diagonal block in registers: lane l (and its mirror l + 16) holds column l, pivots and row entries travel by
      // shuffles, everything is statically indexed (fully unrolled)
      const int l = tid & (CQ_B - 1);
      T col[CQ_B];
#pragma unroll
      for (int i = 0; i < CQ_B; ++i) col[i] = (i <= l) ? S[(b0 + i) * P + b0 + l] : t_zero<T>();
      double my_di = 1.0, dmn = 1e300, dmx = 0.0;
      bool anybad = false;
#pragma unroll
      for (int j = 0; j < CQ_B; ++j) {
        const double d2 = __shfl_sync(0xffffffffu, t_real(col[j]), j);
        const bool bad = !(d2 > 0.0) || !isfinite(d2);
        const double d = bad ? 1.0 : sqrt(d2);
        const double di = 1.0 / d;
        anybad |= bad;
        if (b0 + j < k) { dmn = fmin(dmn, d); dmx = fmax(dmx, d); }
        if (l == j) { col[j] = t_from<T>(d, 0.0); my_di = di; }
        else if (l > j) col[j] = t_scale(col[j], di);
#pragma unroll
        for (int i = j + 1; i < CQ_B; ++i) {
          const T rji = shfl_t(col[j], i);          // R[j][i]: entry j of lane i's column
          if (i <= l) col[i] = t_sub(col[i], t_mul(t_conj(rji), col[j]));
        }
      }
      if (tid < CQ_B) {
#pragma unroll
        for (int i = 0; i < CQ_B; ++i)
          if (i <= l) S[(b0 + i) * P + b0 + l] = col[i];
        dinv[b0 + l] = my_di;
      }
      if (tid == 0) {
        if (anybad) s_bad = 1;
        s_dmin = fmin(s_dmin, dmn); s_dmax = fmax(s_dmax, dmx);
      }
    }
    __syncthreads();
    for (int l = b0 + CQ_B + tid; l < kp; l += CQ_T) {
      T x[CQ_B];
#pragma unroll
      for (int i = 0; i < CQ_B; ++i) {
        T a = S[(b0 + i) * P + l];
#pragma unroll
        for (int t = 0; t < CQ_B; ++t)
          if (t < i) a = t_sub(a, t_mul(t_conj(S[(b0 + t) * P + b0 + i]), x[t]));
        x[i] = t_scale(a, dinv[b0 + i]);
      }
#pragma unroll
      for (int i = 0; i < CQ_B; ++i) S[(b0 + i) * P + l] = x[i];
    }
    __syncthreads();
    const int nt = nbk - jb - 1;
    const int ti = tid / CQ_B, tl = tid % CQ_B;       // entry (ti, tl) of a 16 x 16 tile
    for (int I = 0; I < nt; ++I)
      for (int L = I; L < nt; ++L) {
        const int i = b0 + CQ_B * (1 + I) + ti, l = b0 + CQ_B * (1 + L) + tl;
        if (l >= i) {
          T a = S[i * P + l];
#pragma unroll
          for (int t = 0; t < CQ_B; ++t) a = t_sub(a, t_mul(t_conj(S[(b0 + t) * P + i]), S[(b0 + t) * P + l]));
          S[i * P + l] = a;
        }
      }
    __syncthreads();
  }

  if (Rout != nullptr) {
    T* ro = Rout + (size_t)blockIdx.x * k * k;
    if (Rprev == nullptr) {
      for (int idx = tid; idx < k * k; idx += CQ_T) {
        const int i = idx % k, j = idx / k;
        ro[idx] = (i <= j) ? S[i * P + j] : t_zero<T>();
      }
    } else {
      const T* rp = Rprev + (size_t)blockIdx.x * k * k;
      for (int idx = tid; idx < k * k; idx += CQ_T) {
        const int i = idx % k, j = idx / k;
        T a = t_zero<T>();
        for (int l = i; l <= j; ++l) t_fma(a, S[i * P + l], rp[(size_t)j * k + l]);
        ro[idx] = a;                                // zero below the diagonal (empty sum)
      }
    }
  }
  if (tid == 0 && status != nullptr) {
    status[2 * blockIdx.x] = s_bad ? -1.0 : s_dmin / s_dmax;
    status[2 * blockIdx.x + 1] = s_dmax;
  }

  if (Xout == nullptr) return;
  // X = R^-1 by blocks of CQ_B.  Diagonal blocks first (one thread per column, back-substitution inside the block) ...
  const int nb = kp / CQ_B;
  if (tid < kp) {
    const int c = tid, b0 = (c / CQ_B) * CQ_B;
    // column c of the diagonal block: x[c] = 1/R[c][c]; x[i] = -(sum_{l=i+1..c} R[i][l] x[l]) / R[i][i], i = c-1 .. b0
    T x[CQ_B];
    const int lc = c - b0;
    x[lc] = t_from<T>(dinv[c], 0.0);
    for (int li = lc - 1; li >= 0; --li) {
      T a = t_zero<T>();
      for (int ll = li + 1; ll <= lc; ++ll) t_fma(a, S[(b0 + li) * P + b0 + ll], x[ll]);
      x[li] = t_scale(a, -dinv[b0 + li]);
    }
    // the strictly-upper entries of X go (transposed) into the strictly lower triangle; diag(X) = dinv
    for (int li = 0; li < lc; ++li) S[c * P + b0 + li] = x[li];
  }
  __syncthreads();
  auto Xat = [&](int i, int j) -> T { return i == j ? t_from<T>(dinv[i], 0.0) : S[j * P + i]; };   // i < j or i == j
  // ... then block super-diagonals d = 1 .. nb-1:  X[I][J] = -X[I][I] * sum_{L=I+1..J} R[I][L] X[L][J],  J = I + d
  for (int d = 1; d < nb; ++d) {
    const int nblk = nb - d;
    // phase 1: W[I] = sum_L R[I][L] X[L][J]  (16 x 16 per block) into registers, then to the target (lower) slots
    for (int e = tid; e < nblk * CQ_B * CQ_B; e += CQ_T) {
      const int I = e / (CQ_B * CQ_B), li = (e / CQ_B) % CQ_B, lj = e % CQ_B;
      const int J = I + d, i = I * CQ_B + li, j = J * CQ_B + lj;
      T a = t_zero<T>();
      for (int l = (I + 1) * CQ_B; l <= j; ++l) t_fma(a, S[i * P + l], Xat(l, j));
      S[j * P + i] = a;                            // slot of X[i][j] (transposed storage) holds W for now
    }
    __syncthreads();
    // phase 2: X[I][J] = -X[I][I] * W  (X[I][I] upper triangular 16 x 16)
    T keep[CQ_KEEP];                               // results are parked in registers: W is still being read by other threads
    int cnt = 0;
    for (int e = tid; e < nblk * CQ_B * CQ_B; e += CQ_T, ++cnt) {
      const int I = e / (CQ_B * CQ_B), li = (e / CQ_B) % CQ_B, lj = e % CQ_B;
      const int J = I + d, i = I * CQ_B + li, j = J * CQ_B + lj;
      T a = t_zero<T>();
      for (int ll = li; ll < CQ_B; ++ll) t_fma(a, Xat(i, I * CQ_B + ll), S[j * P + I * CQ_B + ll]);
      keep[cnt] = t_scale(a, -1.0);
    }
    __syncthreads();
    cnt = 0;
    for (int e = tid; e < nblk * CQ_B * CQ_B; e += CQ_T, ++cnt) {
      const int I = e / (CQ_B * CQ_B), li = (e / CQ_B) % CQ_B, lj = e % CQ_B;
      const int J = I + d, i = I * CQ_B + li, j = J * CQ_B + lj;
      S[j * P + i] = keep[cnt];
    }
    __syncthreads();
  }
  T* xo = Xout + (size_t)blockIdx.x * k * k;
  for (int idx = tid; idx < k * k; idx += CQ_T) {
    const int i = idx % k, j = idx / k;
    xo[idx] = (i < j) ? S[j * P + i] : (i == j ? t_from<T>(dinv[i], 0.0) : t_zero<T>());
  }
}

template <class T>
size_t chol_smem(int k) {
  const int kp = (k + CQ_B - 1) / CQ_B * CQ_B;
  return sizeof(T) * (size_t)kp * (kp + 1) + sizeof(double) * kp;
}

template <class T>
void gram_partials(const T* A, int m, int k, int64_t lda, int64_t bA, int nsplit, T* Gp, int batch) {
  GemmArgs g;   // Gp[b][z] = A[z-th row chunk]^H A[z-th row chunk]
  g.M = k; g.N = k; g.K = m / nsplit;
  g.A = A; g.sAm = lda; g.sAk = 1; g.conjA = true; g.bA1 = m / nsplit; g.bA2 = bA;
  g.B = A; g.sBk = 1; g.sBn = lda; g.bB1 = m / nsplit; g.bB2 = bA;
  g.C = Gp; g.sCm = 1; g.sCn = k; g.bC1 = (int64_t)k * k; g.bC2 = (int64_t)nsplit * k * k;
  g.batch1 = nsplit; g.batch2 = batch;
  gemm<T>(g);
}

}  // namespace

template <class T>
bool cholqr2_fits(int m, int k) {
  return k >= 8 && m >= 2 * k && chol_smem<T>(k) <= 220 * 1024;
}

// A (m x k, lda, batch stride bA) = Q R.  R: k x k upper triangular (dense, ld k, zeros below), batch stride k*k.
// Q (optional): m x k, ldq, batch stride bQ.  Returns false if any matrix of the batch is rejected (ill conditioned /
// not positive definite): outputs are then undefined and the caller must use the Householder path.
namespace {
template <class T>
bool cholqr2_impl(const T* A, int m, int k, int64_t lda, int64_t bA, T* R, T* Q, int64_t ldq, int64_t bQ, int batch, double* h_diag);
}

// Two column panels when the k x k Cholesky does not fit one SM's shared memory (ComplexF64 beyond k = 117, Float64 beyond
// k = 165) but k/2 does: block classical Gram-Schmidt with re-orthogonalisation around CholeskyQR2 of each panel,
//     [Q1, R11] = cholqr2(A1);  twice: { S = Q1^H P;  P -= Q1 S;  R12 += S }  (P starts as A2);  [Q2, R22] = cholqr2(P),
// all GEMMs.  The panels are accepted or rejected by their own conditioning test; a rejection sends the caller to Householder.
template <class T>
bool cholqr2_two_panel(const T* A, int m, int k, int64_t lda, int64_t bA, T* R, T* Q, int64_t ldq, int64_t bQ, int batch) {
  const int k1 = (k / 2 + CQ_B - 1) / CQ_B * CQ_B, k2 = k - k1;
  if (k2 < 8 || m < 2 * k || !cholqr2_fits<T>(m, k1) || !cholqr2_fits<T>(m, k2)) return false;
  DevBuf Qw;
  if (Q == nullptr) {                                  // R-only call: the panels of Q are still needed as projectors
    Qw.alloc(sizeof(T) * (size_t)m * k * batch);
    Q = Qw.as<T>(); ldq = m; bQ = (int64_t)m * k;
  }
  const bool want_q = Qw.p == nullptr;
  DevBuf R11(sizeof(T) * (size_t)k1 * k1 * batch), R22(sizeof(T) * (size_t)k2 * k2 * batch);
  DevBuf R12(sizeof(T) * (size_t)k1 * k2 * batch), S2(sizeof(T) * (size_t)k1 * k2 * batch);
  std::vector<double> d1(2 * (size_t)batch), d2(2 * (size_t)batch);     // (min, max) of diag(R1) of each panel's first pass
  if (!cholqr2_impl<T>(A, m, k1, lda, bA, R11.as<T>(), Q, ldq, bQ, batch, d1.data())) return false;
  T* P = Q + (int64_t)k1 * ldq;
  {
    Copy4 c; c.n0 = m; c.n1 = k2; c.n2 = batch; c.s0 = 1; c.s1 = lda; c.s2 = bA; c.d0 = 1; c.d1 = ldq; c.d2 = bQ;
    copy4<T>(A + (int64_t)k1 * lda, P, c);
  }
  for (int pass = 0; pass < 2; ++pass) {
    T* S = pass == 0 ? R12.as<T>() : S2.as<T>();
    GemmArgs g;   // S = Q1^H P
    g.M = k1; g.N = k2; g.K = m;
    g.A = Q; g.sAm = ldq; g.sAk = 1; g.conjA = true; g.bA1 = bQ;
    g.B = P; g.sBk = 1; g.sBn = ldq; g.bB1 = bQ;
    g.C = S; g.sCm = 1; g.sCn = k1; g.bC1 = (int64_t)k1 * k2;
    g.batch1 = batch;
    gemm<T>(g);
    GemmArgs u;   // P -= Q1 S
    u.M = m; u.N = k2; u.K = k1;
    u.A = Q; u.sAm = 1; u.sAk = ldq; u.bA1 = bQ;
    u.B = S; u.sBk = 1; u.sBn = k1; u.bB1 = (int64_t)k1 * k2;
    u.C = P; u.sCm = 1; u.sCn = ldq; u.bC1 = bQ;
    u.alpha = -1.0; u.beta = 1.0;
    u.batch1 = batch;
    gemm<T>(u);
  }
  axpy<T>((int64_t)k1 * k2 * batch, t_one<T>(), S2.as<T>(), R12.as<T>());
  DevBuf Q2;
  if (want_q) Q2.alloc(sizeof(T) * (size_t)m * k2 * batch);
  if (!cholqr2_impl<T>(P, m, k2, ldq, bQ, R22.as<T>(), want_q ? Q2.as<T>() : nullptr, m, (int64_t)m * k2, batch, d2.data()))
    return false;
  // the conditioning estimate of the whole matrix is the diagonal spread of the assembled R (each panel only saw its own)
  for (int b = 0; b < batch; ++b) {
    const double ratio = std::min(d1[2 * b], d2[2 * b]) / std::max(d1[2 * b + 1], d2[2 * b + 1]);
    if (!(ratio >= 1e-4)) {
      if (debug_svd()) fprintf(stderr, "[ttn] cholqr2 %d x %d (two panels): min/max diag(R) = %.3g -> rejected\n", m, k, ratio);
      return false;
    }
  }
  if (want_q) {
    Copy4 c; c.n0 = m; c.n1 = k2; c.n2 = batch; c.s0 = 1; c.s1 = m; c.s2 = (int64_t)m * k2; c.d0 = 1; c.d1 = ldq; c.d2 = bQ;
    copy4<T>(Q2.as<T>(), P, c);
  }
  // R = [R11 R12; 0 R22]
  const int64_t kk = (int64_t)k * k;
  fill<T>(R, kk * batch, t_zero<T>());
  Copy4 a; a.n0 = k1; a.n1 = k1; a.n2 = batch; a.s0 = 1; a.s1 = k1; a.s2 = (int64_t)k1 * k1; a.d0 = 1; a.d1 = k; a.d2 = kk;
  copy4<T>(R11.as<T>(), R, a);
  Copy4 b; b.n0 = k1; b.n1 = k2; b.n2 = batch; b.s0 = 1; b.s1 = k1; b.s2 = (int64_t)k1 * k2; b.d0 = 1; b.d1 = k; b.d2 = kk;
  copy4<T>(R12.as<T>(), R + (int64_t)k1 * k, b);
  Copy4 c; c.n0 = k2; c.n1 = k2; c.n2 = batch; c.s0 = 1; c.s1 = k2; c.s2 = (int64_t)k2 * k2; c.d0 = 1; c.d1 = k; c.d2 = kk;
  copy4<T>(R22.as<T>(), R + (int64_t)k1 * k + k1, c);
  return true;
}

template <class T>
bool cholqr2(const T* A, int m, int k, int64_t lda, int64_t bA, T* R, T* Q, int64_t ldq, int64_t bQ, int batch) {
  if (batch <= 0) return false;
  if (!cholqr2_fits<T>(m, k)) return cholqr2_two_panel<T>(A, m, k, lda, bA, R, Q, ldq, bQ, batch);
  return cholqr2_impl<T>(A, m, k, lda, bA, R, Q, ldq, bQ, batch, nullptr);
}

namespace {
template <class T>
bool cholqr2_impl(const T* A, int m, int k, int64_t lda, int64_t bA, T* R, T* Q, int64_t ldq, int64_t bQ, int batch, double* h_diag) {
  if (!cholqr2_fits<T>(m, k) || batch <= 0) return false;
  int nsplit = 1;
  if (batch * ((k + 63) / 64) * ((k + 63) / 64) < ctx().sm_count)
    for (int s : {8, 4, 2})
      if (m % s == 0 && m / s >= 64) { nsplit = s; break; }
  const size_t smem = chol_smem<T>(k);
  static int attr_dev = -1;   // function attributes are per device (ttn_init may re-bind)
  if (attr_dev != ctx().device) {
    TTN_CUDA(cudaFuncSetAttribute(chol_inv_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    attr_dev = ctx().device;
  }
  const size_t kk = (size_t)k * k;
  DevBuf Gp(sizeof(T) * kk * nsplit * batch), R1(sizeof(T) * kk * batch), X(sizeof(T) * kk * batch), st(sizeof(double) * 2 * batch);
  gram_partials<T>(A, m, k, lda, bA, nsplit, Gp.as<T>(), batch);
  // first Cholesky.  The inverse is only computed when an explicit Q is wanted; an R-only call (SVD preconditioner) can stop
  // after this kernel if the matrix turns out to be well conditioned (below).
  {
    ProfScope prof_scope_(KF_QR_PANEL);
    chol_inv_kernel<T><<<batch, CQ_T, smem, ctx().stream>>>(Gp.as<T>(), nsplit, k, nullptr, R1.as<T>(), Q ? X.as<T>() : nullptr,
                                                           st.as<double>());
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
  std::vector<double> h(2 * (size_t)batch);
  read_back(h.data(), st.p, sizeof(double) * 2 * batch);
  double worst = 1.0;
  for (int b = 0; b < batch; ++b) {
    const double v = h[2 * b];
    if (!(v >= 1e-4)) return false;                 // ill conditioned / not positive definite: Householder path
    worst = std::min(worst, v);
    if (h_diag) { h_diag[2 * b] = v * h[2 * b + 1]; h_diag[2 * b + 1] = h[2 * b + 1]; }
  }
  // One pass is enough when cond(A) is small: the loss of CholeskyQR is eps*cond^2 (relative, in R and in Q^H Q - I);
  // min/max diag(R1) >= 0.3 means cond(A) of a few units (cfg2's bonds: 0.39 ... 0.78), i.e. a few tens of eps — the level of
  // the rounding of the K = 512 GEMMs around it.
  // An explicit Q always takes the second pass: diag(R1) bounds cond(A) from one side only (a Kahan-like matrix has equal
  // diagonals and a growing R^-1), and only the second Gram matrix verifies Q1^H Q1 = I.  The R-only call feeds the Jacobi
  // SVD, whose result is checked through the singular values themselves.
  const bool single = worst >= 0.3 && Q == nullptr;
  if (debug_svd()) fprintf(stderr, "[ttn] cholqr2 %d x %d batch %d: min/max diag(R1) = %.3g -> %s\n", m, k, batch, worst, single ? "one pass" : "two passes");
  if (single) {
    TTN_CUDA(cudaMemcpyAsync(R, R1.p, sizeof(T) * kk * batch, cudaMemcpyDeviceToDevice, ctx().stream));
    if (Q != nullptr) {
      GemmArgs g;   // Q = A X1
      g.M = m; g.N = k; g.K = k;
      g.A = A; g.sAm = 1; g.sAk = lda; g.bA1 = bA;
      g.B = X.p; g.sBk = 1; g.sBn = k; g.bB1 = (int64_t)kk;
      g.C = Q; g.sCm = 1; g.sCn = ldq; g.bC1 = bQ;
      g.batch1 = batch;
      gemm<T>(g);
    }
    return true;                                     // (workspaces are stream-ordered: no sync needed to release them)
  }
  if (Q == nullptr) {
    // second pass needs X1 = R1^-1 after all: redo the (cheap, k x k) factorisation with the inverse
    ProfScope prof_scope_(KF_QR_PANEL);
    chol_inv_kernel<T><<<batch, CQ_T, smem, ctx().stream>>>(Gp.as<T>(), nsplit, k, nullptr, R1.as<T>(), X.as<T>(), nullptr);
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
  DevBuf R2(sizeof(T) * kk * batch), Q1(sizeof(T) * (size_t)m * k * batch);
  {
    GemmArgs g;   // Q1 = A X1
    g.M = m; g.N = k; g.K = k;
    g.A = A; g.sAm = 1; g.sAk = lda; g.bA1 = bA;
    g.B = X.p; g.sBk = 1; g.sBn = k; g.bB1 = (int64_t)kk;
    g.C = Q1.p; g.sCm = 1; g.sCn = m; g.bC1 = (int64_t)m * k;
    g.batch1 = batch;
    gemm<T>(g);
  }
  gram_partials<T>(Q1.as<T>(), m, k, m, (int64_t)m * k, nsplit, Gp.as<T>(), batch);
  {
    ProfScope prof_scope_(KF_QR_PANEL);
    chol_inv_kernel<T><<<batch, CQ_T, smem, ctx().stream>>>(Gp.as<T>(), nsplit, k, nullptr, R2.as<T>(), Q ? X.as<T>() : nullptr,
                                                           st.as<double>());
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
  // min/max diag(R1) only bounds cond(A) from below.  The second Gram matrix is the direct evidence: Q1^H Q1 = I + O(eps cond^2),
  // so diag(R2) must sit at 1; a spread means the first pass lost orthogonality (cond(A) >~ 1e7) and the result is rejected.
  read_back(h.data(), st.p, sizeof(double) * 2 * batch);
  for (int b = 0; b < batch; ++b) {
    const double v = h[2 * b];
    if (!(v >= 0.9)) {
      if (debug_svd()) fprintf(stderr, "[ttn] cholqr2 %d x %d: second pass min/max diag(R2) = %.3g -> rejected\n", m, k, v);
      return false;
    }
  }
  {
    GemmArgs g;   // R = R2 R1
    g.M = k; g.N = k; g.K = k;
    g.A = R2.p; g.sAm = 1; g.sAk = k; g.bA1 = (int64_t)kk;
    g.B = R1.p; g.sBk = 1; g.sBn = k; g.bB1 = (int64_t)kk;
    g.C = R; g.sCm = 1; g.sCn = k; g.bC1 = (int64_t)kk;
    g.batch1 = batch;
    gemm<T>(g);
  }
  if (Q != nullptr) {
    GemmArgs g;   // Q = Q1 X2
    g.M = m; g.N = k; g.K = k;
    g.A = Q1.p; g.sAm = 1; g.sAk = m; g.bA1 = (int64_t)m * k;
    g.B = X.p; g.sBk = 1; g.sBn = k; g.bB1 = (int64_t)kk;
    g.C = Q; g.sCm = 1; g.sCn = ldq; g.bC1 = bQ;
    g.batch1 = batch;
    gemm<T>(g);
  }
  return true;
}
}  // namespace

template bool cholqr2_fits<double>(int, int);
template bool cholqr2_fits<zc>(int, int);
template bool cholqr2<double>(const double*, int, int, int64_t, int64_t, double*, double*, int64_t, int64_t, int);
template bool cholqr2<zc>(const zc*, int, int, int64_t, int64_t, zc*, zc*, int64_t, int64_t, int);

}  // namespace ttn
