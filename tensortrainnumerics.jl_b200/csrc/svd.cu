// Left singular vectors + singular values of a bond-sized matrix: Householder QR preconditioning followed
// by one-sided Jacobi on the square triangular factor (SURVEY.md §7.3 "SVD accuracy vs speed").
//
//   p <= q (wide / square):  Theta^H = Q~ R   ->  L = R^H (p x p);  Jacobi on the columns of L:  L V = U Sigma
//   p >  q (tall)         :  Theta   = Q  R   ->  Jacobi on the columns of R: R V = U_R Sigma;  U Sigma = Q [U_R Sigma; 0]
//
// Only U·Sigma (orthogonal columns, unsorted) and the sorted singular values are produced; callers obtain the
// other factor by projection (Sigma·V^H = U^H·Theta, a DMMA GEMM), which is exact for any orthonormal U and needs
// neither V accumulation nor a division by small singular values.
#include "ttn_internal.h"

namespace ttn {

bool debug_svd() {
  static const bool on = getenv("TTN_DEBUG_SVD") != nullptr;
  return on;
}

namespace {

// squared column norms of W (m x n, ld m): one warp per column
template <class T>
__global__ void col_norms2_kernel(const T* __restrict__ W, int m, int n, double* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const T* x = W + (int64_t)warp * m;
  double a = 0.0;
  for (int i = lane; i < m; i += 32) a += t_abs2(x[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (lane == 0) out[warp] = a;
}

// dst[perm[i], c] = src[i, c]   (p x k, ld p)
template <class T>
__global__ void scatter_rows_kernel(const T* __restrict__ src, T* __restrict__ dst, int p, int k, const int* __restrict__ perm) {
  const int64_t total = (int64_t)p * k;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx % p);
    const int64_t c = idx / p;
    dst[perm[i] + c * p] = src[idx];
  }
}

// Range normalisation of the working copy.  The rotation tests of one-sided Jacobi multiply four entries (|x_p^H x_q|^2
// against ||x_p||^2 ||x_q||^2): from a largest entry of about 1e-73 on they underflow to zero, from about 1e+77 on they
// overflow, and either way the rotation is skipped and the columns are taken as orthogonal.  A matrix whose largest entry
// lies outside [2^-64, 2^64] is therefore scaled by 2^-e (largest entry in [1/2, 1)) before the factorisation and U Sigma,
// Sigma by 2^e after it; powers of two scale exactly, and a matrix inside the range is not touched (e = 0).
__host__ __device__ inline double amax_of(double a) { return fabs(a); }
__host__ __device__ inline double amax_of(zc a) { return fmax(fabs(a.x), fabs(a.y)); }

// amax[b] = max |W_b| (as the bit pattern of a non-negative double, which orders like the value); grid (nblk, batch)
template <class T>
__global__ void amax_kernel(const T* __restrict__ W, int64_t n, int64_t bW, unsigned long long* __restrict__ amax) {
  __shared__ double red[32];
  W += blockIdx.y * bW;
  double m = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    m = fmax(m, amax_of(W[i]));                      // fmax drops NaN: a non-finite input is reported by the Jacobi stage
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, red[w]);
    atomicMax(amax + blockIdx.y, (unsigned long long)__double_as_longlong(m));
  }
}

__device__ inline int range_exponent(unsigned long long bits) {
  const double m = __longlong_as_double((long long)bits);
  if (!(m > 0.0) || !isfinite(m) || (m >= 0x1p-64 && m <= 0x1p64)) return 0;
  int e;
  frexp(m, &e);
  return max(e, -1020);                              // 2^-e stays finite for a subnormal largest entry
}

// W_b *= 2^-e_b (sign = -1) or 2^e_b (sign = +1); with norms, the k norms of matrix b as well
template <class T>
__global__ void pow2_scale_kernel(T* __restrict__ W, int64_t n, int64_t bW, const unsigned long long* __restrict__ amax, int sign,
                                  double* __restrict__ norms, int k) {
  const int e = range_exponent(amax[blockIdx.y]);
  if (e == 0) return;
  const double s = ldexp(1.0, sign * e);
  W += blockIdx.y * bW;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) W[i] = t_scale(W[i], s);
  if (norms && blockIdx.x == 0)
    for (int j = threadIdx.x; j < k; j += blockDim.x) norms[blockIdx.y * (int64_t)k + j] *= s;
}

inline int range_blocks(int64_t n) { return (int)std::min<int64_t>(128, std::max<int64_t>(1, (n + 4095) / 4096)); }

// finds the scale of every matrix of the batch and applies 2^-e to the working copy W (n entries per matrix, stride bW)
template <class T>
void range_normalise(T* W, int64_t n, int64_t bW, int batch, DevBuf& amax) {
  amax.alloc(sizeof(unsigned long long) * (size_t)batch);
  TTN_CUDA(cudaMemsetAsync(amax.p, 0, amax.bytes, ctx().stream));
  const dim3 grid(range_blocks(n), batch);
  amax_kernel<T><<<grid, 256, 0, ctx().stream>>>(W, n, bW, amax.as<unsigned long long>());
  TTN_CHECK_LAUNCH();
  pow2_scale_kernel<T><<<grid, 256, 0, ctx().stream>>>(W, n, bW, amax.as<unsigned long long>(), -1, nullptr, 0);
  TTN_CHECK_LAUNCH();
  ctx().launches += 2;
}

}  // namespace

template <class T>
void svd_left(const T* Theta, int p, int q, int64_t rs, int64_t cs, bool conj, SvdLeft& out, int batch, int64_t bT) {
  ttn_assert(p > 0 && q > 0 && batch > 0, 2, "svd_left: empty matrix");
  const int k = std::min(p, q);
  out.p = p; out.q = q; out.k = k;
  out.norms.alloc(sizeof(double) * (size_t)k * batch);
  out.X.alloc(sizeof(T) * (size_t)p * k * batch);
  T* X = out.X.as<T>();
  const int64_t bX = (int64_t)p * k;
  DevBuf amax;   // largest entry of every matrix, for the range normalisation of the working copy

  // Square bond matrices of the size DMRG / MALS produce are preconditioned like wide ones (Theta^H = Q R, Jacobi on R^H):
  // their spectra decay, and one-sided Jacobi applied directly needs 17-32 sweeps on them against ~10 on the triangular
  // factor (Drmac-Veselic preconditioning); small squares stay direct, the QR would cost more than the sweeps it saves.
  const bool direct = (p == q) && p < 256;
  if (direct) {
    Copy4 c; c.n0 = p; c.n1 = q; c.n2 = batch; c.s0 = rs; c.s1 = cs; c.s2 = bT; c.d0 = 1; c.d1 = p; c.d2 = bX; c.conj = conj;
    copy4<T>(Theta, X, c);
    range_normalise<T>(X, bX, bX, batch, amax);
    out.sweeps = jacobi_orth<T>(X, p, p, p, out.norms.as<double>(), batch, bX, k);
  } else if (p <= q) {
    // W (q x p) = Theta_eff^H
    DevBuf W(sizeof(T) * (size_t)q * p * batch);
    const int64_t bW = (int64_t)q * p;
    Copy4 c; c.n0 = q; c.n1 = p; c.n2 = batch; c.s0 = cs; c.s1 = rs; c.s2 = bT; c.d0 = 1; c.d1 = q; c.d2 = bW; c.conj = !conj;
    copy4<T>(Theta, W.as<T>(), c);
    range_normalise<T>(W.as<T>(), bW, bW, batch, amax);
    // Poor man's column pivoting: order the columns of W = Theta^H (the rows of Theta) by decreasing norm before the unpivoted
    // QR, so that R^H comes out closer to the graded form on which one-sided Jacobi converges fastest (Drmac-Veselic); the
    // row permutation is undone on U Sigma at the end.  DMRG sweep at chi = 1024: 12-17 sweeps per 2048^2 SVD (mean 14.6)
    // become 12-16 (mean 13.3), Jacobi time -9 %.
    const bool sorted = batch == 1 && p >= 256;
    DevBuf dperm;
    if (sorted) {
      DevBuf n2(sizeof(double) * p);
      col_norms2_kernel<T><<<(p + 7) / 8, 256, 0, ctx().stream>>>(W.as<T>(), q, p, n2.as<double>());
      TTN_CHECK_LAUNCH();
      ctx().launches++;
      std::vector<double> hn(p);
      read_back(hn.data(), n2.p, sizeof(double) * p);
      for (double& v : hn)
        if (!std::isfinite(v)) v = 0.0;   // keeps the comparator a strict weak order; the Jacobi stage reports the NaN
      std::vector<int> perm(p);
      for (int j = 0; j < p; ++j) perm[j] = j;
      std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return hn[a] > hn[b]; });
      std::vector<double> ones(p, 1.0);
      dperm.alloc(sizeof(int) * p);
      DevBuf dones(sizeof(double) * p), W2(sizeof(T) * (size_t)q * p);
      TTN_CUDA(cudaMemcpyAsync(dperm.p, perm.data(), sizeof(int) * p, cudaMemcpyHostToDevice, ctx().stream));
      TTN_CUDA(cudaMemcpyAsync(dones.p, ones.data(), sizeof(double) * p, cudaMemcpyHostToDevice, ctx().stream));
      gather_cols<T>(W.as<T>(), q, q, dperm.as<int>(), dones.as<double>(), p, W2.as<T>(), 1, q);
      TTN_CUDA(cudaStreamSynchronize(ctx().stream));   // perm / ones are host stack data
      W = std::move(W2);
    }
    DevBuf Rb(sizeof(T) * (size_t)p * p * batch);
    const bool have_r = cholqr2<T>(W.as<T>(), q, p, q, bW, Rb.as<T>(), nullptr, 0, 0, batch);
    if (!have_r) {
      DevBuf tau(sizeof(T) * (size_t)p * batch);
      qr_factor<T>(W.as<T>(), q, p, q, tau.as<T>(), batch, bW, p);
    }
    // X = R^H (lower triangular p x p): X[i,j] = conj(R[j,i]), j <= i
    Copy4 t; t.n0 = p; t.n1 = p; t.n2 = batch; t.s0 = 1; t.s1 = have_r ? p : q; t.s2 = have_r ? bX : bW;
    t.d0 = p; t.d1 = 1; t.d2 = bX; t.conj = true; t.tri = 1;
    copy4<T>(have_r ? Rb.as<T>() : W.as<T>(), X, t);
    out.sweeps = jacobi_orth<T>(X, p, p, p, out.norms.as<double>(), batch, bX, k);
    if (sorted) {
      DevBuf Xs(sizeof(T) * (size_t)p * k);
      scatter_rows_kernel<T><<<ctx().sm_count * 4, 256, 0, ctx().stream>>>(X, Xs.as<T>(), p, k, dperm.as<int>());
      TTN_CHECK_LAUNCH();
      ctx().launches++;
      out.X = std::move(Xs);
      X = out.X.as<T>();
    }
  } else {
    DevBuf W(sizeof(T) * (size_t)p * q * batch);
    const int64_t bW = (int64_t)p * q;
    Copy4 c; c.n0 = p; c.n1 = q; c.n2 = batch; c.s0 = rs; c.s1 = cs; c.s2 = bT; c.d0 = 1; c.d1 = p; c.d2 = bW; c.conj = conj;
    copy4<T>(Theta, W.as<T>(), c);
    range_normalise<T>(W.as<T>(), bW, bW, batch, amax);
    DevBuf Xr(sizeof(T) * (size_t)q * q * batch), Qe(sizeof(T) * (size_t)p * q * batch);
    const int64_t bR = (int64_t)q * q;
    const bool have_q = cholqr2<T>(W.as<T>(), p, q, p, bW, Xr.as<T>(), Qe.as<T>(), p, bW, batch);
    if (have_q) {
      out.sweeps = jacobi_orth<T>(Xr.as<T>(), q, q, q, out.norms.as<double>(), batch, bR, k);
      GemmArgs g;   // X = Q (R V) = Q * Xr
      g.M = p; g.N = q; g.K = q;
      g.A = Qe.p; g.sAm = 1; g.sAk = p; g.bA1 = bW;
      g.B = Xr.p; g.sBk = 1; g.sBn = q; g.bB1 = bR;
      g.C = X; g.sCm = 1; g.sCn = p; g.bC1 = bX;
      g.batch1 = batch;
      gemm<T>(g);
    } else {
      Qe.release();
      DevBuf tau(sizeof(T) * (size_t)q * batch);
      qr_factor<T>(W.as<T>(), p, q, p, tau.as<T>(), batch, bW, q);
      // Xr (q x q) = R
      Copy4 t; t.n0 = q; t.n1 = q; t.n2 = batch; t.s0 = 1; t.s1 = p; t.s2 = bW; t.d0 = 1; t.d1 = q; t.d2 = bR; t.tri = 1;
      copy4<T>(W.as<T>(), Xr.as<T>(), t);
      out.sweeps = jacobi_orth<T>(Xr.as<T>(), q, q, q, out.norms.as<double>(), batch, bR, k);
      // X = Q [Xr; 0]
      fill<T>(X, (int64_t)p * q * batch, t_zero<T>());
      Copy4 u; u.n0 = q; u.n1 = q; u.n2 = batch; u.s0 = 1; u.s1 = q; u.s2 = bR; u.d0 = 1; u.d1 = p; u.d2 = bX;
      copy4<T>(Xr.as<T>(), X, u);
      qr_apply<T>(W.as<T>(), p, q, p, tau.as<T>(), X, q, p, false, batch, bW, q, bX);
    }
  }

  {   // undo the range normalisation on U Sigma and Sigma
    const dim3 grid(range_blocks(bX), batch);
    pow2_scale_kernel<T><<<grid, 256, 0, ctx().stream>>>(X, bX, bX, amax.as<unsigned long long>(), 1, out.norms.as<double>(), k);
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
  if (debug_svd()) fprintf(stderr, "[ttn] svd_left %d x %d batch %d: %d Jacobi sweeps\n", p, q, batch, out.sweeps);
  // singular values to the host, sorted descending per batch element
  std::vector<double> h((size_t)k * batch);
  read_back(h.data(), out.norms.p, sizeof(double) * h.size());
  for (double v : h)
    if (!std::isfinite(v)) throw Error(5, "svd_left: the Jacobi SVD produced a non-finite singular value (non-finite input?)");
  out.sigma.resize(h.size());
  out.perm.resize(h.size());
  std::vector<int> idx(k);
  for (int b = 0; b < batch; ++b) {
    const double* hb = h.data() + (size_t)b * k;
    for (int j = 0; j < k; ++j) idx[j] = j;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int c2) { return hb[a] > hb[c2]; });
    for (int j = 0; j < k; ++j) {
      out.perm[(size_t)b * k + j] = idx[j];
      out.sigma[(size_t)b * k + j] = hb[idx[j]];
    }
  }
}

template void svd_left<double>(const double*, int, int, int64_t, int64_t, bool, SvdLeft&, int, int64_t);
template void svd_left<zc>(const zc*, int, int, int64_t, int64_t, bool, SvdLeft&, int, int64_t);

}  // namespace ttn
