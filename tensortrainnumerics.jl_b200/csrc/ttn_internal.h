// Internal declarations shared by the sm_100a kernels and the host-side sweep drivers of libttn_b200.
// Nothing in here crosses the C ABI (see include/ttn_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cuComplex.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <stdexcept>
#include <algorithm>
#include <complex>

namespace ttn {

typedef cuDoubleComplex zc;

// ---------------------------------------------------------------------------------------------
// errors: C++ exceptions inside the library, converted to status codes at the ABI boundary
// ---------------------------------------------------------------------------------------------
struct Error : public std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define TTN_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      throw ::ttn::Error(6, std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " +    \
                                __FILE__ + ":" + std::to_string(__LINE__));                   \
  } while (0)

#define TTN_CHECK_LAUNCH() TTN_CUDA(cudaGetLastError())

inline void ttn_assert(bool c, int code, const char* msg) {
  if (!c) throw Error(code, msg);
}

// ---------------------------------------------------------------------------------------------
// context: one device, one stream, launch counter
// ---------------------------------------------------------------------------------------------
enum KernelFamily { KF_GEMM = 0, KF_COPY = 1, KF_APPLY = 2, KF_QR_PANEL = 3, KF_QR_APPLY = 4, KF_JACOBI = 5, KF_REDUCE = 6,
                    KF_GATHER = 7, KF_COUNT = 8 };
struct ProfRec { int fam; cudaEvent_t a, b; };
struct Context {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // host <-> device copies that overlap the compute stream (created on first use)
  int sm_count = 148;
  long long launches = 0;  // kernels launched by this library since the last reset
  bool inited = false;
  bool prof_on = false;    // per-kernel-family CUDA-event timing (bench.py roofline pass only)
  std::vector<ProfRec> prof;
  int last_jacobi_sweeps = 0;  // diagnostics: sweeps used by the most recent Jacobi SVD (batch element 0)
  double flops_gemm = 0.0, flops_heig = 0.0;   // real FLOPs the DMMA GEMMs / the Gram-path eigensolver were asked to execute (roofline accounting)
  long long gram_calls = 0, gram_fallbacks = 0;   // tt_compress! calls that took the Gram path / were redone by the Jacobi path
  int gram_last_flags = 0;
  bool gemm_bulk = true;            // TMA-staged (cp.async.bulk + mbarrier) big-tile GEMM when the operands allow it
  bool gemm_thin = true;            // streaming kernel for thin right-multiplications (N, K <= 32, shared B): the middle contraction of the local operators
  bool gram_compress = true;        // Gram path of tt_compress! for truncerr == 0 (heig.cu)
  void* host_stage = nullptr;       // pinned staging area of the small device -> host reads (flags, singular values): a pageable
  size_t host_stage_bytes = 0;      // destination would make the read a staged, driver-serialised copy that stalls other host threads
  int gram_jacobi_min = 640;        // Gram-block Jacobi (DMMA, two streams) for matrices with min(m, n) >= this (measured crossover)
};
Context& ctx();
/// true when TTN_DEBUG_SVD is set in the environment (read once): the SVD, CholeskyQR2 and Gram-path code then print diagnostics to stderr
bool debug_svd();
/// pinned host scratch of at least `bytes` bytes owned by the calling thread's context (valid until the next call)
void* host_stage(size_t bytes);
/// blocking device -> host read on the library stream; small reads go through the pinned staging area
void read_back(void* dst, const void* src, size_t bytes);
// brackets the launches of one kernel family with CUDA events on the library stream when profiling is enabled
struct ProfScope {
  bool on;
  ProfRec r;
  explicit ProfScope(int fam) : on(ctx().prof_on) {
    if (!on) return;
    r.fam = fam;
    cudaEventCreate(&r.a);
    cudaEventCreate(&r.b);
    cudaEventRecord(r.a, ctx().stream);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(r.b, ctx().stream);
    ctx().prof.push_back(r);
  }
};

void devbuf_cache_trim();   // returns the exact-size block cache of DevBuf to the stream-ordered pool
// stream-ordered device buffer (cudaMallocAsync pool on the context stream, exact-size cache for blocks >= 256 KB)
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() {}
  explicit DevBuf(size_t b) { alloc(b); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void alloc(size_t b);
  void release();
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// ---------------------------------------------------------------------------------------------
// scalar helpers (host + device) so that kernels can be written once for double and complex
// ---------------------------------------------------------------------------------------------
template <class T> struct is_cplx { static const bool value = false; };
template <> struct is_cplx<zc> { static const bool value = true; };

__host__ __device__ inline double t_real(double a) { return a; }
__host__ __device__ inline double t_real(zc a) { return a.x; }
__host__ __device__ inline double t_imag(double) { return 0.0; }
__host__ __device__ inline double t_imag(zc a) { return a.y; }
__host__ __device__ inline double t_abs2(double a) { return a * a; }
__host__ __device__ inline double t_abs2(zc a) { return a.x * a.x + a.y * a.y; }
__host__ __device__ inline double t_conj(double a) { return a; }
__host__ __device__ inline zc t_conj(zc a) { return make_cuDoubleComplex(a.x, -a.y); }
__host__ __device__ inline double t_mul(double a, double b) { return a * b; }
__host__ __device__ inline zc t_mul(zc a, zc b) { return make_cuDoubleComplex(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__host__ __device__ inline double t_add(double a, double b) { return a + b; }
__host__ __device__ inline zc t_add(zc a, zc b) { return make_cuDoubleComplex(a.x + b.x, a.y + b.y); }
__host__ __device__ inline double t_sub(double a, double b) { return a - b; }
__host__ __device__ inline zc t_sub(zc a, zc b) { return make_cuDoubleComplex(a.x - b.x, a.y - b.y); }
__host__ __device__ inline double t_scale(double a, double s) { return a * s; }
__host__ __device__ inline zc t_scale(zc a, double s) { return make_cuDoubleComplex(a.x * s, a.y * s); }
template <class T> __host__ __device__ inline T t_zero();
template <> __host__ __device__ inline double t_zero<double>() { return 0.0; }
template <> __host__ __device__ inline zc t_zero<zc>() { return make_cuDoubleComplex(0.0, 0.0); }
template <class T> __host__ __device__ inline T t_one();
template <> __host__ __device__ inline double t_one<double>() { return 1.0; }
template <> __host__ __device__ inline zc t_one<zc>() { return make_cuDoubleComplex(1.0, 0.0); }
template <class T> __host__ __device__ inline T t_from(double re, double im);
template <> __host__ __device__ inline double t_from<double>(double re, double) { return re; }
template <> __host__ __device__ inline zc t_from<zc>(double re, double im) { return make_cuDoubleComplex(re, im); }
// fused multiply-add  acc += a*b
__host__ __device__ inline void t_fma(double& acc, double a, double b) { acc += a * b; }
__host__ __device__ inline void t_fma(zc& acc, zc a, zc b) {
  acc.x += a.x * b.x - a.y * b.y;
  acc.y += a.x * b.y + a.y * b.x;
}

// ---------------------------------------------------------------------------------------------
// strided-batched GEMM on the FP64 tensor pipe (gemm.cu)
//   C[b](i,j) = alpha * sum_k opA(A[b])(i,k) * opB(B[b])(k,j) + beta * C[b](i,j)
// Every operand is addressed with explicit element strides, so transposes / index permutations of
// TT cores and environments never need a separate permute pass.
// ---------------------------------------------------------------------------------------------
struct GemmArgs {
  int M = 0, N = 0, K = 0;
  const void* A = nullptr; int64_t sAm = 1, sAk = 0; bool conjA = false;
  const void* B = nullptr; int64_t sBk = 1, sBn = 0; bool conjB = false;
  void* C = nullptr;       int64_t sCm = 1, sCn = 0;
  double alpha = 1.0, beta = 0.0;
  int batch1 = 1, batch2 = 1;                       // two batch dimensions, b = b1 + batch1*b2
  int64_t bA1 = 0, bA2 = 0, bB1 = 0, bB2 = 0, bC1 = 0, bC2 = 0;
  // fused all-gather epilogue (shard.cu): the finished C tile is also stored to `npeer` mapped peer buffers (same strides)
  int npeer = 0;
  void* Cpeer[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};
template <class T> void gemm(const GemmArgs& g);
double gemm_flops(const GemmArgs& g, bool cplx);

// ---------------------------------------------------------------------------------------------
// bandwidth-bound helpers (elementwise.cu)
// ---------------------------------------------------------------------------------------------
// dst[i0*d0 + i1*d1 + i2*d2 + i3*d3] = alpha * op(src[i0*s0 + i1*s1 + i2*s2 + i3*s3]),  i0 fastest
struct Copy4 {
  int64_t n0 = 1, n1 = 1, n2 = 1, n3 = 1;
  int64_t s0 = 1, s1 = 0, s2 = 0, s3 = 0;
  int64_t d0 = 1, d1 = 0, d2 = 0, d3 = 0;
  double alpha = 1.0;
  bool conj = false;
  int tri = 0;  // 0: all;  1: keep i0 <= i1 (upper), zero elsewhere;  2: keep i0 >= i1 (lower), zero elsewhere
};
template <class T> void copy4(const T* src, T* dst, const Copy4& c);
template <class T> void fill(T* dst, int64_t n, T v);
template <class T> void set_identity(T* dst, int64_t m, int64_t n, int64_t ld);  // dst (m x n) = [I;0]
// real -> complex / complex -> real-part conversions
void real_to_cplx(const double* src, zc* dst, int64_t n);
void cplx_to_real(const zc* src, double* dst, int64_t n);
// A(i,j) *= f(vec[j]) (axis=1) or f(vec[i]) (axis=0);  mode 0: v, 1: sqrt(v), 2: 1/sqrt(v) (0 if v<=tiny), 3: 1/v (0 if v<=tiny)
template <class T> void diag_scale(T* A, int64_t m, int64_t n, int64_t rs, int64_t cs, const double* vec, int mode, int axis,
                                   int batch = 1, int64_t bA = 0, int64_t bvec = 0);
// y = a*x + y ; y = a*y ; scalars are T
template <class T> void axpy(int64_t n, T a, const T* x, T* y);
template <class T> void scal(int64_t n, T a, T* x);
// out[j] = sum_i conj(X[i + j*ldx]) * y[i], j < nv  (deterministic two-pass reduction); result on host
template <class T> void multi_dot(int64_t n, int nv, const T* X, int64_t ldx, const T* y, T* host_out);
// y -= sum_j h[j] * X[:,j]
template <class T> void multi_axpy(int64_t n, int nv, const T* X, int64_t ldx, const T* h_host, T* y, double sign);
template <class T> double nrm2(int64_t n, const T* x);
template <class T> T dotc(int64_t n, const T* x, const T* y);

// ---------------------------------------------------------------------------------------------
// TTO x TTV apply (apply.cu): y[i,(a,nu),(b,mu)] = sum_j A[i,j,a,b] x[j,nu,mu]   (+ batch of x)
// ---------------------------------------------------------------------------------------------
template <class T>
void apply_core(const T* A, const T* x, T* y, int n_out, int n_in, int Rl, int Rr, int rl, int rr, int batch,
                int64_t bx, int64_t by);

// ---------------------------------------------------------------------------------------------
// Householder QR (qr.cu), column-major, in place, batched
// ---------------------------------------------------------------------------------------------
// A (m x n, lda) -> R in the upper triangle, Householder vectors below (unit diagonal implicit), tau[k], k=min(m,n)
template <class T> void qr_factor(T* A, int m, int n, int64_t lda, T* tau, int batch = 1, int64_t bA = 0, int64_t btau = 0);
// C (m x nc, ldc) <- Q * C  (trans=false, reflectors applied last-to-first)  or  Q^H * C (trans=true)
// where Q = H_0 ... H_{k-1} is held in (A, tau) as produced by qr_factor;  col0: only columns >= col0 of C
template <class T> void qr_apply(const T* A, int m, int k, int64_t lda, const T* tau, T* C, int nc, int64_t ldc, bool trans,
                                 int batch = 1, int64_t bA = 0, int64_t btau = 0, int64_t bC = 0);
// CholeskyQR2 on the DMMA pipe for tall-skinny, well-conditioned matrices (cholqr.cu).  R: k x k upper (ld k, batch stride
// k*k); Q optional.  Returns false when the shape is not served or a matrix is rejected as ill conditioned: the caller
// then uses the Householder path above.
template <class T> bool cholqr2_fits(int m, int k);
template <class T> bool cholqr2(const T* A, int m, int k, int64_t lda, int64_t bA, T* R, T* Q, int64_t ldq, int64_t bQ, int batch);
// thin Q (m x k) explicitly
template <class T> void qr_form_q(const T* A, int m, int k, int64_t lda, const T* tau, T* Q, int64_t ldq,
                                  int batch = 1, int64_t bA = 0, int64_t btau = 0, int64_t bQ = 0);

// ---------------------------------------------------------------------------------------------
// one-sided Jacobi SVD (jacobi.cu)
// ---------------------------------------------------------------------------------------------
// Orthogonalises the n columns (length m) of X in place: X <- X*V with X^H X diagonal.  Column norms
// (unsorted singular values) are written to norms[n] (device).  Returns the number of sweeps used.
template <class T> int jacobi_orth(T* X, int m, int n, int64_t ldx, double* norms, int batch = 1, int64_t bX = 0,
                                   int64_t bnorms = 0);
// single-matrix path on an 8-CTA cluster (jacobi_cluster.cu); false if the shape is not served
template <class T> bool jacobi_cluster(T* X, int m, int n, int64_t ldx, int batch, int64_t bX, double tol, int* d_sweeps);
// Gram-block Jacobi on the DMMA pipe for one large matrix (jacobi_gram.cu); returns sweeps, or -1 if the shape is not served
template <class T> int jacobi_gram(T* X, int m, int n, int64_t ldx, double tol, int max_sweeps);
// dst (m x r) column j = X[:, perm[j]] * scale[j]   (perm/scale device arrays; per batch strides)
template <class T> void gather_cols(const T* X, int m, int64_t ldx, const int* perm, const double* scale, int r, T* dst,
                                    int64_t rs, int64_t cs, int batch = 1, int64_t bX = 0, int64_t bperm = 0,
                                    int64_t bdst = 0);

// Top eigenpairs of small Hermitian PSD matrices (heig.cu): the SVD engine of the Gram path of tt_compress!.
template <class T> int heig_max_n();
template <class T>
bool heig_top(const T* G, int n, int64_t ldg, int64_t bG, int nsplit, int64_t sG, int nev, int batch, double* lam, T* U, int* flags);
template <class T>
void heig_finalize(const T* U, int n, int nev, int batch, const double* lam, const double* w_in, T* out1, int64_t ld1, int64_t b1,
                   T* out2, int64_t ld2, int64_t b2, double* sig_out, int64_t bsig, double* sig0, int* flags);

// left singular vectors + singular values of a strided p x q matrix (svd.cu)
struct SvdLeft {
  int p = 0, q = 0, k = 0;       // k = min(p,q) singular values
  DevBuf X;                       // p x k (col-major, ld=p), columns orthogonal, unsorted: X = U*diag(sigma)
  DevBuf norms;                   // k doubles per batch (device), unsorted
  std::vector<double> sigma;      // host copy, sorted descending, batch-major (batch x k)
  std::vector<int> perm;          // host: sorted position -> column of X, batch-major
  int sweeps = 0;
};
// Theta(i,j) at Theta + i*rs + j*cs (+ b*bT); conjugated if conj.
template <class T> void svd_left(const T* Theta, int p, int q, int64_t rs, int64_t cs, bool conj, SvdLeft& out,
                                 int batch = 1, int64_t bT = 0);

}  // namespace ttn
