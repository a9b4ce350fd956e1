// extern "C" boundary of libttn_b200.so (declared in include/ttn_b200.h).  Converts the library's internal
// exceptions into status codes, and takes the train and operator handles apart and builds new ones.
#pragma GCC visibility push(default)
#include "../../include/ttn_b200.h"
#pragma GCC visibility pop
#include "tt.h"
#include "solvers.h"
#include <memory>

using namespace ttn;

static thread_local std::string g_err;

#define API_BEGIN try {
#define API_END                                         \
  }                                                     \
  catch (const ttn::Error& e) {                         \
    g_err = e.what();                                   \
    return e.code;                                      \
  }                                                     \
  catch (const std::exception& e) {                     \
    g_err = e.what();                                   \
    return TTN_EINTERNAL;                               \
  }                                                     \
  return TTN_OK;

static void need_init() { ttn_assert(ctx().inited, TTN_ECUDA, "ttn_init has not been called (no CUDA device bound)"); }

extern "C" {

int ttn_init(int device) {
  API_BEGIN
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    throw Error(TTN_ECUDA, std::string("no CUDA device available: ") + cudaGetErrorString(e) +
                               " (libttn_b200 has no CPU fallback)");
  ttn_assert(device >= 0 && device < count, TTN_EARG, "ttn_init: bad device index");
  TTN_CUDA(cudaSetDevice(device));
  Context& c = ctx();
  if (!c.inited || c.device != device) {
    if (c.inited && c.stream) { drain_deferred_releases(true); devbuf_cache_trim(); cudaStreamSynchronize(c.stream); cudaStreamDestroy(c.stream); }
    if (c.copy_stream) { cudaStreamSynchronize(c.copy_stream); cudaStreamDestroy(c.copy_stream); c.copy_stream = nullptr; }
    if (c.host_stage) { cudaFreeHost(c.host_stage); c.host_stage = nullptr; c.host_stage_bytes = 0; }
    c.device = device;
    TTN_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    cudaDeviceProp prop;
    TTN_CUDA(cudaGetDeviceProperties(&prop, device));
    c.sm_count = prop.multiProcessorCount;
    cudaMemPool_t pool;
    TTN_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thr = UINT64_MAX;
    TTN_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    c.inited = true;
  }
  API_END
}

int ttn_shutdown(void) {
  API_BEGIN
  Context& c = ctx();
  if (c.inited) {
    drain_deferred_releases(true);
    devbuf_cache_trim();
    cudaStreamSynchronize(c.stream);
    cudaStreamDestroy(c.stream);
    c.stream = nullptr;
    if (c.copy_stream) { cudaStreamSynchronize(c.copy_stream); cudaStreamDestroy(c.copy_stream); c.copy_stream = nullptr; }
    if (c.host_stage) { cudaFreeHost(c.host_stage); c.host_stage = nullptr; c.host_stage_bytes = 0; }
    c.inited = false;
  }
  API_END
}

// run-time switches that select between two live paths on the same input, so that tests can compare them; flop counters
int ttn_set_option(const char* key, double value) {
  API_BEGIN
  need_init();
  ttn_assert(key != nullptr, TTN_EARG, "null argument");
  const std::string k(key);
  Context& c = ctx();
  if (k == "gram_compress") c.gram_compress = value != 0.0;
  else if (k == "gemm_bulk") c.gemm_bulk = value != 0.0;
  else if (k == "gemm_thin") c.gemm_thin = value != 0.0;
  else if (k == "gram_jacobi_min") c.gram_jacobi_min = (int)value;
  else if (k == "reset_flops") { c.flops_gemm = 0.0; c.flops_heig = 0.0; }
  else throw Error(TTN_EARG, "ttn_set_option: unknown key " + k);
  API_END
}
int ttn_get_option(const char* key, double* value) {
  API_BEGIN
  need_init();
  ttn_assert(key != nullptr && value != nullptr, TTN_EARG, "null argument");
  const std::string k(key);
  const Context& c = ctx();
  if (k == "gram_compress") *value = c.gram_compress;
  else if (k == "gemm_bulk") *value = c.gemm_bulk;
  else if (k == "gemm_thin") *value = c.gemm_thin;
  else if (k == "gram_jacobi_min") *value = c.gram_jacobi_min;
  else if (k == "gemm_flops") *value = c.flops_gemm;
  else if (k == "heig_flops") *value = c.flops_heig;
  else if (k == "gram_calls") *value = (double)c.gram_calls;
  else if (k == "gram_fallbacks") *value = (double)c.gram_fallbacks;
  else if (k == "gram_last_flags") *value = (double)c.gram_last_flags;
  else throw Error(TTN_EARG, "ttn_get_option: unknown key " + k);
  API_END
}

const char* ttn_last_error(void) { return g_err.c_str(); }
int ttn_version(void) { return 100; }
int ttn_synchronize(void) {
  API_BEGIN
  need_init();
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  API_END
}
long long ttn_launch_count(void) { return ctx().launches; }
int ttn_reset_launch_count(void) { ctx().launches = 0; return TTN_OK; }
void* ttn_stream(void) { return (void*)ctx().stream; }
int ttn_last_jacobi_sweeps(void) { return ctx().last_jacobi_sweeps; }
int ttn_profile(int enable) {
  API_BEGIN
  Context& c = ctx();
  for (auto& r : c.prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  c.prof.clear();
  c.prof_on = enable != 0;
  API_END
}
int ttn_profile_read(double* ms, long long* counts) {
  API_BEGIN
  need_init();
  ttn_assert(ms && counts, TTN_EARG, "null argument");
  Context& c = ctx();
  TTN_CUDA(cudaStreamSynchronize(c.stream));
  for (int i = 0; i < KF_COUNT; ++i) { ms[i] = 0.0; counts[i] = 0; }
  for (auto& r : c.prof) {
    float t = 0.f;
    TTN_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    ms[r.fam] += t;
    counts[r.fam] += 1;
  }
  API_END
}

// ---------------------------------------------------------------------------------------------------------
}  // extern "C"
static cudaStream_t copy_stream() {
  Context& c = ctx();
  if (!c.copy_stream) TTN_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
  return c.copy_stream;
}
// the copy stream waits until the compute stream has reached this point (no host synchronisation)
static void copy_stream_follows_compute() {
  cudaEvent_t ev;
  TTN_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  TTN_CUDA(cudaEventRecord(ev, ctx().stream));
  TTN_CUDA(cudaStreamWaitEvent(copy_stream(), ev, 0));
  cudaEventDestroy(ev);
}
// `ev` (re)recorded at the current end of the copy stream
static void record_on_copy_stream(cudaEvent_t& ev) {
  if (ev) cudaEventDestroy(ev);
  ev = nullptr;
  TTN_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  TTN_CUDA(cudaEventRecord(ev, copy_stream()));
}
namespace {
struct DeferredRelease {
  cudaEvent_t ev;
  std::vector<ttn::DevBuf> bufs;
};
struct DeferredList {
  std::vector<DeferredRelease> v;
  ~DeferredList() {                                   // thread exit: the context may already be gone, just wait and let go
    for (auto& d : v) { cudaEventSynchronize(d.ev); cudaEventDestroy(d.ev); }
  }
};
DeferredList& deferred() {
  static thread_local DeferredList l;
  return l;
}
}  // namespace
void ttn::drain_deferred_releases(bool block) {
  auto& v = deferred().v;
  size_t keep = 0;
  for (size_t i = 0; i < v.size(); ++i) {
    bool done = block ? (cudaEventSynchronize(v[i].ev), true) : cudaEventQuery(v[i].ev) == cudaSuccess;
    if (done) {
      cudaEventDestroy(v[i].ev);
      v[i].bufs.clear();                              // DevBuf destructors: back to the block cache of this thread
    } else {
      if (keep != i) v[keep] = std::move(v[i]);
      ++keep;
    }
  }
  if (!block) cudaGetLastError();                     // cudaErrorNotReady of the queries is not an error
  v.resize(keep);
}
ttn_ttv_s::~ttn_ttv_s() {
  if (ready) { cudaStreamWaitEvent(ttn::ctx().stream, ready, 0); cudaEventDestroy(ready); }
  if (busy) {
    if (cudaEventQuery(busy) == cudaSuccess) {
      cudaEventDestroy(busy);
    } else {
      cudaGetLastError();
      DeferredRelease d;
      d.ev = busy;
      d.bufs = visit([](auto& t) { return std::move(t.cores); });
      deferred().v.push_back(std::move(d));
    }
  }
  ttn::drain_deferred_releases(false);
}

// The two ways an entry point takes a train whose cores it touches.  Neither makes the host wait.
//   read_ttv:  the compute stream waits for a pending ttn_ttv_upload_async of x, so such a handle may go anywhere at once.
//   write_ttv: for the entry points that replace the cores in place; the compute stream also waits for a pending
//              ttn_ttv_download_async of x, so that the old cores go back to the block cache only after the copy engine
//              has read them.
static ttn_ttv_s& read_ttv(ttn_ttv x) {
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  if (x->ready) {
    TTN_CUDA(cudaStreamWaitEvent(ctx().stream, x->ready, 0));
    cudaEventDestroy(x->ready);
    x->ready = nullptr;
  }
  return *x;
}
static ttn_ttv_s& write_ttv(ttn_ttv x) {
  ttn_ttv_s& h = read_ttv(x);
  if (h.busy) TTN_CUDA(cudaStreamWaitEvent(ctx().stream, h.busy, 0));
  return h;
}
// an empty result train of element type `dtype`; the entry point hands it out with `*out = h.release()`
static std::unique_ptr<ttn_ttv_s> new_ttv(int dtype) {
  with_dtype(dtype, [](auto) {});
  auto h = std::make_unique<ttn_ttv_s>();
  h->dtype = dtype;
  return h;
}
// a train shaped from the caller's arrays, its cores allocated but not yet filled
static std::unique_ptr<ttn_ttv_s> alloc_ttv(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot,
                                            int batch) {
  ttn_assert(d >= 1 && batch >= 1 && dims && rks, TTN_EARG, "upload: bad arguments");
  auto h = new_ttv(dtype);
  h->visit([&](auto& t) {
    t.d = d; t.batch = batch;
    t.dims.assign(dims, dims + d);
    t.rks.assign(rks, rks + d + 1);
    if (ot) t.ot.assign(ot, ot + d); else t.ot.assign(d, 0);
    t.cores.resize(d);
    for (int k = 0; k < d; ++k) {
      ttn_assert(dims[k] >= 1 && rks[k] >= 1 && rks[k + 1] >= 1, TTN_EDIM, "upload: dims and ranks must be positive");
      t.alloc_core(k);
    }
  });
  return h;
}
// every core of a train or operator between the device and the caller's host arrays, queued on `s`
template <class H>
static void copy_cores(H& x, void* const* host, cudaMemcpyKind kind, cudaStream_t s) {
  ttn_assert(host != nullptr, TTN_EARG, "null argument");
  x.visit([&](auto& t) {
    for (int k = 0; k < t.d; ++k) {
      void* dev = t.cores[k].p;
      const bool up = kind == cudaMemcpyHostToDevice;
      TTN_CUDA(cudaMemcpyAsync(up ? dev : host[k], up ? host[k] : dev, t.cores[k].bytes, kind, s));
    }
  });
}
// rks / dims / ot of a handle into the caller's array
template <class H, class F>
static void copy_shape(H* x, int64_t* out, F field) {
  ttn_assert(x && out, TTN_EARG, "null argument");
  x->visit([&](auto& t) {
    const std::vector<int64_t>& v = field(t);
    std::copy(v.begin(), v.end(), out);
  });
}
extern "C" {

int ttn_ttv_upload(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot, const void* const* cores,
                   int batch, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "upload: bad arguments");
  auto h = alloc_ttv(dtype, d, dims, rks, ot, batch);
  copy_cores(*h, const_cast<void* const*>(cores), cudaMemcpyHostToDevice, ctx().stream);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  *out = h.release();
  API_END
}
int ttn_ttv_upload_async(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot, const void* const* cores,
                         int batch, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "upload: bad arguments");
  drain_deferred_releases(false);
  auto h = alloc_ttv(dtype, d, dims, rks, ot, batch);
  copy_stream_follows_compute();   // the stream-ordered allocations become usable on the copy stream
  copy_cores(*h, const_cast<void* const*>(cores), cudaMemcpyHostToDevice, copy_stream());
  record_on_copy_stream(h->ready);
  *out = h.release();
  API_END
}
int ttn_ttv_download_async(ttn_ttv x, void* const* cores) {
  API_BEGIN
  need_init();
  ttn_ttv_s& h = read_ttv(x);
  copy_stream_follows_compute();   // everything queued on the compute stream so far has produced x
  copy_cores(h, cores, cudaMemcpyDeviceToHost, copy_stream());
  record_on_copy_stream(h.busy);
  API_END
}
int ttn_copy_synchronize(void) {
  API_BEGIN
  need_init();
  if (ctx().copy_stream) TTN_CUDA(cudaStreamSynchronize(ctx().copy_stream));
  drain_deferred_releases(true);
  API_END
}

int ttn_ttv_info(ttn_ttv x, int* dtype, int* d, int* batch) {
  API_BEGIN
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  if (dtype) *dtype = x->dtype;
  x->visit([&](auto& t) {
    if (d) *d = t.d;
    if (batch) *batch = t.batch;
  });
  API_END
}
int ttn_ttv_ranks(ttn_ttv x, int64_t* rks) {
  API_BEGIN
  copy_shape(x, rks, [](auto& t) -> auto& { return t.rks; });
  API_END
}
int ttn_ttv_dims(ttn_ttv x, int64_t* dims) {
  API_BEGIN
  copy_shape(x, dims, [](auto& t) -> auto& { return t.dims; });
  API_END
}
int ttn_ttv_ot(ttn_ttv x, int64_t* ot) {
  API_BEGIN
  copy_shape(x, ot, [](auto& t) -> auto& { return t.ot; });
  API_END
}
int ttn_ttv_download(ttn_ttv x, void* const* cores) {
  API_BEGIN
  need_init();
  copy_cores(read_ttv(x), cores, cudaMemcpyDeviceToHost, ctx().stream);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  API_END
}
int ttn_ttv_copy(ttn_ttv x, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  auto h = new_ttv(xs.dtype);
  with_dtype(xs.dtype, [&](auto t) { using T = decltype(t); tt_copy(xs.as<T>(), h->as<T>()); });
  *out = h.release();
  API_END
}
int ttn_ttv_complex(ttn_ttv x, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  auto h = new_ttv(TTN_C128);
  if (xs.dtype == TTN_C128) tt_copy(xs.as<zc>(), h->as<zc>());
  else tt_to_complex(xs.as<double>(), h->as<zc>());
  *out = h.release();
  API_END
}
int ttn_ttv_free(ttn_ttv x) {
  API_BEGIN
  delete x;
  API_END
}

int ttn_tto_upload(int dtype, int d, const int64_t* dims, const int64_t* rks, const void* const* cores, ttn_tto* out) {
  API_BEGIN
  need_init();
  ttn_assert(d >= 1 && dims && rks && out, TTN_EARG, "upload: bad arguments");
  auto h = std::make_unique<ttn_tto_s>();
  h->dtype = dtype;
  with_dtype(dtype, [&](auto tag) {
    using T = decltype(tag);
    TTO<T>& t = h->as<T>();
    t.d = d;
    t.dims.assign(dims, dims + d);
    t.rks.assign(rks, rks + d + 1);
    t.cores.resize(d);
    for (int k = 0; k < d; ++k) {
      ttn_assert(dims[k] >= 1 && rks[k] >= 1 && rks[k + 1] >= 1, TTN_EDIM, "upload: dims and ranks must be positive");
      t.cores[k].alloc(sizeof(T) * (size_t)(dims[k] * dims[k] * rks[k] * rks[k + 1]));
    }
  });
  copy_cores(*h, const_cast<void* const*>(cores), cudaMemcpyHostToDevice, ctx().stream);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  *out = h.release();
  API_END
}
int ttn_tto_complex(ttn_tto A, ttn_tto* out) {
  API_BEGIN
  need_init();
  ttn_assert(A && out, TTN_EARG, "null handle");
  auto h = std::make_unique<ttn_tto_s>();
  h->dtype = TTN_C128;
  if (A->dtype == TTN_C128) tto_copy(A->as<zc>(), h->as<zc>()); else tto_to_complex(A->as<double>(), h->as<zc>());
  *out = h.release();
  API_END
}
int ttn_tto_info(ttn_tto A, int* dtype, int* d) {
  API_BEGIN
  ttn_assert(A != nullptr, TTN_EARG, "null handle");
  if (dtype) *dtype = A->dtype;
  if (d) *d = A->visit([](auto& t) { return t.d; });
  API_END
}
int ttn_tto_ranks(ttn_tto A, int64_t* rks) {
  API_BEGIN
  copy_shape(A, rks, [](auto& t) -> auto& { return t.rks; });
  API_END
}
int ttn_tto_dims(ttn_tto A, int64_t* dims) {
  API_BEGIN
  copy_shape(A, dims, [](auto& t) -> auto& { return t.dims; });
  API_END
}
int ttn_tto_download(ttn_tto A, void* const* cores) {
  API_BEGIN
  need_init();
  ttn_assert(A != nullptr, TTN_EARG, "null handle");
  copy_cores(*A, cores, cudaMemcpyDeviceToHost, ctx().stream);
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  API_END
}
int ttn_tto_free(ttn_tto A) {
  API_BEGIN
  delete A;
  API_END
}

// ---------------------------------------------------------------------------------------------------------
static void same_dtype(int a, int b) { ttn_assert(a == b, TTN_EDIM, "element types differ (promote with ttn_*_complex first)"); }

int ttn_apply(ttn_tto A, ttn_ttv x, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(A && y, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  same_dtype(A->dtype, xs.dtype);
  auto h = new_ttv(xs.dtype);
  with_dtype(xs.dtype, [&](auto t) { using T = decltype(t); tt_apply(A->as<T>(), xs.as<T>(), h->as<T>()); });
  *y = h.release();
  API_END
}
int ttn_dot(ttn_ttv a, ttn_ttv b, double* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& as = read_ttv(a);
  ttn_ttv_s& bs = read_ttv(b);
  same_dtype(as.dtype, bs.dtype);
  with_dtype(as.dtype, [&](auto t) {
    using T = decltype(t);
    std::vector<T> v;
    tt_dot(as.as<T>(), bs.as<T>(), v);
    for (size_t i = 0; i < v.size(); ++i) { out[2 * i] = t_real(v[i]); out[2 * i + 1] = t_imag(v[i]); }
  });
  API_END
}
int ttn_norm(ttn_ttv a, double* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& as = read_ttv(a);
  with_dtype(as.dtype, [&](auto t) {
    using T = decltype(t);
    std::vector<T> v;
    tt_dot(as.as<T>(), as.as<T>(), v);
    for (size_t i = 0; i < v.size(); ++i) out[i] = std::sqrt(t_real(v[i]) > 0 ? t_real(v[i]) : 0.0);
  });
  API_END
}
int ttn_add(ttn_ttv x, ttn_ttv y, ttn_ttv* z) {
  API_BEGIN
  need_init();
  ttn_assert(z != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  ttn_ttv_s& ys = read_ttv(y);
  same_dtype(xs.dtype, ys.dtype);
  auto h = new_ttv(xs.dtype);
  with_dtype(xs.dtype, [&](auto t) { using T = decltype(t); tt_add(xs.as<T>(), ys.as<T>(), h->as<T>()); });
  *z = h.release();
  API_END
}
int ttn_scale(ttn_ttv x, double re, double im, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(y != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  ttn_assert(xs.dtype == TTN_C128 || im == 0.0, TTN_EARG, "complex scalar on a real TT (promote first)");
  auto h = new_ttv(xs.dtype);
  with_dtype(xs.dtype, [&](auto t) { using T = decltype(t); tt_scale(xs.as<T>(), t_from<T>(re, im), h->as<T>()); });
  *y = h.release();
  API_END
}
int ttn_orthogonalize(ttn_ttv x, int center, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(y != nullptr, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  auto h = new_ttv(xs.dtype);
  with_dtype(xs.dtype, [&](auto t) { using T = decltype(t); tt_orthogonalize(xs.as<T>(), center, h->as<T>()); });
  *y = h.release();
  API_END
}
int ttn_compress(ttn_ttv x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride) {
  API_BEGIN
  need_init();
  write_ttv(x).visit([&](auto& t) { tt_compress(t, max_bond, truncerr, sweeps, sigma_out, sigma_stride); });
  API_END
}
int ttn_apply_compress(ttn_tto A, ttn_ttv x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride,
                       ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(A && y, TTN_EARG, "null handle");
  ttn_ttv_s& xs = read_ttv(x);
  same_dtype(A->dtype, xs.dtype);
  auto h = new_ttv(xs.dtype);
  with_dtype(xs.dtype, [&](auto t) {
    using T = decltype(t);
    tt_apply_compress(A->as<T>(), xs.as<T>(), h->as<T>(), max_bond, truncerr, sweeps, sigma_out, sigma_stride);
  });
  *y = h.release();
  API_END
}
int ttn_bond_truncate(ttn_ttv x, int k, int64_t max_bond, double truncerr, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_ttv_s& xs = write_ttv(x);
  xs.visit([&](auto& t) { tt_bond_truncate(t, k, max_bond, truncerr, nullptr, 0); });
  if (y) {
    auto h = new_ttv(xs.dtype);
    with_dtype(xs.dtype, [&](auto t) { using T = decltype(t); tt_orthogonalize(xs.as<T>(), k, h->as<T>()); });
    *y = h.release();
  }
  API_END
}

int ttn_swap_sites(ttn_ttv x, int k, int mode, int64_t max_bond, double tol) {
  API_BEGIN
  need_init();
  ttn_assert(mode == 0 || mode == 1, TTN_EARG, "mode must be 0 (relative threshold) or 1 (tail norm)");
  write_ttv(x).visit([&](auto& t) { tt_swap_sites(t, k, mode, max_bond, tol); });
  API_END
}
int ttn_merge_sites_diag(ttn_ttv x, int k) {
  API_BEGIN
  need_init();
  write_ttv(x).visit([&](auto& t) { tt_merge_diag(t, k); });
  API_END
}
int ttn_split_site(ttn_ttv x, int k, int64_t coarse, int mode, int64_t max_bond, double tol) {
  API_BEGIN
  need_init();
  ttn_assert(mode == 0 || mode == 1, TTN_EARG, "mode must be 0 (relative threshold) or 1 (tail norm)");
  write_ttv(x).visit([&](auto& t) { tt_split_site(t, k, coarse, mode, max_bond, tol); });
  API_END
}

// ---------------------------------------------------------------------------------------------------------
// solvers
// ---------------------------------------------------------------------------------------------------------
int ttn_solver_params_default(ttn_solver_params* p) {
  if (!p) return TTN_EARG;
  p->N = 2; p->tol = 1e-12;
  p->sweep_schedule = nullptr; p->n_sweep_schedule = 0;
  p->rmax_schedule = nullptr; p->n_rmax_schedule = 0;
  p->rmax = 0; p->sweep_count = 2; p->it_solver = 0;
  p->linsolv_maxiter = 200; p->linsolv_tol = 1e-6; p->itslv_thresh = 256; p->krylovdim = 30; p->symmetrize = 0;
  return TTN_OK;
}
int ttn_tdvp_params_default(ttn_tdvp_params* p) {
  if (!p) return TTN_EARG;
  p->two_site = 0; p->steps = nullptr; p->n_steps = 0; p->normalize = 1; p->sweeps = 1; p->imaginary_time = 0;
  p->max_bond = INT64_MAX; p->truncerr = 0.0; p->krylovdim = 30; p->krylov_tol = 1e-12; p->krylov_maxiter = 100;
  return TTN_OK;
}

}  // extern "C"
// The prologue of every solver wrapper: A, x0 and the result share x0's element type; run(T tag, A, x0, x) runs the sweep
// into the new train, which is handed out once it has returned.
template <class F>
static void solve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, F&& run) {
  need_init();
  ttn_assert(A && p && x, TTN_EARG, "null argument");
  ttn_ttv_s& x0s = read_ttv(x0);
  same_dtype(A->dtype, x0s.dtype);
  auto h = new_ttv(x0s.dtype);
  with_dtype(x0s.dtype, [&](auto t) { using T = decltype(t); run(t, A->as<T>(), x0s.as<T>(), h->as<T>()); });
  *x = h.release();
}
// the right-hand side of a linear solve, of A's element type
static ttn_ttv_s& rhs(ttn_tto A, ttn_ttv b) {
  ttn_ttv_s& bs = read_ttv(b);
  ttn_assert(A != nullptr, TTN_EARG, "null argument");
  same_dtype(A->dtype, bs.dtype);
  return bs;
}
// the eigenvalue (and rank) history of a sweep, as far as the caller's arrays reach
static void history_out(const std::vector<double>& Ev, const std::vector<int64_t>& rh, double* E, int64_t* r_hist, int cap_E,
                        int* n_E) {
  if (n_E) *n_E = (int)Ev.size();
  for (int i = 0; i < (int)Ev.size() && i < cap_E; ++i) {
    if (E) E[i] = Ev[i];
    if (r_hist) r_hist[i] = rh[i];
  }
}
extern "C" {

int ttn_als_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual) {
  API_BEGIN
  ttn_ttv_s& bs = rhs(A, b);
  solve(A, x0, p, x, [&](auto t, auto& At, auto& x0t, auto& xt) { als_linsolve(At, bs.as<decltype(t)>(), x0t, *p, xt, residual); });
  API_END
}
int ttn_als_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int cap_E, int* n_E) {
  API_BEGIN
  std::vector<double> Ev;
  solve(A, x0, p, x, [&](auto, auto& At, auto& x0t, auto& xt) { als_eigsolve(At, x0t, *p, xt, Ev); });
  history_out(Ev, {}, E, nullptr, cap_E, n_E);
  API_END
}
int ttn_als_gen_eigsolv(ttn_tto A, ttn_tto S, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int cap_E, int* n_E) {
  API_BEGIN
  ttn_assert(A && S, TTN_EARG, "null argument");
  same_dtype(A->dtype, S->dtype);
  std::vector<double> Ev;
  solve(A, x0, p, x, [&](auto t, auto& At, auto& x0t, auto& xt) { als_gen_eigsolve(At, S->as<decltype(t)>(), x0t, *p, xt, Ev); });
  history_out(Ev, {}, E, nullptr, cap_E, n_E);
  API_END
}
int ttn_mals_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual) {
  API_BEGIN
  ttn_ttv_s& bs = rhs(A, b);
  solve(A, x0, p, x, [&](auto t, auto& At, auto& x0t, auto& xt) { mals_linsolve(At, bs.as<decltype(t)>(), x0t, *p, xt, residual); });
  API_END
}
int ttn_mals_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int64_t* r_hist, int cap_E,
                      int* n_E) {
  API_BEGIN
  std::vector<double> Ev;
  std::vector<int64_t> rh;
  solve(A, x0, p, x, [&](auto, auto& At, auto& x0t, auto& xt) { mals_eigsolve(At, x0t, *p, xt, Ev, rh); });
  history_out(Ev, rh, E, r_hist, cap_E, n_E);
  API_END
}
int ttn_dmrg_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual) {
  API_BEGIN
  ttn_ttv_s& bs = rhs(A, b);
  solve(A, x0, p, x, [&](auto t, auto& At, auto& x0t, auto& xt) { dmrg_linsolve(At, bs.as<decltype(t)>(), x0t, *p, xt, residual); });
  API_END
}
int ttn_dmrg_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int64_t* r_hist, int cap_E,
                      int* n_E) {
  API_BEGIN
  std::vector<double> Ev;
  std::vector<int64_t> rh;
  solve(A, x0, p, x, [&](auto, auto& At, auto& x0t, auto& xt) { dmrg_eigsolve(At, x0t, *p, xt, Ev, rh); });
  history_out(Ev, rh, E, r_hist, cap_E, n_E);
  API_END
}
// ---- multi-GPU DMRG: replicated sweep, sharded Lanczos matvec (shard.cu) -----------------------------------------
int ttn_shard_ctx_create(int dtype, int64_t max_elems, int rank, int nranks, ttn_shard_ctx* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "shard ctx: bad arguments");
  *out = shard_ctx_create(dtype, max_elems, rank, nranks);
  API_END
}
int ttn_shard_ctx_handles(ttn_shard_ctx c, void* handles384) {
  API_BEGIN
  need_init();
  shard_ctx_handles(c, handles384);
  API_END
}
int ttn_shard_ctx_bind(ttn_shard_ctx c, const void* all_handles) {
  API_BEGIN
  need_init();
  shard_ctx_bind(c, all_handles);
  API_END
}
int ttn_shard_ctx_free(ttn_shard_ctx c) {
  API_BEGIN
  delete c;
  API_END
}
int ttn_dmrg_eigsolve_sharded(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_shard_ctx sc, ttn_ttv* x, double* E,
                              int64_t* r_hist, int cap_E, int* n_E) {
  API_BEGIN
  ttn_assert(sc != nullptr, TTN_EARG, "null shard context");
  std::vector<double> Ev;
  std::vector<int64_t> rh;
  solve(A, x0, p, x, [&](auto t, auto& At, auto& x0t, auto& xt) {
    same_dtype(sc->dtype, A->dtype);
    dmrg_eigsolve(At, x0t, *p, xt, Ev, rh, &sc->as<decltype(t)>());
    ttn_assert(shard_ctx_error(sc) == 0, TTN_ECUDA,
               "sharded DMRG: a peer did not publish its slice within the epoch timeout (TTN_SHARD_TIMEOUT_S); the result is invalid");
  });
  history_out(Ev, rh, E, r_hist, cap_E, n_E);
  API_END
}
int ttn_tdvp(ttn_tto H, ttn_ttv u0, const ttn_tdvp_params* p, ttn_ttv* u) {
  API_BEGIN
  need_init();
  ttn_assert(H && p && u, TTN_EARG, "null argument");
  ttn_ttv_s& u0s = read_ttv(u0);
  same_dtype(H->dtype, u0s.dtype);
  // real-time evolution of a real state runs on its complex promotion (tdvp.jl:167-172)
  const bool promote = u0s.dtype != TTN_C128 && !p->imaginary_time;
  auto h = new_ttv(promote ? TTN_C128 : u0s.dtype);
  if (promote) {
    TT<zc> uc;
    TTO<zc> Hc;
    tt_to_complex(u0s.as<double>(), uc);
    tto_to_complex(H->as<double>(), Hc);
    tdvp_run(Hc, uc, *p, h->as<zc>());
  } else {
    with_dtype(u0s.dtype, [&](auto t) { using T = decltype(t); tdvp_run(H->as<T>(), u0s.as<T>(), *p, h->as<T>()); });
  }
  *u = h.release();
  API_END
}

// ---------------------------------------------------------------------------------------------------------
// kernel-level entry points
// ---------------------------------------------------------------------------------------------------------
int ttn_gemm(int dtype, int M, int N, int K, const void* A, int64_t sAm, int64_t sAk, int conjA, const void* B, int64_t sBk,
             int64_t sBn, int conjB, void* C, int64_t sCm, int64_t sCn, double alpha, double beta, int batch, int64_t bA,
             int64_t bB, int64_t bC) {
  API_BEGIN
  need_init();
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.sAm = sAm; g.sAk = sAk; g.conjA = conjA != 0;
  g.B = B; g.sBk = sBk; g.sBn = sBn; g.conjB = conjB != 0;
  g.C = C; g.sCm = sCm; g.sCn = sCn;
  g.alpha = alpha; g.beta = beta;
  // the batch is the outer dimension, which gemm() splits into launches of at most 65535 CTAs along grid.z
  g.batch1 = 1; g.batch2 = batch; g.bA2 = bA; g.bB2 = bB; g.bC2 = bC;
  with_dtype(dtype, [&](auto t) { gemm<decltype(t)>(g); });
  API_END
}

int ttn_matvec2_host(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid, const void* H,
                     const void* V, void* Y, int symmetrize) {
  API_BEGIN
  need_init();
  with_dtype(dtype, [&](auto t) { matvec2_host<decltype(t)>(w_l, w_r, chi_l, chi_r, nn, G, Amid, H, V, Y, symmetrize != 0); });
  API_END
}
int ttn_matvec2_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                       const void* H, ttn_matvec* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "null argument");
  *out = matvec2_create(dtype, w_l, w_r, chi_l, chi_r, nn, G, Amid, H);
  API_END
}
int ttn_matvec2_apply(ttn_matvec mv, const void* V_dev, void* Y_dev) {
  API_BEGIN
  need_init();
  matvec2_apply(mv, V_dev, Y_dev);
  API_END
}
int ttn_matvec2_free(ttn_matvec mv) {
  API_BEGIN
  delete mv;
  API_END
}
int ttn_shard_range(int chi, int rank, int nranks, int* c0, int* cp) {
  API_BEGIN
  ttn_assert(chi >= 1 && nranks >= 1 && rank >= 0 && rank < nranks && c0 && cp, TTN_EARG, "shard_range: bad arguments");
  shard_range(chi, rank, nranks, c0, cp);
  API_END
}
int ttn_shard_matvec_create(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid,
                            const void* H, int rank, int nranks, ttn_shard_matvec* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr, TTN_EARG, "null argument");
  *out = shard_create(dtype, w_l, w_r, chi_l, chi_r, nn, G, Amid, H, rank, nranks);
  API_END
}
int ttn_shard_matvec_handles(ttn_shard_matvec mv, void* handles192) {
  API_BEGIN
  need_init();
  shard_handles(mv, handles192);
  API_END
}
int ttn_shard_matvec_bind(ttn_shard_matvec mv, const void* all_handles) {
  API_BEGIN
  need_init();
  shard_bind_handles(mv, all_handles);
  API_END
}
int ttn_shard_matvec_apply(ttn_shard_matvec mv, const void* V_dev, void** Y_dev) {
  API_BEGIN
  need_init();
  ttn_assert(Y_dev != nullptr, TTN_EARG, "null argument");
  *Y_dev = shard_apply_any(mv, V_dev);
  API_END
}
int ttn_shard_eigsolve(ttn_shard_matvec mv, void* x_dev, int krylovdim, int maxiter, double tol, double* theta, int* matvecs) {
  API_BEGIN
  need_init();
  ttn_assert(theta != nullptr, TTN_EARG, "null argument");
  *theta = shard_eigsolve(mv, x_dev, krylovdim, maxiter, tol, matvecs);
  API_END
}
int ttn_shard_matvec_slice(ttn_shard_matvec mv, int* c0, int* cp) {
  API_BEGIN
  ttn_assert(mv && c0 && cp, TTN_EARG, "null argument");
  shard_slice(mv, c0, cp);
  API_END
}
int ttn_shard_matvec_error(ttn_shard_matvec mv, int* err) {
  API_BEGIN
  need_init();
  ttn_assert(mv && err, TTN_EARG, "null argument");
  *err = shard_error(mv);
  API_END
}
int ttn_shard_matvec_free(ttn_shard_matvec mv) {
  API_BEGIN
  delete mv;
  API_END
}
int ttn_env_left_host(int dtype, int n, int w_l, int w_r, int r_l, int r_r, const void* G, const void* x, const void* A,
                      void* Gout) {
  API_BEGIN
  need_init();
  with_dtype(dtype, [&](auto t) { env_host<decltype(t)>(true, n, w_l, w_r, r_l, r_r, G, x, A, Gout); });
  API_END
}
int ttn_env_right_host(int dtype, int n, int w_l, int w_r, int r_l, int r_r, const void* H, const void* x, const void* A,
                       void* Hout) {
  API_BEGIN
  need_init();
  with_dtype(dtype, [&](auto t) { env_host<decltype(t)>(false, n, w_l, w_r, r_l, r_r, H, x, A, Hout); });
  API_END
}

}  // extern "C"
template <class T>
static void svdtrunc_host(int m, int n, const void* A, int64_t max_bond, double truncerr, void* U, double* s, void* Vt,
                          int* r_out) {
  DevBuf dA(sizeof(T) * (size_t)m * n);
  TTN_CUDA(cudaMemcpyAsync(dA.p, A, dA.bytes, cudaMemcpyHostToDevice, ctx().stream));
  DevBuf dU, dSVt;
  std::vector<double> sig;
  const int r = split_left<T>(dA.as<T>(), m, n, 1, m, false,
                              [&](const double* sg, int k) { return rank_tailnorm(sg, k, max_bond, truncerr); }, dU, dSVt, &sig);
  // Vt = S^{-1} (S Vt)
  std::vector<double> sr(sig.begin(), sig.begin() + r);
  DevBuf ds(sizeof(double) * r);
  TTN_CUDA(cudaMemcpyAsync(ds.p, sr.data(), ds.bytes, cudaMemcpyHostToDevice, ctx().stream));
  diag_scale<T>(dSVt.as<T>(), r, n, 1, r, ds.as<double>(), 3, 0);
  TTN_CUDA(cudaMemcpyAsync(U, dU.p, sizeof(T) * (size_t)m * r, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(Vt, dSVt.p, sizeof(T) * (size_t)r * n, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  for (int j = 0; j < r; ++j) s[j] = sig[j];
  *r_out = r;
}
extern "C" {
int ttn_svdtrunc_host(int dtype, int m, int n, const void* A, int64_t max_bond, double truncerr, void* U, double* s, void* Vt,
                      int* r_out) {
  API_BEGIN
  need_init();
  ttn_assert(m >= 1 && n >= 1 && max_bond >= 1, TTN_EARG, "svdtrunc: bad shape");
  with_dtype(dtype, [&](auto t) { svdtrunc_host<decltype(t)>(m, n, A, max_bond, truncerr, U, s, Vt, r_out); });
  API_END
}

}  // extern "C"
// Test / benchmark hook of the small Hermitian eigensolver behind the Gram path of tt_compress! (csrc/heig.cu)
template <class T>
static void heig_host(int n, int nev, int batch, const void* G, double* lam, void* U, int* flags) {
  DevBuf dG(sizeof(T) * (size_t)n * n * batch), dl(sizeof(double) * (size_t)nev * batch), dU(sizeof(T) * (size_t)n * nev * batch),
      df(sizeof(int) * (size_t)batch);
  TTN_CUDA(cudaMemcpyAsync(dG.p, G, dG.bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaMemsetAsync(df.p, 0, df.bytes, ctx().stream));
  ttn_assert(heig_top<T>(dG.as<T>(), n, n, (int64_t)n * n, 1, 0, nev, batch, dl.as<double>(), dU.as<T>(), df.as<int>()), TTN_EARG,
             "heig: shape not served");
  TTN_CUDA(cudaMemcpyAsync(lam, dl.p, dl.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(U, dU.p, dU.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(flags, df.p, df.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}
extern "C" {
int ttn_heig_host(int dtype, int n, int nev, int batch, const void* G, double* lam, void* U, int* flags) {
  API_BEGIN
  need_init();
  ttn_assert(n >= 1 && nev >= 1 && nev <= n && batch >= 1, TTN_EARG, "heig: bad shape");
  with_dtype(dtype, [&](auto t) { heig_host<decltype(t)>(n, nev, batch, G, lam, U, flags); });
  API_END
}
}
template <class T>
static void qr_host(int m, int n, const void* A, void* Q, void* R) {
  const int k = std::min(m, n);
  DevBuf dA(sizeof(T) * (size_t)m * n), tau(sizeof(T) * (size_t)k), dQ(sizeof(T) * (size_t)m * k), dR(sizeof(T) * (size_t)k * n);
  TTN_CUDA(cudaMemcpyAsync(dA.p, A, dA.bytes, cudaMemcpyHostToDevice, ctx().stream));
  qr_factor<T>(dA.as<T>(), m, n, m, tau.as<T>());
  qr_form_q<T>(dA.as<T>(), m, k, m, tau.as<T>(), dQ.as<T>(), m);
  Copy4 t; t.n0 = k; t.n1 = n; t.s0 = 1; t.s1 = m; t.d0 = 1; t.d1 = k; t.tri = 1;
  copy4<T>(dA.as<T>(), dR.as<T>(), t);
  TTN_CUDA(cudaMemcpyAsync(Q, dQ.p, dQ.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaMemcpyAsync(R, dR.p, dR.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}
extern "C" {
int ttn_qr_host(int dtype, int m, int n, const void* A, void* Q, void* R) {
  API_BEGIN
  need_init();
  ttn_assert(m >= 1 && n >= 1, TTN_EARG, "qr: bad shape");
  with_dtype(dtype, [&](auto t) { qr_host<decltype(t)>(m, n, A, Q, R); });
  API_END
}

// The four truncation rules of the path evaluated on a host spectrum (pure host code, no device needed: CPU parity tests).
int ttn_rank_rule(int rule, const double* s, int len, double tol, int64_t max_bond, int* r) {
  API_BEGIN
  ttn_assert(s != nullptr && r != nullptr && len >= 1, TTN_EARG, "rank_rule: bad arguments");
  switch (rule) {
    case 0: *r = rank_tailnorm(s, len, max_bond, tol); break;                       // _svdtrunc
    case 1: *r = std::min(sv_trunc_count(s, len, tol), len); break;                  // sv_trunc (count)
    case 2: *r = cut_off_index(s, len, tol); break;                                  // cut_off_index
    case 3: {                                                                        // relative threshold (qtt_tools.jl:680-685)
      int k = len;
      if (tol > 0) { k = 0; for (int j = 0; j < len; ++j) k += s[j] > tol * s[0]; k = std::max(1, k); }
      *r = k;
      break;
    }
    default: ttn_assert(false, TTN_EARG, "rank_rule: unknown rule");
  }
  API_END
}

// r_and_d_to_rks(rks, dims; rmax) on the host (rank schedules of the eigen-solvers); `rks`, `out`: d + 1 values
int ttn_r_and_d_to_rks(const int64_t* rks, const int64_t* dims, int d, int64_t rmax, int64_t* out) {
  API_BEGIN
  ttn_assert(rks && dims && out && d >= 1, TTN_EARG, "r_and_d_to_rks: bad arguments");
  const std::vector<int64_t> r = r_and_d_to_rks(std::vector<int64_t>(rks, rks + d + 1), std::vector<int64_t>(dims, dims + d), rmax);
  for (int i = 0; i <= d; ++i) out[i] = r[i];
  API_END
}

int ttn_dev_alloc(size_t bytes, void** out) {
  API_BEGIN
  need_init();
  TTN_CUDA(cudaMalloc(out, bytes));
  API_END
}
int ttn_dev_free(void* p) {
  API_BEGIN
  need_init();
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  TTN_CUDA(cudaFree(p));
  API_END
}
int ttn_h2d(void* dst, const void* src, size_t bytes) {
  API_BEGIN
  need_init();
  TTN_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  API_END
}
int ttn_d2h(void* dst, const void* src, size_t bytes) {
  API_BEGIN
  need_init();
  TTN_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx().stream));
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  API_END
}

}  // extern "C"
