// extern "C" boundary of libttn_b200.so (declared in include/ttn_b200.h).  Converts the library's internal
// exceptions into status codes; nothing else lives here.
#pragma GCC visibility push(default)
#include "../../include/ttn_b200.h"
#pragma GCC visibility pop
#include "tt.h"
#include "solvers.h"

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
template <class T>
static void upload_tt(TT<T>& t, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot, const void* const* cores,
                      int batch) {
  t.d = d; t.batch = batch;
  t.dims.assign(dims, dims + d);
  t.rks.assign(rks, rks + d + 1);
  if (ot) t.ot.assign(ot, ot + d); else t.ot.assign(d, 0);
  t.cores.clear();
  t.cores.resize(d);
  for (int k = 0; k < d; ++k) {
    ttn_assert(dims[k] >= 1 && rks[k] >= 1 && rks[k + 1] >= 1, TTN_EDIM, "upload: dims and ranks must be positive");
    t.alloc_core(k);
    TTN_CUDA(cudaMemcpyAsync(t.cores[k].p, cores[k], t.cores[k].bytes, cudaMemcpyHostToDevice, ctx().stream));
  }
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}
extern "C" {

int ttn_ttv_upload(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot, const void* const* cores,
                   int batch, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(d >= 1 && batch >= 1 && out, TTN_EARG, "upload: bad arguments");
  ttn_assert(dtype == TTN_F64 || dtype == TTN_C128, TTN_EARG, "upload: bad dtype");
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = dtype;
  try {
    if (dtype == TTN_F64) upload_tt(h->r, d, dims, rks, ot, cores, batch);
    else upload_tt(h->c, d, dims, rks, ot, cores, batch);
  } catch (...) { delete h; throw; }
  *out = h;
  API_END
}

#define TTV_FIELD(x, f) ((x)->dtype == TTN_F64 ? (x)->r.f : (x)->c.f)

}  // extern "C"
static cudaStream_t copy_stream() {
  Context& c = ctx();
  if (!c.copy_stream) TTN_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
  return c.copy_stream;
}
// the compute stream waits for a pending asynchronous upload of x (no host synchronisation)
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
      d.bufs = std::move(dtype == TTN_F64 ? r.cores : c.cores);
      deferred().v.push_back(std::move(d));
    }
  }
  ttn::drain_deferred_releases(false);
}

static void await_ready(ttn_ttv x) {
  if (x && x->ready) {
    TTN_CUDA(cudaStreamWaitEvent(ctx().stream, x->ready, 0));
    cudaEventDestroy(x->ready);
    x->ready = nullptr;
  }
}
extern "C" {

int ttn_ttv_upload_async(int dtype, int d, const int64_t* dims, const int64_t* rks, const int64_t* ot, const void* const* cores,
                         int batch, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(d >= 1 && batch >= 1 && out, TTN_EARG, "upload: bad arguments");
  ttn_assert(dtype == TTN_F64 || dtype == TTN_C128, TTN_EARG, "upload: bad dtype");
  drain_deferred_releases(false);
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = dtype;
  try {
    auto setup = [&](auto& t) {
      t.d = d; t.batch = batch;
      t.dims.assign(dims, dims + d);
      t.rks.assign(rks, rks + d + 1);
      if (ot) t.ot.assign(ot, ot + d); else t.ot.assign(d, 0);
      t.cores.clear();
      t.cores.resize(d);
      for (int k = 0; k < d; ++k) {
        ttn_assert(dims[k] >= 1 && rks[k] >= 1 && rks[k + 1] >= 1, TTN_EDIM, "upload: dims and ranks must be positive");
        t.alloc_core(k);
      }
      // the stream-ordered allocations become usable on the copy stream once the compute stream reaches this point
      cudaEvent_t ev;
      TTN_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      TTN_CUDA(cudaEventRecord(ev, ctx().stream));
      TTN_CUDA(cudaStreamWaitEvent(copy_stream(), ev, 0));
      cudaEventDestroy(ev);
      for (int k = 0; k < d; ++k)
        TTN_CUDA(cudaMemcpyAsync(t.cores[k].p, cores[k], t.cores[k].bytes, cudaMemcpyHostToDevice, copy_stream()));
    };
    if (dtype == TTN_F64) setup(h->r); else setup(h->c);
    TTN_CUDA(cudaEventCreateWithFlags(&h->ready, cudaEventDisableTiming));
    TTN_CUDA(cudaEventRecord(h->ready, copy_stream()));
  } catch (...) { delete h; throw; }
  *out = h;
  API_END
}
int ttn_ttv_wait(ttn_ttv x) {
  API_BEGIN
  need_init();
  await_ready(x);
  API_END
}
int ttn_ttv_download_async(ttn_ttv x, void* const* cores) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  await_ready(x);
  cudaEvent_t ev;
  TTN_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  TTN_CUDA(cudaEventRecord(ev, ctx().stream));            // everything queued on the compute stream so far has produced x
  TTN_CUDA(cudaStreamWaitEvent(copy_stream(), ev, 0));
  cudaEventDestroy(ev);
  const int d = TTV_FIELD(x, d);
  for (int k = 0; k < d; ++k) {
    const DevBuf& b = x->dtype == TTN_F64 ? x->r.cores[k] : x->c.cores[k];
    TTN_CUDA(cudaMemcpyAsync(cores[k], b.p, b.bytes, cudaMemcpyDeviceToHost, copy_stream()));
  }
  if (x->busy) cudaEventDestroy(x->busy);
  TTN_CUDA(cudaEventCreateWithFlags(&x->busy, cudaEventDisableTiming));
  TTN_CUDA(cudaEventRecord(x->busy, copy_stream()));
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
  if (d) *d = TTV_FIELD(x, d);
  if (batch) *batch = TTV_FIELD(x, batch);
  API_END
}
int ttn_ttv_ranks(ttn_ttv x, int64_t* rks) {
  API_BEGIN
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  const auto& v = TTV_FIELD(x, rks);
  std::copy(v.begin(), v.end(), rks);
  API_END
}
int ttn_ttv_dims(ttn_ttv x, int64_t* dims) {
  API_BEGIN
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  const auto& v = TTV_FIELD(x, dims);
  std::copy(v.begin(), v.end(), dims);
  API_END
}
int ttn_ttv_ot(ttn_ttv x, int64_t* ot) {
  API_BEGIN
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  const auto& v = TTV_FIELD(x, ot);
  std::copy(v.begin(), v.end(), ot);
  API_END
}
int ttn_ttv_download(ttn_ttv x, void* const* cores) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  await_ready(x);
  const int d = TTV_FIELD(x, d);
  for (int k = 0; k < d; ++k) {
    const DevBuf& b = x->dtype == TTN_F64 ? x->r.cores[k] : x->c.cores[k];
    TTN_CUDA(cudaMemcpyAsync(cores[k], b.p, b.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  }
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
  API_END
}
int ttn_ttv_copy(ttn_ttv x, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(x && out, TTN_EARG, "null handle");
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = x->dtype;
  try {
    if (x->dtype == TTN_F64) tt_copy(x->r, h->r); else tt_copy(x->c, h->c);
  } catch (...) { delete h; throw; }
  *out = h;
  API_END
}
int ttn_ttv_complex(ttn_ttv x, ttn_ttv* out) {
  API_BEGIN
  need_init();
  ttn_assert(x && out, TTN_EARG, "null handle");
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = TTN_C128;
  try {
    if (x->dtype == TTN_C128) tt_copy(x->c, h->c);
    else tt_to_complex(x->r, h->c);
  } catch (...) { delete h; throw; }
  *out = h;
  API_END
}
int ttn_ttv_free(ttn_ttv x) {
  API_BEGIN
  delete x;
  API_END
}

}  // extern "C"
template <class T>
static void upload_tto(TTO<T>& t, int d, const int64_t* dims, const int64_t* rks, const void* const* cores) {
  t.d = d;
  t.dims.assign(dims, dims + d);
  t.rks.assign(rks, rks + d + 1);
  t.cores.clear();
  t.cores.resize(d);
  for (int k = 0; k < d; ++k) {
    t.cores[k].alloc(sizeof(T) * (size_t)(dims[k] * dims[k] * rks[k] * rks[k + 1]));
    TTN_CUDA(cudaMemcpyAsync(t.cores[k].p, cores[k], t.cores[k].bytes, cudaMemcpyHostToDevice, ctx().stream));
  }
  TTN_CUDA(cudaStreamSynchronize(ctx().stream));
}
extern "C" {
int ttn_tto_upload(int dtype, int d, const int64_t* dims, const int64_t* rks, const void* const* cores, ttn_tto* out) {
  API_BEGIN
  need_init();
  ttn_assert(d >= 1 && out, TTN_EARG, "upload: bad arguments");
  ttn_assert(dtype == TTN_F64 || dtype == TTN_C128, TTN_EARG, "upload: bad dtype");
  ttn_tto h = new ttn_tto_s();
  h->dtype = dtype;
  try {
    if (dtype == TTN_F64) upload_tto(h->r, d, dims, rks, cores); else upload_tto(h->c, d, dims, rks, cores);
  } catch (...) { delete h; throw; }
  *out = h;
  API_END
}
int ttn_tto_complex(ttn_tto A, ttn_tto* out) {
  API_BEGIN
  need_init();
  ttn_assert(A && out, TTN_EARG, "null handle");
  ttn_tto h = new ttn_tto_s();
  h->dtype = TTN_C128;
  try {
    if (A->dtype == TTN_C128) tto_copy(A->c, h->c); else tto_to_complex(A->r, h->c);
  } catch (...) { delete h; throw; }
  *out = h;
  API_END
}
int ttn_tto_info(ttn_tto A, int* dtype, int* d) {
  API_BEGIN
  ttn_assert(A != nullptr, TTN_EARG, "null handle");
  if (dtype) *dtype = A->dtype;
  if (d) *d = A->dtype == TTN_F64 ? A->r.d : A->c.d;
  API_END
}
int ttn_tto_ranks(ttn_tto A, int64_t* rks) {
  API_BEGIN
  ttn_assert(A && rks, TTN_EARG, "null handle");
  const auto& v = A->dtype == TTN_F64 ? A->r.rks : A->c.rks;
  std::copy(v.begin(), v.end(), rks);
  API_END
}
int ttn_tto_dims(ttn_tto A, int64_t* dims) {
  API_BEGIN
  ttn_assert(A && dims, TTN_EARG, "null handle");
  const auto& v = A->dtype == TTN_F64 ? A->r.dims : A->c.dims;
  std::copy(v.begin(), v.end(), dims);
  API_END
}
int ttn_tto_download(ttn_tto A, void* const* cores) {
  API_BEGIN
  need_init();
  ttn_assert(A && cores, TTN_EARG, "null handle");
  const int d = A->dtype == TTN_F64 ? A->r.d : A->c.d;
  for (int k = 0; k < d; ++k) {
    const DevBuf& b = A->dtype == TTN_F64 ? A->r.cores[k] : A->c.cores[k];
    TTN_CUDA(cudaMemcpyAsync(cores[k], b.p, b.bytes, cudaMemcpyDeviceToHost, ctx().stream));
  }
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
  ttn_assert(A && x && y, TTN_EARG, "null handle");
  same_dtype(A->dtype, x->dtype);
  await_ready(x);
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = x->dtype;
  try {
    if (x->dtype == TTN_F64) tt_apply(A->r, x->r, h->r); else tt_apply(A->c, x->c, h->c);
  } catch (...) { delete h; throw; }
  *y = h;
  API_END
}
int ttn_dot(ttn_ttv a, ttn_ttv b, double* out) {
  API_BEGIN
  need_init();
  ttn_assert(a && b && out, TTN_EARG, "null handle");
  same_dtype(a->dtype, b->dtype);
  if (a->dtype == TTN_F64) {
    std::vector<double> v;
    tt_dot(a->r, b->r, v);
    for (size_t i = 0; i < v.size(); ++i) { out[2 * i] = v[i]; out[2 * i + 1] = 0.0; }
  } else {
    std::vector<zc> v;
    tt_dot(a->c, b->c, v);
    for (size_t i = 0; i < v.size(); ++i) { out[2 * i] = v[i].x; out[2 * i + 1] = v[i].y; }
  }
  API_END
}
int ttn_norm(ttn_ttv a, double* out) {
  API_BEGIN
  need_init();
  ttn_assert(a && out, TTN_EARG, "null handle");
  if (a->dtype == TTN_F64) {
    std::vector<double> v;
    tt_dot(a->r, a->r, v);
    for (size_t i = 0; i < v.size(); ++i) out[i] = std::sqrt(v[i] > 0 ? v[i] : 0.0);
  } else {
    std::vector<zc> v;
    tt_dot(a->c, a->c, v);
    for (size_t i = 0; i < v.size(); ++i) out[i] = std::sqrt(v[i].x > 0 ? v[i].x : 0.0);
  }
  API_END
}
int ttn_add(ttn_ttv x, ttn_ttv y, ttn_ttv* z) {
  API_BEGIN
  need_init();
  ttn_assert(x && y && z, TTN_EARG, "null handle");
  same_dtype(x->dtype, y->dtype);
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = x->dtype;
  try {
    if (x->dtype == TTN_F64) tt_add(x->r, y->r, h->r); else tt_add(x->c, y->c, h->c);
  } catch (...) { delete h; throw; }
  *z = h;
  API_END
}
int ttn_scale(ttn_ttv x, double re, double im, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(x && y, TTN_EARG, "null handle");
  ttn_assert(x->dtype == TTN_C128 || im == 0.0, TTN_EARG, "complex scalar on a real TT (promote first)");
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = x->dtype;
  try {
    if (x->dtype == TTN_F64) tt_scale(x->r, re, h->r); else tt_scale(x->c, make_cuDoubleComplex(re, im), h->c);
  } catch (...) { delete h; throw; }
  *y = h;
  API_END
}
int ttn_orthogonalize(ttn_ttv x, int center, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(x && y, TTN_EARG, "null handle");
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = x->dtype;
  try {
    if (x->dtype == TTN_F64) tt_orthogonalize(x->r, center, h->r); else tt_orthogonalize(x->c, center, h->c);
  } catch (...) { delete h; throw; }
  *y = h;
  API_END
}
int ttn_compress(ttn_ttv x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  await_ready(x);
  if (x->dtype == TTN_F64) tt_compress(x->r, max_bond, truncerr, sweeps, sigma_out, sigma_stride);
  else tt_compress(x->c, max_bond, truncerr, sweeps, sigma_out, sigma_stride);
  API_END
}
int ttn_apply_compress(ttn_tto A, ttn_ttv x, int64_t max_bond, double truncerr, int sweeps, double* sigma_out, int64_t sigma_stride,
                       ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(A && x && y, TTN_EARG, "null handle");
  same_dtype(A->dtype, x->dtype);
  await_ready(x);
  ttn_ttv h = new ttn_ttv_s();
  h->dtype = x->dtype;
  try {
    if (x->dtype == TTN_F64) tt_apply_compress(A->r, x->r, h->r, max_bond, truncerr, sweeps, sigma_out, sigma_stride);
    else tt_apply_compress(A->c, x->c, h->c, max_bond, truncerr, sweeps, sigma_out, sigma_stride);
  } catch (...) { delete h; throw; }
  *y = h;
  API_END
}
int ttn_bond_truncate(ttn_ttv x, int k, int64_t max_bond, double truncerr, ttn_ttv* y) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  if (x->dtype == TTN_F64) tt_bond_truncate(x->r, k, max_bond, truncerr, nullptr, 0);
  else tt_bond_truncate(x->c, k, max_bond, truncerr, nullptr, 0);
  if (y) {
    ttn_ttv h = new ttn_ttv_s();
    h->dtype = x->dtype;
    try {
      if (x->dtype == TTN_F64) tt_orthogonalize(x->r, k, h->r); else tt_orthogonalize(x->c, k, h->c);
    } catch (...) { delete h; throw; }
    *y = h;
  }
  API_END
}

int ttn_swap_sites(ttn_ttv x, int k, int mode, int64_t max_bond, double tol) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  ttn_assert(mode == 0 || mode == 1, TTN_EARG, "mode must be 0 (relative threshold) or 1 (tail norm)");
  if (x->dtype == TTN_F64) tt_swap_sites(x->r, k, mode, max_bond, tol);
  else tt_swap_sites(x->c, k, mode, max_bond, tol);
  API_END
}
int ttn_merge_sites_diag(ttn_ttv x, int k) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  if (x->dtype == TTN_F64) tt_merge_diag(x->r, k); else tt_merge_diag(x->c, k);
  API_END
}
int ttn_split_site(ttn_ttv x, int k, int64_t coarse, int mode, int64_t max_bond, double tol) {
  API_BEGIN
  need_init();
  ttn_assert(x != nullptr, TTN_EARG, "null handle");
  ttn_assert(mode == 0 || mode == 1, TTN_EARG, "mode must be 0 (relative threshold) or 1 (tail norm)");
  if (x->dtype == TTN_F64) tt_split_site(x->r, k, coarse, mode, max_bond, tol);
  else tt_split_site(x->c, k, coarse, mode, max_bond, tol);
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

#define SOLVER_PROLOGUE(A, x0)                                         \
  need_init();                                                         \
  ttn_assert(A && x0 && p && x, TTN_EARG, "null argument");            \
  same_dtype(A->dtype, x0->dtype);                                     \
  ttn_ttv h = new ttn_ttv_s();                                         \
  h->dtype = x0->dtype;

int ttn_als_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    ttn_assert(b != nullptr, TTN_EARG, "null argument");
    same_dtype(A->dtype, b->dtype);
    if (x0->dtype == TTN_F64) als_linsolve(A->r, b->r, x0->r, *p, h->r, residual);
    else als_linsolve(A->c, b->c, x0->c, *p, h->c, residual);
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
int ttn_als_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int cap_E, int* n_E) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    std::vector<double> Ev;
    if (x0->dtype == TTN_F64) als_eigsolve(A->r, x0->r, *p, h->r, Ev);
    else als_eigsolve(A->c, x0->c, *p, h->c, Ev);
    if (n_E) *n_E = (int)Ev.size();
    if (E) for (int i = 0; i < (int)Ev.size() && i < cap_E; ++i) E[i] = Ev[i];
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
int ttn_als_gen_eigsolv(ttn_tto A, ttn_tto S, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int cap_E, int* n_E) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    ttn_assert(S != nullptr, TTN_EARG, "null argument");
    same_dtype(A->dtype, S->dtype);
    std::vector<double> Ev;
    if (x0->dtype == TTN_F64) als_gen_eigsolve(A->r, S->r, x0->r, *p, h->r, Ev);
    else als_gen_eigsolve(A->c, S->c, x0->c, *p, h->c, Ev);
    if (n_E) *n_E = (int)Ev.size();
    if (E) for (int i = 0; i < (int)Ev.size() && i < cap_E; ++i) E[i] = Ev[i];
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
int ttn_mals_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    ttn_assert(b != nullptr, TTN_EARG, "null argument");
    same_dtype(A->dtype, b->dtype);
    if (x0->dtype == TTN_F64) mals_linsolve(A->r, b->r, x0->r, *p, h->r, residual);
    else mals_linsolve(A->c, b->c, x0->c, *p, h->c, residual);
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
int ttn_mals_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int64_t* r_hist, int cap_E,
                      int* n_E) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    std::vector<double> Ev;
    std::vector<int64_t> rh;
    if (x0->dtype == TTN_F64) mals_eigsolve(A->r, x0->r, *p, h->r, Ev, rh);
    else mals_eigsolve(A->c, x0->c, *p, h->c, Ev, rh);
    if (n_E) *n_E = (int)Ev.size();
    for (int i = 0; i < (int)Ev.size() && i < cap_E; ++i) {
      if (E) E[i] = Ev[i];
      if (r_hist) r_hist[i] = rh[i];
    }
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
int ttn_dmrg_linsolve(ttn_tto A, ttn_ttv b, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* residual) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    ttn_assert(b != nullptr, TTN_EARG, "null argument");
    same_dtype(A->dtype, b->dtype);
    if (x0->dtype == TTN_F64) dmrg_linsolve(A->r, b->r, x0->r, *p, h->r, residual);
    else dmrg_linsolve(A->c, b->c, x0->c, *p, h->c, residual);
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
int ttn_dmrg_eigsolve(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_ttv* x, double* E, int64_t* r_hist, int cap_E,
                      int* n_E) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  try {
    std::vector<double> Ev;
    std::vector<int64_t> rh;
    if (x0->dtype == TTN_F64) dmrg_eigsolve(A->r, x0->r, *p, h->r, Ev, rh);
    else dmrg_eigsolve(A->c, x0->c, *p, h->c, Ev, rh);
    if (n_E) *n_E = (int)Ev.size();
    for (int i = 0; i < (int)Ev.size() && i < cap_E; ++i) {
      if (E) E[i] = Ev[i];
      if (r_hist) r_hist[i] = rh[i];
    }
  } catch (...) { delete h; throw; }
  *x = h;
  API_END
}
// ---- multi-GPU DMRG: replicated sweep, sharded Lanczos matvec (shard.cu) -----------------------------------------
int ttn_shard_ctx_create(int dtype, int64_t max_elems, int rank, int nranks, ttn_shard_ctx* out) {
  API_BEGIN
  need_init();
  ttn_assert(out != nullptr && (dtype == TTN_F64 || dtype == TTN_C128), TTN_EARG, "shard ctx: bad arguments");
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
  if (c) shard_ctx_free(c);
  API_END
}
int ttn_dmrg_eigsolve_sharded(ttn_tto A, ttn_ttv x0, const ttn_solver_params* p, ttn_shard_ctx sc, ttn_ttv* x, double* E,
                              int64_t* r_hist, int cap_E, int* n_E) {
  API_BEGIN
  SOLVER_PROLOGUE(A, x0)
  ttn_assert(sc != nullptr, TTN_EARG, "null shard context");
  active_shard_ctx() = sc;
  try {
    std::vector<double> Ev;
    std::vector<int64_t> rh;
    if (x0->dtype == TTN_F64) dmrg_eigsolve(A->r, x0->r, *p, h->r, Ev, rh);
    else dmrg_eigsolve(A->c, x0->c, *p, h->c, Ev, rh);
    active_shard_ctx() = nullptr;
    ttn_assert(shard_ctx_error(sc) == 0, TTN_ECUDA,
               "sharded DMRG: a peer did not publish its slice within the epoch timeout (TTN_SHARD_TIMEOUT_S); the result is invalid");
    if (n_E) *n_E = (int)Ev.size();
    for (int i = 0; i < (int)Ev.size() && i < cap_E; ++i) {
      if (E) E[i] = Ev[i];
      if (r_hist) r_hist[i] = rh[i];
    }
  } catch (...) { active_shard_ctx() = nullptr; delete h; throw; }
  *x = h;
  API_END
}
int ttn_tdvp(ttn_tto H, ttn_ttv u0, const ttn_tdvp_params* p, ttn_ttv* u) {
  API_BEGIN
  need_init();
  ttn_assert(H && u0 && p && u, TTN_EARG, "null argument");
  same_dtype(H->dtype, u0->dtype);
  ttn_ttv h = new ttn_ttv_s();
  try {
    tdvp_drive(H, u0, *p, h);
  } catch (...) { delete h; throw; }
  *u = h;
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
  if (dtype == TTN_F64) gemm<double>(g); else gemm<zc>(g);
  API_END
}

int ttn_matvec2_host(int dtype, int w_l, int w_r, int chi_l, int chi_r, int nn, const void* G, const void* Amid, const void* H,
                     const void* V, void* Y, int symmetrize) {
  API_BEGIN
  need_init();
  if (dtype == TTN_F64) matvec2_host<double>(w_l, w_r, chi_l, chi_r, nn, G, Amid, H, V, Y, symmetrize != 0);
  else matvec2_host<zc>(w_l, w_r, chi_l, chi_r, nn, G, Amid, H, V, Y, symmetrize != 0);
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
  matvec2_free(mv);
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
  shard_free(mv);
  API_END
}
int ttn_env_left_host(int dtype, int n, int w_l, int w_r, int r_l, int r_r, const void* G, const void* x, const void* A,
                      void* Gout) {
  API_BEGIN
  need_init();
  if (dtype == TTN_F64) env_host<double>(true, n, w_l, w_r, r_l, r_r, G, x, A, Gout);
  else env_host<zc>(true, n, w_l, w_r, r_l, r_r, G, x, A, Gout);
  API_END
}
int ttn_env_right_host(int dtype, int n, int w_l, int w_r, int r_l, int r_r, const void* H, const void* x, const void* A,
                       void* Hout) {
  API_BEGIN
  need_init();
  if (dtype == TTN_F64) env_host<double>(false, n, w_l, w_r, r_l, r_r, H, x, A, Hout);
  else env_host<zc>(false, n, w_l, w_r, r_l, r_r, H, x, A, Hout);
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
  if (dtype == TTN_F64) svdtrunc_host<double>(m, n, A, max_bond, truncerr, U, s, Vt, r_out);
  else svdtrunc_host<zc>(m, n, A, max_bond, truncerr, U, s, Vt, r_out);
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
  if (dtype == TTN_F64) heig_host<double>(n, nev, batch, G, lam, U, flags); else heig_host<zc>(n, nev, batch, G, lam, U, flags);
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
  if (dtype == TTN_F64) qr_host<double>(m, n, A, Q, R); else qr_host<zc>(m, n, A, Q, R);
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
