// C ABI of the uml_b200 engine (see include/uml_b200.h): device binding, model/batch residency, predict calls.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <nvtx3/nvToolsExt.h>
#include <sched.h>

#include "uml_common.cuh"
#include "mlp_rescore.cuh"

// NVTX ranges around the phases of a call (stage / score / re-score / exchange); free when no tool is attached
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

namespace uml {
cudaError_t launch_finite_scan(const float* x, int64_t ld, int64_t rows, int n_features, StageResult* result,
                               cudaStream_t stream);
cudaError_t launch_push_bytes(const void* src, void* const* dst, int n_dst, int64_t bytes, int sm_count,
                              cudaStream_t stream);
cudaError_t launch_labels_take(const void* labels, int label_bytes, int64_t n, const double* classes, int n_classes,
                               double* out, cudaStream_t stream);
cudaError_t launch_labels_count_equal(const void* labels, int label_bytes, int64_t n, const double* classes,
                                      int n_classes, const double* targets, unsigned long long* count,
                                      cudaStream_t stream);
}

using uml::FlagList;
using uml::LinearDeviceModel;
using uml::LinearLaunch;
using uml::StageResult;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static thread_local std::string g_create_error;

constexpr int kSmallRows = 64;              // online path: batches up to this many rows take the one-kernel fp64 route
constexpr int64_t kSmallBytes = 256 << 10;   // ... when their raw feature block fits the pinned request buffer

struct HostMirror {  // pinned; device counters are copied here
  int flag_count;
  int pad;
  unsigned long long counters[4];
  StageResult stage;
  uml::SmallResult small[kSmallRows];
};

// Host threads that gather a pageable source chunk into a pinned bounce buffer: cudaMemcpy from pageable memory is
// staged by the driver on one thread; a few threads doing plain memcpy into page-locked memory keep the link busy.
namespace uml {
int narrow_f64_to_f32(const double* src, float* dst, size_t n);  // host_narrow.cpp
}

class CopyPool {
 public:
  struct Task {  // `rows` runs of n bytes (rows == 1: one contiguous run)
    char* dst;
    const char* src;
    size_t n;
    size_t rows = 1, dpitch = 0, spitch = 0;
    // narrow != nullptr: the run is float64 and is written as float32 (n = source bytes, dst advances half as fast);
    // *narrow is set when a value does not survive the round trip (the caller then re-sends the chunk as float64)
    std::atomic<int>* narrow = nullptr;
  };
  explicit CopyPool(int n_threads) {
    for (int i = 0; i < n_threads; ++i) workers_.emplace_back([this] { loop(); });
  }
  ~CopyPool() {
    {
      std::lock_guard<std::mutex> g(mu_);
      stop_ = true;
    }
    cv_work_.notify_all();
    for (auto& t : workers_) t.join();
  }
  // copy every task; the calling thread works too and returns when all are done
  void run(const std::vector<Task>& tasks) {
    if (tasks.empty()) return;
    auto job = std::make_shared<Job>();
    job->tasks = tasks.data();
    job->n = tasks.size();
    {
      std::lock_guard<std::mutex> g(mu_);
      job_ = job;
      ++generation_;
    }
    cv_work_.notify_all();
    work(*job);
    std::unique_lock<std::mutex> g(mu_);
    cv_done_.wait(g, [&] { return job->done.load() == job->n; });
    job_.reset();
  }

 private:
  // a job owns its counters, so a worker that wakes up late only ever sees an exhausted index range of an old job
  struct Job {
    const Task* tasks = nullptr;
    size_t n = 0;
    std::atomic<size_t> next{0}, done{0};
  };
  void work(Job& job) {
    for (;;) {
      const size_t i = job.next.fetch_add(1);
      if (i >= job.n) return;
      const Task& t = job.tasks[i];
      if (t.narrow) {
        // (also "lossy" for NaN: such chunks travel as float64 and the staging kernel reports them)
        if (uml::narrow_f64_to_f32(reinterpret_cast<const double*>(t.src), reinterpret_cast<float*>(t.dst), t.n / 8))
          t.narrow->store(1, std::memory_order_relaxed);
      } else {
        for (size_t r = 0; r < t.rows; ++r) memcpy(t.dst + r * t.dpitch, t.src + r * t.spitch, t.n);
      }
      if (job.done.fetch_add(1) + 1 == job.n) {
        std::lock_guard<std::mutex> g(mu_);
        cv_done_.notify_all();
      }
    }
  }
  void loop() {
    uint64_t seen = 0;
    for (;;) {
      std::shared_ptr<Job> job;
      {
        std::unique_lock<std::mutex> g(mu_);
        cv_work_.wait(g, [&] { return stop_ || generation_ != seen; });
        if (stop_) return;
        seen = generation_;
        job = job_;
      }
      if (job) work(*job);
    }
  }
  std::vector<std::thread> workers_;
  std::mutex mu_;
  std::condition_variable cv_work_, cv_done_;
  std::shared_ptr<Job> job_;
  uint64_t generation_ = 0;
  bool stop_ = false;
};

struct SmallGraph {  // one captured H2D -> linear_small_kernel -> D2H per (model, rows, features, dtype)
  uint64_t model_uid = 0;
  int n_rows = 0, n_features = 0, dtype = 0;
  cudaGraphExec_t exec = nullptr;
  uint64_t last_use = 0;
};

struct uml_engine {
  int device = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev[6] = {};
  cudaEvent_t chunk_ev[8] = {};
  uml_device_info info{};
  PFN_encodeTiled encode = nullptr;
  std::string last_error;
  // device scratch
  int* d_flag_count = nullptr;
  unsigned long long* d_counters = nullptr;
  StageResult* d_stage = nullptr;
  int32_t* d_flag_rows = nullptr;
  int64_t flag_cap = 0;
  int32_t* d_labels = nullptr;
  int64_t labels_cap = 0;
  void* d_chunk[3] = {nullptr, nullptr, nullptr};  // raw source chunks (staging / predict_host)
  int64_t chunk_cap = 0;
  float* d_xchunk[3] = {nullptr, nullptr, nullptr};  // converted fp32 chunks (predict_host)
  int64_t xchunk_cap = 0;
  double* d_vchunk[3] = {nullptr, nullptr, nullptr};  // class values of a chunk (predict_host_values)
  int64_t vchunk_cap = 0;
  double* d_classes = nullptr;
  int classes_cap = 0;
  void* h_bounce[3] = {nullptr, nullptr, nullptr};  // pinned bounce buffers for pageable sources
  int64_t bounce_cap = 0;
  void* h_result[3] = {nullptr, nullptr, nullptr};  // pinned landing slots for labels / values bound for pageable outputs
  int64_t result_cap = 0;
  CopyPool* pool = nullptr;
  // online path (B <= kSmallRows): pinned request buffer, its device twin, result slots, cached graphs
  void* h_req = nullptr;
  void* d_req = nullptr;
  uml::SmallResult* d_small = nullptr;
  std::vector<SmallGraph> small_graphs;
  uint64_t small_tick = 0;
  // asynchronous host call (uml_linear_predict_host_values_begin / _poll / _finish): one in flight per engine
  std::thread async_thread;
  std::atomic<int64_t> async_rows_done{0};
  std::atomic<int> async_finished{1};
  int async_status = UML_OK;
  uml_stats async_stats{};

  bool small_graph_ok = true;
  HostMirror* h = nullptr;
};

static std::atomic<uint64_t> g_model_uid{1};

struct uml_model {
  uml_engine* e = nullptr;
  uint64_t uid = 0;  // changes whenever the device operands are re-uploaded (keys the cached small-batch graphs)
  LinearDeviceModel dm{};
  int n_features_in = 0;
  int n_classes_in = 0;  // as passed by the caller (1 for sklearn's binary layout)
  std::vector<double> coef64, intercept64;  // caller's values (expanded), before any affine fold
  float* d_wt = nullptr;
  float* d_bias = nullptr;
  double* d_w64 = nullptr;
  double* d_b64 = nullptr;
};

struct uml_batch {
  uml_engine* e = nullptr;
  float* x = nullptr;
  double* x64 = nullptr;
  int64_t n_rows = 0, ld = 0, ld64 = 0;
  int n_features = 0;
  bool owns = false;
  bool lossless = true;
  int tf32_exact = -1;  // every fp32 feature is a tf32 value: 1 yes, 0 no, -1 not scanned yet (wrapped device rows)
  bool has_map = false;
  CUtensorMap map{};  // boxes of 128 rows x 32 features
};

struct uml_mlp {
  uml_engine* e = nullptr;
  uml::MlpDeviceModel dm{};
  float* d_w1t = nullptr;
  float* d_b1 = nullptr;
  float* d_w2t = nullptr;
  float* d_b2 = nullptr;
  double* d_w64 = nullptr;  // w1 | b1 | w2 | b2 packed
  float* d_w1_tiles = nullptr;  // tensor-core B operand: tf32 hi | lo rows, pre-swizzled
  uml::MlpHostModel host;
};

#define UML_FAIL(E, CODE, ...)                              \
  do {                                                      \
    char _buf[512];                                         \
    snprintf(_buf, sizeof(_buf), __VA_ARGS__);              \
    if (E) (E)->last_error = _buf; else g_create_error = _buf; \
    return (CODE);                                          \
  } while (0)

#define UML_CUDA(E, CALL)                                                                              \
  do {                                                                                                 \
    cudaError_t _err = (CALL);                                                                         \
    if (_err != cudaSuccess) {                                                                         \
      UML_FAIL(E, _err == cudaErrorMemoryAllocation ? UML_ERR_NOMEM : UML_ERR_CUDA, "%s failed: %s", #CALL, \
               cudaGetErrorString(_err));                                                              \
    }                                                                                                  \
  } while (0)

static int dtype_size(int dt) {
  switch (dt) {
    case UML_F32: return 4;
    case UML_F64: return 8;
    case UML_I64: return 8;
    case UML_I32: return 4;
    case UML_U8: return 1;
    default: return 0;
  }
}

extern "C" {

int uml_abi_version(void) { return UML_B200_ABI_VERSION; }

const char* uml_last_error(const uml_engine* e) { return e ? e->last_error.c_str() : g_create_error.c_str(); }

int uml_engine_create(uml_engine** out, int device_id) {
  if (!out) UML_FAIL((uml_engine*)nullptr, UML_ERR_INVALID, "uml_engine_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t err = cudaGetDeviceCount(&n);
  if (err != cudaSuccess || n == 0)
    UML_FAIL((uml_engine*)nullptr, UML_ERR_NO_DEVICE, "no CUDA device visible (%s); uml_b200 has no CPU fallback",
             err != cudaSuccess ? cudaGetErrorString(err) : "device count 0");
  if (device_id < 0 || device_id >= n)
    UML_FAIL((uml_engine*)nullptr, UML_ERR_INVALID, "device_id %d out of range [0,%d)", device_id, n);
  uml_engine* e = new uml_engine();
  e->device = device_id;
  auto fail = [&](const char* what, cudaError_t ce) {
    char buf[256];
    snprintf(buf, sizeof(buf), "%s: %s", what, cudaGetErrorString(ce));
    g_create_error = buf;
    delete e;
    return (int)UML_ERR_CUDA;
  };
  if ((err = cudaSetDevice(device_id)) != cudaSuccess) return fail("cudaSetDevice", err);
  cudaDeviceProp prop;
  if ((err = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return fail("cudaGetDeviceProperties", err);
  e->info.device_id = device_id;
  e->info.sm_count = prop.multiProcessorCount;
  e->info.cc_major = prop.major;
  e->info.cc_minor = prop.minor;
  e->info.total_mem_bytes = (int64_t)prop.totalGlobalMem;
  e->info.l2_bytes = prop.l2CacheSize;
  cudaDeviceGetAttribute(&e->info.sm_clock_khz, cudaDevAttrClockRate, device_id);
  cudaDeviceGetAttribute(&e->info.mem_clock_khz, cudaDevAttrMemoryClockRate, device_id);
  strncpy(e->info.name, prop.name, sizeof(e->info.name) - 1);
  if (prop.major != 10) {
    char buf[256];
    snprintf(buf, sizeof(buf), "device %d (%s) is compute capability %d.%d; this library is built for sm_100a only",
             device_id, prop.name, prop.major, prop.minor);
    g_create_error = buf;
    delete e;
    return UML_ERR_NO_DEVICE;
  }
  if ((err = cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking)) != cudaSuccess)
    return fail("cudaStreamCreate", err);
  if ((err = cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking)) != cudaSuccess)
    return fail("cudaStreamCreate", err);
  e->stream = e->own_stream;
  for (auto& ev : e->ev)
    if ((err = cudaEventCreate(&ev)) != cudaSuccess) return fail("cudaEventCreate", err);
  for (auto& ev : e->chunk_ev)
    if ((err = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", err);
  if ((err = cudaMalloc(&e->d_flag_count, sizeof(int))) != cudaSuccess) return fail("cudaMalloc", err);
  if ((err = cudaMalloc(&e->d_counters, 4 * sizeof(unsigned long long))) != cudaSuccess) return fail("cudaMalloc", err);
  if ((err = cudaMalloc(&e->d_stage, sizeof(StageResult))) != cudaSuccess) return fail("cudaMalloc", err);
  if ((err = cudaHostAlloc((void**)&e->h, sizeof(HostMirror), cudaHostAllocMapped)) != cudaSuccess)
    return fail("cudaHostAlloc", err);
  memset(e->h, 0, sizeof(HostMirror));
  // the scoring steps do not memset these: the re-score kernel hands the flag list back empty (linear_kernels.cu)
  if ((err = cudaMemset(e->d_flag_count, 0, sizeof(int))) != cudaSuccess) return fail("cudaMemset", err);
  if ((err = cudaMemset(e->d_counters, 0, 4 * sizeof(unsigned long long))) != cudaSuccess) return fail("cudaMemset", err);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  err = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (err != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return fail("cuTensorMapEncodeTiled lookup", err);
  e->encode = (PFN_encodeTiled)fn;
  *out = e;
  return UML_OK;
}

void uml_engine_destroy(uml_engine* e) {
  if (!e) return;
  if (e->async_thread.joinable()) e->async_thread.join();
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  cudaFree(e->d_flag_count);
  cudaFree(e->d_counters);
  cudaFree(e->d_stage);
  cudaFree(e->d_flag_rows);
  cudaFree(e->d_labels);
  for (auto p : e->d_chunk) cudaFree(p);
  for (auto p : e->d_xchunk) cudaFree(p);
  for (auto p : e->d_vchunk) cudaFree(p);
  cudaFree(e->d_classes);
  for (auto p : e->h_bounce)
    if (p) cudaFreeHost(p);
  for (auto p : e->h_result)
    if (p) cudaFreeHost(p);
  delete e->pool;
  for (auto& g : e->small_graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (e->h_req) cudaFreeHost(e->h_req);  // d_req / d_small are device aliases of pinned host memory
  if (e->h) cudaFreeHost(e->h);
  for (auto ev : e->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto ev : e->chunk_ev)
    if (ev) cudaEventDestroy(ev);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  delete e;
}

int uml_engine_info(const uml_engine* e, uml_device_info* out) {
  if (!e || !out) return UML_ERR_INVALID;
  *out = e->info;
  return UML_OK;
}

int uml_engine_set_stream(uml_engine* e, void* cuda_stream) {
  if (!e) return UML_ERR_INVALID;
  e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
  return UML_OK;
}

int uml_engine_synchronize(uml_engine* e) {
  if (!e) return UML_ERR_INVALID;
  UML_CUDA(e, cudaSetDevice(e->device));
  UML_CUDA(e, cudaStreamSynchronize(e->stream));
  UML_CUDA(e, cudaStreamSynchronize(e->copy_stream));
  return UML_OK;
}

int uml_host_alloc(uml_engine* e, void** out, int64_t bytes) {
  if (!e || !out || bytes < 0) return UML_ERR_INVALID;
  UML_CUDA(e, cudaSetDevice(e->device));
  UML_CUDA(e, cudaHostAlloc(out, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocDefault));
  return UML_OK;
}

int uml_device_alloc(uml_engine* e, void** out, int64_t bytes) {
  if (!e || !out || bytes < 0) return UML_ERR_INVALID;
  UML_CUDA(e, cudaSetDevice(e->device));
  UML_CUDA(e, cudaMalloc(out, (size_t)(bytes > 0 ? bytes : 1)));
  return UML_OK;
}

int uml_device_free(uml_engine* e, void* p) {
  if (!e) return UML_ERR_INVALID;
  UML_CUDA(e, cudaSetDevice(e->device));
  if (p) UML_CUDA(e, cudaFree(p));
  return UML_OK;
}

int uml_host_free(uml_engine* e, void* p) {
  if (!e) return UML_ERR_INVALID;
  if (p) UML_CUDA(e, cudaFreeHost(p));
  return UML_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------------------------
static int upload_model(uml_engine* e, uml_model* m, const std::vector<double>& w, const std::vector<double>& b) {
  const int C = m->dm.n_classes, F = m->dm.n_features;
  const int cp = (C + 1 + 3) / 4 * 4;
  const int f_pad = (F + uml::kChunkF - 1) / uml::kChunkF * uml::kChunkF;
  std::vector<float> wt((size_t)f_pad * cp, 0.f), bias(cp, 0.f);
  float bmax = 0.f;
  for (int c = 0; c < C; ++c) {
    bias[c] = (float)b[c];
    bmax = fmaxf(bmax, fabsf(bias[c]));
  }
  bias[C] = bmax;
  for (int f = 0; f < F; ++f) {
    float wmax = 0.f;
    for (int c = 0; c < C; ++c) {
      const float v = (float)w[(size_t)c * F + f];
      wt[(size_t)f * cp + c] = v;
      wmax = fmaxf(wmax, fabsf(v));
    }
    wt[(size_t)f * cp + C] = wmax;
  }
  auto ensure = [&](void** p, size_t bytes) -> cudaError_t {
    if (*p) cudaFree(*p);
    *p = nullptr;
    return cudaMalloc(p, bytes);
  };
  UML_CUDA(e, ensure((void**)&m->d_wt, wt.size() * 4));
  UML_CUDA(e, ensure((void**)&m->d_bias, bias.size() * 4));
  // fp64 weights feature-major: w64t[f][stride], the classes of one feature contiguous (zero padded)
  const int stride = uml::linear_w64_stride(C);
  std::vector<double> w64t((size_t)F * stride, 0.0);
  for (int c = 0; c < C; ++c)
    for (int f = 0; f < F; ++f) w64t[(size_t)f * stride + c] = w[(size_t)c * F + f];
  UML_CUDA(e, ensure((void**)&m->d_w64, w64t.size() * 8));
  UML_CUDA(e, ensure((void**)&m->d_b64, b.size() * 8));
  UML_CUDA(e, cudaMemcpy(m->d_wt, wt.data(), wt.size() * 4, cudaMemcpyHostToDevice));
  UML_CUDA(e, cudaMemcpy(m->d_bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice));
  UML_CUDA(e, cudaMemcpy(m->d_w64, w64t.data(), w64t.size() * 8, cudaMemcpyHostToDevice));
  UML_CUDA(e, cudaMemcpy(m->d_b64, b.data(), b.size() * 8, cudaMemcpyHostToDevice));
  m->dm.wt = m->d_wt;
  m->dm.bias = m->d_bias;
  m->dm.w64 = m->d_w64;
  m->dm.b64 = m->d_b64;
  m->dm.w64_stride = stride;
  m->dm.cp = cp;
  m->dm.f_pad = f_pad;
  m->uid = g_model_uid.fetch_add(1);
  return UML_OK;
}

int uml_linear_load(uml_engine* e, uml_model** out, const void* coef, const void* intercept, int n_classes,
                    int n_features, int dtype) {
  if (!e || !out || !coef || !intercept) return UML_ERR_INVALID;
  *out = nullptr;
  if (n_classes < 1 || n_features < 1) UML_FAIL(e, UML_ERR_INVALID, "n_classes=%d n_features=%d", n_classes, n_features);
  if (dtype != UML_F32 && dtype != UML_F64) UML_FAIL(e, UML_ERR_INVALID, "coef dtype must be F32 or F64");
  UML_CUDA(e, cudaSetDevice(e->device));
  auto get = [&](const void* p, size_t i) -> double {
    return dtype == UML_F64 ? ((const double*)p)[i] : (double)((const float*)p)[i];
  };
  uml_model* m = new uml_model();
  m->e = e;
  m->n_features_in = n_features;
  m->n_classes_in = n_classes;
  const int C = n_classes == 1 ? 2 : n_classes;  // binary: scores > 0  <=>  argmax([0, s]) with first-max ties
  const int F = n_features;
  m->coef64.assign((size_t)C * F, 0.0);
  m->intercept64.assign(C, 0.0);
  const int c0 = n_classes == 1 ? 1 : 0;
  for (int c = 0; c < n_classes; ++c) {
    for (int f = 0; f < F; ++f) m->coef64[(size_t)(c + c0) * F + f] = get(coef, (size_t)c * F + f);
    m->intercept64[c + c0] = get(intercept, c);
  }
  m->dm.n_classes = C;
  m->dm.n_features = F;
  int rc = upload_model(e, m, m->coef64, m->intercept64);
  if (rc != UML_OK) {
    uml_model_free(m);
    return rc;
  }
  *out = m;
  return UML_OK;
}

int uml_linear_set_affine(uml_engine* e, uml_model* m, const double* shift, const double* scale) {
  if (!e || !m) return UML_ERR_INVALID;
  UML_CUDA(e, cudaSetDevice(e->device));
  const int C = m->dm.n_classes, F = m->dm.n_features;
  std::vector<double> w = m->coef64, b = m->intercept64;
  // s_c = sum_f ((x_f - shift_f) * scale_f) w_cf + b_c = sum_f x_f (scale_f w_cf) + (b_c - sum_f shift_f scale_f w_cf)
  for (int c = 0; c < C; ++c) {
    double acc = b[c];
    for (int f = 0; f < F; ++f) {
      const double sc = scale ? scale[f] : 1.0;
      const double sh = shift ? shift[f] : 0.0;
      const double wf = w[(size_t)c * F + f] * sc;
      w[(size_t)c * F + f] = wf;
      acc -= sh * wf;
    }
    b[c] = acc;
  }
  return upload_model(e, m, w, b);
}

void uml_model_free(uml_model* m) {
  if (!m) return;
  if (m->e) cudaSetDevice(m->e->device);
  cudaFree(m->d_wt);
  cudaFree(m->d_bias);
  cudaFree(m->d_w64);
  cudaFree(m->d_b64);
  delete m;
}

// ---------------------------------------------------------------------------------------------------------------
// batch
// ---------------------------------------------------------------------------------------------------------------
static int encode_map(uml_engine* e, CUtensorMap* map, const float* x, int64_t n_rows, int F, int64_t ld,
                      int box_rows = uml::kTileRows) {
  if (((uintptr_t)x & 15) != 0 || (ld % 4) != 0) UML_FAIL(e, UML_ERR_UNSUPPORTED, "rows must be 16-byte aligned with ld %% 4 == 0");
  if (n_rows >= (1ll << 31) - uml::kTileRows) UML_FAIL(e, UML_ERR_UNSUPPORTED, "more than 2^31 rows in one batch");
  cuuint64_t gdim[2] = {(cuuint64_t)F, (cuuint64_t)n_rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)uml::kChunkF, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = e->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)x, gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) UML_FAIL(e, UML_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for %lld x %d ld %lld", (int)r,
                                  (long long)n_rows, F, (long long)ld);
  return UML_OK;
}

int uml_batch_from_device(uml_engine* e, uml_batch** out, const void* dev_ptr, int64_t n_rows, int n_features,
                          int64_t ld) {
  if (!e || !out || (!dev_ptr && n_rows > 0) || n_rows < 0 || n_features < 1 || ld < n_features) return UML_ERR_INVALID;
  *out = nullptr;
  UML_CUDA(e, cudaSetDevice(e->device));
  uml_batch* b = new uml_batch();
  b->e = e;
  b->x = (float*)dev_ptr;
  b->n_rows = n_rows;
  b->n_features = n_features;
  b->ld = ld;
  b->owns = false;
  if (n_rows > 0) {
    int rc = encode_map(e, &b->map, b->x, n_rows, n_features, ld);
    if (rc == UML_OK) b->has_map = true;
    else if (rc != UML_ERR_UNSUPPORTED) {
      delete b;
      return rc;
    }
  }
  *out = b;
  return UML_OK;
}

static int ensure_chunks(uml_engine* e, int64_t bytes) {
  if (e->chunk_cap >= bytes) return UML_OK;
  for (auto& p : e->d_chunk) {
    cudaFree(p);
    p = nullptr;
  }
  e->chunk_cap = 0;
  for (auto& p : e->d_chunk) UML_CUDA(e, cudaMalloc(&p, (size_t)bytes));
  e->chunk_cap = bytes;
  return UML_OK;
}

struct SrcLayout {
  bool feature_major;
  int64_t pitch_elems;
  int elem;
};

static int classify_layout(uml_engine* e, int64_t n_rows, int F, int64_t rs, int64_t cs, int dtype, SrcLayout* L) {
  const int elem = dtype_size(dtype);
  if (!elem) UML_FAIL(e, UML_ERR_INVALID, "unknown dtype %d", dtype);
  L->elem = elem;
  if (cs == elem || F == 1) {
    if (rs % elem != 0 || rs < (int64_t)F * elem) {
      if (n_rows > 1) UML_FAIL(e, UML_ERR_UNSUPPORTED, "row stride %lld not a multiple of the element size / overlaps", (long long)rs);
      rs = (int64_t)F * elem;
    }
    L->feature_major = false;
    L->pitch_elems = rs / elem;
    return UML_OK;
  }
  if (rs == elem || n_rows == 1) {
    if (cs % elem != 0 || cs < n_rows * elem) UML_FAIL(e, UML_ERR_UNSUPPORTED, "column stride %lld unsupported", (long long)cs);
    L->feature_major = true;
    L->pitch_elems = cs / elem;
    return UML_OK;
  }
  UML_FAIL(e, UML_ERR_UNSUPPORTED, "features must be contiguous along rows or along columns (strides %lld, %lld bytes)",
           (long long)rs, (long long)cs);
}

// copy rows [r0, r0+rows) of the host source into device chunk buffer `dst` (compact: pitch = F or rows elements)
static cudaError_t copy_chunk_h2d(void* dst, const void* host, const SrcLayout& L, int64_t r0, int64_t rows, int F,
                                  cudaStream_t s) {
  const char* src = (const char*)host;
  if (!L.feature_major) {
    const size_t width = (size_t)F * L.elem;
    const size_t spitch = (size_t)L.pitch_elems * L.elem;
    if (spitch == width) return cudaMemcpyAsync(dst, src + (size_t)r0 * spitch, width * rows, cudaMemcpyHostToDevice, s);
    return cudaMemcpy2DAsync(dst, width, src + (size_t)r0 * spitch, spitch, width, (size_t)rows, cudaMemcpyHostToDevice, s);
  }
  const size_t width = (size_t)rows * L.elem;
  const size_t spitch = (size_t)L.pitch_elems * L.elem;
  return cudaMemcpy2DAsync(dst, width, src + (size_t)r0 * L.elem, spitch, width, (size_t)F, cudaMemcpyHostToDevice, s);
}

static bool host_ptr_is_pinned(const void* p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    (void)cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

static bool lossy_capable(int dtype) { return dtype == UML_F64 || dtype == UML_I64 || dtype == UML_I32; }

// gather tasks for rows [r0, r0+rows) of the host source into a compact chunk (row-major [rows][F] or feature-major
// [F][rows]) at `dst`; contiguous runs are cut into <= 1 MiB pieces so the pool's threads share them
static void build_gather_tasks(std::vector<CopyPool::Task>& tasks, char* dst, const void* host, const SrcLayout& L,
                               int64_t r0, int64_t rows, int F, std::atomic<int>* narrow = nullptr) {
  tasks.clear();
  const char* src = (const char*)host;
  const size_t piece = 1u << 20;
  // narrow (float64 source only, contiguous runs): the destination holds float32, so it advances half as fast
  auto add_run = [&](char* d, const char* s_, size_t n) {
    for (size_t o = 0; o < n; o += piece) {
      CopyPool::Task t{d + (narrow ? o / 2 : o), s_ + o, std::min(piece, n - o)};
      t.narrow = narrow;
      tasks.push_back(t);
    }
  };
  if (!L.feature_major) {
    const size_t width = (size_t)F * L.elem, spitch = (size_t)L.pitch_elems * L.elem;
    if (spitch == width) {
      add_run(dst, src + (size_t)r0 * spitch, width * (size_t)rows);
    } else {
      // strided rows (a column slice of a wider C-order array): blocks of rows, each row its own run
      const int64_t rows_per_task = std::max<int64_t>(1, (int64_t)(piece / width));
      for (int64_t r = 0; r < rows; r += rows_per_task) {
        const int64_t n = std::min(rows_per_task, rows - r);
        tasks.push_back({dst + (size_t)r * width, src + (size_t)(r0 + r) * spitch, width, (size_t)n, width, spitch});
      }
    }
  } else {
    const size_t run = (size_t)rows * L.elem, spitch = (size_t)L.pitch_elems * L.elem;
    for (int f = 0; f < F; ++f)
      add_run(dst + (size_t)f * (narrow ? run / 2 : run), src + (size_t)f * spitch + (size_t)r0 * L.elem, run);
  }
}

// CPUs this process can use: scheduler affinity, capped by the cgroup CPU quota (v2 cpu.max, v1 cfs_quota_us)
static int usable_cpus(int* logical = nullptr) {
  int n = (int)std::thread::hardware_concurrency();
  cpu_set_t set;
  if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
  if (n <= 0) n = 4;
  if (logical) *logical = n;  // CPUs the scheduler may place threads on (before the quota)
  auto read_two = [](const char* path, long long* a, long long* b) -> bool {
    FILE* f = fopen(path, "r");
    if (!f) return false;
    char first[64] = {0};
    const int got = fscanf(f, "%63s %lld", first, b);
    fclose(f);
    if (got < 1 || strcmp(first, "max") == 0) return false;
    *a = atoll(first);
    return got == 2;
  };
  long long quota = 0, period = 0;
  if (read_two("/sys/fs/cgroup/cpu.max", &quota, &period) && quota > 0 && period > 0) {
    n = std::min<long long>(n, std::max<long long>(1, quota / period));
  } else {
    FILE* fq = fopen("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "r");
    FILE* fp = fopen("/sys/fs/cgroup/cpu/cpu.cfs_period_us", "r");
    if (fq && fp && fscanf(fq, "%lld", &quota) == 1 && fscanf(fp, "%lld", &period) == 1 && quota > 0 && period > 0)
      n = std::min<long long>(n, std::max<long long>(1, quota / period));
    if (fq) fclose(fq);
    if (fp) fclose(fp);
  }
  return n;
}

// pinned bounce buffers (3 slots) + the copy pool, created on first use
static int ensure_bounce(uml_engine* e, int64_t bytes) {
  if (e->bounce_cap < bytes) {
    for (auto& p : e->h_bounce) {
      if (p) cudaFreeHost(p);
      p = nullptr;
    }
    e->bounce_cap = 0;
    for (auto& p : e->h_bounce) UML_CUDA(e, cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault));
    e->bounce_cap = bytes;
  }
  if (!e->pool) {
    int n = 0;
    if (const char* env = getenv("UML_B200_COPY_THREADS")) n = atoi(env);
    // default: sized from the CPU time this process may really use (affinity and cgroup quota - the GPU boxes give a
    // container a 16-CPU quota on 128 logical CPUs).  The gather threads are stalled on host memory most of the time
    // and idle between chunks, so 1.5 x the quota is where the 10M x 64 float64 frame gathers fastest on those boxes
    // (threads: pipeline ms  10: 98, 14: 99, 20: 77-89, 24: 70, 28: 74, 32: 70, 40: 77-116, 56: 133 - past ~2 x the
    // quota CFS throttles every thread for the rest of the period).  Never more than the logical CPUs minus two (the
    // caller's thread fills the result list meanwhile), at most 32, and the CPUs are shared by the ranks of this node
    // (torchrun exports LOCAL_WORLD_SIZE).
    if (n <= 0) {
      int ranks = 1;
      if (const char* lw = getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, atoi(lw));
      int logical = 0;
      const int quota = usable_cpus(&logical);
      n = std::min(32, std::max(1, std::min(logical - 2, quota * 3 / 2) / ranks));
    }
    e->pool = new CopyPool(n - 1);  // the calling thread is the n-th worker
  }
  return UML_OK;
}

static bool want_bounce(const void* host_ptr, int64_t bytes) {
  return bytes >= (8ll << 20) && !host_ptr_is_pinned(host_ptr) && !getenv("UML_B200_NO_BOUNCE");
}

int uml_stage_rows(uml_engine* e, uml_batch** out, const void* host_ptr, int64_t n_rows, int n_features,
                   int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, uint32_t flags) {
  if (!e || !out || (!host_ptr && n_rows > 0) || n_rows < 0 || n_features < 1) return UML_ERR_INVALID;
  *out = nullptr;
  UML_CUDA(e, cudaSetDevice(e->device));
  (void)cudaGetLastError();
  SrcLayout L{};
  int rc = UML_OK;
  if (n_rows > 0 && (rc = classify_layout(e, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype, &L)) != UML_OK)
    return rc;
  const int F = n_features;
  const int64_t ld = (F + 3) / 4 * 4;
  const bool check = !(flags & UML_STAGE_SKIP_FINITE_CHECK);
  // float64 / int64 / int32 values may not survive the fp32 down-cast (|int32| > 2^24 does not)
  const bool want64 = (flags & UML_STAGE_KEEP_F64) && (src_dtype == UML_F64 || src_dtype == UML_I64 || src_dtype == UML_I32);

  uml_batch* b = new uml_batch();
  b->e = e;
  b->n_rows = n_rows;
  b->n_features = F;
  b->ld = ld;
  b->owns = true;
  auto bail = [&](int code) {
    uml_batch_free(b);
    return code;
  };
  if (n_rows == 0) {
    *out = b;
    return UML_OK;
  }
  cudaError_t ce;
  if ((ce = cudaMalloc((void**)&b->x, (size_t)n_rows * ld * 4)) != cudaSuccess) {
    e->last_error = std::string("cudaMalloc(batch): ") + cudaGetErrorString(ce);
    return bail(ce == cudaErrorMemoryAllocation ? UML_ERR_NOMEM : UML_ERR_CUDA);
  }
  if (want64) {
    b->ld64 = F;
    if ((ce = cudaMalloc((void**)&b->x64, (size_t)n_rows * F * 8)) != cudaSuccess) {
      e->last_error = std::string("cudaMalloc(batch f64): ") + cudaGetErrorString(ce);
      return bail(ce == cudaErrorMemoryAllocation ? UML_ERR_NOMEM : UML_ERR_CUDA);
    }
  }
  cudaStream_t cs = e->stream;
#define STAGE_CUDA(CALL)                                                            \
  do {                                                                              \
    cudaError_t _e2 = (CALL);                                                       \
    if (_e2 != cudaSuccess) {                                                       \
      e->last_error = std::string(#CALL) + ": " + cudaGetErrorString(_e2);          \
      cudaStreamSynchronize(cs);                                                    \
      cudaStreamSynchronize(e->copy_stream);                                        \
      return bail(UML_ERR_CUDA);                                                    \
    }                                                                               \
  } while (0)
  STAGE_CUDA(cudaMemsetAsync(e->d_stage, 0, sizeof(StageResult), cs));

  // already the resident layout and page-locked: one straight H2D, then the finiteness scan (a large pageable source
  // goes through the chunked path instead, where host threads feed pinned bounce buffers)
  const bool direct = !L.feature_major && src_dtype == UML_F32 && L.pitch_elems == ld &&
                      !want_bounce(host_ptr, n_rows * (int64_t)F * L.elem);
  if (direct) {
    STAGE_CUDA(cudaMemcpyAsync(b->x, host_ptr, (size_t)n_rows * ld * 4, cudaMemcpyHostToDevice, cs));
    if (check) STAGE_CUDA(uml::launch_finite_scan(b->x, ld, n_rows, F, e->d_stage, cs));
  } else {
    // chunked: H2D of raw source bytes on the copy stream, transpose/convert kernel on the compute stream
    const int64_t row_bytes = (int64_t)F * L.elem;
    int64_t chunk_rows = std::max<int64_t>(1024, (64ll << 20) / row_bytes);
    chunk_rows = std::min<int64_t>((chunk_rows + 31) / 32 * 32, std::max<int64_t>(n_rows, 1));
    int rc2 = ensure_chunks(e, chunk_rows * row_bytes);
    if (rc2 != UML_OK) return bail(rc2);
    // pageable frames: a few host threads gather each chunk into a pinned bounce buffer (see CopyPool)
    const bool bounce = want_bounce(host_ptr, n_rows * row_bytes);
    if (bounce && (rc2 = ensure_bounce(e, chunk_rows * row_bytes)) != UML_OK) return bail(rc2);
    std::vector<CopyPool::Task> tasks;
    int slot = 0;
    bool used[3] = {false, false, false};
    for (int64_t r0 = 0; r0 < n_rows; r0 += chunk_rows, slot = (slot + 1) % 3) {
      const int64_t rows = std::min(chunk_rows, n_rows - r0);
      if (used[slot]) STAGE_CUDA(cudaStreamWaitEvent(e->copy_stream, e->chunk_ev[3 + slot], 0));  // convert done
      if (bounce) {
        if (used[slot]) STAGE_CUDA(cudaEventSynchronize(e->chunk_ev[slot]));  // previous H2D has left the bounce buffer
        build_gather_tasks(tasks, (char*)e->h_bounce[slot], host_ptr, L, r0, rows, F);
        e->pool->run(tasks);
        STAGE_CUDA(cudaMemcpyAsync(e->d_chunk[slot], e->h_bounce[slot], (size_t)(rows * row_bytes), cudaMemcpyHostToDevice,
                                   e->copy_stream));
      } else
      STAGE_CUDA(copy_chunk_h2d(e->d_chunk[slot], host_ptr, L, r0, rows, F, e->copy_stream));
      STAGE_CUDA(cudaEventRecord(e->chunk_ev[slot], e->copy_stream));
      STAGE_CUDA(cudaStreamWaitEvent(cs, e->chunk_ev[slot], 0));
      STAGE_CUDA(uml::launch_stage_convert(e->d_chunk[slot], src_dtype, L.feature_major, L.feature_major ? rows : F,
                                           rows, F, b->x + r0 * ld, ld, b->x64 ? b->x64 + r0 * b->ld64 : nullptr,
                                           b->ld64, e->d_stage, check, cs));
      STAGE_CUDA(cudaEventRecord(e->chunk_ev[3 + slot], cs));
      used[slot] = true;
    }
  }
  STAGE_CUDA(cudaMemcpyAsync(&e->h->stage, e->d_stage, sizeof(StageResult), cudaMemcpyDeviceToHost, cs));
  STAGE_CUDA(cudaStreamSynchronize(cs));
#undef STAGE_CUDA
  if (check && e->h->stage.nonfinite) {
    e->last_error = "Input X contains NaN or infinity.";
    return bail(UML_ERR_NONFINITE);
  }
  b->lossless = direct ? true : e->h->stage.lossy == 0;
  if (check || !direct) b->tf32_exact = e->h->stage.not_tf32 == 0 ? 1 : 0;  // the scan / conversion pass saw every value
  if (b->x64 && b->lossless) {
    cudaFree(b->x64);
    b->x64 = nullptr;
  }
  rc = encode_map(e, &b->map, b->x, n_rows, F, ld);
  if (rc == UML_OK) b->has_map = true;
  else if (rc != UML_ERR_UNSUPPORTED) return bail(rc);
  *out = b;
  return UML_OK;
}

int uml_batch_info(const uml_batch* b, int64_t* n_rows, int* n_features, int64_t* ld, const void** dev_ptr,
                   int* lossless) {
  if (!b) return UML_ERR_INVALID;
  if (n_rows) *n_rows = b->n_rows;
  if (n_features) *n_features = b->n_features;
  if (ld) *ld = b->ld;
  if (dev_ptr) *dev_ptr = b->x;
  if (lossless) *lossless = b->lossless ? 1 : 0;
  return UML_OK;
}

void uml_batch_free(uml_batch* b) {
  if (!b) return;
  if (b->e) cudaSetDevice(b->e->device);
  if (b->owns) cudaFree(b->x);
  cudaFree(b->x64);
  delete b;
}

// ---------------------------------------------------------------------------------------------------------------
// predict
// ---------------------------------------------------------------------------------------------------------------
static int ensure_flags(uml_engine* e, int64_t rows) {
  if (e->flag_cap >= rows) return UML_OK;
  cudaFree(e->d_flag_rows);
  e->d_flag_rows = nullptr;
  e->flag_cap = 0;
  UML_CUDA(e, cudaMalloc((void**)&e->d_flag_rows, (size_t)rows * 4));
  e->flag_cap = rows;
  return UML_OK;
}

static int ensure_labels(uml_engine* e, int64_t rows) {
  if (e->labels_cap >= rows) return UML_OK;
  cudaFree(e->d_labels);
  e->d_labels = nullptr;
  e->labels_cap = 0;
  UML_CUDA(e, cudaMalloc((void**)&e->d_labels, (size_t)rows * 4));
  e->labels_cap = rows;
  return UML_OK;
}

// enqueue the scoring of one resident block of rows on e->stream; no host synchronisation.
// ev_k (optional) brackets the scoring kernel, ev_r the fp64 re-score.
static int enqueue_predict(uml_engine* e, const uml_model* m, const LinearLaunch& l, const CUtensorMap* map, int mode,
                           bool timed, int* launches, int* path) {
  FlagList fl{e->d_flag_count, e->d_flag_rows, (int)std::min<int64_t>(e->flag_cap, INT32_MAX), e->d_counters};
  const bool exact = mode == UML_PREDICT_EXACT;
  std::string why;
  const bool tma = map != nullptr && uml::linear_tma_supported(m->dm, &why);
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[1], e->stream));
  if (tma) {
    NvtxRange r_score("uml:score");
    std::string err;
    bool need_rescore = false;
    cudaError_t ce = uml::launch_linear_tma(*map, m->dm, l, exact, fl, e->info.sm_count, e->stream, &err, &need_rescore);
    if (ce != cudaSuccess) UML_FAIL(e, UML_ERR_CUDA, "linear_argmax_tma launch: %s %s", cudaGetErrorString(ce), err.c_str());
    *launches += 1;
    *path = 1;
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
    if (need_rescore) {  // UML_B200_RESCORE_MODE=kernel; in queue mode flagged rows are re-scored by a warp of the tile kernel
      NvtxRange r_rescore("uml:rescore_f64");
      UML_CUDA(e, uml::launch_rescore_f64(m->dm, l, fl, false, e->info.sm_count, e->stream));
      *launches += 1;
    }
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[3], e->stream));
  } else {
    NvtxRange r_score("uml:score_f64_generic");
    UML_CUDA(e, uml::launch_rescore_f64(m->dm, l, fl, true, e->info.sm_count, e->stream));
    *launches += 1;
    *path = 2;
    if (timed) {
      UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
      UML_CUDA(e, cudaEventRecord(e->ev[3], e->stream));
    }
  }
  return UML_OK;
}

static int finish_stats(uml_engine* e, uml_stats* stats, int64_t n_rows, int launches, int path, bool timed,
                        bool kernel_events = true) {
  // counters -> pinned mirror, then synchronise and report
  UML_CUDA(e, cudaMemcpyAsync(&e->h->flag_count, e->d_flag_count, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  UML_CUDA(e, cudaMemcpyAsync(e->h->counters, e->d_counters, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                              e->stream));
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[4], e->stream));
  UML_CUDA(e, cudaStreamSynchronize(e->stream));
  if (stats) {
    stats->n_rows = n_rows;
    stats->n_ambiguous = (int64_t)e->h->counters[0];
    stats->n_nonfinite = (int64_t)e->h->counters[1];
    stats->n_flagged = (int64_t)e->h->counters[2];
    stats->kernel_launches = launches;
    stats->path = path;
    if (timed) {
      float ms = 0.f;
      if (kernel_events) {
        if (cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]) == cudaSuccess) stats->kernel_ms = ms;
        if (cudaEventElapsedTime(&ms, e->ev[2], e->ev[3]) == cudaSuccess) stats->recheck_ms = ms;
      }
      if (cudaEventElapsedTime(&ms, e->ev[0], e->ev[4]) == cudaSuccess) stats->total_ms = ms;
      (void)cudaGetLastError();  // never leave a stale error behind for the next launch check
    }
  }
  if (e->h->counters[1] > 0) UML_FAIL(e, UML_ERR_NONFINITE, "Input X contains NaN or infinity.");
  return UML_OK;
}

static int predict_common(uml_engine* e, const uml_model* m, const uml_batch* b, int32_t* labels_out,
                          int labels_on_device, void* const* peers, int n_peers, int64_t row_offset, int label_bytes,
                          int mode, uml_stats* stats) {
  if (!e || !m || !b) return UML_ERR_INVALID;
  if (!labels_out && b->n_rows > 0 && n_peers == 0) return UML_ERR_INVALID;
  if (mode != UML_PREDICT_FAST && mode != UML_PREDICT_EXACT) UML_FAIL(e, UML_ERR_INVALID, "mode %d", mode);
  if (n_peers < 0 || n_peers > 8) UML_FAIL(e, UML_ERR_INVALID, "n_peers %d (max 8)", n_peers);
  if (n_peers > 0 && label_bytes != 1 && label_bytes != 4) UML_FAIL(e, UML_ERR_INVALID, "label_bytes %d", label_bytes);
  if (n_peers > 0 && label_bytes == 1 && m->dm.n_classes > 256)
    UML_FAIL(e, UML_ERR_UNSUPPORTED, "byte labels need n_classes <= 256 (model has %d)", m->dm.n_classes);
  if (b->n_features != m->n_features_in)
    UML_FAIL(e, UML_ERR_SHAPE, "X has %d features, but the estimator is expecting %d features as input.",
             b->n_features, m->n_features_in);
  UML_CUDA(e, cudaSetDevice(e->device));
  (void)cudaGetLastError();
  if (stats) memset(stats, 0, sizeof(*stats));
  if (b->n_rows == 0) return UML_OK;
  const bool exact = mode == UML_PREDICT_EXACT;
  const bool timed = stats != nullptr;
  int rc;
  if (exact && (rc = ensure_flags(e, b->n_rows)) != UML_OK) return rc;
  int32_t* d_labels = labels_out;
  const bool wire_u8 = n_peers > 0 && label_bytes == 1;
  if (!labels_out && n_peers > 0 && !wire_u8) {
    // fused exchange: entry 0 is this rank's own full-length vector -> it is the local label target
    d_labels = static_cast<int32_t*>(peers[0]) + row_offset;
    peers += 1;
    n_peers -= 1;
  } else if (!labels_out && wire_u8) {
    d_labels = nullptr;  // byte vectors everywhere (own vector included among the peers); no int32 copy kept
  } else if (!labels_on_device || !labels_out) {
    if ((rc = ensure_labels(e, b->n_rows)) != UML_OK) return rc;
    d_labels = e->d_labels;
  }
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[0], e->stream));
  if (stats || !labels_on_device) {
    // synchronous call: the counters are read back at the end, start them from zero.  The asynchronous step (device
    // labels, no stats) needs no memset at all: the flag list is handed back empty by the previous re-score kernel.
    UML_CUDA(e, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), e->stream));
    UML_CUDA(e, cudaMemsetAsync(e->d_flag_count, 0, sizeof(int), e->stream));
  }
  LinearLaunch l{};
  l.x = b->x;
  l.x64 = b->x64;
  l.ld = b->ld;
  l.ld64 = b->ld64;
  l.n_rows = b->n_rows;
  l.labels = d_labels;
  l.n_peers = n_peers;
  l.wire_u8 = wire_u8 ? 1 : 0;
  for (int i = 0; i < n_peers; ++i) l.peers[i] = peers[i];
  l.row_offset = row_offset;
  int launches = 0, path = 0;
  rc = enqueue_predict(e, m, l, b->has_map ? &b->map : nullptr, mode, timed, &launches, &path);
  if (rc != UML_OK) return rc;
  int64_t d2h = 0;
  if (!labels_on_device && labels_out) {
    UML_CUDA(e, cudaMemcpyAsync(labels_out, d_labels, (size_t)b->n_rows * 4, cudaMemcpyDeviceToHost, e->stream));
    d2h = b->n_rows * 4;
  }
  if (stats || !labels_on_device) {
    rc = finish_stats(e, stats, b->n_rows, launches, path, timed);
    if (stats) {
      stats->d2h_bytes = d2h;
    }
    return rc;
  }
  return UML_OK;
}

int uml_linear_predict(uml_engine* e, const uml_model* m, const uml_batch* b, int32_t* labels_out,
                       int labels_on_device, int mode, uml_stats* stats) {
  return predict_common(e, m, b, labels_out, labels_on_device, nullptr, 0, 0, 4, mode, stats);
}

int uml_linear_predict_peers(uml_engine* e, const uml_model* m, const uml_batch* b, void* const* peer_labels,
                             int n_peers, int64_t row_offset, int label_bytes, int mode, uml_stats* stats) {
  if (!peer_labels || n_peers < 1) return UML_ERR_INVALID;
  // peer_labels[0] must be this rank's own vector (local target); labels land at peer_labels[i] + row_offset for all i
  return predict_common(e, m, b, nullptr, 1, peer_labels, n_peers, row_offset, label_bytes, mode, stats);
}

// labels (device, int32 or uint8 indices) -> classes_[idx] as float64 in HOST memory: the device-side classes_.take of
// sklearn/linear_model/_base.py:423 followed by the float conversion of the canonical predictor (README.md:92)
int uml_labels_take(uml_engine* e, const void* labels_dev, int label_bytes, int64_t n, const double* classes_host,
                    int n_classes, double* out_host) {
  if (!e || (!labels_dev && n > 0) || !classes_host || n_classes < 1 || (!out_host && n > 0) || n < 0) return UML_ERR_INVALID;
  if (label_bytes != 1 && label_bytes != 4) UML_FAIL(e, UML_ERR_INVALID, "label_bytes %d", label_bytes);
  UML_CUDA(e, cudaSetDevice(e->device));
  if (n == 0) return UML_OK;
  double* d_classes = nullptr;
  double* d_out = nullptr;
  UML_CUDA(e, cudaMalloc((void**)&d_classes, (size_t)n_classes * 8));
  cudaError_t ce = cudaMalloc((void**)&d_out, (size_t)n * 8);
  if (ce != cudaSuccess) {
    cudaFree(d_classes);
    UML_FAIL(e, UML_ERR_NOMEM, "uml_labels_take: %s", cudaGetErrorString(ce));
  }
  auto done = [&](int rc) {
    cudaStreamSynchronize(e->stream);
    cudaFree(d_classes);
    cudaFree(d_out);
    return rc;
  };
  if ((ce = cudaMemcpyAsync(d_classes, classes_host, (size_t)n_classes * 8, cudaMemcpyHostToDevice, e->stream)) != cudaSuccess ||
      (ce = uml::launch_labels_take(labels_dev, label_bytes, n, d_classes, n_classes, d_out, e->stream)) != cudaSuccess ||
      (ce = cudaMemcpyAsync(out_host, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream)) != cudaSuccess ||
      (ce = cudaStreamSynchronize(e->stream)) != cudaSuccess) {
    e->last_error = std::string("uml_labels_take: ") + cudaGetErrorString(ce);
    return done(UML_ERR_CUDA);
  }
  return done(UML_OK);
}

// number of rows whose predicted class value equals the target (the numerator of accuracy_score in the reference's
// evaluator, README.md:94-100); targets are float64 in HOST memory
int uml_labels_count_equal(uml_engine* e, const void* labels_dev, int label_bytes, int64_t n, const double* classes_host,
                           int n_classes, const double* targets_host, int64_t* count_out) {
  if (!e || (!labels_dev && n > 0) || !classes_host || n_classes < 1 || (!targets_host && n > 0) || !count_out || n < 0)
    return UML_ERR_INVALID;
  if (label_bytes != 1 && label_bytes != 4) UML_FAIL(e, UML_ERR_INVALID, "label_bytes %d", label_bytes);
  UML_CUDA(e, cudaSetDevice(e->device));
  *count_out = 0;
  if (n == 0) return UML_OK;
  double* d_classes = nullptr;
  double* d_targets = nullptr;
  UML_CUDA(e, cudaMalloc((void**)&d_classes, (size_t)n_classes * 8));
  cudaError_t ce = cudaMalloc((void**)&d_targets, (size_t)n * 8);
  if (ce != cudaSuccess) {
    cudaFree(d_classes);
    UML_FAIL(e, UML_ERR_NOMEM, "uml_labels_count_equal: %s", cudaGetErrorString(ce));
  }
  auto done = [&](int rc) {
    cudaStreamSynchronize(e->stream);
    cudaFree(d_classes);
    cudaFree(d_targets);
    return rc;
  };
  if ((ce = cudaMemcpyAsync(d_classes, classes_host, (size_t)n_classes * 8, cudaMemcpyHostToDevice, e->stream)) != cudaSuccess ||
      (ce = cudaMemcpyAsync(d_targets, targets_host, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream)) != cudaSuccess ||
      (ce = cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), e->stream)) != cudaSuccess ||
      (ce = uml::launch_labels_count_equal(labels_dev, label_bytes, n, d_classes, n_classes, d_targets, e->d_counters, e->stream)) != cudaSuccess ||
      (ce = cudaMemcpyAsync(e->h->counters, e->d_counters, sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream)) != cudaSuccess ||
      (ce = cudaStreamSynchronize(e->stream)) != cudaSuccess) {
    e->last_error = std::string("uml_labels_count_equal: ") + cudaGetErrorString(ce);
    return done(UML_ERR_CUDA);
  }
  *count_out = (int64_t)e->h->counters[0];
  return done(UML_OK);
}

int uml_labels_push(uml_engine* e, const void* src, void* const* dst, int n_dst, int64_t bytes) {
  if (!e || (!src && bytes > 0) || !dst || n_dst < 1 || n_dst > 8 || bytes < 0) return UML_ERR_INVALID;
  UML_CUDA(e, cudaSetDevice(e->device));
  UML_CUDA(e, uml::launch_push_bytes(src, dst, n_dst, bytes, e->info.sm_count, e->stream));
  return UML_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// host rows -> host labels
// ---------------------------------------------------------------------------------------------------------------
// are the first rows of a host source tf32 values once cast to fp32 (low 13 mantissa bits zero)?  A cheap guess used
// to pick the MLP kernel for the chunk pipeline; correctness never depends on it
static bool host_sample_is_tf32(const void* host, const SrcLayout& L, int64_t n_rows, int F, int dtype) {
  const int64_t rows = std::min<int64_t>(n_rows, 2048);
  const char* base = (const char*)host;
  for (int64_t r = 0; r < rows; ++r)
    for (int f = 0; f < F; ++f) {
      const size_t i = L.feature_major ? (size_t)f * L.pitch_elems + r : (size_t)r * L.pitch_elems + f;
      float v;
      switch (dtype) {
        case UML_F64: v = (float)((const double*)base)[i]; break;
        case UML_I64: v = (float)((const long long*)base)[i]; break;
        case UML_I32: v = (float)((const int*)base)[i]; break;
        case UML_U8: v = (float)((const unsigned char*)base)[i]; break;
        default: v = ((const float*)base)[i]; break;
      }
      uint32_t bits;
      memcpy(&bits, &v, 4);
      if (bits & 0x1fffu) return false;
    }
  return true;
}

// B <= kSmallRows: request block -> pinned (device-mapped) buffer -> linear_small_kernel (replayed as a CUDA graph) ->
// labels written straight into pinned host memory.  fp64 from the caller's own values, so the result is the
// exact-mode result for either mode.
static int predict_host_small(uml_engine* e, const uml_model* m, const void* host_ptr, int n_rows, int F,
                              const SrcLayout& L, int src_dtype, int32_t* labels_out, double* values_out,
                              const double* classes, int n_classes, uml_stats* stats) {
  NvtxRange r_all("uml:predict_host_small");
  const size_t width = (size_t)F * L.elem;
  const size_t bytes = width * (size_t)n_rows;
  if (!e->h_req) {
    // zero-copy: the kernel reads the request straight from page-locked host memory over PCIe (16 KiB for 32 x 64
    // float64) and writes the labels straight back - no H2D / D2H copy nodes on the latency path
    UML_CUDA(e, cudaHostAlloc(&e->h_req, (size_t)kSmallBytes, cudaHostAllocMapped));
    UML_CUDA(e, cudaHostGetDevicePointer(&e->d_req, e->h_req, 0));
    void* d_small = nullptr;
    UML_CUDA(e, cudaHostGetDevicePointer(&d_small, e->h->small, 0));
    e->d_small = (uml::SmallResult*)d_small;
  }
  // gather into the pinned request buffer as compact row-major rows (the kernel reads any order, but a compact
  // block keeps the H2D copy one contiguous piece)
  {
    const char* src = (const char*)host_ptr;
    char* dst = (char*)e->h_req;
    if (!L.feature_major) {
      const size_t spitch = (size_t)L.pitch_elems * L.elem;
      if (spitch == width) memcpy(dst, src, bytes);
      else for (int r = 0; r < n_rows; ++r) memcpy(dst + (size_t)r * width, src + (size_t)r * spitch, width);
    } else {
      // feature-major request (a pandas block): typed transpose into rows
      const size_t pitch = (size_t)L.pitch_elems;
      auto transpose = [&](auto* d, const auto* s_) {
        for (int f = 0; f < F; ++f)
          for (int r = 0; r < n_rows; ++r) d[(size_t)r * F + f] = s_[(size_t)f * pitch + r];
      };
      switch (L.elem) {
        case 8: transpose((uint64_t*)dst, (const uint64_t*)src); break;
        case 4: transpose((uint32_t*)dst, (const uint32_t*)src); break;
        default: transpose((uint8_t*)dst, (const uint8_t*)src); break;
      }
    }
  }
  uml::SrcView view{e->d_req, src_dtype, (long long)F, 1};
  auto enqueue = [&](cudaStream_t s) -> cudaError_t { return uml::launch_linear_small(m->dm, view, n_rows, e->d_small, s); };
  static const bool no_graph = getenv("UML_B200_NO_GRAPH") != nullptr;
  bool launched = false;
  if (e->small_graph_ok && !no_graph) {
    SmallGraph* hit = nullptr;
    for (auto& g : e->small_graphs)
      if (g.model_uid == m->uid && g.n_rows == n_rows && g.n_features == F && g.dtype == src_dtype) hit = &g;
    if (!hit) {
      cudaGraph_t graph = nullptr;
      cudaGraphExec_t exec = nullptr;
      cudaError_t ce = cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal);
      if (ce == cudaSuccess) {
        cudaError_t body = enqueue(e->stream);
        ce = cudaStreamEndCapture(e->stream, &graph);
        if (body != cudaSuccess) ce = body;
      }
      if (ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {
        (void)cudaGetLastError();
        e->small_graph_ok = false;  // capture is not available here (e.g. the caller's stream is itself capturing)
      } else {
        if (e->small_graphs.size() >= 16) {  // evict the least recently used
          size_t lru = 0;
          for (size_t i = 1; i < e->small_graphs.size(); ++i)
            if (e->small_graphs[i].last_use < e->small_graphs[lru].last_use) lru = i;
          cudaGraphExecDestroy(e->small_graphs[lru].exec);
          e->small_graphs.erase(e->small_graphs.begin() + (long)lru);
        }
        e->small_graphs.push_back({m->uid, n_rows, F, src_dtype, exec, 0});
        hit = &e->small_graphs.back();
      }
    }
    if (hit) {
      hit->last_use = ++e->small_tick;
      UML_CUDA(e, cudaGraphLaunch(hit->exec, e->stream));
      launched = true;
    }
  }
  if (!launched) UML_CUDA(e, enqueue(e->stream));
  UML_CUDA(e, cudaStreamSynchronize(e->stream));
  int64_t n_bad = 0, n_amb = 0;
  for (int r = 0; r < n_rows; ++r) {
    const uml::SmallResult& q = e->h->small[r];
    if (labels_out) labels_out[r] = q.label;
    if (values_out) values_out[r] = (q.label >= 0 && q.label < n_classes) ? classes[q.label] : NAN;
    n_bad += q.status & 1;
    n_amb += (q.status >> 1) & 1;
  }
  if (stats) {
    stats->n_rows = n_rows;
    stats->n_nonfinite = n_bad;
    stats->n_ambiguous = n_amb;
    stats->kernel_launches = 1;
    stats->path = 4;
    stats->h2d_bytes = (int64_t)bytes;  // read by the kernel over PCIe (zero-copy), not by a copy engine
    stats->d2h_bytes = (int64_t)sizeof(uml::SmallResult) * n_rows;
  }
  if (n_bad > 0) UML_FAIL(e, UML_ERR_NONFINITE, "Input X contains NaN or infinity.");
  return UML_OK;
}

static int predict_host_impl(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows, int n_features,
                             int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out,
                             double* values_out, const double* classes, int n_classes, int mode, int64_t chunk_rows,
                             uml_stats* stats, std::atomic<int64_t>* progress = nullptr, const uml_mlp* mlp = nullptr) {
  // exactly one of m (linear classifier) and mlp (2-layer MLP) scores the chunks
  if (!e || (!m && !mlp) || (!host_ptr && n_rows > 0) || (!labels_out && !values_out && n_rows > 0) || n_rows < 0 ||
      n_features < 1)
    return UML_ERR_INVALID;
  if (values_out && (!classes || n_classes < 1)) return UML_ERR_INVALID;
  if (mode != UML_PREDICT_FAST && mode != UML_PREDICT_EXACT) UML_FAIL(e, UML_ERR_INVALID, "mode %d", mode);
  if (mlp) {
    if (n_features != mlp->dm.n_in)
      UML_FAIL(e, UML_ERR_SHAPE, "X has %d features, but the module is expecting %d features as input.", n_features,
               mlp->dm.n_in);
  } else if (n_features != m->n_features_in) {
    UML_FAIL(e, UML_ERR_SHAPE, "X has %d features, but the estimator is expecting %d features as input.", n_features,
             m->n_features_in);
  }
  UML_CUDA(e, cudaSetDevice(e->device));
  (void)cudaGetLastError();
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n_rows == 0) return UML_OK;
  SrcLayout L{};
  int rc = classify_layout(e, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype, &L);
  if (rc != UML_OK) return rc;
  const int F = n_features;
  if (!mlp && n_rows <= kSmallRows && (int64_t)F * L.elem * n_rows <= kSmallBytes) {
    rc = predict_host_small(e, m, host_ptr, (int)n_rows, F, L, src_dtype, labels_out, values_out, classes, n_classes, stats);
    if (progress && rc == UML_OK) progress->store(n_rows);
    return rc;
  }

  NvtxRange r_all("uml:predict_host");
  const int64_t ld = (F + 3) / 4 * 4;
  const bool exact = mode == UML_PREDICT_EXACT;
  const int64_t row_bytes = (int64_t)F * L.elem;
  if (chunk_rows <= 0) chunk_rows = std::max<int64_t>(4096, (32ll << 20) / std::max<int64_t>(ld * 4, row_bytes));
  chunk_rows = std::min<int64_t>((chunk_rows + 127) / 128 * 128, (n_rows + 127) / 128 * 128);
  const bool direct = !L.feature_major && src_dtype == UML_F32 && L.pitch_elems == ld;
  // pageable sources of any size worth the trouble go through pinned bounce buffers filled by the copy pool
  const bool bounce = want_bounce(host_ptr, n_rows * row_bytes);

  if (!direct && (rc = ensure_chunks(e, chunk_rows * row_bytes)) != UML_OK) return rc;
  if (e->xchunk_cap < chunk_rows * ld) {
    for (auto& p : e->d_xchunk) {
      cudaFree(p);
      p = nullptr;
    }
    e->xchunk_cap = 0;
    for (auto& p : e->d_xchunk) UML_CUDA(e, cudaMalloc((void**)&p, (size_t)chunk_rows * ld * 4));
    e->xchunk_cap = chunk_rows * ld;
  }
  // bytes of one row as it travels: `direct` rows keep their padding up to ld
  const int64_t wire_row_bytes = direct ? ld * 4 : row_bytes;
  if (bounce && (rc = ensure_bounce(e, chunk_rows * wire_row_bytes)) != UML_OK) return rc;
  if (values_out) {
    if (e->vchunk_cap < chunk_rows) {
      for (auto& p : e->d_vchunk) {
        cudaFree(p);
        p = nullptr;
      }
      e->vchunk_cap = 0;
      for (auto& p : e->d_vchunk) UML_CUDA(e, cudaMalloc((void**)&p, (size_t)chunk_rows * 8));
      e->vchunk_cap = chunk_rows;
    }
    if (e->classes_cap < n_classes) {
      cudaFree(e->d_classes);
      e->d_classes = nullptr;
      e->classes_cap = 0;
      UML_CUDA(e, cudaMalloc((void**)&e->d_classes, (size_t)n_classes * 8));
      e->classes_cap = n_classes;
    }
  }
  if ((rc = ensure_labels(e, 3 * chunk_rows)) != UML_OK) return rc;
  if (exact && (rc = ensure_flags(e, chunk_rows)) != UML_OK) return rc;
  // A device-to-host copy into PAGEABLE memory blocks the calling thread until the chunk's whole pipeline has drained,
  // which would serialise gather / H2D / scoring.  Pageable outputs therefore land in pinned slots first and are
  // copied out by the host when the slot comes round again (three chunks later) or at the end.
  // (the asynchronous variant always does: the flush is also where a finished prefix is published to the poller)
  const bool result_bounce = progress != nullptr || (labels_out && !host_ptr_is_pinned(labels_out)) ||
                             (values_out && !host_ptr_is_pinned(values_out));
  if (result_bounce && e->result_cap < chunk_rows * 12) {
    for (auto& p : e->h_result) {
      if (p) cudaFreeHost(p);
      p = nullptr;
    }
    e->result_cap = 0;
    for (auto& p : e->h_result) UML_CUDA(e, cudaHostAlloc(&p, (size_t)(chunk_rows * 12), cudaHostAllocDefault));
    e->result_cap = chunk_rows * 12;
  }
  struct Pending {
    int64_t r0 = 0, rows = 0;
    bool live = false;
  } pending[3];
  auto flush_slot = [&](int sl) -> cudaError_t {
    if (!pending[sl].live) return cudaSuccess;
    cudaError_t fe = cudaEventSynchronize(e->chunk_ev[3 + sl]);  // recorded after the slot's D2H copies
    if (fe != cudaSuccess) return fe;
    const char* base = (const char*)e->h_result[sl];
    if (values_out) memcpy(values_out + pending[sl].r0, base, (size_t)pending[sl].rows * 8);
    if (labels_out) memcpy(labels_out + pending[sl].r0, base + (size_t)chunk_rows * 8, (size_t)pending[sl].rows * 4);
    pending[sl].live = false;
    if (progress) progress->store(pending[sl].r0 + pending[sl].rows, std::memory_order_release);  // slots flush in row order
    return cudaSuccess;
  };

  // MLP: tensor cores when the features look like tf32 values (a host-side sample of the first rows decides; rows that
  // are not are caught in the kernel and re-scored, so a wrong guess costs time, never labels), CUDA cores otherwise
  bool mlp_tc = false, mlp_ffma = false;
  if (mlp) {
    std::string why;
    mlp_tc = uml::mlp_tc_supported(mlp->dm, &why);
    if (mlp_tc) {
      const char* env = getenv("UML_B200_MLP_TC");
      if (env && env[0] == '0') mlp_tc = false;
      else if (!(env && env[0] == '1')) mlp_tc = host_sample_is_tf32(host_ptr, L, n_rows, F, src_dtype);
    }
    mlp_ffma = !mlp_tc && uml::mlp_tma_supported(mlp->dm, &why);
  }

  const bool timed = stats != nullptr;
  cudaStream_t cs = e->stream;
  // errors inside the pipeline: both streams must be idle before returning - async copies still reference the
  // caller's host_ptr / labels_out
#define HOST_CUDA(CALL)                                                          \
  do {                                                                           \
    cudaError_t _e3 = (CALL);                                                    \
    if (_e3 != cudaSuccess) {                                                    \
      cudaStreamSynchronize(cs);                                                 \
      cudaStreamSynchronize(e->copy_stream);                                     \
      UML_FAIL(e, _e3 == cudaErrorMemoryAllocation ? UML_ERR_NOMEM : UML_ERR_CUDA, "%s failed: %s", #CALL, \
               cudaGetErrorString(_e3));                                         \
    }                                                                            \
  } while (0)
  if (timed) HOST_CUDA(cudaEventRecord(e->ev[0], cs));
  HOST_CUDA(cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), cs));
  HOST_CUDA(cudaMemsetAsync(e->d_flag_count, 0, sizeof(int), cs));
  HOST_CUDA(cudaMemsetAsync(e->d_stage, 0, sizeof(StageResult), cs));
  if (values_out) HOST_CUDA(cudaMemcpyAsync(e->d_classes, classes, (size_t)n_classes * 8, cudaMemcpyHostToDevice, cs));
  HOST_CUDA(cudaEventRecord(e->chunk_ev[6], cs));
  HOST_CUDA(cudaStreamWaitEvent(e->copy_stream, e->chunk_ev[6], 0));
  int launches = 0, path = 0;
  int64_t h2d = 0, d2h = 0;
  bool used[3] = {false, false, false};
  int slot = 0;
  std::vector<CopyPool::Task> tasks;
  bool wire_f32 = bounce && !direct && src_dtype == UML_F64 && (L.feature_major || L.pitch_elems == F) &&
                  !getenv("UML_B200_NO_NARROW");
  // UML_B200_PROFILE_HOST=1: host-side seconds per phase of this call on stderr (diagnostics, not a product feature)
  static const bool prof = getenv("UML_B200_PROFILE_HOST") != nullptr;
  double t_wait = 0, t_gather = 0, t_enqueue = 0;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };
  // ... and, for the first chunks, a device timeline from CUDA events on both streams (H2D / convert+score+D2H), which
  // is what shows the overlap of the pipeline without nsys
  constexpr int kTl = 12;
  cudaEvent_t tl[kTl][4] = {};
  int tl_n = 0;
  if (prof)
    for (auto& row : tl)
      for (auto& ev : row) cudaEventCreate(&ev);
  for (int64_t r0 = 0; r0 < n_rows; r0 += chunk_rows, slot = (slot + 1) % 3) {
    const int64_t rows = std::min(chunk_rows, n_rows - r0);
    float* xc = e->d_xchunk[slot];
    void* raw = direct ? (void*)xc : e->d_chunk[slot];
    const int tli = (prof && tl_n < kTl) ? tl_n++ : -1;
    bool chunk_narrow = false;  // this chunk crossed PCIe as fp32 (lossless float64 source)
    // (1) H2D on the copy stream, once the previous user of this slot has finished scoring (the re-score reads the
    //     raw chunk, so that includes it)
    if (used[slot]) HOST_CUDA(cudaStreamWaitEvent(e->copy_stream, e->chunk_ev[3 + slot], 0));
    if (result_bounce) HOST_CUDA(flush_slot(slot));
    if (tli >= 0) cudaEventRecord(tl[tli][0], e->copy_stream);
    {
      NvtxRange r_h2d("uml:h2d");
      if (bounce) {
        auto t0 = now();
        if (used[slot]) HOST_CUDA(cudaEventSynchronize(e->chunk_ev[slot]));  // the slot's previous H2D has left the bounce buffer
        auto t1 = now();
        t_wait += secs(t0, t1);
        if (direct) {  // already the resident layout (padding included): one contiguous run
          tasks.clear();
          const char* src0 = (const char*)host_ptr + (size_t)r0 * ld * 4;
          const size_t total = (size_t)rows * ld * 4, piece = 1u << 20;
          for (size_t o = 0; o < total; o += piece)
            tasks.push_back({(char*)e->h_bounce[slot] + o, src0 + o, std::min(piece, total - o)});
        }
        auto t2 = now();
        if (direct) {
          e->pool->run(tasks);
        } else {
          // float64 frames whose values are exactly representable in fp32 (integer / pixel domains) cross PCIe as fp32:
          // the gather threads convert while they copy and check every value; the first chunk that is not lossless
          // (and every chunk after it) travels as float64, as before
          chunk_narrow = wire_f32;
          if (chunk_narrow) {
            std::atomic<int> lossy{0};
            build_gather_tasks(tasks, (char*)e->h_bounce[slot], host_ptr, L, r0, rows, F, &lossy);
            e->pool->run(tasks);
            if (lossy.load()) {
              wire_f32 = false;
              chunk_narrow = false;
            }
          }
          if (!chunk_narrow) {
            build_gather_tasks(tasks, (char*)e->h_bounce[slot], host_ptr, L, r0, rows, F);
            e->pool->run(tasks);
          }
        }
        auto t3 = now();
        t_gather += secs(t2, t3);
        HOST_CUDA(cudaMemcpyAsync(raw, e->h_bounce[slot], (size_t)(rows * (chunk_narrow ? wire_row_bytes / 2 : wire_row_bytes)),
                                  cudaMemcpyHostToDevice, e->copy_stream));
        t_enqueue += secs(t3, now());
      } else if (direct) {
        HOST_CUDA(cudaMemcpyAsync(xc, (const char*)host_ptr + (size_t)r0 * ld * 4, (size_t)rows * ld * 4,
                                  cudaMemcpyHostToDevice, e->copy_stream));
      } else {
        HOST_CUDA(copy_chunk_h2d(raw, host_ptr, L, r0, rows, F, e->copy_stream));
      }
    }
    h2d += rows * (chunk_narrow ? wire_row_bytes / 2 : wire_row_bytes);
    if (tli >= 0) cudaEventRecord(tl[tli][1], e->copy_stream);
    HOST_CUDA(cudaEventRecord(e->chunk_ev[slot], e->copy_stream));
    HOST_CUDA(cudaStreamWaitEvent(cs, e->chunk_ev[slot], 0));
    if (tli >= 0) cudaEventRecord(tl[tli][2], cs);
    // (2) transpose / down-cast (+ finiteness) on the compute stream
    if (!direct) {
      NvtxRange r_stage("uml:stage_convert");
      HOST_CUDA(uml::launch_stage_convert(raw, chunk_narrow ? (int)UML_F32 : src_dtype, L.feature_major,
                                          L.feature_major ? rows : F, rows, F, xc, ld, nullptr, 0, e->d_stage, true, cs));
      launches += 1;
    } else if (!exact) {
      HOST_CUDA(uml::launch_finite_scan(xc, ld, rows, F, e->d_stage, cs));
      launches += 1;
    }
    // (3) score
    CUtensorMap map;
    bool has_map = encode_map(e, &map, xc, rows, F, ld) == UML_OK;
    LinearLaunch l{};
    l.x = xc;
    l.ld = ld;
    l.n_rows = rows;
    l.labels = e->d_labels + (int64_t)slot * chunk_rows;
    if (!mlp && exact && !direct && !chunk_narrow && lossy_capable(src_dtype)) {  // (the reference MLP predictor casts to
      // float32; a chunk that travelled as fp32 was checked lossless on the host: its fp32 rows ARE the caller's values)
      // flagged rows are re-scored from the caller's own values (the raw chunk is still resident): float64 / int
      // features that do not survive the fp32 down-cast still get sklearn's float64 labels (_base.py:366-396)
      l.src.base = raw;
      l.src.dtype = src_dtype;
      l.src.row_stride = L.feature_major ? 1 : F;
      l.src.col_stride = L.feature_major ? rows : 1;
    }
    if (mlp) {
      uml::MlpTcLaunch out{};
      out.n_rows = rows;
      out.labels = l.labels;
      out.x = xc;
      out.ld = ld;
      FlagList fl{e->d_flag_count, e->d_flag_rows, (int)std::min<int64_t>(e->flag_cap, INT32_MAX), e->d_counters};
      if (mlp_tc && has_map) {
        bool need_rescore = false;
        HOST_CUDA(uml::launch_mlp_tc(map, mlp->dm, out, exact, fl, e->info.sm_count, cs, &need_rescore));
        launches += 1;
        path = 5;
        if (need_rescore) {
          HOST_CUDA(uml::launch_mlp_rescore_f64(mlp->dm, xc, ld, rows, out, fl, false, e->info.sm_count, cs));
          launches += 1;
        }
      } else if (mlp_ffma && has_map) {
        HOST_CUDA(uml::launch_mlp_tma(map, mlp->dm, xc, rows, out.labels, exact, fl, e->info.sm_count, cs));
        launches += 1;
        path = 3;
        if (exact) {
          HOST_CUDA(uml::launch_mlp_rescore_f64(mlp->dm, xc, ld, rows, out, fl, false, e->info.sm_count, cs));
          launches += 1;
        }
      } else {
        HOST_CUDA(uml::launch_mlp_rescore_f64(mlp->dm, xc, ld, rows, out, fl, true, e->info.sm_count, cs));
        launches += 1;
        path = 2;
      }
      rc = UML_OK;
    } else {
      rc = enqueue_predict(e, m, l, has_map ? &map : nullptr, mode, false, &launches, &path);
    }
    if (rc != UML_OK) {
      cudaStreamSynchronize(cs);
      cudaStreamSynchronize(e->copy_stream);
      return rc;
    }
    // (4) labels (or class values) back
    char* land = result_bounce ? (char*)e->h_result[slot] : nullptr;
    if (values_out) {
      HOST_CUDA(uml::launch_labels_take(l.labels, 4, rows, e->d_classes, n_classes, e->d_vchunk[slot], cs));
      launches += 1;
      HOST_CUDA(cudaMemcpyAsync(land ? (void*)land : (void*)(values_out + r0), e->d_vchunk[slot], (size_t)rows * 8,
                                cudaMemcpyDeviceToHost, cs));
      d2h += rows * 8;
    }
    if (labels_out) {
      HOST_CUDA(cudaMemcpyAsync(land ? (void*)(land + (size_t)chunk_rows * 8) : (void*)(labels_out + r0), l.labels,
                                (size_t)rows * 4, cudaMemcpyDeviceToHost, cs));
      d2h += rows * 4;
    }
    if (result_bounce) {
      pending[slot].r0 = r0;
      pending[slot].rows = rows;
      pending[slot].live = true;
    }
    if (tli >= 0) cudaEventRecord(tl[tli][3], cs);
    HOST_CUDA(cudaEventRecord(e->chunk_ev[3 + slot], cs));
    used[slot] = true;
  }
  HOST_CUDA(cudaMemcpyAsync(&e->h->stage, e->d_stage, sizeof(StageResult), cudaMemcpyDeviceToHost, cs));
#undef HOST_CUDA
  if (prof && tl_n > 0) {
    cudaStreamSynchronize(cs);
    cudaStreamSynchronize(e->copy_stream);
    fprintf(stderr, "uml predict_host timeline (ms since the first H2D began; chunk: h2d [begin,end]  convert+score+d2h [begin,end])\n");
    for (int i = 0; i < tl_n; ++i) {
      float a = 0, b2 = 0, c = 0, d = 0;
      cudaEventElapsedTime(&a, tl[0][0], tl[i][0]);
      cudaEventElapsedTime(&b2, tl[0][0], tl[i][1]);
      cudaEventElapsedTime(&c, tl[0][0], tl[i][2]);
      cudaEventElapsedTime(&d, tl[0][0], tl[i][3]);
      fprintf(stderr, "  chunk %2d: h2d [%7.3f, %7.3f]  compute [%7.3f, %7.3f]\n", i, a, b2, c, d);
    }
    (void)cudaGetLastError();
  }
  if (prof)
    for (auto& row : tl)
      for (auto& ev : row)
        if (ev) cudaEventDestroy(ev);
  if (prof)
    fprintf(stderr, "uml predict_host: rows %lld chunk_rows %lld bounce %d direct %d | wait-for-slot %.4f s, gather %.4f s, "
                    "memcpyAsync enqueue %.4f s\n", (long long)n_rows, (long long)chunk_rows, (int)bounce, (int)direct, t_wait,
            t_gather, t_enqueue);
  rc = finish_stats(e, stats, n_rows, launches, path, timed, false);
  cudaStreamSynchronize(e->copy_stream);
  for (int sl = 0; sl < 3; ++sl)
    if (flush_slot(sl) != cudaSuccess && rc == UML_OK) rc = UML_ERR_CUDA;
  if (stats) {
    stats->h2d_bytes = h2d;
    stats->d2h_bytes = d2h;
  }
  // NaN/Inf in the caller's values (the staging kernel checks the source dtype, so a finite float64 that overflows
  // fp32 is not an error here - exact mode re-scores such rows from the float64 source)
  if (rc == UML_OK && e->h->stage.nonfinite) UML_FAIL(e, UML_ERR_NONFINITE, "Input X contains NaN or infinity.");
  return rc;
}

int uml_linear_predict_host(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows, int n_features,
                            int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out,
                            int mode, int64_t chunk_rows, uml_stats* stats) {
  if (!labels_out && n_rows > 0) return UML_ERR_INVALID;
  return predict_host_impl(e, m, host_ptr, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype, labels_out,
                           nullptr, nullptr, 0, mode, chunk_rows, stats);
}

int uml_linear_predict_host_values(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows,
                                   int n_features, int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype,
                                   const double* classes_host, int n_classes, double* values_out, int mode,
                                   int64_t chunk_rows, uml_stats* stats) {
  if ((!values_out && n_rows > 0) || !classes_host || n_classes < 1) return UML_ERR_INVALID;
  if (m && n_classes < m->dm.n_classes) UML_FAIL(e, UML_ERR_INVALID, "classes_ has %d entries, the model scores %d classes", n_classes, m->dm.n_classes);
  return predict_host_impl(e, m, host_ptr, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype, nullptr,
                           values_out, classes_host, n_classes, mode, chunk_rows, stats);
}

// asynchronous variant: the whole pipeline runs on a library thread so that the caller (Python building the
// List[float] of the predictor contract) can consume labels_out[0, rows_done) while the rest of the batch is still
// crossing PCIe.  One call in flight per engine; no other call on the engine until _finish.
static int async_begin(uml_engine* e, const uml_model* m, const uml_mlp* mlp, const void* host_ptr, int64_t n_rows,
                       int n_features, int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype,
                       int32_t* labels_out, int mode, int64_t chunk_rows) {
  if (!e || (!m && !mlp) || (!labels_out && n_rows > 0)) return UML_ERR_INVALID;
  if (!e->async_finished.load() || e->async_thread.joinable())
    UML_FAIL(e, UML_ERR_INVALID, "an asynchronous call is already in flight on this engine (call uml_async_finish first)");
  e->async_rows_done.store(0);
  e->async_finished.store(0);
  e->async_status = UML_OK;
  memset(&e->async_stats, 0, sizeof(e->async_stats));
  e->async_thread = std::thread([=]() {
    e->async_status = predict_host_impl(e, m, host_ptr, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype,
                                        labels_out, nullptr, nullptr, 0, mode, chunk_rows, &e->async_stats,
                                        &e->async_rows_done, mlp);
    e->async_finished.store(1, std::memory_order_release);
  });
  return UML_OK;
}

int uml_linear_predict_host_begin(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows, int n_features,
                                  int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out,
                                  int mode, int64_t chunk_rows) {
  if (!m) return UML_ERR_INVALID;
  return async_begin(e, m, nullptr, host_ptr, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype, labels_out,
                     mode, chunk_rows);
}

// the MLP predictor through the same chunk pipeline: labels_out[i] = argmax class index of row i, i.e. what
// `module(features).argmax(1)` yields (tests/integration/pytorch_app/quickstart.py:68-70)
int uml_mlp_predict_host(uml_engine* e, const uml_mlp* m, const void* host_ptr, int64_t n_rows, int n_features,
                         int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out, int mode,
                         int64_t chunk_rows, uml_stats* stats) {
  if (!e || !m || (!labels_out && n_rows > 0)) return UML_ERR_INVALID;
  return predict_host_impl(e, nullptr, host_ptr, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype,
                           labels_out, nullptr, nullptr, 0, mode, chunk_rows, stats, nullptr, m);
}

int uml_mlp_predict_host_begin(uml_engine* e, const uml_mlp* m, const void* host_ptr, int64_t n_rows, int n_features,
                               int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out,
                               int mode, int64_t chunk_rows) {
  if (!m) return UML_ERR_INVALID;
  return async_begin(e, nullptr, m, host_ptr, n_rows, n_features, row_stride_bytes, col_stride_bytes, src_dtype, labels_out,
                     mode, chunk_rows);
}

int uml_async_poll(uml_engine* e, int64_t* rows_done, int* finished) {
  if (!e) return UML_ERR_INVALID;
  const int fin = e->async_finished.load(std::memory_order_acquire);  // read first: rows_done is final once it is set
  if (rows_done) *rows_done = e->async_rows_done.load(std::memory_order_acquire);
  if (finished) *finished = fin;
  return UML_OK;
}

int uml_async_finish(uml_engine* e, uml_stats* stats) {
  if (!e) return UML_ERR_INVALID;
  if (e->async_thread.joinable()) e->async_thread.join();
  if (stats) *stats = e->async_stats;
  return e->async_status;
}

int uml_linear_predict_proba(uml_engine* e, const uml_model* m, const uml_batch* b, float* proba_out, int proba_on_device) {
  if (!e || !m || !b || (!proba_out && b->n_rows > 0)) return UML_ERR_INVALID;
  if (b->n_features != m->n_features_in)
    UML_FAIL(e, UML_ERR_SHAPE, "X has %d features, but the estimator is expecting %d features as input.",
             b->n_features, m->n_features_in);
  UML_CUDA(e, cudaSetDevice(e->device));
  (void)cudaGetLastError();
  if (b->n_rows == 0) return UML_OK;
  NvtxRange r_all("uml:predict_proba");
  const int C = m->dm.n_classes;
  float* d_out = proba_out;
  if (!proba_on_device) UML_CUDA(e, cudaMalloc((void**)&d_out, (size_t)b->n_rows * C * 4));
  cudaError_t ce = uml::launch_linear_proba(m->dm, b->x, b->ld, b->n_rows, d_out, e->info.sm_count, e->stream);
  if (ce == cudaSuccess && !proba_on_device) {
    ce = cudaMemcpyAsync(proba_out, d_out, (size_t)b->n_rows * C * 4, cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
  }
  if (!proba_on_device) {
    cudaStreamSynchronize(e->stream);
    cudaFree(d_out);
  }
  if (ce != cudaSuccess) UML_FAIL(e, UML_ERR_CUDA, "uml_linear_predict_proba: %s", cudaGetErrorString(ce));
  return UML_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// MLP: PytorchModel(in, hidden, out) of tests/integration/pytorch_app/quickstart.py
// ---------------------------------------------------------------------------------------------------------------
int uml_mlp_load(uml_engine* e, uml_mlp** out, const float* w1, const float* b1, const float* w2, const float* b2,
                 int n_in, int n_hidden, int n_out) {
  if (!e || !out || !w1 || !b1 || !w2 || !b2) return UML_ERR_INVALID;
  *out = nullptr;
  if (n_in < 1 || n_hidden < 1 || n_out < 2 || n_hidden > 256)
    UML_FAIL(e, UML_ERR_UNSUPPORTED, "MLP shape %d -> %d -> %d (need hidden <= 256, out >= 2)", n_in, n_hidden, n_out);
  {  // the fp64 re-score kernel keeps W1, W2 and eight row strips in shared memory
    const size_t need = ((size_t)n_in * n_hidden + (size_t)n_out * (n_hidden + 1) + 2 * (size_t)n_hidden + n_out + n_in +
                         8 * ((size_t)n_in + n_hidden)) * 8;
    if (need > (size_t)uml::kMaxSmemBytes)
      UML_FAIL(e, UML_ERR_UNSUPPORTED, "MLP shape %d -> %d -> %d: fp64 weights (%zu B) exceed the shared memory of one SM", n_in,
               n_hidden, n_out, need);
  }
  UML_CUDA(e, cudaSetDevice(e->device));
  const int F = n_in, H = n_hidden, C = n_out;
  const int HP = H + 4, cp = (C + 1 + 3) / 4 * 4;
  const int f_pad = (F + uml::kChunkF - 1) / uml::kChunkF * uml::kChunkF;
  std::vector<float> w1t((size_t)f_pad * HP, 0.f), b1p(HP, 0.f), w2t((size_t)H * cp, 0.f), b2p(cp, 0.f);
  for (int f = 0; f < F; ++f) {
    float wmax = 0.f;
    for (int n = 0; n < H; ++n) {
      const float v = w1[(size_t)n * F + f];  // torch Linear weight: (out, in)
      w1t[(size_t)f * HP + n] = v;
      wmax = fmaxf(wmax, fabsf(v));
    }
    w1t[(size_t)f * HP + H] = wmax;
  }
  float bmax = 0.f;
  for (int n = 0; n < H; ++n) {
    b1p[n] = b1[n];
    bmax = fmaxf(bmax, fabsf(b1[n]));
  }
  b1p[H] = bmax;
  double row_sum_max = 0.0;
  for (int c = 0; c < C; ++c) {
    double rs = 0.0;
    for (int n = 0; n < H; ++n) rs += fabs((double)w2[(size_t)c * H + n]);
    row_sum_max = std::max(row_sum_max, rs);
  }
  for (int n = 0; n < H; ++n) {
    float wmax = 0.f;
    for (int c = 0; c < C; ++c) {
      const float v = w2[(size_t)c * H + n];
      w2t[(size_t)n * cp + c] = v;
      wmax = fmaxf(wmax, fabsf(v));
    }
    w2t[(size_t)n * cp + C] = wmax;
  }
  bmax = 0.f;
  for (int c = 0; c < C; ++c) {
    b2p[c] = b2[c];
    bmax = fmaxf(bmax, fabsf(b2[c]));
  }
  b2p[C] = bmax;
  // fp64 operands of the re-score, laid out as the kernels keep them in shared memory
  const std::vector<double> w64 = uml::mlp_rs_build_pack(w1, b1, w2, b2, F, H, C);

  uml_mlp* m = new uml_mlp();
  m->e = e;
  m->host.w1.assign(w1, w1 + (size_t)H * F);
  m->host.b1.assign(b1, b1 + H);
  m->host.w2.assign(w2, w2 + (size_t)C * H);
  m->host.b2.assign(b2, b2 + C);
  std::vector<float> tiles;
  if (f_pad <= 128 && (H == 16 || H == 32)) tiles = uml::mlp_tc_build_w1_tiles(w1, H, F, f_pad);
  auto up = [&](void** dst, const void* src, size_t bytes) -> cudaError_t {
    cudaError_t ce = cudaMalloc(dst, bytes);
    if (ce != cudaSuccess) return ce;
    return cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
  };
  cudaError_t ce;
  if ((ce = up((void**)&m->d_w1t, w1t.data(), w1t.size() * 4)) != cudaSuccess ||
      (ce = up((void**)&m->d_b1, b1p.data(), b1p.size() * 4)) != cudaSuccess ||
      (ce = up((void**)&m->d_w2t, w2t.data(), w2t.size() * 4)) != cudaSuccess ||
      (ce = up((void**)&m->d_b2, b2p.data(), b2p.size() * 4)) != cudaSuccess ||
      (ce = up((void**)&m->d_w64, w64.data(), w64.size() * 8)) != cudaSuccess ||
      (!tiles.empty() && (ce = up((void**)&m->d_w1_tiles, tiles.data(), tiles.size() * 4)) != cudaSuccess)) {
    e->last_error = std::string("uml_mlp_load: ") + cudaGetErrorString(ce);
    uml_mlp_free(m);
    return ce == cudaErrorMemoryAllocation ? UML_ERR_NOMEM : UML_ERR_CUDA;
  }
  m->dm.w1t = m->d_w1t;
  m->dm.b1 = m->d_b1;
  m->dm.w2t = m->d_w2t;
  m->dm.b2 = m->d_b2;
  m->dm.rs_pack = m->d_w64;
  m->dm.n_in = F;
  m->dm.n_hidden = H;
  m->dm.n_classes = C;
  m->dm.cp = cp;
  m->dm.f_pad = f_pad;
  m->dm.w2_abs_row_sum_max = row_sum_max;
  m->dm.w1_tiles = m->d_w1_tiles;
  m->dm.host = &m->host;
  *out = m;
  return UML_OK;
}

void uml_mlp_free(uml_mlp* m) {
  if (!m) return;
  if (m->e) cudaSetDevice(m->e->device);
  cudaFree(m->d_w1t);
  cudaFree(m->d_b1);
  cudaFree(m->d_w2t);
  cudaFree(m->d_b2);
  cudaFree(m->d_w64);
  cudaFree(m->d_w1_tiles);
  delete m;
}

// is every fp32 feature of the batch a tf32 value?  Known from staging; wrapped device rows are scanned once (one
// HBM pass, cached in the batch handle - the handle is logically const for the caller)
static int batch_tf32_exact(uml_engine* e, const uml_batch* b) {
  if (b->tf32_exact >= 0) return b->tf32_exact;
  cudaError_t ce;
  if ((ce = cudaMemsetAsync(e->d_stage, 0, sizeof(StageResult), e->stream)) != cudaSuccess ||
      (ce = uml::launch_finite_scan(b->x, b->ld, b->n_rows, b->n_features, e->d_stage, e->stream)) != cudaSuccess ||
      (ce = cudaMemcpyAsync(&e->h->stage, e->d_stage, sizeof(StageResult), cudaMemcpyDeviceToHost, e->stream)) != cudaSuccess ||
      (ce = cudaStreamSynchronize(e->stream)) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  const_cast<uml_batch*>(b)->tf32_exact = e->h->stage.not_tf32 == 0 ? 1 : 0;
  return b->tf32_exact;
}

static int mlp_predict_common(uml_engine* e, const uml_mlp* m, const uml_batch* b, int32_t* labels_out,
                              int labels_on_device, void* const* peers, int n_peers, int64_t row_offset,
                              int label_bytes, int mode, uml_stats* stats) {
  if (!e || !m || !b) return UML_ERR_INVALID;
  if (!labels_out && b->n_rows > 0 && n_peers == 0) return UML_ERR_INVALID;
  if (mode != UML_PREDICT_FAST && mode != UML_PREDICT_EXACT) UML_FAIL(e, UML_ERR_INVALID, "mode %d", mode);
  if (n_peers < 0 || n_peers > 8) UML_FAIL(e, UML_ERR_INVALID, "n_peers %d (max 8)", n_peers);
  if (n_peers > 0 && label_bytes != 1 && label_bytes != 4) UML_FAIL(e, UML_ERR_INVALID, "label_bytes %d", label_bytes);
  if (n_peers > 0 && label_bytes == 1 && m->dm.n_classes > 256)
    UML_FAIL(e, UML_ERR_UNSUPPORTED, "byte labels need n_classes <= 256 (model has %d)", m->dm.n_classes);
  if (b->n_features != m->dm.n_in)
    UML_FAIL(e, UML_ERR_SHAPE, "X has %d features, but the module is expecting %d features as input.", b->n_features,
             m->dm.n_in);
  UML_CUDA(e, cudaSetDevice(e->device));
  (void)cudaGetLastError();
  if (stats) memset(stats, 0, sizeof(*stats));
  if (b->n_rows == 0) return UML_OK;
  const bool exact = mode == UML_PREDICT_EXACT;
  const bool timed = stats != nullptr;
  const bool sync_call = stats || (!labels_on_device && labels_out);
  int rc;
  if (exact && (rc = ensure_flags(e, b->n_rows)) != UML_OK) return rc;

  // kernel choice: tensor cores when every feature is a tf32 value (integer / pixel domains), CUDA cores otherwise.
  // UML_B200_MLP_TC=0 / 1 forces the choice (1: rows that are not tf32-exact are caught in the kernel and re-scored)
  std::string why;
  bool use_tc = b->has_map && uml::mlp_tc_supported(m->dm, &why);
  if (use_tc) {
    const char* env = getenv("UML_B200_MLP_TC");
    if (env && env[0] == '0') use_tc = false;
    else if (!(env && env[0] == '1')) use_tc = batch_tf32_exact(e, b) == 1;
  }
  const bool use_ffma = !use_tc && b->has_map && uml::mlp_tma_supported(m->dm, &why);

  uml::MlpTcLaunch out{};
  out.n_rows = b->n_rows;
  out.row_offset = row_offset;
  out.x = b->x;
  out.ld = b->ld;
  const bool wire_u8 = n_peers > 0 && label_bytes == 1;
  out.wire_u8 = wire_u8 ? 1 : 0;
  int32_t* d_labels = labels_out;
  if (n_peers > 0) {
    out.n_peers = n_peers;
    for (int i = 0; i < n_peers; ++i) out.peers[i] = peers[i];
    d_labels = nullptr;
  } else if (!labels_on_device) {
    if ((rc = ensure_labels(e, b->n_rows)) != UML_OK) return rc;
    d_labels = e->d_labels;
  }
  out.labels = d_labels;
  // the CUDA-core kernel has no peer stores: it writes int32 labels to scratch and a thin kernel scatters them
  uml::MlpTcLaunch ffma_out = out;
  if (use_ffma && n_peers > 0) {
    if ((rc = ensure_labels(e, b->n_rows)) != UML_OK) return rc;
    ffma_out.labels = e->d_labels;
  }

  FlagList fl{e->d_flag_count, e->d_flag_rows, (int)std::min<int64_t>(e->flag_cap, INT32_MAX), e->d_counters};
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[0], e->stream));
  if (sync_call) {
    UML_CUDA(e, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), e->stream));
    UML_CUDA(e, cudaMemsetAsync(e->d_flag_count, 0, sizeof(int), e->stream));
  }
  int launches = 0, path = 3;
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[1], e->stream));
  if (use_tc) {
    NvtxRange r_score("uml:mlp_score_tcgen05");
    bool need_rescore = false;
    UML_CUDA(e, uml::launch_mlp_tc(b->map, m->dm, out, exact, fl, e->info.sm_count, e->stream, &need_rescore));
    launches += 1;
    path = 5;
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
    if (need_rescore) {  // UML_B200_MLP_RESCORE_MODE=kernel; in queue mode four warps of the scoring kernel do it
      NvtxRange r_rescore("uml:mlp_rescore_f64");
      UML_CUDA(e, uml::launch_mlp_rescore_f64(m->dm, b->x, b->ld, b->n_rows, out, fl, false, e->info.sm_count, e->stream));
      launches += 1;
    }
  } else if (use_ffma) {
    NvtxRange r_score("uml:mlp_score_ffma");
    UML_CUDA(e, uml::launch_mlp_tma(b->map, m->dm, b->x, b->n_rows, ffma_out.labels, exact, fl, e->info.sm_count, e->stream));
    launches += 1;
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
    if (exact) {
      UML_CUDA(e, uml::launch_mlp_rescore_f64(m->dm, b->x, b->ld, b->n_rows, ffma_out, fl, false, e->info.sm_count, e->stream));
      launches += 1;
    }
    if (n_peers > 0) {
      UML_CUDA(e, uml::launch_labels_scatter(e->d_labels, b->n_rows, out.peers, n_peers, out.wire_u8, row_offset,
                                             e->info.sm_count, e->stream));
      launches += 1;
    }
  } else {
    NvtxRange r_score("uml:mlp_score_f64_generic");
    UML_CUDA(e, uml::launch_mlp_rescore_f64(m->dm, b->x, b->ld, b->n_rows, out, fl, true, e->info.sm_count, e->stream));
    launches += 1;
    path = 2;
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
  }
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[3], e->stream));
  int64_t d2h = 0;
  if (!labels_on_device && labels_out) {
    UML_CUDA(e, cudaMemcpyAsync(labels_out, d_labels, (size_t)b->n_rows * 4, cudaMemcpyDeviceToHost, e->stream));
    d2h = b->n_rows * 4;
  }
  if (sync_call) {
    rc = finish_stats(e, stats, b->n_rows, launches, path, timed);
    if (stats) stats->d2h_bytes = d2h;
    return rc;
  }
  return UML_OK;
}

int uml_mlp_predict(uml_engine* e, const uml_mlp* m, const uml_batch* b, int32_t* labels_out, int labels_on_device,
                    int mode, uml_stats* stats) {
  if (b && !labels_out && b->n_rows > 0) return UML_ERR_INVALID;
  return mlp_predict_common(e, m, b, labels_out, labels_on_device, nullptr, 0, 0, 4, mode, stats);
}

int uml_mlp_predict_peers(uml_engine* e, const uml_mlp* m, const uml_batch* b, void* const* peer_labels, int n_peers,
                          int64_t row_offset, int label_bytes, int mode, uml_stats* stats) {
  if (!peer_labels || n_peers < 1) return UML_ERR_INVALID;
  return mlp_predict_common(e, m, b, nullptr, 1, peer_labels, n_peers, row_offset, label_bytes, mode, stats);
}

// class probabilities of the MLP (PytorchModel.forward): the kernel choice of mlp_predict_common, each tile kernel with
// its softmax epilogue, and the fp64 kernel behind it for the rows it flags (features that are not tf32 values on the
// tensor-core path, NaN/Inf anywhere).  Always synchronous: a non-finite row is an error the caller must see.
int uml_mlp_predict_proba(uml_engine* e, const uml_mlp* m, const uml_batch* b, float* proba_out, int proba_on_device,
                          uml_stats* stats) {
  if (!e || !m || !b || (!proba_out && b->n_rows > 0)) return UML_ERR_INVALID;
  if (b->n_features != m->dm.n_in)
    UML_FAIL(e, UML_ERR_SHAPE, "X has %d features, but the module is expecting %d features as input.", b->n_features,
             m->dm.n_in);
  if (proba_on_device && (reinterpret_cast<uintptr_t>(proba_out) & 15u))
    UML_FAIL(e, UML_ERR_UNSUPPORTED, "uml_mlp_predict_proba: device proba_out %p is not 16-byte aligned", (void*)proba_out);
  UML_CUDA(e, cudaSetDevice(e->device));
  (void)cudaGetLastError();
  if (stats) memset(stats, 0, sizeof(*stats));
  if (b->n_rows == 0) return UML_OK;
  const bool timed = stats != nullptr;
  int rc;
  if ((rc = ensure_flags(e, b->n_rows)) != UML_OK) return rc;

  std::string why;  // same choice as mlp_predict_common (UML_B200_MLP_TC=0 / 1 forces it)
  bool use_tc = b->has_map && uml::mlp_tc_supported(m->dm, &why);
  if (use_tc) {
    const char* env = getenv("UML_B200_MLP_TC");
    if (env && env[0] == '0') use_tc = false;
    else if (!(env && env[0] == '1')) use_tc = batch_tf32_exact(e, b) == 1;
  }
  const bool use_ffma = !use_tc && b->has_map && uml::mlp_tma_supported(m->dm, &why);

  NvtxRange r_all("uml:mlp_predict_proba");
  const size_t bytes = (size_t)b->n_rows * m->dm.n_classes * 4;
  struct Scratch {  // device landing buffer of a host-output call
    float* p = nullptr;
    ~Scratch() { cudaFree(p); }
  } scratch;
  float* d_out = proba_out;
  if (!proba_on_device) {
    UML_CUDA(e, cudaMalloc((void**)&scratch.p, bytes));
    d_out = scratch.p;
  }
  FlagList fl{e->d_flag_count, e->d_flag_rows, (int)std::min<int64_t>(e->flag_cap, INT32_MAX), e->d_counters};
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[0], e->stream));
  UML_CUDA(e, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), e->stream));
  UML_CUDA(e, cudaMemsetAsync(e->d_flag_count, 0, sizeof(int), e->stream));
  int launches = 0, path = 2;
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[1], e->stream));
  if (use_tc || use_ffma) {
    if (use_tc) {
      NvtxRange r_score("uml:mlp_proba_tcgen05");
      uml::MlpTcLaunch out{};
      out.n_rows = b->n_rows;
      out.x = b->x;
      out.ld = b->ld;
      UML_CUDA(e, uml::launch_mlp_tc_proba(b->map, m->dm, out, d_out, fl, e->info.sm_count, e->stream));
      path = 5;
    } else {
      NvtxRange r_score("uml:mlp_proba_ffma");
      UML_CUDA(e, uml::launch_mlp_tma(b->map, m->dm, b->x, b->n_rows, nullptr, false, fl, e->info.sm_count, e->stream, d_out));
      path = 3;
    }
    launches += 1;
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
    NvtxRange r_rescore("uml:mlp_proba_f64");
    UML_CUDA(e, uml::launch_mlp_proba_f64(m->dm, b->x, b->ld, b->n_rows, d_out, fl, false, e->info.sm_count, e->stream));
    launches += 1;
  } else {
    NvtxRange r_score("uml:mlp_proba_f64_generic");
    UML_CUDA(e, uml::launch_mlp_proba_f64(m->dm, b->x, b->ld, b->n_rows, d_out, fl, true, e->info.sm_count, e->stream));
    launches += 1;
    if (timed) UML_CUDA(e, cudaEventRecord(e->ev[2], e->stream));
  }
  if (timed) UML_CUDA(e, cudaEventRecord(e->ev[3], e->stream));
  int64_t d2h = 0;
  if (!proba_on_device) {
    UML_CUDA(e, cudaMemcpyAsync(proba_out, d_out, bytes, cudaMemcpyDeviceToHost, e->stream));
    d2h = (int64_t)bytes;
  }
  rc = finish_stats(e, stats, b->n_rows, launches, path, timed);
  if (stats) stats->d2h_bytes = d2h;
  return rc;
}

}  // extern "C"
