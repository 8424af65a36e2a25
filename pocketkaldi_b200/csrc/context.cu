// Context, error plumbing, batch metadata, timers and launch accounting of libpkb200.

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <memory>

#include "common.cuh"

namespace pkb {

namespace {
thread_local char g_error[1024] = "";
}

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

int DevBuf::ensure(size_t bytes) {
  if (bytes <= cap) return PKB_OK;
  if (p) {
    cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  // round up so that repeated, slightly growing requests do not reallocate
  size_t want = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    // the failure is returned here: clear it, or the next launch's error check reports it again
    cudaGetLastError();
    p = nullptr;
    set_error("cudaMalloc(%zu bytes): %s", want, cudaGetErrorString(e));
    return PKB_ERR_CUDA;
  }
  cap = want;
  // PKB_ALLOC_FILL=<byte>: debugging aid that makes reads of never-written device memory deterministic
  static const char *fill = getenv("PKB_ALLOC_FILL");
  if (fill != nullptr) cudaMemset(p, atoi(fill), want);
  return PKB_OK;
}

void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}

Ctx::~Ctx() {
  for (auto &s : spans) {
    cudaEventDestroy(s.e0);
    cudaEventDestroy(s.e1);
  }
  for (auto &e : free_events) cudaEventDestroy(e);
  if (err_host) cudaFreeHost(err_host);
  if (t0) cudaEventDestroy(t0);
  if (t1) cudaEventDestroy(t1);
  if (stream) cudaStreamDestroy(stream);
}

int upload(Ctx *c, void *dst, const void *src, size_t bytes) {
  if (bytes == 0) return PKB_OK;
  PKB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return PKB_OK;
}

int check_device_error(Ctx *c, const char *who) {
  if (c->err_host == nullptr) return PKB_OK;
  const int code = *static_cast<volatile int *>(c->err_host);
  if (code == 0) return PKB_OK;
  *c->err_host = 0;
  set_error("%s: a kernel gave up waiting for its peer CTAs (code %d: softmax exchange of the "
            "output layer); the results of this call are invalid", who, code);
  return PKB_ERR_CUDA;
}

LaunchScope::LaunchScope(Ctx *ctx, int cls) : c(ctx), timed(false) {
  span.cls = cls;
  c->launches[cls]++;
  if (!c->profile) return;
  cudaEvent_t ev[2];
  for (int i = 0; i < 2; ++i) {
    if (!c->free_events.empty()) {
      ev[i] = c->free_events.back();
      c->free_events.pop_back();
    } else if (cudaEventCreate(&ev[i]) != cudaSuccess) {
      return;
    }
  }
  span.e0 = ev[0];
  span.e1 = ev[1];
  cudaEventRecord(span.e0, c->stream);
  timed = true;
}

LaunchScope::~LaunchScope() {
  if (!timed) return;
  cudaEventRecord(span.e1, c->stream);
  c->spans.push_back(span);
}

// ---------------------------------------------------------------- batch metadata
static int finish_meta(BatchMeta *m) {
  const int n = m->n_utts;
  m->sample_off.assign(n + 1, 0);
  m->frame_off.assign(n + 1, 0);
  m->tile_prefix.assign(n + 1, 0);
  for (int u = 0; u < n; ++u) {
    m->sample_off[u + 1] = m->sample_off[u] + m->num_samples[u];
    m->frame_off[u + 1] = m->frame_off[u] + m->num_frames[u];
    int64_t tiles = (m->num_frames[u] + kFramesPerTile - 1) / kFramesPerTile;
    int64_t next = m->tile_prefix[u] + tiles;
    if (next > INT32_MAX) {
      set_error("batch too large: more than 2^31 fbank tiles");
      return PKB_ERR_INVALID;
    }
    m->tile_prefix[u + 1] = static_cast<int32_t>(next);
  }
  m->total_samples = m->sample_off[n];
  m->total_frames = m->frame_off[n];
  m->n_tiles = m->tile_prefix[n];
  m->tile_utt.resize(m->n_tiles);
  for (int u = 0; u < n; ++u)
    for (int32_t i = m->tile_prefix[u]; i < m->tile_prefix[u + 1]; ++i) m->tile_utt[i] = u;
  return PKB_OK;
}

int BatchMeta::build_from_samples(const int32_t *ns, int n) {
  PKB_REQUIRE(n >= 0, "n_utts must be >= 0");
  n_utts = n;
  num_samples.assign(ns, ns + n);
  num_frames.resize(n);
  for (int u = 0; u < n; ++u) {
    PKB_REQUIRE(ns[u] >= 0, "num_samples[%d] < 0", u);
    num_frames[u] = pkb_fbank_num_frames(ns[u]);
  }
  return finish_meta(this);
}

int BatchMeta::build_from_frames(const int32_t *nf, int n) {
  PKB_REQUIRE(n >= 0, "n_utts must be >= 0");
  n_utts = n;
  num_frames.assign(nf, nf + n);
  num_samples.assign(n, 0);
  for (int u = 0; u < n; ++u) PKB_REQUIRE(nf[u] >= 0, "num_frames[%d] < 0", u);
  return finish_meta(this);
}

int BatchMeta::upload(cudaStream_t stream) {
  const size_t n1 = static_cast<size_t>(n_utts) + 1;
  // layout: int64 sample_off[n1], int64 frame_off[n1], int32 num_samples[n1], num_frames[n1], tile_prefix[n1]
  const size_t bytes = n1 * (2 * sizeof(int64_t) + 3 * sizeof(int32_t)) + tile_utt.size() * sizeof(int32_t);
  std::vector<char> host(bytes);
  char *h = host.data();
  size_t o_so = 0, o_fo = o_so + n1 * 8, o_ns = o_fo + n1 * 8, o_nf = o_ns + n1 * 4,
         o_tp = o_nf + n1 * 4, o_tu = o_tp + n1 * 4;
  if (!tile_utt.empty()) memcpy(h + o_tu, tile_utt.data(), tile_utt.size() * 4);
  memcpy(h + o_so, sample_off.data(), n1 * 8);
  memcpy(h + o_fo, frame_off.data(), n1 * 8);
  if (n_utts) {
    memcpy(h + o_ns, num_samples.data(), n_utts * 4);
    memcpy(h + o_nf, num_frames.data(), n_utts * 4);
  }
  memcpy(h + o_tp, tile_prefix.data(), n1 * 4);
  PKB_TRY(dev.ensure(bytes));
  PKB_CUDA(cudaMemcpyAsync(dev.p, h, bytes, cudaMemcpyHostToDevice, stream));
  PKB_CUDA(cudaStreamSynchronize(stream));  // host staging vector goes out of scope
  char *d = dev.as<char>();
  d_sample_off = reinterpret_cast<const int64_t *>(d + o_so);
  d_frame_off = reinterpret_cast<const int64_t *>(d + o_fo);
  d_num_samples = reinterpret_cast<const int32_t *>(d + o_ns);
  d_num_frames = reinterpret_cast<const int32_t *>(d + o_nf);
  d_tile_prefix = reinterpret_cast<const int32_t *>(d + o_tp);
  d_tile_utt = reinterpret_cast<const int32_t *>(d + o_tu);
  return PKB_OK;
}

}  // namespace pkb

using pkb::Ctx;

extern "C" {

const char *pkb_last_error(void) { return pkb::g_error; }

const char *pkb_version(void) { return "pkb200 0.1 sm_100a"; }

int pkb_fbank_num_frames(int num_samples) {
  // Fbank::CalcNumFrames, src/fbank.cc:35-42
  if (num_samples < pkb::kFrame) return 0;
  return 1 + (num_samples - pkb::kFrame) / pkb::kShift;
}

int pkb_create(int device, pkb_ctx_t **out) {
  if (!out) {
    pkb::set_error("pkb_create: out pointer is NULL");
    return PKB_ERR_INVALID;
  }
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    pkb::set_error("pkb_create: no CUDA device (%s); libpkb200 has no CPU fallback",
                   e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return PKB_ERR_CUDA;
  }
  PKB_REQUIRE(device >= 0 && device < count, "pkb_create: device %d out of range [0,%d)", device,
              count);
  PKB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  PKB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    pkb::set_error("pkb_create: device %d is sm_%d%d; libpkb200 is built for sm_100a only", device,
                   prop.major, prop.minor);
    return PKB_ERR_CUDA;
  }
  std::unique_ptr<pkb_ctx, decltype(&pkb_destroy)> c(new pkb_ctx(), pkb_destroy);
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  snprintf(c->name, sizeof(c->name), "%s", prop.name);
  PKB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  PKB_CUDA(cudaEventCreate(&c->t0));
  PKB_CUDA(cudaEventCreate(&c->t1));
  PKB_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&c->err_host), sizeof(int), cudaHostAllocMapped));
  PKB_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void **>(&c->err_dev), c->err_host, 0));
  *c->err_host = 0;
  PKB_TRY(pkb::build_fbank_tables(c.get()));
  *out = c.release();
  return PKB_OK;
}

void pkb_destroy(pkb_ctx_t *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  delete c;
}

int pkb_sync(pkb_ctx_t *c) {
  PKB_REQUIRE(c, "pkb_sync: ctx is NULL");
  PKB_CUDA(cudaSetDevice(c->device));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_sync");
}

int pkb_fbank_set_options(pkb_ctx_t *c, int window_type, float dither, uint64_t dither_seed) {
  PKB_REQUIRE(c, "pkb_fbank_set_options: ctx is NULL");
  PKB_REQUIRE(window_type == PKB_WINDOW_HAMMING || window_type == PKB_WINDOW_POVEY,
              "pkb_fbank_set_options: unknown window type %d", window_type);
  PKB_REQUIRE(dither >= 0.0f, "pkb_fbank_set_options: negative dither");
  PKB_CUDA(cudaSetDevice(c->device));
  PKB_CUDA(cudaStreamSynchronize(c->stream));  // kernels in flight read the window table
  if (window_type != c->window_type) {
    c->window_type = window_type;
    PKB_TRY(pkb::build_fbank_tables(c));
  }
  c->dither = dither;
  c->dither_seed = dither_seed;
  return PKB_OK;
}

int pkb_device_sm_count(pkb_ctx_t *c) { return c ? c->sm_count : 0; }
const char *pkb_device_name(pkb_ctx_t *c) { return c ? c->name : ""; }

int pkb_host_alloc(void **ptr, uint64_t bytes) {
  PKB_REQUIRE(ptr, "pkb_host_alloc: ptr is NULL");
  PKB_CUDA(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
  return PKB_OK;
}

void pkb_host_free(void *ptr) {
  if (ptr) cudaFreeHost(ptr);
}

int pkb_timer_start(pkb_ctx_t *c) {
  PKB_REQUIRE(c, "pkb_timer_start: ctx is NULL");
  PKB_CUDA(cudaEventRecord(c->t0, c->stream));
  return PKB_OK;
}

int pkb_timer_stop(pkb_ctx_t *c, float *elapsed_ms) {
  PKB_REQUIRE(c && elapsed_ms, "pkb_timer_stop: NULL argument");
  PKB_CUDA(cudaEventRecord(c->t1, c->stream));
  PKB_CUDA(cudaEventSynchronize(c->t1));
  PKB_CUDA(cudaEventElapsedTime(elapsed_ms, c->t0, c->t1));
  return pkb::check_device_error(c, "pkb_timer_stop");
}

int pkb_profile_enable(pkb_ctx_t *c, int on) {
  PKB_REQUIRE(c, "pkb_profile_enable: ctx is NULL");
  c->profile = on != 0;
  return PKB_OK;
}

static int drain_spans(pkb_ctx_t *c) {
  if (c->spans.empty()) return PKB_OK;
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  for (auto &s : c->spans) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, s.e0, s.e1) == cudaSuccess) c->total_ms[s.cls] += ms;
    c->free_events.push_back(s.e0);
    c->free_events.push_back(s.e1);
  }
  c->spans.clear();
  return PKB_OK;
}

int pkb_profile_reset(pkb_ctx_t *c) {
  PKB_REQUIRE(c, "pkb_profile_reset: ctx is NULL");
  PKB_TRY(drain_spans(c));
  for (int i = 0; i < PKB_KERNEL_CLASSES; ++i) {
    c->launches[i] = 0;
    c->total_ms[i] = 0.0;
  }
  return PKB_OK;
}

int pkb_profile_get(pkb_ctx_t *c, int64_t *launches, double *total_ms) {
  PKB_REQUIRE(c, "pkb_profile_get: ctx is NULL");
  PKB_TRY(drain_spans(c));
  for (int i = 0; i < PKB_KERNEL_CLASSES; ++i) {
    if (launches) launches[i] = c->launches[i];
    if (total_ms) total_ms[i] = c->total_ms[i];
  }
  return PKB_OK;
}

int pkb_flush_l2(pkb_ctx_t *c) {
  PKB_REQUIRE(c, "pkb_flush_l2: ctx is NULL");
  const size_t bytes = size_t(256) << 20;  // > 126 MB L2
  PKB_TRY(c->s_flush.ensure(bytes));
  PKB_CUDA(cudaMemsetAsync(c->s_flush.p, 0, bytes, c->stream));
  return PKB_OK;
}

}  // extern "C"
