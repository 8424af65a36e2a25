// Shared declarations of libpkb200: context, error plumbing, launch accounting.
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <utility>
#include <vector>

#include "pkb200.h"

namespace pkb {

constexpr int kSampleRate = 16000;
constexpr int kShift = PKB_FRAME_SHIFT;    // src/fbank.cc:15
constexpr int kFrame = PKB_FRAME_LENGTH;   // src/fbank.cc:16
constexpr int kNfft = 512;                 // src/fbank.cc:24-33
constexpr int kMel = PKB_FBANK_DIM;        // src/fbank.h:10
constexpr int kCmvnWindow = 600;           // src/cmvn.h:10
constexpr int kCmvnGlobal = 200;           // src/cmvn.h:11

void set_error(const char *fmt, ...);

#define PKB_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t pkb_e_ = (expr);                                                         \
    if (pkb_e_ != cudaSuccess) {                                                         \
      pkb::set_error("%s: %s (%s:%d)", #expr, cudaGetErrorString(pkb_e_), __FILE__,      \
                     __LINE__);                                                          \
      return PKB_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define PKB_TRY(expr)                  \
  do {                                 \
    int pkb_rc_ = (expr);              \
    if (pkb_rc_ != PKB_OK) return pkb_rc_; \
  } while (0)

#define PKB_REQUIRE(cond, ...)         \
  do {                                 \
    if (!(cond)) {                     \
      pkb::set_error(__VA_ARGS__);     \
      return PKB_ERR_INVALID;          \
    }                                  \
  } while (0)

// Grow-only device allocation, freed when the buffer is destroyed.
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
  ~DevBuf() { release(); }
  int ensure(size_t bytes);
  void release();
  template <typename T> T *as() const { return static_cast<T *>(p); }
};

// Tables the fbank kernel stages into shared memory (all device pointers).
struct FbankTables {
  const float *hamming;       // [400]                     src/fbank.cc:249-256
  const float2 *tw_pass;      // [16][16] W256^(j*k1) at [k1*16+j]
  const float2 *tw_real;      // [16][16] W512^(k1+16*k2) at [k2*16+k1]
  const float4 *mel_w;        // [4][32]  weights of lane entries 4q..4q+3
  const uint32_t *mel_bins;   // [4][32]  four packed uint8 FFT-bin indices
  const uint32_t *mel_ctl;    // [32]     flush mask | first slot << 16
  const uint32_t *mel_sum;    // [40]     first slot | slot count << 16
};

struct ProfSpan {
  int cls;
  cudaEvent_t e0, e1;
};

// ---- metadata of a packed utterance batch (host side + device copy) -------
struct BatchMeta {
  int n_utts = 0;
  int64_t total_samples = 0;
  int64_t total_frames = 0;
  int n_tiles = 0;                      // fbank tiles of kFramesPerTile frames
  std::vector<int32_t> num_samples, num_frames, tile_prefix;
  std::vector<int32_t> tile_utt;        // utterance of every fbank tile
  std::vector<int64_t> sample_off, frame_off;
  // device copies (one allocation)
  DevBuf dev;
  const int32_t *d_num_samples = nullptr, *d_num_frames = nullptr, *d_tile_prefix = nullptr;
  const int32_t *d_tile_utt = nullptr;
  const int64_t *d_sample_off = nullptr, *d_frame_off = nullptr;
  int build_from_samples(const int32_t *ns, int n);
  int build_from_frames(const int32_t *nf, int n);
  int upload(cudaStream_t stream);
};

struct Ctx {
  int device = 0;
  int sm_count = 0;
  char name[256] = {0};
  cudaStream_t stream = nullptr;
  // front-end tables
  DevBuf tables;
  FbankTables fb{};
  // options the reference does not have (pkb_fbank_set_options); defaults = the reference
  int window_type = PKB_WINDOW_HAMMING;
  float dither = 0.0f;
  uint64_t dither_seed = 0;
  // CMVN per-frame smoothing tables for the current global stats
  DevBuf cmvn_tab;           // float alpha[600], scale[600], global[41]
  float cmvn_global[PKB_CMVN_STATS_DIM] = {0};
  bool cmvn_valid = false;
  // scratch for the host-buffer entry points
  DevBuf s_in, s_raw, s_out, s_flush;
  BatchMeta meta;
  // device -> host error word (mapped pinned memory): a kernel that gives up on a bounded wait
  // stores a code here instead of trapping, which would poison the whole CUDA context
  int *err_host = nullptr;
  int *err_dev = nullptr;
  // timers / profiling
  cudaEvent_t t0 = nullptr, t1 = nullptr;
  bool profile = false;
  int64_t launches[PKB_KERNEL_CLASSES] = {0};
  double total_ms[PKB_KERNEL_CLASSES] = {0};
  std::vector<ProfSpan> spans;
  std::vector<cudaEvent_t> free_events;
  ~Ctx();  // the caller has made the device current and drained the stream
};

// Host -> device upload ordered on the context stream and complete on return. Plain cudaMemcpy
// from pageable memory may return before the DMA has landed, and the context stream is
// non-blocking (no implicit ordering against the legacy stream), so a kernel queued right after it
// could read stale bytes.
int upload(Ctx *c, void *dst, const void *src, size_t bytes);

// Reports (and clears) an error word left by a kernel; call after a stream synchronisation.
int check_device_error(Ctx *c, const char *who);

// RAII launch accounting: counts every launch, and with profiling on brackets
// it with an event pair on the context stream.
struct LaunchScope {
  Ctx *c;
  ProfSpan span;
  bool timed;
  LaunchScope(Ctx *ctx, int cls);
  ~LaunchScope();
};

constexpr int kFramesPerTile = 8;

// ---- kernels' host launchers ---------------------------------------------
int launch_fbank_i16(Ctx *c, const int16_t *d_pcm, const BatchMeta &m, float *d_raw);
int launch_fbank_f32(Ctx *c, const float *d_wave, const BatchMeta &m, float *d_raw);
// raw -> out (fp32). When planes != nullptr also writes the padded BF16 planes
// consumed by the first nnet GEMM (see nnet.cuh).
struct PaddedPlanes {
  __nv_bfloat16 *hi = nullptr;  // [padded rows][dim_pad]
  __nv_bfloat16 *lo = nullptr;  // nullptr in PKB_PREC_BF16
  const int64_t *d_pad_off = nullptr;  // [n_utts] first padded row of each utterance
  int left = 0, right = 0, dim_pad = 0;
  int fp16 = 0;  // planes hold FP16 bit patterns instead of BF16 (PKB_PREC_FP16)
};

// 16-bit GEMM operand encoding of v: BF16 (default) or FP16 bits, stored in __nv_bfloat16 slots.
__host__ __device__ inline __nv_bfloat16 operand_bits(float v, int fp16) {
  if (fp16) {
    const __half_raw hr = static_cast<__half_raw>(__float2half_rn(v));
    __nv_bfloat16_raw br;
    br.x = hr.x;
    return __nv_bfloat16(br);
  }
  return __float2bfloat16_rn(v);
}
__host__ __device__ inline float operand_value(__nv_bfloat16 b, int fp16) {
  if (fp16) {
    const __nv_bfloat16_raw br = static_cast<__nv_bfloat16_raw>(b);
    __half_raw hr;
    hr.x = br.x;
    return __half2float(__half(hr));
  }
  return __bfloat162float(b);
}
int prepare_cmvn_tables(Ctx *c, const float *global_stats);
int launch_cmvn(Ctx *c, const float *d_raw, const BatchMeta &m, float *d_out,
                const PaddedPlanes *planes);
int launch_synth_pcm(Ctx *c, int16_t *d_pcm, const BatchMeta &m, uint64_t seed,
                     uint64_t first_utt);
int launch_checksum(Ctx *c, const float *d, int64_t n, double *d_sum);

int build_fbank_tables(Ctx *c);

}  // namespace pkb

struct pkb_ctx : pkb::Ctx {};
