// Streaming entry points: n_streams audio streams advance in lock step, chunk by chunk, with
// carried state, so that the concatenated outputs equal the whole-utterance outputs of
// Fbank::Compute -> CMVN::GetFrame -> AcousticModel::Compute (src/fbank.cc:267-292,
// src/cmvn.cc:103-115, src/am.cc:90-115). The reference has no streaming API (SURVEY.md
// section 5); the carried state is exactly what its whole-utterance loops keep implicitly:
//   * PCM tail: the samples after the start of the next frame (N - T*160, < 400 of them),
//   * CMVN: the float running sums of ComputeStats (src/cmvn.cc:35-71), the frame counter and a
//     600-frame ring of raw features for the sliding-window subtraction,
//   * splice: the last left+right normalised frames (src/am.cc:65-88); a frame is emitted once
//     its right context exists, pkb_stream_flush replicates the last frame as the reference does
//     at the utterance end.

#include <stdlib.h>

#include <algorithm>
#include <memory>

#include "decoder.cuh"
#include "nnet.cuh"

namespace pkb {
namespace {

// next[s][0..tail) = prev[s][prev_len - tail .. prev_len)
__global__ void stream_tail_kernel(const int16_t *__restrict__ prev, int prev_stride, int prev_len,
                                   int16_t *__restrict__ next, int next_stride, int tail, int n_streams) {
  const int s = blockIdx.y;
  if (s >= n_streams) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < tail; i += gridDim.x * blockDim.x)
    next[static_cast<size_t>(s) * next_stride + i] =
        prev[static_cast<size_t>(s) * prev_stride + prev_len - tail + i];
}

// carry rows: next[s][0..carry) = prev[s][prev_rows - carry .. prev_rows)
__global__ void stream_shift_kernel(const __nv_bfloat16 *__restrict__ prev, int prev_rows,
                                    __nv_bfloat16 *__restrict__ next, int next_rows, int carry,
                                    int dim_pad, int n_streams) {
  const int s = blockIdx.y;
  if (s >= n_streams) return;
  const int n = carry * dim_pad;
  const __nv_bfloat16 *src = prev + (static_cast<size_t>(s) * prev_rows + prev_rows - carry) * dim_pad;
  __nv_bfloat16 *dst = next + static_cast<size_t>(s) * next_rows * dim_pad;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

// rows [from, from + count) of every stream := row from - 1 (utterance-end replication)
__global__ void stream_replicate_kernel(__nv_bfloat16 *__restrict__ win, int rows, int from, int count,
                                        int dim_pad, int n_streams) {
  const int s = blockIdx.y;
  if (s >= n_streams) return;
  __nv_bfloat16 *base = win + static_cast<size_t>(s) * rows * dim_pad;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count * dim_pad; i += gridDim.x * blockDim.x)
    base[static_cast<size_t>(from) * dim_pad + i] = base[static_cast<size_t>(from - 1) * dim_pad + (i % dim_pad)];
}

// One thread per (stream, dim): continues the recurrence of cmvn_kernel (cmvn.cu) from the
// carried state for `n_new` frames starting at global frame index t0.
__global__ void cmvn_stream_kernel(const float *__restrict__ raw /* [S][n_new][40] */, int n_new,
                                   const int64_t *__restrict__ t_in, int64_t *__restrict__ t_out,
                                   const float *__restrict__ tab, float *__restrict__ stat,
                                   float *__restrict__ ring /* [S][600][40] */,
                                   __nv_bfloat16 *__restrict__ p_hi, __nv_bfloat16 *__restrict__ p_lo,
                                   int win_rows, int carry, int left, int dim_pad, int n_streams,
                                   int fp16) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = g / kMel, d = g % kMel;
  // the frame index of the first new frame lives on the device (two slots used alternately), so
  // that a captured launch sequence can be replayed without new kernel arguments
  const int64_t t0 = *t_in;
  if (g == 0) *t_out = t0 + n_new;
  if (s >= n_streams) return;
  const float gd = tab[2 * kCmvnWindow + d];
  float st = stat[s * kMel + d];
  float *rg = ring + static_cast<size_t>(s) * kCmvnWindow * kMel + d;
  __nv_bfloat16 *ph = p_hi + static_cast<size_t>(s) * win_rows * dim_pad + d;
  __nv_bfloat16 *pl = p_lo ? p_lo + static_cast<size_t>(s) * win_rows * dim_pad + d : nullptr;
  for (int k = 0; k < n_new; ++k) {
    const int64_t t = t0 + k;
    const float x = raw[(static_cast<size_t>(s) * n_new + k) * kMel + d];
    double acc = (t > 0 ? static_cast<double>(st) : 0.0) + static_cast<double>(x);
    const int slot = static_cast<int>(t % kCmvnWindow);
    if (t >= kCmvnWindow) acc += -1.0 * static_cast<double>(rg[static_cast<size_t>(slot) * kMel]);
    rg[static_cast<size_t>(slot) * kMel] = x;
    st = static_cast<float>(acc);
    const int ti = t < kCmvnWindow ? static_cast<int>(t) : kCmvnWindow - 1;
    float sm = st;
    if (t < kCmvnWindow - 1) sm = __fadd_rn(sm, __fmul_rn(tab[ti], gd));
    const float v = __fadd_rn(x, __fmul_rn(-tab[kCmvnWindow + ti], sm));
    const __nv_bfloat16 h = operand_bits(v, fp16);
    const __nv_bfloat16 l = operand_bits(v - operand_value(h, fp16), fp16);
    const size_t row = static_cast<size_t>(carry + k) * dim_pad;
    ph[row] = h;
    if (pl) pl[row] = l;
    if (t == 0)  // utterance start: the left context replicates frame 0 (src/am.cc:75)
      for (int r = 0; r < left; ++r) {
        ph[static_cast<size_t>(r) * dim_pad] = h;
        if (pl) pl[static_cast<size_t>(r) * dim_pad] = l;
      }
  }
  stat[s * kMel + d] = st;
}

}  // namespace
}  // namespace pkb

struct pkb_stream {
  pkb::Ctx *c = nullptr;
  pkb_am *am = nullptr;
  int S = 0, C = 0;
  float scale = 1.0f;
  float global[PKB_CMVN_STATS_DIM];
  int L = 0, R = 0, Dp = 0, P = 0;
  int max_new = 0, max_rows = 0, pcm_stride = 0;
  int tail = 0;                   // carried samples per stream
  int prev_pcm_len = 0, prev_pcm_stride = 0;
  int64_t n_feat = 0, n_emit = 0; // frames normalised / emitted so far
  int prev_rows = 0;              // rows per stream of the current feature window
  int pcur = 0, fcur = 0;         // ping-pong indices of the PCM and feature windows
  int meta_len = -1;              // window length the cached fbank metadata was built for
  pkb::DevBuf pcm[2], raw, stat, ring, win_hi[2], win_lo[2], out;
  pkb::DevBuf out16, out_off;     // compact output form (pkb_stream_set_compact)
  pkb::DevBuf tcount;             // int64[2]: frame index of the next new frame, slots used alternately
  bool compact = false;
  pkb::Workspace ws;
  pkb::BatchMeta meta;
  // Steady state (every push has the same shapes from the second one on): the launch sequence of a
  // push -- tail copy, H2D, fbank, window shift, CMVN, the nnet stages, D2H -- is captured once per
  // ping-pong parity into a CUDA graph and replayed. Tensor maps, kernel attributes and argument
  // marshalling then cost nothing per chunk.
  struct Shape { int win_len, n_new, carry, rows, emit, tail_in, prev_rows, prev_len; };
  Shape last_shape{};
  bool have_last = false;
  // indexed by the two ping-pong indices (pcur * 2 + fcur)
  cudaGraphExec_t gexec[4] = {nullptr, nullptr, nullptr, nullptr};
  const void *g_pcm[4] = {nullptr, nullptr, nullptr, nullptr};
  void *g_out[4] = {nullptr, nullptr, nullptr, nullptr}, *g_out2[4] = {nullptr, nullptr, nullptr, nullptr};
  int64_t g_launches[4][PKB_KERNEL_CLASSES] = {};
  bool graphs_off = false;
  int64_t replays = 0;         // pushes run by replaying a captured graph
  pkb_decoder *dec = nullptr;  // advanced over the emitted rows of every push (pkb_stream_set_decoder)
  void drop_graphs() {
    for (cudaGraphExec_t &g : gexec) {
      if (g) cudaGraphExecDestroy(g);
      g = nullptr;
    }
  }
  ~pkb_stream() {
    if (dec) dec->st = nullptr;
    drop_graphs();
  }
};

namespace {

// Runs the nnet over the current feature window (rows per stream = `rows`), advances the attached
// decoder over the first `emit` rows of every stream and copies those rows to the host unless
// loglik_out is NULL.
int stream_emit(pkb_stream *st, int rows, int emit, void *loglik_out, float *off_out) {
  pkb::Ctx *c = st->c;
  pkb_am *am = st->am;
  if (emit <= 0) return PKB_OK;
  const int64_t gemm_rows = static_cast<int64_t>(st->S) * rows - (st->L + st->R);
  PKB_TRY(pkb::workspace_ensure(am, &st->ws, gemm_rows));
  if (st->compact) {
    PKB_TRY(st->out16.ensure(static_cast<size_t>(gemm_rows) * st->P * sizeof(uint16_t)));
    PKB_TRY(st->out_off.ensure(static_cast<size_t>(gemm_rows) * sizeof(float)));
  } else {
    PKB_TRY(st->out.ensure(static_cast<size_t>(gemm_rows) * st->P * sizeof(float)));
  }
  pkb::InputView in;
  in.hi = st->win_hi[st->fcur].as<__nv_bfloat16>();
  in.lo = am->planes == 2 ? st->win_lo[st->fcur].as<__nv_bfloat16>() : nullptr;
  in.rows = gemm_rows;
  in.cols = (st->L + st->R + 1) * st->Dp;
  in.pitch_elems = st->Dp;
  const int max_frames = pkb_stream_max_frames(st);
  if (st->compact) {
    PKB_TRY(pkb::nnet_forward(am, &st->ws, in, pkb::kFinalCompact, st->scale, nullptr, st->out16.as<uint16_t>(),
                              st->out_off.as<float>()));
    const size_t row_bytes = static_cast<size_t>(st->P) * sizeof(uint16_t);
    PKB_CUDA(cudaMemcpy2DAsync(loglik_out, max_frames * row_bytes, st->out16.p, rows * row_bytes,
                               emit * row_bytes, st->S, cudaMemcpyDeviceToHost, c->stream));
    PKB_CUDA(cudaMemcpy2DAsync(off_out, max_frames * sizeof(float), st->out_off.p, rows * sizeof(float),
                               emit * sizeof(float), st->S, cudaMemcpyDeviceToHost, c->stream));
    return PKB_OK;
  }
  PKB_TRY(pkb::nnet_forward(am, &st->ws, in, pkb::kFinalLoglik, st->scale, st->out.as<float>()));
  if (st->dec) PKB_TRY(pkb::decoder_enqueue_advance(st->dec, st->out.as<float>(), rows, nullptr, emit));
  if (!loglik_out) return PKB_OK;
  const size_t row_bytes = static_cast<size_t>(st->P) * sizeof(float);
  PKB_CUDA(cudaMemcpy2DAsync(loglik_out, max_frames * row_bytes, st->out.p, rows * row_bytes,
                             emit * row_bytes, st->S, cudaMemcpyDeviceToHost, c->stream));
  return PKB_OK;
}

}  // namespace

namespace pkb {
void stream_drop_graphs(pkb_stream *st) { st->drop_graphs(); }
}  // namespace pkb

extern "C" {

int pkb_stream_create(pkb_ctx_t *c, pkb_am_t *am, int n_streams, int chunk_samples,
                      const float *global_stats, float prob_scale, pkb_stream_t **out) {
  PKB_REQUIRE(c && am && out && global_stats, "pkb_stream_create: NULL argument");
  PKB_REQUIRE(am->c == c, "pkb_stream_create: model belongs to another context");
  PKB_REQUIRE(n_streams > 0, "pkb_stream_create: n_streams must be positive");
  PKB_REQUIRE(chunk_samples > 0 && chunk_samples % pkb::kShift == 0,
              "pkb_stream_create: chunk_samples must be a positive multiple of %d", pkb::kShift);
  PKB_REQUIRE(am->feat_dim == pkb::kMel,
              "pkb_stream_create: the model's feature dim must be %d", pkb::kMel);
  PKB_CUDA(cudaSetDevice(c->device));
  std::unique_ptr<pkb_stream, decltype(&pkb_stream_destroy)> st(new pkb_stream(), pkb_stream_destroy);
  st->c = c;
  st->am = am;
  st->S = n_streams;
  st->C = chunk_samples;
  st->scale = prob_scale;
  memcpy(st->global, global_stats, sizeof(st->global));
  st->L = am->left;
  st->R = am->right;
  st->Dp = am->feat_dim_pad;
  st->P = am->num_pdfs;
  st->max_new = chunk_samples / pkb::kShift + 1;
  st->max_rows = st->L + st->R + std::max(st->max_new, st->R);  // flush appends R replicated rows
  st->pcm_stride = pkb::kFrame + chunk_samples;
  const size_t S = n_streams;
  for (int i = 0; i < 2; ++i) {
    PKB_TRY(st->pcm[i].ensure(S * st->pcm_stride * sizeof(int16_t)));
    PKB_TRY(st->win_hi[i].ensure(S * st->max_rows * st->Dp * 2));
    if (am->planes == 2) PKB_TRY(st->win_lo[i].ensure(S * st->max_rows * st->Dp * 2));
  }
  PKB_TRY(st->raw.ensure(S * st->max_new * pkb::kMel * sizeof(float)));
  PKB_TRY(st->stat.ensure(S * pkb::kMel * sizeof(float)));
  PKB_TRY(st->ring.ensure(S * pkb::kCmvnWindow * pkb::kMel * sizeof(float)));
  PKB_TRY(st->tcount.ensure(2 * sizeof(int64_t)));
  cudaMemsetAsync(st->tcount.p, 0, 2 * sizeof(int64_t), c->stream);
  cudaMemsetAsync(st->stat.p, 0, S * pkb::kMel * sizeof(float), c->stream);
  for (int i = 0; i < 2; ++i) {
    cudaMemsetAsync(st->win_hi[i].p, 0, S * st->max_rows * st->Dp * 2, c->stream);
    if (am->planes == 2) cudaMemsetAsync(st->win_lo[i].p, 0, S * st->max_rows * st->Dp * 2, c->stream);
  }
  PKB_TRY(pkb::prepare_cmvn_tables(c, global_stats));
  *out = st.release();
  return PKB_OK;
}

void pkb_stream_destroy(pkb_stream_t *st) {
  if (!st) return;
  if (st->c) {
    cudaSetDevice(st->c->device);
    cudaStreamSynchronize(st->c->stream);
  }
  delete st;
}

int pkb_stream_max_frames(const pkb_stream_t *st) { return st ? st->max_new + st->R : 0; }

int pkb_stream_graph_replays(const pkb_stream_t *st, int64_t *replays) {
  PKB_REQUIRE(st && replays, "pkb_stream_graph_replays: NULL argument");
  *replays = st->replays;
  return PKB_OK;
}

namespace {

// Queues one push on the context stream: nothing here touches the stream object's host state, so
// the same function serves the eager path and the capture of a CUDA graph.
int stream_enqueue_push(pkb_stream *st, const pkb_stream::Shape &sh, const int16_t *pcm, void *out,
                        float *off_out) {
  pkb::Ctx *c = st->c;
  pkb_am *am = st->am;
  const int S = st->S, C = st->C;
  const int pn = st->pcur ^ 1;
  // ---- assemble [tail | chunk] per stream
  int16_t *pw = st->pcm[pn].as<int16_t>();
  if (sh.tail_in > 0) {
    pkb::LaunchScope scope(c, PKB_KERNEL_MISC);
    pkb::stream_tail_kernel<<<dim3(2, S), 256, 0, c->stream>>>(
        st->pcm[st->pcur].as<int16_t>(), st->prev_pcm_stride, sh.prev_len, pw, sh.win_len, sh.tail_in, S);
    PKB_CUDA(cudaGetLastError());
  }
  PKB_CUDA(cudaMemcpy2DAsync(pw + sh.tail_in, static_cast<size_t>(sh.win_len) * 2, pcm,
                             static_cast<size_t>(C) * 2, static_cast<size_t>(C) * 2, S,
                             cudaMemcpyHostToDevice, c->stream));
  if (sh.n_new <= 0) return PKB_OK;
  // ---- fbank of the new frames (same kernel as the batch path)
  PKB_TRY(pkb::launch_fbank_i16(c, pw, st->meta, st->raw.as<float>()));
  // ---- feature window: carried context rows + the new frames
  const int fn = st->fcur ^ 1;
  __nv_bfloat16 *hi = st->win_hi[fn].as<__nv_bfloat16>();
  __nv_bfloat16 *lo = am->planes == 2 ? st->win_lo[fn].as<__nv_bfloat16>() : nullptr;
  if (st->n_feat > 0) {
    pkb::LaunchScope scope(c, PKB_KERNEL_MISC);
    pkb::stream_shift_kernel<<<dim3(2, S), 256, 0, c->stream>>>(
        st->win_hi[st->fcur].as<__nv_bfloat16>(), sh.prev_rows, hi, sh.rows, sh.carry, st->Dp, S);
    if (lo)
      pkb::stream_shift_kernel<<<dim3(2, S), 256, 0, c->stream>>>(
          st->win_lo[st->fcur].as<__nv_bfloat16>(), sh.prev_rows, lo, sh.rows, sh.carry, st->Dp, S);
    PKB_CUDA(cudaGetLastError());
  }
  {
    pkb::LaunchScope scope(c, PKB_KERNEL_CMVN);
    const int threads = S * pkb::kMel;
    int64_t *tc = st->tcount.as<int64_t>();
    pkb::cmvn_stream_kernel<<<(threads + 127) / 128, 128, 0, c->stream>>>(
        st->raw.as<float>(), sh.n_new, tc + st->fcur, tc + fn, c->cmvn_tab.as<float>(), st->stat.as<float>(),
        st->ring.as<float>(), hi, lo, sh.rows, sh.carry, st->L, st->Dp, S, am->fp16);
    PKB_CUDA(cudaGetLastError());
  }
  if (sh.emit > 0) {
    // stream_emit reads the window through st->fcur
    const int keep = st->fcur;
    st->fcur = fn;
    const int rc = stream_emit(st, sh.rows, sh.emit, out, off_out);
    st->fcur = keep;
    PKB_TRY(rc);
  }
  return PKB_OK;
}

int stream_push(pkb_stream *st, const int16_t *pcm, void *out, float *off_out, int32_t *frames_out,
                const char *who) {
  PKB_REQUIRE(st && pcm, "%s: NULL argument", who);
  pkb::Ctx *c = st->c;
  PKB_CUDA(cudaSetDevice(c->device));
  const int S = st->S, C = st->C;
  // ---- shapes of this push from the carried state
  pkb_stream::Shape sh;
  sh.tail_in = st->tail;
  sh.prev_len = st->prev_pcm_len;
  sh.prev_rows = st->prev_rows;
  sh.win_len = st->tail + C;
  sh.n_new = pkb_fbank_num_frames(sh.win_len);
  sh.carry = static_cast<int>(st->n_feat - st->n_emit) + st->L;
  sh.rows = sh.n_new > 0 ? sh.carry + sh.n_new : 0;
  sh.emit = sh.n_new > 0 ? std::max(0, sh.rows - (st->L + st->R)) : 0;
  PKB_REQUIRE(sh.rows <= st->max_rows, "%s: window overflow (%d rows)", who, sh.rows);
  PKB_REQUIRE(!st->dec || !st->dec->flushed, "%s: the stream was flushed: finish its decoder first", who);
  PKB_REQUIRE(sh.emit == 0 || out || st->dec, "%s: the output buffer is NULL", who);
  PKB_REQUIRE(sh.emit == 0 || !st->compact || off_out, "%s: the offset buffer is NULL", who);
  if (st->dec) pkb::decoder_begin_step(st->dec);
  if (sh.n_new > 0) {
    if (st->meta_len != sh.win_len) {
      std::vector<int32_t> ns(S, sh.win_len);
      PKB_TRY(st->meta.build_from_samples(ns.data(), S));
      PKB_TRY(st->meta.upload(c->stream));
      st->meta_len = sh.win_len;
    }
    PKB_TRY(pkb::prepare_cmvn_tables(c, st->global));
  }
  static const bool graphs_env_off = getenv("PKB_STREAM_GRAPH") != nullptr && atoi(getenv("PKB_STREAM_GRAPH")) == 0;
  const bool steady = st->have_last && memcmp(&sh, &st->last_shape, sizeof(sh)) == 0 && sh.emit > 0;
  const int par = st->pcur * 2 + st->fcur;
  bool done = false;
  if (steady && !graphs_env_off && !st->graphs_off && !c->profile) {
    if (st->gexec[par] != nullptr &&
        (st->g_pcm[par] != pcm || st->g_out[par] != out || st->g_out2[par] != off_out)) {
      cudaGraphExecDestroy(st->gexec[par]);  // other host buffers: capture again
      st->gexec[par] = nullptr;
    }
    if (st->gexec[par] == nullptr) {
      int64_t before[PKB_KERNEL_CLASSES];
      memcpy(before, c->launches, sizeof(before));
      cudaGraph_t graph = nullptr;
      int rc = PKB_OK;
      if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        rc = stream_enqueue_push(st, sh, pcm, out, off_out);
        const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
        if (rc == PKB_OK && e == cudaSuccess && graph != nullptr &&
            cudaGraphInstantiate(&st->gexec[par], graph, 0) == cudaSuccess) {
          for (int k = 0; k < PKB_KERNEL_CLASSES; ++k) {
            st->g_launches[par][k] = c->launches[k] - before[k];
            c->launches[k] = before[k];
          }
          st->g_pcm[par] = pcm;
          st->g_out[par] = out;
          st->g_out2[par] = off_out;
        } else {
          st->gexec[par] = nullptr;
          st->graphs_off = true;  // something in the sequence cannot be captured here: stay eager
          memcpy(c->launches, before, sizeof(before));
          cudaGetLastError();
        }
        if (graph) cudaGraphDestroy(graph);
      } else {
        st->graphs_off = true;
        cudaGetLastError();
      }
    }
    if (st->gexec[par] != nullptr) {
      PKB_CUDA(cudaGraphLaunch(st->gexec[par], c->stream));
      ++st->replays;
      for (int k = 0; k < PKB_KERNEL_CLASSES; ++k) c->launches[k] += st->g_launches[par][k];
      done = true;
    }
  }
  if (!done) PKB_TRY(stream_enqueue_push(st, sh, pcm, out, off_out));
  // ---- advance the carried state
  st->pcur ^= 1;
  st->prev_pcm_stride = sh.win_len;
  st->prev_pcm_len = sh.win_len;
  st->tail = sh.win_len - sh.n_new * pkb::kShift;
  if (sh.n_new > 0) {
    st->n_feat += sh.n_new;
    st->prev_rows = sh.rows;
    st->fcur ^= 1;
    st->n_emit += sh.emit;
  }
  st->last_shape = sh;
  st->have_last = true;
  if (frames_out) *frames_out = sh.emit;
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, who);
}

}  // namespace

int pkb_stream_push_i16(pkb_stream_t *st, const int16_t *pcm, float *loglik_out, int32_t *frames_out) {
  PKB_REQUIRE(st && !st->compact, "pkb_stream_push_i16: the stream writes the compact output (use pkb_stream_push_compact_i16)");
  return stream_push(st, pcm, loglik_out, nullptr, frames_out, "pkb_stream_push_i16");
}

int pkb_stream_push_compact_i16(pkb_stream_t *st, const int16_t *pcm, uint16_t *h16_out, float *off_out,
                                int32_t *frames_out) {
  PKB_REQUIRE(st && st->compact, "pkb_stream_push_compact_i16: switch the compact output on first (pkb_stream_set_compact)");
  return stream_push(st, pcm, h16_out, off_out, frames_out, "pkb_stream_push_compact_i16");
}

int pkb_stream_set_compact(pkb_stream_t *st, int on) {
  PKB_REQUIRE(st, "pkb_stream_set_compact: stream is NULL");
  PKB_REQUIRE(!on || st->am->softmax_last, "pkb_stream_set_compact: the model does not end in a softmax");
  PKB_REQUIRE(!on || !st->dec, "pkb_stream_set_compact: the attached decoder reads the FP32 rows");
  if ((on != 0) == st->compact) return PKB_OK;
  PKB_CUDA(cudaSetDevice(st->c->device));
  PKB_CUDA(cudaStreamSynchronize(st->c->stream));
  st->drop_graphs();
  st->compact = on != 0;
  return PKB_OK;
}

int pkb_stream_set_decoder(pkb_stream_t *st, pkb_decoder_t *dec) {
  PKB_REQUIRE(st, "pkb_stream_set_decoder: stream is NULL");
  if (dec == st->dec) return PKB_OK;
  if (dec) {
    PKB_REQUIRE(dec->c == st->c && dec->am == st->am && dec->n == st->S,
                "pkb_stream_set_decoder: the decoder has another context, model or stream count");
    PKB_REQUIRE(!st->compact, "pkb_stream_set_decoder: the decoder reads the FP32 rows (switch the compact output off)");
    PKB_REQUIRE(!dec->st, "pkb_stream_set_decoder: the decoder is attached to another stream");
  }
  PKB_CUDA(cudaSetDevice(st->c->device));
  PKB_CUDA(cudaStreamSynchronize(st->c->stream));
  st->drop_graphs();  // the captured pushes advance the old decoder, or none
  if (st->dec) st->dec->st = nullptr;
  st->dec = dec;
  if (dec) dec->st = st;
  return PKB_OK;
}

static int stream_flush(pkb_stream_t *st, void *loglik_out, float *off_out, int32_t *frames_out) {
  PKB_REQUIRE(st, "pkb_stream_flush: stream is NULL");
  pkb::Ctx *c = st->c;
  PKB_CUDA(cudaSetDevice(c->device));
  if (st->dec) pkb::decoder_begin_step(st->dec);
  int emit = 0;
  const int pending = static_cast<int>(st->n_feat - st->n_emit);
  if (pending > 0) {
    PKB_REQUIRE((loglik_out || st->dec) && (!st->compact || off_out), "pkb_stream_flush: output buffer is NULL");
    // rows = carry (pending + L); append R replicas of the last frame (src/am.cc:76)
    const int carry = pending + st->L;
    const int rows = carry + st->R;
    PKB_REQUIRE(rows <= st->max_rows, "pkb_stream_flush: window overflow");
    // the window is stored with row pitch prev_rows per stream: re-pitch into the other buffer
    const int nxt = st->fcur ^ 1;
    pkb_am *am = st->am;
    __nv_bfloat16 *hi = st->win_hi[nxt].as<__nv_bfloat16>();
    __nv_bfloat16 *lo = am->planes == 2 ? st->win_lo[nxt].as<__nv_bfloat16>() : nullptr;
    {
      pkb::LaunchScope scope(c, PKB_KERNEL_MISC);
      pkb::stream_shift_kernel<<<dim3(2, st->S), 256, 0, c->stream>>>(
          st->win_hi[st->fcur].as<__nv_bfloat16>(), st->prev_rows, hi, rows, carry, st->Dp, st->S);
      pkb::stream_replicate_kernel<<<dim3(1, st->S), 256, 0, c->stream>>>(hi, rows, carry, st->R, st->Dp, st->S);
      if (lo) {
        pkb::stream_shift_kernel<<<dim3(2, st->S), 256, 0, c->stream>>>(
            st->win_lo[st->fcur].as<__nv_bfloat16>(), st->prev_rows, lo, rows, carry, st->Dp, st->S);
        pkb::stream_replicate_kernel<<<dim3(1, st->S), 256, 0, c->stream>>>(lo, rows, carry, st->R, st->Dp, st->S);
      }
      PKB_CUDA(cudaGetLastError());
    }
    st->fcur = nxt;
    st->prev_rows = rows;
    emit = rows - (st->L + st->R);
    PKB_TRY(stream_emit(st, rows, emit, loglik_out, off_out));
    st->n_emit += emit;
  }
  if (frames_out) *frames_out = emit;
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  // reset for a new utterance
  st->tail = 0;
  st->n_feat = st->n_emit = 0;
  st->prev_rows = 0;
  st->have_last = false;
  if (st->dec) st->dec->flushed = true;
  PKB_CUDA(cudaMemsetAsync(st->stat.p, 0, static_cast<size_t>(st->S) * pkb::kMel * sizeof(float), c->stream));
  PKB_CUDA(cudaMemsetAsync(st->tcount.p, 0, 2 * sizeof(int64_t), c->stream));
  return pkb::check_device_error(c, "pkb_stream_flush");
}

int pkb_stream_flush(pkb_stream_t *st, float *loglik_out, int32_t *frames_out) {
  PKB_REQUIRE(st && !st->compact, "pkb_stream_flush: the stream writes the compact output (use pkb_stream_flush_compact)");
  return stream_flush(st, loglik_out, nullptr, frames_out);
}

int pkb_stream_flush_compact(pkb_stream_t *st, uint16_t *h16_out, float *off_out, int32_t *frames_out) {
  PKB_REQUIRE(st && st->compact, "pkb_stream_flush_compact: switch the compact output on first");
  return stream_flush(st, h16_out, off_out, frames_out);
}

}  // extern "C"
