// The best path of a lattice at any acoustic scale, graph scale and word insertion penalty, with
// its words, their times and its frame alignment (pkb_batch_best_path, pkb_decoder_best_path): a
// forward pass in the tropical semiring, one thread block per utterance, in the fold order of
// include/pkb200.h, then a traceback.
//
// The forward pass is the walk of lattice_walk.cuh with min as its fold: a candidate replaces the
// held value only when it is strictly smaller. The walk saves alpha(t, src) per record, so the
// winner at a node of value v is re-identified exactly as the first candidate in fold order whose
// alpha(t, src) + c(r) equals v (computed with the same double operations): every earlier candidate
// was larger and no later one replaced it. No back-pointers are stored. The traceback starts at the
// best final node and, per node, searches the emitting records of the previous time, then the
// epsilon records of its own time, with the whole block; the winner's saved alpha is the value of
// the next node. It stops at (0, start) of value 0, whose held initial value no candidate replaced.
// One thread then walks the path forward, summing its costs in path order and writing its words,
// their times and the alignment at the start of the utterance's record range; they are gathered
// into place afterwards.

#include <limits.h>
#include <math.h>

#include <algorithm>

#include "lattice_walk.cuh"

namespace pkb {
namespace {

using lattice_walk::kSmemState;
using lattice_walk::kThreads;
using lattice_walk::scaled_cost;

// work: per block the sort order [, per-state arrays]
struct BestArgs : lattice_walk::WalkArgs {
  double wp;
  int *path;                        // the path's records, last first, at the same offsets as alpha
  int32_t *words, *word_t, *ali;    // [records]: utterance u's from first[u] on
  double *cost, *gcost, *acost;     // [n_utts]
  int32_t *n_words, *n_frames;      // [n_utts]
};

// c(r): the scaled cost plus the word insertion penalty on a word
__device__ __forceinline__ double path_cost(const BestArgs &A, const pkb_lattice_arc_t &r) {
  const double c = scaled_cost(A, r);
  return r.olabel ? __dadd_rn(c, A.wp) : c;
}

__global__ void __launch_bounds__(kThreads) best_path_kernel(BestArgs A) {
  __shared__ lattice_walk::Shared sh;
  __shared__ int s_first, s_final;
  __shared__ double s_cost;
  extern __shared__ double smem_state[];
  const int w = blockIdx.x, u = A.u0 + w, tid = threadIdx.x;
  const long long na = A.n_arcs[u];
  auto result = [&](double cost, double g, double a, int nw, int nf) {
    if (tid == 0) {
      A.cost[u] = cost;
      A.gcost[u] = g;
      A.acost[u] = a;
      A.n_words[u] = nw;
      A.n_frames[u] = nf;
    }
  };
  if (na < 0) {
    result(NAN, NAN, NAN, static_cast<int>(na), 0);
    return;
  }
  if (!(A.best[u] < INFINITY)) {  // no complete path
    result(INFINITY, INFINITY, INFINITY, 0, 0);
    return;
  }
  const long long f0 = A.first[u];
  const pkb_lattice_arc_t *recs = A.arcs + f0;
  double *alpha = A.alpha + (f0 - A.rec0);
  int *path = A.path + (f0 - A.rec0);
  const int S = A.num_states, NA = A.num_arcs;
  char *g = A.work + A.work_stride * w;
  int *perm = reinterpret_cast<int *>(g);  // [NA]
  char *st = A.smem_state ? reinterpret_cast<char *>(smem_state) : g + ((sizeof(int) * NA + 7) & ~size_t(7));
  double *X = reinterpret_cast<double *>(st);  // [S] costs of the current time
  double *Y = X + S;                           // [S] costs of the next time
  int *done = reinterpret_cast<int *>(Y + S);  // [S] Kahn state
  int *fill = done + S;                        // [S]
  int *seg = fill + S;                         // [S + 1]

  const lattice_walk::Walk W{recs, na, NA, S, tid, perm, fill, seg, sh};
  const int T = W.last_time();
  const int err = W.forward(X, Y, done, S, A.start, T, alpha,
                            [&](const pkb_lattice_arc_t &r) { return path_cost(A, r); },
                            [](double held, double c) { return c < held ? c : held; });
  if (err) {
    result(NAN, NAN, NAN, -err, 0);
    return;
  }
  // the best final node: the least alpha(T, s) + graph_scale x final(s), ties to the lowest state
  if (tid == 0) {
    double best = INFINITY;
    int bs = -1;
    for (int s = 0; s < S; ++s) {
      const float f = A.final_w[s];
      if (f < INFINITY) {
        const double v = X[s] + __dmul_rn(A.gs, static_cast<double>(f));
        if (v < best) {
          best = v;
          bs = s;
        }
      }
    }
    s_cost = best;
    s_final = bs;
  }
  __syncthreads();
  const double cost = s_cost;
  const int fin = s_final;
  if (fin < 0) {
    result(INFINITY, INFINITY, INFINITY, 0, 0);
    return;
  }

  // the first record of [lo, hi) into s whose candidate equals v, or -1
  auto first_match = [&](long long lo, long long hi, int s, double v) {
    if (tid == 0) s_first = INT_MAX;
    __syncthreads();
    for (long long i = lo + tid; i < hi; i += kThreads) {
      const pkb_lattice_arc_t &r = recs[i];
      if (r.dst == s && __dadd_rn(alpha[i], path_cost(A, r)) == v) {
        atomicMin(&s_first, static_cast<int>(i - lo));
        break;
      }
    }
    __syncthreads();
    const int k = s_first;
    __syncthreads();
    return k == INT_MAX ? -1ll : lo + k;
  };
  // traceback from (T, fin): eps(t) is [eps_beg, eps_end), emit(t - 1) is [emit_beg, eps_beg)
  int s = fin, len = 0;
  double v = X[fin];
  long long eps_end = na;
  for (int t = T; len < na; --t) {
    const long long eps_beg = t > 0 ? W.group_end(max(0ll, eps_end - NA), 2 * t - 1) : 0;
    const long long emit_beg = t > 0 ? W.group_end(max(0ll, eps_beg - NA), 2 * t - 2) : 0;
    long long r = -1;
    while (len < na && !(t == 0 && s == A.start && v == 0.0)) {
      r = t > 0 ? first_match(emit_beg, eps_beg, s, v) : -1;
      const bool emitting = r >= 0;
      if (!emitting) r = first_match(eps_beg, eps_end, s, v);
      if (r < 0) break;
      if (tid == 0) path[len] = static_cast<int>(r);
      ++len;
      s = recs[r].src;
      v = alpha[r];
      if (emitting) break;
    }
    if (r < 0 || t == 0) break;
    eps_end = emit_beg;
  }
  __syncthreads();
  if (tid == 0) {
    int32_t *words = A.words + f0, *word_t = A.word_t + f0, *ali = A.ali + f0;
    double gc = 0.0, ac = 0.0;
    int nw = 0;
    for (int k = len - 1; k >= 0; --k) {
      const pkb_lattice_arc_t r = recs[path[k]];
      gc += static_cast<double>(r.graph_cost);
      ac += static_cast<double>(r.acoustic_cost);
      if (r.olabel) {
        words[nw] = r.olabel;
        word_t[nw] = r.t;
        ++nw;
      }
      if (r.ilabel) ali[r.t] = r.ilabel;
    }
    gc += static_cast<double>(A.final_w[fin]);
    result(cost, gc, ac, nw, T);
  }
}

// Moves utterance u's words, word times and alignment from the start of its record range to their
// offsets in the packed results.
__global__ void best_path_gather_kernel(const int32_t *__restrict__ words, const int32_t *__restrict__ word_t,
                                        const int32_t *__restrict__ ali, const long long *__restrict__ first,
                                        const int32_t *__restrict__ n_words, const int32_t *__restrict__ n_frames,
                                        const long long *__restrict__ off, int n_utts, int32_t *__restrict__ words_out,
                                        int32_t *__restrict__ word_t_out, int32_t *__restrict__ ali_out) {
  const int u = blockIdx.x;
  const long long f0 = first[u], wo = off[u], fo = off[n_utts + u];
  for (int i = threadIdx.x; i < n_words[u]; i += blockDim.x) {
    words_out[wo + i] = words[f0 + i];
    word_t_out[wo + i] = word_t[f0 + i];
  }
  for (int i = threadIdx.x; i < n_frames[u]; i += blockDim.x) ali_out[fo + i] = ali[f0 + i];
}

}  // namespace

int LatticeResults::best_path(float acoustic_scale, float graph_scale, float word_penalty, double *cost_out,
                              double *graph_cost_out, double *acoustic_cost_out, int32_t *n_words_out,
                              int32_t *n_frames_out, const char *who) {
  PKB_REQUIRE(total >= 0, "%s: no lattice: %s", who, why.c_str());
  PKB_REQUIRE(acoustic_scale > 0.0f && acoustic_scale < INFINITY,
              "%s: acoustic_scale must be finite and > 0 (got %g)", who, acoustic_scale);
  PKB_REQUIRE(graph_scale >= 0.0f && graph_scale < INFINITY, "%s: graph_scale must be finite and >= 0 (got %g)",
              who, graph_scale);
  PKB_REQUIRE(std::isfinite(word_penalty), "%s: word_penalty must be finite (got %g)", who, word_penalty);
  PKB_REQUIRE(cost_out && graph_cost_out && acoustic_cost_out && n_words_out && n_frames_out,
              "%s: NULL output argument", who);
  bp.n_words = -1;
  bp.n_frames = 0;
  const int U = static_cast<int>(n_arcs.size());
  if (U == 0) {
    bp.n_words = 0;
    return PKB_OK;
  }
  PKB_CUDA(cudaSetDevice(c->device));
  const long long R = std::max<long long>(total, 1);
  const int S = fst->num_states, NA = std::max(fst->num_arcs, 1);
  PKB_REQUIRE(S < (1 << 30), "pkb best path: %d states are too many", S);
  // per call: words, word times and alignment at the start of each record range; the costs, counts
  // and output offsets of every utterance
  DevBuf scratch;
  PKB_TRY(scratch.ensure(sizeof(double) * 3 * U + sizeof(long long) * 2 * U + sizeof(int32_t) * (3 * R + 2 * U)));
  double *d_cost = scratch.as<double>(), *d_gcost = d_cost + U, *d_acost = d_gcost + U;
  long long *d_off = reinterpret_cast<long long *>(d_acost + U);
  int32_t *d_nw = reinterpret_cast<int32_t *>(d_off + 2 * U), *d_nf = d_nw + U;
  int32_t *d_words = d_nf + U, *d_word_t = d_words + R, *d_ali = d_word_t + R;
  // per block: the sort order, and the per-state arrays when they do not fit in shared memory
  const size_t state_bytes =
      sizeof(double) * 2 * static_cast<size_t>(S) + sizeof(int) * (3 * static_cast<size_t>(S) + 1);
  const bool smem_state = state_bytes <= kSmemState;
  const size_t stride = (((sizeof(int) * NA + 7) & ~size_t(7)) + (smem_state ? 0 : state_bytes) + 255) & ~size_t(255);
  // utterances in waves whose alpha, path and workspace fit the budget
  std::vector<size_t> bytes(U);
  for (int u = 0; u < U; ++u) bytes[u] = stride + (sizeof(double) + sizeof(int)) * std::max<int64_t>(n_arcs[u], 0);
  std::vector<int> wave_start;
  size_t wave_max = 0;
  PKB_TRY(plan_waves(bytes, &wave_start, &wave_max));
  DevBuf wave_buf;
  PKB_TRY(wave_buf.ensure(wave_max));
  // the static shared memory and the per-state arrays together can pass the default 48 KiB
  if (smem_state)
    PKB_CUDA(cudaFuncSetAttribute(best_path_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(state_bytes)));
  BestArgs A{};
  static_cast<lattice_walk::WalkArgs &>(A) = lattice_walk::walk_args(*this, acoustic_scale, graph_scale);
  A.wp = word_penalty;
  A.work_stride = stride;
  A.smem_state = smem_state;
  A.words = d_words;
  A.word_t = d_word_t;
  A.ali = d_ali;
  A.cost = d_cost;
  A.gcost = d_gcost;
  A.acost = d_acost;
  A.n_words = d_nw;
  A.n_frames = d_nf;
  for (size_t i = 0; i + 1 < wave_start.size(); ++i) {
    const int u0 = wave_start[i], m = wave_start[i + 1] - u0;
    long long recs = 0;
    for (int u = u0; u < u0 + m; ++u) recs += std::max<int64_t>(n_arcs[u], 0);
    A.u0 = u0;
    A.work = wave_buf.as<char>();
    A.alpha = reinterpret_cast<double *>(wave_buf.as<char>() + stride * m);
    A.path = reinterpret_cast<int *>(A.alpha + recs);
    A.rec0 = first[u0];
    LaunchScope scope(c, PKB_KERNEL_MISC);
    best_path_kernel<<<m, kThreads, smem_state ? state_bytes : 0, c->stream>>>(A);
    PKB_CUDA(cudaGetLastError());
  }
  PKB_CUDA(cudaMemcpyAsync(cost_out, d_cost, sizeof(double) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(graph_cost_out, d_gcost, sizeof(double) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(acoustic_cost_out, d_acost, sizeof(double) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_words_out, d_nw, sizeof(int32_t) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_frames_out, d_nf, sizeof(int32_t) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  std::vector<long long> off(2 * U);
  long long n_words = 0, n_frames = 0;
  for (int u = 0; u < U; ++u) {
    off[u] = n_words;
    off[U + u] = n_frames;
    n_words += std::max(n_words_out[u], 0);
    n_frames += n_frames_out[u];
  }
  PKB_TRY(bp.words.ensure(sizeof(int32_t) * 2 * std::max(n_words, 1ll)));
  PKB_TRY(bp.ali.ensure(sizeof(int32_t) * std::max(n_frames, 1ll)));
  PKB_CUDA(cudaMemcpyAsync(d_off, off.data(), sizeof(long long) * 2 * U, cudaMemcpyHostToDevice, c->stream));
  {
    LaunchScope scope(c, PKB_KERNEL_MISC);
    best_path_gather_kernel<<<U, 256, 0, c->stream>>>(d_words, d_word_t, d_ali, d_first(), d_nw, d_nf, d_off, U,
                                                      bp.words.as<int32_t>(), bp.words.as<int32_t>() + n_words,
                                                      bp.ali.as<int32_t>());
    PKB_CUDA(cudaGetLastError());
  }
  // the host copy of off must outlive the copy
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  bp.n_words = n_words;
  bp.n_frames = n_frames;
  return check_device_error(c, who);
}

int LatticeResults::best_path_get(int32_t *words_out, int32_t *word_t_out, int32_t *ali_out, const char *who) {
  PKB_REQUIRE(total >= 0, "%s: no lattice: %s", who, why.c_str());
  PKB_REQUIRE(bp.n_words >= 0, "%s: no best path since the latest lattice", who);
  PKB_CUDA(cudaSetDevice(c->device));
  const int32_t *d_words = bp.words.as<int32_t>();
  if (words_out && bp.n_words > 0)
    PKB_CUDA(cudaMemcpyAsync(words_out, d_words, sizeof(int32_t) * bp.n_words, cudaMemcpyDeviceToHost, c->stream));
  if (word_t_out && bp.n_words > 0)
    PKB_CUDA(cudaMemcpyAsync(word_t_out, d_words + bp.n_words, sizeof(int32_t) * bp.n_words,
                             cudaMemcpyDeviceToHost, c->stream));
  if (ali_out && bp.n_frames > 0)
    PKB_CUDA(cudaMemcpyAsync(ali_out, bp.ali.p, sizeof(int32_t) * bp.n_frames, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return check_device_error(c, who);
}

}  // namespace pkb
