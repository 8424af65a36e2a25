// Arc and frame posteriors over the kept records of a lattice (pkb_batch_posteriors,
// pkb_decoder_posteriors): a forward-backward pass in the log semiring, one thread block per
// utterance, in the fold order of include/pkb200.h.
//
// The forward pass is the walk of lattice_walk.cuh with lse as its fold. The block then walks the
// groups backward, with the costs of two times live as per-state double arrays (in shared memory
// when they fit):
//   backward          the records of a group are already grouped by source (the FST's arcs are
//                     sorted by source state), so a node folds its outgoing epsilon records, then
//                     its outgoing emitting records, from two contiguous ranges; the epsilon records
//                     of a time in Kahn levels, a node once every head is complete.
// The forward pass saves alpha(t, src) per record (8 bytes), so the backward pass finishes each
// record's posterior as soon as beta at its head is known. The frame posteriors of time t are the
// emitting posteriors of the group grouped by pdf with the same stable sort, summed in record
// order, thresholded and written in pdf order. The backward pass produces times in descending
// order, so an utterance's entries are written from the end of its record range downwards and
// gathered into (t, pdf) order afterwards. No float atomics: repeated calls are bit-identical.

#include <math.h>

#include <algorithm>

#include "lattice_walk.cuh"

namespace pkb {
namespace {

using lattice_walk::kThreads;
using lattice_walk::kSmemState;
using lattice_walk::scaled_cost;

// work: per block sort order and group posteriors [, per-state arrays]
struct PostArgs : lattice_walk::WalkArgs {
  const int32_t *tid2pdf;
  int num_pdfs;
  float min_post;
  float *arc_post;          // [records]
  pkb_frame_post_t *tail;   // [records]: utterance u's entries end at first[u] + n_arcs[u]
  double *total;            // [n_utts]
  long long *n_post;        // [n_utts]
};

// -log(exp(-a) + exp(-b)); +inf is the identity
__device__ __forceinline__ double lse(double a, double b) {
  const double m = fmin(a, b), M = fmax(a, b);
  return M == INFINITY ? m : m - log1p(exp(m - M));
}

__device__ __forceinline__ double arc_posterior(double total, double alpha, double c, double beta) {
  return total < INFINITY ? exp(total - ((alpha + c) + beta)) : 0.0;
}

__global__ void __launch_bounds__(kThreads) posterior_kernel(PostArgs A) {
  __shared__ lattice_walk::Shared sh;
  __shared__ double s_total;
  extern __shared__ double smem_state[];
  const int w = blockIdx.x, u = A.u0 + w, tid = threadIdx.x;
  const long long na = A.n_arcs[u];
  if (na < 0) {
    if (tid == 0) {
      A.total[u] = NAN;
      A.n_post[u] = na;
    }
    return;
  }
  const long long f0 = A.first[u];
  if (!(A.best[u] < INFINITY)) {  // no complete path, so no records
    for (long long i = tid; i < na; i += kThreads) A.arc_post[f0 + i] = 0.0f;
    if (tid == 0) {
      A.total[u] = INFINITY;
      A.n_post[u] = 0;
    }
    return;
  }
  const pkb_lattice_arc_t *recs = A.arcs + f0;
  double *alpha = A.alpha + (f0 - A.rec0);
  const int S = A.num_states, P = A.num_pdfs, K = max(S, P), NA = A.num_arcs;
  char *g = A.work + A.work_stride * w;
  int *perm = reinterpret_cast<int *>(g);                                           // [NA]
  double *pd = reinterpret_cast<double *>(g + ((sizeof(int) * NA + 7) & ~size_t(7)));  // [NA]
  char *st = A.smem_state ? reinterpret_cast<char *>(smem_state) : reinterpret_cast<char *>(pd + NA);
  double *X = reinterpret_cast<double *>(st);  // [S] costs of the current time
  double *Y = X + S;                           // [S] costs of the neighbouring time
  double *acc = Y + S;                         // [K] frame posteriors by pdf
  int *done = reinterpret_cast<int *>(acc + K);  // [S] Kahn state: 0 open, 1 folded this level, 2 complete
  int *fill = done + S;                        // [K]
  int *seg = fill + K;                         // [K + 1]
  int *eb = seg + K + 1, *ee = eb + S, *mb = ee + S, *me = mb + S;  // [S] each: runs by source

  const lattice_walk::Walk W{recs, na, NA, K, tid, perm, fill, seg, sh};
  const int T = W.last_time();
  const int err = W.forward(X, Y, done, S, A.start, T, alpha,
                            [&](const pkb_lattice_arc_t &r) { return scaled_cost(A, r); },
                            [](double held, double c) { return lse(held, c); });
  if (err) {
    for (long long i = tid; i < na; i += kThreads) A.arc_post[f0 + i] = NAN;
    if (tid == 0) {
      A.total[u] = NAN;
      A.n_post[u] = -err;
    }
    return;
  }
  if (tid == 0) {
    double tot = INFINITY;
    for (int s = 0; s < S; ++s) {
      const float f = A.final_w[s];
      if (f < INFINITY) tot = lse(tot, X[s] + __dmul_rn(A.gs, static_cast<double>(f)));
    }
    s_total = tot;
  }
  __syncthreads();
  const double total = s_total;

  // ---- backward: beta(t, .) in X, beta(t + 1, .) in Y
  long long end = na;
  int nout = 0;
  for (int t = T; t >= 0; --t) {
    const long long m_beg = t < T ? W.group_end(max(0ll, end - NA), 2 * t) : end;
    const long long e_beg = t > 0 ? W.group_end(max(0ll, m_beg - NA), 2 * t - 1) : 0;
    const pkb_lattice_arc_t *E = recs + e_beg, *M = recs + m_beg;
    const int ne = static_cast<int>(m_beg - e_beg), nm = static_cast<int>(end - m_beg);
    if (nm > 0) {
      // posteriors of emit(t), then its frame posteriors
      for (int i = tid; i < nm; i += kThreads) {
        const pkb_lattice_arc_t &r = M[i];
        const double p = arc_posterior(total, alpha[m_beg + i], scaled_cost(A, r), Y[r.dst]);
        pd[i] = p;
        A.arc_post[f0 + m_beg + i] = static_cast<float>(p);
      }
      W.group_by_key(nm, [&](int i) { return A.tid2pdf[M[i].ilabel]; });
      const int per = (P + kThreads - 1) / kThreads, k0 = min(P, tid * per), k1 = min(P, k0 + per);
      int cnt = 0;
      for (int k = k0; k < k1; ++k) {
        if (seg[k + 1] == seg[k]) continue;
        double sum = 0.0;
        for (int j = seg[k]; j < seg[k + 1]; ++j) sum += pd[perm[j]];
        acc[k] = sum;
        cnt += static_cast<float>(sum) >= A.min_post;
      }
      int base = 0, kept = 0;
      lattice_walk::Scan(sh.tmp.scan).ExclusiveSum(cnt, base, kept);
      pkb_frame_post_t *out = A.tail + f0 + na - nout - kept;
      for (int k = k0; k < k1; ++k) {
        if (seg[k + 1] == seg[k]) continue;
        const float v = static_cast<float>(acc[k]);
        if (v >= A.min_post) out[base++] = pkb_frame_post_t{t, k, v};
      }
      nout += kept;
    }
    // beta(t, s): the final weight at T, then the outgoing epsilon and emitting records of s in
    // record order
    for (int s = tid; s < S; s += kThreads) {
      eb[s] = ee[s] = mb[s] = me[s] = 0;
      done[s] = 0;
    }
    __syncthreads();
    for (int i = tid; i < ne; i += kThreads) {
      const int s = E[i].src;
      if (i == 0 || E[i - 1].src != s) eb[s] = i;
      if (i == ne - 1 || E[i + 1].src != s) ee[s] = i + 1;
    }
    for (int i = tid; i < nm; i += kThreads) {
      const int s = M[i].src;
      if (i == 0 || M[i - 1].src != s) mb[s] = i;
      if (i == nm - 1 || M[i + 1].src != s) me[s] = i + 1;
    }
    __syncthreads();
    for (;;) {
      for (int s = tid; s < S; s += kThreads) {
        if (done[s]) continue;
        bool ready = true;
        for (int i = eb[s]; i < ee[s] && ready; ++i) ready = done[E[i].dst] == 2;
        if (!ready) continue;
        double b = INFINITY;
        if (t == T) {
          const float f = A.final_w[s];
          if (f < INFINITY) b = __dmul_rn(A.gs, static_cast<double>(f));
        }
        for (int i = eb[s]; i < ee[s]; ++i) b = lse(b, scaled_cost(A, E[i]) + X[E[i].dst]);
        for (int i = mb[s]; i < me[s]; ++i) b = lse(b, scaled_cost(A, M[i]) + Y[M[i].dst]);
        X[s] = b;
        done[s] = 1;
      }
      __syncthreads();
      int progress = 0;
      for (int s = tid; s < S; s += kThreads)
        if (done[s] == 1) {
          done[s] = 2;
          progress = 1;
        }
      if (!__syncthreads_or(progress)) break;
    }
    for (int i = tid; i < ne; i += kThreads) {
      const pkb_lattice_arc_t &r = E[i];
      A.arc_post[f0 + e_beg + i] = static_cast<float>(arc_posterior(total, alpha[e_beg + i], scaled_cost(A, r), X[r.dst]));
    }
    __syncthreads();
    double *tx = X;
    X = Y;
    Y = tx;
    end = e_beg;
  }
  if (tid == 0) {
    A.total[u] = total;
    A.n_post[u] = nout;
  }
}

// Moves utterance u's frame entries from the end of its record range to out + off[u].
__global__ void posterior_gather_kernel(const pkb_frame_post_t *__restrict__ tail, const long long *__restrict__ first,
                                        const long long *__restrict__ n_arcs, const long long *__restrict__ n_post,
                                        const long long *__restrict__ off, pkb_frame_post_t *__restrict__ out) {
  const int u = blockIdx.x;
  const long long k = n_post[u];
  if (k <= 0) return;
  const pkb_frame_post_t *src = tail + first[u] + n_arcs[u] - k;
  for (long long i = threadIdx.x; i < k; i += blockDim.x) out[off[u] + i] = src[i];
}

}  // namespace

int LatticeResults::posteriors(float acoustic_scale, float graph_scale, float min_post, double *total_out,
                               int64_t *n_post_out, const char *who) {
  PKB_REQUIRE(total >= 0, "%s: no lattice: %s", who, why.c_str());
  PKB_REQUIRE(acoustic_scale > 0.0f && acoustic_scale < INFINITY,
              "%s: acoustic_scale must be finite and > 0 (got %g)", who, acoustic_scale);
  PKB_REQUIRE(graph_scale >= 0.0f && graph_scale < INFINITY, "%s: graph_scale must be finite and >= 0 (got %g)",
              who, graph_scale);
  PKB_REQUIRE(min_post >= 0.0f && min_post <= 1.0f, "%s: min_post must be in [0, 1] (got %g)", who, min_post);
  PKB_REQUIRE(total_out && n_post_out, "%s: NULL output argument", who);
  post.n_arcs = -1;
  post.n_frames = 0;
  const int U = static_cast<int>(n_arcs.size());
  if (U == 0) {
    post.n_arcs = 0;
    return PKB_OK;
  }
  PKB_CUDA(cudaSetDevice(c->device));
  const long long R = total;
  const int S = fst->num_states, P = num_pdfs, K = std::max(S, P), NA = std::max(fst->num_arcs, 1);
  PKB_REQUIRE(K < (1 << 30), "pkb posteriors: %d states or pdfs are too many", K);
  // results: arc posteriors; per call: frame entries at the end of each record range, totals,
  // codes and the entries' output offsets
  PKB_TRY(post.arc.ensure(sizeof(float) * std::max(R, 1ll)));
  const size_t tail_bytes = (sizeof(pkb_frame_post_t) * std::max(R, 1ll) + 7) & ~size_t(7);
  DevBuf scratch;
  PKB_TRY(scratch.ensure(tail_bytes + sizeof(double) * U + sizeof(long long) * (2 * U + 1)));
  pkb_frame_post_t *d_tail = scratch.as<pkb_frame_post_t>();
  double *d_total = reinterpret_cast<double *>(scratch.as<char>() + tail_bytes);
  long long *d_npost = reinterpret_cast<long long *>(d_total + U);
  long long *d_off = d_npost + U;
  // per block: sort order and group posteriors (NA each), and the per-state arrays when they do
  // not fit in shared memory
  const size_t state_bytes = sizeof(double) * (2 * static_cast<size_t>(S) + K) +
                             sizeof(int) * (5 * static_cast<size_t>(S) + 2 * static_cast<size_t>(K) + 1);
  const bool smem_state = state_bytes <= kSmemState;
  const size_t stride = ((((sizeof(int) * NA + 7) & ~size_t(7)) + sizeof(double) * NA +
                          (smem_state ? 0 : state_bytes)) + 255) & ~size_t(255);
  // utterances in waves whose alpha and workspace fit the budget
  std::vector<size_t> bytes(U);
  for (int u = 0; u < U; ++u) bytes[u] = stride + sizeof(double) * std::max<int64_t>(n_arcs[u], 0);
  std::vector<int> wave_start;
  size_t wave_max = 0;
  PKB_TRY(plan_waves(bytes, &wave_start, &wave_max));
  DevBuf wave_buf;
  PKB_TRY(wave_buf.ensure(wave_max));
  // the static shared memory and the per-state arrays together can pass the default 48 KiB
  if (smem_state)
    PKB_CUDA(cudaFuncSetAttribute(posterior_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(state_bytes)));
  PostArgs A{};
  static_cast<lattice_walk::WalkArgs &>(A) = lattice_walk::walk_args(*this, acoustic_scale, graph_scale);
  A.tid2pdf = d_tid2pdf;
  A.num_pdfs = P;
  A.min_post = min_post;
  A.work_stride = stride;
  A.smem_state = smem_state;
  A.arc_post = post.arc.as<float>();
  A.tail = d_tail;
  A.total = d_total;
  A.n_post = d_npost;
  for (size_t i = 0; i + 1 < wave_start.size(); ++i) {
    const int u0 = wave_start[i], m = wave_start[i + 1] - u0;
    A.u0 = u0;
    A.work = wave_buf.as<char>();
    A.alpha = reinterpret_cast<double *>(wave_buf.as<char>() + stride * m);
    A.rec0 = first[u0];
    LaunchScope scope(c, PKB_KERNEL_MISC);
    posterior_kernel<<<m, kThreads, smem_state ? state_bytes : 0, c->stream>>>(A);
    PKB_CUDA(cudaGetLastError());
  }
  static_assert(sizeof(long long) == sizeof(int64_t), "int64_t is long long");
  PKB_CUDA(cudaMemcpyAsync(total_out, d_total, sizeof(double) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_post_out, d_npost, sizeof(long long) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  std::vector<long long> off(U);
  long long n_frames = 0;
  for (int u = 0; u < U; ++u) {
    off[u] = n_frames;
    n_frames += std::max<long long>(n_post_out[u], 0);
  }
  PKB_TRY(post.frames.ensure(sizeof(pkb_frame_post_t) * std::max(n_frames, 1ll)));
  PKB_CUDA(cudaMemcpyAsync(d_off, off.data(), sizeof(long long) * U, cudaMemcpyHostToDevice, c->stream));
  {
    LaunchScope scope(c, PKB_KERNEL_MISC);
    posterior_gather_kernel<<<U, 256, 0, c->stream>>>(d_tail, d_first(), d_n_arcs(), d_npost, d_off,
                                                       post.frames.as<pkb_frame_post_t>());
    PKB_CUDA(cudaGetLastError());
  }
  // the host copy of off must outlive the copy
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  post.n_arcs = R;
  post.n_frames = n_frames;
  return check_device_error(c, who);
}

int LatticeResults::posteriors_get(float *arc_post_out, pkb_frame_post_t *frame_post_out, const char *who) {
  PKB_REQUIRE(total >= 0, "%s: no lattice: %s", who, why.c_str());
  PKB_REQUIRE(post.n_arcs >= 0, "%s: no posteriors since the latest lattice", who);
  PKB_CUDA(cudaSetDevice(c->device));
  if (arc_post_out && post.n_arcs > 0)
    PKB_CUDA(cudaMemcpyAsync(arc_post_out, post.arc.p, sizeof(float) * post.n_arcs, cudaMemcpyDeviceToHost,
                             c->stream));
  if (frame_post_out && post.n_frames > 0)
    PKB_CUDA(cudaMemcpyAsync(frame_post_out, post.frames.p, sizeof(pkb_frame_post_t) * post.n_frames,
                             cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return check_device_error(c, who);
}

}  // namespace pkb
