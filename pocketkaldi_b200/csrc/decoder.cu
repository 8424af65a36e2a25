// GPU token-passing Viterbi beam search (SURVEY 8(f)-4): one thread block per utterance walks the
// frames of its utterance with the log-likelihood rows already resident in HBM, so neither the
// [frames x pdfs] matrix nor one host core per utterance is needed to get from PCM to words.
//
// Reference: Decoder::Decode / InitDecoding / ProcessEmitting / ProcessNonemitting / BestPath
// (src/decoder.cc:39-339), Fst::IterateArcs (src/fst.cc:94-129), pk_decodable_loglikelihood
// (src/decodable.cc:24-31). What is kept exactly:
//   * arc cost arithmetic: total = double(token cost) + double(arc weight) + double(acoustic cost),
//     stored back as float (src/decoder.cc:276-291, Token::cost_ is a float);
//   * the beam: weight_cutoff = float(best + beam) on the previous frame's tokens (:141-200 with
//     fewer than kBeamSize = 30000 tokens), next cutoff = min over kept arcs of total + beam,
//     ProcessNonemitting(float(next cutoff)) (:203-237);
//   * BestPath: min over tokens of cost + final(state), weight = that + final(state) once more
//     (the reference adds the final weight twice, :300-339).
// What differs: the reference tightens the next cutoff while it walks the token list, so arcs seen
// early are tested against a looser bound and may create tokens that the final bound would not;
// those tokens lie outside the next frame's beam and are dropped there. Here every arc is tested
// against the final (tightest) bound. The max-active estimate by sampling (:141-200, more than
// 30000 tokens) is replaced by a hard per-utterance capacity that fails the utterance. Ties between
// equal float costs are broken by arc index instead of by list order.

#include <math.h>

#include <algorithm>
#include <memory>

#include "decoder.cuh"

namespace pkb {

namespace {

constexpr int kVitThreads = 256;
// kVitGroup lanes share one token's arcs: 8 for graphs with a few arcs per state, a whole warp for
// dense ones (the launcher picks by the average out-degree)
constexpr unsigned long long kEmptyVal = ~0ull;
constexpr uint32_t kNoArc = 0xffffffffu;

// total order on floats / doubles as unsigned integers
__device__ __forceinline__ uint32_t ord32(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unord32(uint32_t o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ unsigned long long ord64(double d) {
  const unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(d));
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double unord64(unsigned long long o) {
  return __longlong_as_double(static_cast<long long>((o >> 63) ? (o & 0x7fffffffffffffffull) : ~o));
}
__device__ __forceinline__ unsigned long long pack(float cost, uint32_t arc) {
  return (static_cast<unsigned long long>(ord32(cost)) << 32) | arc;
}
__device__ __forceinline__ float cost_of(unsigned long long v) { return unord32(static_cast<uint32_t>(v >> 32)); }

struct FstDev {
  int num_states, start, has_eps;
  const float *final_w;
  const int32_t *arc_begin, *arc_src, *arc_dst, *arc_il, *arc_ol;
  const float *arc_w;
};

// One frame's tokens: open-addressing table state -> (cost, winning arc) plus the list of used slots.
struct Tab {
  int *keys;                 // state + 1, 0 = empty
  unsigned long long *vals;  // pack(cost, arc); kEmptyVal when unused
  int *bp;                   // index of the token's newest word record, -1 none, -2 not resolved yet
  int *list;                 // slots in use
};

struct Work {
  Tab tab[2];
  int *frontier[2];
  int *inq;        // [H] slot is queued for the epsilon closure
  int *log_prev;   // word records: previous record, output label
  int *log_ol;
};

__device__ __forceinline__ uint32_t hash_state(int s) { return static_cast<uint32_t>(s) * 2654435761u; }

// slot of `state`, or -1
__device__ __forceinline__ int tab_find(const Tab &t, int state, uint32_t mask) {
  uint32_t s = hash_state(state) & mask;
  for (uint32_t n = 0; n <= mask; ++n) {
    const int k = t.keys[s];
    if (k == state + 1) return static_cast<int>(s);
    if (k == 0) return -1;
    s = (s + 1) & mask;
  }
  return -1;
}

// slot of `state`, claiming an empty one (and appending it to the list) when it is new; -1 on overflow
__device__ __forceinline__ int tab_insert(const Tab &t, int state, uint32_t mask, int *n_tok, int max_tok) {
  uint32_t s = hash_state(state) & mask;
  for (uint32_t n = 0; n <= mask; ++n) {  // bounded: a full table (capacity overflow) must not spin
    int k = *reinterpret_cast<volatile int *>(&t.keys[s]);
    if (k == 0) {
      k = atomicCAS(&t.keys[s], 0, state + 1);
      if (k == 0) {
        const int i = atomicAdd(n_tok, 1);
        if (i >= max_tok) return -1;
        t.list[i] = static_cast<int>(s);
        t.bp[s] = -2;
        return static_cast<int>(s);
      }
    }
    if (k == state + 1) return static_cast<int>(s);
    s = (s + 1) & mask;
  }
  return -1;
}


// End of an advance, once the live tokens of stream u are saved in the carry: the best-so-far
// hypothesis (lowest cost, ties to the lowest state, no final weight), then -- when the word-record
// store is more than half full -- its compaction to the records the live tokens can reach.
__device__ void carry_end_advance(const Carry &cr, int u, int n_tok, int T, int *log_prev, int *log_ol,
                                  int *mark, int max_log, int max_words, int n_log, int err, bool alive) {
  __shared__ unsigned long long e_min;
  __shared__ int e_idx, e_sum[kVitThreads];
  const int tid = threadIdx.x;
  const size_t base = static_cast<size_t>(u) * cr.cap;
  int *ts = cr.tok_state + base, *tb = cr.tok_bp + base;
  const float *tc = cr.tok_cost + base;
  if (tid == 0) { e_min = ~0ull; e_idx = -1; }
  __syncthreads();
  if (!err && alive)
    for (int i = tid; i < n_tok; i += kVitThreads) atomicMin(&e_min, pack(tc[i], static_cast<uint32_t>(ts[i])));
  __syncthreads();
  if (e_min != ~0ull)
    for (int i = tid; i < n_tok; i += kVitThreads)
      if (ts[i] == static_cast<int>(static_cast<uint32_t>(e_min))) e_idx = i;
  // compaction: mark what the live tokens reach (a walk stops at a record already marked)
  const bool compact = !err && n_log > max_log / 2;
  if (compact)
    for (int i = tid; i < n_tok; i += kVitThreads)
      for (int r = tb[i]; r >= 0 && atomicExch(&mark[r], 1) == 0; r = log_prev[r]) {}
  __syncthreads();
  if (tid == 0) {
    const long long frames = cr.frames[u] + T;
    cr.frames[u] = frames;
    cr.p_frames[u] = frames;
    int32_t *wo = cr.p_words + static_cast<size_t>(u) * max_words;
    if (err) {
      cr.p_nw[u] = -err;
      cr.p_cost[u] = 0.0f;
    } else if (e_idx < 0) {
      cr.p_nw[u] = 0;  // no token survives: the reference has no hypothesis either
      cr.p_cost[u] = 0.0f;
    } else {
      cr.p_cost[u] = cost_of(e_min);
      int nw = 0;
      for (int r = tb[e_idx]; r >= 0; r = log_prev[r]) ++nw;
      cr.p_nw[u] = nw;
      int k = nw;
      for (int r = tb[e_idx]; r >= 0; r = log_prev[r])
        if (--k < max_words) wo[k] = log_ol[r];
    }
  }
  int kept = n_log;
  if (compact) {
    // exclusive scan of the marks: mark[r] becomes the new index of record r, -1 when dropped
    const int per = (n_log + kVitThreads - 1) / kVitThreads;
    const int r0 = min(tid * per, n_log), r1 = min(r0 + per, n_log);
    int cnt = 0;
    for (int r = r0; r < r1; ++r) cnt += mark[r];
    e_sum[tid] = cnt;
    __syncthreads();
    if (tid == 0) {
      int run = 0;
      for (int i = 0; i < kVitThreads; ++i) { const int v = e_sum[i]; e_sum[i] = run; run += v; }
      e_idx = run;
    }
    __syncthreads();
    int k = e_sum[tid];
    for (int r = r0; r < r1; ++r) mark[r] = mark[r] ? k++ : -1;
    __syncthreads();
    kept = e_idx;
    for (int r = tid; r < n_log; r += kVitThreads)
      if (mark[r] >= 0 && log_prev[r] >= 0) log_prev[r] = mark[log_prev[r]];
    __syncthreads();
    // move forward in order (new index <= old index): read a block of records, then write it
    for (int b = 0; b < n_log; b += kVitThreads) {
      const int r = b + tid;
      const int to = r < n_log ? mark[r] : -1;
      const int lp = to >= 0 ? log_prev[r] : 0, lo = to >= 0 ? log_ol[r] : 0;
      __syncthreads();
      if (to >= 0) { log_prev[to] = lp; log_ol[to] = lo; }
      __syncthreads();
    }
    for (int i = tid; i < n_tok; i += kVitThreads)
      if (tb[i] >= 0) tb[i] = mark[tb[i]];
    __syncthreads();
    for (int r = tid; r < n_log; r += kVitThreads) mark[r] = 0;
  }
  if (tid == 0) {
    int *h = cr.hdr + 4 * u;
    h[0] = err ? 0 : n_tok;
    h[1] = kept;
    h[2] = err;
    h[3] = alive ? 1 : 0;
  }
  __syncthreads();
}

// End of a finish: the stream starts a fresh utterance at its next advance.
__device__ void carry_reset(const Carry &cr, int u) {
  if (threadIdx.x == 0) {
    cr.hdr[4 * u] = -1;
    cr.frames[u] = 0;
    cr.p_frames[u] = 0;
    cr.p_nw[u] = 0;
    cr.p_cost[u] = 0.0f;
  }
}

// ---------------------------------------------------------------------------------------------
// Lattice mode of the batch search (Lattice in decoder.cuh). Only the lattice instantiations
// reference this block's shared state.
constexpr int kLatScanMax = 16 * (kVitThreads / 32);  // flags per thread x warps of block_scan
constexpr unsigned long long kKept = 1ull << 63;      // a log entry's mark (arc indices are < 2^31)

struct LatShared {
  int count;                    // log entries of the current utterance
  int changed;
  int cnt[kLatScanMax + 1];
  unsigned long long best;      // ord64 of the best final cost
};
__device__ __forceinline__ LatShared &lat_shared() {
  __shared__ LatShared s;
  return s;
}

// Exclusive block-wide prefix count of K flags per thread, in the order (k, thread): pos[k] is the
// number of set flags before flag k of this thread. Returns the total. Everyone must call it.
template <int K>
__device__ int block_scan(const bool (&flag)[K], int (&pos)[K]) {
  int *cnt = lat_shared().cnt;
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const unsigned m = __ballot_sync(0xffffffffu, flag[k]);
    pos[k] = __popc(m & ((1u << lane) - 1u));
    if (lane == 0) cnt[k * (kVitThreads / 32) + wp] = __popc(m);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int run = 0;
    for (int i = 0; i < K * (kVitThreads / 32); ++i) { const int v = cnt[i]; cnt[i] = run; run += v; }
    cnt[K * (kVitThreads / 32)] = run;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) pos[k] += cnt[k * (kVitThreads / 32) + wp];
  const int total = cnt[K * (kVitThreads / 32)];
  __syncthreads();
  return total;
}

// Appends group g to the log in the order (k, thread), i.e. by arc index when arc k of a thread is
// tid + 256 k: the arcs whose flag is set, with their source's cost. Everyone must call it.
template <int K>
__device__ void lat_append_ordered(const Lattice &lat, unsigned long long *lg, int *go, int g,
                                   const bool (&flag)[K], const float (&src_cost)[K], int *err) {
  LatShared &ls = lat_shared();
  const int base = ls.count;
  int pos[K];
  const int total = block_scan<K>(flag, pos);
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int r = base + pos[k];
    if (flag[k] && r < lat.max_arcs)
      lg[r] = (static_cast<unsigned long long>(threadIdx.x + k * kVitThreads) << 32) | __float_as_uint(src_cost[k]);
  }
  if (threadIdx.x == 0) {
    go[g] = base;
    ls.count = base + total;
    if (base + total > lat.max_arcs && !*err) *err = 4;
  }
  __syncthreads();
}

// After a pass that appended with atomics: a log past max_arcs fails the utterance with 4, unless
// the pass already failed it otherwise (the reported code does not depend on the order of atomics).
__device__ __forceinline__ void lat_check_overflow(const Lattice &lat, int *err) {
  if (threadIdx.x == 0 && !*err && lat_shared().count > lat.max_arcs) *err = 4;
  __syncthreads();
}

// Sorts a[0, n) ascending: bitonic network whose comparators all put the minimum first, so that
// the missing elements up to the next power of two act as +inf and are never touched.
__device__ void block_sort(unsigned long long *a, int n) {
  int P = 1;
  while (P < n) P <<= 1;
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j >= 1; j >>= 1) {
      for (int idx = threadIdx.x; idx < P / 2; idx += kVitThreads) {
        const int i = (idx / j) * 2 * j + idx % j;
        const int l = j == (k >> 1) ? (i ^ (k - 1)) : i + j;
        if (l < n) {
          const unsigned long long x = a[i], y = a[l];
          if (x > y) { a[i] = y; a[l] = x; }
        }
      }
      __syncthreads();
    }
  }
}

// Backward pass over utterance u's log once its search is complete, with `best` finite:
//   beta(T, s) = final(s); beta(t, s) = min over logged arcs leaving (t, s) of
//   (w + ac) + beta(head), epsilon arcs of a time relaxed to a fixpoint (also at T);
//   an arc is kept when beta(head) is finite and ((alpha(tail) + w) + ac) + beta(head) <= best + beam,
// all in double, ac re-read from the row. `beta` keeps two times, b = t & 1: reset(b), get(b, s)
// (+inf when absent) and relax(b, s, v) (min; true when it lowered the value). The kept arcs are
// then moved to the front of the log as (group << 32 | arc) and, unless the log was written in
// arc order, sorted. Returns the kept count.
template <class Reset, class Get, class Relax>
__device__ int lattice_prune(const FstDev &fst, const Lattice &lat, unsigned long long *lg, const int *go, int T,
                             const float *ll0, int num_pdfs, const int32_t *tid2pdf, double best, bool sort,
                             int *err, Reset reset, Get get, Relax relax) {
  LatShared &ls = lat_shared();
  const int tid = threadIdx.x;
  const double bound = best + static_cast<double>(lat.beam);
  auto beta = [&](int b, int s, bool at_end) {
    const double v = get(b, s);
    return at_end ? fmin(v, static_cast<double>(__ldg(&fst.final_w[s]))) : v;
  };
  for (int t = T; t >= 0; --t) {
    const int b = t & 1;
    const bool end = t == T;
    reset(b);
    if (!end) {
      // emitting arcs from t to t + 1
      const float *ll = ll0 + static_cast<int64_t>(t) * num_pdfs;
      for (int i = go[2 * t + 1] + tid; i < go[2 * t + 2]; i += kVitThreads) {
        const unsigned long long e = lg[i];
        const int a = static_cast<int>(e >> 32);
        const double bh = beta(b ^ 1, __ldg(&fst.arc_dst[a]), t + 1 == T);
        if (bh == INFINITY) continue;
        const double w = static_cast<double>(__ldg(&fst.arc_w[a]));
        const double ac = static_cast<double>(-__ldg(&ll[__ldg(&tid2pdf[__ldg(&fst.arc_il[a])])]));
        relax(b, __ldg(&fst.arc_src[a]), (w + ac) + bh);
        if (((static_cast<double>(__uint_as_float(static_cast<uint32_t>(e))) + w) + ac) + bh <= bound)
          lg[i] = e | kKept;
      }
      __syncthreads();
    }
    // epsilon arcs within t
    const int p0 = go[2 * t], p1 = go[2 * t + 1];
    if (p1 > p0) {
      for (int round = 0;; ++round) {
        if (tid == 0) ls.changed = 0;
        __syncthreads();
        for (int i = p0 + tid; i < p1; i += kVitThreads) {
          const int a = static_cast<int>(lg[i] >> 32);
          const double bh = beta(b, __ldg(&fst.arc_dst[a]), end);
          if (bh != INFINITY && relax(b, __ldg(&fst.arc_src[a]), static_cast<double>(__ldg(&fst.arc_w[a])) + bh))
            ls.changed = 1;
        }
        __syncthreads();
        const int changed = ls.changed;
        __syncthreads();
        if (!changed) break;
        if (round == 4096) {
          if (tid == 0) *err = 3;
          __syncthreads();
          return 0;
        }
      }
      for (int i = p0 + tid; i < p1; i += kVitThreads) {
        const unsigned long long e = lg[i];
        const int a = static_cast<int>(e >> 32);
        const double bh = beta(b, __ldg(&fst.arc_dst[a]), end);
        const double w = static_cast<double>(__ldg(&fst.arc_w[a]));
        if (bh != INFINITY && ((static_cast<double>(__uint_as_float(static_cast<uint32_t>(e))) + w) + 0.0) + bh <= bound)
          lg[i] = e | kKept;
      }
      __syncthreads();
    }
    if (*err) return 0;
  }
  // kept arcs to the front, in order (a write never passes a read of a later block of entries)
  const int n_log = go[2 * T + 1];
  int kept = 0;
  for (int b0 = 0; b0 < n_log; b0 += kVitThreads) {
    const int r = b0 + tid;
    const unsigned long long e = r < n_log ? lg[r] : 0ull;
    bool keep[1] = {(e & kKept) != 0};
    int pos[1];
    unsigned long long key = 0;
    if (keep[0]) {
      int lo = 0, hi = 2 * T + 1;  // the last group that starts at or before r
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (go[mid] <= r) lo = mid; else hi = mid - 1;
      }
      key = (static_cast<unsigned long long>(lo) << 32) | ((e >> 32) & 0x7fffffffull);
    }
    const int total = block_scan<1>(keep, pos);
    if (keep[0]) lg[kept + pos[0]] = key;
    kept += total;
    __syncthreads();
  }
  if (sort) block_sort(lg, kept);
  return kept;
}

template <int kVitGroup, bool kResume, bool kLattice>
__global__ void __launch_bounds__(kVitThreads)
viterbi_kernel(FstDev fst, float beam, int max_tok, uint32_t mask, int max_log, int max_words,
               const float *__restrict__ loglik, int num_pdfs, const int64_t *__restrict__ row_off,
               const int32_t *__restrict__ num_frames, int n_utts, const int32_t *__restrict__ tid2pdf,
               char *work_base, size_t work_stride, int tables_in_smem, int32_t *__restrict__ words_out,
               int32_t *__restrict__ n_words_out, float *__restrict__ weight_out, Carry cr, Lattice lat) {
  __shared__ int s_ntok[2], s_nfront[2], s_log, s_err, s_unres;
  __shared__ unsigned long long s_min;
  // resumable lattice mode: the lattice's own error, so that a lattice that does not fit fails
  // only the lattice and the search goes on (the batch search stops at its first error of either kind)
  __shared__ int s_laterr;
  int *const lerr = kResume ? &s_laterr : &s_err;
  // the lattice is still being logged: checked at points where every thread sees the same flags
  auto lat_live = [&]() { return !kResume || (!s_err && !s_laterr); };

  // carve this block's workspace. Small graphs (every state fits the token capacity chosen by the
  // launcher) keep the two token tables, the lists and the queue in shared memory: the per-frame
  // chain of dependent look-ups and atomics then never leaves the SM. The word records stay global.
  extern __shared__ __align__(16) char s_tab[];
  const uint32_t H = mask + 1;
  char *gp = work_base + static_cast<size_t>(blockIdx.x) * work_stride;
  char *wp = tables_in_smem ? s_tab : gp;
  Work w;
  for (int i = 0; i < 2; ++i) {
    w.tab[i].vals = reinterpret_cast<unsigned long long *>(wp); wp += sizeof(unsigned long long) * H;
  }
  for (int i = 0; i < 2; ++i) {
    w.tab[i].keys = reinterpret_cast<int *>(wp); wp += sizeof(int) * H;
    w.tab[i].bp = reinterpret_cast<int *>(wp); wp += sizeof(int) * H;
    w.tab[i].list = reinterpret_cast<int *>(wp); wp += sizeof(int) * max_tok;
    w.frontier[i] = reinterpret_cast<int *>(wp); wp += sizeof(int) * max_tok;
  }
  w.inq = reinterpret_cast<int *>(wp); wp += sizeof(int) * H;
  if (tables_in_smem) wp = gp;  // the global workspace then holds the word records only
  w.log_prev = reinterpret_cast<int *>(wp); wp += sizeof(int) * max_log;
  w.log_ol = reinterpret_cast<int *>(wp);
  int *mark = w.log_ol + max_log;  // resumable search: compaction marks

  const int tid = threadIdx.x;
  if (tables_in_smem) {
    // the invariant the global workspace gets from the launcher's memset
    for (uint32_t i = tid; i < H; i += kVitThreads) {
      for (int k = 0; k < 2; ++k) {
        w.tab[k].keys[i] = 0;
        w.tab[k].vals[i] = kEmptyVal;
      }
      w.inq[i] = 0;
    }
    __syncthreads();
  }
  constexpr int kVitGroups = kVitThreads / kVitGroup;
  const int grp = tid / kVitGroup, gl = tid % kVitGroup;

  // Epsilon closure of table `c` (ProcessNonemitting, src/decoder.cc:203-237) under `cutoff`, then
  // the word back-pointers of every token of the frame. `p` is the previous frame's table.
  auto close_and_resolve = [&](int c, int p, double cutoff) {
    const Tab &tc = w.tab[c];
    if (fst.has_eps) {
      // frontier = every token of the frame
      const int n0 = s_ntok[c];
      for (int i = tid; i < n0; i += kVitThreads) w.frontier[0][i] = tc.list[i];
      if (tid == 0) { s_nfront[0] = n0 < max_tok ? n0 : max_tok; s_nfront[1] = 0; }
      __syncthreads();
      int fb = 0;
      for (;;) {
        const int nf = s_nfront[fb];
        if (nf == 0) break;
        // the queue flags of this round's states are cleared before any of them is expanded, so an
        // improvement that lands while a state is being expanded always re-queues it
        for (int i = tid; i < nf; i += kVitThreads) w.inq[w.frontier[fb][i]] = 0;
        __syncthreads();
        for (int i = tid; i < nf; i += kVitThreads) {
          const int slot = w.frontier[fb][i];
          const int state = tc.keys[slot] - 1;
          const float cost = cost_of(*reinterpret_cast<volatile unsigned long long *>(&tc.vals[slot]));
          for (int a = __ldg(&fst.arc_begin[state]); a < __ldg(&fst.arc_begin[state + 1]); ++a) {
            if (__ldg(&fst.arc_il[a]) != 0) continue;
            const double total = static_cast<double>(cost) + static_cast<double>(__ldg(&fst.arc_w[a]));
            if (total > cutoff) continue;
            const int s2 = tab_insert(tc, __ldg(&fst.arc_dst[a]), mask, &s_ntok[c], max_tok);
            if (s2 < 0) { s_err = 1; continue; }
            // InsertTok replaces only on a strictly lower cost (src/decoder.cc:127-134): CAS loop
            const unsigned long long nv = pack(static_cast<float>(total), static_cast<uint32_t>(a));
            unsigned long long old = *reinterpret_cast<volatile unsigned long long *>(&tc.vals[s2]);
            bool won = false;
            while ((nv >> 32) < (old >> 32)) {
              const unsigned long long seen = atomicCAS(&tc.vals[s2], old, nv);
              if (seen == old) { won = true; break; }
              old = seen;
            }
            if (won && atomicExch(&w.inq[s2], 1) == 0) {
              const int j = atomicAdd(&s_nfront[fb ^ 1], 1);
              if (j < max_tok) w.frontier[fb ^ 1][j] = s2; else s_err = 1;
            }
          }
        }
        __syncthreads();
        if (tid == 0) { s_nfront[fb] = 0; if (s_nfront[fb ^ 1] > max_tok) s_nfront[fb ^ 1] = max_tok; }
        fb ^= 1;
        __syncthreads();
        if (s_err) break;
      }
    }
    // word back-pointers (Decoder::InsertTok, src/decoder.cc:107-117): a token inherits the record of
    // the token its winning arc left from, plus one new record when that arc carries an output label
    for (int pass = 0; pass < 256; ++pass) {
      if (tid == 0) s_unres = 0;
      __syncthreads();
      const int n = min(s_ntok[c], max_tok);
      for (int i = tid; i < n; i += kVitThreads) {
        const int slot = tc.list[i];
        if (tc.bp[slot] != -2) continue;
        const uint32_t a = static_cast<uint32_t>(tc.vals[slot]);
        int pb;
        if (a == kNoArc) {
          pb = -1;  // the start token
        } else {
          const int src = __ldg(&fst.arc_src[a]);
          if (__ldg(&fst.arc_il[a]) != 0) {
            const int ps = tab_find(w.tab[p], src, mask);
            pb = ps >= 0 ? w.tab[p].bp[ps] : -1;
          } else {
            const int cs = tab_find(tc, src, mask);
            pb = cs >= 0 ? *reinterpret_cast<volatile int *>(&tc.bp[cs]) : -1;
            if (pb == -2) { atomicAdd(&s_unres, 1); continue; }
          }
          const int ol = __ldg(&fst.arc_ol[a]);
          if (ol != 0) {
            const int r = atomicAdd(&s_log, 1);
            if (r >= max_log) { s_err = 2; pb = -1; }
            else { w.log_prev[r] = pb; w.log_ol[r] = ol; pb = r; }
          }
        }
        tc.bp[slot] = pb;
      }
      __syncthreads();
      const int unres = s_unres;  // read by everyone before thread 0 may reset it in the next pass
      __syncthreads();
      if (unres == 0) break;
      if (pass == 255 && tid == 0) s_err = 3;
    }
    __syncthreads();
  };

  auto clear_tab = [&](int c) {
    const Tab &t = w.tab[c];
    const int n = min(s_ntok[c], max_tok);
    for (int i = tid; i < n; i += kVitThreads) {
      const int slot = t.list[i];
      t.keys[slot] = 0;
      t.vals[slot] = kEmptyVal;
      w.inq[slot] = 0;
    }
    __syncthreads();
    if (tid == 0) s_ntok[c] = 0;
    __syncthreads();
  };

  // lattice mode: group g of the log, the epsilon arcs of table c's final tokens under `cutoff`
  // (the closure's bound), in token-list order; lattice_prune sorts the kept ones
  auto lat_log_eps = [&](unsigned long long *lg, int *go, int c, int g, double cutoff) {
    LatShared &ls = lat_shared();
    if (tid == 0) go[g] = ls.count;
    __syncthreads();
    if (fst.has_eps) {
      const Tab &tc = w.tab[c];
      const int n = min(s_ntok[c], max_tok);
      for (int i = grp; i < n; i += kVitGroups) {
        const int slot = tc.list[i];
        const float cost = cost_of(tc.vals[slot]);
        const int state = tc.keys[slot] - 1;
        const int a1 = __ldg(&fst.arc_begin[state + 1]);
        for (int a = __ldg(&fst.arc_begin[state]) + gl; a < a1; a += kVitGroup) {
          if (__ldg(&fst.arc_il[a]) != 0) continue;
          if (static_cast<double>(cost) + static_cast<double>(__ldg(&fst.arc_w[a])) > cutoff) continue;
          const int r = atomicAdd(&ls.count, 1);
          if (r < lat.max_arcs) lg[r] = (static_cast<unsigned long long>(a) << 32) | __float_as_uint(cost);
        }
      }
    }
    __syncthreads();
    lat_check_overflow(lat, lerr);
  };

  // ---- BestPath (src/decoder.cc:300-339) of table c into utterance u's outputs
  auto best_path = [&](int u, int cb, bool alive) {
    if (tid == 0) s_min = ~0ull;
    __syncthreads();
    const Tab &tb = w.tab[cb];
    const int n = (alive && !s_err) ? min(s_ntok[cb], max_tok) : 0;
    for (int i = tid; i < n; i += kVitThreads) {
      const int slot = tb.list[i];
      const float c = cost_of(tb.vals[slot]) + fst.final_w[tb.keys[slot] - 1];
      if (c != INFINITY) atomicMin(&s_min, pack(c, static_cast<uint32_t>(slot)));
    }
    __syncthreads();
    if (tid == 0) {
      int32_t *wo = words_out + static_cast<size_t>(u) * max_words;
      if (s_err) {
        n_words_out[u] = -s_err;
        weight_out[u] = 0.0f;
      } else if (s_min == ~0ull) {
        n_words_out[u] = 0;  // no token in a final state: Hypothesis({}, 0)
        weight_out[u] = 0.0f;
      } else {
        const int slot = static_cast<int>(static_cast<uint32_t>(s_min));
        float weight = cost_of(s_min);
        weight += fst.final_w[tb.keys[slot] - 1];
        weight_out[u] = weight;
        int nw = 0;
        for (int r = tb.bp[slot]; r >= 0; r = w.log_prev[r]) ++nw;
        n_words_out[u] = nw;
        int k = nw;
        for (int r = tb.bp[slot]; r >= 0; r = w.log_prev[r]) {
          --k;
          if (k < max_words) wo[k] = w.log_ol[r];
        }
      }
    }
    if (kResume) carry_reset(cr, u);
    __syncthreads();
  };

  for (int u = blockIdx.x; u < n_utts; u += gridDim.x) {
    const int T = kResume ? (cr.finish ? 0 : num_frames ? num_frames[u] : cr.uniform_frames) : num_frames[u];
    const float *ll0 = loglik + (kResume ? static_cast<int64_t>(u) * cr.frame_stride : row_off[u]) * num_pdfs;
    const int *hdr = kResume ? cr.hdr + 4 * u : nullptr;
    const bool fresh = !kResume || hdr[0] < 0;
    // resumable lattice mode: frames of the utterance before this launch (all of them at a finish)
    // (clamped: a stream past max_frames has a lattice or a search error and logs nothing more)
    const int t0 = kResume && kLattice ? static_cast<int>(min(cr.frames[u], static_cast<long long>(lat.max_frames))) : 0;
    unsigned long long *lg = kLattice ? lat.log + static_cast<size_t>(u) * lat.max_arcs : nullptr;
    int *go = kLattice ? lat.grp + static_cast<size_t>(u) * lat.grp_stride + 2 * t0 : nullptr;
    if (kLattice && tid == 0) lat_shared().count = kResume && !fresh ? lat.state[2 * u] : 0;
    if (tid == 0) { s_ntok[0] = s_ntok[1] = 0; s_log = fresh ? 0 : hdr[1]; s_err = fresh ? 0 : hdr[2]; }
    if (kResume && kLattice && tid == 0) {
      const int e = fresh ? 0 : lat.state[2 * u + 1];
      s_laterr = e == 0 && s_err == 0 && t0 + T > lat.max_frames ? 5 : e;
    }
    __syncthreads();
    if (kResume && kLattice && lat_live()) {
      // this launch's rows, kept for the backward pass of the finish
      float *keep = lat.rows + (static_cast<size_t>(u) * lat.max_frames + t0) * num_pdfs;
      for (int64_t i = tid; i < static_cast<int64_t>(T) * num_pdfs; i += kVitThreads) keep[i] = ll0[i];
    }
    int cur = 0;
    if (fresh) {
      // ---- InitDecoding (src/decoder.cc:82-101): the start state at cost 0, then its epsilon closure
      if (tid == 0) {
        const int s = tab_insert(w.tab[0], fst.start, mask, &s_ntok[0], max_tok);
        w.tab[0].vals[s] = pack(0.0f, kNoArc);
      }
      __syncthreads();
      close_and_resolve(0, 1, INFINITY);
      if (kLattice && !s_err && lat_live()) lat_log_eps(lg, go, 0, 0, INFINITY);
    } else {
      // ---- the carried tokens of the previous advance
      const int n = hdr[2] ? 0 : hdr[0];
      const size_t base = static_cast<size_t>(u) * cr.cap;
      for (int i = tid; i < n; i += kVitThreads) {
        const int s = tab_insert(w.tab[0], cr.tok_state[base + i], mask, &s_ntok[0], max_tok);
        w.tab[0].vals[s] = pack(cr.tok_cost[base + i], kNoArc);
        w.tab[0].bp[s] = cr.tok_bp[base + i];
      }
      __syncthreads();
    }
    bool alive = fresh || hdr[3] != 0;

    for (int f = 0; f < T && alive && !s_err; ++f) {
      const int prev = cur;
      cur ^= 1;
      const Tab &tp = w.tab[prev], &tc = w.tab[cur];
      const int n_prev = s_ntok[prev];
      const float *ll = ll0 + static_cast<int64_t>(f) * num_pdfs;
      // ---- GetCutoff (src/decoder.cc:141-200) below kBeamSize tokens: best cost + beam
      if (tid == 0) s_min = ~0ull;
      __syncthreads();
      {
        uint32_t m = 0xffffffffu;
        for (int i = tid; i < n_prev; i += kVitThreads) m = min(m, static_cast<uint32_t>(tp.vals[tp.list[i]] >> 32));
        atomicMin(&s_min, static_cast<unsigned long long>(m));
      }
      __syncthreads();
      const float best = unord32(static_cast<uint32_t>(s_min));
      const float weight_cutoff = static_cast<float>(static_cast<double>(best) + static_cast<double>(beam));
      __syncthreads();
      // ---- ProcessEmitting, pass 1: the bound on the next frame (min over kept arcs of total + beam)
      if (tid == 0) s_min = ~0ull;
      __syncthreads();
      {
        // eight lanes per token, lanes over its arcs: 32 tokens of the block are in flight at once
        unsigned long long m = ~0ull;
        for (int i = grp; i < n_prev; i += kVitGroups) {
          const int slot = tp.list[i];
          const float cost = cost_of(tp.vals[slot]);
          if (cost > weight_cutoff) continue;
          const int state = tp.keys[slot] - 1;
          const int a1 = __ldg(&fst.arc_begin[state + 1]);
          for (int a = __ldg(&fst.arc_begin[state]) + gl; a < a1; a += kVitGroup) {
            const int il = __ldg(&fst.arc_il[a]);
            if (il == 0) continue;
            const int pdf = __ldg(&tid2pdf[il]);
            const float ac = -__ldg(&ll[pdf]);
            const double total = static_cast<double>(cost) + static_cast<double>(__ldg(&fst.arc_w[a])) +
                                 static_cast<double>(ac);
            m = min(m, ord64(total));
          }
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((tid & 31) == 0) atomicMin(&s_min, m);
      }
      __syncthreads();
      if (s_min == ~0ull) { alive = false; break; }  // no arc left the beam: the reference has no tokens either
      const double next_cutoff = unord64(s_min) + static_cast<double>(beam);
      const bool lat_on = kLattice && lat_live();
      if (lat_on) {
        if (tid == 0) go[2 * f + 1] = lat_shared().count;
        __syncthreads();
      }
      // ---- pass 2: create / improve the tokens of this frame
      for (int i = grp; i < n_prev; i += kVitGroups) {
        const int slot = tp.list[i];
        const float cost = cost_of(tp.vals[slot]);
        if (cost > weight_cutoff) continue;
        const int state = tp.keys[slot] - 1;
        const int a1 = __ldg(&fst.arc_begin[state + 1]);
        for (int a = __ldg(&fst.arc_begin[state]) + gl; a < a1; a += kVitGroup) {
          const int il = __ldg(&fst.arc_il[a]);
          if (il == 0) continue;
          const int pdf = __ldg(&tid2pdf[il]);
          const float ac = -__ldg(&ll[pdf]);
          const double total = static_cast<double>(cost) + static_cast<double>(__ldg(&fst.arc_w[a])) +
                               static_cast<double>(ac);
          if (total > next_cutoff) continue;
          if (lat_on) {
            const int r = atomicAdd(&lat_shared().count, 1);
            if (r < lat.max_arcs) lg[r] = (static_cast<unsigned long long>(a) << 32) | __float_as_uint(cost);
          }
          const int s2 = tab_insert(tc, __ldg(&fst.arc_dst[a]), mask, &s_ntok[cur], max_tok);
          if (s2 < 0) { s_err = 1; continue; }
          atomicMin(&tc.vals[s2], pack(static_cast<float>(total), static_cast<uint32_t>(a)));
        }
      }
      __syncthreads();
      if (kLattice && lat_live()) lat_check_overflow(lat, lerr);
      // ProcessEmitting returns the bound as a float (src/decoder.cc:240)
      if (!s_err) close_and_resolve(cur, prev, static_cast<double>(static_cast<float>(next_cutoff)));
      if (kLattice && !s_err && lat_live())
        lat_log_eps(lg, go, cur, 2 * (f + 1), static_cast<double>(static_cast<float>(next_cutoff)));
      clear_tab(prev);
    }

    if (kResume && !cr.finish) {
      const Tab &tb = w.tab[cur];
      const int n = (alive && !s_err) ? min(s_ntok[cur], max_tok) : 0;
      const size_t base = static_cast<size_t>(u) * cr.cap;
      for (int i = tid; i < n; i += kVitThreads) {
        const int slot = tb.list[i];
        cr.tok_state[base + i] = tb.keys[slot] - 1;
        cr.tok_cost[base + i] = cost_of(tb.vals[slot]);
        cr.tok_bp[base + i] = tb.bp[slot];
      }
      if (kLattice && tid == 0) {
        lat.state[2 * u] = lat_shared().count;
        lat.state[2 * u + 1] = s_laterr;
      }
      __syncthreads();
      carry_end_advance(cr, u, n, T, w.log_prev, w.log_ol, mark, max_log, max_words, s_log, s_err, alive);
    } else if (kLattice) {
      // best complete path: min over the final tokens of double(alpha) + double(final)
      LatShared &ls = lat_shared();
      if (tid == 0) {
        ls.best = ~0ull;
        // a stream with an error of either kind has no lattice: its groups may end past max_frames
        if (lat_live()) go[2 * T + 1] = ls.count;
      }
      __syncthreads();
      const Tab &tb = w.tab[cur];
      const int n = (alive && !s_err) ? min(s_ntok[cur], max_tok) : 0;
      for (int i = tid; i < n; i += kVitThreads) {
        const int slot = tb.list[i];
        const double c = static_cast<double>(cost_of(tb.vals[slot])) +
                         static_cast<double>(fst.final_w[tb.keys[slot] - 1]);
        if (c != INFINITY) atomicMin(&ls.best, ord64(c));
      }
      __syncthreads();
      if (kResume) best_path(u, cur, alive);  // a finish returns the words too
    } else {
      best_path(u, cur, alive);
    }
    if (s_err) {
      // a capacity overflow leaves claimed slots that are in no list: wipe both tables
      for (uint32_t i = tid; i < H; i += kVitThreads) {
        for (int k = 0; k < 2; ++k) {
          w.tab[k].keys[i] = 0;
          w.tab[k].vals[i] = kEmptyVal;
        }
        w.inq[i] = 0;
      }
      __syncthreads();
      if (tid == 0) s_ntok[0] = s_ntok[1] = 0;
      __syncthreads();
    } else {
      clear_tab(0);
      clear_tab(1);
    }
    if (kLattice && (!kResume || cr.finish)) {
      // backward pass with beta keyed by state in the two (clean) token tables; a finish reads the
      // utterance's t0 frames from the row store (ll0 with frame_stride = max_frames)
      const unsigned long long bst = lat_shared().best;
      const double best = bst == ~0ull ? INFINITY : unord64(bst);
      int kept = 0;
      if (!s_err && lat_live() && best != INFINITY) {
        auto reset = [&](int b) { clear_tab(b); };
        auto get = [&](int b, int s) -> double {
          const int sl = tab_find(w.tab[b], s, mask);
          if (sl < 0) return INFINITY;
          const unsigned long long v = *reinterpret_cast<volatile unsigned long long *>(&w.tab[b].vals[sl]);
          return v == kEmptyVal ? INFINITY : unord64(v);
        };
        auto relax = [&](int b, int s, double v) -> bool {
          const int sl = tab_insert(w.tab[b], s, mask, &s_ntok[b], max_tok);
          if (sl < 0) { s_err = 1; return false; }
          const unsigned long long o = ord64(v);
          return atomicMin(&w.tab[b].vals[sl], o) > o;
        };
        kept = lattice_prune(fst, lat, lg, go - 2 * t0, T + t0, ll0, num_pdfs, tid2pdf, best, true, &s_err, reset,
                             get, relax);
        if (s_err) {
          // an overflowing insert leaves a claimed slot in no list
          for (uint32_t i = tid; i < H; i += kVitThreads)
            for (int k = 0; k < 2; ++k) { w.tab[k].keys[i] = 0; w.tab[k].vals[i] = kEmptyVal; }
          __syncthreads();
          if (tid == 0) s_ntok[0] = s_ntok[1] = 0;
          __syncthreads();
        } else {
          clear_tab(0);
          clear_tab(1);
        }
      }
      if (tid == 0) {
        // a lattice error of the resumable search came first: the search's errors stop the logging
        const int e = kResume && s_laterr ? s_laterr : s_err;
        lat.n_out[u] = e ? -e : kept;
        lat.best_out[u] = e ? INFINITY : best;
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Small graphs (pocketkaldi's own territory: command / small-vocabulary grammars): every state has a
// slot, so the token table is three dense shared-memory arrays per frame and the search runs
// arc-parallel over the whole FST -- all lanes busy, 32-bit native shared-memory atomics, each
// thread keeps the totals of its arcs in registers across the passes of a frame.
//   cost[s]  ord32(token cost), kInactive when the state holds no token
//   warc[s]  winning arc; epsilon arcs carry bit 31 so that an emitting arc of equal cost wins, as
//            it does in the reference where emitting arcs are inserted first (src/decoder.cc:127-134)
//   bp[s]    newest word record of the token
constexpr uint32_t kInactive = 0xffffffffu;

template <int kArcsPerThread, bool kResume, bool kLattice>
__global__ void __launch_bounds__(kVitThreads, kArcsPerThread <= 8 ? 3 : 1)
viterbi_dense_kernel(FstDev fst, int num_arcs, float beam, int max_log, int max_words,
                     const float *__restrict__ loglik, int num_pdfs, const int64_t *__restrict__ row_off,
                     const int32_t *__restrict__ num_frames, int n_utts, const int32_t *__restrict__ tid2pdf,
                     char *work_base, size_t work_stride, int32_t *__restrict__ words_out,
                     int32_t *__restrict__ n_words_out, float *__restrict__ weight_out, Carry cr, Lattice lat) {
  extern __shared__ __align__(16) char s_dense[];
  __shared__ int s_log, s_err, s_unres, s_changed;
  __shared__ unsigned long long s_min;
  __shared__ unsigned int s_best;
  // resumable lattice mode: the lattice's own error (see viterbi_kernel)
  __shared__ int s_laterr;
  int *const lerr = kResume ? &s_laterr : &s_err;
  auto lat_live = [&]() { return !kResume || (!s_err && !s_laterr); };
  const int S = fst.num_states;
  uint32_t *cost[2], *warc[2];
  int *bp[2];
  {
    uint32_t *p = reinterpret_cast<uint32_t *>(s_dense);
    cost[0] = p; cost[1] = p + S; warc[0] = p + 2 * S; warc[1] = p + 3 * S;
    bp[0] = reinterpret_cast<int *>(p + 4 * S); bp[1] = reinterpret_cast<int *>(p + 5 * S);
  }
  int *log_prev = reinterpret_cast<int *>(work_base + static_cast<size_t>(blockIdx.x) * work_stride);
  int *log_ol = log_prev + max_log;
  const int tid = threadIdx.x;
  // acoustic costs of the frame, one slot per DISTINCT pdf the graph's arcs read (a word-loop
  // graph reads each pdf from ~15 arcs): bit set of used pdfs, its per-word prefix counts, the pdf
  // of every slot and two frames of costs
  const int W = (num_pdfs + 31) >> 5;
  const int Dmax = min(num_arcs, num_pdfs);
  uint32_t *s_bits = reinterpret_cast<uint32_t *>(s_dense) + 6 * S;
  int *s_wpre = reinterpret_cast<int *>(s_bits + W);
  int *s_pdf = s_wpre + W;
  float *s_ll = reinterpret_cast<float *>(s_pdf + Dmax);  // [2][Dmax]
  __shared__ int s_D;

  // this thread's arcs (the same in every pass of every frame)
  // source | destination << 16 (at most 2048 states; source 0xffff: no arc), weight, and the pdf
  // of an emitting arc (-1: epsilon arc)
  uint32_t a_sd[kArcsPerThread];
  float a_w[kArcsPerThread];
  int a_pdf[kArcsPerThread];
#pragma unroll
  for (int k = 0; k < kArcsPerThread; ++k) {
    const int a = tid + k * kVitThreads;
    const bool ok = a < num_arcs;
    a_sd[k] = ok ? (static_cast<uint32_t>(__ldg(&fst.arc_src[a])) | (static_cast<uint32_t>(__ldg(&fst.arc_dst[a])) << 16))
                 : 0xffffu;
    a_w[k] = ok ? __ldg(&fst.arc_w[a]) : 0.0f;
    const int il = ok ? __ldg(&fst.arc_il[a]) : 0;
    a_pdf[k] = (ok && il != 0) ? __ldg(&tid2pdf[il]) : -1;
  }
  auto src_of = [&](int k) { return static_cast<int>(a_sd[k] & 0xffffu); };
  auto dst_of = [&](int k) { return static_cast<int>(a_sd[k] >> 16); };
  auto has_arc = [&](int k) { return (a_sd[k] & 0xffffu) != 0xffffu; };
  // slots of the distinct pdfs; a_pdf[k] becomes the slot of arc k's pdf
  for (int w = tid; w < W; w += kVitThreads) s_bits[w] = 0u;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kArcsPerThread; ++k)
    if (a_pdf[k] >= 0) atomicOr(&s_bits[a_pdf[k] >> 5], 1u << (a_pdf[k] & 31));
  __syncthreads();
  if (tid < 32) {
    int running = 0;
    for (int base = 0; base < W; base += 32) {
      const int w = base + tid;
      const int cnt = w < W ? __popc(s_bits[w]) : 0;
      int inc = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (tid >= o) inc += t;
      }
      if (w < W) s_wpre[w] = running + inc - cnt;
      running += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (tid == 0) s_D = running;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kArcsPerThread; ++k) {
    if (a_pdf[k] < 0) continue;
    const int pdf = a_pdf[k];
    const int slot = s_wpre[pdf >> 5] + __popc(s_bits[pdf >> 5] & ((1u << (pdf & 31)) - 1u));
    s_pdf[slot] = pdf;  // every arc of the pdf writes the same value
    a_pdf[k] = slot;
  }
  __syncthreads();
  const int D = s_D;
  // The acoustic costs of the NEXT frame are loaded (one load per distinct pdf) while the current
  // frame is searched: the row's DRAM latency is off the critical path of the frame step.

  // epsilon closure of frame table c under `cutoff`, winners, word back-pointers
  auto finish_frame = [&](int c, int p, double cutoff, const double (&td)[kArcsPerThread], const bool (&live)[kArcsPerThread]) {
    if (fst.has_eps) {
      for (int round = 0; round < 4096; ++round) {
        if (tid == 0) s_changed = 0;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kArcsPerThread; ++k) {
          if (!has_arc(k) || a_pdf[k] >= 0) continue;
          const uint32_t cs = *reinterpret_cast<volatile uint32_t *>(&cost[c][src_of(k)]);
          if (cs == kInactive) continue;
          const double total = static_cast<double>(unord32(cs)) + static_cast<double>(a_w[k]);
          if (total > cutoff) continue;
          const uint32_t o = ord32(static_cast<float>(total));
          if (atomicMin(&cost[c][dst_of(k)], o) > o) s_changed = 1;
        }
        __syncthreads();
        const int changed = s_changed;  // read by everyone before thread 0 resets it
        __syncthreads();
        if (!changed) break;
      }
    }
    // winners against the final costs: emitting arcs from the totals kept in registers, epsilon
    // arcs from their source's final cost
#pragma unroll
    for (int k = 0; k < kArcsPerThread; ++k) {
      if (!has_arc(k)) continue;
      const uint32_t a = static_cast<uint32_t>(tid + k * kVitThreads);
      if (a_pdf[k] >= 0) {
        if (live[k] && ord32(static_cast<float>(td[k])) == cost[c][dst_of(k)]) atomicMin(&warc[c][dst_of(k)], a);
      } else if (fst.has_eps) {
        const uint32_t cs = cost[c][src_of(k)];
        if (cs == kInactive) continue;
        const double total = static_cast<double>(unord32(cs)) + static_cast<double>(a_w[k]);
        if (total <= cutoff && ord32(static_cast<float>(total)) == cost[c][dst_of(k)])
          atomicMin(&warc[c][dst_of(k)], a | 0x80000000u);
      }
    }
    __syncthreads();
    // word back-pointers (Decoder::InsertTok, src/decoder.cc:107-117)
    for (int s = tid; s < S; s += kVitThreads) bp[c][s] = cost[c][s] != kInactive ? -2 : -1;
    for (int pass = 0; pass < 256; ++pass) {
      if (tid == 0) s_unres = 0;
      __syncthreads();
      for (int s = tid; s < S; s += kVitThreads) {
        if (bp[c][s] != -2) continue;
        const uint32_t wa = warc[c][s];
        int pb;
        if (wa == kInactive) {
          pb = -1;  // the start token
        } else {
          const int a = static_cast<int>(wa & 0x7fffffffu);
          const int src = __ldg(&fst.arc_src[a]);
          if (wa >> 31) {
            pb = *reinterpret_cast<volatile int *>(&bp[c][src]);
            if (pb == -2) { atomicAdd(&s_unres, 1); continue; }
          } else {
            pb = bp[p][src];
          }
          const int ol = __ldg(&fst.arc_ol[a]);
          if (ol != 0) {
            const int r = atomicAdd(&s_log, 1);
            if (r >= max_log) { s_err = 2; pb = -1; }
            else { log_prev[r] = pb; log_ol[r] = ol; pb = r; }
          }
        }
        bp[c][s] = pb;
      }
      __syncthreads();
      const int unres = s_unres;
      __syncthreads();
      if (unres == 0) break;
      if (pass == 255 && tid == 0) s_err = 3;
    }
    __syncthreads();
  };

  // Closes a frame: clears the previous table, reduces the best cost of the new one (the next
  // frame's GetCutoff) and re-arms the two shared minima. Everyone is past a barrier on entry.
  auto end_frame = [&](int c, int p) {
    if (tid == 0) {
      s_best = kInactive;
      s_min = ~0ull;
    }
    __syncthreads();
    uint32_t m = kInactive;
    for (int s = tid; s < S; s += kVitThreads) {
      cost[p][s] = kInactive;
      warc[p][s] = kInactive;
      m = min(m, cost[c][s]);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0 && m != kInactive) atomicMin(&s_best, m);
    __syncthreads();
  };

  // lattice mode: group g of the log, the emitting arcs still live after pass 2 (source costs in
  // table p) or the epsilon arcs of table c's final tokens under `cutoff`, in arc order
  auto lat_log = [&](unsigned long long *lg, int *go, int g, int tab, bool emitting, double cutoff,
                     const bool (&live)[kArcsPerThread]) {
    bool flag[kArcsPerThread];
    float alpha[kArcsPerThread];
#pragma unroll
    for (int k = 0; k < kArcsPerThread; ++k) {
      const uint32_t cs = has_arc(k) ? cost[tab][src_of(k)] : kInactive;
      alpha[k] = unord32(cs);
      if (emitting) flag[k] = live[k];
      else flag[k] = fst.has_eps && has_arc(k) && a_pdf[k] < 0 && cs != kInactive &&
                     static_cast<double>(alpha[k]) + static_cast<double>(a_w[k]) <= cutoff;
    }
    lat_append_ordered<kArcsPerThread>(lat, lg, go, g, flag, alpha, lerr);
  };

  // ---- BestPath (src/decoder.cc:300-339) of table c into utterance u's outputs
  auto best_path = [&](int u, int c, bool alive) {
    if (tid == 0) s_min = ~0ull;
    __syncthreads();
    if (alive && !s_err) {
      for (int s = tid; s < S; s += kVitThreads) {
        if (cost[c][s] == kInactive) continue;
        const float cs = unord32(cost[c][s]) + fst.final_w[s];
        if (cs != INFINITY) atomicMin(&s_min, pack(cs, static_cast<uint32_t>(s)));
      }
    }
    __syncthreads();
    if (tid == 0) {
      int32_t *wo = words_out + static_cast<size_t>(u) * max_words;
      if (s_err) {
        n_words_out[u] = -s_err;
        weight_out[u] = 0.0f;
      } else if (s_min == ~0ull) {
        n_words_out[u] = 0;
        weight_out[u] = 0.0f;
      } else {
        const int s = static_cast<int>(static_cast<uint32_t>(s_min));
        float weight = cost_of(s_min);
        weight += fst.final_w[s];
        weight_out[u] = weight;
        int nw = 0;
        for (int r = bp[c][s]; r >= 0; r = log_prev[r]) ++nw;
        n_words_out[u] = nw;
        int k = nw;
        for (int r = bp[c][s]; r >= 0; r = log_prev[r]) {
          --k;
          if (k < max_words) wo[k] = log_ol[r];
        }
      }
    }
    if (kResume) carry_reset(cr, u);
    __syncthreads();
  };

  for (int u = blockIdx.x; u < n_utts; u += gridDim.x) {
    const int T = kResume ? (cr.finish ? 0 : num_frames ? num_frames[u] : cr.uniform_frames) : num_frames[u];
    const float *ll0 = loglik + (kResume ? static_cast<int64_t>(u) * cr.frame_stride : row_off[u]) * num_pdfs;
    const int *hdr = kResume ? cr.hdr + 4 * u : nullptr;
    const bool fresh = !kResume || hdr[0] < 0;
    // resumable lattice mode: frames of the utterance before this launch (all of them at a finish)
    // (clamped: a stream past max_frames has a lattice or a search error and logs nothing more)
    const int t0 = kResume && kLattice ? static_cast<int>(min(cr.frames[u], static_cast<long long>(lat.max_frames))) : 0;
    unsigned long long *lg = kLattice ? lat.log + static_cast<size_t>(u) * lat.max_arcs : nullptr;
    int *go = kLattice ? lat.grp + static_cast<size_t>(u) * lat.grp_stride + 2 * t0 : nullptr;
    for (int s = tid; s < S; s += kVitThreads) {
      cost[0][s] = cost[1][s] = kInactive;
      warc[0][s] = warc[1][s] = kInactive;
      bp[0][s] = bp[1][s] = -1;
    }
    if (kLattice && tid == 0) lat_shared().count = kResume && !fresh ? lat.state[2 * u] : 0;
    if (tid == 0) { s_log = fresh ? 0 : hdr[1]; s_err = fresh ? 0 : hdr[2]; }
    if (kResume && kLattice && tid == 0) {
      const int e = fresh ? 0 : lat.state[2 * u + 1];
      s_laterr = e == 0 && s_err == 0 && t0 + T > lat.max_frames ? 5 : e;
    }
    __syncthreads();
    int cur = 0;
    if (fresh) {
      // ---- InitDecoding (src/decoder.cc:82-101)
      if (tid == 0) cost[0][fst.start] = ord32(0.0f);
    } else if (hdr[2] == 0) {
      // ---- the carried tokens of the previous advance
      const size_t base = static_cast<size_t>(u) * cr.cap;
      for (int i = tid; i < hdr[0]; i += kVitThreads) {
        const int s = cr.tok_state[base + i];
        cost[0][s] = ord32(cr.tok_cost[base + i]);
        bp[0][s] = cr.tok_bp[base + i];
      }
    }
    if (T > 0)
      for (int d = tid; d < D; d += kVitThreads) s_ll[d] = __ldg(&ll0[s_pdf[d]]);
    __syncthreads();
    if (kResume && kLattice && lat_live()) {
      // this launch's rows, kept for the backward pass of the finish
      float *keep = lat.rows + (static_cast<size_t>(u) * lat.max_frames + t0) * num_pdfs;
      for (int64_t i = tid; i < static_cast<int64_t>(T) * num_pdfs; i += kVitThreads) keep[i] = ll0[i];
    }
    if (fresh) {
      double td[kArcsPerThread];
      bool live[kArcsPerThread];
#pragma unroll
      for (int k = 0; k < kArcsPerThread; ++k) { td[k] = 0.0; live[k] = false; }
      finish_frame(0, 1, INFINITY, td, live);
      if (kLattice && lat_live()) lat_log(lg, go, 0, 0, false, INFINITY, live);
    }
    end_frame(0, 1);
    bool alive = fresh || hdr[3] != 0;
    for (int f = 0; f < T && alive && !s_err; ++f) {
      const int prev = cur;
      cur ^= 1;
      const float *ll_cur = s_ll + (f & 1) * Dmax;
      float ll_next[kArcsPerThread];  // D <= num_arcs <= kArcsPerThread * kVitThreads
      {
        const float *lln = ll0 + static_cast<int64_t>(f + 1) * num_pdfs;
#pragma unroll
        for (int k = 0; k < kArcsPerThread; ++k) {
          const int d = tid + k * kVitThreads;
          ll_next[k] = (f + 1 < T && d < D) ? __ldg(&lln[s_pdf[d]]) : 0.0f;
        }
      }
      // ---- GetCutoff below kBeamSize tokens: the best cost was reduced when the table was finished
      if (s_best == kInactive) { alive = false; break; }
      const float weight_cutoff = static_cast<float>(static_cast<double>(unord32(s_best)) + static_cast<double>(beam));
      // ---- ProcessEmitting, pass 1: totals of this thread's arcs, bound on the next frame
      double td[kArcsPerThread];
      bool live[kArcsPerThread];
      {
        unsigned long long m = ~0ull;
#pragma unroll
        for (int k = 0; k < kArcsPerThread; ++k) {
          live[k] = false;
          td[k] = 0.0;
          if (a_pdf[k] < 0) continue;
          const uint32_t cs = cost[prev][src_of(k)];
          if (cs == kInactive) continue;
          const float c = unord32(cs);
          if (c > weight_cutoff) continue;
          const float ac = -ll_cur[a_pdf[k]];
          td[k] = static_cast<double>(c) + static_cast<double>(a_w[k]) + static_cast<double>(ac);
          live[k] = true;
          m = min(m, ord64(td[k]));
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((tid & 31) == 0) atomicMin(&s_min, m);
      }
      __syncthreads();
      if (s_min == ~0ull) { alive = false; break; }
      const double next_cutoff = unord64(s_min) + static_cast<double>(beam);
      // ---- pass 2: token costs of this frame
#pragma unroll
      for (int k = 0; k < kArcsPerThread; ++k) {
        live[k] = live[k] && td[k] <= next_cutoff;
        if (live[k]) atomicMin(&cost[cur][dst_of(k)], ord32(static_cast<float>(td[k])));
      }
      __syncthreads();
      if (kLattice && lat_live()) lat_log(lg, go, 2 * f + 1, prev, true, 0.0, live);
      finish_frame(cur, prev, static_cast<double>(static_cast<float>(next_cutoff)), td, live);
      if (kLattice && lat_live())
        lat_log(lg, go, 2 * (f + 1), cur, false, static_cast<double>(static_cast<float>(next_cutoff)), live);
      {
        float *ll_nx = s_ll + ((f + 1) & 1) * Dmax;  // last read two frames ago
#pragma unroll
        for (int k = 0; k < kArcsPerThread; ++k) {
          const int d = tid + k * kVitThreads;
          if (d < D) ll_nx[d] = ll_next[k];
        }
      }
      end_frame(cur, prev);
    }

    if (kResume && !cr.finish) {
      __shared__ int s_nsave;
      if (tid == 0) s_nsave = 0;
      __syncthreads();
      if (alive && !s_err) {
        const size_t base = static_cast<size_t>(u) * cr.cap;
        for (int s = tid; s < S; s += kVitThreads) {
          if (cost[cur][s] == kInactive) continue;
          const int i = atomicAdd(&s_nsave, 1);
          cr.tok_state[base + i] = s;
          cr.tok_cost[base + i] = unord32(cost[cur][s]);
          cr.tok_bp[base + i] = bp[cur][s];
        }
      }
      if (kLattice && tid == 0) {
        lat.state[2 * u] = lat_shared().count;
        lat.state[2 * u + 1] = s_laterr;
      }
      __syncthreads();
      carry_end_advance(cr, u, s_nsave, T, log_prev, log_ol, log_ol + max_log, max_log, max_words, s_log, s_err,
                        alive);
      continue;
    }
    if (kLattice) {
      // best complete path: min over the final tokens of double(alpha) + double(final)
      LatShared &ls = lat_shared();
      if (tid == 0) {
        ls.best = ~0ull;
        // a stream with an error of either kind has no lattice: its groups may end past max_frames
        if (lat_live()) go[2 * T + 1] = ls.count;
      }
      __syncthreads();
      if (alive && !s_err)
        for (int s = tid; s < S; s += kVitThreads) {
          if (cost[cur][s] == kInactive) continue;
          const double c = static_cast<double>(unord32(cost[cur][s])) + static_cast<double>(fst.final_w[s]);
          if (c != INFINITY) atomicMin(&ls.best, ord64(c));
        }
      __syncthreads();
      const double best = ls.best == ~0ull ? INFINITY : unord64(ls.best);
      if (kResume) best_path(u, cur, alive);  // a finish returns the words too, before beta takes the arrays
      int kept = 0;
      if (alive && !s_err && lat_live() && best != INFINITY) {
        // backward pass with beta in the cost / warc arrays the search is done with: 2 S doubles;
        // a finish reads the utterance's t0 frames from the row store (ll0 with frame_stride = max_frames)
        unsigned long long *bt = reinterpret_cast<unsigned long long *>(s_dense);
        auto reset = [&](int b) {
          for (int s = tid; s < S; s += kVitThreads) bt[b * S + s] = kEmptyVal;
          __syncthreads();
        };
        auto get = [&](int b, int s) -> double {
          const unsigned long long v = *reinterpret_cast<volatile unsigned long long *>(&bt[b * S + s]);
          return v == kEmptyVal ? INFINITY : unord64(v);
        };
        auto relax = [&](int b, int s, double v) -> bool {
          const unsigned long long o = ord64(v);
          return atomicMin(&bt[b * S + s], o) > o;
        };
        kept = lattice_prune(fst, lat, lg, go - 2 * t0, T + t0, ll0, num_pdfs, tid2pdf, best, false, &s_err, reset,
                             get, relax);
      }
      if (tid == 0) {
        const int e = kResume && s_laterr ? s_laterr : s_err;  // as in viterbi_kernel
        lat.n_out[u] = e ? -e : kept;
        lat.best_out[u] = e ? INFINITY : best;
      }
      __syncthreads();
      continue;
    }
    best_path(u, cur, alive);
  }
}

// The kept arcs of utterance u (lattice_prune's keys) as records from out + first[u] on.
__global__ void __launch_bounds__(kVitThreads)
lattice_expand_kernel(FstDev fst, Lattice lat, const float *__restrict__ loglik, int num_pdfs,
                      const int64_t *__restrict__ row_off, const int32_t *__restrict__ tid2pdf,
                      const long long *__restrict__ first, pkb_lattice_arc_t *__restrict__ out) {
  const int u = blockIdx.x;
  const long long n = lat.n_out[u];
  const unsigned long long *lg = lat.log + static_cast<size_t>(u) * lat.max_arcs;
  pkb_lattice_arc_t *o = out + first[u];
  for (long long i = threadIdx.x; i < n; i += kVitThreads) {
    const unsigned long long key = lg[i];
    const int t = static_cast<int>(key >> 33), a = static_cast<int>(key & 0xffffffffull);
    const int il = __ldg(&fst.arc_il[a]);
    pkb_lattice_arc_t r;
    r.t = t;
    r.src = __ldg(&fst.arc_src[a]);
    r.dst = __ldg(&fst.arc_dst[a]);
    r.ilabel = il;
    r.olabel = __ldg(&fst.arc_ol[a]);
    r.graph_cost = __ldg(&fst.arc_w[a]);
    r.acoustic_cost = il ? -__ldg(&loglik[(row_off[u] + t) * num_pdfs + __ldg(&tid2pdf[il])]) : 0.0f;
    o[i] = r;
  }
}

// the two value arrays lead every block's workspace
__global__ void viterbi_init_kernel(char *work_base, size_t work_stride, uint32_t n) {
  unsigned long long *vals = reinterpret_cast<unsigned long long *>(work_base + work_stride * blockIdx.y);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    vals[i] = kEmptyVal;
}

}  // namespace

int fst_build(Ctx *c, int num_states, int start, const float *final_w, const int32_t *first_arc,
              int num_arcs, const int32_t *arcs_raw, pkb_fst **out) {
  PKB_REQUIRE(c && out, "pkb_fst: NULL argument");
  PKB_REQUIRE(num_states > 0 && num_arcs >= 0, "pkb_fst: %d states, %d arcs", num_states, num_arcs);
  PKB_REQUIRE(start >= 0 && start < num_states, "pkb_fst: start state %d out of range", start);
  PKB_REQUIRE(final_w && first_arc && (arcs_raw || num_arcs == 0), "pkb_fst: NULL table");
  // arcs of state s: [first_arc[s], first arc of the next state that has arcs) -- Fst::CountArcs,
  // src/fst.cc:94-110
  std::vector<int32_t> begin(num_states + 1, num_arcs), src(num_arcs, 0);
  int32_t next = num_arcs;
  for (int s = num_states - 1; s >= 0; --s) {
    if (first_arc[s] >= 0) {
      PKB_REQUIRE(first_arc[s] <= next, "pkb_fst: arcs are not sorted by source state (state %d)", s);
      begin[s] = first_arc[s];
      next = first_arc[s];
    } else {
      begin[s] = next;
    }
  }
  bool has_eps = false;
  int max_il = 0;
  std::vector<int32_t> dst(num_arcs), il(num_arcs), ol(num_arcs);
  std::vector<float> wt(num_arcs);
  for (int s = 0; s < num_states; ++s)
    for (int a = begin[s]; a < begin[s + 1]; ++a) src[a] = s;
  for (int a = 0; a < num_arcs; ++a) {
    dst[a] = arcs_raw[4 * a];
    il[a] = arcs_raw[4 * a + 1];
    ol[a] = arcs_raw[4 * a + 2];
    memcpy(&wt[a], &arcs_raw[4 * a + 3], sizeof(float));
    PKB_REQUIRE(dst[a] >= 0 && dst[a] < num_states, "pkb_fst: arc %d leads to state %d", a, dst[a]);
    PKB_REQUIRE(il[a] >= 0, "pkb_fst: arc %d has a negative input label", a);
    has_eps = has_eps || il[a] == 0;
    max_il = std::max(max_il, il[a]);
  }
  std::unique_ptr<pkb_fst, decltype(&pkb_fst_destroy)> f(new pkb_fst(), pkb_fst_destroy);
  f->c = c;
  f->num_states = num_states;
  f->num_arcs = num_arcs;
  f->start = start;
  f->has_eps = has_eps;
  f->max_ilabel = max_il;
  const size_t n1 = static_cast<size_t>(num_states) + 1, na = std::max(num_arcs, 1);
  const size_t bytes = 4 * (static_cast<size_t>(num_states) + n1 + 5 * na);
  std::vector<char> host(bytes, 0);
  char *h = host.data();
  size_t o_fin = 0, o_beg = o_fin + 4 * num_states, o_src = o_beg + 4 * n1, o_dst = o_src + 4 * na,
         o_il = o_dst + 4 * na, o_ol = o_il + 4 * na, o_w = o_ol + 4 * na;
  memcpy(h + o_fin, final_w, 4 * static_cast<size_t>(num_states));
  memcpy(h + o_beg, begin.data(), 4 * n1);
  if (num_arcs) {
    memcpy(h + o_src, src.data(), 4 * static_cast<size_t>(num_arcs));
    memcpy(h + o_dst, dst.data(), 4 * static_cast<size_t>(num_arcs));
    memcpy(h + o_il, il.data(), 4 * static_cast<size_t>(num_arcs));
    memcpy(h + o_ol, ol.data(), 4 * static_cast<size_t>(num_arcs));
    memcpy(h + o_w, wt.data(), 4 * static_cast<size_t>(num_arcs));
  }
  PKB_TRY(f->buf.ensure(bytes));
  PKB_TRY(upload(c, f->buf.p, h, bytes));
  const char *d = f->buf.as<char>();
  f->d_final = reinterpret_cast<const float *>(d + o_fin);
  f->d_arc_begin = reinterpret_cast<const int32_t *>(d + o_beg);
  f->d_arc_src = reinterpret_cast<const int32_t *>(d + o_src);
  f->d_arc_dst = reinterpret_cast<const int32_t *>(d + o_dst);
  f->d_arc_il = reinterpret_cast<const int32_t *>(d + o_il);
  f->d_arc_ol = reinterpret_cast<const int32_t *>(d + o_ol);
  f->d_arc_w = reinterpret_cast<const float *>(d + o_w);
  *out = f.release();
  return PKB_OK;
}

namespace {

FstDev fst_dev(const pkb_fst *fst) {
  FstDev fd;
  fd.num_states = fst->num_states;
  fd.start = fst->start;
  fd.has_eps = fst->has_eps ? 1 : 0;
  fd.final_w = fst->d_final;
  fd.arc_begin = fst->d_arc_begin;
  fd.arc_src = fst->d_arc_src;
  fd.arc_dst = fst->d_arc_dst;
  fd.arc_il = fst->d_arc_il;
  fd.arc_ol = fst->d_arc_ol;
  fd.arc_w = fst->d_arc_w;
  return fd;
}

// Kernel, token capacity and workspace of a search over `fst`. The resumable search keeps its blocks'
// compaction marks after the word records (log_arrays = 3 instead of 2) and runs one block per stream.
VitPlan plan_viterbi(const Ctx *c, const pkb_fst *fst, const ViterbiConfig &cfg, int num_pdfs, int n_utts,
                     bool resume) {
  VitPlan p;
  const size_t log_bytes = (resume ? 3 : 2) * sizeof(int) * static_cast<size_t>(cfg.max_log);
  p.dense = fst->num_states <= 2048 && fst->num_arcs <= 16 * kVitThreads;
  if (p.dense) {
    // dense kernel: no token capacity to run out of; the global workspace holds the word records only
    p.max_tok = fst->num_states;
    p.stride = (log_bytes + 255) & ~static_cast<size_t>(255);
    // one resident wave at most (the workspace is per block); the kernels are built for three
    // blocks per SM up to eight arcs per thread
    p.grid = resume ? n_utts : std::min(n_utts, c->sm_count * 4);
    p.smem = sizeof(uint32_t) * (6 * static_cast<size_t>(fst->num_states) +
                                 2 * static_cast<size_t>((num_pdfs + 31) / 32) +
                                 3 * static_cast<size_t>(std::min(fst->num_arcs, num_pdfs)));
    p.variant = fst->num_arcs <= 4 * kVitThreads ? 4 : fst->num_arcs <= 8 * kVitThreads ? 8 : 16;
    return p;
  }
  // a graph with at most 512 states can never hold more tokens than states: its tables go to
  // shared memory (capacity = the state count), whatever max_tokens says
  p.small = fst->num_states <= 512;
  p.max_tok = p.small ? std::max(16, fst->num_states) : cfg.max_tokens;
  p.H = 64;
  while (p.H < 2u * static_cast<uint32_t>(p.max_tok)) p.H <<= 1;
  const size_t table_bytes = 2 * sizeof(unsigned long long) * p.H +
                             2 * (2 * sizeof(int) * p.H + 2 * sizeof(int) * p.max_tok) + sizeof(int) * p.H;
  const size_t stride_raw = (p.small ? 0 : table_bytes) + log_bytes;
  p.stride = (stride_raw + 255) & ~static_cast<size_t>(255);
  // persistent blocks: a few per SM, each walking its share of the utterances with one workspace
  p.grid = resume ? n_utts : std::min(n_utts, c->sm_count * 8);
  p.smem = p.small ? table_bytes : 0;
  p.variant = static_cast<double>(fst->num_arcs) >= 12.0 * fst->num_states ? 32 : 8;
  return p;
}

// Invariant the table kernel relies on (and restores per utterance): keys 0, values empty, queue
// flags 0. The dense kernel's workspace needs nothing; the resumable search's marks start at 0.
int init_workspace(Ctx *c, const VitPlan &p, DevBuf *work) {
  const size_t bytes = p.stride * p.grid;
  PKB_CUDA(cudaMemsetAsync(work->p, 0, bytes, c->stream));
  if (!p.dense && !p.small) {
    LaunchScope scope(c, PKB_KERNEL_MISC);
    viterbi_init_kernel<<<dim3(4, p.grid), 256, 0, c->stream>>>(work->as<char>(), p.stride, 2 * p.H);
    PKB_CUDA(cudaGetLastError());
  }
  return PKB_OK;
}

template <bool kResume, bool kLattice>
int launch_plan(Ctx *c, const pkb_fst *fst, const VitPlan &p, const ViterbiConfig &cfg, const float *d_loglik,
                int num_pdfs, const int64_t *d_row_off, const int32_t *d_num_frames, int n_utts,
                const int32_t *d_tid2pdf, DevBuf *work, int32_t *d_words, int32_t *d_n_words, float *d_weight,
                const Carry &cr, const Lattice &lat) {
  const FstDev fd = fst_dev(fst);
  LaunchScope scope(c, PKB_KERNEL_MISC);
#define PKB_VIT_DENSE(APT)                                                                                   \
  do {                                                                                                       \
    if (p.smem > 48 * 1024)                                                                                  \
      PKB_CUDA(cudaFuncSetAttribute(viterbi_dense_kernel<APT, kResume, kLattice>,                            \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(p.smem))); \
    viterbi_dense_kernel<APT, kResume, kLattice><<<p.grid, kVitThreads, p.smem, c->stream>>>(                \
        fd, fst->num_arcs, cfg.beam, cfg.max_log, cfg.max_words, d_loglik, num_pdfs, d_row_off,              \
        d_num_frames, n_utts, d_tid2pdf, work->as<char>(), p.stride, d_words, d_n_words, d_weight, cr, lat); \
  } while (0)
  // (staging each frame's log-likelihood row in shared memory with cp.async was measured slower in
  // the table kernel, 44 vs 26 ms for 128 utterances: the larger carve-out takes the L1 space that
  // keeps the FST hot)
#define PKB_VIT_LAUNCH(G)                                                                                    \
  do {                                                                                                       \
    if (p.smem > 48 * 1024)                                                                                  \
      PKB_CUDA(cudaFuncSetAttribute(viterbi_kernel<G, kResume, kLattice>,                                    \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(p.smem))); \
    viterbi_kernel<G, kResume, kLattice><<<p.grid, kVitThreads, p.smem, c->stream>>>(                        \
        fd, cfg.beam, p.max_tok, p.H - 1, cfg.max_log, cfg.max_words, d_loglik, num_pdfs, d_row_off,         \
        d_num_frames, n_utts, d_tid2pdf, work->as<char>(), p.stride, p.small ? 1 : 0, d_words, d_n_words,    \
        d_weight, cr, lat);                                                                                  \
  } while (0)
  if (p.dense) {
    if (p.variant == 4) PKB_VIT_DENSE(4);
    else if (p.variant == 8) PKB_VIT_DENSE(8);
    else PKB_VIT_DENSE(16);
  } else {
    if (p.variant == 32) PKB_VIT_LAUNCH(32);
    else PKB_VIT_LAUNCH(8);
  }
#undef PKB_VIT_DENSE
#undef PKB_VIT_LAUNCH
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

}  // namespace

int launch_viterbi(Ctx *c, const pkb_fst *fst, const ViterbiConfig &cfg, const float *d_loglik,
                   int num_pdfs, const int64_t *d_row_off, const int32_t *d_num_frames, int n_utts,
                   const int32_t *d_tid2pdf, int n_tids, DevBuf *work, int32_t *d_words,
                   int32_t *d_n_words, float *d_weight) {
  (void)n_tids;
  if (n_utts == 0) return PKB_OK;
  PKB_REQUIRE(cfg.max_tokens >= 16 && cfg.max_log >= 16 && cfg.max_words >= 1 && cfg.beam > 0.0f,
              "pkb_batch_decode: bad configuration");
  const VitPlan p = plan_viterbi(c, fst, cfg, num_pdfs, n_utts, false);
  PKB_TRY(work->ensure(p.stride * p.grid));
  if (!p.dense && !p.small) PKB_TRY(init_workspace(c, p, work));
  return launch_plan<false, false>(c, fst, p, cfg, d_loglik, num_pdfs, d_row_off, d_num_frames, n_utts, d_tid2pdf,
                                   work, d_words, d_n_words, d_weight, Carry{}, Lattice{});
}

int launch_lattice(Ctx *c, const pkb_fst *fst, const ViterbiConfig &cfg, const float *d_loglik, int num_pdfs,
                   const int64_t *d_row_off, const int32_t *d_num_frames, int n_utts, const int32_t *d_tid2pdf,
                   DevBuf *work, const Lattice &lat) {
  if (n_utts == 0) return PKB_OK;
  PKB_REQUIRE(cfg.max_tokens >= 16 && cfg.max_log >= 16 && cfg.beam > 0.0f && lat.max_arcs > 0 && lat.beam > 0.0f,
              "pkb_batch_lattice: bad configuration");
  const VitPlan p = plan_viterbi(c, fst, cfg, num_pdfs, n_utts, false);
  PKB_TRY(work->ensure(p.stride * p.grid));
  if (!p.dense && !p.small) PKB_TRY(init_workspace(c, p, work));
  return launch_plan<false, true>(c, fst, p, cfg, d_loglik, num_pdfs, d_row_off, d_num_frames, n_utts, d_tid2pdf,
                                  work, nullptr, nullptr, nullptr, Carry{}, lat);
}

int lattice_expand(Ctx *c, const pkb_fst *fst, const Lattice &lat, const float *d_loglik, int num_pdfs,
                   const int64_t *d_row_off, int n_utts, const int32_t *d_tid2pdf, const long long *d_first,
                   pkb_lattice_arc_t *d_out) {
  if (n_utts == 0) return PKB_OK;
  LaunchScope scope(c, PKB_KERNEL_MISC);
  lattice_expand_kernel<<<n_utts, kVitThreads, 0, c->stream>>>(fst_dev(fst), lat, d_loglik, num_pdfs, d_row_off,
                                                               d_tid2pdf, d_first, d_out);
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

int ResumableSearch::setup(Ctx *ctx, const pkb_fst *graph, const ViterbiConfig &config, const int32_t *tid2pdf,
                           int n_tids, int pdfs, int streams) {
  PKB_REQUIRE(config.max_tokens >= 16 && config.max_log >= 16 && config.max_words >= 1 && config.beam > 0.0f,
              "pkb_decoder_create: bad configuration");
  c = ctx;
  fst = graph;
  cfg = config;
  num_pdfs = pdfs;
  n = streams;
  plan = plan_viterbi(c, fst, cfg, num_pdfs, n, true);
  PKB_TRY(work.ensure(plan.stride * plan.grid));
  PKB_TRY(init_workspace(c, plan, &work));
  const size_t S = n, cap = plan.max_tok, mw = cfg.max_words;
  // carry: frames, header, tokens
  PKB_TRY(carry.ensure(S * (sizeof(long long) + 4 * sizeof(int) + cap * 3 * sizeof(int))));
  char *p = carry.as<char>();
  cr = Carry{};
  cr.frames = reinterpret_cast<long long *>(p); p += S * sizeof(long long);
  cr.hdr = reinterpret_cast<int *>(p); p += S * 4 * sizeof(int);
  cr.tok_state = reinterpret_cast<int *>(p); p += S * cap * sizeof(int);
  cr.tok_cost = reinterpret_cast<float *>(p); p += S * cap * sizeof(float);
  cr.tok_bp = reinterpret_cast<int *>(p);
  cr.cap = plan.max_tok;
  PKB_CUDA(cudaMemsetAsync(carry.p, 0, S * sizeof(long long), c->stream));
  PKB_CUDA(cudaMemsetAsync(cr.hdr, 0xff, S * 4 * sizeof(int), c->stream));  // every stream fresh
  // best-so-far block (copied to the host after every advance), then the finish results
  partial_bytes = S * (sizeof(long long) + mw * sizeof(int32_t) + sizeof(int32_t) + sizeof(float));
  const size_t final_bytes = S * (mw * sizeof(int32_t) + sizeof(int32_t) + sizeof(float));
  PKB_TRY(out.ensure(partial_bytes + final_bytes));
  PKB_CUDA(cudaMemsetAsync(out.p, 0, partial_bytes + final_bytes, c->stream));
  p = out.as<char>();
  cr.p_frames = reinterpret_cast<long long *>(p); p += S * sizeof(long long);
  cr.p_words = reinterpret_cast<int32_t *>(p); p += S * mw * sizeof(int32_t);
  cr.p_nw = reinterpret_cast<int32_t *>(p); p += S * sizeof(int32_t);
  cr.p_cost = reinterpret_cast<float *>(p); p += S * sizeof(float);
  f_words = reinterpret_cast<int32_t *>(p); p += S * mw * sizeof(int32_t);
  f_nw = reinterpret_cast<int32_t *>(p); p += S * sizeof(int32_t);
  f_weight = reinterpret_cast<float *>(p);
  PKB_TRY(d_tid2pdf.ensure(static_cast<size_t>(n_tids) * sizeof(int32_t)));
  PKB_TRY(upload(c, d_tid2pdf.p, tid2pdf, static_cast<size_t>(n_tids) * sizeof(int32_t)));
  return PKB_OK;
}

int ResumableSearch::set_lattice(float lattice_beam, int max_frames, int max_arcs) {
  lat = Lattice{};
  lat_first = nullptr;
  lat_row_off = nullptr;
  for (DevBuf *b : {&lat_log, &lat_aux, &lat_rows, &lat_arcs}) b->release();
  if (lattice_beam == 0.0f) return PKB_OK;
  Lattice l{};
  l.max_frames = max_frames > 0 ? max_frames : 6000;
  // as pkb_batch_lattice: the most the search can log in an utterance of max_frames frames, capped
  // so that the log count (an int that passes max_arcs by at most one group) cannot wrap
  const int64_t bound = static_cast<int64_t>(l.max_frames + 1) * std::max(fst->num_arcs, 1);
  l.max_arcs = max_arcs > 0 ? max_arcs
                            : static_cast<int>(std::min<int64_t>(bound, INT32_MAX - std::max(fst->num_arcs, 1)));
  l.grp_stride = 2 * (l.max_frames + 1);
  l.beam = lattice_beam;
  // per stream: the log; the row store; then group offsets, state, kept count, best cost, first
  // record and row offset
  const size_t S = n;
  const size_t grp_bytes = (S * l.grp_stride * sizeof(int) + 7) & ~static_cast<size_t>(7);
  const size_t state_bytes = (S * 2 * sizeof(int) + 7) & ~static_cast<size_t>(7);
  int rc = lat_log.ensure(S * l.max_arcs * sizeof(unsigned long long));
  if (rc == PKB_OK) rc = lat_rows.ensure(S * l.max_frames * num_pdfs * sizeof(float));
  if (rc == PKB_OK) rc = lat_aux.ensure(grp_bytes + state_bytes + 4 * S * sizeof(int64_t));
  if (rc == PKB_OK) {
    char *p = lat_aux.as<char>();
    l.log = lat_log.as<unsigned long long>();
    l.rows = lat_rows.as<float>();
    l.grp = reinterpret_cast<int *>(p); p += grp_bytes;
    l.state = reinterpret_cast<int *>(p); p += state_bytes;
    l.n_out = reinterpret_cast<long long *>(p); p += S * sizeof(int64_t);
    l.best_out = reinterpret_cast<double *>(p); p += S * sizeof(int64_t);
    lat_first = reinterpret_cast<long long *>(p); p += S * sizeof(int64_t);
    lat_row_off = reinterpret_cast<int64_t *>(p);
    std::vector<int64_t> off(S);
    for (size_t s = 0; s < S; ++s) off[s] = static_cast<int64_t>(s) * l.max_frames;
    rc = upload(c, lat_row_off, off.data(), S * sizeof(int64_t));
  }
  if (rc != PKB_OK) {
    // the decoder stays usable without lattices (and the failed allocation is not reported again
    // by the next launch's error check)
    cudaGetLastError();
    lat_first = nullptr;
    lat_row_off = nullptr;
    for (DevBuf *b : {&lat_log, &lat_aux, &lat_rows, &lat_arcs}) b->release();
    return rc;
  }
  lat = l;
  return PKB_OK;
}

int ResumableSearch::advance(const float *d_loglik, int frame_stride, const int32_t *d_n_frames,
                             int uniform_frames) {
  Carry a = cr;
  a.frame_stride = frame_stride;
  a.uniform_frames = uniform_frames;
  if (lat.log)
    return launch_plan<true, true>(c, fst, plan, cfg, d_loglik, num_pdfs, nullptr, d_n_frames, n,
                                   d_tid2pdf.as<int32_t>(), &work, nullptr, nullptr, nullptr, a, lat);
  return launch_plan<true, false>(c, fst, plan, cfg, d_loglik, num_pdfs, nullptr, d_n_frames, n,
                                  d_tid2pdf.as<int32_t>(), &work, nullptr, nullptr, nullptr, a, Lattice{});
}

int ResumableSearch::finish() {
  Carry a = cr;
  a.finish = 1;
  if (lat.log) {
    // the backward pass reads the row store: stream s's rows start at row s * max_frames
    a.frame_stride = lat.max_frames;
    return launch_plan<true, true>(c, fst, plan, cfg, lat.rows, num_pdfs, nullptr, nullptr, n,
                                   d_tid2pdf.as<int32_t>(), &work, f_words, f_nw, f_weight, a, lat);
  }
  return launch_plan<true, false>(c, fst, plan, cfg, nullptr, num_pdfs, nullptr, nullptr, n,
                                  d_tid2pdf.as<int32_t>(), &work, f_words, f_nw, f_weight, a, Lattice{});
}

int ResumableSearch::expand_lattice(int64_t *n_out, double *best_out, int64_t *total) {
  static_assert(sizeof(long long) == sizeof(int64_t), "int64_t is long long");
  PKB_CUDA(cudaMemcpyAsync(n_out, lat.n_out, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(best_out, lat.best_out, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  std::vector<long long> first(n);
  int64_t sum = 0;
  for (int s = 0; s < n; ++s) {
    first[s] = sum;
    sum += std::max<int64_t>(n_out[s], 0);
  }
  PKB_TRY(lat_arcs.ensure(std::max<int64_t>(sum, 1) * sizeof(pkb_lattice_arc_t)));
  PKB_CUDA(cudaMemcpyAsync(lat_first, first.data(), sizeof(long long) * n, cudaMemcpyHostToDevice, c->stream));
  PKB_TRY(lattice_expand(c, fst, lat, lat.rows, num_pdfs, lat_row_off, n, d_tid2pdf.as<int32_t>(), lat_first,
                         lat_arcs.as<pkb_lattice_arc_t>()));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  *total = sum;
  return PKB_OK;
}

}  // namespace pkb
