// N-best lists of distinct word sequences over the kept records of a lattice (pkb_batch_nbest,
// pkb_decoder_nbest), one thread block per utterance.
//
// A node (t, state) holds up to n entries (graph, acoustic, word history), in the order of
// include/pkb200.h: cost = graph + acoustic, then graph, then the word sequences compared from the
// last word backwards, then acoustic; histories within a list are distinct. The block walks the
// records in time order with the lists of two times live, as per-state arrays in its global
// workspace:
//   emit(t)  every destination merges the lists of its incoming arcs, extended by the arc, into its
//            top n. The group's records are first grouped by destination (a counting sort), so one
//            warp owns one destination: no locks, and no dependence on scheduling.
//   eps(t)   Jacobi passes over the group (each pass reads the previous pass's lists, a destination
//            merges its own list with its incoming arcs) until no list changes. Merging is
//            idempotent in this order, so the fixpoint does not depend on the pass order; an
//            epsilon-acyclic group settles in depth + 1 passes.
//   T        every node's list with its final weight added to the graph cost is merged into the
//            answer, and each history is traced back to its words.
// A merge is a k-way merge of its input lists by head: the lane that owns the least head pops it,
// and a popped entry whose history is already in the output is skipped. Lists extended by one arc
// stay sorted up to rounding of the double sums; the merge does not depend on that, and the host
// restatement in tests/test_gpu_nbest.py runs the same merge.
//
// Word histories are interned per utterance in an open-addressing table of (parent id, word) keys;
// a history's id is its slot + 1 (0: the empty history). Two entries have the same word sequence
// exactly when they have the same id, so equality needs no walk, and the slot order that the
// atomics produce never reaches the output. A candidate through a labelled arc is compared by its
// (parent, word) pair and interned only when it is popped.

#include <math.h>

#include <algorithm>
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "decoder.cuh"

namespace pkb {
namespace {

constexpr int kNbThreads = 512;
constexpr int kNbWarps = kNbThreads / 32;
constexpr unsigned long long kNoKey = ~0ull;
constexpr int kEpsPassFactor = 4;  // epsilon passes the history store is sized for

struct Entry {
  double g, a;  // graph and acoustic cost
  int h;        // history id
  int pad;
};
static_assert(sizeof(Entry) == 24, "Entry is 24 bytes");

// A candidate: history (p, 0) is the id p, (p, w) with w != 0 is history p followed by word w.
struct Key {
  double c, g, a;
  int p, w;
  bool ok;
};

struct Hist {
  unsigned long long *keys;  // slots: parent << 32 | word, kNoKey when free
  unsigned long long mask;
  long long cap;             // insertions allowed
  int *count;                // insertions made
};

struct NbestArgs {
  const pkb_lattice_arc_t *arcs;
  const long long *first, *n_arcs;
  const double *best;
  const long long *stats;   // [n_utts][3]: T, labelled emitting records, labelled epsilon records
  const float *final_w;
  int num_states, start, n, max_words, u0;
  int num_scratch;          // max(arcs of the graph, states)
  char *work;
  size_t work_stride;
  unsigned long long *keys;
  const long long *slot_off;  // [wave + 1] first slot of each utterance of the wave
  const long long *hist_cap;  // [wave]
  int *hist_count;            // [wave]
  int32_t *words;             // [n_utts][n][max_words]
  int32_t *n_words;           // [n_utts][n]
  double *graph, *acoustic;   // [n_utts][n]
  int32_t *n_hyps;            // [n_utts]
};

__device__ __forceinline__ unsigned long long hist_key(int p, int w) {
  return (static_cast<unsigned long long>(static_cast<unsigned>(p)) << 32) | static_cast<unsigned>(w);
}

// Id of history p followed by word w; 0 (with *ovf set) once the store is full.
__device__ int intern(const Hist &hs, int p, int w, int *ovf) {
  const unsigned long long key = hist_key(p, w);
  unsigned long long x = key * 0x9E3779B97F4A7C15ull;
  unsigned long long s = (x ^ (x >> 29)) & hs.mask;
  for (;;) {
    unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(&hs.keys[s]);
    if (k == kNoKey) {
      if (*reinterpret_cast<volatile int *>(hs.count) >= hs.cap) {
        *ovf = 1;
        return 0;
      }
      k = atomicCAS(&hs.keys[s], kNoKey, key);
      if (k == kNoKey) {
        atomicAdd(hs.count, 1);
        return static_cast<int>(s + 1);
      }
    }
    if (k == key) return static_cast<int>(s + 1);
    s = (s + 1) & hs.mask;
  }
}

// Takes the last word off history (p, w): false when it is empty.
__device__ __forceinline__ bool pop_word(const Hist &hs, int &p, int &w, int &last) {
  if (w) {
    last = w;
    w = 0;
    return true;
  }
  if (!p) return false;
  const unsigned long long k = hs.keys[p - 1];
  last = static_cast<int>(k & 0xffffffffull);
  p = static_cast<int>(k >> 32);
  return true;
}

// Word sequences compared from the last word backwards; a suffix of the other comes first.
__device__ int hist_cmp(const Hist &hs, int p1, int w1, int p2, int w2) {
  for (;;) {
    if (!w1 && !w2 && p1 == p2) return 0;
    int l1 = 0, l2 = 0;
    const bool e1 = !pop_word(hs, p1, w1, l1), e2 = !pop_word(hs, p2, w2, l2);
    if (e1 || e2) return e1 == e2 ? 0 : (e1 ? -1 : 1);
    if (l1 != l2) return l1 < l2 ? -1 : 1;
  }
}

__device__ bool key_less(const Hist &hs, const Key &x, const Key &y) {
  if (!y.ok) return x.ok;
  if (!x.ok) return false;
  if (x.c != y.c) return x.c < y.c;
  if (x.g != y.g) return x.g < y.g;
  const int h = hist_cmp(hs, x.p, x.w, y.p, y.w);
  if (h) return h < 0;
  return x.a < y.a;
}

// One input of a merge: a list extended by an arc of weight w, acoustic cost ac and output label
// word (0: none).
struct In {
  const Entry *list;
  int len;
  float w, ac;
  int word;
};

__device__ __forceinline__ Key extend(const Entry &e, const In &in) {
  Key k;
  k.g = e.g + static_cast<double>(in.w);
  k.a = e.a + static_cast<double>(in.ac);
  k.c = k.g + k.a;
  k.p = e.h;
  k.w = in.word;
  k.ok = true;
  return k;
}

// The least head over this lane's inputs i = lane, lane + 32, ... (cursors in cur[i]).
template <class Input>
__device__ Key lane_head(const Hist &hs, int k, const Input &input, const int *cur, int lane, int *which) {
  Key best;
  best.ok = false;
  *which = -1;
  for (int i = lane; i < k; i += 32) {
    const In in = input(i);
    if (cur[i] >= in.len) continue;
    const Key c = extend(in.list[cur[i]], in);
    if (key_less(hs, c, best)) {
      best = c;
      *which = i;
    }
  }
  return best;
}

// Merges inputs 0..k-1 into out (up to n entries of distinct histories); the whole warp calls it.
// Returns the number of entries.
template <class Input>
__device__ int warp_merge(const Hist &hs, int k, const Input &input, int *cur, Entry *out, int n, int *ovf) {
  const int lane = threadIdx.x & 31;
  for (int i = lane; i < k; i += 32) cur[i] = 0;
  __syncwarp();
  int which;
  Key mine = lane_head(hs, k, input, cur, lane, &which);
  int cnt = 0;
  while (cnt < n) {
    Key best = mine;
    int bl = lane;
    for (int off = 16; off; off >>= 1) {
      Key o;
      o.c = __shfl_xor_sync(0xffffffffu, best.c, off);
      o.g = __shfl_xor_sync(0xffffffffu, best.g, off);
      o.a = __shfl_xor_sync(0xffffffffu, best.a, off);
      o.p = __shfl_xor_sync(0xffffffffu, best.p, off);
      o.w = __shfl_xor_sync(0xffffffffu, best.w, off);
      o.ok = __shfl_xor_sync(0xffffffffu, best.ok, off);
      const int ol = __shfl_xor_sync(0xffffffffu, bl, off);
      if (key_less(hs, o, best) || (!key_less(hs, best, o) && ol < bl)) {
        best = o;
        bl = ol;
      }
    }
    if (!best.ok) break;
    if (lane == bl) {
      ++cur[which];
      mine = lane_head(hs, k, input, cur, lane, &which);
    }
    int id = best.p;
    if (best.w) {
      if (lane == 0) id = intern(hs, best.p, best.w, ovf);
      id = __shfl_sync(0xffffffffu, id, 0);
    }
    bool dup = false;
    for (int j = lane; j < cnt; j += 32) dup |= out[j].h == id;
    if (!__any_sync(0xffffffffu, dup)) {
      if (lane == 0) out[cnt] = Entry{best.g, best.a, id, 0};
      ++cnt;
      __syncwarp();
    }
  }
  return cnt;
}

__device__ __forceinline__ int group_of(const pkb_lattice_arc_t &r) { return 2 * r.t + (r.ilabel != 0); }

// Per utterance: T (the last emitting record's t + 1), labelled emitting and labelled epsilon
// records. Block n_utts counts the states entered by a labelled emitting / epsilon arc of the graph.
__global__ void __launch_bounds__(kNbThreads)
nbest_scan_kernel(const pkb_lattice_arc_t *__restrict__ arcs, const long long *__restrict__ first,
                  const long long *__restrict__ n_arcs, int n_utts, const int32_t *__restrict__ arc_dst,
                  const int32_t *__restrict__ arc_il, const int32_t *__restrict__ arc_ol, int num_arcs,
                  int num_states, int *flags, long long *stats) {
  using Reduce = cub::BlockReduce<long long, kNbThreads>;
  __shared__ typename Reduce::TempStorage tmp;
  long long v0 = 0, v1 = 0, v2 = 0;
  if (blockIdx.x < n_utts) {
    const int u = blockIdx.x;
    const long long n = n_arcs[u] > 0 ? n_arcs[u] : 0;
    const pkb_lattice_arc_t *r = arcs + first[u];
    for (long long i = threadIdx.x; i < n; i += kNbThreads) {
      if (r[i].ilabel) v0 = max(v0, static_cast<long long>(r[i].t) + 1);
      if (r[i].olabel) (r[i].ilabel ? v1 : v2) += 1;
    }
  } else {
    for (int a = threadIdx.x; a < num_arcs; a += kNbThreads)
      if (arc_ol[a]) flags[(arc_il[a] ? 0 : num_states) + arc_dst[a]] = 1;
    __syncthreads();
    for (int s = threadIdx.x; s < num_states; s += kNbThreads) {
      v1 += flags[s];
      v2 += flags[num_states + s];
    }
  }
  const long long t_max = Reduce(tmp).Reduce(v0, [](long long x, long long y) { return max(x, y); });
  __syncthreads();
  const long long s1 = Reduce(tmp).Sum(v1);
  __syncthreads();
  const long long s2 = Reduce(tmp).Sum(v2);
  if (threadIdx.x == 0) {
    long long *o = stats + 3 * static_cast<long long>(blockIdx.x);
    o[0] = t_max;
    o[1] = s1;
    o[2] = s2;
  }
}

__global__ void __launch_bounds__(kNbThreads) nbest_kernel(NbestArgs A) {
  using Scan = cub::BlockScan<int, kNbThreads>;
  __shared__ typename Scan::TempStorage scan_tmp;
  __shared__ int s_end, s_ovf;
  const int w = blockIdx.x, u = A.u0 + w;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int S = A.num_states, n = A.n;
  const long long na = A.n_arcs[u];
  if (na < 0 || !(A.best[u] < INFINITY)) {
    if (tid == 0) A.n_hyps[u] = na < 0 ? static_cast<int32_t>(na) : 0;
    return;
  }
  const pkb_lattice_arc_t *recs = A.arcs + A.first[u];
  const int T = static_cast<int>(A.stats[3 * static_cast<long long>(u)]);
  Hist hs;
  hs.keys = A.keys + A.slot_off[w];
  hs.mask = static_cast<unsigned long long>(A.slot_off[w + 1] - A.slot_off[w]) - 1;
  hs.cap = A.hist_cap[w];
  hs.count = A.hist_count + w;
  // workspace: lists and counts of two times, then the counting sort (segment starts, fill
  // pointers, record order) and the merge cursors
  char *p = A.work + A.work_stride * w;
  Entry *X = reinterpret_cast<Entry *>(p);
  Entry *Y = X + static_cast<size_t>(S) * n;
  int *cX = reinterpret_cast<int *>(Y + static_cast<size_t>(S) * n);
  int *cY = cX + S;
  int *seg = cY + S;           // [S + 1]
  int *fill = seg + S + 1;     // [S]
  int *perm = fill + S;        // [num_scratch]
  int *cur = perm + A.num_scratch;  // [num_scratch]
  if (tid == 0) s_ovf = 0;
  for (int s = tid; s < S; s += kNbThreads) cX[s] = s == A.start;
  if (tid == 0) X[static_cast<size_t>(A.start) * n] = Entry{0.0, 0.0, 0, 0};
  __syncthreads();

  // the end of the group that starts at pos (records are sorted by group)
  auto group_end = [&](long long pos, int g) {
    if (tid == 0) {
      long long lo = pos, hi = na;
      while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (group_of(recs[mid]) <= g) lo = mid + 1;
        else hi = mid;
      }
      s_end = static_cast<int>(lo - pos);
    }
    __syncthreads();
    const int e = s_end;
    __syncthreads();
    return e;
  };
  // groups records [0, m) of r by destination: seg[d] .. seg[d + 1] index perm
  auto sort_by_dst = [&](const pkb_lattice_arc_t *r, int m) {
    for (int s = tid; s < S; s += kNbThreads) fill[s] = 0;
    __syncthreads();
    for (int i = tid; i < m; i += kNbThreads) atomicAdd(&fill[r[i].dst], 1);
    __syncthreads();
    const int per = (S + kNbThreads - 1) / kNbThreads, s0 = min(S, tid * per), s1 = min(S, s0 + per);
    int sum = 0;
    for (int s = s0; s < s1; ++s) sum += fill[s];
    int base = 0;
    Scan(scan_tmp).ExclusiveSum(sum, base);
    __syncthreads();
    for (int s = s0; s < s1; ++s) {
      const int c = fill[s];
      seg[s] = base;
      fill[s] = base;
      base += c;
    }
    if (tid == kNbThreads - 1) seg[S] = m;
    __syncthreads();
    for (int i = tid; i < m; i += kNbThreads) perm[atomicAdd(&fill[r[i].dst], 1)] = i;
    __syncthreads();
  };
  // merges destination d of the sorted group r into out; with own, d's list in X is its first
  // input. The cursors of d live at cur + seg[d] + d (an epsilon group has one more input per
  // destination than records).
  auto pull = [&](const pkb_lattice_arc_t *r, int d, bool own, Entry *out) {
    const int b = seg[d], k = seg[d + 1] - b + own;
    const Entry *Xc = X;
    const int *cXc = cX;
    auto input = [&](int i) {
      if (own && i == 0) return In{Xc + static_cast<size_t>(d) * n, cXc[d], 0.0f, 0.0f, 0};
      const pkb_lattice_arc_t &a = r[perm[b + i - own]];
      return In{Xc + static_cast<size_t>(a.src) * n, cXc[a.src], a.graph_cost, a.acoustic_cost, a.olabel};
    };
    const int c = warp_merge(hs, k, input, cur + b + d, out, n, &s_ovf);
    if (lane == 0) cY[d] = c;
  };

  int err = 0;
  long long pos = 0;
  for (int t = 0;; ++t) {
    // epsilon closure of time t in X, each pass's new lists in Y
    int m = group_end(pos, 2 * t);
    if (m > 0) {
      const pkb_lattice_arc_t *r = recs + pos;
      sort_by_dst(r, m);
      const long long max_pass = static_cast<long long>(m + 1) * (n + 1);
      for (long long pass = 0;; ++pass) {
        if (pass == max_pass) {
          err = 6;
          break;
        }
        for (int d = warp; d < S; d += kNbWarps)
          if (seg[d + 1] > seg[d]) pull(r, d, true, Y + static_cast<size_t>(d) * n);
        __syncthreads();
        bool changed = false;
        for (int d = warp; d < S; d += kNbWarps) {
          if (seg[d + 1] == seg[d]) continue;
          const int c = cY[d];
          bool diff = c != cX[d];
          const Entry *o = X + static_cast<size_t>(d) * n, *q = Y + static_cast<size_t>(d) * n;
          for (int j = lane; j < c && !diff; j += 32)
            diff = __double_as_longlong(o[j].g) != __double_as_longlong(q[j].g) ||
                   __double_as_longlong(o[j].a) != __double_as_longlong(q[j].a) || o[j].h != q[j].h;
          changed |= diff;
        }
        __syncthreads();
        for (int d = warp; d < S; d += kNbWarps) {
          if (seg[d + 1] == seg[d]) continue;
          const int c = cY[d];
          for (int j = lane; j < c; j += 32) X[static_cast<size_t>(d) * n + j] = Y[static_cast<size_t>(d) * n + j];
          if (lane == 0) cX[d] = c;
        }
        if (!__syncthreads_or(changed)) break;
      }
      pos += m;
    }
    if (t == T || err) break;
    // emitting arcs of time t: X -> Y
    m = group_end(pos, 2 * t + 1);
    for (int s = tid; s < S; s += kNbThreads) cY[s] = 0;
    if (m > 0) {
      const pkb_lattice_arc_t *r = recs + pos;
      sort_by_dst(r, m);
      for (int d = warp; d < S; d += kNbWarps)
        if (seg[d + 1] > seg[d]) pull(r, d, false, Y + static_cast<size_t>(d) * n);
      pos += m;
    }
    __syncthreads();
    Entry *te = X;
    X = Y;
    Y = te;
    int *tc = cX;
    cX = cY;
    cY = tc;
    // no thread writes s_ovf between this barrier and the next one (in group_end)
    if (s_ovf) break;
  }
  __syncthreads();
  if (!err && s_ovf) err = 7;
  if (err) {
    if (tid == 0) A.n_hyps[u] = -err;
    return;
  }
  // final nodes into the answer (in Y), then the histories back to words
  __shared__ int s_cnt;
  if (warp == 0) {
    const float *fin = A.final_w;
    auto input = [&](int s) {
      const float f = __ldg(&fin[s]);
      return In{X + static_cast<size_t>(s) * n, isinf(f) ? 0 : cX[s], f, 0.0f, 0};
    };
    const int c = warp_merge(hs, S, input, cur, Y, n, &s_ovf);
    if (lane == 0) s_cnt = c;
  }
  __syncthreads();
  const int cnt = s_cnt;
  const size_t o = static_cast<size_t>(u) * n;
  for (int i = tid; i < cnt; i += kNbThreads) {
    const Entry e = Y[i];
    int len = 0;
    for (int h = e.h; h; h = static_cast<int>(hs.keys[h - 1] >> 32)) ++len;
    int j = len;
    for (int h = e.h; h; h = static_cast<int>(hs.keys[h - 1] >> 32)) {
      --j;
      if (j < A.max_words) A.words[(o + i) * A.max_words + j] = static_cast<int>(hs.keys[h - 1] & 0xffffffffull);
    }
    A.n_words[o + i] = len;
    A.graph[o + i] = e.g;
    A.acoustic[o + i] = e.a;
  }
  if (tid == 0) A.n_hyps[u] = cnt;
}

}  // namespace

int plan_waves(const std::vector<size_t> &bytes, std::vector<int> *starts, size_t *most) {
  size_t free_b = 0, total_b = 0;
  PKB_CUDA(cudaMemGetInfo(&free_b, &total_b));
  const size_t budget = std::min<size_t>(free_b / 2, size_t(8) << 30);
  const int U = static_cast<int>(bytes.size());
  starts->assign(1, 0);
  size_t top = 0;
  for (int u0 = 0; u0 < U;) {
    int m = 0;
    size_t sum = 0;
    while (u0 + m < U && (m == 0 || sum + bytes[u0 + m] <= budget)) sum += bytes[u0 + m++];
    top = std::max(top, sum);
    u0 += m;
    starts->push_back(u0);
  }
  if (most) *most = top;
  return PKB_OK;
}

int LatticeResults::nbest(int n, int max_words, int32_t *words_out, int32_t *n_words_out,
                          double *graph_cost_out, double *acoustic_cost_out, int32_t *n_hyps_out, const char *who) {
  PKB_REQUIRE(total >= 0, "%s: no lattice: %s", who, why.c_str());
  PKB_REQUIRE(n >= 1 && n <= 1024, "%s: n must be in [1, 1024] (got %d)", who, n);
  PKB_REQUIRE(max_words > 0, "%s: max_words must be > 0 (got %d)", who, max_words);
  PKB_REQUIRE(words_out && n_words_out && graph_cost_out && acoustic_cost_out && n_hyps_out,
              "%s: NULL output argument", who);
  const int U = static_cast<int>(n_arcs.size());
  if (U == 0) return PKB_OK;
  PKB_CUDA(cudaSetDevice(c->device));
  const int S = fst->num_states;
  const int scratch = std::max(fst->num_arcs, S) + S + 1;  // merge cursors at seg[d] + d
  // sizes: statistics and flags, then the outputs
  const size_t stats_bytes = 3 * sizeof(long long) * (U + 1);
  const size_t flag_bytes = (2 * sizeof(int) * S + 7) & ~static_cast<size_t>(7);
  const size_t words_bytes = sizeof(int32_t) * U * static_cast<size_t>(n) * max_words;
  const size_t nw_bytes = (sizeof(int32_t) * U * static_cast<size_t>(n) + 7) & ~static_cast<size_t>(7);
  const size_t cost_bytes = sizeof(double) * U * static_cast<size_t>(n);
  const size_t nh_bytes = (sizeof(int32_t) * U + 7) & ~static_cast<size_t>(7);
  const size_t fixed = stats_bytes + flag_bytes + words_bytes + nw_bytes + 2 * cost_bytes + nh_bytes;
  const size_t stride = ((2 * sizeof(Entry) * S * static_cast<size_t>(n) + sizeof(int) * (4 * S + 1) +
                          2 * sizeof(int) * scratch) + 255) & ~static_cast<size_t>(255);
  // the first pass sizes the word-history stores
  PKB_TRY(nbest_work.ensure(fixed));
  char *p = nbest_work.as<char>();
  long long *d_stats = reinterpret_cast<long long *>(p); p += stats_bytes;
  int *d_flags = reinterpret_cast<int *>(p); p += flag_bytes;
  int32_t *d_words = reinterpret_cast<int32_t *>(p); p += words_bytes;
  int32_t *d_nw = reinterpret_cast<int32_t *>(p); p += nw_bytes;
  double *d_graph = reinterpret_cast<double *>(p); p += cost_bytes;
  double *d_ac = reinterpret_cast<double *>(p); p += cost_bytes;
  int32_t *d_nh = reinterpret_cast<int32_t *>(p);
  PKB_CUDA(cudaMemsetAsync(d_flags, 0, flag_bytes, c->stream));
  PKB_CUDA(cudaMemsetAsync(d_words, 0, fixed - stats_bytes - flag_bytes, c->stream));
  {
    LaunchScope scope(c, PKB_KERNEL_MISC);
    nbest_scan_kernel<<<U + 1, kNbThreads, 0, c->stream>>>(arcs.as<pkb_lattice_arc_t>(), d_first(), d_n_arcs(), U,
                                                          fst->d_arc_dst, fst->d_arc_il, fst->d_arc_ol,
                                                          fst->num_arcs, S, d_flags, d_stats);
    PKB_CUDA(cudaGetLastError());
  }
  std::vector<long long> stats(3 * (U + 1));
  PKB_CUDA(cudaMemcpyAsync(stats.data(), d_stats, stats_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  const long long s_emit = stats[3 * U + 1], s_eps = stats[3 * U + 2];
  // histories an utterance can intern: each merge interns at most n, and a merge that interns has
  // a labelled incoming record; per time at most min(labelled records, states entered by a
  // labelled arc) such merges, for epsilon groups once per pass (sized for kEpsPassFactor passes)
  std::vector<long long> cap(U), slots(U);
  for (int u = 0; u < U; ++u) {
    const long long T = stats[3 * u], le = stats[3 * u + 1], lp = stats[3 * u + 2];
    cap[u] = n * (std::min(le, T * s_emit) + kEpsPassFactor * std::min(lp, (T + 1) * s_eps));
    long long sl = 64;
    while (sl < (cap[u] + 64) + (cap[u] + 64) / 2) sl <<= 1;
    PKB_REQUIRE(sl <= (1ll << 30), "pkb nbest: utterance %d needs %lld word-history slots (more than 2^30)", u, sl);
    slots[u] = sl;
  }
  // utterances in waves whose workspace fits the budget
  std::vector<size_t> bytes(U);
  for (int u = 0; u < U; ++u) bytes[u] = stride + slots[u] * sizeof(unsigned long long) + 4 * sizeof(long long);
  std::vector<int> wave_start;
  PKB_TRY(plan_waves(bytes, &wave_start, nullptr));
  DevBuf wave_buf;
  for (size_t w = 0; w + 1 < wave_start.size(); ++w) {
    const int u0 = wave_start[w], m = wave_start[w + 1] - u0;
    const size_t key_bytes = [&] {
      size_t s = 0;
      for (int i = 0; i < m; ++i) s += slots[u0 + i] * sizeof(unsigned long long);
      return s;
    }();
    const size_t meta_bytes = (sizeof(long long) * (2 * m + 1) + sizeof(int) * m + 255) & ~static_cast<size_t>(255);
    PKB_TRY(wave_buf.ensure(stride * m + key_bytes + meta_bytes));
    char *q = wave_buf.as<char>();
    NbestArgs A{};
    A.work = q; q += stride * m;
    A.keys = reinterpret_cast<unsigned long long *>(q); q += key_bytes;
    long long *d_meta = reinterpret_cast<long long *>(q);
    std::vector<long long> hm(2 * m + 1);
    for (int i = 0; i < m; ++i) {
      hm[i + 1] = hm[i] + slots[u0 + i];
      hm[m + 1 + i] = cap[u0 + i];
    }
    PKB_CUDA(cudaMemcpyAsync(d_meta, hm.data(), sizeof(long long) * hm.size(), cudaMemcpyHostToDevice, c->stream));
    A.slot_off = d_meta;
    A.hist_cap = d_meta + m + 1;
    A.hist_count = reinterpret_cast<int *>(d_meta + 2 * m + 1);
    PKB_CUDA(cudaMemsetAsync(A.hist_count, 0, sizeof(int) * m, c->stream));
    PKB_CUDA(cudaMemsetAsync(A.keys, 0xff, key_bytes, c->stream));
    A.arcs = arcs.as<pkb_lattice_arc_t>();
    A.first = d_first();
    A.n_arcs = d_n_arcs();
    A.best = d_best();
    A.stats = d_stats;
    A.final_w = fst->d_final;
    A.num_states = S;
    A.start = fst->start;
    A.n = n;
    A.max_words = max_words;
    A.u0 = u0;
    A.num_scratch = scratch;
    A.work_stride = stride;
    A.words = d_words;
    A.n_words = d_nw;
    A.graph = d_graph;
    A.acoustic = d_ac;
    A.n_hyps = d_nh;
    {
      LaunchScope scope(c, PKB_KERNEL_MISC);
      nbest_kernel<<<m, kNbThreads, 0, c->stream>>>(A);
      PKB_CUDA(cudaGetLastError());
    }
    // the host copy of hm must outlive the copy
    PKB_CUDA(cudaStreamSynchronize(c->stream));
  }
  PKB_CUDA(cudaMemcpyAsync(words_out, d_words, words_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_words_out, d_nw, sizeof(int32_t) * U * static_cast<size_t>(n), cudaMemcpyDeviceToHost,
                           c->stream));
  PKB_CUDA(cudaMemcpyAsync(graph_cost_out, d_graph, cost_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(acoustic_cost_out, d_ac, cost_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_hyps_out, d_nh, sizeof(int32_t) * U, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return check_device_error(c, who);
}

}  // namespace pkb
