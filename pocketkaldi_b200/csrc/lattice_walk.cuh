// The forward walk over the kept records of one utterance's lattice that the posterior kernel
// (posterior.cu) and the best-path kernel (best_path.cu) share: one thread block per utterance, the
// groups eps(0), emit(0), eps(1), ... in time order, and a fold of each node's incoming records in
// the order of include/pkb200.h. The kernels differ only in the fold (log-add or min) and the cost
// of a record.
//
//   emit(t)   the group's records are grouped by destination with a stable counting sort (below),
//             then one thread per destination folds its incoming records in record order into
//             alpha(t + 1, dst).
//   eps(t)    Kahn levels over the group: a node is folded once every source is complete, so the
//             fold order is fixed and the result does not depend on scheduling. Nodes left over when
//             the levels stop lie on a cycle of epsilon records: the utterance fails with -8.
// The walk saves alpha(t, src) per record (8 bytes), which the kernels read afterwards.
#pragma once

#include <algorithm>
#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include "decoder.cuh"

namespace pkb {
namespace lattice_walk {

constexpr int kThreads = 512;
constexpr int kItems = 4;                      // records per thread of a sort tile
constexpr int kTile = kThreads * kItems;       // records per sort tile
constexpr int kTileBits = 11;                  // log2(kTile)
static_assert((1 << kTileBits) == kTile, "tile bits");
constexpr size_t kSmemState = 48 << 10;        // per-state arrays go to shared memory up to this

using Scan = cub::BlockScan<int, kThreads>;
using Sort = cub::BlockRadixSort<unsigned long long, kThreads, kItems>;

// Static shared memory of a walking block.
struct Shared {
  union {
    typename Scan::TempStorage scan;
    typename Sort::TempStorage sort;
  } tmp;
  int tkey[kTile];
};

// Launch arguments of a walking kernel over the records of a LatticeResults (walk_args fills the
// lattice's part).
struct WalkArgs {
  const pkb_lattice_arc_t *arcs;
  const long long *first, *n_arcs;
  const double *best;
  const float *final_w;
  int num_states, num_arcs, start, u0;
  double as, gs;
  char *work;               // per block: workspace [, per-state arrays]
  size_t work_stride;
  bool smem_state;          // per-state arrays in dynamic shared memory
  double *alpha;            // alpha(t, src) of record first[u] + i at alpha[first[u] - rec0 + i]
  long long rec0;
};

inline WalkArgs walk_args(const LatticeResults &L, float acoustic_scale, float graph_scale) {
  WalkArgs A{};
  A.arcs = L.arcs.as<pkb_lattice_arc_t>();
  A.first = L.d_first();
  A.n_arcs = L.d_n_arcs();
  A.best = L.d_best();
  A.final_w = L.fst->d_final;
  A.num_states = L.fst->num_states;
  A.num_arcs = std::max(L.fst->num_arcs, 1);
  A.start = L.fst->start;
  A.as = acoustic_scale;
  A.gs = graph_scale;
  return A;
}

// graph_scale x graph_cost + acoustic_scale x acoustic_cost in double (include/pkb200.h)
__device__ __forceinline__ double scaled_cost(const WalkArgs &A, const pkb_lattice_arc_t &r) {
  return __dadd_rn(__dmul_rn(A.gs, static_cast<double>(r.graph_cost)),
                   __dmul_rn(A.as, static_cast<double>(r.acoustic_cost)));
}

__device__ __forceinline__ int group_of(const pkb_lattice_arc_t &r) { return 2 * r.t + (r.ilabel != 0); }

__device__ __forceinline__ int bit_width(unsigned x) { return 32 - __clz(x); }

// One block's view of utterance records recs[0, na), in groups of at most NA records. perm [NA],
// fill [K] and seg [K + 1] are the workspace of group_by_key, for keys in [0, K).
struct Walk {
  const pkb_lattice_arc_t *recs;
  long long na;
  int NA, K, tid;
  int *perm, *fill, *seg;
  Shared &sh;

  // the first index in [lo, min(na, lo + NA)] whose group is > grp (a group holds at most NA
  // records); every thread probes once per round, so two rounds cover 2^18 records
  __device__ __forceinline__ long long group_end(long long lo, int grp) const {
    long long a = lo, b = min(na, lo + NA);
    while (b > a) {
      const long long step = (b - a + kThreads - 1) / kThreads, p = a + tid * step;
      const int k = __syncthreads_count(p < b && group_of(recs[p]) <= grp);
      if (k == 0) break;
      const long long nb = min(b, a + k * step);
      a += (k - 1) * step + 1;
      b = nb;
    }
    return a;
  }

  // Groups records [0, m) by key(i) in [0, K) stably: key k's records are perm[seg[k] .. seg[k + 1])
  // in ascending order. Counts and a scan give the segments; then tiles of kTile records in order
  // are radix-sorted by (key, index) and appended to their segments.
  template <class Key>
  __device__ __forceinline__ void group_by_key(int m, Key key) const {
    __syncthreads();
    for (int k = tid; k < K; k += kThreads) fill[k] = 0;
    __syncthreads();
    for (int i = tid; i < m; i += kThreads) atomicAdd(&fill[key(i)], 1);
    __syncthreads();
    const int per = (K + kThreads - 1) / kThreads, k0 = min(K, tid * per), k1 = min(K, k0 + per);
    int sum = 0;
    for (int k = k0; k < k1; ++k) sum += fill[k];
    int base = 0;
    Scan(sh.tmp.scan).ExclusiveSum(sum, base);
    __syncthreads();
    for (int k = k0; k < k1; ++k) {
      const int c = fill[k];
      seg[k] = base;
      fill[k] = base;
      base += c;
    }
    if (tid == 0) seg[K] = m;
    const int end_bit = kTileBits + bit_width(static_cast<unsigned>(K));
    for (int b0 = 0; b0 < m; b0 += kTile) {
      unsigned long long keys[kItems];
      for (int j = 0; j < kItems; ++j) {
        const int li = tid * kItems + j;
        keys[j] = b0 + li < m ? (static_cast<unsigned long long>(key(b0 + li)) << kTileBits) | li : ~0ull;
      }
      __syncthreads();
      Sort(sh.tmp.sort).Sort(keys, 0, end_bit);
      for (int j = 0; j < kItems; ++j) {
        const int r = tid * kItems + j;
        sh.tkey[r] = r < m - b0 ? static_cast<int>(keys[j] >> kTileBits) : -1;
      }
      __syncthreads();
      // the first rank of each key's run in this tile moves its fill pointer back by that rank,
      // every rank then lands at fill + rank, and the run's last rank moves it past the run
      for (int j = 0; j < kItems; ++j) {
        const int r = tid * kItems + j, k = sh.tkey[r];
        if (k >= 0 && (r == 0 || sh.tkey[r - 1] != k)) fill[k] -= r;
      }
      __syncthreads();
      for (int j = 0; j < kItems; ++j) {
        const int r = tid * kItems + j, k = sh.tkey[r];
        if (k >= 0) perm[fill[k] + r] = b0 + static_cast<int>(keys[j] & (kTile - 1));
      }
      __syncthreads();
      for (int j = 0; j < kItems; ++j) {
        const int r = tid * kItems + j, k = sh.tkey[r];
        if (k >= 0 && (r == kTile - 1 || sh.tkey[r + 1] != k)) fill[k] += r + 1;
      }
    }
    __syncthreads();
  }

  // T: the last emitting record's t + 1 (records end with eps(T))
  __device__ __forceinline__ int last_time() const {
    if (na == 0) return 0;
    const pkb_lattice_arc_t last = recs[na - 1];
    if (last.ilabel) return last.t + 1;
    const long long b = group_end(max(0ll, na - NA), 2 * last.t - 1);
    return b > 0 ? recs[b - 1].t + 1 : 0;
  }

  // The forward pass over S states from alpha(0, start) = 0 up to time T: each node folds
  // fold(held, alpha(t, src) + cost(r)) over its incoming records, emitting records of time t - 1
  // in record order, then the epsilon records of time t in record order, starting from +inf (0 at
  // (0, start)). Saves alpha(t, src) of record i at alpha[i]. Returns 0, or 8 when the epsilon
  // records of a time form a cycle. On return X holds alpha(T, .); Y and done [S] are workspace.
  template <class Cost, class Fold>
  __device__ __forceinline__ int forward(double *&X, double *&Y, int *done, int S, int start, int T,
                                         double *alpha, Cost cost, Fold fold) const {
    for (int s = tid; s < S; s += kThreads) X[s] = s == start ? 0.0 : INFINITY;
    long long pos = 0;
    for (int t = 0;; ++t) {
      const long long e_end = group_end(pos, 2 * t);
      const int ne = static_cast<int>(e_end - pos);
      if (ne > 0) {
        const pkb_lattice_arc_t *E = recs + pos;
        group_by_key(ne, [&](int i) { return E[i].dst; });
        for (int s = tid; s < S; s += kThreads) done[s] = seg[s + 1] > seg[s] ? 0 : 2;
        __syncthreads();
        for (;;) {
          for (int d = tid; d < S; d += kThreads) {
            if (done[d]) continue;
            bool ready = true;
            for (int j = seg[d]; j < seg[d + 1] && ready; ++j) ready = done[E[perm[j]].src] == 2;
            if (!ready) continue;
            double a = X[d];
            for (int j = seg[d]; j < seg[d + 1]; ++j) {
              const pkb_lattice_arc_t &r = E[perm[j]];
              a = fold(a, X[r.src] + cost(r));
            }
            X[d] = a;
            done[d] = 1;
          }
          __syncthreads();
          int progress = 0;
          for (int d = tid; d < S; d += kThreads)
            if (done[d] == 1) {
              done[d] = 2;
              progress = 1;
            }
          if (!__syncthreads_or(progress)) break;
        }
        int open = 0;
        for (int d = tid; d < S && !open; d += kThreads) open = done[d] == 0;
        if (__syncthreads_or(open)) return 8;
      }
      const long long m_end = t < T ? group_end(e_end, 2 * t + 1) : e_end;
      for (long long i = pos + tid; i < m_end; i += kThreads) alpha[i] = X[recs[i].src];
      if (t == T) return 0;
      const int nm = static_cast<int>(m_end - e_end);
      const pkb_lattice_arc_t *M = recs + e_end;
      for (int s = tid; s < S; s += kThreads) Y[s] = INFINITY;
      if (nm > 0) {
        group_by_key(nm, [&](int i) { return M[i].dst; });
        for (int d = tid; d < S; d += kThreads) {
          if (seg[d + 1] == seg[d]) continue;
          double a = INFINITY;
          for (int j = seg[d]; j < seg[d + 1]; ++j) {
            const pkb_lattice_arc_t &r = M[perm[j]];
            a = fold(a, X[r.src] + cost(r));
          }
          Y[d] = a;
        }
      }
      __syncthreads();
      double *tx = X;
      X = Y;
      Y = tx;
      pos = m_end;
    }
  }
};

}  // namespace lattice_walk
}  // namespace pkb
