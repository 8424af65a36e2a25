// Online sliding-window cepstral mean normalisation for sm_100a, plus the
// synthetic-PCM generator and the checksum reduction used by the batch pipeline.
//
// Replaces CMVN::GetFrame called for t = 0..T-1 (src/cmvn.cc:103-115):
//   ComputeStats (:35-71)  stats_t = float( double(stats_{t-1}) + x_t - x_{t-600} )
//   SmoothStats  (:73-92)  stats += float(min(600-n,200)/Gc) * G     (float mul, float add)
//   Apply        (:94-101) y = x + (-float(1/count)) * stats         (float mul, float add)
// The running sum is a float that is widened to double only inside a step, so
// the recurrence is inherently sequential per (utterance, dimension). The
// kernel keeps that exact rounding sequence -- one thread per chain -- which
// makes the output bit-identical to the reference for identical raw input;
// parallelism comes from the n_utts * 40 independent chains. The frame-count
// element of the stats vector depends only on t, so alpha_t and scale_t are
// tabulated on the host with the reference's double/float arithmetic.

#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace pkb {

namespace {

constexpr int kCmvnUnroll = 8;

// Where one thread's pair of chains (dims d, d + 1 of one utterance) reads and writes. Everything
// is indexed by frame with a stride of one frame.
struct CmvnChain {
  const float *x;         // raw[t * 40 + d]
  float *y;               // out[t * 40 + d] or nullptr
  __nv_bfloat16 *ph, *pl; // planes[(left + t) * dim_pad + d] or nullptr
  int dim_pad;
  float gd[2];            // global stats of the two dims
};

// RN32(a + b + c) for binary32 a, b, c without widening: Boldo & Melquiond's three-term sum
// (two TwoSums, then the two error terms added with rounding to odd, emulated with a
// round-down / round-up pair). Exact for any inputs short of overflow / underflow.
__device__ __forceinline__ float sum3_rn(float a, float b, float c) {
  const float uh = __fadd_rn(b, c);
  const float ub = __fsub_rn(uh, b);
  const float ul = __fadd_rn(__fsub_rn(b, __fsub_rn(uh, ub)), __fsub_rn(c, ub));
  const float th = __fadd_rn(a, uh);
  const float tb = __fsub_rn(th, a);
  const float tl = __fadd_rn(__fsub_rn(a, __fsub_rn(th, tb)), __fsub_rn(uh, tb));
  const float vd = __fadd_rd(tl, ul), vu = __fadd_ru(tl, ul);
  const float v = (vd == vu || (__float_as_uint(vd) & 1u)) ? vd : vu;
  return __fadd_rn(th, v);
}

// The reference forms double(stat) + x - x_old and rounds to float once per frame
// (src/cmvn.cc:35-71). When every value that entered the chain is 0 or has 2^-6 <= |v| < 2^12, all
// three terms are multiples of 2^-29 below 2^23, both double additions are exact, and the
// step is RN32 of the exact three-term sum -- which sum3_rn delivers on the FP32 pipe (the FP64
// pipe of this part issues one warp instruction per 16 cycles). A chain that has seen a value
// outside that range (digital silence gives log(FLT_EPSILON) = -15.9, which is fine; energies
// within 1.6 % of 1.0 or non-finite values are not) stays on the FP64 path.
__device__ __forceinline__ bool cmvn_out_of_range(float x) {
  const uint32_t u = __float_as_uint(x) & 0x7fffffffu;
  return u != 0u && (u - 0x3C800000u) >= (0x45800000u - 0x3C800000u);
}

// One frame of the recurrence (ComputeStats -> SmoothStats -> Apply, src/cmvn.cc:35-101) for the
// thread's two independent chains (the compiler interleaves them: twice the work per dependent
// step of latency).
//   kSub:   the window is full, the frame 600 steps back leaves the sum (t >= 600)
//   kAlpha: fewer than 600 frames seen, the global stats are blended in (t < 599)
//   kF64:   widen like the reference (only needed for kSub, see above)
template <bool kSub, bool kAlpha, bool kF64, int kPlanes, bool kFp16, bool kOut>
__device__ __forceinline__ void cmvn_frame(const CmvnChain &c, int t, int i, float2 x, float2 xold,
                                           float (&stat)[2], float alpha, float sc) {
  // t = first frame of the group, i = compile-time index inside it: every address below is one
  // group base plus an immediate offset
  const float xv[2] = {x.x, x.y}, xo[2] = {xold.x, xold.y};
  float v[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    if (!kSub) {
      // double(stat) + double(x) rounded to float == the float sum: the double sum is exact when
      // the exponents are within 29 of each other and cannot reach a rounding boundary otherwise
      stat[e] = __fadd_rn(stat[e], xv[e]);
    } else if (kF64) {
      double acc = static_cast<double>(stat[e]) + static_cast<double>(xv[e]);
      acc += -1.0 * static_cast<double>(xo[e]);
      stat[e] = static_cast<float>(acc);
    } else {
      stat[e] = sum3_rn(stat[e], xv[e], -xo[e]);
    }
    float s = stat[e];
    if (kAlpha) s = __fadd_rn(s, __fmul_rn(alpha, c.gd[e]));
    v[e] = __fadd_rn(xv[e], __fmul_rn(-sc, s));
  }
  // streaming stores: the outputs are not read again by this kernel and must not evict the
  // raw rows that are (x[t - 600])
  if (kOut) __stcs(reinterpret_cast<float2 *>(c.y + static_cast<int64_t>(t) * kMel + i * kMel), make_float2(v[0], v[1]));
  if (kPlanes >= 1) {
    // plane rows are kMel elements apart (feat_dim_pad == kMel: 40 is a multiple of 8)
    const __nv_bfloat16 h0 = operand_bits(v[0], kFp16), h1 = operand_bits(v[1], kFp16);
    __stcs(reinterpret_cast<unsigned int *>(c.ph + static_cast<int64_t>(t) * kMel + i * kMel),
           static_cast<unsigned int>(__bfloat16_as_ushort(h0)) |
               (static_cast<unsigned int>(__bfloat16_as_ushort(h1)) << 16));
    if (kPlanes == 2) {
      const __nv_bfloat16 l0 = operand_bits(v[0] - operand_value(h0, kFp16), kFp16);
      const __nv_bfloat16 l1 = operand_bits(v[1] - operand_value(h1, kFp16), kFp16);
      __stcs(reinterpret_cast<unsigned int *>(c.pl + static_cast<int64_t>(t) * kMel + i * kMel),
             static_cast<unsigned int>(__bfloat16_as_ushort(l0)) |
                 (static_cast<unsigned int>(__bfloat16_as_ushort(l1)) << 16));
    }
  }
}

// cp.async: 8 bytes global -> shared without passing through a register; completion is tracked
// per thread in commit groups.
__device__ __forceinline__ void cp_async8(float2 *smem_dst, const float *gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(
                   static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))),
               "l"(gmem_src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(kPending) : "memory");
}


// One thread per pair of chains (utterance, dims 2k and 2k + 1): 20 threads per utterance. The
// recurrence is a handful of dependent FP32 operations per frame, so what limits the kernel is
// latency: every thread streams its x[t] and x[t - 600] pairs through a private shared-memory ring
// with cp.async, kCmvnGroups - 1 groups of 8 frames ahead of the group it is consuming, and no thread
// ever reads another thread's slots (no block-level synchronisation in the loop).
// Frames t < 600 fill the window (global stats blended in through the alpha / scale tables, which
// hold alpha = 0 at t = 599); frames t >= 600 slide it. 600 is a multiple of the group size, so a
// group lies in one phase.
constexpr int kCmvnThreadsPerUtt = kMel / 2;
constexpr int kCmvnGroups = 4;  // ring depth: 4 groups of kCmvnUnroll frames (32 frames)

template <int kPlanes, bool kFp16, bool kOut, int kBlock>
__global__ void __launch_bounds__(kBlock, kBlock == 160 ? 2 : 16)
cmvn_kernel(const float *__restrict__ raw, const int64_t *__restrict__ frame_off,
            const int32_t *__restrict__ num_frames, int n_utts,
            const float *__restrict__ tab /* alpha[600], scale[600], global[41] */,
            float *__restrict__ out, __nv_bfloat16 *__restrict__ p_hi,
            __nv_bfloat16 *__restrict__ p_lo, const int64_t *__restrict__ pad_off, int left,
            int right, int dim_pad) {
  static_assert(kCmvnWindow % kCmvnUnroll == 0, "a group must not straddle the two phases");
  static_assert(kMel % 2 == 0, "two dims per thread");
  constexpr int kCmvnRing = kCmvnGroups * kCmvnUnroll;  // frames in flight per chain (power of two)
  __shared__ float s_alpha[kCmvnWindow];
  __shared__ float s_scale[kCmvnWindow];
  extern __shared__ float2 s_ring[];  // [2][kCmvnRing][kBlock]: x, then x_old
  for (int i = threadIdx.x; i < kCmvnWindow; i += kBlock) {
    s_alpha[i] = tab[i];
    s_scale[i] = tab[kCmvnWindow + i];
  }
  __syncthreads();
  const int64_t g = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  const int u = static_cast<int>(g / kCmvnThreadsPerUtt);
  const int d = 2 * static_cast<int>(g % kCmvnThreadsPerUtt);
  if (u >= n_utts) return;
  const int T = num_frames[u];
  if (T == 0) return;
  CmvnChain c;
  c.gd[0] = tab[2 * kCmvnWindow + d];
  c.gd[1] = tab[2 * kCmvnWindow + d + 1];
  c.x = raw + frame_off[u] * kMel + d;
  c.y = kOut ? out + frame_off[u] * kMel + d : nullptr;
  c.dim_pad = dim_pad;
  c.ph = kPlanes >= 1 ? p_hi + (pad_off[u] + left) * dim_pad + d : nullptr;
  c.pl = kPlanes == 2 ? p_lo + (pad_off[u] + left) * dim_pad + d : nullptr;

  float2 *rx = s_ring + threadIdx.x;
  float2 *ro = rx + kCmvnRing * kBlock;
  const int T8 = T & ~(kCmvnUnroll - 1);  // whole groups run without per-frame bounds checks
  // one commit group per call (possibly empty) keeps the wait count static
  auto issue = [&](int t0) {
    if (t0 < T8) {
      const float *px = c.x + static_cast<int64_t>(t0) * kMel;
      float2 *dx = rx + (t0 & (kCmvnRing - 1)) * kBlock;
#pragma unroll
      for (int i = 0; i < kCmvnUnroll; ++i) cp_async8(dx + i * kBlock, px + i * kMel);
      if (t0 >= kCmvnWindow) {
        float2 *dxo = ro + (t0 & (kCmvnRing - 1)) * kBlock;
#pragma unroll
        for (int i = 0; i < kCmvnUnroll; ++i) cp_async8(dxo + i * kBlock, px + (i - kCmvnWindow) * kMel);
      }
    }
    cp_async_commit();
  };

  float stat[2] = {0.0f, 0.0f};
  bool wide = false;
  const float scale_full = s_scale[kCmvnWindow - 1];
  const float2 zero2 = make_float2(0.0f, 0.0f);
#pragma unroll
  for (int k = 0; k < kCmvnGroups - 1; ++k) issue(k * kCmvnUnroll);
  for (int t0 = 0; t0 < T8; t0 += kCmvnUnroll) {
    issue(t0 + (kCmvnGroups - 1) * kCmvnUnroll);
    cp_async_wait<kCmvnGroups - 1>();  // the group of t0 has landed
    const float2 *gx = rx + (t0 & (kCmvnRing - 1)) * kBlock;
    float2 xv[kCmvnUnroll];
    bool w = wide;
#pragma unroll
    for (int i = 0; i < kCmvnUnroll; ++i) {
      xv[i] = gx[i * kBlock];
      w = w || cmvn_out_of_range(xv[i].x) || cmvn_out_of_range(xv[i].y);
    }
    wide = w;
    if (t0 < kCmvnWindow) {
      const float *pa = s_alpha + t0, *ps = s_scale + t0;
#pragma unroll
      for (int i = 0; i < kCmvnUnroll; ++i)
        cmvn_frame<false, true, false, kPlanes, kFp16, kOut>(c, t0, i, xv[i], zero2, stat, pa[i], ps[i]);
    } else {
      const float2 *go = ro + (t0 & (kCmvnRing - 1)) * kBlock;
      float2 xp[kCmvnUnroll];
#pragma unroll
      for (int i = 0; i < kCmvnUnroll; ++i) xp[i] = go[i * kBlock];
      if (w) {
#pragma unroll
        for (int i = 0; i < kCmvnUnroll; ++i)
          cmvn_frame<true, false, true, kPlanes, kFp16, kOut>(c, t0, i, xv[i], xp[i], stat, 0.0f, scale_full);
      } else {
#pragma unroll
        for (int i = 0; i < kCmvnUnroll; ++i)
          cmvn_frame<true, false, false, kPlanes, kFp16, kOut>(c, t0, i, xv[i], xp[i], stat, 0.0f, scale_full);
      }
    }
  }
  // the last T % 8 frames, one at a time straight from global memory
  for (int t = T8; t < T; ++t) {
    const float2 x = *reinterpret_cast<const float2 *>(c.x + static_cast<int64_t>(t) * kMel);
    wide = wide || cmvn_out_of_range(x.x) || cmvn_out_of_range(x.y);
    if (t < kCmvnWindow) {
      cmvn_frame<false, true, false, kPlanes, kFp16, kOut>(c, t, 0, x, zero2, stat, s_alpha[t], s_scale[t]);
    } else {
      const float2 xo = *reinterpret_cast<const float2 *>(c.x + static_cast<int64_t>(t - kCmvnWindow) * kMel);
      if (wide) cmvn_frame<true, false, true, kPlanes, kFp16, kOut>(c, t, 0, x, xo, stat, 0.0f, scale_full);
      else cmvn_frame<true, false, false, kPlanes, kFp16, kOut>(c, t, 0, x, xo, stat, 0.0f, scale_full);
    }
  }

  // replicated edge rows of the padded planes (AcousticModel::SpliceFeats clamps at the
  // utterance edges, src/am.cc:65-88): copies of this thread's own first / last element
  if (kPlanes >= 1) {
    typedef unsigned int u32;
    const u32 h0 = *reinterpret_cast<const u32 *>(c.ph);
    const u32 h1 = *reinterpret_cast<const u32 *>(c.ph + static_cast<int64_t>(T - 1) * dim_pad);
    for (int r = 1; r <= left; ++r) *reinterpret_cast<u32 *>(c.ph - static_cast<int64_t>(r) * dim_pad) = h0;
    for (int r = 0; r < right; ++r) *reinterpret_cast<u32 *>(c.ph + static_cast<int64_t>(T + r) * dim_pad) = h1;
    if (kPlanes == 2) {
      const u32 l0 = *reinterpret_cast<const u32 *>(c.pl);
      const u32 l1 = *reinterpret_cast<const u32 *>(c.pl + static_cast<int64_t>(T - 1) * dim_pad);
      for (int r = 1; r <= left; ++r) *reinterpret_cast<u32 *>(c.pl - static_cast<int64_t>(r) * dim_pad) = l0;
      for (int r = 0; r < right; ++r) *reinterpret_cast<u32 *>(c.pl + static_cast<int64_t>(T + r) * dim_pad) = l1;
    }
  }
}

// splitmix64 finaliser; must match pocketkaldi_b200/synth.py
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

__global__ void synth_pcm_kernel(int16_t *__restrict__ pcm, const int64_t *__restrict__ sample_off,
                                 const int32_t *__restrict__ num_samples, int n_utts, uint64_t seed,
                                 uint64_t first_utt) {
  const int u = blockIdx.y;
  if (u >= n_utts) return;
  const uint64_t key = mix64(seed * 0x9E3779B97F4A7C15ull + (first_utt + u));
  const int n = num_samples[u];
  int16_t *dst = pcm + sample_off[u];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint64_t h = mix64(key + static_cast<uint64_t>(i) * 0x9E3779B97F4A7C15ull);
    const int64_t s = static_cast<int64_t>((h & 0xffff) + ((h >> 16) & 0xffff) +
                                           ((h >> 32) & 0xffff) + (h >> 48)) - 2 * 65535;
    dst[i] = static_cast<int16_t>((s * 5196) >> 16);
  }
}

__global__ void checksum_kernel(const float *__restrict__ x, int64_t n, double *sum) {
  double acc = 0.0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    acc += static_cast<double>(x[i]);
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ double s[32];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (blockDim.x >> 5); ++i) t += s[i];
    atomicAdd(sum, t);
  }
}

}  // namespace

// Host restatement of the count-dependent part of SmoothStats / Apply
// (src/cmvn.cc:73-101): for n = min(t+1, 600) frames in the window,
// alpha = float(min(600-n, 200) / Gc) (0 once n == 600), count' = n + alpha*Gc
// in float, scale = float(1 / double(count')).
int prepare_cmvn_tables(Ctx *c, const float *global_stats) {
  if (c->cmvn_valid && memcmp(c->cmvn_global, global_stats, sizeof(c->cmvn_global)) == 0)
    return PKB_OK;
  PKB_REQUIRE(global_stats[kMel] > 0.0f, "cmvn: global frame count must be positive");
  std::vector<float> tab(2 * kCmvnWindow + PKB_CMVN_STATS_DIM);
  const float gc = global_stats[kMel];
  for (int t = 0; t < kCmvnWindow; ++t) {
    float count_f = static_cast<float>(t + 1);
    double count = count_f;
    float alpha = 0.0f;
    if (count < kCmvnWindow) {
      double from_global = kCmvnWindow - count;
      double global_count = gc;
      if (from_global > kCmvnGlobal) from_global = kCmvnGlobal;
      alpha = static_cast<float>(from_global / global_count);
      volatile float prod = alpha * gc;
      count_f = count_f + prod;
    }
    double cnt = count_f;
    tab[t] = alpha;
    tab[kCmvnWindow + t] = static_cast<float>(1 / cnt);
  }
  memcpy(&tab[2 * kCmvnWindow], global_stats, sizeof(float) * PKB_CMVN_STATS_DIM);
  PKB_TRY(c->cmvn_tab.ensure(tab.size() * sizeof(float)));
  PKB_CUDA(cudaMemcpyAsync(c->cmvn_tab.p, tab.data(), tab.size() * sizeof(float),
                           cudaMemcpyHostToDevice, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));  // tab is a stack-scoped host vector
  memcpy(c->cmvn_global, global_stats, sizeof(c->cmvn_global));
  c->cmvn_valid = true;
  return PKB_OK;
}

int launch_cmvn(Ctx *c, const float *d_raw, const BatchMeta &m, float *d_out,
                const PaddedPlanes *planes) {
  if (m.n_utts == 0 || m.total_frames == 0) return PKB_OK;
  PKB_REQUIRE(c->cmvn_valid, "cmvn: tables not prepared");
  const int64_t threads = static_cast<int64_t>(m.n_utts) * kCmvnThreadsPerUtt;
  // a chain is sequential in t, so parallelism is n_utts * 20 threads: small batches run as
  // single-warp blocks spread over all SM sub-partitions instead of a few 5-warp blocks
  const int block = threads >= static_cast<int64_t>(c->sm_count) * 2 * 160 ? 160 : 32;
  const int grid = static_cast<int>((threads + block - 1) / block);
  // per-thread rings: x and x_old pairs
  const size_t dyn_smem = static_cast<size_t>(2) * kCmvnGroups * kCmvnUnroll * block * sizeof(float2);
  LaunchScope scope(c, PKB_KERNEL_CMVN);
  __nv_bfloat16 *hi = planes ? planes->hi : nullptr, *lo = planes ? planes->lo : nullptr;
  const int n_planes = hi ? (lo ? 2 : 1) : 0;
  const bool fp16 = planes && planes->fp16;
  PKB_REQUIRE(!planes || planes->dim_pad == kMel, "cmvn: operand planes must have a row pitch of %d elements", kMel);
#define PKB_CMVN_LAUNCH3(PL, FP, OUT, BLK)                                                               \
  do {                                                                                                  \
    if (dyn_smem > 40 * 1024)                                                                           \
      cudaFuncSetAttribute(cmvn_kernel<PL, FP, OUT, BLK>,                                               \
                           cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dyn_smem));    \
    cmvn_kernel<PL, FP, OUT, BLK><<<grid, BLK, dyn_smem, c->stream>>>(                                  \
        d_raw, m.d_frame_off, m.d_num_frames, m.n_utts, c->cmvn_tab.as<float>(), d_out, hi, lo,         \
        planes ? planes->d_pad_off : nullptr, planes ? planes->left : 0, planes ? planes->right : 0,    \
        planes ? planes->dim_pad : 0);                                                                  \
  } while (0)
#define PKB_CMVN_LAUNCH2(PL, FP, OUT)                    \
  do {                                                   \
    if (block == 160) PKB_CMVN_LAUNCH3(PL, FP, OUT, 160); \
    else PKB_CMVN_LAUNCH3(PL, FP, OUT, 32);               \
  } while (0)
#define PKB_CMVN_LAUNCH(PL, FP)                  \
  do {                                           \
    if (d_out) PKB_CMVN_LAUNCH2(PL, FP, true);   \
    else PKB_CMVN_LAUNCH2(PL, FP, false);        \
  } while (0)
  PKB_REQUIRE(d_out || n_planes > 0, "cmvn: no output requested");
  if (n_planes == 0) PKB_CMVN_LAUNCH2(0, false, true);
  else if (n_planes == 1 && !fp16) PKB_CMVN_LAUNCH(1, false);
  else if (n_planes == 1 && fp16) PKB_CMVN_LAUNCH(1, true);
  else if (n_planes == 2 && !fp16) PKB_CMVN_LAUNCH(2, false);
  else PKB_CMVN_LAUNCH(2, true);
#undef PKB_CMVN_LAUNCH3
#undef PKB_CMVN_LAUNCH2
#undef PKB_CMVN_LAUNCH
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

int launch_synth_pcm(Ctx *c, int16_t *d_pcm, const BatchMeta &m, uint64_t seed,
                     uint64_t first_utt) {
  if (m.n_utts == 0) return PKB_OK;
  int max_n = 0;
  for (int32_t n : m.num_samples) max_n = std::max(max_n, n);
  if (max_n == 0) return PKB_OK;
  // grid.y is limited to 65535: loop over slabs of utterances
  const int bx = std::min((max_n + 255) / 256, 64);
  for (int u0 = 0; u0 < m.n_utts; u0 += 32768) {
    const int nu = std::min(32768, m.n_utts - u0);
    LaunchScope scope(c, PKB_KERNEL_MISC);
    synth_pcm_kernel<<<dim3(bx, nu), 256, 0, c->stream>>>(d_pcm, m.d_sample_off + u0,
                                                          m.d_num_samples + u0, nu, seed,
                                                          first_utt + u0);
    PKB_CUDA(cudaGetLastError());
  }
  return PKB_OK;
}

int launch_checksum(Ctx *c, const float *d, int64_t n, double *d_sum) {
  PKB_CUDA(cudaMemsetAsync(d_sum, 0, sizeof(double), c->stream));
  if (n == 0) return PKB_OK;
  const int grid = static_cast<int>(std::min<int64_t>((n + 255) / 256, c->sm_count * 8));
  LaunchScope scope(c, PKB_KERNEL_MISC);
  checksum_kernel<<<grid, 256, 0, c->stream>>>(d, n, d_sum);
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

}  // namespace pkb
