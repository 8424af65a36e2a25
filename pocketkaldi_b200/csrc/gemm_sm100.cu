// Warp-specialised persistent GEMM for sm_100a: TMA -> shared memory (128-byte
// swizzle) -> tcgen05.mma (BF16 x BF16 -> FP32 accumulator in TMEM) -> tcgen05.ld
// epilogue with the fused element-wise layers.
//
// Replaces GEMM<float>::Gemm (src/gemm.cc:69-125) and its AVX2 micro-kernel
// (src/gemm_haswell.cc:72-632) for LinearLayer::Propagate (src/nnet.cc:22-36), with
// ReLULayer / NormalizeLayer (src/nnet.cc:49-75) and the exp/sum half of
// SoftmaxLayer (src/vector.cc:264-277) folded into the epilogue. Weights are used
// in their on-disk [out][in] layout (K-major for both operands), so the transpose
// of LinearLayer::LinearLayer (src/nnet.cc:16-17) disappears.
//
// CTA: warp 0 lane 0 TMA producer, warp 1 lane 0 MMA issuer, warp 2 TMEM allocator, warps 4+
// epilogue (TMEM lane quadrant = warp % 4; 8 warps for single-plane hidden stages, 4 in BF16X3,
// 16 = two teams of 8 for the output stage). Three pipelines: smem full/empty ring (TMA <-> MMA),
// TMEM full/empty double buffer (MMA <-> epilogue), static persistent tile loop with N fastest
// so that co-resident CTAs share the activation tile in L2 (output stage with softmax: grouped
// schedule, see get_tile). Hidden stages (and the BF16X3 output stage) run as CTA pairs
// (cta_group::2): one 256-row MMA tile per cluster of two, each CTA loading half of the W tile.
//
// BF16X3 / FP16X3: every operand is carried as two 16-bit planes (hi, lo = rn16(x - hi)) and
// each K step issues hi*hi + lo*hi + hi*lo into the same accumulator, which brings
// the product error down to ~2^-16 (2^-22) relative (FP32-class for this workload).
//
// FP16C8 (operand mode 3): the same first-order correction at two thirds of the tensor work.
// The two cross terms only need ~4 bits because they are 2^-11 of the product, so they are
// carried as FP8 (E4M3) planes and run at twice the FP16 MMA rate:
//   acc = [ e4m3(a_lo * 2^11) * e4m3(W16 * 2^4)  +  e4m3(a16 * 2^2) * e4m3(W_lo * 2^13) ]   (kind::f8f6f4)
//   acc = a16 * W16 + acc * 2^-15                                  (first kind::f16 MMA: scale-input-d)
// i.e. all correction k-blocks of a tile are accumulated first at 2^15 times the final scale and
// the first main MMA folds them in. One smem slot holds either a 64-wide FP16 k-block or a
// 128-wide FP8 k-block (same bytes, same 128-byte swizzle, same descriptor advance).

#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "gemm_sm100.cuh"

namespace pkb {

namespace {

constexpr int kMainThreads = 128;   // warps 0-3: TMA producer, MMA issuer, TMEM allocator, spare
// FINAL: two teams of 8 epilogue warps, team t owns TMEM accumulator stage t (every other tile),
// so one team's softmax exchange latency is covered by the other team's work.
// Hidden stages: one team; 8 warps (two per lane quadrant, half of the columns each) when there
// is one operand plane, 4 in BF16X3 where the staging tiles are twice as large and the MMA time
// per tile is three times longer anyway.
// Measured on B200 (config 3, 1024 utterances): a second hidden epilogue team (16 warps, 96
// registers, one pipeline stage less) is 5 % slower than one team, and dropping the back-off
// sleeps of the producer / MMA waits changes nothing -- the hidden stages are bound by the
// TMA -> MMA stream, not by the epilogue (PKB_GEMM_DEBUG=1 prints the per-tile cycle split).
// One output-stage team of 16 warps (four column quarters per lane quadrant) is correct but 6-14 %
// slower than two teams: pass 2 is bound by the turnaround of each warp's single TMA staging tile
// and the exchange latency, which only another team's work can cover.
// `planes` is the operand mode of the main loop: 1 = one 16-bit plane, 2 = hi + lo planes (three
// MMAs per product), 3 = FP16 + FP8 corrections (two MMA-equivalents per product).
// Accumulator stages in TMEM. The output stage's drain (two passes over the accumulator with the
// cross-CTA softmax exchange in between, ~17k cycles) is twice as long as a single-plane MMA fill
// (8k), so two 256-column stages leave that stage epilogue-bound. Four 128-column stages with one
// epilogue team each were measured on B200 and are not used: a 128x128 tcgen05.mma of one CTA
// reads 8 KB of shared memory per 64 cycles, exactly the 128 B/cycle the SM has, and the fill
// slows down by more than the extra stages gain (output stage 38.8 -> 50.0 ms per config-3 step).
// Releasing the stage after ONE pass (pass 1 also writes the logits through TMA stores, the warp
// finishes its 32 x 128 block in place from L2 once the lse is known) was measured too: the MMA
// warp no longer waits for TMEM, but the extra write + read + write of every output tile competes
// with the operand loads (wait for shared-memory stages 3.7k -> 7.3k cycles per tile) and the
// in-place finish takes as long as the pass it replaces (41.3 -> 45.5 ms, 43.3 ms with CTA pairs).
constexpr int kAccStages = 2;
constexpr int epi_teams(bool final) { return final ? 2 : 1; }
constexpr int team_warps(bool final, int planes) { return final ? 8 : (planes == 2 ? 4 : kHidWarps); }
constexpr int epi_warps(bool final, int planes) { return epi_teams(final) * team_warps(final, planes); }
constexpr int num_threads(bool final, int planes) { return kMainThreads + 32 * epi_warps(final, planes); }
// bytes of epilogue staging per warp of a hidden stage: one 32 x 128-byte tile per 16-bit output
// plane, or the FP16 tile plus two 32 x 64-byte FP8 tiles
constexpr uint32_t hid_stage_bytes(int planes, bool out8) { return (out8 || planes == 2) ? 8192u : 4096u; }
// Output stage epilogue: one row per lane, rows staged in shared memory and written by TMA bulk
// tensor stores. An accumulator-fragment variant (tcgen05.ld 16x256b, four lanes writing 32
// contiguous bytes of a row straight to global memory: no staging, no proxy fences, 64 KB more
// shared memory for the operand ring) was measured on B200 and dropped: its stores are whole
// sectors but four times as many L1->L2 write requests as full 128-byte lines, and pass 2 went
// from 8.9k to 14.8k cycles per tile and team (output stage 43.5 -> 56.6 ms per config-3 step).
constexpr uint32_t kFinalStageBytes = 16u * 4096u;
constexpr int kMaxStages = 8;
// clock64 probes of the pipeline phases (PKB_GEMM_DEBUG=1 prints them). Compiled in only with
// -DPKB_GEMM_PROBES: even switched off at run time they cost the hidden stages cycles.
#ifdef PKB_GEMM_PROBES
constexpr bool kProbes = true;
#else
constexpr bool kProbes = false;
#endif
constexpr uint32_t kSmemBudget = 227 * 1024;

// ---------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Bounded wait: a pipeline bug turns into a trap (reported as a launch failure)
// instead of hanging the GPU.
template <int kSleepNs = 0>
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (kSleepNs > 0) __nanosleep(kSleepNs);  // keep the spinning lane off the issue port
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}

__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar,
                                            int c_inner, int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}

// shared -> global bulk tensor store of one {32 cols x 32 rows} FP32 box (clipped at the
// tensor's edges by the TMA unit)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, uint32_t src, int c_inner,
                                             int c_outer) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(src), "r"(c_inner), "r"(c_outer)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int kPending>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of a cluster share one 256-row MMA tile. In a cluster
// launch bit 24 of a shared-window address selects the CTA of the pair; clearing it addresses
// the same offset in the leader (even) CTA (cute::Sm100MmaPeerBitMask).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t *bar, uint32_t rank) {
  asm volatile(
      "{\n"
      ".reg .b32 ra;\n"
      "mapa.shared::cluster.u32 ra, %0, %1;\n"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(rank)
      : "memory");
}
// both CTAs of a pair load their part of a stage and signal the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_pair(void *dst, const CUtensorMap *map, uint64_t *bar,
                                                 int c_inner, int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c_inner),
      "r"(c_outer)
      : "memory");
}

template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t *dst, uint32_t ncols) {
  if (CG == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(dst)),
                 "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(dst)),
                 "r"(ncols)
                 : "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_relinquish() {
  if (CG == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if (CG == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, BF16 inputs, FP32 accumulate.
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  if (CG == 1)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// Same for FP8 (E4M3) operands: K = 32 per instruction.
template <int CG>
__device__ __forceinline__ void umma_f8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                        uint32_t idesc, uint32_t accumulate) {
  if (CG == 1)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D = A * B + D * 2^-15 (scale-input-d of kind::f16): folds the FP8 correction sum, which was
// accumulated at 2^15 times the final scale, into the first main MMA of a tile.
template <int CG>
__device__ __forceinline__ void umma_f16_fold15(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                                uint32_t idesc) {
  if (CG == 1)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, 1, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p, 15;\n"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc)
        : "memory");
  else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, 1, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p, 15;\n"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc)
        : "memory");
}

// Arrives on `bar` once all previously issued tcgen05.mma of this thread finished; for a CTA
// pair the arrival is multicast to the barrier at the same offset in both CTAs.
template <int CG>
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  if (CG == 1) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
  } else {
    const uint16_t mask = 3;
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
        "[%0], %1;" ::"r"(smem_u32(bar)),
        "h"(mask)
        : "memory");
  }
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte-swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes
// apart (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout SWIZZLE_128B=2 [61,64)).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// cute::UMMA::InstrDescriptor for kind::f16: D=F32 (1<<4), A=B=BF16 (1<<7, 1<<10),
// both K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29).
// fmt: 1 = BF16, 0 = F16 for both operands.
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, uint32_t fmt) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "r"(addr)
               : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u32(uint32_t *p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

__device__ __forceinline__ float exp2f_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
  __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t *>(&v);
}

// two floats -> two E4M3 bytes (a in the low byte), round to nearest, saturating
__device__ __forceinline__ uint32_t pack_e4m3x2(float a, float b) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  return pack_e4m3x2(a, b) | (pack_e4m3x2(c, d) << 16);
}

struct SmemLayout {
  uint32_t stage_bytes, a_plane, w_plane, stages, epi_off, epi_bytes, bar_off, total;
};

__host__ __device__ inline SmemLayout smem_layout(int block_n, int planes, bool final, int cg, bool out8) {
  SmemLayout L;
  L.a_plane = kBlockM * kBlockK * 2;
  L.w_plane = (block_n / cg) * kBlockK * 2;  // a CTA pair splits the W tile
  // operand mode 3 streams one plane pair per slot (FP8 x FP8 or FP16 x FP16)
  L.stage_bytes = (planes == 2 ? 2 : 1) * (L.a_plane + L.w_plane);
  // epilogue staging: one 32-row x 128-byte tile per warp (and per plane for BF16 outputs)
  // FINAL adds the CTA's fixed bias and log-prior column tiles (2 x block_n floats) and a 128-row (max, sum) scratch per team
  // (and per row one more float for the compact mode's max(z - log_prior))
  L.epi_bytes = final ? kFinalStageBytes + 2 * block_n * 4 + 3 * 128 * 8 + 3 * 128 * 4
                      : epi_warps(false, planes) * hid_stage_bytes(planes, out8);
  uint32_t avail = kSmemBudget - 1024 /* alignment slack */ - 256 /* barriers */ - L.epi_bytes;
  L.stages = avail / L.stage_bytes;
  if (L.stages > kMaxStages) L.stages = kMaxStages;
  L.epi_off = L.stages * L.stage_bytes;
  L.bar_off = L.epi_off + L.epi_bytes;
  L.total = L.bar_off + 256 + 1024;
  return L;
}

// ---------------------------------------------------------------- kernel
// Persistent tile schedule. Default: tiles dealt round-robin with N fastest. Grouped (final
// softmax stage): the grid is a whole number of groups of n_tiles_n CTAs; a group owns one
// row block per iteration and each of its CTAs always owns the same column tile, so the CTAs
// that exchange softmax partials are a fixed team working on the same iteration.
// With CTA pairs (CG == 2) the unit of scheduling is the cluster: it owns a pair of
// consecutive row blocks, CTA `rank` of the pair taking row block 2*pair + rank (which may lie
// past the end of the matrix for an odd block count; such a CTA computes on zero rows).
template <int CG>
__device__ __forceinline__ bool get_tile(const GemmParams &p, int it, uint32_t rank, int &m_blk,
                                         int &n_blk) {
  const int unit = static_cast<int>(blockIdx.x) / CG;
  const int n_units = static_cast<int>(gridDim.x) / CG;
  const int m_units = (p.m_tiles + CG - 1) / CG;
  int mu;
  if (p.group_sched) {
    const int groups = n_units / p.n_tiles_n;
    mu = unit / p.n_tiles_n + it * groups;
    n_blk = unit % p.n_tiles_n;
  } else {
    const int tile = unit + it * n_units;
    mu = tile / p.n_tiles_n;
    n_blk = tile % p.n_tiles_n;
  }
  m_blk = mu * CG + static_cast<int>(rank);
  return mu < m_units;
}

// Operand maps. PLANES 1/2: a_hi (a_lo) x w_hi (w_lo) 16-bit planes. PLANES 3 (FP16C8):
//   a_hi = a16, a_lo = e4m3(a_lo * 2^11), a_x = e4m3(a16 * 2^2);  w_hi = W16, w_lo = e4m3(W_lo * 2^13),
//   w_x = e4m3(W16 * 2^4); correction phase A = a_lo x w_x, phase B = a_x x w_lo, main = a_hi x w_hi.
// OUT8 (hidden stages only): the epilogue writes the FP16C8 operand triple of the next stage.
template <int BN, int PLANES, bool FINAL, int CG, bool OUT8>
__global__ void __launch_bounds__(num_threads(FINAL, PLANES), 1)
gemm_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
            const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
            const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ CUtensorMap tm_a_x,
            const __grid_constant__ CUtensorMap tm_w_x, const GemmParams p) {
  static_assert(!(FINAL && OUT8), "the output stage writes FP32 / compact rows");
  extern __shared__ uint8_t smem_raw[];
  const SmemLayout L = smem_layout(BN, PLANES, FINAL, CG, OUT8);
  // 1024-byte alignment by pointer arithmetic on the shared array (not through an integer): the
  // compiler keeps the address space and emits LDS / STS instead of generic loads and stores
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + L.bar_off);
  uint64_t *full = bars;                       // [stages]
  uint64_t *empty = bars + kMaxStages;         // [stages]
  uint64_t *tfull = bars + 2 * kMaxStages;     // [kAccStages <= 4]
  uint64_t *tempty = bars + 2 * kMaxStages + 4;  // [kAccStages <= 4]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kMaxStages + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t S = L.stages;
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;

  if (warp == 0 && lane == 0) {
    if (FINAL) tma_prefetch_desc(&tm_out);
    tma_prefetch_desc(&tm_a_hi);
    tma_prefetch_desc(&tm_w_hi);
    if (PLANES >= 2) {
      tma_prefetch_desc(&tm_a_lo);
      tma_prefetch_desc(&tm_w_lo);
    }
    if (PLANES == 3) {
      tma_prefetch_desc(&tm_a_x);
      tma_prefetch_desc(&tm_w_x);
    }
  }
  if (warp == 1 && lane == 0) {
    for (uint32_t s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < kAccStages; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], CG * team_warps(FINAL, PLANES));  // both CTAs of a pair release the leader
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc<CG>(tmem_slot, kAccStages * BN);
    tmem_relinquish<CG>();
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();  // peers' barriers are initialised too
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      int m_blk, n_blk;
      for (int it = 0; get_tile<CG>(p, it, cta_rank, m_blk, n_blk); ++it) {
        const int m0 = m_blk * kBlockM;
        const int n0 = n_blk * BN + static_cast<int>(cta_rank) * (BN / CG);  // this CTA's W rows
        if (PLANES == 3) {
          // FP8 correction phases: 128-element (= 128-byte) k-blocks, A: a_lo8 x W_hi8, B: a_hi8 x W_lo8
          for (int kb = 0; kb < 2 * p.num_kb8; ++kb) {
            const bool phase_b = kb >= p.num_kb8;
            const int k0 = (phase_b ? kb - p.num_kb8 : kb) * 128;
            const CUtensorMap *ma = phase_b ? &tm_a_x : &tm_a_lo;
            const CUtensorMap *mw = phase_b ? &tm_w_lo : &tm_w_x;
            mbar_wait<64>(&empty[s], ph ^ 1);
            uint8_t *st = smem + s * L.stage_bytes;
            if (CG == 1) {
              mbar_expect_tx(&full[s], L.stage_bytes);
              tma_load_2d(st, ma, &full[s], k0, m0);
              tma_load_2d(st + L.a_plane, mw, &full[s], k0, n0);
            } else {
              if (leader) mbar_expect_tx(&full[s], 2 * L.stage_bytes);
              tma_load_2d_pair(st, ma, &full[s], k0, m0);
              tma_load_2d_pair(st + L.a_plane, mw, &full[s], k0, n0);
            }
            if (++s == S) { s = 0; ph ^= 1; }
          }
        }
        constexpr int kWOff = PLANES == 2 ? 2 : 1;  // W planes follow the A planes of a slot
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait<64>(&empty[s], ph ^ 1);
          uint8_t *st = smem + s * L.stage_bytes;
          if (CG == 1) {
            mbar_expect_tx(&full[s], L.stage_bytes);
            tma_load_2d(st, &tm_a_hi, &full[s], kb * kBlockK, m0);
            tma_load_2d(st + kWOff * L.a_plane, &tm_w_hi, &full[s], kb * kBlockK, n0);
            if (PLANES == 2) {
              tma_load_2d(st + L.a_plane, &tm_a_lo, &full[s], kb * kBlockK, m0);
              tma_load_2d(st + 2 * L.a_plane + L.w_plane, &tm_w_lo, &full[s], kb * kBlockK, n0);
            }
          } else {
            // the leader's barrier collects the bytes of both CTAs' loads
            if (leader) mbar_expect_tx(&full[s], 2 * L.stage_bytes);
            tma_load_2d_pair(st, &tm_a_hi, &full[s], kb * kBlockK, m0);
            tma_load_2d_pair(st + kWOff * L.a_plane, &tm_w_hi, &full[s], kb * kBlockK, n0);
            if (PLANES == 2) {
              tma_load_2d_pair(st + L.a_plane, &tm_a_lo, &full[s], kb * kBlockK, m0);
              tma_load_2d_pair(st + 2 * L.a_plane + L.w_plane, &tm_w_lo, &full[s], kb * kBlockK, n0);
            }
          }
          if (++s == S) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && leader) {  // a CTA pair's MMAs are issued by the leader alone
      const uint32_t idesc = make_idesc(kBlockM * CG, BN, p.fp16 ? 0u : 1u);
      uint32_t s = 0, ph = 0;
      int m_blk, n_blk;
      for (int it = 0; get_tile<CG>(p, it, cta_rank, m_blk, n_blk); ++it) {
        const uint32_t as = it % kAccStages, aph = (it / kAccStages) & 1;
        long long tw0 = 0, tw_full = 0;
        if (kProbes && p.dbg != nullptr) tw0 = clock64();
        mbar_wait<32>(&tempty[as], aph ^ 1);
        tc_fence_after();
        if (kProbes && p.dbg != nullptr) p.dbg[static_cast<size_t>(blockIdx.x) * 16 + 6] += clock64() - tw0;
        const uint32_t d_tmem = tmem_base + as * BN;
        if (PLANES == 3) {
          // correction sum first (FP8, K = 32 per instruction = the same 32-byte descriptor step)
          const uint32_t idesc8 = make_idesc(kBlockM * CG, BN, 0u);  // E4M3 is format 0 of kind::f8f6f4
          for (int kb = 0; kb < 2 * p.num_kb8; ++kb) {
            mbar_wait(&full[s], ph);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + s * L.stage_bytes);
            const uint64_t a8 = make_smem_desc(sa);
            const uint64_t w8 = make_smem_desc(sa + L.a_plane);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t adv = static_cast<uint64_t>((k * 32) >> 4);
              umma_f8<CG>(d_tmem, a8 + adv, w8 + adv, idesc8, (kb | k) != 0);
            }
            umma_commit<CG>(&empty[s]);
            if (++s == S) { s = 0; ph ^= 1; }
          }
        }
        constexpr int kWOff = PLANES == 2 ? 2 : 1;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          if (kProbes && p.dbg != nullptr) tw0 = clock64();
          mbar_wait(&full[s], ph);
          tc_fence_after();
          if (kProbes && p.dbg != nullptr) tw_full += clock64() - tw0;
          const uint32_t sa = smem_u32(smem + s * L.stage_bytes);
          const uint32_t sw = sa + kWOff * L.a_plane;
          const uint64_t a_hi = make_smem_desc(sa);
          const uint64_t w_hi = make_smem_desc(sw);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            const uint64_t adv = static_cast<uint64_t>((k * kUmmaK * 2) >> 4);
            if (PLANES == 3 && k == 0) {
              // the tile's first main MMA folds the correction sum in (acc * 2^-15 + a16 * W16)
              if (kb == 0) umma_f16_fold15<CG>(d_tmem, a_hi + adv, w_hi + adv, idesc);
              else umma_bf16<CG>(d_tmem, a_hi + adv, w_hi + adv, idesc, 1);
            } else {
              umma_bf16<CG>(d_tmem, a_hi + adv, w_hi + adv, idesc, PLANES == 3 ? 1u : ((kb | k) != 0));
            }
          }
          if (PLANES == 2) {
            const uint64_t a_lo = make_smem_desc(sa + L.a_plane);
            const uint64_t w_lo = make_smem_desc(sw + L.w_plane);
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              const uint64_t adv = static_cast<uint64_t>((k * kUmmaK * 2) >> 4);
              umma_bf16<CG>(d_tmem, a_lo + adv, w_hi + adv, idesc, 1);
              umma_bf16<CG>(d_tmem, a_hi + adv, w_lo + adv, idesc, 1);
            }
          }
          umma_commit<CG>(&empty[s]);  // frees the smem stage (in both CTAs) once these MMAs retire
          if (++s == S) { s = 0; ph ^= 1; }
        }
        umma_commit<CG>(&tfull[as]);  // accumulator complete
        if (kProbes && p.dbg != nullptr) p.dbg[static_cast<size_t>(blockIdx.x) * 16 + 7] += tw_full;
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;  // TMEM lane quadrant
    // FINAL: team = accumulator stage; inside a team two warps per lane quadrant, each owning
    // half of the tile's columns
    constexpr int kTeams = epi_teams(FINAL);
    constexpr int kTeamWarps = team_warps(FINAL, PLANES);
    const int team = (warp - 4) / kTeamWarps;
    const int wt = (warp - 4) % kTeamWarps;
    constexpr int kHalves = kTeamWarps / 4;  // warps per lane quadrant
    const int chalf = wt >> 2;
    constexpr int kTeamThreads = 32 * kTeamWarps;
    // per-warp staging tile: 32 rows x 128 bytes, 16-byte chunks XOR-swizzled by (row & 7);
    // rows are written by their owner lane and read back 4 rows per instruction so that
    // every global store covers whole 128-byte lines
    uint8_t *stg = smem + L.epi_off + (warp - 4) * (FINAL ? 4096u : hid_stage_bytes(PLANES, OUT8));
    // OUT8: the two FP8 tiles (32 rows x 64 bytes, 16-byte chunks XOR-swizzled by (row >> 1) & 3)
    // follow the FP16 tile
    const uint32_t stg8_w = smem_u32(stg) + 4096 + lane * 64;
    const uint32_t stg_w = smem_u32(stg) + lane * 128;          // this lane's row
    // grouped schedule: this CTA's column tile never changes, keep its bias / log-prior in smem
    float *s_bias = reinterpret_cast<float *>(smem + L.epi_off + (FINAL ? kFinalStageBytes : 16u * 4096u));
    float *s_lp = s_bias + BN;
    constexpr int kEpiThreads = 32 * epi_warps(FINAL, PLANES);
    if (FINAL && p.group_sched) {
      const int nb = (static_cast<int>(blockIdx.x) / CG) % p.n_tiles_n;
      for (int i = threadIdx.x - kMainThreads; i < BN; i += kEpiThreads) {
        // padding columns (zero weights) get a bias of -inf in the softmax modes: their logit is
        // -inf, exp() == 0, without any per-element masking in pass 1; pass 2 never stores them
        s_bias[i] = (p.final_mode != 0 && nb * BN + i >= p.N_valid) ? -INFINITY : p.bias[nb * BN + i];
        s_lp[i] = p.log_prior[nb * BN + i];
      }
      named_bar_sync(3, kEpiThreads);
    }
    const int t_row = lane >> 3, t_chunk = lane & 7;            // transposed read role
    int m_blk, n_blk;
    for (int it = team; get_tile<CG>(p, it, cta_rank, m_blk, n_blk); it += kTeams) {
      const uint32_t as = it % kAccStages, aph = (it / kAccStages) & 1;
      const int m0 = m_blk * kBlockM;
      const int n0 = n_blk * BN;
      const int wrow0 = m0 + q * 32;  // first row of this warp
      const int row = wrow0 + lane;
      const bool row_ok = row < p.M;

      float rs = 1.0f;
      if (p.in_sumsq != nullptr && row_ok) {
        float ss = 0.0f;
        for (int i = 0; i < p.in_sumsq_tiles; ++i)
          ss += p.in_sumsq[static_cast<size_t>(row) * p.in_sumsq_tiles + i];
        rs = sqrtf(p.in_dim / ss);  // NormalizeLayer: no floor (src/nnet.cc:71-73)
      }
      rs *= p.acc_scale;  // FP16C8 weights are stored times a power of two (1 otherwise)

      long long tk0 = 0, tk1 = 0, tk2 = 0, tk3 = 0, tk4 = 0, tkm = 0;
      const bool dbg_on = kProbes && p.dbg != nullptr && warp == 4 && lane == 0;  // team 0
      if (dbg_on) tk0 = clock64();
      mbar_wait<32>(&tfull[as], aph);
      tc_fence_after();
      if (dbg_on) tk1 = clock64();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;

      if (!FINAL) {
        float sumsq = 0.0f;
        constexpr int kGroups = BN / 64 / kHalves;  // 64-column groups per warp
#pragma unroll 1
        for (int g = chalf * kGroups; g < (chalf + 1) * kGroups; ++g) {
          const int col0 = n0 + g * 64;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t v[32];
            if (dbg_on) tk2 = clock64();
            tmem_ld32(taddr + g * 64 + h * 32, v);
            tmem_ld_wait();
            if (dbg_on) { const long long t = clock64(); tk3 += t - tk2; tk2 = t; }
            float z[32];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b = __ldg(reinterpret_cast<const float4 *>(p.bias + col0 + h * 32 + i));
              z[i + 0] = fmaf(__uint_as_float(v[i + 0]), rs, b.x);
              z[i + 1] = fmaf(__uint_as_float(v[i + 1]), rs, b.y);
              z[i + 2] = fmaf(__uint_as_float(v[i + 2]), rs, b.z);
              z[i + 3] = fmaf(__uint_as_float(v[i + 3]), rs, b.w);
            }
            if (p.relu == 1) {
#pragma unroll
              for (int i = 0; i < 32; ++i) z[i] = fmaxf(z[i], 0.0f);
            } else if (p.relu == 2) {  // sigmoid (not a reference layer type; parity unpinned)
              // padding columns (z = 0) would become 0.5 and add 0.25 each to the NormalizeLayer
              // sum of squares of the row: keep them 0 like ReLU and "no activation" do
#pragma unroll
              for (int i = 0; i < 32; ++i)
                z[i] = col0 + h * 32 + i < p.N_valid ? 1.0f / (1.0f + expf(-z[i])) : 0.0f;
            }
            if (p.out_sumsq != nullptr) {
#pragma unroll
              for (int i = 0; i < 32; ++i) sumsq = fmaf(z[i], z[i], sumsq);
            }
            uint32_t hi[16];
#pragma unroll
            for (int i = 0; i < 16; ++i)
              hi[i] = p.fp16 ? pack_f16(z[2 * i], z[2 * i + 1]) : pack_bf16(z[2 * i], z[2 * i + 1]);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              st_shared_v4(stg_w + (((h * 4 + j) ^ (lane & 7)) << 4), hi[4 * j], hi[4 * j + 1],
                           hi[4 * j + 2], hi[4 * j + 3]);
            if (dbg_on) tkm += clock64() - tk2;
            if (OUT8) {
              // next stage's FP8 correction operands: e4m3((z - fp16(z)) * 2^11) and e4m3(fp16(z) * 2^2)
              uint32_t l8[8], h8[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float f[4], r[4];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const __half2 hh = *reinterpret_cast<const __half2 *>(&hi[2 * i + e]);
                  f[2 * e] = __low2float(hh);
                  f[2 * e + 1] = __high2float(hh);
                  r[2 * e] = (z[4 * i + 2 * e] - f[2 * e]) * 2048.0f;
                  r[2 * e + 1] = (z[4 * i + 2 * e + 1] - f[2 * e + 1]) * 2048.0f;
                }
                l8[i] = pack_e4m3x4(r[0], r[1], r[2], r[3]);
                h8[i] = pack_e4m3x4(f[0] * 4.0f, f[1] * 4.0f, f[2] * 4.0f, f[3] * 4.0f);
              }
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const uint32_t o = ((h * 2 + j) ^ ((lane >> 1) & 3)) << 4;
                st_shared_v4(stg8_w + o, l8[4 * j], l8[4 * j + 1], l8[4 * j + 2], l8[4 * j + 3]);
                st_shared_v4(stg8_w + 2048 + o, h8[4 * j], h8[4 * j + 1], h8[4 * j + 2], h8[4 * j + 3]);
              }
            }
            if (PLANES == 2 && !OUT8) {
              uint32_t lo[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                if (p.fp16) {
                  const __half2 hh = *reinterpret_cast<const __half2 *>(&hi[i]);
                  lo[i] = pack_f16(z[2 * i] - __low2float(hh), z[2 * i + 1] - __high2float(hh));
                } else {
                  const __nv_bfloat162 hh = *reinterpret_cast<__nv_bfloat162 *>(&hi[i]);
                  lo[i] = pack_bf16(z[2 * i] - __low2float(hh), z[2 * i + 1] - __high2float(hh));
                }
              }
#pragma unroll
              for (int j = 0; j < 4; ++j)
                st_shared_v4(stg_w + 4096 + (((h * 4 + j) ^ (lane & 7)) << 4), lo[4 * j],
                             lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
            }
          }
          __syncwarp();
          if (dbg_on) tk2 = clock64();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = 4 * i + t_row;
            if (wrow0 + rr < p.M) {
              const uint32_t src = smem_u32(stg) + rr * 128 + ((t_chunk ^ (rr & 7)) << 4);
              const size_t off = static_cast<size_t>(wrow0 + rr) * p.ld_out + col0 + t_chunk * 8;
              *reinterpret_cast<uint4 *>(p.out_hi + off) = ld_shared_v4(src);
              if (PLANES == 2 && !OUT8) *reinterpret_cast<uint4 *>(p.out_lo + off) = ld_shared_v4(src + 4096);
            }
          }
          if (OUT8) {
            // 64-byte rows: four lanes per row, eight rows per instruction
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = 8 * i + (lane >> 2), ch = lane & 3;
              if (wrow0 + rr < p.M) {
                const uint32_t src = smem_u32(stg) + 4096 + rr * 64 + ((ch ^ ((rr >> 1) & 3)) << 4);
                const size_t off = static_cast<size_t>(wrow0 + rr) * p.ld_out + col0 + ch * 16;
                *reinterpret_cast<uint4 *>(p.out8_lo + off) = ld_shared_v4(src);
                *reinterpret_cast<uint4 *>(p.out8_hi + off) = ld_shared_v4(src + 2048);
              }
            }
          }
          __syncwarp();
          if (dbg_on) tk4 += clock64() - tk2;
        }
        // all TMEM reads of this accumulator are done: hand it back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (leader) mbar_arrive(&tempty[as]); else mbar_arrive_remote(&tempty[as], 0);
        }
        if (p.out_sumsq != nullptr && row_ok)
          p.out_sumsq[(static_cast<size_t>(row) * p.n_tiles_n + n_blk) * kHalves + chalf] = sumsq;
        if (dbg_on) {
          const long long tk5 = clock64();
          long long *d = p.dbg + static_cast<size_t>(blockIdx.x) * 16;
          d[0] += tk1 - tk0;        // wait for the accumulator
          d[1] += tk3;              // TMEM loads
          d[2] += tk4;              // staged global stores
          d[3] += tk5 - tk1;        // whole tile after the wait
          d[4] += tkm;              // bias / ReLU / pack / staging writes
          d[5] += 1;
        }
      } else {
        // ---- pass 1 (softmax only): per-row (max, sum exp) over this warp's half of the
        //      tile's columns, exchanged with the warps / CTAs that own the other columns
        constexpr int kChunks = BN / 32 / kHalves;  // 32-column chunks per epilogue warp
        static_assert(kChunks % 2 == 0, "the compact output packs two 32-column chunks per staging row");
        const int cbase = chalf * (BN / kHalves);
        const float kLog2e = 1.4426950408889634f;
        float lse = 0.0f, off16 = 0.0f;
        if (p.final_mode != 0) {
          float run_max = -INFINITY, run_sum = 0.0f;
          float run_mzl = -INFINITY;  // compact mode: max over columns of z - log_prior
          const bool compact = p.final_mode == 3;
          // the per-row maximum of z - log_prior is exchanged for the compact output and for the
          // near-tie count of the refinement pass (p.near_cnt)
          const bool want_mzl = compact || p.near_cnt != nullptr;
#pragma unroll 1
          for (int c = 0; c < kChunks; ++c) {
            const int col0 = n0 + cbase + c * 32;
            const int nvalid = p.N_valid - col0;
            if (nvalid <= 0) break;
            uint32_t v[32];
            tmem_ld32(taddr + cbase + c * 32, v);
            tmem_ld_wait();
            float z[32];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b = *reinterpret_cast<const float4 *>(s_bias + cbase + c * 32 + i);
              z[i + 0] = fmaf(__uint_as_float(v[i + 0]), rs, b.x);
              z[i + 1] = fmaf(__uint_as_float(v[i + 1]), rs, b.y);
              z[i + 2] = fmaf(__uint_as_float(v[i + 2]), rs, b.z);
              z[i + 3] = fmaf(__uint_as_float(v[i + 3]), rs, b.w);
            }
            float cmax = z[0];
#pragma unroll
            for (int i = 1; i < 32; ++i) cmax = fmaxf(cmax, z[i]);
            if (want_mzl) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                const float4 lp = *reinterpret_cast<const float4 *>(s_lp + cbase + c * 32 + i);
                run_mzl = fmaxf(run_mzl, fmaxf(fmaxf(z[i] - lp.x, z[i + 1] - lp.y),
                                               fmaxf(z[i + 2] - lp.z, z[i + 3] - lp.w)));
              }
            }
            const float nm = fmaxf(run_max, cmax);
            const float off = -nm * kLog2e;
            float acc = 0.0f;
#pragma unroll
            for (int i = 0; i < 32; ++i) acc += exp2f_fast(fmaf(z[i], kLog2e, off));
            run_sum = run_sum * exp2f_fast((run_max - nm) * kLog2e) + acc;
            run_max = nm;
          }
          // (1) fold the two column halves of this CTA through shared memory, then publish one
          //     (max, sum) per row and column tile, row-fastest so that every warp-wide access
          //     to the exchange buffer is one contiguous 256-byte segment
          const int rit = q * 32 + lane;  // row inside the tile
          // (kTeams * (kHalves - 1) == 2 or 3 scratch planes of 128 rows)
          float2 *s_half = reinterpret_cast<float2 *>(s_lp + BN) + team * (kHalves - 1) * kBlockM;
          float *s_half_mzl = reinterpret_cast<float *>(reinterpret_cast<float2 *>(s_lp + BN) + 3 * kBlockM) +
                              team * (kHalves - 1) * kBlockM;
          if (chalf != 0) {
            s_half[(chalf - 1) * kBlockM + rit] = make_float2(run_max, run_sum);
            if (want_mzl) s_half_mzl[(chalf - 1) * kBlockM + rit] = run_mzl;
          }
          if (dbg_on) tk2 = clock64();
          if (kHalves > 1) named_bar_sync(4 + team, kTeamThreads);
          unsigned long long *xbase =
              reinterpret_cast<unsigned long long *>(p.lse_part) + static_cast<size_t>(m_blk) * p.n_tiles_n * kBlockM;
          uint32_t *zbase = reinterpret_cast<uint32_t *>(p.mzl_part) + static_cast<size_t>(m_blk) * p.n_tiles_n * kBlockM;
          if (chalf == 0) {
            float nm = run_max, sm = run_sum;
#pragma unroll
            for (int h = 0; h < kHalves - 1; ++h) {
              const float2 o = s_half[h * kBlockM + rit];
              const float m2 = fmaxf(nm, o.x);
              sm = sm * exp2f_fast((nm - m2) * kLog2e) + o.y * exp2f_fast((o.x - m2) * kLog2e);
              nm = m2;
            }
            // one 64-bit word per (row, column tile): max in the low half, sum in the high half.
            // The buffer is pre-filled with 0xFF bytes by the launcher and an all-ones high half
            // (a NaN no computation below produces: sums are canonicalised) means "not written
            // yet" -- the data is its own ready flag, no counter, no release / acquire chain.
            if (sm != sm) sm = __int_as_float(0x7fc00000);
            st_relaxed_u64(xbase + n_blk * kBlockM + rit,
                           static_cast<unsigned long long>(__float_as_uint(nm)) |
                               (static_cast<unsigned long long>(__float_as_uint(sm)) << 32));
            if (want_mzl) {
              float mz = run_mzl;
#pragma unroll
              for (int h = 0; h < kHalves - 1; ++h) mz = fmaxf(mz, s_half_mzl[h * kBlockM + rit]);
              if (mz != mz) mz = __int_as_float(0x7fc00000);
              st_relaxed_u32(zbase + n_blk * kBlockM + rit, __float_as_uint(mz));
            }
          }
          // the scratch planes may be rewritten for this team's next tile only after they were read
          if (kHalves > 1) named_bar_sync(4 + team, kTeamThreads);
          if (dbg_on) tk3 = clock64();
          // (2) every lane collects the partials of its own row from the peer CTAs of this row
          //     block, kPollGroup loads in flight, polling until each word has been written.
          //     Measured (ncu cycles of the config-3 FP16 output stage, 12 column tiles): groups
          //     of 4 beat 1 / 2 / 3 / 6 / 8 / 12 / 16 (+15 % / +4 % / +1.5 % / +0.7 % / +3.7 % /
          //     +8 % / +9 %): re-polling a wide group while the last peer is late costs more than
          //     the extra round trips of a narrow one; the 100 ns back-off beats 0 / 200 / 400 ns.
          constexpr int kPollGroup = 4;
          {
            float mx = -INFINITY, ssum = 0.0f, mz = -INFINITY;
            const long long t0 = clock64();
            for (int j0 = 0; j0 < p.n_tiles_n; j0 += kPollGroup) {
              unsigned long long w[kPollGroup];
              uint32_t zz[kPollGroup];
              while (true) {
                bool ready = true;
#pragma unroll
                for (int j = 0; j < kPollGroup; ++j) {
                  const bool in = j0 + j < p.n_tiles_n;
                  w[j] = in ? ld_relaxed_u64(xbase + (j0 + j) * kBlockM + rit) : 0xff800000ull;  // (-inf, 0)
                  zz[j] = (in && want_mzl) ? ld_relaxed_u32(zbase + (j0 + j) * kBlockM + rit) : 0xff800000u;
                  ready = ready && static_cast<uint32_t>(w[j] >> 32) != 0xffffffffu && zz[j] != 0xffffffffu;
                }
                if (ready) break;
                // A peer that never arrives (it cannot with a co-resident grid) must not hang the
                // device, and a trap would poison the whole context: give up after ~20 s of
                // cycles, leave an error code for the host (check_device_error) and carry on.
                if (clock64() - t0 > 40000000000ll) {
                  if (p.err_flag != nullptr) *reinterpret_cast<volatile int *>(p.err_flag) = 1;
                  break;
                }
                __nanosleep(100);
              }
#pragma unroll
              for (int j = 0; j < kPollGroup; ++j) {
                const float ex = __uint_as_float(static_cast<uint32_t>(w[j]));
                const float ey = __uint_as_float(static_cast<uint32_t>(w[j] >> 32));
                const float nm = fmaxf(mx, ex);
                ssum = ssum * exp2f_fast((mx - nm) * kLog2e) + ey * exp2f_fast((ex - nm) * kLog2e);
                mx = nm;
                mz = fmaxf(mz, __uint_as_float(zz[j]));
              }
            }
            lse = mx + logf(ssum);
            if (want_mzl) {
              // reference point of this frame's 16-bit values: the largest max(z - lse, floor) - lp
              // unless the floor binds (softmax below 1e-20), which only moves the point
              off16 = mz - lse;
              if (compact && n_blk == 0 && chalf == 0 && row_ok) p.out_off[row] = off16;
            }
          }
        }
        if (dbg_on) tk4 = clock64();
        // ---- pass 2: final values -> swizzled staging tile -> TMA bulk tensor store; the TMA
        //      unit clips rows >= M and columns >= N_valid. One staging tile per warp: the
        //      previous store must have read it before it is rewritten (the other team's work
        //      fills that gap).
        const bool vec_ok = (p.ld_f32 & 3) == 0;
        const float floor_v = p.log_floor, sc = p.scale;
        if (p.final_mode == 3) {
          // compact: two 32-column chunks fill one 128-byte staging row of halves
          const bool vec16_ok = (p.ld_f32 & 7) == 0;
          const bool count_near = p.near_cnt != nullptr;
          const __half2 near2 = __float2half2_rn(-p.near_margin);
          __half2 cnt2 = __float2half2_rn(0.0f);  // <= 128 columns per thread: exact in FP16
#pragma unroll 1
          for (int c = 0; c < kChunks; c += 2) {
            const int col0 = n0 + cbase + c * 32;
            if (p.N_valid - col0 <= 0) break;
            uint32_t hbits[32];
#pragma unroll
            for (int hc = 0; hc < 2; ++hc) {
              uint32_t v[32];
              tmem_ld32(taddr + cbase + (c + hc) * 32, v);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                const float4 b = *reinterpret_cast<const float4 *>(s_bias + cbase + (c + hc) * 32 + i);
                const float4 lp = *reinterpret_cast<const float4 *>(s_lp + cbase + (c + hc) * 32 + i);
                const float t0 = fmaxf(fmaf(__uint_as_float(v[i + 0]), rs, b.x) - lse, floor_v) - lp.x - off16;
                const float t1 = fmaxf(fmaf(__uint_as_float(v[i + 1]), rs, b.y) - lse, floor_v) - lp.y - off16;
                const float t2 = fmaxf(fmaf(__uint_as_float(v[i + 2]), rs, b.z) - lse, floor_v) - lp.z - off16;
                const float t3 = fmaxf(fmaf(__uint_as_float(v[i + 3]), rs, b.w) - lse, floor_v) - lp.w - off16;
                hbits[hc * 16 + i / 2] = pack_f16(t0, t1);
                hbits[hc * 16 + i / 2 + 1] = pack_f16(t2, t3);
              }
            }
            if (count_near) {
              // columns within near_margin of this frame's best one: the stored value is the
              // distance from it. Padding columns (zero weights) are masked by their index.
              if (col0 + 64 <= p.N_valid) {
#pragma unroll
                for (int i = 0; i < 32; ++i)
                  cnt2 = __hadd2(cnt2, __hgt2(*reinterpret_cast<const __half2 *>(&hbits[i]), near2));
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  const __half2 g = __hgt2(*reinterpret_cast<const __half2 *>(&hbits[i]), near2);
                  const __half zero = __float2half(0.0f);
                  cnt2 = __hadd2(cnt2, __halves2half2(col0 + 2 * i < p.N_valid ? __low2half(g) : zero,
                                                      col0 + 2 * i + 1 < p.N_valid ? __high2half(g) : zero));
                }
              }
            }
            if (vec16_ok) {
              if (lane == 0) tma_store_wait_read<0>();
              __syncwarp();
#pragma unroll
              for (int j = 0; j < 8; ++j)
                st_shared_v4(stg_w + ((j ^ (lane & 7)) << 4), hbits[4 * j], hbits[4 * j + 1], hbits[4 * j + 2],
                             hbits[4 * j + 3]);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                tma_store_2d(&tm_out, smem_u32(stg), col0, wrow0);
                tma_store_commit();
              }
            } else if (row_ok) {
              uint16_t *dst = p.out_h16 + static_cast<size_t>(row) * p.ld_f32 + col0;
#pragma unroll
              for (int i = 0; i < 64; ++i)
                if (col0 + i < p.N_valid)
                  dst[i] = static_cast<uint16_t>((i & 1) ? (hbits[i >> 1] >> 16) : (hbits[i >> 1] & 0xffffu));
            }
          }
          if (count_near && row_ok) {
            const int n = static_cast<int>(__low2float(cnt2) + __high2float(cnt2));
            if (n > 0) atomicAdd(p.near_cnt + row, n);
          }
        } else {
        const bool count_near = p.near_cnt != nullptr && p.final_mode == 2;
        const float near_thr = off16 - p.near_margin;
        int near_n = 0;
#pragma unroll 1
        for (int c = 0; c < kChunks; ++c) {
          const int col0 = n0 + cbase + c * 32;
          const int nvalid = p.N_valid - col0;
          if (nvalid <= 0) break;
          uint32_t v[32];
          long long q0 = 0, q1 = 0, q2 = 0, q3 = 0;
          if (dbg_on) q0 = clock64();
          tmem_ld32(taddr + cbase + c * 32, v);
          tmem_ld_wait();
          if (dbg_on) q1 = clock64();
          float z[32];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b = p.group_sched
                                 ? *reinterpret_cast<const float4 *>(s_bias + cbase + c * 32 + i)
                                 : __ldg(reinterpret_cast<const float4 *>(p.bias + col0 + i));
            z[i + 0] = fmaf(__uint_as_float(v[i + 0]), rs, b.x);
            z[i + 1] = fmaf(__uint_as_float(v[i + 1]), rs, b.y);
            z[i + 2] = fmaf(__uint_as_float(v[i + 2]), rs, b.z);
            z[i + 3] = fmaf(__uint_as_float(v[i + 3]), rs, b.w);
          }
          if (p.final_mode == 1) {  // softmax probabilities (Nnet::Propagate)
#pragma unroll
            for (int i = 0; i < 32; ++i) z[i] = expf(z[i] - lse);
          } else if (p.final_mode == 2) {  // scaled log-likelihood (src/am.cc:106-112, decodable.cc:15)
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 lp = *reinterpret_cast<const float4 *>(s_lp + cbase + c * 32 + i);
              z[i + 0] = fmaxf(z[i + 0] - lse, floor_v) - lp.x;
              z[i + 1] = fmaxf(z[i + 1] - lse, floor_v) - lp.y;
              z[i + 2] = fmaxf(z[i + 2] - lse, floor_v) - lp.z;
              z[i + 3] = fmaxf(z[i + 3] - lse, floor_v) - lp.w;
            }
            if (count_near) {
              if (nvalid >= 32) {
#pragma unroll
                for (int i = 0; i < 32; ++i) near_n += z[i] > near_thr ? 1 : 0;
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) near_n += (i < nvalid && z[i] > near_thr) ? 1 : 0;
              }
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) z[i] *= sc;
          }
          if (vec_ok) {
            if (dbg_on) q2 = clock64();
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
            if (dbg_on) q3 = clock64();
#pragma unroll
            for (int j = 0; j < 8; ++j)
              st_shared_v4(stg_w + ((j ^ (lane & 7)) << 4), __float_as_uint(z[4 * j]),
                           __float_as_uint(z[4 * j + 1]), __float_as_uint(z[4 * j + 2]),
                           __float_as_uint(z[4 * j + 3]));
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&tm_out, smem_u32(stg), col0, wrow0);
              tma_store_commit();
            }
            if (dbg_on) {
              long long *d = p.dbg + static_cast<size_t>(blockIdx.x) * 16;
              d[8] += q1 - q0;             // pass 2: TMEM load
              d[9] += q2 - q1;             // pass 2: math
              d[10] += q3 - q2;            // pass 2: wait for the staging tile (previous TMA store)
              d[11] += clock64() - q3;     // pass 2: staging writes, proxy fence, TMA issue
            }
          } else if (row_ok) {
            float *dst = p.out_f32 + static_cast<size_t>(row) * p.ld_f32 + col0;
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (i < nvalid) dst[i] = z[i];
          }
        }
        if (count_near && row_ok && near_n > 0) atomicAdd(p.near_cnt + row, near_n);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (leader) mbar_arrive(&tempty[as]); else mbar_arrive_remote(&tempty[as], 0);
        }
        if (dbg_on) {
          const long long tk5 = clock64();
          long long *d = p.dbg + static_cast<size_t>(blockIdx.x) * 16;
          d[0] += tk1 - tk0;  // wait for the accumulator
          d[1] += tk2 - tk1;  // pass 1
          d[2] += tk3 - tk2;  // publish + peer wait
          d[3] += tk4 - tk3;  // combine partials
          d[4] += tk5 - tk4;  // pass 2
          d[5] += kTeams;  // tiles of this CTA (team 0 times every other one)
        }
      }
    }
    // shared memory must stay valid until the last bulk stores have read it
    if (FINAL && lane == 0) tma_store_wait_read<0>();
  }

  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<CG>(tmem_base, kAccStages * BN);
  }
}

template <int BN, int PLANES, bool FINAL, int CG, bool OUT8>
int launch_one(Ctx *c, const GemmMaps &mp, const GemmParams &p) {
  const CUtensorMap *a_hi = mp.a_hi, *a_lo = mp.a_lo, *w_hi = mp.w_hi, *w_lo = mp.w_lo;
  const CUtensorMap *a_x = PLANES == 3 ? mp.a_x : mp.a_hi, *w_x = PLANES == 3 ? mp.w_x : mp.w_hi;
  // output map of the final stage's TMA stores, boxes of 32 rows x 128 bytes; it needs a 16-byte
  // row pitch (hidden stages pass a dummy copy of the A map)
  CUtensorMap out_map = *a_hi;
  if (FINAL && p.final_mode == 3) {
    if ((p.ld_f32 & 7) == 0)
      PKB_TRY(encode_tensor_map(&out_map, CU_TENSOR_MAP_DATA_TYPE_UINT16, p.out_h16, p.N_valid, p.M,
                                static_cast<uint64_t>(p.N_valid) * sizeof(uint16_t), 64, 32,
                                CU_TENSOR_MAP_L2_PROMOTION_NONE));
  } else if (FINAL && (p.ld_f32 & 3) == 0) {
    PKB_TRY(encode_tensor_map(&out_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, p.out_f32, p.N_valid, p.M,
                              static_cast<uint64_t>(p.N_valid) * sizeof(float), 32, 32,
                              CU_TENSOR_MAP_L2_PROMOTION_NONE));
  }
  const SmemLayout L = smem_layout(BN, PLANES, FINAL, CG, OUT8);
  auto kern = gemm_kernel<BN, PLANES, FINAL, CG, OUT8>;
  PKB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
  GemmParams pp = p;
  pp.m_tiles = (p.M + kBlockM - 1) / kBlockM;
  pp.group_sched = 0;
  const int m_units = (pp.m_tiles + CG - 1) / CG;
  const int max_units = c->sm_count / CG;
  int grid = CG * static_cast<int>(std::min<int64_t>(static_cast<int64_t>(m_units) * p.n_tiles_n, max_units));
  if (FINAL && p.final_mode != 0) {
    if (p.n_tiles_n > c->sm_count) {
      set_error("launch_gemm: %d column tiles exceed the %d SMs of the device", p.n_tiles_n, c->sm_count);
      return PKB_ERR_UNSUPPORTED;
    }
    if (max_units / p.n_tiles_n < 1) {
      set_error("launch_gemm: %d column tiles of CTA %s do not fit the %d SMs of the device", p.n_tiles_n,
                CG == 2 ? "pairs" : "singles", c->sm_count);
      return PKB_ERR_UNSUPPORTED;
    }
    pp.group_sched = 1;
    grid = CG * std::min(max_units / p.n_tiles_n, m_units) * p.n_tiles_n;
  }
  pp.err_flag = c->err_dev;
  static const bool dbg_env = kProbes && getenv("PKB_GEMM_DEBUG") != nullptr;
  long long *dbg = nullptr;
  if (dbg_env) {
    cudaMalloc(&dbg, sizeof(long long) * 16 * grid);
    cudaMemsetAsync(dbg, 0, sizeof(long long) * 16 * grid, c->stream);
  }
  pp.dbg = dbg;
  {
  LaunchScope scope(c, FINAL ? PKB_KERNEL_GEMM_FINAL : PKB_KERNEL_GEMM);
  if (FINAL && p.final_mode != 0) {
    // the column tiles of a row block exchange softmax partials through global memory and wait
    // for each other: a cooperative launch guarantees that all CTAs are co-resident
    // (+1: a CTA pair may work on one row block past the end of the matrix)
    // exchange buffers: all-ones words mean "not written yet" (see the epilogue)
    const size_t words = (static_cast<size_t>((p.M + kBlockM - 1) / kBlockM) + 1) * p.n_tiles_n * kBlockM;
    PKB_CUDA(cudaMemsetAsync(p.lse_part, 0xFF, words * sizeof(float2), c->stream));
    if (p.final_mode == 3 || p.near_cnt != nullptr)
      PKB_CUDA(cudaMemsetAsync(p.mzl_part, 0xFF, words * sizeof(float), c->stream));
    CUtensorMap m0 = *a_hi, m1 = *a_lo, m2 = *w_hi, m3 = *w_lo, m5 = *a_x, m6 = *w_x;
    void *args[] = {&m0, &m1, &m2, &m3, &out_map, &m5, &m6, &pp};
    if (CG == 1) {
      PKB_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(kern), dim3(grid),
                                           dim3(num_threads(FINAL, PLANES)), args, L.total, c->stream));
    } else {
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3(grid);
      cfg.blockDim = dim3(num_threads(FINAL, PLANES));
      cfg.dynamicSmemBytes = L.total;
      cfg.stream = c->stream;
      cudaLaunchAttribute attr[2];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      attr[1].id = cudaLaunchAttributeCooperative;
      attr[1].val.cooperative = 1;
      cfg.attrs = attr;
      // Nsight Compute rejects a cooperative launch of a cluster kernel (LaunchFailed, grid shown
      // as 0). Under an injected tool kernels are serialised anyway, so co-residency of the
      // grid (<= one CTA per SM) holds without the attribute.
      static const bool tool_attached = getenv("CUDA_INJECTION64_PATH") != nullptr ||
                                        getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR") != nullptr ||
                                        getenv("NV_NSIGHT_INJECTION_PORT_BASE") != nullptr;
      cfg.numAttrs = tool_attached ? 1 : 2;
      PKB_CUDA(cudaLaunchKernelEx(&cfg, kern, m0, m1, m2, m3, out_map, m5, m6, pp));
    }
  } else if (CG == 2) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(num_threads(FINAL, PLANES));
    cfg.dynamicSmemBytes = L.total;
    cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    PKB_CUDA(cudaLaunchKernelEx(&cfg, kern, *a_hi, *a_lo, *w_hi, *w_lo, out_map, *a_x, *w_x, pp));
  } else {
    kern<<<grid, num_threads(FINAL, PLANES), L.total, c->stream>>>(*a_hi, *a_lo, *w_hi, *w_lo, out_map, *a_x,
                                                               *w_x, pp);
  }
  PKB_CUDA(cudaGetLastError());
  }
  if (dbg) {
    std::vector<long long> h(16 * grid);
    cudaStreamSynchronize(c->stream);
    cudaMemcpy(h.data(), dbg, sizeof(long long) * 16 * grid, cudaMemcpyDeviceToHost);
    cudaFree(dbg);
    double s[16] = {0};
    for (int b = 0; b < grid; ++b)
      for (int k = 0; k < 16; ++k) s[k] += h[16 * b + k];
    const double n = s[5] > 0 ? s[5] : 1;
    if (FINAL)
      fprintf(stderr, "[pkb gemm final] tiles/cta=%.0f cycles/tile: wait_acc=%.0f pass1=%.0f sync=%.0f combine=%.0f pass2=%.0f (tmem_ld=%.0f math=%.0f stage_wait=%.0f stage_write=%.0f) | mma: wait_tmem=%.0f wait_smem=%.0f\n",
              n / grid, s[0] / n, s[1] / n, s[2] / n, s[3] / n, s[4] / n, s[8] / n, s[9] / n, s[10] / n, s[11] / n, s[6] / n, s[7] / n);
    else
      fprintf(stderr, "[pkb gemm kb=%d] tiles/cta=%.0f cycles/tile: wait_acc=%.0f tmem_ld=%.0f math=%.0f stores=%.0f epilogue=%.0f | mma: wait_tmem=%.0f wait_smem=%.0f\n",
              p.num_kb, n / grid, s[0] / n, s[1] / n, s[4] / n, s[2] / n, s[3] / n, s[6] / n * CG, s[7] / n * CG);
  }
  return PKB_OK;
}

}  // namespace

int gemm_max_smem_bytes(int block_n, int planes) { return smem_layout(block_n, planes, true, 1, false).total; }

int encode_tensor_map(CUtensorMap *map, CUtensorMapDataType type, const void *base, uint64_t cols,
                      uint64_t rows, uint64_t pitch_bytes, uint32_t box_cols, uint32_t box_rows,
                      CUtensorMapL2promotion l2) {
  typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                    const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                    const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static const EncodeTiledFn fn = [] {
    void *sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
                    q == cudaDriverEntryPointSuccess && sym != nullptr;
    return ok ? reinterpret_cast<EncodeTiledFn>(sym) : nullptr;
  }();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return PKB_ERR_CUDA;
  }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, type, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) type=%d cols=%llu rows=%llu pitch=%llu box=%ux%u", (int)r,
              (int)type, (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)pitch_bytes,
              box_cols, box_rows);
    return PKB_ERR_CUDA;
  }
  return PKB_OK;
}

int launch_gemm(Ctx *c, int block_n, int planes, bool final, int cta_group, bool out8,
                const GemmMaps &maps, const GemmParams &p) {
  if (p.num_tiles <= 0) return PKB_OK;
  GemmMaps m = maps;
  if (planes == 1) { m.a_lo = m.a_hi; m.w_lo = m.w_hi; }
  if (out8 && (final || planes == 1)) {
    set_error("launch_gemm: the FP8 operand triple is written by hidden stages of operand mode 2 or 3");
    return PKB_ERR_INVALID;
  }
  if (cta_group == 2 && block_n != 256) {
    set_error("launch_gemm: cta_group 2 is built for block_n 256 only");
    return PKB_ERR_INVALID;
  }
#define PKB_GEMM_CASE(BN, PL, FN, CGV, O8) \
  if (block_n == BN && planes == PL && final == FN && cta_group == CGV && out8 == O8) \
    return launch_one<BN, PL, FN, CGV, O8>(c, m, p);
  // CTA pairs (the W maps must have box rows block_n / 2)
  PKB_GEMM_CASE(256, 1, false, 2, false)
  PKB_GEMM_CASE(256, 2, false, 2, false)
  PKB_GEMM_CASE(256, 2, true, 2, false)
  PKB_GEMM_CASE(256, 2, false, 2, true)
  PKB_GEMM_CASE(256, 3, false, 2, true)
  PKB_GEMM_CASE(256, 3, true, 2, false)
  // single CTAs
  PKB_GEMM_CASE(128, 1, false, 1, false)
  PKB_GEMM_CASE(128, 1, true, 1, false)
  PKB_GEMM_CASE(128, 2, false, 1, false)
  PKB_GEMM_CASE(128, 2, true, 1, false)
  PKB_GEMM_CASE(256, 1, false, 1, false)
  PKB_GEMM_CASE(256, 1, true, 1, false)
  PKB_GEMM_CASE(256, 2, false, 1, false)
  PKB_GEMM_CASE(256, 2, true, 1, false)
  PKB_GEMM_CASE(128, 2, false, 1, true)
  PKB_GEMM_CASE(256, 2, false, 1, true)
  PKB_GEMM_CASE(128, 3, false, 1, true)
  PKB_GEMM_CASE(256, 3, false, 1, true)
  PKB_GEMM_CASE(128, 3, true, 1, false)
  PKB_GEMM_CASE(256, 3, true, 1, false)
#undef PKB_GEMM_CASE
  set_error("launch_gemm: unsupported configuration block_n=%d planes=%d final=%d cta_group=%d out8=%d",
            block_n, planes, final ? 1 : 0, cta_group, out8 ? 1 : 0);
  return PKB_ERR_INVALID;
}

}  // namespace pkb
