// Interface of the sm_100a tcgen05 GEMM that replaces pocketkaldi's packed SGEMM
// (src/gemm.cc:69-304 driver + src/gemm_haswell.cc:72-632 AVX2 6x16 micro-kernel)
// together with the element-wise layers that follow a LinearLayer
// (src/nnet.cc:22-75) and the first half of the softmax / AM epilogue
// (src/vector.cc:264-277, src/am.cc:106-112).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "common.cuh"

namespace pkb {

constexpr int kBlockM = 128;   // rows (frames) per CTA tile = TMEM lanes
constexpr int kBlockK = 64;    // one 128-byte swizzle row of BF16
constexpr int kUmmaK = 16;     // K of one tcgen05.mma kind::f16

// Epilogue description of one fused GEMM stage:
//   acc      = A[M x K] * W[N x K]^T                       (FP32 in TMEM)
//   z        = acc * rowscale(row) + bias[col]             rowscale = sqrt(D / sum_sq(row)) of the
//                                                          preceding NormalizeLayer, else 1
//   hidden   : y = relu ? max(z, 0) : z ; optional per-row sum of y^2 (for a following
//              NormalizeLayer); stored as BF16 hi (+ lo = bf16(y - hi) in BF16X3)
//   final    : FP32 output, row m of the GEMM -> row m of the output (the caller keeps the
//              padded-row layout and compacts per utterance when copying out). Tiles leave the
//              SM through shared memory and TMA bulk tensor stores. With a SoftmaxLayer the CTAs that
//              own the column tiles of one row block exchange per-row (max, sum exp) partials
//              through global memory while the accumulators stay in TMEM, then write
//              softmax(z) or prob_scale * (max(log softmax(z), log 1e-20) - log_prior) once --
//              no second pass over the [frames x pdfs] matrix.
struct GemmParams {
  int M;               // rows of A / D
  int n_tiles_n;       // N_pad / block_n
  int num_tiles;       // m_tiles * n_tiles_n
  int m_tiles;         // set by the launcher
  int group_sched;     // set by the launcher: grouped schedule of the final softmax stage
  int num_kb;          // K_pad / kBlockK
  int num_kb8;         // operand mode 3: 128-wide FP8 k-blocks per correction phase (ceil(K_pad / 128))
  float acc_scale;     // operand mode 3: 2^-g, undoes the power-of-two scaling of the stored weights
  uint8_t *out8_lo, *out8_hi;  // OUT8: [M][ld_out] E4M3 planes of the next stage's correction operands
  int N_valid;         // logical N (columns >= N_valid are padding)
  const float *bias;   // [N_pad], zero in the padding
  const float *in_sumsq;  // [M][in_sumsq_tiles] partial sums of squares, or nullptr
  int in_sumsq_tiles;
  float in_dim;        // D of the NormalizeLayer feeding this stage
  float *out_sumsq;    // [M][n_tiles_n * sumsq_parts(planes)] or nullptr
  int relu;            // activation behind the linear layer: 0 none, 1 ReLU, 2 sigmoid
  int fp16;            // operands (and hidden outputs) are FP16 instead of BF16
  __nv_bfloat16 *out_hi, *out_lo;  // [M][ld_out]
  int ld_out;
  float *out_f32;      // final: [M][ld_f32], GEMM row m -> output row m (padded-row layout)
  int ld_f32;
  // final_mode: 0 raw logits, 1 softmax probabilities, 2 scale*(max(log softmax, log_floor) - log_prior),
  // 3 compact log-likelihoods: t = max(log softmax, log_floor) - log_prior is written as
  //   out_h16[row][col] = fp16(t - off[row]),  out_off[row] = max_col(z - log_prior) - lse
  // i.e. half the bytes, exact at the top of every frame (the values a decoder compares), the
  // consumer finishes prob_scale * (float(h) + off) (pk_decodable_loglikelihood, src/decodable.cc:24-31)
  int final_mode;
  uint16_t *out_h16;   // compact: [M][ld_f32] IEEE half bits (padded-row layout like out_f32)
  float *out_off;      // compact: [M]
  float *mzl_part;     // compact / near_cnt: [M][n_tiles_n] per-tile max(z - log_prior), exchanged like lse_part
  // refinement (final_mode 2 and 3): near_cnt[row] += number of columns whose log-likelihood lies
  // within near_margin of the row's best one (the best column counts itself: >= 2 means a near-tie).
  // Zeroed by the caller; nullptr switches the count off.
  int *near_cnt;
  float near_margin;
  float2 *lse_part;    // final softmax: [m_tiles + 1][n_tiles_n][128] (max, sum exp) exchanged between the
                       // column tiles; filled with 0xFF bytes (= not written yet) by the launcher
  const float *log_prior;  // [N_pad]
  float scale, log_floor;
  int *err_flag;       // set by the launcher: mapped host word for "gave up waiting" reports
  long long *dbg;      // optional phase-cycle counters [grid][8] (PKB_GEMM_DEBUG=1), else nullptr
};

// Encodes a 2-D tensor map with 128-byte swizzle: inner dim `cols` elements, outer dim `rows`, row
// pitch `pitch_bytes`, box {box_cols, box_rows}. The only caller of cuTensorMapEncodeTiled.
int encode_tensor_map(CUtensorMap *map, CUtensorMapDataType type, const void *base, uint64_t cols,
                      uint64_t rows, uint64_t pitch_bytes, uint32_t box_cols, uint32_t box_rows,
                      CUtensorMapL2promotion l2);

// K-major GEMM operand map: 16-bit elements (box {64, box_rows}) or, with fp8, E4M3 bytes (box
// {128, box_rows}); either way one 128-byte swizzle row per box row. pitch_bytes may be smaller
// than the row: overlapping rows implement the splice of AcousticModel::SpliceFeats
// (src/am.cc:65-88).
inline int make_operand_map(CUtensorMap *map, const void *base, bool fp8, uint64_t cols, uint64_t rows,
                            uint64_t pitch_bytes, uint32_t box_rows) {
  return encode_tensor_map(map, fp8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base,
                           cols, rows, pitch_bytes, fp8 ? 128 : kBlockK, box_rows,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

// Operand maps of one launch (see gemm_kernel): a_x / w_x are only read in operand mode 3.
struct GemmMaps {
  const CUtensorMap *a_hi, *a_lo, *a_x, *w_hi, *w_lo, *w_x;
};

// block_n in {128, 256}; planes (operand mode) in {1 one 16-bit plane, 2 hi + lo planes, 3 FP16 +
// FP8 corrections}; final: FP32 / compact output mode; out8: a hidden stage that writes the
// operand triple of a mode-3 successor.
// cta_group 2 (block_n 256): clusters of two CTAs share one 256-row tcgen05 tile,
// each loading half of the W tile (w maps with box rows block_n / 2).
int launch_gemm(Ctx *c, int block_n, int planes, bool final, int cta_group, bool out8,
                const GemmMaps &maps, const GemmParams &p);

int gemm_max_smem_bytes(int block_n, int planes);

// Epilogue warps of a single-plane hidden stage: two per TMEM lane quadrant.
constexpr int kHidWarps = 8;
// Sum-of-squares partials one hidden tile writes per row (= epilogue warps per lane quadrant)
// for operand mode `planes`.
inline int sumsq_parts(int planes) { return planes == 2 ? 1 : kHidWarps / 4; }

}  // namespace pkb
