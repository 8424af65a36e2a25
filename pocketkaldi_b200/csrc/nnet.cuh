// Device-resident acoustic model and the fused forward pass.
#pragma once

#include <string>
#include <vector>

#include "common.cuh"
#include "gemm_sm100.cuh"

namespace pkb {

// One LinearLayer with the element-wise layers fused behind it.
struct Stage {
  int in_dim = 0, out_dim = 0;  // logical K, N
  int k_pad = 0, n_pad = 0;     // K padded to 64, N padded to block_n
  int block_n = 128;
  bool relu = false;            // ReLULayer follows       (src/nnet.cc:49-60)
  bool sigmoid = false;         // sigmoid follows (PKB_LAYER_SIGMOID; not a reference layer type)
  bool normalize = false;       // NormalizeLayer follows  (src/nnet.cc:62-75)
  DevBuf w_hi, w_lo, bias;      // [n_pad][k_pad] BF16 planes, [n_pad] FP32
  // operand mode 3 (FP16C8): w_hi holds fp16(W * 2^w_exp); E4M3 planes [n_pad][k_pad8]
  bool c8 = false;
  int w_exp = 0;                // g: stored weights are W * 2^g with max |W * 2^g| in [1, 2)
  int k_pad8 = 0;               // K padded to 128
  DevBuf w8_hi, w8_lo;          // e4m3(W16 * 2^4), e4m3((W * 2^g - W16) * 2^13)
  // weight maps [tile][operand]: tile 0 has box rows block_n, tile 1 block_n / 2 (the W half of a
  // CTA pair); operands 0, 1, 2 are GemmMaps::w_hi, w_lo, w_x and map w_hi; w_lo (FP16C8: w8_lo,
  // one plane: w_hi); w8_hi (FP16C8) or w_hi
  CUtensorMap w_map[2][3];
};

// How the final stage's logits are turned into the caller's output.
enum FinalMode {
  kFinalRaw = 0,     // z                                   (stack without SoftmaxLayer)
  kFinalProb = 1,    // softmax(z)                          (Nnet::Propagate, src/nnet.cc:149-163)
  kFinalLoglik = 2,  // s*(log(max(softmax(z),1e-20))-lp)   (AcousticModel::Compute + decodable scale)
  kFinalCompact = 3, // fp16(log(max(softmax(z),1e-20)) - lp - off[row]) + off[row]: half the bytes
};

// A [rows][cols] BF16 matrix (one or two planes) as the first GEMM's A operand.
// pitch_elems < cols describes overlapping rows (the splice view).
struct InputView {
  const __nv_bfloat16 *hi = nullptr, *lo = nullptr;
  int64_t rows = 0;
  int cols = 0;
  int pitch_elems = 0;
};

// Per-batch scratch of the forward pass.
struct Workspace {
  int64_t rows = 0;  // M of every GEMM
  DevBuf act_hi[2], act_lo[2], sumsq[2], lse_part, mzl_part, row_map;
  DevBuf act8_lo[2], act8_hi[2];  // FP16C8: E4M3 correction operands of the hidden activations
  bool fast_only = false;         // only single-plane passes run on this workspace (FP16R first pass)
  // padded feature planes of the batch pipeline
  DevBuf feat_hi, feat_lo, pad_off;
};

// Scratch of the selective second pass of PKB_PREC_FP16R (nnet_forward_refined).
struct Refine {
  DevBuf near_cnt, list, n_sel;   // [rows] near-tie counts, selected rows, their number
  DevBuf in_hi, in_lo;            // gathered (spliced) input rows of the selected frames
  DevBuf out_f32, out_h16, out_off;
  Workspace ws;
  int32_t *h_n_sel = nullptr;     // pinned host copy of n_sel
  int64_t last_rows = 0, last_selected = 0;  // of the latest forward pass (pkb_batch_refine_stats)
  ~Refine() {
    if (h_n_sel) cudaFreeHost(h_n_sel);
  }
};

}  // namespace pkb

struct pkb_am {
  pkb::Ctx *c = nullptr;
  int precision = PKB_PREC_BF16;
  int planes = 1;  // 16-bit planes of the input features and of stage 0
  int fp16 = 0;    // operands are FP16 instead of BF16 (PKB_PREC_FP16, _FP16X3, _FP16C8)
  int c8 = 0;      // PKB_PREC_FP16C8 / _FP16R: stages after the first run in operand mode 3
  // PKB_PREC_FP16R: one FP16 MMA per product for every frame, then the frames whose two best
  // pdfs lie within refine_margin of each other are recomputed with the FP16C8 operands
  int refine = 0;
  float refine_margin = 0.02f;  // tools/refine_margin_stats.py: 3x the largest error spread seen
  int left = 0, right = 0, num_pdfs = 0;
  int input_dim = 0;   // nnet input dim
  int feat_dim = 0;    // input_dim / (left + right + 1) when divisible, else 0
  int feat_dim_pad = 0;
  bool softmax_last = false;
  // stages[0] reads feat_dim_pad columns per context frame (the padded splice view) when
  // feat_dim > 0, the input_dim columns of a row otherwise
  std::vector<pkb::Stage> stages;
  pkb::DevBuf log_prior;  // [num_pdfs], log taken at load (src/am.cc:42-43)
  std::vector<int32_t> tid2pdf;
  // scratch of the synchronous host-buffer entry points (pkb_am_compute, pkb_nnet_propagate)
  pkb::Workspace ws;
  pkb::Refine rf;
  pkb::BatchMeta meta;
  pkb::DevBuf in_f32, out_f32;
};

namespace pkb {

int am_build(Ctx *c, int n_layers, const int32_t *types, const float *const *weights,
             const float *const *biases, const int32_t *out_dims, const int32_t *in_dims,
             const float *prior, int num_pdfs, int left, int right, const int32_t *tid2pdf,
             int n_tid2pdf, int precision, pkb_am **out);

// Sizes `ws` for `rows` GEMM rows of model `am`.
int workspace_ensure(pkb_am *am, Workspace *ws, int64_t rows);

// Runs every stage. d_out is [ws->rows][out_dim]: GEMM row m -> output row m. For a padded
// batch the rows of utterance u start at pad_off[u] and the (left+right) rows between two
// utterances hold garbage; copy_rows_compact() removes them on the way out.
// kFinalCompact writes d_h16 [ws->rows][out_dim] (IEEE half bits) and d_off [ws->rows] instead of
// d_out; prob_scale is then left to the consumer.
// fast: every stage as one 16-bit plane (the hi planes of whatever the model holds).
// near_cnt (kFinalLoglik / kFinalCompact): see GemmParams::near_cnt.
int nnet_forward(pkb_am *am, Workspace *ws, const InputView &in, FinalMode mode, float prob_scale,
                 float *d_out, uint16_t *d_h16 = nullptr, float *d_off = nullptr, bool fast = false,
                 int *near_cnt = nullptr, float near_margin = 0.0f);

// nnet_forward for every precision; PKB_PREC_FP16R log-likelihoods take two passes:
//   1. nnet_forward(fast) over all rows, counting per row the pdfs within am->refine_margin of
//      the best one;
//   2. the rows with a near-tie (count >= 2; row_map[row] >= 0 when a row map is given) are
//      gathered, run through the FP16C8 stages and scattered over the first pass's output.
// One host synchronisation in between (the number of selected rows sizes the second pass).
int nnet_forward_refined(pkb_am *am, Workspace *ws, Refine *rf, const InputView &in,
                         const int32_t *row_map, FinalMode mode, float prob_scale, float *d_out,
                         uint16_t *d_h16 = nullptr, float *d_off = nullptr);

// Device (padded rows) -> host (compact frames) copy of frames [frame0, frame0 + n): one
// cudaMemcpyAsync per utterance touched.
int copy_rows_compact(Ctx *c, void *host_dst, const void *d_padded, const BatchMeta &m,
                      const std::vector<int64_t> &pad_off, int cols, int64_t frame0, int64_t n,
                      size_t elem_bytes = sizeof(float));

// Sum over the valid rows (row_map[m] >= 0) of a padded [rows][cols] matrix, in double.
int launch_checksum_rows(Ctx *c, const float *d, int cols, int64_t rows, const int32_t *row_map,
                         double *d_sum);

// float [F][dim] -> padded BF16 planes with replicated edge frames + row map.
int launch_pack_padded(Ctx *c, const float *d_feats, const BatchMeta &m, int dim, int dim_pad,
                       int left, int right, const int64_t *d_pad_off, __nv_bfloat16 *hi,
                       __nv_bfloat16 *lo, int32_t *row_map, int fp16);
// float [rows][groups * group] -> BF16 planes [rows][groups * group_pad]: column k goes to
// (k / group) * group_pad + k % group, the padding columns are zero.
int launch_pack_plain(Ctx *c, const float *d_in, int64_t rows, int groups, int group, int group_pad,
                      __nv_bfloat16 *hi, __nv_bfloat16 *lo, int fp16);
// row_map for a padded batch without packing (the CMVN kernel wrote the planes).
int launch_row_map(Ctx *c, const BatchMeta &m, int left, int right, const int64_t *d_pad_off,
                   int32_t *row_map, int64_t rows);

// Padded-row bookkeeping: pad_off[u] = frame_off[u] + u*(left+right); returns total padded
// rows and the GEMM row count (padded rows - (left+right), 0 for an empty batch).
void padded_rows(const BatchMeta &m, int left, int right, std::vector<int64_t> *pad_off,
                 int64_t *padded, int64_t *gemm_rows);

}  // namespace pkb
