// Acoustic model on the device: weight packing, the fused layer plan, the forward
// pass and the small kernels around the GEMMs (pack / row map / finalize).
//
// Reference path: AcousticModel::Compute (src/am.cc:90-115) = SpliceFeats (:65-88)
// -> Nnet::Propagate (src/nnet.cc:149-163: Linear / ReLU / Normalize / Softmax layers,
// :22-75) -> floor 1e-20, log, minus log-prior (src/am.cc:106-112), then the
// decodable's prob_scale (src/decodable.cc:15).

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_fp8.h>

#include <algorithm>
#include <memory>

#include "nnet.cuh"

namespace pkb {

namespace {

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// ---------------------------------------------------------------- kernels
__global__ void pack_padded_kernel(const float *__restrict__ feats,
                                   const int64_t *__restrict__ frame_off,
                                   const int32_t *__restrict__ num_frames,
                                   const int64_t *__restrict__ pad_off, int n_utts, int dim,
                                   int dim_pad, int left, int right, int64_t total_frames,
                                   __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo,
                                   int32_t *__restrict__ row_map, int fp16) {
  // one thread per (frame, padded column)
  const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t f = g / dim_pad;
  const int d = static_cast<int>(g % dim_pad);
  if (f >= total_frames) return;
  int a = 0, b = n_utts - 1;
  while (a < b) {  // largest u with frame_off[u] <= f (utterances with 0 frames are skipped)
    int mid = (a + b + 1) >> 1;
    if (frame_off[mid] <= f) a = mid; else b = mid - 1;
  }
  const int u = a;
  const int t = static_cast<int>(f - frame_off[u]);
  const int T = num_frames[u];
  const float v = d < dim ? feats[f * dim + d] : 0.0f;
  const __nv_bfloat16 h = operand_bits(v, fp16);
  const __nv_bfloat16 l = operand_bits(v - operand_value(h, fp16), fp16);
  const int64_t base = pad_off[u];
  const int64_t row = base + left + t;
  hi[row * dim_pad + d] = h;
  if (lo) lo[row * dim_pad + d] = l;
  if (t == 0)
    for (int r = 0; r < left; ++r) {
      hi[(base + r) * dim_pad + d] = h;
      if (lo) lo[(base + r) * dim_pad + d] = l;
    }
  if (t == T - 1)
    for (int r = 0; r < right; ++r) {
      hi[(row + 1 + r) * dim_pad + d] = h;
      if (lo) lo[(row + 1 + r) * dim_pad + d] = l;
    }
  if (d == 0 && row_map) row_map[base + t] = static_cast<int32_t>(f);
}

__global__ void row_map_kernel(const int64_t *__restrict__ frame_off,
                               const int32_t *__restrict__ num_frames,
                               const int64_t *__restrict__ pad_off, int n_utts,
                               int32_t *__restrict__ row_map) {
  const int u = blockIdx.y;
  if (u >= n_utts) return;
  const int T = num_frames[u];
  const int64_t base = pad_off[u], f0 = frame_off[u];
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x)
    row_map[base + t] = static_cast<int32_t>(f0 + t);
}

// one thread per (row, padded column); input column k goes to (k / group) * group_pad + k % group
__global__ void pack_plain_kernel(const float *__restrict__ in, int64_t rows, int dim, int dim_pad,
                                  int group, int group_pad, __nv_bfloat16 *__restrict__ hi,
                                  __nv_bfloat16 *__restrict__ lo, int fp16) {
  const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t r = g / dim_pad;
  const int d = static_cast<int>(g % dim_pad);
  if (r >= rows) return;
  const int j = d % group_pad;
  const float v = j < group ? in[r * dim + d / group_pad * group + j] : 0.0f;
  const __nv_bfloat16 h = operand_bits(v, fp16);
  hi[g] = h;
  if (lo) lo[g] = operand_bits(v - operand_value(h, fp16), fp16);
}

// FP16C8 weight planes from the FP32 matrix (one thread per element of the padded planes).
__global__ void pack_c8_kernel(const float *__restrict__ W, int out_dim, int in_dim, int n_pad, int k_pad,
                               int k_pad8, float sg, __nv_bfloat16 *__restrict__ w16, uint8_t *__restrict__ h8,
                               uint8_t *__restrict__ l8) {
  const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int o = static_cast<int>(g / k_pad8), k = static_cast<int>(g % k_pad8);
  if (o >= n_pad) return;
  float w = 0.0f;
  if (o < out_dim && k < in_dim) w = W[static_cast<int64_t>(o) * in_dim + k] * sg;
  const __half h = __float2half_rn(w);
  const float wf = __half2float(h);
  if (k < k_pad) {
    const __half_raw hr = static_cast<__half_raw>(h);
    __nv_bfloat16_raw br;
    br.x = hr.x;
    w16[static_cast<int64_t>(o) * k_pad + k] = __nv_bfloat16(br);
  }
  h8[g] = static_cast<uint8_t>(__nv_cvt_float_to_fp8(wf * 16.0f, __NV_SATFINITE, __NV_E4M3));
  l8[g] = static_cast<uint8_t>(__nv_cvt_float_to_fp8((w - wf) * 8192.0f, __NV_SATFINITE, __NV_E4M3));
}

// ---------------------------------------------------------------- weight packing
// What both packings share: the N tiling, the zero-padded bias, the device planes (`planes` 16-bit
// ones, and the two E4M3 ones of FP16C8) and the weight maps. The caller sets the K layout first
// (k_pad; c8 and k_pad8 for FP16C8) and fills the planes.
int alloc_stage(Ctx *c, Stage *st, const float *b, int out_dim, int in_dim, int planes) {
  st->in_dim = in_dim;
  st->out_dim = out_dim;
  const int n128 = round_up(out_dim, 128), n256 = round_up(out_dim, 256);
  // wide tiles unless they cost more than 6% extra padding
  st->block_n = (n256 * 100 <= n128 * 106) ? 256 : 128;
  st->n_pad = st->block_n == 256 ? n256 : n128;
  std::vector<float> bias(st->n_pad, 0.0f);
  memcpy(bias.data(), b, sizeof(float) * out_dim);
  PKB_TRY(st->bias.ensure(sizeof(float) * st->n_pad));
  PKB_TRY(upload(c, st->bias.p, bias.data(), sizeof(float) * st->n_pad));
  const size_t e16 = static_cast<size_t>(st->n_pad) * st->k_pad, e8 = static_cast<size_t>(st->n_pad) * st->k_pad8;
  PKB_TRY(st->w_hi.ensure(e16 * 2));
  if (planes == 2) PKB_TRY(st->w_lo.ensure(e16 * 2));
  if (st->c8) {
    PKB_TRY(st->w8_hi.ensure(e8));
    PKB_TRY(st->w8_lo.ensure(e8));
  }
  const uint64_t p16 = static_cast<uint64_t>(st->k_pad) * 2, p8 = static_cast<uint64_t>(st->k_pad8);
  for (int t = 0; t < 2; ++t) {
    CUtensorMap *m = st->w_map[t];
    const uint32_t box_rows = st->block_n >> t;
    PKB_TRY(make_operand_map(&m[0], st->w_hi.p, false, st->k_pad, st->n_pad, p16, box_rows));
    m[1] = m[2] = m[0];
    if (planes == 2) PKB_TRY(make_operand_map(&m[1], st->w_lo.p, false, st->k_pad, st->n_pad, p16, box_rows));
    if (st->c8) {
      PKB_TRY(make_operand_map(&m[1], st->w8_lo.p, true, st->k_pad8, st->n_pad, p8, box_rows));
      PKB_TRY(make_operand_map(&m[2], st->w8_hi.p, true, st->k_pad8, st->n_pad, p8, box_rows));
    }
  }
  return PKB_OK;
}

// W[out][in] float -> BF16 planes [n_pad][k_pad]; column k of the source goes to column
// (k / group) * group_pad + k % group (group = group_pad = in_dim: the identity).
int pack_stage(Ctx *c, Stage *st, const float *W, const float *b, int out_dim, int in_dim,
               int group, int group_pad, int planes, int fp16) {
  st->k_pad = round_up(in_dim / group * group_pad, kBlockK);
  PKB_TRY(alloc_stage(c, st, b, out_dim, in_dim, planes));
  const size_t elems = static_cast<size_t>(st->n_pad) * st->k_pad;
  std::vector<__nv_bfloat16> hi(elems, operand_bits(0.0f, fp16)), lo;
  if (planes == 2) lo.assign(elems, operand_bits(0.0f, fp16));
  for (int o = 0; o < out_dim; ++o) {
    const float *src = W + static_cast<size_t>(o) * in_dim;
    __nv_bfloat16 *dh = hi.data() + static_cast<size_t>(o) * st->k_pad;
    __nv_bfloat16 *dl = planes == 2 ? lo.data() + static_cast<size_t>(o) * st->k_pad : nullptr;
    for (int k = 0; k < in_dim; ++k) {
      const int kk = (k / group) * group_pad + (k % group);
      const __nv_bfloat16 h = operand_bits(src[k], fp16);
      dh[kk] = h;
      if (dl) dl[kk] = operand_bits(src[k] - operand_value(h, fp16), fp16);
    }
  }
  PKB_TRY(upload(c, st->w_hi.p, hi.data(), elems * 2));
  if (planes == 2) PKB_TRY(upload(c, st->w_lo.p, lo.data(), elems * 2));
  return PKB_OK;
}

// Operand mode 3 (FP16C8) planes of W[out][in]: W16 = fp16(W * 2^g) with max |W * 2^g| in [1, 2),
// W_hi8 = e4m3(W16 * 2^4), W_lo8 = e4m3((W * 2^g - W16) * 2^13); see gemm_sm100.cu.
int pack_stage_c8(Ctx *c, Stage *st, const float *W, const float *b, int out_dim, int in_dim) {
  st->c8 = true;
  st->k_pad = round_up(in_dim, kBlockK);
  st->k_pad8 = round_up(in_dim, 128);
  float wmax = 0.0f;
  for (size_t i = 0; i < static_cast<size_t>(out_dim) * in_dim; ++i) wmax = std::max(wmax, fabsf(W[i]));
  PKB_REQUIRE(std::isfinite(wmax), "linear layer: non-finite weight");
  int e = 0;
  if (wmax > 0.0f) frexpf(wmax, &e);  // wmax = m * 2^e, m in [0.5, 1)
  st->w_exp = wmax > 0.0f ? 1 - e : 0; // W * 2^g has its maximum in [1, 2)
  const float sg = ldexpf(1.0f, st->w_exp);
  PKB_TRY(alloc_stage(c, st, b, out_dim, in_dim, 1));
  // the planes are rounded on the device: 2 x 8.8 M scalar FP8 conversions on the host would
  // dominate the model load of the config-3 net
  DevBuf tmp;
  const size_t wbytes = static_cast<size_t>(out_dim) * in_dim * sizeof(float);
  PKB_TRY(tmp.ensure(wbytes));
  PKB_TRY(upload(c, tmp.p, W, wbytes));
  const int64_t threads = static_cast<int64_t>(st->n_pad) * st->k_pad8;
  pack_c8_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, c->stream>>>(
      tmp.as<float>(), out_dim, in_dim, st->n_pad, st->k_pad, st->k_pad8, sg, st->w_hi.as<__nv_bfloat16>(),
      st->w8_hi.as<uint8_t>(), st->w8_lo.as<uint8_t>());
  PKB_CUDA(cudaGetLastError());
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return PKB_OK;
}

}  // namespace

void padded_rows(const BatchMeta &m, int left, int right, std::vector<int64_t> *pad_off,
                 int64_t *padded, int64_t *gemm_rows) {
  pad_off->resize(m.n_utts);
  const int64_t ctx = left + right;
  for (int u = 0; u < m.n_utts; ++u) (*pad_off)[u] = m.frame_off[u] + u * ctx;
  *padded = m.total_frames + static_cast<int64_t>(m.n_utts) * ctx;
  *gemm_rows = m.total_frames > 0 ? *padded - ctx : 0;
}

int am_build(Ctx *c, int n_layers, const int32_t *types, const float *const *weights,
             const float *const *biases, const int32_t *out_dims, const int32_t *in_dims,
             const float *prior, int num_pdfs, int left, int right, const int32_t *tid2pdf,
             int n_tid2pdf, int precision, pkb_am **out) {
  PKB_REQUIRE(c && out, "pkb_am_create: NULL argument");
  PKB_REQUIRE(precision >= PKB_PREC_BF16 && precision <= PKB_PREC_FP16R,
              "pkb_am_create: unknown precision %d", precision);
  PKB_REQUIRE(left >= 0 && right >= 0, "pkb_am_create: negative context");
  PKB_REQUIRE(n_layers > 0 && types, "pkb_am_create: empty layer list");
  PKB_CUDA(cudaSetDevice(c->device));
  std::unique_ptr<pkb_am, decltype(&pkb_am_destroy)> am(new pkb_am(), pkb_am_destroy);
  am->c = c;
  am->precision = precision;
  am->refine = precision == PKB_PREC_FP16R ? 1 : 0;
  am->c8 = (precision == PKB_PREC_FP16C8 || am->refine) ? 1 : 0;
  if (am->refine) {
    if (const char *e = getenv("PKB_REFINE_MARGIN")) am->refine_margin = static_cast<float>(atof(e));
  }
  am->planes = (precision == PKB_PREC_BF16X3 || precision == PKB_PREC_FP16X3 || am->c8) ? 2 : 1;
  am->fp16 = (precision == PKB_PREC_FP16 || precision == PKB_PREC_FP16X3 || am->c8) ? 1 : 0;
  am->left = left;
  am->right = right;
  int lin = 0;
  int i = 0;
  int prev_out = -1;
  while (i < n_layers) {
    if (types[i] != 0) {
      set_error("layer %d: type %d without a preceding linear layer is not supported", i, types[i]);
      return PKB_ERR_UNSUPPORTED;
    }
    if (am->softmax_last) {
      set_error("layer %d: layers after softmax are not supported", i);
      return PKB_ERR_UNSUPPORTED;
    }
    const int od = out_dims[lin], id = in_dims[lin];
    PKB_REQUIRE(od > 0 && id > 0 && (prev_out < 0 || id == prev_out),
                "linear layer %d: shape [%d x %d] does not follow output dim %d", lin, od, id, prev_out);
    int group = id, group_pad = id;
    if (lin == 0) {
      am->input_dim = id;
      const int w = left + right + 1;
      if (id % w == 0) {  // stage 0 reads the padded splice view: feat_dim_pad columns per frame
        am->feat_dim = group = id / w;
        am->feat_dim_pad = group_pad = round_up(am->feat_dim, 8);  // 16-byte row pitch for the TMA view
      }
    }
    am->stages.emplace_back();
    Stage &st = am->stages.back();
    // FP16C8: stage 0 reads the 16-bit feature planes (three MMAs), later stages the FP8 triple
    PKB_TRY((am->c8 && lin > 0) ? pack_stage_c8(c, &st, weights[lin], biases[lin], od, id)
                                : pack_stage(c, &st, weights[lin], biases[lin], od, id, group, group_pad,
                                             am->planes, am->fp16));
    prev_out = od;
    ++lin;
    ++i;
    if (i < n_layers && types[i] == 1) { st.relu = true; ++i; }
    else if (i < n_layers && types[i] == PKB_LAYER_SIGMOID) { st.sigmoid = true; ++i; }
    if (i < n_layers && types[i] == 2) { st.normalize = true; ++i; }
    if (i < n_layers && types[i] == 3) { am->softmax_last = true; ++i; }
    if (i < n_layers && types[i] != 0) {
      set_error("layer %d: type %d in an unsupported position (supported: linear [relu | sigmoid] "
                "[normalize] ... linear [softmax])", i, types[i]);
      return PKB_ERR_UNSUPPORTED;
    }
  }
  const Stage &last = am->stages.back();
  if (last.relu || last.sigmoid || last.normalize) {
    set_error("relu / sigmoid / normalize after the last linear layer is not supported");
    return PKB_ERR_UNSUPPORTED;
  }
  am->num_pdfs = num_pdfs > 0 ? num_pdfs : last.out_dim;
  PKB_REQUIRE(prior == nullptr || am->num_pdfs == last.out_dim, "num_pdfs %d != nnet output dim %d",
              am->num_pdfs, last.out_dim);
  // log prior: log in double, stored float (src/am.cc:42-43, src/vector.cc:333-339)
  // padded to the last stage's n_pad so that the epilogue can use vector loads
  const int lp_len = std::max(am->num_pdfs, last.n_pad);
  std::vector<float> lp(lp_len, 0.0f);
  if (prior)
    for (int j = 0; j < am->num_pdfs; ++j) lp[j] = static_cast<float>(log(static_cast<double>(prior[j])));
  PKB_TRY(am->log_prior.ensure(sizeof(float) * lp_len));
  PKB_TRY(upload(c, am->log_prior.p, lp.data(), sizeof(float) * lp_len));
  if (tid2pdf && n_tid2pdf > 0) am->tid2pdf.assign(tid2pdf, tid2pdf + n_tid2pdf);
  *out = am.release();
  return PKB_OK;
}

int workspace_ensure(pkb_am *am, Workspace *ws, int64_t rows) {
  ws->rows = rows;
  if (rows == 0) return PKB_OK;
  size_t max_hidden = 0;
  int max_tiles = 1;
  const size_t ns = am->stages.size();
  for (size_t i = 0; i + 1 < ns; ++i) {
    max_hidden = std::max<size_t>(max_hidden, am->stages[i].n_pad);
    max_tiles = std::max(max_tiles, am->stages[i].n_pad / am->stages[i].block_n);
  }
  const int bufs = ns > 2 ? 2 : (ns > 1 ? 1 : 0);
  for (int i = 0; i < bufs; ++i) {
    PKB_TRY(ws->act_hi[i].ensure(static_cast<size_t>(rows) * max_hidden * 2));
    if (am->c8 && !ws->fast_only) {
      PKB_TRY(ws->act8_lo[i].ensure(static_cast<size_t>(rows) * max_hidden));
      PKB_TRY(ws->act8_hi[i].ensure(static_cast<size_t>(rows) * max_hidden));
    } else if (am->planes == 2 && !am->c8) {
      PKB_TRY(ws->act_lo[i].ensure(static_cast<size_t>(rows) * max_hidden * 2));
    }
    PKB_TRY(ws->sumsq[i].ensure(static_cast<size_t>(rows) * max_tiles * 2 * sizeof(float)));
  }
  const Stage &last = am->stages.back();
  // softmax exchange: one word per row and column tile (128-column tiles at most), one row block
  // more than the matrix has (a CTA pair may work one block past the end)
  const size_t words = (static_cast<size_t>((rows + kBlockM - 1) / kBlockM) + 1) * kBlockM * (last.n_pad / 128);
  PKB_TRY(ws->lse_part.ensure(words * sizeof(float2)));
  PKB_TRY(ws->mzl_part.ensure(words * sizeof(float)));
  return PKB_OK;
}

int nnet_forward(pkb_am *am, Workspace *ws, const InputView &in, FinalMode mode_out, float prob_scale,
                 float *d_out, uint16_t *d_h16, float *d_off, bool fast, int *near_cnt, float near_margin) {
  Ctx *c = am->c;
  const int64_t rows = ws->rows;
  if (rows == 0) return PKB_OK;
  PKB_REQUIRE(rows <= INT32_MAX, "nnet_forward: %lld rows exceed the 2^31 limit of one launch",
              static_cast<long long>(rows));
  PKB_REQUIRE(in.rows == rows, "nnet_forward: input rows %lld != workspace rows %lld",
              static_cast<long long>(in.rows), static_cast<long long>(rows));
  const size_t ns = am->stages.size();
  // AcousticModel::Compute (src/am.cc:106-112) floors and takes the log of the nnet output, which
  // only means something for a SoftmaxLayer output; raw logits would silently differ from it
  if ((mode_out == kFinalLoglik || mode_out == kFinalCompact) && !am->softmax_last) {
    set_error("log-likelihoods need a model whose last layer is a softmax (AcousticModel::Compute "
              "takes log(max(p, 1e-20)) of the nnet output)");
    return PKB_ERR_UNSUPPORTED;
  }
  const __nv_bfloat16 *a_hi = in.hi, *a_lo = in.lo;
  const uint8_t *a8_lo = nullptr, *a8_hi = nullptr;  // FP16C8 operand triple of the current stage
  int a_cols = in.cols, a_pitch = in.pitch_elems;
  const float *in_sumsq = nullptr;
  int in_sumsq_tiles = 0;
  float in_dim = 0.0f;
  const int m_tiles = static_cast<int>((rows + kBlockM - 1) / kBlockM);
  for (size_t i = 0; i < ns; ++i) {
    const Stage &st = am->stages[i];
    const bool final = i + 1 == ns;
    // operand mode of this stage and the form its epilogue has to produce for the next one
    const int mode = fast ? 1 : (st.c8 ? 3 : am->planes);
    const bool out8 = !fast && !final && am->c8;
    CUtensorMap tm_a_hi, tm_a_lo, tm_a_x;
    PKB_TRY(make_operand_map(&tm_a_hi, a_hi, false, a_cols, rows, static_cast<uint64_t>(a_pitch) * 2, kBlockM));
    if (mode == 2) {
      PKB_TRY(make_operand_map(&tm_a_lo, a_lo, false, a_cols, rows, static_cast<uint64_t>(a_pitch) * 2, kBlockM));
      tm_a_x = tm_a_hi;
    } else if (mode == 3) {
      PKB_TRY(make_operand_map(&tm_a_lo, a8_lo, true, a_cols, rows, static_cast<uint64_t>(a_pitch), kBlockM));
      PKB_TRY(make_operand_map(&tm_a_x, a8_hi, true, a_cols, rows, static_cast<uint64_t>(a_pitch), kBlockM));
    } else {
      tm_a_lo = tm_a_hi;
      tm_a_x = tm_a_hi;
    }
    const int block_n = st.block_n;
    GemmParams p{};
    p.M = static_cast<int>(rows);
    p.n_tiles_n = st.n_pad / block_n;
    const int64_t tiles = static_cast<int64_t>(m_tiles) * p.n_tiles_n;
    PKB_REQUIRE(tiles <= INT32_MAX, "nnet_forward: too many tiles");
    p.num_tiles = static_cast<int>(tiles);
    p.num_kb = st.k_pad / kBlockK;
    p.num_kb8 = st.c8 ? st.k_pad8 / 128 : 0;
    p.acc_scale = st.c8 ? ldexpf(1.0f, -st.w_exp) : 1.0f;
    p.N_valid = st.out_dim;
    p.bias = st.bias.as<float>();
    p.in_sumsq = in_sumsq;
    p.in_sumsq_tiles = in_sumsq_tiles;
    p.in_dim = in_dim;
    p.relu = st.relu ? 1 : (st.sigmoid ? 2 : 0);
    p.fp16 = am->fp16;
    if (!final) {
      const int buf = static_cast<int>(i & 1);
      p.out_hi = ws->act_hi[buf].as<__nv_bfloat16>();
      p.out_lo = (!fast && am->planes == 2 && !am->c8) ? ws->act_lo[buf].as<__nv_bfloat16>() : nullptr;
      p.out8_lo = out8 ? ws->act8_lo[buf].as<uint8_t>() : nullptr;
      p.out8_hi = out8 ? ws->act8_hi[buf].as<uint8_t>() : nullptr;
      p.ld_out = st.n_pad;
      p.out_sumsq = st.normalize ? ws->sumsq[buf].as<float>() : nullptr;
    } else {
      p.out_f32 = d_out;
      p.ld_f32 = st.out_dim;
      // softmax + AM epilogue are fused into this GEMM (no second pass over the output)
      p.final_mode = am->softmax_last ? (mode_out == kFinalCompact ? 3 : (mode_out == kFinalLoglik ? 2 : (mode_out == kFinalProb ? 1 : 0))) : 0;
      if (p.final_mode == 3) {
        PKB_REQUIRE(d_h16 && d_off, "nnet_forward: the compact output needs its two buffers");
        p.out_h16 = d_h16;
        p.out_off = d_off;
      }
      p.mzl_part = ws->mzl_part.as<float>();
      if (near_cnt != nullptr && (p.final_mode == 2 || p.final_mode == 3)) {
        p.near_cnt = near_cnt;
        p.near_margin = near_margin;
      }
      p.lse_part = ws->lse_part.as<float2>();
      p.log_prior = am->log_prior.as<float>();
      p.scale = prob_scale;
      p.log_floor = static_cast<float>(log(static_cast<double>(static_cast<float>(1.0e-20))));
    }
    // CTA pairs (cta_group::2) whenever the tile is 256 wide and there is at least one full pair
    // of row blocks: always for hidden stages; for the output stage only in the multi-MMA modes,
    // where the halved W tile is what makes a second pipeline stage fit (its BF16/FP16 variant is
    // bound by the epilogue, not by operand traffic, and measured no gain from pairing)
    const bool want_pair = !final || mode >= 2;
    int cg = (want_pair && block_n == 256 && m_tiles >= 2) ? 2 : 1;
    // the grouped schedule of the softmax stage needs one CTA (pair) per column tile on the device
    if (final && p.final_mode != 0 && cg == 2 && (c->sm_count / 2) / p.n_tiles_n < 1) cg = 1;
    const CUtensorMap *w = st.w_map[cg == 2 ? 1 : 0];
    const GemmMaps maps{&tm_a_hi, &tm_a_lo, &tm_a_x, &w[0], &w[1], &w[2]};
    PKB_TRY(launch_gemm(c, block_n, mode, final, cg, out8, maps, p));
    if (!final) {
      a_hi = p.out_hi;
      a_lo = p.out_lo;
      a8_lo = p.out8_lo;
      a8_hi = p.out8_hi;
      a_cols = st.n_pad;
      a_pitch = st.n_pad;
      in_sumsq = p.out_sumsq;
      in_sumsq_tiles = p.n_tiles_n * sumsq_parts(mode);
      in_dim = static_cast<float>(st.out_dim);
    }
  }
  return PKB_OK;
}

namespace {
// Rows whose near-tie count reached 2, in row order inside a block of 1024 rows.
__global__ void __launch_bounds__(1024) select_rows_kernel(const int *__restrict__ near_cnt,
                                                           const int32_t *__restrict__ row_map,
                                                           int64_t rows, int32_t *__restrict__ list,
                                                           int *__restrict__ n_sel) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  const int64_t r = static_cast<int64_t>(blockIdx.x) * 1024 + threadIdx.x;
  const bool sel = r < rows && near_cnt[r] >= 2 && (row_map == nullptr || row_map[r] >= 0);
  const unsigned m = __ballot_sync(0xffffffffu, sel);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) s_warp[warp] = __popc(m);
  __syncthreads();
  if (warp == 0) {
    const int v = s_warp[lane];
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    s_warp[lane] = inc - v;
    if (lane == 31) s_base = inc > 0 ? atomicAdd(n_sel, inc) : 0;
  }
  __syncthreads();
  if (sel) list[s_base + s_warp[warp] + __popc(m & ((1u << lane) - 1u))] = static_cast<int32_t>(r);
}

// dst[i][0 .. v16) = src[list[i] * pitch16 .. + v16) in 16-byte units, for one or two planes.
__global__ void gather_rows_kernel(const uint4 *__restrict__ hi, const uint4 *__restrict__ lo,
                                   const int32_t *__restrict__ list, int n, int v16, int pitch16,
                                   uint4 *__restrict__ g_hi, uint4 *__restrict__ g_lo) {
  const int64_t total = static_cast<int64_t>(n) * v16;
  for (int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; g < total;
       g += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(g / v16), j = static_cast<int>(g % v16);
    const int64_t src = static_cast<int64_t>(list[i]) * pitch16 + j;
    g_hi[g] = hi[src];
    if (lo != nullptr) g_lo[g] = lo[src];
  }
}

// dst[list[i]][0 .. v) = src[i][0 .. v) in units of T.
template <typename T>
__global__ void scatter_rows_kernel(const T *__restrict__ src, const int32_t *__restrict__ list, int n,
                                    int v, T *__restrict__ dst) {
  const int64_t total = static_cast<int64_t>(n) * v;
  for (int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; g < total;
       g += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(g / v), j = static_cast<int>(g % v);
    dst[static_cast<int64_t>(list[i]) * v + j] = src[g];
  }
}

int launch_scatter(Ctx *c, const void *src, const int32_t *list, int n, size_t row_bytes, void *dst) {
  const int grid_cap = c->sm_count * 16;
  LaunchScope scope(c, PKB_KERNEL_MISC);
  if (row_bytes % 16 == 0) {
    const int v = static_cast<int>(row_bytes / 16);
    const int grid = static_cast<int>(std::min<int64_t>((static_cast<int64_t>(n) * v + 255) / 256, grid_cap));
    scatter_rows_kernel<uint4><<<grid, 256, 0, c->stream>>>(static_cast<const uint4 *>(src), list, n, v,
                                                            static_cast<uint4 *>(dst));
  } else if (row_bytes % 4 == 0) {
    const int v = static_cast<int>(row_bytes / 4);
    const int grid = static_cast<int>(std::min<int64_t>((static_cast<int64_t>(n) * v + 255) / 256, grid_cap));
    scatter_rows_kernel<uint32_t><<<grid, 256, 0, c->stream>>>(static_cast<const uint32_t *>(src), list, n, v,
                                                               static_cast<uint32_t *>(dst));
  } else {
    const int v = static_cast<int>(row_bytes / 2);
    const int grid = static_cast<int>(std::min<int64_t>((static_cast<int64_t>(n) * v + 255) / 256, grid_cap));
    scatter_rows_kernel<uint16_t><<<grid, 256, 0, c->stream>>>(static_cast<const uint16_t *>(src), list, n, v,
                                                               static_cast<uint16_t *>(dst));
  }
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}
}  // namespace

int nnet_forward_refined(pkb_am *am, Workspace *ws, Refine *rf, const InputView &in,
                         const int32_t *row_map, FinalMode mode, float prob_scale, float *d_out,
                         uint16_t *d_h16, float *d_off) {
  if (!am->refine || (mode != kFinalLoglik && mode != kFinalCompact))
    return nnet_forward(am, ws, in, mode, prob_scale, d_out, d_h16, d_off);
  Ctx *c = am->c;
  const int64_t rows = ws->rows;
  rf->last_rows = rows;
  rf->last_selected = 0;
  if (rows == 0) return PKB_OK;
  PKB_REQUIRE(in.cols % 8 == 0 && in.pitch_elems % 8 == 0,
              "nnet_forward_refined: input rows must be multiples of 16 bytes");
  PKB_TRY(rf->near_cnt.ensure(static_cast<size_t>(rows) * sizeof(int)));
  PKB_TRY(rf->list.ensure(static_cast<size_t>(rows) * sizeof(int32_t)));
  PKB_TRY(rf->n_sel.ensure(sizeof(int)));
  if (rf->h_n_sel == nullptr)
    PKB_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&rf->h_n_sel), sizeof(int32_t), cudaHostAllocDefault));
  PKB_CUDA(cudaMemsetAsync(rf->near_cnt.p, 0, static_cast<size_t>(rows) * sizeof(int), c->stream));
  PKB_CUDA(cudaMemsetAsync(rf->n_sel.p, 0, sizeof(int), c->stream));
  // pass 1: one FP16 MMA per product
  PKB_TRY(nnet_forward(am, ws, in, mode, prob_scale, d_out, d_h16, d_off, true, rf->near_cnt.as<int>(),
                       am->refine_margin));
  {
    LaunchScope scope(c, PKB_KERNEL_MISC);
    select_rows_kernel<<<static_cast<unsigned>((rows + 1023) / 1024), 1024, 0, c->stream>>>(
        rf->near_cnt.as<int>(), row_map, rows, rf->list.as<int32_t>(), rf->n_sel.as<int>());
    PKB_CUDA(cudaGetLastError());
  }
  PKB_CUDA(cudaMemcpyAsync(rf->h_n_sel, rf->n_sel.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  const int n = *rf->h_n_sel;
  rf->last_selected = n;
  if (n == 0) return PKB_OK;
  // pass 2 over the selected rows: buffers grow with some headroom so that a slightly larger
  // selection in the next batch does not reallocate
  const size_t cap = static_cast<size_t>(n) + static_cast<size_t>(n) / 8 + 128;
  const size_t in_bytes = static_cast<size_t>(in.cols) * 2;
  const int out_dim = am->stages.back().out_dim;
  if (rf->in_hi.cap < static_cast<size_t>(n) * in_bytes) {
    PKB_TRY(rf->in_hi.ensure(cap * in_bytes));
    PKB_TRY(rf->in_lo.ensure(cap * in_bytes));
  }
  if (mode == kFinalCompact) {
    if (rf->out_h16.cap < static_cast<size_t>(n) * out_dim * 2) PKB_TRY(rf->out_h16.ensure(cap * out_dim * 2));
    if (rf->out_off.cap < static_cast<size_t>(n) * sizeof(float)) PKB_TRY(rf->out_off.ensure(cap * sizeof(float)));
  } else if (rf->out_f32.cap < static_cast<size_t>(n) * out_dim * sizeof(float)) {
    PKB_TRY(rf->out_f32.ensure(cap * out_dim * sizeof(float)));
  }
  if (rf->ws.rows < n || rf->ws.act_hi[0].p == nullptr) {
    PKB_TRY(workspace_ensure(am, &rf->ws, static_cast<int64_t>(cap)));
  }
  rf->ws.rows = n;
  {
    const int v16 = in.cols / 8, pitch16 = in.pitch_elems / 8;
    const int grid = static_cast<int>(std::min<int64_t>((static_cast<int64_t>(n) * v16 + 255) / 256,
                                                        static_cast<int64_t>(c->sm_count) * 16));
    LaunchScope scope(c, PKB_KERNEL_MISC);
    gather_rows_kernel<<<grid, 256, 0, c->stream>>>(
        reinterpret_cast<const uint4 *>(in.hi), reinterpret_cast<const uint4 *>(in.lo),
        rf->list.as<int32_t>(), n, v16, pitch16, rf->in_hi.as<uint4>(), rf->in_lo.as<uint4>());
    PKB_CUDA(cudaGetLastError());
  }
  InputView in2;
  in2.hi = rf->in_hi.as<__nv_bfloat16>();
  in2.lo = rf->in_lo.as<__nv_bfloat16>();
  in2.rows = n;
  in2.cols = in.cols;
  in2.pitch_elems = in.cols;
  PKB_TRY(nnet_forward(am, &rf->ws, in2, mode, prob_scale, rf->out_f32.as<float>(),
                       rf->out_h16.as<uint16_t>(), rf->out_off.as<float>()));
  if (mode == kFinalCompact) {
    PKB_TRY(launch_scatter(c, rf->out_h16.p, rf->list.as<int32_t>(), n, static_cast<size_t>(out_dim) * 2, d_h16));
    PKB_TRY(launch_scatter(c, rf->out_off.p, rf->list.as<int32_t>(), n, sizeof(float), d_off));
  } else {
    PKB_TRY(launch_scatter(c, rf->out_f32.p, rf->list.as<int32_t>(), n, static_cast<size_t>(out_dim) * 4, d_out));
  }
  return PKB_OK;
}

int copy_rows_compact(Ctx *c, void *host_dst, const void *d_padded, const BatchMeta &m,
                      const std::vector<int64_t> &pad_off, int cols, int64_t frame0, int64_t n,
                      size_t elem_bytes) {
  if (n <= 0) return PKB_OK;
  // first utterance whose frame range reaches past frame0
  int u = static_cast<int>(std::upper_bound(m.frame_off.begin(), m.frame_off.end(), frame0) -
                           m.frame_off.begin()) - 1;
  if (u < 0) u = 0;
  const int64_t end = frame0 + n;
  char *dst = static_cast<char *>(host_dst);
  const size_t row_bytes = static_cast<size_t>(cols) * elem_bytes;
  while (u < m.n_utts && m.frame_off[u] < end) {
    const int64_t a = std::max<int64_t>(frame0, m.frame_off[u]);
    const int64_t b = std::min<int64_t>(end, m.frame_off[u + 1]);
    if (b <= a) { ++u; continue; }
    const int64_t prow = pad_off[u] + (a - m.frame_off[u]);
    // a run of whole utterances of equal length is one strided 2-D copy (source pitch = padded
    // utterance, destination pitch = compact utterance) instead of one copy per utterance
    int run = 1;
    const int64_t T = m.num_frames[u];
    if (a == m.frame_off[u] && b == m.frame_off[u + 1] && T > 0) {
      // equal lengths imply equal padded pitch: pad_off[v + 1] - pad_off[v] = T_v + left + right
      while (u + run < m.n_utts && m.num_frames[u + run] == T && m.frame_off[u + run + 1] <= end)
        ++run;
    }
    if (run > 1) {
      const size_t src_pitch = static_cast<size_t>(pad_off[u + 1] - pad_off[u]) * row_bytes;
      PKB_CUDA(cudaMemcpy2DAsync(dst + (a - frame0) * row_bytes, static_cast<size_t>(T) * row_bytes,
                                 reinterpret_cast<const char *>(d_padded) + prow * row_bytes, src_pitch,
                                 static_cast<size_t>(T) * row_bytes, run, cudaMemcpyDeviceToHost,
                                 c->stream));
    } else {
      PKB_CUDA(cudaMemcpyAsync(dst + (a - frame0) * row_bytes,
                               reinterpret_cast<const char *>(d_padded) + prow * row_bytes,
                               (b - a) * row_bytes, cudaMemcpyDeviceToHost, c->stream));
    }
    u += run;
  }
  return PKB_OK;
}

namespace {
__global__ void checksum_rows_kernel(const float *__restrict__ x, int cols, int64_t rows,
                                     const int32_t *__restrict__ row_map, double *sum) {
  double acc = 0.0;
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    if (row_map[r] < 0) continue;
    const float *row = x + r * cols;
    for (int j = threadIdx.x; j < cols; j += blockDim.x) acc += static_cast<double>(row[j]);
  }
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

int launch_checksum_rows(Ctx *c, const float *d, int cols, int64_t rows, const int32_t *row_map,
                         double *d_sum) {
  PKB_CUDA(cudaMemsetAsync(d_sum, 0, sizeof(double), c->stream));
  if (rows == 0) return PKB_OK;
  const int grid = static_cast<int>(std::min<int64_t>(rows, static_cast<int64_t>(c->sm_count) * 16));
  LaunchScope scope(c, PKB_KERNEL_MISC);
  checksum_rows_kernel<<<grid, 256, 0, c->stream>>>(d, cols, rows, row_map, d_sum);
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

int launch_pack_padded(Ctx *c, const float *d_feats, const BatchMeta &m, int dim, int dim_pad,
                       int left, int right, const int64_t *d_pad_off, __nv_bfloat16 *hi,
                       __nv_bfloat16 *lo, int32_t *row_map, int fp16) {
  if (m.total_frames == 0) return PKB_OK;
  const int64_t threads = m.total_frames * dim_pad;
  const int grid = static_cast<int>((threads + 255) / 256);
  LaunchScope scope(c, PKB_KERNEL_MISC);
  pack_padded_kernel<<<grid, 256, 0, c->stream>>>(d_feats, m.d_frame_off, m.d_num_frames, d_pad_off,
                                                  m.n_utts, dim, dim_pad, left, right,
                                                  m.total_frames, hi, lo, row_map, fp16);
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

int launch_pack_plain(Ctx *c, const float *d_in, int64_t rows, int groups, int group, int group_pad,
                      __nv_bfloat16 *hi, __nv_bfloat16 *lo, int fp16) {
  if (rows == 0) return PKB_OK;
  const int dim_pad = groups * group_pad;
  const int64_t threads = rows * dim_pad;
  const int grid = static_cast<int>((threads + 255) / 256);
  LaunchScope scope(c, PKB_KERNEL_MISC);
  pack_plain_kernel<<<grid, 256, 0, c->stream>>>(d_in, rows, groups * group, dim_pad, group, group_pad, hi,
                                                 lo, fp16);
  PKB_CUDA(cudaGetLastError());
  return PKB_OK;
}

int launch_row_map(Ctx *c, const BatchMeta &m, int left, int right, const int64_t *d_pad_off,
                   int32_t *row_map, int64_t rows) {
  (void)left;
  (void)right;
  if (rows == 0) return PKB_OK;
  PKB_CUDA(cudaMemsetAsync(row_map, 0xFF, static_cast<size_t>(rows) * sizeof(int32_t), c->stream));
  int max_t = 0;
  for (int32_t t : m.num_frames) max_t = std::max(max_t, t);
  const int bx = std::max(1, std::min((max_t + 255) / 256, 16));
  for (int u0 = 0; u0 < m.n_utts; u0 += 32768) {
    const int nu = std::min(32768, m.n_utts - u0);
    LaunchScope scope(c, PKB_KERNEL_MISC);
    row_map_kernel<<<dim3(bx, nu), 256, 0, c->stream>>>(m.d_frame_off + u0, m.d_num_frames + u0,
                                                        d_pad_off + u0, nu, row_map);
    PKB_CUDA(cudaGetLastError());
  }
  return PKB_OK;
}

}  // namespace pkb
