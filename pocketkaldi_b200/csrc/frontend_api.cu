// Host-buffer entry points of the front end: the batched equivalents of
// Fbank::Compute (src/fbank.cc:267-292) and CMVN::GetFrame (src/cmvn.cc:103-115).

#include "common.cuh"

using pkb::BatchMeta;
using pkb::Ctx;

namespace {

template <typename SampleT>
int fbank_host(pkb_ctx_t *c, const SampleT *wave, const int32_t *num_samples, int n_utts,
               float *feats_out, int32_t *num_frames_out) {
  PKB_REQUIRE(c, "pkb_fbank: ctx is NULL");
  PKB_REQUIRE(n_utts == 0 || num_samples, "pkb_fbank: num_samples is NULL");
  PKB_CUDA(cudaSetDevice(c->device));
  BatchMeta &m = c->meta;
  PKB_TRY(m.build_from_samples(num_samples, n_utts));
  if (num_frames_out)
    for (int u = 0; u < n_utts; ++u) num_frames_out[u] = m.num_frames[u];
  if (m.total_frames == 0) return PKB_OK;
  PKB_REQUIRE(wave && feats_out, "pkb_fbank: wave / feats_out is NULL");
  PKB_TRY(m.upload(c->stream));
  const size_t in_bytes = static_cast<size_t>(m.total_samples) * sizeof(SampleT);
  const size_t out_bytes = static_cast<size_t>(m.total_frames) * pkb::kMel * sizeof(float);
  PKB_TRY(c->s_in.ensure(in_bytes));
  PKB_TRY(c->s_raw.ensure(out_bytes));
  PKB_CUDA(cudaMemcpyAsync(c->s_in.p, wave, in_bytes, cudaMemcpyHostToDevice, c->stream));
  if (sizeof(SampleT) == 2)
    PKB_TRY(pkb::launch_fbank_i16(c, c->s_in.as<int16_t>(), m, c->s_raw.as<float>()));
  else
    PKB_TRY(pkb::launch_fbank_f32(c, c->s_in.as<float>(), m, c->s_raw.as<float>()));
  PKB_CUDA(cudaMemcpyAsync(feats_out, c->s_raw.p, out_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return PKB_OK;
}

}  // namespace

extern "C" {

int pkb_fbank_f32(pkb_ctx_t *c, const float *wave, const int32_t *num_samples, int n_utts,
                  float *feats_out, int32_t *num_frames_out) {
  return fbank_host<float>(c, wave, num_samples, n_utts, feats_out, num_frames_out);
}

int pkb_fbank_i16(pkb_ctx_t *c, const int16_t *pcm, const int32_t *num_samples, int n_utts,
                  float *feats_out, int32_t *num_frames_out) {
  return fbank_host<int16_t>(c, pcm, num_samples, n_utts, feats_out, num_frames_out);
}

int pkb_cmvn(pkb_ctx_t *c, const float *raw, const int32_t *num_frames, int n_utts,
             const float *global_stats, float *out) {
  PKB_REQUIRE(c, "pkb_cmvn: ctx is NULL");
  PKB_REQUIRE(global_stats, "pkb_cmvn: global_stats is NULL");
  PKB_REQUIRE(n_utts == 0 || num_frames, "pkb_cmvn: num_frames is NULL");
  PKB_CUDA(cudaSetDevice(c->device));
  BatchMeta &m = c->meta;
  PKB_TRY(m.build_from_frames(num_frames, n_utts));
  if (m.total_frames == 0) return PKB_OK;
  PKB_REQUIRE(raw && out, "pkb_cmvn: raw / out is NULL");
  PKB_TRY(pkb::prepare_cmvn_tables(c, global_stats));
  PKB_TRY(m.upload(c->stream));
  const size_t bytes = static_cast<size_t>(m.total_frames) * pkb::kMel * sizeof(float);
  PKB_TRY(c->s_raw.ensure(bytes));
  PKB_TRY(c->s_out.ensure(bytes));
  PKB_CUDA(cudaMemcpyAsync(c->s_raw.p, raw, bytes, cudaMemcpyHostToDevice, c->stream));
  PKB_TRY(pkb::launch_cmvn(c, c->s_raw.as<float>(), m, c->s_out.as<float>(), nullptr));
  PKB_CUDA(cudaMemcpyAsync(out, c->s_out.p, bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return PKB_OK;
}

}  // extern "C"
