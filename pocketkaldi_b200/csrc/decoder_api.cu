// Online decoding entry points (pkb_decoder_*): the resumable GPU search of decoder.cu for
// n_streams streams that advance chunk by chunk, fed from host rows or, attached to a pkb_stream,
// from the rows its push just computed on the device.

#include <algorithm>
#include <memory>

#include "decoder.cuh"
#include "nnet.cuh"

namespace pkb {

int check_decode_graph(const Ctx *c, const pkb_am *am, const pkb_fst *fst, const char *who) {
  PKB_REQUIRE(fst->c == c, "%s: the FST belongs to another context", who);
  PKB_REQUIRE(!am->tid2pdf.empty(), "%s: the model has no tid2pdf map", who);
  PKB_REQUIRE(fst->max_ilabel < static_cast<int>(am->tid2pdf.size()),
              "%s: the graph uses input label %d but the model's tid2pdf map has %zu entries", who,
              fst->max_ilabel, am->tid2pdf.size());
  for (int32_t v : am->tid2pdf)
    PKB_REQUIRE(v >= 0 && v < am->num_pdfs, "%s: tid2pdf entry %d outside [0, %d)", who, v, am->num_pdfs);
  return PKB_OK;
}

int check_decode_outputs(int max_words, const void *words_out, const void *n_words_out, const void *weight_out,
                         const char *who) {
  PKB_REQUIRE(max_words > 0 && words_out && n_words_out && weight_out, "%s: bad output arguments", who);
  return PKB_OK;
}

int decoder_enqueue_advance(pkb_decoder *dec, const float *d_rows, int frame_stride, const int32_t *d_n_frames,
                            int uniform_frames) {
  PKB_TRY(dec->search.advance(d_rows, frame_stride, d_n_frames, uniform_frames));
  PKB_CUDA(cudaMemcpyAsync(dec->partial.p, dec->search.out.p, dec->search.partial_bytes, cudaMemcpyDeviceToHost,
                           dec->c->stream));
  return PKB_OK;
}

}  // namespace pkb

pkb_decoder::~pkb_decoder() {
  if (partial.p) cudaFreeHost(partial.p);
}

extern "C" {

int pkb_decoder_create(pkb_ctx_t *c, const pkb_am_t *am, const pkb_fst_t *fst, int n_streams, float beam,
                       int max_tokens, int max_words, int max_records, pkb_decoder_t **out) {
  PKB_REQUIRE(c && am && fst && out, "pkb_decoder_create: NULL argument");
  PKB_REQUIRE(am->c == c, "pkb_decoder_create: model belongs to another context");
  PKB_REQUIRE(n_streams > 0 && max_words > 0, "pkb_decoder_create: n_streams and max_words must be positive");
  PKB_TRY(pkb::check_decode_graph(c, am, fst, "pkb_decoder_create"));
  PKB_CUDA(cudaSetDevice(c->device));
  pkb::ViterbiConfig cfg;
  if (beam > 0.0f) cfg.beam = beam;
  if (max_tokens > 0) cfg.max_tokens = max_tokens;
  if (max_records > 0) cfg.max_log = max_records;
  cfg.max_words = max_words;
  std::unique_ptr<pkb_decoder, decltype(&pkb_decoder_destroy)> dec(new pkb_decoder(), pkb_decoder_destroy);
  dec->c = c;
  dec->am = am;
  dec->n = n_streams;
  PKB_TRY(dec->search.setup(c, fst, cfg, am->tid2pdf.data(), static_cast<int>(am->tid2pdf.size()), am->num_pdfs,
                            n_streams));
  PKB_CUDA(cudaHostAlloc(&dec->partial.p, dec->search.partial_bytes, cudaHostAllocDefault));
  memset(dec->partial.p, 0, dec->search.partial_bytes);
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  *out = dec.release();
  return PKB_OK;
}

void pkb_decoder_destroy(pkb_decoder_t *dec) {
  if (!dec) return;
  if (dec->c) {
    cudaSetDevice(dec->c->device);
    cudaStreamSynchronize(dec->c->stream);
  }
  if (dec->st) pkb_stream_set_decoder(dec->st, nullptr);
  delete dec;
}

int pkb_decoder_advance(pkb_decoder_t *dec, const float *loglik, int frame_stride, const int32_t *n_frames) {
  PKB_REQUIRE(dec && n_frames && frame_stride >= 0, "pkb_decoder_advance: bad argument");
  int most = 0;
  for (int s = 0; s < dec->n; ++s) {
    PKB_REQUIRE(n_frames[s] >= 0 && n_frames[s] <= frame_stride,
                "pkb_decoder_advance: stream %d has %d frames, the stride is %d", s, n_frames[s], frame_stride);
    most = std::max(most, n_frames[s]);
  }
  PKB_REQUIRE(loglik || most == 0, "pkb_decoder_advance: loglik is NULL");
  pkb::Ctx *c = dec->c;
  PKB_CUDA(cudaSetDevice(c->device));
  const size_t row_bytes = static_cast<size_t>(dec->am->num_pdfs) * sizeof(float);
  const size_t bytes = static_cast<size_t>(dec->n) * frame_stride * row_bytes;
  if (bytes) {
    PKB_TRY(dec->rows.ensure(bytes));
    PKB_TRY(pkb::upload(c, dec->rows.p, loglik, bytes));
  }
  PKB_TRY(dec->nfr.ensure(static_cast<size_t>(dec->n) * sizeof(int32_t)));
  PKB_TRY(pkb::upload(c, dec->nfr.p, n_frames, static_cast<size_t>(dec->n) * sizeof(int32_t)));
  PKB_TRY(pkb::decoder_enqueue_advance(dec, dec->rows.as<float>(), frame_stride, dec->nfr.as<int32_t>(), 0));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_decoder_advance");
}

int pkb_decoder_partial(pkb_decoder_t *dec, int32_t *words_out, int32_t *n_words_out, float *cost_out,
                        int64_t *frames_out) {
  PKB_REQUIRE(dec, "pkb_decoder_partial: decoder is NULL");
  const size_t S = dec->n, mw = dec->search.cfg.max_words;
  const char *p = static_cast<const char *>(dec->partial.p);
  if (frames_out) memcpy(frames_out, p, S * sizeof(int64_t));
  p += S * sizeof(int64_t);
  if (words_out) memcpy(words_out, p, S * mw * sizeof(int32_t));
  p += S * mw * sizeof(int32_t);
  if (n_words_out) memcpy(n_words_out, p, S * sizeof(int32_t));
  p += S * sizeof(int32_t);
  if (cost_out) memcpy(cost_out, p, S * sizeof(float));
  return PKB_OK;
}

int pkb_decoder_finish(pkb_decoder_t *dec, int32_t *words_out, int32_t *n_words_out, float *weight_out) {
  PKB_REQUIRE(dec, "pkb_decoder_finish: decoder is NULL");
  PKB_TRY(pkb::check_decode_outputs(dec->search.cfg.max_words, words_out, n_words_out, weight_out,
                                    "pkb_decoder_finish"));
  pkb::Ctx *c = dec->c;
  PKB_CUDA(cudaSetDevice(c->device));
  pkb::ResumableSearch &r = dec->search;
  PKB_TRY(r.finish());
  const size_t S = dec->n;
  PKB_CUDA(cudaMemcpyAsync(words_out, r.f_words, S * r.cfg.max_words * sizeof(int32_t), cudaMemcpyDeviceToHost,
                           c->stream));
  PKB_CUDA(cudaMemcpyAsync(n_words_out, r.f_nw, S * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaMemcpyAsync(weight_out, r.f_weight, S * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  // the best-so-far block now describes fresh utterances
  PKB_CUDA(cudaMemcpyAsync(dec->partial.p, r.out.p, r.partial_bytes, cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  dec->flushed = false;
  return pkb::check_device_error(c, "pkb_decoder_finish");
}

}  // extern "C"
