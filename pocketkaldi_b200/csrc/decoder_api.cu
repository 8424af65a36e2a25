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

int check_nbest_args(int n, int max_words, const void *words_out, const void *n_words_out,
                     const void *graph_cost_out, const void *acoustic_cost_out, const void *n_hyps_out,
                     const char *who) {
  PKB_REQUIRE(n >= 1 && n <= 1024, "%s: n must be in [1, 1024] (got %d)", who, n);
  PKB_REQUIRE(max_words > 0, "%s: max_words must be > 0 (got %d)", who, max_words);
  PKB_REQUIRE(words_out && n_words_out && graph_cost_out && acoustic_cost_out && n_hyps_out,
              "%s: NULL output argument", who);
  return PKB_OK;
}

int decoder_enqueue_advance(pkb_decoder *dec, const float *d_rows, int frame_stride, const int32_t *d_n_frames,
                            int uniform_frames) {
  PKB_TRY(dec->search.advance(d_rows, frame_stride, d_n_frames, uniform_frames));
  PKB_CUDA(cudaMemcpyAsync(dec->partial.p, dec->search.out.p, dec->search.partial_bytes, cudaMemcpyDeviceToHost,
                           dec->c->stream));
  return PKB_OK;
}

void decoder_begin_step(pkb_decoder *dec) {
  dec->in_utt = true;
  dec->lat_total = -1;
  dec->lat_why = "an advance, push or flush came after the latest pkb_decoder_finish";
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
  pkb::decoder_begin_step(dec);
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
  dec->in_utt = false;
  dec->lat_total = -1;
  dec->lat_why = "the latest pkb_decoder_finish ran without lattices";
  PKB_TRY(pkb::check_device_error(c, "pkb_decoder_finish"));
  if (r.lat.log) {
    // the words above are complete and the utterance is over: a lattice that cannot be expanded
    // (the records of a large graph can take gigabytes) is reported by pkb_decoder_lattice instead
    dec->lat_n.resize(S);
    dec->lat_best.resize(S);
    int64_t total = 0;
    if (r.expand_lattice(dec->lat_n.data(), dec->lat_best.data(), &total) == PKB_OK) {
      dec->lat_total = total;
    } else {
      dec->lat_why = std::string("expanding the lattices of the latest pkb_decoder_finish failed: ") + pkb_last_error();
      cudaGetLastError();
    }
  }
  return PKB_OK;
}

int pkb_decoder_set_lattice(pkb_decoder_t *dec, float lattice_beam, int max_frames, int max_arcs) {
  PKB_REQUIRE(dec, "pkb_decoder_set_lattice: decoder is NULL");
  PKB_REQUIRE(lattice_beam >= 0.0f, "pkb_decoder_set_lattice: lattice_beam must be >= 0 (got %g)", lattice_beam);
  PKB_REQUIRE(max_frames <= (1 << 24), "pkb_decoder_set_lattice: max_frames %d is more than %d", max_frames, 1 << 24);
  // the log count is an int and passes max_arcs by at most one group (at most the graph's arcs)
  const int arcs_cap = INT32_MAX - std::max(dec->search.fst->num_arcs, 1);
  PKB_REQUIRE(max_arcs <= arcs_cap, "pkb_decoder_set_lattice: max_arcs %d is more than %d", max_arcs, arcs_cap);
  PKB_REQUIRE(!dec->in_utt,
              "pkb_decoder_set_lattice: only between utterances (after create or pkb_decoder_finish)");
  pkb::Ctx *c = dec->c;
  PKB_CUDA(cudaSetDevice(c->device));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  // the attached stream's captured pushes launch the advance with the old lattice arguments (or
  // none): they are captured again
  if (dec->st) pkb::stream_drop_graphs(dec->st);
  dec->lat_total = -1;
  dec->lat_why = "pkb_decoder_set_lattice came after the latest pkb_decoder_finish";
  return dec->search.set_lattice(lattice_beam, max_frames, max_arcs);
}

int pkb_decoder_lattice(pkb_decoder_t *dec, int64_t *n_arcs_out, double *best_cost_out) {
  PKB_REQUIRE(dec && n_arcs_out && best_cost_out, "pkb_decoder_lattice: NULL argument");
  PKB_REQUIRE(dec->lat_total >= 0, "pkb_decoder_lattice: no lattice: %s", dec->lat_why.c_str());
  memcpy(n_arcs_out, dec->lat_n.data(), sizeof(int64_t) * dec->n);
  memcpy(best_cost_out, dec->lat_best.data(), sizeof(double) * dec->n);
  return PKB_OK;
}

int pkb_decoder_lattice_get(pkb_decoder_t *dec, pkb_lattice_arc_t *arcs_out) {
  PKB_REQUIRE(dec, "pkb_decoder_lattice_get: decoder is NULL");
  PKB_REQUIRE(dec->lat_total >= 0, "pkb_decoder_lattice_get: no lattice: %s", dec->lat_why.c_str());
  if (dec->lat_total == 0) return PKB_OK;
  PKB_REQUIRE(arcs_out, "pkb_decoder_lattice_get: NULL argument");
  pkb::Ctx *c = dec->c;
  PKB_CUDA(cudaSetDevice(c->device));
  PKB_CUDA(cudaMemcpyAsync(arcs_out, dec->search.lat_arcs.p, sizeof(pkb_lattice_arc_t) * dec->lat_total,
                           cudaMemcpyDeviceToHost, c->stream));
  PKB_CUDA(cudaStreamSynchronize(c->stream));
  return pkb::check_device_error(c, "pkb_decoder_lattice_get");
}

int pkb_decoder_nbest(pkb_decoder_t *dec, int n, int max_words, int32_t *words_out, int32_t *n_words_out,
                      double *graph_cost_out, double *acoustic_cost_out, int32_t *n_hyps_out) {
  PKB_REQUIRE(dec, "pkb_decoder_nbest: decoder is NULL");
  PKB_REQUIRE(dec->lat_total >= 0, "pkb_decoder_nbest: no lattice: %s", dec->lat_why.c_str());
  PKB_TRY(pkb::check_nbest_args(n, max_words, words_out, n_words_out, graph_cost_out, acoustic_cost_out,
                                n_hyps_out, "pkb_decoder_nbest"));
  pkb::Ctx *c = dec->c;
  PKB_CUDA(cudaSetDevice(c->device));
  const pkb::ResumableSearch &r = dec->search;
  pkb::LatticeRecords lr;
  lr.arcs = r.lat_arcs.as<pkb_lattice_arc_t>();
  lr.first = r.lat_first;
  lr.n_arcs = r.lat.n_out;
  lr.best = r.lat.best_out;
  lr.n_utts = dec->n;
  PKB_TRY(pkb::launch_nbest(c, r.fst, lr, n, max_words, &dec->nbest_work, words_out, n_words_out, graph_cost_out,
                            acoustic_cost_out, n_hyps_out));
  return pkb::check_device_error(c, "pkb_decoder_nbest");
}

}  // extern "C"
