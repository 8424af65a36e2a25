// GPU token-passing Viterbi beam search over a pocketkaldi FST (SURVEY 8(f)-4).
//
// Replaces, for whole batches whose log-likelihoods are already resident on the device,
// Decoder::Decode + BestPath (src/decoder.cc:39-339) over Fst (src/fst.cc:29-129) with the
// decodable look-up of src/decodable.cc:24-31 -- the consumer that otherwise pulls the
// [frames x pdfs] matrix over PCIe and walks it on one host core per utterance.
#pragma once

#include <string>
#include <vector>

#include "common.cuh"

struct pkb_fst {
  pkb::Ctx *c = nullptr;
  int num_states = 0, num_arcs = 0, start = 0;
  bool has_eps = false;  // some arc has input label 0
  int max_ilabel = 0;    // largest input label (must index the model's tid2pdf map)
  pkb::DevBuf buf;       // one allocation, pointers below
  const float *d_final = nullptr;      // [num_states]
  const int32_t *d_arc_begin = nullptr;  // [num_states + 1]: arcs of state s are [begin[s], begin[s + 1])
  const int32_t *d_arc_src = nullptr;    // [num_arcs]
  const int32_t *d_arc_dst = nullptr, *d_arc_il = nullptr, *d_arc_ol = nullptr;
  const float *d_arc_w = nullptr;
};

namespace pkb {

// Builds the device FST from the file layout of src/fst.cc:29-92: final[state], first_arc[state]
// (-1: no arcs) and arcs {next_state, input_label, output_label, weight} sorted by source state.
int fst_build(Ctx *c, int num_states, int start, const float *final_w, const int32_t *first_arc,
              int num_arcs, const int32_t *arcs_raw /* 4 x int32 per arc, weight as float bits */,
              pkb_fst **out);

struct ViterbiConfig {
  float beam = 16.0f;        // Decoder::beam_ (src/decoder.cc:29)
  int max_tokens = 4096;     // tokens created per frame and utterance; more fail the utterance
  int max_log = 1 << 18;     // word back-pointer records per utterance
  int max_words = 256;       // words returned per utterance
  int max_active = 0;        // tokens expanded per frame, ties at the cutoff included (0: no limit)
};

// Kernel choice and workspace of one search (launch_viterbi picks the same for both entry points).
struct VitPlan {
  bool dense = false;   // dense shared-memory kernel (small graphs) instead of the hash-table kernel
  bool small = false;   // table kernel with its tables in shared memory
  int variant = 0;      // arcs per thread (dense) or lanes per token (table)
  int max_tok = 0;      // token capacity per frame
  uint32_t H = 0;       // hash-table slots
  int grid = 0;
  size_t stride = 0;    // global workspace bytes per block
  size_t smem = 0;      // dynamic shared memory
};

// Carried state of the resumable search (pkb_decoder): what one stream keeps in global memory
// between launches. A launch restores the tokens into its tables, runs the new frames with the
// per-frame code of the batch search and saves them back.
struct Carry {
  int *hdr;              // [n][4]: live tokens (-1: fresh utterance), word records used, error, alive
  long long *frames;     // [n] frames decoded in this utterance
  int *tok_state;        // [n][cap] live tokens: state, cost, newest word record
  float *tok_cost;
  int *tok_bp;
  int cap;
  int frame_stride;      // the rows of stream s start at row s * frame_stride
  int uniform_frames;    // new frames of every stream when num_frames is NULL
  int finish;            // BestPath of the current tokens, then a fresh utterance
  long long *p_frames;   // best-so-far per stream: frames, [n][max_words] words, word count, cost
  int32_t *p_words;
  int32_t *p_nw;
  float *p_cost;
};

// Lattice output of the batch search (pkb_batch_lattice). Utterance u logs every arc the search
// relaxed under its bounds as (arc << 32 | float bits of the tail's cost) at log + u * max_arcs, in
// the groups eps(0), emit(0), eps(1), ..., whose start offsets go to grp + u * grp_stride
// (2 (T + 1) ints; grp[2T + 1] is the log's length). After the last frame the block runs the
// backward pass and leaves the kept arcs at the start of its log as (group << 32 | arc), in order.
struct Lattice {
  unsigned long long *log;
  int *grp;
  long long *n_out;    // [n] kept arcs, or -(error code)
  double *best_out;    // [n] min over final nodes of double(alpha) + double(final)
  int max_arcs, grp_stride;
  float beam;          // lattice beam
  // Resumable search only (pkb_decoder_set_lattice). Groups are indexed by utterance time, so an
  // advance that starts at frame t0 logs emit(t) / eps(t + 1) at grp[2 (t0 + t) + 1 / + 2]. Each
  // advance copies its rows to rows + (s * max_frames + t0) * num_pdfs for the backward pass of
  // the finish, which reads them back as its loglik with frame_stride = max_frames.
  int *state;          // [n][2]: log length, lattice error (4 arcs, 5 frames; apart from the search's)
  float *rows;         // [n][max_frames][num_pdfs]
  int max_frames;
};

// Decodes n_utts utterances. loglik: [rows][num_pdfs] scaled log-likelihoods where utterance u owns
// rows [row_off[u], row_off[u] + num_frames[u]). tid2pdf: device map of input labels.
// words_out [n_utts][max_words] in spoken order, n_words_out[u] (-1: the search failed: token or
// log capacity exceeded), weight_out[u] = Hypothesis::weight() of Decoder::BestPath.
int launch_viterbi(Ctx *c, const pkb_fst *fst, const ViterbiConfig &cfg, const float *d_loglik,
                   int num_pdfs, const int64_t *d_row_off, const int32_t *d_num_frames, int n_utts,
                   const int32_t *d_tid2pdf, int n_tids, DevBuf *work, int32_t *d_words,
                   int32_t *d_n_words, float *d_weight);

// The search of launch_viterbi in lattice mode: per utterance lat.n_out / lat.best_out and the kept
// arcs in lat.log (see Lattice); LatticeResults::expand turns them into records.
int launch_lattice(Ctx *c, const pkb_fst *fst, const ViterbiConfig &cfg, const float *d_loglik, int num_pdfs,
                   const int64_t *d_row_off, const int32_t *d_num_frames, int n_utts, const int32_t *d_tid2pdf,
                   DevBuf *work, const Lattice &lat);
// Log entries per utterance of a lattice search over `frames` frames: max_arcs, or for max_arcs <= 0
// the most the search can log, (frames + 1) x arcs of the graph. The log count is an int that passes
// max_arcs by at most one group (at most the graph's arcs), so the default is capped at
// INT32_MAX - arcs and a larger max_arcs is rejected.
int lattice_max_arcs(const pkb_fst *fst, int frames, int max_arcs, const char *who, int *out);

// Utterances in waves whose bytes (bytes[u] per utterance) stay within 8 GiB or half the free device
// memory, whichever is less, with at least one utterance each: wave i is [starts[i], starts[i + 1]).
// *most (if not NULL): the bytes of the largest wave.
int plan_waves(const std::vector<size_t> &bytes, std::vector<int> *starts, size_t *most);

// Results of the latest posteriors call, kept on the device for the _get call: one float per
// record, and every utterance's frame entries back to back.
struct PosteriorResults {
  DevBuf arc, frames;
  int64_t n_arcs = -1;   // records covered (-1: no valid results)
  int64_t n_frames = 0;  // frame entries
};

// Results of the latest best-path call, kept on the device for the _get call: every utterance's
// words, then every utterance's word times, and every utterance's alignment, back to back.
struct BestPathResults {
  DevBuf words, ali;
  int64_t n_words = -1;  // words (-1: no valid results)
  int64_t n_frames = 0;  // alignment entries
};

// The lattice of the latest search of a batch or decoder and what is computed from it: utterance u's
// n_arcs[u] kept records (or its negative code) from arcs + first[u] on, and its best cost. Every
// operation takes the name of its entry point for its messages and checks the results are valid.
struct LatticeResults {
  Ctx *c = nullptr;
  const pkb_fst *fst = nullptr;          // the graph the records belong to
  const int32_t *d_tid2pdf = nullptr;    // its input labels' pdfs, in [0, num_pdfs)
  int num_pdfs = 0;
  DevBuf arcs;                           // the records, every utterance's back to back
  DevBuf meta;                           // device copy of n_arcs, first and best
  std::vector<int64_t> n_arcs;
  std::vector<long long> first;
  std::vector<double> best;
  int64_t total = -1;                    // records (-1: not valid, for the reason in why)
  std::string why = "no lattice search yet";
  DevBuf nbest_work;                     // outputs of nbest
  PosteriorResults post;                 // results of posteriors, valid as the records are
  BestPathResults bp;                    // results of best_path, valid as the records are

  long long *d_n_arcs() const { return meta.as<long long>(); }
  long long *d_first() const { return d_n_arcs() + n_arcs.size(); }
  double *d_best() const { return reinterpret_cast<double *>(d_first() + n_arcs.size()); }
  void invalidate(std::string reason) {
    total = -1;
    why = std::move(reason);
    post.n_arcs = -1;
    bp.n_words = -1;
  }
  // After launch_lattice (or the finish of a resumable search) over n_utts utterances whose rows
  // start at d_loglik + d_row_off[u] * num_pdfs: copies lat.n_out / lat.best_out to the host and
  // writes the kept arcs as records. Valid when it returns PKB_OK.
  int expand(Ctx *ctx, const pkb_fst *graph, const Lattice &lat, int n_utts, const float *d_loglik, int pdfs,
             const int64_t *d_row_off, const int32_t *tid2pdf, const char *who);
  int get(pkb_lattice_arc_t *arcs_out, const char *who) const;
  // N-best lists of distinct word sequences per utterance (nbest.cu), with the arguments and host
  // outputs of pkb_batch_nbest. nbest_work keeps the outputs and statistics; the per-block lists
  // (2 x states x n x 24 bytes) and word-history tables are allocated per call.
  int nbest(int n, int max_words, int32_t *words_out, int32_t *n_words_out, double *graph_cost_out,
            double *acoustic_cost_out, int32_t *n_hyps_out, const char *who);
  // Arc and frame posteriors per utterance (posterior.cu), with the arguments and host outputs of
  // pkb_batch_posteriors. Alpha (8 bytes per record) and the per-block workspace are allocated per
  // call, in waves.
  int posteriors(float acoustic_scale, float graph_scale, float min_post, double *total_out, int64_t *n_post_out,
                 const char *who);
  // Copies the results of the latest posteriors out (either output may be NULL).
  int posteriors_get(float *arc_post_out, pkb_frame_post_t *frame_post_out, const char *who);
  // The best path per utterance at the given scales and word insertion penalty (best_path.cu), with
  // the arguments and host outputs of pkb_batch_best_path. Alpha and the path (12 bytes per record)
  // and the per-block workspace are allocated per call, in waves.
  int best_path(float acoustic_scale, float graph_scale, float word_penalty, double *cost_out,
                double *graph_cost_out, double *acoustic_cost_out, int32_t *n_words_out, int32_t *n_frames_out,
                const char *who);
  // Copies the words, word times and alignments of the latest best_path out (any may be NULL).
  int best_path_get(int32_t *words_out, int32_t *word_t_out, int32_t *ali_out, const char *who);
};

// The resumable search behind pkb_decoder: n streams, one thread block each, whose tokens and word
// records stay in global memory between launches. advance() decodes the next rows of every stream
// (stream s: rows [s * frame_stride, s * frame_stride + n_frames[s]) of d_loglik, or uniform_frames
// rows each when d_n_frames is NULL) and leaves the best-so-far block in `out`; its arguments stay
// fixed for fixed inputs, so it can be captured into a CUDA graph. finish() applies BestPath to the
// current tokens (f_words / f_nw / f_weight, as launch_viterbi) and starts a fresh utterance.
struct ResumableSearch {
  Ctx *c = nullptr;
  const pkb_fst *fst = nullptr;
  ViterbiConfig cfg;
  int num_pdfs = 0, n = 0;
  VitPlan plan;
  DevBuf work, carry, out, d_tid2pdf;
  Carry cr{};
  size_t partial_bytes = 0;  // the best-so-far block at the start of `out`
  int32_t *f_words = nullptr, *f_nw = nullptr;
  float *f_weight = nullptr;
  // lattice mode (set_lattice): lat.log == nullptr when off. lat_aux holds the group offsets, the
  // per-stream state, the finish results and the row offsets of the row store.
  Lattice lat{};
  DevBuf lat_log, lat_aux, lat_rows;
  int64_t *lat_row_off = nullptr;
  int setup(Ctx *ctx, const pkb_fst *graph, const ViterbiConfig &config, const int32_t *tid2pdf, int n_tids,
            int pdfs, int streams);
  // lattice_beam > 0 switches lattice mode on (buffers for max_frames > 0 frames and max_arcs > 0
  // log entries per stream), 0 off. Only between utterances.
  int set_lattice(float lattice_beam, int max_frames, int max_arcs);
  int advance(const float *d_loglik, int frame_stride, const int32_t *d_n_frames, int uniform_frames);
  int finish();
};

// Checks shared by pkb_batch_decode and pkb_decoder_create / _finish: the FST is from context c, the
// model has a tid2pdf map that covers the graph's input labels and points into its pdfs; the
// output arguments exist.
int check_decode_graph(const Ctx *c, const pkb_am *am, const pkb_fst *fst, const char *who);
int check_decode_outputs(int max_words, const void *words_out, const void *n_words_out, const void *weight_out,
                         const char *who);

}  // namespace pkb

// n_streams searches of pkb_decoder_create (include/pkb200.h).
struct pkb_decoder {
  pkb::Ctx *c = nullptr;
  const pkb_am *am = nullptr;
  int n = 0;
  pkb::ResumableSearch search;
  pkb::DevBuf rows, nfr;        // staging of the host-fed advance: rows, frames per stream
  struct { void *p = nullptr; } partial;  // pinned host copy of the best-so-far block
  pkb_stream *st = nullptr;     // attached stream (pkb_stream_set_decoder)
  bool flushed = false;         // the attached stream was flushed: finish before its next push
  bool in_utt = false;          // an advance, push or flush since create or the last finish
  pkb::LatticeResults lat;      // of the latest finish in lattice mode, valid until the next advance, push or flush
  pkb_decoder() = default;
  pkb_decoder(const pkb_decoder &) = delete;
  pkb_decoder &operator=(const pkb_decoder &) = delete;
  ~pkb_decoder();
};

namespace pkb {
// Queues an advance over device rows and the copy of its best-so-far block to the host.
int decoder_enqueue_advance(pkb_decoder *dec, const float *d_rows, int frame_stride, const int32_t *d_n_frames,
                            int uniform_frames);
// Host state of a decoder whose utterance moves on (an advance, or a push / flush of the attached
// stream, whose captured graph advances the decoder without host code): the lattice results of
// the last finish stop being valid and lattice mode can no longer change.
void decoder_begin_step(pkb_decoder *dec);
// Destroys the captured CUDA graphs of a stream's pushes (stream_api.cu).
void stream_drop_graphs(pkb_stream *st);
}  // namespace pkb
