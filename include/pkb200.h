/* pkb200.h -- C ABI of the B200-native acoustic front half of pocketkaldi.
 *
 * This is the drop-in boundary: plain pointers and sizes, int return codes, no
 * CUDA or torch types. Every entry point names the reference interface it
 * replaces (paths relative to the pocketkaldi tree). All matrices crossing the
 * boundary are frame-major float32: element (frame t, dim d) at [t * dim + d],
 * which is byte-for-byte the reference's column-major pk_matrix_t
 * {nrow = dim, ncol = frames} (src/matrix.h:19-24, src/matrix.cc:136-144).
 *
 * Batches: the reference processes one utterance per call; every batched call
 * here takes `n_utts` utterances packed back to back with a per-utterance
 * length array, and n_utts == 1 reproduces the reference call exactly.
 *
 * There is no CPU fallback. Every function fails with PKB_ERR_CUDA when no
 * sm_100 device is usable.
 *
 * Threading: like the reference's per-utterance objects, a pkb_ctx_t and everything
 * created from it (models, batches, streams) must be used by one host thread at a
 * time; different contexts (also on the same GPU) are independent and may be driven
 * concurrently -- that is how bench.py overlaps the D2H copy of one chunk with the
 * kernels of the next.
 */
#ifndef PKB200_H_
#define PKB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes (0 == success; message via pkb_last_error) ------------- */
#define PKB_OK 0
#define PKB_ERR_INVALID 1     /* bad argument / shape (the reference asserts)       */
#define PKB_ERR_IO 2          /* reference: Status::IOError   (src/status.h:42)     */
#define PKB_ERR_CORRUPT 3     /* reference: Status::Corruption (src/status.h:45)    */
#define PKB_ERR_CUDA 4        /* CUDA runtime / driver failure, or no sm_100 device */
#define PKB_ERR_UNSUPPORTED 5 /* layer stack outside {Linear,ReLU,Normalize,Softmax} patterns */

/* ---- GEMM arithmetic of the nnet (src/gemm.cc, src/gemm_haswell.cc) ------- */
#define PKB_PREC_BF16 0   /* one BF16 tcgen05 MMA per product, FP32 accumulate      */
#define PKB_PREC_BF16X3 1 /* split BF16 (hi+lo), 3 MMAs: FP32-class accuracy; parity mode */
#define PKB_PREC_FP16 2   /* one FP16 MMA per product (11-bit significand, BF16 speed); operands
                             must stay below 65504 in magnitude                              */
#define PKB_PREC_FP16X3 3 /* split FP16 (hi+lo), 3 MMAs: the most accurate mode (error ~2^-22)  */
#define PKB_PREC_FP16C8 4 /* FP16 product + the two first-order correction terms through FP8 (E4M3)
                             operands at twice the MMA rate: 2 MMA-equivalents per product,
                             error ~2^-15. Meets the parity bar; the first layer (whose spliced
                             input view has a 40-byte row pitch in FP8) runs as FP16X3        */
#define PKB_PREC_FP16R 5  /* FP16 with selective refinement (log-likelihood outputs): every frame is
                             computed with one FP16 MMA per product (error ~1e-2 at most), and the
                             frames whose two best pdfs lie within the refinement margin (default
                             0.02, pkb_am_set_refine_margin) -- the only ones whose ranking that
                             error can change: the FP16 error differs by at most 7e-3 between the
                             leading pdfs of a frame on the BASELINE nets, tools/
                             refine_margin_stats.py -- are recomputed with the FP16C8 operands.
                             Other outputs (pkb_nnet_propagate, streams) run as FP16C8        */

/* ---- fixed front-end geometry (src/fbank.h:7-13, src/cmvn.h:10-11) -------- */
#define PKB_FBANK_DIM 40
#define PKB_FRAME_LENGTH 400
#define PKB_FRAME_SHIFT 160
#define PKB_CMVN_STATS_DIM 41

typedef struct pkb_ctx pkb_ctx_t;     /* one per GPU: stream, tables, scratch       */
typedef struct pkb_am pkb_am_t;       /* device-resident AcousticModel              */
typedef struct pkb_batch pkb_batch_t; /* device-resident utterance batch (pipeline) */
typedef struct pkb_stream pkb_stream_t; /* streaming state for one audio stream set */

/* Thread-local message of the last failing call on this thread. */
const char *pkb_last_error(void);

/* Library / build identification: "pkb200 <version> sm_100a". */
const char *pkb_version(void);

/* ---- context --------------------------------------------------------------*/
/* Creates the per-GPU context on CUDA device `device` (replaces the table
 * set-up of Fbank::Fbank, src/fbank.cc:258-265, and pk_srfft_init,
 * src/srfft.cc:343-356). */
int pkb_create(int device, pkb_ctx_t **ctx);
/* Every object created on a context (models, batches, streams, events) must be destroyed
 * before the context itself. */
void pkb_destroy(pkb_ctx_t *ctx);
/* Blocks until all work queued on the context's stream has finished. */
int pkb_sync(pkb_ctx_t *ctx);
/* Number of SMs / device name of the context's GPU. */
int pkb_device_sm_count(pkb_ctx_t *ctx);
const char *pkb_device_name(pkb_ctx_t *ctx);

/* ---- fbank (Fbank::Compute, src/fbank.cc:267-292) ---------------------------*/
/* Fbank::CalcNumFrames, src/fbank.cc:35-42. */
int pkb_fbank_num_frames(int num_samples);

/* wave: all utterances' samples back to back (utterance u starts at
 * sum(num_samples[0..u-1])), float in int16 range, unscaled, exactly what
 * pk_16kpcm_read produces (src/pcm_reader.cc:189-211).
 * feats_out: [sum_u T_u][40] raw log-mel. num_frames_out[u] = T_u (may be NULL). */
int pkb_fbank_f32(pkb_ctx_t *ctx, const float *wave, const int32_t *num_samples,
                  int n_utts, float *feats_out, int32_t *num_frames_out);
/* Same, from 16-bit PCM (skips the float conversion of pcm_reader.cc). */
int pkb_fbank_i16(pkb_ctx_t *ctx, const int16_t *pcm, const int32_t *num_samples,
                  int n_utts, float *feats_out, int32_t *num_frames_out);

/* Front-end options that BASELINE.json's north_star names but the reference does not have
 * (its Fbank is fixed: no dither, Hamming window -- src/fbank.cc:44-100,249-256). Both default to
 * the reference's behaviour and are PARITY UNPINNED: no reference output exists for them; they
 * follow Kaldi's definitions and are covered by property tests only.
 *   window_type  PKB_WINDOW_HAMMING, or PKB_WINDOW_POVEY = pow(0.5 - 0.5 cos(2 pi i / 399), 0.85)
 *   dither       every sample of every frame window gets dither * N(0,1) added before DC removal
 *                (Kaldi's --dither); the noise is a counter-based stream keyed by (dither_seed,
 *                utterance index in the call, frame, sample), so runs are reproducible. 0 = off. */
#define PKB_WINDOW_HAMMING 0
#define PKB_WINDOW_POVEY 1
int pkb_fbank_set_options(pkb_ctx_t *ctx, int window_type, float dither, uint64_t dither_seed);

/* ---- CMVN (CMVN::CMVN + GetFrame for t = 0..T-1, src/cmvn.cc:103-125) -----*/
/* raw / out: [sum_u T_u][40]; global_stats: 40 sums + count
 * (the "cmvn_stats" VEC0 of pk_load, src/pocketkaldi.cc:96-104). The float
 * running sum of ComputeStats (src/cmvn.cc:35-71) is reproduced step by step,
 * so out equals the reference bit for bit on identical raw input. */
int pkb_cmvn(pkb_ctx_t *ctx, const float *raw, const int32_t *num_frames, int n_utts,
             const float *global_stats, float *out);

/* ---- acoustic model (AcousticModel, src/am.h:21-50) -----------------------*/
/* AcousticModel::Read (src/am.cc:23-63): keys nnet, prior, left_context,
 * right_context, num_pdfs, tid2pdf of the model .conf; NNT0/LAY0/MAT0/VEC0
 * readers of src/nnet.cc:80-147, src/matrix.cc:287-319, src/vector.cc:392-425. */
int pkb_am_load(pkb_ctx_t *ctx, const char *conf_path, int precision, pkb_am_t **am);

/* A layer type the reference does not have (its set is {Linear, ReLU, Normalize, Softmax},
 * src/nnet.h:28-33; 4 and 5 are the converter's ADD / MUL): logistic sigmoid, accepted where a
 * ReLU is. BASELINE.json's north_star names it; PARITY UNPINNED (no reference output exists),
 * checked against a float64 evaluation only. The file loader accepts it as LAY0 type 6. */
#define PKB_LAYER_SIGMOID 6

/* Same model from memory. layer_types[i] in {0 linear, 1 relu, 2 normalize,
 * 3 softmax} (src/nnet.h:28-33) or PKB_LAYER_SIGMOID; for linear layer number j (in order)
 * weights[j] is W[out][in] row-major as on disk, biases[j] is b[out],
 * out_dims[j] / in_dims[j] its shape. prior holds probabilities (log is taken
 * here, as src/am.cc:42-43 does). tid2pdf may be NULL. */
int pkb_am_create(pkb_ctx_t *ctx, int n_layers, const int32_t *layer_types,
                  const float *const *weights, const float *const *biases,
                  const int32_t *out_dims, const int32_t *in_dims, const float *prior,
                  int num_pdfs, int left_context, int right_context,
                  const int32_t *tid2pdf, int n_tid2pdf, int precision, pkb_am_t **am);
void pkb_am_destroy(pkb_am_t *am);
int pkb_am_num_pdfs(const pkb_am_t *am);        /* AcousticModel::num_pdfs, src/am.h:38 */
/* PKB_PREC_FP16R: log-likelihood distance between a frame's two best pdfs below which the frame is
 * recomputed with the FP16C8 operands (>= 0; 0 refines exact ties only). */
int pkb_am_set_refine_margin(pkb_am_t *am, float margin);
int pkb_am_input_dim(const pkb_am_t *am);       /* nnet input dim = (L+R+1) * feat dim  */
int pkb_am_left_context(const pkb_am_t *am);
int pkb_am_right_context(const pkb_am_t *am);
/* AcousticModel::TransitionIdToPdfId, src/am.h:30-32. -1 when out of range. */
int pkb_am_tid2pdf(const pkb_am_t *am, int transition_id);
int pkb_am_num_tids(const pkb_am_t *am);

/* AcousticModel::Compute (src/am.cc:90-115) followed by the decodable's scale
 * (pk_decodable_init, src/decodable.cc:8-17; pass prob_scale = 1 for the bare
 * AcousticModel::Compute). feats: [sum_u T_u][feat_dim] CMVN output;
 * loglik_out: [sum_u T_u][num_pdfs] =
 *   prob_scale * (log(max(softmax(z), 1e-20)) - log(prior)). */
int pkb_am_compute(pkb_ctx_t *ctx, pkb_am_t *am, const float *feats,
                   const int32_t *num_frames, int n_utts, int feat_dim, float prob_scale,
                   float *loglik_out);

/* ---- event-gated results (SURVEY 8(f)-1: lazy / chunked decodable) ------------
 * pk_decodable_init (src/decodable.cc:8-17) blocks until the whole [pdfs x frames] matrix is
 * in host memory, although the decoder consumes it strictly frame by frame
 * (Decoder::Decode / ProcessEmitting, src/decoder.cc:49,252-279). An event marks a point of the
 * context's stream; the host can wait for it without waiting for later work. */
typedef struct pkb_event pkb_event_t;
int pkb_event_create(pkb_ctx_t *ctx, pkb_event_t **ev);
void pkb_event_destroy(pkb_event_t *ev);
int pkb_event_record(pkb_ctx_t *ctx, pkb_event_t *ev); /* after everything queued so far      */
int pkb_event_wait(pkb_event_t *ev);                   /* blocks the calling host thread      */
int pkb_event_query(pkb_event_t *ev, int *done);       /* *done = 1 once the point is reached */

/* pkb_am_compute for ONE utterance that returns as soon as the work is queued. The result is
 * copied out in chunks of chunk_frames frames; events[i] is recorded right after the copy of
 * frames [i*chunk_frames, (i+1)*chunk_frames) so that a consumer may read them while later
 * chunks are still in flight. n_events must be >= ceil(num_frames / chunk_frames). loglik_out
 * must stay valid until the last event has completed and should be page-locked
 * (pkb_host_alloc), otherwise each copy blocks the caller and nothing overlaps. */
int pkb_am_compute_chunked(pkb_ctx_t *ctx, pkb_am_t *am, const float *feats, int32_t num_frames,
                           int feat_dim, float prob_scale, float *loglik_out, int chunk_frames,
                           pkb_event_t *const *events, int n_events);

/* Nnet::Propagate (src/nnet.cc:149-163): the layer stack only, no splice, no
 * prior. in: [rows][in_dim]; out: [rows][out_dim of the last layer]. */
int pkb_nnet_propagate(pkb_ctx_t *ctx, pkb_am_t *am, const float *in, int rows, int in_dim,
                       float *out);

/* ---- fused path (the three hot stages of pk_process, src/pocketkaldi.cc:192-216)
 * 16-bit PCM -> fbank -> CMVN -> splice -> nnet -> scaled log-likelihoods.
 * feats_out (optional, may be NULL) receives the CMVN features. */
int pkb_pcm_to_loglik_i16(pkb_ctx_t *ctx, pkb_am_t *am, const int16_t *pcm,
                          const int32_t *num_samples, int n_utts, const float *global_stats,
                          float prob_scale, float *loglik_out, float *feats_out,
                          int32_t *num_frames_out);

/* ---- device-resident batch pipeline ---------------------------------------
 * The throughput path: buffers live in HBM across calls, nothing is allocated
 * or copied inside pkb_batch_run. `am` may be NULL for a front-end-only batch. */
#define PKB_STAGE_FBANK 1
#define PKB_STAGE_CMVN 2
#define PKB_STAGE_NNET 4
#define PKB_STAGE_ALL 7
/* Together with PKB_STAGE_CMVN on a batch that has a model: do not materialise the FP32 copy of
 * the CMVN features (PKB_BUF_FEATS keeps its previous content); the nnet consumes the 16-bit
 * operand planes the CMVN kernel writes anyway. Saves 160 of the 560 bytes the stage moves per
 * frame. */
#define PKB_STAGE_NO_FEATS 8

#define PKB_BUF_PCM 0    /* int16  [sum samples]            */
#define PKB_BUF_RAW 1    /* float  [frames][40] raw fbank   */
#define PKB_BUF_FEATS 2  /* float  [frames][40] after CMVN  */
#define PKB_BUF_LOGLIK 3 /* float  [frames][num_pdfs]       */
/* compact output (pkb_batch_set_compact): IEEE half bits and one float offset per frame;
 * loglik[t][p] = prob_scale * (half(LOGLIK16[t][p]) + LOGLIK_OFF[t])                  */
#define PKB_BUF_LOGLIK16 4   /* uint16 [frames][num_pdfs] */
#define PKB_BUF_LOGLIK_OFF 5 /* float  [frames]           */

int pkb_batch_create(pkb_ctx_t *ctx, pkb_am_t *am, int n_utts, const int32_t *num_samples,
                     const float *global_stats, float prob_scale, pkb_batch_t **batch);
void pkb_batch_destroy(pkb_batch_t *batch);
int64_t pkb_batch_num_frames(const pkb_batch_t *batch);
int64_t pkb_batch_num_samples(const pkb_batch_t *batch);
/* Asynchronous host -> device copy of the packed PCM on the context stream. */
int pkb_batch_set_pcm_i16(pkb_batch_t *batch, const int16_t *pcm);
/* Fills the PCM buffer on the device with the counter-based synthetic stream
 * of pocketkaldi_b200/synth.py: utterance u gets id first_utt_id + u. */
int pkb_batch_synth_pcm(pkb_batch_t *batch, uint64_t seed, uint64_t first_utt_id);
/* Queues the selected stages on the context stream (asynchronous). */
int pkb_batch_run(pkb_batch_t *batch, int stages);
/* Asynchronous device -> host copy of a whole buffer (PKB_BUF_*), or of the
 * rows [frame0, frame0 + n_frames) of a per-frame buffer. */
int pkb_batch_get(pkb_batch_t *batch, int which, void *host_dst);
int pkb_batch_get_rows(pkb_batch_t *batch, int which, int64_t frame0, int64_t n_frames,
                       void *host_dst);
/* SURVEY 8(f)-1, second half: the [frames x pdfs] FP32 matrix (12 KB per frame at 3000 pdfs) is
 * what limits end-to-end throughput over PCIe. With the compact output on, the nnet stage writes
 *   h[t][p]  = fp16( log(max(softmax(z)[p], 1e-20)) - log_prior[p] - off[t] )
 *   off[t]   = max_p(z[p] - log_prior[p]) - logsumexp(z)        (FP32)
 * instead of PKB_BUF_LOGLIK: half the bytes. The frame's best pdf is stored as exactly 0 and a
 * value d below it carries at most d * 2^-11 of rounding error (<= 7.8e-3 up to d = 32), so the
 * per-frame ordering of pdfs -- what the decoder compares -- is preserved. The consumer finishes
 * prob_scale * (float(h) + off) per look-up (pk_decodable_loglikelihood, src/decodable.cc:24-31;
 * pkb_loglik16_expand for a whole block). Needs a model that ends in a softmax.
 * Switching releases the buffer of the other form. */
int pkb_batch_set_compact(pkb_batch_t *batch, int on);
/* PKB_PREC_FP16R: GEMM rows of the latest pkb_batch_run (frames plus the context rows between
 * utterances) and how many frames its second pass recomputed. Zeros for other precisions. */
int pkb_batch_refine_stats(const pkb_batch_t *batch, int64_t *rows, int64_t *refined);
/* Host-side expansion of a block of compact rows: out[t][p] = prob_scale * (half(h[t][p]) + off[t]).
 * Does not touch the GPU. */
int pkb_loglik16_expand(const uint16_t *h, const float *off, int64_t n_frames, int num_pdfs,
                        float prob_scale, float *out);
/* ---- GPU Viterbi (SURVEY 8(f)-4) ----------------------------------------------------------
 * Decoder::Decode + BestPath (src/decoder.cc:39-339) over an Fst (src/fst.cc:29-129) for every
 * utterance of a batch, one thread block per utterance, reading the log-likelihood rows where
 * pkb_batch_run left them in HBM: the [frames x pdfs] matrix never crosses PCIe and no host core
 * walks it. Costs, the beam (16 in the reference) and the best-path rule are the reference's;
 * differences (tightest instead of running cutoff, hard token capacity instead of the sampled
 * max-active estimate, tie-breaking) are listed in pocketkaldi_b200/csrc/decoder.cu. */
typedef struct pkb_fst pkb_fst_t;
/* Fst::Read (src/fst.cc:29-92): "pk::fst_0" file. */
int pkb_fst_load(pkb_ctx_t *ctx, const char *path, pkb_fst_t **fst);
/* Same from memory: final[num_states], first_arc[num_states] (-1: no arcs), and num_arcs arcs of
 * four 32-bit words {next_state, input_label, output_label, weight (float bits)} sorted by
 * source state -- the file's own layout. */
int pkb_fst_create(pkb_ctx_t *ctx, int num_states, int start_state, const float *final_weights,
                   const int32_t *first_arc, int num_arcs, const int32_t *arcs, pkb_fst_t **fst);
void pkb_fst_destroy(pkb_fst_t *fst);
/* Decodes every utterance of the batch from its FP32 log-likelihood buffer (the nnet stage must
 * have run with the compact output off; the model needs its tid2pdf map). beam <= 0 selects the
 * reference's 16. words_out: [n_utts][max_words] output labels in spoken order; n_words_out[u] =
 * number of words of utterance u (it may exceed max_words: the list is then truncated), or a
 * negative code when the search ran out of its per-utterance capacity (max_tokens tokens per
 * frame; 0 selects 4096); weight_out[u] = Hypothesis::weight(). Synchronous. */
int pkb_batch_decode(pkb_batch_t *batch, const pkb_fst_t *fst, float beam, int max_tokens,
                     int max_words, int32_t *words_out, int32_t *n_words_out, float *weight_out);

/* ---- lattices of the batch search -------------------------------------------------------------
 * Every arc the search of pkb_batch_decode relaxed under its beam, kept when the best complete path
 * through it costs at most best + lattice_beam (backward costs in double over the search's arcs).
 * Arcs come sorted by source time; within one time, epsilon arcs before emitting arcs, each group in
 * ascending FST arc index. */
typedef struct {           /* 28 bytes, no padding */
  int32_t t;               /* time of the source node; an emitting arc reads row t and ends at t + 1 */
  int32_t src, dst;        /* FST states of the source / destination nodes */
  int32_t ilabel, olabel;
  float graph_cost;        /* the arc's FST weight */
  float acoustic_cost;     /* -loglik[t][tid2pdf[ilabel]] (scaled rows); 0 for an epsilon arc */
} pkb_lattice_arc_t;
/* Searches every utterance like pkb_batch_decode (same beam / max_tokens defaults) and keeps its
 * lattice pruned to lattice_beam (> 0, may be +inf) on the device. max_arcs: unpruned arcs per
 * utterance, 8 bytes of device log each (<= 0: (frames of the longest utterance + 1) x arcs of the
 * graph, which no utterance can exceed; a word loop keeps nearly all its arcs inside the beam, so a
 * caller short of memory passes less). n_arcs_out[u]: kept arcs, or a
 * negative code (-1 tokens, -2 word records, -3 epsilon closure, -4 more than max_arcs arcs);
 * best_cost_out[u]: min over final nodes of alpha + final (+inf: no final node or a failed search).
 * Synchronous. */
int pkb_batch_lattice(pkb_batch_t *batch, const pkb_fst_t *fst, float beam, float lattice_beam, int max_tokens,
                      int max_arcs, int64_t *n_arcs_out, double *best_cost_out);
/* The arcs of the latest pkb_batch_lattice, every utterance's back to back in utterance order. */
int pkb_batch_lattice_get(pkb_batch_t *batch, pkb_lattice_arc_t *arcs_out);
/* ---- N-best lists over a lattice ----------------------------------------------------------------
 * A path of a lattice runs from (0, start) to (T, s) with final(s) finite, where T is the last
 * emitting record's t + 1 (0 without one); an emitting record goes from (t, src) to (t + 1, dst), an
 * epsilon record from (t, src) to (t, dst). Along a path, its words are the nonzero olabels in path
 * order, its graph cost ((g1 + g2) + ...) + final(s) and its acoustic cost (a1 + a2) + ..., both
 * summed in double in path order from the records' floats; cost = graph + acoustic. A word sequence
 * is represented by its best path: least cost, then least graph cost. The N-best list holds the n
 * first distinct word sequences ordered by cost, then graph cost, then the word sequences compared
 * from the last word backwards (a suffix of the other comes first), then acoustic cost. The list is
 * taken over the lattice's paths: a sequence whose cost is above best + lattice_beam may have had
 * cheaper alignments pruned, so its cost is then only an upper bound on its best cost over the
 * search's arcs. A zero-frame utterance whose start state is final gives one empty sequence of cost
 * final(start).
 * Device memory per call: the outputs, 2 x states x n x 24 bytes of lists per utterance in flight,
 * and a word-history table of 8-byte slots for at least 1.5 x n x (min(labelled emitting records,
 * T x states entered by a labelled emitting arc) + 4 x min(labelled epsilon records, (T + 1) x states
 * entered by a labelled epsilon arc)) histories per utterance in flight; utterances run in waves of
 * at most 8 GiB (or half the free memory) of these.
 * n_hyps_out codes besides those of the lattice: -6 an epsilon closure that did not settle in
 * (records of the group + 1) x (n + 1) passes (only cycles that never settle), -7 more word
 * histories than the table holds (only an epsilon closure of more than 4 passes can need more). */
/* N-best lists of the latest pkb_batch_lattice of this batch (fst: the graph of that call; another
 * one is rejected). 1 <= n <= 1024, max_words > 0. words_out [n_utts][n][max_words] in spoken order,
 * n_words_out / graph_cost_out / acoustic_cost_out [n_utts][n] (n_words may exceed max_words: the
 * list is then truncated, as in pkb_batch_decode); n_hyps_out[u]: entries of utterance u (<= n;
 * 0 when the lattice has no complete path), or that lattice's negative code. Synchronous; the
 * lattice itself is left unchanged. */
int pkb_batch_nbest(pkb_batch_t *batch, const pkb_fst_t *fst, int n, int max_words, int32_t *words_out,
                    int32_t *n_words_out, double *graph_cost_out, double *acoustic_cost_out, int32_t *n_hyps_out);

/* ---- online decoding: the GPU Viterbi search, chunk by chunk ----------------------------------
 * n_streams searches whose tokens and word records stay on the device between calls, so that
 * log-likelihood rows can arrive in any split: decoding a stream's rows 1, 7, 16 or all frames at a
 * time gives bit-identical words and weight to pkb_batch_decode over the same rows. Streams advance
 * together and finish together. */
typedef struct pkb_decoder pkb_decoder_t;
/* n_streams searches over `fst` with `am`'s tid2pdf map (the checks of pkb_batch_decode apply).
 * The decoder keeps pointers to both: the model and the FST must outlive it.
 * beam <= 0: 16; max_tokens <= 0: 4096 tokens per frame (graphs of more than 2048 states or 4096
 * arcs); max_words: words returned per stream; max_records <= 0: 2^18 word records per stream.
 * When an advance leaves the record store more than half full it is compacted to the word histories
 * of the live tokens, so its use grows with the words spoken, not with frames x tokens. A stream
 * whose live history does not fit, or whose tokens overflow, reports a negative word count. */
int pkb_decoder_create(pkb_ctx_t *ctx, const pkb_am_t *am, const pkb_fst_t *fst, int n_streams, float beam,
                       int max_tokens, int max_words, int max_records, pkb_decoder_t **dec);
/* Detaches the decoder from its stream, if any. */
void pkb_decoder_destroy(pkb_decoder_t *dec);
/* Host rows: loglik [n_streams][frame_stride][num_pdfs]; stream s contributes its first n_frames[s]
 * rows (n_frames[s] <= frame_stride). Synchronous. */
int pkb_decoder_advance(pkb_decoder_t *dec, const float *loglik, int frame_stride, const int32_t *n_frames);
/* Best-so-far per stream as of the last advance (or push / flush of the attached stream): the words
 * ([n_streams][max_words], spoken order) of the lowest-cost token of the last frame, ties to the
 * lowest state, without final weights; n_words_out < 0 when the search failed; its cost; frames
 * decoded in this utterance. Any output may be NULL. Reads a host copy: no device work. */
int pkb_decoder_partial(pkb_decoder_t *dec, int32_t *words_out, int32_t *n_words_out, float *cost_out,
                        int64_t *frames_out);
/* BestPath of every stream as pkb_batch_decode returns it, then a fresh utterance (InitDecoding).
 * Synchronous. */
int pkb_decoder_finish(pkb_decoder_t *dec, int32_t *words_out, int32_t *n_words_out, float *weight_out);
/* Lattices of the online search: with lattice_beam > 0 (may be +inf) every pkb_decoder_finish also
 * leaves each stream's lattice on the device, bit-identical to pkb_batch_lattice over the same rows
 * with the same beam, lattice_beam and max_tokens, however the rows were split across advances or
 * pushes; words, weights and partials stay exactly those of a decoder without lattices. Each
 * advance copies its rows into a per-stream store for the backward pass of the finish.
 * max_frames (<= 0: 6000, 60 s): frames per utterance and stream the store keeps; max_arcs: log
 * entries per stream as in pkb_batch_lattice (<= 0: (max_frames + 1) x arcs of the graph; at most
 * INT32_MAX - arcs of the graph, the default capped there). Device
 * memory per stream: 8 max_arcs + 4 max_frames x num_pdfs bytes. lattice_beam = 0 switches lattices
 * off and frees the buffers; negative or NaN is rejected. Only between utterances (after create or
 * pkb_decoder_finish); an attached stream captures its CUDA graphs again. A failed allocation
 * leaves the decoder working without lattices. */
int pkb_decoder_set_lattice(pkb_decoder_t *dec, float lattice_beam, int max_frames, int max_arcs);
/* Per stream, for the latest finish: kept arcs or a negative code (those of pkb_batch_lattice, and
 * -5 more than max_frames frames; a lattice error fails only that stream's lattice) and the best
 * cost. Valid until the next advance, push or flush; rejected after one, or when the latest finish
 * ran without lattices. If the finish could not expand the lattices into records (their device
 * buffer could not be allocated), the finish still succeeds with its words and this call is
 * rejected with the reason. */
int pkb_decoder_lattice(pkb_decoder_t *dec, int64_t *n_arcs_out, double *best_cost_out);
/* The arcs of the latest finish, every stream's back to back in stream order (same validity). */
int pkb_decoder_lattice_get(pkb_decoder_t *dec, pkb_lattice_arc_t *arcs_out);
/* pkb_batch_nbest for the lattices of the latest pkb_decoder_finish; valid when pkb_decoder_lattice is. */
int pkb_decoder_nbest(pkb_decoder_t *dec, int n, int max_words, int32_t *words_out, int32_t *n_words_out,
                      double *graph_cost_out, double *acoustic_cost_out, int32_t *n_hyps_out);

/* Sum over all elements of a per-frame float buffer, computed on the device
 * in double (a cheap whole-output fingerprint for full-size runs). */
int pkb_batch_checksum(pkb_batch_t *batch, int which, double *sum_out);

/* ---- streaming (carried state; no reference equivalent: the reference has no
 * streaming API, SURVEY.md section 5) ---------------------------------------
 * n_streams concurrent streams advance in lock step, chunk_samples new samples
 * per stream per call (a multiple of 160). Concatenated outputs equal the
 * whole-utterance outputs except for the last right_context frames, which are
 * emitted by pkb_stream_flush. */
int pkb_stream_create(pkb_ctx_t *ctx, pkb_am_t *am, int n_streams, int chunk_samples,
                      const float *global_stats, float prob_scale, pkb_stream_t **st);
void pkb_stream_destroy(pkb_stream_t *st);
/* pcm: [n_streams][chunk_samples]; loglik_out: [n_streams][max_frames][num_pdfs]
 * with max_frames = pkb_stream_max_frames(); frames_out = frames produced per
 * stream by this call (identical for every stream). */
int pkb_stream_max_frames(const pkb_stream_t *st);
int pkb_stream_push_i16(pkb_stream_t *st, const int16_t *pcm, float *loglik_out,
                        int32_t *frames_out);
int pkb_stream_flush(pkb_stream_t *st, float *loglik_out, int32_t *frames_out);
/* From the second chunk of an utterance on every push has the same shapes; its launch sequence
 * (tail copy, H2D, fbank, CMVN, nnet stages, D2H) is then captured once into a CUDA graph and
 * replayed, provided the caller passes the same host buffers every time (other buffers are
 * captured again). PKB_STREAM_GRAPH=0 in the environment keeps every push eager.
 * Compact output of a stream (see pkb_batch_set_compact): h16_out [n_streams][max_frames][num_pdfs]
 * half bits and off_out [n_streams][max_frames] offsets instead of the FP32 rows. */
int pkb_stream_set_compact(pkb_stream_t *st, int on);
/* Number of pushes so far that replayed a captured CUDA graph (0 with PKB_STREAM_GRAPH=0). */
int pkb_stream_graph_replays(const pkb_stream_t *st, int64_t *replays);
int pkb_stream_push_compact_i16(pkb_stream_t *st, const int16_t *pcm, uint16_t *h16_out, float *off_out,
                                int32_t *frames_out);
int pkb_stream_flush_compact(pkb_stream_t *st, uint16_t *h16_out, float *off_out, int32_t *frames_out);
/* Attaches a decoder of the same context, model and n_streams (NULL detaches). Every push and flush
 * then advances it over the rows it emitted, on the device and inside the captured CUDA graph of
 * the steady state; loglik_out may then be NULL (decode-only: no row crosses PCIe) and
 * pkb_decoder_partial reads the result. Decoding reads the FP32 rows: a compact stream cannot have a
 * decoder. After pkb_stream_flush, pkb_decoder_finish must be called before the next push.
 * Destroying the stream leaves the decoder usable. */
int pkb_stream_set_decoder(pkb_stream_t *st, pkb_decoder_t *dec);

/* ---- batched ingestion (SURVEY 8(f)-2) --------------------------------------
 * Host-side readers that feed the batch pipeline without the reference's detour through
 * float: pk_16kpcm_read (src/pcm_reader.cc:45-220) parses one strict 44-byte RIFF/WAVE file
 * (PCM, mono, 16 kHz, 8/16/32 bit) into an unscaled float vector, and main.cc:34-46 walks a
 * .scp list one file at a time. Here the same header checks (same messages, PKB_ERR_CORRUPT /
 * PKB_ERR_IO like Status::Corruption / IOError) are applied, 8/16-bit samples go straight to
 * int16 (typically pinned) staging, and a list is read by several host threads.
 * These functions do not touch the GPU and work without one. */
int pkb_wav_probe(const char *path, int32_t *num_samples, int32_t *bits_per_sample);
/* 8- and 16-bit files; a 32-bit file is PKB_ERR_UNSUPPORTED (use the f32 reader). */
int pkb_wav_read_i16(const char *path, int16_t *dst, int32_t capacity, int32_t *num_samples);
/* 8/16/32-bit files, unscaled: element-for-element what pk_16kpcm_read returns. */
int pkb_wav_read_f32(const char *path, float *dst, int32_t capacity, int32_t *num_samples);

/* A list of wave files: one path per line, trailing CR/LF trimmed (pk_readable_readline,
 * src/util.cc:130-160). Every header is validated when the list is opened, so sizes are known
 * before the batch is created. Unlike the reference CLI a last line without a newline is not
 * an error. */
typedef struct pkb_wavlist pkb_wavlist_t;
int pkb_scp_open(const char *scp_path, pkb_wavlist_t **list);
/* Same, from an array of paths. */
int pkb_wavlist_create(const char *const *paths, int n_paths, pkb_wavlist_t **list);
void pkb_wavlist_destroy(pkb_wavlist_t *list);
int pkb_wavlist_size(const pkb_wavlist_t *list);
const char *pkb_wavlist_path(const pkb_wavlist_t *list, int i);
/* [size] samples per file: the num_samples argument of pkb_batch_create. */
const int32_t *pkb_wavlist_num_samples(const pkb_wavlist_t *list);
/* Reads files [first, first + count) back to back into dst (the layout pkb_batch_set_pcm_i16
 * expects) with n_threads host threads (<= 0: one per hardware thread, at most 16). */
int pkb_wavlist_read_i16(const pkb_wavlist_t *list, int first, int count, int16_t *dst,
                         int n_threads);

/* ---- pinned host memory for callers that want overlapped copies ------------*/
int pkb_host_alloc(void **ptr, uint64_t bytes);
void pkb_host_free(void *ptr);

/* ---- measurement -----------------------------------------------------------
 * CUDA events on the context stream (the stream every kernel of this library
 * is launched on). */
int pkb_timer_start(pkb_ctx_t *ctx);
int pkb_timer_stop(pkb_ctx_t *ctx, float *elapsed_ms); /* synchronises */
/* With profiling on, every kernel launch is bracketed by an event pair and
 * accumulated per kernel class. */
#define PKB_KERNEL_FBANK 0
#define PKB_KERNEL_CMVN 1
#define PKB_KERNEL_GEMM 2       /* hidden-layer GEMMs (fused bias/ReLU/normalize epilogue)    */
#define PKB_KERNEL_GEMM_FINAL 3 /* output-layer GEMM (fused log-softmax / prior / scale)      */
#define PKB_KERNEL_MISC 4
#define PKB_KERNEL_CLASSES 5
int pkb_profile_enable(pkb_ctx_t *ctx, int on);
int pkb_profile_reset(pkb_ctx_t *ctx);
/* launches[c] / total_ms[c] for c in PKB_KERNEL_*; launches are counted even
 * with profiling off, times only with it on. */
int pkb_profile_get(pkb_ctx_t *ctx, int64_t *launches, double *total_ms);
/* Flushes L2 by writing a scratch buffer larger than the cache. */
int pkb_flush_l2(pkb_ctx_t *ctx);

#ifdef __cplusplus
}
#endif
#endif /* PKB200_H_ */
