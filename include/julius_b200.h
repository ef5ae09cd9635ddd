/* julius_b200.h -- C-ABI of libjb200.so: B200-native acoustic scoring + pass-1 beam for Julius.
 *
 * Plain C: pointers, sizes, opaque handles.  No torch / CUDA types.  Every
 * entry point names the reference interface it stands in for (file:line in
 * julius-speech/julius 4.6); INTEGRATION.md shows the reference-side binding.
 *
 * Conventions
 *   - all functions return 0 on success or a negative error code; the message
 *     is available from jb200_last_error() (thread-local).
 *   - "host" variants take ordinary host pointers and include the H2D/D2H copies;
 *     "device" variants take device pointers on the handle's device and enqueue
 *     on the given CUDA stream (a cudaStream_t passed as void*; NULL = the
 *     handle's own stream).
 *   - scores are log10 likelihoods, exactly the values the reference keeps in
 *     HMMWork.outprob_cache[t][state-id] (libsent/include/sent/hmm_calc.h:115).
 *   - there is NO CPU fallback: creating a handle without a usable sm_100 GPU fails.
 */
#ifndef JULIUS_B200_H
#define JULIUS_B200_H

#include <stdint.h>
#include "jb200_model.h"

#ifdef __cplusplus
extern "C" {
#endif

#define JB200_OK              0
#define JB200_ERR_ARG        -1
#define JB200_ERR_CUDA       -2
#define JB200_ERR_NODEVICE   -3
#define JB200_ERR_UNSUPPORTED -4
#define JB200_ERR_CAPACITY   -5

/* arithmetic mode of the GMM scorer */
#define JB200_GMM_EXACT 0   /* reference's fp32 statement order + addlog table: bit-identical scores */
#define JB200_GMM_FAST  1   /* FMA + exact log-sum-exp: <=1e-4 relative (BASELINE.json tolerance)  */

int jb200_version(void);
const char *jb200_last_error(void);
int jb200_device_count(void);
/* number of kernels launched by this library since load (bench.py "gpu_launches") */
int64_t jb200_launch_count(void);

/* ------------------------------------------------------------------------------------
 * GMM state scorer.   Stands in for, per frame and for ALL states at once,
 *   outprob_state()  libsent/src/phmm/outprob.c:183-249   (batch_computation branch :230-240)
 *   calc_mix()       libsent/src/phmm/calc_mix.c:40-81
 *   gprune_none/safe/beam/heu (compute_gaussset)  libsent/src/phmm/gprune_*.c
 *   addlog_array()   libsent/src/phmm/addlog.c:102-123
 *   outprob_cd()     libsent/src/phmm/outprob.c:286-400   (pseudo-phone sets)
 * ---------------------------------------------------------------------------------- */
typedef struct jb200_gmm jb200_gmm;

/* The descriptor is checked before anything is uploaded: with n_gauss > 0, state_off must be non-decreasing
 * from 0 to n_gauss (a state has at most 64 mixture slots), cd_off must be non-decreasing from 0 to n_cdset_states
 * and every cd_states entry a state id; otherwise JB200_ERR_ARG (JB200_ERR_UNSUPPORTED for dim, -tmix, -iwcd1 best
 * or a mixture count the kernels are not built for).  A state with no mixture slots (state_off[s] == state_off[s+1])
 * scores LOG_ZERO, as outprob_state does for an empty mixture list.  n_gauss == 0 describes the state / cd-set layout
 * of a DNN-HMM only: state_off may then be NULL and the state columns cannot be scored. */
int jb200_gmm_create(const jb200_gmm_desc *desc, int device, int mode, jb200_gmm **out);
void jb200_gmm_destroy(jb200_gmm *h);
/* row stride (floats) of the score matrix: n_states + n_cdsets rounded up to 4 */
int jb200_gmm_score_stride(const jb200_gmm *h);
int jb200_gmm_n_states(const jb200_gmm *h);
int jb200_gmm_n_cdsets(const jb200_gmm *h);

/* feats [T][dim] (host) -> scores [T][n_states] (host), log10. */
int jb200_gmm_score_host(jb200_gmm *h, const float *feats, int T, float *scores);
/* feats [T][dim] (host) -> full rows [T][stride] (host): states then cd-set scores */
int jb200_gmm_score_rows_host(jb200_gmm *h, const float *feats, int T, float *rows);
/* device: d_feats [T][dim] -> d_rows [T][stride]; state columns and cd-set columns are both filled */
int jb200_gmm_score_device(jb200_gmm *h, const float *d_feats, int T, float *d_rows, void *stream);
/* device: fill only the cd-set columns of rows whose state columns are already present */
int jb200_gmm_cdsets_device(jb200_gmm *h, float *d_rows, int T, void *stream);
/* per-Gaussian ln scores of ONE frame, without mixture weights (the calcmix hook's
 * contract, plugin/calcmix.c:226-323): feat [dim] (host) -> gauss [n_gauss] (host) */
int jb200_gmm_gauss_host(jb200_gmm *h, const float *feat, float *gauss);

/* ------------------------------------------------------------------------------------
 * DNN-HMM state scorer (tensor cores).  Stands in for, for all frames of a batch at once,
 *   dnn_calc_outprob()   libsent/src/phmm/calc_dnn.c:774-868   (GEMV stack, table logistic,
 *                        log-softmax through addlog_array, minus log10 state prior)
 *   cuda_calc_outprob()  libsent/src/phmm/calc_dnn_cuda.cu:294-321 (the reference's own GPU path)
 * in [T][in_dim] already spliced feature vectors -> scores [T][out_dim], log10.
 * Arithmetic: bf16 x3 split products with fp32 accumulation (<= 1e-4 relative, see DESIGN.md).
 * ---------------------------------------------------------------------------------- */
typedef struct jb200_dnn jb200_dnn;
int jb200_dnn_create(const jb200_dnn_desc *desc, int device, jb200_dnn **out);
void jb200_dnn_destroy(jb200_dnn *h);
int jb200_dnn_in_dim(const jb200_dnn *h);
int jb200_dnn_out_dim(const jb200_dnn *h);
int jb200_dnn_score_host(jb200_dnn *h, const float *in, int T, float *scores);

/* ------------------------------------------------------------------------------------
 * Pass-1 decoder (lexicon-tree token passing).  Stands in for
 *   get_back_trellis_init/_proceed/_end, finalize_1st_pass   libjulius/src/beam.c:1825,2663,3052,3133
 *   outprob_style()                                         libjulius/src/outprob_style.c:354-494
 *   max_successor_prob(_iw)()                               libjulius/src/factoring_sub.c:942-1143
 *   bt_store/bt_relocate_rw/bt_sort_rw                      libjulius/src/backtrellis.c:190-267,438-478
 * run for a whole BATCH of utterances, one thread-block per utterance; a launch covers all frames of the
 * utterances, or one time slice of them (batch pipeline, streams: see the end of this header) -- the kernels are
 * resumable, an utterance's state lives in its device work area between launches.
 * ---------------------------------------------------------------------------------- */
typedef struct jb200_decoder jb200_decoder;

/* one word-trellis atom (libjulius/include/julius/trellis.h:28-45) */
typedef struct {
  int32_t wid;
  int32_t begintime;
  int32_t endtime;
  float backscore;
  float lscore;
  int32_t last;        /* index of last_tre within the same utterance's atom list, -1 = sentence start */
} jb200_atom;

typedef struct {
  int32_t status;      /* 0 = success, -1 = search failed (J_RESULT_STATUS_FAIL) */
  int32_t n_frames;
  int32_t n_atoms;
  int32_t n_words;     /* pass-1 best sequence length */
  float score;         /* pass1_score */
  int64_t atom_offset; /* first atom of this utterance in the batch atom array */
  int32_t word_offset; /* first word in the batch word array */
  int32_t overflow;    /* non-zero if a device-side capacity was exceeded (result invalid) */
} jb200_utt_result;

/* am: GMM scorer (owns device + cd-set layout).  max_utts / max_frames size the work areas. */
int jb200_decoder_create(const jb200_tree_desc *tree, jb200_gmm *am, int max_utts, int max_frames,
                         jb200_decoder **out);
void jb200_decoder_destroy(jb200_decoder *d);
/* DNN-HMM: score frames with `dnn` instead of the GMMs of `am` (am then only carries the state /
 * cd-set layout: a descriptor with n_gauss == 0 is accepted by jb200_gmm_create for this purpose). */
int jb200_decoder_attach_dnn(jb200_decoder *d, jb200_dnn *dnn);

/* End-to-end: host feature vectors -> GPU scoring -> GPU beam -> host results.
 *   feats       [sum T_u][dim]   concatenated utterances (host)
 *   frame_off   [n_utts+1]       utterance boundaries in frames
 * Results stay owned by the decoder until the next call; read them with jb200_decoder_results(). */
int jb200_decode_batch_host(jb200_decoder *d, const float *feats, const int32_t *frame_off, int n_utts);
/* Same, but the state-score matrix is given ([sum T_u][n_states], host, log10): used to
 * check the beam in isolation on the reference's own score matrix. */
int jb200_decode_batch_scores_host(jb200_decoder *d, const float *scores, const int32_t *frame_off, int n_utts);
/* Device-resident input (bench "value"): d_feats on the decoder's device. */
int jb200_decode_batch_device(jb200_decoder *d, const float *d_feats, const int32_t *frame_off, int n_utts);
/* copy results of the last batch device->host (called implicitly by the *_host variants) */
int jb200_decoder_fetch(jb200_decoder *d);
int jb200_decoder_results(jb200_decoder *d, const jb200_utt_result **utts, const jb200_atom **atoms,
                          const int32_t **words);
/* timing of the last batch in milliseconds (CUDA events on the decoder's stream):
 * [0]=H2D, [1]=acoustic scoring, [2]=beam, [3]=D2H */
int jb200_decoder_last_timing(jb200_decoder *d, float ms[4]);
/* wait for the last batch's kernels and refresh the timing (device variant, no D2H) */
int jb200_decoder_sync_timing(jb200_decoder *d);
/* bytes moved device->host by the last fetch (results + atoms + words) */
int64_t jb200_decoder_last_d2h_bytes(const jb200_decoder *d);
/* how often (frames, since create) the beam cut had to fall back to the plain sequential replay (0 unless forced) */
int64_t jb200_decoder_misspeculations(jb200_decoder *d);
/* beam-cut replay counters since create: out[0] fall-backs to the plain sequential loop, out[1] replay ticks (tree
 * levels with the single-thread replay), out[2] extractions replayed */
int jb200_decoder_heap_stats(jb200_decoder *d, int64_t out[3]);
/* beam cuts that select the top of the token set (sort_token_upward) since create: out[0] how many,
 * out[1] how many of them were answered by the closed form (score, pre-order position) instead of a replay */
int jb200_decoder_select_stats(jb200_decoder *d, int64_t out[2]);
/* of the closed-form answers, how many needed the exact treatment of re-inserted elements (closed form with relocations) */
int64_t jb200_decoder_relocated_selects(jb200_decoder *d);
/* how many utterances (thread blocks) are co-resident on the device for this decoder */
int jb200_decoder_resident_utts(const jb200_decoder *d);
/* SM-cycle totals per kernel phase of the first n_utts utterances of the last batch: cycles [n_utts][8]
 * 0 clear, 1 count/atoms, 2 expand, 3 creators, 4 order sort, 5 materialise+outprob, 6 heap select, 7 rest */
int jb200_decoder_phase_cycles(jb200_decoder *d, int64_t *cycles, int n_utts);
/* per-frame token counts of utterance u of the last batch (debug / roofline accounting):
 * counts [T][2] = (tokens created, survivors) */
int jb200_decoder_frame_counts(jb200_decoder *d, int u, int32_t *counts, int max_frames);

/* ------------------------------------------------------------------------------------
 * Batch pipeline.  With frames_per_slice > 0 a GMM batch is cut into time slices: the scoring of slice c+1 runs on its
 * own CUDA stream beside the token passing of slice c (the FP32-bound scoring kernel and the latency-bound beam kernel
 * share the SMs), provided the batch leaves room for a scoring thread block on every SM (n_utts <= 3/4 of
 * jb200_decoder_resident_utts()).  Results are bit-identical to the unsliced batch.  0 (default, or JB200_PIPE_FRAMES
 * in the environment) = one launch per batch.  jb200_decoder_last_timing() then reports [1] = the scoring the beam had
 * to wait for (slice 0) and [2] = everything after; pipeline_info gives the slice count and how long the scoring stream
 * was busy (overlapped).
 * ---------------------------------------------------------------------------------- */
int jb200_decoder_set_pipeline(jb200_decoder *d, int frames_per_slice);
int jb200_decoder_pipeline_info(jb200_decoder *d, int32_t *n_slices, float *score_busy_ms);

/* ------------------------------------------------------------------------------------
 * Frame-synchronous operation ("streams").  The reference drives pass 1 one frame at a time,
 *   get_back_trellis_init -> get_back_trellis_proceed(t) ... -> get_back_trellis_end -> finalize_1st_pass
 *   (decode_proceed, libjulius/src/pass1.c:112-254; real-time input realtime-1stpass.c:681-, interim result
 *   bt_current_max, beam.c:876-921 / :2983-2993),
 * because with live input the utterance's length is not known in advance.  A stream is that call sequence: n_streams
 * (<= max_utts) independent utterances advance together, each feed hands every stream its next n_new[s] >= 0 frames
 * (feature vectors packed stream-major) and decodes them on the device; last[s] != 0 marks the end of stream s's
 * utterance (its final frames, possibly none, come with the same call), after which jb200_stream_result() returns what
 * jb200_decoder_results() returns for a batch.  Frame for frame the trellis is identical to the batch decode of the
 * same vectors, whatever the feed sizes.  Per-stream capacity: max_frames / n_streams frames.
 * ---------------------------------------------------------------------------------- */
int jb200_stream_open(jb200_decoder *d, int n_streams);          /* all streams at the start of an utterance */
int jb200_stream_restart(jb200_decoder *d, int stream);          /* one stream starts its next utterance */
int jb200_stream_feed_host(jb200_decoder *d, const float *feats, const int32_t *n_new, const uint8_t *last, int want_interim);
/* the same on a given state-score matrix ([sum n_new][n_states], host, log10) instead of feature vectors */
int jb200_stream_feed_scores_host(jb200_decoder *d, const float *scores, const int32_t *n_new, const uint8_t *last, int want_interim);
/* frames decoded so far; alive = 0 once the beam ran empty (get_back_trellis_proceed's FALSE, beam.c:3012-3015) */
int jb200_stream_status(jb200_decoder *d, int stream, int32_t *frames_done, int32_t *alive, int32_t *ended);
/* interim result of the last feed that asked for one (want_interim): the best word sequence ending at the last decoded
 * frame, as bt_current_max publishes it in r->result.pass1 (word_num 0 = no word has ended there) */
int jb200_stream_partial(jb200_decoder *d, int stream, int32_t *words, int max_words, int32_t *n_words, float *score, int32_t *frame);
int jb200_stream_result(jb200_decoder *d, int stream, const jb200_utt_result **utt, const jb200_atom **atoms, const int32_t **words);

#ifdef __cplusplus
}
#endif
#endif /* JULIUS_B200_H */
