/*
 * fpnmt.h — C ABI of libfpnmt.so, the B200 (sm_100a) caption-inference engine.
 *
 * The reference (samkoesnadi/fpn-MT-image-captioning) is pure Python/TensorFlow and has no FFI; the
 * boundary this library sits behind is the reference's Python builder API.  Each entry point names the
 * reference interface it replaces (paths relative to the reference repo).  The host-side Python mirror
 * (fpn-mt-image-captioning_b200/fpnmt) binds these symbols with ctypes; see INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes only (no C++/torch types); every function returns 0 on success or
 * an FPNMT_ERR_* code and leaves a message retrievable with fpnmt_last_error(); device pointers are raw
 * CUDA device addresses (e.g. torch.Tensor.data_ptr() or a DLPack capsule's data field) on the engine's
 * device; all work is enqueued on the caller's stream (cudaStream_t passed as void*; NULL = default stream);
 * one handle per GPU; calls on one handle must be serialised by the caller.  There is no CPU fallback.
 */
#ifndef FPNMT_H_
#define FPNMT_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define FPNMT_API __attribute__((visibility("default")))
#else
#define FPNMT_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

enum {
  FPNMT_OK = 0,
  FPNMT_ERR_INVALID = 1,     /* bad argument / shape / configuration            */
  FPNMT_ERR_STATE = 2,       /* call order (e.g. encode before finalize)        */
  FPNMT_ERR_CUDA = 3,        /* CUDA runtime / driver error                     */
  FPNMT_ERR_MISSING = 4      /* a required weight was never set                 */
};

enum { FPNMT_BACKBONE_MOBILENETV2 = 0, FPNMT_BACKBONE_RESNET50 = 1, FPNMT_BACKBONE_DENSENET121 = 2 };
enum { FPNMT_PREC_BF16 = 0,      /* bf16 operands, fp32 accumulate, bf16 activations                          */
       FPNMT_PREC_BF16X3 = 1 };  /* 3-term split-bf16 products (~fp32 operand precision), fp32 accumulate:
                                    the parity mode; same kernels, 3x the tensor work                        */
enum { FPNMT_SCORE_LOG = 0,      /* beam score = sum of log-probs                                             */
       FPNMT_SCORE_PROB = 1 };   /* beam score = product of softmax probabilities (reference, pipeline.py:117-123) */
/* fpnmt_config.kernel_opts: each bit switches ONE fused kernel back to its unfused equivalent (A/B timing and the
 * fused-vs-unfused parity tests).  0 = every fused path on (the product configuration). */
enum { FPNMT_OPT_NO_XATTN = 1,       /* separate q2 / cross-attention / o2+LN kernels instead of xattn_kernel          */
       FPNMT_OPT_NO_STEM = 2,        /* explicit im2col + GEMM stem instead of stem_kernel                              */
       FPNMT_OPT_NO_TGEMM = 4,       /* decoder Dense layers through igemm + separate LayerNorm                         */
       FPNMT_OPT_ENC_ATT_SIMT = 8,   /* CUDA-core encoder attention instead of the tensor-core flash kernel             */
       FPNMT_OPT_NO_PDL = 32,        /* no programmatic dependent launch (process-wide: the last created engine wins)    */
       FPNMT_OPT_DEC_ATT_SIMT = 256, /* CUDA-core decode self-attention in bf16 mode (instead of the mma.sync kernel)          */
       FPNMT_OPT_TGEMM_WIDE = 512,   /* bf16 Dense layers on tgemmw_kernel (128 rows per CTA, two CTAs per SM, TMA-store
                                        epilogue: least SM time, best when several lanes share the GPU) even with lanes < 2.
                                        Default: tgemmw_kernel when fpnmt_config.lanes >= 2, else tgemm_kernel (lowest
                                        latency of a single chain)                                                         */
       FPNMT_OPT_NO_TGEMM_WIDE = 1024, /* never tgemmw_kernel                                                             */
       FPNMT_OPT_NO_DENSE_1X1 = 8192, /* 1x1 convolutions in the 2-D pixel-tile geometry of the other convolutions (default: as a
                                        GEMM over 128 consecutive pixels per tile)                                          */
       FPNMT_OPT_NO_B_STATIONARY = 32768, /* igemm_kernel streams the weight chunks with every tile (default: a panel <= 96 KB of a
                                        single output-channel tile stays in shared memory for all tiles of the CTA)            */
       FPNMT_OPT_NO_TMA_STORE = 16384, /* igemm_kernel writes its bf16 outputs with 16-byte LSU stores instead of bulk tensor stores */
       FPNMT_OPT_NO_VSTATS = 4096,   /* keep the [rows][V] fp32 logits between the vocabulary projection and k_beam_step (default with
                                        the wide Dense kernels, log scores and beam <= 8: per-tile softmax partials + 8 candidates)  */
       FPNMT_OPT_NO_KV_SHARE = 2048, /* ancestry cache mode: every beam reads its own lineage's cache rows even when another
                                        beam of the image has the same token history (default: read the first such beam's rows;
                                        identical bits, 8x less cache traffic under the reference's beam initialisation)    */
       FPNMT_OPT_DSTEP_TAPS = 128    /* fused decoder: also keep every layer's LayerNorm outputs (fpnmt_get_tap "decL_outK") */ };
enum { FPNMT_CACHE_ANCESTRY = 0,     /* KV cache never moves; an ancestry table maps (beam, position) -> physical row    */
       FPNMT_CACHE_PHYSICAL = 1 };   /* KV cache rows are gathered by beam parent after every step (bandwidth kernel)    */
enum { FPNMT_DECODE_AUTO = 0,        /* the faster path for the configuration: today the per-operator chain                */
       FPNMT_DECODE_CHAIN = 1,       /* per-operator kernel chain (tgemm / attention / xattn / beam kernels), 38 per step   */
       FPNMT_DECODE_FUSED = 2 };     /* group-stationary fused decoder (dstep_kernel): ONE launch runs every layer, the
                                        vocabulary projection and the beam tail of all steps (bf16, log scores, beam <= 16) */

typedef struct fpnmt_config {
  int32_t backbone;      /* FPNMT_BACKBONE_* — models/mobilenet.py:43, models/resnet.py:78, models/densenet.py:73 */
  int32_t image_size;    /* IMAGE_INPUT_SIZE, common/common_definitions.py:18 (multiple of 256)                  */
  int32_t batch;         /* images per call (the reference predicts one image at a time, pipeline.py:93)         */
  int32_t beam;          /* BEAM_SEARCH_N, common/common_definitions.py:22                                       */
  int32_t vocab;         /* target_vocab_size, utils/pipeline.py:19                                              */
  int32_t max_len;       /* max_seq_len, utils/pipeline.py:12 / test.py:13                                       */
  int32_t num_layers;    /* common/common_definitions.py:56                                                      */
  int32_t d_model;       /* :57 (must be 512)                                                                    */
  int32_t num_heads;     /* :59 (must be 8)                                                                      */
  int32_t dff;           /* :58                                                                                  */
  int32_t precision;     /* FPNMT_PREC_*                                                                         */
  int32_t score_mode;    /* FPNMT_SCORE_*                                                                        */
  int32_t start_id;      /* tokenizer.word_index['<start>'], pipeline.py:89                                      */
  int32_t end_id;        /* tokenizer.word_index['<end>'],   pipeline.py:90                                      */
  int32_t true_beam;     /* 0 = reference init (all beams identical, pipeline.py:101-102); 1 = only beam 0 alive  */
  int32_t use_graphs;    /* 1 = replay the encode / decode-step programs as CUDA graphs                          */
  /* ---- the eight words below were `reserved[8]` in ABI 0.1; all-zero selects the defaults ---- */
  int32_t kernel_opts;   /* FPNMT_OPT_* bit mask; a bit not defined above is refused (FPNMT_ERR_INVALID)          */
  int32_t cache_mode;    /* FPNMT_CACHE_*                                                                         */
  int32_t decode_path;   /* FPNMT_DECODE_*                                                                        */
  float length_penalty;  /* EXTENSION (not in the reference): alpha of the length normalisation applied when a beam
                            finishes, score / ((5 + len) / 6)^alpha; 0 = reference ordering                        */
  int32_t finished_beams;/* EXTENSION: 1 = a beam that emitted <end> is frozen and competes with its final score;
                            the image stops when its best beam is a finished one.  0 = reference (pipeline.py:143-148:
                            stop the moment the top beam emits <end>, finished lower beams keep decoding)          */
  int32_t dec_groups;    /* unused, must be 0 or 1 (the batch is decoded as one chain); kept so the layout does not change */
  int32_t lanes;         /* batches in flight (fpnmt_submit / fpnmt_collect): the handle holds this many complete engines
                            (own activations, KV cache, beam state, streams; ONE shared copy of the GEMM weights) on the one GPU, 0/1 = one,
                            at most 16.  Two lanes overlap
                            the throughput-bound encoder of batch i+1 with the latency-bound decode of batch i.            */
  int32_t reserved[1];   /* must be 0                                                                               */
} fpnmt_config;

typedef struct fpnmt_handle fpnmt_handle;

/* Library / build information ("sm_100a", kernel list).  Never fails. */
FPNMT_API const char* fpnmt_version(void);
/* Thread-local message of the last failing call. */
FPNMT_API const char* fpnmt_last_error(void);

/* Replaces: Transformer(...) / Encoder(...) / FeatureExtractor(...) construction
 * (models/transformer.py:344-357, :246-264; models/retinanet.py:266-304). */
FPNMT_API int fpnmt_create(const fpnmt_config* cfg, int device, fpnmt_handle** out);
FPNMT_API int fpnmt_destroy(fpnmt_handle* h);

/* Replaces: checkpoint restore / load_weights (utils/pipeline.py:38-48, models/retinanet.py:277-278).
 * `key` is the variable path of SURVEY.md Appendix B (e.g. "transformer/decoder/dec_layers/0/mha1/wq/kernel");
 * `data` is HOST float32 in Keras layout (Dense (in,out); Conv2D (kh,kw,Cin,Cout); Depthwise (kh,kw,C,1));
 * the library copies it. */
FPNMT_API int fpnmt_set_weight(fpnmt_handle* h, const char* key, const float* data, const int64_t* shape, int ndim);
/* Folds BatchNorm, concatenates projections, converts to bf16 (split into hi/lo for BF16X3), uploads, builds
 * the kernel programs and tensor maps. */
FPNMT_API int fpnmt_finalize_weights(fpnmt_handle* h);

/* Replaces: Encoder.call(x, training=False, mask=None) (models/transformer.py:266-303).
 * images: float32 NHWC [batch, S, S, 3] in [-1,1] (dataset.py:19-26), DEVICE pointer unless images_on_host != 0
 * (then a pinned/pageable HOST pointer; the H2D copy is enqueued on `stream`).
 * memory_out: optional DEVICE float32 [batch, 16*(S/512)^2.., d_model] = encoder output; may be NULL. */
FPNMT_API int fpnmt_encode(fpnmt_handle* h, const float* images, int images_on_host, float* memory_out, void* stream);

/* Replaces: FeatureExtractor.call(inp) (models/retinanet.py:306-307).  Runs the CNN part only and copies the five
 * head outputs (P3..P7 order, NHWC float32, DEVICE pointers, sizes batch*(S/16>>i)^2*d_model) out. */
FPNMT_API int fpnmt_features(fpnmt_handle* h, const float* images, int images_on_host, float* const out5[5], void* stream);

/* Copies a named intermediate of the last fpnmt_encode (e.g. "C3","C4","C5","P3".."P7","tokens0".."tokens4",
 * "enc_layer0"..) to a DEVICE float32 buffer of `capacity` floats; writes its element count to *count. */
FPNMT_API int fpnmt_get_tap(fpnmt_handle* h, const char* name, float* out, size_t capacity, size_t* count, void* stream);

/* Replaces: Transformer.call(inp=enc_output, tar, training=False, look_ahead_mask) (models/transformer.py:359-374)
 * for teacher-forced parity: memory DEVICE float32 [batch,16,d_model] (NULL = reuse the last fpnmt_encode result),
 * tokens DEVICE int32 [batch, t]; logits_out DEVICE float32 [batch, t, vocab].  Computed with the KV-cached
 * step program (position by position), which is mathematically the causal-masked full forward. */
FPNMT_API int fpnmt_decode_logits(fpnmt_handle* h, const float* memory, const int32_t* tokens, int t, float* logits_out,
                        void* stream);

/* Replaces: Decoder.call(x, enc_output, training=False, look_ahead_mask, padding_mask) (models/transformer.py:321-341): the
 * output of the last decoder layer (before final_layer) for teacher-forced tokens; arguments as fpnmt_decode_logits,
 * hidden_out DEVICE float32 [batch, t, d_model].  The attention-weights dict comes from fpnmt_decode_attention. */
FPNMT_API int fpnmt_decode_hidden(fpnmt_handle* h, const float* memory, const int32_t* tokens, int t, float* hidden_out,
                                  void* stream);

/* The attention-weights dict of Decoder.call (models/transformer.py:337-338) for teacher-forced tokens; memory / tokens /
 * t as fpnmt_decode_logits (NULL memory = the last encode).  self_out DEVICE float32 [num_layers][batch][heads][t][t]:
 * "decoder_layer{l+1}_block1", causal softmax(q k^T / 8) with exact zeros above the diagonal; cross_out DEVICE float32
 * [num_layers][batch][heads][t][n_memory]: "decoder_layer{l+1}_block2", the softmax over the memory tokens (token j = P6
 * cell (j / w6, j % w6)).  Either output may be NULL, not both.  The probabilities are computed by extra kernels in the
 * teacher-forced step program; not available with decode_path = FUSED (FPNMT_ERR_STATE). */
FPNMT_API int fpnmt_decode_attention(fpnmt_handle* h, const float* memory, const int32_t* tokens, int t, float* self_out,
                                     float* cross_out, void* stream);

/* Replaces: the body of the decode loop, utils/pipeline.py:115-141, on caller-provided logits (the decode-tail
 * kernels alone): logits DEVICE float32 [batch*beam, vocab], scores_in DEVICE float32 [batch*beam];
 * outputs DEVICE int32 parent[batch*beam], token[batch*beam], float32 scores_out[batch*beam]. */
FPNMT_API int fpnmt_beam_step(fpnmt_handle* h, const float* logits, const float* scores_in, int32_t* parent, int32_t* token,
                    float* scores_out, void* stream);
/* fpnmt_beam_step through the logits-free decode tail: the same step with the vocabulary projection's per-tile softmax
 * partials and candidates in place of the logits (what fpnmt_op_vocab_stats writes; the beam-search decode of the bf16 mode
 * with the wide Dense kernels runs this kernel branch).  stat DEVICE float32 [batch*beam][tiles][2] = (max, sum exp(x - max))
 * of the tile's valid tokens; val DEVICE float32 [batch*beam][tiles][8] the tile's 8 largest logits, descending, ties lower
 * id first, -inf padded; idx DEVICE int32 [batch*beam][tiles][8] their token ids in [0, vocab), 0x7fffffff where padded.
 * stat and val 16-byte aligned.  FPNMT_ERR_INVALID (nothing launched) for score_mode PROB, beam > 8 or tiles outside
 * 1..192. */
FPNMT_API int fpnmt_beam_step_vstats(fpnmt_handle* h, const float* stat, const float* val, const int32_t* idx, int tiles,
                                     const float* scores_in, int32_t* parent, int32_t* token, float* scores_out, void* stream);

/* Sampling parameters of fpnmt_sample / fpnmt_op_sample_step.  Row (image b, sample n) at step t, logits z (fp32, the
 * vocabulary projection):
 *   1. p = softmax(z / temperature) over all V tokens.
 *   2. top-k: K1 = {i : z_i >= z_(k)}, z_(k) the k-th largest logit; every token tied with it is kept (|K1| may exceed k).
 *   3. top-p: p renormalised over K1; K2 = {i in K1 : p_i >= tau}, tau the largest value for which the tokens of K1 with
 *      p_j >= tau hold at least top_p of K1's mass.  Ties at tau are kept; K2 always holds the arg-max.
 *   4. u = (philox4x32_10(counter = (t, b, n, 0), key = (seed & 0xffffffff, seed >> 32))[0] >> 8) * 2^-24.
 *   5. token = the smallest id i in K2 with sum_{j in K2, j <= i} p_j > u * sum_{K2} p.
 *   6. log-probability of a sample = sum over its emitted steps, <end> included, of log_softmax(z)[token] at temperature 1
 *      with no filtering: the caption's log-likelihood under the model.
 * temperature 0 is greedy: the arg-max, lowest token id on ties (identical for every n; on an engine with the reference beam
 * initialisation that is the caption fpnmt_generate returns).  Vocabulary entries with logit -1e9 get p = 0 and are never
 * drawn. */
typedef struct fpnmt_sampling {
  float temperature;     /* >= 0; 0 = greedy (arg-max, lowest token id on ties)        */
  int32_t top_k;         /* 0 = off; else keep tokens whose logit >= the k-th largest  */
  float top_p;           /* (0, 1]; 1 = off                                            */
  uint64_t seed;
  int32_t reserved[4];   /* must be 0 */
} fpnmt_sampling;

/* N = beam independent sampled captions per image (see fpnmt_sampling): encoder (images != NULL; NULL = the memory of the
 * last fpnmt_encode / fpnmt_generate) + a decode in which row (b, n) is sample n of image b.  A sample stops at its first
 * <end>; its row keeps being computed but its tokens are ignored; an image is done when all N of its samples are.
 * out_ids DEVICE-or-HOST int32 [batch][beam][max_len] (0 padded, no <start>, no <end>), out_len int32 [batch][beam]
 * (max_len when <end> never fired), out_logprob float32 [batch][beam] or NULL (same side as the others).
 * outputs_on_host != 0: host outputs, the call synchronises the stream.  early_stop != 0: stop once every sample has
 * emitted <end> (the result is the same either way).  Errors: FPNMT_ERR_INVALID for temperature < 0, top_p outside (0, 1],
 * top_k outside [0, vocab] or non-zero reserved words; FPNMT_ERR_STATE with decode_path = FUSED or while lane 0 holds a
 * submitted batch.  Results are bit-identical run to run, with graphs on or off, early stop on or off and in both cache
 * modes; the call leaves nothing behind that changes a later fpnmt_generate. */
FPNMT_API int fpnmt_sample(fpnmt_handle* h, const float* images, int images_on_host, const fpnmt_sampling* sampling,
                           int32_t* out_ids, int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop,
                           void* stream);

/* Caption scoring: the log-likelihood of N = beam given captions per image, all positions in one teacher-forced decoder pass
 * (no reference counterpart).  ids DEVICE int32 [batch][beam][t], 1 <= t <= max_len; lens DEVICE int32 [batch][beam].  Row
 * (b, n) is caption n of image b in the layout fpnmt_sample returns: no <start>, no <end>, entries from position len on
 * ignored.
 *   decoder input at position j: <start> for j = 0, else ids[b][n][j-1];
 *   target at position j: ids[b][n][j] for j < len, and <end> at j = len when len < t;
 *   scored positions n_bn = len + 1 when len < t; when len == t, t positions and no <end> term (a truncated caption, as a
 *   sample whose len == max_len).
 * out_token_logprob[b][n][j] = log_softmax(z_j)[target_j] (temperature 1, no filtering) for j < n_bn, exactly 0 beyond;
 * out_logprob[b][n] = the sum of those terms in position order.  Scoring a caption fpnmt_sample produced gives that
 * sample's out_logprob (up to the precision of the two passes).  Position j attends to positions <= j of its caption and to
 * the memory tokens of its image: the memory of the last fpnmt_encode / fpnmt_generate / fpnmt_sample, or of `images` when
 * given.  A caption with len outside [0, t], or with an id outside [0, vocab) among its first len entries, gets NaN in both
 * outputs; ids are clamped before any load and the host never reads ids / lens.  out_logprob float32 [batch][beam],
 * out_token_logprob float32 [batch][beam][t] or NULL, both on the host (outputs_on_host != 0; the call synchronises the
 * stream) or both on the device.  Results are bit-identical run to run, with graphs on or off, under any permutation of the
 * captions among the N slots of an image and for any contents of ids at positions >= len.  The pass leaves nothing behind
 * that changes a later fpnmt_generate / fpnmt_sample.  Errors: FPNMT_ERR_INVALID for t outside [1, max_len] or NULL ids /
 * lens / out_logprob; FPNMT_ERR_STATE with decode_path = FUSED or while lane 0 holds a submitted batch. */
FPNMT_API int fpnmt_score(fpnmt_handle* h, const float* images, int images_on_host, const int32_t* ids, const int32_t* lens, int t,
                          float* out_logprob, float* out_token_logprob, int outputs_on_host, void* stream);

/* N-best beam search: the N = beam most likely captions of every image with their log-likelihoods (no reference counterpart).
 * Always a true beam search with frozen finished beams, whatever the handle's true_beam / finished_beams / length_penalty:
 *   start: at t = 0 only beam 0 is alive (log-score 0, the others -inf);
 *   a beam that emits <end> is frozen: its only candidate is itself, score unchanged;
 *   candidates are ranked by raw / lp(n), lp(n) = ((5 + n) / 6)^length_penalty, n = tokens generated including <end> for a
 *   frozen beam and t + 1 for a live one; ties go to the lower flat index parent * vocab + token.
 * An image is finished when all N of its beams are frozen (nothing can change after that) or after max_len steps; early_stop
 * != 0 ends the decode once every image is finished (the host looks every 4 steps), with identical results.
 * out_ids int32 [batch][beam][max_len]: no <start>, no <end>, 0 from position len on.  out_len int32 [batch][beam]: len <
 * max_len when the caption ended with <end>, max_len when it was truncated (as fpnmt_sample).  out_logprob float32
 * [batch][beam] or NULL: the raw beam score, the sum of the log_softmax terms over min(len + 1, max_len) positions, <end>
 * included; what fpnmt_score returns for that caption with t = max_len.  The N captions of an image come in rank order, by
 * out_logprob / lp(min(len + 1, max_len)) descending, ties to the lower slot; they are pairwise distinct when vocab >= beam.
 * With length_penalty = 0, row 0 is what fpnmt_generate returns on a handle created with true_beam = 1, finished_beams = 1
 * (that decode stops when its top beam freezes, and with alpha = 0 no later beam can overtake it); with length_penalty != 0
 * row 0 may be a longer caption that fpnmt_generate stopped too early to see.
 * images as fpnmt_sample (NULL = the memory of the last fpnmt_encode / generate / sample / score; given images are encoded and
 * become that memory).  Outputs DEVICE, or HOST with outputs_on_host != 0 (the call synchronises the stream).  Results are
 * bit-identical run to run, with graphs on or off, in both cache modes and with or without FPNMT_OPT_NO_KV_SHARE; the call
 * leaves nothing behind that changes a later fpnmt_generate / fpnmt_sample / fpnmt_score.  Errors: FPNMT_ERR_INVALID for a
 * NaN or infinite length_penalty or NULL out_ids / out_len; FPNMT_ERR_STATE with decode_path = FUSED, score_mode = PROB or
 * while lane 0 holds a submitted batch. */
FPNMT_API int fpnmt_beam_search(fpnmt_handle* h, const float* images, int images_on_host, float length_penalty, int32_t* out_ids,
                                int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop, void* stream);

/* Diverse beam search (Vijayakumar et al., "Diverse Beam Search"): N = beam captions per image in G = beam_groups groups of
 * N / G beams, each group a true beam search of width N / G that is pushed away from the tokens the earlier groups chose at
 * the same step.  It is fpnmt_beam_search with these changes (lambda = diversity):
 *   groups: G divides N; beam slot n belongs to group n / (N / G).
 *   start: at t = 0 the first beam of every group is alive (log-score 0), the others are -inf.
 *   step t: for g = 0 .. G-1 in order, group g's N / G new beams are chosen from the candidates of group g's own rows only.
 *     A live candidate (parent p, token v) has raw = score[p] + log_softmax(z_p)[v] and ranking key
 *     raw / lp(t + 1) - lambda * h_g(v), h_g(v) the number of new beams of groups 0 .. g-1 at this step that are live
 *     emissions of v (<end> counts like any token).  A frozen beam's only candidate is itself, key raw / lp(fin_len), never
 *     penalised and never counted in h.  Ties go to the lower flat index parent * vocab + token within the group.  The key
 *     is computed in fp32 as __fsub_rn(__fdiv_rn(raw, lp), __fmul_rn(lambda, (float)h)), without contraction.
 *   stored score: raw; the penalty is never accumulated, so out_logprob is the caption's log-likelihood and fpnmt_score of a
 *     returned caption gives it back.
 *   close: unchanged (all N beams frozen, or max_len steps; early_stop as fpnmt_beam_search).
 *   output order: group-major, slots [g * N / G, (g + 1) * N / G) hold group g; within a group by
 *     out_logprob / lp(min(len + 1, max_len)) descending, ties to the lower slot (the last step's keys carried the penalty,
 *     so the close sorts).
 * Captions are pairwise distinct within a group (vocab >= beam); across groups they may repeat: with lambda = 0 every group
 * holds the same list, that of fpnmt_beam_search at width N / G.  G = 1 is fpnmt_beam_search bit for bit (lambda ignored).
 * Outputs, images, determinism and what the call leaves behind as fpnmt_beam_search.  Errors: FPNMT_ERR_INVALID (nothing
 * launched) for G < 1, G not dividing beam, a negative, NaN or infinite diversity, a NaN or infinite length_penalty or NULL
 * out_ids / out_len; FPNMT_ERR_STATE as fpnmt_beam_search (decode_path = FUSED, score_mode = PROB, lane 0 busy). */
FPNMT_API int fpnmt_beam_search_diverse(fpnmt_handle* h, const float* images, int images_on_host, int beam_groups, float diversity,
                                        float length_penalty, int32_t* out_ids, int32_t* out_len, float* out_logprob,
                                        int outputs_on_host, int early_stop, void* stream);

/* Prompted decoding: fpnmt_sample, fpnmt_beam_search and fpnmt_beam_search_diverse continuing a given caption prefix per image
 * (no reference counterpart; completing a caption a user started, a fixed opening for every caption, keeping the first k
 * words and asking for the best continuations).  prefix_ids DEVICE int32 [batch][p], 1 <= p <= max_len - 1, and prefix_len
 * DEVICE int32 [batch]: image b's prefix is prefix_ids[b][0 .. prefix_len[b]), in the layout of fpnmt_score's ids (no
 * <start>, no <end>), shared by all N = beam samples or beams of the image.  The call is its unprompted twin with one change:
 *   forced step: at a step t < prefix_len[b] every row of image b, live or dead, takes the token prefix_ids[b][t] and keeps
 *     its own parent (parent = self; the physical cache mode's reorder is the identity for that image).  A live row's score
 *     grows by log_softmax(z)[token] at temperature 1 with no filtering, a dead beam stays at -inf.  Nothing is ranked, no
 *     diversity penalty is applied, nothing is counted in h_g and no Philox draw is used: the counter stays (t, b, n, 0), so
 *     the steps from prefix_len[b] on draw what they would draw anyway.
 *   after the prefix: from t = prefix_len[b] the image decodes as the unprompted call does (true-beam start: only beam 0, or
 *     the first beam of every group, is alive, and it now carries the prefix; frozen finished beams; lp(n) with n counting
 *     the prefix tokens too; the N-best close and early stop as before).  A prompted call runs the same number of steps as an
 *     unprompted one: the prefix fills positions 0 .. prefix_len[b] - 1 of the caption.
 *   outputs: the layout of the unprompted call.  out_ids / out_len hold the whole caption, prefix included; out_logprob is the
 *     whole caption's log-likelihood, prefix terms included, so fpnmt_score of a returned caption gives it back.
 *   invalid prefix: an image whose prefix_len is outside [0, p], or one of whose first prefix_len ids is outside [0, vocab) or
 *     equals end_id, comes back with out_len 0, zero ids and NaN out_logprob in all N rows; every other image's result is
 *     bit-identical to what it would be anyway.  The host never reads prefix_ids / prefix_len; ids are clamped before any load.
 * All prefix_len = 0 gives the unprompted call's results bit for bit.  Determinism and what the call leaves behind as the
 * unprompted twin.  Errors: FPNMT_ERR_INVALID (nothing launched) for p outside [1, max_len - 1], NULL prefix_ids /
 * prefix_len and every refusal of the unprompted twin; FPNMT_ERR_STATE with decode_path = FUSED, score_mode = PROB (beam
 * search only) or while lane 0 holds a submitted batch.  fpnmt_generate has no prompted form. */
FPNMT_API int fpnmt_sample_prefix(fpnmt_handle* h, const float* images, int images_on_host, const int32_t* prefix_ids,
                                  const int32_t* prefix_len, int p, const fpnmt_sampling* sampling, int32_t* out_ids,
                                  int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop, void* stream);
/* beam_groups = 1: the prompted fpnmt_beam_search (diversity ignored); > 1: the prompted fpnmt_beam_search_diverse. */
FPNMT_API int fpnmt_beam_search_prefix(fpnmt_handle* h, const float* images, int images_on_host, const int32_t* prefix_ids,
                                       const int32_t* prefix_len, int p, int beam_groups, float diversity, float length_penalty,
                                       int32_t* out_ids, int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop,
                                       void* stream);

/* Constrained decoding: the standard decoding controls for fpnmt_sample, fpnmt_beam_search and fpnmt_beam_search_diverse,
 * prompted or not (no reference counterpart).
 *   no_repeat_ngram  n: 0 = off; 1 <= n <= max_len: no n-gram occurs twice in a caption.
 *   min_len          0 = off; <end> is banned while the caption has fewer than min_len tokens; 0 <= min_len <= max_len.
 *   banned           HOST int32 [n_banned] token ids never emitted (e.g. the padding id 0, <start>, the OOV token), or NULL;
 *                    duplicates allowed; <end> may not be listed (min_len is how <end> is held back).
 * A live row at step t whose caption is w_0 .. w_{t-1} (no <start>, prefix tokens included) has the ban set
 * A(t) = S | E(t) | R(t): S = the banned list; E(t) = {end_id} when t < min_len; R(t) = { w_{j+n-1} : 0 <= j <= t - n,
 * w_{j .. j+n-2} = w_{t-n+1 .. t-1} } for n >= 1 (n = 1: every token already in the caption).  A constraint removes
 * candidates and never changes a score:
 *   beam search (N-best and diverse): a live candidate (parent p, token v) with v in A_p(t) is never ranked nor selected;
 *     everything else is the unconstrained search (raw score = score + log_softmax(z)[v] over all V, length penalty,
 *     diversity penalty and h_g; frozen beams unaffected), so out_logprob is still the caption's log-likelihood and
 *     fpnmt_score of a returned caption gives it back.
 *   sampling: steps 1-5 of fpnmt_sampling run on z' with z'_i = -inf for i in A(t) (top-k is the k-th largest allowed logit;
 *     greedy is the arg-max over allowed tokens, lowest id on ties); step 6, the reported log-probability, is log_softmax of
 *     the unmasked z; the Philox counter is unchanged.
 *   prefix: a forced step (t < prefix_len[b]) takes the prefix token even if it is in A(t); forced tokens count in the
 *     history of R and toward min_len.
 * Errors: FPNMT_ERR_INVALID (nothing launched) for an id outside [0, vocab) or end_id in `banned`, NULL banned with
 * n_banned > 0, n or min_len out of range, non-zero reserved words, vocab - |distinct banned ids| - max_len < beam (that
 * bound keeps at least `beam` allowed tokens for every live row at every step, as |R(t)| + |E(t)| <= max_len), and every
 * refusal of the unconstrained twin; FPNMT_ERR_STATE as the twin (decode_path = FUSED, score_mode = PROB for beam search,
 * lane 0 busy).  All-zero constraints (banned NULL) give the twin's results bit for bit; determinism, graphs, cache modes
 * and what the call leaves behind are as for the twin.  fpnmt_generate has no constrained form. */
typedef struct fpnmt_constraints {
  int32_t no_repeat_ngram;
  int32_t min_len;
  const int32_t* banned;
  int32_t n_banned;
  int32_t reserved[4]; /* must be 0 */
} fpnmt_constraints;
/* prefix_ids / prefix_len / p as fpnmt_sample_prefix, or NULL / NULL / 0 for an unprompted call. */
FPNMT_API int fpnmt_sample_constrained(fpnmt_handle* h, const float* images, int images_on_host, const int32_t* prefix_ids,
                                       const int32_t* prefix_len, int p, const fpnmt_sampling* sampling,
                                       const fpnmt_constraints* constraints, int32_t* out_ids, int32_t* out_len,
                                       float* out_logprob, int outputs_on_host, int early_stop, void* stream);
/* beam_groups = 1: the constrained fpnmt_beam_search (diversity ignored); > 1: the constrained fpnmt_beam_search_diverse.
 * prefix_ids / prefix_len / p as fpnmt_beam_search_prefix, or NULL / NULL / 0 for an unprompted call. */
FPNMT_API int fpnmt_beam_search_constrained(fpnmt_handle* h, const float* images, int images_on_host, const int32_t* prefix_ids,
                                            const int32_t* prefix_len, int p, int beam_groups, float diversity,
                                            float length_penalty, const fpnmt_constraints* constraints, int32_t* out_ids,
                                            int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop,
                                            void* stream);

/* Replaces: Pipeline.predict (utils/pipeline.py:82-154) for a batch: encoder + beam-search decode.
 * out_ids DEVICE-or-HOST int32 [batch, max_len] (0 padded), out_len int32 [batch]: exactly what predict() returns
 * per image (<start> stripped, trailing <end> stripped).  outputs_on_host != 0: results are copied to host and
 * the call synchronises the stream.  early_stop != 0: stop when every image's top beam has emitted <end>
 * (pipeline.py:147); 0: always run max_len steps (throughput runs).
 * step_scores: optional DEVICE float32 [max_len, batch] score of the top beam after each step (may be NULL). */
FPNMT_API int fpnmt_generate(fpnmt_handle* h, const float* images, int images_on_host, int32_t* out_ids, int32_t* out_len,
                   int outputs_on_host, int early_stop, float* step_scores, void* stream);
/* Replaces: the input overlap the reference gets from tf.data (dataset.py:90-92, map(load_image, AUTOTUNE) +
 * prefetch(AUTOTUNE)): double-buffered HOST input.  fpnmt_stage_images enqueues the host->device copy of a whole batch
 * (HOST float32 [batch, S, S, 3]; pinned memory for a truly asynchronous copy) into staging slot 0 or 1 on the engine's
 * own copy stream and returns at once; the buffer must stay valid until the matching fpnmt_generate_staged has been
 * issued and its stream synchronised.  fpnmt_generate_staged is fpnmt_generate on a staged slot: `stream` waits for that
 * slot's copy, runs encoder + decode, and releases the slot as soon as the encoder has consumed it.  Typical loop:
 * stage(0); for i: stage((i+1)&1, batch i+1); generate_staged(i&1, ...).  Error: FPNMT_ERR_STATE if the slot is empty. */
FPNMT_API int fpnmt_stage_images(fpnmt_handle* h, const float* host_images, int slot);
FPNMT_API int fpnmt_generate_staged(fpnmt_handle* h, int slot, int32_t* out_ids, int32_t* out_len, int outputs_on_host,
                                    int early_stop, float* step_scores, void* stream);
/* Replaces: the caller's loop over batches (utils/pipeline.py:156-175 evaluate; test.py:14-21) with `lanes` batches in
 * flight.  fpnmt_submit enqueues one whole batch (host->device copy when images_on_host, encoder, decode) on lane `lane`'s
 * own stream and returns at once; fpnmt_collect hands that batch's result over (outputs as fpnmt_generate; host outputs
 * synchronise the lane's stream, device outputs make `stream` wait for them).  The image buffer must stay valid until the
 * matching collect; device images are ordered after the work already enqueued on `stream`.  With early_stop != 0 the
 * decode needs the host to poll the finished-image counter: submit enqueues the encoder only and collect runs the decode
 * (the encoder of the batch submitted on another lane meanwhile still overlaps it).  A lane holds one batch at a time:
 * FPNMT_ERR_STATE on a second submit before collect, or a collect without submit.  Results are bit-identical to
 * fpnmt_generate on the same images (same kernels, same order per lane).  Typical loop, L = fpnmt_lanes(h):
 *   for i: if (i >= L) collect(i % L, ...batch i-L...); submit(i % L, batch i);   then collect the last L. */
FPNMT_API int fpnmt_lanes(fpnmt_handle* h);
FPNMT_API int fpnmt_submit(fpnmt_handle* h, int lane, const float* images, int images_on_host, int early_stop, void* stream);
FPNMT_API int fpnmt_collect(fpnmt_handle* h, int lane, int32_t* out_ids, int32_t* out_len, int outputs_on_host, void* stream);
/* Same, from an encoder output already in the engine (after fpnmt_encode) — the decode half only. */
FPNMT_API int fpnmt_decode(fpnmt_handle* h, int32_t* out_ids, int32_t* out_len, int outputs_on_host, int early_stop,
                 float* step_scores, void* stream);

/* Per-kernel timing of the encode and decode-step programs (CUDA events, `iters` repetitions each).  Writes a JSON
 * document into buf (NUL terminated, truncated to cap).  Reports algorithmic FLOPs/bytes per kernel. */
FPNMT_API int fpnmt_profile(fpnmt_handle* h, int iters, char* buf, size_t cap);
/* Number of kernel launches issued by this handle since creation (graph replays count their kernel nodes). */
FPNMT_API int64_t fpnmt_launch_count(fpnmt_handle* h);

/* ---- stand-alone operators (used by the parity tests to check single kernels) ------------------------------- */
/* out[pix, co] = act(conv(x) + bias [+ residual]); x DEVICE float32 NHWC [N,H,W,Cin]; kernel HOST float32
 * (kh,kw,Cin,Cout); bias HOST float32 [Cout] or NULL; residual DEVICE float32 (same shape as out, or
 * [N,H/2,W/2,Cout] when res_mode == 2) or NULL; out DEVICE float32 [N,H,W,Cout].  stride 1, zero padding
 * (pad_top, pad_left; the rest implied by the output size == input size). act: 0 none,1 relu,2 leaky(0.2),3 relu6 */
FPNMT_API int fpnmt_op_conv2d(int device, int precision, const float* x, int N, int H, int W, int Cin, const float* kernel,
                    int kh, int kw, int Cout, int pad_top, int pad_left, const float* bias, int act,
                    const float* residual, int res_mode, float* out, int force_bn, void* stream);

/* Replaces: dataset.load_image after the JPEG decode (dataset.py:21-24): tf.image.resize(img, (S, S)) — bilinear,
 * half-pixel centres, no antialias — followed by mobilenet_v2.preprocess_input (x / 127.5 - 1).
 * images_hwc DEVICE uint8 [N, H, W, 3]; out DEVICE float32 NHWC [N, S, S, 3] in [-1, 1] (the layout fpnmt_encode takes). */
FPNMT_API int fpnmt_op_preprocess(int device, const uint8_t* images_hwc, int N, int H, int W, int S, float* out, void* stream);

/* Replaces: dataset.load_image as a whole (dataset.py:19-26) for a batch of JPEG byte strings: tf.io.read_file's result ->
 * tf.image.decode_jpeg(channels=3) -> resize to (S, S) -> x / 127.5 - 1.  jpegs: n HOST pointers to the encoded files,
 * lengths their byte counts; decode runs on the GPU (nvJPEG), the RGB image never visits the host; out DEVICE float32 NHWC
 * [n, S, S, 3]; sizes_out optional HOST int32 [n][2] = decoded (height, width).  FPNMT_ERR_INVALID names the first image that
 * is not a decodable JPEG.  Work is enqueued on `stream`; the encoded bytes must stay valid until it has run. */
FPNMT_API int fpnmt_op_decode_jpeg(int device, const uint8_t* const* jpegs, const size_t* lengths, int n, int S, float* out,
                                   int32_t* sizes_out, void* stream);

/* out[r, f] = epilogue( x[r, :] @ kernel[:, f] + bias[f] [+ residual[r, f]] ) with the skinny-row Dense kernel of the
 * decoder step (tf.keras.layers.Dense, models/transformer.py:117-122, 165-168, 211-214, 357): x DEVICE float32 [R, K];
 * kernel HOST float32 (K, F) Keras layout; bias HOST [F] or NULL; residual DEVICE float32 [R, F] or NULL; out DEVICE
 * float32 [R, F].  gamma/beta HOST [F] != NULL (F must be 512): the epilogue is LayerNormalization(epsilon=eps) of
 * (dense + residual) (models/transformer.py:192,198,230,235,241), computed by a 4-CTA cluster. act as fpnmt_op_conv2d.
 * force_bn: 0 = automatic, 32 / 64 = rows per CTA of tgemm_kernel, 128 = the wide-row kernel of FPNMT_OPT_TGEMM_WIDE. */
FPNMT_API int fpnmt_op_dense(int device, int precision, const float* x, int R, int K, const float* kernel, int F,
                   const float* bias, int act, const float* residual, const float* gamma, const float* beta, float eps,
                   float* out, int force_bn, void* stream);
/* The vocabulary projection of the logits-free decode tail (bf16 only, the wide-row Dense kernel in its softmax-partials
 * epilogue): logits z[r, f] = x[r, :] @ kernel[:, f] + bias[f] are never stored; for every row r < R and 128-feature tile t
 * (ftiles = ceil(F / 128)) the kernel writes stat[r][t] = (max, sum exp(z - max)) over the tile's features f < F,
 * val[r][t][0..7] the 8 largest z, descending, ties lower f first, -inf padded, and idx[r][t][0..7] their f (0x7fffffff
 * where padded).  x DEVICE float32 [R, K]; kernel HOST float32 (K, F); bias HOST [F] or NULL; stat / val / idx DEVICE
 * float32 [.][ftiles][2] / float32 [.][ftiles][8] / int32 [.][ftiles][8], 16-byte aligned, written in place: rows >= R
 * and anything else the kernel does not write keep their contents.  K and F multiples of 8; bf16x3 is FPNMT_ERR_INVALID. */
FPNMT_API int fpnmt_op_vocab_stats(int device, int precision, const float* x, int R, int K, const float* kernel, int F,
                                   const float* bias, float* stat, float* val, int32_t* idx, void* stream);
/* fpnmt_op_vocab_stats with the target epilogue of a prompted beam search on the logits-free tail: stat / val / idx as
 * fpnmt_op_vocab_stats writes them, and for every row r < R whose target[r] lies in [0, F), target_logit[r] = z[r, target[r]],
 * the fp32 value the tile's statistics and candidates are computed from (written in place; other entries keep their
 * contents).  target DEVICE int32 [R] (-1 = none), target_logit DEVICE float32 [R]. */
FPNMT_API int fpnmt_op_vocab_stats_target(int device, int precision, const float* x, int R, int K, const float* kernel, int F,
                                          const float* bias, const int32_t* target, float* stat, float* val, int32_t* idx,
                                          float* target_logit, void* stream);
/* fpnmt_op_vocab_stats with the ban-mask epilogue of a constrained beam search on the logits-free tail: stat is written
 * exactly as fpnmt_op_vocab_stats writes it (over every feature), and val / idx hold each tile's 8 largest ALLOWED
 * logits (features f with bit f % 32 of mask[r][f / 32] clear), -inf / 0x7fffffff padded.  mask DEVICE uint32
 * [R][ceil(F / 32)].  target / target_logit (both NULL, or both set) as fpnmt_op_vocab_stats_target. */
FPNMT_API int fpnmt_op_vocab_stats_mask(int device, int precision, const float* x, int R, int K, const float* kernel, int F,
                                        const float* bias, const uint32_t* mask, const int32_t* target, float* stat, float* val,
                                        int32_t* idx, float* target_logit, void* stream);
/* The ban sets of fpnmt_constraints for `rows` given captions: mask[r] (DEVICE uint32 [rows][ceil(vocab / 32)]) = the bits of
 * A(len[r]) for the caption hist[r][0 .. len[r]) (DEVICE int32 hist [rows][ld], len [rows], clamped to [0, ld]; ids outside
 * [0, vocab) never set a bit).  no_repeat_ngram, min_len and banned / n_banned as fpnmt_constraints (banned HOST; the refusals
 * are those of the entry points, except the vocab - |S| - max_len bound). */
FPNMT_API int fpnmt_op_ban_mask(int device, const int32_t* hist, int ld, const int32_t* len, int rows, int vocab, int end_id,
                                int no_repeat_ngram, int min_len, const int32_t* banned, int n_banned, uint32_t* mask,
                                void* stream);

/* Encoder bandwidth kernels one at a time (the launchers of the engine's program, which choose the kernel by precision
 * and shape exactly as the engine does).  Activations are DEVICE float32, uploaded into bf16 (or bf16x3 hi + lo)
 * activations and read back after the kernel.  Channel views: a tensor with ld channels per pixel (in_ld / out_ld,
 * 0 = C, multiples of 8) of which the kernel reads or writes the first C, as DenseNet's stage buffers are used.  `out`
 * is read as well as written: its incoming contents are uploaded first, so values the kernel does not write (other
 * columns, other pixels) come back unchanged.  Host arrays are float32; all calls synchronise `stream`. */

/* MobileNetV2 DepthwiseConv2D 3x3 with BatchNorm folded in (models/retinanet.py backbone): out[n,yo,xo,c] =
 * act(sum_{ky,kx} x[n, yo*stride+ky-pad_top, xo*stride+kx-pad_left, c] * kernel[ky,kx,c] + bias[c]), taps outside the
 * image are zero.  x [N,H,W,in_ld]; kernel HOST (3,3,C,1); bias HOST [C] or NULL; out [N,Ho,Wo,out_ld]; stride 1 or 2;
 * act as fpnmt_op_conv2d.  bf16 stride 1 runs the 4-outputs-per-thread kernel, everything else the generic one. */
FPNMT_API int fpnmt_op_depthwise3x3(int device, int precision, const float* x, int N, int H, int W, int C, int in_ld,
                                    const float* kernel, const float* bias, int stride, int pad_top, int pad_left, int Ho,
                                    int Wo, int act, float* out, int out_ld, void* stream);
/* kind 0: MaxPooling2D k x k / stride, out-of-image taps ignored (-inf padding) or, with zero_pad, counted as 0
 * (ZeroPadding2D + valid pool); kind 1: AveragePooling2D 2x2 / 2 (Ho = H/2, Wo = W/2); kind 2: out[n,y,x] = x[n,2y,2x]
 * (the stride-2 1x1 input of a ResNet stage, Ho = (H+1)/2, Wo = (W+1)/2).  x [N,H,W,in_ld]; out [N,Ho,Wo,out_ld]. */
FPNMT_API int fpnmt_op_pool(int device, int precision, int kind, const float* x, int N, int H, int W, int C, int in_ld, int k,
                            int stride, int pad_top, int pad_left, int Ho, int Wo, int zero_pad, float* out, int out_ld,
                            void* stream);
/* DenseNet pre-activation BatchNormalization + ReLU: out[p,c] = max(x[p,c] * scale[c] + shift[c], 0).
 * x [pixels,in_ld]; scale / shift HOST [C]; out [pixels,out_ld]. */
FPNMT_API int fpnmt_op_scale_shift_relu(int device, int precision, const float* x, int64_t pixels, int C, int in_ld,
                                        const float* scale, const float* shift, float* out, int out_ld, void* stream);
/* The co-attention score map, Conv2D(1, 3x3, padding='same') on 256 channels (models/retinanet.py:287): x [N,H,W,256];
 * kernel HOST (3,3,256,1); bias HOST [1]; out [N,H,W].  bf16 only (the one-channel CUDA-core kernel); bf16x3 runs
 * fpnmt_op_conv2d with Cout = 1 and is rejected here with FPNMT_ERR_INVALID. */
FPNMT_API int fpnmt_op_score_conv(int device, int precision, const float* x, int N, int H, int W, const float* kernel,
                                  const float* bias, float* out, void* stream);
/* CoAttention_CNN (coattention.py:13-32): out[n,p,c] = softmax_p(score[n,:])[p] * cls[n,p,c].  score [N,HW];
 * cls and out [N,HW,C]. */
FPNMT_API int fpnmt_op_coattention(int device, int precision, const float* score, const float* cls, int N, int HW, int C,
                                   float* out, void* stream);
/* Encoder token pre-amble (transformer.py:279-296): out[n*HW+p] = LayerNormalization(epsilon=eps)(x[n*HW+p]) + pos[p],
 * d_model 512.  x and out [N*HW,512]; gamma / beta HOST [512]; pos HOST [HW,512]. */
FPNMT_API int fpnmt_op_tokens_ln_pos(int device, int precision, const float* x, int N, int HW, const float* gamma,
                                     const float* beta, float eps, const float* pos, float* out, void* stream);
/* Cross-level attention of the Multi-Transformer encoder (head dim 64): for view v, head h, image b,
 * out[b*Tq+i, (v*heads+h)*64 + d] = softmax_j(q_i . k_j / 8) v_j with q_i = q[b*Tq+i, (v*heads+h)*64 ..],
 * k_j = kv[v][b*tk[v]+j, k_col + h*64 ..], v_j = kv[v][b*tk[v]+j, v_col + h*64 ..].  q and out [B*Tq, nviews*heads*64];
 * kv HOST array of nviews DEVICE pointers to [B*tk[v], kv_ld]; tk HOST [nviews]; Tq <= 16 (else FPNMT_ERR_INVALID).
 * Kernel choice as the engine's: bf16 with nviews > 1 one launch of all views, bf16 with one view the tensor-core kernel,
 * bf16x3 or force_simt the fp32 CUDA-core kernel once per view. */
FPNMT_API int fpnmt_op_enc_attention(int device, int precision, const float* q, const float* const* kv, const int* tk,
                                     int nviews, int kv_ld, int k_col, int v_col, int B, int Tq, int heads, int force_simt,
                                     float* out, void* stream);

/* Decoder kernels one at a time, with the conventions of the encoder operators above (DEVICE float32 activations uploaded
 * into bf16 or bf16x3 activations; every tensor the kernel writes is uploaded first and read back whole; integer tables
 * are HOST int32 and checked on the host, an entry out of range is FPNMT_ERR_INVALID).  Head dim 64, d = heads * 64. */

/* Decode self-attention of step t (transformer.py:131-153 with the KV cache of pipeline.py): for row r and head h,
 * out[r, h*64 ..] = softmax_j(q . k_j / 8) v_j over the cached positions j < t, K/V read from cache row anc[t&1][r][j] * T + j,
 * and the new position t with k, v = qkv[r, d + h*64 ..], qkv[r, 2d + h*64 ..]; those are appended to the cache at row
 * r * T + t.  qkv [rows, 3d]; kc, vc [rows*T, d] (read and written); kc2 / vc2 NULL (ancestry mode) or the second buffer
 * pair of the physical mode, which odd steps read and append to; anc HOST [2][rows][T] (entries in [0, rows)); rep HOST
 * [2][rows] (representative row of each row's token-history class per step parity, entries in [0, rows)) or NULL; beam =
 * rows per image (1..32); out [rows, d].  kernel 0: the engine's choice (bf16x3 the split CUDA-core kernel, bf16 the
 * mma.sync kernel, which reads rep when beam <= 8 divides rows), 1: the CUDA-core kernel, 2: the mma.sync kernel (bf16 only). */
FPNMT_API int fpnmt_op_dec_self_attention(int device, int precision, const float* qkv, float* kc, float* vc, float* kc2,
                                          float* vc2, const int* anc, const int* rep, int rows, int T, int t, int heads, int beam,
                                          int kernel, float* out, void* stream);
/* Decode cross-attention over the memory tokens of the row's image (the CUDA-core kernel, split in bf16x3):
 * out[r, h*64 ..] = softmax_j(q[r, h*64 ..] . k_j / 8) v_j, k_j = kv[(r/beam)*Tk + j, k_col + h*64 ..], v_j likewise at
 * v_col.  q and out [rows, d]; kv [rows/beam*Tk, kv_ld]. */
FPNMT_API int fpnmt_op_dec_cross_attention(int device, int precision, const float* q, const float* kv, int kv_ld, int k_col,
                                           int v_col, int rows, int beam, int Tk, int heads, float* out, void* stream);
/* The fused decoder cross-attention block (bf16 only, d_model 512, 8 heads) of `layer` on images [b0, b0 + B) of a batch
 * of Btot: out2 = LayerNorm(softmax_j((out1 . wq + bq)_h K_h^T / 8) V_h . wo + bo + out1) over rows r of those images,
 * K and V of layer l at columns l*1024 and l*1024 + 512 of ckv [Btot*n_mem, L*1024] (n_mem <= 16, beam <= 16).  First the
 * fold kernels build the per-image operands of all Btot images and L layers, then one block kernel runs on the slice.
 * wq, wo HOST [L][512][512] as stored (Dense kernels, in x out); bq HOST [L][512]; bo, gamma, beta HOST [512] of `layer`;
 * out1 [Btot*beam, 512]; out2 [Btot*beam, 512] (rows outside the slice come back unchanged).  Optional outputs of the
 * fold: Mt [L*Btot*128, 512], Nt [L*Btot*512, 128], sbias [L*Btot*128] (see csrc/xattn.cuh). */
FPNMT_API int fpnmt_op_xattn(int device, int precision, const float* ckv, const float* wq, const float* bq, const float* wo,
                             const float* bo, const float* gamma, const float* beta, int Btot, int n_mem, int L, int layer,
                             int b0, int B, int beam, const float* out1, float* out2, float* Mt, float* Nt, float* sbias,
                             void* stream);
/* Physical KV-cache reorder after decode step tt = t - 1 (pipeline.py:134-137): for each cache c and row r,
 * dst[c][r*T + j] = src[c][((r/beam)*beam + parent[tt][r])*T + j] for j <= tt; t = 0 copies nothing.  src and dst
 * [ncaches][rows*T][D] (dst read and written); parent HOST [T][rows], entries in [0, beam). */
FPNMT_API int fpnmt_op_kv_reorder(int device, int precision, const float* src, float* dst, int ncaches, const int* parent,
                                  int rows, int beam, int T, int D, int t, void* stream);
/* Decoder input: out[r] = emb[tokens[r]] + pos[t].  tokens HOST [rows] in [0, V); emb HOST [V][C]; pos HOST [T][C]; t in
 * [0, T); out [rows, C]. */
FPNMT_API int fpnmt_op_embed_pos(int device, int precision, const int* tokens, int rows, const float* emb, int V,
                                 const float* pos, int T, int C, int t, float* out, void* stream);
/* LayerNormalization(epsilon=eps) of fp32 rows (d_model 512), the unfused decoder's LayerNorm: x [rows, 512] read as
 * float32; gamma / beta HOST [512]; out [rows, 512]. */
FPNMT_API int fpnmt_op_layernorm_rows(int device, int precision, const float* x, int rows, const float* gamma,
                                      const float* beta, float eps, float* out, void* stream);

/* One sampling step (the kernel of fpnmt_sample) on caller logits: logits DEVICE float32 [rows][V]; row r is sample
 * r % samples_per_image of image r / samples_per_image at step t; sampling as fpnmt_sample.  Outputs DEVICE: token int32
 * [rows], logprob float32 [rows] (log_softmax at temperature 1 of the token) or NULL, u_out float32 [rows] (the row's
 * Philox uniform) or NULL.  V in [1, 51200]. */
FPNMT_API int fpnmt_op_sample_step(int device, const float* logits, int rows, int V, int samples_per_image, int t,
                                   const fpnmt_sampling* sampling, int32_t* token, float* logprob, float* u_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FPNMT_H_ */
