// Launchers for the CUDA-core (bandwidth-bound) kernels of the hot path.
#pragma once
#include "common.cuh"

namespace fpnmt {

// Opt-in shared-memory sizes are a per-DEVICE function attribute: Engine::init calls these for its device (a static
// "done once per process" guard would leave a second engine on another GPU of the same process without them).
int elementwise_set_attributes();
int attention_set_attributes();
void set_dec_att_simt(bool v);   // bf16 mode: CUDA-core decode self-attention instead of the mma.sync kernel (A/B, parity tests)
int beam_set_attributes();

// ---- elementwise.cu -----------------------------------------------------------------------------
// fp32 NHWC image (pointer read from a device slot so a captured graph can be re-pointed) -> im2col matrix [N*Ho*Wo][Kpad] for the Cin=3 stem convolutions (k = (ky*kw+kx)*3+c).
int launch_im2col_stem(const float* const* img_slot, int N, int H, int W, int kh, int kw, int stride, int pad_t, int pad_l, int Ho,
                       int Wo, Act out, cudaStream_t s);
// NHWC max-pool k x k / stride, padding handled by ignoring out-of-bounds taps (== -inf padding); with
// zero_pad the out-of-bounds taps contribute 0 (ZeroPadding2D + valid pool).
int launch_maxpool(Act in, int N, int H, int W, int k, int stride, int pad_t, int pad_l, int Ho, int Wo, bool zero_pad,
                   Act out, cudaStream_t s);
int launch_avgpool2(Act in, int N, int H, int W, Act out, cudaStream_t s);
int launch_subsample2(Act in, int N, int H, int W, Act out, cudaStream_t s);     // out[n,y,x] = in[n,2y,2x]
// depthwise 3x3 (+ per-channel bias, ReLU6); w = [9][C] fp32 with BN folded in
int launch_depthwise3x3(Act in, int N, int H, int W, int stride, int pad_t, int pad_l, int Ho, int Wo, const float* w,
                        const float* bias, int act, Act out, cudaStream_t s);
// out = relu(in * scale[c] + shift[c])   (DenseNet pre-activation BN)
int launch_scale_shift_relu(Act in, size_t pixels, const float* scale, const float* shift, Act out, cudaStream_t s);
// CoAttention_CNN: out[b,p,c] = softmax_p(score[b,:])[p] * cls[b,p,c]
int launch_coattention(Act score, Act cls, int N, int HW, Act out, cudaStream_t s);
// 3x3 "same" convolution of a 256-channel bf16 map to ONE channel (the co-attention score), w = fp32 [9][256], bias [1]
int launch_conv3x3_c1(Act in, const float* w, const float* bias, int N, int H, int W, Act out, cudaStream_t s);
// Encoder pre-amble: out[b*HW+p] = LN(in[b*HW+p]) + pos[p]   (C = 512)
int launch_tokens_ln_pos(Act in, int N, int HW, const float* gamma, const float* beta, float eps, const float* pos,
                         Act out, cudaStream_t s);
// y = LN(x) over rows of fp32 x[rows][C]
int launch_layernorm_rows(const float* x, int rows, int C, const float* gamma, const float* beta, float eps, Act out,
                          cudaStream_t s);
// Decoder input: out[r] = emb[tok[r]] + pos[*step]
int launch_embed_pos(const int* tokens, const float* emb, const float* pos, const int* step, int rows, int C, Act out,
                     cudaStream_t s);
// dataset.py:19-26 minus the JPEG decode: uint8 HWC [N,H,W,3] -> bilinear (TF2 half-pixel) resize to SxS -> x/127.5-1, fp32 NHWC
int launch_preprocess(const uint8_t* img, int N, int H, int W, int S, float* out, cudaStream_t s);
// fp32 rows -> activation view (used for uploads / tests)
int launch_f32_to_act(const float* x, size_t rows, int C, Act out, cudaStream_t s);
int launch_act_to_f32(Act in, size_t rows, float* out, cudaStream_t s);

// ---- attention.cu -------------------------------------------------------------------------------
// Encoder cross-level attention for one (layer, view): q (B*16 rows) vs K/V of a static view (B*Tk rows).
// force_simt: fp32 CUDA-core kernel even in bf16 mode (FPNMT_OPT_ENC_ATT_SIMT; compares the two paths on identical inputs)
int launch_enc_attention(Act q, int q_col, Act kv, int k_col, int v_col, int B, int Tq, int Tk, int heads, Act out,
                         int out_col, bool force_simt, cudaStream_t s);
// All (<= 4) cross-level attentions of one encoder layer as ONE launch (bf16 mode): view v uses K/V tensor kvs[v] with tks[v]
// keys and the query / output column block cols[v].
int launch_enc_attention_views(Act q, const Act* kvs, const int* tks, const int* cols, int nviews, int k_col, int v_col, int B,
                               int Tq, int heads, Act out, cudaStream_t s);
// Decoder self-attention, one new position per row, KV cache with beam-ancestry indirection.
// qkv: [rows][3*d] (q|k|v) of the new position; caches [rows][T][d]; anc [2][..][T] physical row per position, the two
// step parities `anc_stride` ints apart (rows may be a slice of a larger batch: anc_stride = total rows * T).
// kcache2 / vcache2 (p != nullptr): physical cache mode - odd steps read and append to the second buffer pair.
// Kernel choice: DEC_ATT_AUTO is the engine's (bf16x3: the split CUDA-core kernel; bf16: the mma.sync kernel, or the CUDA-core
// kernel under FPNMT_OPT_DEC_ATT_SIMT); DEC_ATT_SIMT / DEC_ATT_MMA force one of the two bf16 kernels (MMA needs plain bf16).
enum DecAttKernel { DEC_ATT_AUTO = 0, DEC_ATT_SIMT = 1, DEC_ATT_MMA = 2 };
int launch_dec_self_attention(Act qkv, Act kcache, Act vcache, Act kcache2, Act vcache2, const int* anc, size_t anc_stride,
                              const int* step, int rows, int T, int heads, Act out, cudaStream_t s, const int* rep_e = nullptr,
                              const int* rep_o = nullptr, int N = 1, DecAttKernel kernel = DEC_ATT_AUTO);
// rep_e / rep_o (bf16 tensor-core kernel only, beam N <= 8 dividing rows): BeamState::rep of the two step parities - the warp
// of a class representative computes every member of its token-history class (members = MMA rows).  nullptr: every row is
// its own class.
// Decoder cross-attention over the 16 memory tokens of the row's image.
int launch_dec_cross_attention(Act q, Act kv, int k_col, int v_col, int rows, int beam, int Tk, int heads, Act out,
                               cudaStream_t s);
// Normalised attention probabilities of the beam-0 row b * N of every image at step t = *step, for one decoder layer:
// self_out[b][h][t][j] = softmax_j(q_h . k_j / 8) for j <= t (K of position j at cache row anc[t & 1][b * N][j] * T + j) and
// exactly 0 for t < j < tlen; cross_out[b][h][t][j] for the n_mem memory tokens, from q2 against the K columns k_col of kv or,
// when Mt is set, from the fused cross-attention block's folded operands (scores = Mt . out1 + sbias, padding never read).
// Either output may be nullptr.  fp32 arithmetic on bf16 / bf16x3 operands.
struct DecProbArgs {
  Act qkv, kc;                  // layer's QKV projection [rows][3d] and K cache [rows * T][d]
  const int* anc;               // ancestry table of the parity 0, the second parity anc_stride ints further
  size_t anc_stride;
  int T;
  Act q;                        // q2 [rows][d] or, with Mt, out1 [rows][512]
  Act kv;                       // cross K/V of the memory [B * n_mem][..] (unused with Mt)
  int k_col;
  const bf16* Mt;               // [B][128 (h,j)][512] folded operand of this layer, or nullptr
  const float* sbias;           // [B][128] score bias of this layer (with Mt)
  int n_mem;
  const int* step;
  int N, heads, tlen;
  float* self_out;              // [B][heads][tlen][tlen] of this layer
  float* cross_out;             // [B][heads][tlen][n_mem] of this layer
};
int launch_dec_attention_probs(const DecProbArgs& a, int B, cudaStream_t s);

// ---- beam.cu ------------------------------------------------------------------------------------
struct BeamState {
  int B, N, V, T;            // images, beam width, vocab, max steps
  int Btot;                  // images of the whole batch when this state is a slice of it (stride of the [T][..] logs)
  int start_id, end_id;
  int prob_mode;             // 1: product of probabilities (reference), 0: sum of log-probs
  float* score[2];           // [B*N] double-buffered beam scores
  int* seq[2];               // [B*N][T+1] token sequences (seq[.][0] = <start>)
  int* anc[2];               // [B*N][T] physical cache row per position
  int* rep[2];               // [B*N] per step parity (may be null): representative row = the first beam of the image with the
                             // same token history.  Beams with equal histories hold bit-identical K/V (same inputs, same
                             // instructions), so the beam kernel points a beam's ancestry at its representative's cache rows:
                             // under the reference's beam initialisation (all beams identical, pipeline.py:101-102) the
                             // attention kernels then read ONE set of cache lines per image instead of one per beam (8x less
                             // HBM traffic); every row still computes and appends its own K/V and its own attention.
  int* last_tok;             // [B*N] token fed to the next step
  int* step;                 // device scalar: current step t (0-based)
  int* done;                 // [B] 1 once the image's top beam has emitted <end>
  int* n_done;               // [2]: number of finished images, image-completion counter
  int* img_count;            // [B] rows of the image whose candidates are ready (elects the block that merges)
  int* out_ids;              // [B][T]
  int* out_len;              // [B]
  float* cand_val;           // [B*N][N] per-row candidates (phase 1 -> phase 2)
  int* cand_idx;             // [B*N][N]
  float* step_logprob;       // optional [T][B] log-prob (or prob) increment of the chosen top beam, may be null
  int* parent_out;           // optional [T][B*N] parents chosen per step (debug / parity), may be null
  int* token_out;            // optional [T][B*N]
  long long* dbg;            // optional globaltimer stamps of image 0 (FPNMT_DBG_OP=beam_step), else nullptr
  // EXTENSION (fpnmt_config.finished_beams / length_penalty; 0 / 0 = the reference, pipeline.py:143-148): a beam that has
  // emitted <end> is frozen - it contributes ONE candidate (itself, score unchanged) to the next ranking instead of V - and
  // candidates are ranked by score / lp[length] with lp[len] = ((5 + len) / 6)^alpha (host table, lp[.] = 1 for alpha = 0).
  int finished_mode;
  int* fin_len[2];           // [B*N] per step parity: 0 = live beam, else the length (tokens incl. <end>) at which it finished
  const float* lp;           // [T + 1] length-penalty table
  // Logits-free decode tail (log score mode, beam <= 8): the vocabulary projection (tgemmw_kernel, TgemmParams::vs_*) leaves
  // per (row, 128-token tile) softmax partials and its 8 largest logits; phase 1 of k_beam_step merges those instead of
  // scanning a [rows][V] fp32 logits tensor (which is then never written).  nullptr = the logits path.
  const float2* vs_stat;     // [B*N][vs_tiles] (max, sum exp(x - max))
  const float* vs_val;       // [B*N][vs_tiles][8] largest logits of the tile, -inf padded
  const int* vs_idx;         // [B*N][vs_tiles][8] token ids
  int vs_tiles;
  int physical;              // 1: "physical" KV-cache mode - the ancestry tables stay the identity (never written here) and
                             // launch_kv_reorder moves the cache rows by beam parent after every step
  // N-best outputs (fpnmt_beam_search; launch_beam_step_nbest, finished_mode = 1): an image closes when all N beams are frozen
  // or at t = T - 1, and its close writes every beam, in rank order, instead of beam 0 into out_ids / out_len.
  struct NBest {
    int* ids;                // [B][N][T] caption of each beam, 0 padded (no <start>, no <end>)
    int* len;                // [B][N]
    float* score;            // [B][N] raw beam score (sum of log_softmax terms, <end> included)
    void* unused;            // 32 bytes in all: the kernel parameters after BeamState keep their 16-byte alignment, so the
                             // generate instantiations of k_beam_step keep their vector constant loads (same code)
  } nb;
};
static_assert(sizeof(BeamState::NBest) == 32, "see BeamState::NBest::unused");
// true_beam = 0 reproduces the reference (all beams start identical, pipeline.py:101-102); 1 starts beams 1..N-1 dead
int launch_beam_init(const BeamState& st, int true_beam, cudaStream_t s);
// Next-step decoder input written by the beam kernel: x[row] = emb[token] + pos[step + 1] (emb == nullptr: skip).
struct BeamEmbed {
  const float* emb;          // [V][D] fp32
  const float* pos;          // [T][D] fp32
  Act x;                     // [B*N][D]
  int D;
};
// One beam-search step on fp32 logits [B*N][ld]: row softmax statistics + candidate scores + row-local top-N, then
// (last block of each image) merge N x N candidates, emit parents/tokens/scores, reorder sequences + ancestry, handle
// <end>, write the next decoder input, advance the step counter.  Buffers are double-buffered on (step & 1).
int launch_beam_step(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, cudaStream_t s);
// The same step with the N-best close (BeamState::nb): needs finished_mode and log scores.
int launch_beam_step_nbest(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, cudaStream_t s);
// The refusals of launch_beam_step (set_last_error + 1), for callers that must refuse before launching anything else.
int check_beam_step(const BeamState& st, int ld);
// Physical KV-cache reorder by beam parent (pipeline.py:134-137 applied to the cache instead of an indirection table), ALL
// layers and both of K / V in one launch: after decode step tt = *step - 1, for every row r of the batch
//   buf[(tt + 1) & 1][c][r][0..tt] = buf[tt & 1][c][(r / N) * N + parent[tt][r]][0..tt]      c = 0 .. ncaches - 1
// where a cache row's live positions are one contiguous span of (tt + 1) * row_bytes bytes.  `bufs` is a device array of
// 2 * ncaches base pointers ([parity][cache]); parent = BeamState::parent_out ([T][rows_total], local beam index).
int launch_kv_reorder(const bf16* const* bufs, int ncaches, const int* parent, int rows, int rows_total, int N, int T, int row_bytes,
                      const int* step, cudaStream_t s);

// ---- sample.cu ----------------------------------------------------------------------------------
// Sampled decoding (fpnmt_sampling, include/fpnmt.h): row r = (image r / N, sample r % N) of fp32 logits [rows][V] draws one
// token from softmax(z / temperature) restricted to the top-k logits (ties kept) and then to the nucleus of top_p of that
// mass, with the Philox4x32-10 uniform of counter (t, image, sample, 0) and key (seed lo, seed hi).
struct SampleParams {       // device copy of fpnmt_sampling read by every step (changing it needs no graph re-capture)
  float temperature;
  int top_k;
  float top_p;
  int pad;
  unsigned long long seed;
};
struct SampleState {
  int rows, V, N, T;         // rows = images * N samples, vocab, samples per image, max steps
  int start_id, end_id;
  const SampleParams* params;
  int* step;                 // device step counter (advanced by the kernel), or nullptr: step t0
  int t0;
  // engine decode state (ids == nullptr: stand-alone step, nothing below is touched)
  int* last_tok;             // [rows] token fed to the next step
  int* ids;                  // [rows][T] caption of each sample, 0 padded (no <start>, no <end>)
  int* len;                  // [rows]
  int* fin;                  // [rows] 1 once the sample emitted <end> (or ran T steps)
  float* lp;                 // [rows] sum of log_softmax(z)[token] (temperature 1) over the emitted steps
  int* img_fin;              // [images] finished samples of the image
  int* n_done;               // [2]: finished images, row-completion counter of the step
  // per-step outputs, each optional
  int* tok_out;              // [rows]
  float* lp_out;             // [rows] log_softmax(z)[token] at temperature 1
  float* u_out;              // [rows] the row's uniform
};
int sample_set_attributes();
// step 0, last_tok = <start>, identity ancestry [2][rows][T] in `anc`, per-row and per-image state cleared
int launch_sample_init(const SampleState& st, int* anc, cudaStream_t s);
int launch_sample_step(const SampleState& st, const float* logits, cudaStream_t s);

// ---- score.cu -----------------------------------------------------------------------------------
// Caption scoring (fpnmt_score, include/fpnmt.h): row r = c * t + j is position j of caption c = b * N + n.
struct ScoreArgs {
  int caps, t, V;            // captions (B * N), positions per caption, vocab
  int start_id, end_id;
  const int* ids;            // [caps][t] caption tokens (no <start>, no <end>)
  const int* lens;           // [caps]
  int* tgt;                  // [caps * t] target id of each row (written by score_embed)
  int* bad;                  // [caps] 1: length outside [0, t] or an id outside [0, V) among the first len
  float* tok_lp;             // [caps * t] log_softmax(z)[target]
  float* lp;                 // [caps] sum over the scored positions
};
// x[r] = emb[input token] + pos[j] (input: <start> at j = 0, else ids[c][j - 1] clamped to [0, V)), tgt, bad
int launch_score_embed(const ScoreArgs& a, const float* emb, const float* pos, Act x, cudaStream_t s);
// causal self-attention of every caption over its own t positions: qkv [caps * t][3d] (q | k | v) -> out [caps * t][d]
// (fp32 CUDA-core arithmetic on bf16 or split bf16x3 operands)
int launch_score_self_attention(Act qkv, int caps, int t, int heads, Act out, cudaStream_t s);
// tok_lp[i] = log_softmax(logits[i])[tgt[i]] for i < rows, fp32 logits [rows][V]
int launch_score_rows(const float* logits, int rows, int V, const int* tgt, float* tok_lp, cudaStream_t s);
// lp[c] = sum of tok_lp over the scored positions of caption c; 0 after them; NaN everywhere for a flagged caption
int launch_score_sum(const ScoreArgs& a, cudaStream_t s);

}  // namespace fpnmt
