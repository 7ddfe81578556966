// Group-stationary fused decoder (bf16 mode; opt-in: fpnmt_config.decode_path = FPNMT_DECODE_FUSED): ONE kernel runs whole
// decode steps - every layer of the KV-cached decoder (models/transformer.py:224-243, 321-341), the vocabulary projection
// (:357,372) and the beam-search tail (utils/pipeline.py:115-148) - for all T steps of a decode, replacing the 38-kernel
// chain per step of the per-operator path (2 432 launches per C2 batch -> 1).
//
// Why it can be one kernel: a decoder row (image, beam) only ever needs its own activations, the K/V cache rows of ITS image
// (through the beam ancestry) and the 16 memory tokens of its image.  A GROUP of 8 co-resident CTAs therefore owns
// floor(32 / beam) images = up to 32 rows for the whole decode and never synchronises with another group: no grid-wide
// barrier, no kernel boundary between the ~45 dependent GEMM / attention / LayerNorm phases of a step.
//
//   CTA c of the group = attention head c = output-feature slice c of every Dense layer:
//     qkv    : [q_c | k_c] and [v_c]                      (2 UMMA tiles, K = 512)   -> self-attention of head c in this CTA
//     o1/q2/o2: features c*64 .. c*64+63                   (1 tile,  K = 512)        -> LayerNorm over the row via an exchange
//     ffn1   : hidden features c*256 .. +255, LeakyReLU   (2 tiles, K = 512)        -> stays in shared memory (bf16 operand)
//     ffn2   : ALL 512 features over its K slice c*256..  (4 tiles, K = 256)        -> split-K partial sums, reduced over the group
//     final  : vocabulary slice c (ceil(V/8) rounded to 128), accumulators of all its tiles resident in TMEM at once
//   Orientation as in tgemm: the WEIGHT tile is the tcgen05 A operand (M = 128 features = TMEM lanes), the 32 rows are the
//   B operand (N = 32), D^T[feature][row] accumulates in TMEM.  The weights of one CTA form one contiguous stream in its
//   consumption order (packed on the host), pulled by a producer warp with TMA (128-row x 64 boxes, SWIZZLE_128B, two boxes
//   per mbarrier) through a 3 x 32 KB ring that runs ahead of the phase chain - the weights never depend on data.
//   Between phases the 8 CTAs exchange their slices through small group-private global buffers (L2 resident) guarded by a
//   barrier among the 16 worker warps of each CTA (monotonic counter in global memory: fence + atomic arrive, acquire-load
//   spin; the producer and MMA warps never take part, so the weight stream is not throttled by the phase barriers).  The
//   launch is cooperative, at most floor(SMs / 8) groups at a time, which guarantees that the CTAs of a group are resident.
//   (The first version used 8-CTA hardware clusters with DSMEM mbarriers: a B200 schedules only 15 such clusters of 220 KB
//   CTAs at once - cudaOccupancyMaxActiveClusters - so the 16th group of a 64-image batch ran as a second wave: 2x the time.)
//   Residual streams and LayerNorm inputs stay fp32 end to end (the per-operator path rounds them to bf16 between kernels).
//   Self-attention: beams with the same token history hold bit-identical K/V (DstepParams::rep), so when every image of the
//   group has one shared ancestry the K/V lines are read once per image, not once per beam (always the case under the
//   reference's beam initialisation); otherwise each row walks its own ancestry.
//   Tail: per-row max / sum-exp / top-N candidates are taken straight from the TMEM accumulators of the vocabulary tiles -
//   the [rows][V] logits are never written (teacher-forcing mode writes them for the parity tests) - merged over the group,
//   and the image's beams are ranked with the tf.math.top_k order (value descending, lower flat index first).
//
// Status (C2, B200, profiles/r02_*dstep*): parity slightly better than the chain (fp32 residuals, unfolded cross-attention);
// 374 us per decode step against 342 us for the chain, so decode_path AUTO still selects the chain.  Measured phase times per
// layer at t = 63: GEMM phases ~20 us (0.3 us per 32 KB group when streaming, ~1.5 us hand-off per job), self-attention
// 13 us, the six exchange barriers + operand staging ~20 us, cross-attention 3.5 us; vocabulary GEMM ~27 us, tail ~50 us.
#pragma once
#include "common.cuh"
#include "kernels.cuh"

namespace fpnmt {

constexpr int DS_ROWS = 32;              // rows per cluster == UMMA N
constexpr int DS_CTAS = 8;               // CTAs per cluster == attention heads
constexpr int DS_WORKER_WARPS = 16;
constexpr int DS_THREADS = (2 + DS_WORKER_WARPS) * 32;   // producer warp + MMA warp + workers
constexpr int DS_RING = 3;               // weight ring slots of two 16 KB TMA boxes each
constexpr int DS_SLOT = 16384;           // bytes per TMA box: one [128 features x 64 k] bf16 tile
constexpr int DS_MAX_VTILES = 14;        // vocabulary tiles of one CTA resident in TMEM (32 columns each)

// fp32 parameter block of one decoder layer (offsets in floats)
enum { DSB_Q = 0, DSB_K = 512, DSB_V = 1024, DSB_O1 = 1536, DSB_Q2 = 2048, DSB_O2 = 2560, DSB_F1 = 3072, DSB_F2 = 5120,
       DSB_LN1G = 5632, DSB_LN1B = 6144, DSB_LN2G = 6656, DSB_LN2B = 7168, DSB_LN3G = 7680, DSB_LN3B = 8192, DSB_SIZE = 8704 };
// bytes of one (layer, CTA) weight stream: QK 8 x 16K, V 8 x 8K, o1/q2/o2 24 x 8K, ffn1 16 x 16K, ffn2 16 x 16K
constexpr size_t DS_LAYER_STREAM = 8 * 16384 + 8 * 8192 + 24 * 8192 + 16 * 16384 + 16 * 16384;

struct DstepParams {
  int B, N, R;               // images, beam width, rows = B * N
  int ipc;                   // images per cluster = 32 / N
  int L, T, V;               // decoder layers, max steps, vocabulary
  int vslice, ntv;           // vocabulary features per CTA (multiple of 128), tiles per CTA (vslice / 128)
  int n_mem;                 // memory tokens per image (<= 16)
  int t0, nsteps;            // first step of this launch, number of steps
  int group0, ngroups;       // first CTA group of this launch (set by dstep_launch), groups of the whole batch
  int* gbar;                 // [ngroups] barrier counters of the groups (zeroed by dstep_launch)
  int* rep;                  // [2][R] (step parity) representative row of each beam: the first beam of its image with the
                             // same token history.  Beams with equal histories hold bit-identical K/V (same tokens, same image,
                             // computed by the same instructions), so attention reads the representative's cache rows - under
                             // the reference's beam initialisation (all beams identical, pipeline.py:101-102) one set of K/V
                             // lines per image instead of one per beam.  Every row still computes everything else itself.
  int mode;                  // 0 = beam search; 1 = teacher forcing: write the fp32 logits of every row, no beam tail
  const uint8_t* wstream;    // [L][8] layer streams, then [8] final-layer streams of ntv * 8 * 16 KB: plain [rows][64] bf16 tiles
  size_t final_off;          // byte offset of the final-layer streams
  size_t stream_bytes;       // total bytes
  const float* lparams;      // [L][DSB_SIZE]
  const float* vbias;        // [8 * vslice] final-layer bias (0 beyond V)
  const float* emb;          // [V][512] fp32 embedding table
  const float* pos;          // [T][512] fp32 positional table
  bf16* kcache;              // [L][R][T][512]
  bf16* vcache;
  const bf16* ckv;           // cross-attention K/V of the memory: [B * n_mem][ckv_ld], K of layer l at l*1024, V at l*1024+512
  int ckv_ld;
  // cluster-private exchange buffers (indexed by cluster * 32 + local row)
  bf16* x_att;               // [clusters*32][512] attention outputs (self, then cross)
  float* x_pre;              // [clusters*32][512] pre-LayerNorm sums
  float* x_part;             // [clusters][8][32][512] ffn2 split-K partial sums
  float* x_stat;             // [clusters*32][8][2] per-CTA (max, sum-exp) of the row's vocabulary slice
  float* x_cval;             // [clusters*32][8][N] per-CTA top-N logits of the row
  int* x_cidx;               // [clusters*32][8][N] their vocabulary ids (0x7fffffff = none)
  float* logits_out;         // mode 1: [R][ld_logits]
  int ld_logits;
  float* dbg;                // optional [L][3][clusters*32][512] LayerNorm outputs (parity taps), else nullptr
  long long* timeline;       // -DFPNMT_DBG_STAMPS builds only: globaltimer stamps of cluster 0 / CTA 0 in the last step
  BeamState st;
};

size_t dstep_smem_bytes();
int dstep_set_attributes();
int dstep_max_groups(int num_sms);   // CTA groups one cooperative launch can hold
int dstep_launch(const DstepParams& p, cudaStream_t stream);

}  // namespace fpnmt
