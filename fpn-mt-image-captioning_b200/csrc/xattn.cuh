// Fused decoder cross-attention block (bf16 mode): one tcgen05 kernel per layer and decode step replaces
//   q2 = out1 . Wq + bq ;  att = softmax(q2_h K_h^T / 8) V_h  (16 memory tokens) ;  out2 = LN(att . Wo + bo + out1)
// (models/transformer.py:232-235 with MultiHeadAttention :131-153), i.e. three kernels of the step.
//
// The memory K/V of an image are constant during its decode, so the projections around the attention are folded into
// per-image operands once per batch (k_xattn_fold, CUDA cores, ~6 GFLOP):
//   Mt[l][b][(h,j)][k] = 1/8 * sum_d K_b,h[j][d] * Wq[k][h*64+d]        scores^T = Mt . out1^T + sbias    (128 x 512)
//   Nt[l][b][f][(h,j)] =       sum_d V_b,h[j][d] * Wo[h*64+d][f]        out2^T   = Nt . P^T + bo          (512 x 128)
// With 8 heads x 16 tokens = 128 (h,j) pairs the score matrix of one image is exactly one UMMA M = 128 tile: lane = (h,j),
// column = beam row; the softmax over j is a 16-lane shuffle reduction on the TMEM-loaded accumulator; P^T is written to
// shared memory as the K-major B operand of the second GEMM chain (4 feature tiles x K = 128); the epilogue adds the
// residual and applies LayerNorm over the 512 features, all inside one CTA per image.
#pragma once
#include "common.cuh"

namespace fpnmt {

constexpr int XA_THREADS = 192;     // TMA warp + MMA warp + 4 epilogue warps
constexpr int XA_NROWS = 16;        // UMMA N: beam rows of one image, padded to 16
constexpr int XA_PAIRS = 128;       // heads x memory tokens

struct XattnParams {
  int B, beam, R;            // images of this launch, beam width (<= 16), rows = B * beam
  int b0, Btot;              // first image of this launch within the batch, images of the whole batch (operand index)
  int layer;                 // decoder layer (selects the per-image operands)
  const float* sbias;        // [L][B][128] score bias (bq . K / 8; -1e30 for padded tokens)
  const float* obias;        // [512] output-projection bias of this layer
  const float* gamma;        // LayerNorm2
  const float* beta;
  float eps;
  Act res;                   // out1 [R][512] (also the B operand of the first GEMM, through tmX)
  Act out;                   // out2 [R][512]
  long long* dbg;            // optional globaltimer stamps (FPNMT_DBG_OP), else nullptr
};

struct XattnOp {
  CUtensorMap tmM, tmN, tmX;
  XattnParams p;
};

size_t xattn_smem_bytes();
int xattn_set_attributes();
int xattn_launch(const XattnOp& op, cudaStream_t stream);
// Mt: [L*B*128][512] bf16, Nt: [L*B*512][128] bf16, x: out1 view.
// x / out are the row views of images [b0, b0 + B) of a batch of Btot images.
int make_xattn_op(XattnOp* op, const bf16* Mt, const bf16* Nt, int L, int Btot, int b0, int B, int beam, int layer,
                  const float* sbias, const float* obias, const float* gamma, const float* beta, const Act& x, const Act& out);

// Folding kernels (once per batch, all layers): ckv = cross K/V activations [B*n_mem][L*2*512] (K at l*1024, V at +512).
// wq: bf16 [L][512 k][512 (h,d)] (the Dense kernel of mha2/wq as stored, in -> out); woT: bf16 [L][512 f][512 (h,d)] (the
// mha2 output Dense kernel TRANSPOSED); bq: per-layer fp32 bias pointers.
// Host side of the fold operands of one layer (512 x 512 each, bf16 bits): wq_bf16 = the mha2/wq Dense kernel as stored,
// woT_bf16[f][(h,d)] = the mha2 output Dense kernel wo[(h,d)][f] transposed.
void xattn_fold_weights(const float* wq, const float* wo, uint16_t* wq_bf16, uint16_t* woT_bf16);
int launch_xattn_fold(const Act& ckv, int B, int n_mem, int L, const bf16* wq, const float* const* bq, const bf16* woT,
                      bf16* Mt, bf16* Nt, float* sbias, cudaStream_t s);

}  // namespace fpnmt
