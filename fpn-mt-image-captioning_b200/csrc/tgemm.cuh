// Skinny-row Dense kernel for the decoder step (and the 16-token encoder layers): out[r][f] = X[r][:] . Wt[f][:].
//
// With only R = batch*beam (512) activation rows, the classic orientation (rows = MMA M) makes every CTA pull a
// 128-row x K activation panel that only exists once the previous kernel has finished, so each of the ~50 small
// GEMMs of a decode step serialises ~150 KB of dependent loads behind the kernel boundary.  This kernel swaps the
// roles: the WEIGHT tile [128 features x K] is the tcgen05 A operand (M = 128 features = TMEM lanes) and is
// prefetched by TMA BEFORE griddepcontrol.wait (weights are static, so under programmatic dependent launch they
// stream in while the producer kernel is still running); the activation tile [BN rows x K] (BN = 32/64) is the B
// operand and the only dependent load (4-8 KB per k-chunk).  The accumulator is D^T: lane = feature, column = row.
// Epilogues:
//   plain : + bias[f] (+ residual[r][f]) -> activation -> bf16 (hi/lo) or fp32, warp-coalesced along features
//   LN    : a cluster of 4 CTAs (the 4 feature tiles of a 512-wide output) reduces per-row mean / M2 through shared
//           memory + DSMEM (Chan's parallel variance), then writes LayerNorm(x + residual) as 64-byte row segments.
#pragma once
#include "common.cuh"

namespace fpnmt {

constexpr int TG_BM = 128;       // features per tile (UMMA M)
constexpr int TG_BK = 64;        // K elements per chunk (one 128 B swizzle row)
constexpr int TG_THREADS = 192;  // TMA warp + MMA warp + 4 epilogue warps
constexpr int TG_A_SLOTS = 8;    // weight chunks resident in shared memory (8 x 16 KB: a full K = 512 panel)
constexpr int TG_B_STAGES = 8;   // a full K = 512 activation panel in flight

struct TgemmParams {
  int R, F;              // activation rows, output features
  int kchunks;           // ceil(K / 64)
  int nterms, w_lo_off;  // 1 = bf16; 3 = bf16x3 (W.hi*X.hi + W.lo*X.hi + W.hi*X.lo), K offset of the weight low halves
  int ftiles, rtiles;    // ceil(F / 128), ceil(R / BN)
  int rt_per_item;       // row tiles handled by one CTA (consecutive)
  int stationary;        // 1: the weight panel (<= 8 chunks) stays in shared memory for all row tiles of the CTA
  const float* bias;     // [F] (padded to a multiple of 128) or nullptr
  int act;
  Act out;               // bf16 output view [R][ld] (p may be nullptr)
  float* out_f32;        // optional fp32 output [R][ld_f32]
  int ld_f32;
  int has_res;
  Act res;               // residual [R][F], added before activation / LayerNorm
  const float* gamma;    // LN fusion when != nullptr (requires F == 512, BN == 32, cluster of 4 feature tiles)
  const float* beta;
  float eps;
  long long* dbg;        // optional timeline buffer (globaltimer stamps of block 0), normally nullptr
  // tgemmw_kernel only - vocabulary projection WITHOUT a logits tensor (decode tail, utils/pipeline.py:115-131): instead of the
  // [R][F] outputs each (row, 128-feature tile) leaves its softmax partials and its TG_VS_N best logits, which k_beam_step merges.
  float2* vs_stat;       // [R][ftiles] (max, sum of exp(x - max)) over the tile's valid features, or nullptr = normal outputs
  float* vs_val;         // [R][ftiles][TG_VS_N] largest logits of the tile, descending, ties -> lower feature first (-inf padded)
  int* vs_idx;           // [R][ftiles][TG_VS_N] their feature indices (0x7fffffff where padded)
};
constexpr int TG_VS_N = 8;   // candidates kept per (row, tile): covers beam widths <= 8

struct TgemmOp {
  CUtensorMap tmW, tmX_hi, tmX_lo;
  TgemmParams p;
  int BN;        // 32 or 64 (tgemm_kernel); 64 or 128 (tgemmw_kernel)
  int wide;      // 1: tgemmw_kernel (tgemmw.cu)
  int grid;
  int cluster;   // 1, or 4 (LayerNorm)
  double flops;
  // vocabulary projection without logits (p.vs_stat) of a prompted beam search: tgemmw_target_kernel also writes
  // tgt_logit[r] = z[r][tgt[r]] for every row r whose tgt[r] lies in [0, F) (device [R] each; nullptr = tgemmw_kernel)
  const int* tgt = nullptr;
  float* tgt_logit = nullptr;
  // constrained beam search on the same tail: tgemmw_mask_kernel keeps banned features out of every row's candidates (mask
  // [2][R][ceil(F / 32)] bits by the parity of *mask_step, nullptr: parity 0; tgt may then be nullptr)
  const uint32_t* mask = nullptr;
  const int* mask_step = nullptr;
};

size_t tgemm_smem_bytes(int BN);
int tgemm_launch(const TgemmOp& op, cudaStream_t stream);
int tgemm_set_attributes();

// x: activation view [R][ld] (C == K); wt: [F][K] bf16 (split: [F][2K]).  BN = 0 selects automatically.
int make_tgemm_op(TgemmOp* op, int R, const Act& x, const bf16* wt, int F, int K, bool split, const float* bias, int act,
                  const Act& out, float* out_f32, int ld_f32, const Act* res, const float* gamma, const float* beta,
                  float eps, int num_sms, int force_bn = 0);

// Wide-row, two-CTAs-per-SM variant (tgemmw.cu): BN = 128 rows per CTA, K streamed through a 96 KB ring, bf16 mode only.
size_t tgemmw_smem_bytes(int BN);
int tgemmw_launch(const TgemmOp& op, cudaStream_t stream);
int tgemmw_set_attributes();
bool tgemmw_supports(bool split, bool has_res, bool ln, int F, int K);
int make_tgemmw_op(TgemmOp* op, int R, const Act& x, const bf16* wt, int F, int K, const float* bias, int act, const Act& out,
                   float* out_f32, int ld_f32, const Act* res, const float* gamma, const float* beta, float eps, int num_sms,
                   float2* vs_stat = nullptr, float* vs_val = nullptr, int* vs_idx = nullptr);

}  // namespace fpnmt
