// Caption scoring (fpnmt_score): the teacher-forced decoder over all B * N * t positions of N given captions per image as
// rows of ONE pass.  Row r = c * t + j is position j of caption c = b * N + n.  The Dense layers and the cross-attention run
// on the engine's existing kernels; this file holds what the parallel pass needs beyond them:
//   score_embed          : decoder input emb[token] + pos[j] of every row, the row's target id and the caption's NaN flag
//   score_self_attention : causal self-attention of every position straight from the layer's QKV projection (no KV cache)
//   score_rows           : log_softmax(z)[target] of a chunk of fp32 logits rows
//   score_sum            : per-caption sum of its scored terms in position order, zero / NaN fill
// Every reduction has a fixed order, so results are bit-identical run to run and independent of the other captions.
#include <math.h>

#include "attention.cuh"
#include "kernels.cuh"

namespace fpnmt {

// Scored positions of a caption of length len (clamped; a caption with len outside [0, t] is NaN in the end anyway).
__device__ __forceinline__ int scored_positions(int len, int t) {
  len = min(max(len, 0), t);
  return len < t ? len + 1 : t;
}

// One thread per (row, 8 channels).  Token ids are clamped into [0, V) before any load: a bad id cannot fault, it only
// raises the caption's flag.  Same arithmetic as k_embed_pos (fp32 emb + pos, then st_act8).
__global__ void k_score_embed(ScoreArgs a, const float* __restrict__ emb, const float* __restrict__ pos, Act x) {
  pdl_launch();
  pdl_wait();
  const int groups = x.C / 8;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int t = a.t;
  if (idx >= (size_t)a.caps * t * groups) return;
  const int g = (int)(idx % groups);
  const int r = (int)(idx / groups);
  const int c = r / t, j = r % t;
  const int* cid = a.ids + (size_t)c * t;
  const int tok = j == 0 ? a.start_id : min(max(cid[j - 1], 0), a.V - 1);
  const float* e = emb + (size_t)tok * x.C + g * 8;
  const float* p = pos + (size_t)j * x.C + g * 8;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = e[i] + p[i];
  st_act8(x, (size_t)r, g * 8, v);
  if (g == 0) {
    const int len = a.lens[c];
    // unscored rows (j > len) get token 0: their term is computed and then replaced by 0 in k_score_sum
    a.tgt[r] = j < len ? min(max(cid[j], 0), a.V - 1) : (j == len ? a.end_id : 0);
    if (j == 0) {
      int bad = len < 0 || len > t;
      for (int k = 0; k < len && !bad; ++k) bad = cid[k] < 0 || cid[k] >= a.V;
      a.bad[c] = bad;
    }
  }
}

// ---- causal self-attention ------------------------------------------------------------------------------------------------
// One warp per (row, head): the query of position j against the K/V of positions 0 .. j of its caption, read straight from
// the layer's QKV projection (warp_attend: fp32 CUDA-core arithmetic on bf16 or split bf16x3 operands, online softmax across
// 32-position chunks).  Every row walks the same chunks whatever the other rows hold, so a row's result depends on its
// caption's positions <= j only.
constexpr int SC_WARPS = 4;
template <bool SPLIT>
__global__ void __launch_bounds__(SC_WARPS * 32) k_score_self_attention(Act qkv, int rows, int t, int heads, Act out) {
  __shared__ WarpScratchT<SPLIT> s_ws[SC_WARPS];
  pdl_launch();
  pdl_wait();
  const int gw = blockIdx.x * SC_WARPS + (threadIdx.x >> 5);
  if (gw >= rows * heads) return;
  const int lane = threadIdx.x & 31;
  WarpScratchT<SPLIT>& ws = s_ws[threadIdx.x >> 5];
  const int row = gw / heads, h = gw % heads;
  const int j = row % t;
  const size_t base = (size_t)row - j;
  const int d = heads * DH;
  const float2 qv = ld_pair(qkv, row, h * DH, lane);
  ws.q[lane * 2] = qv.x * 0.125f;       // 1/sqrt(64)
  ws.q[lane * 2 + 1] = qv.y * 0.125f;
  __syncwarp();
  float m = -INFINITY, l = 0.f, o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i] = 0.f;
  warp_attend<SPLIT>(ws, qkv, d + h * DH, qkv, 2 * d + h * DH, j + 1, [&](int pos) { return base + pos; }, lane, m, l, o);
  pv_reduce(o);
  if (lane < 8) {
    const float inv = 1.f / l;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] *= inv;
    st_act8(out, (size_t)row, h * DH + lane * 8, o);
  }
}

// ---- log-probability of the target of each logits row ---------------------------------------------------------------------
// One block per row: max, sum exp(z - max) in a fixed order (per-thread strided partials, xor-tree warp reductions, the 8
// warp partials summed in warp order), then z[target] - max - log(sum).
constexpr int SR_THREADS = 256;
__global__ void __launch_bounds__(SR_THREADS) k_score_rows(const float* __restrict__ logits, int V, const int* __restrict__ tgt,
                                                           float* __restrict__ tok_lp) {
  __shared__ float s_red[SR_THREADS / 32];
  pdl_launch();
  pdl_wait();
  const int row = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* z = logits + (size_t)row * V;
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < V; i += SR_THREADS) mx = fmaxf(mx, z[i]);
  mx = warp_max(mx);
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = s_red[0];
#pragma unroll
  for (int w = 1; w < SR_THREADS / 32; ++w) mx = fmaxf(mx, s_red[w]);
  __syncthreads();
  float sum = 0.f;
  for (int i = threadIdx.x; i < V; i += SR_THREADS) sum += expf(z[i] - mx);
  sum = warp_sum(sum);
  if (lane == 0) s_red[warp] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < SR_THREADS / 32; ++w) s += s_red[w];
    const int k = min(max(tgt[row], 0), V - 1);
    tok_lp[row] = z[k] - mx - logf(s);
  }
}

// One thread per caption: the sum of its scored terms in position order; terms past them become 0, and a caption with a bad
// length or id gets NaN in every output.
__global__ void k_score_sum(ScoreArgs a) {
  pdl_launch();
  pdl_wait();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.caps) return;
  const int t = a.t;
  const int n = scored_positions(a.lens[c], t);
  const bool bad = a.bad[c] != 0;
  float* tl = a.tok_lp + (size_t)c * t;
  float s = 0.f;
  for (int j = 0; j < t; ++j) {
    if (bad) tl[j] = NAN;
    else if (j < n) s += tl[j];
    else tl[j] = 0.f;
  }
  a.lp[c] = bad ? NAN : s;
}

int launch_score_embed(const ScoreArgs& a, const float* emb, const float* pos, Act x, cudaStream_t s) {
  const size_t n = (size_t)a.caps * a.t * (x.C / 8);
  FPNMT_CUDA_OK(launch_k(k_score_embed, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, a, emb, pos, x));
  return 0;
}

int launch_score_self_attention(Act qkv, int caps, int t, int heads, Act out, cudaStream_t s) {
  const int rows = caps * t, warps = rows * heads;
  const dim3 grid((warps + SC_WARPS - 1) / SC_WARPS), block(SC_WARPS * 32);
  if (qkv.lo)
    FPNMT_CUDA_OK(launch_k(k_score_self_attention<true>, grid, block, 0, s, qkv, rows, t, heads, out));
  else
    FPNMT_CUDA_OK(launch_k(k_score_self_attention<false>, grid, block, 0, s, qkv, rows, t, heads, out));
  return 0;
}

int launch_score_rows(const float* logits, int rows, int V, const int* tgt, float* tok_lp, cudaStream_t s) {
  FPNMT_CUDA_OK(launch_k(k_score_rows, dim3(rows), dim3(SR_THREADS), 0, s, logits, V, tgt, tok_lp));
  return 0;
}

int launch_score_sum(const ScoreArgs& a, cudaStream_t s) {
  FPNMT_CUDA_OK(launch_k(k_score_sum, dim3((a.caps + 127) / 128), dim3(128), 0, s, a));
  return 0;
}

}  // namespace fpnmt
