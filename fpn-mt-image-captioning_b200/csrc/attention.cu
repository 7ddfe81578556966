// Attention kernels (CUDA cores; head dim 64).  All softmax arithmetic in fp32.
//   enc_attention       : 16 baseline queries vs. a static pyramid view (Tk in {1024,256,64,4}), flash-style
//                         single pass with online softmax; one block per (image, head), 4 queries per warp.
//   dec_self_attention  : one new query per (row, head) against the KV cache through the beam-ancestry table.
//   dec_cross_attention : one query per (row, head) against the 16 memory tokens of the row's image.
//   dec_attention_probs : the normalised probabilities of both for the beam-0 rows (inspection, teacher forcing).
#include <stdlib.h>

#include <algorithm>

#include "attention.cuh"
#include "kernels.cuh"
#include "xattn.cuh"

namespace fpnmt {

#define LAUNCH_CHECK() FPNMT_CUDA_OK(cudaGetLastError())

// ---------------------------------------------------------------------------------------- encoder
// block = 128 threads = 4 warps; warp w handles queries 4w..4w+3 of the 16; lanes own keys in chunks of 32
// for the score pass and own 2 output dims for the value pass.
__global__ void __launch_bounds__(128) k_enc_attention(Act q, int q_col, Act kv, int k_col, int v_col, int Tq, int Tk,
                                                       Act out, int out_col) {
  pdl_launch();
  pdl_wait();
  __shared__ float sq[16][DH];
  const int b = blockIdx.x, h = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float scale = 0.125f;   // 1/sqrt(64)
  for (int i = threadIdx.x; i < Tq * DH; i += blockDim.x) {
    const int qi = i / DH, d = i % DH;
    sq[qi][d] = ld_act(q, (size_t)b * Tq + qi, q_col + h * DH + d) * scale;
  }
  __syncthreads();
  constexpr int QW = 4;
  float m[QW], l[QW], o0[QW], o1[QW];
#pragma unroll
  for (int i = 0; i < QW; ++i) { m[i] = -INFINITY; l[i] = 0.f; o0[i] = 0.f; o1[i] = 0.f; }
  for (int k0 = 0; k0 < Tk; k0 += 32) {
    const int key = k0 + lane;
    float sc[QW];
#pragma unroll
    for (int i = 0; i < QW; ++i) sc[i] = -INFINITY;
    if (key < Tk) {
      float kr[DH];
      ld_row64(kv, (size_t)b * Tk + key, k_col + h * DH, kr);
#pragma unroll
      for (int i = 0; i < QW; ++i) {
        float a = 0.f;
#pragma unroll
        for (int d = 0; d < DH; ++d) a = fmaf(sq[warp * QW + i][d], kr[d], a);
        sc[i] = a;
      }
    }
    float p[QW];
#pragma unroll
    for (int i = 0; i < QW; ++i) {
      const float mn = fmaxf(m[i], warp_max(sc[i]));
      const float corr = __expf(m[i] - mn);
      p[i] = (key < Tk) ? __expf(sc[i] - mn) : 0.f;
      l[i] = l[i] * corr + warp_sum(p[i]);
      o0[i] *= corr;
      o1[i] *= corr;
      m[i] = mn;
    }
    const int kmax = min(32, Tk - k0);
    for (int j = 0; j < kmax; ++j) {
      const float2 v = ld_pair(kv, (size_t)b * Tk + k0 + j, v_col + h * DH, lane);
#pragma unroll
      for (int i = 0; i < QW; ++i) {
        const float pj = __shfl_sync(0xffffffffu, p[i], j);
        o0[i] = fmaf(pj, v.x, o0[i]);
        o1[i] = fmaf(pj, v.y, o1[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < QW; ++i) {
    const int qi = warp * QW + i;
    if (qi < Tq) {
      const float inv = 1.f / l[i];
      st_pair(out, (size_t)b * Tq + qi, out_col + h * DH, lane, o0[i] * inv, o1[i] * inv);
    }
  }
}
// ---------------------------------------------------------------------------------------- encoder, tensor-core path
// bf16 mode.  One block (4 warps) per (image, head): the <= 16 baseline queries form exactly one m16 MMA row block, so
// S = Q K^T and O = P V run on mma.sync.m16n8k16 (bf16 in, fp32 accumulate) flash-style: each warp walks the key axis
// in tiles of 64 keys (its K and V tiles staged in swizzled shared memory by 16-byte cp.async, fragments read with
// ldmatrix / ldmatrix.trans), keeps online-softmax statistics in registers, and the four warps' partial (m, l, O) are
// merged through shared memory at the end.  (tcgen05 needs M >= 64 rows per tile; 16 queries per head do not fill it.)
__device__ __forceinline__ void mma_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}

constexpr int EA_WARPS = 4;
constexpr int EA_TILE = 64;                       // keys per tile
constexpr int EA_TILE_BYTES = EA_TILE * DH * 2;   // 8 KB
constexpr int EA_SMEM = EA_WARPS * 2 * EA_TILE_BYTES + EA_WARPS * 16 * 2 * 4;

// blockIdx.z selects the pyramid view: all (up to 4) cross-level attentions of an encoder layer run as ONE launch, the
// long view first (z = 0), so the short ones fill the tail instead of paying a launch each.
struct EncAttViews {
  Act kv[4];
  int Tk[4];
  int col[4];      // query / output column block of the view
};
__global__ void __launch_bounds__(EA_WARPS * 32) k_enc_attention_mma(Act q, EncAttViews views, int k_col, int v_col, int Tq,
                                                                    Act out) {
  extern __shared__ __align__(128) uint8_t ea_smem[];
  pdl_launch();
  pdl_wait();
  const int b = blockIdx.x, h = blockIdx.y;
  const Act kv = views.kv[blockIdx.z];
  const int Tk = views.Tk[blockIdx.z];
  const int q_col = views.col[blockIdx.z], out_col = q_col;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  uint8_t* sK = ea_smem + warp * 2 * EA_TILE_BYTES;
  uint8_t* sV = sK + EA_TILE_BYTES;
  float* sM = reinterpret_cast<float*>(ea_smem + EA_WARPS * 2 * EA_TILE_BYTES);   // [EA_WARPS][16]
  float* sL = sM + EA_WARPS * 16;
  const uint32_t sK_u = smem_u32(sK), sV_u = smem_u32(sV);

  // Q fragments (rows g and g+8 of the 16-query block; 4 k-steps of 16 dims)
  uint32_t qa[4][4];
  {
    const bf16* q0 = q.p + (size_t)(b * Tq + g) * q.ld + q_col + h * DH;
    const bf16* q1 = q0 + (size_t)8 * q.ld;
    const bool ok0 = g < Tq, ok1 = g + 8 < Tq;
#pragma unroll
    for (int s4 = 0; s4 < 4; ++s4) {
      const int c = s4 * 16 + 2 * t;
      qa[s4][0] = ok0 ? *reinterpret_cast<const uint32_t*>(q0 + c) : 0u;
      qa[s4][1] = ok1 ? *reinterpret_cast<const uint32_t*>(q1 + c) : 0u;
      qa[s4][2] = ok0 ? *reinterpret_cast<const uint32_t*>(q0 + c + 8) : 0u;
      qa[s4][3] = ok1 ? *reinterpret_cast<const uint32_t*>(q1 + c + 8) : 0u;
    }
  }
  float o_acc[8][4];
#pragma unroll
  for (int d = 0; d < 8; ++d)
#pragma unroll
    for (int i = 0; i < 4; ++i) o_acc[d][i] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;      // rows g and g+8 (this thread's quad share)

  const int ntiles = (Tk + EA_TILE - 1) / EA_TILE;
  for (int tile = warp; tile < ntiles; tile += EA_WARPS) {
    const int key0 = tile * EA_TILE;
    // ---- stage K and V tiles: 64 keys x 8 chunks of 16 B each, chunk index swizzled with (key & 7)
#pragma unroll 4
    for (int it = 0; it < 16; ++it) {
      const int c = it * 32 + lane;
      const int key = c >> 3, ch = c & 7;
      const bool ok = key0 + key < Tk;
      const bf16* src = kv.p + (size_t)(b * Tk + (ok ? key0 + key : 0)) * kv.ld + h * DH + ch * 8;
      const uint32_t off = key * 128 + ((ch ^ (key & 7)) << 4);
      cp16(sK_u + off, src + k_col, ok);
      cp16(sV_u + off, src + v_col, ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    // ---- S = Q K^T for the 64 keys (8 n-tiles of 8 keys)
    float s_acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
      for (int i = 0; i < 4; ++i) s_acc[j][i] = 0.f;
      const int key = 8 * j + (lane & 7);
#pragma unroll
      for (int sp = 0; sp < 2; ++sp) {              // two k-steps (32 dims) per ldmatrix.x4
        uint32_t kb[4];
        const int ch = 4 * sp + (lane >> 3);
        ldsm_x4(kb, sK_u + key * 128 + ((ch ^ (key & 7)) << 4));
        mma_16816(s_acc[j], qa[2 * sp], kb[0], kb[1]);
        mma_16816(s_acc[j], qa[2 * sp + 1], kb[2], kb[3]);
      }
    }
    // ---- online softmax (scale 1/sqrt(64)); keys beyond Tk are masked
    float tm0 = -INFINITY, tm1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int kk = key0 + 8 * j + 2 * t;
      s_acc[j][0] = kk < Tk ? s_acc[j][0] * 0.125f : -INFINITY;
      s_acc[j][1] = kk + 1 < Tk ? s_acc[j][1] * 0.125f : -INFINITY;
      s_acc[j][2] = kk < Tk ? s_acc[j][2] * 0.125f : -INFINITY;
      s_acc[j][3] = kk + 1 < Tk ? s_acc[j][3] * 0.125f : -INFINITY;
      tm0 = fmaxf(tm0, fmaxf(s_acc[j][0], s_acc[j][1]));
      tm1 = fmaxf(tm1, fmaxf(s_acc[j][2], s_acc[j][3]));
    }
    tm0 = fmaxf(tm0, __shfl_xor_sync(0xffffffffu, tm0, 1));
    tm0 = fmaxf(tm0, __shfl_xor_sync(0xffffffffu, tm0, 2));
    tm1 = fmaxf(tm1, __shfl_xor_sync(0xffffffffu, tm1, 1));
    tm1 = fmaxf(tm1, __shfl_xor_sync(0xffffffffu, tm1, 2));
    const float n0 = fmaxf(m0, tm0), n1 = fmaxf(m1, tm1);
    const float c0 = __expf(m0 - n0), c1 = __expf(m1 - n1);
    m0 = n0;
    m1 = n1;
    float ps0 = 0.f, ps1 = 0.f;
    uint32_t pa[4][4];                               // P as A fragments: k-step kk covers keys 16kk .. 16kk+15
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float p0 = __expf(s_acc[j][0] - n0), p1 = __expf(s_acc[j][1] - n0);
      const float p2 = __expf(s_acc[j][2] - n1), p3 = __expf(s_acc[j][3] - n1);
      ps0 += p0 + p1;
      ps1 += p2 + p3;
      pa[j >> 1][(j & 1) * 2] = pack2(p0, p1);       // a0 / a2: row g
      pa[j >> 1][(j & 1) * 2 + 1] = pack2(p2, p3);   // a1 / a3: row g+8
    }
    l0 = l0 * c0 + ps0;
    l1 = l1 * c1 + ps1;
#pragma unroll
    for (int d = 0; d < 8; ++d) {
      o_acc[d][0] *= c0;
      o_acc[d][1] *= c0;
      o_acc[d][2] *= c1;
      o_acc[d][3] *= c1;
    }
    // ---- O += P V
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {              // two 8-dim n-tiles per ldmatrix.x4.trans
        uint32_t vb[4];
        const int mi = lane >> 3;
        const int key = 16 * kk + (mi & 1) * 8 + (lane & 7);
        const int ch = 2 * dp + (mi >> 1);
        ldsm_x4_t(vb, sV_u + key * 128 + ((ch ^ (key & 7)) << 4));
        mma_16816(o_acc[2 * dp], pa[kk], vb[0], vb[1]);
        mma_16816(o_acc[2 * dp + 1], pa[kk], vb[2], vb[3]);
      }
    }
    __syncwarp();
  }
  // ---- merge the four warps: quad-reduce l, publish (m, l) and O, then every thread finishes 8 output values
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  __syncthreads();                                   // all tiles consumed: the K/V area becomes the O exchange buffer
  float* sO = reinterpret_cast<float*>(ea_smem);     // [EA_WARPS][16][64]
  if (t == 0) {
    sM[warp * 16 + g] = m0;
    sM[warp * 16 + g + 8] = m1;
    sL[warp * 16 + g] = l0;
    sL[warp * 16 + g + 8] = l1;
  }
#pragma unroll
  for (int d = 0; d < 8; ++d) {
    float* r0 = sO + (warp * 16 + g) * DH + 8 * d + 2 * t;
    float* r1 = sO + (warp * 16 + g + 8) * DH + 8 * d + 2 * t;
    r0[0] = o_acc[d][0];
    r0[1] = o_acc[d][1];
    r1[0] = o_acc[d][2];
    r1[1] = o_acc[d][3];
  }
  __syncthreads();
  {
    const int row = threadIdx.x >> 3, d0 = (threadIdx.x & 7) * 8;
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < EA_WARPS; ++w) M = fmaxf(M, sM[w * 16 + row]);
    float L = 0.f, o[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int w = 0; w < EA_WARPS; ++w) {
      const float mw = sM[w * 16 + row];
      const float sc = (mw == -INFINITY) ? 0.f : __expf(mw - M);
      L += sL[w * 16 + row] * sc;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = fmaf(sO[(w * 16 + row) * DH + d0 + i], sc, o[i]);
    }
    if (row < Tq) {
      const float inv = 1.f / L;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] *= inv;
      st_act8(out, (size_t)b * Tq + row, out_col + h * DH + d0, o);
    }
  }
}

// Function attributes are per device: called from Engine::init for every device an engine is created on.
int dec_attention_set_attributes();   // defined next to k_dec_self_attention_mma below
int attention_set_attributes() {
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_enc_attention_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, EA_SMEM));
  return dec_attention_set_attributes();
}

int launch_enc_attention(Act q, int q_col, Act kv, int k_col, int v_col, int B, int Tq, int Tk, int heads, Act out,
                         int out_col, bool force_simt, cudaStream_t s) {
  if (Tq > 16) {
    set_last_error("enc_attention: Tq must be <= 16");
    return 1;
  }
  dim3 grid(B, heads);
  if (!kv.lo && !q.lo && !out.lo && !force_simt) {   // bf16 mode: tensor-core flash kernel
    if (q_col != out_col) {
      set_last_error("enc_attention: the tensor-core path writes the output at the query's column block");
      return 1;
    }
    EncAttViews views{};
    views.kv[0] = kv;
    views.Tk[0] = Tk;
    views.col[0] = q_col;
    FPNMT_CUDA_OK(launch_k(k_enc_attention_mma, dim3(grid), dim3(EA_WARPS * 32), (size_t)EA_SMEM, s, q, views, k_col, v_col, Tq, out));
    return 0;
  }
  FPNMT_CUDA_OK(launch_k(k_enc_attention, dim3(grid), dim3(128), 0, s, q, q_col, kv, k_col, v_col, Tq, Tk, out, out_col));
  LAUNCH_CHECK();
  return 0;
}

// All views of one encoder layer in a single launch (bf16 tensor-core path only; view v reads the query columns
// [col[v], col[v]+heads*64) and writes its output there).
int launch_enc_attention_views(Act q, const Act* kvs, const int* tks, const int* cols, int nviews, int k_col, int v_col, int B,
                               int Tq, int heads, Act out, cudaStream_t s) {
  if (Tq > 16 || nviews < 1 || nviews > 4 || q.lo || out.lo) {
    set_last_error("enc_attention_views: Tq <= 16, 1..4 views, plain bf16 activations");
    return 1;
  }
  EncAttViews views{};
  for (int v = 0; v < nviews; ++v) {
    if (kvs[v].lo) {
      set_last_error("enc_attention_views: plain bf16 K/V");
      return 1;
    }
    views.kv[v] = kvs[v];
    views.Tk[v] = tks[v];
    views.col[v] = cols[v];
  }
  FPNMT_CUDA_OK(launch_k(k_enc_attention_mma, dim3(B, heads, nviews), dim3(EA_WARPS * 32), (size_t)EA_SMEM, s, q, views, k_col, v_col,
                         Tq, out));
  return 0;
}

// ---------------------------------------------------------------------------------------- decoder attention

constexpr int DEC_WARPS = 4;

// one warp per (row, head).  Position t = *step is the new token: its K/V come from `qkv` and are appended to the
// cache at [row][t]; positions t' < t are read from cache row anc[row][t'] (the beam's ancestor at that time).
template <bool SPLIT>
__global__ void __launch_bounds__(DEC_WARPS * 32, SPLIT ? 4 : 8) k_dec_self_attention(Act qkv, Act kc0, Act vc0, Act kc1, Act vc1,
                                                                       const int* __restrict__ anc_base, size_t anc_stride,
                                                                       const int* __restrict__ step, int rows, int T,
                                                                       int heads, Act out) {
  __shared__ WarpScratchT<SPLIT> s_ws[DEC_WARPS];
  pdl_launch();
  pdl_wait();
  const int gw = blockIdx.x * DEC_WARPS + (threadIdx.x >> 5);
  if (gw >= rows * heads) return;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  WarpScratchT<SPLIT>& ws = s_ws[w];
  const int row = gw / heads, h = gw % heads;
  const int d = heads * DH;
  // The ancestry entries of the first 64 positions are fetched for BOTH parities of the double-buffered table together
  // with the step counter, so the address of the K/V rows is one memory round trip away instead of two.
  const int* anc_e = anc_base + (size_t)row * T;
  const int* anc_o = anc_e + anc_stride;
  int a_e[2], a_o[2];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int pos = c * 32 + lane;
    a_e[c] = pos < T ? __ldg(anc_e + pos) : 0;
    a_o[c] = pos < T ? __ldg(anc_o + pos) : 0;
  }
  const int t = *step;
  const bool second = kc1.p != nullptr && (t & 1);      // physical cache mode: odd steps live in the second buffer pair
  const Act kc = second ? kc1 : kc0, vc = second ? vc1 : vc0;
  const int* anc = (t & 1) ? anc_o : anc_e;
  const int a0 = (t & 1) ? a_o[0] : a_e[0], a1 = (t & 1) ? a_o[1] : a_e[1];
  const float2 qv = ld_pair(qkv, row, h * DH, lane);
  const float2 kn = ld_pair(qkv, row, d + h * DH, lane);
  const float2 vn = ld_pair(qkv, row, 2 * d + h * DH, lane);
  ws.q[lane * 2] = qv.x * 0.125f;       // 1/sqrt(64)
  ws.q[lane * 2 + 1] = qv.y * 0.125f;
  st_pair(kc, (size_t)row * T + t, h * DH, lane, kn.x, kn.y);     // append the new K/V to the cache
  st_pair(vc, (size_t)row * T + t, h * DH, lane, vn.x, vn.y);
  __syncwarp();
  float m = -INFINITY, l = 0.f, o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i] = 0.f;
  warp_attend<SPLIT>(ws, kc, h * DH, vc, h * DH, t,
                     [&](int pos) { return (size_t)(pos < 32 ? a0 : pos < 64 ? a1 : anc[pos]) * T + pos; }, lane, m, l, o);
  pv_reduce(o);
  {   // the new position itself (K/V still in registers): fold it in on lanes 0..7
    const float sc = warp_sum((qv.x * kn.x + qv.y * kn.y) * 0.125f);
    const float mn = fmaxf(m, sc);
    const float corr = __expf(m - mn);
    const float p = __expf(sc - mn);
    l = l * corr + p;
    // v_new dims lane*8 .. +7 live on lanes 4*lane .. 4*lane+3 (2 dims each)
    float vnew[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      vnew[2 * i] = __shfl_sync(0xffffffffu, vn.x, (lane & 7) * 4 + i);
      vnew[2 * i + 1] = __shfl_sync(0xffffffffu, vn.y, (lane & 7) * 4 + i);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = o[i] * corr + p * vnew[i];
  }
  if (lane < 8) {
    const float inv = 1.f / l;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] *= inv;
    st_act8(out, (size_t)row, h * DH + lane * 8, o);
  }
}
static bool g_dec_att_simt = false;   // FPNMT_OPT_DEC_ATT_SIMT: CUDA-core decode self-attention in bf16 mode too
void set_dec_att_simt(bool v) { g_dec_att_simt = v; }

// ---- bf16 mode: the same attention on mma.sync.m16n8k16 ---------------------------------------------------------------
// The CUDA-core kernel above is bound by instruction issue, not by HBM (ncu at t = 40: 1 800 instructions per warp, issue
// slots 55 % busy, DRAM 42 %): per cached position a lane unpacks and multiplies 16 values and takes part in 3 shuffles.
// Here a warp still owns one (row, head), but the arithmetic is two small tensor-core products per 32-position chunk:
//   S^T = K_chunk[32 x 64] . q[64]      A = K rows from shared memory (ldmatrix), B = the query in column 0 of an n8 tile
//   o   = p[32] . V_chunk[32 x 64]      A = the probabilities in row 0 of an m16 tile (bf16 hi + lo parts: two MMAs, so the
//                                       probabilities keep ~16 mantissa bits), B = V rows (ldmatrix.trans)
// 7/8 of each MMA is padding - the tensor pipe is idle in this kernel anyway; what matters is ~4x fewer issued instructions.
// K and V rows of the chunk are staged with cp.async into a 128-byte-row XOR-swizzled tile (conflict-free for both the
// 16-byte copies and ldmatrix); the new position's K/V (from the QKV projection) is written into the tile directly and
// appended to the cache.  Online softmax across chunks as before.
struct __align__(128) DecAttTile {
  uint4 k[32 * 8];
  uint4 v[32 * 8];
};

// Launch shape: 8 KB of staging per warp limits an SM to 27 warps with 4-warp CTAs (6 CTAs x (32 + 1) KB), i.e. 3 552 resident
// warps for the 4 096 (row, head) pairs of C2 - ncu: 1.15 waves.  With 14 warps per CTA two CTAs fit an SM (2 x 113 KB):
// 28 warps per SM, 293 CTAs <= 296 slots, one wave.
//
// Round 2, token-history classes: beams of an image with the same token history (BeamState::rep; under the reference's beam
// initialisation ALL beams of an image, pipeline.py:101-102) read the same cache rows - so the warp of the class representative
// computes the attention of every member at once, flash-attention style with the MEMBERS as the MMA rows:
//   S[member][pos] = Q[member][:] . K[pos][:]     A = the members' queries (m16: up to 8 members + padding), B = K rows (ldmatrix)
//   O[member][:]  += P[member][pos] . V[pos][:]    A = P straight from the S accumulator layout (bf16 hi + lo), B = V (ldmatrix.trans)
// - the instruction count of ONE row serves the whole class (the old layout used 1 of 16 MMA rows and 1 of 8 columns), every
// member's row is still computed and written, and the warps of the other members only append their K/V and leave.  Warps are
// ordered beam-major, so with one class per image whole CTAs of non-representatives retire at once.  Without `rep` (teacher
// forcing, true beams that have diverged) every row is its own class: one member per warp, as before.
constexpr int DEC_MMA_WARPS = 14;
__global__ void __launch_bounds__(DEC_MMA_WARPS * 32, 2) k_dec_self_attention_mma(Act qkv, Act kc0, Act vc0, Act kc1, Act vc1,
                                                                              const int* __restrict__ anc_base, size_t anc_stride,
                                                                              const int* __restrict__ step, const int* __restrict__ rep_e,
                                                                              const int* __restrict__ rep_o, int rows, int T,
                                                                              int heads, int N, Act out) {
  extern __shared__ __align__(128) uint8_t s_tile_raw[];
  DecAttTile* s_tile = reinterpret_cast<DecAttTile*>(s_tile_raw);
  pdl_launch();
  pdl_wait();
  const int gw = blockIdx.x * DEC_MMA_WARPS + (threadIdx.x >> 5);
  if (gw >= rows * heads) return;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int per_beam = (rows / N) * heads;               // beam-major warp order: gw = n * (B * heads) + b * heads + h
  const int n_beam = gw / per_beam, bh = gw % per_beam;
  const int b = bh / heads, h = bh % heads;
  const int row = b * N + n_beam;
  const int d = heads * DH;
  const int g = lane >> 2, tq = lane & 3;
  const uint32_t sK = smem_u32(s_tile[w].k), sV = smem_u32(s_tile[w].v);
  const int* anc_e = anc_base + (size_t)row * T;
  const int* anc_o = anc_e + anc_stride;
  int a_e[2], a_o[2];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int pos = c * 32 + lane;
    a_e[c] = pos < T ? __ldg(anc_e + pos) : 0;
    a_o[c] = pos < T ? __ldg(anc_o + pos) : 0;
  }
  // representative rows of this image's beams for both step parities (the parity is known once `step` has arrived)
  int r_e = b * N + lane, r_o = b * N + lane;
  if (rep_e && lane < N) {
    r_e = rep_e[b * N + lane];
    r_o = rep_o[b * N + lane];
  }
  const int t = *step;
  const bool second = kc1.p != nullptr && (t & 1);      // physical cache mode: odd steps live in the second buffer pair
  const Act kc = second ? kc1 : kc0, vc = second ? vc1 : vc0;
  const int* anc = (t & 1) ? anc_o : anc_e;
  const int a0 = (t & 1) ? a_o[0] : a_e[0], a1 = (t & 1) ? a_o[1] : a_e[1];
  const int r_l = (t & 1) ? r_o : r_e;                   // lane l < N: representative row of beam l
  const int my_rep = __shfl_sync(0xffffffffu, r_l, n_beam);
  const bf16* qrow = qkv.p + (size_t)row * qkv.ld + h * DH;
  const uint32_t knew = *reinterpret_cast<const uint32_t*>(qrow + d + 2 * lane);
  const uint32_t vnew = *reinterpret_cast<const uint32_t*>(qrow + 2 * d + 2 * lane);
  *reinterpret_cast<uint32_t*>(kc.p + ((size_t)row * T + t) * kc.ld + h * DH + 2 * lane) = knew;     // every row appends its own K/V
  *reinterpret_cast<uint32_t*>(vc.p + ((size_t)row * T + t) * vc.ld + h * DH + 2 * lane) = vnew;
  if (my_rep != row) return;                             // a member of another beam's class: that beam's warp computes this row
  const unsigned members = __ballot_sync(0xffffffffu, lane < N && r_l == row);
  const int nm = __popc(members);
  // MMA row g = g-th member of the class (rows >= nm are padding)
  const int mrow = g < nm ? b * N + (int)__fns(members, 0, g + 1) : row;
  uint32_t qa[4][4];
  {
    const bf16* q0 = qkv.p + (size_t)mrow * qkv.ld + h * DH;
    const bool ok0 = g < nm;
#pragma unroll
    for (int s4 = 0; s4 < 4; ++s4) {
      const int c = s4 * 16 + 2 * tq;
      qa[s4][0] = ok0 ? *reinterpret_cast<const uint32_t*>(q0 + c) : 0u;
      qa[s4][1] = 0u;
      qa[s4][2] = ok0 ? *reinterpret_cast<const uint32_t*>(q0 + c + 8) : 0u;
      qa[s4][3] = 0u;
    }
  }
  float m = -INFINITY, l = 0.f;                          // row g of the class (this thread's quad share)
  float o[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
  const int Tk = t + 1;                                  // cached positions 0..t-1 and the new one
  for (int k0 = 0; k0 < Tk; k0 += 32) {
    const int kmax = min(32, Tk - k0);
    const int pos = k0 + lane;
    const unsigned my_row = pos < t ? (unsigned)((size_t)(pos < 32 ? a0 : pos < 64 ? a1 : anc[pos]) * T + pos) : 0u;
    // ---- stage the chunk: lane -> (position 4i + lane/8, 16-byte unit lane%8); rows past the new position are zero-filled
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int pp = 4 * i + (lane >> 3), u = lane & 7;
      const unsigned r = __shfl_sync(0xffffffffu, my_row, pp);
      const int gp = k0 + pp;
      const uint32_t off = (uint32_t)(pp * 128 + ((u ^ (pp & 7)) << 4));
      if (gp != t) {
        cp16(sK + off, kc.p + (size_t)r * kc.ld + h * DH + u * 8, gp < t);
        cp16(sV + off, vc.p + (size_t)r * vc.ld + h * DH + u * 8, gp < t);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (t >= k0 && t < k0 + 32) {                        // the new position: straight from the registers
      const int pn = t - k0;
      const uint32_t off = (uint32_t)(pn * 128 + (((lane >> 2) ^ (pn & 7)) << 4) + (lane & 3) * 4);
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sK + off), "r"(knew) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sV + off), "r"(vnew) : "memory");
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    // ---- S = Q K^T for the 32 positions (4 n-tiles of 8)
    float sa[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      sa[j][0] = sa[j][1] = sa[j][2] = sa[j][3] = 0.f;
      if (8 * j < kmax) {
        const int key = 8 * j + (lane & 7);
#pragma unroll
        for (int sp = 0; sp < 2; ++sp) {                 // two k-steps (32 dims) per ldmatrix.x4
          uint32_t kb[4];
          const int ch = 4 * sp + (lane >> 3);
          ldsm_x4(kb, sK + (uint32_t)(key * 128 + ((ch ^ (key & 7)) << 4)));
          mma_16816(sa[j], qa[2 * sp], kb[0], kb[1]);
          mma_16816(sa[j], qa[2 * sp + 1], kb[2], kb[3]);
        }
      }
    }
    // ---- online softmax of row g (scale 1/sqrt(64)); positions beyond the new one are masked
    float tm = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int kk = 8 * j + 2 * tq;
      sa[j][0] = kk < kmax ? sa[j][0] * 0.125f : -INFINITY;
      sa[j][1] = kk + 1 < kmax ? sa[j][1] * 0.125f : -INFINITY;
      tm = fmaxf(tm, fmaxf(sa[j][0], sa[j][1]));
    }
    tm = fmaxf(tm, __shfl_xor_sync(0xffffffffu, tm, 1));
    tm = fmaxf(tm, __shfl_xor_sync(0xffffffffu, tm, 2));
    const float mn = fmaxf(m, tm);
    const float corr = __expf(m - mn);
    m = mn;
    float ps = 0.f;
    uint32_t ah[2][4], al[2][4];                         // P as A fragments (bf16 hi + lo parts): k-step kt = positions 16kt..16kt+15
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float p0 = __expf(sa[j][0] - mn), p1 = __expf(sa[j][1] - mn);   // exp(-inf) = 0 for the masked entries
      ps += p0 + p1;
      const __nv_bfloat162 hh = __floats2bfloat162_rn(p0, p1);
      const float2 hf = __bfloat1622float2(hh);
      const __nv_bfloat162 ll = __floats2bfloat162_rn(p0 - hf.x, p1 - hf.y);
      ah[j >> 1][(j & 1) * 2] = *reinterpret_cast<const uint32_t*>(&hh);      // a0 / a2: row g
      al[j >> 1][(j & 1) * 2] = *reinterpret_cast<const uint32_t*>(&ll);
      ah[j >> 1][(j & 1) * 2 + 1] = 0u;                                        // a1 / a3: row g + 8 (padding)
      al[j >> 1][(j & 1) * 2 + 1] = 0u;
    }
    l = l * corr + ps;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      o[nb][0] *= corr;
      o[nb][1] *= corr;
    }
    // ---- O += P V
#pragma unroll
    for (int kt = 0; kt < 2; ++kt) {
      if (kt * 16 < kmax) {
        const int r = kt * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          uint32_t bq[4];
          ldsm_x4_t(bq, sV + (uint32_t)(r * 128 + (((np * 2 + (lane >> 4)) ^ (r & 7)) << 4)));
          mma_16816(o[2 * np], ah[kt], bq[0], bq[1]);
          mma_16816(o[2 * np], al[kt], bq[0], bq[1]);
          mma_16816(o[2 * np + 1], ah[kt], bq[2], bq[3]);
          mma_16816(o[2 * np + 1], al[kt], bq[2], bq[3]);
        }
      }
    }
    __syncwarp();                                        // the tile is restaged by the next chunk
  }
  l += __shfl_xor_sync(0xffffffffu, l, 1);
  l += __shfl_xor_sync(0xffffffffu, l, 2);
  if (g < nm) {                                          // row g of the accumulators: dims nb*8 + 2*tq, +1 of member g
    const float inv = 1.f / l;
    bf16* orow = out.p + (size_t)mrow * out.ld + h * DH + 2 * tq;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const __nv_bfloat162 v2 = __floats2bfloat162_rn(o[nb][0] * inv, o[nb][1] * inv);
      *reinterpret_cast<__nv_bfloat162*>(orow + nb * 8) = v2;
    }
  }
}

int dec_attention_set_attributes() {
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_dec_self_attention_mma, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(DEC_MMA_WARPS * sizeof(DecAttTile))));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_dec_self_attention_mma, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return 0;
}

int launch_dec_self_attention(Act qkv, Act kcache, Act vcache, Act kcache2, Act vcache2, const int* anc, size_t anc_stride,
                              const int* step, int rows, int T, int heads, Act out, cudaStream_t s, const int* rep_e,
                              const int* rep_o, int N, DecAttKernel kernel) {
  const int warps = rows * heads;
  const bool plain = !kcache.lo && !qkv.lo && !out.lo;
  if (kernel == DEC_ATT_MMA && !plain) {
    set_last_error("dec_self_attention: the mma.sync kernel needs plain bf16 activations");
    return 1;
  }
  const bool simt = kernel == DEC_ATT_SIMT || (kernel == DEC_ATT_AUTO && g_dec_att_simt);
  if (kcache.lo)
    FPNMT_CUDA_OK(launch_k(k_dec_self_attention<true>, dim3((warps + DEC_WARPS - 1) / DEC_WARPS), dim3(DEC_WARPS * 32), 0, s,
                           qkv, kcache, vcache, kcache2, vcache2, anc, anc_stride, step, rows, T, heads, out));
  else if (!plain || simt)
    FPNMT_CUDA_OK(launch_k(k_dec_self_attention<false>, dim3((warps + DEC_WARPS - 1) / DEC_WARPS), dim3(DEC_WARPS * 32), 0, s,
                           qkv, kcache, vcache, kcache2, vcache2, anc, anc_stride, step, rows, T, heads, out));
  else {
    // The kernel finds beam n of image b at row b * N + n, so N must divide the rows; otherwise every row is its own image
    // and its own class (rep_e / rep_o index rows by that layout and would name representatives of other images).
    const int n = (N >= 1 && rows % N == 0) ? N : 1;
    const bool classes = n == N && N <= 8;
    FPNMT_CUDA_OK(launch_k(k_dec_self_attention_mma, dim3((warps + DEC_MMA_WARPS - 1) / DEC_MMA_WARPS), dim3(DEC_MMA_WARPS * 32),
                           DEC_MMA_WARPS * sizeof(DecAttTile), s,
                           qkv, kcache, vcache, kcache2, vcache2, anc, anc_stride, step, classes ? rep_e : nullptr,
                           classes ? rep_o : nullptr, rows, T, heads, n, out));
  }
  return 0;
}

template <bool SPLIT>
__global__ void __launch_bounds__(DEC_WARPS * 32, SPLIT ? 4 : 8) k_dec_cross_attention(Act q, Act kv, int k_col, int v_col, int rows,
                                                                        int beam, int Tk, int heads, Act out) {
  __shared__ WarpScratchT<SPLIT> s_ws[DEC_WARPS];
  pdl_launch();
  pdl_wait();
  const int gw = blockIdx.x * DEC_WARPS + (threadIdx.x >> 5);
  if (gw >= rows * heads) return;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  WarpScratchT<SPLIT>& ws = s_ws[w];
  const int row = gw / heads, h = gw % heads;
  const int img = row / beam;
  const float2 qv = ld_pair(q, row, h * DH, lane);
  ws.q[lane * 2] = qv.x * 0.125f;
  ws.q[lane * 2 + 1] = qv.y * 0.125f;
  __syncwarp();
  float m = -INFINITY, l = 0.f, o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i] = 0.f;
  warp_attend<SPLIT>(ws, kv, k_col + h * DH, kv, v_col + h * DH, Tk, [&](int pos) { return (size_t)img * Tk + pos; }, lane, m, l, o);
  pv_reduce(o);
  if (lane < 8) {
    const float inv = 1.f / l;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] *= inv;
    st_act8(out, (size_t)row, h * DH + lane * 8, o);
  }
}
int launch_dec_cross_attention(Act q, Act kv, int k_col, int v_col, int rows, int beam, int Tk, int heads, Act out,
                               cudaStream_t s) {
  const int warps = rows * heads;
  if (kv.lo)
    FPNMT_CUDA_OK(launch_k(k_dec_cross_attention<true>, dim3((warps + DEC_WARPS - 1) / DEC_WARPS), dim3(DEC_WARPS * 32), 0, s,
                           q, kv, k_col, v_col, rows, beam, Tk, heads, out));
  else
    FPNMT_CUDA_OK(launch_k(k_dec_cross_attention<false>, dim3((warps + DEC_WARPS - 1) / DEC_WARPS), dim3(DEC_WARPS * 32), 0, s,
                           q, kv, k_col, v_col, rows, beam, Tk, heads, out));
  return 0;
}

// ---- attention probabilities for inspection (Engine::decode_logits with attention outputs) ------------------------------
// Block (b, h, z): the beam-0 row b * N of image b; z = 0 the self-attention row t = *step of head h, z = 1 the cross-attention
// row.  Scores are recomputed from the operands the layer's attention kernels read, one warp per key position (lanes split
// the dot product), then normalised in fp32 over the block.  Runs after the layer's cross-attention block, when the new K of
// position t is in the cache and q2 / out1 are final.
__device__ __forceinline__ float dot_row(const float* x, const Act& a, size_t pix, int c0, int K, int lane) {
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc = fmaf(x[k], ld_act(a, pix, c0 + k), acc);
  return warp_sum(acc);
}

constexpr int DP_THREADS = 128;

__global__ void __launch_bounds__(DP_THREADS) k_dec_attention_probs(DecProbArgs a) {
  extern __shared__ float s_sc[];                     // [max(tlen, n_mem)] scores, then unnormalised probabilities
  __shared__ float s_x[512];                          // the query (64) or, on the fused path, the out1 row (512)
  __shared__ float s_red[DP_THREADS / 32];
  pdl_launch();
  pdl_wait();
  const int b = blockIdx.x, h = blockIdx.y, cross = blockIdx.z;
  float* out = cross ? a.cross_out : a.self_out;
  if (!out) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = DP_THREADS / 32;
  const int t = *a.step;
  const size_t row = (size_t)b * a.N;
  const bool folded = cross && a.Mt;
  const int kd = folded ? a.q.C : DH;
  const int n = cross ? a.n_mem : t + 1;
  if (folded)
    for (int k = threadIdx.x; k < kd; k += DP_THREADS) s_x[k] = ld_act(a.q, row, k);
  else
    for (int k = threadIdx.x; k < DH; k += DP_THREADS) s_x[k] = ld_act(cross ? a.q : a.qkv, row, h * DH + k) * 0.125f;   // 1/sqrt(64)
  __syncthreads();
  for (int j = warp; j < n; j += nw) {
    float s;
    if (!cross) {
      const int* anc = a.anc + (size_t)(t & 1) * a.anc_stride + row * a.T;
      s = dot_row(s_x, a.kc, (size_t)anc[j] * a.T + j, h * DH, DH, lane);
    } else if (folded) {
      const Act m{const_cast<bf16*>(a.Mt), kd, kd, 0};
      const size_t pair = (size_t)b * XA_PAIRS + h * 16 + j;    // (head, token) pairs padded to 16 tokens per head
      s = dot_row(s_x, m, pair, 0, kd, lane) + a.sbias[pair];
    } else {
      s = dot_row(s_x, a.kv, (size_t)b * a.n_mem + j, a.k_col + h * DH, DH, lane);
    }
    if (lane == 0) s_sc[j] = s;
  }
  __syncthreads();
  float m = -INFINITY;
  for (int j = threadIdx.x; j < n; j += DP_THREADS) m = fmaxf(m, s_sc[j]);
  m = warp_max(m);
  if (lane == 0) s_red[warp] = m;
  __syncthreads();
  m = s_red[0];
  for (int w = 1; w < nw; ++w) m = fmaxf(m, s_red[w]);
  __syncthreads();
  float l = 0.f;
  for (int j = threadIdx.x; j < n; j += DP_THREADS) {
    const float e = expf(s_sc[j] - m);
    s_sc[j] = e;
    l += e;
  }
  l = warp_sum(l);
  if (lane == 0) s_red[warp] = l;
  __syncthreads();
  l = s_red[0];
  for (int w = 1; w < nw; ++w) l += s_red[w];
  const int width = cross ? a.n_mem : a.tlen;   // self rows are causal: exact zeros after position t
  float* dst = out + (((size_t)b * a.heads + h) * a.tlen + t) * width;
  for (int j = threadIdx.x; j < width; j += DP_THREADS) dst[j] = j < n ? s_sc[j] / l : 0.f;
}

int launch_dec_attention_probs(const DecProbArgs& a, int B, cudaStream_t s) {
  if (a.Mt && (a.q.C > 512 || a.n_mem > 16 || a.q.lo)) {
    set_last_error("dec_attention_probs: unsupported shape");
    return 1;
  }
  const size_t smem = (size_t)std::max(a.tlen, a.n_mem) * sizeof(float);
  FPNMT_CUDA_OK(launch_k(k_dec_attention_probs, dim3(B, a.heads, 2), dim3(DP_THREADS), smem, s, a));
  return 0;
}

}  // namespace fpnmt
