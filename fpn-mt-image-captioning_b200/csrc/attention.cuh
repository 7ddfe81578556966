// Device helpers shared by the attention kernels (attention.cu) and the caption-scoring kernels (score.cu): head-dim-64
// row access, the cp.async wrapper and the warp-level online-softmax attention of one query.
#pragma once
#include "common.cuh"

namespace fpnmt {

constexpr int DH = 64;

// Load 64 contiguous channels [col, col+64) of one row into 64 floats spread as 2 per lane (lane*2, lane*2+1).
__device__ __forceinline__ float2 ld_pair(const Act& a, size_t row, int col, int lane) {
  const bf16* q = a.p + row * (size_t)a.ld + col + lane * 2;
  __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(q);
  float2 v = __bfloat1622float2(h);
  if (a.lo) {
    float2 l = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(q + a.lo));
    v.x += l.x;
    v.y += l.y;
  }
  return v;
}
__device__ __forceinline__ void st_pair(const Act& a, size_t row, int col, int lane, float x, float y) {
  bf16* q = a.p + row * (size_t)a.ld + col + lane * 2;
  __nv_bfloat162 h = __floats2bfloat162_rn(x, y);
  *reinterpret_cast<__nv_bfloat162*>(q) = h;
  if (a.lo) {
    float2 hf = __bfloat1622float2(h);
    *reinterpret_cast<__nv_bfloat162*>(q + a.lo) = __floats2bfloat162_rn(x - hf.x, y - hf.y);
  }
}
// Full 64-wide row segment into registers of ONE lane (used when a lane owns a key).
__device__ __forceinline__ void ld_row64(const Act& a, size_t row, int col, float* f) {
#pragma unroll
  for (int i = 0; i < 8; ++i) ld_act8(a, row, col + i * 8, f + i * 8);
}

__device__ __forceinline__ void cp16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}

// Warp-level attention of ONE query over Tk cached positions.  The query (pre-scaled) lives in shared memory
// (broadcast reads).  `krow(pos)` maps a position to the row of the K/V views.
// Value pass layout: lane = pg * 8 + dg owns output dims dg*8 .. dg*8+7 for the positions p = pg (mod 4).  The V rows of
// the 32-position chunk are copied into per-warp shared memory with cp.async (16 B units, consecutive lanes = consecutive
// units, so the global reads are 128 B row segments and the shared writes are conflict-free) WHILE the score pass still
// reads the K rows into registers: the two dependent DRAM round trips of the chunk (K, then V) become one.  The
// probabilities and cache rows of the chunk sit in per-warp shared arrays, and the four position groups are summed by
// two xor-shuffles at the end.
template <bool SPLIT>
struct __align__(16) WarpScratchT {
  uint4 v[(SPLIT ? 2 : 1) * 32 * 8];   // V rows of the current chunk: [hi | lo][position][8 x 16 B]
  float q[DH];                         // pre-scaled query
  unsigned row[32];                    // K/V rows of the current chunk
};

template <bool SPLIT>
__device__ __forceinline__ void v_stage_async(const Act& vc, int v_col, WarpScratchT<SPLIT>& ws, int kmax, int lane) {
  const uint32_t dst0 = (uint32_t)__cvta_generic_to_shared(ws.v);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int u = i * 32 + lane, r = u >> 3;
    const bool ok = r < kmax;
    const bf16* src = vc.p + (size_t)ws.row[ok ? r : 0] * vc.ld + v_col + (u & 7) * 8;
    cp16(dst0 + u * 16, src, ok);
    if constexpr (SPLIT) cp16(dst0 + (256 + u) * 16, src + vc.lo, ok);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

// Score and value pass share one mapping: lane = pg * 8 + dg handles the positions pp = pg (mod 4) of the chunk and the
// dims dg*8 .. dg*8+7.  Per load instruction a warp therefore covers 4 positions x 128 contiguous bytes (4 L1 wavefronts;
// the earlier "one key row per lane" layout touched 32 different lines per instruction and was bound by the L1 tag
// stage), the 8-dim partial dot products are summed over the 8 dg lanes with three xor-shuffles, and the probabilities
// stay in the registers of exactly the lanes that need them for the value pass.
template <bool SPLIT, typename RowFn>
__device__ __forceinline__ void warp_attend(WarpScratchT<SPLIT>& ws, const Act& kc, int k_col, const Act& vc, int v_col, int Tk,
                                            RowFn krow, int lane, float& m, float& l, float* o) {
  const int pg = lane >> 3, dg = lane & 7;
  float q8[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) q8[j] = ws.q[dg * 8 + j];
  for (int k0 = 0; k0 < Tk; k0 += 32) {
    const int pos = k0 + lane;
    const int kmax = min(32, Tk - k0);
    ws.row[lane] = (pos < Tk) ? (unsigned)krow(pos) : 0u;
    __syncwarp();
    v_stage_async<SPLIT>(vc, v_col, ws, kmax, lane);
    float sc[8];
    {
      uint4 kh[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int pp = pg + 4 * i;
        const bf16* src = kc.p + (size_t)ws.row[pp < kmax ? pp : 0] * kc.ld + k_col + dg * 8;
        kh[i] = *reinterpret_cast<const uint4*>(src);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float f[8];
        unpack8(kh[i], f);
        float a = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) a = fmaf(q8[j], f[j], a);
        sc[i] = a;
      }
      if constexpr (SPLIT) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int pp = pg + 4 * i;
          const bf16* src = kc.p + (size_t)ws.row[pp < kmax ? pp : 0] * kc.ld + k_col + dg * 8 + kc.lo;
          kh[i] = *reinterpret_cast<const uint4*>(src);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float f[8];
          unpack8(kh[i], f);
          float a = sc[i];
#pragma unroll
          for (int j = 0; j < 8; ++j) a = fmaf(q8[j], f[j], a);
          sc[i] = a;
        }
      }
    }
    float cmax = -INFINITY;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sc[i] += __shfl_xor_sync(0xffffffffu, sc[i], 1);
      sc[i] += __shfl_xor_sync(0xffffffffu, sc[i], 2);
      sc[i] += __shfl_xor_sync(0xffffffffu, sc[i], 4);
      if (pg + 4 * i >= kmax) sc[i] = -INFINITY;
      cmax = fmaxf(cmax, sc[i]);
    }
    cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, 8));
    cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, 16));
    const float mn = fmaxf(m, cmax);
    const float corr = __expf(m - mn);
    float psum = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sc[i] = (pg + 4 * i < kmax) ? __expf(sc[i] - mn) : 0.f;      // sc[] now holds the probabilities
      psum += sc[i];
    }
    psum += __shfl_xor_sync(0xffffffffu, psum, 8);
    psum += __shfl_xor_sync(0xffffffffu, psum, 16);
    l = l * corr + psum;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] *= corr;
    m = mn;
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int pp = pg + 4 * i;
      if (pp < kmax) {
        float f[8];
        unpack8(ws.v[pp * 8 + dg], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(sc[i], f[j], o[j]);
        if constexpr (SPLIT) {
          unpack8(ws.v[256 + pp * 8 + dg], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = fmaf(sc[i], f[j], o[j]);
        }
      }
    }
    __syncwarp();
  }
}

// sum the four position groups; afterwards lanes 0..7 hold dims lane*8 .. lane*8+7
__device__ __forceinline__ void pv_reduce(float* o) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    o[i] += __shfl_xor_sync(0xffffffffu, o[i], 8);
    o[i] += __shfl_xor_sync(0xffffffffu, o[i], 16);
  }
}

}  // namespace fpnmt
