// Skinny-row Dense kernel (see tgemm.cuh): weights = tcgen05 A operand prefetched before the grid dependency,
// activations = B operand, accumulator D^T[feature][row] in TMEM, plain or cluster-LayerNorm epilogue.
//   warp 0     : TMA producer (one lane).  A ring: 8 x 16 KB weight chunks; B ring: 8 x (BN x 128 B) activation chunks.
//   warp 1     : TMEM allocator + MMA issuer (one lane): tcgen05.mma 128 x BN x 16, two accumulator buffers.
//   warps 2..5 : epilogue; warp w owns TMEM lanes 32*(w%4).. (features), each thread one feature x BN rows.
#include "tgemm.cuh"

#include <stdlib.h>

#include "tensormap.cuh"

namespace fpnmt {

constexpr int TG_A_BYTES = TG_BM * TG_BK * 2;          // 16 KB
constexpr int TG_LN_STRIDE = 132;                      // floats per row of the transposed scratch: 16-byte aligned rows with a
                                                       // 4-bank skew (feature-major writes and float4 row reads both conflict-free)
constexpr int TG_LN_BYTES = 32 * TG_LN_STRIDE * 4 + 128;

size_t tgemm_smem_bytes(int BN) {
  return (size_t)TG_A_SLOTS * TG_A_BYTES + (size_t)TG_B_STAGES * BN * TG_BK * 2 + TG_LN_BYTES + 4 * 32 * 8 /*partials*/ +
         32 * 8 /*cta stats*/ + 2 * TG_BM * 4 /*LayerNorm gamma, beta of the tile*/ + 512 /*barriers*/ + 1024 /*align slack*/;
}

__device__ __forceinline__ long long tg_timer() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float2 ld_dsmem_f2(const float2* local, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local)), "r"(rank));
  float2 v;
  asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(remote) : "memory");
  return v;
}

template <int BN>
__global__ void __launch_bounds__(TG_THREADS, 1)
tgemm_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX_hi,
             const __grid_constant__ CUtensorMap tmX_lo, const TgemmParams p) {
  constexpr int B_BYTES = BN * TG_BK * 2;
  constexpr int TMEM_COLS = 2 * BN;
  constexpr int CHUNKS = BN / 32;
  constexpr uint32_t IDESC = umma_idesc_bf16(TG_BM, BN);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = sA + TG_A_SLOTS * TG_A_BYTES;
  float* sLN = reinterpret_cast<float*>(sB + TG_B_STAGES * B_BYTES);
  float2* sPart = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(sLN) + TG_LN_BYTES);   // [4][32] (mean, M2)
  float2* sStat = sPart + 4 * 32;                                                            // [32] CTA-level (mean, M2)
  float* sGB = reinterpret_cast<float*>(sStat + 32);                                         // [2][128] gamma, beta of this feature tile
  uint64_t* bars = reinterpret_cast<uint64_t*>(sGB + 2 * TG_BM);
  uint64_t* fullA = bars;                          // [8]
  uint64_t* emptyA = bars + TG_A_SLOTS;            // [8]
  uint64_t* fullB = bars + 2 * TG_A_SLOTS;         // [8]
  uint64_t* emptyB = fullB + TG_B_STAGES;          // [8]
  uint64_t* tfull = emptyB + TG_B_STAGES;          // [2]
  uint64_t* tempty = tfull + 2;                    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool is_ln = p.gamma != nullptr;

  const int item = blockIdx.x;
  const int ftile = item % p.ftiles;                 // the ftiles CTAs of a row group form the LayerNorm cluster
  const int rgroup = item / p.ftiles;
  const int rt0 = rgroup * p.rt_per_item;
  const int rt1 = min(p.rtiles, rt0 + p.rt_per_item);
  const int kiters = p.nterms * p.kchunks;

#ifdef FPNMT_DBG_STAMPS   // build.py --dbg-stamps: globaltimer timeline of block 0 (FPNMT_DBG_OP=<op name>); off in product builds
  __shared__ long long* s_dbg;
  if (threadIdx.x == 0) {
    s_dbg = nullptr;
    if (p.dbg && blockIdx.x == 0) {
      const long long inst = (long long)atomicAdd((unsigned long long*)p.dbg, 1ull);
      s_dbg = p.dbg + 16 + (inst % 8) * 16;
      s_dbg[0] = tg_timer();
    }
  }
#define DBG(k) do { if (s_dbg) s_dbg[k] = tg_timer(); } while (0)
#else
#define DBG(k) do { } while (0)
#endif
  pdl_launch();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmX_hi);
    if (p.nterms > 1) tma_prefetch_desc(&tmX_lo);
    for (int s = 0; s < TG_A_SLOTS; ++s) {         // (only the first TG_A_SLOTS / 4 of each are used: one per group)
      mbar_init(&fullA[s], 1);
      mbar_init(&emptyA[s], 1);
    }
    for (int s = 0; s < TG_B_STAGES; ++s) {
      mbar_init(&fullB[s], 1);
      mbar_init(&emptyB[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) DBG(1);

  // The k-chunks move through the pipeline in GROUPS of 4 (one mbarrier per group and operand): the TMA producer and the
  // MMA issuer are single threads whose mbarrier instructions (~90 cycles each, even when already complete) sit on the
  // critical path of a latency-bound kernel, so one wait / one commit per 16 tcgen05.mma instead of per 4.
  constexpr int G = 4;                             // k-chunks per group
  constexpr int NG = TG_A_SLOTS / G;               // groups resident per operand (2)
  const int ngroups = (kiters + G - 1) / G;
  if (warp == 0) {
    // ---------------------------------------------------------------------------------- TMA producer
    // convergent warp, one elected lane issues (see umma_bf16_pred in common.cuh)
    const uint32_t leader = elect_one() ? 1u : 0u;
    {
      auto load_a_group = [&](int g, int slot) {   // chunks g*G .. of the weight panel -> A slots slot*G ..
        const int c0 = g * G, n = min(G, kiters - c0);
        mbar_expect_tx_pred(&fullA[slot], n * TG_A_BYTES, leader);
        int term = c0 / p.kchunks, kc = c0 % p.kchunks;
        for (int i = 0; i < n; ++i) {
          tma_load_2d_pred(sA + (slot * G + i) * TG_A_BYTES, &tmW, &fullA[slot], (term == 1 ? p.w_lo_off : 0) + kc * TG_BK, ftile * TG_BM, leader);
          if (++kc == p.kchunks) { kc = 0; ++term; }
        }
      };
      const int npre = ngroups < NG ? ngroups : NG;
      for (int g = 0; g < npre; ++g) load_a_group(g, g);   // static weights: issued before the grid dependency resolves
      pdl_wait();
      if (leader) DBG(2);
      int gA = 0, gB = 0;                          // groups issued so far
      for (int rt = rt0; rt < rt1; ++rt) {
        for (int g = 0; g < ngroups; ++g) {
          if (!p.stationary || rt == rt0) {
            if (gA >= npre) {
              const int slot = gA % NG;
              mbar_wait(&emptyA[slot], ((gA / NG) & 1) ^ 1);
              load_a_group(g, slot);
            }
            ++gA;
          }
          const int sb = gB % NG;
          if (gB >= NG) mbar_wait(&emptyB[sb], ((gB / NG) & 1) ^ 1);
          const int c0 = g * G, n = min(G, kiters - c0);
          mbar_expect_tx_pred(&fullB[sb], n * B_BYTES, leader);
          int term = c0 / p.kchunks, kc = c0 % p.kchunks;
          for (int i = 0; i < n; ++i) {
            tma_load_2d_pred(sB + (sb * G + i) * B_BYTES, term == 2 ? &tmX_lo : &tmX_hi, &fullB[sb], kc * TG_BK, rt * BN, leader);
            if (++kc == p.kchunks) { kc = 0; ++term; }
          }
          ++gB;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---------------------------------------------------------------------------------- MMA issuer
    // The whole warp runs the (uniform) loop and waits on the barriers; one elected lane issues (see umma_bf16_pred).
    const uint32_t leader = elect_one() ? 1u : 0u;
    {
      int gA = 0, gB = 0, acc = 0;
      uint32_t acc_phase = 0;
      for (int rt = rt0; rt < rt1; ++rt) {
        mbar_wait(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int g = 0; g < ngroups; ++g) {
          int sa;
          if (!p.stationary || rt == rt0) {
            sa = gA % NG;
            mbar_wait(&fullA[sa], (gA / NG) & 1);
            ++gA;
          } else {
            sa = g;                                // stationary panel: group g lives in slot g
          }
          const int sb = gB % NG;
          mbar_wait(&fullB[sb], (gB / NG) & 1);
          ++gB;
          tc_fence_after();
          if (g == 0 && rt == rt0 && leader) DBG(3);
          if (g == 0 && rt > rt0 && rt - rt0 <= 4 && leader) DBG(8 + (rt - rt0));
          const int n = min(G, kiters - g * G);
          const uint64_t adesc0 = umma_desc_sw128(smem_u32(sA + sa * G * TG_A_BYTES));
          const uint64_t bdesc0 = umma_desc_sw128(smem_u32(sB + sb * G * B_BYTES));
          if (n == G) {                            // full group: 16 back-to-back MMAs, descriptors advance by constants
#pragma unroll
            for (int i = 0; i < G; ++i)
#pragma unroll
              for (int k = 0; k < TG_BK / 16; ++k)
                umma_bf16_pred(d_tmem, adesc0 + (uint64_t)(i * (TG_A_BYTES >> 4) + 2 * k), bdesc0 + (uint64_t)(i * (B_BYTES >> 4) + 2 * k),
                          IDESC, (g > 0 || i > 0 || k > 0) ? 1u : 0u, leader);
          } else {
            for (int i = 0; i < n; ++i)
#pragma unroll
              for (int k = 0; k < TG_BK / 16; ++k)
                umma_bf16_pred(d_tmem, adesc0 + (uint64_t)(i * (TG_A_BYTES >> 4) + 2 * k), bdesc0 + (uint64_t)(i * (B_BYTES >> 4) + 2 * k),
                          IDESC, (g > 0 || i > 0 || k > 0) ? 1u : 0u, leader);
          }
          umma_commit_pred(&emptyB[sb], leader);
          if (!p.stationary) umma_commit_pred(&emptyA[sa], leader);
        }
        umma_commit_pred(&tfull[acc], leader);
        if (rt == rt0 && leader) DBG(4);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------------------------- epilogue (128 threads)
    // Per 32-row chunk: (A) thread = feature: TMEM -> registers, + bias, transposed write to the padded scratch;
    // (B) thread = (row, 32 consecutive features): + residual (prefetched 16-byte loads), activation or cluster
    // LayerNorm, 16-byte row-contiguous stores.  No per-element branches anywhere.
    const int e = warp - 2;                 // 0..3
    const int quarter = warp & 3;           // TMEM lane window of this warp
    const int fl = quarter * 32 + lane;     // phase A: feature within the tile == TMEM lane
    const int f = ftile * TG_BM + fl;
    const float bias = (p.bias && f < p.F) ? __ldg(p.bias + f) : 0.f;
    const int fo = ftile * TG_BM + e * 32;  // phase B: first of this thread's 32 features
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool direct_f32 = !is_ln && p.out_f32 != nullptr && p.out.p == nullptr && !p.has_res && p.act != ACT_RELU6;
    if (is_ln && e < 2) {   // static LayerNorm parameters of this feature tile -> shared memory, before the dependency resolves
      const float* g = (e == 0 ? p.gamma : p.beta) + ftile * TG_BM + lane * 4;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(sGB + e * TG_BM + lane * 4)), "l"(g) : "memory");
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    pdl_wait();
    __syncwarp();
    for (int rt = rt0; rt < rt1; ++rt) {
#pragma unroll 1
      for (int ch = 0; ch < CHUNKS; ++ch) {
        const int row = rt * BN + ch * 32 + lane;
        const bool row_ok = row < p.R;
        uint4 rh[4], rl[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) rh[g] = rl[g] = make_uint4(0u, 0u, 0u, 0u);
        if (p.has_res && row_ok) {   // in flight while the MMAs of the tile are still running
          const bf16* q = p.res.p + (size_t)row * p.res.ld + fo;
#pragma unroll
          for (int g = 0; g < 4; ++g)
            if (fo + g * 8 < p.F) rh[g] = *reinterpret_cast<const uint4*>(q + g * 8);
          if (p.res.lo) {
#pragma unroll
            for (int g = 0; g < 4; ++g)
              if (fo + g * 8 < p.F) rl[g] = *reinterpret_cast<const uint4*>(q + p.res.lo + g * 8);
          }
        }
        if (ch == 0) {
          mbar_wait(&tfull[acc], acc_phase);
          tc_fence_after();
          if (e == 0 && lane == 0 && rt == rt0) DBG(5);
        }
        {
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + ch * 32, r);
          tmem_ld_wait();
          if (ch == CHUNKS - 1) {           // accumulator drained: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            mbar_arrive(&tempty[acc]);
          }
          if (direct_f32) {
            // fp32-only output without residual (the vocabulary projection): store straight from the accumulator layout.
            // Thread = feature, so each of the 32 predicated stores of a warp covers 128 contiguous bytes of one row;
            // no shared-memory transpose, no barriers.
            const int rb = rt * BN + ch * 32;
            float* o = p.out_f32 + (size_t)rb * p.ld_f32 + f;     // running pointer: one 64-bit add per store
            const size_t ldb = (size_t)p.ld_f32;
            const int nvalid = (f < p.F) ? min(32, p.R - rb) : 0;  // rows this thread may write
            if (p.act == ACT_LEAKY) {
#pragma unroll
              for (int c = 0; c < 32; ++c) {
                const float v = __uint_as_float(r[c]) + bias;
                r[c] = __float_as_uint(v >= 0.f ? v : 0.2f * v);
              }
            } else if (p.act == ACT_RELU) {
#pragma unroll
              for (int c = 0; c < 32; ++c) r[c] = __float_as_uint(fmaxf(__uint_as_float(r[c]) + bias, 0.f));
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c) r[c] = __float_as_uint(__uint_as_float(r[c]) + bias);
            }
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              if (c < nvalid) *o = __uint_as_float(r[c]);
              o += ldb;
            }
            if (e == 0 && lane == 0 && rt == rt0) DBG(6 + ch);
            continue;
          }
#pragma unroll
          for (int c = 0; c < 32; ++c) sLN[c * TG_LN_STRIDE + fl] = __uint_as_float(r[c]) + bias;
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        float x[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 q4 = *reinterpret_cast<const float4*>(sLN + lane * TG_LN_STRIDE + e * 32 + i * 4);
          x[4 * i] = q4.x; x[4 * i + 1] = q4.y; x[4 * i + 2] = q4.z; x[4 * i + 3] = q4.w;
        }
        if (p.has_res) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float t[8];
            unpack8(rh[g], t);
#pragma unroll
            for (int i = 0; i < 8; ++i) x[g * 8 + i] += t[i];
          }
          if (p.res.lo) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float t[8];
              unpack8(rl[g], t);
#pragma unroll
              for (int i = 0; i < 8; ++i) x[g * 8 + i] += t[i];
            }
          }
        }
        if (!is_ln) {
          if (p.act == ACT_RELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = fmaxf(x[i], 0.f);
          } else if (p.act == ACT_LEAKY) {
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = x[i] >= 0.f ? x[i] : 0.2f * x[i];
          } else if (p.act == ACT_RELU6) {
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = fminf(fmaxf(x[i], 0.f), 6.f);
          }
          if (row_ok) {
            if (p.out.p) {
#pragma unroll
              for (int g = 0; g < 4; ++g)
                if (fo + g * 8 < p.F) st_act8(p.out, (size_t)row, fo + g * 8, x + g * 8);
            }
            if (p.out_f32) {
              float* o = p.out_f32 + (size_t)row * p.ld_f32 + fo;
#pragma unroll
              for (int g = 0; g < 8; ++g)
                if (fo + g * 4 < p.F) *reinterpret_cast<float4*>(o + g * 4) = make_float4(x[g * 4], x[g * 4 + 1], x[g * 4 + 2], x[g * 4 + 3]);
            }
          }
        } else {
          // ---- LayerNorm over the 512 features of each row: 4 CTAs x 4 threads hold one row (Chan's parallel variance)
          float sum = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) sum += x[i];
          const float m = sum * (1.f / 32.f);
          float m2 = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float d = x[i] - m;
            m2 = fmaf(d, d, m2);
          }
          sPart[e * 32 + lane] = make_float2(m, m2);
          asm volatile("cp.async.wait_group 0;" ::: "memory");   // the staged gamma / beta (issued before the grid dependency)
          asm volatile("bar.sync 1, 128;" ::: "memory");
          {
            const float2 a0 = sPart[lane], a1 = sPart[32 + lane], a2 = sPart[64 + lane], a3 = sPart[96 + lane];
            const float mc = 0.25f * (a0.x + a1.x + a2.x + a3.x);
            const float d0 = a0.x - mc, d1 = a1.x - mc, d2 = a2.x - mc, d3 = a3.x - mc;
            const float m2c = a0.y + a1.y + a2.y + a3.y + 32.f * (d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3);
            if (e == 0) sStat[lane] = make_float2(mc, m2c);
          }
          cluster_sync_all();                                  // #1: every CTA's row statistics are published
          const float2 s0 = ld_dsmem_f2(&sStat[lane], 0), s1 = ld_dsmem_f2(&sStat[lane], 1), s2 = ld_dsmem_f2(&sStat[lane], 2),
                       s3 = ld_dsmem_f2(&sStat[lane], 3);
          const float mean = 0.25f * (s0.x + s1.x + s2.x + s3.x);
          const float e0 = s0.x - mean, e1 = s1.x - mean, e2 = s2.x - mean, e3 = s3.x - mean;
          const float M2 = s0.y + s1.y + s2.y + s3.y + 128.f * (e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3);
          const float rstd = rsqrtf(M2 * (1.f / 512.f) + p.eps);
          if (row_ok) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float o[8];
              const float4 ga = *reinterpret_cast<const float4*>(sGB + e * 32 + g * 8);
              const float4 gb = *reinterpret_cast<const float4*>(sGB + e * 32 + g * 8 + 4);
              const float4 ba = *reinterpret_cast<const float4*>(sGB + TG_BM + e * 32 + g * 8);
              const float4 bb = *reinterpret_cast<const float4*>(sGB + TG_BM + e * 32 + g * 8 + 4);
              const float gg[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
              const float be[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) o[i] = (x[g * 8 + i] - mean) * rstd * gg[i] + be[i];
              st_act8(p.out, (size_t)row, fo + g * 8, o);
            }
          }
          cluster_sync_all();                                  // #2: nobody exits while its statistics are still being read
                                                               //     (after the stores: off the critical path of the output)
        }
        if (e == 0 && lane == 0 && rt == rt0) DBG(6 + ch);
        if (CHUNKS > 1 || rt + 1 < rt1) asm volatile("bar.sync 1, 128;" ::: "memory");   // scratch is reused
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }
  if (is_ln && warp < 2) {   // the TMA / MMA warps take part in the cluster barriers of the LN epilogue
    cluster_sync_all();
    cluster_sync_all();
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) DBG(8);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
#undef DBG
}

template <int BN>
static int launch_bn(const TgemmOp& op, cudaStream_t stream) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(op.grid);
  cfg.blockDim = dim3(TG_THREADS);
  cfg.dynamicSmemBytes = tgemm_smem_bytes(BN);
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (op.cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = op.cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  FPNMT_CUDA_OK(cudaLaunchKernelEx(&cfg, tgemm_kernel<BN>, op.tmW, op.tmX_hi, op.tmX_lo, op.p));
  return 0;
}

int tgemm_launch(const TgemmOp& op, cudaStream_t stream) {
  if (op.wide) return tgemmw_launch(op, stream);
  if (op.BN == 32) return launch_bn<32>(op, stream);
  if (op.BN == 64) return launch_bn<64>(op, stream);
  set_last_error("tgemm_launch: unsupported BN");
  return 1;
}

int tgemm_set_attributes() {
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemm_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tgemm_smem_bytes(32)));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemm_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tgemm_smem_bytes(64)));
  return 0;
}

int make_tgemm_op(TgemmOp* op, int R, const Act& x, const bf16* wt, int F, int K, bool split, const float* bias, int act,
                  const Act& out, float* out_f32, int ld_f32, const Act* res, const float* gamma, const float* beta,
                  float eps, int num_sms, int force_bn) {
  TgemmParams& p = op->p;
  p = TgemmParams{};
  if (x.C != K) {
    set_last_error("make_tgemm_op: activation view width != K");
    return 1;
  }
  if (split && !x.lo) {
    set_last_error("make_tgemm_op: split mode needs a split activation view");
    return 1;
  }
  const bool ln = gamma != nullptr;
  if (ln && (F != 512 || !out.p)) {
    set_last_error("make_tgemm_op: the LayerNorm epilogue needs F == 512 and a bf16 output view");
    return 1;
  }
  int BN = force_bn ? force_bn : ((ln || F < 1024) ? 32 : 64);
  if (ln) BN = 32;
  p.R = R;
  p.F = F;
  p.kchunks = (K + TG_BK - 1) / TG_BK;
  p.nterms = split ? 3 : 1;
  p.w_lo_off = split ? K : 0;
  p.ftiles = (F + TG_BM - 1) / TG_BM;
  p.rtiles = (R + BN - 1) / BN;
  int rgroups = num_sms / p.ftiles;
  if (rgroups < 1) rgroups = 1;
  if (rgroups > p.rtiles) rgroups = p.rtiles;
  if (ln) rgroups = p.rtiles;
  p.rt_per_item = (p.rtiles + rgroups - 1) / rgroups;
  rgroups = (p.rtiles + p.rt_per_item - 1) / p.rt_per_item;
  p.stationary = (p.nterms * p.kchunks <= TG_A_SLOTS) ? 1 : 0;
  p.bias = bias;
  p.act = act;
  p.out = out;
  p.out_f32 = out_f32;
  p.ld_f32 = ld_f32;
  p.has_res = res ? 1 : 0;
  if (res) p.res = *res;
  p.gamma = gamma;
  p.beta = beta;
  p.eps = eps;
  op->BN = BN;
  op->wide = 0;
  op->grid = p.ftiles * rgroups;
  op->cluster = ln ? 4 : 1;
  op->flops = 2.0 * (double)R * (double)F * (double)K;
  const uint64_t kw_total = split ? 2 * (uint64_t)K : (uint64_t)K;
  int rc = encode_tmap_2d(&op->tmW, wt, kw_total, (uint64_t)F, kw_total, TG_BM);
  if (rc) return rc;
  rc = encode_tmap_2d(&op->tmX_hi, x.p, (uint64_t)K, (uint64_t)R, (uint64_t)x.ld, BN);
  if (rc) return rc;
  return encode_tmap_2d(&op->tmX_lo, split ? x.p + x.lo : x.p, (uint64_t)K, (uint64_t)R, (uint64_t)x.ld, BN);
}

}  // namespace fpnmt
