// Wide-row variant of the skinny-row Dense kernel (tgemm.cuh), built for THROUGHPUT when several decode lanes share the GPU.
//
// tgemm_kernel<32/64> keeps a whole K = 512 weight panel (128 KB) plus the activation panel resident: ~180-210 KB of shared
// memory, so one CTA owns an SM for its ~6 us of (latency-bound) life, every 32/64-row tile pulls the full weight panel
// through L2 again (60 MB of weights x 16 row tiles ~ 1 GB of L2->SM traffic per decode step), and kernels of concurrent lanes
// (fpnmt_submit) cannot share an SM.  Measured: four co-running decode chains sustain 211 us per step where one alone needs 347.
//
// This kernel trades a little single-chain latency for SM time:
//   * 128 activation rows per CTA, and because 128 rows fill the UMMA M dimension the NATURAL orientation: the activation tile is
//     the tcgen05 A operand (M = 128 rows = TMEM lanes), the weight tile the B operand (N = 128 features = TMEM columns).
//     tcgen05.mma 128 x 128 x 16 runs at the full tensor rate (65 clk; N = 32 takes 41 clk for a quarter of the work) and the
//     weight panel is fetched once per 128 rows - 4x less L2->SM traffic and 4x fewer CTAs than 32-row tiles;
//   * the K loop streams through a 96 KB ring (3 x [16 KB activations + 16 KB weights], one mbarrier per stage), so a CTA needs
//     ~100 KB of shared memory and TWO CTAs are resident per SM (TMEM: 128 or 256 columns each);
//   * epilogue thread = row: tcgen05.ld hands it 32 CONSECUTIVE features of its row, so bias / activation / 16-byte stores and
//     the LayerNorm sums need no transpose, no shared-memory scratch and no block barrier (tgemm_kernel's D^T layout pays a
//     transpose through shared memory and a barrier per 32-row chunk: ~0.9 us each on one warp per scheduler).
//     LayerNorm(x.W + b + residual): pass 1 reduces (mean, M2) of the CTA's 128 features in registers, ONE exchange over the
//     4-CTA cluster (DSMEM), pass 2 reads the accumulator from TMEM again, normalises and stores.
// bf16 mode only (the BF16X3 parity mode keeps tgemm_kernel).  Reference: the Dense layers of models/transformer.py:104-119,
// 224-243 (decoder layer), :357,372 (final_layer).
//   warp 0     : TMA producer (convergent, elected lane issues); weights of the first ring pass go out before griddepcontrol.wait
//   warp 1     : TMEM allocator + tcgen05.mma issuer
//   warps 2..5 : epilogue
#include "tgemm.cuh"

#include "tensormap.cuh"

namespace fpnmt {

constexpr int TW_ROWS = 128;                           // activation rows per CTA == UMMA M == TMEM lanes
constexpr int TW_TILE_BYTES = 128 * TG_BK * 2;         // 16 KB: [128 rows or features][64 k] bf16, SWIZZLE_128B
constexpr int TW_STAGE_BYTES = 2 * TW_TILE_BYTES;      // activations | weights
constexpr int TW_STAGES = 3;
constexpr int TW_RING_BYTES = TW_STAGES * TW_STAGE_BYTES;

size_t tgemmw_smem_bytes(int) {
  return (size_t)TW_RING_BYTES + 3 * TG_BM * 4 /*bias, gamma, beta of the feature tile*/ + TW_ROWS * 8 /*row statistics*/ +
         256 /*barriers*/ + 1024 /*align slack*/;
}

__device__ __forceinline__ void tw_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ long long tw_timer() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ float2 tw_ld_dsmem_f2(const float2* local, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local)), "r"(rank));
  float2 v;
  asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(remote) : "memory");
  return v;
}
// Output tile staging for the TMA store: two [128 rows][64 features] bf16 sub-tiles with 128-byte rows in the SWIZZLE_128B
// pattern (16-byte chunk index XOR row % 8) - the layout cp.async.bulk.tensor expects for that swizzle mode, and a bank-conflict
// free target for "thread = row" 16-byte writes (rows l, l+8, l+16, l+24 share banks: 4 wavefronts for 512 B, the minimum).
// Stores of 16 B per lane to 32 different rows straight to global memory cost ~0.9 us per 32-feature chunk (32 partial lines per
// instruction); the bulk tensor store writes whole lines and runs asynchronously.
__device__ __forceinline__ void tw_stage_chunk(uint8_t* stg, int lr, int ch, const float* x) {
  uint8_t* rowp = stg + (ch >> 1) * TW_TILE_BYTES + lr * 128;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int lc = (ch & 1) * 4 + g;
    *reinterpret_cast<uint4*>(rowp + ((lc ^ (lr & 7)) << 4)) = pack8(x + g * 8);
  }
}
__device__ __forceinline__ void tw_tma_store_2d(const CUtensorMap* m, const void* smem, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(m), "r"(smem_u32(smem)), "r"(c0),
               "r"(c1)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tw_tma_store_wait() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// sub-tile `sub` of the staging buffer is complete in every epilogue thread's view -> one thread issues its bulk store
__device__ __forceinline__ void tw_store_subtile(const CUtensorMap* m, uint8_t* stg, int sub, int f0, int F, int row0, bool issuer) {
  fence_proxy_async();
  asm volatile("bar.sync 1, 128;" ::: "memory");
  if (issuer && f0 + sub * 64 < F) tw_tma_store_2d(m, stg + sub * TW_TILE_BYTES, f0 + sub * 64, row0);
}
// activation with the selector hoisted out of the element loop (a per-element switch compiles to an indirect branch each)
__device__ __forceinline__ void tw_act32(float* x, int act) {
  if (act == ACT_RELU) {
#pragma unroll
    for (int i = 0; i < 32; ++i) x[i] = fmaxf(x[i], 0.f);
  } else if (act == ACT_LEAKY) {
#pragma unroll
    for (int i = 0; i < 32; ++i) x[i] = x[i] >= 0.f ? x[i] : 0.2f * x[i];
  } else if (act == ACT_RELU6) {
#pragma unroll
    for (int i = 0; i < 32; ++i) x[i] = fminf(fmaxf(x[i], 0.f), 6.f);
  }
}
// accumulator chunk -> registers: this thread's row (TMEM lane), 32 consecutive features, + bias (shared-memory broadcast)
__device__ __forceinline__ void tw_load_chunk(uint32_t taddr, const float* sBias32, float* x) {
  uint32_t r[32];
  tmem_ld32(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 b = *reinterpret_cast<const float4*>(sBias32 + 4 * i);
    x[4 * i] = __uint_as_float(r[4 * i]) + b.x;
    x[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + b.y;
    x[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + b.z;
    x[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + b.w;
  }
}

// The kernel body.  TGT (tgemmw_target_kernel, vocabulary tile without logits only): the row whose target id tgt[row] lies in
// [0, F) also writes the fp32 logit of that feature, the value its tile's statistics and candidates are computed from, to
// tgt_logit[row] (-1 or an id >= F: nothing written).  MASK (tgemmw_mask_kernel, with TGT; tgt may then be nullptr): the
// top-8 candidates of a row skip the features banned in its mask row, mask + (par * R + row) * ceil(F / 32) with par =
// *mask_step & 1 (mask_step nullptr: 0); a 32-feature chunk is one mask word.  The (max, sum exp) statistics stay unmasked.
template <bool TGT, bool MASK = false>
__device__ __forceinline__ void tgemmw_body(const CUtensorMap& tmW, const CUtensorMap& tmX, const CUtensorMap& tmO,
                                            const TgemmParams p, const int* __restrict__ tgt, float* __restrict__ tgt_logit,
                                            const uint32_t* __restrict__ mask = nullptr, const int* __restrict__ mask_step = nullptr) {
  constexpr int STAGES = TW_STAGES;
  constexpr int BN = 128;                          // features per tile == UMMA N == TMEM columns of one accumulator
  constexpr int CHUNKS = BN / 32;
  constexpr uint32_t IDESC = umma_idesc_bf16(TW_ROWS, BN);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* ring = smem;
  float* sBias = reinterpret_cast<float*>(smem + TW_RING_BYTES);                             // [128] bias | gamma | beta
  float* sGam = sBias + TG_BM;
  float* sBet = sGam + TG_BM;
  float2* sStat = reinterpret_cast<float2*>(sBet + TG_BM);                                   // [128 rows] CTA-level (mean, M2)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStat + TW_ROWS);
  uint64_t* full = bars;                           // [STAGES]
  uint64_t* empty = bars + 4;                      // [STAGES]
  uint64_t* tfull = bars + 8;                      // [2]
  uint64_t* tempty = bars + 10;                    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool is_ln = p.gamma != nullptr;
  const int item = blockIdx.x;
  const int ftile = item % p.ftiles;
  const int rgroup = item / p.ftiles;
  const int rt0 = rgroup * p.rt_per_item;
  const int rt1 = min(p.rtiles, rt0 + p.rt_per_item);
  const int kiters = p.kchunks;
  const bool multi = p.rt_per_item > 1;            // several row tiles per CTA: two accumulators

#ifdef FPNMT_DBG_STAMPS   // build.py --dbg-stamps: globaltimer timeline of block 0 (FPNMT_DBG_OP=<op name>); off in product builds
  __shared__ long long* s_dbg;
  if (threadIdx.x == 0) {
    s_dbg = nullptr;
    if (p.dbg && blockIdx.x == 0) {
      const long long inst = (long long)atomicAdd((unsigned long long*)p.dbg, 1ull);
      s_dbg = p.dbg + 16 + (inst % 8) * 16;
      s_dbg[0] = tw_timer();
    }
  }
#define DBG(k) do { if (s_dbg) s_dbg[k] = tw_timer(); } while (0)
#else
#define DBG(k) do { } while (0)
#endif
  pdl_launch();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmO);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (multi) tmem_alloc<2 * BN>(tmem_slot);
    else tmem_alloc<BN>(tmem_slot);
  }
  if (warp >= 2) {                                 // static per-feature vectors of this tile (never written by a kernel)
    const int t = threadIdx.x - 64;                // 0..127
    const int f = ftile * TG_BM + t;
    sBias[t] = (p.bias && f < p.F) ? __ldg(p.bias + f) : 0.f;
    if (is_ln) {
      sGam[t] = __ldg(p.gamma + f);
      sBet[t] = __ldg(p.beta + f);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) DBG(1);

  if (warp == 0) {
    // ---------------------------------------------------------------------------------- TMA producer
    const uint32_t leader = elect_one() ? 1u : 0u;
    const int total = (rt1 - rt0) * kiters;
    const int npre = total < STAGES ? total : STAGES;
    for (int i = 0; i < npre; ++i) {               // static weights of the first ring pass: before the grid dependency resolves
      mbar_expect_tx_pred(&full[i], TW_STAGE_BYTES, leader);
      tma_load_2d_pred(ring + i * TW_STAGE_BYTES + TW_TILE_BYTES, &tmW, &full[i], (i % kiters) * TG_BK, ftile * TG_BM, leader);
    }
    pdl_wait();
    if (leader) DBG(2);
    int it = 0;
    for (int rt = rt0; rt < rt1; ++rt) {
      for (int kc = 0; kc < kiters; ++kc, ++it) {
        const int s = it % STAGES;
        uint8_t* st = ring + s * TW_STAGE_BYTES;
        if (it >= npre) {
          mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
          mbar_expect_tx_pred(&full[s], TW_STAGE_BYTES, leader);
          tma_load_2d_pred(st + TW_TILE_BYTES, &tmW, &full[s], kc * TG_BK, ftile * TG_BM, leader);
        }
        tma_load_2d_pred(st, &tmX, &full[s], kc * TG_BK, rt * TW_ROWS, leader);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---------------------------------------------------------------------------------- MMA issuer (convergent warp)
    // D[row][feature] += X[row][k] . W[feature][k]: the activation tile is the A operand (M = 128 rows = TMEM lanes), the
    // weight tile the B operand (N = 128 features = TMEM columns) - the natural orientation, possible because 128 rows fill M.
    const uint32_t leader = elect_one() ? 1u : 0u;
    int it = 0, acc = 0;
    uint32_t acc_phase = 0;
    for (int rt = rt0; rt < rt1; ++rt) {
      if (multi) {
        mbar_wait(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
      }
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kc = 0; kc < kiters; ++kc, ++it) {
        const int s = it % STAGES;
        mbar_wait(&full[s], (it / STAGES) & 1);
        tc_fence_after();
        if (leader && it == 0) DBG(3);
        if (leader && !is_ln && (it & 1) && it < 8) DBG(9 + (it >> 1));
        const uint64_t adesc = umma_desc_sw128(smem_u32(ring + s * TW_STAGE_BYTES));
        const uint64_t bdesc = umma_desc_sw128(smem_u32(ring + s * TW_STAGE_BYTES + TW_TILE_BYTES));
#pragma unroll
        for (int k = 0; k < TG_BK / 16; ++k)
          umma_bf16_pred(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), IDESC, (kc > 0 || k > 0) ? 1u : 0u, leader);
        umma_commit_pred(&empty[s], leader);
      }
      umma_commit_pred(&tfull[acc], leader);
      if (leader && rt == rt0) DBG(4);
      if (multi && ++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------------------------- epilogue (128 threads)
    // thread = row (TMEM lane); per 32-feature chunk it holds 32 CONSECUTIVE features of its row: 16-byte stores and the
    // LayerNorm sums need no transpose, no shared-memory scratch and no block barrier.
    const int quarter = warp & 3;           // TMEM lane window of this warp
    const int lr = quarter * 32 + lane;     // row within the tile
    const int f0 = ftile * TG_BM;
    const bool issuer = warp == 2 && lane == 0;
    const bool use_tma_store = !multi && p.out.p != nullptr && p.out_f32 == nullptr;
    pdl_wait();
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int rt = rt0; rt < rt1; ++rt) {
      const int row = rt * TW_ROWS + lr;
      const bool row_ok = row < p.R;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN;
      uint4 rh[4];                          // residual of chunk 0: in flight while the MMAs still run
#pragma unroll
      for (int g = 0; g < 4; ++g) rh[g] = make_uint4(0u, 0u, 0u, 0u);
      const bf16* resp = (is_ln && p.has_res && row_ok) ? p.res.p + (size_t)row * p.res.ld + f0 : nullptr;
      if (resp) {
#pragma unroll
        for (int g = 0; g < 4; ++g) rh[g] = *reinterpret_cast<const uint4*>(resp + g * 8);
      }
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      if (warp == 2 && lane == 0 && rt == rt0) DBG(5);
      if (p.vs_stat) {
        // ---- vocabulary tile without logits: online (max, sum-exp) and the TG_VS_N largest logits of this row's 128 features,
        // all in this thread's registers (thread = row).  The list is kept sorted by a compare-exchange chain; scanning the
        // features in ascending order with strict comparisons gives the tf.math.top_k tie order (lower index first).
        // (Measured alternative: an unsorted set with a tracked worst slot - 8 selects + a 3-level tree per insertion - is 2.5x
        // slower, 65 vs 26 us for the C2 projection: the insertion body runs for nearly every element because some lane of the
        // warp always qualifies, so instruction count matters more than the length of the dependent chain.)
        float m = -INFINITY, ssum = 0.f;
        int tg = -1;                                          // target feature of this row (TGT)
        if constexpr (TGT) tg = (row_ok && (!MASK || tgt)) ? __ldcg(tgt + row) : -1;
        const uint32_t* mrow = nullptr;                       // this row's ban mask (MASK)
        if constexpr (MASK) {
          const int par = mask_step ? (__ldcg(mask_step) & 1) : 0;
          mrow = mask + ((size_t)par * p.R + row) * ((p.F + 31) / 32);
        }
        float bv[TG_VS_N];
        int bi[TG_VS_N];
#pragma unroll
        for (int k = 0; k < TG_VS_N; ++k) {
          bv[k] = -INFINITY;
          bi[k] = 0x7fffffff;
        }
#pragma unroll 1
        for (int ch = 0; ch < CHUNKS; ++ch) {
          float x[32];
          tw_load_chunk(taddr + ch * 32, sBias + ch * 32, x);
          if (multi && ch == CHUNKS - 1) {
            tc_fence_before();
            mbar_arrive(&tempty[acc]);
          }
          const int fo = f0 + ch * 32;
          float cm = -INFINITY;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (fo + i >= p.F) x[i] = -INFINITY;     // padding features of the last tile
            cm = fmaxf(cm, x[i]);
          }
          if constexpr (TGT) {
            const int d = tg - fo;
            if (d >= 0 && d < 32 && tg < p.F) {      // this chunk holds the target: select it without indexing the registers
              float z = x[0];
#pragma unroll
              for (int i = 1; i < 32; ++i) z = d == i ? x[i] : z;
              tgt_logit[row] = z;
            }
          }
          if (cm > -INFINITY) {
            const float mn = fmaxf(m, cm);
            float cs = 0.f;
#pragma unroll
            for (int i = 0; i < 32; ++i) cs += __expf(x[i] - mn);
            ssum = ssum * __expf(m - mn) + cs;
            m = mn;
          }
          uint32_t mw = 0u;                                   // banned features of this chunk (MASK): never candidates
          float cma = cm;
          if constexpr (MASK) {
            mw = (row_ok && fo < p.F) ? __ldcg(mrow + (fo >> 5)) : 0u;   // padding chunks: no mask word (already -inf)
            if (mw) {
              cma = -INFINITY;
#pragma unroll
              for (int i = 0; i < 32; ++i) cma = ((mw >> i) & 1u) ? cma : fmaxf(cma, x[i]);
            }
          }
          if (cma > bv[TG_VS_N - 1]) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (x[i] > bv[TG_VS_N - 1] && !((mw >> i) & 1u)) {
                bv[TG_VS_N - 1] = x[i];
                bi[TG_VS_N - 1] = fo + i;
#pragma unroll
                for (int k = TG_VS_N - 1; k > 0; --k) {
                  const bool sw = bv[k] > bv[k - 1];
                  const float tv = sw ? bv[k - 1] : bv[k];
                  const int ti = sw ? bi[k - 1] : bi[k];
                  bv[k - 1] = sw ? bv[k] : bv[k - 1];
                  bi[k - 1] = sw ? bi[k] : bi[k - 1];
                  bv[k] = tv;
                  bi[k] = ti;
                }
              }
            }
          }
        }
        if (row_ok) {
          const size_t slot = (size_t)row * p.ftiles + ftile;
          p.vs_stat[slot] = make_float2(m, ssum);
          float4* vo = reinterpret_cast<float4*>(p.vs_val + slot * TG_VS_N);
          int4* io = reinterpret_cast<int4*>(p.vs_idx + slot * TG_VS_N);
#pragma unroll
          for (int k = 0; k < TG_VS_N / 4; ++k) {
            vo[k] = make_float4(bv[4 * k], bv[4 * k + 1], bv[4 * k + 2], bv[4 * k + 3]);
            io[k] = make_int4(bi[4 * k], bi[4 * k + 1], bi[4 * k + 2], bi[4 * k + 3]);
          }
        }
      } else if (!is_ln) {
#pragma unroll 1
        for (int ch = 0; ch < CHUNKS; ++ch) {
          float x[32];
          tw_load_chunk(taddr + ch * 32, sBias + ch * 32, x);
          if (multi && ch == CHUNKS - 1) {  // accumulator drained: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            mbar_arrive(&tempty[acc]);
          }
          tw_act32(x, p.act);
          const int fo = f0 + ch * 32;
          if (use_tma_store) {              // single tile: the ring is idle, the output tile is staged in it and bulk-stored
            tw_stage_chunk(ring, lr, ch, x);
            if (ch & 1) tw_store_subtile(&tmO, ring, ch >> 1, f0, p.F, rt * TW_ROWS, issuer);
          } else if (row_ok) {
            if (p.out.p) {
              bf16* o = p.out.p + (size_t)row * p.out.ld + fo;
#pragma unroll
              for (int g = 0; g < 4; ++g)
                if (fo + g * 8 < p.F) *reinterpret_cast<uint4*>(o + g * 8) = pack8(x + g * 8);
            }
            if (p.out_f32) {
              float* o = p.out_f32 + (size_t)row * p.ld_f32 + fo;
#pragma unroll
              for (int g = 0; g < 8; ++g)
                if (fo + g * 4 < p.F) *reinterpret_cast<float4*>(o + g * 4) = make_float4(x[g * 4], x[g * 4 + 1], x[g * 4 + 2], x[g * 4 + 3]);
            }
          }
          if (warp == 2 && lane == 0 && ch < 2) DBG(6 + ch);
        }
      } else {
        // ---- LayerNorm over the 512 features of a row held by the 4 CTAs of the cluster.  Pass 1: (mean, M2) of this CTA's
        // 128 features, chunk by chunk (Chan's parallel variance); the sums are NOT kept - pass 2 reads the accumulator again.
        float mean_c = 0.f, m2_c = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < CHUNKS; ++ch) {
          float x[32];
          tw_load_chunk(taddr + ch * 32, sBias + ch * 32, x);
          uint4 rn[4];                      // next chunk's residual while this one is reduced
#pragma unroll
          for (int g = 0; g < 4; ++g) rn[g] = make_uint4(0u, 0u, 0u, 0u);
          if (resp && ch + 1 < CHUNKS) {
#pragma unroll
            for (int g = 0; g < 4; ++g) rn[g] = *reinterpret_cast<const uint4*>(resp + (ch + 1) * 32 + g * 8);
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float t[8];
            unpack8(rh[g], t);
#pragma unroll
            for (int i = 0; i < 8; ++i) x[g * 8 + i] += t[i];
          }
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
          // merge (32 ch features; mean_c, m2_c) with (32; m, m2)
          const float na = 32.f * ch, nab = na + 32.f;
          const float dl = m - mean_c;
          m2_c = m2_c + m2 + dl * dl * (na * 32.f / nab);
          mean_c = mean_c + dl * (32.f / nab);
#pragma unroll
          for (int g = 0; g < 4; ++g) rh[g] = rn[g];
          if (warp == 2 && lane == 0 && ch < 2) DBG(6 + ch);
        }
        sStat[lr] = make_float2(mean_c, m2_c);
        if (warp == 2 && lane == 0) DBG(9);
        if (resp) {                         // chunk 0's residual again for pass 2 (L1 / L2 hit), in flight over the exchange
#pragma unroll
          for (int g = 0; g < 4; ++g) rh[g] = *reinterpret_cast<const uint4*>(resp + g * 8);
        }
        tw_cluster_sync();                                   // #1: every CTA's row statistics are published
        if (warp == 2 && lane == 0) DBG(10);
        const float2 s0 = tw_ld_dsmem_f2(&sStat[lr], 0), s1 = tw_ld_dsmem_f2(&sStat[lr], 1), s2 = tw_ld_dsmem_f2(&sStat[lr], 2),
                     s3 = tw_ld_dsmem_f2(&sStat[lr], 3);
        const float mean = 0.25f * (s0.x + s1.x + s2.x + s3.x);
        const float e0 = s0.x - mean, e1 = s1.x - mean, e2 = s2.x - mean, e3 = s3.x - mean;
        const float M2 = s0.y + s1.y + s2.y + s3.y + 128.f * (e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3);
        const float rstd = rsqrtf(M2 * (1.f / 512.f) + p.eps);
#pragma unroll 1
        for (int ch = 0; ch < CHUNKS; ++ch) {
          float x[32];
          tw_load_chunk(taddr + ch * 32, sBias + ch * 32, x);
          uint4 rn[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) rn[g] = make_uint4(0u, 0u, 0u, 0u);
          if (resp && ch + 1 < CHUNKS) {
#pragma unroll
            for (int g = 0; g < 4; ++g) rn[g] = *reinterpret_cast<const uint4*>(resp + (ch + 1) * 32 + g * 8);
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float t[8];
            unpack8(rh[g], t);
#pragma unroll
            for (int i = 0; i < 8; ++i) x[g * 8 + i] += t[i];
          }
          {
            float y[32];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const float4 ga = *reinterpret_cast<const float4*>(sGam + ch * 32 + g * 8);
              const float4 gb = *reinterpret_cast<const float4*>(sGam + ch * 32 + g * 8 + 4);
              const float4 ba = *reinterpret_cast<const float4*>(sBet + ch * 32 + g * 8);
              const float4 bb = *reinterpret_cast<const float4*>(sBet + ch * 32 + g * 8 + 4);
              const float gg[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
              const float be[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) y[g * 8 + i] = (x[g * 8 + i] - mean) * rstd * gg[i] + be[i];
            }
            tw_stage_chunk(ring, lr, ch, y);
            if (ch & 1) tw_store_subtile(&tmO, ring, ch >> 1, f0, p.F, rt * TW_ROWS, issuer);
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) rh[g] = rn[g];
        }
        if (warp == 2 && lane == 0) DBG(11);
        tw_cluster_sync();                                   // #2: nobody exits while its statistics are still being read
      }
      if (multi && ++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (issuer) DBG(12);
    if (issuer) tw_tma_store_wait();        // the bulk stores have left shared memory and are globally performed
  }
  if (is_ln && warp < 2) {   // the TMA / MMA warps take part in the cluster barriers of the LayerNorm epilogue
    tw_cluster_sync();
    tw_cluster_sync();
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) DBG(8);
#undef DBG
  if (warp == 1) {
    tc_fence_after();
    if (multi) tmem_dealloc<2 * BN>(tmem_base);
    else tmem_dealloc<BN>(tmem_base);
  }
}

__global__ void __launch_bounds__(TG_THREADS, 2)
tgemmw_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX,
              const __grid_constant__ CUtensorMap tmO, const TgemmParams p) {
  tgemmw_body<false>(tmW, tmX, tmO, p, nullptr, nullptr);
}
// The vocabulary projection of a prompted beam search on the logits-free tail: tgemmw_kernel + the target logit (TgemmOp::tgt)
__global__ void __launch_bounds__(TG_THREADS, 2)
tgemmw_target_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX,
                     const __grid_constant__ CUtensorMap tmO, const TgemmParams p, const int* __restrict__ tgt,
                     float* __restrict__ tgt_logit) {
  tgemmw_body<true>(tmW, tmX, tmO, p, tgt, tgt_logit);
}
// The vocabulary projection of a constrained beam search on the logits-free tail: tgemmw_target_kernel + the ban masks
// (TgemmOp::mask): every row's candidates are its allowed features only
__global__ void __launch_bounds__(TG_THREADS, 2)
tgemmw_mask_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX,
                   const __grid_constant__ CUtensorMap tmO, const TgemmParams p, const int* __restrict__ tgt,
                   float* __restrict__ tgt_logit, const uint32_t* __restrict__ mask, const int* __restrict__ mask_step) {
  tgemmw_body<true, true>(tmW, tmX, tmO, p, tgt, tgt_logit, mask, mask_step);
}

int tgemmw_launch(const TgemmOp& op, cudaStream_t stream) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(op.grid);
  cfg.blockDim = dim3(TG_THREADS);
  cfg.dynamicSmemBytes = tgemmw_smem_bytes(128);
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
  if (op.mask)
    FPNMT_CUDA_OK(cudaLaunchKernelEx(&cfg, tgemmw_mask_kernel, op.tmW, op.tmX_hi, op.tmX_lo, op.p, op.tgt, op.tgt_logit, op.mask,
                                     op.mask_step));
  else if (op.tgt) FPNMT_CUDA_OK(cudaLaunchKernelEx(&cfg, tgemmw_target_kernel, op.tmW, op.tmX_hi, op.tmX_lo, op.p, op.tgt, op.tgt_logit));
  else FPNMT_CUDA_OK(cudaLaunchKernelEx(&cfg, tgemmw_kernel, op.tmW, op.tmX_hi, op.tmX_lo, op.p));
  return 0;
}

int tgemmw_set_attributes() {
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemmw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tgemmw_smem_bytes(128)));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemmw_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemmw_target_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tgemmw_smem_bytes(128)));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemmw_target_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemmw_mask_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tgemmw_smem_bytes(128)));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(tgemmw_mask_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return 0;
}

// Whether the wide kernel can run this Dense layer: bf16 storage, and a residual only together with the LayerNorm epilogue.
bool tgemmw_supports(bool split, bool has_res, bool ln, int F, int K) {
  if (split || (has_res && !ln) || (K % 8) != 0) return false;
  return !ln || F == 512;
}

int make_tgemmw_op(TgemmOp* op, int R, const Act& x, const bf16* wt, int F, int K, const float* bias, int act, const Act& out,
                   float* out_f32, int ld_f32, const Act* res, const float* gamma, const float* beta, float eps, int num_sms,
                   float2* vs_stat, float* vs_val, int* vs_idx) {
  TgemmParams& p = op->p;
  p = TgemmParams{};
  if (x.C != K) {
    set_last_error("make_tgemmw_op: activation view width != K");
    return 1;
  }
  const bool ln = gamma != nullptr;
  if (ln && (F != 512 || !out.p)) {
    set_last_error("make_tgemmw_op: the LayerNorm epilogue needs F == 512 and a bf16 output view");
    return 1;
  }
  const int BN = TW_ROWS;
  p.R = R;
  p.F = F;
  p.kchunks = (K + TG_BK - 1) / TG_BK;
  p.nterms = 1;
  p.ftiles = (F + TG_BM - 1) / TG_BM;
  p.rtiles = (R + BN - 1) / BN;
  int rgroups = 2 * num_sms / p.ftiles;            // two resident CTAs per SM
  if (rgroups < 1) rgroups = 1;
  if (rgroups > p.rtiles || ln) rgroups = p.rtiles;
  p.rt_per_item = (p.rtiles + rgroups - 1) / rgroups;
  rgroups = (p.rtiles + p.rt_per_item - 1) / p.rt_per_item;
  p.stationary = 0;
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
  p.vs_stat = vs_stat;
  p.vs_val = vs_val;
  p.vs_idx = vs_idx;
  op->BN = BN;
  op->wide = 1;
  op->grid = p.ftiles * rgroups;
  op->cluster = ln ? 4 : 1;
  op->flops = 2.0 * (double)R * (double)F * (double)K;
  int rc = encode_tmap_2d(&op->tmW, wt, (uint64_t)K, (uint64_t)F, (uint64_t)K, TG_BM);
  if (rc) return rc;
  rc = encode_tmap_2d(&op->tmX_hi, x.p, (uint64_t)K, (uint64_t)R, (uint64_t)x.ld, BN);
  if (rc) return rc;
  op->tmX_lo = op->tmX_hi;
  if (out.p)   // output map of the bulk tensor store (kept in the tmX_lo slot): [R][F] bf16, boxes of 128 rows x 64 features
    rc = encode_tmap_2d(&op->tmX_lo, out.p, (uint64_t)F, (uint64_t)R, (uint64_t)out.ld, TW_ROWS);
  return rc;
}

}  // namespace fpnmt
