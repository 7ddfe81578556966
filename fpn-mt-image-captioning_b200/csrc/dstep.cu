// Group-stationary fused decoder kernel (design: dstep.cuh).
//   warp 0      : weight producer - TMA boxes of the packed weight stream through a 3 x 32 KB ring
//   warp 1      : TMEM allocator + tcgen05.mma issuer (M = 128 features x N = 32 rows x K = 16 per instruction)
//   warps 2..17 : workers - operand staging (embedding, LayerNorm), TMEM epilogues, attention, cluster exchanges, beam tail
#include "dstep.cuh"

#include "tensormap.cuh"

namespace fpnmt {

constexpr int DS_GROUP = 2 * DS_SLOT;                   // bytes per ring slot: two TMA boxes on one mbarrier
constexpr int DS_XB_BYTES = 32768;                      // [32 rows][512] bf16 operand: 8 k-chunks of [32][64] (4 KB, SW128)
constexpr int DS_HB_BYTES = 16384;                      // [32 rows][256] bf16 hidden slice
constexpr int DS_EXTRA_BYTES = 16384;                   // XB | HB | EXTRA = 64 KB: V staging (attention) / selection scratch (tail)
constexpr int DS_OFF_XB = DS_RING * DS_GROUP;
constexpr int DS_OFF_HB = DS_OFF_XB + DS_XB_BYTES;
constexpr int DS_OFF_EXTRA = DS_OFF_HB + DS_HB_BYTES;
constexpr int DS_OFF_Q = DS_OFF_EXTRA + DS_EXTRA_BYTES;   // QS | KS | VS: [32][64] fp32 each
constexpr int DS_OFF_RES = DS_OFF_Q + 3 * 32 * 64 * 4;    // [32][64] fp32 residual slice of this CTA
constexpr int DS_CKV_STRIDE = 144;                        // bytes per staged memory-token row (128 B of K or V + 16 B skew)
constexpr int DS_CKV_ROWS = 64;                           // images of the cluster x memory tokens that fit the staging buffer
constexpr int DS_OFF_CKV = DS_OFF_RES + 32 * 64 * 4;      // cross-attention K | V of the cluster's images, head `cta`
constexpr int DS_OFF_MISC = DS_OFF_CKV + 2 * DS_CKV_ROWS * DS_CKV_STRIDE;
constexpr int DS_MISC_BYTES = 4096;
constexpr int DS_OFF_VB = DS_OFF_MISC + DS_MISC_BYTES;     // final-layer bias of this CTA's vocabulary slice (fp32)
constexpr int DS_OFF_ANC = DS_OFF_VB + DS_MAX_VTILES * 128 * 4;   // beam ancestry of the group's rows as local row bytes [32][64]
constexpr int DS_ANC_T = 64;                               // longest decode whose ancestry fits the byte table
constexpr int DS_SMEM = DS_OFF_ANC + 32 * DS_ANC_T + 1024;
constexpr int DS_W = DS_WORKER_WARPS * 32;                // 512 worker threads
constexpr int DS_CAP = 64;                                // threshold-selection list capacity per (warp, row)
constexpr int DS_NMAX = 16;                               // beam width limit of the fused path
constexpr int NONE_IDX = 0x7fffffff;

size_t dstep_smem_bytes() { return DS_SMEM; }

// ---------------------------------------------------------------------------------------------- small PTX helpers
__device__ __forceinline__ int ds_ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void ds_tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void ds_worker_sync() { asm volatile("bar.sync 1, %0;" ::"n"(DS_W) : "memory"); }
__device__ __forceinline__ void ds_cp16(uint32_t dst, const void* src, bool ok) {
  const int sz = ok ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ bool ds_better(float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); }

// ---------------------------------------------------------------------------------------------- the kernel
__global__ void __launch_bounds__(DS_THREADS, 1) dstep_kernel(const __grid_constant__ CUtensorMap tmW, const DstepParams p) {
  extern __shared__ uint8_t ds_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ds_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* ring = smem;
  uint8_t* XB = smem + DS_OFF_XB;
  uint8_t* HB = smem + DS_OFF_HB;
  uint8_t* SCR = XB;                                               // 64 KB scratch (XB | HB | EXTRA) when no GEMM reads them
  float* QS = reinterpret_cast<float*>(smem + DS_OFF_Q);
  float* KS = QS + 32 * 64;
  float* VS = KS + 32 * 64;
  float* RES = reinterpret_cast<float*>(smem + DS_OFF_RES);
  uint8_t* CKS = smem + DS_OFF_CKV;                                // staged cross-attention K rows, then V rows
  float* VBS = reinterpret_cast<float*>(smem + DS_OFF_VB);         // [ntv * 128]
  uint8_t* ANC8 = smem + DS_OFF_ANC;                               // [32][DS_ANC_T]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + DS_OFF_MISC);
  uint64_t* full = bars;                       // [DS_RING]
  uint64_t* empty = bars + DS_RING;            // [DS_RING]
  uint64_t* x_ready = bars + 2 * DS_RING;      // workers -> MMA warp: the B operand of the next GEMM job is in shared memory
  uint64_t* acc_ready = x_ready + 1;           // MMA warp -> workers: the accumulators of the job are complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_ready + 1);
  unsigned* s_rowidx = reinterpret_cast<unsigned*>(smem + DS_OFF_MISC + 256);   // [16 warps][32]
  int* s_small = reinterpret_cast<int*>(smem + DS_OFF_MISC + 256 + 2048);       // 448 ints of small per-phase state

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x % DS_CTAS;                    // rank inside the 8-CTA group == attention head
  const int cid = p.group0 + blockIdx.x / DS_CTAS;         // group (== "cluster" of the design notes) handled by this CTA
  const int nclusters = p.ngroups;
  const int N = p.N;
  const int row_base = cid * p.ipc * N;
  const int nrows = min(p.R - row_base, p.ipc * N);        // valid rows of this cluster (whole images)
  const int nimg = nrows / N;

  if (threadIdx.x == 0) {
    for (int s = 0; s < DS_RING; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(x_ready, 1);
    mbar_init(acc_ready, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ weight producer
    // The weight stream of this CTA, viewed as a [rows][64] bf16 matrix, is pulled in GROUPS of two TMA boxes (2 x 128 rows
    // x 64 = 32 KB, SWIZZLE_128B) that complete on one mbarrier: the single issuing threads of the producer and MMA warps
    // pay ~250 cycles of barrier wait / commit per group, which at one 16 KB box per barrier (4 tcgen05.mma) capped the
    // stream at ~45 GB/s per SM - measured 0.3-0.45 us per box in the MMA warp even with the data resident.
    // The decode also streams 200-400 MB of K/V cache per step through the 126 MB L2, so the weights do not survive from one
    // step to the next: the producer prefetches the stream into L2 DS_AHEAD groups ahead of its TMA loads.
    const uint32_t leader = elect_one() ? 1u : 0u;
    uint32_t it = 0;                                               // group counter
    if (leader) tma_prefetch_desc(&tmW);
    const int per_step = p.L * 28 + p.ntv * 4;                    // groups of one decode step
    auto group_row = [&](int idx) -> int {                         // stream row (128 B units) of group `idx` of a step
      if (idx < p.L * 28) {
        const int l = idx / 28, i = idx - l * 28;
        return (int)((((size_t)l * DS_CTAS + cta) * DS_LAYER_STREAM) >> 7) + i * 256;
      }
      return (int)((p.final_off + (size_t)cta * p.ntv * 8 * 16384) >> 7) + (idx - p.L * 28) * 256;
    };
    const int total = p.nsteps * per_step;
    constexpr int DS_AHEAD = 12;
    auto l2_prefetch = [&](int n) {
      if (n < total && leader)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p.wstream + (size_t)group_row(n % per_step) * 128), "n"(DS_GROUP) : "memory");
    };
    for (int n = 0; n < DS_AHEAD; ++n) l2_prefetch(n);
    for (int n = 0; n < total; ++n) {
      const uint32_t slot = it % DS_RING;
      const int row = group_row(n % per_step);
      l2_prefetch(n + DS_AHEAD);
      if (it >= DS_RING) mbar_wait(&empty[slot], ((it / DS_RING) & 1) ^ 1);
      mbar_expect_tx_pred(&full[slot], DS_GROUP, leader);
      tma_load_2d_pred(ring + slot * DS_GROUP, &tmW, &full[slot], 0, row, leader);
      tma_load_2d_pred(ring + slot * DS_GROUP + DS_SLOT, &tmW, &full[slot], 0, row + 128, leader);
#ifdef FPNMT_DBG_STAMPS   // issue times of the ffn1 groups of layer 0 in the last step (CTA 0): timeline[174 ..]
      if (p.timeline && blockIdx.x == 0 && leader && n / per_step == p.nsteps - 1 && n % per_step >= 12 && n % per_step < 20) {
        long long t_;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
        p.timeline[174 + n % per_step - 12] = t_;
      }
#endif
      ++it;
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    const uint32_t leader = elect_one() ? 1u : 0u;
    constexpr uint32_t IDESC = umma_idesc_bf16(128, DS_ROWS);
    const uint32_t ring_a = smem_u32(ring), xb_a = smem_u32(XB), hb_a = smem_u32(HB);
    uint32_t it = 0, job = 0;                                      // `it` counts 16 KB units: group = it / 2, half = it & 1
#ifdef FPNMT_DBG_STAMPS
    bool mstamp = false;
    int n_ms = 0;
#define MSTAMP() do { if (mstamp && leader && n_ms < 24) { long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); p.timeline[150 + n_ms++] = t_; } } while (0)
#else
#define MSTAMP() do { } while (0)
#endif
    // one 16 KB unit of the ring: waits for its group at the first half, releases the group after the second half
    auto unit_begin = [&]() -> uint32_t {
      const uint32_t grp = it >> 1, slot = grp % DS_RING;
      if (!(it & 1)) {
        mbar_wait(&full[slot], (grp / DS_RING) & 1);
        MSTAMP();
        tc_fence_after();
      }
      return ring_a + slot * DS_GROUP + (it & 1) * DS_SLOT;
    };
    auto unit_end = [&]() {
      if (it & 1) {
        MSTAMP();   // all MMAs of the group issued
        umma_commit_pred(&empty[(it >> 1) % DS_RING], leader);
      }
      ++it;
    };
    auto tile = [&](uint32_t acc_col, int nchunks, uint32_t b_addr) {   // 128-feature tile: one k-chunk per unit
      for (int kc = 0; kc < nchunks; ++kc) {
        const uint64_t adesc = umma_desc_sw128(unit_begin());
        const uint64_t bdesc = umma_desc_sw128(b_addr + kc * 4096);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16_pred(tmem_base + acc_col, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), IDESC, (kc > 0 || k > 0) ? 1u : 0u, leader);
        unit_end();
      }
    };
    auto tile64 = [&](uint32_t acc_col, uint32_t b_addr) {        // 64-feature tile, K = 512: 4 units of two 8 KB k-chunks;
      for (int s2 = 0; s2 < 4; ++s2) {                             // rows 64..127 of the A descriptor read the neighbouring
        const uint32_t a0 = unit_begin();                          // bytes (lanes 64..127 of the accumulator are never used)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint64_t adesc = umma_desc_sw128(a0 + h * 8192);
          const uint64_t bdesc = umma_desc_sw128(b_addr + (2 * s2 + h) * 4096);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_pred(tmem_base + acc_col, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), IDESC, (s2 > 0 || h > 0 || k > 0) ? 1u : 0u, leader);
        }
        unit_end();
      }
    };
    auto begin_job = [&]() {
      mbar_wait(x_ready, job & 1);
      tc_fence_after();
    };
    auto end_job = [&]() {
      umma_commit_pred(acc_ready, leader);
      ++job;
    };
    for (int s = 0; s < p.nsteps; ++s) {
      for (int l = 0; l < p.L; ++l) {
        begin_job(); tile(0, 8, xb_a); tile64(32, xb_a); end_job();                        // qkv
        begin_job(); tile64(0, xb_a); end_job();                                           // o1
        begin_job(); tile64(0, xb_a); end_job();                                           // q2
        begin_job(); tile64(0, xb_a); end_job();                                           // o2
#ifdef FPNMT_DBG_STAMPS
        mstamp = p.timeline && blockIdx.x == 0 && s == p.nsteps - 1 && l == 0;
#endif
        begin_job(); MSTAMP(); tile(0, 8, xb_a); tile(32, 8, xb_a); end_job(); MSTAMP();   // ffn1
#ifdef FPNMT_DBG_STAMPS
        mstamp = false;
#endif
        begin_job();
        for (int ft = 0; ft < 4; ++ft) tile(64 + 32 * ft, 4, hb_a);                        // ffn2 split-K partials
        end_job();
      }
      begin_job();
      for (int vt = 0; vt < p.ntv; ++vt) tile(32 * vt, 8, xb_a);                           // vocabulary slice
      end_job();
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------------------------------ workers
    const int ww = warp - 2;                       // worker warp 0..15
    const int wt = ww * 32 + lane;                 // worker thread 0..511
    const int q = warp & 3;                        // TMEM lane quarter of this warp
    const int g = ww >> 2;                         // column (row) group: rows g*8 .. g*8+7
    const int r16 = wt >> 4, p16 = wt & 15;        // (row, 1/16 of the row) mapping
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * 8);
    uint32_t job = 0;
    int xtarget = 0;
    const size_t xrow0 = (size_t)cid * 32;         // first row of this cluster in the exchange buffers
#ifdef FPNMT_DBG_STAMPS   // build.py --dbg-stamps + FPNMT_DBG_OP=dstep: phase timeline of the launch's last step (cluster 0, CTA 0)
    int n_stamp = 0;
    bool stamp_on = false;
#define DSTAMP() do { if (stamp_on && n_stamp < 120) { long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); p.timeline[1 + n_stamp++] = t_; p.timeline[0] = n_stamp; } } while (0)
#define DSTAMPL() do { if (l == 0) DSTAMP(); } while (0)
#else
#define DSTAMP() do { } while (0)
#define DSTAMPL() do { } while (0)
#endif

    auto signal_x_ready = [&]() {                  // every worker has written its part of the operand
      fence_proxy_async();
      tc_fence_before();
      ds_worker_sync();
      if (wt == 0) mbar_arrive(x_ready);
    };
    // Only ONE worker warp polls the mbarrier; the other 15 sleep in the hardware barrier.  (With all 512 worker threads
    // spinning in mbarrier.try_wait the MMA warp's tcgen05.mma stream ran 3-4x slower: the polls compete with the MMA operand
    // reads for the shared-memory pipe.)
    auto wait_acc = [&]() {
      if (ww == 0) mbar_wait(acc_ready, job & 1);
      ds_worker_sync();
      tc_fence_after();
      ++job;
    };
    // Barrier among the workers of the group's 8 CTAs: a monotonic counter in global memory (zeroed before the launch),
    // arrive = fence + atomic add by one thread after a CTA barrier, wait = acquire-load spin, second CTA barrier to release
    // the other workers (the pattern of a cooperative grid barrier, restricted to 8 co-resident CTAs).
    auto xsync = [&]() {
      ds_worker_sync();
      if (wt == 0) {
        __threadfence();
        atomicAdd(p.gbar + cid, 1);
        xtarget += DS_CTAS;
        while (ds_ld_acquire(p.gbar + cid) < xtarget) {
        }
      }
      ds_worker_sync();
    };
    // Row mapping of the staging phases: thread (r16, p16) holds the float4 chunks p16 + 16 i (i = 0..7) of row r16, i.e.
    // x[4i .. 4i+3] = features 64 i + 4 p16 .. +3.  The 16 lanes of a row then read 256 contiguous bytes per load instruction
    // (a per-thread contiguous 128 B slice made every load touch 32 different lines and was bound by the L1 wavefront rate:
    // 9 us per LayerNorm staging instead of ~1 us), chunk i lands in k-chunk i of the operand, and the 16 lanes write one
    // 128 B operand row per store instruction.  x -> bf16 operand (SW128 K-major) + this CTA's fp32 residual slice.
    auto store_operand = [&](const float* x) {
      uint8_t* base = XB + r16 * 128 + (((p16 >> 1) ^ (r16 & 7)) << 4) + (p16 & 1) * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        *reinterpret_cast<uint2*>(base + i * 4096) = make_uint2(pack2(x[4 * i], x[4 * i + 1]), pack2(x[4 * i + 2], x[4 * i + 3]));
        if (i == cta) *reinterpret_cast<float4*>(RES + r16 * 64 + p16 * 4) = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
      }
    };
    // LayerNorm (eps 1e-6) of the exchanged pre-activation rows; every CTA normalises all 32 rows itself
    auto ln_load = [&](const float* gam, const float* bet, int l, int which) {
      float x[32];
      const float4* src = reinterpret_cast<const float4*>(p.x_pre + (xrow0 + r16) * 512) + p16;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 v = __ldcg(src + 16 * i);
        x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
      }
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) s += x[i];
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float mean = s * (1.f / 512.f);
      float m2 = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float d = x[i] - mean;
        m2 = fmaf(d, d, m2);
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
      const float rstd = rsqrtf(m2 * (1.f / 512.f) + 1e-6f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 ga = __ldg(reinterpret_cast<const float4*>(gam) + p16 + 16 * i);
        const float4 be = __ldg(reinterpret_cast<const float4*>(bet) + p16 + 16 * i);
        x[4 * i] = (x[4 * i] - mean) * rstd * ga.x + be.x;
        x[4 * i + 1] = (x[4 * i + 1] - mean) * rstd * ga.y + be.y;
        x[4 * i + 2] = (x[4 * i + 2] - mean) * rstd * ga.z + be.z;
        x[4 * i + 3] = (x[4 * i + 3] - mean) * rstd * ga.w + be.w;
      }
      store_operand(x);
      if (p.dbg && cta == 0) {
        float4* d = reinterpret_cast<float4*>(p.dbg + (((size_t)(l * 3 + which) * nclusters * 32) + xrow0 + r16) * 512) + p16;
#pragma unroll
        for (int i = 0; i < 8; ++i) d[16 * i] = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
      }
    };
    auto load_att_operand = [&]() {                // x_att rows (bf16) -> operand, no conversion
      // 16-byte chunks p16 + 16 i (8 features each): k-chunk 2 i + (p16 >> 3), position p16 & 7 inside its 128 B row
      const uint4* src = reinterpret_cast<const uint4*>(p.x_att + (xrow0 + r16) * 512) + p16;
      uint8_t* base = XB + (p16 >> 3) * 4096 + r16 * 128 + (((p16 & 7) ^ (r16 & 7)) << 4);
      uint4 v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = __ldcg(src + 16 * i);
#pragma unroll
      for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(base + i * 8192) = v[i];
    };
    // 64-feature Dense slice epilogue: acc + bias + residual slice -> exchanged pre-LayerNorm rows
    auto epi_slice = [&](const float* bias) {
      if (q < 2) {
        float v[8];
        ds_tmem_ld8(t_lane, v);
        const int f = q * 32 + lane;
        const float b = __ldg(bias + cta * 64 + f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int row = g * 8 + j;
          p.x_pre[(xrow0 + row) * 512 + cta * 64 + f] = v[j] + b + RES[row * 64 + f];
        }
      }
    };

    for (int i = wt; i < p.ntv * 128; i += DS_W) VBS[i] = __ldg(p.vbias + cta * p.vslice + i);
    const bool anc_smem = p.T <= DS_ANC_T && (p.T & 3) == 0;   // (16-byte aligned ancestry rows)
    for (int s = 0; s < p.nsteps; ++s) {
      const int t = p.t0 + s;
      const int cur = t & 1, nxt = cur ^ 1;
#ifdef FPNMT_DBG_STAMPS
      stamp_on = p.timeline && wt == 0 && cid == 0 && cta == 0 && s == p.nsteps - 1;
#endif
      DSTAMP();   // step start
      // ---- decoder input: x = embedding[token] + pos[t]  (transformer.py:326-329; no sqrt(d) scaling, :327 is commented out)
      bool anc_differs = false;
      {
        float x[32];
        if (r16 < nrows) {
          const int tok = __ldcg(p.st.last_tok + row_base + r16);
          const float4* e = reinterpret_cast<const float4*>(p.emb + (size_t)tok * 512) + p16;
          const float4* ps = reinterpret_cast<const float4*>(p.pos + (size_t)t * 512) + p16;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 a = __ldg(e + 16 * i), b = __ldg(ps + 16 * i);
            x[4 * i] = a.x + b.x; x[4 * i + 1] = a.y + b.y; x[4 * i + 2] = a.z + b.z; x[4 * i + 3] = a.w + b.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) x[i] = 0.f;
        }
        store_operand(x);
        // beam ancestry of the group's rows for this step -> shared memory (local row index, one byte per position): the
        // six attention phases and prefetch passes of the step then need no dependent global load for the cache addresses
        if (anc_smem && r16 < nrows && p16 * 4 < t) {
          // ancestry of the row's REPRESENTATIVE (DstepParams::rep); teacher forcing keeps every row on its own
          const int rrow = (p.mode == 0) ? __ldcg(p.rep + (size_t)cur * p.R + row_base + r16) : row_base + r16;
          const int4 a = __ldcg(reinterpret_cast<const int4*>(p.st.anc[cur] + (size_t)rrow * p.T) + p16);
          *reinterpret_cast<uchar4*>(ANC8 + r16 * DS_ANC_T + p16 * 4) =
              make_uchar4((unsigned char)(a.x - row_base), (unsigned char)(a.y - row_base), (unsigned char)(a.z - row_base), (unsigned char)(a.w - row_base));
          // does this row share the ancestry of its image's first beam?  (positions >= t are not compared)
          const int4 f = __ldcg(reinterpret_cast<const int4*>(p.st.anc[cur] + (size_t)(row_base + (r16 / N) * N) * p.T) + p16);
          const int rem = t - p16 * 4;
          anc_differs = (a.x != f.x) | (rem > 1 && a.y != f.y) | (rem > 2 && a.z != f.z) | (rem > 3 && a.w != f.w);
        }
      }
      // uniform == every image of the group has ONE ancestry shared by all its beams (always true under the reference's
      // beam initialisation, pipeline.py:101-102; usually false for a true beam search): the attention phases then read each
      // K/V line once per image instead of once per beam.  bar.red doubles as the worker barrier.
      bool uniform;
      {
        int r;
        asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %1, 0;\n\tbar.red.or.pred q, 1, %2, p;\n\tselp.b32 %0, 1, 0, q;\n\t}\n"
                     : "=r"(r) : "r"(anc_differs ? 1 : 0), "n"(DS_W) : "memory");
        uniform = anc_smem && !r;
      }
      signal_x_ready();
      DSTAMP();   // embedding staged

      for (int l = 0; l < p.L; ++l) {
        const float* lp = p.lparams + (size_t)l * DSB_SIZE;
        // cross-attention K / V rows of the cluster's images for head `cta` (constant during the decode): staged with cp.async
        // now, consumed after the q2 projection.  Row = (local image, memory token), 128 B of K resp. V, skewed by 16 B.
        const bool ckv_staged = p.ipc * p.n_mem <= DS_CKV_ROWS;
        if (ckv_staged) {
          const int nck = p.ipc * p.n_mem * 16;                       // 16-byte units: rows x (8 of K + 8 of V)
          for (int u = wt; u < nck; u += DS_W) {
            const int rowi2 = u >> 4, part = u & 15;                  // part 0..7: K, 8..15: V
            const int img = min(cid * p.ipc + rowi2 / p.n_mem, p.B - 1);
            const bf16* src = p.ckv + ((size_t)img * p.n_mem + rowi2 % p.n_mem) * p.ckv_ld + (size_t)l * 1024 + (part >> 3) * 512 + cta * 64 + (part & 7) * 8;
            ds_cp16(smem_u32(CKS + (part >> 3) * DS_CKV_ROWS * DS_CKV_STRIDE + rowi2 * DS_CKV_STRIDE + (part & 7) * 16), src, true);
          }
          asm volatile("cp.async.commit_group;" ::: "memory");
        }
        // ================================================================== qkv epilogue -> self-attention of head `cta`
        wait_acc();
        DSTAMPL();   // qkv accumulators ready
        {
          float v[8];
          ds_tmem_ld8(t_lane, v);                                   // tile [q_c | k_c]
          const int f = q * 32 + lane;
          const float b = __ldg(lp + (q < 2 ? DSB_Q + cta * 64 + f : DSB_K + cta * 64 + f - 64));
          float* dst = (q < 2 ? QS : KS) + (f & 63);
          const float sc = q < 2 ? 0.125f : 1.f;                    // 1 / sqrt(depth) folded into q (transformer.py:91-92)
#pragma unroll
          for (int j = 0; j < 8; ++j) dst[(g * 8 + j) * 64] = (v[j] + b) * sc;
          if (q < 2) {
            ds_tmem_ld8(t_lane + 32, v);                            // tile [v_c]
            const float bv = __ldg(lp + DSB_V + cta * 64 + f);
#pragma unroll
            for (int j = 0; j < 8; ++j) VS[(g * 8 + j) * 64 + f] = v[j] + bv;
          }
        }
        tc_fence_before();
        ds_worker_sync();
        DSTAMPL();   // qkv epilogue done
        // append K/V of position t to the cache (bf16)
        if (r16 < nrows) {
          const float* src = (p16 < 8 ? KS : VS) + r16 * 64 + (p16 & 7) * 8;
          bf16* dstc = (p16 < 8 ? p.kcache : p.vcache) + (((size_t)l * p.R + row_base + r16) * p.T + t) * 512 + cta * 64 + (p16 & 7) * 8;
          *reinterpret_cast<uint4*>(dstc) = pack8(src);
        }
        // self-attention (transformer.py:88-102 with the causal mask implicit)
        if (uniform) {
          // ---- uniform ancestry: task = (image, 16-position chunk); the task's K/V lines are loaded ONCE (registers) and
          // used by all N beams of the image; per (row, chunk) partial (max, sum, o[64]) go to shared memory and are merged
          // with the new position afterwards.  K/V traffic per CTA: t x 256 B per image instead of per row.
          float* part = reinterpret_cast<float*>(SCR);                    // [32 rows][4 chunks][68]
          const int pg = lane >> 3, dg = lane & 7;
          const bf16* kc_l = p.kcache + (size_t)l * p.R * p.T * 512 + cta * 64 + dg * 8;
          const bf16* vc_l = p.vcache + (size_t)l * p.R * p.T * 512 + cta * 64 + dg * 8;
          for (int task = ww; task < nimg * 4; task += DS_WORKER_WARPS) {
            const int il = task >> 2, c = task & 3;
            float kf[4][8];
            uint4 vh[4];
            bool ok[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int pos = 16 * c + pg + 4 * i;
              ok[i] = pos < t;
              const size_t off = ok[i] ? ((size_t)(row_base + (int)ANC8[il * N * DS_ANC_T + pos]) * p.T + pos) * 512 : 0;
              const uint4 kq = ok[i] ? __ldcg(reinterpret_cast<const uint4*>(kc_l + off)) : make_uint4(0u, 0u, 0u, 0u);
              vh[i] = ok[i] ? __ldcg(reinterpret_cast<const uint4*>(vc_l + off)) : make_uint4(0u, 0u, 0u, 0u);
              unpack8(kq, kf[i]);
            }
            for (int n = 0; n < N; ++n) {
              const int lr = il * N + n;
              float q8[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) q8[j] = QS[lr * 64 + dg * 8 + j];
              float sc[4], cmax = -INFINITY;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                float a = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) a = fmaf(q8[j], kf[i][j], a);
                a += __shfl_xor_sync(0xffffffffu, a, 1);
                a += __shfl_xor_sync(0xffffffffu, a, 2);
                a += __shfl_xor_sync(0xffffffffu, a, 4);
                sc[i] = ok[i] ? a : -INFINITY;
                cmax = fmaxf(cmax, sc[i]);
              }
              cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, 8));
              cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, 16));
              float psum = 0.f, o[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) o[j] = 0.f;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float pr = ok[i] ? __expf(sc[i] - cmax) : 0.f;
                psum += pr;
                float f[8];
                unpack8(vh[i], f);
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = fmaf(pr, f[j], o[j]);
              }
              psum += __shfl_xor_sync(0xffffffffu, psum, 8);
              psum += __shfl_xor_sync(0xffffffffu, psum, 16);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                o[j] += __shfl_xor_sync(0xffffffffu, o[j], 8);
                o[j] += __shfl_xor_sync(0xffffffffu, o[j], 16);
              }
              if (pg == 0) {
                float* pp = part + (lr * 4 + c) * 68;
                *reinterpret_cast<float4*>(pp + 4 + dg * 8) = make_float4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<float4*>(pp + 8 + dg * 8) = make_float4(o[4], o[5], o[6], o[7]);
                if (dg == 0) {
                  pp[0] = cmax;
                  pp[1] = psum;
                }
              }
            }
          }
          ds_worker_sync();
          for (int rr = 0; rr < 2; ++rr) {       // merge the chunk partials of a row with the new position (K/V in fp32 shared memory)
            const int lr = ww * 2 + rr;
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = 0.f;
            if (lr < nrows) {
              const float scn = warp_sum(QS[lr * 64 + 2 * lane] * KS[lr * 64 + 2 * lane] + QS[lr * 64 + 2 * lane + 1] * KS[lr * 64 + 2 * lane + 1]);
              const float* pp = part + lr * 4 * 68;
              float M = scn;
#pragma unroll
              for (int c = 0; c < 4; ++c) M = fmaxf(M, pp[c * 68]);
              const float pn = __expf(scn - M);
              float lsum = pn;
              const int d8 = (lane & 7) * 8;
#pragma unroll
              for (int i = 0; i < 8; ++i) o[i] = pn * VS[lr * 64 + d8 + i];
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                const float mc = pp[c * 68];
                if (mc > -INFINITY) {
                  const float w = __expf(mc - M);
                  lsum = fmaf(pp[c * 68 + 1], w, lsum);
                  const float4 a = *reinterpret_cast<const float4*>(pp + c * 68 + 4 + d8), b = *reinterpret_cast<const float4*>(pp + c * 68 + 8 + d8);
                  o[0] = fmaf(a.x, w, o[0]); o[1] = fmaf(a.y, w, o[1]); o[2] = fmaf(a.z, w, o[2]); o[3] = fmaf(a.w, w, o[3]);
                  o[4] = fmaf(b.x, w, o[4]); o[5] = fmaf(b.y, w, o[5]); o[6] = fmaf(b.z, w, o[6]); o[7] = fmaf(b.w, w, o[7]);
                }
              }
              const float inv = 1.f / lsum;
#pragma unroll
              for (int i = 0; i < 8; ++i) o[i] *= inv;
            }
            if (lane < 8) *reinterpret_cast<uint4*>(p.x_att + (xrow0 + lr) * 512 + cta * 64 + lane * 8) = pack8(o);
          }
        } else {
          uint4* vst = reinterpret_cast<uint4*>(SCR + ww * 4096);       // V rows of the current 32-position chunk
          unsigned* rowi = s_rowidx + ww * 32;
          const int pg = lane >> 3, dg = lane & 7;
          const bf16* kc_l = p.kcache + (size_t)l * p.R * p.T * 512 + cta * 64;
          const bf16* vc_l = p.vcache + (size_t)l * p.R * p.T * 512 + cta * 64;
          for (int rr = 0; rr < 2; ++rr) {
            const int lr = ww * 2 + rr;
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = 0.f;
            float m = -INFINITY, lsum = 0.f;
            if (lr < nrows) {
              const int* anc = p.st.anc[cur] + (size_t)(row_base + lr) * p.T;
              float q8[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) q8[j] = QS[lr * 64 + dg * 8 + j];
              for (int k0 = 0; k0 < t; k0 += 32) {
                const int pos = k0 + lane;
                const int kmax = min(32, t - k0);
                const int arow = (pos < t) ? (anc_smem ? row_base + (int)ANC8[lr * DS_ANC_T + pos] : __ldcg(anc + pos)) : 0;
                rowi[lane] = (pos < t) ? (unsigned)(arow * p.T + pos) : 0u;
                __syncwarp();
                {
                  const uint32_t d0 = smem_u32(vst);
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const int u = i * 32 + lane, r = u >> 3;
                    const bool ok = r < kmax;
                    ds_cp16(d0 + u * 16, vc_l + (size_t)rowi[ok ? r : 0] * 512 + (u & 7) * 8, ok);
                  }
                  asm volatile("cp.async.commit_group;" ::: "memory");
                }
                float sc[8];
                {
                  uint4 kh[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const int pp = pg + 4 * i;
                    kh[i] = __ldcg(reinterpret_cast<const uint4*>(kc_l + (size_t)rowi[pp < kmax ? pp : 0] * 512 + dg * 8));
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
                  sc[i] = (pg + 4 * i < kmax) ? __expf(sc[i] - mn) : 0.f;
                  psum += sc[i];
                }
                psum += __shfl_xor_sync(0xffffffffu, psum, 8);
                psum += __shfl_xor_sync(0xffffffffu, psum, 16);
                lsum = lsum * corr + psum;
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
                    unpack8(vst[pp * 8 + dg], f);
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = fmaf(sc[i], f[j], o[j]);
                  }
                }
                __syncwarp();
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {          // sum the four position groups: lanes 0..7 hold dims lane*8 .. +7
                o[i] += __shfl_xor_sync(0xffffffffu, o[i], 8);
                o[i] += __shfl_xor_sync(0xffffffffu, o[i], 16);
              }
              // the new position itself (K/V in shared memory, fp32)
              const float scn = warp_sum(QS[lr * 64 + 2 * lane] * KS[lr * 64 + 2 * lane] + QS[lr * 64 + 2 * lane + 1] * KS[lr * 64 + 2 * lane + 1]);
              const float mn = fmaxf(m, scn);
              const float corr = __expf(m - mn);
              const float pn = __expf(scn - mn);
              lsum = lsum * corr + pn;
              const float inv = 1.f / lsum;
#pragma unroll
              for (int i = 0; i < 8; ++i) o[i] = (o[i] * corr + pn * VS[lr * 64 + (lane & 7) * 8 + i]) * inv;
            }
            if (lane < 8) *reinterpret_cast<uint4*>(p.x_att + (xrow0 + lr) * 512 + cta * 64 + lane * 8) = pack8(o);
          }
        }
        DSTAMPL();   // self-attention done
        xsync();                                                    // A: attention heads of all CTAs
        DSTAMPL();   // barrier A
        load_att_operand();
        signal_x_ready();
        DSTAMPL();   // att operand staged
        // ================================================================== o1 + residual -> LayerNorm1
        wait_acc();
        DSTAMPL();   // o1 accumulators ready
        epi_slice(lp + DSB_O1);
        tc_fence_before();
        DSTAMPL();   // o1 epilogue
        xsync();                                                    // B
        DSTAMPL();   // barrier B
        ln_load(lp + DSB_LN1G, lp + DSB_LN1B, l, 0);
        signal_x_ready();
        DSTAMPL();   // LN1 staged
        // ================================================================== q2 -> cross-attention over the memory tokens
        wait_acc();
        DSTAMPL();   // q2 accumulators ready
        if (q < 2) {
          float v[8];
          ds_tmem_ld8(t_lane, v);
          const int f = q * 32 + lane;
          const float b = __ldg(lp + DSB_Q2 + cta * 64 + f);
#pragma unroll
          for (int j = 0; j < 8; ++j) QS[(g * 8 + j) * 64 + f] = (v[j] + b) * 0.125f;
        }
        tc_fence_before();
        ds_worker_sync();
        if (ckv_staged) {
          asm volatile("cp.async.wait_group 0;" ::: "memory");
          ds_worker_sync();
          const int il = min(r16 / N, p.ipc - 1);                   // local image of the row
          const int j = p16;                                        // memory token of this thread
          const uint8_t* kb = CKS + (il * p.n_mem) * DS_CKV_STRIDE;
          const uint8_t* vb = kb + DS_CKV_ROWS * DS_CKV_STRIDE;
          float sc = -INFINITY;
          if (j < p.n_mem) {
            const uint4* kr = reinterpret_cast<const uint4*>(kb + j * DS_CKV_STRIDE);
            float a = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float f[8];
              unpack8(kr[i], f);
#pragma unroll
              for (int d = 0; d < 8; ++d) a = fmaf(QS[r16 * 64 + i * 8 + d], f[d], a);
            }
            sc = a;
          }
          float mx = sc;
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          float pr = (j < p.n_mem) ? __expf(sc - mx) : 0.f;
          float sm = pr;
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
          pr /= sm;
          float o4[4] = {0.f, 0.f, 0.f, 0.f};
          for (int jj = 0; jj < p.n_mem; ++jj) {
            const float pj = __shfl_sync(0xffffffffu, pr, (lane & 16) | jj);
            const uint2 u = *reinterpret_cast<const uint2*>(vb + jj * DS_CKV_STRIDE + p16 * 8);
            o4[0] = fmaf(pj, __uint_as_float(u.x << 16), o4[0]);
            o4[1] = fmaf(pj, __uint_as_float(u.x & 0xffff0000u), o4[1]);
            o4[2] = fmaf(pj, __uint_as_float(u.y << 16), o4[2]);
            o4[3] = fmaf(pj, __uint_as_float(u.y & 0xffff0000u), o4[3]);
          }
          *reinterpret_cast<uint2*>(p.x_att + (xrow0 + r16) * 512 + cta * 64 + p16 * 4) = make_uint2(pack2(o4[0], o4[1]), pack2(o4[2], o4[3]));
        } else {
          const int img = min((row_base + r16) / N, p.B - 1);
          const int j = p16;                                        // memory token of this thread
          const bf16* kv = p.ckv + (size_t)img * p.n_mem * p.ckv_ld + (size_t)l * 1024 + cta * 64;
          float sc = -INFINITY;
          if (j < p.n_mem) {
            const uint4* kr = reinterpret_cast<const uint4*>(kv + (size_t)j * p.ckv_ld);
            float a = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float f[8];
              unpack8(__ldg(kr + i), f);
#pragma unroll
              for (int d = 0; d < 8; ++d) a = fmaf(QS[r16 * 64 + i * 8 + d], f[d], a);
            }
            sc = a;
          }
          float mx = sc;
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          float pr = (j < p.n_mem) ? __expf(sc - mx) : 0.f;
          float sm = pr;
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
          pr /= sm;
          float o4[4] = {0.f, 0.f, 0.f, 0.f};
          const bf16* vr = kv + 512 + p16 * 4;                      // this thread's 4 output dims
          for (int jj = 0; jj < p.n_mem; ++jj) {
            const float pj = __shfl_sync(0xffffffffu, pr, (lane & 16) | jj);
            const uint2 u = __ldg(reinterpret_cast<const uint2*>(vr + (size_t)jj * p.ckv_ld));
            o4[0] = fmaf(pj, __uint_as_float(u.x << 16), o4[0]);
            o4[1] = fmaf(pj, __uint_as_float(u.x & 0xffff0000u), o4[1]);
            o4[2] = fmaf(pj, __uint_as_float(u.y << 16), o4[2]);
            o4[3] = fmaf(pj, __uint_as_float(u.y & 0xffff0000u), o4[3]);
          }
          *reinterpret_cast<uint2*>(p.x_att + (xrow0 + r16) * 512 + cta * 64 + p16 * 4) = make_uint2(pack2(o4[0], o4[1]), pack2(o4[2], o4[3]));
        }
        DSTAMPL();   // cross-attention done
        xsync();                                                    // C
        load_att_operand();
        signal_x_ready();
        DSTAMPL();   // barrier C + operand staged
        // ================================================================== o2 + residual -> LayerNorm2
        wait_acc();
        DSTAMPL();   // o2 accumulators ready
        epi_slice(lp + DSB_O2);
        tc_fence_before();
        xsync();                                                    // D
        ln_load(lp + DSB_LN2G, lp + DSB_LN2B, l, 1);
        signal_x_ready();
        DSTAMPL();   // barrier D + LN2 staged
        // ================================================================== ffn1 + LeakyReLU(0.2) -> hidden slice operand
        wait_acc();
        DSTAMPL();   // ffn1 accumulators ready
#pragma unroll
        for (int ft = 0; ft < 2; ++ft) {
          float v[8];
          ds_tmem_ld8(t_lane + 32 * ft, v);
          const int hf = ft * 128 + q * 32 + lane;
          const float b = __ldg(lp + DSB_F1 + cta * 256 + hf);
          uint8_t* base = HB + (hf >> 6) * 4096 + (hf & 7) * 2;
          const int c16 = (hf & 63) >> 3;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int row = g * 8 + j;
            float y = v[j] + b;
            y = y >= 0.f ? y : 0.2f * y;
            *reinterpret_cast<bf16*>(base + row * 128 + ((c16 ^ (row & 7)) << 4)) = __float2bfloat16_rn(y);
          }
        }
        signal_x_ready();
        DSTAMPL();   // hidden operand staged
        // ================================================================== ffn2 split-K partials -> reduce -> LayerNorm3
        wait_acc();
        DSTAMPL();   // ffn2 accumulators ready
#pragma unroll
        for (int ft = 0; ft < 4; ++ft) {
          float v[8];
          ds_tmem_ld8(t_lane + 64 + 32 * ft, v);
          float* dst = p.x_part + (((size_t)cid * DS_CTAS + cta) * 32 + g * 8) * 512 + ft * 128 + q * 32 + lane;
#pragma unroll
          for (int j = 0; j < 8; ++j) dst[j * 512] = v[j];
        }
        tc_fence_before();
        DSTAMPL();   // partials written
        xsync();                                                    // E
        DSTAMPL();   // barrier E
        {
          float4 a = __ldg(reinterpret_cast<const float4*>(lp + DSB_F2 + cta * 64 + p16 * 4));
          const float4 rs = *reinterpret_cast<const float4*>(RES + r16 * 64 + p16 * 4);
          a.x += rs.x; a.y += rs.y; a.z += rs.z; a.w += rs.w;
#pragma unroll
          for (int c2 = 0; c2 < DS_CTAS; ++c2) {
            const float4 v = __ldcg(reinterpret_cast<const float4*>(p.x_part + (((size_t)cid * DS_CTAS + c2) * 32 + r16) * 512 + cta * 64 + p16 * 4));
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
          }
          *reinterpret_cast<float4*>(p.x_pre + (xrow0 + r16) * 512 + cta * 64 + p16 * 4) = a;
        }
        DSTAMPL();   // reduced
        xsync();                                                    // F
        ln_load(lp + DSB_LN3G, lp + DSB_LN3B, l, 2);
        signal_x_ready();
        DSTAMPL();   // barrier F + LN3 staged (layer end)
      }

      // ==================================================================== vocabulary projection epilogue + beam tail
      wait_acc();
      DSTAMP();   // vocabulary accumulators ready
      const int vbase = cta * p.vslice + q * 32 + lane;             // vocabulary id of this thread in tile 0
      if (p.mode == 1) {
        for (int vt = 0; vt < p.ntv; ++vt) {
          float v[8];
          ds_tmem_ld8(t_lane + 32 * vt, v);
          const int vid = vbase + vt * 128;
          const float b = VBS[vt * 128 + q * 32 + lane];
          if (vid < p.V) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (g * 8 + j < nrows) p.logits_out[(size_t)(row_base + g * 8 + j) * p.ld_logits + vid] = v[j] + b;
          }
        }
        tc_fence_before();
        ds_worker_sync();
        continue;
      }
      // ---- per (warp, row): maxima, selection threshold, sum of exponentials, top-N of the warp's 32 x ntv logits
      float* s_lv = reinterpret_cast<float*>(SCR);                   // [16][8][CAP]   (XB | HB | EXTRA: free during the tail)
      int* s_li = reinterpret_cast<int*>(SCR + 32768);               // [16][8][CAP]
      float* s_wv = QS;                                              // [16][8][DS_NMAX] warp-level winners (QS | KS | VS: free)
      int* s_wi = reinterpret_cast<int*>(QS + 2048);                 // [16][8][DS_NMAX]
      float* s_wm = QS + 4096;                                       // [16][8] warp max
      float* s_ws = s_wm + 128;                                      // [16][8] warp sum-exp
      int* s_cnt = s_small;                                          // [16][8]
      {
        float lmax[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) lmax[j] = -INFINITY;
        for (int vt = 0; vt < p.ntv; ++vt) {
          float v[8];
          ds_tmem_ld8(t_lane + 32 * vt, v);
          const int vid = vbase + vt * 128;
          if (vid < p.V) {
            const float b = VBS[vt * 128 + q * 32 + lane];
#pragma unroll
            for (int j = 0; j < 8; ++j) lmax[j] = fmaxf(lmax[j], v[j] + b);
          }
        }
        // Selection threshold of a row: split the 32 lanes into G >= N groups of 32 / G lanes (G = 8, 16: a power of two);
        // each group's maximum is an element of its own, so at least N elements reach tau = the smallest group maximum.
        // 5 shuffles per row (an exact N-th largest of the 32 lane maxima by rank counting cost 32 and ~4x the time); the
        // bound is a little looser - ~18 survivors per (warp, row) instead of ~9 at V = 10^4 - hence the list capacity of 64.
        float tau[8], wmax[8];
        const int gl = N <= 8 ? 4 : 2;               // lanes per group
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float gm = lmax[j];
          for (int o = 1; o < gl; o <<= 1) gm = fmaxf(gm, __shfl_xor_sync(0xffffffffu, gm, o));   // group maximum
          float mn = gm, mx = gm;
          for (int o = gl; o < 32; o <<= 1) {
            mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          }
          tau[j] = mn;
          wmax[j] = mx;
        }
        DSTAMP();   // tail: maxima + thresholds
        if (lane < 8) s_cnt[ww * 8 + lane] = 0;
        __syncwarp();
        float sum[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) sum[j] = 0.f;
        for (int vt = 0; vt < p.ntv; ++vt) {
          float v[8];
          ds_tmem_ld8(t_lane + 32 * vt, v);
          const int vid = vbase + vt * 128;
          if (vid < p.V) {
            const float b = VBS[vt * 128 + q * 32 + lane];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float x = v[j] + b;
              sum[j] += __expf(x - wmax[j]);
              if (x >= tau[j]) {
                const int pos = atomicAdd(&s_cnt[ww * 8 + j], 1);
                if (pos < DS_CAP) {
                  s_lv[(ww * 8 + j) * DS_CAP + pos] = x;
                  s_li[(ww * 8 + j) * DS_CAP + pos] = vid;
                }
              }
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float sj = warp_sum(sum[j]);
          if (lane == 0) {
            s_wm[ww * 8 + j] = wmax[j];
            s_ws[ww * 8 + j] = (wmax[j] > -INFINITY) ? sj : 0.f;
          }
        }
        __syncwarp();
        DSTAMP();   // tail: pass 2 (sum-exp + survivor lists)
        for (int j = 0; j < 8; ++j) {
          const int cnt = s_cnt[ww * 8 + j];
          float* wv = s_wv + (ww * 8 + j) * DS_NMAX;
          int* wi = s_wi + (ww * 8 + j) * DS_NMAX;
          if (cnt <= DS_CAP) {                       // rank the few survivors by counting (value desc, id asc)
            const float* lv = s_lv + (ww * 8 + j) * DS_CAP;
            const int* li = s_li + (ww * 8 + j) * DS_CAP;
            for (int e0 = lane; e0 < cnt; e0 += 32) {
              const float v = lv[e0];
              const int id = li[e0];
              int rank = 0;
              for (int e = 0; e < cnt; ++e) rank += ds_better(lv[e], li[e], v, id) ? 1 : 0;
              if (rank < N) {
                wv[rank] = v;
                wi[rank] = id;
              }
            }
            if (lane >= cnt && lane < N) {
              wv[lane] = -INFINITY;
              wi[lane] = NONE_IDX;
            }
          } else {
            // exact fallback for massive ties: N rounds of "best element strictly after the previous winner"
            float pv = INFINITY;
            int pi = -1;
            for (int k = 0; k < N; ++k) {
              float bv = -INFINITY;
              int bi = NONE_IDX;
              for (int vt = 0; vt < p.ntv; ++vt) {
                float v[8];
                ds_tmem_ld8(t_lane + 32 * vt, v);
                const int vid = vbase + vt * 128;
                if (vid < p.V) {
                  float x = 0.f;
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj)
                    if (jj == j) x = v[jj];
                  x += VBS[vt * 128 + q * 32 + lane];
                  const bool after = (x < pv) || (x == pv && vid > pi);
                  if (after && ds_better(x, vid, bv, bi)) {
                    bv = x;
                    bi = vid;
                  }
                }
              }
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ds_better(ov, oi, bv, bi)) {
                  bv = ov;
                  bi = oi;
                }
              }
              if (lane == 0) {
                wv[k] = bv;
                wi[k] = bi;
              }
              pv = bv;
              pi = bi;
            }
          }
        }
      }
      tc_fence_before();
      ds_worker_sync();
      DSTAMP();   // warp-level selection done
      // ---- CTA level: merge the 4 quarter-warps of every row -> exchanged per-CTA candidates and (max, sum-exp)
      {
        const int gr = r16 >> 3, jr = r16 & 7;      // the 4 warps gr*4 .. gr*4+3 hold row r16 (as their local row jr)
        const int n4 = 4 * N;
        for (int e = p16; e < n4; e += 16) {
          const int wq = gr * 4 + e / N, k = e % N;
          const float v = s_wv[(wq * 8 + jr) * DS_NMAX + k];
          const int id = s_wi[(wq * 8 + jr) * DS_NMAX + k];
          int rank = 0;
          for (int qi = 0, e2 = 0; qi < 4; ++qi) {
            const float* v2p = s_wv + ((gr * 4 + qi) * 8 + jr) * DS_NMAX;
            const int* i2p = s_wi + ((gr * 4 + qi) * 8 + jr) * DS_NMAX;
            for (int k2 = 0; k2 < N; ++k2, ++e2) {
              const float v2 = v2p[k2];
              const int i2 = i2p[k2];
              rank += (v2 > v || (v2 == v && (i2 < id || (i2 == id && e2 < e)))) ? 1 : 0;
            }
          }
          if (rank < N) {
            p.x_cval[((xrow0 + r16) * DS_CTAS + cta) * N + rank] = v;
            p.x_cidx[((xrow0 + r16) * DS_CTAS + cta) * N + rank] = id;
          }
        }
        if (p16 == 0) {
          float M = -INFINITY;
#pragma unroll
          for (int i = 0; i < 4; ++i) M = fmaxf(M, s_wm[(gr * 4 + i) * 8 + jr]);
          float S = 0.f;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float mi = s_wm[(gr * 4 + i) * 8 + jr];
            if (mi > -INFINITY) S += s_ws[(gr * 4 + i) * 8 + jr] * __expf(mi - M);
          }
          p.x_stat[((xrow0 + r16) * DS_CTAS + cta) * 2] = M;
          p.x_stat[((xrow0 + r16) * DS_CTAS + cta) * 2 + 1] = S;
        }
      }
      DSTAMP();   // CTA-level merge done
      xsync();                                                      // T1: candidates of all vocabulary slices
      DSTAMP();   // barrier T1
      // ---- per image (CTA i handles images i, i+8, ..): row top-N over the 8 slices, then N x N -> N beams
      for (int im = cta; im < nimg; im += DS_CTAS) {
        float* m_v = reinterpret_cast<float*>(SCR);                  // [N][8N] logits
        int* m_i = reinterpret_cast<int*>(SCR + 8192);               // [N][8N] vocabulary ids
        float* r_c = reinterpret_cast<float*>(SCR + 16384);          // [N][N] row winners: candidate scores
        int* r_i = reinterpret_cast<int*>(SCR + 16384 + 1024);       // [N][N] ids
        float* s_lse = reinterpret_cast<float*>(SCR + 16384 + 2048); // [N]
        int* s_parent = s_small + 128;                               // [N]
        int* s_token = s_small + 160;                                // [N]
        const int n8 = 8 * N;
        const int rows0 = row_base + im * N;                         // first global row of the image
        const size_t xr0 = xrow0 + (size_t)im * N;
        ds_worker_sync();                                            // scratch reuse across the image loop
        for (int e = wt; e < N * n8; e += DS_W) {
          const int n = e / n8, k = e % n8;
          m_v[e] = __ldcg(p.x_cval + (xr0 + n) * n8 + k);
          m_i[e] = __ldcg(p.x_cidx + (xr0 + n) * n8 + k);
        }
        if (wt < N) {
          float M = -INFINITY;
          float ms[DS_CTAS], ss[DS_CTAS];
#pragma unroll
          for (int c2 = 0; c2 < DS_CTAS; ++c2) {
            ms[c2] = __ldcg(p.x_stat + ((xr0 + wt) * DS_CTAS + c2) * 2);
            ss[c2] = __ldcg(p.x_stat + ((xr0 + wt) * DS_CTAS + c2) * 2 + 1);
            M = fmaxf(M, ms[c2]);
          }
          float S = 0.f;
#pragma unroll
          for (int c2 = 0; c2 < DS_CTAS; ++c2)
            if (ms[c2] > -INFINITY) S += ss[c2] * __expf(ms[c2] - M);
          s_lse[wt] = M + logf(S);
        }
        ds_worker_sync();
        for (int e = wt; e < N * n8; e += DS_W) {
          const int n = e / n8, k = e % n8;
          const float v = m_v[e];
          const int id = m_i[e];
          int rank = 0;
          for (int k2 = 0; k2 < n8; ++k2) {
            const float v2 = m_v[n * n8 + k2];
            const int i2 = m_i[n * n8 + k2];
            rank += (v2 > v || (v2 == v && (i2 < id || (i2 == id && k2 < k)))) ? 1 : 0;
          }
          if (rank < N) {
            // candidate score of pipeline.py:117-123 in the log domain: beam log-prob + log_softmax(logit)
            const float score = __ldcg(p.st.score[cur] + rows0 + n);
            r_c[n * N + rank] = (id != NONE_IDX) ? score + (v - s_lse[n]) : -INFINITY;
            r_i[n * N + rank] = (id != NONE_IDX) ? n * p.V + id : NONE_IDX;        // flat index over the N x V candidates
          }
        }
        ds_worker_sync();
        for (int e = wt; e < N * N; e += DS_W) {
          const float c = r_c[e];
          const int f = r_i[e];
          if (f == NONE_IDX) continue;
          int rank = 0;
          for (int e2 = 0; e2 < N * N; ++e2) rank += ds_better(r_c[e2], r_i[e2], c, f) ? 1 : 0;
          if (rank < N) {                                            // new beam `rank` (pipeline.py:127-131, 140-141)
            const int par = f / p.V, tok = f - par * p.V;
            s_parent[rank] = par;
            s_token[rank] = tok;
            p.st.score[nxt][rows0 + rank] = c;
            p.st.last_tok[rows0 + rank] = tok;
            if (p.st.parent_out) p.st.parent_out[(size_t)t * p.st.B * N + rows0 + rank] = par;
            if (p.st.token_out) p.st.token_out[(size_t)t * p.st.B * N + rows0 + rank] = tok;
            if (rank == 0 && p.st.step_logprob) p.st.step_logprob[(size_t)t * p.st.B + rows0 / N] = c;
          }
        }
        ds_worker_sync();
        if (wt < N) {   // representative of new beam wt: first new beam with the same (parent's representative, token)
          const int* rc = p.rep + (size_t)cur * p.R + rows0;
          const int mine = (t == 0) ? rows0 : __ldcg(rc + s_parent[wt]);
          int first = wt;
          for (int j = 0; j < wt; ++j) {
            const int other = (t == 0) ? rows0 : __ldcg(rc + s_parent[j]);
            if (other == mine && s_token[j] == s_token[wt]) {
              first = j;
              break;
            }
          }
          p.rep[(size_t)nxt * p.R + rows0 + wt] = rows0 + first;
        }
        const int T = p.T;
        for (int n = ww; n < N; n += DS_WORKER_WARPS) {              // reorder sequences + ancestry (pipeline.py:134-137)
          const int par = s_parent[n], tok = s_token[n];
          const int* sseq = p.st.seq[cur] + (size_t)(rows0 + par) * (T + 1);
          int* dseq = p.st.seq[nxt] + (size_t)(rows0 + n) * (T + 1);
          for (int j = lane; j <= t; j += 32) dseq[j] = __ldcg(sseq + j);
          const int* sanc = p.st.anc[cur] + (size_t)(rows0 + par) * T;
          int* danc = p.st.anc[nxt] + (size_t)(rows0 + n) * T;
          for (int j = lane; j < t; j += 32) danc[j] = __ldcg(sanc + j);
          if (lane == 0) {
            dseq[t + 1] = tok;
            danc[t] = rows0 + par;
          }
        }
        ds_worker_sync();
        if (ww == 0) {                                               // top beam is rank 0 (pipeline.py:143-148)
          const int b = rows0 / N;
          const int top_tok = s_token[0];
          if (!p.st.done[b] && (top_tok == p.st.end_id || t == T - 1)) {
            const int* res = p.st.seq[nxt] + (size_t)rows0 * (T + 1);
            const int len = (top_tok == p.st.end_id) ? t : t + 1;    // strip <start> and a trailing <end>
            for (int j = lane; j < len; j += 32) p.st.out_ids[(size_t)b * T + j] = res[1 + j];
            __syncwarp();
            if (lane == 0) {
              p.st.out_len[b] = len;
              p.st.done[b] = 1;
              atomicAdd(p.st.n_done, 1);
            }
          }
        }
      }
      DSTAMP();   // image merge + bookkeeping done
      xsync();                                                      // T2: next tokens / ancestry / scores of the cluster
      DSTAMP();   // barrier T2 (step end)
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

int dstep_set_attributes() {
  FPNMT_CUDA_OK(cudaFuncSetAttribute(dstep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DS_SMEM));
  return 0;
}

int dstep_max_groups(int num_sms) { return num_sms / DS_CTAS; }   // 1 CTA per SM (220 KB of shared memory)

// The 8 CTAs of a group wait on each other, so every CTA of a launch must be resident: cooperative launches of at most
// floor(SMs / 8) groups; more groups run as consecutive launches (groups never interact).
int dstep_launch(const DstepParams& p0, cudaStream_t stream) {
  if (p0.N < 1 || p0.N > DS_NMAX || p0.ntv < 1 || p0.ntv > DS_MAX_VTILES || p0.n_mem < 1 || p0.n_mem > 16 || p0.nsteps < 1 ||
      p0.t0 < 0 || p0.t0 + p0.nsteps > p0.T || !p0.gbar) {
    set_last_error("dstep_launch: configuration outside the fused decoder's limits");
    return 1;
  }
  int dev = 0, sms = 0;
  FPNMT_CUDA_OK(cudaGetDevice(&dev));
  FPNMT_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int per_launch = dstep_max_groups(sms);
  CUtensorMap tmW;   // the whole weight stream as [rows][64] bf16, box 128 rows x 64, SWIZZLE_128B
  {
    const int rc = encode_tmap_2d(&tmW, reinterpret_cast<const bf16*>(p0.wstream), 64, p0.stream_bytes >> 7, 64, 128);
    if (rc) return rc;
  }
  DstepParams p = p0;
  p.ngroups = (p.B + p.ipc - 1) / p.ipc;
  FPNMT_CUDA_OK(cudaMemsetAsync(p.gbar, 0, (size_t)p.ngroups * sizeof(int), stream));
  for (int g0 = 0; g0 < p.ngroups; g0 += per_launch) {
    p.group0 = g0;
    const int ng = p.ngroups - g0 < per_launch ? p.ngroups - g0 : per_launch;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(ng * DS_CTAS);
    cfg.blockDim = dim3(DS_THREADS);
    cfg.dynamicSmemBytes = DS_SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FPNMT_CUDA_OK(cudaLaunchKernelEx(&cfg, dstep_kernel, tmW, p));
  }
  return 0;
}

}  // namespace fpnmt
