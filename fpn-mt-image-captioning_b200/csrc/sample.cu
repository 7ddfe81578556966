// Sampled caption decoding (temperature, top-k, nucleus), ONE kernel per decode step over fp32 logits [rows][V]:
//   k_sample_step   one CTA per row: row max / arg-max and sum of exponentials at temperature 1 (for the log-probability),
//                   top-k threshold by a radix select on order-preserving uint32 logit keys (integer counts), tempered
//                   probabilities as fixed-point integer masses (2^-40 of the row maximum's probability), top-p threshold by a
//                   radix select over those masses, and the draw by a block scan in vocabulary order.  Every reduction that
//                   decides the token is an integer one, so the token does not depend on the order in which threads add;
//                   the one float reduction (the log-partition function) runs in a fixed tree.  Then the row update: token
//                   fed to the next step, frozen flag / length / log-probability / caption of the sample, the image's
//                   finished-sample counter, and the device step counter (last CTA).
//   k_sample_init   step 0, <start> fed to every row, identity ancestry in both step parities, per-row state cleared.
#include "../../include/fpnmt.h"
#include "kernels.cuh"

namespace fpnmt {

#define LAUNCH_CHECK() FPNMT_CUDA_OK(cudaGetLastError())

constexpr int SAMPLE_THREADS = 256;
constexpr int SAMPLE_MAX_SMEM = 200 * 1024;             // the row of logits (then of tempered probabilities) in shared memory
constexpr float SAMPLE_MASS_SCALE = 1099511627776.f;    // 2^40: fixed-point unit of the probability mass (row maximum = 2^40)

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k.x += 0x9E3779B9u;
      k.y += 0xBB67AE85u;
    }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// order-preserving uint32 key of a float: a < b  <=>  key(a) < key(b)
__device__ __forceinline__ uint32_t fkey(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ unsigned long long mass_of(float e) { return __float2ull_rn(e * SAMPLE_MASS_SCALE); }

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct SampleSmem {
  unsigned long long hist[256];
  unsigned long long wsum[SAMPLE_THREADS / 32];
  float wm[SAMPLE_THREADS / 32], ws[SAMPLE_THREADS / 32];
  int wi[SAMPLE_THREADS / 32];
  uint32_t sel_prefix;
  unsigned long long sel_rem;
  float m, lse1;
  int mi, tok;
  uint32_t u24;
};
// the step's shared state; MASK adds the largest allowed logit (per warp, of the row) and its lowest index (the other kernels
// keep SampleSmem's layout)
template <bool MASK>
struct SampleStepSmem : SampleSmem {};
template <>
struct SampleStepSmem<true> : SampleSmem {
  float wma[SAMPLE_THREADS / 32], ma;
  int wmai[SAMPLE_THREADS / 32];
};

// Block sum of a uint64 (exact: integer addition), result in every thread.
__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v, SampleSmem& sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum_u64(v);
  __syncthreads();                     // sm.wsum may still be read by a previous call
  if (lane == 0) sm.wsum[warp] = v;
  __syncthreads();
  unsigned long long t = 0;
#pragma unroll
  for (int w = 0; w < SAMPLE_THREADS / 32; ++w) t += sm.wsum[w];
  return t;
}

// Largest key tau such that sum_{i : key(i) >= tau} w(i) >= target (1 <= target <= sum of all w), by four 8-bit radix
// passes from the top digit.  Histogram atomics add integers: the result is independent of their order.
template <typename KeyW>
__device__ uint32_t radix_select_desc(const float* s_row, int V, unsigned long long target, KeyW keyw, SampleSmem& sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t prefix = 0, mask = 0;
  unsigned long long rem = target;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    __syncthreads();                   // previous pass' selection has been read
    for (int i = tid; i < 256; i += SAMPLE_THREADS) sm.hist[i] = 0ull;
    __syncthreads();
    for (int i = tid; i < V; i += SAMPLE_THREADS) {
      uint32_t key;
      const unsigned long long w = keyw(s_row[i], &key);
      if (w && (key & mask) == prefix) atomicAdd(&sm.hist[(key >> shift) & 255u], w);
    }
    __syncthreads();
    if (warp == 0) {
      // lane owns bins 8*lane .. 8*lane+7; `above` = mass of the lanes with higher bins
      unsigned long long h[8], tot = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        h[j] = sm.hist[8 * lane + j];
        tot += h[j];
      }
      unsigned long long incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_down_sync(0xffffffffu, incl, o);
        if (lane + o < 32) incl += v;
      }
      const unsigned long long above = incl - tot;
      if (above < rem && rem <= incl) {            // exactly one lane (rem <= mass of the prefix class)
        unsigned long long acc = above;
        int bin = 8 * lane;
#pragma unroll
        for (int j = 7; j >= 0; --j) {
          if (acc + h[j] >= rem) {
            bin = 8 * lane + j;
            break;
          }
          acc += h[j];
        }
        sm.sel_prefix = prefix | ((uint32_t)bin << shift);
        sm.sel_rem = rem - acc;
      }
    }
    __syncthreads();
    prefix = sm.sel_prefix;
    rem = sm.sel_rem;
    mask |= 255u << shift;
  }
  return prefix;
}

// The step body.  PREFIX (k_sample_step_prefix): a row of an image inside its prefix (step t < pfx_len[image]) takes the
// prefix token pfx_ids[image][t] (top-k, top-p and the draw skipped) and adds its log-probability with the expression of the
// free path.  MASK (k_sample_step_constrained): after the log-partition function, the banned logits of the staged row become
// -inf, so the arg-max, top-k, the masses (taken relative to the largest ALLOWED logit: relative to a banned maximum the allowed
// masses could all round to 0) and the draw see allowed tokens only; the log-probability still reads the unmasked logit.  The
// row's CTA then writes its own ban set of step t + 1.
template <bool PREFIX, bool MASK = false>
__device__ __forceinline__ void sample_step_body(const SampleState& st, const float* __restrict__ logits,
                                                 const int* __restrict__ pfx_ids, const int* __restrict__ pfx_len,
                                                 const BanMask& ban) {
  extern __shared__ float4 s_row4[];
  float* s_row = reinterpret_cast<float*>(s_row4);
  __shared__ SampleStepSmem<MASK> sm;
  pdl_launch();
  pdl_wait();
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = SAMPLE_THREADS / 32;
  const int V = st.V;
  const int t = st.step ? *st.step : st.t0;
  const SampleParams prm = *st.params;
  const float* x = logits + (size_t)row * V;

  // ---- stage the row, thread maxima with the lowest index of the maximum
  float m = -INFINITY;
  int mi = 0x7fffffff;
  if ((V & 3) == 0) {
    const float4* x4 = reinterpret_cast<const float4*>(x);
    for (int i = tid; i < V / 4; i += SAMPLE_THREADS) {
      const float4 q = __ldcs(x4 + i);
      s_row4[i] = q;
      const float v4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (v4[j] > m) {              // indices of one thread ascend: strict > keeps the lowest
          m = v4[j];
          mi = 4 * i + j;
        }
    }
  } else {
    for (int i = tid; i < V; i += SAMPLE_THREADS) {
      const float v = __ldcs(x + i);
      s_row[i] = v;
      if (v > m) {
        m = v;
        mi = i;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > m || (om == m && oi < mi)) {
      m = om;
      mi = oi;
    }
  }
  if (lane == 0) {
    sm.wm[warp] = m;
    sm.wi[warp] = mi;
  }
  __syncthreads();
  if (tid == 0) {
    float bm = sm.wm[0];
    int bi = sm.wi[0];
#pragma unroll
    for (int w = 1; w < NW; ++w)
      if (sm.wm[w] > bm || (sm.wm[w] == bm && sm.wi[w] < bi)) {
        bm = sm.wm[w];
        bi = sm.wi[w];
      }
    sm.m = bm;
    sm.mi = bi;
    // uniform of the row: counter (t, image, sample, 0), key = the seed's two words; u = u24 * 2^-24 (exact in fp32 / fp64)
    const int b = row / st.N, n = row - b * st.N;
    sm.u24 = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)n, 0u),
                           make_uint2((uint32_t)(prm.seed & 0xffffffffull), (uint32_t)(prm.seed >> 32))).x >> 8;
  }
  __syncthreads();
  m = sm.m;
  // ---- log-partition function at temperature 1 (fixed reduction tree: bit-identical run to run)
  float s1 = 0.f;
  float ma = -INFINITY;                                  // MASK: this thread's largest allowed logit (lowest index)
  int mai = 0x7fffffff;
  if constexpr (MASK) {
    const uint32_t* mk = ban_row(ban, t, row);
    for (int i = tid; i < V; i += SAMPLE_THREADS) {     // own entries: the same slots the sum reads, no barrier
      const float v = s_row[i];
      s1 += expf(v - m);
      if ((__ldcg(mk + (i >> 5)) >> (i & 31)) & 1u) s_row[i] = -INFINITY;
      else if (v > ma) {
        ma = v;
        mai = i;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, ma, o);
      const int oi = __shfl_xor_sync(0xffffffffu, mai, o);
      if (om > ma || (om == ma && oi < mai)) {
        ma = om;
        mai = oi;
      }
    }
    if (lane == 0) {
      sm.wma[warp] = ma;
      sm.wmai[warp] = mai;
    }
  } else {
    for (int i = tid; i < V; i += SAMPLE_THREADS) s1 += expf(s_row[i] - m);
  }
  s1 = warp_sum(s1);
  if (lane == 0) sm.ws[warp] = s1;
  __syncthreads();
  if (tid == 0) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) a += sm.ws[w];
    sm.lse1 = m + logf(a);
    sm.tok = sm.mi;                                      // temperature 0: arg-max, lowest token id on ties
    if constexpr (MASK) {                                //   over the allowed tokens
      float bm = sm.wma[0];
      int bi = sm.wmai[0];
#pragma unroll
      for (int w = 1; w < NW; ++w)
        if (sm.wma[w] > bm || (sm.wma[w] == bm && sm.wmai[w] < bi)) {
          bm = sm.wma[w];
          bi = sm.wmai[w];
        }
      sm.ma = bm;
      sm.tok = bi;
    }
    if constexpr (PREFIX) {                              // forced step of a prompted decode: the prefix token
      const int b = row / st.N;
      if (t < pfx_len[b]) sm.tok = pfx_ids[(size_t)b * st.T + t];
    }
  }
  bool forced = false;
  if constexpr (PREFIX) forced = t < pfx_len[row / st.N];

  if (prm.temperature > 0.f && !forced) {
    // ---- top-k: K1 = {i : z_i >= z_(k)}, every token tied with the k-th largest logit kept
    uint32_t k1 = 0u;
    if (prm.top_k > 0 && prm.top_k < V)
      k1 = radix_select_desc(s_row, V, (unsigned long long)prm.top_k,
                             [](float z, uint32_t* key) -> unsigned long long { *key = fkey(z); return 1ull; }, sm);
    // ---- tempered probabilities relative to the row maximum, 0 outside K1; fixed-point masses of those
    __syncthreads();
    float mref = m;
    if constexpr (MASK) mref = sm.ma;
    unsigned long long w1 = 0ull;
    for (int i = tid; i < V; i += SAMPLE_THREADS) {
      const float z = s_row[i];
      const float e = fkey(z) >= k1 ? expf((z - mref) / prm.temperature) : 0.f;
      s_row[i] = e;
      w1 += mass_of(e);
    }
    // ---- top-p: K2 = {i in K1 : p_i >= tau}, tau the largest value whose upper set holds top_p of K1's mass
    uint32_t k2 = 0u;                                    // bits of a non-negative float order like the float
    if (prm.top_p < 1.f) {
      const unsigned long long W1 = block_sum_u64(w1, sm);
      unsigned long long target = (unsigned long long)ceil((double)prm.top_p * (double)W1);
      target = target < 1ull ? 1ull : (target > W1 ? W1 : target);
      k2 = radix_select_desc(s_row, V, target,
                             [](float e, uint32_t* key) -> unsigned long long { *key = __float_as_uint(e); return mass_of(e); }, sm);
    }
    __syncthreads();
    // ---- draw: the smallest token i of K2 with sum_{j in K2, j <= i} p_j > u * sum_{K2} p, on the integer masses;
    // thread `tid` owns the contiguous vocabulary chunk [tid * chunk, (tid + 1) * chunk)
    const int chunk = (V + SAMPLE_THREADS - 1) / SAMPLE_THREADS;
    const int c0 = min(V, tid * chunk), c1 = min(V, c0 + chunk);
    unsigned long long loc = 0ull;
    for (int i = c0; i < c1; ++i) {
      const float e = s_row[i];
      if (__float_as_uint(e) >= k2) loc += mass_of(e);
    }
    unsigned long long incl = loc;                       // block inclusive scan in thread (= vocabulary) order
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) sm.wsum[warp] = incl;
    __syncthreads();
    unsigned long long base = 0ull, W2 = 0ull;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      if (w < warp) base += sm.wsum[w];
      W2 += sm.wsum[w];
    }
    incl += base;
    const unsigned long long excl = incl - loc;
    // cum * 2^24 > u24 * W2, compared exactly in 128 bits
    const unsigned long long u24 = sm.u24;
    const unsigned long long thr_lo = u24 * W2, thr_hi = __umul64hi(u24, W2);
    auto above = [&](unsigned long long cum) {
      const unsigned long long hi = cum >> 40, lo = cum << 24;
      return hi > thr_hi || (hi == thr_hi && lo > thr_lo);
    };
    if (loc && !above(excl) && above(incl)) {            // the crossing lies in this chunk: exactly one thread
      unsigned long long cum = excl;
      for (int i = c0; i < c1; ++i) {
        const float e = s_row[i];
        if (__float_as_uint(e) >= k2) cum += mass_of(e);
        if (above(cum)) {
          sm.tok = i;
          break;
        }
      }
    }
  }
  __syncthreads();

  // ---- outputs of the step and the row update
  if (tid == 0) {
    const int tok = sm.tok;
    const int b = row / st.N;
    const float lp = x[tok] - sm.lse1;                   // log_softmax at temperature 1, no filtering
    if (st.tok_out) st.tok_out[row] = tok;
    if (st.lp_out) st.lp_out[row] = lp;
    if (st.u_out) st.u_out[row] = (float)sm.u24 * 5.9604644775390625e-8f;
    if (st.ids) {                                        // engine: one sample of an image
      const int T = st.T;
      if (!st.fin[row]) {
        st.lp[row] += lp;
        const int len = st.len[row];
        const bool end = tok == st.end_id;
        if (!end) {
          st.ids[(size_t)row * T + len] = tok;
          st.len[row] = len + 1;
        }
        if (end || t == T - 1) {
          st.fin[row] = 1;
          if (atomicAdd(st.img_fin + b, 1) == st.N - 1) atomicAdd(st.n_done, 1);
        }
      }
      st.last_tok[row] = tok;                            // a finished row keeps being computed; its tokens are ignored
      __threadfence();
      if (atomicAdd(st.n_done + 1, 1) == st.rows - 1) {  // last row of the step advances the step counter
        st.n_done[1] = 0;
        *st.step = t + 1;
      }
    }
  }
  if constexpr (MASK) {                                  // the row's ban set of step t + 1 from its caption (thread 0 is in warp 0)
    if (warp == 0) {
      __syncwarp();
      if (t + 1 < st.T) ban_row_warp(ban_row(ban, t + 1, row), ban, st.ids + (size_t)row * st.T, __ldcg(st.len + row));
    }
  }
}

__global__ void __launch_bounds__(SAMPLE_THREADS) k_sample_step(SampleState st, const float* __restrict__ logits) {
  sample_step_body<false>(st, logits, nullptr, nullptr, BanMask{});
}
// the step of a prompted decode (pfx_ids [images][T], pfx_len [images]: launch_prefix_load's buffers)
__global__ void __launch_bounds__(SAMPLE_THREADS) k_sample_step_prefix(SampleState st, const float* __restrict__ logits,
                                                                       const int* __restrict__ pfx_ids,
                                                                       const int* __restrict__ pfx_len) {
  sample_step_body<true>(st, logits, pfx_ids, pfx_len, BanMask{});
}
// the step of a constrained decode (prompted or not: pfx_len 0), with the ban sets of `ban`.  The minimum of 5 blocks per SM
// gives ptxas a 48-register budget: with the thread count alone it picks 40 and spills one register across the masses loop.
__global__ void __launch_bounds__(SAMPLE_THREADS, 5) k_sample_step_constrained(SampleState st, const float* __restrict__ logits,
                                                                            const int* __restrict__ pfx_ids,
                                                                            const int* __restrict__ pfx_len, BanMask ban) {
  sample_step_body<true, true>(st, logits, pfx_ids, pfx_len, ban);
}

__global__ void k_sample_init(SampleState st, int* anc) {
  pdl_launch();
  pdl_wait();
  const int rows = st.rows, T = st.T;
  const size_t i0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  if (i0 == 0) {
    *st.step = 0;
    st.n_done[0] = 0;
    st.n_done[1] = 0;
  }
  for (size_t i = i0; i < (size_t)rows; i += stride) {
    st.last_tok[i] = st.start_id;
    st.len[i] = 0;
    st.fin[i] = 0;
    st.lp[i] = 0.f;
    if (i % st.N == 0) st.img_fin[i / st.N] = 0;
  }
  for (size_t j = i0; j < (size_t)rows * T; j += stride) st.ids[j] = 0;
  for (size_t j = i0; j < (size_t)2 * rows * T; j += stride) anc[j] = (int)((j / T) % rows);   // identity, both parities
}

int sample_set_attributes() {   // per device
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_sample_step, cudaFuncAttributeMaxDynamicSharedMemorySize, SAMPLE_MAX_SMEM));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_sample_step_prefix, cudaFuncAttributeMaxDynamicSharedMemorySize, SAMPLE_MAX_SMEM));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_sample_step_constrained, cudaFuncAttributeMaxDynamicSharedMemorySize, SAMPLE_MAX_SMEM));
  return 0;
}

int check_sampling(const fpnmt_sampling& sp, int V) {
  return !(sp.temperature >= 0.f) || !(sp.top_p > 0.f && sp.top_p <= 1.f) || sp.top_k < 0 || sp.top_k > V || sp.reserved[0] ||
         sp.reserved[1] || sp.reserved[2] || sp.reserved[3];
}

int launch_sample_init(const SampleState& st, int* anc, cudaStream_t s) {
  FPNMT_CUDA_OK(launch_k(k_sample_init, dim3(148), dim3(256), 0, s, st, anc));
  return 0;
}

static size_t sample_smem(const SampleState& st) {   // 0: refused
  const size_t smem = ((size_t)st.V * 4 + 15) / 16 * 16;
  if (st.V < 1 || smem > (size_t)SAMPLE_MAX_SMEM || st.rows < 1 || st.N < 1) {
    set_last_error("sample_step: vocabulary must be 1 .. 51200 and rows >= 1");
    return 0;
  }
  return smem;
}
int launch_sample_step(const SampleState& st, const float* logits, cudaStream_t s) {
  const size_t smem = sample_smem(st);
  if (!smem) return 1;
  FPNMT_CUDA_OK(launch_k(k_sample_step, dim3(st.rows), dim3(SAMPLE_THREADS), smem, s, st, logits));
  return 0;
}
int launch_sample_step_prefix(const SampleState& st, const int* pfx_ids, const int* pfx_len, const float* logits, cudaStream_t s) {
  if (!pfx_ids || !pfx_len || !st.ids) {
    set_last_error("sample_step_prefix: needs the prefix buffers and the engine's decode state");
    return 1;
  }
  const size_t smem = sample_smem(st);
  if (!smem) return 1;
  FPNMT_CUDA_OK(launch_k(k_sample_step_prefix, dim3(st.rows), dim3(SAMPLE_THREADS), smem, s, st, logits, pfx_ids, pfx_len));
  return 0;
}

int launch_sample_step_constrained(const SampleState& st, const int* pfx_ids, const int* pfx_len, const float* logits,
                                   const BanMask& ban, cudaStream_t s) {
  if (!pfx_ids || !pfx_len || !st.ids || !ban.mask || !ban.cfg || ban.rows != st.rows || ban.V != st.V ||
      ban.W != (st.V + 31) / 32) {
    set_last_error("sample_step_constrained: needs the prefix buffers, the ban masks of every row and the engine's decode state");
    return 1;
  }
  const size_t smem = sample_smem(st);
  if (!smem) return 1;
  FPNMT_CUDA_OK(launch_k(k_sample_step_constrained, dim3(st.rows), dim3(SAMPLE_THREADS), smem, s, st, logits, pfx_ids, pfx_len,
                         ban));
  return 0;
}

}  // namespace fpnmt
