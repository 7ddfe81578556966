// Decode tail of one beam-search step (reference: /root/reference/utils/pipeline.py:115-148), ONE kernel per step:
//   k_beam_step   phase 1: per (image, beam) row of fp32 logits: max, sum-exp, candidate score (prob mode:
//                 softmax * beam_prob; log mode: log_softmax + beam_logprob), row-local top-N with tf.math.top_k tie
//                 order (lower index first); 128-bit streaming loads, values kept in registers, warp-shuffle rounds.
//                 phase 2 (last block of each image): merge N x N candidates (ties -> lower flat index n*V+v), emit
//                 parent/token/score, reorder token sequences and the KV-cache ancestry table by parent, handle <end>
//                 on the top beam, write the next step's embedding+position rows, advance the device step counter.
//                 NBEST = true (fpnmt_beam_search, fpnmt_beam_search_diverse) ranks the N x N candidates in G groups of
//                 N / G beams with a diversity penalty (G = 1: one ranking, as above) and differs where an image closes:
//                 when all N beams are frozen, and then with every beam's caption, length and score.
//   k_kv_reorder            : physical KV-cache reorder by parent, all layers in one launch (the bandwidth-bound
//                             alternative to the ancestry table; fpnmt_config.cache_mode = FPNMT_CACHE_PHYSICAL).
#include "kernels.cuh"

namespace fpnmt {

#define LAUNCH_CHECK() FPNMT_CUDA_OK(cudaGetLastError())


__global__ void k_beam_init(BeamState st, int true_beam, int beam_groups) {
  pdl_launch();
  pdl_wait();
  const int rows = st.B * st.N;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    *st.step = 0;
    *st.n_done = 0;
    st.n_done[1] = 0;   // block-completion counter used by k_beam_merge
  }
  if (i < st.B) {
    st.done[i] = 0;
    st.out_len[i] = 0;
    st.img_count[i] = 0;
  }
  if (i < rows) {
    const int n = i % st.N;
    float s0 = st.prob_mode ? 1.f : 0.f;
    if (true_beam && n % (st.N / beam_groups) != 0) s0 = st.prob_mode ? 0.f : -INFINITY;   // first beam of each group alive
    st.score[0][i] = s0;
    if (st.finished_mode) st.fin_len[0][i] = 0;
    st.seq[0][(size_t)i * (st.T + 1)] = st.start_id;
    st.last_tok[i] = st.start_id;
    if (st.rep[0]) st.rep[0][i] = i - n;                   // every beam starts from <start>: one history per image
    if (st.pf.tgt) st.pf.tgt[i] = st.pf.len[i / st.N] > 0 ? st.pf.ids[(size_t)(i / st.N) * st.T] : -1;   // step 0's targets
  }
  for (size_t j = i; j < (size_t)st.B * st.T; j += (size_t)gridDim.x * blockDim.x) st.out_ids[j] = 0;
}
int launch_beam_init(const BeamState& st, int true_beam, cudaStream_t s, int beam_groups) {
  if (beam_groups < 1 || st.N % beam_groups) {
    set_last_error("beam_init: beam_groups must divide the beam width");
    return 1;
  }
  const int rows = st.B * st.N;
  FPNMT_CUDA_OK(launch_k(k_beam_init, dim3((rows + 255) / 256), dim3(256), 0, s, st, true_beam, beam_groups));
  return 0;
}

// (value, index) arg-max with tf.math.top_k ordering: larger value first, equal values -> lower index
__device__ __forceinline__ bool better(float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); }

__device__ __forceinline__ void warp_argmax(float& v, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (better(ov, oi, v, i)) {
      v = ov;
      i = oi;
    }
  }
}

// One launch per decode step.  grid = B*N blocks, one per (image, beam) row of logits:
//   phase 1 (every block)  online softmax statistics of the row (one pass, one block reduction), candidate scores in
//                          registers, per-WARP top-N by shuffle arg-max rounds in which only the owning lane rescans its
//                          registers, then warp 0 merges the NW*N survivors -> cand_val/cand_idx[row][N] (sorted).
//   phase 2 (last block of each image, elected by an atomic counter)  merge the N x N candidates (ties -> lower flat
//                          index n*V+v), emit parent/token/score, reorder token sequences and the KV ancestry table,
//                          handle <end>, write the NEXT step's decoder input rows (embedding + position), and let the
//                          last image advance the device step counter.
//   PREFIX (prompted N-best decode, BeamState::pf): at a step inside the image's prefix every row's one candidate is the prefix
//                          token, scored with the expression of the free branch, and phase 2 keeps every beam on its own row.
//   MASK (constrained decode, `ban`; only with NBEST and PREFIX): a live unforced row ranks allowed tokens only (its lse stays
//                          over all V), and phase 2 writes every new beam's ban set of step t + 1.  `ban` is the last parameter,
//                          so the other instantiations keep their parameter offsets and code.
template <int THREADS, bool NBEST = false, bool PREFIX = false, bool MASK = false>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 4 : 2) k_beam_step(BeamState st, const float* __restrict__ logits, int ld, BeamEmbed em,
                                                                                BanMask ban) {
  constexpr int NW = THREADS / 32;
  extern __shared__ float4 s_row4[];                       // the row's logits (later: candidate scores), nv4*THREADS float4
  __shared__ float s_m[NW], s_s[NW];
  __shared__ float s_cv[NW * 32];
  __shared__ int s_ci[NW * 32];
  __shared__ int s_parent[32], s_token[32], s_rep[32];
  __shared__ int s_last;
  const int row = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef FPNMT_DBG_STAMPS   // build.py --dbg-stamps (see igemm.cu): timeline of image 0 (its last block: phase 2)
  long long* dbg = (st.dbg && row < st.N) ? st.dbg + 16 : nullptr;
#define BDBG(k) do { if (dbg && tid == 0) { long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); dbg[k] = t_; } } while (0)
#else
#define BDBG(k) do { } while (0)
#endif
  if (row == 0) BDBG(0);
  pdl_launch();
  pdl_wait();
  if (row == 0) BDBG(1);
  const int V = st.V, N = st.N, T = st.T;
  const int t = *st.step;
  const float score = st.score[t & 1][row];
  const float* x = logits + (size_t)row * ld;
  // finished-beam extension: a frozen beam's only candidate is itself (token <end>, score unchanged)
  const bool row_frozen = st.finished_mode && st.fin_len[t & 1][row] > 0;
  int ftok = -1;                                           // forced token of the image at this step (prompted decode), or -1
  if constexpr (PREFIX) {
    if (t < st.pf.len[row / N]) ftok = st.pf.ids[(size_t)(row / N) * T + t];
  }
  if (row_frozen) {
    if (tid < N) {
      st.cand_val[(size_t)row * N + tid] = tid == 0 ? score : -INFINITY;
      st.cand_idx[(size_t)row * N + tid] = tid == 0 ? st.end_id : 0x7fffffff;
    }
  } else if (st.vs_stat) {
    // ---- phase 1 without logits: merge the per-tile softmax partials and candidates left by the vocabulary projection
    const int nt = st.vs_tiles, nc = nt * 8;
    float* s_lv2 = reinterpret_cast<float*>(s_row4);        // [nc] candidate scores that reach the threshold
    int* s_li2 = reinterpret_cast<int*>(s_lv2 + nc);        // [nc] their token ids
    __shared__ float s_tau;
    __shared__ int s_cnt2;
    const float2* stt = st.vs_stat + (size_t)row * nt;
    const float* cvv = st.vs_val + (size_t)row * nc;
    const int* cii = st.vs_idx + (size_t)row * nc;
    float tm = -INFINITY, ts = 0.f;                          // this thread's tiles: (max, sum relative to it)
    for (int i = tid; i < nt; i += THREADS) {
      const float2 q = __ldcg(stt + i);
      if (q.x > -INFINITY) {
        const float mn = fmaxf(tm, q.x);
        ts = ts * __expf(tm - mn) + q.y * __expf(q.x - mn);
        tm = mn;
      }
    }
    {
      const float wm = warp_max(tm);
      const float wsum = warp_sum(tm > -INFINITY ? ts * __expf(tm - wm) : 0.f);
      if (lane == 0) {
        s_m[warp] = wm;
        s_s[warp] = wsum;
      }
    }
    // tile maxima: the N-th largest of them bounds the N-th best logit of the row from below.  MASK: each tile's best ALLOWED
    // logit (its first candidate; the projection skipped the banned ones) - a banned tile maximum would lift tau above every
    // allowed candidate.  N distinct tiles still reach tau, and a tile holds at most N - 1 <= 7 better allowed logits.
    if constexpr (MASK) {
      for (int i = tid; i < nt; i += THREADS) s_cv[i] = __ldcg(cvv + (size_t)i * 8);
    } else {
      for (int i = tid; i < nt; i += THREADS) s_cv[i] = __ldcg(stt + i).x;
    }
    if (tid == 0) {
      s_cnt2 = 0;
      s_tau = -INFINITY;
    }
    __syncthreads();
    float m = s_m[0];
#pragma unroll
    for (int w = 1; w < NW; ++w) m = fmaxf(m, s_m[w]);
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) sum += s_m[w] > -INFINITY ? s_s[w] * __expf(s_m[w] - m) : 0.f;
    const float lse = m + logf(sum);
    if (PREFIX && ftok >= 0) {                               // forced step: the prefix token is the row's one candidate
      if (tid < N) {
        st.cand_val[(size_t)row * N + tid] = tid == 0 ? score + (__ldcg(st.pf.tgt_logit + row) - lse) : -INFINITY;
        st.cand_idx[(size_t)row * N + tid] = tid == 0 ? ftok : 0x7fffffff;
      }
    } else {
    for (int i = tid; i < nt; i += THREADS) {
      const float g = s_cv[i];
      int rank = 0;
      for (int j = 0; j < nt; ++j) {
        const float gj = s_cv[j];
        rank += (gj > g || (gj == g && j < i)) ? 1 : 0;
      }
      if (rank == N - 1) s_tau = g;                          // ranks are a permutation: exactly one writer (none if nt < N)
    }
    __syncthreads();
    const float tau_raw = s_tau;
    for (int c = tid; c < nc; c += THREADS) {
      const int e = __ldcg(cii + c);
      const float v = __ldcg(cvv + c);
      if (e != 0x7fffffff && v >= tau_raw) {
        const int pos = atomicAdd(&s_cnt2, 1);
        s_lv2[pos] = score + (v - lse);                      // log score mode (the launcher rejects prob mode here)
        s_li2[pos] = e;
      }
    }
    __syncthreads();
    const int cnt = s_cnt2;
    for (int c = tid; c < cnt; c += THREADS) {
      const float v = s_lv2[c];
      const int e = s_li2[c];
      int rank = 0;
      for (int j = 0; j < cnt; ++j) rank += better(s_lv2[j], s_li2[j], v, e) ? 1 : 0;
      if (rank < N) {
        st.cand_val[(size_t)row * N + rank] = v;
        st.cand_idx[(size_t)row * N + rank] = e;
      }
    }
    if (cnt < N && tid >= cnt && tid < N) {                  // fewer than N valid tokens (tiny vocabularies): pad
      st.cand_val[(size_t)row * N + tid] = -INFINITY;
      st.cand_idx[(size_t)row * N + tid] = 0x7fffffff;
    }
    }   // !forced
  } else {
  const int nv4 = (V + 4 * THREADS - 1) / (4 * THREADS);  // float4 slots per thread; slot i of thread tid = elements
  float* s_row = reinterpret_cast<float*>(s_row4);        //   (i*THREADS + tid)*4 .. +3 (conflict-free, coalesced)

  // ---- stage the row in shared memory with 16-byte cp.async: every load of the row is in flight at once and no
  // registers are tied up (every row block of the step is resident at the same time); then one pass for the maxima
  {
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(s_row4);
#pragma unroll 4
    for (int i = 0; i < nv4; ++i) {
      const int e = (i * THREADS + tid) * 4;
      if (e + 3 < V) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s0 + (uint32_t)(i * THREADS + tid) * 16u), "l"(x + e) : "memory");
      } else {
        float4 q;
        q.x = (e < V) ? x[e] : -INFINITY;
        q.y = (e + 1 < V) ? x[e + 1] : -INFINITY;
        q.z = (e + 2 < V) ? x[e + 2] : -INFINITY;
        q.w = (e + 3 < V) ? x[e + 3] : -INFINITY;
        s_row4[i * THREADS + tid] = q;
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  if (row == 0) BDBG(2);
  float m = -INFINITY;
#pragma unroll 4
  for (int i = 0; i < nv4; ++i) {
    const float4 q = s_row4[i * THREADS + tid];               // own slots only: no barrier needed
    m = fmaxf(m, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
  }
  const float tmax_v = m;                                  // this thread's largest logit
  // ---- row max and sum of exponentials, ONE block barrier: every thread sums its own slots relative to its own
  // maximum (it only re-reads what it wrote itself), warps and then the block combine (max, rescaled sum) pairs.
  float sum = 0.f;
  if (tmax_v > -INFINITY) {
#pragma unroll 4
    for (int i = 0; i < nv4; ++i) {
      const float4 q = s_row4[i * THREADS + tid];
      // __expf (2^x on the SFU, ~2 ulp): the sum only enters lse, where 1e-7 relative is far below the parity tolerance;
      // the candidate scores themselves (cand(), prob mode) keep the accurate expf
      sum += __expf(q.x - tmax_v) + __expf(q.y - tmax_v) + __expf(q.z - tmax_v) + __expf(q.w - tmax_v);   // exp(-inf) = 0: padding
    }
  }
  {
    const float wm = warp_max(tmax_v);
    sum = warp_sum(tmax_v > -INFINITY ? sum * __expf(tmax_v - wm) : 0.f);
    if (lane == 0) {
      s_m[warp] = wm;
      s_s[warp] = sum;
    }
    float tsel = tmax_v;
    if constexpr (MASK) {
      // banned tokens -> -inf in the staged row (own slots: no barrier), after the unmasked statistics above; the thread
      // maxima behind tau, the pre-filter, the gather and the exact fallback below then see allowed tokens only.  A forced
      // row keeps its row: it reads its prefix token's logit.
      if (!(PREFIX && ftok >= 0)) {
        const uint32_t* mk = ban_row(ban, t, row);
        tsel = -INFINITY;
        for (int i = 0; i < nv4; ++i) {
          const int e = (i * THREADS + tid) * 4;
          float4 q = s_row4[i * THREADS + tid];
          const uint32_t bits = e < V ? (__ldcg(mk + (e >> 5)) >> (e & 31)) & 15u : 0u;
          if (bits) {
            if (bits & 1u) q.x = -INFINITY;
            if (bits & 2u) q.y = -INFINITY;
            if (bits & 4u) q.z = -INFINITY;
            if (bits & 8u) q.w = -INFINITY;
            s_row4[i * THREADS + tid] = q;
          }
          tsel = fmaxf(tsel, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
        }
      }
    }
    s_cv[warp * 32 + lane] = tsel;                          // thread maxima, for the selection threshold below
  }
  constexpr int CAP = 128;
  __shared__ float s_lv[CAP];
  __shared__ int s_li[CAP];
  __shared__ int s_cnt;
  if (tid == 0) s_cnt = 0;
  __syncthreads();
  if (row == 0) BDBG(3);
  m = s_m[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) m = fmaxf(m, s_m[w]);
  sum = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) sum += s_s[w] * __expf(s_m[w] - m);
  // ---- candidate score of a logit (pipeline.py:117,122 in prob mode; the same ordering in the log domain otherwise).
  // Every step of it is monotone non-decreasing in floating point, so max_e cand(v_e) == cand(max_e v_e) exactly.
  const float lse = m + logf(sum);
  const bool prob = st.prob_mode != 0;
  auto cand = [&](float vv) -> float { return prob ? (expf(vv - m) / sum) * score : score + (vv - lse); };
  if (PREFIX && ftok >= 0) {                                 // forced step: the prefix token is the row's one candidate
    if (tid < N) {
      st.cand_val[(size_t)row * N + tid] = tid == 0 ? cand(s_row[ftok]) : -INFINITY;
      st.cand_idx[(size_t)row * N + tid] = tid == 0 ? ftok : 0x7fffffff;
    }
  } else {

  // ---- row-local top-N (tf.math.top_k order: value descending, lower index first).
  // Fast path: the 32 "lane groups" (threads with the same lane id, one per warp) hold 32 disjoint parts of the row; the
  // N-th largest of their maxima, tau, is a lower bound of the N-th largest candidate (N distinct elements reach it), so
  // every winner satisfies c >= tau.  Those few elements (typically N..2N of V) are gathered into a shared list and
  // ranked by counting (rank = number of better entries; no serial arg-max rounds).  If more than CAP elements reach tau
  // (massive ties, e.g. the reference's probability underflow regime where every candidate is 0), the exact but slower
  // rescan path below takes over.  Every warp derives tau redundantly from the shared maxima: no extra barrier.
  float tau, tau_raw;
  {
    float g = s_cv[lane];
#pragma unroll
    for (int w = 1; w < NW; ++w) g = fmaxf(g, s_cv[w * 32 + lane]);
    int rank = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float gj = __shfl_sync(0xffffffffu, g, j);
      rank += (gj > g || (gj == g && j < lane)) ? 1 : 0;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, rank == N - 1);      // ranks are a permutation of 0..31
    tau_raw = __shfl_sync(0xffffffffu, g, __ffs(hit) - 1);
    tau = cand(tau_raw);
  }
  // Raw-logit pre-filter: cand() is monotone non-decreasing, so if cand(v_lo) < tau STRICTLY, every element below v_lo has
  // c <= cand(v_lo) < tau and cannot qualify; the exact comparison runs on the survivors.  When the plateau of equal
  // candidate scores reaches the margin (probability underflow, dead beams: all candidates tie) the filter is disabled
  // and the tie handling below sees every element, exactly as before.
  const float v_lo0 = tau_raw - 1e-2f * fmaxf(1.f, fabsf(tau_raw));
  const float v_lo = (cand(v_lo0) < tau) ? v_lo0 : -INFINITY;
  {
#pragma unroll 2
    for (int i = 0; i < nv4; ++i) {
      const float4 q = s_row4[i * THREADS + tid];
      const float v4[4] = {q.x, q.y, q.z, q.w};
      if (!(fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)) >= v_lo)) continue;      // the common case: nothing near the threshold
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int e = (i * THREADS + tid) * 4 + j;
        if (e < V && v4[j] >= v_lo) {
          const float c = cand(v4[j]);
          if (c >= tau) {
            const int pos = atomicAdd(&s_cnt, 1);
            if (pos < CAP) {
              s_lv[pos] = c;
              s_li[pos] = e;
            }
          }
        }
      }
    }
  }
  __syncthreads();
  if (row == 0) BDBG(4);
  const int cnt = s_cnt;
  if (cnt <= CAP && cnt >= N) {
    if (tid < cnt) {
      const float v = s_lv[tid];
      const int e = s_li[tid];
      int rank = 0;
      for (int j = 0; j < cnt; ++j) rank += better(s_lv[j], s_li[j], v, e) ? 1 : 0;
      if (rank < N) {
        st.cand_val[(size_t)row * N + rank] = v;
        st.cand_idx[(size_t)row * N + rank] = e;            // published by the block barrier + thread 0's fence below
      }
    }
  } else {
    // ---- exact fallback: candidate scores written back to shared memory; per-warp top-N by shuffle arg-max rounds
    // in which the owning lane knocks its winner out (-inf) and rescans its slots; then warp 0 merges the survivors.
    for (int i = 0; i < nv4; ++i) {
      float4 q = s_row4[i * THREADS + tid];
      const int e = (i * THREADS + tid) * 4;
      q.x = (e < V) ? cand(q.x) : -INFINITY;
      q.y = (e + 1 < V) ? cand(q.y) : -INFINITY;
      q.z = (e + 2 < V) ? cand(q.z) : -INFINITY;
      q.w = (e + 3 < V) ? cand(q.w) : -INFINITY;
      s_row4[i * THREADS + tid] = q;
    }
    unsigned long long taken_lo = 0ull;                     // knocked-out slots of this thread (up to 64 elements;
    unsigned long long taken_hi = 0ull;                     //  second word for rows longer than 16 float4 per thread)
    float bv;
    int bi;
    auto is_taken = [&](int s) { return s < 64 ? ((taken_lo >> s) & 1ull) != 0 : ((taken_hi >> (s - 64)) & 1ull) != 0; };
    auto rescan = [&]() {
      bv = -INFINITY;
      bi = 0x7fffffff;
      for (int i = 0; i < nv4; ++i) {
        const float4 q = s_row4[i * THREADS + tid];
        const float c4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int e = (i * THREADS + tid) * 4 + j;
          if (e < V && !is_taken(4 * i + j) && better(c4[j], e, bv, bi)) {
            bv = c4[j];
            bi = e;
          }
        }
      }
    };
    rescan();
    for (int k = 0; k < N; ++k) {
      float wv = bv;
      int wi = bi;
      warp_argmax(wv, wi);
      if (lane == 0) {
        s_cv[warp * 32 + k] = wv;
        s_ci[warp * 32 + k] = wi;
      }
      if (wi == bi && bi != 0x7fffffff) {                  // element indices are unique -> exactly one owner
        const int slot = 4 * ((bi >> 2) / THREADS) + (bi & 3);
        if (slot < 64) taken_lo |= 1ull << slot;
        else taken_hi |= 1ull << (slot - 64);
        rescan();
      }
    }
    __syncthreads();
    if (warp == 0) {
      float cv[NW];
      int ci[NW];
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const bool ok = lane < N;
        cv[w] = ok ? s_cv[w * 32 + lane] : -INFINITY;
        ci[w] = ok ? s_ci[w * 32 + lane] : 0x7fffffff;
      }
      for (int k = 0; k < N; ++k) {
        float b2 = -INFINITY;
        int i2 = 0x7fffffff;
#pragma unroll
        for (int w = 0; w < NW; ++w)
          if (ci[w] != 0x7fffffff && better(cv[w], ci[w], b2, i2)) {
            b2 = cv[w];
            i2 = ci[w];
          }
        warp_argmax(b2, i2);
#pragma unroll
        for (int w = 0; w < NW; ++w)
          if (ci[w] == i2) ci[w] = 0x7fffffff;
        if (lane == 0) {
          st.cand_val[(size_t)row * N + k] = b2;
          st.cand_idx[(size_t)row * N + k] = i2;
        }
      }
    }
  }
  }   // !forced
  }   // !row_frozen
  __syncthreads();
  if (row == 0) BDBG(5);
  if (tid == 0) {
    __threadfence();                                        // candidates visible before the image counter moves
    s_last = (atomicAdd(st.img_count + row / N, 1) == N - 1);
  }
  __syncthreads();
  if (row == 0) BDBG(6);
  if (!s_last) return;
  BDBG(7);

  // =================================================================== phase 2: this block closes image b
  __threadfence();
  const int b = row / N;
  const int cur = t & 1, nxt = cur ^ 1;
  const int NN = N * N;
  const int rows0 = b * N;
  // N x N candidates of the image, ranked by counting over the flat index order (pipeline.py:127-131)
  float* s_fv = reinterpret_cast<float*>(s_row4);           // [N*N] values   (the row staging area is free now;
  int* s_ff = reinterpret_cast<int*>(s_fv + 1024);          // [N*N] flat ids  the launcher sizes it >= 8 KB)
  if (tid < 32) {
    s_parent[tid] = 0;
    s_token[tid] = 0;
  }
  if (tid == 0) st.img_count[b] = 0;                        // re-armed for the next step
  float* s_key = s_fv + 2048;                               // [N*N] ranking keys (== values unless the extension is on)
  for (int c = tid; c < NN; c += THREADS) {
    const int tok = __ldcg(st.cand_idx + (size_t)rows0 * N + c);
    const bool ok = tok != 0x7fffffff;
    const float val = ok ? __ldcg(st.cand_val + (size_t)rows0 * N + c) : -INFINITY;
    s_fv[c] = val;
    s_ff[c] = ok ? (c / N) * V + tok : 0x7fffffff;          // flat index over the N x V candidates
    float key = val;
    if (st.finished_mode && ok) {                           // length-normalised score of the candidate
      const int fl = st.fin_len[cur][rows0 + c / N];
      key = val / st.lp[fl > 0 ? fl : t + 1];
    }
    s_key[c] = key;
  }
  __syncthreads();
  BDBG(8);
  if constexpr (NBEST) {
    // Beam groups (fpnmt_beam_search_diverse; G = 1 is the single ranking of the branch below): the new beams of group g are
    // slots [g * M, (g + 1) * M), M = N / G, chosen in group order among the M * N candidates of the group's own rows.  A
    // live candidate's key loses lambda * h, h = the number of new beams of groups 0 .. g-1 that are live emissions of its
    // token; a frozen beam is never penalised and never counted.  Phase 1's top-N per row suffices: at most g * M <= N - M
    // tokens carry a penalty and it only lowers keys, so a row's M best penalised candidates are among its N best raw ones.
    __shared__ int s_live[32];                              // token of each new beam, -1 for a frozen one
    const int G = (int)st.nb.groups[0];
    const float lambda = st.nb.groups[1];
    const int M = N / G, MN = M * N;
    if (PREFIX && ftok >= 0) {
      // forced step: new beam n is row n's one candidate (parent = n, the prefix token); no ranking, no penalty
      if (tid < N) {
        const int n = tid;
        const float v = s_fv[n * N];
        const int fl = st.fin_len[cur][rows0 + n];
        s_parent[n] = n;
        s_token[n] = ftok;
        st.fin_len[nxt][rows0 + n] = fl > 0 ? fl : (ftok == st.end_id ? t + 1 : 0);
        st.score[nxt][rows0 + n] = v;
        st.last_tok[rows0 + n] = ftok;
        if (st.parent_out) st.parent_out[(size_t)t * st.B * N + rows0 + n] = n;
        if (st.token_out) st.token_out[(size_t)t * st.B * N + rows0 + n] = ftok;
        if (n == 0 && st.step_logprob) st.step_logprob[(size_t)t * st.B + b] = v;
      }
    } else
    for (int g = 0; g < G; ++g) {
      const int c0 = g * MN;
      if (g > 0) {
        __syncthreads();                                    // group g - 1's tokens are in s_live
        for (int c = c0 + tid; c < c0 + MN; c += THREADS) {
          const int f = s_ff[c];
          if (f == 0x7fffffff || st.fin_len[cur][rows0 + c / N] > 0) continue;
          const int tok = f - (c / N) * V;
          int h = 0;
          for (int m = 0; m < g * M; ++m) h += s_live[m] == tok ? 1 : 0;
          s_key[c] = __fsub_rn(s_key[c], __fmul_rn(lambda, (float)h));
        }
        __syncthreads();
      }
      for (int c = c0 + tid; c < c0 + MN; c += THREADS) {
        const int f = s_ff[c];
        if (f == 0x7fffffff) continue;
        const float v = s_fv[c], key = s_key[c];
        int rank = 0;
        for (int j = c0; j < c0 + MN; ++j) rank += better(s_key[j], s_ff[j], key, f) ? 1 : 0;
        if (rank < M) {
          const int n = g * M + rank;                       // new beam n (ties -> lower flat index within the group)
          const int par = f / V;
          const int tok = f - par * V;
          const int fl = st.fin_len[cur][rows0 + par];
          s_parent[n] = par;
          s_token[n] = tok;
          s_live[n] = fl > 0 ? -1 : tok;
          st.fin_len[nxt][rows0 + n] = fl > 0 ? fl : (tok == st.end_id ? t + 1 : 0);
          st.score[nxt][rows0 + n] = v;                     // raw: the penalty only ranks, it is never accumulated
          st.last_tok[rows0 + n] = tok;
          if (st.parent_out) st.parent_out[(size_t)t * st.B * N + rows0 + n] = par;
          if (st.token_out) st.token_out[(size_t)t * st.B * N + rows0 + n] = tok;
          if (n == 0 && st.step_logprob) st.step_logprob[(size_t)t * st.B + b] = v;
        }
      }
    }
  } else {
  for (int c = tid; c < NN; c += THREADS) {
    const int f = s_ff[c];
    if (f == 0x7fffffff) continue;
    const float v = s_fv[c], key = s_key[c];
    int rank = 0;
    for (int j = 0; j < NN; ++j) rank += better(s_key[j], s_ff[j], key, f) ? 1 : 0;
    if (rank < N) {                                         // new beam `rank` (scores sorted, ties -> lower flat index)
      const int par = f / V;                                // pipeline.py:130
      const int tok = f - par * V;                          // pipeline.py:131
      s_parent[rank] = par;
      s_token[rank] = tok;
      if (st.finished_mode) {
        const int fl = st.fin_len[cur][rows0 + par];
        st.fin_len[nxt][rows0 + rank] = fl > 0 ? fl : (tok == st.end_id ? t + 1 : 0);
      }
      st.score[nxt][rows0 + rank] = v;
      st.last_tok[rows0 + rank] = tok;
      if (st.parent_out) st.parent_out[(size_t)t * st.B * N + rows0 + rank] = par;
      if (st.token_out) st.token_out[(size_t)t * st.B * N + rows0 + rank] = tok;
      if (rank == 0 && st.step_logprob) st.step_logprob[(size_t)t * st.B + b] = v;
    }
  }
  }
  if constexpr (PREFIX) {                                    // the token whose logit step t + 1's vocabulary projection reports
    if (st.pf.tgt && tid < N)
      st.pf.tgt[rows0 + tid] = t + 1 < st.pf.len[b] ? st.pf.ids[(size_t)b * T + t + 1] : -1;
  }
  __syncthreads();
  BDBG(9);
  // representative of each new beam: the first new beam with the same token history (parents equivalent, same token)
  if (tid < N) {
    int m_sel = tid;
    if (st.rep[0]) {
      const int* rc = st.rep[cur] + rows0;
      const int rn = rc[s_parent[tid]], tk = s_token[tid];
      for (int m = 0; m < tid; ++m)
        if (s_token[m] == tk && rc[s_parent[m]] == rn) {
          m_sel = m;
          break;
        }
      st.rep[nxt][rows0 + tid] = rows0 + m_sel;
    }
    s_rep[tid] = m_sel;
  }
  __syncthreads();
  for (int n = warp; n < N; n += NW) {
    const int par = s_parent[n], tok = s_token[n];
    const int* sseq = st.seq[cur] + (size_t)(rows0 + par) * (T + 1);
    int* dseq = st.seq[nxt] + (size_t)(rows0 + n) * (T + 1);
    for (int j = lane; j <= t; j += 32) dseq[j] = sseq[j];            // pipeline.py:134-137
    if (!st.physical) {                                               // ancestry cache mode: move the indirection, not the cache
      const int apar = s_parent[s_rep[n]];                            // the representative's lineage: identical K/V bits
      const int* sanc = st.anc[cur] + (size_t)(rows0 + apar) * T;
      int* danc = st.anc[nxt] + (size_t)(rows0 + n) * T;
      for (int j = lane; j < t; j += 32) danc[j] = sanc[j];
      if (lane == 0) danc[t] = rows0 + apar;
    }
    if (lane == 0) dseq[t + 1] = tok;
    if constexpr (MASK) {                                             // the new beam's ban set of step t + 1 from its caption
      __syncwarp();
      if (t + 1 < T) ban_row_warp(ban_row(ban, t + 1, rows0 + n), ban, dseq + 1, t + 1);
    }
  }
  BDBG(10);
  // next step's decoder input: x[row] = embedding[token] + pos[t + 1]   (transformer.py:326-329)
  if (em.emb && t + 1 < T) {
    const int groups = em.D / 8;
    for (int i = tid; i < N * groups; i += THREADS) {
      const int n = i / groups, g = i % groups;
      const float* ep = em.emb + (size_t)s_token[n] * em.D + g * 8;
      const float* pp = em.pos + (size_t)(t + 1) * em.D + g * 8;
      const float4 a0 = *reinterpret_cast<const float4*>(ep), a1 = *reinterpret_cast<const float4*>(ep + 4);
      const float4 p0 = *reinterpret_cast<const float4*>(pp), p1 = *reinterpret_cast<const float4*>(pp + 4);
      const float o[8] = {a0.x + p0.x, a0.y + p0.y, a0.z + p0.z, a0.w + p0.w, a1.x + p1.x, a1.y + p1.y, a1.z + p1.z, a1.w + p1.w};
      st_act8(em.x, (size_t)(rows0 + n), g * 8, o);
    }
  }
  __syncthreads();
  BDBG(11);
  // top beam is rank 0 (scores are sorted; tf.argmax returns the first maximum) — pipeline.py:143-148
  if (warp == 0) {
    if constexpr (NBEST) {
      // N-best: the image is finished once all N beams are frozen (later steps only re-rank the frozen beams in the same
      // order) or after T steps; every beam is written, in rank order within its group, stripped of <start> and of the
      // <end> it froze on
      bool all_frozen = true;
      for (int n = 0; n < N; ++n) all_frozen = all_frozen && st.fin_len[nxt][rows0 + n] > 0;
      if (!st.done[b] && (all_frozen || t == T - 1)) {
        // output slot of lane n's beam: its rank within its group by score / lp(min(len + 1, T)), ties to the lower slot.
        // This step's keys carried the diversity penalty, so for G > 1 slot order need not be that order; for G = 1 the
        // keys are exactly the ranking's and this is the identity.
        const int M = N / (int)st.nb.groups[0];
        float okey = -INFINITY;
        if (lane < N) {
          const int fl = st.fin_len[nxt][rows0 + lane];
          okey = __fdiv_rn(st.score[nxt][rows0 + lane], st.lp[fl > 0 ? fl : t + 1]);
        }
        int oslot = (lane / M) * M;
        for (int m = 0; m < N; ++m) {
          const float km = __shfl_sync(0xffffffffu, okey, m);
          if (m / M == lane / M && (km > okey || (km == okey && m < lane))) ++oslot;
        }
        for (int n = 0; n < N; ++n) {
          const int o = rows0 + __shfl_sync(0xffffffffu, oslot, n);
          const int fl = st.fin_len[nxt][rows0 + n];
          const int len = fl > 0 ? fl - 1 : t + 1;
          const int* res = st.seq[nxt] + (size_t)(rows0 + n) * (T + 1);
          int* dst = st.nb.ids + (size_t)o * T;
          for (int j = lane; j < T; j += 32) dst[j] = j < len ? res[1 + j] : 0;
          if (lane == 0) {
            st.nb.len[o] = len;
            st.nb.score[o] = st.score[nxt][rows0 + n];
          }
        }
        __syncwarp();
        if (lane == 0) {
          st.done[b] = 1;
          atomicAdd(st.n_done, 1);
        }
      }
    } else {
    const int top_tok = s_token[0];
    // extension: the image stops when its best beam is a frozen one; its caption ends before the <end> it froze on
    const int top_fin = st.finished_mode ? st.fin_len[nxt][rows0] : 0;
    if (!st.done[b] && (top_tok == st.end_id || t == T - 1)) {
      const int* res = st.seq[nxt] + (size_t)rows0 * (T + 1);
      const int len = top_fin > 0 ? top_fin - 1 : (top_tok == st.end_id) ? t : t + 1;   // strip <start> and a trailing <end>
      for (int j = lane; j < len; j += 32) st.out_ids[(size_t)b * T + j] = res[1 + j];
      __syncwarp();
      if (lane == 0) {
        st.out_len[b] = len;
        st.done[b] = 1;
        atomicAdd(st.n_done, 1);
      }
    }
    }
    // last image to finish advances the step counter
    if (lane == 0) {
      __threadfence();
      const int prev = atomicAdd(st.n_done + 1, 1);
      if (prev == st.B - 1) {
        st.n_done[1] = 0;
        *st.step = t + 1;
      }
    }
  }
  BDBG(12);
}
int beam_set_attributes() {   // per device (Engine::init)
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<512, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<256, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<512, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<256, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FPNMT_CUDA_OK(cudaFuncSetAttribute(k_beam_step<512, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  return 0;
}
int check_beam_step(const BeamState& st, int ld) {
  if (st.N > 32 || (ld & 3)) {
    set_last_error("beam_step: beam width must be <= 32 and logits ld a multiple of 4");
    return 1;
  }
  if (st.vs_stat) {
    if (st.prob_mode || st.N > 8 || st.vs_tiles > 192 || st.vs_tiles < 1) {
      set_last_error("beam_step: the logits-free tail needs log scores, beam <= 8 and <= 192 vocabulary tiles");
      return 1;
    }
  } else {
    const int threads = st.V <= 16384 ? 256 : 512;
    const int nv4 = (st.V + 4 * threads - 1) / (4 * threads);
    if (nv4 > 32 || (size_t)nv4 * threads * 16 > 200 * 1024) {
      set_last_error("beam_step: vocabulary too large (max 65536)");
      return 1;
    }
  }
  return 0;
}
template <bool NBEST, bool PREFIX = false, bool MASK = false>
static int launch_step(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, cudaStream_t s,
                       const BanMask& ban = BanMask{}) {
  if (check_beam_step(st, ld)) return 1;
  if (st.vs_stat) {                                         // logits-free tail: merge the vocabulary projection's candidates
    size_t smem = (size_t)st.vs_tiles * 8 * 8;
    if (smem < 12288) smem = 12288;
    FPNMT_CUDA_OK(launch_k(k_beam_step<256, NBEST, PREFIX, MASK>, dim3(st.B * st.N), dim3(256), smem, s, st, logits, ld, em, ban));
    return 0;
  }
  const int threads = st.V <= 16384 ? 256 : 512;
  const int nv4 = (st.V + 4 * threads - 1) / (4 * threads);
  size_t smem = (size_t)nv4 * threads * 16;
  if (smem < 12288) smem = 12288;                           // phase 2 keeps the N x N merge lists (values, flat ids, keys) there
  if (threads == 256)
    FPNMT_CUDA_OK(launch_k(k_beam_step<256, NBEST, PREFIX, MASK>, dim3(st.B * st.N), dim3(256), smem, s, st, logits, ld, em, ban));
  else
    FPNMT_CUDA_OK(launch_k(k_beam_step<512, NBEST, PREFIX, MASK>, dim3(st.B * st.N), dim3(512), smem, s, st, logits, ld, em, ban));
  return 0;
}
int launch_beam_step(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, cudaStream_t s) {
  return launch_step<false>(st, logits, ld, em, s);
}
int check_beam_groups(const BeamState& st, int beam_groups, float diversity) {
  if (beam_groups < 1 || st.N % beam_groups) {
    set_last_error("beam_search: beam_groups must be >= 1 and divide the beam width");
    return 1;
  }
  if (!(diversity >= 0.f) || diversity == INFINITY) {
    set_last_error("beam_search: diversity must be finite and >= 0");
    return 1;
  }
  return 0;
}
int launch_beam_step_nbest(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, cudaStream_t s) {
  if (!st.finished_mode || st.prob_mode || !st.nb.ids || !st.nb.len || !st.nb.score || !st.nb.groups) {
    set_last_error("beam_step_nbest: needs finished beams, log scores, the N-best outputs and the beam-group words");
    return 1;
  }
  return launch_step<true>(st, logits, ld, em, s);
}
int launch_beam_step_prefix(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, cudaStream_t s) {
  if (!st.pf.ids || !st.pf.len || (st.vs_stat && (!st.pf.tgt || !st.pf.tgt_logit))) {
    set_last_error("beam_step_prefix: needs the prefix buffers (and on the logits-free tail the target ids and logits)");
    return 1;
  }
  if (!st.finished_mode || st.prob_mode || !st.nb.ids || !st.nb.len || !st.nb.score || !st.nb.groups) {
    set_last_error("beam_step_prefix: needs finished beams, log scores, the N-best outputs and the beam-group words");
    return 1;
  }
  return launch_step<true, true>(st, logits, ld, em, s);
}
int launch_beam_step_constrained(const BeamState& st, const float* logits, int ld, const BeamEmbed& em, const BanMask& ban,
                                 cudaStream_t s) {
  if (!ban.mask || !ban.cfg || ban.rows != st.B * st.N || ban.V != st.V || ban.W != (st.V + 31) / 32) {
    set_last_error("beam_step_constrained: needs the ban masks of every row");
    return 1;
  }
  if (!st.pf.ids || !st.pf.len || (st.vs_stat && (!st.pf.tgt || !st.pf.tgt_logit))) {
    set_last_error("beam_step_constrained: needs the prefix buffers (and on the logits-free tail the target ids and logits)");
    return 1;
  }
  if (!st.finished_mode || st.prob_mode || !st.nb.ids || !st.nb.len || !st.nb.score || !st.nb.groups) {
    set_last_error("beam_step_constrained: needs finished beams, log scores, the N-best outputs and the beam-group words");
    return 1;
  }
  return launch_step<true, true, true>(st, logits, ld, em, s, ban);
}

// Step 0's ban sets (hist == nullptr) and fpnmt_op_ban_mask: one warp per row
__global__ void k_ban_rows(BanMask bm, int t, const int* __restrict__ hist, int ld, const int* __restrict__ len) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= bm.rows) return;
  const int n = len ? len[row] : 0;
  ban_row_warp(ban_row(bm, t, row), bm, hist ? hist + (size_t)row * ld : nullptr, hist ? min(max(n, 0), ld) : 0);
}
int launch_ban_rows(const BanMask& bm, int t, const int* hist, int ld, const int* len, cudaStream_t s) {
  k_ban_rows<<<(bm.rows + 3) / 4, 128, 0, s>>>(bm, t, hist, ld, len);
  LAUNCH_CHECK();
  return 0;
}

// Prompted decode: one block per image copies and checks its prefix (see kernels.cuh)
__global__ void k_prefix_load(const int* __restrict__ prefix_ids, const int* __restrict__ prefix_len, int p, int T, int V,
                              int end_id, int* __restrict__ dst_ids, int* __restrict__ dst_len, int* __restrict__ bad) {
  const int b = blockIdx.x;
  const int len = prefix_len[b];
  const bool len_bad = len < 0 || len > p;
  const int n = len_bad ? 0 : len;
  int bad_id = 0;
  for (int j = threadIdx.x; j < T; j += blockDim.x) {
    int v = 0;
    if (j < n) {
      const int id = prefix_ids[(size_t)b * p + j];
      bad_id |= (id < 0 || id >= V || id == end_id) ? 1 : 0;
      v = min(max(id, 0), V - 1);
    }
    dst_ids[(size_t)b * T + j] = v;
  }
  const int any_bad = __syncthreads_or(bad_id) || len_bad;
  if (threadIdx.x == 0) {
    bad[b] = any_bad ? 1 : 0;
    dst_len[b] = any_bad ? 0 : n;
  }
}
int launch_prefix_load(const int* prefix_ids, const int* prefix_len, int p, int B, int T, int V, int end_id, int* dst_ids,
                       int* dst_len, int* bad, cudaStream_t s) {
  if (p < 1 || p > T) {
    set_last_error("prefix_load: prefix width must be 1 .. max_len");
    return 1;
  }
  k_prefix_load<<<B, 128, 0, s>>>(prefix_ids, prefix_len, p, T, V, end_id, dst_ids, dst_len, bad);
  LAUNCH_CHECK();
  return 0;
}

__global__ void k_prefix_flag(const int* __restrict__ bad, int N, int T, int* __restrict__ ids, int* __restrict__ len,
                              float* __restrict__ logprob) {
  const int b = blockIdx.x;
  if (!bad[b]) return;
  for (int j = threadIdx.x; j < N * T; j += blockDim.x) ids[(size_t)b * N * T + j] = 0;
  if (threadIdx.x < N) {
    len[b * N + threadIdx.x] = 0;
    logprob[b * N + threadIdx.x] = __int_as_float(0x7fc00000);
  }
}
int launch_prefix_flag(const int* bad, int B, int N, int T, int* ids, int* len, float* logprob, cudaStream_t s) {
  k_prefix_flag<<<B, 128, 0, s>>>(bad, N, T, ids, len, logprob);
  LAUNCH_CHECK();
  return 0;
}

// Physical KV-cache reorder (see kernels.cuh).  grid (rows, ncaches): one block streams the live span of one cache row -
// (tt + 1) * row_bytes contiguous bytes - from its parent's row of the source buffer to its own row of the other buffer with
// 16-byte loads / stores, 4 in flight per thread.  Bandwidth kernel: 2 x live bytes of HBM traffic, nothing else.
__global__ void __launch_bounds__(256) k_kv_reorder(const bf16* const* __restrict__ bufs, int ncaches, const int* __restrict__ parent,
                                                    int rows_total, int N, int T, int row_bytes, const int* __restrict__ step) {
  pdl_launch();
  pdl_wait();
  const int tt = *step - 1;                        // the decode step that has just been closed by the beam kernel
  if (tt < 0) return;
  const int r = blockIdx.x, c = blockIdx.y;
  const int src_row = (r / N) * N + parent[(size_t)tt * rows_total + r];
  const size_t row_stride = (size_t)T * row_bytes;
  const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(bufs[(tt & 1) * ncaches + c]) + src_row * row_stride);
  uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(const_cast<bf16*>(bufs[((tt + 1) & 1) * ncaches + c])) + r * row_stride);
  const int n = (tt + 1) * (row_bytes / 16);
  int i = threadIdx.x;
  for (; i + 3 * 256 < n; i += 4 * 256) {
    const uint4 a = __ldcs(src + i), b = __ldcs(src + i + 256), d = __ldcs(src + i + 512), e = __ldcs(src + i + 768);
    __stcs(dst + i, a);
    __stcs(dst + i + 256, b);
    __stcs(dst + i + 512, d);
    __stcs(dst + i + 768, e);
  }
  for (; i < n; i += 256) __stcs(dst + i, __ldcs(src + i));
}
int launch_kv_reorder(const bf16* const* bufs, int ncaches, const int* parent, int rows, int rows_total, int N, int T, int row_bytes,
                      const int* step, cudaStream_t s) {
  if (row_bytes % 16) {
    set_last_error("kv_reorder: cache rows must be a multiple of 16 bytes");
    return 1;
  }
  FPNMT_CUDA_OK(launch_k(k_kv_reorder, dim3(rows, ncaches), dim3(256), 0, s, bufs, ncaches, parent, rows_total, N, T, row_bytes, step));
  return 0;
}

}  // namespace fpnmt
