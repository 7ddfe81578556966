// extern "C" surface of libfpnmt.so (see include/fpnmt.h).
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "engine.cuh"
#include "tgemm.cuh"

namespace fpnmt {
static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
static int g_pdl_mode = 1;   // 0 = off, 1 = every kernel, 2 = tcgen05 GEMM kernels only (fpnmt_config.kernel_opts)
void set_pdl_mode(int mode) { g_pdl_mode = mode; }
bool pdl_enabled() { return g_pdl_mode != 0; }
bool pdl_small_enabled() { return g_pdl_mode == 1; }
}  // namespace fpnmt

using namespace fpnmt;

struct fpnmt_handle {
  Engine* eng;                   // lane 0: every single-batch entry point runs here
  std::vector<Engine*> lanes;    // lanes[0] == eng; fpnmt_submit / fpnmt_collect address the others
  cudaEvent_t last_encode = nullptr;   // encoder-done event of the most recent fpnmt_submit (owned by that lane)
};

extern "C" {

FPNMT_API const char* fpnmt_version(void) {
  return "fpnmt 0.1 (sm_100a; tcgen05 implicit-GEMM igemm_kernel<32|64|128|256> + skinny-row tgemm_kernel<32|64> (cluster LayerNorm epilogue), TMA, TMEM; CUDA-core tail kernels)";
}
FPNMT_API const char* fpnmt_last_error(void) { return g_last_error.c_str(); }

FPNMT_API int fpnmt_create(const fpnmt_config* cfg, int device, fpnmt_handle** out) {
  if (!cfg || !out) {
    set_last_error("fpnmt_create: NULL argument");
    return FPNMT_ERR_INVALID;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_last_error("fpnmt_create: no CUDA device (this library has no CPU fallback)");
    return FPNMT_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) {
    set_last_error("fpnmt_create: bad device index");
    return FPNMT_ERR_INVALID;
  }
  if (cfg->lanes < 0 || cfg->lanes > 16) {
    set_last_error("fpnmt_create: lanes must be 0..16");
    return FPNMT_ERR_INVALID;
  }
  const int L = cfg->lanes < 1 ? 1 : cfg->lanes;
  fpnmt_handle* h = new fpnmt_handle{nullptr, {}};
  for (int l = 0; l < L; ++l) {
    Engine* e = new (std::nothrow) Engine(*cfg, device);
    int rc = e ? e->init() : FPNMT_ERR_INVALID;
    if (rc) {
      delete e;
      for (size_t i = h->lanes.size(); i-- > 0;) delete h->lanes[i];
      delete h;
      return rc;
    }
    if (!h->lanes.empty()) e->share_weights_of(h->lanes[0]);   // one device copy of the GEMM weights for all lanes
    h->lanes.push_back(e);
  }
  h->eng = h->lanes[0];
  *out = h;
  return FPNMT_OK;
}

FPNMT_API int fpnmt_destroy(fpnmt_handle* h) {
  if (!h) return FPNMT_OK;
  for (size_t i = h->lanes.size(); i-- > 0;) delete h->lanes[i];   // the lead lane (owner of the shared weights) last
  delete h;
  return FPNMT_OK;
}

#define CHECK_H(h)                                 \
  if (!(h) || !(h)->eng) {                         \
    set_last_error("NULL handle");                 \
    return FPNMT_ERR_INVALID;                      \
  }

FPNMT_API int fpnmt_set_weight(fpnmt_handle* h, const char* key, const float* data, const int64_t* shape, int ndim) {
  CHECK_H(h);
  for (Engine* e : h->lanes) {
    const int rc = e->set_weight(key, data, shape, ndim);
    if (rc) return rc;
  }
  return FPNMT_OK;
}
FPNMT_API int fpnmt_finalize_weights(fpnmt_handle* h) {
  CHECK_H(h);
  for (Engine* e : h->lanes) {
    const int rc = e->finalize();
    if (rc) return rc;
  }
  return FPNMT_OK;
}
FPNMT_API int fpnmt_lanes(fpnmt_handle* h) { return h ? (int)h->lanes.size() : 0; }
FPNMT_API int fpnmt_submit(fpnmt_handle* h, int lane, const float* images, int on_host, int early_stop, void* stream) {
  CHECK_H(h);
  if (lane < 0 || lane >= (int)h->lanes.size()) {
    set_last_error("fpnmt_submit: lane out of range (fpnmt_config.lanes)");
    return FPNMT_ERR_INVALID;
  }
  const int rc = h->lanes[lane]->submit(images, on_host, early_stop, (cudaStream_t)stream, h->last_encode);
  if (!rc) h->last_encode = h->lanes[lane]->encode_done_event();
  return rc;
}
FPNMT_API int fpnmt_collect(fpnmt_handle* h, int lane, int32_t* out_ids, int32_t* out_len, int outputs_on_host, void* stream) {
  CHECK_H(h);
  if (lane < 0 || lane >= (int)h->lanes.size()) {
    set_last_error("fpnmt_collect: lane out of range (fpnmt_config.lanes)");
    return FPNMT_ERR_INVALID;
  }
  return h->lanes[lane]->collect(out_ids, out_len, outputs_on_host, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_encode(fpnmt_handle* h, const float* images, int on_host, float* memory_out, void* stream) {
  CHECK_H(h);
  return h->eng->encode(images, on_host, memory_out, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_features(fpnmt_handle* h, const float* images, int on_host, float* const out5[5], void* stream) {
  CHECK_H(h);
  return h->eng->features(images, on_host, out5, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_get_tap(fpnmt_handle* h, const char* name, float* out, size_t capacity, size_t* count, void* stream) {
  CHECK_H(h);
  return h->eng->get_tap(name, out, capacity, count, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_decode_logits(fpnmt_handle* h, const float* memory, const int32_t* tokens, int t, float* logits_out,
                        void* stream) {
  CHECK_H(h);
  return h->eng->decode_logits(memory, tokens, t, logits_out, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_decode_hidden(fpnmt_handle* h, const float* memory, const int32_t* tokens, int t, float* hidden_out,
                                  void* stream) {
  CHECK_H(h);
  if (!hidden_out) {
    set_last_error("decode_hidden: hidden_out is NULL");
    return FPNMT_ERR_INVALID;
  }
  return h->eng->decode_logits(memory, tokens, t, nullptr, (cudaStream_t)stream, hidden_out);
}
FPNMT_API int fpnmt_decode_attention(fpnmt_handle* h, const float* memory, const int32_t* tokens, int t, float* self_out,
                                     float* cross_out, void* stream) {
  CHECK_H(h);
  if (!self_out && !cross_out) {
    set_last_error("decode_attention: self_out and cross_out are both NULL");
    return FPNMT_ERR_INVALID;
  }
  return h->eng->decode_logits(memory, tokens, t, nullptr, (cudaStream_t)stream, nullptr, self_out, cross_out);
}
FPNMT_API int fpnmt_beam_step(fpnmt_handle* h, const float* logits, const float* scores_in, int32_t* parent, int32_t* token,
                    float* scores_out, void* stream) {
  CHECK_H(h);
  return h->eng->beam_step(logits, scores_in, parent, token, scores_out, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_beam_step_vstats(fpnmt_handle* h, const float* stat, const float* val, const int32_t* idx, int tiles,
                                     const float* scores_in, int32_t* parent, int32_t* token, float* scores_out, void* stream) {
  CHECK_H(h);
  if (!stat || !val || !idx || !scores_in || !parent || !token || !scores_out || (((uintptr_t)stat | (uintptr_t)val) & 15)) {
    set_last_error("beam_step_vstats: NULL argument or stat / val not 16-byte aligned");
    return FPNMT_ERR_INVALID;
  }
  return h->eng->beam_step(nullptr, scores_in, parent, token, scores_out, (cudaStream_t)stream, (const float2*)stat, val, idx,
                           tiles);
}
FPNMT_API int fpnmt_generate(fpnmt_handle* h, const float* images, int on_host, int32_t* out_ids, int32_t* out_len,
                   int outputs_on_host, int early_stop, float* step_scores, void* stream) {
  CHECK_H(h);
  return h->eng->generate(images, on_host, out_ids, out_len, outputs_on_host, early_stop, step_scores,
                          (cudaStream_t)stream);
}
FPNMT_API int fpnmt_sample(fpnmt_handle* h, const float* images, int images_on_host, const fpnmt_sampling* sampling,
                           int32_t* out_ids, int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop,
                           void* stream) {
  CHECK_H(h);
  if (!sampling) {
    set_last_error("sample: NULL sampling parameters");
    return FPNMT_ERR_INVALID;
  }
  return h->eng->sample(images, images_on_host, *sampling, out_ids, out_len, out_logprob, outputs_on_host, early_stop,
                        (cudaStream_t)stream);
}
FPNMT_API int fpnmt_score(fpnmt_handle* h, const float* images, int images_on_host, const int32_t* ids, const int32_t* lens, int t,
                          float* out_logprob, float* out_token_logprob, int outputs_on_host, void* stream) {
  CHECK_H(h);
  return h->eng->score(images, images_on_host, ids, lens, t, out_logprob, out_token_logprob, outputs_on_host, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_beam_search(fpnmt_handle* h, const float* images, int images_on_host, float length_penalty, int32_t* out_ids,
                                int32_t* out_len, float* out_logprob, int outputs_on_host, int early_stop, void* stream) {
  CHECK_H(h);
  return h->eng->beam_search(images, images_on_host, length_penalty, out_ids, out_len, out_logprob, outputs_on_host, early_stop,
                             (cudaStream_t)stream);
}
FPNMT_API int fpnmt_stage_images(fpnmt_handle* h, const float* host_images, int slot) {
  CHECK_H(h);
  return h->eng->stage_images(host_images, slot);
}
FPNMT_API int fpnmt_generate_staged(fpnmt_handle* h, int slot, int32_t* out_ids, int32_t* out_len, int outputs_on_host,
                                    int early_stop, float* step_scores, void* stream) {
  CHECK_H(h);
  return h->eng->generate_staged(slot, out_ids, out_len, outputs_on_host, early_stop, step_scores, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_decode(fpnmt_handle* h, int32_t* out_ids, int32_t* out_len, int outputs_on_host, int early_stop,
                 float* step_scores, void* stream) {
  CHECK_H(h);
  return h->eng->decode(out_ids, out_len, outputs_on_host, early_stop, step_scores, (cudaStream_t)stream);
}
FPNMT_API int fpnmt_profile(fpnmt_handle* h, int iters, char* buf, size_t cap) {
  CHECK_H(h);
  return h->eng->profile(iters, buf, cap);
}
FPNMT_API int64_t fpnmt_launch_count(fpnmt_handle* h) {
  if (!h || !h->eng) return 0;
  int64_t n = 0;
  for (Engine* e : h->lanes) n += e->launches;
  return n;
}

// ---- stand-alone convolution operator -----------------------------------------------------------------
static inline uint16_t f2bf_host(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0x7fc0;
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline float bf2f_host(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

FPNMT_API int fpnmt_op_conv2d(int device, int precision, const float* x, int N, int H, int W, int Cin, const float* kernel, int kh,
                    int kw, int Cout, int pad_top, int pad_left, const float* bias, int act, const float* residual,
                    int res_mode, float* out, int force_bn, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (Cin % 8) {
    set_last_error("op_conv2d: Cin must be a multiple of 8");
    return FPNMT_ERR_INVALID;
  }
  FPNMT_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  FPNMT_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error("op_conv2d: device is not sm_100");
    return FPNMT_ERR_CUDA;
  }
  int rc = igemm_set_attributes();
  if (rc) return rc;
  const bool split = precision == FPNMT_PREC_BF16X3;
  const int K = kh * kw * Cin;
  const size_t ldw = split ? 2 * (size_t)K : (size_t)K;
  std::vector<uint16_t> hw((size_t)Cout * ldw);
  for (int t = 0; t < kh * kw; ++t)
    for (int ci = 0; ci < Cin; ++ci)
      for (int o = 0; o < Cout; ++o) {
        const float f = kernel[((size_t)t * Cin + ci) * Cout + o];
        const uint16_t hi = f2bf_host(f);
        hw[(size_t)o * ldw + (size_t)t * Cin + ci] = hi;
        if (split) hw[(size_t)o * ldw + K + (size_t)t * Cin + ci] = f2bf_host(f - bf2f_host(hi));
      }
  std::vector<void*> tmp;
  auto dal = [&](size_t b) {
    void* p = nullptr;
    cudaMalloc(&p, b ? b : 16);
    tmp.push_back(p);
    return p;
  };
  auto cleanup = [&]() {
    for (void* p : tmp) cudaFree(p);
  };
  bf16* dw = (bf16*)dal(hw.size() * 2);
  float* dbias = nullptr;
  if (bias) {
    dbias = (float*)dal((size_t)(Cout + 32) * 4);
    cudaMemsetAsync(dbias, 0, (size_t)(Cout + 32) * 4, s);
    cudaMemcpyAsync(dbias, bias, (size_t)Cout * 4, cudaMemcpyHostToDevice, s);
  }
  cudaMemcpyAsync(dw, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice, s);
  auto mk = [&](size_t pix, int C) {
    Act a;
    const int cs = C < 8 ? 8 : (C + 7) / 8 * 8;
    a.C = C;
    a.ld = split ? 2 * cs : cs;
    a.lo = split ? cs : 0;
    a.p = (bf16*)dal(pix * a.ld * 2);
    return a;
  };
  const size_t pix = (size_t)N * H * W;
  Act ax = mk(pix, Cin), ao = mk(pix, Cout), ar{nullptr, 0, 0, 0};
  rc = launch_f32_to_act(x, pix, Cin, ax, s);
  if (!rc && residual) {
    const size_t rpix = res_mode == RES_UP2 ? (size_t)N * (H / 2) * (W / 2) : pix;
    ar = mk(rpix, Cout);
    rc = launch_f32_to_act(residual, rpix, Cout, ar, s);
  }
  IgemmOp op;
  ConvGeom g{N, H, W, Cin, Cout, kh, kw, pad_top, pad_left};
  if (!rc)
    rc = make_igemm_op(&op, g, ax, dw, split, dbias, act, ao, nullptr, 0, residual ? res_mode : RES_NONE, ar,
                       prop.multiProcessorCount, force_bn);
  if (!rc) rc = igemm_launch(op, s);
  if (!rc) rc = launch_act_to_f32(ao, pix, out, s);
  cudaError_t e = cudaStreamSynchronize(s);
  cleanup();
  if (!rc && e != cudaSuccess) {
    set_last_error(std::string("op_conv2d: ") + cudaGetErrorString(e));
    return FPNMT_ERR_CUDA;
  }
  return rc;
}

// ---- input preprocessing operator ------------------------------------------------------------------------
FPNMT_API int fpnmt_op_preprocess(int device, const uint8_t* images_hwc, int N, int H, int W, int S, float* out, void* stream) {
  if (!images_hwc || !out || N < 1 || H < 1 || W < 1 || S < 1) {
    set_last_error("op_preprocess: bad arguments");
    return FPNMT_ERR_INVALID;
  }
  FPNMT_CUDA_OK(cudaSetDevice(device));
  return launch_preprocess(images_hwc, N, H, W, S, out, (cudaStream_t)stream);
}

// ---- stand-alone skinny-row Dense operator (tgemm) -----------------------------------------------------
}  // extern "C"
// Keras Dense kernel (K, F) -> the engine's [F][K] bf16 weight rows ([F][2K], hi | lo, when split)
static std::vector<uint16_t> dense_weights(const float* kernel, int K, int F, bool split) {
  const size_t ldw = split ? 2 * (size_t)K : (size_t)K;
  std::vector<uint16_t> hw((size_t)F * ldw);
  for (int k = 0; k < K; ++k)
    for (int o = 0; o < F; ++o) {
      const float f = kernel[(size_t)k * F + o];
      const uint16_t hi = f2bf_host(f);
      hw[(size_t)o * ldw + k] = hi;
      if (split) hw[(size_t)o * ldw + K + k] = f2bf_host(f - bf2f_host(hi));
    }
  return hw;
}
extern "C" {

FPNMT_API int fpnmt_op_dense(int device, int precision, const float* x, int R, int K, const float* kernel, int F,
                   const float* bias, int act, const float* residual, const float* gamma, const float* beta, float eps,
                   float* out, int force_bn, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (K % 8 || F % 8) {
    set_last_error("op_dense: K and F must be multiples of 8");
    return FPNMT_ERR_INVALID;
  }
  FPNMT_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  FPNMT_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error("op_dense: device is not sm_100");
    return FPNMT_ERR_CUDA;
  }
  int rc = tgemm_set_attributes();
  if (!rc) rc = tgemmw_set_attributes();
  if (rc) return rc;
  const bool split = precision == FPNMT_PREC_BF16X3;
  const bool wide = force_bn >= 128;          // the wide-row two-CTAs-per-SM kernel (tgemmw.cu)
  if (wide && !tgemmw_supports(split, residual != nullptr, gamma != nullptr, F, K)) {
    set_last_error("op_dense: the wide-row kernel needs bf16 precision and a residual only together with LayerNorm");
    return FPNMT_ERR_INVALID;
  }
  const std::vector<uint16_t> hw = dense_weights(kernel, K, F, split);
  std::vector<void*> tmp;
  auto dal = [&](size_t b) {
    void* p = nullptr;
    cudaMalloc(&p, b ? b : 16);
    tmp.push_back(p);
    return p;
  };
  bf16* dw = (bf16*)dal(hw.size() * 2);
  cudaMemcpyAsync(dw, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice, s);
  auto upl = [&](const float* h, int n) {
    float* d = (float*)dal((size_t)(n + 128) * 4);
    cudaMemsetAsync(d, 0, (size_t)(n + 128) * 4, s);
    cudaMemcpyAsync(d, h, (size_t)n * 4, cudaMemcpyHostToDevice, s);
    return d;
  };
  float* dbias = bias ? upl(bias, F) : nullptr;
  float* dg = gamma ? upl(gamma, F) : nullptr;
  float* db = beta ? upl(beta, F) : nullptr;
  auto mk = [&](size_t rows, int C) {
    Act a;
    a.C = C;
    a.ld = split ? 2 * C : C;
    a.lo = split ? C : 0;
    a.p = (bf16*)dal(rows * a.ld * 2);
    return a;
  };
  Act ax = mk(R, K), ao = mk(R, F), ar{nullptr, 0, 0, 0};
  rc = launch_f32_to_act(x, R, K, ax, s);
  if (!rc && residual) {
    ar = mk(R, F);
    rc = launch_f32_to_act(residual, R, F, ar, s);
  }
  TgemmOp op;
  if (!rc && wide)
    rc = make_tgemmw_op(&op, R, ax, dw, F, K, dbias, act, ao, nullptr, 0, residual ? &ar : nullptr, dg, db, eps, prop.multiProcessorCount);
  else if (!rc)
    rc = make_tgemm_op(&op, R, ax, dw, F, K, split, dbias, act, ao, nullptr, 0, residual ? &ar : nullptr, dg, db, eps,
                       prop.multiProcessorCount, force_bn);
  if (!rc) rc = tgemm_launch(op, s);
  if (!rc) rc = launch_act_to_f32(ao, R, out, s);
  cudaError_t e = cudaStreamSynchronize(s);
  for (void* p : tmp) cudaFree(p);
  if (!rc && e != cudaSuccess) {
    set_last_error(std::string("op_dense: ") + cudaGetErrorString(e));
    return FPNMT_ERR_CUDA;
  }
  return rc;
}

}  // extern "C"

// ---- stand-alone encoder bandwidth operators ------------------------------------------------------------
// Each one uploads fp32 tensors into activations of the requested precision, calls the engine's launcher (which picks the
// kernel exactly as the engine's program does) and reads the result back.  A tensor of `ld` channels per pixel is one
// activation of ld channels; the operator sees its first C channels, as through Engine::chan_view.  The output tensor
// is uploaded too, so columns the kernel must not touch come back unchanged.
namespace {
struct OpScratch {
  cudaStream_t s;
  bool split;
  int rc = 0;
  std::vector<void*> tmp;
  OpScratch(cudaStream_t st, int precision) : s(st), split(precision == FPNMT_PREC_BF16X3) {}
  ~OpScratch() {
    cudaStreamSynchronize(s);
    for (void* p : tmp) cudaFree(p);
  }
  void* alloc(size_t b) {
    void* p = nullptr;
    if (cudaMalloc(&p, b ? b : 16) != cudaSuccess) {
      set_last_error("stand-alone operator: cudaMalloc failed");
      rc = FPNMT_ERR_CUDA;
      return nullptr;
    }
    tmp.push_back(p);
    return p;
  }
  // host fp32 [n] -> device, zero-padded so that 16-byte vector loads at the end stay inside the allocation
  const float* upload(const float* h, size_t n) {
    if (!h) return nullptr;
    float* d = (float*)alloc((n + 32) * 4);
    if (!d) return nullptr;
    cudaMemsetAsync(d, 0, (n + 32) * 4, s);
    cudaMemcpyAsync(d, h, n * 4, cudaMemcpyHostToDevice, s);
    return d;
  }
  const int* upload_i(const int* h, size_t n) {
    int* d = (int*)alloc(n * 4);
    if (d) cudaMemcpyAsync(d, h, n * 4, cudaMemcpyHostToDevice, s);
    return d;
  }
  // activation of `ld` channels per row (the engine's layout: hi at [c], lo at [ld + c] in bf16x3), filled from device
  // fp32 [rows][ld] when src != NULL; the returned view covers the first C channels
  Act act(size_t rows, int C, int ld, const float* src) {
    Act a{nullptr, ld, split ? 2 * ld : ld, split ? ld : 0};
    a.p = (bf16*)alloc(rows * a.ld * 2);
    if (a.p && src && !rc) rc = launch_f32_to_act(src, rows, ld, a, s);
    a.C = C;
    return a;
  }
  // device fp32 [rows][ld] <- the whole activation (the columns beyond C included)
  void read_back(Act a, size_t rows, float* out) {
    a.C = a.lo ? a.lo : a.ld;
    if (!rc) rc = launch_act_to_f32(a, rows, out, s);
  }
  int finish(const char* name) {
    const cudaError_t e = cudaStreamSynchronize(s);
    if (!rc && e != cudaSuccess) {
      set_last_error(std::string(name) + ": " + cudaGetErrorString(e));
      return FPNMT_ERR_CUDA;
    }
    return rc;
  }
};

int op_invalid(const char* msg) {
  set_last_error(msg);
  return FPNMT_ERR_INVALID;
}
int op_device(int device, const char* name) {
  FPNMT_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  FPNMT_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error(std::string(name) + ": device is not sm_100");
    return FPNMT_ERR_CUDA;
  }
  return 0;
}
// channels per pixel of a channel-view buffer: 0 means C; must hold C and keep 16-byte rows
bool view_ld(int C, int* ld) {
  if (*ld == 0) *ld = C;
  return C > 0 && C % 8 == 0 && *ld >= C && *ld % 8 == 0;
}
bool bad_precision(int precision) { return precision != FPNMT_PREC_BF16 && precision != FPNMT_PREC_BF16X3; }
bool all_in(const int* v, size_t n, int lo, int hi) {
  for (size_t i = 0; i < n; ++i)
    if (v[i] < lo || v[i] >= hi) return false;
  return true;
}
}  // namespace

extern "C" {

FPNMT_API int fpnmt_op_depthwise3x3(int device, int precision, const float* x, int N, int H, int W, int C, int in_ld,
                                    const float* kernel, const float* bias, int stride, int pad_top, int pad_left, int Ho,
                                    int Wo, int act, float* out, int out_ld, void* stream) {
  if (!x || !kernel || !out || N < 1 || H < 1 || W < 1 || Ho < 1 || Wo < 1 || (stride != 1 && stride != 2) ||
      bad_precision(precision) || !view_ld(C, &in_ld) || !view_ld(C, &out_ld))
    return op_invalid("op_depthwise3x3: bad arguments (C and the lds multiples of 8, stride 1 or 2)");
  int rc = op_device(device, "op_depthwise3x3");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const float* dw = o.upload(kernel, (size_t)9 * C);
  const float* db = o.upload(bias, (size_t)C);
  const size_t ipix = (size_t)N * H * W, opix = (size_t)N * Ho * Wo;
  Act ax = o.act(ipix, C, in_ld, x), ao = o.act(opix, C, out_ld, out);
  if (!o.rc) o.rc = launch_depthwise3x3(ax, N, H, W, stride, pad_top, pad_left, Ho, Wo, dw, db, act, ao, o.s);
  o.read_back(ao, opix, out);
  return o.finish("op_depthwise3x3");
}

FPNMT_API int fpnmt_op_pool(int device, int precision, int kind, const float* x, int N, int H, int W, int C, int in_ld, int k,
                            int stride, int pad_top, int pad_left, int Ho, int Wo, int zero_pad, float* out, int out_ld,
                            void* stream) {
  if (!x || !out || N < 1 || H < 1 || W < 1 || Ho < 1 || Wo < 1 || bad_precision(precision) || !view_ld(C, &in_ld) ||
      !view_ld(C, &out_ld))
    return op_invalid("op_pool: bad arguments (C and the lds multiples of 8)");
  if ((kind == 0 && (k < 1 || stride < 1)) || (kind == 1 && (Ho != H / 2 || Wo != W / 2)) ||
      (kind == 2 && (Ho != (H + 1) / 2 || Wo != (W + 1) / 2)) || kind < 0 || kind > 2)
    return op_invalid("op_pool: kind 0 (max, k >= 1), 1 (avg 2x2, Ho = H/2) or 2 (subsample, Ho = (H+1)/2)");
  int rc = op_device(device, "op_pool");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const size_t ipix = (size_t)N * H * W, opix = (size_t)N * Ho * Wo;
  Act ax = o.act(ipix, C, in_ld, x), ao = o.act(opix, C, out_ld, out);
  if (!o.rc) {
    if (kind == 0) o.rc = launch_maxpool(ax, N, H, W, k, stride, pad_top, pad_left, Ho, Wo, zero_pad != 0, ao, o.s);
    else if (kind == 1) o.rc = launch_avgpool2(ax, N, H, W, ao, o.s);
    else o.rc = launch_subsample2(ax, N, H, W, ao, o.s);
  }
  o.read_back(ao, opix, out);
  return o.finish("op_pool");
}

FPNMT_API int fpnmt_op_scale_shift_relu(int device, int precision, const float* x, int64_t pixels, int C, int in_ld,
                                        const float* scale, const float* shift, float* out, int out_ld, void* stream) {
  if (!x || !scale || !shift || !out || pixels < 1 || bad_precision(precision) || !view_ld(C, &in_ld) || !view_ld(C, &out_ld))
    return op_invalid("op_scale_shift_relu: bad arguments (C and the lds multiples of 8)");
  int rc = op_device(device, "op_scale_shift_relu");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const float *dsc = o.upload(scale, (size_t)C), *dsh = o.upload(shift, (size_t)C);
  Act ax = o.act((size_t)pixels, C, in_ld, x), ao = o.act((size_t)pixels, C, out_ld, out);
  if (!o.rc) o.rc = launch_scale_shift_relu(ax, (size_t)pixels, dsc, dsh, ao, o.s);
  o.read_back(ao, (size_t)pixels, out);
  return o.finish("op_scale_shift_relu");
}

FPNMT_API int fpnmt_op_score_conv(int device, int precision, const float* x, int N, int H, int W, const float* kernel,
                                  const float* bias, float* out, void* stream) {
  if (precision != FPNMT_PREC_BF16)
    return op_invalid("op_score_conv: the one-channel score kernel is a bf16-mode kernel (bf16x3 runs op_conv2d with Cout = 1)");
  if (!x || !kernel || !bias || !out || N < 1 || H < 1 || W < 1 || N > 65535 || (H + 7) / 8 > 65535)
    return op_invalid("op_score_conv: bad arguments");
  int rc = op_device(device, "op_score_conv");
  if (rc) return rc;
  rc = elementwise_set_attributes();
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const float *dw = o.upload(kernel, (size_t)9 * 256), *db = o.upload(bias, 1);
  const size_t pix = (size_t)N * H * W;
  Act ax = o.act(pix, 256, 256, x), ao = o.act(pix, 1, 8, nullptr);
  if (!o.rc) o.rc = launch_f32_to_act(out, pix, 1, ao, o.s);
  if (!o.rc) o.rc = launch_conv3x3_c1(ax, dw, db, N, H, W, ao, o.s);
  if (!o.rc) o.rc = launch_act_to_f32(ao, pix, out, o.s);
  return o.finish("op_score_conv");
}

FPNMT_API int fpnmt_op_coattention(int device, int precision, const float* score, const float* cls, int N, int HW, int C,
                                   float* out, void* stream) {
  if (!score || !cls || !out || N < 1 || N > 65535 || HW < 1 || bad_precision(precision) || C < 8 || C % 8)
    return op_invalid("op_coattention: bad arguments (C a multiple of 8)");
  int rc = op_device(device, "op_coattention");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const size_t pix = (size_t)N * HW;
  Act as = o.act(pix, 1, 8, nullptr), ac = o.act(pix, C, C, cls), ao = o.act(pix, C, C, out);
  if (!o.rc) o.rc = launch_f32_to_act(score, pix, 1, as, o.s);
  if (!o.rc) o.rc = launch_coattention(as, ac, N, HW, ao, o.s);
  o.read_back(ao, pix, out);
  return o.finish("op_coattention");
}

FPNMT_API int fpnmt_op_tokens_ln_pos(int device, int precision, const float* x, int N, int HW, const float* gamma,
                                     const float* beta, float eps, const float* pos, float* out, void* stream) {
  if (!x || !gamma || !beta || !pos || !out || N < 1 || HW < 1 || bad_precision(precision))
    return op_invalid("op_tokens_ln_pos: bad arguments");
  int rc = op_device(device, "op_tokens_ln_pos");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const float *dg = o.upload(gamma, 512), *db = o.upload(beta, 512), *dp = o.upload(pos, (size_t)HW * 512);
  const size_t rows = (size_t)N * HW;
  Act ax = o.act(rows, 512, 512, x), ao = o.act(rows, 512, 512, out);
  if (!o.rc) o.rc = launch_tokens_ln_pos(ax, N, HW, dg, db, eps, dp, ao, o.s);
  o.read_back(ao, rows, out);
  return o.finish("op_tokens_ln_pos");
}

FPNMT_API int fpnmt_op_enc_attention(int device, int precision, const float* q, const float* const* kv, const int* tk,
                                     int nviews, int kv_ld, int k_col, int v_col, int B, int Tq, int heads, int force_simt,
                                     float* out, void* stream) {
  const int width = heads * 64;
  if (!q || !kv || !tk || !out || nviews < 1 || nviews > 4 || B < 1 || B > 65535 || Tq < 1 || heads < 1 || heads > 65535 ||
      bad_precision(precision) || kv_ld % 8 || k_col < 0 || v_col < 0 || k_col % 8 || v_col % 8 || k_col + width > kv_ld ||
      v_col + width > kv_ld)
    return op_invalid("op_enc_attention: bad arguments (1..4 views, K/V columns multiples of 8 inside kv_ld)");
  for (int v = 0; v < nviews; ++v)
    if (!kv[v] || tk[v] < 1) return op_invalid("op_enc_attention: every view needs K/V and tk >= 1");
  int rc = op_device(device, "op_enc_attention");
  if (rc) return rc;
  rc = attention_set_attributes();
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const size_t qrows = (size_t)B * Tq;
  const int qw = nviews * width;
  Act aq = o.act(qrows, qw, qw, q), ao = o.act(qrows, qw, qw, out), akv[4];
  int cols[4];
  for (int v = 0; v < nviews; ++v) {
    akv[v] = o.act((size_t)B * tk[v], kv_ld, kv_ld, kv[v]);
    cols[v] = v * width;
  }
  // kernel choice of Engine::build_mt_encoder: one views launch in bf16 mode, else one launch per view
  if (!o.rc && !o.split && !force_simt && nviews > 1) {
    o.rc = launch_enc_attention_views(aq, akv, tk, cols, nviews, k_col, v_col, B, Tq, heads, ao, o.s);
  } else {
    for (int v = 0; v < nviews && !o.rc; ++v)
      o.rc = launch_enc_attention(aq, cols[v], akv[v], k_col, v_col, B, Tq, tk[v], heads, ao, cols[v], force_simt != 0, o.s);
  }
  o.read_back(ao, qrows, out);
  return o.finish("op_enc_attention");
}


// ---- stand-alone decoder operators ----------------------------------------------------------------------------------
FPNMT_API int fpnmt_op_dec_self_attention(int device, int precision, const float* qkv, float* kc, float* vc, float* kc2,
                                          float* vc2, const int* anc, const int* rep, int rows, int T, int t, int heads, int beam,
                                          int kernel, float* out, void* stream) {
  if (!qkv || !kc || !vc || !anc || !out || (!kc2) != (!vc2) || rows < 1 || T < 1 || t < 0 || t >= T || heads < 1 ||
      beam < 1 || beam > 32 || kernel < 0 || kernel > 2 || bad_precision(precision) ||
      (kernel == DEC_ATT_MMA && precision != FPNMT_PREC_BF16) || (size_t)rows * heads > (1u << 30) || (size_t)rows * T > (1u << 26))
    return op_invalid("op_dec_self_attention: bad arguments (0 <= t < T, beam 1..32, kernel 0..2, mma only in bf16)");
  if (!all_in(anc, (size_t)2 * rows * T, 0, rows) || (rep && !all_in(rep, (size_t)2 * rows, 0, rows)))
    return op_invalid("op_dec_self_attention: anc and rep entries must be rows in [0, rows)");
  int rc = op_device(device, "op_dec_self_attention");
  if (rc) return rc;
  rc = attention_set_attributes();
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const int d = heads * 64;
  const size_t crows = (size_t)rows * T;
  const int* danc = o.upload_i(anc, (size_t)2 * rows * T);
  const int* drep = rep ? o.upload_i(rep, (size_t)2 * rows) : nullptr;
  const int* dstep = o.upload_i(&t, 1);
  const Act none{nullptr, 0, 0, 0};
  Act aq = o.act(rows, 3 * d, 3 * d, qkv), ao = o.act(rows, d, d, out);
  Act ak = o.act(crows, d, d, kc), av = o.act(crows, d, d, vc);
  Act ak2 = kc2 ? o.act(crows, d, d, kc2) : none, av2 = vc2 ? o.act(crows, d, d, vc2) : none;
  if (!o.rc)
    o.rc = launch_dec_self_attention(aq, ak, av, ak2, av2, danc, crows, dstep, rows, T, heads, ao, o.s, drep,
                                     drep ? drep + rows : nullptr, beam, (DecAttKernel)kernel);
  o.read_back(ao, rows, out);
  o.read_back(ak, crows, kc);
  o.read_back(av, crows, vc);
  if (kc2) {
    o.read_back(ak2, crows, kc2);
    o.read_back(av2, crows, vc2);
  }
  return o.finish("op_dec_self_attention");
}

FPNMT_API int fpnmt_op_dec_cross_attention(int device, int precision, const float* q, const float* kv, int kv_ld, int k_col,
                                           int v_col, int rows, int beam, int Tk, int heads, float* out, void* stream) {
  const int d = heads * 64;
  if (!q || !kv || !out || rows < 1 || beam < 1 || rows % beam || Tk < 1 || heads < 1 || (size_t)rows * heads > (1u << 30) ||
      bad_precision(precision) || kv_ld < 8 || kv_ld % 8 || k_col < 0 || v_col < 0 || k_col % 8 || v_col % 8 ||
      k_col + d > kv_ld || v_col + d > kv_ld)
    return op_invalid("op_dec_cross_attention: bad arguments (beam divides rows, K/V columns multiples of 8 inside kv_ld)");
  int rc = op_device(device, "op_dec_cross_attention");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  Act aq = o.act(rows, d, d, q), ao = o.act(rows, d, d, out);
  Act akv = o.act((size_t)(rows / beam) * Tk, kv_ld, kv_ld, kv);
  if (!o.rc) o.rc = launch_dec_cross_attention(aq, akv, k_col, v_col, rows, beam, Tk, heads, ao, o.s);
  o.read_back(ao, rows, out);
  return o.finish("op_dec_cross_attention");
}

FPNMT_API int fpnmt_op_xattn(int device, int precision, const float* ckv, const float* wq, const float* bq, const float* wo,
                             const float* bo, const float* gamma, const float* beta, int Btot, int n_mem, int L, int layer,
                             int b0, int B, int beam, const float* out1, float* out2, float* Mt, float* Nt, float* sbias,
                             void* stream) {
  if (precision != FPNMT_PREC_BF16)
    return op_invalid("op_xattn: the fused cross-attention block is a bf16-mode kernel (bf16x3 runs the unfused path)");
  if (!ckv || !wq || !bq || !wo || !bo || !gamma || !beta || !out1 || !out2 || Btot < 1 || Btot > 65535 || n_mem < 1 ||
      n_mem > 16 || L < 1 || L > 64 || layer < 0 || layer >= L || b0 < 0 || B < 1 || b0 + B > Btot || beam < 1 || beam > 16)
    return op_invalid("op_xattn: bad arguments (n_mem and beam 1..16, 0 <= layer < L, images [b0, b0 + B) inside Btot)");
  int rc = op_device(device, "op_xattn");
  if (rc) return rc;
  rc = xattn_set_attributes();
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const size_t W = (size_t)512 * 512;
  std::vector<uint16_t> hwq((size_t)L * W), hwo((size_t)L * W);
  for (int l = 0; l < L; ++l) xattn_fold_weights(wq + l * W, wo + l * W, &hwq[l * W], &hwo[l * W]);
  bf16* dq = (bf16*)o.alloc(hwq.size() * 2);
  bf16* d_o = (bf16*)o.alloc(hwo.size() * 2);
  const float* dbq = o.upload(bq, (size_t)L * 512);
  std::vector<const float*> hb(L);
  for (int l = 0; l < L; ++l) hb[l] = dbq ? dbq + (size_t)l * 512 : nullptr;
  const float** db = (const float**)o.alloc(L * sizeof(float*));
  const float *dbo = o.upload(bo, 512), *dg = o.upload(gamma, 512), *dbe = o.upload(beta, 512);
  bf16* dMt = (bf16*)o.alloc((size_t)L * Btot * 128 * 512 * 2);
  bf16* dNt = (bf16*)o.alloc((size_t)L * Btot * 512 * 128 * 2);
  float* dsb = (float*)o.alloc((size_t)L * Btot * 128 * 4);
  if (o.rc) return o.finish("op_xattn");
  cudaMemcpyAsync(dq, hwq.data(), hwq.size() * 2, cudaMemcpyHostToDevice, o.s);
  cudaMemcpyAsync(d_o, hwo.data(), hwo.size() * 2, cudaMemcpyHostToDevice, o.s);
  cudaMemcpyAsync(db, hb.data(), L * sizeof(float*), cudaMemcpyHostToDevice, o.s);
  const size_t rows = (size_t)Btot * beam;
  Act ac = o.act((size_t)Btot * n_mem, L * 1024, L * 1024, ckv);
  Act ax = o.act(rows, 512, 512, out1), ay = o.act(rows, 512, 512, out2);
  if (!o.rc) o.rc = launch_xattn_fold(ac, Btot, n_mem, L, dq, db, d_o, dMt, dNt, dsb, o.s);
  Act xv = ax, yv = ay;                   // row views of the slice, as Engine's build_chain makes them
  xv.p += (size_t)b0 * beam * ax.ld;
  yv.p += (size_t)b0 * beam * ay.ld;
  XattnOp op;
  if (!o.rc) o.rc = make_xattn_op(&op, dMt, dNt, L, Btot, b0, B, beam, layer, dsb, dbo, dg, dbe, xv, yv);
  if (!o.rc) o.rc = xattn_launch(op, o.s);
  o.read_back(ay, rows, out2);
  if (Mt) o.read_back(Act{dMt, 512, 512, 0}, (size_t)L * Btot * 128, Mt);
  if (Nt) o.read_back(Act{dNt, 128, 128, 0}, (size_t)L * Btot * 512, Nt);
  if (sbias && !o.rc) cudaMemcpyAsync(sbias, dsb, (size_t)L * Btot * 128 * 4, cudaMemcpyDeviceToDevice, o.s);
  return o.finish("op_xattn");
}

FPNMT_API int fpnmt_op_kv_reorder(int device, int precision, const float* src, float* dst, int ncaches, const int* parent,
                                  int rows, int beam, int T, int D, int t, void* stream) {
  if (!src || !dst || !parent || ncaches < 1 || ncaches > 65535 || rows < 1 || beam < 1 || rows % beam || T < 1 || t < 0 ||
      t > T || D < 8 || D % 8 || bad_precision(precision) || (size_t)rows * T > (1u << 26))
    return op_invalid("op_kv_reorder: bad arguments (beam divides rows, 0 <= t <= T, D a multiple of 8)");
  if (!all_in(parent, (size_t)T * rows, 0, beam)) return op_invalid("op_kv_reorder: parent entries must be beams in [0, beam)");
  int rc = op_device(device, "op_kv_reorder");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const size_t crows = (size_t)rows * T, all = crows * ncaches;
  const int* dpar = o.upload_i(parent, (size_t)T * rows);
  const int* dstep = o.upload_i(&t, 1);
  Act as = o.act(all, D, D, src), ad = o.act(all, D, D, dst);
  // bufs[parity][cache]: the kernel reads parity (t-1)&1 and writes the other, as after decode step t-1 of the engine
  const int tt = t - 1;
  std::vector<const bf16*> hp((size_t)2 * ncaches);
  for (int c = 0; c < ncaches; ++c) {
    hp[(size_t)(tt & 1) * ncaches + c] = as.p + c * crows * as.ld;
    hp[(size_t)((tt + 1) & 1) * ncaches + c] = ad.p + c * crows * ad.ld;
  }
  const bf16** dp = (const bf16**)o.alloc(hp.size() * sizeof(bf16*));
  if (!o.rc) {
    cudaMemcpyAsync(dp, hp.data(), hp.size() * sizeof(bf16*), cudaMemcpyHostToDevice, o.s);
    o.rc = launch_kv_reorder(dp, ncaches, dpar, rows, rows, beam, T, as.ld * 2, dstep, o.s);
  }
  o.read_back(ad, all, dst);
  return o.finish("op_kv_reorder");
}

FPNMT_API int fpnmt_op_embed_pos(int device, int precision, const int* tokens, int rows, const float* emb, int V,
                                 const float* pos, int T, int C, int t, float* out, void* stream) {
  if (!tokens || !emb || !pos || !out || rows < 1 || V < 1 || T < 1 || t < 0 || t >= T || C < 8 || C % 8 ||
      bad_precision(precision) || (size_t)rows * C > (1u << 30))
    return op_invalid("op_embed_pos: bad arguments (C a multiple of 8, 0 <= t < T)");
  if (!all_in(tokens, rows, 0, V)) return op_invalid("op_embed_pos: tokens must be in [0, V)");
  int rc = op_device(device, "op_embed_pos");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const int *dtok = o.upload_i(tokens, rows), *dstep = o.upload_i(&t, 1);
  const float *demb = o.upload(emb, (size_t)V * C), *dpos = o.upload(pos, (size_t)T * C);
  Act ao = o.act(rows, C, C, out);
  if (!o.rc) o.rc = launch_embed_pos(dtok, demb, dpos, dstep, rows, C, ao, o.s);
  o.read_back(ao, rows, out);
  return o.finish("op_embed_pos");
}

FPNMT_API int fpnmt_op_layernorm_rows(int device, int precision, const float* x, int rows, const float* gamma,
                                      const float* beta, float eps, float* out, void* stream) {
  if (!x || !gamma || !beta || !out || rows < 1 || bad_precision(precision))
    return op_invalid("op_layernorm_rows: bad arguments");
  int rc = op_device(device, "op_layernorm_rows");
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, precision);
  const float *dg = o.upload(gamma, 512), *db = o.upload(beta, 512);
  Act ao = o.act(rows, 512, 512, out);
  if (!o.rc) o.rc = launch_layernorm_rows(x, rows, 512, dg, db, eps, ao, o.s);
  o.read_back(ao, rows, out);
  return o.finish("op_layernorm_rows");
}

FPNMT_API int fpnmt_op_vocab_stats(int device, int precision, const float* x, int R, int K, const float* kernel, int F,
                                   const float* bias, float* stat, float* val, int32_t* idx, void* stream) {
  if (precision != FPNMT_PREC_BF16)
    return op_invalid("op_vocab_stats: the logits-free vocabulary projection is a bf16-mode kernel (the wide-row Dense kernel)");
  if (!x || !kernel || !stat || !val || !idx || R < 1 || K < 8 || K % 8 || F < 8 || F % 8 ||
      (((uintptr_t)stat | (uintptr_t)val | (uintptr_t)idx) & 15))
    return op_invalid("op_vocab_stats: bad arguments (K and F multiples of 8, outputs 16-byte aligned)");
  int rc = op_device(device, "op_vocab_stats");
  if (rc) return rc;
  rc = tgemmw_set_attributes();
  if (rc) return rc;
  int sms = 0;
  FPNMT_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  OpScratch o((cudaStream_t)stream, precision);
  const std::vector<uint16_t> hw = dense_weights(kernel, K, F, false);
  bf16* dw = (bf16*)o.alloc(hw.size() * 2);
  const float* db = o.upload(bias, (size_t)F);
  Act ax = o.act(R, K, K, x);
  if (o.rc) return o.finish("op_vocab_stats");
  cudaMemcpyAsync(dw, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice, o.s);
  // the op of the engine's beam-search chain (Engine::build_decoder, logits-free tail), writing the caller's buffers
  const Act none{nullptr, 0, 0, 0};
  TgemmOp op;
  o.rc = make_tgemmw_op(&op, R, ax, dw, F, K, db, ACT_NONE, none, nullptr, 0, nullptr, nullptr, nullptr, 1e-6f, sms,
                        (float2*)stat, val, idx);
  if (!o.rc) o.rc = tgemm_launch(op, o.s);
  return o.finish("op_vocab_stats");
}

FPNMT_API int fpnmt_op_sample_step(int device, const float* logits, int rows, int V, int samples_per_image, int t,
                                   const fpnmt_sampling* sampling, int32_t* token, float* logprob, float* u_out, void* stream) {
  if (!logits || !sampling || !token || rows < 1 || V < 1 || V > 51200 || samples_per_image < 1 || t < 0)
    return op_invalid("op_sample_step: bad arguments (rows >= 1, 1 <= V <= 51200, samples_per_image >= 1, t >= 0)");
  const fpnmt_sampling& sp = *sampling;
  if (!(sp.temperature >= 0.f) || !(sp.top_p > 0.f && sp.top_p <= 1.f) || sp.top_k < 0 || sp.top_k > V || sp.reserved[0] ||
      sp.reserved[1] || sp.reserved[2] || sp.reserved[3])
    return op_invalid("op_sample_step: temperature >= 0, top_p in (0, 1], 0 <= top_k <= V and reserved words 0");
  int rc = op_device(device, "op_sample_step");
  if (rc) return rc;
  rc = sample_set_attributes();
  if (rc) return rc;
  OpScratch o((cudaStream_t)stream, FPNMT_PREC_BF16);
  const SampleParams prm{sp.temperature, sp.top_k, sp.top_p, 0, (unsigned long long)sp.seed};
  SampleParams* dp = (SampleParams*)o.alloc(sizeof prm);
  if (o.rc) return o.finish("op_sample_step");
  cudaMemcpyAsync(dp, &prm, sizeof prm, cudaMemcpyHostToDevice, o.s);
  SampleState st{};
  st.rows = rows; st.V = V; st.N = samples_per_image; st.T = 0;
  st.params = dp;
  st.t0 = t;
  st.tok_out = token;
  st.lp_out = logprob;
  st.u_out = u_out;
  o.rc = launch_sample_step(st, logits, o.s);
  return o.finish("op_sample_step");
}

}  // extern "C"
