// Engine implementation: weight preparation (BN folding, projection fusion, bf16 / split-bf16 conversion),
// program construction for the three backbones + FPN + heads + Multi-Transformer encoder + KV-cached decoder,
// and execution (eager or CUDA-graph replay).
//
// Reference behaviour followed (paths relative to the reference repo):
//   backbones            models/mobilenet.py:55-72, models/resnet.py:97-112, models/densenet.py:89-103 (+ SURVEY App. C)
//   FPN                  models/retinanet.py:105-141
//   head sub-model       models/retinanet.py:25-102, 283-301 ; models/coattention.py:13-32
//   encoder pre-amble    models/transformer.py:279-296 ; encoder layers :176-200, :298-299
//   decoder              models/transformer.py:224-243, :321-341, :359-374
//   beam loop            utils/pipeline.py:82-154
#include "engine.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>

namespace fpnmt {

static const char* TR = "transformer";
static const std::string RN = "transformer/encoder/feature_extractor/retinanet_model";
static const std::string HM = "transformer/encoder/feature_extractor/model";

#define RC(expr)            \
  do {                      \
    int _rc = (expr);       \
    if (_rc) return _rc;    \
  } while (0)

static int fail(int code, const std::string& msg) {
  set_last_error(msg);
  return code;
}

// --------------------------------------------------------------------------------------------- basics
Engine::Engine(const fpnmt_config& cfg, int device) : cfg_(cfg), dev_(device) { split_ = cfg.precision == FPNMT_PREC_BF16X3; }

Engine::~Engine() {
  cudaSetDevice(dev_);
  if (cnn_graph_) cudaGraphExecDestroy(cnn_graph_);
  if (enc_graph_) cudaGraphExecDestroy(enc_graph_);
  if (step_graph_) cudaGraphExecDestroy(step_graph_);
  if (loop_graph_) cudaGraphExecDestroy(loop_graph_);
  if (sample_graph_) cudaGraphExecDestroy(sample_graph_);
  if (nbest_graph_) cudaGraphExecDestroy(nbest_graph_);
  if (nbest_pfx_graph_) cudaGraphExecDestroy(nbest_pfx_graph_);
  if (sample_pfx_graph_) cudaGraphExecDestroy(sample_pfx_graph_);
  if (nbest_con_graph_) cudaGraphExecDestroy(nbest_con_graph_);
  if (sample_con_graph_) cudaGraphExecDestroy(sample_con_graph_);
  for (auto& kv : score_graphs_)
    if (kv.second) cudaGraphExecDestroy(kv.second);
  if (cap_stream_) cudaStreamDestroy(cap_stream_);
  if (copy_stream_) {
    cudaStreamSynchronize(copy_stream_);
    cudaStreamDestroy(copy_stream_);
  }
  for (int i = 0; i < 2; ++i) {
    if (stage_ready_[i]) cudaEventDestroy(stage_ready_[i]);
    if (stage_free_[i]) cudaEventDestroy(stage_free_[i]);
  }
  if (lane_dec_stream_) {
    cudaStreamSynchronize(lane_dec_stream_);
    cudaStreamDestroy(lane_dec_stream_);
  }
  if (lane_enc_ev_) cudaEventDestroy(lane_enc_ev_);
  if (lane_stream_) {
    cudaStreamSynchronize(lane_stream_);
    cudaStreamDestroy(lane_stream_);
  }
  if (lane_in_ev_) cudaEventDestroy(lane_in_ev_);
  if (lane_out_ev_) cudaEventDestroy(lane_out_ev_);
  if (h_pinned_) cudaFreeHost(h_pinned_);
  for (void* p : allocs_) cudaFree(p);
}

int Engine::init() {
  const fpnmt_config& c = cfg_;
  if (c.d_model != 512 || c.num_heads != 8) return fail(FPNMT_ERR_INVALID, "d_model must be 512 and num_heads 8");
  if (c.batch < 1 || c.beam < 1 || c.beam > 32 || c.vocab < 8 || c.max_len < 1 || c.num_layers < 1)
    return fail(FPNMT_ERR_INVALID, "bad batch / beam / vocab / max_len / num_layers");
  if (c.vocab % 8) return fail(FPNMT_ERR_INVALID, "vocab must be a multiple of 8");
  if (c.image_size < 256 || c.image_size % 256) return fail(FPNMT_ERR_INVALID, "image_size must be a multiple of 256");
  if (c.dff % 8) return fail(FPNMT_ERR_INVALID, "dff must be a multiple of 8");
  if (c.backbone < 0 || c.backbone > 2) return fail(FPNMT_ERR_INVALID, "unknown backbone");
  // a word or bit that selects nothing is refused rather than silently running the defaults
  const int32_t known_opts = FPNMT_OPT_NO_XATTN | FPNMT_OPT_NO_STEM | FPNMT_OPT_NO_TGEMM | FPNMT_OPT_ENC_ATT_SIMT | FPNMT_OPT_NO_PDL |
                             FPNMT_OPT_DEC_ATT_SIMT | FPNMT_OPT_TGEMM_WIDE | FPNMT_OPT_NO_TGEMM_WIDE | FPNMT_OPT_NO_DENSE_1X1 |
                             FPNMT_OPT_NO_B_STATIONARY | FPNMT_OPT_NO_TMA_STORE | FPNMT_OPT_NO_VSTATS | FPNMT_OPT_NO_KV_SHARE |
                             FPNMT_OPT_DSTEP_TAPS;
  if (c.kernel_opts & ~known_opts) return fail(FPNMT_ERR_INVALID, "kernel_opts sets a bit that no FPNMT_OPT_* defines");
  if (c.dec_groups < 0 || c.dec_groups > 1) return fail(FPNMT_ERR_INVALID, "dec_groups must be 0 or 1 (the batch decodes as one chain)");
  if (c.reserved[0]) return fail(FPNMT_ERR_INVALID, "fpnmt_config.reserved must be 0");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  cudaDeviceProp prop;
  FPNMT_CUDA_OK(cudaGetDeviceProperties(&prop, dev_));
  if (prop.major != 10) return fail(FPNMT_ERR_CUDA, "this library contains sm_100a code only; device is not Blackwell");
  num_sms_ = prop.multiProcessorCount;
  RC(igemm_set_attributes());
  RC(tgemm_set_attributes());
  RC(tgemmw_set_attributes());
  RC(xattn_set_attributes());
  RC(elementwise_set_attributes());
  RC(attention_set_attributes());
  RC(beam_set_attributes());
  RC(sample_set_attributes());
  RC(stem_set_attributes());
  use_xattn_ = !(c.kernel_opts & FPNMT_OPT_NO_XATTN);
  use_stem_ = !(c.kernel_opts & FPNMT_OPT_NO_STEM);
  use_tgemm_ = !(c.kernel_opts & FPNMT_OPT_NO_TGEMM);
  set_dec_att_simt((c.kernel_opts & FPNMT_OPT_DEC_ATT_SIMT) != 0);   // process-wide, like the PDL mode
  set_pdl_enabled(!(c.kernel_opts & FPNMT_OPT_NO_PDL));
  if (c.cache_mode < 0 || c.cache_mode > 1 || c.decode_path < 0 || c.decode_path > 2 || c.length_penalty < 0.f)
    return fail(FPNMT_ERR_INVALID, "bad cache_mode / decode_path / length_penalty");
  FPNMT_CUDA_OK(cudaStreamCreateWithFlags(&cap_stream_, cudaStreamNonBlocking));
  FPNMT_CUDA_OK(cudaMallocHost(&h_pinned_, 64));
  return 0;
}

// Timeline buffer for the op named by FPNMT_DBG_OP - only in builds with -DFPNMT_DBG_STAMPS (build.py --dbg-stamps); the
// product build has neither the stamps in the kernels nor this environment lookup.
long long* Engine::dbg_timeline(const std::string& name) {
#ifdef FPNMT_DBG_STAMPS
  const char* dn = getenv("FPNMT_DBG_OP");
  if (dn && name == dn) {
    dbg_buf_ = (long long*)dalloc(192 * sizeof(long long));
    if (dbg_buf_) cudaMemset(dbg_buf_, 0, 192 * sizeof(long long));
    return dbg_buf_;
  }
#endif
  (void)name;
  return nullptr;
}

void* Engine::dalloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    set_last_error("cudaMalloc of " + std::to_string(bytes) + " bytes failed (engine holds " + std::to_string(alloc_bytes_) + ")");
    return nullptr;
  }
  allocs_.push_back(p);
  alloc_bytes_ += bytes;
  return p;
}

Tensor Engine::new_act(int N, int H, int W, int C) {
  Tensor t;
  t.N = N; t.H = H; t.W = W;
  const int cs = std::max(8, (C + 7) / 8 * 8);
  t.a.C = C;
  t.a.ld = split_ ? 2 * cs : cs;
  t.a.lo = split_ ? cs : 0;
  t.a.p = (bf16*)dalloc((size_t)N * H * W * t.a.ld * sizeof(bf16));
  return t;
}
Tensor Engine::chan_view(const Tensor& t, int c0, int C) {
  Tensor v = t;
  v.a.p = t.a.p + c0;
  v.a.C = C;
  return v;
}

int Engine::set_weight(const char* key, const float* data, const int64_t* shape, int ndim) {
  if (!key || !data || ndim < 1 || ndim > 4) return fail(FPNMT_ERR_INVALID, "set_weight: bad arguments");
  HostW w;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    w.shape.push_back(shape[i]);
    n *= (size_t)shape[i];
  }
  w.data.assign(data, data + n);
  hw_[key] = std::move(w);
  return 0;
}
const HostW* Engine::W(const std::string& key) {
  auto it = hw_.find(key);
  if (it == hw_.end()) {
    set_last_error("missing weight: " + key);
    return nullptr;
  }
  return &it->second;
}

int Engine::upload_f32(const std::vector<float>& v, float** out) {
  *out = (float*)dalloc(std::max<size_t>(v.size(), 4) * sizeof(float));
  if (!*out) return FPNMT_ERR_CUDA;
  FPNMT_CUDA_OK(cudaMemcpy(*out, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}
int Engine::prep_vec(const std::string& key, float** out) {
  const HostW* w = W(key);
  if (!w) return FPNMT_ERR_MISSING;
  return upload_f32(w->data, out);
}

void xattn_fold_weights(const float* wq, const float* wo, uint16_t* wq_bf16, uint16_t* woT_bf16) {
  for (size_t i = 0; i < 512 * 512; ++i) wq_bf16[i] = f2bf(wq[i]);
  for (int hd = 0; hd < 512; ++hd)
    for (int f = 0; f < 512; ++f) woT_bf16[(size_t)f * 512 + hd] = f2bf(wo[(size_t)hd * 512 + f]);
}

int Engine::upload_gemm(const std::vector<float>& wt, const std::vector<float>& bias, int Cout, int K, GemmW* out) {
  if (K % 8) return fail(FPNMT_ERR_INVALID, "upload_gemm: K must be a multiple of 8");
  if (weight_lead_) {                               // follower lane: the lead lane's device copy (see engine.cuh)
    if (gemm_log_pos_ >= weight_lead_->gemm_log_.size() || weight_lead_->gemm_log_[gemm_log_pos_].Cout != Cout ||
        weight_lead_->gemm_log_[gemm_log_pos_].K != K || weight_lead_->split_ != split_)
      return fail(FPNMT_ERR_STATE, "lane weight sharing: finalize sequences of the lanes differ");
    *out = weight_lead_->gemm_log_[gemm_log_pos_++];
    return 0;
  }
  const size_t ldw = split_ ? 2 * (size_t)K : (size_t)K;
  std::vector<uint16_t> h((size_t)Cout * ldw);
  for (int r = 0; r < Cout; ++r)
    for (int k = 0; k < K; ++k) {
      const float f = wt[(size_t)r * K + k];
      const uint16_t hi = f2bf(f);
      h[r * ldw + k] = hi;
      if (split_) h[r * ldw + K + k] = f2bf(f - bf2f(hi));
    }
  out->w = (bf16*)dalloc(h.size() * 2);
  if (!out->w) return FPNMT_ERR_CUDA;
  FPNMT_CUDA_OK(cudaMemcpy(out->w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  std::vector<float> b = bias;
  b.resize((size_t)(Cout + 31) / 32 * 32, 0.f);   // the epilogue reads bias in 32-column units
  RC(upload_f32(b, &out->bias));
  out->Cout = Cout;
  out->K = K;
  gemm_log_.push_back(*out);
  return 0;
}

// Conv2D kernel (kh,kw,Cin,Cout) [+bias] [+ following inference BatchNorm folded] -> Wt[Cout][kh*kw*Cin (padded to kpad)]
int Engine::prep_conv(const std::string& kernel_key, const std::string& bias_key, const std::string& bn, float eps,
                      GemmW* out, int kpad) {
  const HostW* k = W(kernel_key);
  if (!k) return FPNMT_ERR_MISSING;
  if (k->shape.size() != 4) return fail(FPNMT_ERR_INVALID, kernel_key + ": conv kernel must be rank 4");
  const int kh = (int)k->shape[0], kw = (int)k->shape[1], cin = (int)k->shape[2], cout = (int)k->shape[3];
  const int K = kh * kw * cin;
  const int Kp = kpad ? kpad : K;
  std::vector<float> scale(cout, 1.f), shift(cout, 0.f);
  if (k->data.size() != (size_t)K * cout) return fail(FPNMT_ERR_INVALID, kernel_key + ": element count does not match its shape");
  if (kpad && kpad < K) return fail(FPNMT_ERR_INVALID, kernel_key + ": more taps x channels than the layer takes");
  if (!bias_key.empty()) {
    const HostW* b = W(bias_key);
    if (!b) return FPNMT_ERR_MISSING;
    if (b->data.size() != (size_t)cout) return fail(FPNMT_ERR_INVALID, bias_key + ": expected " + std::to_string(cout) + " values");
    for (int o = 0; o < cout; ++o) shift[o] = b->data[o];
  }
  if (!bn.empty()) {
    const HostW *g = W(bn + "/gamma"), *be = W(bn + "/beta"), *m = W(bn + "/moving_mean"), *v = W(bn + "/moving_variance");
    if (!g || !be || !m || !v) return FPNMT_ERR_MISSING;
    if (g->data.size() != (size_t)cout || be->data.size() != (size_t)cout || m->data.size() != (size_t)cout || v->data.size() != (size_t)cout)
      return fail(FPNMT_ERR_INVALID, bn + ": BatchNorm vectors must have " + std::to_string(cout) + " values (the convolution's filters)");
    for (int o = 0; o < cout; ++o) {
      const float s = g->data[o] / sqrtf(v->data[o] + eps);
      shift[o] = (shift[o] - m->data[o]) * s + be->data[o];
      scale[o] = s;
    }
  }
  std::vector<float> wt((size_t)cout * Kp, 0.f);
  for (int t = 0; t < kh * kw; ++t)
    for (int ci = 0; ci < cin; ++ci) {
      const float* src = &k->data[((size_t)t * cin + ci) * cout];
      for (int o = 0; o < cout; ++o) wt[(size_t)o * Kp + (size_t)t * cin + ci] = src[o] * scale[o];
    }
  return upload_gemm(wt, shift, cout, Kp, out);
}

// Dense layers sharing one input, concatenated along the output axis: Wt[sum out][in]
int Engine::prep_dense_cat(const std::vector<std::string>& names, GemmW* out) {
  int in = -1, tot = 0;
  for (auto& n : names) {
    const HostW* k = W(n + "/kernel");
    if (!k) return FPNMT_ERR_MISSING;
    if (k->shape.size() != 2 || k->data.size() != (size_t)(k->shape[0] * k->shape[1]))
      return fail(FPNMT_ERR_INVALID, n + "/kernel: Dense kernel must be rank 2 (in, out)");
    if (in < 0) in = (int)k->shape[0];
    if ((int)k->shape[0] != in) return fail(FPNMT_ERR_INVALID, "prep_dense_cat: input dims differ");
    tot += (int)k->shape[1];
  }
  std::vector<float> wt((size_t)tot * in), bias(tot);
  int o0 = 0;
  for (auto& n : names) {
    const HostW *k = W(n + "/kernel"), *b = W(n + "/bias");
    if (!b) return FPNMT_ERR_MISSING;
    const int co = (int)k->shape[1];
    if (b->data.size() != (size_t)co) return fail(FPNMT_ERR_INVALID, n + "/bias: expected " + std::to_string(co) + " values");
    for (int i = 0; i < in; ++i)
      for (int o = 0; o < co; ++o) wt[(size_t)(o0 + o) * in + i] = k->data[(size_t)i * co + o];
    for (int o = 0; o < co; ++o) bias[o0 + o] = b->data[o];
    o0 += co;
  }
  return upload_gemm(wt, bias, tot, in, out);
}

// Dense layers whose outputs are summed, inputs concatenated: y = [x0|x1|..] @ [W0;W1;..] + sum(b)
int Engine::prep_dense_stack(const std::vector<std::string>& names, GemmW* out) {
  int co = -1, tot = 0;
  for (auto& n : names) {
    const HostW* k = W(n + "/kernel");
    if (!k) return FPNMT_ERR_MISSING;
    if (k->shape.size() != 2 || k->data.size() != (size_t)(k->shape[0] * k->shape[1]))
      return fail(FPNMT_ERR_INVALID, n + "/kernel: Dense kernel must be rank 2 (in, out)");
    if (co < 0) co = (int)k->shape[1];
    if ((int)k->shape[1] != co) return fail(FPNMT_ERR_INVALID, "prep_dense_stack: output dims differ (" + n + ")");
    tot += (int)k->shape[0];
  }
  std::vector<float> wt((size_t)co * tot), bias(co, 0.f);
  int i0 = 0;
  for (auto& n : names) {
    const HostW *k = W(n + "/kernel"), *b = W(n + "/bias");
    if (!b) return FPNMT_ERR_MISSING;
    if (b->data.size() != (size_t)co) return fail(FPNMT_ERR_INVALID, n + "/bias: expected " + std::to_string(co) + " values");
    const int in = (int)k->shape[0];
    for (int i = 0; i < in; ++i)
      for (int o = 0; o < co; ++o) wt[(size_t)o * tot + i0 + i] = k->data[(size_t)i * co + o];
    for (int o = 0; o < co; ++o) bias[o] += b->data[o];
    i0 += in;
  }
  return upload_gemm(wt, bias, co, tot, out);
}

int Engine::prep_bn_affine(const std::string& bn, float eps, int C, float** scale, float** shift) {
  const HostW *g = W(bn + "/gamma"), *be = W(bn + "/beta"), *m = W(bn + "/moving_mean"), *v = W(bn + "/moving_variance");
  if (!g || !be || !m || !v) return FPNMT_ERR_MISSING;
  std::vector<float> s(C), t(C);
  for (int c = 0; c < C; ++c) {
    s[c] = g->data[c] / sqrtf(v->data[c] + eps);
    t[c] = be->data[c] - m->data[c] * s[c];
  }
  RC(upload_f32(s, scale));
  return upload_f32(t, shift);
}

int Engine::prep_depthwise(const std::string& key, const std::string& bn, float eps, float** w, float** bias) {
  const HostW* k = W(key);
  if (!k) return FPNMT_ERR_MISSING;
  const int C = (int)k->shape[2];
  const HostW *g = W(bn + "/gamma"), *be = W(bn + "/beta"), *m = W(bn + "/moving_mean"), *v = W(bn + "/moving_variance");
  if (!g || !be || !m || !v) return FPNMT_ERR_MISSING;
  std::vector<float> wt(9 * (size_t)C), b(C);
  for (int c = 0; c < C; ++c) {
    const float s = g->data[c] / sqrtf(v->data[c] + eps);
    for (int t = 0; t < 9; ++t) wt[(size_t)t * C + c] = k->data[(size_t)t * C + c] * s;
    b[c] = be->data[c] - m->data[c] * s;
  }
  RC(upload_f32(wt, w));
  return upload_f32(b, bias);
}

// --------------------------------------------------------------------------------------------- op builders
int Engine::add_conv(Program& prog, const std::string& name, const Tensor& in, const GemmW& gw, int kh, int kw, int pad_t,
                     int pad_l, int act, int res_mode, const Tensor* res, const Tensor& out, float* out_f32, int ld_f32) {
  if (!in.a.p || (!out.a.p && !out_f32)) return FPNMT_ERR_CUDA;
  ConvGeom g{in.N, in.H, in.W, in.a.C, gw.Cout, kh, kw, pad_t, pad_l};
  // A 1x1 convolution is a GEMM over the pixels: run it in the dense geometry (128 consecutive pixels per tile, plain 2-D
  // operand boxes) unless the residual is the half-resolution map of an FPN lateral.
  if (kh == 1 && kw == 1 && pad_t == 0 && pad_l == 0 && res_mode != RES_UP2 && !(cfg_.kernel_opts & FPNMT_OPT_NO_DENSE_1X1)) {
    g.W = in.N * in.H * in.W;
    g.N = 1;
    g.H = 1;
  }
  if (gw.K < kh * kw * in.a.C) return fail(FPNMT_ERR_INVALID, name + ": weight K smaller than kh*kw*Cin");
  if (out.a.p && gw.Cout != out.a.C)
    return fail(FPNMT_ERR_INVALID, name + ": the kernel has " + std::to_string(gw.Cout) + " filters, the layer's output " + std::to_string(out.a.C) + " channels");
  IgemmOp op;
  Act r{nullptr, 0, 0, 0};
  if (res) r = res->a;
  // a K-padded weight (stem im2col) is addressed with Cin == K
  RC(make_igemm_op(&op, g, in.a, gw.w, split_, gw.bias, act, out.a, out_f32, ld_f32, res_mode, r, num_sms_, 0,
                   !(cfg_.kernel_opts & FPNMT_OPT_NO_TMA_STORE), !(cfg_.kernel_opts & FPNMT_OPT_NO_B_STATIONARY)));
  op.p.dbg = dbg_timeline(name);
  Op o;
  o.name = name;
  o.kind = "igemm";
  o.flops = op.flops * (split_ ? 3.0 : 1.0);
  const double esz = split_ ? 4.0 : 2.0;
  o.bytes = (double)in.pixels() * in.a.C * esz + (double)gw.Cout * gw.K * esz +
            (double)in.pixels() * gw.Cout * (out_f32 ? 4.0 : esz) + (res ? (double)res->pixels() * gw.Cout * esz : 0.0);
  o.run = [op](cudaStream_t s) { return igemm_launch(op, s); };
  prog.push_back(std::move(o));
  return 0;
}

int Engine::add_dense(Program& prog, const std::string& name, const Tensor& in, const GemmW& gw, int act, const Tensor* res,
                      const Tensor& out, float* out_f32, int ld_f32, const float* gamma, const float* beta) {
  if (!in.a.p || (!out.a.p && !out_f32)) return FPNMT_ERR_CUDA;
  if (gw.K != in.a.C) return fail(FPNMT_ERR_INVALID, name + ": Dense kernel takes " + std::to_string(gw.K) + " inputs, the layer feeds " + std::to_string(in.a.C));
  if (out.a.p && gw.Cout != out.a.C)
    return fail(FPNMT_ERR_INVALID, name + ": Dense kernel has " + std::to_string(gw.Cout) + " outputs, the layer's output " + std::to_string(out.a.C));
  if (out_f32 && gw.Cout > ld_f32) return fail(FPNMT_ERR_INVALID, name + ": Dense kernel has more outputs than the fp32 output row");
  const int R = (int)in.pixels();
  TgemmOp op;
  const bool want_wide = (cfg_.kernel_opts & FPNMT_OPT_TGEMM_WIDE) || (cfg_.lanes >= 2 && !(cfg_.kernel_opts & FPNMT_OPT_NO_TGEMM_WIDE));
  if (want_wide && out_f32 == nullptr && tgemmw_supports(split_, res != nullptr, gamma != nullptr, gw.Cout, gw.K))
    RC(make_tgemmw_op(&op, R, in.a, gw.w, gw.Cout, gw.K, gw.bias, act, out.a, out_f32, ld_f32, res ? &res->a : nullptr, gamma, beta,
                      1e-6f, num_sms_));
  else
    RC(make_tgemm_op(&op, R, in.a, gw.w, gw.Cout, gw.K, split_, gw.bias, act, out.a, out_f32, ld_f32, res ? &res->a : nullptr,
                     gamma, beta, 1e-6f, num_sms_));
  op.p.dbg = dbg_timeline(name);
  Op o;
  o.name = name;
  o.kind = "tgemm";
  o.flops = op.flops * (split_ ? 3.0 : 1.0);
  const double esz = split_ ? 4.0 : 2.0;
  o.bytes = (double)R * gw.K * esz + (double)gw.Cout * gw.K * esz + (double)R * gw.Cout * (out_f32 ? 4.0 : esz) +
            (res ? (double)R * gw.Cout * esz : 0.0);
  o.run = [op](cudaStream_t s) { return tgemm_launch(op, s); };
  prog.push_back(std::move(o));
  return 0;
}

int Engine::add_stem(Program& p, const std::string& name, int kh, int pad, int cout, const GemmW& gw, int Kp, int act,
                     const Tensor& out) {
  const int B = cfg_.batch, S = cfg_.image_size;
  StemOp so;
  const int ks = (kh + 1) / 2;
  bf16* wp = (bf16*)dalloc((size_t)cout * ks * ks * 12 * sizeof(bf16));
  if (!wp) return FPNMT_ERR_CUDA;
  RC(make_stem_op(&so, img_slot_, B, S, S, kh, pad, cout, gw.w, Kp, wp, gw.bias, act, out.a, num_sms_));
  so.p.dbg = dbg_timeline(name);
  Op o;
  o.name = name;
  o.kind = "igemm";
  o.flops = so.flops;
  o.bytes = (double)B * S * S * 3 * 4 + (double)out.pixels() * cout * 2;
  o.run = [so](cudaStream_t s) { return stem_launch(so, s); };
  p.push_back(std::move(o));
  stem_fused_ = true;
  return 0;
}

static Op ew_op(const std::string& name, std::function<int(cudaStream_t)> fn, double bytes, const char* kind = "elementwise") {
  Op o;
  o.name = name;
  o.kind = kind;
  o.run = std::move(fn);
  o.bytes = bytes;
  return o;
}

// im2col + GEMM stem for the Cin=3 first convolution (7x7 s2 pad 3 for ResNet/DenseNet)
int Engine::build_stem_resnet_like(Program& p, const std::string& conv_key, const std::string& bn_key, float eps,
                                   Tensor* out) {
  const int B = cfg_.batch, S = cfg_.image_size, So = S / 2;
  const int Kp = 152;   // 7*7*3 = 147 padded to a multiple of 8
  if (use_stem_ && !split_) {   // bf16 mode: fused tcgen05 stem kernel, no im2col matrix in HBM
    GemmW gw;
    RC(prep_conv(conv_key, "", bn_key, eps, &gw, Kp));
    Tensor y = new_act(B, So, So, 64);
    RC(add_stem(p, "stem_fused", 7, 3, 64, gw, Kp, ACT_RELU, y));
    *out = y;
    return 0;
  }
  Tensor col = new_act(1, 1, B * So * So, Kp);
  const float** slot = img_slot_;
  Act ca = col.a;
  p.push_back(ew_op("stem_im2col", [=](cudaStream_t s) { return launch_im2col_stem(slot, B, S, S, 7, 7, 2, 3, 3, So, So, ca, s); },
                    (double)B * S * S * 3 * 4 + (double)col.pixels() * Kp * (split_ ? 4 : 2)));
  GemmW gw;
  RC(prep_conv(conv_key, "", bn_key, eps, &gw, Kp));
  Tensor y = new_act(B, So, So, 64);
  Tensor yrows = y;
  yrows.N = 1; yrows.H = 1; yrows.W = B * So * So;
  RC(add_conv(p, "stem_conv", col, gw, 1, 1, 0, 0, ACT_RELU, RES_NONE, nullptr, yrows));
  // the GEMM saw K = Kp input channels
  *out = y;
  return 0;
}

int Engine::build_resnet50(Program& p, Tensor c[3]) {
  const int B = cfg_.batch;
  Tensor x;
  RC(build_stem_resnet_like(p, RN + "/conv1/kernel", RN + "/bn_conv1", 1e-5f, &x));
  {   // pool1: 3x3 s2 'same' (even size -> pad bottom/right only)
    Tensor y = new_act(B, x.H / 2, x.W / 2, 64);
    Act xa = x.a, ya = y.a;
    const int H = x.H, W = x.W;
    p.push_back(ew_op("pool1", [=](cudaStream_t s) { return launch_maxpool(xa, B, H, W, 3, 2, 0, 0, H / 2, W / 2, false, ya, s); },
                      (double)x.pixels() * 64 * 2 * 1.25));
    x = y;
  }
  const int nblk[4] = {3, 4, 6, 3};
  int ti = 0;
  for (int st = 0; st < 4; ++st) {
    const int f = 64 << st;
    for (int b = 0; b < nblk[st]; ++b) {
      char nm[8];
      snprintf(nm, sizeof nm, "%d%c", st + 2, 'a' + b);
      const std::string n(nm);
      Tensor xin = x;
      if (b == 0 && st > 0) {   // stride 2 on the first 1x1 (and on the shortcut): subsample once
        Tensor sub = new_act(B, x.H / 2, x.W / 2, x.a.C);
        Act xa = x.a, sa = sub.a;
        const int H = x.H, W = x.W;
        p.push_back(ew_op("res" + n + "_subsample", [=](cudaStream_t s) { return launch_subsample2(xa, B, H, W, sa, s); },
                          (double)sub.pixels() * x.a.C * 4));
        xin = sub;
      }
      GemmW wa, wb, wc;
      RC(prep_conv(RN + "/res" + n + "_branch2a/kernel", "", RN + "/bn" + n + "_branch2a", 1e-5f, &wa));
      RC(prep_conv(RN + "/res" + n + "_branch2b/kernel", "", RN + "/bn" + n + "_branch2b", 1e-5f, &wb));
      RC(prep_conv(RN + "/res" + n + "_branch2c/kernel", "", RN + "/bn" + n + "_branch2c", 1e-5f, &wc));
      Tensor ya = new_act(B, xin.H, xin.W, f), yb = new_act(B, xin.H, xin.W, f), yc = new_act(B, xin.H, xin.W, 4 * f);
      RC(add_conv(p, "res" + n + "_2a", xin, wa, 1, 1, 0, 0, ACT_RELU, RES_NONE, nullptr, ya));
      RC(add_conv(p, "res" + n + "_2b", ya, wb, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, yb));
      Tensor sc = xin;
      if (b == 0) {
        GemmW w1;
        RC(prep_conv(RN + "/res" + n + "_branch1/kernel", "", RN + "/bn" + n + "_branch1", 1e-5f, &w1));
        sc = new_act(B, xin.H, xin.W, 4 * f);
        RC(add_conv(p, "res" + n + "_1", xin, w1, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, sc));
      }
      RC(add_conv(p, "res" + n + "_2c", yb, wc, 1, 1, 0, 0, ACT_RELU, RES_SAME, &sc, yc));
      x = yc;
    }
    if (st >= 1) c[ti++] = x;
  }
  return 0;
}

int Engine::build_mobilenetv2(Program& p, Tensor c[3]) {
  const int B = cfg_.batch, S = cfg_.image_size, So = S / 2;
  const float eps = 1e-3f;
  // Conv1: ZeroPadding2D(((0,1),(0,1))) + 3x3 s2 valid
  const int Kp = 32;
  GemmW g1;
  RC(prep_conv(RN + "/Conv1/kernel", "", RN + "/bn_Conv1", eps, &g1, Kp));
  Tensor x = new_act(B, So, So, 32);
  if (use_stem_ && !split_) {   // bf16 mode: fused tcgen05 stem kernel, no im2col matrix in HBM
    RC(add_stem(p, "Conv1_fused", 3, 0, 32, g1, Kp, ACT_RELU6, x));
  } else {
    Tensor col = new_act(1, 1, B * So * So, Kp);
    const float** slot = img_slot_;
    Act ca = col.a;
    p.push_back(ew_op("Conv1_im2col", [=](cudaStream_t s) { return launch_im2col_stem(slot, B, S, S, 3, 3, 2, 0, 0, So, So, ca, s); },
                      (double)B * S * S * 3 * 4 + (double)col.pixels() * Kp * (split_ ? 4 : 2)));
    Tensor xr = x;
    xr.N = 1; xr.H = 1; xr.W = B * So * So;
    RC(add_conv(p, "Conv1", col, g1, 1, 1, 0, 0, ACT_RELU6, RES_NONE, nullptr, xr));
  }
  auto depthwise = [&](const std::string& name, const Tensor& in, int stride, Tensor* out) -> int {
    float *w, *b;
    RC(prep_depthwise(RN + "/" + name + "/depthwise_kernel", RN + "/" + name + "_BN", eps, &w, &b));
    const int Ho = in.H / stride, Wo = in.W / stride;
    Tensor y = new_act(B, Ho, Wo, in.a.C);
    Act ia = in.a, ya = y.a;
    const int H = in.H, Wd = in.W;
    const int pad = stride == 1 ? 1 : 0;
    p.push_back(ew_op(name, [=](cudaStream_t s) { return launch_depthwise3x3(ia, B, H, Wd, stride, pad, pad, Ho, Wo, w, b, ACT_RELU6, ya, s); },
                      ((double)in.pixels() + y.pixels()) * in.a.C * 2));
    *out = y;
    return 0;
  };
  {   // expanded_conv
    Tensor d;
    RC(depthwise("expanded_conv_depthwise", x, 1, &d));
    GemmW gp;
    RC(prep_conv(RN + "/expanded_conv_project/kernel", "", RN + "/expanded_conv_project_BN", eps, &gp));
    Tensor y = new_act(B, d.H, d.W, 16);
    RC(add_conv(p, "expanded_conv_project", d, gp, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, y));
    x = y;
  }
  const int blocks[16][2] = {{24, 2}, {24, 1}, {32, 2}, {32, 1}, {32, 1}, {64, 2}, {64, 1}, {64, 1}, {64, 1}, {96, 1},
                             {96, 1}, {96, 1}, {160, 2}, {160, 1}, {160, 1}, {320, 1}};
  for (int k = 1; k <= 16; ++k) {
    const int cout = blocks[k - 1][0], stride = blocks[k - 1][1];
    const int cin = x.a.C;
    const std::string pre = "block_" + std::to_string(k);
    GemmW ge, gp;
    RC(prep_conv(RN + "/" + pre + "_expand/kernel", "", RN + "/" + pre + "_expand_BN", eps, &ge));
    Tensor e = new_act(B, x.H, x.W, 6 * cin);
    RC(add_conv(p, pre + "_expand", x, ge, 1, 1, 0, 0, ACT_RELU6, RES_NONE, nullptr, e));
    Tensor d;
    RC(depthwise(pre + "_depthwise", e, stride, &d));
    RC(prep_conv(RN + "/" + pre + "_project/kernel", "", RN + "/" + pre + "_project_BN", eps, &gp));
    Tensor y = new_act(B, d.H, d.W, cout);
    const bool add = (stride == 1 && cin == cout);
    RC(add_conv(p, pre + "_project", d, gp, 1, 1, 0, 0, ACT_NONE, add ? RES_SAME : RES_NONE, add ? &x : nullptr, y));
    x = y;
    if (k == 5) c[0] = x;    // block_5_add
    if (k == 12) c[1] = x;   // block_12_add
  }
  GemmW gl;
  RC(prep_conv(RN + "/Conv_1/kernel", "", RN + "/Conv_1_bn", eps, &gl));
  Tensor y = new_act(B, x.H, x.W, 1280);
  RC(add_conv(p, "Conv_1", x, gl, 1, 1, 0, 0, ACT_RELU6, RES_NONE, nullptr, y));
  c[2] = y;                  // out_relu
  return 0;
}

int Engine::build_densenet121(Program& p, Tensor c[3]) {
  const int B = cfg_.batch;
  const float eps = 1.001e-5f;
  Tensor x;
  RC(build_stem_resnet_like(p, RN + "/conv1/conv/kernel", RN + "/conv1/bn", eps, &x));
  const int nblk[4] = {6, 12, 24, 16};
  int cch = 64;
  int H = x.H / 2, Wd = x.W / 2;
  Tensor buf = new_act(B, H, Wd, cch + 32 * nblk[0]);
  {   // pool1: ZeroPadding2D(1) + 3x3 s2 valid, written into the first 64 channels of the stage buffer
    Act xa = x.a, ya = chan_view(buf, 0, 64).a;
    const int Hi = x.H, Wi = x.W;
    p.push_back(ew_op("pool1", [=](cudaStream_t s) { return launch_maxpool(xa, B, Hi, Wi, 3, 2, 1, 1, Hi / 2, Wi / 2, true, ya, s); },
                      (double)x.pixels() * 64 * 2 * 1.25));
  }
  int ti = 0;
  for (int si = 0; si < 4; ++si) {
    const int stage = si + 2;
    for (int b = 1; b <= nblk[si]; ++b) {
      const std::string pre = RN + "/conv" + std::to_string(stage) + "_block" + std::to_string(b);
      const std::string sn = "conv" + std::to_string(stage) + "_block" + std::to_string(b);
      float *sc, *sh;
      RC(prep_bn_affine(pre + "_0_bn", eps, cch, &sc, &sh));
      Tensor t0 = new_act(B, H, Wd, cch);
      Act ia = chan_view(buf, 0, cch).a, ta = t0.a;
      const size_t pix = t0.pixels();
      p.push_back(ew_op(sn + "_0_bn_relu", [=](cudaStream_t s) { return launch_scale_shift_relu(ia, pix, sc, sh, ta, s); },
                        (double)pix * cch * 4));
      GemmW g1, g2;
      RC(prep_conv(pre + "_1_conv/kernel", "", pre + "_1_bn", eps, &g1));
      RC(prep_conv(pre + "_2_conv/kernel", "", "", 0.f, &g2));
      Tensor y1 = new_act(B, H, Wd, 128);
      RC(add_conv(p, sn + "_1_conv", t0, g1, 1, 1, 0, 0, ACT_RELU, RES_NONE, nullptr, y1));
      RC(add_conv(p, sn + "_2_conv", y1, g2, 3, 3, 1, 1, ACT_NONE, RES_NONE, nullptr, chan_view(buf, cch, 32)));
      cch += 32;
    }
    if (si >= 1) c[ti++] = chan_view(buf, 0, cch);
    if (si < 3) {
      const std::string pre = RN + "/pool" + std::to_string(stage);
      float *sc, *sh;
      RC(prep_bn_affine(pre + "_bn", eps, cch, &sc, &sh));
      Tensor t0 = new_act(B, H, Wd, cch);
      Act ia = chan_view(buf, 0, cch).a, ta = t0.a;
      const size_t pix = t0.pixels();
      p.push_back(ew_op("pool" + std::to_string(stage) + "_bn_relu",
                        [=](cudaStream_t s) { return launch_scale_shift_relu(ia, pix, sc, sh, ta, s); }, (double)pix * cch * 4));
      GemmW g;
      RC(prep_conv(pre + "_conv/kernel", "", "", 0.f, &g));
      Tensor y = new_act(B, H, Wd, cch / 2);
      RC(add_conv(p, "pool" + std::to_string(stage) + "_conv", t0, g, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, y));
      cch /= 2;
      Tensor nbuf = new_act(B, H / 2, Wd / 2, cch + 32 * nblk[si + 1]);
      Act ya = y.a, na = chan_view(nbuf, 0, cch).a;
      const int Hi = H, Wi = Wd;
      p.push_back(ew_op("pool" + std::to_string(stage) + "_pool", [=](cudaStream_t s) { return launch_avgpool2(ya, B, Hi, Wi, na, s); },
                        (double)y.pixels() * cch * 2 * 1.25));
      buf = nbuf;
      H /= 2;
      Wd /= 2;
    }
  }
  return 0;
}

// FPN (retinanet.py:105-141) + per-level head sub-model (retinanet.py:283-301) + token pre-amble (transformer.py:279-296)
int Engine::build_fpn_heads(Program& p, Tensor c[3]) {
  const int B = cfg_.batch;
  const int F = 256, D = cfg_.d_model;
  taps_["C3"] = c[0]; taps_["C4"] = c[1]; taps_["C5"] = c[2];
  GemmW c5r, p5w, c4r, p4w, c3r, p3w, p6w, p7w;
  RC(prep_conv(RN + "/C5_reduced/kernel", RN + "/C5_reduced/bias", "", 0, &c5r));
  RC(prep_conv(RN + "/P5/kernel", RN + "/P5/bias", "", 0, &p5w));
  RC(prep_conv(RN + "/C4_reduced/kernel", RN + "/C4_reduced/bias", "", 0, &c4r));
  RC(prep_conv(RN + "/P4/kernel", RN + "/P4/bias", "", 0, &p4w));
  RC(prep_conv(RN + "/C3_reduced/kernel", RN + "/C3_reduced/bias", "", 0, &c3r));
  RC(prep_conv(RN + "/P3/kernel", RN + "/P3/bias", "", 0, &p3w));
  RC(prep_conv(RN + "/conv2d/kernel", RN + "/conv2d/bias", "", 0, &p6w));
  RC(prep_conv(RN + "/conv2d_1/kernel", RN + "/conv2d_1/bias", "", 0, &p7w));
  Tensor P[5];
  Tensor p5f = new_act(B, c[2].H, c[2].W, F);
  RC(add_conv(p, "C5_reduced", c[2], c5r, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, p5f));
  P[2] = new_act(B, p5f.H, p5f.W, F);
  RC(add_conv(p, "P5", p5f, p5w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, P[2]));
  Tensor p4m = new_act(B, c[1].H, c[1].W, F);   // lateral 1x1 with the nearest-2x upsample + add fused into the epilogue
  RC(add_conv(p, "C4_reduced+P5_upsampled", c[1], c4r, 1, 1, 0, 0, ACT_NONE, RES_UP2, &p5f, p4m));
  P[1] = new_act(B, p4m.H, p4m.W, F);
  RC(add_conv(p, "P4", p4m, p4w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, P[1]));
  Tensor p3m = new_act(B, c[0].H, c[0].W, F);
  RC(add_conv(p, "C3_reduced+P4_upsampled", c[0], c3r, 1, 1, 0, 0, ACT_NONE, RES_UP2, &p4m, p3m));
  P[0] = new_act(B, p3m.H, p3m.W, F);
  RC(add_conv(p, "P3", p3m, p3w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, P[0]));
  auto pool2 = [&](const std::string& name, const Tensor& in, Tensor* out) {
    Tensor y = new_act(B, in.H / 2, in.W / 2, in.a.C);
    Act ia = in.a, ya = y.a;
    const int H = in.H, W = in.W;
    p.push_back(ew_op(name, [=](cudaStream_t s) { return launch_maxpool(ia, B, H, W, 2, 2, 0, 0, H / 2, W / 2, false, ya, s); },
                      (double)in.pixels() * in.a.C * 2 * 1.25));
    *out = y;
  };
  {
    Tensor t = new_act(B, p5f.H, p5f.W, F);
    RC(add_conv(p, "P6_conv", p5f, p6w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, t));
    pool2("P6", t, &P[3]);
    Tensor t2 = new_act(B, P[3].H, P[3].W, F);
    RC(add_conv(p, "P7_conv", P[3], p7w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, t2));
    pool2("P7", t2, &P[4]);
  }
  const char* pn[5] = {"P3", "P4", "P5", "P6", "P7"};
  for (int i = 0; i < 5; ++i) taps_[pn[i]] = P[i];

  // shared head weights
  GemmW t0w, r1w, c1w, scw, clw, h4w, h5w;
  {   // first trunk convs of both sub-models share their input: one conv with Cout = 512 ([reg | cls])
    const HostW *kr = W(RN + "/regression_submodel/pyramid_regression_0/kernel"), *br = W(RN + "/regression_submodel/pyramid_regression_0/bias");
    const HostW *kc = W(RN + "/classification_submodel/pyramid_classification_0/kernel"), *bc = W(RN + "/classification_submodel/pyramid_classification_0/bias");
    if (!kr || !br || !kc || !bc) return FPNMT_ERR_MISSING;
    const int K = 9 * F;
    std::vector<float> wt((size_t)2 * F * K), bias(2 * F);
    for (int t = 0; t < 9; ++t)
      for (int ci = 0; ci < F; ++ci)
        for (int o = 0; o < F; ++o) {
          wt[(size_t)o * K + t * F + ci] = kr->data[((size_t)t * F + ci) * F + o];
          wt[(size_t)(F + o) * K + t * F + ci] = kc->data[((size_t)t * F + ci) * F + o];
        }
    for (int o = 0; o < F; ++o) {
      bias[o] = br->data[o];
      bias[F + o] = bc->data[o];
    }
    RC(upload_gemm(wt, bias, 2 * F, K, &t0w));
  }
  RC(prep_conv(RN + "/regression_submodel/pyramid_regression_1/kernel", RN + "/regression_submodel/pyramid_regression_1/bias", "", 0, &r1w));
  RC(prep_conv(RN + "/classification_submodel/pyramid_classification_1/kernel", RN + "/classification_submodel/pyramid_classification_1/bias", "", 0, &c1w));
  RC(prep_conv(HM + "/conv2d_2/kernel", HM + "/conv2d_2/bias", "", 0, &scw));
  float *score_w = nullptr, *score_b = nullptr;      // fp32 [9][256] (HWIO with O = 1 is already tap-major) + bias
  if (!split_ && F == 256) {
    RC(prep_vec(HM + "/conv2d_2/kernel", &score_w));
    RC(prep_vec(HM + "/conv2d_2/bias", &score_b));
  }
  RC(prep_conv(HM + "/conv2d_3/kernel", HM + "/conv2d_3/bias", "", 0, &clw));
  RC(prep_conv(HM + "/conv2d_4/kernel", HM + "/conv2d_4/bias", "", 0, &h4w));
  RC(prep_conv(HM + "/conv2d_5/kernel", HM + "/conv2d_5/bias", "", 0, &h5w));

  for (int i = 0; i < 5; ++i) {
    const std::string L = pn[i];
    const Tensor& x = P[i];
    Tensor t0 = new_act(B, x.H, x.W, 2 * F);
    RC(add_conv(p, L + "_trunk0", x, t0w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, t0));
    Tensor r1 = new_act(B, x.H, x.W, F), c1 = new_act(B, x.H, x.W, F);
    RC(add_conv(p, L + "_reg1", chan_view(t0, 0, F), r1w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, r1));
    RC(add_conv(p, L + "_cls1", chan_view(t0, F, F), c1w, 3, 3, 1, 1, ACT_RELU, RES_NONE, nullptr, c1));
    Tensor score = new_act(B, x.H, x.W, 1), cmap = new_act(B, x.H, x.W, F);
    if (score_w) {   // bf16 mode: dedicated CUDA-core kernel (a 1-channel GEMM wastes the tensor-core tile)
      Act ia = r1.a, oa = score.a;
      const int hh = x.H, ww = x.W;
      const float *sw = score_w, *sb = score_b;
      Op o = ew_op(L + "_score", [=](cudaStream_t s) { return launch_conv3x3_c1(ia, sw, sb, B, hh, ww, oa, s); },
                   (double)r1.pixels() * F * 2 + (double)score.pixels() * 2);
      o.flops = 2.0 * (double)r1.pixels() * 9.0 * F;
      p.push_back(std::move(o));
    } else {
      RC(add_conv(p, L + "_score", r1, scw, 3, 3, 1, 1, ACT_NONE, RES_NONE, nullptr, score));
    }
    RC(add_conv(p, L + "_clsmap", c1, clw, 3, 3, 1, 1, ACT_NONE, RES_NONE, nullptr, cmap));
    Tensor co = new_act(B, x.H, x.W, F);
    {
      Act sa = score.a, ca = cmap.a, oa = co.a;
      const int HW = x.H * x.W;
      p.push_back(ew_op(L + "_coattention", [=](cudaStream_t s) { return launch_coattention(sa, ca, B, HW, oa, s); },
                        (double)co.pixels() * F * 4));
    }
    Tensor h4 = new_act(B, x.H, x.W, F);
    RC(add_conv(p, L + "_conv4", co, h4w, 3, 3, 1, 1, ACT_LEAKY, RES_NONE, nullptr, h4));
    Tensor hp;
    pool2(L + "_pool", h4, &hp);
    feat_[i] = new_act(B, hp.H, hp.W, D);
    RC(add_conv(p, L + "_conv5", hp, h5w, 3, 3, 1, 1, ACT_LEAKY, RES_NONE, nullptr, feat_[i]));
    taps_["feat" + std::to_string(i)] = feat_[i];
  }
  return 0;
}

// Multi-Transformer encoder (transformer.py:266-303).  Views after reordering [P3,P4,P5,P7 | P6]: the four
// static views feed K/V only, so their projections for all layers are hoisted into one GEMM per view.
int Engine::build_mt_encoder(Program& p) {
  const int B = cfg_.batch, D = cfg_.d_model, L = cfg_.num_layers, H = cfg_.num_heads, FF = cfg_.dff;
  const int order[5] = {0, 1, 2, 4, 3};   // transformer.py:253 with BASELINE_INDEX = 3
  // positional table (transformer.py:22-43), input_vocab_size = ceil(S/16)^2 (pipeline.py:20)
  const int npos = ((cfg_.image_size + 15) / 16) * ((cfg_.image_size + 15) / 16);
  std::vector<float> pos((size_t)npos * D);
  for (int ps = 0; ps < npos; ++ps)
    for (int i = 0; i < D; ++i) {
      const double rate = 1.0 / pow(10000.0, (double)(2 * (i / 2)) / (double)(float)D);
      const double ang = ps * rate;
      pos[(size_t)ps * D + i] = (float)((i % 2 == 0) ? sin(ang) : cos(ang));
    }
  float *d_pos, *g0, *b0;
  RC(upload_f32(pos, &d_pos));
  RC(prep_vec(std::string(TR) + "/encoder/layernorm1/gamma", &g0));
  RC(prep_vec(std::string(TR) + "/encoder/layernorm1/beta", &b0));
  Tensor tok[5];
  int ntok[5];
  for (int v = 0; v < 5; ++v) {
    const Tensor& f = feat_[order[v]];
    ntok[v] = f.H * f.W;
    tok[v] = rows_act(B * ntok[v], D);
    Act fa = f.a, ta = tok[v].a;
    const int hw = ntok[v];
    p.push_back(ew_op("tokens" + std::to_string(v) + "_ln_pos",
                      [=](cudaStream_t s) { return launch_tokens_ln_pos(fa, B, hw, g0, b0, 1e-6f, d_pos, ta, s); },
                      (double)B * hw * D * 4));
    taps_["tokens" + std::to_string(v)] = tok[v];
  }
  n_base_ = ntok[4];
  if (n_base_ > 16) return fail(FPNMT_ERR_INVALID, "baseline view has more than 16 tokens (image_size > 512 unsupported)");
  // hoisted K/V projections: per view one GEMM [B*n, 512] x [512, L*2*512]
  Tensor kv[4];
  for (int v = 0; v < 4; ++v) {
    std::vector<std::string> names;
    for (int l = 0; l < L; ++l) {
      const std::string m = std::string(TR) + "/encoder/enc_layers/" + std::to_string(l) + "/mhas/" + std::to_string(v);
      names.push_back(m + "/wk");
      names.push_back(m + "/wv");
    }
    GemmW g;
    RC(prep_dense_cat(names, &g));
    kv[v] = rows_act(B * ntok[v], L * 2 * D);
    RC(add_conv(p, "enc_kv_view" + std::to_string(v), tok[v], g, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, kv[v]));
  }
  Tensor base = tok[4];
  const int R = B * n_base_;
  for (int l = 0; l < L; ++l) {
    const std::string e = std::string(TR) + "/encoder/enc_layers/" + std::to_string(l);
    const std::string ln = "enc" + std::to_string(l);
    GemmW gq, go, g1, g2;
    RC(prep_dense_cat({e + "/mhas/0/wq", e + "/mhas/1/wq", e + "/mhas/2/wq", e + "/mhas/3/wq"}, &gq));
    RC(prep_dense_stack({e + "/mhas/0/dense", e + "/mhas/1/dense", e + "/mhas/2/dense", e + "/mhas/3/dense"}, &go));
    RC(prep_dense_cat({e + "/ffn1"}, &g1));
    RC(prep_dense_cat({e + "/ffn2"}, &g2));
    Tensor q = rows_act(R, 4 * D), att = rows_act(R, 4 * D);
    RC(add_conv(p, ln + "_q", base, gq, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, q));
    const bool force_simt = (cfg_.kernel_opts & FPNMT_OPT_ENC_ATT_SIMT) != 0;
    if (!split_ && !force_simt) {
      // bf16 mode: the four cross-level attentions of the layer as one launch (long view first)
      struct V4 { Act kv[4]; int tk[4]; int col[4]; } v4;
      double bytes = 0, flops = 0;
      for (int v = 0; v < 4; ++v) {
        v4.kv[v] = kv[v].a;
        v4.tk[v] = ntok[v];
        v4.col[v] = v * D;
        bytes += (double)B * ntok[v] * 2 * D * 2;
        flops += 4.0 * B * n_base_ * ntok[v] * D;
      }
      Act qa = q.a, oa = att.a;
      const int tq = n_base_, kc = l * 2 * D, vc = l * 2 * D + D;
      Op o = ew_op(ln + "_attn_views", [=](cudaStream_t s) { return launch_enc_attention_views(qa, v4.kv, v4.tk, v4.col, 4, kc, vc, B, tq, H, oa, s); },
                   bytes, "attention");
      o.flops = flops;
      p.push_back(std::move(o));
    } else {
    for (int v = 0; v < 4; ++v) {
      Act qa = q.a, ka = kv[v].a, oa = att.a;
      const int tk = ntok[v], tq = n_base_, kc = l * 2 * D, vc = l * 2 * D + D, qc = v * D;
      Op o = ew_op(ln + "_attn_view" + std::to_string(v),
                   [=](cudaStream_t s) { return launch_enc_attention(qa, qc, ka, kc, vc, B, tq, tk, H, oa, qc, force_simt, s); },
                   (double)B * tk * 2 * D * 2, "attention");
      o.flops = 4.0 * B * tq * tk * D;
      p.push_back(std::move(o));
    }
    }
    Tensor none;
    float *g1p, *b1p, *g2p, *b2p;
    RC(prep_vec(e + "/layernorm1/gamma", &g1p));
    RC(prep_vec(e + "/layernorm1/beta", &b1p));
    RC(prep_vec(e + "/layernorm2/gamma", &g2p));
    RC(prep_vec(e + "/layernorm2/beta", &b2p));
    Tensor out1 = rows_act(R, D), hdn = rows_act(R, FF), out2 = rows_act(R, D);
    if (use_tgemm_) {
      // skinny-row tgemm (R = 16 B rows): residual + LayerNorm fused into the epilogue, as in the decoder step
      RC(add_dense(p, ln + "_out+res+ln", att, go, ACT_NONE, &base, out1, nullptr, 0, g1p, b1p));
      RC(add_dense(p, ln + "_ffn1", out1, g1, ACT_LEAKY, nullptr, hdn));
      RC(add_dense(p, ln + "_ffn2+res+ln", hdn, g2, ACT_NONE, &out1, out2, nullptr, 0, g2p, b2p));
    } else {
      float* y = (float*)dalloc((size_t)R * D * 4);
      RC(add_conv(p, ln + "_out+res", att, go, 1, 1, 0, 0, ACT_NONE, RES_SAME, &base, none, y, D));
      {
        Act oa = out1.a;
        p.push_back(ew_op(ln + "_ln1", [=](cudaStream_t s) { return launch_layernorm_rows(y, R, D, g1p, b1p, 1e-6f, oa, s); }, (double)R * D * 6));
      }
      RC(add_conv(p, ln + "_ffn1", out1, g1, 1, 1, 0, 0, ACT_LEAKY, RES_NONE, nullptr, hdn));
      float* y2 = (float*)dalloc((size_t)R * D * 4);
      RC(add_conv(p, ln + "_ffn2+res", hdn, g2, 1, 1, 0, 0, ACT_NONE, RES_SAME, &out1, none, y2, D));
      {
        Act oa = out2.a;
        p.push_back(ew_op(ln + "_ln2", [=](cudaStream_t s) { return launch_layernorm_rows(y2, R, D, g2p, b2p, 1e-6f, oa, s); }, (double)R * D * 6));
      }
    }
    base = out2;
    taps_["enc_layer" + std::to_string(l)] = out2;
  }
  enc_out_ = base;
  taps_["memory"] = base;
  return 0;
}

__global__ void k_anc_identity(int* anc, int rows, int T);

// KV-cached decoder step programs (transformer.py:224-243, 321-341, 372) + decode tail (pipeline.py:115-148)
int Engine::build_decoder() {
  const int B = cfg_.batch, N = cfg_.beam, D = cfg_.d_model, L = cfg_.num_layers, H = cfg_.num_heads, FF = cfg_.dff;
  const int V = cfg_.vocab, T = cfg_.max_len;
  const int R = B * N;
  // beam state
  bs_.B = B; bs_.N = N; bs_.V = V; bs_.T = T;
  bs_.start_id = cfg_.start_id; bs_.end_id = cfg_.end_id;
  bs_.prob_mode = cfg_.score_mode == FPNMT_SCORE_PROB;
  for (int i = 0; i < 2; ++i) {
    bs_.score[i] = (float*)dalloc((size_t)R * 4);
    bs_.seq[i] = (int*)dalloc((size_t)R * (T + 1) * 4);
    bs_.anc[i] = nullptr;
  }
  int* anc = (int*)dalloc((size_t)2 * R * T * 4);   // [2][R][T] contiguous (the attention kernel indexes by step&1)
  bs_.anc[0] = anc;
  bs_.anc[1] = anc + (size_t)R * T;
  bs_.last_tok = (int*)dalloc((size_t)R * 4);
  {
    int* rep = (cfg_.kernel_opts & FPNMT_OPT_NO_KV_SHARE) ? nullptr : (int*)dalloc((size_t)2 * R * 4);
    bs_.rep[0] = rep;
    bs_.rep[1] = rep ? rep + R : nullptr;
  }
  bs_.step = (int*)dalloc(16);
  bs_.done = (int*)dalloc((size_t)B * 4);
  bs_.n_done = (int*)dalloc(16);
  bs_.img_count = (int*)dalloc((size_t)B * 4);
  FPNMT_CUDA_OK(cudaMemset(bs_.img_count, 0, (size_t)B * 4));
  bs_.finished_mode = cfg_.finished_beams ? 1 : 0;
  if (bs_.finished_mode) {   // extension: frozen finished beams + length penalty lp[len] = ((5 + len) / 6)^alpha
    bs_.fin_len[0] = (int*)dalloc((size_t)R * 4);
    bs_.fin_len[1] = (int*)dalloc((size_t)R * 4);
    std::vector<float> lp(T + 2);
    for (int i = 0; i < T + 2; ++i) lp[i] = powf((5.f + (float)i) / 6.f, cfg_.length_penalty);
    float* dlp;
    RC(upload_f32(lp, &dlp));
    bs_.lp = dlp;
    if (!bs_.fin_len[0] || !bs_.fin_len[1]) return FPNMT_ERR_CUDA;
    FPNMT_CUDA_OK(cudaMemset(bs_.fin_len[0], 0, (size_t)R * 4));
    FPNMT_CUDA_OK(cudaMemset(bs_.fin_len[1], 0, (size_t)R * 4));
  } else if (cfg_.length_penalty != 0.f) {
    return fail(FPNMT_ERR_INVALID, "length_penalty needs finished_beams = 1 (it only orders beams of different lengths)");
  }
  bs_.out_ids = (int*)dalloc((size_t)B * T * 4);
  bs_.out_len = (int*)dalloc((size_t)B * 4);
  bs_.cand_val = (float*)dalloc((size_t)R * N * 4);
  bs_.cand_idx = (int*)dalloc((size_t)R * N * 4);
  step_scores_ = (float*)dalloc((size_t)T * B * 4);
  bs_.step_logprob = step_scores_;
  bs_.parent_out = (int*)dalloc((size_t)T * R * 4);
  bs_.token_out = (int*)dalloc((size_t)T * R * 4);
  logits_ = (float*)dalloc((size_t)R * V * 4);
  forced_tokens_ = (int*)dalloc((size_t)B * T * 4);
  forced_logits_ = nullptr;
  if (!logits_ || !forced_tokens_) return FPNMT_ERR_CUDA;
  FPNMT_CUDA_OK(cudaMemset(anc, 0, (size_t)2 * R * T * 4));

  // decoder positional table (transformer.py:315)
  std::vector<float> pos((size_t)T * D);
  for (int ps = 0; ps < T; ++ps)
    for (int i = 0; i < D; ++i) {
      const double rate = 1.0 / pow(10000.0, (double)(2 * (i / 2)) / (double)(float)D);
      pos[(size_t)ps * D + i] = (float)((i % 2 == 0) ? sin(ps * rate) : cos(ps * rate));
    }
  float *d_pos, *d_emb;
  RC(upload_f32(pos, &d_pos));
  RC(prep_vec(std::string(TR) + "/decoder/embedding/embeddings", &d_emb));
  dec_emb_ = d_emb;
  dec_pos_ = d_pos;

  // cross-attention K/V of the memory for all layers: one GEMM [B*16,512] x [512, L*2*512] per batch
  {
    std::vector<std::string> names;
    for (int l = 0; l < L; ++l) {
      const std::string m = std::string(TR) + "/decoder/dec_layers/" + std::to_string(l) + "/mha2";
      names.push_back(m + "/wk");
      names.push_back(m + "/wv");
    }
    GemmW g;
    RC(prep_dense_cat(names, &g));
    Tensor ckv = rows_act(B * n_base_, L * 2 * D);
    RC(add_conv(dec_init_prog_, "dec_cross_kv", enc_out_, g, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, ckv));
    taps_["cross_kv"] = ckv;
    dec_ckv_ = ckv;

    // Group-stationary fused decoder (dstep.cuh): one kernel per decode instead of 38 per step.  Needs the bf16 mode,
    // log-domain scores and the reference beam semantics; everything else takes the per-operator chain below.
    {
      const int vslice = ((V + DS_CTAS - 1) / DS_CTAS + 127) / 128 * 128;
      const bool want = cfg_.decode_path == FPNMT_DECODE_FUSED;
      use_dstep_ = want && !split_ && cfg_.score_mode == FPNMT_SCORE_LOG && N <= 16 && D == 512 &&
                   H == 8 && FF == 2048 && vslice / 128 <= DS_MAX_VTILES && n_base_ <= 16 && cfg_.cache_mode == FPNMT_CACHE_ANCESTRY &&
                   !cfg_.finished_beams && cfg_.length_penalty == 0.f;
      if (want && !use_dstep_)
        return fail(FPNMT_ERR_INVALID, "decode_path FUSED needs precision bf16, score_mode log, beam <= 16, dff 2048, vocab <= 14336, "
                                       "cache_mode ancestry and the reference beam semantics");
      if (use_dstep_) return build_dstep(ckv, d_emb, d_pos);
    }

    // Fused cross-attention block (bf16 mode): per-image folded operands, recomputed once per batch (xattn.cuh)
    const bool xattn = use_xattn_ && use_tgemm_ && !split_ && N <= XA_NROWS && n_base_ <= 16 && D == 512 && H == 8;
    bf16 *xMt = nullptr, *xNt = nullptr;
    float* xSb = nullptr;
    if (xattn) {
      xMt = (bf16*)dalloc((size_t)L * B * 128 * 512 * 2);
      xNt = (bf16*)dalloc((size_t)L * B * 512 * 128 * 2);
      xSb = (float*)dalloc((size_t)L * B * 128 * 4);
      if (!xMt || !xNt || !xSb) return FPNMT_ERR_CUDA;
      // bf16 copies of the projection weights for the mma.sync fold kernels: Wq as stored [k][(h,d)], Wo transposed [f][(h,d)]
      std::vector<uint16_t> hwq((size_t)L * 512 * 512), hwo((size_t)L * 512 * 512);
      std::vector<const float*> hb(L);
      for (int l = 0; l < L; ++l) {
        const std::string m = std::string(TR) + "/decoder/dec_layers/" + std::to_string(l) + "/mha2";
        const HostW *kq = W(m + "/wq/kernel"), *ko = W(m + "/dense/kernel");
        if (!kq || !ko) return FPNMT_ERR_MISSING;
        if (kq->data.size() != 512 * 512 || ko->data.size() != 512 * 512) return fail(FPNMT_ERR_INVALID, m + ": projection kernels must be 512x512");
        xattn_fold_weights(kq->data.data(), ko->data.data(), &hwq[(size_t)l * 512 * 512], &hwo[(size_t)l * 512 * 512]);
        float* b2;
        RC(prep_vec(m + "/wq/bias", &b2));
        hb[l] = b2;
      }
      bf16* dq = (bf16*)dalloc(hwq.size() * 2);
      bf16* d_o = (bf16*)dalloc(hwo.size() * 2);
      const float** db = (const float**)dalloc(L * sizeof(float*));
      if (!dq || !d_o || !db) return FPNMT_ERR_CUDA;
      FPNMT_CUDA_OK(cudaMemcpy(dq, hwq.data(), hwq.size() * 2, cudaMemcpyHostToDevice));
      FPNMT_CUDA_OK(cudaMemcpy(d_o, hwo.data(), hwo.size() * 2, cudaMemcpyHostToDevice));
      FPNMT_CUDA_OK(cudaMemcpy(db, hb.data(), L * sizeof(float*), cudaMemcpyHostToDevice));
      Act ca = ckv.a;
      const int nm = n_base_;
      Op o = ew_op("xattn_fold", [=](cudaStream_t s) { return launch_xattn_fold(ca, B, nm, L, dq, db, d_o, xMt, xNt, xSb, s); },
                   (double)L * B * 2 * 128 * 512 * 2, "elementwise");
      o.flops = 2.0 * 2.0 * L * B * 128.0 * 512.0 * 64.0;
      dec_init_prog_.push_back(std::move(o));
    }

    // ---- per-layer weights and buffers
    const bool physical = cfg_.cache_mode == FPNMT_CACHE_PHYSICAL;
    bs_.physical = physical ? 1 : 0;
    if (physical) {   // the ancestry tables stay the identity in this mode
      k_anc_identity<<<148, 256>>>(anc, R, T);
      FPNMT_CUDA_OK(cudaGetLastError());
    }
    struct LayerW : DecLayerW {
      Tensor qkv, att, out1, q2, att2, out2, hdn, out3, kc, vc, kc2, vc2;
      float* y;
    };
    std::vector<LayerW> lw(L);
    for (int l = 0; l < L; ++l) {
      const std::string d = std::string(TR) + "/decoder/dec_layers/" + std::to_string(l);
      LayerW& w = lw[l];
      RC(prep_dense_cat({d + "/mha1/wq", d + "/mha1/wk", d + "/mha1/wv"}, &w.gqkv));
      RC(prep_dense_cat({d + "/mha1/dense"}, &w.go1));
      RC(prep_dense_cat({d + "/mha2/wq"}, &w.gq2));
      RC(prep_dense_cat({d + "/mha2/dense"}, &w.go2));
      RC(prep_dense_cat({d + "/ffn1"}, &w.g1));
      RC(prep_dense_cat({d + "/ffn2"}, &w.g2));
      const char* lnn[6] = {"/layernorm1/gamma", "/layernorm1/beta", "/layernorm2/gamma", "/layernorm2/beta", "/layernorm3/gamma", "/layernorm3/beta"};
      for (int i = 0; i < 6; ++i) RC(prep_vec(d + lnn[i], &w.lnp[i]));
      w.qkv = rows_act(R, 3 * D); w.att = rows_act(R, D); w.out1 = rows_act(R, D); w.q2 = rows_act(R, D);
      w.att2 = rows_act(R, D); w.out2 = rows_act(R, D); w.hdn = rows_act(R, FF); w.out3 = rows_act(R, D);
      w.kc = rows_act(R * T, D); w.vc = rows_act(R * T, D);
      if (physical) {   // second buffer pair: every step's reorder gathers from one pair into the other
        w.kc2 = rows_act(R * T, D);
        w.vc2 = rows_act(R * T, D);
        if (!w.kc2.a.p || !w.vc2.a.p) return FPNMT_ERR_CUDA;
      }
      w.y = (float*)dalloc((size_t)R * D * 4);
    }
    GemmW gf;
    RC(prep_dense_cat({std::string(TR) + "/final_layer"}, &gf));
    dec_lw_.assign(lw.begin(), lw.end());
    dec_final_ = gf;
    Tensor x = rows_act(R, D);
    Tensor none;
    bs_.dbg = dbg_timeline("beam_step");

    // ---- the step-0 embedding program and the program of one step
    {   // step 0 input (embedding of <start> + pos[0]); later steps' inputs are written by the beam kernel
      Act xa = x.a;
      const int* tok = bs_.last_tok;
      const int* step = bs_.step;
      embed_prog_.push_back(ew_op("embed_pos", [=](cudaStream_t s) { return launch_embed_pos(tok, d_emb, d_pos, step, R, D, xa, s); }, (double)R * D * 6));
    }
    const BeamEmbed em{d_emb, d_pos, x.a, D};
    beam_embed_ = em;
    // attention-probability launches of step_attn_prog_: position in step_prog_ they follow, the op
    std::vector<std::pair<size_t, Op>> prob_ops;
    for (int l = 0; l < L; ++l) {
      LayerW& w = lw[l];
      const std::string ln = "dec" + std::to_string(l);
      // Dense layers of the step: skinny-row tgemm (weights prefetched before the grid dependency, LayerNorm fused
      // into the epilogue by a 4-CTA cluster) or, with FPNMT_TGEMM=0, the generic igemm + separate LayerNorm kernels.
      auto dense = [&](const std::string& nm, const Tensor& in, const GemmW& g, int act, const Tensor& out) -> int {
        if (use_tgemm_) return add_dense(step_prog_, nm, in, g, act, nullptr, out);
        return add_conv(step_prog_, nm, in, g, 1, 1, 0, 0, act, RES_NONE, nullptr, out);
      };
      auto dense_res_ln = [&](const std::string& nm, const std::string& lnn2, const Tensor& in, const GemmW& g, const Tensor& res,
                              float* gam, float* bet, const Tensor& out) -> int {
        if (use_tgemm_) return add_dense(step_prog_, nm + "+ln", in, g, ACT_NONE, &res, out, nullptr, 0, gam, bet);
        float* y = w.y;
        RC(add_conv(step_prog_, nm, in, g, 1, 1, 0, 0, ACT_NONE, RES_SAME, &res, none, y, D));
        Act oa = out.a;
        step_prog_.push_back(ew_op(lnn2, [=](cudaStream_t s) { return launch_layernorm_rows(y, R, D, gam, bet, 1e-6f, oa, s); }, (double)R * D * 6));
        return 0;
      };
      RC(dense(ln + "_qkv", x, w.gqkv, ACT_NONE, w.qkv));
      {
        Act qa = w.qkv.a, ka = w.kc.a, va = w.vc.a, oa = w.att.a, ka2 = w.kc2.a, va2 = w.vc2.a;
        const size_t anc_stride = (size_t)R * T;
        const int* step = bs_.step;
        const int *rep_e = bs_.rep[0], *rep_o = bs_.rep[1];
        Op o = ew_op(ln + "_self_attn",
                     [=](cudaStream_t s) {
                       // teacher forcing (decode_logits) has no beam step and therefore no reorder: it stays in the first buffer pair
                       const Act none{nullptr, 0, 0, 0};
                       return launch_dec_self_attention(qa, ka, va, forced_mode_ ? none : ka2, forced_mode_ ? none : va2, anc, anc_stride, step, R, T, H, oa, s,
                                                        forced_mode_ ? nullptr : rep_e, forced_mode_ ? nullptr : rep_o, N);
                     },
                     (double)R * (T / 2) * 2 * D * 2, "attention");
        step_prog_.push_back(std::move(o));
      }
      RC(dense_res_ln(ln + "_o1+res", ln + "_ln1", w.att, w.go1, x, w.lnp[0], w.lnp[1], w.out1));
      size_t prob_at = 0;   // the probabilities read the new K of position t, q2 / out1: after the cross-attention block
      if (xattn) {
        XattnOp xo;
        RC(make_xattn_op(&xo, xMt, xNt, L, B, 0, B, N, l, xSb, w.go2.bias, w.lnp[2], w.lnp[3], w.out1.a, w.out2.a));
        xo.p.dbg = dbg_timeline(ln + "_xattn");
        Op o;
        o.name = ln + "_xattn(q2+cross_attn+o2+res+ln)";
        o.kind = "xattn";
        o.flops = 2.0 * R * D * D * 2.0 + 4.0 * R * n_base_ * D;          // the two projections + the attention proper
        o.bytes = (double)B * 2 * 128 * 512 * 2 + (double)R * D * 2 * 2;  // folded per-image operands + activations
        o.run = [xo](cudaStream_t s) { return xattn_launch(xo, s); };
        step_prog_.push_back(std::move(o));
        prob_at = step_prog_.size();
      } else {
        RC(dense(ln + "_q2", w.out1, w.gq2, ACT_NONE, w.q2));
        {
          Act qa = w.q2.a, oa = w.att2.a, ka = ckv.a;
          const int kcx = l * 2 * D, vcx = l * 2 * D + D, tk = n_base_;
          step_prog_.push_back(ew_op(ln + "_cross_attn", [=](cudaStream_t s) { return launch_dec_cross_attention(qa, ka, kcx, vcx, R, N, tk, H, oa, s); },
                                     (double)B * tk * 2 * D * 2, "attention"));
          prob_at = step_prog_.size();
        }
        RC(dense_res_ln(ln + "_o2+res", ln + "_ln2", w.att2, w.go2, w.out1, w.lnp[2], w.lnp[3], w.out2));
      }
      {
        DecProbArgs pa{};
        pa.qkv = w.qkv.a;
        pa.kc = w.kc.a;
        pa.anc = anc;
        pa.anc_stride = (size_t)R * T;
        pa.T = T;
        pa.q = xattn ? w.out1.a : w.q2.a;
        pa.kv = ckv.a;
        pa.k_col = l * 2 * D;
        pa.Mt = xattn ? xMt + (size_t)l * B * 128 * 512 : nullptr;
        pa.sbias = xattn ? xSb + (size_t)l * B * 128 : nullptr;
        pa.n_mem = n_base_;
        pa.step = bs_.step;
        pa.N = N;
        pa.heads = H;
        const int nm = n_base_;
        // output pointers and row count are those of the decode_logits call that runs the program
        Op o = ew_op(ln + "_attn_probs",
                     [=](cudaStream_t s) {
                       DecProbArgs q = pa;
                       const size_t tl = (size_t)attn_tlen_;
                       q.tlen = attn_tlen_;
                       q.self_out = attn_self_ ? attn_self_ + (size_t)l * B * H * tl * tl : nullptr;
                       q.cross_out = attn_cross_ ? attn_cross_ + (size_t)l * B * H * tl * nm : nullptr;
                       return launch_dec_attention_probs(q, B, s);
                     },
                     (double)B * H * (T / 2 + nm) * D * 2, "attention");
        prob_ops.emplace_back(prob_at, std::move(o));
      }
      RC(dense(ln + "_ffn1", w.out2, w.g1, ACT_LEAKY, w.hdn));
      RC(dense_res_ln(ln + "_ffn2+res", ln + "_ln3", w.hdn, w.g2, w.out2, w.lnp[4], w.lnp[5], w.out3));
      // per-layer decoder states of the last executed step (parity taps, same names in the fused decoder)
      taps_[ln + "_out1"] = w.out1;
      taps_[ln + "_out2"] = w.out2;
      taps_[ln + "_out3"] = w.out3;
      x = w.out3;
    }
    float* lg = logits_;
    if (use_tgemm_) RC(add_dense(step_prog_, "final_layer", x, gf, ACT_NONE, nullptr, none, lg, V));
    else RC(add_conv(step_prog_, "final_layer", x, gf, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, none, lg, V));
    // teacher forcing: embed the forced token, then the shared layer stack
    step_forced_prog_ = embed_prog_;
    step_forced_prog_.insert(step_forced_prog_.end(), step_prog_.begin(), step_prog_.end());
    step_attn_prog_ = embed_prog_;   // the same launches with the probability kernels after the operands they read
    size_t k = 0;
    for (size_t i = 0; i < step_prog_.size(); ++i) {
      step_attn_prog_.push_back(step_prog_[i]);
      for (; k < prob_ops.size() && prob_ops[k].first == i + 1; ++k) step_attn_prog_.push_back(prob_ops[k].second);
    }
    // Logits-free decode tail (bf16 mode, log scores, beam <= 8, wide Dense kernels): the beam-search chain replaces the
    // vocabulary projection's [rows][V] fp32 output (20.5 MB written and read back per step at C2) by per-tile softmax
    // partials + 8 candidates (2.9 MB); teacher forcing (decode_logits) keeps the logits version built above.
    const int vtiles = (V + TG_BM - 1) / TG_BM;
    const bool want_wide = (cfg_.kernel_opts & FPNMT_OPT_TGEMM_WIDE) || (cfg_.lanes >= 2 && !(cfg_.kernel_opts & FPNMT_OPT_NO_TGEMM_WIDE));
    const bool vstats = use_tgemm_ && want_wide && !split_ && !bs_.prob_mode && N <= TG_VS_N && vtiles <= 192 &&
                        !(cfg_.kernel_opts & FPNMT_OPT_NO_VSTATS);
    BeamState bsv = bs_;
    if (vstats) {
      float2* vst = (float2*)dalloc((size_t)R * vtiles * sizeof(float2));
      float* vval = (float*)dalloc((size_t)R * vtiles * TG_VS_N * sizeof(float));
      int* vidx = (int*)dalloc((size_t)R * vtiles * TG_VS_N * sizeof(int));
      if (!vst || !vval || !vidx) return FPNMT_ERR_CUDA;
      TgemmOp op;
      RC(make_tgemmw_op(&op, R, x.a, gf.w, gf.Cout, gf.K, gf.bias, ACT_NONE, none.a, nullptr, 0, nullptr, nullptr, nullptr, 1e-6f,
                        num_sms_, vst, vval, vidx));
      op.p.dbg = dbg_timeline("final_layer");
      Op o;
      o.name = "final_layer(softmax partials + candidates)";
      o.kind = "tgemm";
      o.flops = op.flops;
      o.bytes = (double)R * gf.K * 2 + (double)gf.Cout * gf.K * 2 + (double)R * vtiles * (8 + 8 * TG_VS_N);
      o.run = [op](cudaStream_t s) { return tgemm_launch(op, s); };
      step_prog_.back() = std::move(o);                      // replaces the logits version in the beam-search chain
      step_final_at_ = step_prog_.size() - 1;
      vs_final_op_ = op;
      bsv.vs_stat = vst;
      bsv.vs_val = vval;
      bsv.vs_idx = vidx;
      bsv.vs_tiles = vtiles;
    }
    {
      Op o = ew_op("beam_step", [=](cudaStream_t s) { return launch_beam_step(bsv, lg, V, em, s); },
                   vstats ? (double)R * vtiles * (8 + 8 * TG_VS_N) + (double)R * (T + 1) * 8
                          : (double)R * V * 4 + (double)R * (T + 1) * 8, "beam");
      o.idempotent = false;
      step_prog_.push_back(std::move(o));
    }
    step_beam_at_ = step_prog_.size() - 1;
    step_bsv_ = bsv;
    if (physical) {
      // KV-cache reorder by beam parent, all layers and K / V in one bandwidth-bound launch (north-star item 3)
      std::vector<const bf16*> hp(2 * 2 * L);
      for (int l = 0; l < L; ++l) {
        hp[2 * l] = lw[l].kc.a.p;
        hp[2 * l + 1] = lw[l].vc.a.p;
        hp[2 * L + 2 * l] = lw[l].kc2.a.p;
        hp[2 * L + 2 * l + 1] = lw[l].vc2.a.p;
      }
      const bf16** dp = (const bf16**)dalloc(hp.size() * sizeof(bf16*));
      if (!dp) return FPNMT_ERR_CUDA;
      FPNMT_CUDA_OK(cudaMemcpy(dp, hp.data(), hp.size() * sizeof(bf16*), cudaMemcpyHostToDevice));
      const int row_bytes = lw[0].kc.a.ld * 2;
      const int* par = bs_.parent_out;
      const int* step = bs_.step;
      Op o = ew_op("kv_reorder_physical", [=](cudaStream_t s) { return launch_kv_reorder(dp, 2 * L, par, R, R, N, T, row_bytes, step, s); },
                   2.0 * 2 * L * (double)R * (T / 2 + 1) * row_bytes, "kvreorder");
      o.idempotent = false;
      step_prog_.push_back(std::move(o));
    }
  }
  return 0;
}

// --------------------------------------------------------------------------------------------- fused decoder (dstep.cuh)
// Appends one [rows x 64] bf16 tile (row r = 128 contiguous bytes) to the weight stream; the kernel pulls 128-row boxes of
// the stream with TMA (SWIZZLE_128B), so consecutive tiles form the exact consumption order of one CTA.
template <typename F>
static void ds_pack_chunk(std::vector<uint16_t>& out, int rows, F get) {
  const size_t base = out.size();
  out.resize(base + (size_t)rows * 64);
  for (int r = 0; r < rows; ++r)
    for (int kk = 0; kk < 64; ++kk) out[base + (size_t)r * 64 + kk] = f2bf(get(r, kk));
}

int Engine::build_dstep(const Tensor& ckv, const float* d_emb, const float* d_pos) {
  const int B = cfg_.batch, N = cfg_.beam, L = cfg_.num_layers, V = cfg_.vocab, T = cfg_.max_len;
  const int R = B * N;
  DstepParams& p = dsp_;
  p = DstepParams{};
  p.B = B; p.N = N; p.R = R;
  p.ipc = DS_ROWS / N;
  p.L = L; p.T = T; p.V = V;
  p.vslice = ((V + DS_CTAS - 1) / DS_CTAS + 127) / 128 * 128;
  p.ntv = p.vslice / 128;
  p.n_mem = n_base_;
  const int clusters = (B + p.ipc - 1) / p.ipc;
  // ---- weight streams
  std::vector<uint16_t> ws;
  ws.reserve(((size_t)L * DS_CTAS * DS_LAYER_STREAM + (size_t)DS_CTAS * p.ntv * 8 * 16384) / 2);
  std::vector<float> lp((size_t)L * DSB_SIZE);
  auto dense_w = [&](const std::string& name, int K, int F) -> const HostW* {
    const HostW* k = W(name + "/kernel");
    if (k && (k->shape.size() != 2 || k->shape[0] != K || k->shape[1] != F)) {
      set_last_error(name + "/kernel: expected shape (" + std::to_string(K) + ", " + std::to_string(F) + ")");
      return nullptr;
    }
    return k;
  };
  auto copy_vec = [&](const std::string& key, float* dst, int n) -> int {
    const HostW* v = W(key);
    if (!v) return FPNMT_ERR_MISSING;
    if ((int)v->data.size() != n) return fail(FPNMT_ERR_INVALID, key + ": expected " + std::to_string(n) + " elements");
    std::copy(v->data.begin(), v->data.end(), dst);
    return 0;
  };
  for (int l = 0; l < L; ++l) {
    const std::string d = std::string(TR) + "/decoder/dec_layers/" + std::to_string(l);
    const HostW *wq = dense_w(d + "/mha1/wq", 512, 512), *wk = dense_w(d + "/mha1/wk", 512, 512), *wv = dense_w(d + "/mha1/wv", 512, 512),
                *wo1 = dense_w(d + "/mha1/dense", 512, 512), *wq2 = dense_w(d + "/mha2/wq", 512, 512),
                *wo2 = dense_w(d + "/mha2/dense", 512, 512), *w1 = dense_w(d + "/ffn1", 512, 2048), *w2 = dense_w(d + "/ffn2", 2048, 512);
    if (!wq || !wk || !wv || !wo1 || !wq2 || !wo2 || !w1 || !w2) return FPNMT_ERR_MISSING;
    for (int c = 0; c < DS_CTAS; ++c) {
      const size_t before = ws.size();
      for (int kc = 0; kc < 8; ++kc)
        ds_pack_chunk(ws, 128, [&](int r, int kk) {
          return r < 64 ? wq->data[(size_t)(kc * 64 + kk) * 512 + c * 64 + r] : wk->data[(size_t)(kc * 64 + kk) * 512 + c * 64 + r - 64];
        });
      for (const HostW* m : {wv, wo1, wq2, wo2})
        for (int kc = 0; kc < 8; ++kc)
          ds_pack_chunk(ws, 64, [&](int r, int kk) { return m->data[(size_t)(kc * 64 + kk) * 512 + c * 64 + r]; });
      for (int ft = 0; ft < 2; ++ft)
        for (int kc = 0; kc < 8; ++kc)
          ds_pack_chunk(ws, 128, [&](int r, int kk) { return w1->data[(size_t)(kc * 64 + kk) * 2048 + c * 256 + ft * 128 + r]; });
      for (int ft = 0; ft < 4; ++ft)
        for (int kc = 0; kc < 4; ++kc)
          ds_pack_chunk(ws, 128, [&](int r, int kk) { return w2->data[(size_t)(c * 256 + kc * 64 + kk) * 512 + ft * 128 + r]; });
      if ((ws.size() - before) * 2 != DS_LAYER_STREAM) return fail(FPNMT_ERR_INVALID, "build_dstep: layer stream size mismatch");
    }
    float* q = lp.data() + (size_t)l * DSB_SIZE;
    RC(copy_vec(d + "/mha1/wq/bias", q + DSB_Q, 512));
    RC(copy_vec(d + "/mha1/wk/bias", q + DSB_K, 512));
    RC(copy_vec(d + "/mha1/wv/bias", q + DSB_V, 512));
    RC(copy_vec(d + "/mha1/dense/bias", q + DSB_O1, 512));
    RC(copy_vec(d + "/mha2/wq/bias", q + DSB_Q2, 512));
    RC(copy_vec(d + "/mha2/dense/bias", q + DSB_O2, 512));
    RC(copy_vec(d + "/ffn1/bias", q + DSB_F1, 2048));
    RC(copy_vec(d + "/ffn2/bias", q + DSB_F2, 512));
    RC(copy_vec(d + "/layernorm1/gamma", q + DSB_LN1G, 512));
    RC(copy_vec(d + "/layernorm1/beta", q + DSB_LN1B, 512));
    RC(copy_vec(d + "/layernorm2/gamma", q + DSB_LN2G, 512));
    RC(copy_vec(d + "/layernorm2/beta", q + DSB_LN2B, 512));
    RC(copy_vec(d + "/layernorm3/gamma", q + DSB_LN3G, 512));
    RC(copy_vec(d + "/layernorm3/beta", q + DSB_LN3B, 512));
  }
  p.final_off = ws.size() * 2;
  {
    const HostW* wf = dense_w(std::string(TR) + "/final_layer", 512, V);
    const HostW* bf = W(std::string(TR) + "/final_layer/bias");
    if (!wf || !bf) return FPNMT_ERR_MISSING;
    if ((int)bf->data.size() != V) return fail(FPNMT_ERR_INVALID, "final_layer/bias: expected vocab elements");
    for (int c = 0; c < DS_CTAS; ++c)
      for (int vt = 0; vt < p.ntv; ++vt)
        for (int kc = 0; kc < 8; ++kc)
          ds_pack_chunk(ws, 128, [&](int r, int kk) {
            const int f = c * p.vslice + vt * 128 + r;
            return f < V ? wf->data[(size_t)(kc * 64 + kk) * V + f] : 0.f;
          });
    std::vector<float> vb((size_t)DS_CTAS * p.vslice, 0.f);
    std::copy(bf->data.begin(), bf->data.end(), vb.begin());
    float* dvb;
    RC(upload_f32(vb, &dvb));
    p.vbias = dvb;
  }
  uint8_t* dws = (uint8_t*)dalloc(ws.size() * 2);
  if (!dws) return FPNMT_ERR_CUDA;
  FPNMT_CUDA_OK(cudaMemcpy(dws, ws.data(), ws.size() * 2, cudaMemcpyHostToDevice));
  p.wstream = dws;
  p.stream_bytes = ws.size() * 2;
  float* dlp;
  RC(upload_f32(lp, &dlp));
  p.lparams = dlp;
  p.emb = d_emb;
  p.pos = d_pos;
  {
    const HostW* e = W(std::string(TR) + "/decoder/embedding/embeddings");
    if (!e || e->shape.size() != 2 || e->shape[0] < V || e->shape[1] != 512)
      return fail(FPNMT_ERR_INVALID, "decoder/embedding/embeddings: expected shape (>= vocab, 512)");
  }
  // ---- caches, exchange buffers
  const size_t cache_elems = (size_t)L * R * T * 512;
  p.kcache = (bf16*)dalloc(cache_elems * 2);
  p.vcache = (bf16*)dalloc(cache_elems * 2);
  p.ckv = ckv.a.p;
  p.ckv_ld = ckv.a.ld;
  const size_t xr = (size_t)clusters * 32;
  p.x_att = (bf16*)dalloc(xr * 512 * 2);
  p.x_pre = (float*)dalloc(xr * 512 * 4);
  p.x_part = (float*)dalloc((size_t)clusters * DS_CTAS * 32 * 512 * 4);
  p.x_stat = (float*)dalloc(xr * DS_CTAS * 2 * 4);
  p.x_cval = (float*)dalloc(xr * DS_CTAS * N * 4);
  p.x_cidx = (int*)dalloc(xr * DS_CTAS * N * 4);
  p.gbar = (int*)dalloc((size_t)clusters * sizeof(int));
  p.rep = (int*)dalloc((size_t)2 * R * sizeof(int));
  p.ngroups = clusters;
  if (!p.gbar || !p.rep || !p.kcache || !p.vcache || !p.x_att || !p.x_pre || !p.x_part || !p.x_stat || !p.x_cval || !p.x_cidx) return FPNMT_ERR_CUDA;
  FPNMT_CUDA_OK(cudaMemset(p.x_att, 0, xr * 512 * 2));
  FPNMT_CUDA_OK(cudaMemset(p.x_pre, 0, xr * 512 * 4));
  p.logits_out = logits_;
  p.ld_logits = V;
  if (cfg_.kernel_opts & FPNMT_OPT_DSTEP_TAPS) {   // LayerNorm outputs of every layer (last executed step), for the parity tests
    float* dbg = (float*)dalloc((size_t)L * 3 * xr * 512 * 4);
    if (!dbg) return FPNMT_ERR_CUDA;
    FPNMT_CUDA_OK(cudaMemset(dbg, 0, (size_t)L * 3 * xr * 512 * 4));
    p.dbg = dbg;
    for (int l = 0; l < L; ++l)
      for (int i = 0; i < 3; ++i)
        taps_f32_["dec" + std::to_string(l) + "_out" + std::to_string(i + 1)] = F32Tap{dbg + (size_t)(l * 3 + i) * xr * 512, xr * 512};
  }
  p.st = bs_;
  p.mode = 0;
  p.timeline = dbg_timeline("dstep");
  RC(dstep_set_attributes());
  // one-step op for the per-op profiler (the product decode is ONE launch of all steps)
  {
    Op o;
    o.name = "dstep(all layers + vocabulary projection + beam tail of one step)";
    o.kind = "dstep";
    o.flops = 2.0 * R * ((double)L * (512.0 * 1536 + 3.0 * 512 * 512 + 2.0 * 512 * 2048) + 512.0 * V);
    o.bytes = (double)ws.size() * 2 + (double)L * R * (T / 2) * 2 * 512 * 2;   // weight streams once + K/V cache at t = T/2
    o.idempotent = false;
    o.run = [this](cudaStream_t s) {
      DstepParams q = dsp_;
      q.t0 = prof_t_;
      q.nsteps = 1;
      if (prof_t_ + 1 < cfg_.max_len) ++prof_t_;
      return dstep_launch(q, s);
    };
    step_prog_.push_back(std::move(o));
  }
  return 0;
}

// --------------------------------------------------------------------------------------------- finalize / run
int Engine::finalize() {
  if (finalized_) return fail(FPNMT_ERR_STATE, "finalize_weights called twice");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  img_slot_ = (const float**)dalloc(16);
  if (!img_slot_) return FPNMT_ERR_CUDA;
  Tensor c[3];
  if (cfg_.backbone == FPNMT_BACKBONE_RESNET50) RC(build_resnet50(cnn_prog_, c));
  else if (cfg_.backbone == FPNMT_BACKBONE_MOBILENETV2) RC(build_mobilenetv2(cnn_prog_, c));
  else RC(build_densenet121(cnn_prog_, c));
  RC(build_fpn_heads(cnn_prog_, c));
  enc_prog_ = cnn_prog_;
  RC(build_mt_encoder(enc_prog_));
  RC(build_decoder());
  FPNMT_CUDA_OK(cudaDeviceSynchronize());
  hw_.clear();   // host staging no longer needed
  finalized_ = true;
  return 0;
}

int Engine::run_program(Program& p, cudaStream_t s) {
  for (auto& op : p) {
    int rc = op.run(s);
    if (rc) {
      set_last_error("op '" + op.name + "' failed: " + fpnmt_last_error());
      return rc;
    }
  }
  launches += (int64_t)p.size();
  return 0;
}

int Engine::capture(Program& p, cudaGraphExec_t* out) {
  cudaGraph_t g;
  FPNMT_CUDA_OK(cudaStreamBeginCapture(cap_stream_, cudaStreamCaptureModeThreadLocal));
  int rc = 0;
  for (auto& op : p) {
    rc = op.run(cap_stream_);
    if (rc) break;
  }
  cudaError_t e = cudaStreamEndCapture(cap_stream_, &g);
  if (rc) return rc;
  FPNMT_CUDA_OK(e);
  FPNMT_CUDA_OK(cudaGraphInstantiate(out, g, 0));
  FPNMT_CUDA_OK(cudaGraphDestroy(g));
  return 0;
}

int Engine::launch_prog(Program& p, cudaGraphExec_t g, cudaStream_t s) {
  if (g) {
    FPNMT_CUDA_OK(cudaGraphLaunch(g, s));
    launches += (int64_t)p.size();
    return 0;
  }
  return run_program(p, s);
}

int Engine::launch_graph(Program& p, cudaGraphExec_t& g, cudaStream_t s) {
  if (cfg_.use_graphs && !g) RC(capture(p, &g));
  return launch_prog(p, g, s);
}

int Engine::poll_done(const int* n_done, cudaStream_t s, bool* done) {
  FPNMT_CUDA_OK(cudaMemcpyAsync(h_pinned_, n_done, 4, cudaMemcpyDeviceToHost, s));
  FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  *done = h_pinned_[0] >= cfg_.batch;
  return 0;
}

// max_len replays of a step program; with early stop the host reads the finished-image counter every 4 steps and stops
// once every image has finished
int Engine::run_steps(Program& p, cudaGraphExec_t& g, const int* n_done, int early_stop, cudaStream_t s) {
  const int T = cfg_.max_len;
  for (int t = 0; t < T; ++t) {
    RC(launch_graph(p, g, s));
    if (early_stop && (t % 4 == 3) && t + 1 < T) {
      bool done = false;
      RC(poll_done(n_done, s, &done));
      if (done) break;
    }
  }
  return 0;
}

// the refusals shared by the decode modes that need the per-operator chain and the lane's own buffers
int Engine::check_decode_entry(const char* entry, const char* fused_reason) {
  const std::string e = entry;
  if (!finalized_) return fail(FPNMT_ERR_STATE, e + " before finalize_weights");
  if (use_dstep_) return fail(FPNMT_ERR_STATE, e + ": the fused decoder " + fused_reason + " (use decode_path = chain)");
  if (lane_state_ != 0) return fail(FPNMT_ERR_STATE, e + ": this lane still holds a submitted batch (call fpnmt_collect first)");
  return 0;
}

// result handoff: device src -> dst on the host (on_host) or the device; nothing for a NULL dst
static int copy_out(void* dst, const void* src, size_t bytes, int on_host, cudaStream_t s) {
  if (dst) FPNMT_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s));
  return 0;
}

// sets a flag for the guard's lifetime (forced_mode_ while a teacher-forced step program is enqueued or captured)
struct FlagGuard {
  bool& f;
  explicit FlagGuard(bool& flag) : f(flag) { f = true; }
  ~FlagGuard() { f = false; }
};

int Engine::set_images(const float* images, int on_host, cudaStream_t s) {
  const size_t n = (size_t)cfg_.batch * cfg_.image_size * cfg_.image_size * 3;
  const float* dptr = images;
  if (!on_host && stem_fused_ && (reinterpret_cast<uintptr_t>(images) & 15))
    return fail(FPNMT_ERR_INVALID, "device images must be 16-byte aligned");
  if (on_host) {
    if (!img_stage_) {
      img_stage_ = (float*)dalloc(n * 4);
      if (!img_stage_) return FPNMT_ERR_CUDA;
    }
    FPNMT_CUDA_OK(cudaMemcpyAsync(img_stage_, images, n * 4, cudaMemcpyHostToDevice, s));
    dptr = img_stage_;
  }
  FPNMT_CUDA_OK(cudaMemcpyAsync(img_slot_, &dptr, sizeof(dptr), cudaMemcpyHostToDevice, s));
  return 0;
}

int Engine::encode(const float* images, int on_host, float* memory_out, cudaStream_t s, bool cnn_only) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "encode before finalize_weights");
  if (!images) return fail(FPNMT_ERR_INVALID, "images is NULL");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  RC(set_images(images, on_host, s));
  if (cnn_only) RC(launch_graph(cnn_prog_, cnn_graph_, s));
  else RC(launch_graph(enc_prog_, enc_graph_, s));
  if (memory_out && !cnn_only) RC(launch_act_to_f32(enc_out_.a, enc_out_.pixels(), memory_out, s));
  return 0;
}

int Engine::features(const float* images, int on_host, float* const out5[5], cudaStream_t s) {
  RC(encode(images, on_host, nullptr, s, true));
  for (int i = 0; i < 5; ++i)
    if (out5[i]) RC(launch_act_to_f32(feat_[i].a, feat_[i].pixels(), out5[i], s));
  return 0;
}

int Engine::get_tap_f32(const std::string& name, float* out, size_t cap, size_t* count, cudaStream_t s) {
  const F32Tap& t = taps_f32_[name];
  if (count) *count = t.count;
  if (!out) return 0;
  if (cap < t.count) return fail(FPNMT_ERR_INVALID, "get_tap: buffer too small");
  FPNMT_CUDA_OK(cudaMemcpyAsync(out, t.p, t.count * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int Engine::get_tap(const char* name, float* out, size_t cap, size_t* count, cudaStream_t s) {
#ifdef FPNMT_DBG_STAMPS
  if (std::string(name) == "dstep_timeline" && use_dstep_ && dsp_.timeline) {   // stamps of the last launch's last step, ns since its start
    if (count) *count = 192;
    if (!out) return 0;
    if (cap < 192) return fail(FPNMT_ERR_INVALID, "get_tap: buffer too small");
    FPNMT_CUDA_OK(cudaStreamSynchronize(s));
    long long h[192];
    FPNMT_CUDA_OK(cudaMemcpy(h, dsp_.timeline, sizeof h, cudaMemcpyDeviceToHost));
    float f[192] = {0};
    f[0] = (float)h[0];
    for (int i = 0; i < (int)h[0] && i < 120; ++i) f[1 + i] = (float)(h[1 + i] - h[1]);
    for (int i = 150; i < 192; ++i) f[i] = h[i] ? (float)(h[i] - h[1]) : 0.f;     // MMA-warp stamps of one job
    FPNMT_CUDA_OK(cudaMemcpy(out, f, sizeof f, cudaMemcpyHostToDevice));
    return 0;
  }
#endif
  if (taps_f32_.count(name)) return get_tap_f32(name, out, cap, count, s);
  auto it = taps_.find(name);
  if (it == taps_.end()) return fail(FPNMT_ERR_INVALID, std::string("unknown tap: ") + name);
  const Tensor& t = it->second;
  const size_t n = t.pixels() * t.a.C;
  if (count) *count = n;
  if (!out) return 0;
  if (cap < n) return fail(FPNMT_ERR_INVALID, "get_tap: buffer too small");
  return launch_act_to_f32(t.a, t.pixels(), out, s);
}

// teacher-forced tail: copy beam-0 logits of every image to logits_out[b][t][:], feed the next forced token
__global__ void k_forced_tail(BeamState st, const float* __restrict__ logits, const int* __restrict__ forced, int tlen,
                              float* __restrict__ out) {
  const int t = *st.step;
  const int b = blockIdx.x;
  const float* src = logits + (size_t)(b * st.N) * st.V;
  float* dst = out + ((size_t)b * tlen + t) * st.V;
  if (out)
    for (int i = threadIdx.x; i < st.V; i += blockDim.x) dst[i] = src[i];
  if (threadIdx.x < st.N && t + 1 < tlen) st.last_tok[b * st.N + threadIdx.x] = forced[(size_t)b * tlen + t + 1];
}
__global__ void k_forced_init(BeamState st, const int* __restrict__ forced, int tlen) {
  const int rows = st.B * st.N;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *st.step = 0;
  if (i < rows) st.last_tok[i] = forced[(size_t)(i / st.N) * tlen];
  for (size_t j = i; j < (size_t)2 * rows * st.T; j += (size_t)gridDim.x * blockDim.x)
    st.anc[0][j] = (int)((j / st.T) % rows);   // identity ancestry in both buffers
}
// teacher-forced hidden states: beam-0 row of the last decoder layer's output -> hidden_out[b][t][:]
__global__ void k_forced_hidden(Act x, const int* __restrict__ step, int N, int tlen, float* __restrict__ out) {
  const int t = *step, b = blockIdx.x;
  const bf16* row = x.p + (size_t)(b * N) * x.ld;
  float* dst = out + ((size_t)b * tlen + t) * x.C;
  for (int i = threadIdx.x; i < x.C; i += blockDim.x) {
    float v = __bfloat162float(row[i]);
    if (x.lo) v += __bfloat162float(row[x.lo + i]);
    dst[i] = v;
  }
}
__global__ void k_step_inc(int* step) { *step += 1; }
__global__ void k_anc_identity(int* anc, int rows, int T) {
  const size_t n = (size_t)2 * rows * T;
  for (size_t j = blockIdx.x * (size_t)blockDim.x + threadIdx.x; j < n; j += (size_t)gridDim.x * blockDim.x)
    anc[j] = (int)((j / T) % rows);
}

int Engine::decode_logits(const float* memory, const int32_t* tokens, int t, float* logits_out, cudaStream_t s, float* hidden_out,
                          float* self_out, float* cross_out) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "decode_logits before finalize_weights");
  if (t < 1 || t > cfg_.max_len) return fail(FPNMT_ERR_INVALID, "decode_logits: t out of range");
  if (!tokens || (!logits_out && !hidden_out && !self_out && !cross_out)) return fail(FPNMT_ERR_INVALID, "decode_logits: NULL tokens / output");
  const bool attn = self_out || cross_out;
  if (attn && use_dstep_)
    return fail(FPNMT_ERR_STATE, "decode_attention: the fused decoder does not keep attention operands (use decode_path = chain)");
  const Tensor* last = nullptr;
  if (hidden_out) {
    auto it = taps_.find("dec" + std::to_string(cfg_.num_layers - 1) + "_out3");
    if (it == taps_.end())
      return fail(FPNMT_ERR_STATE, "decode_hidden: the fused decoder keeps layer outputs only with FPNMT_OPT_DSTEP_TAPS (or use decode_path = chain)");
    last = &it->second;
  }
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const int R = cfg_.batch * cfg_.beam;
  if (memory) RC(launch_f32_to_act(memory, enc_out_.pixels(), cfg_.d_model, enc_out_.a, s));
  RC(run_program(dec_init_prog_, s));
  k_forced_init<<<(R + 255) / 256, 256, 0, s>>>(bs_, tokens, t);
  FPNMT_CUDA_OK(cudaGetLastError());
  FlagGuard forced(forced_mode_);
  attn_self_ = self_out;
  attn_cross_ = cross_out;
  attn_tlen_ = t;
  for (int i = 0; i < t; ++i) {
    if (use_dstep_) {   // fused decoder, teacher-forcing mode: one step, fp32 logits of every row written out
      DstepParams q = dsp_;
      q.t0 = i;
      q.nsteps = 1;
      q.mode = 1;
      RC(dstep_launch(q, s));
      launches += 1;
    } else {
      RC(run_program(attn ? step_attn_prog_ : step_forced_prog_, s));
    }
    if (last) {
      k_forced_hidden<<<cfg_.batch, 128, 0, s>>>(last->a, bs_.step, cfg_.beam, t, hidden_out);
      launches += 1;
    }
    k_forced_tail<<<cfg_.batch, 256, 0, s>>>(bs_, logits_, tokens, t, logits_out);
    k_step_inc<<<1, 1, 0, s>>>(bs_.step);
    FPNMT_CUDA_OK(cudaGetLastError());
    launches += 2;
  }
  return 0;
}

int Engine::beam_step(const float* logits, const float* scores_in, int32_t* parent, int32_t* token, float* scores_out,
                      cudaStream_t s, const float2* vs_stat, const float* vs_val, const int* vs_idx, int vs_tiles) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "beam_step before finalize_weights");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const int R = cfg_.batch * cfg_.beam;
  BeamState st = bs_;
  st.vs_stat = vs_stat;
  st.vs_val = vs_val;
  st.vs_idx = vs_idx;
  st.vs_tiles = vs_tiles;
  RC(check_beam_step(st, cfg_.vocab));                     // a refused step launches nothing
  RC(launch_beam_init(bs_, 0, s));
  FPNMT_CUDA_OK(cudaMemcpyAsync(bs_.score[0], scores_in, (size_t)R * 4, cudaMemcpyDeviceToDevice, s));
  RC(launch_beam_step(st, logits, cfg_.vocab, BeamEmbed{nullptr, nullptr, Act{nullptr, 0, 0, 0}, 0}, s));
  launches += 2;
  FPNMT_CUDA_OK(cudaMemcpyAsync(parent, bs_.parent_out, (size_t)R * 4, cudaMemcpyDeviceToDevice, s));
  FPNMT_CUDA_OK(cudaMemcpyAsync(token, bs_.token_out, (size_t)R * 4, cudaMemcpyDeviceToDevice, s));
  FPNMT_CUDA_OK(cudaMemcpyAsync(scores_out, bs_.score[1], (size_t)R * 4, cudaMemcpyDeviceToDevice, s));
  return 0;
}

int Engine::decode(int32_t* out_ids, int32_t* out_len, int on_host, int early_stop, float* step_scores, cudaStream_t s) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "decode before finalize_weights");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const int B = cfg_.batch, T = cfg_.max_len;
  if (use_dstep_) {
    // Fused decoder: the whole fixed-length decode is ONE launch (every cluster runs its images through all T steps on
    // its own); with early stop the host looks at the finished-image counter every 4 steps, as the chain path does.
    RC(launch_beam_init(bs_, cfg_.true_beam, s));
    launches += 1;
    RC(run_program(dec_init_prog_, s));
    DstepParams q = dsp_;
    const int chunk = early_stop ? 4 : T;
    for (int t0 = 0; t0 < T; t0 += chunk) {
      q.t0 = t0;
      q.nsteps = std::min(chunk, T - t0);
      RC(dstep_launch(q, s));
      launches += 1;
      if (early_stop && t0 + chunk < T) {
        bool done = false;
        RC(poll_done(bs_.n_done, s, &done));
        if (done) break;
      }
    }
  } else {
  RC(launch_beam_init(bs_, cfg_.true_beam, s));
  launches += 1;
  RC(run_program(dec_init_prog_, s));
  RC(run_program(embed_prog_, s));
  if (cfg_.use_graphs && !early_stop) {
    // fixed-length decode: all T steps replay as ONE graph (no per-step graph-launch gap; the programmatic-launch chain
    // runs across step boundaries)
    if (!loop_graph_) {
      Program loop;
      Program one = step_prog_;
#ifdef FPNMT_DBG_STAMPS   // developer build only: leave ops out of the timed loop (timing attribution; results are garbage)
      if (const char* sk = getenv("FPNMT_SKIP")) {
        Program kept;
        for (auto& op : one) {
          bool skip = false;
          std::string list = sk;
          size_t pos = 0;
          while (pos <= list.size()) {
            size_t c = list.find(',', pos);
            if (c == std::string::npos) c = list.size();
            const std::string tok = list.substr(pos, c - pos);
            if (!tok.empty() && op.name.find(tok) != std::string::npos) skip = true;
            pos = c + 1;
          }
          if (!skip) kept.push_back(op);
        }
        one = kept;
      }
#endif
      for (int t = 0; t < T; ++t) loop.insert(loop.end(), one.begin(), one.end());
      RC(capture(loop, &loop_graph_));
    }
    FPNMT_CUDA_OK(cudaGraphLaunch(loop_graph_, s));
    launches += (int64_t)T * (int64_t)step_prog_.size();
  } else {
    RC(run_steps(step_prog_, step_graph_, bs_.n_done, early_stop, s));
  }
  }
  RC(copy_out(out_ids, bs_.out_ids, (size_t)B * T * 4, on_host, s));
  RC(copy_out(out_len, bs_.out_len, (size_t)B * 4, on_host, s));
  RC(copy_out(step_scores, step_scores_, (size_t)T * B * 4, 0, s));
  if (on_host) FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

int Engine::generate(const float* images, int on_host, int32_t* out_ids, int32_t* out_len, int out_on_host, int early_stop,
                     float* step_scores, cudaStream_t s) {
  RC(encode(images, on_host, nullptr, s, false));
  return decode(out_ids, out_len, out_on_host, early_stop, step_scores, s);
}

// Sampled decode.  Row r = (image r / N, sample r % N) runs the teacher-forced step program (whole layer stack, fp32 logits
// of every row, input token = BeamState::last_tok, identity ancestry, no KV-share representatives, first buffer pair) and
// k_sample_step draws its next token, so the N rows of an image are N independent samples.  The sampling parameters live in a
// device struct the kernel reads: a captured sample_graph_ serves every parameter set.
int Engine::sample(const float* images, int on_host, const fpnmt_sampling& sp, int32_t* out_ids, int32_t* out_len,
                   float* out_logprob, int out_on_host, int early_stop, cudaStream_t s, const PrefixArg* prefix,
                   const fpnmt_constraints* con) {
  RC(check_decode_entry("sample", "has no sampling tail"));
  const int B = cfg_.batch, N = cfg_.beam, T = cfg_.max_len, V = cfg_.vocab, R = B * N;
  if (check_sampling(sp, V))
    return fail(FPNMT_ERR_INVALID, "sample: temperature >= 0, top_p in (0, 1], 0 <= top_k <= vocab and reserved words 0");
  if (!out_ids || !out_len) return fail(FPNMT_ERR_INVALID, "sample: NULL out_ids / out_len");
  RC(check_prefix(con ? "sample_constrained" : "sample_prefix", prefix));
  RC(check_constraints("sample_constrained", con));
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  if (!ss_.ids) {   // per-row buffers [R][T] + [R] x 3 and the per-image counters, on the first call
    SampleState st{};
    st.rows = R; st.V = V; st.N = N; st.T = T;
    st.start_id = cfg_.start_id; st.end_id = cfg_.end_id;
    st.params = (const SampleParams*)dalloc(sizeof(SampleParams));
    st.step = bs_.step;
    st.last_tok = bs_.last_tok;
    st.n_done = bs_.n_done;
    st.ids = (int*)dalloc((size_t)R * T * 4);
    st.len = (int*)dalloc((size_t)R * 4);
    st.fin = (int*)dalloc((size_t)R * 4);
    st.lp = (float*)dalloc((size_t)R * 4);
    st.img_fin = (int*)dalloc((size_t)B * 4);
    if (!st.params || !st.ids || !st.len || !st.fin || !st.lp || !st.img_fin) return FPNMT_ERR_CUDA;
    sample_prog_ = step_forced_prog_;
    const float* lg = logits_;
    Op o = ew_op("sample_step", [st, lg](cudaStream_t q) { return launch_sample_step(st, lg, q); },
                 (double)R * V * 4 + (double)R * 16, "beam");
    o.idempotent = false;
    sample_prog_.push_back(std::move(o));
    ss_ = st;
  }
  if (prefix && sample_pfx_prog_.empty()) {   // prompted: the same program with the forced-capable sample op
    const SampleState st = ss_;
    const float* lg = logits_;
    const int *pid = pfx_ids_, *pln = pfx_len_;
    sample_pfx_prog_ = sample_prog_;
    Op& o = sample_pfx_prog_.back();
    o.name = "sample_step(prefix)";
    o.run = [st, lg, pid, pln](cudaStream_t q) { return launch_sample_step_prefix(st, pid, pln, lg, q); };
  }
  if (con && sample_con_prog_.empty()) {      // constrained: the same program with the masked sample op
    const SampleState st = ss_;
    const float* lg = logits_;
    const int *pid = pfx_ids_, *pln = pfx_len_;
    const BanMask bm = ban_;
    sample_con_prog_ = sample_prog_;
    Op& o = sample_con_prog_.back();
    o.name = "sample_step(constrained)";
    o.run = [st, lg, pid, pln, bm](cudaStream_t q) { return launch_sample_step_constrained(st, pid, pln, lg, bm, q); };
  }
  const SampleParams prm{sp.temperature, sp.top_k, sp.top_p, 0, (unsigned long long)sp.seed};
  if (images) RC(encode(images, on_host, nullptr, s, false));
  FPNMT_CUDA_OK(cudaMemcpyAsync(const_cast<SampleParams*>(ss_.params), &prm, sizeof prm, cudaMemcpyHostToDevice, s));
  RC(run_program(dec_init_prog_, s));
  if (con) RC(load_constraints(*con, prefix, s));
  else if (prefix) RC(load_prefix(*prefix, s));
  RC(launch_sample_init(ss_, bs_.anc[0], s));
  launches += 1;
  FlagGuard forced(forced_mode_);   // the self-attention launches of the program stay in the first buffer pair, without representatives
  if (con) {
    RC(run_steps(sample_con_prog_, sample_con_graph_, bs_.n_done, early_stop, s));
    if (prefix) {
      RC(launch_prefix_flag(pfx_bad_, B, N, T, ss_.ids, ss_.len, ss_.lp, s));
      launches += 1;
    }
  } else if (prefix) {
    RC(run_steps(sample_pfx_prog_, sample_pfx_graph_, bs_.n_done, early_stop, s));
    RC(launch_prefix_flag(pfx_bad_, B, N, T, ss_.ids, ss_.len, ss_.lp, s));
    launches += 1;
  } else {
    RC(run_steps(sample_prog_, sample_graph_, bs_.n_done, early_stop, s));
  }
  RC(copy_out(out_ids, ss_.ids, (size_t)R * T * 4, out_on_host, s));
  RC(copy_out(out_len, ss_.len, (size_t)R * 4, out_on_host, s));
  RC(copy_out(out_logprob, ss_.lp, (size_t)R * 4, out_on_host, s));
  if (out_on_host) FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

// N-best and diverse beam search.  The whole-batch step program with its beam_step op replaced by the N-best variant (same
// phase 1; phase 2 ranks the beams in beam_groups groups with the diversity penalty, and an image closes when all N beams are
// frozen, writing all of them).  The variant's state is a copy of the op's own (logits or the logits-free partials, KV
// ancestry and representatives, physical reorder by parent_out all unchanged) with finished_mode on, its own fin_len and its
// own length-penalty table followed by the (beam_groups, diversity) words, uploaded on every call: one captured graph serves
// every (G, lambda, alpha) and bs_.lp, which generate reads, is never touched.  fpnmt_beam_search is G = 1.
int Engine::beam_search(const float* images, int on_host, int beam_groups, float diversity, float length_penalty,
                        int32_t* out_ids, int32_t* out_len, float* out_logprob, int out_on_host, int early_stop, cudaStream_t s,
                        const PrefixArg* prefix, const fpnmt_constraints* con) {
  RC(check_decode_entry("beam_search", "has no N-best tail"));
  if (cfg_.score_mode == FPNMT_SCORE_PROB)
    return fail(FPNMT_ERR_STATE, "beam_search: the length penalty and the log-likelihoods need score_mode = log");
  if (!std::isfinite(length_penalty)) return fail(FPNMT_ERR_INVALID, "beam_search: length_penalty must be finite");
  if (check_beam_groups(step_bsv_, beam_groups, diversity)) return FPNMT_ERR_INVALID;
  if (!out_ids || !out_len) return fail(FPNMT_ERR_INVALID, "beam_search: NULL out_ids / out_len");
  RC(check_prefix(con ? "beam_search_constrained" : "beam_search_prefix", prefix));
  RC(check_constraints("beam_search_constrained", con));
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const int B = cfg_.batch, T = cfg_.max_len, R = B * cfg_.beam;
  if (!nbest_bs_.nb.ids) {
    BeamState st = step_bsv_;
    st.finished_mode = 1;
    st.fin_len[0] = (int*)dalloc((size_t)R * 4);
    st.fin_len[1] = (int*)dalloc((size_t)R * 4);
    st.lp = (const float*)dalloc((size_t)(T + 4) * 4);     // lp[0 .. T + 1], then G and lambda (nb.groups)
    st.nb.ids = (int*)dalloc((size_t)R * T * 4);
    st.nb.len = (int*)dalloc((size_t)R * 4);
    st.nb.score = (float*)dalloc((size_t)R * 4);
    if (!st.fin_len[0] || !st.fin_len[1] || !st.lp || !st.nb.ids || !st.nb.len || !st.nb.score) return FPNMT_ERR_CUDA;
    st.nb.groups = st.lp + T + 2;
    nbest_prog_ = step_prog_;
    const float* lg = logits_;
    const BeamEmbed em = beam_embed_;
    const int V = cfg_.vocab;
    Op& o = nbest_prog_[step_beam_at_];
    o.name = "beam_step(n-best)";
    o.run = [st, lg, V, em](cudaStream_t q) { return launch_beam_step_nbest(st, lg, V, em, q); };
    nbest_bs_ = st;
  }
  if (prefix && nbest_pfx_prog_.empty()) {
    // prompted: the forced-capable beam op on nbest_bs_ + the prefix buffers; on the logits-free tail the vocabulary
    // projection also reports the logit of each row's forced token
    BeamState st = nbest_bs_;
    st.pf.ids = pfx_ids_;
    st.pf.len = pfx_len_;
    nbest_pfx_prog_ = nbest_prog_;
    if (st.vs_stat) {
      st.pf.tgt = pfx_tgt_;
      st.pf.tgt_logit = pfx_tgt_logit_;
      TgemmOp op = vs_final_op_;
      op.tgt = pfx_tgt_;
      op.tgt_logit = pfx_tgt_logit_;
      Op& f = nbest_pfx_prog_[step_final_at_];
      f.name = "final_layer(softmax partials + candidates + target logit)";
      f.run = [op](cudaStream_t q) { return tgemm_launch(op, q); };
    }
    const float* lg = logits_;
    const BeamEmbed em = beam_embed_;
    const int V = cfg_.vocab;
    Op& o = nbest_pfx_prog_[step_beam_at_];
    o.name = "beam_step(n-best, prefix)";
    o.run = [st, lg, V, em](cudaStream_t q) { return launch_beam_step_prefix(st, lg, V, em, q); };
    nbest_pfx_bs_ = st;
  }
  if (con && nbest_con_prog_.empty()) {
    // constrained: the prompted program's state (prefix buffers, target logits) with the masked beam op and, on the logits-free
    // tail, the masked vocabulary projection (it reads the ban sets of the step parity in bs_.step)
    BeamState st = nbest_bs_;
    st.pf.ids = pfx_ids_;
    st.pf.len = pfx_len_;
    const BanMask bm = ban_;
    nbest_con_prog_ = nbest_prog_;
    if (st.vs_stat) {
      st.pf.tgt = pfx_tgt_;
      st.pf.tgt_logit = pfx_tgt_logit_;
      TgemmOp op = vs_final_op_;
      op.tgt = pfx_tgt_;
      op.tgt_logit = pfx_tgt_logit_;
      op.mask = bm.mask;
      op.mask_step = st.step;
      Op& f = nbest_con_prog_[step_final_at_];
      f.name = "final_layer(softmax partials + allowed candidates + target logit)";
      f.run = [op](cudaStream_t q) { return tgemm_launch(op, q); };
    }
    const float* lg = logits_;
    const BeamEmbed em = beam_embed_;
    const int V = cfg_.vocab;
    Op& o = nbest_con_prog_[step_beam_at_];
    o.name = "beam_step(n-best, constrained)";
    o.run = [st, lg, V, em, bm](cudaStream_t q) { return launch_beam_step_constrained(st, lg, V, em, bm, q); };
    nbest_con_bs_ = st;
  }
  std::vector<float> lp(T + 4);
  for (int i = 0; i < T + 2; ++i) lp[i] = powf((5.f + (float)i) / 6.f, length_penalty);
  lp[T + 2] = (float)beam_groups;
  lp[T + 3] = beam_groups > 1 ? diversity : 0.f;
  if (images) RC(encode(images, on_host, nullptr, s, false));
  FPNMT_CUDA_OK(cudaMemcpyAsync(const_cast<float*>(nbest_bs_.lp), lp.data(), lp.size() * 4, cudaMemcpyHostToDevice, s));
  // before the init kernel, which writes step 0's targets
  if (con) RC(load_constraints(*con, prefix, s));
  else if (prefix) RC(load_prefix(*prefix, s));
  RC(launch_beam_init(con ? nbest_con_bs_ : prefix ? nbest_pfx_bs_ : nbest_bs_, 1, s, beam_groups));
  launches += 1;
  RC(run_program(dec_init_prog_, s));
  RC(run_program(embed_prog_, s));
  if (con) {
    RC(run_steps(nbest_con_prog_, nbest_con_graph_, nbest_bs_.n_done, early_stop, s));
    if (prefix) {
      RC(launch_prefix_flag(pfx_bad_, B, cfg_.beam, T, nbest_bs_.nb.ids, nbest_bs_.nb.len, nbest_bs_.nb.score, s));
      launches += 1;
    }
  } else if (prefix) {
    RC(run_steps(nbest_pfx_prog_, nbest_pfx_graph_, nbest_bs_.n_done, early_stop, s));
    RC(launch_prefix_flag(pfx_bad_, B, cfg_.beam, T, nbest_bs_.nb.ids, nbest_bs_.nb.len, nbest_bs_.nb.score, s));
    launches += 1;
  } else {
    RC(run_steps(nbest_prog_, nbest_graph_, nbest_bs_.n_done, early_stop, s));
  }
  RC(copy_out(out_ids, nbest_bs_.nb.ids, (size_t)R * T * 4, out_on_host, s));
  RC(copy_out(out_len, nbest_bs_.nb.len, (size_t)R * 4, out_on_host, s));
  RC(copy_out(out_logprob, nbest_bs_.nb.score, (size_t)R * 4, out_on_host, s));
  if (out_on_host) FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

// The refusals of a prefix argument (nothing launched) and, on the first prompted call, the engine's prefix buffers.
int Engine::check_prefix(const char* entry, const PrefixArg* prefix) {
  if (!prefix) return 0;
  const std::string e = entry;
  if (!prefix->ids || !prefix->len) return fail(FPNMT_ERR_INVALID, e + ": NULL prefix_ids / prefix_len");
  if (prefix->p < 1 || prefix->p > cfg_.max_len - 1) return fail(FPNMT_ERR_INVALID, e + ": p must be 1 .. max_len - 1");
  return alloc_prefix();
}
int Engine::alloc_prefix() {
  if (!pfx_ids_) {
    FPNMT_CUDA_OK(cudaSetDevice(dev_));
    const int B = cfg_.batch, R = B * cfg_.beam;
    pfx_ids_ = (int*)dalloc((size_t)B * cfg_.max_len * 4);
    pfx_len_ = (int*)dalloc((size_t)B * 4);
    pfx_bad_ = (int*)dalloc((size_t)B * 4);
    pfx_tgt_ = (int*)dalloc((size_t)R * 4);
    pfx_tgt_logit_ = (float*)dalloc((size_t)R * 4);
    if (!pfx_ids_ || !pfx_len_ || !pfx_bad_ || !pfx_tgt_ || !pfx_tgt_logit_) return FPNMT_ERR_CUDA;
  }
  return 0;
}

// The refusals of a constraint set (nothing launched) and, on the first constrained call, the ban masks and the prefix buffers
// the constrained programs always carry.
int Engine::check_constraints(const char* entry, const fpnmt_constraints* con) {
  if (!con) return 0;
  const std::string e = entry;
  const int V = cfg_.vocab, T = cfg_.max_len;
  if (con->reserved[0] || con->reserved[1] || con->reserved[2] || con->reserved[3])
    return fail(FPNMT_ERR_INVALID, e + ": reserved words must be 0");
  if (con->no_repeat_ngram < 0 || con->no_repeat_ngram > T) return fail(FPNMT_ERR_INVALID, e + ": no_repeat_ngram must be 0 .. max_len");
  if (con->min_len < 0 || con->min_len > T) return fail(FPNMT_ERR_INVALID, e + ": min_len must be 0 .. max_len");
  if (con->n_banned < 0 || (con->n_banned > 0 && !con->banned)) return fail(FPNMT_ERR_INVALID, e + ": NULL banned with n_banned > 0");
  std::vector<char> seen(V, 0);
  int distinct = 0;
  for (int i = 0; i < con->n_banned; ++i) {
    const int v = con->banned[i];
    if (v < 0 || v >= V) return fail(FPNMT_ERR_INVALID, e + ": banned id " + std::to_string(v) + " outside [0, vocab)");
    if (v == cfg_.end_id) return fail(FPNMT_ERR_INVALID, e + ": <end> cannot be banned (min_len holds it back)");
    distinct += seen[v] ? 0 : 1;
    seen[v] = 1;
  }
  if (V - distinct - T < cfg_.beam)
    return fail(FPNMT_ERR_INVALID, e + ": vocab - distinct banned ids - max_len must be >= beam (allowed tokens at every step)");
  RC(alloc_prefix());
  if (!ban_.mask) {
    FPNMT_CUDA_OK(cudaSetDevice(dev_));                      // the entry points set the device only after these checks
    const int W = (V + 31) / 32, R = cfg_.batch * cfg_.beam;
    ban_.mask = (uint32_t*)dalloc((size_t)2 * R * W * 4);
    ban_.cfg = (const uint32_t*)dalloc((size_t)(2 + W) * 4);
    if (!ban_.mask || !ban_.cfg) return FPNMT_ERR_CUDA;
    ban_.rows = R;
    ban_.W = W;
    ban_.V = V;
    ban_.end_id = cfg_.end_id;
  }
  return 0;
}

// (n, min_len, S) -> ban_.cfg, the prefixes (all prefix_len 0 for an unprompted call), then step 0's ban sets
int Engine::load_constraints(const fpnmt_constraints& con, const PrefixArg* prefix, cudaStream_t s) {
  std::vector<uint32_t> h(2 + ban_.W, 0u);
  h[0] = (uint32_t)con.no_repeat_ngram;
  h[1] = (uint32_t)con.min_len;
  for (int i = 0; i < con.n_banned; ++i) h[2 + con.banned[i] / 32] |= 1u << (con.banned[i] % 32);
  FPNMT_CUDA_OK(cudaMemcpyAsync(const_cast<uint32_t*>(ban_.cfg), h.data(), h.size() * 4, cudaMemcpyHostToDevice, s));
  if (prefix) {
    RC(load_prefix(*prefix, s));
  } else {
    FPNMT_CUDA_OK(cudaMemsetAsync(pfx_len_, 0, (size_t)cfg_.batch * 4, s));
  }
  RC(launch_ban_rows(ban_, 0, nullptr, 0, nullptr, s));
  launches += 1;
  return 0;
}

// the caller's prefixes -> pfx_ids_ / pfx_len_ / pfx_bad_ (checked and clamped on the device)
int Engine::load_prefix(const PrefixArg& prefix, cudaStream_t s) {
  RC(launch_prefix_load(prefix.ids, prefix.len, prefix.p, cfg_.batch, cfg_.max_len, cfg_.vocab, cfg_.end_id, pfx_ids_, pfx_len_,
                        pfx_bad_, s));
  launches += 1;
  return 0;
}

// Score program for captions of t positions.  Row r = c * t + j (caption c = b * N + n, position j) of every activation:
// the Dense layers are igemm in its 1x1 dense geometry at B * N * t rows (LayerNorm layers: fp32 residual output, then
// layernorm_rows), the self-attention is causal over the caption's own rows, the cross-attention is the step program's kernel
// with beam := N * t (rows per image).  The vocabulary projection runs in chunks of B * N rows through the [B * N][V] logits
// buffer of the step programs, each followed by score_rows; score_sum closes the pass.
int Engine::build_score(int t, Program& p) {
  const int B = cfg_.batch, N = cfg_.beam, D = cfg_.d_model, H = cfg_.num_heads, V = cfg_.vocab, L = cfg_.num_layers;
  const int R = B * N, rows = R * t;
  const double esz = split_ ? 4.0 : 2.0;
  auto view = [rows](const Tensor& a) {
    Tensor v = a;
    v.N = 1; v.H = 1; v.W = rows;
    return v;
  };
  Tensor x = view(sc_.x), qkv = view(sc_.qkv), att = view(sc_.att), out1 = view(sc_.out1), q2 = view(sc_.q2),
         out2 = view(sc_.out2), hdn = view(sc_.hdn);
  Tensor none;
  float* y = sc_.y;
  const ScoreArgs a{R, t, V, cfg_.start_id, cfg_.end_id, sc_.ids, sc_.lens, sc_.tgt, sc_.bad, sc_.tok_lp, sc_.lp};
  {
    const float *emb = dec_emb_, *pos = dec_pos_;
    const Act xa = x.a;
    p.push_back(ew_op("score_embed", [=](cudaStream_t s) { return launch_score_embed(a, emb, pos, xa, s); },
                      (double)rows * D * (8 + esz) + (double)rows * 8));
  }
  auto dense_ln = [&](const std::string& nm, const Tensor& in, const GemmW& g, const Tensor& res, const float* gam,
                      const float* bet, const Tensor& out) -> int {
    RC(add_conv(p, nm, in, g, 1, 1, 0, 0, ACT_NONE, RES_SAME, &res, none, y, D));
    const Act oa = out.a;
    p.push_back(ew_op(nm + "_ln", [=](cudaStream_t s) { return launch_layernorm_rows(y, rows, D, gam, bet, 1e-6f, oa, s); },
                      (double)rows * D * (4 + esz)));
    return 0;
  };
  for (int l = 0; l < L; ++l) {
    const DecLayerW& w = dec_lw_[l];
    const std::string ln = "score_dec" + std::to_string(l);
    RC(add_conv(p, ln + "_qkv", x, w.gqkv, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, qkv));
    {
      const Act qa = qkv.a, oa = att.a;
      Op o = ew_op(ln + "_self_attn", [=](cudaStream_t s) { return launch_score_self_attention(qa, R, t, H, oa, s); },
                   (double)rows * D * 4 * esz, "attention");
      o.flops = 4.0 * R * D * (double)t * (t + 1) / 2;
      p.push_back(std::move(o));
    }
    RC(dense_ln(ln + "_o1+res", att, w.go1, x, w.lnp[0], w.lnp[1], out1));
    RC(add_conv(p, ln + "_q2", out1, w.gq2, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, q2));
    {
      const Act qa = q2.a, oa = att.a, ka = dec_ckv_.a;
      const int kcx = l * 2 * D, vcx = l * 2 * D + D, tk = n_base_, rows_per_image = N * t;
      p.push_back(ew_op(ln + "_cross_attn",
                        [=](cudaStream_t s) { return launch_dec_cross_attention(qa, ka, kcx, vcx, rows, rows_per_image, tk, H, oa, s); },
                        (double)rows * D * 2 * esz + (double)B * tk * 2 * D * esz, "attention"));
    }
    RC(dense_ln(ln + "_o2+res", att, w.go2, out1, w.lnp[2], w.lnp[3], out2));
    RC(add_conv(p, ln + "_ffn1", out2, w.g1, 1, 1, 0, 0, ACT_LEAKY, RES_NONE, nullptr, hdn));
    RC(dense_ln(ln + "_ffn2+res", hdn, w.g2, out2, w.lnp[4], w.lnp[5], x));
  }
  for (int c = 0; c < t; ++c) {
    Tensor xc = x;
    xc.a.p = x.a.p + (size_t)c * R * x.a.ld;
    xc.W = R;
    RC(add_conv(p, "score_final_layer", xc, dec_final_, 1, 1, 0, 0, ACT_NONE, RES_NONE, nullptr, none, logits_, V));
    const int* tg = sc_.tgt + (size_t)c * R;
    float* tl = sc_.tok_lp + (size_t)c * R;
    const float* lg = logits_;
    p.push_back(ew_op("score_rows", [=](cudaStream_t s) { return launch_score_rows(lg, R, V, tg, tl, s); },
                      (double)R * V * 4 + (double)R * 8));
  }
  p.push_back(ew_op("score_sum", [=](cudaStream_t s) { return launch_score_sum(a, s); }, (double)rows * 8 + (double)R * 8));
  return 0;
}

int Engine::score(const float* images, int on_host, const int32_t* ids, const int32_t* lens, int t, float* out_logprob,
                  float* out_token_logprob, int out_on_host, cudaStream_t s) {
  RC(check_decode_entry("score", "has no per-layer weights for a parallel pass"));
  if (t < 1 || t > cfg_.max_len) return fail(FPNMT_ERR_INVALID, "score: t must lie in [1, max_len]");
  if (!ids || !lens || !out_logprob) return fail(FPNMT_ERR_INVALID, "score: NULL ids / lens / out_logprob");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const int R = cfg_.batch * cfg_.beam, T = cfg_.max_len, D = cfg_.d_model;
  if (!sc_.x.a.p) {   // activations of B * N * max_len rows, on the first call
    const int rows = R * T;
    sc_.x = rows_act(rows, D); sc_.qkv = rows_act(rows, 3 * D); sc_.att = rows_act(rows, D); sc_.out1 = rows_act(rows, D);
    sc_.q2 = rows_act(rows, D); sc_.out2 = rows_act(rows, D); sc_.hdn = rows_act(rows, cfg_.dff);
    sc_.y = (float*)dalloc((size_t)rows * D * 4);
    sc_.ids = (int*)dalloc((size_t)rows * 4);
    sc_.lens = (int*)dalloc((size_t)R * 4);
    sc_.tgt = (int*)dalloc((size_t)rows * 4);
    sc_.bad = (int*)dalloc((size_t)R * 4);
    sc_.tok_lp = (float*)dalloc((size_t)rows * 4);
    sc_.lp = (float*)dalloc((size_t)R * 4);
    if (!sc_.x.a.p || !sc_.qkv.a.p || !sc_.att.a.p || !sc_.out1.a.p || !sc_.q2.a.p || !sc_.out2.a.p || !sc_.hdn.a.p || !sc_.y ||
        !sc_.ids || !sc_.lens || !sc_.tgt || !sc_.bad || !sc_.tok_lp || !sc_.lp) {
      sc_.x.a.p = nullptr;
      return FPNMT_ERR_CUDA;
    }
  }
  auto it = score_progs_.find(t);
  if (it == score_progs_.end()) {
    Program p;
    RC(build_score(t, p));
    it = score_progs_.emplace(t, std::move(p)).first;
  }
  if (images) RC(encode(images, on_host, nullptr, s, false));
  FPNMT_CUDA_OK(cudaMemcpyAsync(sc_.ids, ids, (size_t)R * t * 4, cudaMemcpyDeviceToDevice, s));
  FPNMT_CUDA_OK(cudaMemcpyAsync(sc_.lens, lens, (size_t)R * 4, cudaMemcpyDeviceToDevice, s));
  RC(run_program(dec_init_prog_, s));
  RC(launch_graph(it->second, score_graphs_[t], s));
  RC(copy_out(out_logprob, sc_.lp, (size_t)R * 4, out_on_host, s));
  RC(copy_out(out_token_logprob, sc_.tok_lp, (size_t)R * t * 4, out_on_host, s));
  if (out_on_host) FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

// Double-buffered input (the role of dataset.py:90-92's map/prefetch in the reference's input pipeline): the copy of the
// next batch runs on the engine's own stream, ordered against the compute stream with two events per slot.
int Engine::stage_images(const float* host_images, int slot) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "stage_images before finalize_weights");
  if (!host_images || slot < 0 || slot > 1) return fail(FPNMT_ERR_INVALID, "stage_images: NULL images or slot not 0/1");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const size_t n = (size_t)cfg_.batch * cfg_.image_size * cfg_.image_size * 3;
  if (!copy_stream_) FPNMT_CUDA_OK(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
  if (!stage_buf_[slot]) {
    stage_buf_[slot] = (float*)dalloc(n * 4);
    if (!stage_buf_[slot]) return FPNMT_ERR_CUDA;
    FPNMT_CUDA_OK(cudaEventCreateWithFlags(&stage_ready_[slot], cudaEventDisableTiming));
    FPNMT_CUDA_OK(cudaEventCreateWithFlags(&stage_free_[slot], cudaEventDisableTiming));
  } else {
    FPNMT_CUDA_OK(cudaStreamWaitEvent(copy_stream_, stage_free_[slot], 0));   // last consumer of this slot is done
  }
  FPNMT_CUDA_OK(cudaMemcpyAsync(stage_buf_[slot], host_images, n * 4, cudaMemcpyHostToDevice, copy_stream_));
  FPNMT_CUDA_OK(cudaEventRecord(stage_ready_[slot], copy_stream_));
  stage_filled_[slot] = true;
  return 0;
}

int Engine::generate_staged(int slot, int32_t* out_ids, int32_t* out_len, int out_on_host, int early_stop, float* step_scores,
                            cudaStream_t s) {
  if (slot < 0 || slot > 1 || !stage_filled_[slot]) return fail(FPNMT_ERR_STATE, "generate_staged: slot was not staged");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  FPNMT_CUDA_OK(cudaStreamWaitEvent(s, stage_ready_[slot], 0));
  RC(encode(stage_buf_[slot], 0, nullptr, s, false));
  FPNMT_CUDA_OK(cudaEventRecord(stage_free_[slot], s));
  stage_filled_[slot] = false;
  return decode(out_ids, out_len, out_on_host, early_stop, step_scores, s);
}

// Lane interface.  submit() enqueues a whole batch on the engine's own stream and returns; collect() hands the result over.
// Device-resident images are ordered against the caller's stream with an event (they must stay valid until collect); host
// images are copied into the lane's staging buffer on the lane stream (pinned memory for a truly asynchronous copy; the buffer
// must stay valid until collect).  A fixed-length decode is enqueued completely at submit; an early-stop decode needs the host
// to look at the finished-image counter, so submit enqueues the encoder only and collect drives the decode - the encoder of the
// batch submitted on another lane in between still overlaps it.
int Engine::submit(const float* images, int on_host, int early_stop, cudaStream_t caller, cudaEvent_t prev_encode_done) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "submit before finalize_weights");
  if (lane_state_ != 0) return fail(FPNMT_ERR_STATE, "submit: this lane still holds a batch (call fpnmt_collect first)");
  if (!images) return fail(FPNMT_ERR_INVALID, "images is NULL");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  if (!lane_stream_) {
    // Two streams per lane, encoder and decode chain, at EQUAL priority.  Measured on C2 with 4 lanes: decode streams at the
    // highest priority starve the encoder at every one of its 151 kernel boundaries (2 950 -> 1 960 images/s with the encoder
    // chain below, 2 650 without it); encoder-high is neutral (2 920).
    FPNMT_CUDA_OK(cudaStreamCreateWithFlags(&lane_stream_, cudaStreamNonBlocking));
    FPNMT_CUDA_OK(cudaStreamCreateWithFlags(&lane_dec_stream_, cudaStreamNonBlocking));
    FPNMT_CUDA_OK(cudaEventCreateWithFlags(&lane_in_ev_, cudaEventDisableTiming));
    FPNMT_CUDA_OK(cudaEventCreateWithFlags(&lane_out_ev_, cudaEventDisableTiming));
    FPNMT_CUDA_OK(cudaEventCreateWithFlags(&lane_enc_ev_, cudaEventDisableTiming));
  }
  FPNMT_CUDA_OK(cudaStreamWaitEvent(lane_stream_, lane_out_ev_, 0));   // the previous batch of this lane has left the decode stream
  if (!on_host) {
    FPNMT_CUDA_OK(cudaEventRecord(lane_in_ev_, caller));
    FPNMT_CUDA_OK(cudaStreamWaitEvent(lane_stream_, lane_in_ev_, 0));
  }
  RC(set_images(images, on_host, lane_stream_));
  // Encoders of different lanes run one after the other, in submission order: they are throughput-bound (nothing is gained by
  // running two at once) and a staggered pipeline - one encoder under the decodes of the other lanes - is what the lanes are
  // for.  Without the chain the overlap depends on when the host happens to submit (measured: 2 920 -> 2 960 images/s, and
  // the run-to-run spread of the device-resident figure shrinks).
  if (prev_encode_done) FPNMT_CUDA_OK(cudaStreamWaitEvent(lane_stream_, prev_encode_done, 0));
  RC(launch_graph(enc_prog_, enc_graph_, lane_stream_));
  FPNMT_CUDA_OK(cudaEventRecord(lane_enc_ev_, lane_stream_));
  FPNMT_CUDA_OK(cudaStreamWaitEvent(lane_dec_stream_, lane_enc_ev_, 0));
  if (early_stop) {
    lane_state_ = 2;
    return 0;
  }
  RC(decode(nullptr, nullptr, 0, 0, nullptr, lane_dec_stream_));
  FPNMT_CUDA_OK(cudaEventRecord(lane_out_ev_, lane_dec_stream_));
  lane_state_ = 1;
  return 0;
}

int Engine::collect(int32_t* out_ids, int32_t* out_len, int on_host, cudaStream_t caller) {
  if (lane_state_ == 0) return fail(FPNMT_ERR_STATE, "collect: nothing was submitted on this lane");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  const int B = cfg_.batch, T = cfg_.max_len;
  const int st = lane_state_;
  lane_state_ = 0;
  if (st == 2) {
    RC(decode(out_ids, out_len, on_host, 1, nullptr, lane_dec_stream_));
  } else {
    RC(copy_out(out_ids, bs_.out_ids, (size_t)B * T * 4, on_host, lane_dec_stream_));
    RC(copy_out(out_len, bs_.out_len, (size_t)B * 4, on_host, lane_dec_stream_));
  }
  FPNMT_CUDA_OK(cudaEventRecord(lane_out_ev_, lane_dec_stream_));
  if (on_host) {
    FPNMT_CUDA_OK(cudaStreamSynchronize(lane_dec_stream_));
  } else {
    FPNMT_CUDA_OK(cudaStreamWaitEvent(caller, lane_out_ev_, 0));
  }
  return 0;
}

// --------------------------------------------------------------------------------------------- profiling
// Busy-wait kernel: keeps the GPU occupied while the host enqueues the whole timed program, so that the CUDA-event
// intervals measure device execution only (no host launch gaps).
__global__ void k_spin(long long ns) {
  long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  do {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
  } while (t1 - t0 < ns);
}

int Engine::profile_program(Program& p, int iters, std::string& json, const char* label) {
  cudaStream_t s = cap_stream_;
  const size_t n = p.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) FPNMT_CUDA_OK(cudaEventCreate(&e));
  std::vector<int> reps(n);
  size_t total_launches = 0;
  for (size_t i = 0; i < n; ++i) {
    reps[i] = p[i].idempotent ? iters : 1;
    total_launches += reps[i];
  }
  k_spin<<<1, 1, 0, s>>>((long long)(total_launches * 6000 + 200000));   // ~6 us of host time per launch
  FPNMT_CUDA_OK(cudaEventRecord(ev[0], s));
  for (size_t i = 0; i < n; ++i) {
    for (int r = 0; r < reps[i]; ++r) RC(p[i].run(s));
    FPNMT_CUDA_OK(cudaEventRecord(ev[i + 1], s));
  }
  FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  json += std::string("\"") + label + "\": [";
  for (size_t i = 0; i < n; ++i) {
    float ms = 0;
    FPNMT_CUDA_OK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    char buf[512];
    snprintf(buf, sizeof buf, "%s{\"name\": \"%s\", \"kind\": \"%s\", \"us\": %.3f, \"flops\": %.6g, \"bytes\": %.6g}",
             i ? ", " : "", p[i].name.c_str(), p[i].kind.c_str(), ms * 1000.0 / reps[i], p[i].flops, p[i].bytes);
    json += buf;
  }
  json += "]";
  for (auto& e : ev) cudaEventDestroy(e);
  return 0;
}

int Engine::profile(int iters, char* buf, size_t cap) {
  if (!finalized_) return fail(FPNMT_ERR_STATE, "profile before finalize_weights");
  FPNMT_CUDA_OK(cudaSetDevice(dev_));
  if (iters < 1) iters = 1;
  // requires a prior encode() so that the image slot points at valid data
  std::string json = "{";
  RC(profile_program(enc_prog_, iters, json, "encode"));
  json += ", ";
  cudaStream_t s = cap_stream_;
  RC(launch_beam_init(bs_, cfg_.true_beam, s));
  RC(run_program(dec_init_prog_, s));
  RC(run_program(embed_prog_, s));
  const int warm = cfg_.max_len / 2;
  prof_t_ = 0;
  for (int t = 0; t < warm; ++t) RC(run_program(step_prog_, s));
  RC(profile_program(dec_init_prog_, iters, json, "decode_init"));
  json += ", ";
  RC(profile_program(step_prog_, iters, json, "decode_step"));
  char tail[240];
  snprintf(tail, sizeof tail, ", \"decode_step_t\": %d, \"device_bytes\": %zu, \"dstep_groups_per_launch\": %d}", warm,
           alloc_bytes_, use_dstep_ ? dstep_max_groups(num_sms_) : 0);
  json += tail;
  FPNMT_CUDA_OK(cudaStreamSynchronize(s));
  if (dbg_buf_ && use_dstep_ && dsp_.timeline) {   // FPNMT_DBG_OP=dstep: phase stamps of the last profiled step (cluster 0, CTA 0)
    long long h[16 * 9];
    cudaMemcpy(h, dbg_buf_, sizeof h, cudaMemcpyDeviceToHost);
    fprintf(stderr, "[fpnmt dbg] dstep timeline, %lld stamps (ns since step start):", h[0]);
    for (int i = 0; i < (int)h[0] && i < 120; ++i) fprintf(stderr, " %lld", h[1 + i] - h[1]);
    fprintf(stderr, "\n");
  } else
  if (dbg_buf_) {   // FPNMT_DBG_OP timeline of the last 8 instances (ns relative to each instance's entry)
    long long h[16 * 9];
    cudaMemcpy(h, dbg_buf_, sizeof h, cudaMemcpyDeviceToHost);
    fprintf(stderr, "[fpnmt dbg] %lld instances; stamps: entry setup pdl_wait first_full mma_issued tfull epi_chunk0 epi_chunk1 end tile1_start tile2_start tile3_start tile4_start\n", h[0]);
    for (int i = 0; i < 8; ++i) {
      const long long* t = h + 16 + i * 16;
      fprintf(stderr, "[fpnmt dbg] inst slot %d entry@%lld:", i, t[0]);
      for (int k = 1; k <= 12; ++k) fprintf(stderr, " %6lld", t[k] ? t[k] - t[0] : -1);
      fprintf(stderr, "\n");
    }
  }
  if (cap == 0) return fail(FPNMT_ERR_INVALID, "profile: zero capacity");
  const size_t n = std::min(cap - 1, json.size());
  memcpy(buf, json.data(), n);
  buf[n] = 0;
  return 0;
}

}  // namespace fpnmt
