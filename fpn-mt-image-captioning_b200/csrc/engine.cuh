// Engine: owns weights, activation buffers, the kernel programs (encode / decode step) and their CUDA graphs.
#pragma once
#include <functional>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/fpnmt.h"
#include "igemm.cuh"
#include "kernels.cuh"
#include "tensormap.cuh"
#include "tgemm.cuh"
#include "stem.cuh"
#include "xattn.cuh"
#include "dstep.cuh"

namespace fpnmt {

struct HostW {
  std::vector<int64_t> shape;
  std::vector<float> data;
};

struct GemmW {          // device weight matrix [Cout][K] bf16 (split: [Cout][2K]) + fp32 bias
  bf16* w = nullptr;
  float* bias = nullptr;
  int Cout = 0, K = 0;
};

struct DecLayerW {      // device weights of one decoder layer (shared by the step programs and the score pass)
  GemmW gqkv, go1, gq2, go2, g1, g2;
  float* lnp[6];        // layernorm{1,2,3} gamma, beta
};

struct Tensor {         // NHWC activation (dense rows: N=1,H=1,W=rows)
  Act a{nullptr, 0, 0, 0};
  int N = 0, H = 0, W = 0;
  size_t pixels() const { return (size_t)N * H * W; }
};

struct Op {
  std::string name;
  std::string kind;     // "igemm", "elementwise", "attention", "beam"
  std::function<int(cudaStream_t)> run;
  double flops = 0;     // algorithmic (2*MAC)
  double bytes = 0;     // algorithmic HBM bytes (inputs read once + outputs written once)
  bool idempotent = true;
};
typedef std::vector<Op> Program;

// The caption prefixes of a prompted decode (fpnmt_sample_prefix / fpnmt_beam_search_prefix): DEVICE ids [batch][p] and
// len [batch], never read by the host.
struct PrefixArg {
  const int32_t* ids;
  const int32_t* len;
  int p;
};

class Engine {
 public:
  Engine(const fpnmt_config& cfg, int device);
  ~Engine();
  int init();
  int set_weight(const char* key, const float* data, const int64_t* shape, int ndim);
  int finalize();
  int encode(const float* images, int on_host, float* memory_out, cudaStream_t s, bool cnn_only = false);
  int features(const float* images, int on_host, float* const out5[5], cudaStream_t s);
  int get_tap(const char* name, float* out, size_t cap, size_t* count, cudaStream_t s);
  // self_out / cross_out (either may be nullptr): attention probabilities of the beam-0 rows, [L][B][heads][t][t] and
  // [L][B][heads][t][n_mem] (step_attn_prog_; not with the fused decoder)
  int decode_logits(const float* memory, const int32_t* tokens, int t, float* logits_out, cudaStream_t s, float* hidden_out = nullptr,
                    float* self_out = nullptr, float* cross_out = nullptr);
  // vs_stat != nullptr: the logits-free tail on the caller's softmax partials and candidates ([B*N][vs_tiles], see BeamState)
  int beam_step(const float* logits, const float* scores_in, int32_t* parent, int32_t* token, float* scores_out,
                cudaStream_t s, const float2* vs_stat = nullptr, const float* vs_val = nullptr, const int* vs_idx = nullptr,
                int vs_tiles = 0);
  int decode(int32_t* out_ids, int32_t* out_len, int on_host, int early_stop, float* step_scores, cudaStream_t s);
  int generate(const float* images, int on_host, int32_t* out_ids, int32_t* out_len, int out_on_host, int early_stop,
               float* step_scores, cudaStream_t s);
  // Sampled decode (fpnmt_sample): every row of the batch is one independent sample of its image; the teacher-forced step
  // program with k_sample_step in place of the teacher-forced tail.  images == nullptr: the memory of the last encode.
  // prefix != nullptr: the prompted decode (fpnmt_sample_prefix) on sample_pfx_prog_.  con != nullptr: the constrained decode
  // (fpnmt_sample_constrained, prompted or not) on sample_con_prog_.
  int sample(const float* images, int on_host, const fpnmt_sampling& sp, int32_t* out_ids, int32_t* out_len, float* out_logprob,
             int out_on_host, int early_stop, cudaStream_t s, const PrefixArg* prefix = nullptr,
             const fpnmt_constraints* con = nullptr);
  // Caption scoring (fpnmt_score): the N captions ids [B][N][t] / lens [B][N] (device) of every image through the decoder
  // as B * N * t rows of one teacher-forced pass.  images == nullptr: the memory of the last encode.
  int score(const float* images, int on_host, const int32_t* ids, const int32_t* lens, int t, float* out_logprob,
            float* out_token_logprob, int out_on_host, cudaStream_t s);
  // N-best beam search (fpnmt_beam_search: beam_groups = 1) and diverse beam search (fpnmt_beam_search_diverse): the
  // whole-batch step program with k_beam_step's group ranking and N-best close, true-beam start (first beam of every group),
  // frozen finished beams and this call's length penalty.  images == nullptr: the memory of the last encode.
  // prefix != nullptr: the prompted search (fpnmt_beam_search_prefix) on nbest_pfx_prog_.  con != nullptr: the constrained
  // search (fpnmt_beam_search_constrained, prompted or not) on nbest_con_prog_.
  int beam_search(const float* images, int on_host, int beam_groups, float diversity, float length_penalty, int32_t* out_ids,
                  int32_t* out_len, float* out_logprob, int out_on_host, int early_stop, cudaStream_t s,
                  const PrefixArg* prefix = nullptr, const fpnmt_constraints* con = nullptr);
  int profile(int iters, char* buf, size_t cap);
  int build_dstep(const Tensor& ckv, const float* d_emb, const float* d_pos);
  int get_tap_f32(const std::string& name, float* out, size_t cap, size_t* count, cudaStream_t s);
  int add_stem(Program& p, const std::string& name, int kh, int pad, int cout, const GemmW& gw, int Kp, int act, const Tensor& out);
  // double-buffered host input: copy batch i+1 on the engine's copy stream while batch i runs
  int stage_images(const float* host_images, int slot);
  int generate_staged(int slot, int32_t* out_ids, int32_t* out_len, int outputs_on_host, int early_stop, float* step_scores,
                      cudaStream_t s);
  // Lane interface (fpnmt_submit / fpnmt_collect): one batch in flight per engine on the engine's own stream, so that several
  // engines ("lanes") of one handle overlap the throughput-bound encode of one batch with the latency-bound decode of another.
  void share_weights_of(const Engine* lead) { weight_lead_ = lead; }   // before finalize(); `lead` must outlive this engine
  int submit(const float* images, int on_host, int early_stop, cudaStream_t caller, cudaEvent_t prev_encode_done = nullptr);
  cudaEvent_t encode_done_event() const { return lane_enc_ev_; }   // recorded after the encoder of the last submitted batch
  int collect(int32_t* out_ids, int32_t* out_len, int on_host, cudaStream_t caller);
  const fpnmt_config& config() const { return cfg_; }
  int device() const { return dev_; }
  int64_t launches = 0;

 private:
  cudaStream_t lane_stream_ = nullptr, lane_dec_stream_ = nullptr;   // encoder / decode chain of the lane's batch
  cudaEvent_t lane_in_ev_ = nullptr, lane_out_ev_ = nullptr, lane_enc_ev_ = nullptr;
  int lane_state_ = 0;                    // 0 idle, 1 = fixed-length batch enqueued, 2 = encode enqueued, early-stop decode runs in collect()
  fpnmt_config cfg_;
  int dev_;
  int num_sms_ = 148;
  bool split_ = false;
  bool finalized_ = false;
  std::unordered_map<std::string, HostW> hw_;
  std::vector<void*> allocs_;
  size_t alloc_bytes_ = 0;
  std::map<std::string, Tensor> taps_;

  // programs
  Program cnn_prog_, enc_prog_, dec_init_prog_, embed_prog_, step_prog_, step_forced_prog_;
  Program step_attn_prog_;                // step_forced_prog_ + the attention-probability launches (decode_logits with outputs)
  Program sample_prog_;                   // step_forced_prog_ + k_sample_step (sample; built on its first call)
  // beam search: step_prog_ with its beam_step op (index step_beam_at_, state step_bsv_) replaced by the N-best step on
  // nbest_bs_, a copy of step_bsv_ with its own fin_len, length-penalty table + beam-group words and the N-best outputs (built
  // on its first call; fpnmt_beam_search and fpnmt_beam_search_diverse share it)
  size_t step_beam_at_ = 0;
  BeamState step_bsv_{};
  Program nbest_prog_;
  BeamState nbest_bs_{};
  cudaGraphExec_t nbest_graph_ = nullptr;
  // prompted decode (built on its first call): nbest_prog_ with the beam op replaced by the forced-capable one on nbest_pfx_bs_
  // (nbest_bs_ + the prefix buffers) and, on the logits-free tail, the vocabulary projection (index step_final_at_, op
  // vs_final_op_) by its target variant; sample_pfx_prog_ is sample_prog_ with the forced-capable sample op.  The prefixes
  // are copied into pfx_ids_ / pfx_len_ on every call, so one captured graph serves every prefix.
  size_t step_final_at_ = 0;
  TgemmOp vs_final_op_{};
  Program nbest_pfx_prog_, sample_pfx_prog_;
  BeamState nbest_pfx_bs_{};
  cudaGraphExec_t nbest_pfx_graph_ = nullptr, sample_pfx_graph_ = nullptr;
  int *pfx_ids_ = nullptr, *pfx_len_ = nullptr, *pfx_bad_ = nullptr, *pfx_tgt_ = nullptr;   // [B][T], [B], [B], [B*N]
  float* pfx_tgt_logit_ = nullptr;                                                          // [B*N]
  int check_prefix(const char* entry, const PrefixArg* prefix);
  int alloc_prefix();
  int load_prefix(const PrefixArg& prefix, cudaStream_t s);
  // constrained decode (built on its first call): copies of the prompted programs (an unprompted call runs them with every
  // prefix_len 0) with the beam / sample op replaced by its MASK variant and, on the logits-free tail, the vocabulary projection
  // by tgemmw_mask_kernel.  The ban sets live in ban_ (one buffer pair for both programs); each call uploads (n, min_len, S)
  // and writes step 0's sets, so one captured graph serves every constraint set.
  Program nbest_con_prog_, sample_con_prog_;
  BeamState nbest_con_bs_{};
  cudaGraphExec_t nbest_con_graph_ = nullptr, sample_con_graph_ = nullptr;
  BanMask ban_{};
  int check_constraints(const char* entry, const fpnmt_constraints* con);
  int load_constraints(const fpnmt_constraints& con, const PrefixArg* prefix, cudaStream_t s);
  SampleState ss_{};                      // sampler state: per-row buffers allocated on the first sample call
  cudaGraphExec_t sample_graph_ = nullptr;   // sample_prog_ captured with forced_mode_ set (never step_graph_)
  // score pass: one program (and graph) per caption length t, built on its first call; activations for B * N * max_len rows
  // allocated on the first call and shared by all of them (one layer's set is live at a time)
  struct ScoreBufs {
    Tensor x, qkv, att, out1, q2, out2, hdn;
    float* y = nullptr;
    int *ids = nullptr, *lens = nullptr, *tgt = nullptr, *bad = nullptr;
    float *tok_lp = nullptr, *lp = nullptr;
  } sc_;
  std::map<int, Program> score_progs_;
  std::map<int, cudaGraphExec_t> score_graphs_;
  std::vector<DecLayerW> dec_lw_;         // decoder weights prepared by build_decoder (chain decode path)
  GemmW dec_final_{};
  const float *dec_emb_ = nullptr, *dec_pos_ = nullptr;   // [V][D] embedding, [max_len][D] positional table
  Tensor dec_ckv_;                        // cross-attention K/V of the memory, all layers [B * n_mem][L * 2 * D]
  int build_score(int t, Program& p);
  BeamEmbed beam_embed_{};
  cudaGraphExec_t cnn_graph_ = nullptr, enc_graph_ = nullptr, step_graph_ = nullptr, loop_graph_ = nullptr;
  cudaStream_t cap_stream_ = nullptr;

  // buffers referenced at run time
  const float** img_slot_ = nullptr;      // device slot holding the current image pointer
  float* img_stage_ = nullptr;            // device staging for host images
  float* stage_buf_[2] = {nullptr, nullptr};          // fpnmt_stage_images slots
  cudaEvent_t stage_ready_[2] = {nullptr, nullptr};   // copy of the slot finished (recorded on copy_stream_)
  cudaEvent_t stage_free_[2] = {nullptr, nullptr};    // encoder has consumed the slot (recorded on the compute stream)
  bool stage_filled_[2] = {false, false};
  cudaStream_t copy_stream_ = nullptr;
  Tensor feat_[5];                        // head outputs P3..P7
  Tensor enc_out_;                        // (B*16, 512)
  int n_base_ = 16;                       // tokens of the baseline view
  BeamState bs_{};
  bool use_dstep_ = false;                // group-stationary fused decoder (dstep.cuh) instead of the per-operator chain
  DstepParams dsp_{};
  bool forced_mode_ = false;              // decode_logits is running (physical cache mode: no buffer alternation)
  float* attn_self_ = nullptr;            // attention outputs and row count of the running decode_logits (step_attn_prog_)
  float* attn_cross_ = nullptr;
  int attn_tlen_ = 0;
  int prof_t_ = 0;                        // step index used by the single-step op of the fused decoder in profile()
  struct F32Tap { const float* p; size_t count; };
  std::map<std::string, F32Tap> taps_f32_;
  float* logits_ = nullptr;               // [rows][V]
  int* forced_tokens_ = nullptr;          // [B][T] teacher-forced tokens
  int* forced_len_ = nullptr;
  float* forced_logits_ = nullptr;        // [B][T][V]
  int* h_pinned_ = nullptr;               // pinned scratch for n_done polling
  float* step_scores_ = nullptr;
  long long* dbg_buf_ = nullptr;          // FPNMT_DBG_OP timeline buffer

  // helpers
  void* dalloc(size_t bytes);
  long long* dbg_timeline(const std::string& name);
  Tensor new_act(int N, int H, int W, int C);
  Tensor rows_act(int rows, int C) { return new_act(1, 1, rows, C); }
  static Tensor chan_view(const Tensor& t, int c0, int C);
  const HostW* W(const std::string& key);
  int upload_gemm(const std::vector<float>& wt, const std::vector<float>& bias, int Cout, int K, GemmW* out);
  // Lanes share ONE device copy of the GEMM weights: every lane runs the same finalize sequence on the same host weights, so the
  // i-th upload of a follower lane is the i-th upload of the lead lane (checked by shape).  Without it 8 lanes cycle 8 x 110 MB
  // of identical weights through the 126 MB L2 and every weight tile of the latency-bound decode GEMMs comes from DRAM.
  const Engine* weight_lead_ = nullptr;
  std::vector<GemmW> gemm_log_;
  size_t gemm_log_pos_ = 0;
  int prep_conv(const std::string& kernel_key, const std::string& bias_key, const std::string& bn, float eps, GemmW* out,
                int kpad = 0);
  int prep_dense_cat(const std::vector<std::string>& names, GemmW* out);       // concat along outputs
  int prep_dense_stack(const std::vector<std::string>& names, GemmW* out);     // concat along inputs, biases summed
  int prep_vec(const std::string& key, float** out);
  int prep_bn_affine(const std::string& bn, float eps, int C, float** scale, float** shift);
  int prep_depthwise(const std::string& key, const std::string& bn, float eps, float** w, float** bias);
  int upload_f32(const std::vector<float>& v, float** out);

  int add_conv(Program& prog, const std::string& name, const Tensor& in, const GemmW& gw, int kh, int kw, int pad_t,
               int pad_l, int act, int res_mode, const Tensor* res, const Tensor& out, float* out_f32 = nullptr,
               int ld_f32 = 0);
  // skinny-row Dense (tgemm): out = act(in @ W + b [+ res]) or LayerNorm(in @ W + b + res) when gamma != nullptr
  int add_dense(Program& prog, const std::string& name, const Tensor& in, const GemmW& gw, int act, const Tensor* res,
                const Tensor& out, float* out_f32 = nullptr, int ld_f32 = 0, const float* gamma = nullptr,
                const float* beta = nullptr);
  bool stem_fused_ = false;               // the encode program starts with stem_kernel (needs 16-byte aligned images)
  bool use_stem_ = true;                  // FPNMT_STEM=0: explicit im2col + GEMM stem (always in BF16X3 mode)
  bool use_xattn_ = true;                 // FPNMT_XATTN=0: separate q2 / cross-attention / o2+LN kernels (always in BF16X3 mode)
  bool use_tgemm_ = true;                 // FPNMT_TGEMM=0 routes the decoder GEMMs through igemm + separate LayerNorm
  int build_stem_resnet_like(Program& p, const std::string& conv_key, const std::string& bn_key, float eps, Tensor* out);
  int build_resnet50(Program& p, Tensor c[3]);
  int build_mobilenetv2(Program& p, Tensor c[3]);
  int build_densenet121(Program& p, Tensor c[3]);
  int build_fpn_heads(Program& p, Tensor c[3]);
  int build_mt_encoder(Program& p);
  int build_decoder();
  int run_program(Program& p, cudaStream_t s);
  int capture(Program& p, cudaGraphExec_t* out);
  int launch_prog(Program& p, cudaGraphExec_t g, cudaStream_t s);
  int launch_graph(Program& p, cudaGraphExec_t& g, cudaStream_t s);     // capture g on first use (use_graphs), then launch
  int poll_done(const int* n_done, cudaStream_t s, bool* done);         // synchronises s; done: every image has finished
  int run_steps(Program& p, cudaGraphExec_t& g, const int* n_done, int early_stop, cudaStream_t s);
  int check_decode_entry(const char* entry, const char* fused_reason);
  int set_images(const float* images, int on_host, cudaStream_t s);
  int profile_program(Program& p, int iters, std::string& json, const char* label);
};

}  // namespace fpnmt

// The object behind the C ABI's opaque handle (api.cu, dlapi.cu).
struct fpnmt_handle {
  fpnmt::Engine* eng;                   // lane 0: every single-batch entry point runs here
  std::vector<fpnmt::Engine*> lanes;    // lanes[0] == eng; fpnmt_submit / fpnmt_collect address the others
  cudaEvent_t last_encode = nullptr;    // encoder-done event of the most recent fpnmt_submit (owned by that lane)
};

#define CHECK_H(h)                                 \
  if (!(h) || !(h)->eng) {                         \
    ::fpnmt::set_last_error("NULL handle");        \
    return FPNMT_ERR_INVALID;                      \
  }
