// DLPack-typed twins of the tensor entry points and the in-library NCCL communicator (include/fpnmt_dlpack.h).
// NCCL is opened at run time (dlopen) so that libfpnmt.so has no link-time dependency on it and uses the copy that is
// already in the process when there is one (PyTorch's bundled libnccl); only <nccl.h>'s public types are used.
#include <dlfcn.h>
#include <nccl.h>

#include <mutex>
#include <string>

#include "../../include/fpnmt_dlpack.h"
#include "engine.cuh"

struct fpnmt_handle {          // same layout as in api.cu
  fpnmt::Engine* eng;
  std::vector<fpnmt::Engine*> lanes;
  cudaEvent_t last_encode = nullptr;
};

namespace fpnmt {

static int dl_fail(const std::string& m) {
  set_last_error(m);
  return FPNMT_ERR_INVALID;
}

// Validates one DLTensor argument; on success *ptr = data + byte_offset and *on_host says where it lives.
static int dl_check(const char* what, const DLTensor* t, int code, int device, bool allow_host, bool allow_device,
                    std::initializer_list<int64_t> shape, void** ptr, int* on_host) {
  const std::string w = what;
  if (!t || !t->data) return dl_fail(w + ": NULL tensor");
  const bool host = t->device.device_type == kDLCPU || t->device.device_type == kDLCUDAHost;
  const bool dev = t->device.device_type == kDLCUDA || t->device.device_type == kDLCUDAManaged;
  if (!host && !dev) return dl_fail(w + ": unsupported DLPack device type " + std::to_string((int)t->device.device_type));
  if (host && !allow_host) return dl_fail(w + ": must be a CUDA tensor");
  if (dev && !allow_device) return dl_fail(w + ": must be a host tensor");
  if (dev && t->device.device_id != device)
    return dl_fail(w + ": lives on cuda:" + std::to_string(t->device.device_id) + ", the engine on cuda:" + std::to_string(device));
  if (t->dtype.code != code || t->dtype.bits != 32 || t->dtype.lanes != 1)
    return dl_fail(w + ": dtype must be " + (code == kDLFloat ? "float32" : "int32"));
  if (t->ndim != (int)shape.size()) return dl_fail(w + ": rank " + std::to_string(t->ndim) + ", expected " + std::to_string(shape.size()));
  int i = 0;
  for (int64_t d : shape) {
    if (d >= 0 && t->shape[i] != d)
      return dl_fail(w + ": dimension " + std::to_string(i) + " is " + std::to_string(t->shape[i]) + ", expected " + std::to_string(d));
    ++i;
  }
  if (t->strides) {
    int64_t st = 1;
    for (int k = t->ndim - 1; k >= 0; --k) {
      if (t->shape[k] != 1 && t->strides[k] != st) return dl_fail(w + ": must be compact row-major (C-contiguous)");
      st *= t->shape[k];
    }
  }
  *ptr = (char*)t->data + t->byte_offset;
  if (on_host) *on_host = host ? 1 : 0;
  return 0;
}

// ---- NCCL through dlopen ------------------------------------------------------------------------------------------
struct Nccl {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static Nccl g_nccl;
static std::mutex g_nccl_mu;

static int nccl_open() {
  std::lock_guard<std::mutex> lock(g_nccl_mu);
  if (g_nccl.lib) return 0;
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);     // the copy already in the process (PyTorch's), if any
  if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) {
    set_last_error(std::string("fpnmt_comm: cannot open libnccl.so.2: ") + dlerror());
    return FPNMT_ERR_CUDA;
  }
  Nccl n;
  n.lib = lib;
#define SYM(field, name)                                              \
  *(void**)(&n.field) = dlsym(lib, name);                             \
  if (!n.field) {                                                     \
    set_last_error(std::string("fpnmt_comm: libnccl lacks ") + name); \
    return FPNMT_ERR_CUDA;                                            \
  }
  SYM(GetUniqueId, "ncclGetUniqueId");
  SYM(CommInitRank, "ncclCommInitRank");
  SYM(CommDestroy, "ncclCommDestroy");
  SYM(AllGather, "ncclAllGather");
  SYM(GroupStart, "ncclGroupStart");
  SYM(GroupEnd, "ncclGroupEnd");
  SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
  g_nccl = n;
  return 0;
}
static int nccl_fail(const char* what, ncclResult_t r) {
  set_last_error(std::string("nccl: ") + what + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"));
  return FPNMT_ERR_CUDA;
}
#define NCCL_OK(call, what)                      \
  do {                                           \
    ncclResult_t r_ = (call);                    \
    if (r_ != ncclSuccess) return nccl_fail(what, r_); \
  } while (0)

}  // namespace fpnmt

using namespace fpnmt;

struct fpnmt_comm {
  ncclComm_t comm = nullptr;
  int world = 1, rank = 0, device = 0;
};

static_assert(sizeof(ncclUniqueId) == FPNMT_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");

#define CHECK_HDL(h)                               \
  if (!(h) || !(h)->eng) {                         \
    set_last_error("NULL handle");                 \
    return FPNMT_ERR_INVALID;                      \
  }

extern "C" {

FPNMT_API int fpnmt_set_weight_dl(fpnmt_handle* h, const char* key, const DLTensor* w) {
  CHECK_HDL(h);
  if (!key || !w || !w->data) return dl_fail("set_weight_dl: NULL key / tensor");
  if (w->ndim < 1 || w->ndim > 4) return dl_fail(std::string("set_weight_dl(") + key + "): rank must be 1..4");
  void* p = nullptr;
  std::initializer_list<int64_t> any1 = {-1}, any2 = {-1, -1}, any3 = {-1, -1, -1}, any4 = {-1, -1, -1, -1};
  const auto& shp = w->ndim == 1 ? any1 : w->ndim == 2 ? any2 : w->ndim == 3 ? any3 : any4;
  int rc = dl_check((std::string("set_weight_dl(") + key + ")").c_str(), w, kDLFloat, 0, true, false, shp, &p, nullptr);
  if (rc) return rc;
  return fpnmt_set_weight(h, key, (const float*)p, w->shape, w->ndim);
}

FPNMT_API int fpnmt_encode_dl(fpnmt_handle* h, const DLTensor* images, DLTensor* memory_out, void* stream) {
  CHECK_HDL(h);
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size, nm = (int64_t)(S / 128) * (S / 128);
  void *pi = nullptr, *pm = nullptr;
  int on_host = 0;
  int rc = dl_check("encode_dl: images", images, kDLFloat, h->eng->device(), true, true, {c.batch, S, S, 3}, &pi, &on_host);
  if (rc) return rc;
  if (memory_out) {
    rc = dl_check("encode_dl: memory_out", memory_out, kDLFloat, h->eng->device(), false, true, {c.batch, nm, c.d_model}, &pm, nullptr);
    if (rc) return rc;
  }
  return fpnmt_encode(h, (const float*)pi, on_host, (float*)pm, stream);
}

FPNMT_API int fpnmt_features_dl(fpnmt_handle* h, const DLTensor* images, DLTensor* const out5[5], void* stream) {
  CHECK_HDL(h);
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size;
  void* pi = nullptr;
  int on_host = 0;
  int rc = dl_check("features_dl: images", images, kDLFloat, h->eng->device(), true, true, {c.batch, S, S, 3}, &pi, &on_host);
  if (rc) return rc;
  if (!out5) return dl_fail("features_dl: out5 is NULL");
  float* outs[5];
  for (int i = 0; i < 5; ++i) {
    const int64_t side = (S / 16) >> i;
    void* po = nullptr;
    rc = dl_check(("features_dl: out5[" + std::to_string(i) + "]").c_str(), out5[i], kDLFloat, h->eng->device(), false, true,
                  {c.batch, side, side, c.d_model}, &po, nullptr);
    if (rc) return rc;
    outs[i] = (float*)po;
  }
  return fpnmt_features(h, (const float*)pi, on_host, outs, stream);
}

static int forced_args(fpnmt_handle* h, const char* fn, const DLTensor* memory, const DLTensor* tokens, void** pm, void** pt, int* t) {
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size, nm = (int64_t)(S / 128) * (S / 128);
  const std::string f = fn;
  *pm = nullptr;
  if (memory) {
    int rc = dl_check((f + ": memory").c_str(), memory, kDLFloat, h->eng->device(), false, true, {c.batch, nm, c.d_model}, pm, nullptr);
    if (rc) return rc;
  }
  int rc = dl_check((f + ": tokens").c_str(), tokens, kDLInt, h->eng->device(), false, true, {c.batch, -1}, pt, nullptr);
  if (rc) return rc;
  *t = (int)tokens->shape[1];
  return 0;
}

FPNMT_API int fpnmt_decode_logits_dl(fpnmt_handle* h, const DLTensor* memory, const DLTensor* tokens, DLTensor* logits_out,
                                     void* stream) {
  CHECK_HDL(h);
  void *pm, *pt, *po = nullptr;
  int t = 0;
  int rc = forced_args(h, "decode_logits_dl", memory, tokens, &pm, &pt, &t);
  if (rc) return rc;
  const fpnmt_config& c = h->eng->config();
  rc = dl_check("decode_logits_dl: logits_out", logits_out, kDLFloat, h->eng->device(), false, true, {c.batch, t, c.vocab}, &po, nullptr);
  if (rc) return rc;
  return fpnmt_decode_logits(h, (const float*)pm, (const int32_t*)pt, t, (float*)po, stream);
}

FPNMT_API int fpnmt_decode_hidden_dl(fpnmt_handle* h, const DLTensor* memory, const DLTensor* tokens, DLTensor* hidden_out,
                                     void* stream) {
  CHECK_HDL(h);
  void *pm, *pt, *po = nullptr;
  int t = 0;
  int rc = forced_args(h, "decode_hidden_dl", memory, tokens, &pm, &pt, &t);
  if (rc) return rc;
  const fpnmt_config& c = h->eng->config();
  rc = dl_check("decode_hidden_dl: hidden_out", hidden_out, kDLFloat, h->eng->device(), false, true, {c.batch, t, c.d_model}, &po, nullptr);
  if (rc) return rc;
  return fpnmt_decode_hidden(h, (const float*)pm, (const int32_t*)pt, t, (float*)po, stream);
}

FPNMT_API int fpnmt_decode_attention_dl(fpnmt_handle* h, const DLTensor* memory, const DLTensor* tokens, DLTensor* self_out,
                                        DLTensor* cross_out, void* stream) {
  CHECK_HDL(h);
  void *pm, *pt, *ps = nullptr, *pc = nullptr;
  int t = 0;
  int rc = forced_args(h, "decode_attention_dl", memory, tokens, &pm, &pt, &t);
  if (rc) return rc;
  const fpnmt_config& c = h->eng->config();
  const int64_t nm = (int64_t)(c.image_size / 128) * (c.image_size / 128);
  if (!self_out && !cross_out) return dl_fail("decode_attention_dl: self_out and cross_out are both NULL");
  if (self_out) {
    rc = dl_check("decode_attention_dl: self_out", self_out, kDLFloat, h->eng->device(), false, true,
                  {c.num_layers, c.batch, c.num_heads, t, t}, &ps, nullptr);
    if (rc) return rc;
  }
  if (cross_out) {
    rc = dl_check("decode_attention_dl: cross_out", cross_out, kDLFloat, h->eng->device(), false, true,
                  {c.num_layers, c.batch, c.num_heads, t, nm}, &pc, nullptr);
    if (rc) return rc;
  }
  return fpnmt_decode_attention(h, (const float*)pm, (const int32_t*)pt, t, (float*)ps, (float*)pc, stream);
}

FPNMT_API int fpnmt_generate_dl(fpnmt_handle* h, const DLTensor* images, DLTensor* out_ids, DLTensor* out_len, int early_stop,
                                DLTensor* step_scores, void* stream) {
  CHECK_HDL(h);
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size;
  void *pi = nullptr, *pids = nullptr, *plen = nullptr, *psc = nullptr;
  int img_host = 0, ids_host = 0, len_host = 0;
  int rc = dl_check("generate_dl: images", images, kDLFloat, h->eng->device(), true, true, {c.batch, S, S, 3}, &pi, &img_host);
  if (rc) return rc;
  rc = dl_check("generate_dl: out_ids", out_ids, kDLInt, h->eng->device(), true, true, {c.batch, c.max_len}, &pids, &ids_host);
  if (rc) return rc;
  rc = dl_check("generate_dl: out_len", out_len, kDLInt, h->eng->device(), true, true, {c.batch}, &plen, &len_host);
  if (rc) return rc;
  if (ids_host != len_host) return dl_fail("generate_dl: out_ids and out_len must both be host or both be device tensors");
  if (step_scores) {
    rc = dl_check("generate_dl: step_scores", step_scores, kDLFloat, h->eng->device(), false, true, {c.max_len, c.batch}, &psc, nullptr);
    if (rc) return rc;
  }
  return fpnmt_generate(h, (const float*)pi, img_host, (int32_t*)pids, (int32_t*)plen, ids_host, early_stop, (float*)psc, stream);
}

FPNMT_API int fpnmt_sample_dl(fpnmt_handle* h, const DLTensor* images, const fpnmt_sampling* sampling, DLTensor* out_ids,
                              DLTensor* out_len, DLTensor* out_logprob, int early_stop, void* stream) {
  CHECK_HDL(h);
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size;
  void *pi = nullptr, *pids = nullptr, *plen = nullptr, *plp = nullptr;
  int img_host = 0, ids_host = 0, len_host = 0, lp_host = 0;
  int rc = 0;
  if (images) {
    rc = dl_check("sample_dl: images", images, kDLFloat, h->eng->device(), true, true, {c.batch, S, S, 3}, &pi, &img_host);
    if (rc) return rc;
  }
  rc = dl_check("sample_dl: out_ids", out_ids, kDLInt, h->eng->device(), true, true, {c.batch, c.beam, c.max_len}, &pids, &ids_host);
  if (rc) return rc;
  rc = dl_check("sample_dl: out_len", out_len, kDLInt, h->eng->device(), true, true, {c.batch, c.beam}, &plen, &len_host);
  if (rc) return rc;
  if (ids_host != len_host) return dl_fail("sample_dl: out_ids and out_len must both be host or both be device tensors");
  if (out_logprob) {
    rc = dl_check("sample_dl: out_logprob", out_logprob, kDLFloat, h->eng->device(), true, true, {c.batch, c.beam}, &plp, &lp_host);
    if (rc) return rc;
    if (lp_host != ids_host) return dl_fail("sample_dl: out_logprob must live where out_ids does");
  }
  return fpnmt_sample(h, (const float*)pi, img_host, sampling, (int32_t*)pids, (int32_t*)plen, (float*)plp, ids_host, early_stop,
                      stream);
}

FPNMT_API int fpnmt_beam_search_dl(fpnmt_handle* h, const DLTensor* images, float length_penalty, DLTensor* out_ids,
                                   DLTensor* out_len, DLTensor* out_logprob, int early_stop, void* stream) {
  CHECK_HDL(h);
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size;
  void *pi = nullptr, *pids = nullptr, *plen = nullptr, *plp = nullptr;
  int img_host = 0, ids_host = 0, len_host = 0, lp_host = 0;
  int rc = 0;
  if (images) {
    rc = dl_check("beam_search_dl: images", images, kDLFloat, h->eng->device(), true, true, {c.batch, S, S, 3}, &pi, &img_host);
    if (rc) return rc;
  }
  rc = dl_check("beam_search_dl: out_ids", out_ids, kDLInt, h->eng->device(), true, true, {c.batch, c.beam, c.max_len}, &pids,
                &ids_host);
  if (rc) return rc;
  rc = dl_check("beam_search_dl: out_len", out_len, kDLInt, h->eng->device(), true, true, {c.batch, c.beam}, &plen, &len_host);
  if (rc) return rc;
  if (ids_host != len_host) return dl_fail("beam_search_dl: out_ids and out_len must both be host or both be device tensors");
  if (out_logprob) {
    rc = dl_check("beam_search_dl: out_logprob", out_logprob, kDLFloat, h->eng->device(), true, true, {c.batch, c.beam}, &plp,
                  &lp_host);
    if (rc) return rc;
    if (lp_host != ids_host) return dl_fail("beam_search_dl: out_logprob must live where out_ids does");
  }
  return fpnmt_beam_search(h, (const float*)pi, img_host, length_penalty, (int32_t*)pids, (int32_t*)plen, (float*)plp, ids_host,
                           early_stop, stream);
}

FPNMT_API int fpnmt_score_dl(fpnmt_handle* h, const DLTensor* images, const DLTensor* ids, const DLTensor* lens,
                             DLTensor* out_logprob, DLTensor* out_token_logprob, void* stream) {
  CHECK_HDL(h);
  const fpnmt_config& c = h->eng->config();
  const int64_t S = c.image_size;
  void *pi = nullptr, *pids = nullptr, *plen = nullptr, *plp = nullptr, *ptok = nullptr;
  int img_host = 0, lp_host = 0, tok_host = 0;
  int rc = 0;
  if (images) {
    rc = dl_check("score_dl: images", images, kDLFloat, h->eng->device(), true, true, {c.batch, S, S, 3}, &pi, &img_host);
    if (rc) return rc;
  }
  rc = dl_check("score_dl: ids", ids, kDLInt, h->eng->device(), false, true, {c.batch, c.beam, -1}, &pids, nullptr);
  if (rc) return rc;
  const int64_t t = ids->shape[2];
  if (t < 1 || t > c.max_len) return dl_fail("score_dl: ids must hold 1 .. max_len positions per caption");
  rc = dl_check("score_dl: lens", lens, kDLInt, h->eng->device(), false, true, {c.batch, c.beam}, &plen, nullptr);
  if (rc) return rc;
  rc = dl_check("score_dl: out_logprob", out_logprob, kDLFloat, h->eng->device(), true, true, {c.batch, c.beam}, &plp, &lp_host);
  if (rc) return rc;
  if (out_token_logprob) {
    rc = dl_check("score_dl: out_token_logprob", out_token_logprob, kDLFloat, h->eng->device(), true, true, {c.batch, c.beam, t}, &ptok,
                  &tok_host);
    if (rc) return rc;
    if (tok_host != lp_host) return dl_fail("score_dl: out_token_logprob must live where out_logprob does");
  }
  return fpnmt_score(h, (const float*)pi, img_host, (const int32_t*)pids, (const int32_t*)plen, (int)t, (float*)plp, (float*)ptok,
                     lp_host, stream);
}

// ---- communicator ---------------------------------------------------------------------------------------------------
FPNMT_API int fpnmt_comm_unique_id(uint8_t id_out[FPNMT_UNIQUE_ID_BYTES]) {
  if (!id_out) return dl_fail("comm_unique_id: NULL");
  int rc = nccl_open();
  if (rc) return rc;
  ncclUniqueId id;
  NCCL_OK(g_nccl.GetUniqueId(&id), "ncclGetUniqueId");
  memcpy(id_out, &id, sizeof id);
  return FPNMT_OK;
}

FPNMT_API int fpnmt_comm_create(int world, int rank, const uint8_t id[FPNMT_UNIQUE_ID_BYTES], int device, fpnmt_comm** out) {
  if (!out || !id || world < 1 || rank < 0 || rank >= world) return dl_fail("comm_create: bad world / rank / id");
  int rc = nccl_open();
  if (rc) return rc;
  FPNMT_CUDA_OK(cudaSetDevice(device));
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof uid);
  fpnmt_comm* c = new fpnmt_comm();
  c->world = world;
  c->rank = rank;
  c->device = device;
  ncclResult_t r = g_nccl.CommInitRank(&c->comm, world, uid, rank);
  if (r != ncclSuccess) {
    delete c;
    return nccl_fail("ncclCommInitRank", r);
  }
  *out = c;
  return FPNMT_OK;
}

FPNMT_API int fpnmt_comm_destroy(fpnmt_comm* c) {
  if (!c) return FPNMT_OK;
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  delete c;
  return FPNMT_OK;
}

FPNMT_API int fpnmt_allgather_ids(fpnmt_comm* c, const int32_t* local_ids, const int32_t* local_len, int batch, int max_len,
                                  int32_t* all_ids, int32_t* all_len, void* stream) {
  if (!c || !c->comm) return dl_fail("allgather_ids: NULL communicator");
  if (!local_ids || !all_ids || batch < 1 || max_len < 1 || (!local_len) != (!all_len))
    return dl_fail("allgather_ids: bad arguments");
  FPNMT_CUDA_OK(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  NCCL_OK(g_nccl.GroupStart(), "ncclGroupStart");
  NCCL_OK(g_nccl.AllGather(local_ids, all_ids, (size_t)batch * max_len, ncclInt32, c->comm, s), "ncclAllGather(ids)");
  if (local_len) NCCL_OK(g_nccl.AllGather(local_len, all_len, (size_t)batch, ncclInt32, c->comm, s), "ncclAllGather(len)");
  NCCL_OK(g_nccl.GroupEnd(), "ncclGroupEnd");
  return FPNMT_OK;
}

FPNMT_API int fpnmt_allgather_ids_dl(fpnmt_comm* c, const DLTensor* local_ids, const DLTensor* local_len, DLTensor* all_ids,
                                     DLTensor* all_len, void* stream) {
  if (!c || !c->comm) return dl_fail("allgather_ids_dl: NULL communicator");
  void *pi = nullptr, *pl = nullptr, *ai = nullptr, *al = nullptr;
  int rc = dl_check("allgather_ids_dl: local_ids", local_ids, kDLInt, c->device, false, true, {-1, -1}, &pi, nullptr);
  if (rc) return rc;
  const int64_t b = local_ids->shape[0], t = local_ids->shape[1];
  rc = dl_check("allgather_ids_dl: all_ids", all_ids, kDLInt, c->device, false, true, {b * c->world, t}, &ai, nullptr);
  if (rc) return rc;
  if ((!local_len) != (!all_len)) return dl_fail("allgather_ids_dl: local_len and all_len go together");
  if (local_len) {
    rc = dl_check("allgather_ids_dl: local_len", local_len, kDLInt, c->device, false, true, {b}, &pl, nullptr);
    if (rc) return rc;
    rc = dl_check("allgather_ids_dl: all_len", all_len, kDLInt, c->device, false, true, {b * c->world}, &al, nullptr);
    if (rc) return rc;
  }
  return fpnmt_allgather_ids(c, (const int32_t*)pi, (const int32_t*)pl, (int)b, (int)t, (int32_t*)ai, (int32_t*)al, stream);
}

}  // extern "C"
