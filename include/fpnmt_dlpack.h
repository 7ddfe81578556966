/*
 * fpnmt_dlpack.h — DLPack-typed twins of the tensor-carrying entry points of fpnmt.h, and the in-library NCCL communicator
 * (SURVEY.md §8(b2): "tensors cross as DLManagedTensor* / raw device pointers + shape structs", `fpnmt_allgather_ids`).
 *
 * The structs below are the DLPack v0.8 C ABI (dmlc/dlpack, dlpack.h: DLDevice, DLDataType, DLTensor) restated so that this
 * header has no dependency; a host that already includes <dlpack/dlpack.h> defines FPNMT_HAVE_DLPACK_H first and the real
 * header's definitions are used.  What a `_dl` call checks before it touches memory (FPNMT_ERR_INVALID otherwise, with the
 * offending argument named in fpnmt_last_error()): device type (kDLCUDA on the engine's device for device tensors, kDLCPU /
 * kDLCUDAHost for host tensors), dtype (float32 / int32, lanes 1), rank and shape against the engine's configuration, and
 * compact row-major strides (strides == NULL or the C-contiguous strides).  `byte_offset` is honoured.
 */
#ifndef FPNMT_DLPACK_H_
#define FPNMT_DLPACK_H_

#include "fpnmt.h"

#ifdef __cplusplus
extern "C" {
#endif

#ifndef FPNMT_HAVE_DLPACK_H
#ifndef DLPACK_DLPACK_H_
typedef enum { kDLCPU = 1, kDLCUDA = 2, kDLCUDAHost = 3, kDLCUDAManaged = 13 } DLDeviceType;
typedef struct { DLDeviceType device_type; int32_t device_id; } DLDevice;
typedef enum { kDLInt = 0U, kDLUInt = 1U, kDLFloat = 2U, kDLBfloat = 4U } DLDataTypeCode;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;
typedef struct {
  void* data;
  DLDevice device;
  int32_t ndim;
  DLDataType dtype;
  int64_t* shape;
  int64_t* strides;      /* in elements; NULL = compact row-major */
  uint64_t byte_offset;
} DLTensor;
#endif
#endif

/* fpnmt_set_weight with a HOST float32 DLTensor (kDLCPU / kDLCUDAHost) in Keras layout; the library copies it
 * (utils/pipeline.py:38-48, models/retinanet.py:277-278). */
FPNMT_API int fpnmt_set_weight_dl(fpnmt_handle* h, const char* key, const DLTensor* w);
/* fpnmt_encode: images float32 [batch, S, S, 3] on the engine's GPU or on the host; memory_out (may be NULL) float32
 * [batch, n_memory, d_model] on the GPU (models/transformer.py:266-303). */
FPNMT_API int fpnmt_encode_dl(fpnmt_handle* h, const DLTensor* images, DLTensor* memory_out, void* stream);
/* fpnmt_features: five float32 NHWC outputs [batch, S/16>>i, S/16>>i, d_model] on the GPU (models/retinanet.py:306-307). */
FPNMT_API int fpnmt_features_dl(fpnmt_handle* h, const DLTensor* images, DLTensor* const out5[5], void* stream);
/* fpnmt_decode_logits: memory float32 [batch, n_memory, d_model] or NULL, tokens int32 [batch, t], logits_out float32
 * [batch, t, vocab], all on the GPU (models/transformer.py:359-374). */
FPNMT_API int fpnmt_decode_logits_dl(fpnmt_handle* h, const DLTensor* memory, const DLTensor* tokens, DLTensor* logits_out,
                                     void* stream);
/* Decoder.call(x, enc_output, training=False, look_ahead_mask, padding_mask) (models/transformer.py:321-341): the hidden
 * states of the last decoder layer, before final_layer, for teacher-forced tokens.  memory / tokens as above;
 * hidden_out float32 [batch, t, d_model] on the GPU.  (Raw-pointer twin: fpnmt_decode_hidden in fpnmt.h.) */
FPNMT_API int fpnmt_decode_hidden_dl(fpnmt_handle* h, const DLTensor* memory, const DLTensor* tokens, DLTensor* hidden_out,
                                     void* stream);
/* The attention-weights dict of Decoder.call (models/transformer.py:337-338): memory / tokens as above; self_out float32
 * [num_layers, batch, heads, t, t], cross_out float32 [num_layers, batch, heads, t, n_memory], on the GPU; either may be
 * NULL, not both.  (Raw-pointer twin: fpnmt_decode_attention in fpnmt.h.) */
FPNMT_API int fpnmt_decode_attention_dl(fpnmt_handle* h, const DLTensor* memory, const DLTensor* tokens, DLTensor* self_out,
                                        DLTensor* cross_out, void* stream);
/* fpnmt_generate (utils/pipeline.py:82-154): images as fpnmt_encode_dl; out_ids int32 [batch, max_len], out_len int32 [batch],
 * both on the GPU or both on the host (host outputs synchronise the stream); step_scores float32 [max_len, batch] on the GPU
 * or NULL. */
FPNMT_API int fpnmt_generate_dl(fpnmt_handle* h, const DLTensor* images, DLTensor* out_ids, DLTensor* out_len, int early_stop,
                                DLTensor* step_scores, void* stream);
/* fpnmt_sample: images as fpnmt_encode_dl, or NULL for the memory of the last encode; out_ids int32 [batch, beam, max_len],
 * out_len int32 [batch, beam], out_logprob float32 [batch, beam] or NULL, all on the GPU or all on the host (host outputs
 * synchronise the stream). */
FPNMT_API int fpnmt_sample_dl(fpnmt_handle* h, const DLTensor* images, const fpnmt_sampling* sampling, DLTensor* out_ids,
                              DLTensor* out_len, DLTensor* out_logprob, int early_stop, void* stream);
/* fpnmt_score: images as fpnmt_encode_dl, or NULL for the memory of the last encode; ids int32 [batch, beam, t] and lens int32
 * [batch, beam] on the GPU (t = ids' last dimension); out_logprob float32 [batch, beam] and out_token_logprob float32
 * [batch, beam, t] or NULL, both on the GPU or both on the host (host outputs synchronise the stream). */
FPNMT_API int fpnmt_score_dl(fpnmt_handle* h, const DLTensor* images, const DLTensor* ids, const DLTensor* lens,
                             DLTensor* out_logprob, DLTensor* out_token_logprob, void* stream);
/* fpnmt_beam_search: images as fpnmt_encode_dl, or NULL for the memory of the last encode; out_ids int32 [batch, beam,
 * max_len], out_len int32 [batch, beam], out_logprob float32 [batch, beam] or NULL, all on the GPU or all on the host (host
 * outputs synchronise the stream). */
FPNMT_API int fpnmt_beam_search_dl(fpnmt_handle* h, const DLTensor* images, float length_penalty, DLTensor* out_ids,
                                   DLTensor* out_len, DLTensor* out_logprob, int early_stop, void* stream);
/* fpnmt_beam_search_diverse: tensors and checks as fpnmt_beam_search_dl. */
FPNMT_API int fpnmt_beam_search_diverse_dl(fpnmt_handle* h, const DLTensor* images, int beam_groups, float diversity,
                                           float length_penalty, DLTensor* out_ids, DLTensor* out_len, DLTensor* out_logprob,
                                           int early_stop, void* stream);
/* fpnmt_sample_prefix / fpnmt_beam_search_prefix: prefix_ids int32 [batch, p] (p from its shape) and prefix_len int32 [batch],
 * both on the GPU; images and outputs as fpnmt_sample_dl / fpnmt_beam_search_dl. */
FPNMT_API int fpnmt_sample_prefix_dl(fpnmt_handle* h, const DLTensor* images, const DLTensor* prefix_ids, const DLTensor* prefix_len,
                                     const fpnmt_sampling* sampling, DLTensor* out_ids, DLTensor* out_len, DLTensor* out_logprob,
                                     int early_stop, void* stream);
FPNMT_API int fpnmt_beam_search_prefix_dl(fpnmt_handle* h, const DLTensor* images, const DLTensor* prefix_ids,
                                          const DLTensor* prefix_len, int beam_groups, float diversity, float length_penalty,
                                          DLTensor* out_ids, DLTensor* out_len, DLTensor* out_logprob, int early_stop, void* stream);
/* fpnmt_sample_constrained / fpnmt_beam_search_constrained: prefix_ids / prefix_len as fpnmt_sample_prefix_dl, or both NULL
 * for an unprompted call; constraints a host struct; images and outputs as fpnmt_sample_dl / fpnmt_beam_search_dl. */
FPNMT_API int fpnmt_sample_constrained_dl(fpnmt_handle* h, const DLTensor* images, const DLTensor* prefix_ids,
                                          const DLTensor* prefix_len, const fpnmt_sampling* sampling,
                                          const fpnmt_constraints* constraints, DLTensor* out_ids, DLTensor* out_len,
                                          DLTensor* out_logprob, int early_stop, void* stream);
FPNMT_API int fpnmt_beam_search_constrained_dl(fpnmt_handle* h, const DLTensor* images, const DLTensor* prefix_ids,
                                               const DLTensor* prefix_len, int beam_groups, float diversity, float length_penalty,
                                               const fpnmt_constraints* constraints, DLTensor* out_ids, DLTensor* out_len,
                                               DLTensor* out_logprob, int early_stop, void* stream);

/* ---- in-library communicator: the ONE collective of the path (SURVEY §8e) -------------------------------------------
 * Image batches shard across the GPUs of a box; the only exchange is the all-gather of the caption ids.  The library opens
 * NCCL itself (dlopen of libnccl.so.2: the copy already loaded into the process, e.g. PyTorch's, else the system one), so a
 * host without torch.distributed can run the multi-GPU path.  Bootstrap as NCCL does: rank 0 calls fpnmt_comm_unique_id and
 * hands the 128 bytes to the other ranks over any channel; every rank then calls fpnmt_comm_create (collective). */
typedef struct fpnmt_comm fpnmt_comm;
#define FPNMT_UNIQUE_ID_BYTES 128
FPNMT_API int fpnmt_comm_unique_id(uint8_t id_out[FPNMT_UNIQUE_ID_BYTES]);
FPNMT_API int fpnmt_comm_create(int world, int rank, const uint8_t id[FPNMT_UNIQUE_ID_BYTES], int device, fpnmt_comm** out);
FPNMT_API int fpnmt_comm_destroy(fpnmt_comm* c);
/* all_ids[r * batch + b, :] = rank r's local_ids[b, :] (rank-major), likewise the lengths: DEVICE int32 local_ids
 * [batch, max_len], local_len [batch] -> all_ids [world * batch, max_len], all_len [world * batch]; one grouped NCCL
 * all-gather enqueued on `stream` (no host synchronisation).  local_len / all_len may both be NULL. */
FPNMT_API int fpnmt_allgather_ids(fpnmt_comm* c, const int32_t* local_ids, const int32_t* local_len, int batch, int max_len,
                                  int32_t* all_ids, int32_t* all_len, void* stream);
FPNMT_API int fpnmt_allgather_ids_dl(fpnmt_comm* c, const DLTensor* local_ids, const DLTensor* local_len, DLTensor* all_ids,
                                     DLTensor* all_len, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FPNMT_DLPACK_H_ */
