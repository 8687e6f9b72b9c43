/*
 * vqa_b200.h -- C ABI of libvqa_b200.so: the sm_100a engine behind the reference's
 * VQAModel.forward / VQAInference.predict hot path.
 *
 * The reference (zeyadmohamedabdo/Visual-Question-Answering-VQA-system) is pure Python on
 * PyTorch; it has no FFI of its own.  This header is therefore the boundary a maintainer
 * would bind with ctypes from models/vqa_model.py:243-311 (VQAModel.forward) and
 * api/inference.py:195-323 (predict / predict_batch); INTEGRATION.md shows the stub.
 * Each op kind below names the reference lines it replaces.
 *
 * Conventions
 *   - plain C types only: device pointers as uint64_t, sizes as int32_t, cudaStream_t as void*.
 *   - the caller owns every buffer (weights arena, workspace, inputs, outputs); the library
 *     never allocates or frees device memory and never synchronises the device.  Work is
 *     ordered on the stream it is given: ops marked for lane 1 run on a non-blocking side
 *     stream the plan owns, forked from and joined back into the caller's stream with events
 *     inside the same call, so a run can still be captured in a CUDA graph.
 *   - a plan is bound to one device (vqa_plan_create / vqa_plan_run select it and restore the
 *     caller's current device) and is not re-entrant: it owns its fork / join events and its
 *     workspace, so two runs of one plan must be ordered by the caller (same stream or events)
 *     and a second host thread enqueueing the same plan concurrently gets VQA_E_INVALID.
 *     Independent batches run on separate plans ("slots" in the Python engine).
 *   - every entry point returns 0 on success or a negative VQA_E_* code; vqa_last_error()
 *     returns a thread-local human-readable message.  Nothing aborts the process
 *     (api/main.py:213-221 expects exceptions it can stringify).
 *   - a "plan" is an immutable list of ops (kernel launches) with their tensor maps encoded
 *     once; the Python host builds the list from the model's state_dict (program.py).
 *   - a pointer field whose top bit is set is an external slot: (VQA_EXT_TAG | k) resolves to
 *     ext[k] of vqa_plan_run (model inputs / outputs that change per call).
 */
#ifndef VQA_B200_H_
#define VQA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQA_ABI_VERSION 10

#define VQA_OK            0
#define VQA_E_INVALID    -1   /* bad argument / unsupported shape */
#define VQA_E_CUDA       -2   /* CUDA runtime or driver error (message has the detail) */
#define VQA_E_ALIGN      -3   /* misaligned pointer or stride */
#define VQA_E_UNSUPPORTED -4  /* device is not sm_100 */

#define VQA_EXT_TAG   0x8000000000000000ull
#define VQA_MAX_TAPS   16
#define VQA_MAX_GROUPS 12
#define VQA_LANE_JOIN  4
#define VQA_OP_NI      160
#define VQA_OP_NP     16
#define VQA_OP_NF     4

/* Op kinds.  Field layouts (indices into VqaOp.i / .p / .f) are listed in program.py
 * (FIELDS) and mirrored by the *_I / *_P enums in csrc/op_fields.h (generated); vqa_op_num_fields() lets the
 * host verify both sides agree. */
enum VqaOpKind {
  VQA_OP_INGEST        = 1,  /* NCHW fp32 (models/vqa_model.py:243-258) or uint8 HWC + normalise
                                (data/preprocess.py:117-121) -> phase-packed bf16 stem input */
  VQA_OP_GEMM          = 2,  /* tap-shifted GEMM on tcgen05: every Conv2d+BN(+ReLU)(+residual)
                                (models/cnn_backbone.py:164-197,349-352) and every nn.Linear */
  VQA_OP_MAXPOOL       = 3,  /* MaxPool2d 3x3/2 p1 (models/cnn_backbone.py:353) */
  VQA_OP_SE_SQUEEZE    = 4,  /* adaptive_avg_pool2d partial sums (models/attention_modules.py:116) */
  VQA_OP_SE_EXCITE     = 5,  /* fc1-ReLU-fc2-sigmoid (models/attention_modules.py:123-126) */
  VQA_OP_SPATIAL_MAP   = 6,  /* channel max/mean, 7x7 conv, sigmoid (models/attention_modules.py:223-240) */
  VQA_OP_SCALE_RELAYOUT= 7,  /* x*scale[c]*map[pixel] (attention_modules.py:133-136,243) + layout for next stage */
  VQA_OP_EMBED         = 8,  /* embedding*sqrt(D)+PE (models/text_encoder.py:504-512) */
  VQA_OP_LAYERNORM     = 9,  /* nn.LayerNorm(256) (+ projector row compaction and position add, models/fusion.py:98-112) */
  VQA_OP_SELF_ATTN     = 10, /* masked softmax(QK^T/sqrt(d))V (models/text_encoder.py:229-259) */
  VQA_OP_CROSS_ATTN    = 11, /* softmax(QK^T/sqrt(d))V over 49 image tokens (models/cross_attention.py:164-197) */
  VQA_OP_POOL_GATE_LN  = 12, /* masked mean pools, gate, output_norm (models/fusion.py:299-326) */
  VQA_OP_SOFTMAX_TOPK  = 13, /* softmax + top-k (models/vqa_model.py:336-337, api/inference.py:231-234) */
  VQA_OP_MASK_PREP     = 14, /* attention_mask (int64 | fp32 | absent) -> int32 */
  VQA_OP_GRID_TO_NCHW  = 15, /* padded-flat bf16 grid -> NCHW fp32 (aux['image_features'], models/vqa_model.py:301-309) */
  VQA_OP_COPY_ROWS     = 16, /* fp32 [rows, cols] copy between leading dimensions (logits whose num_answers is not a multiple of 4) */
  VQA_OP_STAGE_TAIL    = 17, /* fused stage tail: SE squeeze+excite, spatial attention, scale, relayout (attention_modules.py:91-136,198-243) */
  VQA_OP_SPLIT_TF32    = 18, /* fp32 -> [tf32 hi | tf32 lo] A operand of the 3xTF32 Linears of the tf32 precision mode */
  VQA_OP_STEM_POOL     = 19, /* fused stem: conv7x7/2 + BN + ReLU + MaxPool2d 3x3/2 (models/cnn_backbone.py:349-354), two conv rows
                                per N = 128 MMA, vertical max carried in registers along runs of pooled rows */
  VQA_OP_MLP_CHAIN     = 20, /* fused post-attention chain of a transformer layer: W_o + residual, LayerNorm, FFN, residual and the next
                                block's LayerNorm + projection (models/text_encoder.py:373-399, models/cross_attention.py:265-299) */
  VQA_OP_ATTN_CHUNKED  = 21, /* masked softmax(QK^T/sqrt(d))V with the keys streamed in chunks of 64 (online softmax): the self-
                                (models/text_encoder.py:229-259) and cross-attention (models/cross_attention.py:164-197) of
                                questions longer than 64 tokens, up to 512 queries and 512 keys */
  VQA_OP_KIND_MAX      = 22
};

typedef struct VqaOp {
  int32_t  kind;
  int32_t  lane;            /* bit 0: 0 = caller's stream, 1 = the plan's side stream (forked at its first op, joined at
                               the end of the run); VQA_LANE_JOIN: wait for the other lane's work issued so far */
  int32_t  i[VQA_OP_NI];
  float    f[VQA_OP_NF];
  uint64_t p[VQA_OP_NP];
} VqaOp;

typedef struct VqaPlan VqaPlan;

/* library / device */
int         vqa_abi_version(void);
const char* vqa_last_error(void);
int         vqa_device_check(int device);            /* 0 iff `device` is compute capability 10.x */
int         vqa_op_num_fields(int kind, int* n_i, int* n_p, int* n_f);

/* plans */
int  vqa_plan_create(const VqaOp* ops, int32_t n_ops, int32_t device, VqaPlan** out);
int  vqa_plan_run(const VqaPlan* plan, const uint64_t* ext, int32_t n_ext, void* stream);
int  vqa_plan_run_range(const VqaPlan* plan, int32_t first, int32_t last,
                        const uint64_t* ext, int32_t n_ext, void* stream);
int  vqa_plan_num_launches(const VqaPlan* plan);      /* kernels one vqa_plan_run launches */
int  vqa_plan_op_kernel_name(const VqaPlan* plan, int32_t op, char* buf, int32_t buflen);
void vqa_plan_destroy(VqaPlan* plan);

/* PIL-exact antialiased bilinear resize of one uint8 HWC image on the device (SURVEY 8f, row f1).
 * Replaces the CPU resize inside the reference transform: transforms.Resize((224,224)) -> Pillow
 * Image.resize(BILINEAR) (data/preprocess.py:117-121, api/inference.py:153-167).  All pointers are device
 * pointers.  bounds_* are int32 [out, 2] = (first input index, count), kk_* int32 [out, ksize_*] the 22-bit
 * fixed-point weights of Pillow's Resample.c (the host computes them: vqa_b200/resize.py::coeffs).  tmp holds
 * the horizontally resized intermediate (in_h * out_w * channels bytes; may be NULL when only one pass is
 * needed).  Horizontal pass first, intermediate rounded to uint8: bit-exact with PIL. */
int vqa_resize_bilinear_u8(const uint8_t* src, int32_t in_h, int32_t in_w, int32_t channels, uint8_t* tmp, uint8_t* dst,
                           int32_t out_h, int32_t out_w, const int32_t* bounds_h, const int32_t* kk_h, int32_t ksize_h,
                           const int32_t* bounds_v, const int32_t* kk_v, int32_t ksize_v, void* stream);

/* Fused top-1 / top-k accuracy accumulation (SURVEY 8f, row f4).  Replaces VQAAccuracy.update's argmax + topk(5) +
 * .cpu() + .item() per batch (utils/metrics.py:56-105, called from training/evaluate.py:77-106 and
 * training/train.py:229-264).  Give either logits (fp32 [batch, num_classes], row pitch ld) or pred_in (int64
 * [batch], the 1-D form of update(): top-1 only); targets int64 [batch] (a target outside [0, num_classes) is never
 * correct but counts in the total).  counters = uint64[3] in device memory {top-1 correct, top-k correct, total},
 * ADDED to (zero them to reset).  pred_out (int64 [batch], argmax with ties to the lower index) and rank_out (int32
 * [batch], rank of the target's logit in its row, num_classes for an invalid target) may be NULL.  All pointers are
 * device pointers; one launch, no synchronisation. */
int vqa_accuracy_update(const float* logits, int32_t ld, int32_t num_classes, const int64_t* pred_in,
                        const int64_t* targets, int32_t batch, int32_t k, uint64_t* counters, int64_t* pred_out,
                        int32_t* rank_out, void* stream);

/* counters (process-wide): kernels launched by this library since load */
uint64_t vqa_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VQA_B200_H_ */
