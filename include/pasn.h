/* pasn.h -- C ABI of the B200-native ProtoASNet prototype head / push library (libpasn_b200.so).
 *
 * The reference (hooman007/ProtoASNet) has no FFI layer: its boundary for this path is the Python
 * duck-type of the model object (SURVEY.md section 8b).  Each entry point below names the reference
 * method(s) it replaces; citations are relative to the reference checkout.  The Python module
 * protoasnet_b200/head.py binds these with ctypes and re-exposes the reference's
 * forward() / push_forward() / compute_occurence_map() / push_prototypes() API; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; the caller owns all buffers
 *   - all calls are asynchronous on `stream`, never allocate, never synchronise, never throw
 *   - return value 0 on success, a negative pasn_status otherwise (pasn_strerror() explains it)
 *   - no per-call state is kept; process-wide state is limited to the measurement / debug hooks at the end of this
 *     header and the sticky fault word (below); one call sequence per stream at a time
 *   - every wait inside the tensor-core kernels is bounded.  A kernel that gives up writes a code into a host-mapped
 *     fault word; from then on pasn_head_forward / pasn_occurrence_only / pasn_head_backward return PASN_ERR_FAULT
 *     (no synchronisation needed to notice: the word lives in pinned host memory)
 *   - there is NO CPU implementation behind this ABI: without a CUDA device the compute calls fail
 */
#ifndef PASN_H_
#define PASN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PASN_ABI_VERSION 2

typedef enum {
  PASN_OK = 0,
  PASN_ERR_INVALID = -1,     /* bad argument / unsupported shape                      */
  PASN_ERR_WORKSPACE = -2,   /* workspace too small                                   */
  PASN_ERR_CUDA = -3,        /* a CUDA runtime call or kernel launch failed           */
  PASN_ERR_UNSUPPORTED = -4, /* requested path (e.g. tcgen05) not available for dims  */
  PASN_ERR_ALIGN = -5,       /* pointer not aligned as required                       */
  PASN_ERR_FAULT = -6        /* an earlier kernel of this process hit a bounded-wait   */
                             /* limit (internal pipeline fault): its results and      */
                             /* everything computed since are invalid                 */
} pasn_status;

/* element type of the feature map (and of the occurrence map, which is returned in the same type).
 * PASN_F16 (torch.autocast's default) runs on the tensor-core families only (fused or tiled, see pasn_path); a shape that only
 * the generic CUDA-core path takes, or dims.path = PASN_PATH_GENERIC, is refused with PASN_ERR_UNSUPPORTED (and a
 * workspace size of 0): the CUDA-core path is the fp32 correctness path.  In fp16 mode the feature map is read exactly, the
 * first-layer weights (add_on_layers.0.weight, occurrence_module.0.weight) are rounded to fp16, and everything after the
 * first layer is bf16 mode's arithmetic.  An fp16 occurrence map saturates to inf above 65504, as any fp16 tensor does. */
typedef enum { PASN_F32 = 0, PASN_BF16 = 1, PASN_F16 = 2 } pasn_dtype;

/* memory format of the backbone feature map handed to the head */
typedef enum {
  PASN_LAYOUT_NCS = 0, /* contiguous NCDHW / NCHW: [N][C][S], S = T*H*W innermost (reference default) */
  PASN_LAYOUT_NSC = 1  /* channels_last(_3d):     [N][S][C], C innermost                              */
} pasn_layout;

/* activation applied to the occurrence module output.  The reference uses abs
 * (src/models/Video_XProtoNet.py:106-109); nothing else is implemented. */
typedef enum { PASN_OCC_ABS = 0 } pasn_occ_act;

/* which kernel family computes the head */
typedef enum {
  PASN_PATH_AUTO = 0,    /* fused kernel when dims/dtype qualify, else tiled, else generic (fp16: never generic) */
  PASN_PATH_GENERIC = 1, /* CUDA-core FFMA kernels, fp32 accumulate, every shape; fp32 / bf16 only              */
  PASN_PATH_TCGEN05 = 2, /* fused tcgen05/TMEM token kernel (bf16 operands, fp32 accumulate; D = 256, S >= 128; */
                         /* fp16 maps: first layer fp16 x fp16)                                                 */
  PASN_PATH_TILED = 3    /* chain of TMA-fed tcgen05 GEMMs: any S / P, D % 128 == 0, C % 64 == 0; bf16 feature   */
                         /* maps in bf16, fp16 maps with an fp16 x fp16 first layer, fp32 feature maps as a     */
                         /* 3-pass bf16 hi/lo split (fp32-grade results)                                        */
} pasn_path;

typedef struct {
  int32_t N; /* clips (or images) in this call                                  */
  int32_t C; /* backbone output channels                                        */
  int32_t D; /* prototype_shape[1]                                              */
  int32_t P; /* prototype_shape[0] (number of prototypes)                       */
  int32_t K; /* num_classes (including the abstention class)                    */
  int32_t S; /* T*H*W (video) or H*W (image)                                    */
  int32_t dtype;   /* pasn_dtype of feat and of occurrence_map                  */
  int32_t layout;  /* pasn_layout of feat                                       */
  int32_t occ_act; /* pasn_occ_act                                              */
  int32_t path;    /* pasn_path                                                 */
} pasn_dims;

/* fp32 master parameters exactly as they sit in the reference state_dict (1x1 kernels flattened):
 *   add_on_layers.{0,2}.{weight,bias}, occurrence_module.{0,2}.{weight,bias}, occurrence_module.4.weight,
 *   prototype_vectors, last_layer.weight
 * (src/models/Video_XProtoNet.py:27-80; src/models/XProtoNet.py:17-49).  In PASN_BF16 mode the conv
 * weights and biases are rounded to bf16 (round-to-nearest-even) on the fly (PASN_F16 mode: the two first-layer weights
 * addon_w1 / occ_w1 to fp16, the rest as in bf16 mode); prototypes and last_layer always stay fp32. */
typedef struct {
  const float* addon_w1; /* [D][C]   */
  const float* addon_b1; /* [D]      */
  const float* addon_w2; /* [D][D]   */
  const float* addon_b2; /* [D]      */
  const float* occ_w1;   /* [D][C]   */
  const float* occ_b1;   /* [D]      */
  const float* occ_w2;   /* [D/2][D] */
  const float* occ_b2;   /* [D/2]    */
  const float* occ_w3;   /* [P][D/2] (bias-free) */
  const float* prototypes; /* [P][D] */
  const float* last_layer; /* [K][P] */
} pasn_weights;

/* optional push arguments of pasn_head_forward: fuse the class-restricted running argmin of
 * src/utils/push_abs_revision.py:288-307 into the similarity kernel, and keep the winner's pooled features in the same
 * pass, as the reference does (:299-302 stashes protoL_input[a, j] from the very forward pass that produced the minimum --
 * the train_push loader draws a random window per __getitem__, src/data/as_dataloader.py:246-255, so a clip cannot be
 * re-fetched later). */
typedef struct {
  const int64_t* labels;      /* [N] ground-truth class of each clip (data_sample["target_AS"])        */
  const int32_t* proto_class; /* [P] class a prototype is restricted to, or -1 for unrestricted        */
                              /*     (abstention prototypes, push_abs_revision.py:231-237)             */
  int64_t global_offset;      /* global index of clip 0 of this call in the unshuffled training set    */
  uint64_t* best_key;         /* [P] in/out running minimum of (orderable(dist) << 32 | global index), stored    */
                              /*     with the top bit flipped: signed int64 order == key order, so ranks merge    */
                              /*     by a plain signed minimum; INT64_MAX = no candidate yet                      */
  float* best_vec;            /* [P][D] in/out or NULL: features_extracted[n*, p, :] of the clip n* that holds    */
                              /*     best_key[p]; rows of prototypes whose best clip is not in this call are kept */
} pasn_push_args;

int pasn_abi_version(void);
const char* pasn_strerror(int status);

/* 1 if a tensor-core path (fused or tiled, per dims.path) can run these dims, else 0 (generic CUDA-core path only) */
int pasn_tcgen05_supported(const pasn_dims* dims);

/* scratch needed by pasn_head_forward / pasn_occurrence_only for these dims */
size_t pasn_head_workspace_bytes(const pasn_dims* dims);

/* size of / fill the derived bf16 (fp16 mode: first layer fp16) weight cache of the tensor-core path that serves these dims (fused: stage images in
 * shared-memory byte order; tiled: row-major bf16 planes); depends on dims.dtype and dims.path; never saved in checkpoints */
size_t pasn_packed_weights_bytes(const pasn_dims* dims);
int pasn_pack_weights(const pasn_weights* w, const pasn_dims* dims, void* packed, void* stream);

/* Replaces Video_XProtoNet.forward / push_forward minus the backbone
 * (src/models/Video_XProtoNet.py:82-98, :111-130; src/models/XProtoNet.py:51-67, :87-106).
 *   feat               [N,C,S] or [N,S,C] (dims.layout), dims.dtype
 *   packed             result of pasn_pack_weights for the same dims, or NULL (then only the generic path can run)
 *   logits             [N,K] fp32
 *   similarity         [N,P] fp32           ((cos+1)/2)
 *   occurrence_map     [N,P,S] dims.dtype, or NULL to skip the store
 *   features_extracted [N,P,D] fp32, or NULL
 *   distance           [N,P] fp32 (= 1 - similarity), or NULL
 *   push               NULL, or the fused running-argmin arguments                                  */
int pasn_head_forward(const void* feat, const pasn_weights* w, const void* packed, const pasn_dims* dims,
                      float* logits, float* similarity, void* occurrence_map, float* features_extracted,
                      float* distance, const pasn_push_args* push, void* workspace, size_t workspace_bytes,
                      void* stream);

/* Replaces Video_XProtoNet.compute_occurence_map minus the backbone (src/models/Video_XProtoNet.py:100-109; called once
 * more per training step by TransformLoss, src/loss/loss.py:302).  Served by the same kernel family as pasn_head_forward
 * for these dims (`packed`, `workspace` as there): the fused token kernel alone (it writes the map on its way), the
 * occurrence branch of the tiled GEMM chain, or the generic CUDA-core path (`packed` NULL or dims.path GENERIC). */
int pasn_occurrence_only(const void* feat, const pasn_weights* w, const void* packed, const pasn_dims* dims,
                         void* occurrence_map, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the head (training: loss.backward() through Video_XProtoNet.forward, src/agents/XProtoNet_Base.py:397,
 * src/agents/Video_XProtoNet_e2e.py:138, and through compute_occurence_map, src/loss/loss.py:302).  Forward
 * intermediates are recomputed, nothing has to be saved by the forward call.  Gradients of the fp32 formulation on the
 * given inputs (a bf16 or fp16 feature map is read exactly, weights are not rounded); sub-gradients as in PyTorch (relu'(0) = 0,
 * d|x|/dx(0) = 0, clamped norms constant).  Shapes the tiled path takes (C % 64 = 0, D % 128 = 0) run on the tensor cores
 * as three-pass bf16 hi/lo GEMMs (fp32-grade products, fp32 accumulation) unless dims.path is PASN_PATH_GENERIC; the
 * rest runs on fp32 CUDA-core kernels.  fp16 feature maps take the tensor-core chain only (PASN_ERR_UNSUPPORTED and a
 * workspace size of 0 otherwise).  grad_logits = grad_similarity = NULL: only the occurrence branch is recomputed
 * and differentiated (backward of pasn_occurrence_only); the other parameter gradients are left untouched.
 *   grad_logits      [N,K] fp32 or NULL     grad_similarity [N,P] fp32 or NULL     grad_occurrence [N,P,S] fp32 or NULL
 *   grads            required; same shapes as pasn_weights; gradients are ADDED to the buffers.  A NULL member is not
 *                    wanted: it is neither computed nor written, and work that serves only unwanted gradients is
 *                    skipped (e.g. prototypes / last_layer alone: the forward recompute and the prototype stage, no
 *                    pooling or branch backward).  A wanted gradient is computed the same way whatever else is wanted.
 *                    Every member NULL and grad_feat NULL: PASN_OK, nothing launched.
 *   grad_feat        [N,C,S] fp32 (always channel-major, whatever dims.layout says about feat), or NULL (not wanted) */
typedef struct {
  float* addon_w1; float* addon_b1; float* addon_w2; float* addon_b2;
  float* occ_w1; float* occ_b1; float* occ_w2; float* occ_b2; float* occ_w3;
  float* prototypes; float* last_layer;
} pasn_grads;
size_t pasn_head_backward_workspace_bytes(const pasn_dims* dims);
int pasn_head_backward(const void* feat, const pasn_weights* w, const pasn_dims* dims, const float* grad_logits,
                       const float* grad_similarity, const float* grad_occurrence, const pasn_grads* grads,
                       float* grad_feat, void* workspace, size_t workspace_bytes, void* stream);

/* Upstream gradients of every output of pasn_head_forward, each fp32 and optional (NULL: no gradient arrives through it). */
typedef struct {
  const float* grad_logits;     /* [N,K]                                                     */
  const float* grad_similarity; /* [N,P]                                                     */
  const float* grad_distance;   /* [N,P]   distance = 1 - similarity                         */
  const float* grad_occurrence; /* [N,P,S]                                                   */
  const float* grad_features;   /* [N,P,D] features_extracted                                */
} pasn_upstream;
/* Backward of Video_XProtoNet.push_forward (src/models/Video_XProtoNet.py:111-130; XProtoNet.py:87-106) and of forward:
 * pasn_head_backward with every upstream gradient of the head (`up` non-NULL).  Same workspace
 * (pasn_head_backward_workspace_bytes), kernel family, add-into-`grads` rule and channel-major fp32 grad_feat.  The
 * distance gradient enters as minus a similarity gradient, the feature gradient is added to d(features_extracted) where
 * the cosine's gradient forms it.  Occurrence-only mode (only the occurrence branch recomputed and differentiated, the
 * other parameter gradients left untouched) is taken when grad_logits, grad_similarity, grad_distance and grad_features
 * are all NULL.  pasn_head_backward(..., gl, gs, go, ...) is this call with {gl, gs, NULL, go, NULL}. */
int pasn_head_backward_ex(const void* feat, const pasn_weights* w, const pasn_dims* dims, const pasn_upstream* up,
                          const pasn_grads* grads, float* grad_feat, void* workspace, size_t workspace_bytes,
                          void* stream);
/* Backward of the last layer alone (a training stage with every other head parameter and the feature map frozen):
 *   grad_last_layer[k][p] += sum_n grad_logits[n][k] * similarity[n][p]
 * grad_logits [N,K] fp32, similarity [N,P] fp32 as pasn_head_forward returned it (no recompute, no workspace), grad_last_layer
 * [K,P] fp32.  One CUDA-core FFMA GEMM whose output tiles are each summed by one block over all N: bit-identical from call
 * to call.  N = 0: no-op. */
int pasn_last_layer_backward(const float* grad_logits, const float* similarity, int32_t N, int32_t P, int32_t K,
                             float* grad_last_layer, void* stream);

/* Loss / metric consumers of the head outputs, on the device (no per-step host round trip):
 *   class_max[n,k] / class_arg[n,k]  max (and global prototype index of the first maximum) of similarity over the
 *                                    prototypes of class k (P/K consecutive prototypes per class)
 *   sums[0] += -sum_n class_max[n, labels[n]]                           ClusterRoiFeat,    src/loss/loss.py:114-138
 *   sums[1] += sum_n sum_{k != labels[n], k != K-1 if abstain} class_max[n,k]   SeparationRoiFeat, src/loss/loss.py:158-187
 *   counts[j] += [j among the top_specific most similar prototypes of [0,n_specific)] + [... top_rest of the rest]
 *   sim_cumsum[j] += sum_n similarity[n,j]                              src/agents/Video_XProtoNet_e2e.py:158-173
 * Any output may be NULL; labels may be NULL when sums is NULL.  P <= 64 when counts is given. */
int pasn_similarity_stats(const float* similarity, const int64_t* labels, int32_t N, int32_t P, int32_t K, int32_t abstain,
                          int32_t n_specific, int32_t top_specific, int32_t top_rest, float* class_max, int32_t* class_arg,
                          double* sums, uint64_t* counts, double* sim_cumsum, void* stream);
/* sum[0] += sum over rows of ||occ[row, 0:S]||_p (p = 1 or 2; L_norm over the spatial dims, src/loss/loss.py:236-250);
 * row_norm[row] = that norm (or NULL).  occ is [rows][S] in `dtype` (any pasn_dtype). */
int pasn_occurrence_lnorm(const void* occ, int32_t dtype, int64_t rows, int32_t S, int32_t p, double* sum, float* row_norm,
                          void* stream);

/* push bookkeeping (src/utils/push_abs_revision.py:242, :299-300, :342-346).
 * A push record is one contiguous buffer  [ best_key: P x u64 | best_vec: P x D x f32 ]  (pasn_push_record_bytes), so that
 * the merge across ranks is ONE all-gather of the records followed by pasn_push_reduce. */
size_t pasn_push_record_bytes(int32_t P, int32_t D);
int pasn_push_init(uint64_t* best_key, int32_t P, void* stream);          /* best_key[:] = +inf / no index */
int pasn_push_decode(const uint64_t* best_key, int32_t P, int64_t* index, /* index[p] = winner or -1       */
                     float* distance, void* stream);                      /* distance[p] fp32 (inf if none)*/
/* gathered = R records back to back (R = 1: this rank's own record).  Per prototype the record with the smallest key
 * wins (lowest distance, ties to the lowest global index):
 *   index[p] / distance[p] / valid[p]   decoded winner (index -1, distance +inf, valid 0 when no rank had a candidate)
 *   vec[p,:]                            its best_vec row (untouched when !valid)                                  */
int pasn_push_reduce(const void* gathered, int32_t R, int32_t P, int32_t D, int64_t* index, float* distance, int32_t* valid,
                     float* vec, void* stream);
/* The merge of a multi-GPU push as ONE kernel over NVLink peer memory instead of a collective call: every rank's record
 * lives in memory all ranks of the node have mapped (torch symmetric memory in protoasnet_b200/push.py).
 *   peer_records [R] device array of device pointers to the ranks' records (this rank's own included)
 *   peer_flags   [R] device array of device pointers to one uint32 epoch flag per rank (zero-initialised, only ever raised)
 * The kernel publishes this rank's record (system-scope release of `epoch` into its flag), waits (bounded) until every
 * peer's flag has reached `epoch`, then reduces like pasn_push_reduce, reading keys and the winners' vectors straight
 * from the peers.  The caller alternates between two record buffers from push to push (epoch parity). */
int pasn_push_merge_peers(const uint64_t* peer_records, const uint64_t* peer_flags, int32_t R, int32_t my_rank, uint32_t epoch,
                          int32_t P, int32_t D, int64_t* index, float* distance, int32_t* valid, float* vec, void* stream);
/* prototype_vectors[p,:] = vec[p,:] where valid[p] != 0 (else unchanged) */
int pasn_push_write_prototypes(float* prototypes, const float* vec, const int32_t* valid, int32_t P, int32_t D,
                               void* stream);
/* Winner side data captured on the device, in the pass that produced the minimum (push_abs_revision.py:301-307): for every
 * prototype p whose best_key[p] names a clip of this call (global index idx in [global_offset, global_offset + N)), copy
 * row (idx - global_offset, p) of each slot's source into row p of its destination; every other row is left untouched.
 *   src row address = src + (idx - global_offset) * clip_stride_bytes + p * proto_stride_bytes   (proto_stride 0: per-clip data)
 *   dst row address = dst + p * row_bytes
 * Called after the scan of a batch on the same stream: keys only decrease and ties go to the lowest global index, so
 * best_key[p] names a clip of the batch exactly when that batch improved p, and the row that survives belongs to the final key.
 * Rows are copied as bytes (16-byte vectors when src, dst and row_bytes are 16-byte aligned). */
#define PASN_CAPTURE_MAX_SLOTS 8
typedef struct {
  const void* src;
  void* dst;
  int64_t row_bytes;
  int64_t clip_stride_bytes;
  int64_t proto_stride_bytes;
} pasn_capture_slot;
int pasn_push_capture(const uint64_t* best_key, int32_t P, int64_t global_offset, int32_t N,
                      const pasn_capture_slot* slots_host, int32_t nslots, void* stream);

/* measurement hooks used by bench.py (not part of the reference-facing contract):
 *   launch_count          number of kernels this library has launched in the process so far
 *   time_main_kernel(1)   record CUDA events around the dominant kernel of every following pasn_head_forward
 *   last_main_kernel_ms   synchronise on those events and return the last duration (ms), <0 if none        */
unsigned long long pasn_debug_launch_count(void);
int pasn_debug_time_main_kernel(int enable);
float pasn_debug_last_main_kernel_ms(void);
/* sticky fault word (0 = none): read it / set it (tests) / clear it */
int pasn_debug_fault(void);
int pasn_debug_set_fault(int code);
/* synchronises `stream` and returns the bounded-wait error code the fused tcgen05 kernels left in `workspace`
 * on the last pasn_head_forward with these dims (0 = none; non-zero = internal pipeline fault, results invalid).  The word is
 * only cleared in front of a call when the process runs with PASN_DEBUG_SYNC=1 (a memset per call otherwise costs ~2 us of a
 * 170 us step); without it read pasn_debug_fault(), the sticky fault word every bounded wait reports into. */
int pasn_debug_sm100_error(const void* workspace, const pasn_dims* dims, void* stream);
/* device buffer of 1024 int64: [0,768) clock64() stamps of CTA 0 of the token kernel per tile phase, [768,1024) globaltimer
 * stamps of the token kernel start/end and of CTA 0 of the prototype kernel (tools/trace_k1.py, trace_k2.py; NULL = off) */
int pasn_debug_set_trace(void* device_buffer);
/* Test hook for the building block of the tiled tensor-core path: one launch of the library's internal tcgen05 GEMM.
 * `desc_host` points at a pasn::tcg::Gemm (protoasnet_b200/csrc/tc_gemm.cuh; tests/test_tc_gemm_gpu.py mirrors it field
 * by field), `desc_bytes` must equal pasn_debug_tc_gemm_desc_bytes(). */
size_t pasn_debug_tc_gemm_desc_bytes(void);
int pasn_debug_tc_gemm(const void* desc_host, size_t desc_bytes, void* stream);
/* device buffer of 64 x 64 int64: globaltimer stamps of CTA 0 of the next (up to 64) GEMM launches of the tiled path, one row
 * per launch (tools/trace_gemm.py; NULL = off) */
int pasn_debug_set_gemm_trace(void* device_buffer);

#ifdef __cplusplus
}
#endif
#endif /* PASN_H_ */
