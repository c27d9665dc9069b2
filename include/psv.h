/*
 * psv.h -- C ABI of the B200-native patch-skipping ViT encoder ("psv").
 *
 * The reference (himanshukumargupta11012/ViT-pruning) has no FFI of its own: its boundary is
 * the Python class API of himanshu/model_utils.py.  This library sits directly below that API;
 * the Python drop-in (vit-pruning_b200/model_utils.py) binds it with ctypes.  Each entry point
 * cites the reference code it replaces (file:line under /root/reference/himanshu unless noted;
 * "HF:" = transformers/models/vit/modeling_vit.py).
 *
 * Conventions
 *   - every function returns PSV_OK (0) or a negative PsvStatus; nothing throws or aborts;
 *     psv_last_error() gives the message for the last failure on that handle;
 *   - all tensor memory is owned by the caller; the handle owns workspaces and packed weights;
 *   - all pointers are DEVICE pointers unless the name says host; tensors are contiguous
 *     row-major and 16-byte aligned;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and nothing
 *     synchronises with the host (the functions are CUDA-graph capturable) unless stated;
 *   - a handle is bound to the device that was current at psv_create and is not thread-safe;
 *   - masks are uint8 (1 = process the token, 0 = skip), the reference's boolean_mask.
 */
#ifndef PSV_H_
#define PSV_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct PsvHandle PsvHandle;

typedef enum {
  PSV_OK = 0,
  PSV_ERR_INVALID = -1,      /* bad argument / shape / alignment */
  PSV_ERR_CUDA = -2,         /* a CUDA runtime or driver call failed */
  PSV_ERR_STATE = -3,        /* call order (e.g. forward before load_weights) */
  PSV_ERR_UNSUPPORTED = -4   /* geometry or mode this build does not cover */
} PsvStatus;

typedef enum {
  PSV_FP32 = 0,              /* fp32 storage + fp32 FFMA GEMMs: the 1e-4 parity mode */
  PSV_BF16 = 1               /* bf16 operands on tcgen05 tensor cores, fp32 accumulate,
                                fp32 residual stream / LayerNorm / softmax */
} PsvPrecision;

typedef enum {               /* element type of a pixel_values buffer */
  PSV_PIXELS_F32 = 0,
  PSV_PIXELS_BF16 = 1,
  PSV_PIXELS_U8_HWC = 2     /* raw uint8 [B, H, W, 3] images: resize + rescale + normalise fused into the patch embedding
                               (see psv_set_u8_input) */
} PsvPixelType;

/* Geometry = the ViTConfig fields the path reads (model_utils.py:184-187; HF ViTConfig). */
typedef struct {
  int32_t hidden;            /* D: 1024 (ViT-L/16), 768 (ViT-B/16) or 384 (DeiT-S/16)       */
  int32_t heads;             /* H: head width hidden/heads must be 64                        */
  int32_t ffn;               /* F: intermediate_size                                         */
  int32_t layers;            /* L                                                            */
  int32_t tokens;            /* N = patches + 1 = 197 (the reference hard-codes 196, :16,:62) */
  int32_t classes;           /* C = num_labels of the classifier (model_utils.py:187)        */
  int32_t image;             /* 224 */
  int32_t patch;             /* 16  */
  int32_t channels;          /* 3   */
  int32_t comp_hidden;       /* 64: compressor hidden width (model_utils.py:28)              */
  int32_t precision;         /* PsvPrecision                                                 */
  int32_t max_batch;         /* workspaces are sized for this many images                    */
  float ln_eps;              /* 1e-12 */
} PsvConfig;

/* Device pointers to the fp32 state-dict tensors of one encoder layer
 * (keys encoder.layer.{i}.*, SURVEY.md 8b).  Linear weights are [out, in] row-major. */
typedef struct {
  const float *ln1_w, *ln1_b;          /* layernorm_before                         */
  const float *q_w, *q_b;              /* attention.attention.query                */
  const float *k_w, *k_b;              /* attention.attention.key                  */
  const float *v_w, *v_b;              /* attention.attention.value                */
  const float *o_w, *o_b;              /* attention.output.dense                   */
  const float *ln2_w, *ln2_b;          /* layernorm_after                          */
  const float *fc1_w, *fc1_b;          /* intermediate.dense                       */
  const float *fc2_w, *fc2_b;          /* output.dense                             */
  const float *c1_w, *c1_b;            /* mlp_layer.0  [comp_hidden, 2*hidden]     */
  const float *c2_w, *c2_b;            /* mlp_layer.2  [1, comp_hidden], [1]       */
} PsvLayerWeights;

typedef struct {
  const float *cls_token;              /* embeddings.cls_token            [1,1,D]       */
  const float *pos_emb;                /* embeddings.position_embeddings  [1,N,D]       */
  const float *patch_w, *patch_b;      /* embeddings.patch_embeddings.projection [D,C,P,P], [D] */
  const float *final_ln_w, *final_ln_b;/* layernorm                                      */
  const float *cls_w, *cls_b;          /* classifier [C,D], [C]                         */
  const PsvLayerWeights *layers;       /* HOST array of `layers` entries                */
} PsvWeights;

/* Per-layer statistics of the dense label pass (model_utils.py:95-113). */
typedef struct {
  float *loss;                 /* [1]      BCE-with-logits on the post-sigmoid scores, :104-108 */
  float *similarity;           /* [B,N-1]  blended similarity, :97-101 (nullable)               */
  uint8_t *accuracy;           /* [B,N-1]  mlp_accuracy_arr, :109 (nullable)                    */
  int64_t *confusion;          /* [2,2]    rows = true (sim < st), cols = predicted, :111-113   */
} PsvLayerStats;

/* ---- lifetime --------------------------------------------------------------------------- */
const char *psv_version(void);
/* Replaces ModifiedViTModel.__init__ (model_utils.py:184-187): allocates workspaces. */
int psv_create(const PsvConfig *cfg, PsvHandle **out);
int psv_destroy(PsvHandle *h);
const char *psv_last_error(const PsvHandle *h);          /* h may be NULL: last create error */
/* Replaces load_state_dict / .to(device) (hi_main.py:130-142).  The library casts and packs
 * into its own buffers (QKV concatenated, compressor split into CLS/token halves, bf16 copies
 * in PSV_BF16 mode); the caller keeps ownership of the inputs.  May be called again to
 * refresh the weights (e.g. after an optimizer step). */
int psv_load_weights(PsvHandle *h, const PsvWeights *w, void *stream);

/* ---- the hot path ----------------------------------------------------------------------- */
/* ViTEmbeddings.forward (model_utils.py:227-229; HF:100-128,153-167).
 * pixels [B,C,H,W] -> hidden fp32 [B,N,D]. */
int psv_embed(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch,
              float *hidden, void *stream);

/* ModifiedViTLayer.forward (model_utils.py:43-121) on the residual stream, IN PLACE:
 * compressor scores -> threshold -> stable compaction -> LN/attention/MLP on the active set ->
 * scatter back; skipped rows are not touched.
 *   hidden        fp32 [B,N,D], updated in place
 *   mlp_threshold the reference's mt (score >= mt means "process")
 *   forced_mask   nullable uint8 [B,N]; replaces the compressor decision (teacher forcing /
 *                 similarity criterion); column 0 is forced to 1 as model_utils.py:67-68
 *   mask_out      nullable uint8 [B,N]   (boolean_mask, :66-68)
 *   scores_out    nullable fp32  [B,N-1] (mlp_output, :65)
 *   n_active_out  nullable int32 [B]     active tokens per image, CLS included */
int psv_layer_forward(PsvHandle *h, int32_t layer, float *hidden, int32_t batch,
                      float mlp_threshold, const uint8_t *forced_mask, uint8_t *mask_out,
                      float *scores_out, int32_t *n_active_out, void *stream);

/* Copies the compaction result of the most recent psv_layer_forward on this handle:
 *   idx_out int32 [B*N] (first T entries valid: flat row ids b*N+t, ascending),
 *   cu_seqlens_out int32 [B+1].  Both nullable. */
int psv_get_compaction(PsvHandle *h, int32_t batch, int32_t *idx_out, int32_t *cu_seqlens_out,
                       void *stream);

/* Dense label pass of one layer (model_utils.py:95-113; `self.training or compute_cosine`).
 * Must be called with the layer INPUT hidden state and the mask/scores that
 * psv_layer_forward produced for it.  Does not modify `hidden_in`. */
int psv_layer_stats(PsvHandle *h, int32_t layer, const float *hidden_in, int32_t batch,
                    const uint8_t *mask, const float *scores, float sim_threshold,
                    const PsvLayerStats *out, void *stream);

/* Similarity ("cosine") skip criterion, pradeep/model_utils.py:73-84: dense pass, blended
 * similarity, mask = [1, sim < st].  mask_out uint8 [B,N], similarity_out nullable [B,N-1]. */
int psv_similarity_mask(PsvHandle *h, int32_t layer, const float *hidden_in, int32_t batch,
                        float sim_threshold, uint8_t *mask_out, float *similarity_out,
                        void *stream);

/* Final LayerNorm + classifier on the CLS row (model_utils.py:241,254).
 * hidden fp32 [B,N,D] -> logits fp32 [B,C]. */
int psv_head(PsvHandle *h, const float *hidden, int32_t batch, float *logits, void *stream);

/* ModifiedViTModel.forward (model_utils.py:189-259): embed -> L layers -> head, one call,
 * no host synchronisation.  Per-layer outputs are nullable:
 *   forced_masks uint8 [L,B,N], masks_out uint8 [L,B,N], scores_out fp32 [L,B,N-1],
 *   n_active_out int32 [L,B].
 * The masks follow the handle's skip criterion (psv_set_skip_criterion) unless forced_masks is given.
 * With use_graph != 0 the launch sequence is captured into a CUDA graph on first use for this
 * (batch, pointer set) and replayed afterwards. */
int psv_forward(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch,
                float mlp_threshold, const uint8_t *forced_masks, float *logits,
                uint8_t *masks_out, float *scores_out, int32_t *n_active_out,
                int32_t use_graph, void *stream);

/* End-to-end call with HOST buffers (what `model(inputs.to(device)).logits.cpu()` does in
 * main_model_utils.py:244-252): copies pixels host->device in chunks overlapped with compute,
 * runs the forward, copies logits (and n_active, nullable, [L,B]) back, and synchronises the
 * stream before returning.  Host buffers should be page-locked for full copy bandwidth. */
int psv_forward_host(PsvHandle *h, const void *host_pixels, int32_t pixel_type, int32_t batch,
                     float mlp_threshold, float *host_logits, int32_t *host_n_active,
                     void *stream);

/* Asynchronous form of psv_forward_host for a double-buffered serving loop: two slots (0, 1).
 * submit enqueues H2D (copy stream) -> forward (`stream`) -> D2H (second copy stream) for one batch and
 * returns immediately; wait blocks the host until that slot's logits (and n_active) have landed.
 * While one slot computes, the other slot's pixels are being copied in.  Host buffers must stay valid
 * (and should be page-locked) until the matching wait returns. */
int psv_forward_host_submit(PsvHandle *h, int32_t slot, const void *host_pixels, int32_t pixel_type,
                            int32_t batch, float mlp_threshold, float *host_logits,
                            int32_t *host_n_active, void *stream);
int psv_forward_host_wait(PsvHandle *h, int32_t slot);

/* ---- compressor training (main_model_utils.py:100-191 with loss_type="cosine") ----------- */
/* One forward + backward of the 12 compressor regressions on a frozen backbone
 * (model_utils.py:95-108, 275-282): runs every layer in skip mode and computes the gradient of
 * sum_l loss_l with respect to the compressor parameters.
 *   grads     fp32, flat, layer-major: for each layer [c1_w (ch*2D), c1_b (ch), c2_w (ch), c2_b (1), pad]
 *             where every layer block is padded with zeros to a multiple of 4 floats
 *   loss_out  fp32 [L] per-layer losses
 * The caller all-reduces `grads` across ranks (NCCL) and applies the optimizer. */
int psv_compressor_grads(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch,
                         float mlp_threshold, float *grads, float *loss_out, void *stream);
/* Gradient of ONE layer's loss (model_utils.py:103-108) with respect to that layer's
 * compressor parameters, given the layer INPUT hidden state and the mask/scores that
 * psv_layer_forward produced for it (this is the backward of the Python drop-in's
 * `layer.loss.backward()`, main_model_utils.py:145-148,168).
 *   grads  fp32 [round_up(ch*2D + ch + ch + 1, 4)], layout [c1_w | c1_b | c2_w | c2_b | pad],
 *          scaled by grad_scale */
int psv_compressor_layer_grads(PsvHandle *h, int32_t layer, const float *hidden_in, int32_t batch,
                               const uint8_t *mask, const float *scores, float grad_scale,
                               float *grads, void *stream);
/* Number of floats in `grads` of psv_compressor_grads (all layers). */
int64_t psv_compressor_param_count(const PsvHandle *h);
/* Fused Adam step on the flat compressor parameters held by the handle (torch.optim.Adam
 * defaults, main_model_utils.py:119), from an (all-reduced) flat gradient; `step` is 1-based. */
int psv_compressor_adam_step(PsvHandle *h, const float *grads, float lr, float beta1, float beta2,
                             float eps, int32_t step, float grad_scale, void *stream);
/* Gradient all-reduce FUSED with the Adam step over NVLink peer memory (data-parallel compressor training, SURVEY.md
 * 8e / C1; the reference trains on one GPU, main_model_utils.py:119,167-169).  `peer_grads[r]` (host array of `world`
 * DEVICE pointers, 16-byte aligned, this rank's own bucket included) is rank r's flat gradient bucket as written by
 * psv_compressor_grads, mapped into this process (CUDA IPC / torch symmetric memory).  One kernel reads all buckets,
 * sums them in rank order (every replica computes the same bits) and applies Adam -- no separate collective, no
 * reduced intermediate.  The caller brackets the call with cross-rank barriers on `stream`: all buckets complete
 * before, no bucket overwritten until every rank has finished reading.  world <= 16. */
int psv_compressor_peer_reduce_adam_step(PsvHandle *h, const float *const *peer_grads, int32_t world, float lr,
                                         float beta1, float beta2, float eps, int32_t step, float grad_scale,
                                         void *stream);
/* Copies the handle's current compressor parameters out (same flat layout as `grads`). */
int psv_get_compressor_params(PsvHandle *h, float *params_out, void *stream);

/* Overwrites the handle's compressor parameters (same flat layout) and refreshes the derived
 * packs; used after an external optimizer step (torch.optim.Adam in the drop-in train()). */
int psv_set_compressor_params(PsvHandle *h, const float *params, void *stream);
/* The Adam moments of the native optimizer (same flat layout as the parameters; zeros before the first step), so a
 * training run can be checkpointed and resumed together with psv_get/set_compressor_params and the caller's step
 * counter (the reference checkpoints with torch.save(model.state_dict()), main_model_utils.py:181-183). */
int psv_get_compressor_adam_state(PsvHandle *h, float *m_out, float *v_out, void *stream);
int psv_set_compressor_adam_state(PsvHandle *h, const float *m, const float *v, void *stream);

/* ---- backbone fine-tuning (main_model_utils.py:108-165 with loss_type = "classification" / "both" / "alternate" and
 * model.vit_train(), model_utils.py:265-273) ------------------------------------------------------------------------ */
/* The patch-skip forward in fp32, keeping per layer the compaction and the packed activations the backward needs
 * (PSV_FP32 handles; fp32 pixel_values, or raw uint8 images after psv_set_u8_input).  logits fp32 [B, C].  It runs in
 * the handle's kv mode (psv_set_kv_mode); in PSV_KV_ALL it also keeps the layer input, LN1 and q|k|v of all
 * batch*tokens rows, and the backward then sends gradient into the skipped tokens through their key / value rows as
 * well.  It decides by the handle's skip criterion (psv_set_skip_criterion); under PSV_SKIP_SIMILARITY every layer first
 * runs its dense pass over all rows (the same split-bf16 tensor-core products as the training forward) and takes
 * [1, sim < sim_threshold] as its mask.  The kv mode, the criterion and the uint8 input setup (size, mean, std) are
 * recorded with the forward: the matching psv_backbone_backward follows them whatever the handle's settings are by then.
 * The skip decisions are hard thresholds: the backward treats them as constants (a skipped token passes its gradient
 * through unchanged), exactly what autograd does in the reference.  `pixels` (fp32 or uint8) must stay valid until the
 * matching psv_backbone_backward has run.  Synchronises the
 * stream once (the backward sizes its GEMMs with the exact per-layer row counts).  Everything the backward reads is kept
 * apart from the inference buffers, so psv_forward*, psv_layer_forward and psv_compressor_grads may run in between; only
 * a later psv_backbone_forward_train replaces the saved state (and with it the pending backward).
 * layer_losses (nullable, device, [L]): the layers' compressor losses (model_utils.py:103-108) as further outputs, for
 * the joint objective of loss_type "both" (main_model_utils.py:131-135, after model.vit_mlp_train()); the forward then
 * also keeps what their backward needs. */
int psv_backbone_forward_train(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch, float mlp_threshold,
                               float *logits, float *layer_losses, void *stream);
/* d loss / d logits [B, C] (fp32, device) -> the gradient with respect to every backbone parameter, flat fp32:
 *   [ cls_token D | position_embeddings N*D | patch projection weight D*(3*16*16) | patch projection bias D |
 *     per layer: layernorm_before w,b (D,D) | q/k/v weights concatenated (3D*D) | q/k/v biases (3D) | attention.output
 *     .dense w,b (D*D, D) | layernorm_after w,b | intermediate.dense w,b (F*D, F) | output.dense w,b (D*F, D) |
 *     final layernorm w,b | classifier w,b (C*D, C) ]
 * (psv_backbone_param_count floats).
 * dlosses / comp_grads (both null or both given; device): the upstream gradients of the L layer losses and the output
 * for the compressor gradients (psv_compressor_param_count floats, the psv_get_compressor_params layout).  With them
 * the backbone gradient includes what the layer losses send back through the compressor inputs (the reference's
 * mlp_input is built from the undetached hidden states, model_utils.py:62-65), as autograd does for loss_type "both";
 * without them the compressors get no gradient, as with vit_train(). */
int psv_backbone_backward(PsvHandle *h, const float *dlogits, const float *dlosses, float *grads, float *comp_grads,
                          void *stream);
int64_t psv_backbone_param_count(const PsvHandle *h);

/* ---- introspection / test hooks --------------------------------------------------------- */
/* Number of kernels the last psv_forward / psv_layer_forward enqueued (bench "gpu_launches"). */
int32_t psv_last_launch_count(const PsvHandle *h);
/* The skip masks the last psv_backbone_forward_train decided, rebuilt from its saved compaction: uint8 [L, batch, N]
 * (device), 1 = the token was processed.  PSV_ERR_STATE before any training forward. */
int psv_backbone_train_masks(PsvHandle *h, uint8_t *masks_out, void *stream);
/* Profiling mode: between begin and end every kernel the library launches (non-graph calls
 * as well as the launches psv_forward captures into a CUDA graph: there the brackets are external event-record
 * nodes between the kernels, so the timeline is the graph replay's own) is bracketed by CUDA events on its stream.
 * psv_profile_end synchronises, writes the
 * kernel kind (0 score/mask, 1 compaction+gather+LN1, 2 GEMM, 3 attention, 4 LayerNorm, 5 im2col,
 * 6 CLS rows, 7 head, 8 similarity, 9 label stats, 10 training, 11 other, 12 CLS half of the compressor) and the duration in ms
 * of each launch, in launch order, into HOST arrays of `capacity` entries and stores the number
 * of launches in *count. */
int psv_profile_begin(PsvHandle *h);
int psv_profile_end(PsvHandle *h, int32_t *kinds, float *ms, int32_t capacity, int32_t *count);
/* Standalone GEMM hook for kernel-level parity tests and roofline timing:
 *   out[M,N] (+)= act(A[M,K] . W[N,K]^T + bias) (+ residual[M,N])
 * a/w element types follow the handle's precision (fp32, or bf16); out_fp32 selects the output
 * type.  bf16 handles offer the three epilogues of the forward: bf16 out (bias required, optional
 * gelu), fp32 store with optional fp32 residual, fp32 accumulate (accumulate=1: out += ...).
 * Uses the same kernels as the forward. */
int psv_gemm(PsvHandle *h, const void *a, const void *w, const float *bias, const float *residual,
             void *out, int32_t out_fp32, int32_t m, int32_t n, int32_t k, int32_t gelu,
             int32_t accumulate, void *stream);

/* Raw-image input (reference main_model_utils.py:54-60: HuggingFace ViTImageProcessor per sample on the host).  After
 * this call `pixel_type = PSV_PIXELS_U8_HWC` is accepted wherever pixels are: the images are uint8 [B, height, width, 3]
 * (height, width <= the model's image size) and the patch-embedding im2col kernel performs Pillow's bilinear resize
 * (fixed-point, horizontal then vertical pass, each rounded to uint8 -- bit-exact), x * (1/255) and (x - mean) / std on
 * the fly.  mean / std: 3 floats each (NULL = 0.5, the ViT default). */
int psv_set_u8_input(PsvHandle *h, int32_t height, int32_t width, const float *mean, const float *std, void *stream);
/* bf16 handles own three tensor-core attention kernels with the same results (within bf16 rounding): the
 * tcgen05/TMEM kernel (faster when images keep many tokens), a query-block mma.sync kernel (short and mixed
 * sequences: the work unit is one head x a block of up to 32 queries of ONE image, blocks aligned to the image's first
 * row, so an image's results do not depend on its neighbours in the batch) and the
 * older one-CTA-per-(image, head) mma.sync kernel (kept for the keep-all-keys mode and as a cross-check).  AUTO picks
 * per layer from the token counts seen by the warm-up forward that precedes a CUDA-graph capture (eager per-layer
 * calls without that information use the packed kernel).  Changing the kind drops the captured graphs. */
#define PSV_ATTENTION_AUTO 0
#define PSV_ATTENTION_MMA 1
#define PSV_ATTENTION_TC 2
#define PSV_ATTENTION_PK 3
int psv_set_attention_kernel(PsvHandle *h, int32_t kind);
/* Which tokens serve as keys / values in the skip layers of psv_forward* / psv_layer_forward (SURVEY.md 8f-4).
 *   PSV_KV_ACTIVE (default): attention among the ACTIVE tokens only -- reference himanshu/model_utils.py:88-91, the
 *                 layer runs on hidden[i][mask[i]], so skipped tokens are neither queries nor keys.
 *   PSV_KV_ALL  : query-only pruning -- reference recap/convprad4.py:99-125 (ModifiedViTSelfAttention: K and V from all
 *                 tokens, `prune_queries` :191-193), :341-352 (layernorm_before on all tokens, residual / LN2 / MLP on the
 *                 kept rows) and :541 (DHSLayer scatters the kept rows back).  LN1 and the q/k/v projection run on all
 *                 batch*tokens rows; everything from the output projection on runs on the active rows as before.
 * Masks, scores and the compaction do not depend on the mode.  Changing it drops the captured graphs.  The training entry
 * points follow it too: psv_compressor_grads runs its skip layers in the mode, psv_backbone_forward_train records it for
 * its backward. */
#define PSV_KV_ACTIVE 0
#define PSV_KV_ALL 1
int psv_set_kv_mode(PsvHandle *h, int32_t mode);
/* Which criterion decides the skip masks of the whole-model entry points.
 *   PSV_SKIP_MLP (default)  : the compressor score, mask = [1, score >= mlp_threshold] -- reference
 *                             himanshu/model_utils.py:62-68.
 *   PSV_SKIP_SIMILARITY     : the oracle ("cosine") criterion of reference pradeep/model_utils.py:73-84 (BASELINE config
 *                             4): before each skip layer a dense pass of that layer over all tokens, the blended
 *                             similarity of its output with the input, mask = [1, sim < sim_threshold] (the mask
 *                             psv_similarity_mask returns).  The compressor scores are still computed (scores_out, the
 *                             joint objective); they no longer decide.
 * Followed by psv_forward, psv_forward_host* and psv_backbone_forward_train (which records it for its backward);
 * caller-supplied forced_masks still take precedence.  psv_layer_forward, psv_layer_stats and psv_similarity_mask do not
 * depend on it (per-layer callers pass forced_mask themselves).  psv_compressor_grads refuses PSV_SKIP_SIMILARITY
 * (PSV_ERR_UNSUPPORTED).  sim_threshold must be finite; it is ignored under PSV_SKIP_MLP.  Changing the mode drops the
 * captured graphs. */
#define PSV_SKIP_MLP 0
#define PSV_SKIP_SIMILARITY 1
int psv_set_skip_criterion(PsvHandle *h, int32_t criterion, float sim_threshold);
/* Which loss the label path (psv_layer_stats, psv_compressor_layer_grads, psv_compressor_grads) computes.
 *   PSV_LOSS_MASK_LABELS (default) : himanshu/model_utils.py:95-113 -- similarity blend 0.3, labels = the layer's own
 *                                    mask, pos_weight = mean/(1 - mean + 1e-16), accuracy / confusion against the mask.
 *   PSV_LOSS_SIMILARITY_LABELS     : donal/model_utils.py:68-80 -- blend 0.5, labels = (similarity < sim_threshold),
 *                                    pos_weight 1.5, prediction = score > mlp_threshold (strict).  For
 *                                    psv_compressor_layer_grads pass those labels ([True, sim < st], i.e. the mask
 *                                    psv_similarity_mask returns) as `mask`; psv_compressor_grads runs the dense label
 *                                    pass of every layer itself (as the reference does every training step). */
#define PSV_LOSS_MASK_LABELS 0
#define PSV_LOSS_SIMILARITY_LABELS 1
int psv_set_loss_variant(PsvHandle *h, int32_t variant, float sim_threshold);
/* Standalone attention hook (bf16 handles: the tcgen05 kernel unless PSV_ATTENTION_MMA is set; fp32 handles: the
 * FFMA kernel):
 *   ctx[r, h*64:(h+1)*64] = softmax(q_r . K_img^T / 8) . V_img      for every packed row r of every image
 * qkv is the packed [total_rows, 3*hidden] activation (row = [q | k | v], heads along columns, element type of
 * the handle's precision), cu_seqlens [batch+1] the DEVICE row offsets of the images (each image at most
 * `tokens` rows), ctx [total_rows, hidden].  This is what reference model_utils.py:91 computes through
 * HF ViTSelfAttention (HF:171-196) on the gathered sub-sequence of one image. */
int psv_attention(PsvHandle *h, const void *qkv, const int32_t *cu_seqlens, int32_t batch, int32_t total_rows,
                  void *ctx, void *stream);

#ifdef __cplusplus
}
#endif
#endif  /* PSV_H_ */
