// Internal declarations shared by the psv translation units (not part of the C ABI).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "psv.h"

namespace psv {

using bf16 = __nv_bfloat16;

// ---------------------------------------------------------------------------------------------
// GEMM epilogue description: out[orow(r), :] = act(acc + bias) + res[rrow(r), :]
//   orow(r) = out_idx ? out_idx[r] : r ;  rrow(r) = res_idx ? res_idx[r] : r
// `m_dev` (nullable) points at the device-resident row count (T = cu_seqlens[B]); the grid is
// sized for `m_max` rows and tiles past *m_dev exit early, so no host sync is needed.
struct GemmArgs {
  const void *a = nullptr;        // [m, k]   activations (float or bf16 by precision)
  const void *w = nullptr;        // [n, k]   weights (float or bf16), K contiguous
  const float *bias = nullptr;    // [n] nullable
  const float *res = nullptr;     // fp32 residual source, row stride n; nullable
  const int32_t *res_idx = nullptr;
  const int32_t *out_idx = nullptr;
  void *out = nullptr;            // [*, n]
  int out_fp32 = 1;               // output element type: 1 float, 0 bf16
  int gelu = 0;
  int accumulate = 0;             // fp32 output only: out[orow] += ... (red.global.add) instead of a store
  int m_max = 0, n = 0, k = 0;
  const int32_t *m_dev = nullptr;
};

// Per-layer packed weights owned by the handle.
struct LayerPack {
  // fp32 masters (always present; fp32 mode computes from these)
  float *ln1_w, *ln1_b, *ln2_w, *ln2_b;
  float *wqkv, *bqkv;          // [3D, D], [3D]
  float *wo, *bo;              // [D, D], [D]
  float *w1, *b1;              // [F, D], [F]
  float *w2, *b2;              // [D, F], [D]
  float *c1;                   // compressor flat params: [c1_w (ch x 2D) | c1_b (ch) | c2_w (ch) | c2_b (1)]
  float *c1_tokT;              // [D, ch] token half of c1_w transposed (derived; see repack_compressor)
  bf16 *c1_tok_hi, *c1_tok_lo; // [ch, D] split-bf16 token half of c1_w (PSV_BF16 only; derived)
  // bf16 copies of the GEMM weights (PSV_BF16 only)
  bf16 *wqkv_h, *wo_h, *w1_h, *w2_h;
};

struct TensorMapCache;   // gemm_tc.cu
struct TrainSave;        // train_backbone.cu: activations kept for the backbone backward
struct BackboneOptim;    // optim.cu: segment table and Adam moments of the backbone optimizer

// kernel kinds reported by the profiling mode (psv_profile_begin / psv_profile_end)
enum KernelKind { KK_SCORE = 0, KK_GATHER_LN = 1, KK_GEMM = 2, KK_ATTENTION = 3, KK_LN = 4, KK_IM2COL = 5,
                  KK_CLS_ROWS = 6, KK_HEAD = 7, KK_SIMILARITY = 8, KK_LABEL_STATS = 9, KK_TRAIN = 10, KK_OTHER = 11,
                  KK_CLS_HALF = 12, KK_BUDGET = 13 };
// a / b index PsvHandle::prof_events (inside a captured graph consecutive launches share one event: b of launch i is
// a of launch i+1, so the timeline costs one external event-record node per kernel)
struct ProfRec { int kind; int a, b; };

}  // namespace psv

struct PsvHandle {
  PsvConfig cfg{};
  int device = 0;
  int sm_count = 148;
  bool weights_loaded = false;
  std::string err;
  int32_t launches = 0;
  bool profiling = false;            // per-launch CUDA-event timing (bench roofline leg)
  std::vector<psv::ProfRec> prof;
  std::vector<cudaEvent_t> prof_events;
  std::vector<cudaGraphExec_t> prof_execs;   // graphs captured while profiling (they hold external event-record nodes)
  int prof_chain = -1;               // last event of the chain while capturing a profiled graph, -1 outside

  // geometry shorthands
  int D = 0, H = 0, F = 0, L = 0, N = 0, C = 0, CH = 0, P = 0, KP = 0;  // KP = channels*patch*patch
  int64_t R = 0;                                                        // max rows = max_batch * N

  // weights
  std::vector<psv::LayerPack> layers;
  float *cls_token = nullptr, *pos_emb = nullptr, *patch_w = nullptr, *patch_b = nullptr;
  float *final_ln_w = nullptr, *final_ln_b = nullptr, *cls_w = nullptr, *cls_b = nullptr;
  psv::bf16 *patch_w_h = nullptr;
  float *comp_params = nullptr;      // flat compressor parameters of all layers (LayerPack::c1 point in here)
  float *adam_m = nullptr, *adam_v = nullptr;
  int64_t comp_per_layer = 0;

  // workspaces
  uint8_t *mask = nullptr;           // [R]
  float *scores = nullptr;           // [max_batch, N-1]
  int32_t *n_active = nullptr;       // [max_batch]   active tokens per image (fp32 score kernel)
  int score_tile_rows = 128;         // rows per tile of the last score_tc launch (<= 128; gather_ln needs it)
  int32_t *n_tile = nullptr;         // [ceil(R/128)][2] active tokens per 128-row tile and image (tcgen05 score kernel)
  int32_t *cu_seqlens = nullptr;     // [max_batch + 1]
  int32_t *idx = nullptr;            // [R]
  int32_t *attn_units = nullptr;     // [max_batch * 7][4] attention work units {first query row, first key row, end key row, image}
  int32_t *attn_unit_count = nullptr;  // [1] number of valid entries (zeroed by the score kernel, appended by the compaction)
  void *act_a = nullptr;             // [R, D]   LN output (operand type)
  void *act_qkv = nullptr;           // [R, 3D]
  void *act_ctx = nullptr;           // [R, D]
  float *x1 = nullptr;               // [R, D]   fp32 post-attention residual (packed)
  void *act_mid = nullptr;           // [R, F]   GELU output; also the im2col buffer
  float *hidden = nullptr;           // [R, D]   residual stream used by psv_forward
  float *dense_out = nullptr;        // [R, D]   dense-pass output for the label path
  int32_t *embed_out_idx = nullptr;  // [max_batch*(N-1)] patch row -> hidden row
  int32_t *embed_pos_idx = nullptr;  // [max_batch*(N-1)] patch row -> position row
  int32_t *iota_rows = nullptr;      // [R] 0..R-1 (identity compaction for the dense pass)
  int32_t *dense_cu = nullptr;       // [max_batch+1] 0,N,2N,...
  int32_t *rows_dev = nullptr;       // [4] scratch device ints (row counts for dense GEMMs)
  void *pixels_dev = nullptr;        // staging for psv_forward_host
  float *logits_dev = nullptr;       // [max_batch, C]
  int32_t *n_active_all = nullptr;   // [L, max_batch]
  float *stat_scratch = nullptr;     // reductions for the label path
  float *hc = nullptr;               // [max_batch, ch] CLS half of the compressor pre-activation
  float *train_dw1 = nullptr;        // compressor training: partial [64, D] blocks of the split-K dW1 product (lazy)
  float *train_delta = nullptr;      // [max_batch*(N-1), ch] d loss / d pre-activation (training path, lazy)
  float *train_preact = nullptr;     // [max_batch*(N-1), ch] compressor pre-activations (bf16-mode training, lazy)
  float *train_dsum = nullptr;       // [max_batch, ch] per-image sums of train_delta (+ 2 coefficient floats)

  // expected active tokens per image of each layer (attention kernel choice; -1 unknown), from the warm-up
  // forward that precedes a graph capture
  std::vector<int> attn_tokens_hint;
  int attention_kernel = PSV_ATTENTION_AUTO;
  int loss_variant = PSV_LOSS_MASK_LABELS;   // psv_set_loss_variant
  float loss_st = 0.9f;              // sim_threshold of the similarity-label variant
  float loss_mt = 0.5f;              // mlp_threshold of the last decision (donal's accuracy / prediction use it)
  uint8_t *label_mask = nullptr;     // [R] labels of the similarity-label variant in psv_compressor_grads (lazy)
  int kv_mode = PSV_KV_ACTIVE;       // psv_set_kv_mode: PSV_KV_ALL = skipped tokens still serve as keys / values
  int train_precision = PSV_TRAIN_SPLIT;   // psv_set_train_precision (backbone fine-tuning on fp32 handles)
  int skip_criterion = PSV_SKIP_MLP; // psv_set_skip_criterion: PSV_SKIP_SIMILARITY = dense pass + [1, sim < skip_st]
  float skip_st = 0.9f;
  uint8_t *crit_mask = nullptr;      // [R] the similarity mask of the layer about to run (lazy, ensure_criterion_buffers)
  bool attn_hint_valid = false;
  float attn_hint_mt = 0.f;
  int budget_mode = PSV_BUDGET_OFF;  // psv_set_token_budget: PSV_BUDGET_EXACT / CAP keep at most budget_keep[l] patches
  std::vector<int32_t> budget_keep;  // [L] (host)

  // CUDA graph cache for psv_forward: one graph per (batch, pixel type, threshold, forced masks, wanted outputs); the
  // kernels write into handle-owned staging buffers (logits_dev, n_active_all, masks_all, scores_all) and the pixel
  // pointer of the root (im2col) node is patched when the caller's input tensor changes
  struct GraphKey {
    int32_t pixel_type, batch; float mt; const void *forced; bool want_masks, want_scores;
    bool operator==(const GraphKey &o) const {
      return pixel_type == o.pixel_type && batch == o.batch && mt == o.mt && forced == o.forced &&
             want_masks == o.want_masks && want_scores == o.want_scores;
    }
  };
  struct GraphEntry {
    GraphKey key; cudaGraphExec_t exec; cudaGraph_t graph; int32_t launches; const void *pixels;
    cudaGraphNode_t root; cudaKernelNodeParams root_params; int root_nparams; std::vector<int> hints;
    uint64_t last_use;
  };
  uint64_t graph_clock = 0;
  std::vector<GraphEntry> graphs;
  uint8_t *masks_all = nullptr;      // [L, R]            staging of the per-layer masks (lazy)
  float *scores_all = nullptr;       // [L, max_batch*196] staging of the per-layer scores (lazy)
  int32_t *hint_host = nullptr;      // pinned [L, max_batch]: token counts of a replay, fetched every 64th replay
  cudaEvent_t hint_event = nullptr;
  bool hint_pending = false;
  int hint_batch = 0;
  uint32_t hint_counter = 0;

  // two-slot asynchronous host pipeline (psv_forward_host_submit / _wait)
  struct HostSlot {
    void *pixels = nullptr; float *logits = nullptr; int32_t *n_active = nullptr;
    cudaEvent_t h2d_done = nullptr, fwd_done = nullptr, d2h_done = nullptr;
    bool busy = false; int launches = 0;
  };
  HostSlot slots[2];
  cudaStream_t d2h_stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_event = nullptr;
  cudaEvent_t start_event = nullptr;

  // raw uint8 input (psv_set_u8_input): source size, normalisation and Pillow's bilinear coefficient tables
  int u8_h = 0, u8_w = 0;
  float u8_mean[3] = {0.5f, 0.5f, 0.5f}, u8_std[3] = {0.5f, 0.5f, 0.5f};
  int32_t *u8_tables = nullptr;      // [fx(S) | cx(2S) | fy(S) | cy(2S)], S = image size

  psv::TensorMapCache *tmaps = nullptr;
  psv::TrainSave *train_save = nullptr;   // lazily allocated by psv_backbone_forward_train
  psv::BackboneOptim *bopt = nullptr;     // lazily allocated by the backbone optimizer entry points
};

namespace psv {

// Counts a kernel launch and, in profiling mode, brackets it with CUDA events on its stream.
// Eager launches: one event before and one after the kernel.  Launches captured into a CUDA graph (psv_forward with
// use_graph while profiling): external event-record nodes, chained, so the timeline is that of the graph replay itself.
struct LaunchScope {
  PsvHandle *h; cudaStream_t s; ProfRec rec; bool on, captured = false;
  int new_event() {
    cudaEvent_t e;
    cudaEventCreate(&e);
    h->prof_events.push_back(e);
    return (int)h->prof_events.size() - 1;
  }
  void record(int i) {
    if (captured) cudaEventRecordWithFlags(h->prof_events[i], s, cudaEventRecordExternal);
    else cudaEventRecord(h->prof_events[i], s);
  }
  LaunchScope(PsvHandle *h_, int kind, cudaStream_t s_) : h(h_), s(s_), on(h_->profiling) {
    ++h->launches;
    if (on) {
      cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
      cudaStreamIsCapturing(s, &st);
      captured = st == cudaStreamCaptureStatusActive;
      rec.kind = kind;
      if (captured && h->prof_chain >= 0) rec.a = h->prof_chain;
      else { rec.a = new_event(); record(rec.a); }
    }
  }
  ~LaunchScope() {
    if (on) {
      rec.b = new_event(); record(rec.b);
      if (captured) h->prof_chain = rec.b;
      h->prof.push_back(rec);
    }
  }
};

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------
// Forward-path kernels are launched with programmaticStreamSerialization: a kernel may start while its
// predecessor is still draining, runs its private prologue (barrier init, TMEM alloc, tensormap prefetch,
// smem carve-up), and must call pdl_wait() before touching ANY global memory a predecessor may write.
#if defined(__CUDACC__)
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Trigger policy: kernels do NOT release their dependents at the top (a dependent grid that becomes resident early only
// spins in pdl_wait() and takes SM resources from the primary's remaining CTAs; measured slower).  The implicit trigger
// at CTA exit is what lets the next grid's launch overlap the primary's tail; pdl_trigger_now() is for the few places
// where an earlier release is known to pay (cls_half_kernel -> score_tc_kernel).
__device__ __forceinline__ void pdl_trigger_now() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
bool pdl_enabled();
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

inline size_t esize(const PsvHandle *h) { return h->cfg.precision == PSV_BF16 ? 2 : 4; }

// Hidden widths the kernels templated on D are instantiated for: DeiT-S/16, ViT-B/16, ViT-L/16.  Their launchers
// dispatch on exactly these and return cudaErrorNotSupported for anything else.
inline bool psv_hidden_supported(int D) { return D == 384 || D == 768 || D == 1024; }

// ---- kernels (one launcher per file); every launcher returns cudaError_t and bumps h->launches
cudaError_t launch_score_mask(PsvHandle *h, const LayerPack &lp, const float *hidden, int batch, float mt,
                              const uint8_t *forced_mask, uint8_t *mask_out, float *scores_out,
                              int32_t *n_active_out, cudaStream_t s);
cudaError_t launch_gather_ln(PsvHandle *h, const LayerPack &lp, const float *hidden, int batch,
                             int32_t *n_active_out, bool tile_counts, cudaStream_t s, bool index_only = false);
// the token budget of `layer` (h->budget_mode != PSV_BUDGET_OFF) applied to h->scores: rewrites h->mask and h->n_active
// (the compaction must then take per-image counts), and mask_out when given
cudaError_t launch_budget_mask(PsvHandle *h, int layer, int batch, float mt, uint8_t *mask_out, cudaStream_t s);
cudaError_t configure_score_tc();
cudaError_t launch_comp_split(PsvHandle *h, const LayerPack &lp, cudaStream_t s);
cudaError_t launch_score_mask_tc(PsvHandle *h, const LayerPack &lp, const float *hidden, int batch, float mt,
                                 const uint8_t *forced_mask, uint8_t *mask_out, float *scores_out, float *preact_out,
                                 cudaStream_t s);
// bf16_out: bf16 output whatever the handle's precision (the PSV_TRAIN_BF16 training forward on fp32 handles)
cudaError_t launch_ln_rows(PsvHandle *h, const float *x, const int32_t *row_idx, const float *gamma,
                           const float *beta, void *out, int rows_max, const int32_t *rows_dev, cudaStream_t s,
                           bool bf16_out = false);
constexpr int kAttentionTcMinTokens = 190;  // mean tokens per image from which the tcgen05 kernel wins (launch_attention)
// have_units: h->attn_units was written for these cu_seqlens by the compaction kernel (else built on demand)
cudaError_t launch_attention(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                             int64_t qkv_rows, int tokens_hint, cudaStream_t s, bool have_units = false);
cudaError_t configure_attention_pk();
cudaError_t launch_attention_pk(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                int64_t qkv_rows, bool have_units, int rows_hint, cudaStream_t s);
cudaError_t launch_gemm(PsvHandle *h, const GemmArgs &g, cudaStream_t s);          // dispatch on precision
cudaError_t launch_gemm_simt(PsvHandle *h, const GemmArgs &g, cudaStream_t s);     // fp32 FFMA
cudaError_t launch_gemm_tc(PsvHandle *h, const GemmArgs &g, cudaStream_t s);       // bf16 tcgen05
cudaError_t launch_im2col(PsvHandle *h, const void *pixels, int pixel_type, int batch, void *patches, cudaStream_t s);
// raw uint8 images with an explicit setup (launch_im2col passes the handle's current one; the training backward the
// one its forward recorded): source size, Pillow coefficient tables [6 * image], mean / std [3]
cudaError_t launch_im2col_u8(PsvHandle *h, const uint8_t *pixels, int batch, void *patches, int src_h, int src_w,
                             const int32_t *tables, const float *mean, const float *std, cudaStream_t s);
size_t pixel_bytes_per_image(const PsvHandle *h, int pixel_type);
cudaError_t launch_cls_rows(PsvHandle *h, float *hidden, int batch, cudaStream_t s);
cudaError_t launch_head(PsvHandle *h, const float *hidden, int batch, float *logits, cudaStream_t s);
cudaError_t launch_cast_bf16(const float *src, bf16 *dst, int64_t n, cudaStream_t s);
cudaError_t launch_similarity(PsvHandle *h, const float *dense_out, const float *hidden_in, int batch,
                              float *sim_out, cudaStream_t s);
cudaError_t launch_label_stats(PsvHandle *h, const float *sim, const uint8_t *mask, const float *scores, int batch,
                               float st, const PsvLayerStats *out, cudaStream_t s);
cudaError_t launch_sim_mask(PsvHandle *h, const float *sim, int batch, float st, uint8_t *mask_out, cudaStream_t s);

// q_rows / kv_tokens: keep-all-keys mode (see attention_mma.cu); nullptr / 0 = queries and keys are the packed rows
cudaError_t launch_attention_simt(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                  cudaStream_t s, const int32_t *q_rows = nullptr, int kv_tokens = 0);
cudaError_t configure_attention_simt();
cudaError_t configure_attention_mma();
cudaError_t launch_attention_mma(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                 cudaStream_t s, const int32_t *q_rows = nullptr, int kv_tokens = 0);
cudaError_t configure_attention_tc();
cudaError_t launch_attention_tc(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                int64_t qkv_rows, cudaStream_t s);
cudaError_t configure_gemm_tc();
bool tmap_encode_available();
cudaError_t launch_comp_repack(PsvHandle *h, const float *c1, float *tokT, cudaStream_t s);
cudaError_t launch_iota(int32_t *p, int64_t n, int mul, cudaStream_t s);
cudaError_t launch_embed_index(PsvHandle *h, cudaStream_t s);
cudaError_t launch_adam(float *p, float *m, float *v, const float *g, int64_t n, float lr, float b1, float b2,
                        float eps, int step, float gscale, cudaStream_t s, const float *clip = nullptr);
constexpr int PSV_MAX_PEERS = 16;
// clip (nullable, device): the global-norm clip coefficient the gradient is multiplied by after grad_scale
cudaError_t launch_adam_peer_reduce(float *p, float *m, float *v, const float *const *peer_grads, int world, int64_t n,
                                    float lr, float b1, float b2, float eps, int step, float gscale, cudaStream_t s,
                                    const float *clip = nullptr);

// `preact` (nullable): pre-activations [batch*(N-1), 64] written by the tcgen05 score kernel for this very input; without
// them the backward kernel recomputes the compressor's first layer in fp32.
cudaError_t enqueue_compressor_layer_grads(PsvHandle *h, int layer, const float *hidden_in, int batch,
                                           const uint8_t *mask, const float *scores, const float *preact,
                                           float grad_scale, float *grads, float *loss_out, cudaStream_t s);

// psv_api.cu: PSV_OK or a status with h->err set
int check_pixel_type(PsvHandle *h, int pixel_type);      // fp32 / bf16 pixel_values, or uint8 HWC after psv_set_u8_input
int ensure_criterion_buffers(PsvHandle *h);              // dense_out and crit_mask for PSV_SKIP_SIMILARITY
int check_budget_criterion(PsvHandle *h, const uint8_t *forced_masks);   // a token budget under PSV_SKIP_SIMILARITY

// attention_train.cu (PSV_TRAIN_BF16): forward writes ctx bf16 [rows, D] and lse fp32 [rows, H]; the backward writes
// dqkv fp32 [rows, 3D] and uses di [rows, H] as scratch
cudaError_t launch_attention_train_fwd(PsvHandle *h, const bf16 *qkv, const int32_t *cu_seqlens, int batch, bf16 *ctx,
                                       float *lse, cudaStream_t s);
cudaError_t launch_attention_train_bwd(PsvHandle *h, const bf16 *qkv, const bf16 *ctx, const float *lse,
                                       const float *dctx, const int32_t *cu_seqlens, int batch, float *di, float *dqkv,
                                       cudaStream_t s);

void train_save_free(PsvHandle *h);            // train_backbone.cu
void backbone_optim_free(PsvHandle *h);        // optim.cu
// optim.cu: the device clip coefficient of the last clipped backbone step whose norm covered the compressor gradient
// (null if there was none), read by the clipped compressor Adam steps
const float *backbone_clip_coef(const PsvHandle *h);
// split-bf16 tensor-core products (train_backbone.cu): fp32 operands as bf16 planes, 3 or 6 passes of launch_gemm_tc
struct SplitPlanes { bf16 *hi, *lo, *mid; };   // mid: third plane (null in the two-plane form)
cudaError_t split_planes(const float *src, int ld, int rows, int cols, bool tr, int ldo, SplitPlanes out, bool three,
                         cudaStream_t s, const int32_t *rows_dev = nullptr);
cudaError_t split_gemm(PsvHandle *h, SplitPlanes a, SplitPlanes w, float *out, int M, int N, int K, const float *bias,
                       const float *res, const int32_t *res_idx, const int32_t *out_idx, const int32_t *m_dev,
                       bool three, cudaStream_t s);
TensorMapCache *tmap_cache_create();
void tmap_cache_destroy(TensorMapCache *);

}  // namespace psv
