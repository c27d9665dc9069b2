// C ABI of include/psv.h: handle lifetime, weight packing, and the launch sequences of the
// patch-skip forward.  No kernel lives here; this file only validates, allocates and enqueues.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "psv_internal.cuh"

using namespace psv;

namespace {

thread_local std::string g_create_error;

int fail(PsvHandle *h, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define PSV_CUDA(h, call)                                                                          \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(h, PSV_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

template <typename T>
cudaError_t dmalloc(T **p, size_t count) {
  return cudaMalloc(reinterpret_cast<void **>(p), count * sizeof(T) + 256);
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- the launch sequence of one ViT layer on a packed row set ---------------------------------
// h->act_a already holds LN1(x) for the packed rows.
//   fp32 mode : x1 = proj + res_src[res_idx] kept in a packed fp32 buffer; out[out_idx] = fc2 + x1.
//   bf16 mode : `out` must already hold the layer input for the rows out_idx (it is the residual stream
//               itself for the skip path); both residual additions are fp32 red.global.add's of the GEMM
//               epilogues into out[out_idx], so no separate x1 buffer and no residual reads.
//   kv_all    : keep-all-keys mode (psv_set_kv_mode, reference recap/convprad4.py:99-125,191-193,341-352): h->act_a holds
//               LN1 of ALL batch*N rows in dense order, q/k/v are projected for all of them, every active token attends to
//               all N tokens of its image; from the output projection on the layer runs on the packed active rows as usual.
int enqueue_layer_core(PsvHandle *h, const LayerPack &lp, int batch, const int32_t *cu, const int32_t *m_dev,
                       int m_max, const float *res_src, const int32_t *res_idx, float *out,
                       const int32_t *out_idx, int attn_tokens_hint, cudaStream_t s, bool kv_all = false) {
  const bool bf = h->cfg.precision == PSV_BF16;
  const int rows_hint = attn_tokens_hint > 0 ? attn_tokens_hint * batch : -1;
  GemmArgs g;
  // K5: QKV projection (HF:228-230), one GEMM over the concatenated weight
  g.rows_hint = kv_all ? batch * h->N : rows_hint;
  g.a = h->act_a; g.w = bf ? (const void *)lp.wqkv_h : (const void *)lp.wqkv; g.bias = lp.bqkv;
  g.out = h->act_qkv; g.out_fp32 = !bf; g.m_max = kv_all ? batch * h->N : m_max; g.n = 3 * h->D; g.k = h->D;
  g.m_dev = kv_all ? nullptr : m_dev;
  PSV_CUDA(h, launch_gemm(h, g, s));
  // K6: attention among the active tokens of each image (kv_all: active queries x all keys)
  if (kv_all) {
    static const bool force_simt = getenv("PSV_DEBUG_ATTENTION_SIMT") != nullptr;
    if (bf && !force_simt) PSV_CUDA(h, launch_attention_mma(h, h->act_qkv, h->act_ctx, cu, batch, s, out_idx, h->N));
    else                   PSV_CUDA(h, launch_attention_simt(h, h->act_qkv, h->act_ctx, cu, batch, s, out_idx, h->N));
  } else {
    PSV_CUDA(h, launch_attention(h, h->act_qkv, h->act_ctx, cu, batch, h->R, attn_tokens_hint, s,
                                 cu == h->cu_seqlens));
  }
  // K7: output projection + first residual (HF:266,337)
  g = GemmArgs();
  g.a = h->act_ctx; g.w = bf ? (const void *)lp.wo_h : (const void *)lp.wo; g.bias = lp.bo;
  g.m_max = m_max; g.n = h->D; g.k = h->D; g.m_dev = m_dev; g.out_fp32 = 1; g.rows_hint = rows_hint;
  if (bf) { g.out = out; g.out_idx = out_idx; g.accumulate = 1; }
  else    { g.res = res_src; g.res_idx = res_idx; g.out = h->x1; }
  PSV_CUDA(h, launch_gemm(h, g, s));
  // K8: layernorm_after (HF:340)
  if (bf) PSV_CUDA(h, launch_ln_rows(h, out, out_idx, lp.ln2_w, lp.ln2_b, h->act_a, m_max, m_dev, s));
  else    PSV_CUDA(h, launch_ln_rows(h, h->x1, nullptr, lp.ln2_w, lp.ln2_b, h->act_a, m_max, m_dev, s));
  if (bf && h->fused_mlp) {
    // K9 + K10/K11 as one kernel (mlp_tc_kernel): FC1 + GELU, then FC2 + second residual + scatter-back
    PSV_CUDA(h, launch_mlp_tc(h, lp, m_max, m_dev, out, out_idx, s));
    return PSV_OK;
  }
  // K9: intermediate dense + erf-GELU (HF:297-298)
  g = GemmArgs();
  g.a = h->act_a; g.w = bf ? (const void *)lp.w1_h : (const void *)lp.w1; g.bias = lp.b1; g.gelu = 1;
  g.out = h->act_mid; g.out_fp32 = !bf; g.m_max = m_max; g.n = h->F; g.k = h->D; g.m_dev = m_dev; g.rows_hint = rows_hint;
  PSV_CUDA(h, launch_gemm(h, g, s));
  // K10/K11: output dense + second residual (HF:309-311) + scatter back to the token rows
  g = GemmArgs();
  g.a = h->act_mid; g.w = bf ? (const void *)lp.w2_h : (const void *)lp.w2; g.bias = lp.b2;
  g.out = out; g.out_idx = out_idx; g.out_fp32 = 1;
  g.m_max = m_max; g.n = h->D; g.k = h->F; g.m_dev = m_dev; g.rows_hint = rows_hint;
  if (bf) g.accumulate = 1; else g.res = h->x1;
  PSV_CUDA(h, launch_gemm(h, g, s));
  return PSV_OK;
}

int enqueue_skip_layer(PsvHandle *h, int layer, float *hidden, int batch, float mt, const uint8_t *forced,
                       uint8_t *mask_out, float *scores_out, int32_t *n_active_out, cudaStream_t s) {
  const LayerPack &lp = h->layers[layer];
  static const bool score_simt = getenv("PSV_DEBUG_SCORE_SIMT") != nullptr;
  const bool tc = h->cfg.precision == PSV_BF16 && !score_simt;
  if (tc) PSV_CUDA(h, launch_score_mask_tc(h, lp, hidden, batch, mt, forced, mask_out, scores_out, nullptr, s));
  else    PSV_CUDA(h, launch_score_mask(h, lp, hidden, batch, mt, forced, mask_out, scores_out, nullptr, s));
  const bool kv_all = h->kv_mode == PSV_KV_ALL;
  PSV_CUDA(h, launch_gather_ln(h, lp, hidden, batch, n_active_out, tc, s, kv_all));
  if (kv_all)     // LN1 of every row: the skipped tokens are keys / values too
    PSV_CUDA(h, launch_ln_rows(h, hidden, nullptr, lp.ln1_w, lp.ln1_b, h->act_a, batch * h->N, nullptr, s));
  return enqueue_layer_core(h, lp, batch, h->cu_seqlens, h->cu_seqlens + batch, batch * h->N, hidden, h->idx,
                            hidden, h->idx, h->attn_tokens_hint[layer], s, kv_all);
}

// dense ViT layer on all tokens: hidden_in -> dense_out (hidden_in untouched); model_utils.py:96
int enqueue_dense_layer(PsvHandle *h, int layer, const float *hidden_in, int batch, float *dense_out,
                        cudaStream_t s) {
  const LayerPack &lp = h->layers[layer];
  const int rows = batch * h->N;
  PSV_CUDA(h, launch_ln_rows(h, hidden_in, nullptr, lp.ln1_w, lp.ln1_b, h->act_a, rows, nullptr, s));
  if (h->cfg.precision == PSV_BF16)        // bf16 epilogues accumulate into the output: seed it with the input
    PSV_CUDA(h, cudaMemcpyAsync(dense_out, hidden_in, (size_t)rows * h->D * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return enqueue_layer_core(h, lp, batch, h->dense_cu, nullptr, rows, hidden_in, nullptr, dense_out, nullptr, h->N, s);
}

int enqueue_embed(PsvHandle *h, const void *pixels, int pixel_type, int batch, float *hidden, cudaStream_t s) {
  const bool bf = h->cfg.precision == PSV_BF16;
  PSV_CUDA(h, launch_im2col(h, pixels, pixel_type, batch, h->act_mid, s));
  GemmArgs g;
  g.a = h->act_mid; g.w = bf ? (const void *)h->patch_w_h : (const void *)h->patch_w; g.bias = h->patch_b;
  g.res = h->pos_emb; g.res_idx = h->embed_pos_idx; g.out = hidden; g.out_idx = h->embed_out_idx; g.out_fp32 = 1;
  g.m_max = batch * (h->N - 1); g.n = h->D; g.k = h->KP;
  PSV_CUDA(h, launch_gemm(h, g, s));
  PSV_CUDA(h, launch_cls_rows(h, hidden, batch, s));
  return PSV_OK;
}

int enqueue_forward(PsvHandle *h, const void *pixels, int pixel_type, int batch, float mt,
                    const uint8_t *forced_masks, float *hidden, float *logits, uint8_t *masks_out,
                    float *scores_out, int32_t *n_active_out, cudaStream_t s) {
  int rc = enqueue_embed(h, pixels, pixel_type, batch, hidden, s);
  if (rc) return rc;
  const size_t bn = (size_t)batch * h->N, bp = (size_t)batch * (h->N - 1);
  const bool similarity = !forced_masks && h->skip_criterion == PSV_SKIP_SIMILARITY;
  for (int l = 0; l < h->L; ++l) {
    const uint8_t *forced = forced_masks ? forced_masks + l * bn : nullptr;
    if (similarity) {
      // pradeep/model_utils.py:73-84: the dense pass of this layer decides (what psv_similarity_mask computes)
      if ((rc = enqueue_dense_layer(h, l, hidden, batch, h->dense_out, s))) return rc;
      PSV_CUDA(h, launch_similarity(h, h->dense_out, hidden, batch, h->stat_scratch, s));
      PSV_CUDA(h, launch_sim_mask(h, h->stat_scratch, batch, h->skip_st, h->crit_mask, s));
      forced = h->crit_mask;
    }
    rc = enqueue_skip_layer(h, l, hidden, batch, mt, forced,
                            masks_out ? masks_out + l * bn : nullptr, scores_out ? scores_out + l * bp : nullptr,
                            n_active_out ? n_active_out + (size_t)l * batch : nullptr, s);
    if (rc) return rc;
  }
  PSV_CUDA(h, launch_head(h, hidden, batch, logits, s));
  return PSV_OK;
}

// true when the token counts fetched from a replay (h->hint_host, [L, batch]) would change an attention-kernel choice
// or moved a layer's row count by more than 25 % against the hints the graphs were captured with
bool hints_drifted(PsvHandle *h, int batch) {
  static const int tc_min = getenv("PSV_ATTN_TC_MIN") ? atoi(getenv("PSV_ATTN_TC_MIN")) : kAttentionTcMinTokens;
  for (int l = 0; l < h->L; ++l) {
    long long t = 0;
    for (int b = 0; b < batch; ++b) t += h->hint_host[(size_t)l * batch + b];
    const int now = (int)(t / batch), was = h->attn_tokens_hint[l];
    if ((now >= tc_min) != (was >= tc_min)) return true;
    if (now > was + was / 4 + 2 || now < was - was / 4 - 2) return true;
  }
  return false;
}

void drop_graphs(PsvHandle *h) {
  for (auto &g : h->graphs) { cudaGraphExecDestroy(g.exec); cudaGraphDestroy(g.graph); }
  h->graphs.clear();
}

int check_ready(PsvHandle *h, int batch) {
  if (!h) return PSV_ERR_INVALID;
  if (!h->weights_loaded) return fail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  if (batch < 1 || batch > h->cfg.max_batch)
    return fail(h, PSV_ERR_INVALID, "batch %d outside [1, max_batch=%d]", batch, h->cfg.max_batch);
  return PSV_OK;
}

}  // namespace

namespace psv {
// pixel_type accepted by the entry points: fp32 / bf16 NCHW pixel_values, or raw uint8 HWC after psv_set_u8_input
int check_pixel_type(PsvHandle *h, int pixel_type) {
  if (pixel_type == PSV_PIXELS_F32 || pixel_type == PSV_PIXELS_BF16) return PSV_OK;
  if (pixel_type == PSV_PIXELS_U8_HWC) {
    if (h->u8_h > 0) return PSV_OK;
    return fail(h, PSV_ERR_STATE, "PSV_PIXELS_U8_HWC needs psv_set_u8_input first");
  }
  return fail(h, PSV_ERR_INVALID, "bad pixel_type");
}
// the similarity criterion's dense-pass output and mask: allocated before any graph capture
int ensure_criterion_buffers(PsvHandle *h) {
  if (!h->dense_out) PSV_CUDA(h, dmalloc(&h->dense_out, (size_t)h->R * h->D));
  if (!h->crit_mask) PSV_CUDA(h, dmalloc(&h->crit_mask, (size_t)h->R));
  return PSV_OK;
}
// Programmatic dependent launch is OFF by default: measured on B200 it gave no gain inside the CUDA graph
// (3.98 ms -> 4.06 ms per step) and one bf16 parity case failed with it, so it stays an experiment (PSV_PDL=1).
bool pdl_enabled() {
  static const bool on = getenv("PSV_PDL") != nullptr;
  return on;
}
// refresh the packs derived from the flat compressor parameters of one layer
cudaError_t refresh_compressor_packs(PsvHandle *h, const LayerPack &lp, cudaStream_t s) {
  cudaError_t e = launch_comp_repack(h, lp.c1, lp.c1_tokT, s);
  if (e == cudaSuccess && h->cfg.precision == PSV_BF16) e = launch_comp_split(h, lp, s);
  return e;
}
cudaError_t launch_gemm(PsvHandle *h, const GemmArgs &g, cudaStream_t s) {
  static const bool force_simt = getenv("PSV_DEBUG_GEMM_SIMT") != nullptr;
  if (h->cfg.precision == PSV_BF16 && !force_simt) return launch_gemm_tc(h, g, s);
  return launch_gemm_simt(h, g, s);
}
// bf16 mode has two tensor-core attention kernels, both correct for every sequence length:
//   attention_tc.cu  (tcgen05 / TMEM)  : 1.3-1.5x faster once images keep >= ~120 tokens (one 128-row tile is full)
//   attention_mma.cu (warp mma.sync)   : faster for short sequences, where a 128-row tile is mostly padding and
//                                        the per-tile latency chain (TMA -> MMA -> softmax -> MMA -> store) dominates
// The choice is a SPEED hint only: `tokens_hint` = expected active tokens per image for this launch (the layer's
// mean from the warm-up forward that precedes graph capture; N for the dense pass; -1 unknown -> mma.sync).
// psv_set_attention_kernel (or PSV_ATTENTION=tc|mma at psv_create) forces one kernel.  The fp32 mode uses the
// FFMA kernel.
cudaError_t launch_attention(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                             int64_t qkv_rows, int tokens_hint, cudaStream_t s, bool have_units) {
  static const bool force_simt = getenv("PSV_DEBUG_ATTENTION_SIMT") != nullptr;
  if (h->cfg.precision == PSV_BF16 && !force_simt) {
    static const int tc_min = getenv("PSV_ATTN_TC_MIN") ? atoi(getenv("PSV_ATTN_TC_MIN")) : kAttentionTcMinTokens;
    int kind = tokens_hint >= tc_min ? PSV_ATTENTION_TC : PSV_ATTENTION_PK;
    if (h->attention_kernel != PSV_ATTENTION_AUTO) kind = h->attention_kernel;
    if (kind == PSV_ATTENTION_TC) return launch_attention_tc(h, qkv, ctx, cu_seqlens, batch, qkv_rows, s);
    if (kind == PSV_ATTENTION_MMA) return launch_attention_mma(h, qkv, ctx, cu_seqlens, batch, s);
    return launch_attention_pk(h, qkv, ctx, cu_seqlens, batch, qkv_rows, have_units,
                               tokens_hint > 0 ? tokens_hint * batch : -1, s);
  }
  return launch_attention_simt(h, qkv, ctx, cu_seqlens, batch, s);
}
}  // namespace psv

extern "C" {
#pragma GCC visibility push(default)

const char *psv_version(void) { return "psv 0.1 (sm_100a)"; }

const char *psv_last_error(const PsvHandle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int psv_create(const PsvConfig *cfg, PsvHandle **out) {
  if (!cfg || !out) return fail(nullptr, PSV_ERR_INVALID, "null argument");
  *out = nullptr;
  if (!psv_hidden_supported(cfg->hidden))
    return fail(nullptr, PSV_ERR_UNSUPPORTED,
                "hidden=%d: this build covers 1024 (ViT-L/16), 768 (ViT-B/16) and 384 (DeiT-S/16)", cfg->hidden);
  if (cfg->heads <= 0 || cfg->hidden != cfg->heads * 64)
    return fail(nullptr, PSV_ERR_UNSUPPORTED, "head width hidden/heads must be 64 (got %d/%d)", cfg->hidden, cfg->heads);
  if (cfg->tokens != 197 || cfg->image != 224 || cfg->patch != 16 || cfg->channels != 3)
    return fail(nullptr, PSV_ERR_UNSUPPORTED, "the path is specialised to 224x224x3 / patch 16 / 197 tokens "
                "(the reference hard-codes 196 patches, model_utils.py:16,62)");
  if (cfg->comp_hidden != 64) return fail(nullptr, PSV_ERR_UNSUPPORTED, "compressor hidden width must be 64");
  if (cfg->ffn % 128 != 0 || cfg->ffn <= 0) return fail(nullptr, PSV_ERR_INVALID, "ffn must be a positive multiple of 128");
  if (cfg->layers < 1 || cfg->classes < 1 || cfg->max_batch < 1)
    return fail(nullptr, PSV_ERR_INVALID, "layers, classes and max_batch must be positive");
  if (cfg->precision != PSV_FP32 && cfg->precision != PSV_BF16)
    return fail(nullptr, PSV_ERR_INVALID, "unknown precision %d", cfg->precision);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, PSV_ERR_CUDA, "no CUDA device: psv has no CPU fallback");

  PsvHandle *h = new PsvHandle();
  h->cfg = *cfg;
  h->D = cfg->hidden; h->H = cfg->heads; h->F = cfg->ffn; h->L = cfg->layers; h->N = cfg->tokens;
  h->C = cfg->classes; h->CH = cfg->comp_hidden; h->P = cfg->patch;
  h->KP = cfg->channels * cfg->patch * cfg->patch;
  h->R = (int64_t)cfg->max_batch * cfg->tokens;
  h->comp_per_layer = (((int64_t)h->CH * 2 * h->D + h->CH + h->CH + 1) + 3) / 4 * 4;   // padded to 16 bytes
  cudaGetDevice(&h->device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, h->device) == cudaSuccess) {
    h->sm_count = prop.multiProcessorCount;
    if (prop.major != 10) {
      int rc = fail(nullptr, PSV_ERR_UNSUPPORTED, "device sm_%d%d: psv is built for sm_100a (B200) only", prop.major, prop.minor);
      delete h;
      return rc;
    }
  }
  const size_t es = esize(h);
  const int D = h->D, F = h->F, N = h->N, MB = cfg->max_batch;
  const int64_t R = h->R;
#define PSV_ALLOC(ptr, count)                                                            \
  do {                                                                                   \
    cudaError_t e__ = dmalloc(&(ptr), (size_t)(count));                                  \
    if (e__ != cudaSuccess) {                                                            \
      int rc__ = fail(nullptr, PSV_ERR_CUDA, "cudaMalloc(%s, %zu elements) failed: %s", #ptr, (size_t)(count), cudaGetErrorString(e__)); \
      psv_destroy(h);                                                                    \
      return rc__;                                                                       \
    }                                                                                    \
  } while (0)
  uint8_t *raw;
  PSV_ALLOC(h->mask, R);
  PSV_ALLOC(h->scores, (size_t)MB * (N - 1));
  PSV_ALLOC(h->n_active, MB);
  PSV_ALLOC(h->n_tile, (size_t)2 * ((R + 7) / 8 + 1));          // tiles are 8..128 rows high
  PSV_ALLOC(h->mlp_flags, (size_t)4 * (R / 256 + 2) + 8);       // ready / passed per (m-pair, CTA rank) + 2 ticket counters
  if (cudaMemset(h->mlp_flags, 0, ((size_t)4 * (R / 256 + 2) + 8) * sizeof(int32_t)) != cudaSuccess) {
    psv_destroy(h);
    return fail(nullptr, PSV_ERR_CUDA, "cudaMemset(mlp_flags) failed");
  }
  PSV_ALLOC(h->cu_seqlens, MB + 1);
  PSV_ALLOC(h->idx, R);
  PSV_ALLOC(h->attn_units, (size_t)4 * MB * ((N + 31) / 32));
  PSV_ALLOC(h->attn_unit_count, 4);
  if (cudaMemset(h->attn_unit_count, 0, 16) != cudaSuccess) { psv_destroy(h); return fail(nullptr, PSV_ERR_CUDA, "cudaMemset failed"); }
  PSV_ALLOC(raw, R * D * es); h->act_a = raw;
  PSV_ALLOC(raw, R * 3 * D * es); h->act_qkv = raw;
  PSV_ALLOC(raw, R * D * es); h->act_ctx = raw;
  PSV_ALLOC(h->x1, R * D);
  { size_t mid = (size_t)R * F * es, col = (size_t)MB * (N - 1) * h->KP * es;
    PSV_ALLOC(raw, mid > col ? mid : col); h->act_mid = raw; }
  PSV_ALLOC(h->hidden, R * D);
  PSV_ALLOC(h->embed_out_idx, (size_t)MB * (N - 1));
  PSV_ALLOC(h->embed_pos_idx, (size_t)MB * (N - 1));
  PSV_ALLOC(h->iota_rows, R);
  PSV_ALLOC(h->dense_cu, MB + 1);
  PSV_ALLOC(h->rows_dev, 4);
  PSV_ALLOC(h->logits_dev, (size_t)MB * h->C);
  PSV_ALLOC(h->n_active_all, (size_t)h->L * MB);
  PSV_ALLOC(h->stat_scratch, (size_t)MB * (N - 1) + 64);
  PSV_ALLOC(h->hc, (size_t)MB * h->CH);
  // weights
  PSV_ALLOC(h->cls_token, D); PSV_ALLOC(h->pos_emb, (size_t)N * D);
  PSV_ALLOC(h->patch_w, (size_t)D * h->KP); PSV_ALLOC(h->patch_b, D);
  PSV_ALLOC(h->final_ln_w, D); PSV_ALLOC(h->final_ln_b, D);
  PSV_ALLOC(h->cls_w, (size_t)h->C * D); PSV_ALLOC(h->cls_b, h->C);
  PSV_ALLOC(h->comp_params, (size_t)h->L * h->comp_per_layer);
  if (cfg->precision == PSV_BF16) PSV_ALLOC(h->patch_w_h, (size_t)D * h->KP);
  h->layers.resize(h->L);
  h->attn_tokens_hint.assign(h->L, -1);
  h->fused_mlp = getenv("PSV_FUSED_MLP") != nullptr;          // experiment, see mlp_tc_kernel (gemm_tc.cu)
  if (const char *force = getenv("PSV_ATTENTION"))
    h->attention_kernel = force[0] == 't' ? PSV_ATTENTION_TC : (force[0] == 'm' ? PSV_ATTENTION_MMA
                        : (force[0] == 'p' ? PSV_ATTENTION_PK : PSV_ATTENTION_AUTO));
  for (int l = 0; l < h->L; ++l) {
    LayerPack &lp = h->layers[l];
    memset(&lp, 0, sizeof lp);
    PSV_ALLOC(lp.ln1_w, D); PSV_ALLOC(lp.ln1_b, D); PSV_ALLOC(lp.ln2_w, D); PSV_ALLOC(lp.ln2_b, D);
    PSV_ALLOC(lp.wqkv, (size_t)3 * D * D); PSV_ALLOC(lp.bqkv, 3 * D);
    PSV_ALLOC(lp.wo, (size_t)D * D); PSV_ALLOC(lp.bo, D);
    PSV_ALLOC(lp.w1, (size_t)F * D); PSV_ALLOC(lp.b1, F);
    PSV_ALLOC(lp.w2, (size_t)D * F); PSV_ALLOC(lp.b2, D);
    PSV_ALLOC(lp.c1_tokT, (size_t)D * h->CH);
    lp.c1 = h->comp_params + (size_t)l * h->comp_per_layer;
    if (cfg->precision == PSV_BF16) {
      PSV_ALLOC(lp.wqkv_h, (size_t)3 * D * D); PSV_ALLOC(lp.wo_h, (size_t)D * D);
      PSV_ALLOC(lp.w1_h, (size_t)F * D); PSV_ALLOC(lp.w2_h, (size_t)D * F);
      PSV_ALLOC(lp.c1_tok_hi, (size_t)h->CH * D); PSV_ALLOC(lp.c1_tok_lo, (size_t)h->CH * D);
    }
  }
#undef PSV_ALLOC
  cudaError_t e = cudaMemset(h->comp_params, 0, (size_t)h->L * h->comp_per_layer * sizeof(float));
  if (e == cudaSuccess) e = configure_attention_simt();
  if (e == cudaSuccess) e = configure_attention_mma();
  if (e == cudaSuccess && cfg->precision == PSV_BF16) e = configure_attention_pk();
  if (e == cudaSuccess && cfg->precision == PSV_BF16) e = configure_attention_tc();
  // attention_tc.cu and attention_pk.cu multiply V rows past an image's last token by P = 0: they must never hold NaN /
  // Inf patterns.  The QKV GEMM's bf16 epilogue stores whole 32-row boxes, so the rows just past the last active row
  // are computed from the LN1 rows past it: act_a must start finite too, or the last image of a batch can read NaN
  // from memory a previous allocation left behind.
  if (e == cudaSuccess) e = cudaMemset(h->act_qkv, 0, (size_t)R * 3 * D * es);
  if (e == cudaSuccess) e = cudaMemset(h->act_a, 0, (size_t)R * D * es);
  if (e == cudaSuccess && cfg->precision == PSV_BF16) e = configure_gemm_tc();
  if (e == cudaSuccess && cfg->precision == PSV_BF16) e = configure_score_tc();
  if (e == cudaSuccess) e = launch_iota(h->iota_rows, R, 1, 0);
  if (e == cudaSuccess) e = launch_iota(h->dense_cu, MB + 1, N, 0);
  if (e == cudaSuccess) e = launch_embed_index(h, 0);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
  for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&h->copy_events[i], cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->start_event, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    int rc = fail(nullptr, PSV_ERR_CUDA, "workspace initialisation failed: %s", cudaGetErrorString(e));
    psv_destroy(h);
    return rc;
  }
  h->tmaps = tmap_cache_create();
  *out = h;
  return PSV_OK;
}

int psv_destroy(PsvHandle *h) {
  if (!h) return PSV_OK;
  DeviceGuard guard(h->device);
  cudaDeviceSynchronize();
  for (auto &e : h->prof_events) cudaEventDestroy(e);
  for (auto &g : h->prof_execs) cudaGraphExecDestroy(g);
  drop_graphs(h);
  if (h->hint_host) cudaFreeHost(h->hint_host);
  if (h->hint_event) cudaEventDestroy(h->hint_event);
  void *ptrs[] = {h->masks_all, h->scores_all, h->mask, h->scores, h->n_active, h->n_tile, h->mlp_flags, h->cu_seqlens, h->idx, h->attn_units, h->attn_unit_count, h->act_a, h->act_qkv, h->act_ctx, h->x1,
                  h->act_mid, h->hidden, h->dense_out, h->crit_mask, h->embed_out_idx, h->embed_pos_idx, h->iota_rows,
                  h->dense_cu, h->rows_dev, h->label_mask, h->pixels_dev, h->logits_dev, h->n_active_all, h->stat_scratch, h->hc, h->train_delta, h->train_dsum, h->train_preact, h->train_planes, h->train_dw1, h->u8_tables,
                  h->cls_token, h->pos_emb, h->patch_w, h->patch_b, h->final_ln_w, h->final_ln_b, h->cls_w,
                  h->cls_b, h->patch_w_h, h->comp_params, h->adam_m, h->adam_v};
  for (void *p : ptrs) if (p) cudaFree(p);
  for (auto &lp : h->layers) {
    void *lpt[] = {lp.ln1_w, lp.ln1_b, lp.ln2_w, lp.ln2_b, lp.wqkv, lp.bqkv, lp.wo, lp.bo, lp.w1, lp.b1, lp.w2,
                   lp.b2, lp.c1_tokT, lp.c1_tok_hi, lp.c1_tok_lo, lp.wqkv_h, lp.wo_h, lp.w1_h, lp.w2_h};
    for (void *p : lpt) if (p) cudaFree(p);
  }
  for (auto &sl : h->slots) {
    if (sl.pixels) cudaFree(sl.pixels);
    if (sl.logits) cudaFree(sl.logits);
    if (sl.n_active) cudaFree(sl.n_active);
    if (sl.h2d_done) cudaEventDestroy(sl.h2d_done);
    if (sl.fwd_done) cudaEventDestroy(sl.fwd_done);
    if (sl.d2h_done) cudaEventDestroy(sl.d2h_done);
  }
  if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (auto &ev : h->copy_events) if (ev) cudaEventDestroy(ev);
  if (h->start_event) cudaEventDestroy(h->start_event);
  if (h->tmaps) tmap_cache_destroy(h->tmaps);
  train_save_free(h);
  delete h;
  return PSV_OK;
}

int psv_load_weights(PsvHandle *h, const PsvWeights *w, void *stream) {
  if (!h || !w || !w->layers) return fail(h, PSV_ERR_INVALID, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  DeviceGuard guard(h->device);
  const int D = h->D, F = h->F, CH = h->CH;
  auto cp = [&](float *dst, const float *src, size_t n) -> cudaError_t {
    if (!src) return cudaErrorInvalidValue;
    return cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, s);
  };
  PSV_CUDA(h, cp(h->cls_token, w->cls_token, D));
  PSV_CUDA(h, cp(h->pos_emb, w->pos_emb, (size_t)h->N * D));
  PSV_CUDA(h, cp(h->patch_w, w->patch_w, (size_t)D * h->KP));
  PSV_CUDA(h, cp(h->patch_b, w->patch_b, D));
  PSV_CUDA(h, cp(h->final_ln_w, w->final_ln_w, D));
  PSV_CUDA(h, cp(h->final_ln_b, w->final_ln_b, D));
  PSV_CUDA(h, cp(h->cls_w, w->cls_w, (size_t)h->C * D));
  PSV_CUDA(h, cp(h->cls_b, w->cls_b, h->C));
  const bool bf = h->cfg.precision == PSV_BF16;
  if (bf) PSV_CUDA(h, launch_cast_bf16(h->patch_w, h->patch_w_h, (int64_t)D * h->KP, s));
  for (int l = 0; l < h->L; ++l) {
    const PsvLayerWeights &lw = w->layers[l];
    LayerPack &lp = h->layers[l];
    PSV_CUDA(h, cp(lp.ln1_w, lw.ln1_w, D)); PSV_CUDA(h, cp(lp.ln1_b, lw.ln1_b, D));
    PSV_CUDA(h, cp(lp.ln2_w, lw.ln2_w, D)); PSV_CUDA(h, cp(lp.ln2_b, lw.ln2_b, D));
    PSV_CUDA(h, cp(lp.wqkv, lw.q_w, (size_t)D * D));
    PSV_CUDA(h, cp(lp.wqkv + (size_t)D * D, lw.k_w, (size_t)D * D));
    PSV_CUDA(h, cp(lp.wqkv + (size_t)2 * D * D, lw.v_w, (size_t)D * D));
    PSV_CUDA(h, cp(lp.bqkv, lw.q_b, D)); PSV_CUDA(h, cp(lp.bqkv + D, lw.k_b, D));
    PSV_CUDA(h, cp(lp.bqkv + 2 * D, lw.v_b, D));
    PSV_CUDA(h, cp(lp.wo, lw.o_w, (size_t)D * D)); PSV_CUDA(h, cp(lp.bo, lw.o_b, D));
    PSV_CUDA(h, cp(lp.w1, lw.fc1_w, (size_t)F * D)); PSV_CUDA(h, cp(lp.b1, lw.fc1_b, F));
    PSV_CUDA(h, cp(lp.w2, lw.fc2_w, (size_t)D * F)); PSV_CUDA(h, cp(lp.b2, lw.fc2_b, D));
    float *c = lp.c1;
    PSV_CUDA(h, cp(c, lw.c1_w, (size_t)CH * 2 * D)); c += (size_t)CH * 2 * D;
    PSV_CUDA(h, cp(c, lw.c1_b, CH)); c += CH;
    PSV_CUDA(h, cp(c, lw.c2_w, CH)); c += CH;
    PSV_CUDA(h, cp(c, lw.c2_b, 1));
    PSV_CUDA(h, refresh_compressor_packs(h, lp, s));
    if (bf) {
      PSV_CUDA(h, launch_cast_bf16(lp.wqkv, lp.wqkv_h, (int64_t)3 * D * D, s));
      PSV_CUDA(h, launch_cast_bf16(lp.wo, lp.wo_h, (int64_t)D * D, s));
      PSV_CUDA(h, launch_cast_bf16(lp.w1, lp.w1_h, (int64_t)F * D, s));
      PSV_CUDA(h, launch_cast_bf16(lp.w2, lp.w2_h, (int64_t)D * F, s));
    }
  }
  h->weights_loaded = true;
  return PSV_OK;
}

int psv_embed(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch, float *hidden, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (!pixels || !hidden || !aligned16(pixels) || !aligned16(hidden))
    return fail(h, PSV_ERR_INVALID, "pixels/hidden must be non-null and 16-byte aligned");
  if ((rc = check_pixel_type(h, pixel_type))) return rc;
  DeviceGuard guard(h->device);
  h->launches = 0;
  return enqueue_embed(h, pixels, pixel_type, batch, hidden, (cudaStream_t)stream);
}

int psv_layer_forward(PsvHandle *h, int32_t layer, float *hidden, int32_t batch, float mlp_threshold,
                      const uint8_t *forced_mask, uint8_t *mask_out, float *scores_out, int32_t *n_active_out,
                      void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (layer < 0 || layer >= h->L) return fail(h, PSV_ERR_INVALID, "layer %d outside [0,%d)", layer, h->L);
  if (!hidden || !aligned16(hidden)) return fail(h, PSV_ERR_INVALID, "hidden must be non-null and 16-byte aligned");
  DeviceGuard guard(h->device);
  h->launches = 0;
  h->loss_mt = mlp_threshold;
  return enqueue_skip_layer(h, layer, hidden, batch, mlp_threshold, forced_mask, mask_out, scores_out,
                            n_active_out, (cudaStream_t)stream);
}

int psv_get_compaction(PsvHandle *h, int32_t batch, int32_t *idx_out, int32_t *cu_seqlens_out, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (idx_out)
    PSV_CUDA(h, cudaMemcpyAsync(idx_out, h->idx, (size_t)batch * h->N * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
  if (cu_seqlens_out)
    PSV_CUDA(h, cudaMemcpyAsync(cu_seqlens_out, h->cu_seqlens, (size_t)(batch + 1) * sizeof(int32_t),
                                cudaMemcpyDeviceToDevice, s));
  return PSV_OK;
}

static int ensure_dense_out(PsvHandle *h) {
  if (h->dense_out) return PSV_OK;
  PSV_CUDA(h, dmalloc(&h->dense_out, (size_t)h->R * h->D));
  return PSV_OK;
}

int psv_layer_stats(PsvHandle *h, int32_t layer, const float *hidden_in, int32_t batch, const uint8_t *mask,
                    const float *scores, float sim_threshold, const PsvLayerStats *out, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (layer < 0 || layer >= h->L) return fail(h, PSV_ERR_INVALID, "layer %d outside [0,%d)", layer, h->L);
  if (!hidden_in || !mask || !scores || !out || !out->loss || !out->confusion)
    return fail(h, PSV_ERR_INVALID, "hidden_in, mask, scores, out->loss and out->confusion are required");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_dense_out(h))) return rc;
  h->launches = 0;
  if ((rc = enqueue_dense_layer(h, layer, hidden_in, batch, h->dense_out, s))) return rc;
  PSV_CUDA(h, launch_similarity(h, h->dense_out, hidden_in, batch, h->stat_scratch, s));
  PSV_CUDA(h, launch_label_stats(h, h->stat_scratch, mask, scores, batch, sim_threshold, out, s));
  return PSV_OK;
}

int psv_similarity_mask(PsvHandle *h, int32_t layer, const float *hidden_in, int32_t batch, float sim_threshold,
                        uint8_t *mask_out, float *similarity_out, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (layer < 0 || layer >= h->L) return fail(h, PSV_ERR_INVALID, "layer %d outside [0,%d)", layer, h->L);
  if (!hidden_in || !mask_out) return fail(h, PSV_ERR_INVALID, "hidden_in and mask_out are required");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_dense_out(h))) return rc;
  h->launches = 0;
  if ((rc = enqueue_dense_layer(h, layer, hidden_in, batch, h->dense_out, s))) return rc;
  float *sim = similarity_out ? similarity_out : h->stat_scratch;
  PSV_CUDA(h, launch_similarity(h, h->dense_out, hidden_in, batch, sim, s));
  PSV_CUDA(h, launch_sim_mask(h, sim, batch, sim_threshold, mask_out, s));
  return PSV_OK;
}

int psv_head(PsvHandle *h, const float *hidden, int32_t batch, float *logits, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (!hidden || !logits) return fail(h, PSV_ERR_INVALID, "null argument");
  DeviceGuard guard(h->device);
  h->launches = 0;
  PSV_CUDA(h, launch_head(h, hidden, batch, logits, (cudaStream_t)stream));
  return PSV_OK;
}

int psv_forward(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch, float mlp_threshold,
                const uint8_t *forced_masks, float *logits, uint8_t *masks_out, float *scores_out,
                int32_t *n_active_out, int32_t use_graph, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (!pixels || !logits || !aligned16(pixels)) return fail(h, PSV_ERR_INVALID, "pixels/logits must be non-null, pixels 16-byte aligned");
  if ((rc = check_pixel_type(h, pixel_type))) return rc;
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (h->skip_criterion == PSV_SKIP_SIMILARITY && !forced_masks && (rc = ensure_criterion_buffers(h))) return rc;
  if (!use_graph) {
    h->launches = 0;
    return enqueue_forward(h, pixels, pixel_type, batch, mlp_threshold, forced_masks, h->hidden, logits, masks_out,
                           scores_out, n_active_out, s);
  }
  // ---- graph path.  A graph is captured once per (batch, pixel type, threshold, forced masks, wanted outputs): the
  // kernels write into handle-owned staging buffers and the caller's buffers receive small device-to-device copies
  // after the replay, and the pixel pointer of the first kernel (im2col) is patched into the instantiated graph when it
  // changes -- so a serving loop that allocates fresh input / output tensors every step still replays ONE graph.
  const bool want_masks = masks_out != nullptr, want_scores = scores_out != nullptr;
  if (want_masks && !h->masks_all) PSV_CUDA(h, dmalloc(&h->masks_all, (size_t)h->L * h->R));
  if (want_scores && !h->scores_all) PSV_CUDA(h, dmalloc(&h->scores_all, (size_t)h->L * h->cfg.max_batch * (h->N - 1)));
  auto copy_out = [&]() -> int {
    const size_t bn = (size_t)batch * h->N, bp = (size_t)batch * (h->N - 1);
    if (logits != h->logits_dev)
      PSV_CUDA(h, cudaMemcpyAsync(logits, h->logits_dev, (size_t)batch * h->C * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (n_active_out && n_active_out != h->n_active_all)
      PSV_CUDA(h, cudaMemcpyAsync(n_active_out, h->n_active_all, (size_t)h->L * batch * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    if (want_masks) PSV_CUDA(h, cudaMemcpyAsync(masks_out, h->masks_all, h->L * bn, cudaMemcpyDeviceToDevice, s));
    if (want_scores) PSV_CUDA(h, cudaMemcpyAsync(scores_out, h->scores_all, h->L * bp * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return PSV_OK;
  };
  PsvHandle::GraphKey key{pixel_type, batch, mlp_threshold, forced_masks, want_masks, want_scores};
  // profiling: always capture a fresh graph (with external event-record nodes between the kernels) and keep it out of
  // the cache; psv_profile_end destroys it
  if (!h->profiling) {
    // attention-kernel / grid-size hints were frozen at capture: every 64th replay the per-layer token counts of a
    // replay are fetched (asynchronously; evaluated at a later call), and graphs whose layers drifted are dropped
    if (h->hint_pending && cudaEventQuery(h->hint_event) == cudaSuccess) {
      h->hint_pending = false;
      if (h->hint_batch == batch && !forced_masks && hints_drifted(h, batch)) {
        drop_graphs(h);
        h->attn_hint_valid = false;                  // falls through to the warm-up + capture below
      }
    }
    // exact hit (same shape AND same input tensor), else -- once kMaxPerShape graphs of this shape exist -- the least
    // recently used one with its im2col node re-pointed at the new input tensor
    constexpr int kMaxPerShape = 4;
    int hit = -1, same_shape = 0, lru = -1;
    for (size_t gi = 0; gi < h->graphs.size(); ++gi) {
      PsvHandle::GraphEntry &g = h->graphs[gi];
      if (!(g.key == key)) continue;
      ++same_shape;
      if (g.pixels == pixels) { hit = (int)gi; break; }
      if (lru < 0 || g.last_use < h->graphs[lru].last_use) lru = (int)gi;
    }
    if (hit < 0 && same_shape >= kMaxPerShape) {
      PsvHandle::GraphEntry &g = h->graphs[lru];
      cudaKernelNodeParams kp = g.root_params;
      void *args[16];
      for (int a = 0; a < g.root_nparams; ++a) args[a] = g.root_params.kernelParams[a];
      const void *px = pixels;
      args[0] = &px;
      kp.kernelParams = args;
      PSV_CUDA(h, cudaGraphExecKernelNodeSetParams(g.exec, g.root, &kp));
      g.pixels = pixels;
      hit = lru;
    }
    if (hit >= 0) {
      PsvHandle::GraphEntry &g = h->graphs[hit];
      g.last_use = ++h->graph_clock;
      h->launches = g.launches;
      PSV_CUDA(h, cudaGraphLaunch(g.exec, s));
      if ((rc = copy_out())) return rc;
      if (!forced_masks && !h->hint_pending && (++h->hint_counter & 63) == 0 && h->hint_host) {
        PSV_CUDA(h, cudaMemcpyAsync(h->hint_host, h->n_active_all, (size_t)h->L * batch * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        PSV_CUDA(h, cudaEventRecord(h->hint_event, s));
        h->hint_pending = true;
        h->hint_batch = batch;
      }
      return PSV_OK;
    }
  }
  // First capture for this mlp_threshold: one eager warm-up forward measures the mean number of active tokens per
  // image of every layer; the captured graph then uses the attention kernel that is faster for that length
  // (launch_attention).  Results do not depend on the choice, only the speed does.
  if (!h->attn_hint_valid || h->attn_hint_mt != mlp_threshold || forced_masks) {
    h->launches = 0;
    rc = enqueue_forward(h, pixels, pixel_type, batch, mlp_threshold, forced_masks, h->hidden, h->logits_dev,
                         want_masks ? h->masks_all : nullptr, want_scores ? h->scores_all : nullptr, h->n_active_all, s);
    if (rc) return rc;
    std::vector<int32_t> na((size_t)h->L * batch);
    PSV_CUDA(h, cudaMemcpyAsync(na.data(), h->n_active_all, na.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    PSV_CUDA(h, cudaStreamSynchronize(s));
    for (int l = 0; l < h->L; ++l) {
      long long t = 0;
      for (int b = 0; b < batch; ++b) t += na[(size_t)l * batch + b];
      h->attn_tokens_hint[l] = (int)(t / batch);
    }
    h->attn_hint_valid = !forced_masks;
    h->attn_hint_mt = mlp_threshold;
  }
  // capture: ThreadLocal mode so unrelated threads (e.g. torch's allocator) are not affected
  cudaStream_t cs = s;
  bool own_stream = false;
  if (cs == nullptr || cs == cudaStreamLegacy || cs == cudaStreamPerThread) {   // legacy stream cannot capture
    PSV_CUDA(h, cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    own_stream = true;
  }
  cudaGraph_t graph = nullptr;
  PSV_CUDA(h, cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
  h->launches = 0;
  h->prof_chain = -1;
  rc = enqueue_forward(h, pixels, pixel_type, batch, mlp_threshold, forced_masks, h->hidden, h->logits_dev,
                       want_masks ? h->masks_all : nullptr, want_scores ? h->scores_all : nullptr, h->n_active_all, cs);
  h->prof_chain = -1;
  cudaError_t ce = cudaStreamEndCapture(cs, &graph);
  if (own_stream) cudaStreamDestroy(cs);
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (ce != cudaSuccess) return fail(h, PSV_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
  cudaGraphExec_t exec = nullptr;
  ce = cudaGraphInstantiate(&exec, graph, 0);
  if (ce != cudaSuccess) { cudaGraphDestroy(graph); return fail(h, PSV_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
  if (h->profiling) {
    cudaGraphDestroy(graph);
    h->prof_execs.push_back(exec);
    PSV_CUDA(h, cudaGraphLaunch(exec, s));
    return copy_out();
  }
  PsvHandle::GraphEntry entry{};
  entry.key = key; entry.exec = exec; entry.graph = graph; entry.launches = h->launches; entry.pixels = pixels;
  entry.hints = h->attn_tokens_hint;
  entry.last_use = ++h->graph_clock;
  {
    // the first node of the captured chain is the im2col kernel whose first parameter is the pixel pointer
    cudaGraphNode_t roots[4];
    size_t nroots = 4;
    cudaGraphNodeType type = cudaGraphNodeTypeEmpty;
    if (cudaGraphGetRootNodes(graph, roots, &nroots) != cudaSuccess || nroots != 1 ||
        cudaGraphNodeGetType(roots[0], &type) != cudaSuccess || type != cudaGraphNodeTypeKernel ||
        cudaGraphKernelNodeGetParams(roots[0], &entry.root_params) != cudaSuccess) {
      cudaGraphExecDestroy(exec); cudaGraphDestroy(graph);
      return fail(h, PSV_ERR_CUDA, "captured graph does not start with the im2col kernel node");
    }
    entry.root = roots[0];
    entry.root_nparams = pixel_type == PSV_PIXELS_U8_HWC ? 14 : 6;
  }
  if (h->graphs.size() >= 16) {
    cudaGraphExecDestroy(h->graphs.front().exec); cudaGraphDestroy(h->graphs.front().graph);
    h->graphs.erase(h->graphs.begin());
  }
  h->graphs.push_back(entry);
  if (!h->hint_host) {
    if (cudaMallocHost((void **)&h->hint_host, (size_t)h->L * h->cfg.max_batch * sizeof(int32_t)) != cudaSuccess) h->hint_host = nullptr;
    else if (cudaEventCreateWithFlags(&h->hint_event, cudaEventDisableTiming) != cudaSuccess) { cudaFreeHost(h->hint_host); h->hint_host = nullptr; }
  }
  PSV_CUDA(h, cudaGraphLaunch(exec, s));
  return copy_out();
}

int psv_forward_host(PsvHandle *h, const void *host_pixels, int32_t pixel_type, int32_t batch, float mlp_threshold,
                     float *host_logits, int32_t *host_n_active, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (!host_pixels || !host_logits) return fail(h, PSV_ERR_INVALID, "null argument");
  if ((rc = check_pixel_type(h, pixel_type))) return rc;
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t img_bytes = pixel_bytes_per_image(h, pixel_type);
  if (!h->pixels_dev) {
    uint8_t *raw;
    PSV_CUDA(h, dmalloc(&raw, (size_t)h->cfg.max_batch * h->cfg.channels * h->cfg.image * h->cfg.image * 4));
    h->pixels_dev = raw;
  }
  // The whole batch is one forward (one packed GEMM set); the H2D copy runs on the copy stream in
  // `chunks` pieces and the forward waits for the last one.  Chunked compute would shrink the GEMMs.
  static const int chunks_env = getenv("PSV_E2E_CHUNKS") ? atoi(getenv("PSV_E2E_CHUNKS")) : 1;
  int chunks = chunks_env < 1 ? 1 : (chunks_env > 8 ? 8 : chunks_env);
  if (chunks > batch) chunks = batch;
  PSV_CUDA(h, cudaEventRecord(h->start_event, s));
  PSV_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->start_event, 0));
  const int per = (batch + chunks - 1) / chunks;
  const float mt = mlp_threshold;
  int total_launches = 0;
  for (int c = 0; c < chunks; ++c) {
    const int b0 = c * per, nb = (b0 + per <= batch) ? per : batch - b0;
    if (nb <= 0) break;
    PSV_CUDA(h, cudaMemcpyAsync((uint8_t *)h->pixels_dev + b0 * img_bytes, (const uint8_t *)host_pixels + b0 * img_bytes,
                                nb * img_bytes, cudaMemcpyHostToDevice, h->copy_stream));
    PSV_CUDA(h, cudaEventRecord(h->copy_events[c], h->copy_stream));
    PSV_CUDA(h, cudaStreamWaitEvent(s, h->copy_events[c], 0));
    if (chunks > 1) {
      rc = psv_forward(h, (uint8_t *)h->pixels_dev + b0 * img_bytes, pixel_type, nb, mt, nullptr,
                       h->logits_dev + (size_t)b0 * h->C, nullptr, nullptr,
                       host_n_active ? h->n_active_all + (size_t)c * h->L * per : nullptr, 1, s);
      if (rc) return rc;
      total_launches += h->launches;
    }
  }
  if (chunks == 1) {
    rc = psv_forward(h, h->pixels_dev, pixel_type, batch, mt, nullptr, h->logits_dev, nullptr, nullptr,
                     host_n_active ? h->n_active_all : nullptr, 1, s);
    if (rc) return rc;
    total_launches = h->launches;
  }
  PSV_CUDA(h, cudaMemcpyAsync(host_logits, h->logits_dev, (size_t)batch * h->C * sizeof(float),
                              cudaMemcpyDeviceToHost, s));
  if (host_n_active) {
    if (chunks == 1) {
      PSV_CUDA(h, cudaMemcpyAsync(host_n_active, h->n_active_all, (size_t)h->L * batch * sizeof(int32_t),
                                  cudaMemcpyDeviceToHost, s));
    } else {
      for (int c = 0; c < chunks; ++c) {
        const int b0 = c * per, nb = (b0 + per <= batch) ? per : batch - b0;
        if (nb <= 0) break;
        for (int l = 0; l < h->L; ++l)
          PSV_CUDA(h, cudaMemcpyAsync(host_n_active + (size_t)l * batch + b0,
                                      h->n_active_all + (size_t)c * h->L * per + (size_t)l * nb,
                                      nb * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
      }
    }
  }
  PSV_CUDA(h, cudaStreamSynchronize(s));
  h->launches = total_launches;
  return PSV_OK;
}

static void profile_release(PsvHandle *h) {
  for (auto &e : h->prof_events) cudaEventDestroy(e);
  for (auto &g : h->prof_execs) cudaGraphExecDestroy(g);
  h->prof_events.clear(); h->prof_execs.clear(); h->prof.clear();
  h->prof_chain = -1;
}

int psv_profile_begin(PsvHandle *h) {
  if (!h) return PSV_ERR_INVALID;
  DeviceGuard guard(h->device);
  profile_release(h);
  h->profiling = true;
  return PSV_OK;
}

int psv_profile_end(PsvHandle *h, int32_t *kinds, float *ms, int32_t capacity, int32_t *count) {
  if (!h || !count) return fail(h, PSV_ERR_INVALID, "null argument");
  h->profiling = false;
  DeviceGuard guard(h->device);
  int n = 0;
  int rc = PSV_OK;
  for (auto &r : h->prof) {
    float t = 0.f;
    cudaError_t e = cudaEventSynchronize(h->prof_events[r.b]);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, h->prof_events[r.a], h->prof_events[r.b]);
    if (e != cudaSuccess && rc == PSV_OK) rc = fail(h, PSV_ERR_CUDA, "profile event failed: %s", cudaGetErrorString(e));
    if (n < capacity && kinds && ms) { kinds[n] = r.kind; ms[n] = t; }
    ++n;
  }
  profile_release(h);
  *count = n;
  return rc;
}

int psv_compressor_grads(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch, float mlp_threshold,
                         float *grads, float *loss_out, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (!pixels || !grads || !loss_out || !aligned16(pixels)) return fail(h, PSV_ERR_INVALID, "null or misaligned argument");
  if ((rc = check_pixel_type(h, pixel_type))) return rc;
  if (h->skip_criterion != PSV_SKIP_MLP)
    return fail(h, PSV_ERR_UNSUPPORTED, "psv_compressor_grads trains under the mlp criterion (PSV_SKIP_MLP) only");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  h->launches = 0;
  h->loss_mt = mlp_threshold;
  if ((rc = enqueue_embed(h, pixels, pixel_type, batch, h->hidden, s))) return rc;
  static const bool score_simt = getenv("PSV_DEBUG_SCORE_SIMT") != nullptr;
  for (int l = 0; l < h->L; ++l) {
    const LayerPack &lp = h->layers[l];
    // forward decision of layer l, then its loss/gradient from the layer INPUT (still intact in h->hidden),
    // then the rest of the skip layer updates the stream in place
    const bool tc = h->cfg.precision == PSV_BF16 && !score_simt;
    if (tc && !h->train_preact)
      PSV_CUDA(h, dmalloc(&h->train_preact, (size_t)h->cfg.max_batch * (h->N - 1) * h->CH));
    if (tc) PSV_CUDA(h, launch_score_mask_tc(h, lp, h->hidden, batch, mlp_threshold, nullptr, nullptr, nullptr,
                                             h->train_preact, s));
    else    PSV_CUDA(h, launch_score_mask(h, lp, h->hidden, batch, mlp_threshold, nullptr, nullptr, nullptr, nullptr, s));
    const uint8_t *labels = h->mask;                 // himanshu: the labels are the layer's own decisions (:103)
    if (h->loss_variant == PSV_LOSS_SIMILARITY_LABELS) {
      // donal/model_utils.py:68-75: labels = (similarity of the DENSE layer output with the input < st), every step
      if ((rc = ensure_dense_out(h))) return rc;
      if (!h->label_mask) PSV_CUDA(h, dmalloc(&h->label_mask, (size_t)h->R));
      if ((rc = enqueue_dense_layer(h, l, h->hidden, batch, h->dense_out, s))) return rc;
      PSV_CUDA(h, launch_similarity(h, h->dense_out, h->hidden, batch, h->stat_scratch, s));
      PSV_CUDA(h, launch_sim_mask(h, h->stat_scratch, batch, h->loss_st, h->label_mask, s));
      labels = h->label_mask;
    }
    PSV_CUDA(h, enqueue_compressor_layer_grads(h, l, h->hidden, batch, labels, h->scores, tc ? h->train_preact : nullptr,
                                               1.0f, grads + (size_t)l * h->comp_per_layer, loss_out + l, s));
    // the rest of the skip layer as enqueue_skip_layer runs it, in either kv mode
    const bool kv_all = h->kv_mode == PSV_KV_ALL;
    PSV_CUDA(h, launch_gather_ln(h, lp, h->hidden, batch, nullptr, tc, s, kv_all));
    if (kv_all)
      PSV_CUDA(h, launch_ln_rows(h, h->hidden, nullptr, lp.ln1_w, lp.ln1_b, h->act_a, batch * h->N, nullptr, s));
    if ((rc = enqueue_layer_core(h, lp, batch, h->cu_seqlens, h->cu_seqlens + batch, batch * h->N, h->hidden, h->idx,
                                 h->hidden, h->idx, h->attn_tokens_hint[l], s, kv_all)))
      return rc;
  }
  return PSV_OK;
}

// ---- two-slot asynchronous host pipeline --------------------------------------------------------
// submit(slot): H2D of the pixels on the copy stream -> forward (CUDA graph) on `stream` -> D2H of logits /
// n_active on the D2H stream.  Nothing blocks the host; while slot A computes, slot B's pixels are in flight.
int psv_forward_host_submit(PsvHandle *h, int32_t slot, const void *host_pixels, int32_t pixel_type, int32_t batch,
                            float mlp_threshold, float *host_logits, int32_t *host_n_active, void *stream) {
  int rc = check_ready(h, batch);
  if (rc) return rc;
  if (slot < 0 || slot > 1) return fail(h, PSV_ERR_INVALID, "slot must be 0 or 1");
  if (!host_pixels || !host_logits) return fail(h, PSV_ERR_INVALID, "null argument");
  if ((rc = check_pixel_type(h, pixel_type))) return rc;
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  PsvHandle::HostSlot &sl = h->slots[slot];
  if (sl.busy) return fail(h, PSV_ERR_STATE, "slot %d has a forward in flight: call psv_forward_host_wait first", slot);
  if (!sl.pixels) {
    uint8_t *raw;
    PSV_CUDA(h, dmalloc(&raw, (size_t)h->cfg.max_batch * h->cfg.channels * h->cfg.image * h->cfg.image * 4));
    sl.pixels = raw;
    PSV_CUDA(h, dmalloc(&sl.logits, (size_t)h->cfg.max_batch * h->C));
    PSV_CUDA(h, dmalloc(&sl.n_active, (size_t)h->L * h->cfg.max_batch));
    PSV_CUDA(h, cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming));
    PSV_CUDA(h, cudaEventCreateWithFlags(&sl.fwd_done, cudaEventDisableTiming));
    PSV_CUDA(h, cudaEventCreateWithFlags(&sl.d2h_done, cudaEventDisableTiming));
    if (!h->d2h_stream) PSV_CUDA(h, cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
  }
  const size_t bytes = (size_t)batch * pixel_bytes_per_image(h, pixel_type);
  // the slot's previous forward (already waited for by the host) is complete, so its buffers are free
  PSV_CUDA(h, cudaMemcpyAsync(sl.pixels, host_pixels, bytes, cudaMemcpyHostToDevice, h->copy_stream));
  PSV_CUDA(h, cudaEventRecord(sl.h2d_done, h->copy_stream));
  PSV_CUDA(h, cudaStreamWaitEvent(s, sl.h2d_done, 0));
  rc = psv_forward(h, sl.pixels, pixel_type, batch, mlp_threshold, nullptr, sl.logits, nullptr, nullptr, sl.n_active, 1, s);
  if (rc) return rc;
  sl.launches = h->launches;
  PSV_CUDA(h, cudaEventRecord(sl.fwd_done, s));
  PSV_CUDA(h, cudaStreamWaitEvent(h->d2h_stream, sl.fwd_done, 0));
  PSV_CUDA(h, cudaMemcpyAsync(host_logits, sl.logits, (size_t)batch * h->C * sizeof(float), cudaMemcpyDeviceToHost,
                              h->d2h_stream));
  if (host_n_active)
    PSV_CUDA(h, cudaMemcpyAsync(host_n_active, sl.n_active, (size_t)h->L * batch * sizeof(int32_t),
                                cudaMemcpyDeviceToHost, h->d2h_stream));
  PSV_CUDA(h, cudaEventRecord(sl.d2h_done, h->d2h_stream));
  sl.busy = true;
  return PSV_OK;
}

int psv_forward_host_wait(PsvHandle *h, int32_t slot) {
  if (!h || slot < 0 || slot > 1) return fail(h, PSV_ERR_INVALID, "bad handle or slot");
  PsvHandle::HostSlot &sl = h->slots[slot];
  if (!sl.busy) return fail(h, PSV_ERR_STATE, "slot %d has nothing in flight", slot);
  PSV_CUDA(h, cudaEventSynchronize(sl.d2h_done));
  sl.busy = false;
  h->launches = sl.launches;
  return PSV_OK;
}

int32_t psv_last_launch_count(const PsvHandle *h) { return h ? h->launches : 0; }

int64_t psv_compressor_param_count(const PsvHandle *h) { return h ? (int64_t)h->L * h->comp_per_layer : 0; }

int psv_get_compressor_params(PsvHandle *h, float *params_out, void *stream) {
  if (!h || !params_out) return fail(h, PSV_ERR_INVALID, "null argument");
  if (!h->weights_loaded) return fail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  DeviceGuard guard(h->device);
  PSV_CUDA(h, cudaMemcpyAsync(params_out, h->comp_params, (size_t)h->L * h->comp_per_layer * sizeof(float),
                              cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return PSV_OK;
}

int psv_set_compressor_params(PsvHandle *h, const float *params, void *stream) {
  if (!h || !params) return fail(h, PSV_ERR_INVALID, "null argument");
  if (!h->weights_loaded) return fail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  PSV_CUDA(h, cudaMemcpyAsync(h->comp_params, params, (size_t)h->L * h->comp_per_layer * sizeof(float),
                              cudaMemcpyDeviceToDevice, s));
  for (int l = 0; l < h->L; ++l) PSV_CUDA(h, refresh_compressor_packs(h, h->layers[l], s));
  return PSV_OK;
}

int psv_compressor_adam_step(PsvHandle *h, const float *grads, float lr, float beta1, float beta2, float eps,
                             int32_t step, float grad_scale, void *stream) {
  if (!h || !grads) return fail(h, PSV_ERR_INVALID, "null argument");
  if (!h->weights_loaded) return fail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  if (step < 1) return fail(h, PSV_ERR_INVALID, "step is 1-based");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = (int64_t)h->L * h->comp_per_layer;
  if (!h->adam_m) {
    PSV_CUDA(h, dmalloc(&h->adam_m, (size_t)n));
    PSV_CUDA(h, dmalloc(&h->adam_v, (size_t)n));
    PSV_CUDA(h, cudaMemsetAsync(h->adam_m, 0, n * sizeof(float), s));
    PSV_CUDA(h, cudaMemsetAsync(h->adam_v, 0, n * sizeof(float), s));
  }
  PSV_CUDA(h, launch_adam(h->comp_params, h->adam_m, h->adam_v, grads, n, lr, beta1, beta2, eps, step, grad_scale, s));
  for (int l = 0; l < h->L; ++l) PSV_CUDA(h, refresh_compressor_packs(h, h->layers[l], s));
  return PSV_OK;
}

int psv_get_compressor_adam_state(PsvHandle *h, float *m_out, float *v_out, void *stream) {
  if (!h || !m_out || !v_out) return fail(h, PSV_ERR_INVALID, "null argument");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t bytes = (size_t)h->L * h->comp_per_layer * sizeof(float);
  if (!h->adam_m) {                                 // no step taken yet: the moments are zero
    PSV_CUDA(h, cudaMemsetAsync(m_out, 0, bytes, s));
    PSV_CUDA(h, cudaMemsetAsync(v_out, 0, bytes, s));
    return PSV_OK;
  }
  PSV_CUDA(h, cudaMemcpyAsync(m_out, h->adam_m, bytes, cudaMemcpyDeviceToDevice, s));
  PSV_CUDA(h, cudaMemcpyAsync(v_out, h->adam_v, bytes, cudaMemcpyDeviceToDevice, s));
  return PSV_OK;
}

int psv_set_compressor_adam_state(PsvHandle *h, const float *m, const float *v, void *stream) {
  if (!h || !m || !v) return fail(h, PSV_ERR_INVALID, "null argument");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)h->L * h->comp_per_layer;
  if (!h->adam_m) {
    PSV_CUDA(h, dmalloc(&h->adam_m, n));
    PSV_CUDA(h, dmalloc(&h->adam_v, n));
  }
  PSV_CUDA(h, cudaMemcpyAsync(h->adam_m, m, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  PSV_CUDA(h, cudaMemcpyAsync(h->adam_v, v, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return PSV_OK;
}

int psv_compressor_peer_reduce_adam_step(PsvHandle *h, const float *const *peer_grads, int32_t world, float lr,
                                         float beta1, float beta2, float eps, int32_t step, float grad_scale,
                                         void *stream) {
  if (!h || !peer_grads) return fail(h, PSV_ERR_INVALID, "null argument");
  if (!h->weights_loaded) return fail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  if (step < 1) return fail(h, PSV_ERR_INVALID, "step is 1-based");
  if (world < 1 || world > PSV_MAX_PEERS) return fail(h, PSV_ERR_INVALID, "world must be 1..%d", PSV_MAX_PEERS);
  for (int r = 0; r < world; ++r)
    if (!peer_grads[r] || !aligned16(peer_grads[r])) return fail(h, PSV_ERR_INVALID, "peer bucket %d is null or not 16-byte aligned", r);
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = (int64_t)h->L * h->comp_per_layer;
  if (!h->adam_m) {
    PSV_CUDA(h, dmalloc(&h->adam_m, (size_t)n));
    PSV_CUDA(h, dmalloc(&h->adam_v, (size_t)n));
    PSV_CUDA(h, cudaMemsetAsync(h->adam_m, 0, n * sizeof(float), s));
    PSV_CUDA(h, cudaMemsetAsync(h->adam_v, 0, n * sizeof(float), s));
  }
  PSV_CUDA(h, launch_adam_peer_reduce(h->comp_params, h->adam_m, h->adam_v, peer_grads, world, n, lr, beta1, beta2, eps,
                                      step, grad_scale, s));
  for (int l = 0; l < h->L; ++l) PSV_CUDA(h, refresh_compressor_packs(h, h->layers[l], s));
  return PSV_OK;
}

int psv_gemm(PsvHandle *h, const void *a, const void *w, const float *bias, const float *residual, void *out,
             int32_t out_fp32, int32_t m, int32_t n, int32_t k, int32_t gelu, int32_t accumulate, void *stream) {
  if (!h || !a || !w || !out) return fail(h, PSV_ERR_INVALID, "null argument");
  if (m < 1 || n % 128 != 0 || k % 64 != 0) return fail(h, PSV_ERR_INVALID, "need m>=1, n%%128==0, k%%64==0");
  if (h->cfg.precision == PSV_FP32 && !out_fp32) return fail(h, PSV_ERR_INVALID, "fp32 handles write fp32");
  DeviceGuard guard(h->device);
  GemmArgs g;
  g.a = a; g.w = w; g.bias = bias; g.res = residual; g.out = out; g.out_fp32 = out_fp32; g.gelu = gelu;
  g.m_max = m; g.n = n; g.k = k; g.accumulate = accumulate;
  if (accumulate && h->cfg.precision == PSV_FP32) return fail(h, PSV_ERR_INVALID, "accumulate is a bf16-mode epilogue");
  h->launches = 0;
  PSV_CUDA(h, launch_gemm(h, g, (cudaStream_t)stream));
  return PSV_OK;
}

int psv_set_u8_input(PsvHandle *h, int32_t height, int32_t width, const float *mean, const float *std, void *stream) {
  if (!h) return PSV_ERR_INVALID;
  const int S = h->cfg.image;
  if (height < 1 || width < 1 || height > S || width > S)
    return fail(h, PSV_ERR_UNSUPPORTED, "u8 input %dx%d: the fused resize only up-scales (1..%d per side)", height, width, S);
  if (h->cfg.channels != 3) return fail(h, PSV_ERR_UNSUPPORTED, "u8 input needs 3 channels");
  // unchanged geometry and normalisation: nothing to rebuild, and the captured graphs stay valid (the drop-in calls
  // this on every raw-image forward)
  {
    bool same = h->u8_tables && h->u8_h == height && h->u8_w == width;
    for (int c = 0; c < 3 && same; ++c)
      same = h->u8_mean[c] == (mean ? mean[c] : 0.5f) && h->u8_std[c] == (std ? std[c] : 0.5f);
    if (same) return PSV_OK;
  }
  DeviceGuard guard(h->device);
  // Pillow's precompute_coeffs + normalize_coeffs_8bpc for the bilinear filter (support 1 when up-scaling: two taps)
  std::vector<int32_t> t((size_t)6 * S, 0);
  auto fill = [&](int in_size, int32_t *first, int32_t *coef) {
    const double scale = (double)in_size / (double)S, support = 1.0;
    for (int xx = 0; xx < S; ++xx) {
      const double center = (xx + 0.5) * scale;
      int xmin = (int)(center - support + 0.5); if (xmin < 0) xmin = 0;
      int xmax = (int)(center + support + 0.5); if (xmax > in_size) xmax = in_size;
      xmax -= xmin;
      double k[4] = {0, 0, 0, 0}, ww = 0.0;
      for (int x = 0; x < xmax && x < 4; ++x) {
        double a = (x + xmin - center + 0.5); if (a < 0) a = -a;
        k[x] = a < 1.0 ? 1.0 - a : 0.0;
        ww += k[x];
      }
      first[xx] = xmin;
      for (int x = 0; x < 2; ++x) {
        const double w = (x < xmax && ww != 0.0) ? k[x] / ww : 0.0;
        coef[2 * xx + x] = (int32_t)(0.5 + w * (double)(1 << 22));
      }
    }
  };
  fill(width, t.data(), t.data() + S);
  fill(height, t.data() + 3 * S, t.data() + 4 * S);
  if (!h->u8_tables) PSV_CUDA(h, dmalloc(&h->u8_tables, (size_t)6 * S));
  cudaStream_t s = (cudaStream_t)stream;
  PSV_CUDA(h, cudaMemcpyAsync(h->u8_tables, t.data(), t.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  PSV_CUDA(h, cudaStreamSynchronize(s));             // `t` is a stack-lifetime host buffer
  h->u8_h = height; h->u8_w = width;
  for (int c = 0; c < 3; ++c) { h->u8_mean[c] = mean ? mean[c] : 0.5f; h->u8_std[c] = std ? std[c] : 0.5f; }
  drop_graphs(h);                                             // captured graphs baked the previous geometry in
  return PSV_OK;
}

int psv_set_attention_kernel(PsvHandle *h, int32_t kind) {
  if (!h) return PSV_ERR_INVALID;
  if (kind != PSV_ATTENTION_AUTO && kind != PSV_ATTENTION_MMA && kind != PSV_ATTENTION_TC && kind != PSV_ATTENTION_PK)
    return fail(h, PSV_ERR_INVALID, "unknown attention kernel %d", kind);
  h->attention_kernel = kind;
  drop_graphs(h);                                             // captured graphs baked the previous choice in
  return PSV_OK;
}

int psv_set_loss_variant(PsvHandle *h, int32_t variant, float sim_threshold) {
  if (!h) return PSV_ERR_INVALID;
  if (variant != PSV_LOSS_MASK_LABELS && variant != PSV_LOSS_SIMILARITY_LABELS)
    return fail(h, PSV_ERR_INVALID, "unknown loss variant %d", variant);
  h->loss_variant = variant;
  h->loss_st = sim_threshold;
  return PSV_OK;
}

int psv_set_kv_mode(PsvHandle *h, int32_t mode) {
  if (!h) return PSV_ERR_INVALID;
  if (mode != PSV_KV_ACTIVE && mode != PSV_KV_ALL) return fail(h, PSV_ERR_INVALID, "unknown kv mode %d", mode);
  h->kv_mode = mode;
  drop_graphs(h);                                             // captured graphs baked the previous mode in
  return PSV_OK;
}

int psv_set_skip_criterion(PsvHandle *h, int32_t criterion, float sim_threshold) {
  if (!h) return PSV_ERR_INVALID;
  if (criterion != PSV_SKIP_MLP && criterion != PSV_SKIP_SIMILARITY)
    return fail(h, PSV_ERR_INVALID, "unknown skip criterion %d", criterion);
  if (!std::isfinite(sim_threshold)) return fail(h, PSV_ERR_INVALID, "sim_threshold must be finite");
  h->skip_criterion = criterion;
  h->skip_st = sim_threshold;
  drop_graphs(h);                                             // captured graphs baked the previous criterion in
  h->attn_hint_valid = false;                                 // and their token counts
  return PSV_OK;
}

int psv_attention(PsvHandle *h, const void *qkv, const int32_t *cu_seqlens, int32_t batch, int32_t total_rows,
                  void *ctx, void *stream) {
  if (!h || !qkv || !cu_seqlens || !ctx) return fail(h, PSV_ERR_INVALID, "null argument");
  if (batch < 1 || total_rows < 1) return fail(h, PSV_ERR_INVALID, "batch and total_rows must be positive");
  if (!aligned16(qkv) || !aligned16(ctx)) return fail(h, PSV_ERR_INVALID, "qkv/ctx must be 16-byte aligned");
  DeviceGuard guard(h->device);
  h->launches = 0;
  // AUTO resolves to the tcgen05 kernel here (hint = full length); psv_set_attention_kernel selects the other one
  PSV_CUDA(h, launch_attention(h, qkv, ctx, cu_seqlens, batch, total_rows, h->N, (cudaStream_t)stream));
  return PSV_OK;
}

#pragma GCC visibility pop
}  // extern "C"
