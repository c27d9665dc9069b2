// K1/K2: fused compressor MLP -> sigmoid -> threshold -> skip mask  (reference model_utils.py:62-68)
// and the stable per-image compaction + gather + LayerNorm1       (model_utils.py:88-91, HF:333).
//
// score_mask_kernel: one CTA per image.  The reference materialises cat([CLS.repeat(196), tok])
// [B,196,2D] and runs Linear(2D,64); here the CLS half  W1[:, :D].cls + b1  is computed once per
// image and the token half is a 196 x 64 x D fp32 FFMA mini-GEMM tiled through shared memory,
// fused with ReLU, the 64-wide dot with w2, the sigmoid and the `>= mt` decision.  fp32 FFMA
// keeps scores within ~1e-7 of the reference so masks are bit-exact outside the 1e-4 band.
//
// gather_ln_kernel: grid (B, SLICES).  Each CTA recomputes the image's row offset (sum of
// n_active of the preceding images -- a few hundred L2 hits, cheaper than a separate scan
// launch), ranks the image's active tokens with warp ballots (ascending token order = the
// bit-exact idx contract), writes idx / cu_seqlens, and LayerNorms its slice of the active rows
// straight from the residual stream into the packed [T, D] GEMM operand.
#include "psv_internal.cuh"

namespace psv {

namespace {

constexpr int SC_TOK_PER_THREAD = 7;
constexpr int SC_HID_PER_THREAD = 8;
constexpr int SC_KC = 32;                       // k-chunk staged in shared memory
constexpr int SC_THREADS = 224;                 // 28 token groups x 8 hidden groups
constexpr int SC_NP = 196;                      // patch tokens (hard-coded 196 in the reference, :16,:62)
constexpr int SC_XS_STRIDE = 197;

template <int D>
__global__ void __launch_bounds__(SC_THREADS)
score_mask_kernel(const float *__restrict__ hidden,      // [B, N, D]
                  const float *__restrict__ comp,        // flat compressor params of this layer
                  const float *__restrict__ c1_tokT,     // [D, 64]  token half of W1, transposed
                  float mt, const uint8_t *__restrict__ forced,   // nullable [B, N]
                  uint8_t *__restrict__ mask,            // [B, N] workspace
                  float *__restrict__ scores,            // [B, 196] workspace
                  int32_t *__restrict__ n_active,        // [B]
                  uint8_t *__restrict__ mask_out, float *__restrict__ scores_out,
                  int32_t *__restrict__ n_active_out, int32_t *__restrict__ unit_count) {
  constexpr int CH = 64;
  if (blockIdx.x == 0 && threadIdx.x == 0) *unit_count = 0;     // the compaction kernel appends the attention work units
  constexpr int N = SC_NP + 1;
  __shared__ float xs[SC_KC][SC_XS_STRIDE];
  __shared__ __align__(16) float ws[SC_KC][CH];
  __shared__ float hc[CH];
  __shared__ int count;

  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float *w1 = comp;                          // [64, 2D]
  const float *b1 = comp + (size_t)CH * 2 * D;
  const float *w2 = b1 + CH;
  const float *b2 = w2 + CH;
  const float *xb = hidden + (size_t)b * N * D;

  if (tid == 0) count = 0;
  // CLS half: hc[j] = b1[j] + W1[j, 0:D] . cls
  for (int j = warp; j < CH; j += SC_THREADS / 32) {
    const float *wr = w1 + (size_t)j * 2 * D;
    float acc = 0.f;
    for (int k = lane * 4; k < D; k += 128) {
      float4 wv = *reinterpret_cast<const float4 *>(wr + k);
      float4 xv = *reinterpret_cast<const float4 *>(xb + k);
      acc = fmaf(wv.x, xv.x, acc); acc = fmaf(wv.y, xv.y, acc);
      acc = fmaf(wv.z, xv.z, acc); acc = fmaf(wv.w, xv.w, acc);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) hc[j] = acc + b1[j];
  }

  const int hg = tid & 7, tg = tid >> 3;           // hidden group 0..7, token group 0..27
  float acc[SC_TOK_PER_THREAD][SC_HID_PER_THREAD];
#pragma unroll
  for (int i = 0; i < SC_TOK_PER_THREAD; ++i)
#pragma unroll
    for (int j = 0; j < SC_HID_PER_THREAD; ++j) acc[i][j] = 0.f;

  const float *xt = xb + D;                        // patch tokens start at row 1
  for (int k0 = 0; k0 < D; k0 += SC_KC) {
    __syncthreads();
    // token tile: 196 rows x 32 floats, 8 lanes per row (float4 each), stored transposed
    for (int e = tid; e < SC_NP * (SC_KC / 4); e += SC_THREADS) {
      int row = e >> 3, kq = e & 7;
      float4 v = *reinterpret_cast<const float4 *>(xt + (size_t)row * D + k0 + kq * 4);
      xs[kq * 4 + 0][row] = v.x; xs[kq * 4 + 1][row] = v.y;
      xs[kq * 4 + 2][row] = v.z; xs[kq * 4 + 3][row] = v.w;
    }
    // weight tile: 32 rows (k) x 64 floats, already k-major in c1_tokT
    for (int e = tid; e < SC_KC * (CH / 4); e += SC_THREADS) {
      int kr = e >> 4, q = e & 15;
      *reinterpret_cast<float4 *>(&ws[kr][q * 4]) =
          *reinterpret_cast<const float4 *>(c1_tokT + (size_t)(k0 + kr) * CH + q * 4);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < SC_KC; ++k) {
      float4 wa = *reinterpret_cast<const float4 *>(&ws[k][hg * 8]);
      float4 wb = *reinterpret_cast<const float4 *>(&ws[k][hg * 8 + 4]);
      float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
      for (int i = 0; i < SC_TOK_PER_THREAD; ++i) {
        float xv = xs[k][tg * SC_TOK_PER_THREAD + i];
#pragma unroll
        for (int j = 0; j < SC_HID_PER_THREAD; ++j) acc[i][j] = fmaf(xv, wv[j], acc[i][j]);
      }
    }
  }

  // ReLU, dot with w2 over the 64 hidden units (8 here, 8 lanes across), sigmoid, threshold
  float w2v[SC_HID_PER_THREAD], hcv[SC_HID_PER_THREAD];
#pragma unroll
  for (int j = 0; j < SC_HID_PER_THREAD; ++j) { w2v[j] = w2[hg * 8 + j]; hcv[j] = hc[hg * 8 + j]; }
  const float bias2 = b2[0];
  int local = 0;
#pragma unroll
  for (int i = 0; i < SC_TOK_PER_THREAD; ++i) {
    float z = 0.f;
#pragma unroll
    for (int j = 0; j < SC_HID_PER_THREAD; ++j) z = fmaf(fmaxf(acc[i][j] + hcv[j], 0.f), w2v[j], z);
    z += __shfl_xor_sync(0xffffffffu, z, 1);
    z += __shfl_xor_sync(0xffffffffu, z, 2);
    z += __shfl_xor_sync(0xffffffffu, z, 4);
    if (hg == 0) {
      const int t = tg * SC_TOK_PER_THREAD + i;
      const float s = 1.0f / (1.0f + expf(-(z + bias2)));
      uint8_t m = forced ? (forced[(size_t)b * N + 1 + t] != 0) : (s >= mt);
      local += m;
      mask[(size_t)b * N + 1 + t] = m;
      scores[(size_t)b * SC_NP + t] = s;
      if (mask_out) mask_out[(size_t)b * N + 1 + t] = m;
      if (scores_out) scores_out[(size_t)b * SC_NP + t] = s;
    }
  }
  if (hg == 0 && local) atomicAdd(&count, local);
  __syncthreads();
  if (tid == 0) {
    mask[(size_t)b * N] = 1;                       // CLS column is always processed (:67-68)
    if (mask_out) mask_out[(size_t)b * N] = 1;
    n_active[b] = count + 1;
    if (n_active_out) n_active_out[b] = count + 1;
  }
}

// ---------------------------------------------------------------------------------------------
constexpr int GL_THREADS = 256;
constexpr int GL_SLICES = 4;

template <typename OutT> struct Store4;
template <> struct Store4<float> {
  static __device__ __forceinline__ void st(float *p, float a, float b, float c, float d) {
    *reinterpret_cast<float4 *>(p) = make_float4(a, b, c, d);
  }
};
template <> struct Store4<bf16> {
  static __device__ __forceinline__ void st(bf16 *p, float a, float b, float c, float d) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    uint2 v;
    v.x = *reinterpret_cast<uint32_t *>(&lo);
    v.y = *reinterpret_cast<uint32_t *>(&hi);
    *reinterpret_cast<uint2 *>(p) = v;
  }
};

// LayerNorm of one row held by a warp (D/128 float4 per lane): two-pass fp32 statistics.
template <int D, typename OutT>
__device__ __forceinline__ void warp_layernorm_row(const float *__restrict__ src, OutT *__restrict__ dst,
                                                   const float *__restrict__ gamma,
                                                   const float *__restrict__ beta, float eps, int lane) {
  constexpr int V = D / 128;
  float4 v[V];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    v[i] = *reinterpret_cast<const float4 *>(src + (i * 32 + lane) * 4);
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * (1.0f / D);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    sq += (a * a + b * b) + (c * c + d * d);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = 1.0f / sqrtf(sq * (1.0f / D) + eps);
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = (i * 32 + lane) * 4;
    float4 g = *reinterpret_cast<const float4 *>(gamma + c);
    float4 be = *reinterpret_cast<const float4 *>(beta + c);
    Store4<OutT>::st(dst + c, (v[i].x - mean) * rstd * g.x + be.x, (v[i].y - mean) * rstd * g.y + be.y,
                     (v[i].z - mean) * rstd * g.z + be.z, (v[i].w - mean) * rstd * g.w + be.w);
  }
}

// LayerNorm of one row that was staged in shared memory by a bulk copy (TMA-staged variant of the gather, below)
template <int D, typename OutT>
__device__ __forceinline__ void warp_layernorm_row_smem(const float *src, OutT *__restrict__ dst,
                                                        const float *__restrict__ gamma, const float *__restrict__ beta,
                                                        float eps, int lane) {
  warp_layernorm_row<D, OutT>(src, dst, gamma, beta, eps, lane);
}
__device__ __forceinline__ uint32_t gl_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
constexpr int GL_RING = 2;               // staged rows per warp

// TMA_STAGE (PSV_GATHER_TMA=1, north-star item "TMA-staged gather of active tokens with fused LayerNorm"): every warp
// brings its rows into shared memory with cp.async.bulk (one 3 KB bulk copy per row, completion on an mbarrier, up to
// GL_RING rows in flight per warp) and normalises them from there; the default path loads the row with six 16-byte
// ld.global per lane.  Same arithmetic, same bits.
template <int D, typename OutT, bool TMA_STAGE>
__global__ void __launch_bounds__(GL_THREADS)
gather_ln_kernel(const float *__restrict__ hidden, const uint8_t *__restrict__ mask,
                 const int32_t *__restrict__ n_active, const int2 *__restrict__ n_tile,
                 const float *__restrict__ gamma,
                 const float *__restrict__ beta, float eps, int N, int B, int tile_rows,
                 int32_t *__restrict__ idx, int32_t *__restrict__ cu_seqlens, int32_t *__restrict__ n_active_out,
                 int4 *__restrict__ units, int32_t *__restrict__ unit_count, OutT *__restrict__ out) {
  __shared__ int warp_sums[GL_THREADS / 32];
  __shared__ int warp_cnt[8];
  __shared__ int16_t tok_of_rank[256];
  __shared__ int s_offset;
  const int b = blockIdx.x, slice = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_launch_dependents();
  pdl_wait();

  // row offset of this image = sum of the active counts of the images before it.  Counts come either per image
  // (fp32 score kernel) or per 128-row tile of the flat [B*N] row space (tcgen05 score kernel: n_tile[t] = counts
  // of the tile's first / second image; a tile touches at most two images because N > 128).
  int part = 0, nb_tiles = 0;
  if (n_tile) {
    const int t0 = (b * N) / tile_rows, t1 = (b * N + N - 1) / tile_rows;
    for (int i = tid; i < t0; i += GL_THREADS) { const int2 c = n_tile[i]; part += c.x + c.y; }
    if (tid == 0 && (t0 * tile_rows) / N < b) part += n_tile[t0].x;      // the previous image's share of tile t0
    for (int t = t0; t <= t1; ++t) {
      const int2 c = n_tile[t];
      nb_tiles += (b == (t * tile_rows) / N) ? c.x : c.y;
    }
  } else {
    for (int i = tid; i < b; i += GL_THREADS) part += n_active[i];
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if (lane == 0) warp_sums[warp] = part;
  // rank the active tokens of this image (N <= 256)
  const int t = tid;
  const bool on = (t < N) && mask[(size_t)b * N + t];
  const unsigned ball = __ballot_sync(0xffffffffu, on);
  if (lane == 0) warp_cnt[warp] = __popc(ball);
  __syncthreads();
  if (tid == 0) {
    int s = 0;
    for (int w = 0; w < GL_THREADS / 32; ++w) s += warp_sums[w];
    s_offset = s;
  }
  int before = 0;
  for (int w = 0; w < warp; ++w) before += warp_cnt[w];
  if (on) tok_of_rank[before + __popc(ball & ((1u << lane) - 1u))] = (int16_t)t;
  __syncthreads();
  const int offset = s_offset;
  const int nb = n_tile ? nb_tiles : n_active[b];
  if (slice == 0 && tid == 0) {
    cu_seqlens[b] = offset;
    if (n_active_out) n_active_out[b] = nb;
    if (b == B - 1) cu_seqlens[B] = offset + nb;
  }
  // attention work units of this image (attention_pk.cu): one per block of 32 queries, appended to a flat table; the
  // score kernel zeroed the counter.  The order of the table is arbitrary, the units themselves are not.
  if (slice == 0 && tid < 32) {
    const int nu = (nb + 31) >> 5;
    int base = 0;
    if (tid == 0) base = atomicAdd(unit_count, nu);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (tid < nu) units[base + tid] = make_int4(offset + tid * 32, offset, offset + nb, b);
  }
  const int chunk = (nb + GL_SLICES - 1) / GL_SLICES;
  const int r_end = min(nb, (slice + 1) * chunk);
  if (TMA_STAGE && out) {
    extern __shared__ __align__(128) uint8_t stage_raw[];        // [warps][GL_RING][D] fp32 + barriers
    float *stage = reinterpret_cast<float *>(stage_raw) + (size_t)warp * GL_RING * D;
    uint64_t *bar = reinterpret_cast<uint64_t *>(stage_raw + (size_t)(GL_THREADS / 32) * GL_RING * D * 4) + warp * GL_RING;
    if (lane == 0) {
      for (int i = 0; i < GL_RING; ++i)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(gl_smem_u32(&bar[i])));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const int r_first = slice * chunk + warp, step = GL_THREADS / 32;
    auto issue = [&](int r, int slot) {
      if (lane == 0 && r < r_end) {
        const float *src = hidden + (size_t)(b * N + tok_of_rank[r]) * D;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gl_smem_u32(&bar[slot])), "r"(D * 4) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(gl_smem_u32(stage + (size_t)slot * D)), "l"(src), "r"(D * 4), "r"(gl_smem_u32(&bar[slot])) : "memory");
      }
    };
    for (int i = 0; i < GL_RING; ++i) issue(r_first + i * step, i);
    int k = 0;
    for (int r = r_first; r < r_end; r += step, ++k) {
      const int slot = k % GL_RING;
      const uint32_t parity = (uint32_t)(k / GL_RING) & 1u;
      uint32_t ok = 0;
      while (!ok)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(gl_smem_u32(&bar[slot])), "r"(parity) : "memory");
      if (lane == 0) idx[offset + r] = b * N + tok_of_rank[r];
      warp_layernorm_row_smem<D, OutT>(stage + (size_t)slot * D, out + (size_t)(offset + r) * D, gamma, beta, eps, lane);
      __syncwarp();                                   // every lane has read the slot before it is refilled
      issue(r + GL_RING * step, slot);
    }
    return;
  }
  for (int r = slice * chunk + warp; r < r_end; r += GL_THREADS / 32) {
    const int row = b * N + tok_of_rank[r];
    if (lane == 0) idx[offset + r] = row;
    if (out) warp_layernorm_row<D, OutT>(hidden + (size_t)row * D, out + (size_t)(offset + r) * D, gamma, beta, eps, lane);
  }
}

template <int D, typename OutT>
__global__ void __launch_bounds__(GL_THREADS)
ln_rows_kernel(const float *__restrict__ x, const int32_t *__restrict__ row_idx, const float *__restrict__ gamma,
               const float *__restrict__ beta, float eps, int rows_max, const int32_t *__restrict__ rows_dev,
               OutT *__restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const int rows = rows_dev ? min(*rows_dev, rows_max) : rows_max;
  const int lane = threadIdx.x & 31;
  const int wpb = GL_THREADS / 32;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows; r += gridDim.x * wpb)
    warp_layernorm_row<D, OutT>(x + (size_t)(row_idx ? row_idx[r] : r) * D, out + (size_t)r * D, gamma, beta, eps,
                                lane);
}

}  // namespace

cudaError_t launch_score_mask(PsvHandle *h, const LayerPack &lp, const float *hidden, int batch, float mt,
                              const uint8_t *forced_mask, uint8_t *mask_out, float *scores_out,
                              int32_t *n_active_out, cudaStream_t s) {
  LaunchScope scope(h, KK_SCORE, s);
  if (h->D == 1024)
    score_mask_kernel<1024><<<batch, SC_THREADS, 0, s>>>(hidden, lp.c1, lp.c1_tokT, mt, forced_mask, h->mask,
                                                         h->scores, h->n_active, mask_out, scores_out, n_active_out,
                                                         h->attn_unit_count);
  else if (h->D == 768)
    score_mask_kernel<768><<<batch, SC_THREADS, 0, s>>>(hidden, lp.c1, lp.c1_tokT, mt, forced_mask, h->mask,
                                                        h->scores, h->n_active, mask_out, scores_out, n_active_out,
                                                        h->attn_unit_count);
  else if (h->D == 384)
    score_mask_kernel<384><<<batch, SC_THREADS, 0, s>>>(hidden, lp.c1, lp.c1_tokT, mt, forced_mask, h->mask,
                                                        h->scores, h->n_active, mask_out, scores_out, n_active_out,
                                                        h->attn_unit_count);
  else
    return cudaErrorNotSupported;
  return cudaGetLastError();
}

// Gather + LN1 of the active rows of `hidden` into h->act_a; also writes h->idx / h->cu_seqlens.
// index_only: just the compaction (idx / cu_seqlens / n_active) -- the keep-all-keys mode normalises ALL rows itself.
cudaError_t launch_gather_ln(PsvHandle *h, const LayerPack &lp, const float *hidden, int batch,
                             int32_t *n_active_out, bool tile_counts, cudaStream_t s, bool index_only) {
  LaunchScope scope(h, KK_GATHER_LN, s);
  const int2 *n_tile = tile_counts ? (const int2 *)h->n_tile : nullptr;
  dim3 grid(batch, GL_SLICES);
  const float eps = h->cfg.ln_eps;
  cudaError_t e = cudaSuccess;
  static const bool tma_stage = getenv("PSV_GATHER_TMA") != nullptr && atoi(getenv("PSV_GATHER_TMA")) != 0;
  const bool use_tma = tma_stage && !index_only && h->cfg.precision == PSV_BF16;
#define PSV_GL_ARGS(TT)                                                                                             \
  hidden, (const uint8_t *)h->mask, (const int32_t *)h->n_active, n_tile, (const float *)lp.ln1_w,                  \
  (const float *)lp.ln1_b, eps, h->N, batch, h->score_tile_rows, h->idx, h->cu_seqlens, n_active_out,               \
  (int4 *)h->attn_units, h->attn_unit_count, index_only ? (TT *)nullptr : (TT *)h->act_a
#define PSV_GL(DD, TT)                                                                                              \
  e = use_tma ? launch_pdl(gather_ln_kernel<DD, TT, true>, grid, dim3(GL_THREADS),                                  \
                           (size_t)(GL_THREADS / 32) * GL_RING * (DD * 4 + 8), s, PSV_GL_ARGS(TT))                  \
              : launch_pdl(gather_ln_kernel<DD, TT, false>, grid, dim3(GL_THREADS), 0, s, PSV_GL_ARGS(TT))
  if (use_tma) {                                   // > 48 KB of dynamic shared memory: opt in once (outside any capture)
    static bool configured = false;
    if (!configured) {
      cudaFuncSetAttribute(gather_ln_kernel<1024, bf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (GL_THREADS / 32) * GL_RING * (1024 * 4 + 8));
      cudaFuncSetAttribute(gather_ln_kernel<768, bf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (GL_THREADS / 32) * GL_RING * (768 * 4 + 8));
      cudaFuncSetAttribute(gather_ln_kernel<384, bf16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (GL_THREADS / 32) * GL_RING * (384 * 4 + 8));
      configured = true;
    }
  }
  if (!psv_hidden_supported(h->D)) return cudaErrorNotSupported;
  if (h->cfg.precision == PSV_BF16) {
    if (h->D == 1024) PSV_GL(1024, bf16); else if (h->D == 768) PSV_GL(768, bf16); else PSV_GL(384, bf16);
  } else {
    if (h->D == 1024) PSV_GL(1024, float); else if (h->D == 768) PSV_GL(768, float); else PSV_GL(384, float);
  }
#undef PSV_GL
#undef PSV_GL_ARGS
  return e;
}

cudaError_t launch_ln_rows(PsvHandle *h, const float *x, const int32_t *row_idx, const float *gamma,
                           const float *beta, void *out, int rows_max, const int32_t *rows_dev, cudaStream_t s,
                           bool bf16_out) {
  LaunchScope scope(h, KK_LN, s);
  const float eps = h->cfg.ln_eps;
  int grid = min((rows_max + 7) / 8, h->sm_count * 8);
  if (grid < 1) grid = 1;
  cudaError_t e = cudaSuccess;
#define PSV_LN(DD, TT) \
  e = launch_pdl(ln_rows_kernel<DD, TT>, dim3(grid), dim3(GL_THREADS), 0, s, x, row_idx, gamma, beta, eps, rows_max, \
                 rows_dev, (TT *)out)
  if (!psv_hidden_supported(h->D)) return cudaErrorNotSupported;
  if (h->cfg.precision == PSV_BF16 || bf16_out) {
    if (h->D == 1024) PSV_LN(1024, bf16); else if (h->D == 768) PSV_LN(768, bf16); else PSV_LN(384, bf16);
  } else {
    if (h->D == 1024) PSV_LN(1024, float); else if (h->D == 768) PSV_LN(768, float); else PSV_LN(384, float);
  }
#undef PSV_LN
  return e;
}

}  // namespace psv
