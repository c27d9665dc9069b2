// Compressor training path (reference main_model_utils.py:100-191 with loss_type="cosine";
// model_utils.py:95-108, 275-282): loss of one layer's compressor and its gradient with respect to
// the layer's compressor parameters.  The backbone is frozen and the mask is not differentiable, so
// layer l's loss reaches only layer l's four compressor tensors and needs only the layer INPUT.
//
//   y_i   = mask (label, model_utils.py:103)            s_i = sigmoid(z_i)  (the score)
//   pw    = mean(y) / (1 - mean(y) + 1e-16)             (:104-105)
//   loss  = mean_i[(1 - y_i) s_i + (1 + (pw - 1) y_i) softplus(-s_i)]    BCE-with-logits ON THE SCORE (:108)
//   dz_i  = [(1 - y_i) - (1 + (pw - 1) y_i) sigmoid(-s_i)] / M * s_i (1 - s_i)
//   a_ij  = b1_j + W1[j,:D].cls_b + W1[j,D:].x_i        z_i = b2 + sum_j w2_j relu(a_ij)
//   dW2_j = sum_i dz_i relu(a_ij)   db2 = sum_i dz_i    delta_ij = dz_i w2_j [a_ij > 0]
//   db1_j = sum_i delta_ij          dW1[j,D:] = sum_i delta_ij x_i      dW1[j,:D] = sum_b (sum_{i in b} delta_ij) cls_b
//
// All arithmetic is fp32 FFMA (this path is about exactness of the optimisation trajectory, not
// throughput): train_prep (one CTA: label mean, pw, loss) -> comp_bwd (one CTA per image: recompute
// a_ij with the same tiling as the fp32 score kernel, emit delta [M,64], per-image sums and the small
// gradients) -> dw1_tok (split-K FFMA GEMM delta^T . X with atomic accumulation) -> dw1_cls.
#include <cstdlib>

#include "psv_internal.cuh"

namespace psv {
namespace {

constexpr int CH = 64, NP = 196;
// comp_bwd: each image's 196 patch tokens are split over TB_SLICES CTAs (49 tokens each: 7 token groups x 8 hidden
// groups = 56 working threads), so a batch of 64 images fills the GPU (one CTA per image left 84 of 148 SMs idle:
// 222 us per layer).
constexpr int TB_TOK = 7, TB_HID = 8, TB_KC = 32, TB_SLICES = 4, TB_TS = NP / TB_SLICES, TB_TG = TB_TS / TB_TOK;
constexpr int TB_THREADS = 64, TB_XS = TB_TS + 1;
static_assert(TB_TS * TB_SLICES == NP && TB_TG * TB_TOK == TB_TS && TB_TG * 8 <= TB_THREADS, "comp_bwd tiling");

// coef[0] = pw, coef[1] = 1 / M;  loss = mean over the B*196 scores of BCE-with-logits(x, y; pos_weight pw) with
// pw = alpha / (1 - alpha), alpha = mean(y)  (model_utils.py:103-108).  The loss splits into two sums that do not depend
// on pw -- sum[(1 - y) x + sp] + (pw - 1) sum[y sp], sp = softplus(-x) -- so one pass over the scores suffices:
// PREP_CTAS CTAs store their partial (count, S0, S1), the last one to finish (ticket) adds them up in index order
// (deterministic) and writes coef / loss.  (The single-CTA two-pass form took 14.6 us per layer.)
constexpr int PREP_CTAS = 64, PREP_THREADS = 256;
struct PrepScratch { double part[PREP_CTAS][3]; unsigned int ticket; };
__global__ void __launch_bounds__(PREP_THREADS)
train_prep_kernel(const uint8_t *__restrict__ mask, const float *__restrict__ scores, int batch, int N,
                  float fixed_pw, float *__restrict__ coef, float *__restrict__ loss_out, PrepScratch *__restrict__ sc) {
  __shared__ double red[PREP_THREADS / 32][3];
  __shared__ bool last;
  const int total = batch * (N - 1);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double cnt = 0.0, s0 = 0.0, s1 = 0.0;
  for (int e = blockIdx.x * PREP_THREADS + tid; e < total; e += PREP_CTAS * PREP_THREADS) {
    const float y = mask[(size_t)(e / (N - 1)) * N + 1 + e % (N - 1)] ? 1.0f : 0.0f;
    const float x = scores[e];
    const float sp = log1pf(expf(-fabsf(x))) + fmaxf(-x, 0.0f);
    cnt += (double)y;
    s0 += (double)((1.0f - y) * x + sp);
    s1 += (double)(y * sp);
  }
  for (int o = 16; o; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (lane == 0) { red[warp][0] = cnt; red[warp][1] = s0; red[warp][2] = s1; }
  __syncthreads();
  if (tid == 0) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int w = 0; w < PREP_THREADS / 32; ++w) { a += red[w][0]; b += red[w][1]; c += red[w][2]; }
    sc->part[blockIdx.x][0] = a; sc->part[blockIdx.x][1] = b; sc->part[blockIdx.x][2] = c;
    __threadfence();
    last = atomicAdd(&sc->ticket, 1u) == PREP_CTAS - 1;
  }
  __syncthreads();
  if (last && tid == 0) {
    __threadfence();
    double a = 0.0, b = 0.0, c = 0.0;
    for (int i = 0; i < PREP_CTAS; ++i) {
      a += __ldcg(&sc->part[i][0]); b += __ldcg(&sc->part[i][1]); c += __ldcg(&sc->part[i][2]);
    }
    const float alpha = (float)a / (float)total;
    const float pw = fixed_pw > 0.f ? fixed_pw : alpha / (1.0f - alpha + 1e-16f);   // donal/model_utils.py:75 fixes it at 1.5
    coef[0] = pw;
    coef[1] = 1.0f / (float)total;
    if (loss_out) loss_out[0] = (float)((b + ((double)pw - 1.0) * c) / (double)total);
    sc->ticket = 0;                                 // ready for the next layer
  }
}

template <int D>
__global__ void __launch_bounds__(TB_THREADS)
comp_bwd_kernel(const float *__restrict__ hidden, const float *__restrict__ comp, const float *__restrict__ c1_tokT,
                const uint8_t *__restrict__ mask, const float *__restrict__ coef, float grad_scale,
                float *__restrict__ delta,        // [B*196, 64]
                float *__restrict__ dsum,         // [B, 64]   per-image sums of delta
                float *__restrict__ grads) {      // this layer's flat gradient block (small terms, atomics)
  constexpr int N = NP + 1;
  __shared__ float xs[TB_KC][TB_XS];
  __shared__ __align__(16) float ws[TB_KC][CH];
  __shared__ float hc[CH];
  __shared__ float red_w2[TB_TG][CH];
  __shared__ float red_b1[TB_TG][CH];
  __shared__ float red_b2[TB_TG];
  const int b = blockIdx.x, t_first = blockIdx.y * TB_TS, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float *w1 = comp, *b1 = comp + (size_t)CH * 2 * D, *w2 = b1 + CH, *b2 = w2 + CH;
  const float *xb = hidden + (size_t)b * N * D;

  for (int j = warp; j < CH; j += TB_THREADS / 32) {
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
  const int hg = tid & 7, tg = min(tid >> 3, TB_TG - 1);
  const bool worker = (tid >> 3) < TB_TG;
  float acc[TB_TOK][TB_HID];
#pragma unroll
  for (int i = 0; i < TB_TOK; ++i)
#pragma unroll
    for (int j = 0; j < TB_HID; ++j) acc[i][j] = 0.f;
  const float *xt = xb + (size_t)(1 + t_first) * D;
  for (int k0 = 0; k0 < D; k0 += TB_KC) {
    __syncthreads();
    for (int e = tid; e < TB_TS * (TB_KC / 4); e += TB_THREADS) {
      int row = e >> 3, kq = e & 7;
      float4 v = *reinterpret_cast<const float4 *>(xt + (size_t)row * D + k0 + kq * 4);
      xs[kq * 4 + 0][row] = v.x; xs[kq * 4 + 1][row] = v.y;
      xs[kq * 4 + 2][row] = v.z; xs[kq * 4 + 3][row] = v.w;
    }
    for (int e = tid; e < TB_KC * (CH / 4); e += TB_THREADS) {
      int kr = e >> 4, q = e & 15;
      *reinterpret_cast<float4 *>(&ws[kr][q * 4]) =
          *reinterpret_cast<const float4 *>(c1_tokT + (size_t)(k0 + kr) * CH + q * 4);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < TB_KC; ++k) {
      float4 wa = *reinterpret_cast<const float4 *>(&ws[k][hg * 8]);
      float4 wb = *reinterpret_cast<const float4 *>(&ws[k][hg * 8 + 4]);
      float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
      for (int i = 0; i < TB_TOK; ++i) {
        float xv = xs[k][tg * TB_TOK + i];
#pragma unroll
        for (int j = 0; j < TB_HID; ++j) acc[i][j] = fmaf(xv, wv[j], acc[i][j]);
      }
    }
  }
  float w2v[TB_HID], hcv[TB_HID], gw2[TB_HID], gb1[TB_HID];
#pragma unroll
  for (int j = 0; j < TB_HID; ++j) { w2v[j] = w2[hg * 8 + j]; hcv[j] = hc[hg * 8 + j]; gw2[j] = 0.f; gb1[j] = 0.f; }
  const float bias2 = b2[0], pw = coef[0], inv_m = coef[1];
  float gb2 = 0.f;
#pragma unroll
  for (int i = 0; i < TB_TOK; ++i) {
    const int t = t_first + tg * TB_TOK + i;
    float a[TB_HID], z = 0.f;
#pragma unroll
    for (int j = 0; j < TB_HID; ++j) { a[j] = acc[i][j] + hcv[j]; z = fmaf(fmaxf(a[j], 0.f), w2v[j], z); }
    z += __shfl_xor_sync(0xffffffffu, z, 1);
    z += __shfl_xor_sync(0xffffffffu, z, 2);
    z += __shfl_xor_sync(0xffffffffu, z, 4);
    const float s = 1.0f / (1.0f + expf(-(z + bias2)));
    const float y = mask[(size_t)b * N + 1 + t] ? 1.0f : 0.0f;
    const float dl_ds = inv_m * ((1.0f - y) - (1.0f + (pw - 1.0f) * y) / (1.0f + expf(s)));
    const float dz = grad_scale * dl_ds * s * (1.0f - s);
    if (hg == 0) gb2 += dz;
    float dv[TB_HID];
#pragma unroll
    for (int j = 0; j < TB_HID; ++j) {
      gw2[j] = fmaf(dz, fmaxf(a[j], 0.f), gw2[j]);
      dv[j] = a[j] > 0.f ? dz * w2v[j] : 0.f;
      gb1[j] += dv[j];
    }
    if (worker) {
      float *dp = delta + ((size_t)b * NP + t) * CH + hg * 8;
      *reinterpret_cast<float4 *>(dp) = make_float4(dv[0], dv[1], dv[2], dv[3]);
      *reinterpret_cast<float4 *>(dp + 4) = make_float4(dv[4], dv[5], dv[6], dv[7]);
    }
  }
  if (worker) {
#pragma unroll
    for (int j = 0; j < TB_HID; ++j) { red_w2[tg][hg * 8 + j] = gw2[j]; red_b1[tg][hg * 8 + j] = gb1[j]; }
    if (hg == 0) red_b2[tg] = gb2;
  }
  __syncthreads();
  if (tid < CH) {
    float sw = 0.f, sb = 0.f;
    for (int g = 0; g < TB_TG; ++g) { sw += red_w2[g][tid]; sb += red_b1[g][tid]; }
    atomicAdd(dsum + (size_t)b * CH + tid, sb);          // the image's other slices add their share (dsum is zeroed)
    float *g_b1 = grads + (size_t)CH * 2 * D, *g_w2 = g_b1 + CH;
    atomicAdd(g_w2 + tid, sw);
    atomicAdd(g_b1 + tid, sb);
  }
  if (tid == 0) {
    float sb2 = 0.f;
    for (int g = 0; g < TB_TG; ++g) sb2 += red_b2[g];
    atomicAdd(grads + (size_t)CH * 2 * D + 2 * CH, sb2);
  }
}

// Same outputs as comp_bwd_kernel, from the PRE-ACTIVATIONS a[i, j] that the tcgen05 score kernel kept for this
// input (split-bf16 products, ~16 mantissa bits): no second 768-wide product, the kernel is a few MB of traffic.
// grid (batch, 196 / 28), 224 threads: thread = (token of the slice, hidden group of 8).
constexpr int TL_TOK = 28, TL_THREADS = TL_TOK * 8;
__global__ void __launch_bounds__(TL_THREADS)
comp_bwd_light_kernel(const float *__restrict__ preact, const float *__restrict__ comp, int D,
                      const uint8_t *__restrict__ mask, const float *__restrict__ coef, float grad_scale,
                      float *__restrict__ delta, float *__restrict__ dsum, float *__restrict__ grads) {
  constexpr int N = NP + 1;
  __shared__ float red_w2[TL_TOK][CH];
  __shared__ float red_b1[TL_TOK][CH];
  __shared__ float red_b2[TL_TOK];
  const int b = blockIdx.x, tid = threadIdx.x, hg = tid & 7, r = tid >> 3;
  const int t = blockIdx.y * TL_TOK + r;                        // patch token 0..195
  const float *w2 = comp + (size_t)CH * 2 * D + CH, *b2 = w2 + CH;
  const float *ap = preact + ((size_t)b * NP + t) * CH + hg * 8;
  const float4 a0 = *reinterpret_cast<const float4 *>(ap), a1 = *reinterpret_cast<const float4 *>(ap + 4);
  const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
  float w2v[8], z = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) { w2v[j] = w2[hg * 8 + j]; z = fmaf(fmaxf(a[j], 0.f), w2v[j], z); }
  z += __shfl_xor_sync(0xffffffffu, z, 1);
  z += __shfl_xor_sync(0xffffffffu, z, 2);
  z += __shfl_xor_sync(0xffffffffu, z, 4);
  const float pw = coef[0], inv_m = coef[1];
  const float s = 1.0f / (1.0f + expf(-(z + b2[0])));
  const float y = mask[(size_t)b * N + 1 + t] ? 1.0f : 0.0f;
  const float dl_ds = inv_m * ((1.0f - y) - (1.0f + (pw - 1.0f) * y) / (1.0f + expf(s)));
  const float dz = grad_scale * dl_ds * s * (1.0f - s);
  float dv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    dv[j] = a[j] > 0.f ? dz * w2v[j] : 0.f;
    red_w2[r][hg * 8 + j] = dz * fmaxf(a[j], 0.f);
    red_b1[r][hg * 8 + j] = dv[j];
  }
  if (hg == 0) red_b2[r] = dz;
  float *dp = delta + ((size_t)b * NP + t) * CH + hg * 8;
  *reinterpret_cast<float4 *>(dp) = make_float4(dv[0], dv[1], dv[2], dv[3]);
  *reinterpret_cast<float4 *>(dp + 4) = make_float4(dv[4], dv[5], dv[6], dv[7]);
  __syncthreads();
  if (tid < CH) {
    float sw = 0.f, sb = 0.f;
    for (int g = 0; g < TL_TOK; ++g) { sw += red_w2[g][tid]; sb += red_b1[g][tid]; }
    atomicAdd(dsum + (size_t)b * CH + tid, sb);
    float *g_b1 = grads + (size_t)CH * 2 * D, *g_w2 = g_b1 + CH;
    atomicAdd(g_w2 + tid, sw);
    atomicAdd(g_b1 + tid, sb);
  }
  if (tid == CH) {
    float sb2 = 0.f;
    for (int g = 0; g < TL_TOK; ++g) sb2 += red_b2[g];
    atomicAdd(grads + (size_t)CH * 2 * D + 2 * CH, sb2);
  }
}

// part[split][j, c] = sum_{r in split} delta[r, j] * x[r, c]   (x = patch-token rows of the fp32 stream)
// grid (D/128 column blocks, splits); 256 threads: 4 hidden units x 8 columns per thread.  Every split STORES its partial
// [64, D] block; dw1_cls_kernel adds the blocks up in split order -- deterministic (the first version accumulated with
// 2.4 M atomicAdds onto 49 k addresses; the step time is the same either way, 2.67 ms at batch 64).
constexpr int DW_COLS = 128, DW_ROWS = 32, DW_THREADS = 256;
__global__ void __launch_bounds__(DW_THREADS)
dw1_tok_kernel(const float *__restrict__ hidden, const float *__restrict__ delta, int batch, int N, int D,
               float *__restrict__ part) {
  __shared__ __align__(16) float ds[DW_ROWS][CH];
  __shared__ __align__(16) float xs[DW_ROWS][DW_COLS];
  const int c0 = blockIdx.x * DW_COLS;
  const int total = batch * (N - 1);
  const int per = (total + gridDim.y - 1) / gridDim.y;
  const int r_begin = blockIdx.y * per, r_end = min(total, r_begin + per);
  const int tid = threadIdx.x, tj = tid >> 4, tc = tid & 15;     // 16 hidden groups x 16 column groups
  float acc[4][8];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[a][c] = 0.f;
  // software pipeline: the next chunk's global loads (2 + 4 float4 per thread) are in flight while this one is computed
  float4 pd[2], px[4];
  auto fetch = [&](int r0) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int e = tid + i * DW_THREADS, rr = e >> 4, q = e & 15, r = r0 + rr;
      pd[i] = r < r_end ? *reinterpret_cast<const float4 *>(delta + (size_t)r * CH + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + i * DW_THREADS, rr = e >> 5, q = e & 31, r = r0 + rr;
      px[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < r_end) {
        const int b = r / (N - 1), t = r % (N - 1);
        px[i] = *reinterpret_cast<const float4 *>(hidden + ((size_t)b * N + 1 + t) * D + c0 + q * 4);
      }
    }
  };
  if (r_begin < r_end) fetch(r_begin);
  for (int r0 = r_begin; r0 < r_end; r0 += DW_ROWS) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 2; ++i) { const int e = tid + i * DW_THREADS; *reinterpret_cast<float4 *>(&ds[e >> 4][(e & 15) * 4]) = pd[i]; }
#pragma unroll
    for (int i = 0; i < 4; ++i) { const int e = tid + i * DW_THREADS; *reinterpret_cast<float4 *>(&xs[e >> 5][(e & 31) * 4]) = px[i]; }
    __syncthreads();
    if (r0 + DW_ROWS < r_end) fetch(r0 + DW_ROWS);
#pragma unroll 4
    for (int rr = 0; rr < DW_ROWS; ++rr) {
      const float4 dv = *reinterpret_cast<const float4 *>(&ds[rr][tj * 4]);
      const float4 x0 = *reinterpret_cast<const float4 *>(&xs[rr][tc * 8]);
      const float4 x1 = *reinterpret_cast<const float4 *>(&xs[rr][tc * 8 + 4]);
      const float d[4] = {dv.x, dv.y, dv.z, dv.w};
      const float x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[a][c] = fmaf(d[a], x[c], acc[a][c]);
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    float *g = part + ((size_t)blockIdx.y * CH + tj * 4 + a) * D + c0 + tc * 8;
    *reinterpret_cast<float4 *>(g) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
    *reinterpret_cast<float4 *>(g + 4) = make_float4(acc[a][4], acc[a][5], acc[a][6], acc[a][7]);
  }
}

// Tensor-core form of dW1[:, D:] = delta^T . x (the 64 x D x (B*N) product): delta^T as split-bf16 planes [128, Kpad]
// (rows 64..127 and the CLS / padding columns are zero, so the product can run over ALL rows of the stream), x^T by
// split_planes, three stream-K passes of the tcgen05 GEMM into a zeroed [128, D] scratch.  32 stream rows per CTA.
__global__ void __launch_bounds__(256)
delta_planes_kernel(const float *__restrict__ delta, int batch, int N, int kpad, bf16 *__restrict__ hi, bf16 *__restrict__ lo) {
  __shared__ float tile[32][CH + 1];
  const int r0 = blockIdx.x * 32, tid = threadIdx.x;
  for (int e = tid; e < 32 * CH; e += 256) {
    const int rr = e >> 6, j = e & 63, r = r0 + rr;
    const int b = r / N, tok = r - b * N;
    tile[rr][j] = (b < batch && tok > 0) ? delta[((size_t)b * (N - 1) + tok - 1) * CH + j] : 0.f;
  }
  __syncthreads();
  for (int e = tid; e < 32 * CH; e += 256) {
    const int j = e >> 5, rr = e & 31, r = r0 + rr;
    if (r < kpad) {
      const float v = tile[rr][j];
      const bf16 h = __float2bfloat16_rn(v);
      hi[(size_t)j * kpad + r] = h;
      lo[(size_t)j * kpad + r] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
  }
}

// dW1[j, c] = sum_b dsum[b, j] * cls_b[c]    (c < D): one CTA per block of 32 columns, the CLS rows and dsum staged in
// shared memory 64 images at a time, 256 threads = 64 hidden units x 4 column groups of 8.  (One CTA per hidden unit
// with a serial loop over the batch took 33 us per layer.)
constexpr int DC_COLS = 32, DC_IMGS = 64;
__global__ void __launch_bounds__(256)
dw1_cls_kernel(const float *__restrict__ hidden, const float *__restrict__ dsum, int batch, int N, int D,
               float *__restrict__ grads, const float *__restrict__ dw1_tok, int tok_parts) {
  __shared__ __align__(16) float xs[DC_IMGS][DC_COLS];
  __shared__ __align__(16) float ds[DC_IMGS][CH];
  const int c0 = blockIdx.x * DC_COLS, tid = threadIdx.x, j = tid >> 2, cg = tid & 3;
  float acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.f;
  for (int b0 = 0; b0 < batch; b0 += DC_IMGS) {
    const int nb = min(DC_IMGS, batch - b0);
    __syncthreads();
    for (int e = tid; e < DC_IMGS * (DC_COLS / 4); e += 256) {
      const int bb = e >> 3, q = e & 7;
      *reinterpret_cast<float4 *>(&xs[bb][q * 4]) =
          bb < nb ? *reinterpret_cast<const float4 *>(hidden + (size_t)(b0 + bb) * N * D + c0 + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int e = tid; e < DC_IMGS * (CH / 4); e += 256) {
      const int bb = e >> 4, q = e & 15;
      *reinterpret_cast<float4 *>(&ds[bb][q * 4]) =
          bb < nb ? *reinterpret_cast<const float4 *>(dsum + (size_t)(b0 + bb) * CH + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
#pragma unroll 8
    for (int bb = 0; bb < DC_IMGS; ++bb) {               // images in ascending order: the same sum as before
      const float d = ds[bb][j];
      const float4 x0 = *reinterpret_cast<const float4 *>(&xs[bb][cg * 8]);
      const float4 x1 = *reinterpret_cast<const float4 *>(&xs[bb][cg * 8 + 4]);
      acc[0] = fmaf(d, x0.x, acc[0]); acc[1] = fmaf(d, x0.y, acc[1]); acc[2] = fmaf(d, x0.z, acc[2]); acc[3] = fmaf(d, x0.w, acc[3]);
      acc[4] = fmaf(d, x1.x, acc[4]); acc[5] = fmaf(d, x1.y, acc[5]); acc[6] = fmaf(d, x1.z, acc[6]); acc[7] = fmaf(d, x1.w, acc[7]);
    }
  }
  float *g = grads + (size_t)j * 2 * D + c0 + cg * 8;
  *reinterpret_cast<float4 *>(g) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  *reinterpret_cast<float4 *>(g + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
  // the token half: the partial [64 (or 128), D] blocks of dw1_tok_kernel (or the one block of the tensor-core product),
  // added in block order
  float4 t0 = make_float4(0.f, 0.f, 0.f, 0.f), t1 = t0;
  for (int p = 0; p < tok_parts; ++p) {
    const float4 *t = reinterpret_cast<const float4 *>(dw1_tok + ((size_t)p * CH + j) * D + c0 + cg * 8);
    const float4 a = t[0], b = t[1];
    t0.x += a.x; t0.y += a.y; t0.z += a.z; t0.w += a.w;
    t1.x += b.x; t1.y += b.y; t1.z += b.z; t1.w += b.w;
  }
  *reinterpret_cast<float4 *>(g + D) = t0;
  *reinterpret_cast<float4 *>(g + D + 4) = t1;
}

int fail(PsvHandle *h, int code, const char *msg) {
  if (h) h->err = msg;
  return code;
}

}  // namespace

// Enqueue loss + gradient of one layer.  `grads` = that layer's flat block (comp_per_layer floats).
cudaError_t enqueue_compressor_layer_grads(PsvHandle *h, int layer, const float *hidden_in, int batch,
                                           const uint8_t *mask, const float *scores, const float *preact,
                                           float grad_scale, float *grads, float *loss_out, cudaStream_t s) {
  const LayerPack &lp = h->layers[layer];
  cudaError_t e;
  if (!h->train_delta || !h->train_dsum) {          // both or neither: a half-made pair is never left behind
    float *delta = nullptr, *dsum = nullptr;
    e = cudaMalloc((void **)&delta, (size_t)h->cfg.max_batch * (h->N - 1) * CH * sizeof(float));
    if (e != cudaSuccess) return e;
    // dsum | 2 coefficient floats (64 bytes) | PrepScratch (partials + ticket, zeroed once)
    const size_t dsum_bytes = (size_t)h->cfg.max_batch * CH * sizeof(float) + 64;
    e = cudaMalloc((void **)&dsum, dsum_bytes + sizeof(PrepScratch));
    if (e == cudaSuccess) e = cudaMemset(reinterpret_cast<uint8_t *>(dsum) + dsum_bytes, 0, sizeof(PrepScratch));
    if (e != cudaSuccess) { cudaFree(delta); if (dsum) cudaFree(dsum); return e; }
    h->train_delta = delta; h->train_dsum = dsum;
  }
  float *coef = h->train_dsum + (size_t)h->cfg.max_batch * CH;      // 2 floats after dsum
  e = cudaMemsetAsync(grads, 0, (size_t)h->comp_per_layer * sizeof(float), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(h->train_dsum, 0, (size_t)batch * CH * sizeof(float), s);
  if (e != cudaSuccess) return e;
  {
    LaunchScope scope(h, KK_TRAIN, s);
    PrepScratch *sc = reinterpret_cast<PrepScratch *>(reinterpret_cast<uint8_t *>(h->train_dsum) +
                                                      (size_t)h->cfg.max_batch * CH * sizeof(float) + 64);
    train_prep_kernel<<<PREP_CTAS, PREP_THREADS, 0, s>>>(mask, scores, batch, h->N,
                                                         h->loss_variant == PSV_LOSS_SIMILARITY_LABELS ? 1.5f : 0.f, coef,
                                                         loss_out, sc);
  }
  {
    LaunchScope scope(h, KK_TRAIN, s);
    static_assert(NP % TL_TOK == 0, "comp_bwd_light tiling");
    if (preact)
      comp_bwd_light_kernel<<<dim3(batch, NP / TL_TOK), TL_THREADS, 0, s>>>(preact, lp.c1, h->D, mask, coef, grad_scale,
                                                                           h->train_delta, h->train_dsum, grads);
    else if (h->D == 1024)
      comp_bwd_kernel<1024><<<dim3(batch, TB_SLICES), TB_THREADS, 0, s>>>(hidden_in, lp.c1, lp.c1_tokT, mask, coef,
                                                                           grad_scale, h->train_delta, h->train_dsum, grads);
    else if (h->D == 768)
      comp_bwd_kernel<768><<<dim3(batch, TB_SLICES), TB_THREADS, 0, s>>>(hidden_in, lp.c1, lp.c1_tokT, mask, coef,
                                                                          grad_scale, h->train_delta, h->train_dsum, grads);
    else if (h->D == 384)
      comp_bwd_kernel<384><<<dim3(batch, TB_SLICES), TB_THREADS, 0, s>>>(hidden_in, lp.c1, lp.c1_tokT, mask, coef,
                                                                          grad_scale, h->train_delta, h->train_dsum, grads);
    else
      return cudaErrorNotSupported;
  }
  // dW1 token half: the fp32 FFMA split-K kernel, or (PSV_TRAIN_DW1_TC=1) a split-bf16 stream-K product on the tensor
  // cores.  The tensor-core form is correct (same tests) and its three GEMM passes take ~10 us each, but the tcgen05 GEMM
  // wants K-major operands and K is the ROW index here: x must be transposed first (38 MB in, 38 MB out at batch 64),
  // which costs more than the 85 us FFMA kernel it replaces -- 2.91 against 2.67 ms per step at batch 64.  Off by default.
  static const bool want_tc = getenv("PSV_TRAIN_DW1_TC") && atoi(getenv("PSV_TRAIN_DW1_TC")) != 0;
  const bool tc = want_tc && h->D % 128 == 0 && tmap_encode_available();
  const int splits_max = (2 * h->sm_count) / (h->D / DW_COLS) > 2 ? (2 * h->sm_count) / (h->D / DW_COLS) : 2;   // >= the 128 rows of the tensor-core form
  if (!h->train_dw1) {
    float *dw1 = nullptr;
    e = cudaMalloc((void **)&dw1, (size_t)splits_max * CH * h->D * sizeof(float));
    if (e != cudaSuccess) return e;
    h->train_dw1 = dw1;
  }
  int tok_parts = 1;
  if (tc) {
    const int K = batch * h->N, kpad = (K + 63) / 64 * 64;
    if (!h->train_planes) {
      const size_t kmax = ((size_t)h->cfg.max_batch * h->N + 63) / 64 * 64;
      bf16 *planes = nullptr;
      e = cudaMalloc((void **)&planes, (2 * 128 + 2 * (size_t)h->D) * kmax * sizeof(bf16));
      if (e == cudaSuccess) e = cudaMemset(planes, 0, 2 * 128 * kmax * sizeof(bf16));     // rows 64..127 of delta^T stay zero
      if (e == cudaSuccess) e = configure_gemm_tc();
      if (e != cudaSuccess) { cudaFree(planes); return e; }
      h->train_planes = planes;
    }
    const size_t kmax = ((size_t)h->cfg.max_batch * h->N + 63) / 64 * 64;
    // plane storage is sized for max_batch; the operands of this call are laid out densely with row pitch kpad
    SplitPlanes dT{h->train_planes, h->train_planes + 128 * kmax, nullptr};
    SplitPlanes xT{h->train_planes + 2 * 128 * kmax, h->train_planes + 2 * 128 * kmax + (size_t)h->D * kmax, nullptr};
    {
      LaunchScope scope(h, KK_TRAIN, s);
      if (kpad != (int)kmax) {     // a smaller batch than the last call: rows 64..127 must be zero at THIS pitch as well
        e = cudaMemsetAsync(dT.hi + (size_t)64 * kpad, 0, (size_t)64 * kpad * sizeof(bf16), s);
        if (e == cudaSuccess) e = cudaMemsetAsync(dT.lo + (size_t)64 * kpad, 0, (size_t)64 * kpad * sizeof(bf16), s);
        if (e != cudaSuccess) return e;
      }
      delta_planes_kernel<<<(kpad + 31) / 32, 256, 0, s>>>(h->train_delta, batch, h->N, kpad, dT.hi, dT.lo);
    }
    { LaunchScope scope(h, KK_TRAIN, s); e = split_planes(hidden_in, h->D, K, h->D, true, kpad, xT, false, s); }
    if (e == cudaSuccess) e = cudaMemsetAsync(h->train_dw1, 0, (size_t)128 * h->D * sizeof(float), s);
    if (e == cudaSuccess) e = split_gemm(h, dT, xT, h->train_dw1, 128, h->D, kpad, nullptr, nullptr, nullptr, nullptr, nullptr,
                                         false, s, true);
    if (e != cudaSuccess) return e;
  } else {
    LaunchScope scope(h, KK_TRAIN, s);
    const int total = batch * (h->N - 1);
    int splits = splits_max;
    const int max_splits = (total + DW_ROWS - 1) / DW_ROWS;
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
    dw1_tok_kernel<<<dim3(h->D / DW_COLS, splits), DW_THREADS, 0, s>>>(hidden_in, h->train_delta, batch, h->N, h->D,
                                                                         h->train_dw1);
    tok_parts = splits;
  }
  {
    LaunchScope scope(h, KK_TRAIN, s);
    dw1_cls_kernel<<<h->D / DC_COLS, 256, 0, s>>>(hidden_in, h->train_dsum, batch, h->N, h->D, grads, h->train_dw1, tok_parts);
  }
  return cudaGetLastError();
}

}  // namespace psv

using namespace psv;

extern "C" {
#pragma GCC visibility push(default)

int psv_compressor_layer_grads(PsvHandle *h, int32_t layer, const float *hidden_in, int32_t batch,
                               const uint8_t *mask, const float *scores, float grad_scale, float *grads,
                               void *stream) {
  if (!h || !hidden_in || !mask || !scores || !grads) return fail(h, PSV_ERR_INVALID, "null argument");
  if (!h->weights_loaded) return fail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  if (layer < 0 || layer >= h->L || batch < 1 || batch > h->cfg.max_batch)
    return fail(h, PSV_ERR_INVALID, "layer or batch out of range");
  int prev_dev = -1;                              // kernels and the lazy workspaces belong to the handle's device
  cudaGetDevice(&prev_dev);
  if (prev_dev != h->device) cudaSetDevice(h->device);
  h->launches = 0;
  cudaError_t e = enqueue_compressor_layer_grads(h, layer, hidden_in, batch, mask, scores, nullptr, grad_scale, grads, nullptr,
                                                 (cudaStream_t)stream);
  if (prev_dev != h->device && prev_dev >= 0) cudaSetDevice(prev_dev);
  if (e != cudaSuccess) { h->err = std::string("compressor gradient launch failed: ") + cudaGetErrorString(e); return PSV_ERR_CUDA; }
  return PSV_OK;
}

#pragma GCC visibility pop
}
