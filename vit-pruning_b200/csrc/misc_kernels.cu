// Small HBM-bound kernels around the GEMMs: patch extraction (K0 front), CLS rows, the
// classification head (K12), weight casts/repacks, and the label path of model_utils.py:95-113
// (similarity, loss, accuracy, confusion counts) plus the similarity skip criterion.
#include "psv_internal.cuh"

namespace psv {
namespace {

// ---- K0 front: pixels [B,C,H,W] -> patches [B*P2, C*p*p], column = c*p*p + i*p + j -------------
// (matches the flattened conv weight [D, C, p, p] of HF:153-167, so the conv is a plain GEMM)
// One CTA per (image, patch row): it walks the C * p image rows of that stripe with 16-byte loads along the
// image row (896 contiguous bytes for 224 fp32 pixels) and writes 4-element pieces of the patch rows; 32-bit
// index arithmetic only (the first version spent most of its time in 64-bit div/mod per element).
template <typename InT> struct Vec4 { };
template <> struct Vec4<float> {
  static __device__ __forceinline__ void load(const float *p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4 *>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float *p, const float (&v)[4]) {
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct Vec4<bf16> {
  static __device__ __forceinline__ void load(const bf16 *p, float (&v)[4]) {
    const uint2 t = *reinterpret_cast<const uint2 *>(p);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&t.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&t.y));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
  static __device__ __forceinline__ void store(bf16 *p, const float (&v)[4]) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    uint2 t; t.x = *reinterpret_cast<uint32_t *>(&a); t.y = *reinterpret_cast<uint32_t *>(&b);
    *reinterpret_cast<uint2 *>(p) = t;
  }
};
template <typename InT, typename OutT>
__global__ void __launch_bounds__(256)
im2col_kernel(const InT *__restrict__ px, OutT *__restrict__ out, int batch, int C, int img, int p) {
  pdl_wait();
  const int g = img / p;                 // patches per side
  const int b = blockIdx.x / g, py = blockIdx.x % g;
  const int kp = C * p * p, quads = img / 4;
  const int total = C * p * quads;       // float4 pieces of this stripe
  const InT *src0 = px + ((size_t)b * C * img + (size_t)py * p) * img;
  OutT *dst0 = out + ((size_t)b * g * g + (size_t)py * g) * kp;
  for (int e = threadIdx.x; e < total; e += 256) {
    const int x = (e % quads) * 4, ci = e / quads;       // ci = c * p + i
    const int c = ci / p, i = ci - c * p;
    float v[4];
    Vec4<InT>::load(src0 + ((size_t)c * img + i) * img + x, v);
    const int pxx = x / p, j = x - pxx * p;
    Vec4<OutT>::store(dst0 + (size_t)pxx * kp + ci * p + j, v);
  }
}

// Raw uint8 [B, H0, W0, 3] images -> patch rows, with Pillow's bilinear resize (ImagingResample: separable, fixed-point
// coefficients with 22 fractional bits, horizontal pass then vertical pass, each rounded and clipped to uint8), the
// 1/255 rescale and the (x - mean) / std normalisation of HuggingFace's ViTImageProcessor fused in (reference
// main_model_utils.py:54-60 does this per sample on the host).  One CTA per (image, patch row): the horizontally
// resized source rows the stripe needs (at most p * H0 / img + 3) live in shared memory.  Up-scaling only (two taps).
constexpr int U8_MAX_ROWS = 20;
template <typename OutT>
__global__ void __launch_bounds__(256)
im2col_u8_kernel(const uint8_t *__restrict__ src, OutT *__restrict__ out, int H0, int W0, int C, int img, int p,
                 const int32_t *__restrict__ tables, float m0, float m1, float m2, float s0, float s1, float s2) {
  extern __shared__ uint8_t tmp[];                   // [rows][img][C]
  pdl_wait();
  const int g = img / p, b = blockIdx.x / g, py = blockIdx.x % g;
  const int32_t *fx = tables, *cx = fx + img, *fy = cx + 2 * img, *cy = fy + img;
  const uint8_t *sb = src + (size_t)b * H0 * W0 * C;
  if (H0 == img && W0 == img && (img * C) % 16 == 0) {
    // Source already at the model's size: Pillow's two-tap filter degenerates to the identity (coefficients 1 and 0), so
    // the stripe's p source rows -- one contiguous block of the HWC image -- are staged with 16-byte loads and only
    // rescaled / normalised.  Same values as the general path below, ~4x less time for 224 x 224 sources.
    const uint4 *s16 = reinterpret_cast<const uint4 *>(sb + (size_t)py * p * img * C);
    uint4 *t16 = reinterpret_cast<uint4 *>(tmp);
    for (int e = threadIdx.x; e < p * img * C / 16; e += 256) t16[e] = s16[e];
    __syncthreads();
    const int kp = C * p * p, quads = img / 4;
    OutT *dst0 = out + ((size_t)b * g * g + (size_t)py * g) * kp;
    const float inv255 = (float)(1.0 / 255.0);
    for (int e = threadIdx.x; e < C * p * quads; e += 256) {
      const int x = (e % quads) * 4, ci = e / quads;
      const int c = ci / p, i = ci - c * p;
      const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2), stdv = c == 0 ? s0 : (c == 1 ? s1 : s2);
      float v[4];
#pragma unroll
      for (int t = 0; t < 4; ++t)
        v[t] = __fdiv_rn(__fsub_rn(__fmul_rn((float)tmp[(i * img + x + t) * C + c], inv255), mean), stdv);
      const int pxx = x / p, j = x - pxx * p;
      Vec4<OutT>::store(dst0 + (size_t)pxx * kp + ci * p + j, v);
    }
    return;
  }
  const int r_lo = fy[py * p], r_hi = min(fy[py * p + p - 1] + 1, H0 - 1), rows = r_hi - r_lo + 1;
  const int half = 1 << 21;
  for (int e = threadIdx.x; e < rows * img * C; e += 256) {
    const int c = e % C, xx = (e / C) % img, r = e / (C * img);
    const int x0 = fx[xx], x1 = min(x0 + 1, W0 - 1);
    const uint8_t *row = sb + (size_t)(r_lo + r) * W0 * C;
    const int acc = half + (int)row[x0 * C + c] * cx[2 * xx] + (int)row[x1 * C + c] * cx[2 * xx + 1];
    tmp[e] = (uint8_t)min(max(acc >> 22, 0), 255);
  }
  __syncthreads();
  const int kp = C * p * p, quads = img / 4;
  OutT *dst0 = out + ((size_t)b * g * g + (size_t)py * g) * kp;
  const float inv255 = (float)(1.0 / 255.0);
  for (int e = threadIdx.x; e < C * p * quads; e += 256) {
    const int x = (e % quads) * 4, ci = e / quads;
    const int c = ci / p, i = ci - c * p, y = py * p + i;
    const int t0 = fy[y] - r_lo, t1 = min(t0 + 1, rows - 1), k0 = cy[2 * y], k1 = cy[2 * y + 1];
    const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2), stdv = c == 0 ? s0 : (c == 1 ? s1 : s2);
    float v[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int acc = half + (int)tmp[(t0 * img + x + t) * C + c] * k0 + (int)tmp[(t1 * img + x + t) * C + c] * k1;
      const float u = (float)min(max(acc >> 22, 0), 255);
      v[t] = __fdiv_rn(__fsub_rn(__fmul_rn(u, inv255), mean), stdv);
    }
    const int pxx = x / p, j = x - pxx * p;
    Vec4<OutT>::store(dst0 + (size_t)pxx * kp + ci * p + j, v);
  }
}

__global__ void cls_rows_kernel(float *__restrict__ hidden, const float *__restrict__ cls,
                                const float *__restrict__ pos, int batch, int N, int D) {
  pdl_wait();
  const int total = batch * D;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int b = e / D, d = e % D;
    hidden[(size_t)b * N * D + d] = cls[d] + pos[d];
  }
}

// ---- K12: final LayerNorm of the CLS row + classifier ------------------------------------------
// HEAD_IMGS images per CTA: one warp normalises one CLS row (two-pass fp32 statistics, as torch's
// native_layer_norm), then every classifier row that a warp loads serves all the CTA's images and two classes
// are in flight per warp (the kernel is a latency chain of L2 loads and shuffles, not a bandwidth problem).
constexpr int HEAD_IMGS = 4;
__global__ void __launch_bounds__(256)
head_kernel(const float *__restrict__ hidden, const float *__restrict__ gamma, const float *__restrict__ beta,
            const float *__restrict__ cw, const float *__restrict__ cb, float eps, int N, int D, int C, int batch,
            float *__restrict__ logits) {
  extern __shared__ __align__(16) float rows[];          // [HEAD_IMGS][D]
  const int b0 = blockIdx.x * HEAD_IMGS, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nimg = min(HEAD_IMGS, batch - b0);
  pdl_wait();
  if (warp < nimg) {
    const float *x = hidden + (size_t)(b0 + warp) * N * D;
    float *row = rows + warp * D;
    float s = 0.f;
    for (int d = lane * 4; d < D; d += 128) {
      const float4 v = *reinterpret_cast<const float4 *>(x + d);
      *reinterpret_cast<float4 *>(row + d) = v;
      s += (v.x + v.y) + (v.z + v.w);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / D;
    float q = 0.f;
    for (int d = lane * 4; d < D; d += 128) {
      const float4 v = *reinterpret_cast<const float4 *>(row + d);
      const float c0 = v.x - mean, c1 = v.y - mean, c2 = v.z - mean, c3 = v.w - mean;
      q += (c0 * c0 + c1 * c1) + (c2 * c2 + c3 * c3);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = 1.0f / sqrtf(q / D + eps);
    for (int d = lane * 4; d < D; d += 128) {
      float4 v = *reinterpret_cast<const float4 *>(row + d);
      const float4 g = *reinterpret_cast<const float4 *>(gamma + d), be = *reinterpret_cast<const float4 *>(beta + d);
      v.x = (v.x - mean) * rstd * g.x + be.x; v.y = (v.y - mean) * rstd * g.y + be.y;
      v.z = (v.z - mean) * rstd * g.z + be.z; v.w = (v.w - mean) * rstd * g.w + be.w;
      *reinterpret_cast<float4 *>(row + d) = v;
    }
  }
  __syncthreads();
  // classes are split over gridDim.y slices (each CTA repeats the cheap LayerNorm of its images): the classifier is a
  // chain of dependent L2 loads per class pair, so the kernel time is the number of pairs a warp walks through
  const int per = (((C + gridDim.y - 1) / gridDim.y) + 1) & ~1;
  const int c_end = min(C, ((int)blockIdx.y + 1) * per);
  for (int c = blockIdx.y * per + warp * 2; c < c_end; c += 16) {               // classes c and c+1
    const bool two = c + 1 < c_end;
    const float *w0 = cw + (size_t)c * D, *w1 = cw + (size_t)(two ? c + 1 : c) * D;
    float acc[2][HEAD_IMGS];
#pragma unroll
    for (int i = 0; i < HEAD_IMGS; ++i) acc[0][i] = acc[1][i] = 0.f;
    for (int d = lane * 4; d < D; d += 128) {
      const float4 a = *reinterpret_cast<const float4 *>(w0 + d), bq = *reinterpret_cast<const float4 *>(w1 + d);
#pragma unroll
      for (int i = 0; i < HEAD_IMGS; ++i) {
        const float4 r = *reinterpret_cast<const float4 *>(rows + i * D + d);
        acc[0][i] = fmaf(a.x, r.x, acc[0][i]); acc[0][i] = fmaf(a.y, r.y, acc[0][i]);
        acc[0][i] = fmaf(a.z, r.z, acc[0][i]); acc[0][i] = fmaf(a.w, r.w, acc[0][i]);
        acc[1][i] = fmaf(bq.x, r.x, acc[1][i]); acc[1][i] = fmaf(bq.y, r.y, acc[1][i]);
        acc[1][i] = fmaf(bq.z, r.z, acc[1][i]); acc[1][i] = fmaf(bq.w, r.w, acc[1][i]);
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
#pragma unroll
      for (int i = 0; i < HEAD_IMGS; ++i) {
        acc[0][i] += __shfl_xor_sync(0xffffffffu, acc[0][i], o);
        acc[1][i] += __shfl_xor_sync(0xffffffffu, acc[1][i], o);
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < HEAD_IMGS; ++i)
        if (i < nimg) {
          logits[(size_t)(b0 + i) * C + c] = acc[0][i] + cb[c];
          if (two) logits[(size_t)(b0 + i) * C + c + 1] = acc[1][i] + cb[c + 1];
        }
    }
  }
}

__global__ void cast_bf16_kernel(const float *__restrict__ src, bf16 *__restrict__ dst, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i]);
}

// c1_tokT[k][j] = c1_w[j][D + k]
__global__ void comp_repack_kernel(const float *__restrict__ c1, float *__restrict__ tokT, int D, int CH) {
  const int total = D * CH;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int k = e / CH, j = e % CH;
    tokT[e] = c1[(size_t)j * 2 * D + D + k];
  }
}

__global__ void iota_kernel(int32_t *p, int64_t n, int mul) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = (int32_t)(i * mul);
}

__global__ void embed_index_kernel(int32_t *out_idx, int32_t *pos_idx, int64_t n, int NP) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = r / NP;
    const int p = (int)(r % NP);
    out_idx[r] = (int32_t)(b * (NP + 1) + 1 + p);
    pos_idx[r] = 1 + p;
  }
}

// ---- label path: blended similarity per patch token (model_utils.py:96-101) -------------------
// one warp per (image, patch token)
__global__ void __launch_bounds__(256)
similarity_kernel(const float *__restrict__ dense, const float *__restrict__ hid, int batch, int N, int D,
                  float blend, float *__restrict__ sim) {
  const int lane = threadIdx.x & 31;
  const int64_t total = (int64_t)batch * (N - 1);
  for (int64_t w = blockIdx.x * 8 + (threadIdx.x >> 5); w < total; w += (int64_t)gridDim.x * 8) {
    const int64_t b = w / (N - 1);
    const int t = (int)(w % (N - 1)) + 1;
    const float *r = dense + ((size_t)b * N + t) * D;
    const float *c = hid + ((size_t)b * N + t) * D;
    float dot = 0.f, rr = 0.f, cc = 0.f, dd = 0.f;
    for (int d = lane * 4; d < D; d += 128) {
      float4 a = *reinterpret_cast<const float4 *>(r + d);
      float4 x = *reinterpret_cast<const float4 *>(c + d);
      dot += a.x * x.x + a.y * x.y + a.z * x.z + a.w * x.w;
      rr += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
      cc += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
      float e0 = a.x - x.x, e1 = a.y - x.y, e2 = a.z - x.z, e3 = a.w - x.w;
      dd += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      dot += __shfl_xor_sync(0xffffffffu, dot, o); rr += __shfl_xor_sync(0xffffffffu, rr, o);
      cc += __shfl_xor_sync(0xffffffffu, cc, o);   dd += __shfl_xor_sync(0xffffffffu, dd, o);
    }
    if (lane == 0) {
      const float eps = 1e-8f;                       // F.cosine_similarity default
      const float cosv = dot / (fmaxf(sqrtf(rr), eps) * fmaxf(sqrtf(cc), eps));
      const float cs = (cosv + 1.0f) / 2.0f;
      const float ed = dd / rr;
      sim[w] = blend * cs + (1.0f - blend) * (1.0f / (1.0f + ed));    // blend: 0.3 himanshu :99-101, 0.5 donal :72-73
    }
  }
}

// loss / accuracy / confusion of one layer (model_utils.py:103-113); a single CTA is plenty for
// B*196 elements.  BCE-with-logits is applied to the POST-sigmoid score, as the reference does.
// donal != 0: the variant of donal/model_utils.py:68-80 -- labels = (similarity < st) instead of the layer's own mask,
// fixed pos_weight 1.5, prediction = score > mt (strict), accuracy = ((st - sim) * (score - mt) > 0).
__global__ void __launch_bounds__(1024)
label_stats_kernel(const float *__restrict__ sim, const uint8_t *__restrict__ mask,
                   const float *__restrict__ scores, int batch, int N, float st, float *__restrict__ loss,
                   uint8_t *__restrict__ acc_out, float *__restrict__ sim_out, long long *__restrict__ confusion,
                   int donal, float mt) {
  __shared__ double red[32];
  __shared__ unsigned long long cnt[4];
  __shared__ unsigned int pos_count;
  const int NP = N - 1;
  const int total = batch * NP;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) pos_count = 0;
  if (tid < 4) cnt[tid] = 0;
  __syncthreads();
  unsigned int local = 0;
  for (int e = tid; e < total; e += 1024) local += mask[(size_t)(e / NP) * N + 1 + e % NP] != 0;
  for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if (lane == 0 && local) atomicAdd(&pos_count, local);
  __syncthreads();
  const float alpha = (float)pos_count / (float)total;               // labels.mean()
  const float pw = donal ? 1.5f : alpha / (1.0f - alpha + 1e-16f);   // :105 / donal :75
  double lsum = 0.0;
  unsigned int c[4] = {0, 0, 0, 0};
  for (int e = tid; e < total; e += 1024) {
    const float sv = sim[e];
    const float x = scores[e];
    const int tl = sv < st;                                          // true label  (:111)
    const float y = donal ? (float)tl : (mask[(size_t)(e / NP) * N + 1 + e % NP] ? 1.0f : 0.0f);
    const float sp = log1pf(expf(-fabsf(x))) + fmaxf(-x, 0.0f);      // softplus(-x), torch's stable form
    lsum += (double)((1.0f - y) * x + (1.0f + (pw - 1.0f) * y) * sp);
    const int pl = donal ? (x > mt) : (y != 0.0f);                   // predicted   (:112 / donal :79)
    ++c[tl * 2 + pl];
    if (acc_out) acc_out[e] = donal ? (((st - sv) * (x - mt)) > 0.0f) : (((st - sv) * (y - 0.5f)) > 0.0f);   // :109 / donal :77
    if (sim_out) sim_out[e] = sv;
  }
  for (int o = 16; o; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
  if (lane == 0) red[warp] = lsum;
  for (int k = 0; k < 4; ++k) {
    unsigned int v = c[k];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && v) atomicAdd(&cnt[k], (unsigned long long)v);
  }
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int w = 0; w < 32; ++w) t += red[w];
    loss[0] = (float)(t / (double)total);
    for (int k = 0; k < 4; ++k) confusion[k] = (long long)cnt[k];
  }
}

__global__ void sim_mask_kernel(const float *__restrict__ sim, int batch, int N, float st,
                                uint8_t *__restrict__ mask_out) {
  const int total = batch * N;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int b = e / N, t = e % N;
    mask_out[e] = (t == 0) ? 1 : (sim[(size_t)b * (N - 1) + t - 1] < st);
  }
}

__global__ void adam_kernel(float *__restrict__ p, float *__restrict__ m, float *__restrict__ v,
                            const float *__restrict__ g, int64_t n, float lr, float b1, float b2, float eps,
                            float bc1, float bc2_sqrt, float gscale) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// Gradient all-reduce FUSED with the Adam step over NVLink peer memory (one-shot: every rank reads the gradient bucket
// of every rank -- its own included -- straight from that GPU's memory and sums them in rank order, so all replicas
// compute bit-identical updates without a separate collective, an intermediate reduced buffer or a second pass).
// 4.7 MB per rank: the loads are 16-byte vectors, `world` of them in flight per thread.  The caller brackets the launch
// with cross-rank barriers (all buckets written before / nobody overwrites its bucket until all have read it).
struct PeerGrads { const float *p[PSV_MAX_PEERS]; };
__global__ void __launch_bounds__(256)
adam_peer_reduce_kernel(float *__restrict__ p, float *__restrict__ m, float *__restrict__ v, PeerGrads peers, int world,
                        int64_t n4, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt, float gscale) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 g[PSV_MAX_PEERS];
#pragma unroll
    for (int r = 0; r < PSV_MAX_PEERS; ++r)
      if (r < world) g[r] = reinterpret_cast<const float4 *>(peers.p[r])[i];       // peer loads go over NVLink
    float4 s = g[0];
#pragma unroll
    for (int r = 1; r < PSV_MAX_PEERS; ++r)
      if (r < world) { s.x += g[r].x; s.y += g[r].y; s.z += g[r].z; s.w += g[r].w; }
    float4 pi = reinterpret_cast<float4 *>(p)[i], mi = reinterpret_cast<float4 *>(m)[i], vi = reinterpret_cast<float4 *>(v)[i];
    float *ps = &pi.x, *ms = &mi.x, *vs = &vi.x;
    const float *gs = &s.x;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float ge = gs[e] * gscale;
      ms[e] = b1 * ms[e] + (1.0f - b1) * ge;
      vs[e] = b2 * vs[e] + (1.0f - b2) * ge * ge;
      const float denom = sqrtf(vs[e]) / bc2_sqrt + eps;
      ps[e] -= (lr / bc1) * (ms[e] / denom);
    }
    reinterpret_cast<float4 *>(p)[i] = pi; reinterpret_cast<float4 *>(m)[i] = mi; reinterpret_cast<float4 *>(v)[i] = vi;
  }
}

// The two kernels above with global-norm clipping: the scaled gradient is multiplied by the clip coefficient (*clip,
// device, read once per thread), in the order of torch.nn.utils.clip_grad_norm_ followed by the optimizer:
// g = fp32(fp32(g * gscale) * coef).  Separate kernels, so that the unclipped steps keep their code.
__global__ void adam_clip_kernel(float *__restrict__ p, float *__restrict__ m, float *__restrict__ v,
                                 const float *__restrict__ g, int64_t n, float lr, float b1, float b2, float eps,
                                 float bc1, float bc2_sqrt, float gscale, const float *__restrict__ clip) {
  const float coef = *clip;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = __fmul_rn(__fmul_rn(g[i], gscale), coef);
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

__global__ void __launch_bounds__(256)
adam_peer_reduce_clip_kernel(float *__restrict__ p, float *__restrict__ m, float *__restrict__ v, PeerGrads peers,
                             int world, int64_t n4, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt,
                             float gscale, const float *__restrict__ clip) {
  const float coef = *clip;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 g[PSV_MAX_PEERS];
#pragma unroll
    for (int r = 0; r < PSV_MAX_PEERS; ++r)
      if (r < world) g[r] = reinterpret_cast<const float4 *>(peers.p[r])[i];
    float4 s = g[0];
#pragma unroll
    for (int r = 1; r < PSV_MAX_PEERS; ++r)
      if (r < world) { s.x += g[r].x; s.y += g[r].y; s.z += g[r].z; s.w += g[r].w; }
    float4 pi = reinterpret_cast<float4 *>(p)[i], mi = reinterpret_cast<float4 *>(m)[i], vi = reinterpret_cast<float4 *>(v)[i];
    float *ps = &pi.x, *ms = &mi.x, *vs = &vi.x;
    const float *gs = &s.x;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float ge = __fmul_rn(__fmul_rn(gs[e], gscale), coef);
      ms[e] = b1 * ms[e] + (1.0f - b1) * ge;
      vs[e] = b2 * vs[e] + (1.0f - b2) * ge * ge;
      const float denom = sqrtf(vs[e]) / bc2_sqrt + eps;
      ps[e] -= (lr / bc1) * (ms[e] / denom);
    }
    reinterpret_cast<float4 *>(p)[i] = pi; reinterpret_cast<float4 *>(m)[i] = mi; reinterpret_cast<float4 *>(v)[i] = vi;
  }
}

inline int grid_for(int64_t n, int threads, int cap) {
  int64_t g = (n + threads - 1) / threads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

cudaError_t launch_im2col_u8(PsvHandle *h, const uint8_t *pixels, int batch, void *patches, int src_h, int src_w,
                             const int32_t *tables, const float *m, const float *sd, cudaStream_t s) {
  if (src_h <= 0 || src_w <= 0 || !tables) return cudaErrorInvalidValue;
  LaunchScope scope(h, KK_IM2COL, s);
  const int C = h->cfg.channels, img = h->cfg.image, p = h->cfg.patch;
  const int grid = batch * (img / p);    // one CTA per (image, patch row)
  const size_t smem = (size_t)U8_MAX_ROWS * img * C;
  if (h->cfg.precision == PSV_BF16)
    return launch_pdl(im2col_u8_kernel<bf16>, dim3(grid), dim3(256), smem, s, pixels, (bf16 *)patches,
                      src_h, src_w, C, img, p, tables, m[0], m[1], m[2], sd[0], sd[1], sd[2]);
  return launch_pdl(im2col_u8_kernel<float>, dim3(grid), dim3(256), smem, s, pixels, (float *)patches,
                    src_h, src_w, C, img, p, tables, m[0], m[1], m[2], sd[0], sd[1], sd[2]);
}

cudaError_t launch_im2col(PsvHandle *h, const void *pixels, int pixel_type, int batch, void *patches,
                          cudaStream_t s) {
  if (pixel_type == PSV_PIXELS_U8_HWC)
    return launch_im2col_u8(h, (const uint8_t *)pixels, batch, patches, h->u8_h, h->u8_w, h->u8_tables, h->u8_mean,
                            h->u8_std, s);
  LaunchScope scope(h, KK_IM2COL, s);
  const int C = h->cfg.channels, img = h->cfg.image, p = h->cfg.patch;
  const int grid = batch * (img / p);    // one CTA per (image, patch row)
  const bool out_bf16 = h->cfg.precision == PSV_BF16;
  if (pixel_type == PSV_PIXELS_F32) {
    if (out_bf16) return launch_pdl(im2col_kernel<float, bf16>, dim3(grid), dim3(256), 0, s, (const float *)pixels, (bf16 *)patches, batch, C, img, p);
    return launch_pdl(im2col_kernel<float, float>, dim3(grid), dim3(256), 0, s, (const float *)pixels, (float *)patches, batch, C, img, p);
  }
  if (out_bf16) return launch_pdl(im2col_kernel<bf16, bf16>, dim3(grid), dim3(256), 0, s, (const bf16 *)pixels, (bf16 *)patches, batch, C, img, p);
  return launch_pdl(im2col_kernel<bf16, float>, dim3(grid), dim3(256), 0, s, (const bf16 *)pixels, (float *)patches, batch, C, img, p);
}

size_t pixel_bytes_per_image(const PsvHandle *h, int pixel_type) {
  if (pixel_type == PSV_PIXELS_U8_HWC) return (size_t)h->u8_h * h->u8_w * h->cfg.channels;
  return (size_t)h->cfg.channels * h->cfg.image * h->cfg.image * (pixel_type == PSV_PIXELS_F32 ? 4 : 2);
}

cudaError_t launch_cls_rows(PsvHandle *h, float *hidden, int batch, cudaStream_t s) {
  LaunchScope scope(h, KK_CLS_ROWS, s);
  return launch_pdl(cls_rows_kernel, dim3(grid_for((int64_t)batch * h->D, 256, 1024)), dim3(256), 0, s, hidden,
                    (const float *)h->cls_token, (const float *)h->pos_emb, batch, h->N, h->D);
}

cudaError_t launch_head(PsvHandle *h, const float *hidden, int batch, float *logits, cudaStream_t s) {
  LaunchScope scope(h, KK_HEAD, s);
  const int slices = (h->C + 31) / 32;                   // <= 32 classes per CTA: two class pairs per warp
  return launch_pdl(head_kernel, dim3((batch + HEAD_IMGS - 1) / HEAD_IMGS, slices), dim3(256),
                    (size_t)HEAD_IMGS * h->D * sizeof(float), s, hidden, (const float *)h->final_ln_w,
                    (const float *)h->final_ln_b, (const float *)h->cls_w, (const float *)h->cls_b, h->cfg.ln_eps,
                    h->N, h->D, h->C, batch, logits);
}

cudaError_t launch_cast_bf16(const float *src, bf16 *dst, int64_t n, cudaStream_t s) {
  cast_bf16_kernel<<<grid_for(n, 256, 148 * 16), 256, 0, s>>>(src, dst, n);
  return cudaGetLastError();
}

cudaError_t launch_comp_repack(PsvHandle *h, const float *c1, float *tokT, cudaStream_t s) {
  comp_repack_kernel<<<grid_for((int64_t)h->D * h->CH, 256, 1024), 256, 0, s>>>(c1, tokT, h->D, h->CH);
  return cudaGetLastError();
}

cudaError_t launch_iota(int32_t *p, int64_t n, int mul, cudaStream_t s) {
  iota_kernel<<<grid_for(n, 256, 1024), 256, 0, s>>>(p, n, mul);
  return cudaGetLastError();
}

cudaError_t launch_embed_index(PsvHandle *h, cudaStream_t s) {
  const int64_t n = (int64_t)h->cfg.max_batch * (h->N - 1);
  embed_index_kernel<<<grid_for(n, 256, 1024), 256, 0, s>>>(h->embed_out_idx, h->embed_pos_idx, n, h->N - 1);
  return cudaGetLastError();
}

cudaError_t launch_similarity(PsvHandle *h, const float *dense_out, const float *hidden_in, int batch,
                              float *sim_out, cudaStream_t s) {
  LaunchScope scope(h, KK_SIMILARITY, s);
  const int64_t warps = (int64_t)batch * (h->N - 1);
  similarity_kernel<<<grid_for(warps, 8, h->sm_count * 8), 256, 0, s>>>(dense_out, hidden_in, batch, h->N, h->D,
                                                                          h->loss_variant == PSV_LOSS_SIMILARITY_LABELS ? 0.5f : 0.3f,
                                                                          sim_out);
  return cudaGetLastError();
}

cudaError_t launch_label_stats(PsvHandle *h, const float *sim, const uint8_t *mask, const float *scores, int batch,
                               float st, const PsvLayerStats *out, cudaStream_t s) {
  LaunchScope scope(h, KK_LABEL_STATS, s);
  label_stats_kernel<<<1, 1024, 0, s>>>(sim, mask, scores, batch, h->N, st, out->loss, out->accuracy,
                                        out->similarity, (long long *)out->confusion,
                                        h->loss_variant == PSV_LOSS_SIMILARITY_LABELS ? 1 : 0, h->loss_mt);
  return cudaGetLastError();
}

cudaError_t launch_sim_mask(PsvHandle *h, const float *sim, int batch, float st, uint8_t *mask_out,
                            cudaStream_t s) {
  LaunchScope scope(h, KK_OTHER, s);
  sim_mask_kernel<<<grid_for((int64_t)batch * h->N, 256, 1024), 256, 0, s>>>(sim, batch, h->N, st, mask_out);
  return cudaGetLastError();
}

cudaError_t launch_adam(float *p, float *m, float *v, const float *g, int64_t n, float lr, float b1, float b2,
                        float eps, int step, float gscale, cudaStream_t s, const float *clip) {
  const float bc1 = 1.0f - powf(b1, (float)step);
  const float bc2 = 1.0f - powf(b2, (float)step);
  if (clip)
    adam_clip_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(p, m, v, g, n, lr, b1, b2, eps, bc1, sqrtf(bc2), gscale,
                                                                clip);
  else
    adam_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, s>>>(p, m, v, g, n, lr, b1, b2, eps, bc1, sqrtf(bc2), gscale);
  return cudaGetLastError();
}

cudaError_t launch_adam_peer_reduce(float *p, float *m, float *v, const float *const *peer_grads, int world, int64_t n,
                                    float lr, float b1, float b2, float eps, int step, float gscale, cudaStream_t s,
                                    const float *clip) {
  if (world < 1 || world > PSV_MAX_PEERS || n % 4 != 0) return cudaErrorInvalidValue;
  PeerGrads peers;
  for (int r = 0; r < PSV_MAX_PEERS; ++r) peers.p[r] = r < world ? peer_grads[r] : nullptr;
  const float bc1 = 1.0f - powf(b1, (float)step);
  const float bc2 = 1.0f - powf(b2, (float)step);
  if (clip)
    adam_peer_reduce_clip_kernel<<<grid_for(n / 4, 256, 148 * 4), 256, 0, s>>>(p, m, v, peers, world, n / 4, lr, b1, b2,
                                                                                eps, bc1, sqrtf(bc2), gscale, clip);
  else
    adam_peer_reduce_kernel<<<grid_for(n / 4, 256, 148 * 4), 256, 0, s>>>(p, m, v, peers, world, n / 4, lr, b1, b2, eps,
                                                                           bc1, sqrtf(bc2), gscale);
  return cudaGetLastError();
}

}  // namespace psv
