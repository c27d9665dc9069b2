// Backbone fine-tuning path (SURVEY.md 8f-2; reference main_model_utils.py:108-165 with loss_type = "classification" and
// model.vit_train(), model_utils.py:265-273): the gradient of a loss on the logits with respect to EVERY backbone
// parameter (embeddings, 12 layers, final LayerNorm, classifier), through the patch-skip forward.
//
// The skip decisions are hard thresholds, so no gradient flows through the compressors: at every layer the gradient of
// a skipped token passes through unchanged (the token was carried forward), and the gradient of an active token goes
// back through LayerNorm -> attention among the image's ACTIVE tokens -> proj -> LayerNorm -> MLP on the packed rows --
// the adjoints of the forward's gather (hidden[idx] -> packed) and scatter (packed -> hidden[idx]).
// In the keep-all-keys mode (PSV_KV_ALL, reference recap/convprad4.py:99-125) LN1 and q|k|v cover all batch * N rows and
// the active queries attend to all N tokens: a skipped token then also receives gradient through its key / value rows,
// so the QKV and LN1 backward run over all rows; from the output projection on nothing changes.
// Under the similarity criterion (PSV_SKIP_SIMILARITY, reference pradeep/model_utils.py:73-84) each layer of the forward
// first runs its dense pass to decide the mask; the backward is unchanged, the masks being constants either way.
// Raw uint8 images (PSV_PIXELS_U8_HWC): the forward records the resize / normalisation setup and the backward's im2col
// recomputes the patches with it.
//
//   psv_backbone_forward_train : the fp32 forward, keeping per layer the compaction (idx, cu_seqlens) and the packed
//                                activations the backward needs (layer input rows, LN1 out, q|k|v, attention out, x1,
//                                LN2 out, FC1 pre-activation)
//   psv_backbone_backward      : d(logits) -> flat fp32 gradient of all backbone parameters
//
// fp32 only (PSV_FP32 handles): this is the parity-first form of the row -- fp32 FFMA GEMMs for dgrad / wgrad, fp32
// attention backward -- checked against the UNMODIFIED reference's autograd (tests/golden/finetune_*.npz).  It is not a
// tuned path: the forward hot path is what this library optimises.
#include <algorithm>
#include <cstdio>
#include <vector>

#include "psv_internal.cuh"

namespace psv {
namespace {

// ---- C[M,N] (+)= op(A)[M,K] . op(B)[K,N], fp32, arbitrary sizes / leading dimensions -------------------------------------
// A(m,k) = TA ? A[k*lda + m] : A[m*lda + k];   B(k,n) = TB ? B[n*ldb + k] : B[k*ldb + n]
template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
train_gemm_kernel(const float *__restrict__ A, int lda, const float *__restrict__ B, int ldb, float *__restrict__ C,
                  int ldc, int M, int N, int K, int accumulate) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int e = threadIdx.x; e < 16 * 64; e += 256) {
      // A tile: [16 k][64 m]; iterate so that the contiguous global dimension is the fast one
      const int kk = TA ? e / 64 : e % 16, mm = TA ? e % 64 : e / 16;
      const int m = m0 + mm, k = k0 + kk;
      As[kk][mm] = (m < M && k < K) ? (TA ? A[(size_t)k * lda + m] : A[(size_t)m * lda + k]) : 0.f;
      const int kb = TB ? e % 16 : e / 64, nn = TB ? e / 16 : e % 64;
      const int n = n0 + nn, k2 = k0 + kb;
      Bs[kb][nn] = (n < N && k2 < K) ? (TB ? B[(size_t)n * ldb + k2] : B[(size_t)k2 * ldb + n]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) C[(size_t)m * ldc + n] = acc[i][j] + (accumulate ? C[(size_t)m * ldc + n] : 0.f);
    }
  }
}

cudaError_t train_gemm(const float *A, int lda, bool ta, const float *B, int ldb, bool tb, float *C, int ldc, int M,
                       int N, int K, bool accumulate, cudaStream_t s) {
  if (M <= 0 || N <= 0 || K <= 0) return cudaSuccess;
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  const int acc = accumulate ? 1 : 0;
  if (ta && tb)       train_gemm_kernel<true, true><<<grid, 256, 0, s>>>(A, lda, B, ldb, C, ldc, M, N, K, acc);
  else if (ta)        train_gemm_kernel<true, false><<<grid, 256, 0, s>>>(A, lda, B, ldb, C, ldc, M, N, K, acc);
  else if (tb)        train_gemm_kernel<false, true><<<grid, 256, 0, s>>>(A, lda, B, ldb, C, ldc, M, N, K, acc);
  else                train_gemm_kernel<false, false><<<grid, 256, 0, s>>>(A, lda, B, ldb, C, ldc, M, N, K, acc);
  return cudaGetLastError();
}

// ---- small row kernels -----------------------------------------------------------------------------------------------
// dst[r, :] = src[idx ? idx[r] : r, :] (gather) or dst[idx[r], :] = src[r, :] (scatter), `rows` rows of `width` floats;
// rows_dev (nullable): only the first *rows_dev rows -- idx past the layer's active row count is not written
__global__ void rows_copy_kernel(const float *__restrict__ src, float *__restrict__ dst, const int32_t *__restrict__ idx,
                                 int rows, int width, int scatter, const int32_t *__restrict__ rows_dev = nullptr) {
  if (rows_dev) rows = min(rows, *rows_dev);
  const int q = width / 4;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < (int64_t)rows * q; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / q), c = (int)(e % q) * 4;
    const int other = idx ? idx[r] : r;
    const float4 v = *reinterpret_cast<const float4 *>(src + (size_t)(scatter ? r : other) * width + c);
    *reinterpret_cast<float4 *>(dst + (size_t)(scatter ? other : r) * width + c) = v;
  }
}
// out[n] += sum_r x[r, n], any width (the classifier's 100 columns)
__global__ void colsum_slow_kernel(const float *__restrict__ x, int rows, int width, float *__restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= width) return;
  float acc = 0.f;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) acc += x[(size_t)r * width + n];
  atomicAdd(out + n, acc);
}
// out[n] += sum_r x[r, n]   (width % 4 == 0): 32 float4 columns x 8 row lanes per block, grid.y row slices
__global__ void __launch_bounds__(256)
colsum_kernel(const float *__restrict__ x, int rows, int width, float *__restrict__ out) {
  __shared__ float4 part[8][32];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + cx) * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < width)
    for (int r = blockIdx.y * 8 + ry; r < rows; r += gridDim.y * 8) {
      const float4 v = *reinterpret_cast<const float4 *>(x + (size_t)r * width + c);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  part[ry][cx] = acc;
  __syncthreads();
  if (ry == 0 && c < width) {
    for (int i = 1; i < 8; ++i) { acc.x += part[i][cx].x; acc.y += part[i][cx].y; acc.z += part[i][cx].z; acc.w += part[i][cx].w; }
    atomicAdd(out + c, acc.x); atomicAdd(out + c + 1, acc.y); atomicAdd(out + c + 2, acc.z); atomicAdd(out + c + 3, acc.w);
  }
}
__device__ __forceinline__ float gelu_f(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }
// exact erf-GELU (HF "gelu") and its derivative:  Phi(v) + v * phi(v)
__global__ void gelu_fwd_kernel(const float *__restrict__ u, float *__restrict__ g, int64_t n,       // n % 4 == 0
                                const int32_t *__restrict__ rows_dev, int width) {
  if (rows_dev) n = min(n, (int64_t)*rows_dev * width);
  for (int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4; i < n; i += (int64_t)gridDim.x * blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4 *>(u + i);
    *reinterpret_cast<float4 *>(g + i) = make_float4(gelu_f(v.x), gelu_f(v.y), gelu_f(v.z), gelu_f(v.w));
  }
}
__device__ __forceinline__ float gelu_grad_f(float v) {
  const float cdf = 0.5f * (1.0f + erff(v * 0.70710678118654752440f));
  const float pdf = 0.3989422804014327f * expf(-0.5f * v * v);
  return cdf + v * pdf;
}
__global__ void gelu_bwd_kernel(const float *__restrict__ u, float *__restrict__ dg, int64_t n) {      // n % 4 == 0
  for (int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * 4; i < n; i += (int64_t)gridDim.x * blockDim.x * 4) {
    const float4 v = *reinterpret_cast<const float4 *>(u + i);
    float4 d = *reinterpret_cast<const float4 *>(dg + i);
    d.x *= gelu_grad_f(v.x); d.y *= gelu_grad_f(v.y); d.z *= gelu_grad_f(v.z); d.w *= gelu_grad_f(v.w);
    *reinterpret_cast<float4 *>(dg + i) = d;
  }
}
// LayerNorm backward of `rows` rows (one warp per row, D = 32 * V4 * 4):
//   dx[orow] (+)= rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma;   dgamma += dy * xhat;  dbeta += dy
// x rows are read at x_idx ? x_idx[r] : r, dx rows written at the same position of `dx` (add_to_dx: accumulate).
// The per-warp dgamma / dbeta partials meet in shared memory; above D = 768 the [8][D] pair would pass the 48 KB of
// static shared memory, so D = 1024 reduces them in two column halves through [8][D / 2] arrays.
template <int D>
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const float *__restrict__ x, const int32_t *__restrict__ x_idx, const float *__restrict__ dy,
              const float *__restrict__ gamma, float eps, int rows, float *__restrict__ dx, int add_to_dx,
              float *__restrict__ dgamma, float *__restrict__ dbeta) {
  constexpr int V = D / 128;
  constexpr int RC = D <= 768 ? D : D / 2;        // columns reduced per pass
  __shared__ float red_g[8][RC], red_b[8][RC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 ag[V], ab[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { ag[i] = make_float4(0, 0, 0, 0); ab[i] = make_float4(0, 0, 0, 0); }
  for (int r = blockIdx.x * 8 + warp; r < rows; r += gridDim.x * 8) {
    const size_t xr = (size_t)(x_idx ? x_idx[r] : r) * D;
    float4 v[V], d[V];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      v[i] = *reinterpret_cast<const float4 *>(x + xr + (i * 32 + lane) * 4);
      d[i] = *reinterpret_cast<const float4 *>(dy + (size_t)r * D + (i * 32 + lane) * 4);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * (1.0f / D);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
      sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = 1.0f / sqrtf(sq * (1.0f / D) + eps);
    float sg = 0.f, sgx = 0.f;
    float4 g[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const float4 gm = *reinterpret_cast<const float4 *>(gamma + (i * 32 + lane) * 4);
      v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;                   // xhat
      g[i] = make_float4(d[i].x * gm.x, d[i].y * gm.y, d[i].z * gm.z, d[i].w * gm.w);
      sg += (g[i].x + g[i].y) + (g[i].z + g[i].w);
      sgx += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
      ag[i].x += d[i].x * v[i].x; ag[i].y += d[i].y * v[i].y; ag[i].z += d[i].z * v[i].z; ag[i].w += d[i].w * v[i].w;
      ab[i].x += d[i].x; ab[i].y += d[i].y; ab[i].z += d[i].z; ab[i].w += d[i].w;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { sg += __shfl_xor_sync(0xffffffffu, sg, o); sgx += __shfl_xor_sync(0xffffffffu, sgx, o); }
    sg *= (1.0f / D); sgx *= (1.0f / D);
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float4 o4 = make_float4(rstd * (g[i].x - sg - v[i].x * sgx), rstd * (g[i].y - sg - v[i].y * sgx),
                              rstd * (g[i].z - sg - v[i].z * sgx), rstd * (g[i].w - sg - v[i].w * sgx));
      float *dst = dx + xr + (i * 32 + lane) * 4;
      if (add_to_dx) {
        const float4 p = *reinterpret_cast<const float4 *>(dst);
        o4.x += p.x; o4.y += p.y; o4.z += p.z; o4.w += p.w;
      }
      *reinterpret_cast<float4 *>(dst) = o4;
    }
  }
  if constexpr (RC == D) {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      *reinterpret_cast<float4 *>(&red_g[warp][(i * 32 + lane) * 4]) = ag[i];
      *reinterpret_cast<float4 *>(&red_b[warp][(i * 32 + lane) * 4]) = ab[i];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += 256) {
      float sgm = 0.f, sbt = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) { sgm += red_g[w][c]; sbt += red_b[w][c]; }
      atomicAdd(dgamma + c, sgm);
      atomicAdd(dbeta + c, sbt);
    }
  } else {
    // float4 slot i of a lane holds columns (i * 32 + lane) * 4: slots [0, V/2) are the first half, the rest the second
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      if (half) __syncthreads();                      // the first half's sums have been read
#pragma unroll
      for (int i = 0; i < V / 2; ++i) {
        *reinterpret_cast<float4 *>(&red_g[warp][(i * 32 + lane) * 4]) = ag[half * (V / 2) + i];
        *reinterpret_cast<float4 *>(&red_b[warp][(i * 32 + lane) * 4]) = ab[half * (V / 2) + i];
      }
      __syncthreads();
      for (int c = threadIdx.x; c < RC; c += 256) {
        float sgm = 0.f, sbt = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) { sgm += red_g[w][c]; sbt += red_b[w][c]; }
        atomicAdd(dgamma + half * RC + c, sgm);
        atomicAdd(dbeta + half * RC + c, sbt);
      }
    }
  }
}

// out[t, :] += sum_b x[b, t, :]   (position-embedding gradient; t < N)
__global__ void batch_sum_kernel(const float *__restrict__ x, int batch, int N, int D, float *__restrict__ out) {
  const int total = N * D;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int b = 0; b < batch; ++b) acc += x[(size_t)b * total + e];
    out[e] += acc;
  }
}

// ---- attention backward (fp32): one CTA per (head, image), n <= 200 tokens ------------------------------------------------
// Forward (HF:171-196): P = softmax(Q K^T / 8), O = P V.  Given dO:  dV = P^T dO;  dP = dO V^T;  dS = P o (dP - rowsum(P o dP));
// dQ = dS K / 8;  dK = dS^T Q / 8.  Q / 8, K, V, dO of the (image, head) live in shared memory (rows padded to 65 floats).
// Pass 1, a warp per query: the row's log-sum-exp, delta = rowsum(P o dP) and dQ.  Pass 2, a warp per key: the column of P
// and dS is recomputed from the saved row statistics (same fma order, same bits) and dK / dV accumulate in registers --
// no atomics, so the gradients are deterministic.  Shared memory is sized by the layer's longest sequence (n_cap).
// KV_ALL (keep-all-keys mode, the adjoint of attention_simt_kernel with q_rows / kv_tokens): the queries are the image's
// packed active rows (dO packed, q read from the dense q|k|v through q_rows), the keys / values its kv_tokens dense rows.
// dQ goes to the Q columns of each query's dense row, dK / dV to every dense row, and the Q columns of the skipped rows
// are zeroed, so dqkv is complete over all batch * kv_tokens rows.  Queries and keys both fit n_cap (n <= kv_tokens).
constexpr int AB_MAX_N = 200, AB_DH = 64, AB_WARPS = 8, AB_LD = AB_DH + 1;
constexpr size_t ab_smem(int n_cap) { return ((size_t)4 * n_cap * AB_LD + 2 * (size_t)n_cap) * sizeof(float); }
constexpr size_t AB_SMEM = ab_smem(AB_MAX_N);
template <bool KV_ALL>
__global__ void __launch_bounds__(AB_WARPS * 32)
attention_bwd_kernel(const float *__restrict__ qkv, const float *__restrict__ dctx, const int32_t *__restrict__ cu,
                     int D, float *__restrict__ dqkv, int n_cap, const int32_t *__restrict__ q_rows, int kv_tokens) {
  extern __shared__ float sm[];
  float *Qs = sm;                                   // [n][65]   q / 8
  float *Ks = Qs + (size_t)n_cap * AB_LD;           // [nk][65]
  float *Vs = Ks + (size_t)n_cap * AB_LD;           // [nk][65]
  float *dOs = Vs + (size_t)n_cap * AB_LD;          // [n][65]
  float *lse = dOs + (size_t)n_cap * AB_LD;         // [n]
  float *dl = lse + n_cap;                          // [n]
  const int head = blockIdx.x, b = blockIdx.y;
  const int row0 = cu[b], n = cu[b + 1] - row0;     // n queries
  const int nk = KV_ALL ? kv_tokens : n;            // nk keys
  if ((!KV_ALL && n <= 0) || nk > n_cap) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t ld = (size_t)3 * D;
  const size_t key0 = KV_ALL ? (size_t)b * kv_tokens : (size_t)row0;
  const float *base = qkv + key0 * ld + head * AB_DH;
  for (int e = tid; e < nk * AB_DH; e += AB_WARPS * 32) {
    const int j = e >> 6, d = e & 63;
    if (KV_ALL) {
      dqkv[(key0 + j) * ld + head * AB_DH + d] = 0.f;   // pass 1 overwrites the active rows (after the barrier)
      if (j < n) {
        Qs[j * AB_LD + d] = qkv[(size_t)q_rows[row0 + j] * ld + head * AB_DH + d] * 0.125f;
        dOs[j * AB_LD + d] = dctx[(size_t)(row0 + j) * D + head * AB_DH + d];
      }
    } else {
      Qs[j * AB_LD + d] = base[(size_t)j * ld + d] * 0.125f;
    }
    Ks[j * AB_LD + d] = base[(size_t)j * ld + D + d];
    Vs[j * AB_LD + d] = base[(size_t)j * ld + 2 * D + d];
    if (!KV_ALL) dOs[j * AB_LD + d] = dctx[(size_t)(row0 + j) * D + head * AB_DH + d];
  }
  __syncthreads();
  constexpr int NJ = AB_MAX_N / 32 + 1;
  // ---- pass 1: queries
  for (int r = warp; r < n; r += AB_WARPS) {
    float qr[AB_DH], dor[AB_DH];                       // the query's rows in registers: one shared-memory operand per fma
#pragma unroll
    for (int d = 0; d < AB_DH; ++d) { qr[d] = Qs[r * AB_LD + d]; dor[d] = dOs[r * AB_LD + d]; }
    float p[NJ], dp[NJ];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int j = lane + 32 * i;
      float sc = -INFINITY, a = 0.f;
      if (j < nk) {
        sc = 0.f;
        const float *kr = Ks + j * AB_LD, *vr = Vs + j * AB_LD;
#pragma unroll
        for (int d = 0; d < AB_DH; ++d) { sc = fmaf(qr[d], kr[d], sc); a = fmaf(dor[d], vr[d], a); }
      }
      p[i] = sc; dp[i] = a;
      mx = fmaxf(mx, sc);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NJ; ++i) { if (lane + 32 * i < nk) sum += expf(p[i] - mx); }
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float l = mx + logf(sum);
    float dsum = 0.f;
#pragma unroll
    for (int i = 0; i < NJ; ++i) { p[i] = (lane + 32 * i < nk) ? expf(p[i] - l) : 0.f; dsum += p[i] * dp[i]; }
#pragma unroll
    for (int o = 16; o; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
    if (lane == 0) { lse[r] = l; dl[r] = dsum; }
    float dq0 = 0.f, dq1 = 0.f;
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const float ds_own = p[i] * (dp[i] - dsum);          // d loss / d s_j for this lane's key (s = (q/8) . k)
      const int jn = min(32, nk - 32 * i);
      for (int src = 0; src < jn; ++src) {
        const float ds = __shfl_sync(0xffffffffu, ds_own, src);
        const float *kr = Ks + (src + 32 * i) * AB_LD;
        dq0 = fmaf(ds, kr[lane], dq0); dq1 = fmaf(ds, kr[lane + 32], dq1);
      }
    }
    float *dqrow = dqkv + (size_t)(KV_ALL ? q_rows[row0 + r] : row0 + r) * ld + head * AB_DH;
    dqrow[lane] = dq0 * 0.125f; dqrow[lane + 32] = dq1 * 0.125f;
  }
  __syncthreads();
  // ---- pass 2: keys
  for (int j = warp; j < nk; j += AB_WARPS) {
    float kr[AB_DH], vr[AB_DH];
#pragma unroll
    for (int d = 0; d < AB_DH; ++d) { kr[d] = Ks[j * AB_LD + d]; vr[d] = Vs[j * AB_LD + d]; }
    float p[NJ], ds[NJ];
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int r = lane + 32 * i;
      p[i] = 0.f; ds[i] = 0.f;
      if (r < n) {
        float sc = 0.f, a = 0.f;
        const float *qr = Qs + r * AB_LD, *dor = dOs + r * AB_LD;
#pragma unroll
        for (int d = 0; d < AB_DH; ++d) { sc = fmaf(qr[d], kr[d], sc); a = fmaf(dor[d], vr[d], a); }
        p[i] = expf(sc - lse[r]);
        ds[i] = p[i] * (a - dl[r]);
      }
    }
    float dk0 = 0.f, dk1 = 0.f, dv0 = 0.f, dv1 = 0.f;
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int rn = min(32, n - 32 * i);
      for (int src = 0; src < rn; ++src) {
        const float dsb = __shfl_sync(0xffffffffu, ds[i], src), pb = __shfl_sync(0xffffffffu, p[i], src);
        const float *qr = Qs + (src + 32 * i) * AB_LD, *dor = dOs + (src + 32 * i) * AB_LD;
        dk0 = fmaf(dsb, qr[lane], dk0); dk1 = fmaf(dsb, qr[lane + 32], dk1);
        dv0 = fmaf(pb, dor[lane], dv0); dv1 = fmaf(pb, dor[lane + 32], dv1);
      }
    }
    float *o = dqkv + (size_t)(KV_ALL ? b * kv_tokens + j : row0 + j) * ld + head * AB_DH;
    o[D + lane] = dk0; o[D + lane + 32] = dk1;
    o[2 * D + lane] = dv0; o[2 * D + lane + 32] = dv1;
  }
}

// ---- fp32-class GEMMs on the tensor cores: (a_hi + a_lo)(w_hi + w_lo) ~= a_hi w_hi + a_hi w_lo + a_lo w_hi ---------------
// Every operand is split into two bf16 planes (hi = bf16(x), lo = bf16(x - hi): 16 mantissa bits together, the dropped
// lo * lo term is 2^-16 relative) and the product is three passes of the bf16 tcgen05 GEMM (gemm_tc.cu) into the same fp32
// output, store then two red.adds, in launch order (deterministic).  Same idea as the score kernel's split products.
// split_kernel<TR = false>: dst[r, c] = src[r, c];  <TR = true>: dst[c, r] = src[r, c] (32 x 32 tiles through shared
// memory).  dst has `ldo` columns; columns past the source extent are written as zeros (K padding to 64).
// two planes: x ~= hi + lo (16 mantissa bits); three planes (mid != null): x ~= hi + mid + lo (24 bits, fp32-exact)
__device__ __forceinline__ void split_store(float v, bf16 *hi, bf16 *mid, bf16 *lo, size_t at) {
  const bf16 h = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(h);
  hi[at] = h;
  if (mid) {
    const bf16 m = __float2bfloat16_rn(r1);
    mid[at] = m;
    lo[at] = __float2bfloat16_rn(r1 - __bfloat162float(m));
  } else {
    lo[at] = __float2bfloat16_rn(r1);
  }
}
template <bool TR>
__global__ void __launch_bounds__(256)
split_kernel(const float *__restrict__ src, int ld, int rows, int cols, bf16 *__restrict__ hi, bf16 *__restrict__ mid,
             bf16 *__restrict__ lo, int ldo, const int32_t *__restrict__ rows_dev) {
  __shared__ float tile[32][33];
  if (rows_dev) rows = min(rows, *rows_dev);       // packed activations: only the rows the layer kept
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;                 // 32 x 8
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  if (TR) {
    for (int i = ty; i < 32; i += 8) {
      const int r = r0 + i, c = c0 + tx;
      tile[i][tx] = (r < rows && c < cols) ? src[(size_t)r * ld + c] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
      const int c = c0 + i, r = r0 + tx;                                  // dst row = source column
      if (c < cols && r < ldo) {
        split_store(tile[tx][i], hi, mid, lo, (size_t)c * ldo + r);
      }
    }
  } else {
    if (r0 >= rows) return;
    for (int i = ty; i < 32; i += 8) {
      const int r = r0 + i, c = c0 + tx;
      if (r < rows && c < ldo) {
        split_store(c < cols ? src[(size_t)r * ld + c] : 0.f, hi, mid, lo, (size_t)r * ldo + c);
      }
    }
  }
}

// planes of op(src): tr = false -> [rows, ldo >= cols]; tr = true -> [cols, ldo >= rows]; three: also the mid plane
}  // namespace

cudaError_t split_planes(const float *src, int ld, int rows, int cols, bool tr, int ldo, SplitPlanes out, bool three,
                         cudaStream_t s, const int32_t *rows_dev) {
  if (rows <= 0 || cols <= 0) return cudaSuccess;
  bf16 *mid = three ? out.mid : nullptr;
  if (tr) {
    dim3 grid((cols + 31) / 32, (ldo + 31) / 32);
    split_kernel<true><<<grid, 256, 0, s>>>(src, ld, rows, cols, out.hi, mid, out.lo, ldo, nullptr);
  } else {
    dim3 grid((ldo + 31) / 32, (rows + 31) / 32);
    split_kernel<false><<<grid, 256, 0, s>>>(src, ld, rows, cols, out.hi, mid, out.lo, ldo, rows_dev);
  }
  return cudaGetLastError();
}
// out[M, N] (fp32, row stride N) = A[M, K] . W[N, K]^T (+ bias) (+ res rows), operands as split planes, K % 64 == 0, N % 128 == 0
// three: hi hi + hi mid + mid hi + mid mid + hi lo + lo hi (the dropped terms are below 2^-24 relative)
// stream_k: every pass red.adds into `out` (the caller zeroes it) with the (tile, k-block) space cut evenly over the CTA
// pairs -- for products with a long K and few output tiles (dW = delta^T x: 3 tiles, K = the row count)
cudaError_t split_gemm(PsvHandle *h, SplitPlanes a, SplitPlanes w, float *out, int M, int N, int K, const float *bias,
                       const float *res, const int32_t *res_idx, const int32_t *out_idx, const int32_t *m_dev,
                       bool three, cudaStream_t s, bool stream_k) {
  if (M <= 0) return cudaSuccess;
  GemmArgs g;
  g.a = a.hi; g.w = w.hi; g.bias = bias; g.res = res; g.res_idx = res_idx; g.out_idx = out_idx; g.out = out; g.out_fp32 = 1;
  g.m_max = M; g.n = N; g.k = K; g.m_dev = m_dev;
  if (stream_k) { g.accumulate = 1; g.stream_k = 1; }
  cudaError_t e = launch_gemm_tc(h, g, s);
  g.bias = nullptr; g.res = nullptr; g.res_idx = nullptr; g.accumulate = 1;
  g.w = w.lo;
  if (e == cudaSuccess) e = launch_gemm_tc(h, g, s);
  g.a = a.lo; g.w = w.hi;
  if (e == cudaSuccess) e = launch_gemm_tc(h, g, s);
  if (three) {
    g.a = a.hi; g.w = w.mid;
    if (e == cudaSuccess) e = launch_gemm_tc(h, g, s);
    g.a = a.mid; g.w = w.hi;
    if (e == cudaSuccess) e = launch_gemm_tc(h, g, s);
    g.a = a.mid; g.w = w.mid;
    if (e == cudaSuccess) e = launch_gemm_tc(h, g, s);
  }
  return e;
}

namespace {

int grid_for64(int64_t n, int threads, int cap) {
  int64_t g = (n + threads - 1) / threads;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

int tfail(PsvHandle *h, int code, const char *msg) {
  if (h) h->err = msg;
  return code;
}

#define T_CUDA(h, call)                                                                                    \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess) {                                                                              \
      h->err = std::string(#call) + " failed: " + cudaGetErrorString(e__);                                 \
      return PSV_ERR_CUDA;                                                                                 \
    }                                                                                                      \
  } while (0)

}  // namespace

// d loss_l / d (layer input) through the compressor's first Linear (himanshu/model_utils.py:62-65: its input row of patch
// p is [hidden[b, 0] | hidden[b, 1 + p]]):
//   dH[b, 1 + p, c] += g * sum_j delta[b, p, j] * W1[j, D + c];    dH[b, 0, c] += g * sum_j dsum[b, j] * W1[j, c]
// g = *gscale (the upstream gradient of loss_l).  grid (ceil(N / CI_ROWS), batch), D / 4... threads over c.
constexpr int CI_ROWS = 16, CH = 64;            // CH: the compressor's hidden width (train_kernels.cu)
__global__ void __launch_bounds__(256)
comp_input_grad_kernel(const float *__restrict__ delta, const float *__restrict__ dsum, const float *__restrict__ w1,
                       const float *__restrict__ gscale, int N, int D, float *__restrict__ dH) {
  __shared__ float dv[CI_ROWS][CH];
  const int b = blockIdx.y, t0 = blockIdx.x * CI_ROWS;
  const float g = *gscale;
  for (int e = threadIdx.x; e < CI_ROWS * CH; e += blockDim.x) {
    const int r = e / CH, j = e % CH, t = t0 + r;
    float v = 0.f;
    if (t < N) v = t == 0 ? dsum[(size_t)b * CH + j] : delta[((size_t)b * (N - 1) + t - 1) * CH + j];
    dv[r][j] = v * g;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float acc[CI_ROWS];
#pragma unroll
    for (int r = 0; r < CI_ROWS; ++r) acc[r] = 0.f;
    for (int j = 0; j < CH; ++j) {
      const float wc = w1[(size_t)j * 2 * D + c], wt = w1[(size_t)j * 2 * D + D + c];
#pragma unroll
      for (int r = 0; r < CI_ROWS; ++r) acc[r] = fmaf(dv[r][j], (t0 + r == 0) ? wc : wt, acc[r]);
    }
#pragma unroll
    for (int r = 0; r < CI_ROWS; ++r)
      if (t0 + r < N) dH[((size_t)b * N + t0 + r) * D + c] += acc[r];
  }
}
// out[i] = src[i] * *scale
__global__ void scale_copy_kernel(const float *__restrict__ src, const float *__restrict__ scale, float *__restrict__ out, int64_t n) {
  const float g = *scale;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = src[i] * g;
}
// mask[idx[r]] = 1 for the T kept rows of a layer (idx: flat b * N + t)
__global__ void mark_rows_kernel(const int32_t *__restrict__ idx, int T, uint8_t *__restrict__ mask) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < T; r += gridDim.x * blockDim.x) mask[idx[r]] = 1;
}

// activations kept by psv_backbone_forward_train (all packed to the layer's T active rows unless noted)
struct TrainSave {
  int batch = 0;
  bool kv_all = false;                     // the forward ran in PSV_KV_ALL: x0, a1 and qkv hold all batch * N rows in
                                           // dense order; the backward follows this, not the handle's current mode
  int criterion = PSV_SKIP_MLP;            // the skip criterion the forward decided by (and its sim_threshold)
  float sim_threshold = 0.f;
  // uint8 pixels: the psv_set_u8_input setup the forward ran with, for the backward's im2col (the handle's own may change
  // in between); u8_tables is a copy of the handle's coefficient tables (lazy)
  int u8_h = 0, u8_w = 0;
  float u8_mean[3] = {0.f, 0.f, 0.f}, u8_std[3] = {0.f, 0.f, 0.f};
  int32_t *u8_tables = nullptr;
  std::vector<int> T;                      // active rows per layer (host)
  std::vector<int> n_max;                  // longest sequence per layer (host)
  const void *pixels = nullptr; int pixel_type = 0;
  int32_t *idx = nullptr;                  // [L][R]
  int32_t *cu = nullptr;                   // [L][MB + 1]
  float *x0 = nullptr, *a1 = nullptr, *qkv = nullptr, *ctx = nullptr, *x1 = nullptr, *a2 = nullptr, *u = nullptr;   // [L][R, width]
  float *cls = nullptr;                    // [MB, D] final CLS rows (the head's input; h->hidden is shared with psv_forward)
  // backward scratch
  float *dH = nullptr, *dy = nullptr, *dmid = nullptr, *da = nullptr, *dx1 = nullptr, *dctx = nullptr, *dqkv = nullptr, *z = nullptr;
  // the layers' compressor losses as part of the objective (loss_type "both"): per layer d loss_l / d first-layer
  // pre-activation [MB*(N-1), CH], its per-image sums [MB, CH], the compressor gradient for d loss_l = 1, the loss values
  // split-bf16 operand planes of the tensor-core GEMMs (PSV_TRAIN_TC, default on): activation side / weight side
  SplitPlanes pa{nullptr, nullptr, nullptr}, pw{nullptr, nullptr, nullptr};
  bool tc = false, fwd_three = true;       // forward products with three planes (fp32-exact operands): the skip decisions
                                           // and the layer losses then see the same hidden states as the FFMA path
  bool with_comp = false;
  float *delta = nullptr, *dsum = nullptr, *cgrad = nullptr, *closs = nullptr;
  std::vector<void *> all;
};

}  // namespace psv

namespace psv {
void train_save_free(PsvHandle *h) {
  if (!h || !h->train_save) return;
  for (void *p : h->train_save->all) cudaFree(p);
  delete h->train_save;
  h->train_save = nullptr;
}
}  // namespace psv

using namespace psv;

// flat gradient layout (floats), see include/psv.h
static int64_t bb_layer_params(const PsvHandle *h) {
  const int64_t D = h->D, F = h->F;
  return 2 * D + 3 * D * D + 3 * D + D * D + D + 2 * D + F * D + F + D * F + D;
}
static int64_t bb_embed_params(const PsvHandle *h) { return (int64_t)h->D + (int64_t)h->N * h->D + (int64_t)h->D * h->KP + h->D; }

extern "C" {
#pragma GCC visibility push(default)

int64_t psv_backbone_param_count(const PsvHandle *h) {
  if (!h) return 0;
  return bb_embed_params(h) + (int64_t)h->L * bb_layer_params(h) + 2 * h->D + (int64_t)h->C * h->D + h->C;
}

static int ensure_train_save(PsvHandle *h) {
  if (h->train_save) return PSV_OK;
  TrainSave *ts = new TrainSave();
  const int64_t R = h->R, D = h->D, F = h->F, L = h->L, MB = h->cfg.max_batch;
  auto alloc = [&](auto **p, size_t count) -> cudaError_t {
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), count * sizeof(**p) + 256);
    if (e == cudaSuccess) ts->all.push_back(*p);
    return e;
  };
  cudaError_t e = alloc(&ts->idx, (size_t)(L * R));
  if (e == cudaSuccess) e = alloc(&ts->cu, (size_t)(L * (MB + 1)));
  if (e == cudaSuccess) e = alloc(&ts->x0, (size_t)(L * R * D));
  if (e == cudaSuccess) e = alloc(&ts->a1, (size_t)(L * R * D));
  if (e == cudaSuccess) e = alloc(&ts->qkv, (size_t)(L * R * 3 * D));
  if (e == cudaSuccess) e = alloc(&ts->ctx, (size_t)(L * R * D));
  if (e == cudaSuccess) e = alloc(&ts->x1, (size_t)(L * R * D));
  if (e == cudaSuccess) e = alloc(&ts->a2, (size_t)(L * R * D));
  if (e == cudaSuccess) e = alloc(&ts->u, (size_t)(L * R * F));
  if (e == cudaSuccess) e = alloc(&ts->dH, (size_t)(R * D));
  if (e == cudaSuccess) e = alloc(&ts->dy, (size_t)(R * D));
  const size_t mid = (size_t)R * F, col = (size_t)MB * (h->N - 1) * h->KP;
  if (e == cudaSuccess) e = alloc(&ts->dmid, mid > col ? mid : col);
  if (e == cudaSuccess) e = alloc(&ts->da, (size_t)(R * D));
  if (e == cudaSuccess) e = alloc(&ts->dx1, (size_t)(R * D));
  if (e == cudaSuccess) e = alloc(&ts->dctx, (size_t)(R * D));
  if (e == cudaSuccess) e = alloc(&ts->dqkv, (size_t)(R * 3 * D));
  if (e == cudaSuccess) e = alloc(&ts->z, (size_t)(MB * D));
  if (e == cudaSuccess) e = alloc(&ts->cls, (size_t)(MB * D));
  static const bool want_tc = !(getenv("PSV_TRAIN_TC") && atoi(getenv("PSV_TRAIN_TC")) == 0);
  ts->tc = want_tc && D % 128 == 0 && F % 128 == 0 && h->KP % 128 == 0 && tmap_encode_available();
  if (ts->tc) {
    // largest operand: [F, R + 64] (transposed activations, K padded) or [R, F]
    size_t plane = (size_t)(R + 64) * F;
    const size_t wmax = (size_t)F * D > (size_t)3 * D * D ? (size_t)F * D : (size_t)3 * D * D;
    const size_t colp = (size_t)h->KP * (MB * (h->N - 1) + 64);
    if (colp > plane) plane = colp;
    if (e == cudaSuccess) e = alloc(&ts->pa.hi, plane);
    if (e == cudaSuccess) e = alloc(&ts->pa.lo, plane);
    if (e == cudaSuccess) e = alloc(&ts->pw.hi, plane > wmax ? plane : wmax);
    if (e == cudaSuccess) e = alloc(&ts->pw.lo, plane > wmax ? plane : wmax);
    static const bool two = getenv("PSV_TRAIN_FWD_PLANES") && atoi(getenv("PSV_TRAIN_FWD_PLANES")) == 2;
    ts->fwd_three = !two;
    if (ts->fwd_three) {                   // forward operands only: [R, F] activations, [F, D] / [3D, D] weights
      if (e == cudaSuccess) e = alloc(&ts->pa.mid, (size_t)R * F);
      if (e == cudaSuccess) e = alloc(&ts->pw.mid, wmax > (size_t)D * h->KP ? wmax : (size_t)D * h->KP);
    }
    if (e == cudaSuccess) e = configure_gemm_tc();
  }
  if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AB_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AB_SMEM);
  if (e != cudaSuccess) {
    for (void *p : ts->all) cudaFree(p);
    delete ts;
    h->err = std::string("training workspace allocation failed: ") + cudaGetErrorString(e);
    return PSV_ERR_CUDA;
  }
  h->train_save = ts;
  return PSV_OK;
}

static int ensure_train_comp(PsvHandle *h) {
  TrainSave *ts = h->train_save;
  if (ts->delta) return PSV_OK;
  const size_t L = h->L, MB = h->cfg.max_batch;
  float *delta = nullptr, *dsum = nullptr, *cgrad = nullptr, *closs = nullptr;
  cudaError_t e = cudaMalloc((void **)&delta, L * MB * (h->N - 1) * CH * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void **)&dsum, L * MB * CH * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void **)&cgrad, L * (size_t)h->comp_per_layer * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void **)&closs, L * sizeof(float));
  if (e != cudaSuccess) {
    cudaFree(delta); cudaFree(dsum); cudaFree(cgrad); cudaFree(closs);
    h->err = std::string("training workspace allocation failed: ") + cudaGetErrorString(e);
    return PSV_ERR_CUDA;
  }
  ts->delta = delta; ts->dsum = dsum; ts->cgrad = cgrad; ts->closs = closs;
  for (void *p : {(void *)delta, (void *)dsum, (void *)cgrad, (void *)closs}) ts->all.push_back(p);
  return PSV_OK;
}

int psv_backbone_forward_train(PsvHandle *h, const void *pixels, int32_t pixel_type, int32_t batch, float mlp_threshold,
                               float *logits, float *layer_losses, void *stream) {
  if (!h || !pixels || !logits) return tfail(h, PSV_ERR_INVALID, "null argument");
  if (!h->weights_loaded) return tfail(h, PSV_ERR_STATE, "psv_load_weights has not been called");
  if (h->cfg.precision != PSV_FP32)
    return tfail(h, PSV_ERR_UNSUPPORTED, "backbone fine-tuning runs on PSV_FP32 handles (the parity-first form of the path)");
  if (batch < 1 || batch > h->cfg.max_batch) return tfail(h, PSV_ERR_INVALID, "batch outside [1, max_batch]");
  if (int rcp = check_pixel_type(h, pixel_type)) return rcp;
  if (pixel_type == PSV_PIXELS_BF16)
    return tfail(h, PSV_ERR_UNSUPPORTED, "fine-tuning takes fp32 pixel_values or raw uint8 images");
  if (h->N > AB_MAX_N || h->D / h->H != AB_DH) return tfail(h, PSV_ERR_UNSUPPORTED, "fine-tuning supports up to 200 tokens and 64-wide heads");
  if (layer_losses && h->loss_variant != PSV_LOSS_MASK_LABELS)
    return tfail(h, PSV_ERR_UNSUPPORTED, "the joint objective follows himanshu/model_utils.py:95-108 (labels = the layer's own mask)");
  int prev = -1;
  cudaGetDevice(&prev);
  if (prev != h->device) cudaSetDevice(h->device);
  const bool similarity = h->skip_criterion == PSV_SKIP_SIMILARITY;
  int rc = ensure_train_save(h);
  if (!rc && layer_losses) rc = ensure_train_comp(h);
  if (!rc && similarity) rc = ensure_criterion_buffers(h);
  if (!rc && pixel_type == PSV_PIXELS_U8_HWC && !h->train_save->u8_tables) {
    cudaError_t e = cudaMalloc((void **)&h->train_save->u8_tables, (size_t)6 * h->cfg.image * sizeof(int32_t));
    if (e == cudaSuccess) h->train_save->all.push_back(h->train_save->u8_tables);
    else rc = tfail(h, PSV_ERR_CUDA, "training workspace allocation failed");
  }
  if (rc) { if (prev != h->device) cudaSetDevice(prev); return rc; }
  h->train_save->with_comp = layer_losses != nullptr;
  TrainSave &ts = *h->train_save;
  cudaStream_t s = (cudaStream_t)stream;
  const int D = h->D, F = h->F, N = h->N, L = h->L, MB = h->cfg.max_batch;
  const int64_t R = h->R;
  const int rows_max = batch * N;
  const bool kv_all = h->kv_mode == PSV_KV_ALL;
  const float st = h->skip_st;
  // out[out_idx] = A[m, K] . W[N, K]^T + bias (+ res[res_idx]): split-bf16 tensor-core passes, or the FFMA kernel
  auto fwd_gemm = [&](const float *A, int K, const float *W, int N, const float *bias, const float *res,
                      const int32_t *res_idx, float *out, const int32_t *out_idx, int m_max,
                      const int32_t *m_dev) -> cudaError_t {
    if (!ts.tc || N % 128 != 0 || K % 64 != 0) {
      GemmArgs g;
      g.a = A; g.w = W; g.bias = bias; g.res = res; g.res_idx = res_idx; g.out = out; g.out_idx = out_idx; g.out_fp32 = 1;
      g.m_max = m_max; g.n = N; g.k = K; g.m_dev = m_dev;
      return launch_gemm_simt(h, g, s);
    }
    cudaError_t e = split_planes(A, K, m_max, K, false, K, ts.pa, ts.fwd_three, s, m_dev);
    if (e == cudaSuccess) e = split_planes(W, K, N, K, false, K, ts.pw, ts.fwd_three, s);
    if (e == cudaSuccess) e = split_gemm(h, ts.pa, ts.pw, out, m_max, N, K, bias, res, res_idx, out_idx, m_dev, ts.fwd_three, s);
    return e;
  };
  auto body = [&]() -> int {
    // embeddings (model_utils.py:227-229)
    if (pixel_type == PSV_PIXELS_U8_HWC)
      T_CUDA(h, cudaMemcpyAsync(ts.u8_tables, h->u8_tables, (size_t)6 * h->cfg.image * sizeof(int32_t),
                                cudaMemcpyDeviceToDevice, s));
    T_CUDA(h, launch_im2col(h, pixels, pixel_type, batch, h->act_mid, s));
    T_CUDA(h, fwd_gemm((const float *)h->act_mid, h->KP, h->patch_w, D, h->patch_b, h->pos_emb, h->embed_pos_idx, h->hidden,
                       h->embed_out_idx, batch * (N - 1), nullptr));
    T_CUDA(h, launch_cls_rows(h, h->hidden, batch, s));
    for (int l = 0; l < L; ++l) {
      const LayerPack &lp = h->layers[l];
      int32_t *idx = ts.idx + (size_t)l * R, *cu = ts.cu + (size_t)l * (MB + 1);
      float *x0 = ts.x0 + (size_t)l * R * D, *a1 = ts.a1 + (size_t)l * R * D, *qkv = ts.qkv + (size_t)l * R * 3 * D;
      float *ctx = ts.ctx + (size_t)l * R * D, *x1 = ts.x1 + (size_t)l * R * D, *a2 = ts.a2 + (size_t)l * R * D;
      float *u = ts.u + (size_t)l * R * F;
      if (similarity) {
        // the similarity criterion (pradeep/model_utils.py:73-84): the dense layer over all batch * N rows with the
        // forward's split-bf16 products, in backward scratch (no backward runs during a forward), then
        // mask = [1, sim(dense_out, layer input) < st]
        T_CUDA(h, launch_ln_rows(h, h->hidden, nullptr, lp.ln1_w, lp.ln1_b, ts.da, rows_max, nullptr, s));
        T_CUDA(h, fwd_gemm(ts.da, D, lp.wqkv, 3 * D, lp.bqkv, nullptr, nullptr, ts.dqkv, nullptr, rows_max, nullptr));
        T_CUDA(h, launch_attention_simt(h, ts.dqkv, ts.dctx, h->dense_cu, batch, s));
        T_CUDA(h, fwd_gemm(ts.dctx, D, lp.wo, D, lp.bo, h->hidden, nullptr, ts.dx1, nullptr, rows_max, nullptr));
        T_CUDA(h, launch_ln_rows(h, ts.dx1, nullptr, lp.ln2_w, lp.ln2_b, ts.da, rows_max, nullptr, s));
        T_CUDA(h, fwd_gemm(ts.da, D, lp.w1, F, lp.b1, nullptr, nullptr, ts.dmid, nullptr, rows_max, nullptr));
        gelu_fwd_kernel<<<148 * 8, 256, 0, s>>>(ts.dmid, (float *)h->act_mid, (int64_t)rows_max * F, nullptr, F);
        T_CUDA(h, fwd_gemm((const float *)h->act_mid, F, lp.w2, D, lp.b2, ts.dx1, nullptr, h->dense_out, nullptr, rows_max,
                           nullptr));
        T_CUDA(h, launch_similarity(h, h->dense_out, h->hidden, batch, h->stat_scratch, s));
        T_CUDA(h, launch_sim_mask(h, h->stat_scratch, batch, st, h->crit_mask, s));
      }
      // decision + compaction + LN1 (model_utils.py:62-68, 88-91; HF:333); under the similarity criterion the scores are
      // still computed (the joint objective's layer losses read them) and the similarity mask decides
      T_CUDA(h, launch_score_mask(h, lp, h->hidden, batch, mlp_threshold, similarity ? h->crit_mask : nullptr, nullptr,
                                  nullptr, nullptr, s));
      if (layer_losses) {
        // loss_l (model_utils.py:103-108) from the layer INPUT, its compressor gradient for an upstream gradient of 1,
        // and d loss_l / d pre-activation, which the backward sends on into the backbone through W1
        T_CUDA(h, enqueue_compressor_layer_grads(h, l, h->hidden, batch, h->mask, h->scores, nullptr, 1.0f,
                                                 ts.cgrad + (size_t)l * h->comp_per_layer, ts.closs + l, s));
        T_CUDA(h, cudaMemcpyAsync(ts.delta + (size_t)l * MB * (N - 1) * CH, h->train_delta,
                                  (size_t)batch * (N - 1) * CH * sizeof(float), cudaMemcpyDeviceToDevice, s));
        T_CUDA(h, cudaMemcpyAsync(ts.dsum + (size_t)l * MB * CH, h->train_dsum, (size_t)batch * CH * sizeof(float),
                                  cudaMemcpyDeviceToDevice, s));
      }
      T_CUDA(h, launch_gather_ln(h, lp, h->hidden, batch, nullptr, false, s, kv_all));      // kv_all: compaction only
      T_CUDA(h, cudaMemcpyAsync(idx, h->idx, (size_t)rows_max * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
      T_CUDA(h, cudaMemcpyAsync(cu, h->cu_seqlens, (size_t)(batch + 1) * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
      const int32_t *m_dev = h->cu_seqlens + batch;
      if (kv_all) {
        // the layer input, LN1 and q|k|v of ALL rows in dense order: skipped tokens are keys / values too
        // (recap/convprad4.py:341-352); every active query attends to the N tokens of its image
        T_CUDA(h, launch_ln_rows(h, h->hidden, nullptr, lp.ln1_w, lp.ln1_b, a1, rows_max, nullptr, s));
        T_CUDA(h, cudaMemcpyAsync(x0, h->hidden, (size_t)rows_max * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
        T_CUDA(h, fwd_gemm(a1, D, lp.wqkv, 3 * D, lp.bqkv, nullptr, nullptr, qkv, nullptr, rows_max, nullptr));
        T_CUDA(h, launch_attention_simt(h, qkv, ctx, h->cu_seqlens, batch, s, h->idx, N));
      } else {
        // rows past T are never read back: copying the worst case keeps the forward free of host synchronisation
        T_CUDA(h, cudaMemcpyAsync(a1, h->act_a, (size_t)rows_max * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
        rows_copy_kernel<<<grid_for64((int64_t)rows_max * D / 4, 256, 148 * 8), 256, 0, s>>>(h->hidden, x0, h->idx, rows_max, D,
                                                                                               0, m_dev);
        T_CUDA(h, fwd_gemm(a1, D, lp.wqkv, 3 * D, lp.bqkv, nullptr, nullptr, qkv, nullptr, rows_max, m_dev));
        T_CUDA(h, launch_attention_simt(h, qkv, ctx, h->cu_seqlens, batch, s));
      }
      T_CUDA(h, fwd_gemm(ctx, D, lp.wo, D, lp.bo, h->hidden, h->idx, x1, nullptr, rows_max, m_dev));
      T_CUDA(h, launch_ln_rows(h, x1, nullptr, lp.ln2_w, lp.ln2_b, a2, rows_max, m_dev, s));
      T_CUDA(h, fwd_gemm(a2, D, lp.w1, F, lp.b1, nullptr, nullptr, u, nullptr, rows_max, m_dev));
      gelu_fwd_kernel<<<148 * 8, 256, 0, s>>>(u, (float *)h->act_mid, (int64_t)rows_max * F, m_dev, F);
      T_CUDA(h, fwd_gemm((const float *)h->act_mid, F, lp.w2, D, lp.b2, x1, nullptr, h->hidden, h->idx, rows_max, m_dev));
    }
    T_CUDA(h, launch_head(h, h->hidden, batch, logits, s));
    rows_copy_kernel<<<grid_for64((int64_t)batch * D / 4, 256, 148), 256, 0, s>>>(h->hidden, ts.cls, h->dense_cu, batch, D, 0);
    if (layer_losses)
      T_CUDA(h, cudaMemcpyAsync(layer_losses, ts.closs, (size_t)L * sizeof(float), cudaMemcpyDeviceToDevice, s));
    // the backward sizes its GEMMs with the exact row counts and its attention kernel with the longest sequence of each
    // layer: one synchronisation per training step
    std::vector<int32_t> cu_host((size_t)L * (batch + 1));
    for (int l = 0; l < L; ++l)
      T_CUDA(h, cudaMemcpyAsync(cu_host.data() + (size_t)l * (batch + 1), ts.cu + (size_t)l * (MB + 1),
                                (size_t)(batch + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    T_CUDA(h, cudaStreamSynchronize(s));
    ts.T.assign((size_t)L, 0);
    ts.n_max.assign((size_t)L, 0);
    for (int l = 0; l < L; ++l) {
      const int32_t *c = cu_host.data() + (size_t)l * (batch + 1);
      ts.T[l] = c[batch];
      for (int b = 0; b < batch; ++b) ts.n_max[l] = std::max(ts.n_max[l], (int)(c[b + 1] - c[b]));
    }
    ts.batch = batch; ts.pixels = pixels; ts.pixel_type = pixel_type; ts.kv_all = kv_all;
    ts.criterion = h->skip_criterion; ts.sim_threshold = st;
    if (pixel_type == PSV_PIXELS_U8_HWC) {
      ts.u8_h = h->u8_h; ts.u8_w = h->u8_w;
      for (int c = 0; c < 3; ++c) { ts.u8_mean[c] = h->u8_mean[c]; ts.u8_std[c] = h->u8_std[c]; }
    }
    return PSV_OK;
  };
  rc = body();
  if (prev != h->device) cudaSetDevice(prev);
  return rc;
}

int psv_backbone_backward(PsvHandle *h, const float *dlogits, const float *dlosses, float *grads, float *comp_grads,
                          void *stream) {
  if (!h || !dlogits || !grads) return tfail(h, PSV_ERR_INVALID, "null argument");
  if (!h->train_save || h->train_save->batch < 1)
    return tfail(h, PSV_ERR_STATE, "psv_backbone_forward_train has not been called");
  if ((dlosses != nullptr) != (comp_grads != nullptr)) return tfail(h, PSV_ERR_INVALID, "dlosses and comp_grads go together");
  if (dlosses && !h->train_save->with_comp)
    return tfail(h, PSV_ERR_STATE, "the forward did not keep the layers' compressor losses (layer_losses was null)");
  if (!psv_hidden_supported(h->D)) return tfail(h, PSV_ERR_UNSUPPORTED, "no LayerNorm backward for this hidden width");
  int prev = -1;
  cudaGetDevice(&prev);
  if (prev != h->device) cudaSetDevice(h->device);
  TrainSave &ts = *h->train_save;
  cudaStream_t s = (cudaStream_t)stream;
  const int D = h->D, F = h->F, N = h->N, L = h->L, C = h->C, MB = h->cfg.max_batch, KP = h->KP;
  const int64_t R = h->R;
  const int batch = ts.batch;
  const float eps = h->cfg.ln_eps;
  // flat layout
  float *g_cls = grads, *g_pos = g_cls + D, *g_pw = g_pos + (size_t)N * D, *g_pb = g_pw + (size_t)D * KP;
  float *g_layers = g_pb + D;
  const int64_t per = bb_layer_params(h);
  float *g_fln_w = g_layers + (size_t)L * per, *g_fln_b = g_fln_w + D, *g_cw = g_fln_b + D, *g_cb = g_cw + (size_t)C * D;
  auto colsum = [&](const float *x, int rows, int width, float *out) {
    if (rows <= 0) return;
    if (width % 4 != 0) { colsum_slow_kernel<<<dim3((width + 127) / 128, rows < 64 ? rows : 64), 128, 0, s>>>(x, rows, width, out); return; }
    const int gx = (width / 4 + 31) / 32;
    int gy = (148 * 4 + gx - 1) / gx;
    if (gy > (rows + 7) / 8) gy = (rows + 7) / 8;
    colsum_kernel<<<dim3(gx, gy < 1 ? 1 : gy), 256, 0, s>>>(x, rows, width, out);
  };
  auto ln_bwd = [&](const float *x, const int32_t *x_idx, const float *dy, const float *gamma, int rows, float *dx, int add,
                    float *dgamma, float *dbeta) {
    if (rows <= 0) return;
    const int grid = grid_for64(rows, 8, 148 * 4);
    // D is one of the widths psv_create accepts, checked again on entry
    if (D == 1024)     ln_bwd_kernel<1024><<<grid, 256, 0, s>>>(x, x_idx, dy, gamma, eps, rows, dx, add, dgamma, dbeta);
    else if (D == 768) ln_bwd_kernel<768><<<grid, 256, 0, s>>>(x, x_idx, dy, gamma, eps, rows, dx, add, dgamma, dbeta);
    else if (D == 384) ln_bwd_kernel<384><<<grid, 256, 0, s>>>(x, x_idx, dy, gamma, eps, rows, dx, add, dgamma, dbeta);
  };
  // dW[Dout, Din] = dY[rows, Dout]^T . X[rows, Din]   and   dX[rows, Din] = dY[rows, Dout] . W[Dout, Din]
  auto wgrad = [&](const float *dY, int Dout, const float *X, int Din, int rows, float *dW) -> cudaError_t {
    if (!ts.tc || Din % 128 != 0) return train_gemm(dY, Dout, true, X, Din, false, dW, Din, Dout, Din, rows, false, s);
    const int kp = (rows + 63) / 64 * 64;                        // K of this GEMM = the row count, zero-padded to 64
    cudaError_t e = split_planes(dY, Dout, rows, Dout, true, kp, ts.pa, false, s);
    if (e == cudaSuccess) e = split_planes(X, Din, rows, Din, true, kp, ts.pw, false, s);
    if (e == cudaSuccess) e = split_gemm(h, ts.pa, ts.pw, dW, Dout, Din, kp, nullptr, nullptr, nullptr, nullptr, nullptr, false, s);
    return e;
  };
  auto dgrad = [&](const float *dY, int Dout, const float *W, int Din, int rows, float *dX) -> cudaError_t {
    if (!ts.tc || Din % 128 != 0 || Dout % 64 != 0)
      return train_gemm(dY, Dout, false, W, Din, false, dX, Din, rows, Din, Dout, false, s);
    cudaError_t e = split_planes(dY, Dout, rows, Dout, false, Dout, ts.pa, false, s);
    if (e == cudaSuccess) e = split_planes(W, Din, Dout, Din, true, Dout, ts.pw, false, s);      // W^T [Din, Dout]
    if (e == cudaSuccess) e = split_gemm(h, ts.pa, ts.pw, dX, rows, Din, Dout, nullptr, nullptr, nullptr, nullptr, nullptr, false, s);
    return e;
  };
  auto body = [&]() -> int {
    T_CUDA(h, cudaMemsetAsync(grads, 0, (size_t)psv_backbone_param_count(h) * sizeof(float), s));
    T_CUDA(h, cudaMemsetAsync(ts.dH, 0, (size_t)batch * N * D * sizeof(float), s));
    // ---- head (model_utils.py:241,254): logits = LN_f(hidden[b, 0]) . Wc^T + bc, on the CLS rows the forward kept
    T_CUDA(h, launch_ln_rows(h, ts.cls, nullptr, h->final_ln_w, h->final_ln_b, ts.z, batch, nullptr, s));
    T_CUDA(h, train_gemm(dlogits, C, true, ts.z, D, false, g_cw, D, C, D, batch, false, s));              // dWc = dlogits^T z
    colsum(dlogits, batch, C, g_cb);
    T_CUDA(h, train_gemm(dlogits, C, false, h->cls_w, D, false, ts.da, D, batch, D, C, false, s));        // dz = dlogits Wc
    ln_bwd(ts.cls, nullptr, ts.da, h->final_ln_w, batch, ts.dy, 0, g_fln_w, g_fln_b);
    // the CLS rows of dH are rows b * N = dense_cu[b]
    rows_copy_kernel<<<grid_for64((int64_t)batch * D / 4, 256, 148), 256, 0, s>>>(ts.dy, ts.dH, h->dense_cu, batch, D, 1);
    // ---- layers in reverse
    for (int l = L - 1; l >= 0; --l) {
      const LayerPack &lp = h->layers[l];
      const int T = ts.T[l];
      const int32_t *idx = ts.idx + (size_t)l * R, *cu = ts.cu + (size_t)l * (MB + 1);
      const float *x0 = ts.x0 + (size_t)l * R * D, *a1 = ts.a1 + (size_t)l * R * D, *qkv = ts.qkv + (size_t)l * R * 3 * D;
      const float *ctx = ts.ctx + (size_t)l * R * D, *x1 = ts.x1 + (size_t)l * R * D, *a2 = ts.a2 + (size_t)l * R * D;
      const float *u = ts.u + (size_t)l * R * F;
      float *gl = g_layers + (size_t)l * per;
      float *g_ln1w = gl, *g_ln1b = g_ln1w + D, *g_wqkv = g_ln1b + D, *g_bqkv = g_wqkv + (size_t)3 * D * D;
      float *g_wo = g_bqkv + 3 * D, *g_bo = g_wo + (size_t)D * D, *g_ln2w = g_bo + D, *g_ln2b = g_ln2w + D;
      float *g_w1 = g_ln2b + D, *g_b1 = g_w1 + (size_t)F * D, *g_w2 = g_b1 + F, *g_b2 = g_w2 + (size_t)D * F;
      auto compressor_part = [&]() -> int {
        // dH is now d objective / d (output of layer l) -> add what loss_l sends into the layer INPUT; the layer's own
        // main-path contribution has been scattered into dH already (the skipped rows pass through unchanged)
        if (!dlosses) return PSV_OK;
        scale_copy_kernel<<<grid_for64(h->comp_per_layer, 256, 148), 256, 0, s>>>(
            ts.cgrad + (size_t)l * h->comp_per_layer, dlosses + l, comp_grads + (size_t)l * h->comp_per_layer, h->comp_per_layer);
        comp_input_grad_kernel<<<dim3((N + CI_ROWS - 1) / CI_ROWS, batch), 256, 0, s>>>(
            ts.delta + (size_t)l * MB * (N - 1) * CH, ts.dsum + (size_t)l * MB * CH, lp.c1, dlosses + l, N, D, ts.dH);
        T_CUDA(h, cudaGetLastError());
        return PSV_OK;
      };
      if (T <= 0) { if (int rcc = compressor_part()) return rcc; continue; }
      const int64_t tf = (int64_t)T * F, td = (int64_t)T * D;
      float *gact = (float *)h->act_mid;
      // dy = dH[idx]   (adjoint of the scatter-back, model_utils.py:88-91)
      rows_copy_kernel<<<grid_for64(td / 4, 256, 148 * 8), 256, 0, s>>>(ts.dH, ts.dy, idx, T, D, 0);
      // FC2 (HF:309-311): y = x1 + gelu(u) W2^T + b2
      gelu_fwd_kernel<<<grid_for64(tf / 4, 256, 148 * 8), 256, 0, s>>>(u, gact, tf, nullptr, F);
      T_CUDA(h, wgrad(ts.dy, D, gact, F, T, g_w2));                                                       // dW2 = dy^T g
      colsum(ts.dy, T, D, g_b2);
      T_CUDA(h, dgrad(ts.dy, D, lp.w2, F, T, ts.dmid));                                                   // dg = dy W2
      gelu_bwd_kernel<<<grid_for64(tf / 4, 256, 148 * 8), 256, 0, s>>>(u, ts.dmid, tf);                      // du
      // FC1 (HF:297-298)
      T_CUDA(h, wgrad(ts.dmid, F, a2, D, T, g_w1));                                                       // dW1 = du^T a2
      colsum(ts.dmid, T, F, g_b1);
      T_CUDA(h, dgrad(ts.dmid, F, lp.w1, D, T, ts.da));                                                   // da2 = du W1
      // LN2 (HF:340) and the second residual: dx1 = dy + LN2'(da2)
      T_CUDA(h, cudaMemcpyAsync(ts.dx1, ts.dy, (size_t)td * sizeof(float), cudaMemcpyDeviceToDevice, s));
      ln_bwd(x1, nullptr, ts.da, lp.ln2_w, T, ts.dx1, 1, g_ln2w, g_ln2b);
      // proj (HF:266,337)
      T_CUDA(h, wgrad(ts.dx1, D, ctx, D, T, g_wo));                                                       // dWo = dx1^T ctx
      colsum(ts.dx1, T, D, g_bo);
      T_CUDA(h, dgrad(ts.dx1, D, lp.wo, D, T, ts.dctx));                                                  // dctx = dx1 Wo
      if (ts.kv_all) {
        // active queries x all N keys (recap/convprad4.py:99-125): dqkv, LN1 and the layer input over all batch * N rows
        const int rows = batch * N;
        const int n_cap = std::min(AB_MAX_N, (N + 7) / 8 * 8);
        attention_bwd_kernel<true><<<dim3(h->H, batch), AB_WARPS * 32, ab_smem(n_cap), s>>>(qkv, ts.dctx, cu, D, ts.dqkv,
                                                                                           n_cap, idx, N);
        T_CUDA(h, wgrad(ts.dqkv, 3 * D, a1, D, rows, g_wqkv));                                            // dWqkv = dqkv^T a1
        colsum(ts.dqkv, rows, 3 * D, g_bqkv);
        T_CUDA(h, dgrad(ts.dqkv, 3 * D, lp.wqkv, D, rows, ts.da));                                        // da1 = dqkv Wqkv
        // the residual path of the active rows replaces their output gradient; skipped rows keep theirs (pass-through),
        // then every row adds its LN1 backward (dx = dx1 + LN1'(da1) on active rows, dH + LN1'(da1) on skipped ones)
        rows_copy_kernel<<<grid_for64(td / 4, 256, 148 * 8), 256, 0, s>>>(ts.dx1, ts.dH, idx, T, D, 1);
        ln_bwd(x0, nullptr, ts.da, lp.ln1_w, rows, ts.dH, 1, g_ln1w, g_ln1b);
        if (int rcc = compressor_part()) return rcc;
        continue;
      }
      // attention among the active tokens of each image (HF:171-196)
      {
        const int n_cap = std::min(AB_MAX_N, (ts.n_max[l] + 7) / 8 * 8);
        attention_bwd_kernel<false><<<dim3(h->H, batch), AB_WARPS * 32, ab_smem(n_cap), s>>>(qkv, ts.dctx, cu, D, ts.dqkv,
                                                                                            n_cap, nullptr, 0);
      }
      // QKV (HF:228-230)
      T_CUDA(h, wgrad(ts.dqkv, 3 * D, a1, D, T, g_wqkv));                                                 // dWqkv = dqkv^T a1
      colsum(ts.dqkv, T, 3 * D, g_bqkv);
      T_CUDA(h, dgrad(ts.dqkv, 3 * D, lp.wqkv, D, T, ts.da));                                             // da1 = dqkv Wqkv
      // LN1 (HF:333) and the first residual: dx = dx1 + LN1'(da1); back to the token rows (adjoint of the gather)
      ln_bwd(x0, nullptr, ts.da, lp.ln1_w, T, ts.dx1, 1, g_ln1w, g_ln1b);
      rows_copy_kernel<<<grid_for64(td / 4, 256, 148 * 8), 256, 0, s>>>(ts.dx1, ts.dH, idx, T, D, 1);
      if (int rcc = compressor_part()) return rcc;
    }
    // ---- embeddings (HF:100-128,153-167): hidden0[b, 0] = cls + pos[0];  hidden0[b, 1 + p] = patch_p . Wp^T + bp + pos[1 + p]
    batch_sum_kernel<<<grid_for64((int64_t)N * D, 256, 1024), 256, 0, s>>>(ts.dH, batch, N, D, g_pos);
    T_CUDA(h, cudaMemcpyAsync(g_cls, g_pos, (size_t)D * sizeof(float), cudaMemcpyDeviceToDevice, s));     // d cls = d pos[0]
    const int prow = batch * (N - 1);
    rows_copy_kernel<<<grid_for64((int64_t)prow * D / 4, 256, 148 * 8), 256, 0, s>>>(ts.dH, ts.dy, h->embed_out_idx, prow, D, 0);
    if (ts.pixel_type == PSV_PIXELS_U8_HWC)           // the setup of the forward, not the handle's current one
      T_CUDA(h, launch_im2col_u8(h, (const uint8_t *)ts.pixels, batch, ts.dmid, ts.u8_h, ts.u8_w, ts.u8_tables, ts.u8_mean,
                                 ts.u8_std, s));
    else
      T_CUDA(h, launch_im2col(h, ts.pixels, ts.pixel_type, batch, ts.dmid, s));
    T_CUDA(h, wgrad(ts.dy, D, ts.dmid, KP, prow, g_pw));                                                 // dWp = dHp^T patches
    colsum(ts.dy, prow, D, g_pb);
    T_CUDA(h, cudaGetLastError());
    return PSV_OK;
  };
  const int rc = body();
  if (prev != h->device) cudaSetDevice(prev);
  return rc;
}

int psv_backbone_train_masks(PsvHandle *h, uint8_t *masks_out, void *stream) {
  if (!h) return PSV_ERR_INVALID;
  if (!h->train_save || h->train_save->batch < 1)
    return tfail(h, PSV_ERR_STATE, "psv_backbone_forward_train has not been called");
  if (!masks_out) return tfail(h, PSV_ERR_INVALID, "null argument");
  int prev = -1;
  cudaGetDevice(&prev);
  if (prev != h->device) cudaSetDevice(h->device);
  const TrainSave &ts = *h->train_save;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t per = (size_t)ts.batch * h->N;
  auto body = [&]() -> int {
    T_CUDA(h, cudaMemsetAsync(masks_out, 0, (size_t)h->L * per, s));
    for (int l = 0; l < h->L; ++l)
      if (ts.T[l] > 0)
        mark_rows_kernel<<<grid_for64(ts.T[l], 256, 148), 256, 0, s>>>(ts.idx + (size_t)l * h->R, ts.T[l], masks_out + l * per);
    T_CUDA(h, cudaGetLastError());
    return PSV_OK;
  };
  const int rc = body();
  if (prev != h->device) cudaSetDevice(prev);
  return rc;
}

#pragma GCC visibility pop
}
