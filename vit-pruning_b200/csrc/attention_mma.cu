// K6 (bf16 mode): varlen flash-style attention among the ACTIVE tokens of each image on the
// tensor cores (reference model_utils.py:91 -> HF:171-196: softmax(q k^T / 8) v).
//
// One CTA (4 warps) per (head, image); n <= 197 active tokens.  Queries are taken 64 at a time (one
// 16-query block per warp) and keys/values stream through a double-buffered pair of 64-row tiles
// (cp.async prefetch of chunk k+1 while chunk k is multiplied), all in an XOR-swizzled layout
// (16-byte chunk ^= row & 7) so every ldmatrix is bank-conflict free.  40 KB of shared memory per
// CTA keeps 5 CTAs resident per SM, which is what hides the load latency for the typical short
// sequences.  fp32 online softmax (running max / sum in registers, exp2 with the 1/8 scale folded
// in); S = Q K^T and O += P V are mma.sync m16n8k16 bf16 with fp32 accumulators in registers.
//
// Tensor-path note: this is the legacy warp-level mma.sync path (HMMA), not tcgen05 -- attention
// is <= 4 % of the path's FLOPs (SURVEY.md 7.3) and per-image sequences are at most 197 tokens,
// so a whole (image, head) problem is smaller than one 128-row tcgen05 tile; see DESIGN.md.
#include "psv_internal.cuh"

namespace psv {
namespace {

constexpr int AM_THREADS = 128;
constexpr int AM_WARPS = 4;
constexpr int DH = 64;
constexpr int GROUP = 64;                        // queries per pass (16 per warp) and keys per chunk
constexpr int TILE_BYTES = GROUP * DH * 2;       // 8 KB: 64 rows x 128 B
constexpr size_t AM_SMEM = (size_t)5 * TILE_BYTES;   // Q + double-buffered K and V : 40 KB -> 5 CTAs / SM

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// byte offset of (row, 16B-chunk) in a [rows][64] bf16 tile with XOR swizzle
__device__ __forceinline__ uint32_t sw_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, bool valid) {
  const int sz = valid ? 16 : 0;                 // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2_approx(float x) {      // one MUFU.EX2 (ex2(-inf) = +0)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}

// stage `rows16` rows (16-byte chunks, zero-filled past n) of matrix `mat` (0 Q, 1 K, 2 V) starting at
// token `first` into a swizzled [64][128 B] tile
// (`rows` non-null: token i lives in row rows[i] of `base` -- the queries of the keep-all-keys mode)
__device__ __forceinline__ void stage_rows(uint32_t tile, const bf16 *base, size_t ld, int D, int mat, int first,
                                           int rows16, int n, int tid, const int32_t *__restrict__ rows = nullptr) {
  for (int e = tid; e < rows16 * 8; e += AM_THREADS) {
    const int row = e >> 3, chunk = e & 7;
    const bool valid = first + row < n;
    const int tok = valid ? first + row : 0;
    const bf16 *src = base + (size_t)(rows ? (valid ? rows[tok] : 0) : tok) * ld + mat * D + chunk * 8;
    cp_async16(tile + sw_off(row, chunk), src, valid);
  }
}

__global__ void __launch_bounds__(AM_THREADS)
attention_mma_kernel(const bf16 *__restrict__ qkv, bf16 *__restrict__ ctx, const int32_t *__restrict__ cu_seqlens,
                     int D, const int32_t *__restrict__ q_rows, int kv_tokens) {
  extern __shared__ __align__(128) uint8_t smem[];
  pdl_wait();
  const int head = blockIdx.x, b = blockIdx.y;
  const int row0 = cu_seqlens[b];
  const int nq = cu_seqlens[b + 1] - row0;
  if (nq <= 0) return;
  // Default: queries = keys = the image's active tokens, rows row0.. of the packed qkv.  Keep-all-keys mode (kv_tokens
  // = N > 0, reference recap/convprad4.py:99-125,191-193): qkv holds ALL rows in dense order, the keys / values are the
  // image's kv_tokens rows and the queries its active rows q_rows[row0 + i]; ctx stays packed (row0 + i).
  const int n = kv_tokens > 0 ? kv_tokens : nq;                    // keys
  const int n16 = (n + 15) & ~15, nq16_all = (nq + 15) & ~15;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t ld = (size_t)3 * D;
  const bf16 *base = qkv + (size_t)(kv_tokens > 0 ? b * kv_tokens : row0) * ld + head * DH;
  const bf16 *qbase = kv_tokens > 0 ? qkv + head * DH : base;
  const int32_t *qr = kv_tokens > 0 ? q_rows + row0 : nullptr;
  const uint32_t aQ = smem_addr(smem);
  const uint32_t aKV = aQ + TILE_BYTES;            // [buf][K|V] tiles
  const float sl2 = 0.125f * 1.4426950408889634f;  // softmax scale * log2(e)
  const int g = lane >> 2, t = lane & 3;
  const int nkc = (n16 + GROUP - 1) / GROUP;       // key chunks
  // Per-lane ldmatrix offsets inside a [64][128 B] swizzled tile.  All row offsets added later are multiples of
  // 16 rows (2048 B, row & 7 unchanged), so the XOR-swizzled chunk is a per-lane constant for each k-step / dim block.
  uint32_t offQ[4], offK[4], offV[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    offQ[i] = sw_off(warp * 16 + (lane & 15), i * 2 + (lane >> 4));
    offK[i] = sw_off((lane & 7) + ((lane >> 4) << 3), i * 2 + ((lane >> 3) & 1));
    offV[i] = sw_off((lane & 7) + (((lane >> 3) & 1) << 3), i * 2 + (lane >> 4));
  }

  for (int qg = 0; qg < nq; qg += GROUP) {
    const int nq16 = min(GROUP, nq16_all - qg);
    stage_rows(aQ, qbase, ld, D, 0, qg, nq16, nq, tid, qr);
    {
      const int r16 = min(GROUP, n16);
      stage_rows(aKV, base, ld, D, 1, 0, r16, n, tid);
      stage_rows(aKV + TILE_BYTES, base, ld, D, 2, 0, r16, n, tid);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    const bool active = warp * 16 < nq16;          // this warp's 16-query block exists
    uint32_t qf[4][4];
    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;      // rows g and g+8

    for (int kc = 0; kc < nkc; ++kc) {
      const uint32_t aK = aKV + (kc & 1) * 2 * TILE_BYTES, aV = aK + TILE_BYTES;
      if (kc + 1 < nkc) {                           // prefetch the next key chunk into the other buffer
        const int first = (kc + 1) * GROUP, r16 = min(GROUP, n16 - first);
        const uint32_t nK = aKV + ((kc + 1) & 1) * 2 * TILE_BYTES;
        stage_rows(nK, base, ld, D, 1, first, r16, n, tid);
        stage_rows(nK + TILE_BYTES, base, ld, D, 2, first, r16, n, tid);
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      __syncthreads();
      if (active) {
        if (kc == 0) {
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) ldmatrix_x4(aQ + offQ[ks], qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
        }
        const int kbase = kc * GROUP;
        const int nkb = min(GROUP, n16 - kbase) >> 3;              // 8-key blocks in this chunk (even)
        float s[8][4];
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) { s[nb][0] = s[nb][1] = s[nb][2] = s[nb][3] = 0.f; }
        // S = Q K^T : B fragment (k = dim, n = key) straight from the row-major K rows.  k-step outer / key-block
        // inner, so consecutive mma.sync's hit different accumulators (8 independent chains hide the HMMA latency)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
          for (int nb2 = 0; nb2 < 4; ++nb2) {
            if (nb2 * 2 < nkb) {
              // x4: (keys 0-7, dims lo), (keys 0-7, dims hi), (keys 8-15, dims lo), (keys 8-15, dims hi)
              uint32_t b0, b1, b2, b3;
              ldmatrix_x4(aK + nb2 * 2048 + offK[ks], b0, b1, b2, b3);
              mma_bf16(s[nb2 * 2], qf[ks], b0, b1);
              mma_bf16(s[nb2 * 2 + 1], qf[ks], b2, b3);
            }
          }
        }
        // mask keys >= n (only the last chunk can hold any), chunk max
        if (kbase + GROUP > n) {
#pragma unroll
          for (int nb = 0; nb < 8; ++nb) {
            const int key = kbase + nb * 8 + 2 * t;
            if (key >= n) { s[nb][0] = -INFINITY; s[nb][2] = -INFINITY; }
            if (key + 1 >= n) { s[nb][1] = -INFINITY; s[nb][3] = -INFINITY; }
          }
        }
        float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
          cm0 = fmaxf(cm0, fmaxf(s[nb][0], s[nb][1]));
          cm1 = fmaxf(cm1, fmaxf(s[nb][2], s[nb][3]));
        }
        cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1)); cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
        cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1)); cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
        const float nm0 = fmaxf(m0, cm0), nm1 = fmaxf(m1, cm1);    // finite: the chunk's first key is valid
        const float corr0 = ex2_approx((m0 - nm0) * sl2), corr1 = ex2_approx((m1 - nm1) * sl2);
        m0 = nm0; m1 = nm1;
        const float ms0 = m0 * sl2, ms1 = m1 * sl2;                // p = 2^(s*sl2 - m*sl2): one FFMA + one MUFU
        float rs0 = 0.f, rs1 = 0.f;
        uint32_t pf[4][4];                                         // P as A fragments, 4 k-steps of 16 keys
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
          const float p0 = ex2_approx(fmaf(s[nb][0], sl2, -ms0)), p1 = ex2_approx(fmaf(s[nb][1], sl2, -ms0));
          const float p2 = ex2_approx(fmaf(s[nb][2], sl2, -ms1)), p3 = ex2_approx(fmaf(s[nb][3], sl2, -ms1));
          rs0 += p0 + p1; rs1 += p2 + p3;
          pf[nb >> 1][(nb & 1) * 2 + 0] = pack_bf16(p0, p1);
          pf[nb >> 1][(nb & 1) * 2 + 1] = pack_bf16(p2, p3);
        }
        l0 = l0 * corr0 + rs0; l1 = l1 * corr1 + rs1;
        // rescale O only when some row's running max moved (never for the first chunk: O is still zero)
        if (kc > 0 && __any_sync(0xffffffffu, corr0 != 1.0f || corr1 != 1.0f)) {
#pragma unroll
          for (int i = 0; i < 8; ++i) { o[i][0] *= corr0; o[i][1] *= corr0; o[i][2] *= corr1; o[i][3] *= corr1; }
        }
        // O += P V : B fragment (k = key, n = dim) via transposed ldmatrix on the row-major V rows
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          if (ks * 2 < nkb) {
#pragma unroll
            for (int db = 0; db < 4; ++db) {
              // x4.trans: (keys 0-7, dims db*16+0..7), (keys 8-15, same dims), (keys 0-7, dims +8), (keys 8-15, +8)
              uint32_t b0, b1, b2, b3;
              ldmatrix_x4_trans(aV + ks * 2048 + offV[db], b0, b1, b2, b3);
              mma_bf16(o[db * 2], pf[ks], b0, b1);
              mma_bf16(o[db * 2 + 1], pf[ks], b2, b3);
            }
          }
        }
      }
      __syncthreads();                              // everyone is done with this K/V buffer (and with Q at the end)
    }
    if (active) {
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
      const int r0 = qg + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
        const int col = head * DH + nb * 8 + 2 * t;
        if (r0 < nq) *reinterpret_cast<uint32_t *>(ctx + (size_t)(row0 + r0) * D + col) = pack_bf16(o[nb][0] * inv0, o[nb][1] * inv0);
        if (r1 < nq) *reinterpret_cast<uint32_t *>(ctx + (size_t)(row0 + r1) * D + col) = pack_bf16(o[nb][2] * inv1, o[nb][3] * inv1);
      }
    }
  }
}

}  // namespace

cudaError_t configure_attention_mma() {
  return cudaFuncSetAttribute(attention_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AM_SMEM);
}

cudaError_t launch_attention_mma(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                 cudaStream_t s, const int32_t *q_rows, int kv_tokens) {
  LaunchScope scope(h, KK_ATTENTION, s);
  dim3 grid(h->H, batch);
  return launch_pdl(attention_mma_kernel, grid, dim3(AM_THREADS), AM_SMEM, s, (const bf16 *)qkv, (bf16 *)ctx,
                    cu_seqlens, h->D, q_rows, kv_tokens);
}

}  // namespace psv
