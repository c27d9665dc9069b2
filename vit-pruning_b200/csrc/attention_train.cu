// Mixed-precision fine-tuning (PSV_TRAIN_BF16): varlen attention forward and backward on mma.sync m16n8k16 bf16 with
// fp32 accumulation, for packed sequences of up to AB_MAX_N (200) tokens and 64-wide heads (reference model_utils.py:91
// -> HF:171-196: softmax(q k^T / 8) v among the active tokens of one image).
//
//   forward : unit (image, block of 32 queries, head), 2 warps x 16 queries, keys in 32-row chunks, fp32 online softmax
//             (exp2, 1/8 folded in) as attention_pk.cu; P is rounded to bf16 against the running max, ctx is stored
//             bf16 and the fp32 log-sum-exp of every (row, head) is kept for the backward.
//   backward: FlashAttention-2 style in two passes, P recomputed from q, k and the saved log-sum-exp:
//             dq  pass, unit (image, 32-query block, head): Di = rowsum(dO o O) in fp32, dS = P o (dO V^T - Di),
//                       dQ = dS K / 8;
//             dkv pass, unit (image, 32-key block, head):   dV = P^T dO, dK = dS^T Q / 8.
//             MMA operands (Q, K, V, dO, P, dS) are bf16, accumulation fp32.  Di takes the same bf16-rounded dO as the
//             dO V^T product (and O, the saved bf16 ctx): where P is nearly one-hot, dP and Di nearly cancel, and an fp32
//             dO in Di alone would leave its bf16 rounding error (~2^-9 |dO| |v|) uncancelled in dS.  No atomics: every
//             output element is written by one thread after a fixed loop, so results are run-to-run bit-identical.
// Key and query chunks are aligned to the image's first row, so an image's results do not depend on its neighbours in
// the batch.  Tiles are staged through shared memory with plain 16-byte loads (rows outside the image zero-filled) in
// the 128-byte-swizzled layout that makes ldmatrix conflict-free.
#include "tc_common.cuh"

namespace psv {
namespace {

using namespace tc;

constexpr int AT_BLK = 32;               // queries (forward, dq pass) or keys (dkv pass) per unit; rows per chunk
constexpr int AT_THREADS = 64;
constexpr int AT_DH = 64;
constexpr int AT_TILE = AT_BLK * AT_DH * 2;   // 4 KB: one 32 x 64 bf16 tile
constexpr float kSl2 = 0.125f * 1.4426950408889634f;   // softmax scale * log2(e)
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ uint32_t sw_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}

// 32 rows x 64 columns into a swizzled tile: rows [row0, row0 + 32) of src (row stride ld elements, first column col);
// rows at or past `end` are zeros.  bf16 sources are copied, fp32 sources rounded to bf16.
__device__ __forceinline__ void load_tile(uint8_t *tile, const bf16 *__restrict__ src, size_t ld, int col, int row0, int end) {
  for (int p = threadIdx.x; p < AT_BLK * 8; p += AT_THREADS) {
    const int r = p >> 3, ch = p & 7;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (row0 + r < end) v = *reinterpret_cast<const uint4 *>(src + (size_t)(row0 + r) * ld + col + ch * 8);
    *reinterpret_cast<uint4 *>(tile + sw_off(r, ch)) = v;
  }
}
__device__ __forceinline__ void load_tile(uint8_t *tile, const float *__restrict__ src, size_t ld, int col, int row0, int end) {
  for (int p = threadIdx.x; p < AT_BLK * 8; p += AT_THREADS) {
    const int r = p >> 3, ch = p & 7;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (row0 + r < end) {
      const float4 a = *reinterpret_cast<const float4 *>(src + (size_t)(row0 + r) * ld + col + ch * 8);
      const float4 b = *reinterpret_cast<const float4 *>(src + (size_t)(row0 + r) * ld + col + ch * 8 + 4);
      v = make_uint4(pack2(a.x, a.y), pack2(a.z, a.w), pack2(b.x, b.y), pack2(b.z, b.w));
    }
    *reinterpret_cast<uint4 *>(tile + sw_off(r, ch)) = v;
  }
}

// per-lane ldmatrix offsets inside a swizzled 32-row tile (pattern of attention_pk.cu):
//   a[i] : A operand (16 rows of this warp x k-step i of 16 columns)
//   b[i] : B operand from ROWS of the tile (x . row^T products), k-step i, two n8 blocks of rows; +2048 for rows 16..31
//   t[i] : B operand from the tile TRANSPOSED (P . tile products), column block i of 16; +2048 for rows 16..31
struct Offs { uint32_t a[4], b[4], t[4]; };
__device__ __forceinline__ Offs make_offs(int warp, int lane) {
  Offs o;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    o.a[i] = sw_off(warp * 16 + (lane & 15), i * 2 + (lane >> 4));
    o.b[i] = sw_off((lane & 7) + ((lane >> 4) << 3), i * 2 + ((lane >> 3) & 1));
    o.t[i] = sw_off((lane & 7) + (((lane >> 3) & 1) << 3), i * 2 + (lane >> 4));
  }
  return o;
}
// s[16 x 32] = A[16 x 64] . tile[32 x 64]^T
__device__ __forceinline__ void mm_rows(float (&s)[4][4], const uint32_t (&af)[4][4], uint32_t tile, const Offs &o) {
#pragma unroll
  for (int nb = 0; nb < 4; ++nb) { s[nb][0] = s[nb][1] = s[nb][2] = s[nb][3] = 0.f; }
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
    for (int nb2 = 0; nb2 < 2; ++nb2) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4(tile + nb2 * 2048 + o.b[ks], b0, b1, b2, b3);
      mma16816(s[nb2 * 2], af[ks], b0, b1);
      mma16816(s[nb2 * 2 + 1], af[ks], b2, b3);
    }
  }
}
// acc[16 x 64] += P[16 x 32] . tile[32 x 64]   (P as two k16 A fragments)
__device__ __forceinline__ void mm_tr(float (&acc)[8][4], const uint32_t (&pf)[2][4], uint32_t tile, const Offs &o) {
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
    for (int db = 0; db < 4; ++db) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4_t(tile + ks * 2048 + o.t[db], b0, b1, b2, b3);
      mma16816(acc[db * 2], pf[ks], b0, b1);
      mma16816(acc[db * 2 + 1], pf[ks], b2, b3);
    }
  }
}
__device__ __forceinline__ void load_a(uint32_t (&af)[4][4], uint32_t tile, const Offs &o) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) ldsm_x4(tile + o.a[ks], af[ks][0], af[ks][1], af[ks][2], af[ks][3]);
}
// accumulator layout of a 16 x 32 product -> two k16 A fragments
__device__ __forceinline__ void to_a(uint32_t (&pf)[2][4], const float (&p)[4][4]) {
#pragma unroll
  for (int nb = 0; nb < 4; ++nb) {
    pf[nb >> 1][(nb & 1) * 2 + 0] = pack2(p[nb][0], p[nb][1]);
    pf[nb >> 1][(nb & 1) * 2 + 1] = pack2(p[nb][2], p[nb][3]);
  }
}

// image b and block index of a unit: blockIdx.x = b * blocks + block
struct Unit { int lo, hi, r0; };
__device__ __forceinline__ Unit unit_of(const int32_t *__restrict__ cu, int blocks) {
  const int b = blockIdx.x / blocks, blk = blockIdx.x % blocks;
  Unit u;
  u.lo = cu[b]; u.hi = cu[b + 1]; u.r0 = u.lo + blk * AT_BLK;
  return u;
}

__global__ void __launch_bounds__(AT_THREADS)
attn_train_fwd_kernel(const bf16 *__restrict__ qkv, const int32_t *__restrict__ cu, int blocks, int D,
                      bf16 *__restrict__ ctx, float *__restrict__ lse) {
  __shared__ __align__(1024) uint8_t sm[3 * AT_TILE];
  const Unit u = unit_of(cu, blocks);
  if (u.r0 >= u.hi) return;
  const int head = blockIdx.y, H = D / AT_DH;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const size_t ld = (size_t)3 * D;
  const uint32_t aQ = smem_u32(sm), aK = aQ + AT_TILE, aV = aK + AT_TILE;
  const Offs of = make_offs(warp, lane);
  const bool warp_on = u.r0 + warp * 16 < u.hi;
  load_tile(sm, qkv, ld, head * AT_DH, u.r0, u.hi);
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  uint32_t qf[4][4];
  const int nch = (u.hi - u.lo + AT_BLK - 1) / AT_BLK;
  for (int c = 0; c < nch; ++c) {
    const int kbase = u.lo + c * AT_BLK;
    __syncthreads();                                   // previous chunk consumed
    load_tile(sm + AT_TILE, qkv, ld, D + head * AT_DH, kbase, u.hi);
    load_tile(sm + 2 * AT_TILE, qkv, ld, 2 * D + head * AT_DH, kbase, u.hi);
    __syncthreads();
    if (!warp_on) continue;
    if (c == 0) load_a(qf, aQ, of);
    float s[4][4];
    mm_rows(s, qf, aK, of);
    if (kbase + AT_BLK > u.hi) {
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) {
        const int key = kbase + nb * 8 + 2 * t;
        if (key >= u.hi) { s[nb][0] = -INFINITY; s[nb][2] = -INFINITY; }
        if (key + 1 >= u.hi) { s[nb][1] = -INFINITY; s[nb][3] = -INFINITY; }
      }
    }
    float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      cm0 = fmaxf(cm0, fmaxf(s[nb][0], s[nb][1]));
      cm1 = fmaxf(cm1, fmaxf(s[nb][2], s[nb][3]));
    }
    cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1)); cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
    cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1)); cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
    const float nm0 = fmaxf(m0, cm0), nm1 = fmaxf(m1, cm1);      // finite: the chunk's first key is real
    const float corr0 = ex2f((m0 - nm0) * kSl2), corr1 = ex2f((m1 - nm1) * kSl2);
    m0 = nm0; m1 = nm1;
    const float ms0 = m0 * kSl2, ms1 = m1 * kSl2;
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      s[nb][0] = ex2f(fmaf(s[nb][0], kSl2, -ms0)); s[nb][1] = ex2f(fmaf(s[nb][1], kSl2, -ms0));
      s[nb][2] = ex2f(fmaf(s[nb][2], kSl2, -ms1)); s[nb][3] = ex2f(fmaf(s[nb][3], kSl2, -ms1));
      rs0 += s[nb][0] + s[nb][1]; rs1 += s[nb][2] + s[nb][3];
    }
    uint32_t pf[2][4];
    to_a(pf, s);
    l0 = l0 * corr0 + rs0; l1 = l1 * corr1 + rs1;
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] *= corr0; o[i][1] *= corr0; o[i][2] *= corr1; o[i][3] *= corr1; }
    mm_tr(o, pf, aV, of);
  }
  if (!warp_on) return;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
  const int ra = u.r0 + warp * 16 + g, rb = ra + 8;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int col = head * AT_DH + nb * 8 + 2 * t;
    if (ra < u.hi) *reinterpret_cast<uint32_t *>(ctx + (size_t)ra * D + col) = pack2(o[nb][0] * inv0, o[nb][1] * inv0);
    if (rb < u.hi) *reinterpret_cast<uint32_t *>(ctx + (size_t)rb * D + col) = pack2(o[nb][2] * inv1, o[nb][3] * inv1);
  }
  if (t == 0) {                                        // natural-log units: lse = max(s) / 8 + ln(sum exp(s / 8 - max / 8))
    if (ra < u.hi) lse[(size_t)ra * H + head] = m0 * 0.125f + logf(l0);
    if (rb < u.hi) lse[(size_t)rb * H + head] = m1 * 0.125f + logf(l1);
  }
}

// dq pass; also writes Di [rows, H] for the dkv pass
__global__ void __launch_bounds__(AT_THREADS)
attn_train_dq_kernel(const bf16 *__restrict__ qkv, const bf16 *__restrict__ ctx, const float *__restrict__ lse,
                     const float *__restrict__ dctx, const int32_t *__restrict__ cu, int blocks, int D,
                     float *__restrict__ di, float *__restrict__ dqkv) {
  __shared__ __align__(1024) uint8_t sm[4 * AT_TILE];
  __shared__ float s_lse2[AT_BLK], s_di[AT_BLK];
  const Unit u = unit_of(cu, blocks);
  if (u.r0 >= u.hi) return;
  const int head = blockIdx.y, H = D / AT_DH;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const size_t ld = (size_t)3 * D;
  const uint32_t aQ = smem_u32(sm), aO = aQ + AT_TILE, aK = aO + AT_TILE, aV = aK + AT_TILE;
  const Offs of = make_offs(warp, lane);
  const bool warp_on = u.r0 + warp * 16 < u.hi;
  load_tile(sm, qkv, ld, head * AT_DH, u.r0, u.hi);
  load_tile(sm + AT_TILE, dctx, (size_t)D, head * AT_DH, u.r0, u.hi);
  {
    // Di = rowsum(bf16(dO) o O) in fp32: two threads per row, 32 columns each
    const int r = tid >> 1, half = tid & 1, row = u.r0 + r;
    float acc = 0.f;
    if (row < u.hi) {
      const float *dor = dctx + (size_t)row * D + head * AT_DH + half * 32;
      const bf16 *orow = ctx + (size_t)row * D + head * AT_DH + half * 32;
#pragma unroll 8
      for (int j = 0; j < 32; ++j) acc = fmaf(__bfloat162float(__float2bfloat16_rn(dor[j])), __bfloat162float(orow[j]), acc);
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    if (half == 0) {
      s_di[r] = acc;
      s_lse2[r] = row < u.hi ? lse[(size_t)row * H + head] * kLog2e : 0.f;
      if (row < u.hi) di[(size_t)row * H + head] = acc;
    }
  }
  const int la = warp * 16 + g, lb = la + 8;
  float dq[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) { dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f; }
  uint32_t qf[4][4], of4[4][4];
  float lse2a = 0.f, lse2b = 0.f, dia = 0.f, dib = 0.f;
  const int nch = (u.hi - u.lo + AT_BLK - 1) / AT_BLK;
  for (int c = 0; c < nch; ++c) {
    const int kbase = u.lo + c * AT_BLK;
    __syncthreads();
    load_tile(sm + 2 * AT_TILE, qkv, ld, D + head * AT_DH, kbase, u.hi);
    load_tile(sm + 3 * AT_TILE, qkv, ld, 2 * D + head * AT_DH, kbase, u.hi);
    __syncthreads();
    if (!warp_on) continue;
    if (c == 0) {
      load_a(qf, aQ, of); load_a(of4, aO, of);
      lse2a = s_lse2[la]; lse2b = s_lse2[lb]; dia = s_di[la]; dib = s_di[lb];
    }
    float s[4][4], dp[4][4];
    mm_rows(s, qf, aK, of);
    mm_rows(dp, of4, aV, of);
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      const int key = kbase + nb * 8 + 2 * t;
      const bool v0 = key < u.hi, v1 = key + 1 < u.hi;
      const float p0 = v0 ? ex2f(fmaf(s[nb][0], kSl2, -lse2a)) : 0.f, p1 = v1 ? ex2f(fmaf(s[nb][1], kSl2, -lse2a)) : 0.f;
      const float p2 = v0 ? ex2f(fmaf(s[nb][2], kSl2, -lse2b)) : 0.f, p3 = v1 ? ex2f(fmaf(s[nb][3], kSl2, -lse2b)) : 0.f;
      s[nb][0] = p0 * (dp[nb][0] - dia); s[nb][1] = p1 * (dp[nb][1] - dia);
      s[nb][2] = p2 * (dp[nb][2] - dib); s[nb][3] = p3 * (dp[nb][3] - dib);
    }
    uint32_t dsf[2][4];
    to_a(dsf, s);
    mm_tr(dq, dsf, aK, of);
  }
  if (!warp_on) return;
  const int ra = u.r0 + la, rb = u.r0 + lb;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int col = head * AT_DH + nb * 8 + 2 * t;
    if (ra < u.hi) *reinterpret_cast<float2 *>(dqkv + (size_t)ra * ld + col) = make_float2(dq[nb][0] * 0.125f, dq[nb][1] * 0.125f);
    if (rb < u.hi) *reinterpret_cast<float2 *>(dqkv + (size_t)rb * ld + col) = make_float2(dq[nb][2] * 0.125f, dq[nb][3] * 0.125f);
  }
}

// dkv pass: the unit's 32 keys against the image's queries in 32-row chunks
__global__ void __launch_bounds__(AT_THREADS)
attn_train_dkv_kernel(const bf16 *__restrict__ qkv, const float *__restrict__ lse, const float *__restrict__ di,
                      const float *__restrict__ dctx, const int32_t *__restrict__ cu, int blocks, int D,
                      float *__restrict__ dqkv) {
  __shared__ __align__(1024) uint8_t sm[4 * AT_TILE];
  __shared__ float s_lse2[AT_BLK], s_di[AT_BLK];
  const Unit u = unit_of(cu, blocks);                  // r0: the unit's first key
  if (u.r0 >= u.hi) return;
  const int head = blockIdx.y, H = D / AT_DH;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const size_t ld = (size_t)3 * D;
  const uint32_t aK = smem_u32(sm), aV = aK + AT_TILE, aQ = aV + AT_TILE, aO = aQ + AT_TILE;
  const Offs of = make_offs(warp, lane);
  const bool warp_on = u.r0 + warp * 16 < u.hi;
  load_tile(sm, qkv, ld, D + head * AT_DH, u.r0, u.hi);
  load_tile(sm + AT_TILE, qkv, ld, 2 * D + head * AT_DH, u.r0, u.hi);
  float dk[8][4], dv[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
    dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
  }
  uint32_t kf[4][4], vf[4][4];
  const int nch = (u.hi - u.lo + AT_BLK - 1) / AT_BLK;
  for (int c = 0; c < nch; ++c) {
    const int qbase = u.lo + c * AT_BLK;
    __syncthreads();
    load_tile(sm + 2 * AT_TILE, qkv, ld, head * AT_DH, qbase, u.hi);
    load_tile(sm + 3 * AT_TILE, dctx, (size_t)D, head * AT_DH, qbase, u.hi);
    if (tid < AT_BLK) {
      const int row = qbase + tid;
      s_lse2[tid] = row < u.hi ? lse[(size_t)row * H + head] * kLog2e : 0.f;
      s_di[tid] = row < u.hi ? di[(size_t)row * H + head] : 0.f;
    }
    __syncthreads();
    if (!warp_on) continue;
    if (c == 0) { load_a(kf, aK, of); load_a(vf, aV, of); }
    float s[4][4], dp[4][4];
    mm_rows(s, kf, aQ, of);                            // S^T: rows = keys, columns = the chunk's queries
    mm_rows(dp, vf, aO, of);                           // dP^T
    float p[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int qc = nb * 8 + 2 * t + j;
        const bool valid = qbase + qc < u.hi;
        const float l2 = s_lse2[qc], dd = s_di[qc];
        const float pa = valid ? ex2f(fmaf(s[nb][j], kSl2, -l2)) : 0.f;
        const float pb = valid ? ex2f(fmaf(s[nb][j + 2], kSl2, -l2)) : 0.f;
        p[nb][j] = pa; p[nb][j + 2] = pb;
        s[nb][j] = pa * (dp[nb][j] - dd); s[nb][j + 2] = pb * (dp[nb][j + 2] - dd);
      }
    }
    uint32_t pf[2][4], dsf[2][4];
    to_a(pf, p);
    to_a(dsf, s);
    mm_tr(dv, pf, aO, of);
    mm_tr(dk, dsf, aQ, of);
  }
  if (!warp_on) return;
  const int ra = u.r0 + warp * 16 + g, rb = ra + 8;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int col = head * AT_DH + nb * 8 + 2 * t;
    if (ra < u.hi) {
      *reinterpret_cast<float2 *>(dqkv + (size_t)ra * ld + D + col) = make_float2(dk[nb][0] * 0.125f, dk[nb][1] * 0.125f);
      *reinterpret_cast<float2 *>(dqkv + (size_t)ra * ld + 2 * D + col) = make_float2(dv[nb][0], dv[nb][1]);
    }
    if (rb < u.hi) {
      *reinterpret_cast<float2 *>(dqkv + (size_t)rb * ld + D + col) = make_float2(dk[nb][2] * 0.125f, dk[nb][3] * 0.125f);
      *reinterpret_cast<float2 *>(dqkv + (size_t)rb * ld + 2 * D + col) = make_float2(dv[nb][2], dv[nb][3]);
    }
  }
}

int blocks_per_image(const PsvHandle *h) { return (h->N + AT_BLK - 1) / AT_BLK; }

}  // namespace

cudaError_t launch_attention_train_fwd(PsvHandle *h, const bf16 *qkv, const int32_t *cu_seqlens, int batch, bf16 *ctx,
                                       float *lse, cudaStream_t s) {
  if (h->D % AT_DH != 0 || h->D / h->H != AT_DH) return cudaErrorNotSupported;
  LaunchScope scope(h, KK_ATTENTION, s);
  const int blocks = blocks_per_image(h);
  attn_train_fwd_kernel<<<dim3(batch * blocks, h->H), AT_THREADS, 0, s>>>(qkv, cu_seqlens, blocks, h->D, ctx, lse);
  return cudaGetLastError();
}

cudaError_t launch_attention_train_bwd(PsvHandle *h, const bf16 *qkv, const bf16 *ctx, const float *lse,
                                       const float *dctx, const int32_t *cu_seqlens, int batch, float *di, float *dqkv,
                                       cudaStream_t s) {
  if (h->D % AT_DH != 0 || h->D / h->H != AT_DH) return cudaErrorNotSupported;
  const int blocks = blocks_per_image(h);
  {
    LaunchScope scope(h, KK_TRAIN, s);
    attn_train_dq_kernel<<<dim3(batch * blocks, h->H), AT_THREADS, 0, s>>>(qkv, ctx, lse, dctx, cu_seqlens, blocks, h->D,
                                                                           di, dqkv);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  LaunchScope scope(h, KK_TRAIN, s);
  attn_train_dkv_kernel<<<dim3(batch * blocks, h->H), AT_THREADS, 0, s>>>(qkv, lse, di, dctx, cu_seqlens, blocks, h->D,
                                                                          dqkv);
  return cudaGetLastError();
}

}  // namespace psv
