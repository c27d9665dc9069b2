// K6 (bf16 mode), short / mixed sequences: varlen attention over 32-QUERY BLOCKS of one image
// (reference model_utils.py:91 -> HF:171-196: softmax(q k^T / 8) v among the active tokens of one image).
//
// Why a third kernel: with the natural skip profile most images keep 1..60 tokens and a few keep ~190.  One CTA per
// (image, head) (attention_mma.cu) then costs ~14 us per layer even when every image has ONE token -- 3072 CTAs whose
// life is a chain of dependent latencies (cu_seqlens -> ~50 cp.async per thread -> ldmatrix -> store) at 4 CTAs per
// SM -- and the few long images leave a tail (layers with 8 k rows but one 190-token image took 40 us).  Here:
//   * the work unit is (image, block of 32 queries, head); the compaction kernel publishes one descriptor per
//     (image, block) -- {first query row, first key row, one-past-last key row} -- in a flat table (order arbitrary,
//     appended with one atomicAdd per image), so the grid holds exactly the blocks that exist and a 190-token image is
//     six independent units instead of one long CTA;
//   * Q (32 x 64) and K / V (32-key chunks, aligned to the image's first row) arrive by TMA (128B swizzle = the
//     ldmatrix-conflict-free layout) in a small ring: a handful of instructions instead of ~50 cp.async per thread;
//   * 64 threads, 2 warps x 16 queries, mma.sync m16n8k16 bf16 with fp32 online softmax (exp2, 1/8 folded in);
//   * <= 28 KB of shared memory and <= 128 registers: 7-8 resident CTAs per SM hide each other's latency.
// Every row's arithmetic depends on its own image only (chunks are aligned to the image, not to the packed buffer), so
// results do not depend on what else is in the batch: a shard of 128 images gives the bits of the 256-image batch.
// (A first version packed 32 CONSECUTIVE PACKED rows per unit across image boundaries with a block-diagonal mask --
// 2-4x fewer CTAs for the short layers and ~3 us faster there, but the chunk alignment of an image then depends on
// its neighbours and the last bits of the output with it; dropped for that reason.)
// Tensor-path note: like attention_mma.cu this is the warp-level HMMA path on purpose -- a unit is 32 queries x
// <= 197 keys, far below one 128-row tcgen05 tile; the tcgen05/TMEM kernel (attention_tc.cu) serves the long sequences.
#include "tc_common.cuh"

namespace psv {
namespace {

using namespace tc;

constexpr int PK_Q = 32;                 // queries per CTA
constexpr int PK_KC = 32;                // keys per chunk
constexpr int PK_THREADS = 64;
constexpr int DH = 64;
constexpr int Q_BYTES = PK_Q * DH * 2;   // 4 KB
constexpr int KV_BYTES = PK_KC * DH * 2; // 4 KB each for K and V

constexpr int NST = 2;                   // K / V ring stages
constexpr int PK_SMEM = Q_BYTES + NST * 2 * KV_BYTES + 1024 /* alignment slack */;

__device__ __forceinline__ uint32_t sw_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}

// units[u] = {first query row of the block, first key row of the image, one past its last key row, -}; *count_dev units
__global__ void __launch_bounds__(PK_THREADS, 8)
attention_pk_kernel(const __grid_constant__ CUtensorMap map_qkv, bf16 *__restrict__ ctx,
                    const int4 *__restrict__ units, const int32_t *__restrict__ count_dev, int D) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bars[NST + 1];               // [0] Q, [1 + s] K/V stage s
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t aQ = smem_u32(smem), aKV = aQ + Q_BYTES;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int head = blockIdx.y;
  const int g = lane >> 2, t = lane & 3;
  const float sl2 = 0.125f * 1.4426950408889634f;  // softmax scale * log2(e)

  pdl_wait();
  const int n_units = *count_dev;
  int4 U = make_int4(0, 0, 0, 0);
  if ((int)blockIdx.x < n_units) U = units[blockIdx.x];        // independent of the count load: one latency, not two
  if (tid == 0) {
    for (int i = 0; i < NST + 1; ++i) mbar_init(&bars[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_qkv) : "memory");
  }
  // per-lane ldmatrix offsets inside the swizzled tiles (row offsets added later are multiples of 16 rows)
  uint32_t offQ[4], offK[4], offV[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    offQ[i] = sw_off(warp * 16 + (lane & 15), i * 2 + (lane >> 4));
    offK[i] = sw_off((lane & 7) + ((lane >> 4) << 3), i * 2 + ((lane >> 3) & 1));
    offV[i] = sw_off((lane & 7) + (((lane >> 3) & 1) << 3), i * 2 + (lane >> 4));
  }
  uint32_t qph = 0, sph = 0;                       // barrier phases (bit s of sph = stage s)

  for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
    if (unit != (int)blockIdx.x) U = units[unit];
    const int r0 = U.x, lo = U.y, hi = U.z;        // queries r0 .. min(r0 + 32, hi); keys lo .. hi
    const int nch = (hi - lo + PK_KC - 1) / PK_KC;
    const int ra = r0 + warp * 16 + g, rb = ra + 8;
    const bool warp_on = r0 + warp * 16 < hi;      // this warp holds at least one real query
    __syncthreads();                               // barriers initialised / previous unit done with shared memory
    if (tid == 0) {
      mbar_arrive_expect_tx(&bars[0], Q_BYTES);
      tma_load_2d(smem, &map_qkv, &bars[0], head * DH, r0);
      for (int c = 0; c < NST && c < nch; ++c) {
        mbar_arrive_expect_tx(&bars[1 + c], 2 * KV_BYTES);
        tma_load_2d(smem + Q_BYTES + c * 2 * KV_BYTES, &map_qkv, &bars[1 + c], D + head * DH, lo + c * PK_KC);
        tma_load_2d(smem + Q_BYTES + c * 2 * KV_BYTES + KV_BYTES, &map_qkv, &bars[1 + c], 2 * D + head * DH, lo + c * PK_KC);
      }
    }
    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    mbar_wait(&bars[0], qph); qph ^= 1;
    uint32_t qf[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) ldmatrix_x4(aQ + offQ[ks], qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);

    for (int c = 0; c < nch; ++c) {
      const int st = c % NST;
      const uint32_t aK = aKV + st * 2 * KV_BYTES, aV = aK + KV_BYTES;
      mbar_wait(&bars[1 + st], (sph >> st) & 1u); sph ^= 1u << st;
      const int kbase = lo + c * PK_KC;
      if (warp_on) {
        float s[4][4];
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) { s[nb][0] = s[nb][1] = s[nb][2] = s[nb][3] = 0.f; }
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
          for (int nb2 = 0; nb2 < 2; ++nb2) {
            uint32_t b0, b1, b2, b3;
            ldmatrix_x4(aK + nb2 * 2048 + offK[ks], b0, b1, b2, b3);
            mma_bf16(s[nb2 * 2], qf[ks], b0, b1);
            mma_bf16(s[nb2 * 2 + 1], qf[ks], b2, b3);
          }
        }
        // keys past the image's last row (only the last chunk holds any) do not count
        if (kbase + PK_KC > hi) {
#pragma unroll
          for (int nb = 0; nb < 4; ++nb) {
            const int key = kbase + nb * 8 + 2 * t;
            if (key >= hi) { s[nb][0] = -INFINITY; s[nb][2] = -INFINITY; }
            if (key + 1 >= hi) { s[nb][1] = -INFINITY; s[nb][3] = -INFINITY; }
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
        const float nm0 = fmaxf(m0, cm0), nm1 = fmaxf(m1, cm1);    // finite: the chunk's first key is real
        const float corr0 = ex2_approx((m0 - nm0) * sl2), corr1 = ex2_approx((m1 - nm1) * sl2);
        m0 = nm0; m1 = nm1;
        const float ms0 = m0 * sl2, ms1 = m1 * sl2;
        float rs0 = 0.f, rs1 = 0.f;
        uint32_t pf[2][4];
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
          const float p0 = ex2_approx(fmaf(s[nb][0], sl2, -ms0)), p1 = ex2_approx(fmaf(s[nb][1], sl2, -ms0));
          const float p2 = ex2_approx(fmaf(s[nb][2], sl2, -ms1)), p3 = ex2_approx(fmaf(s[nb][3], sl2, -ms1));
          rs0 += p0 + p1; rs1 += p2 + p3;
          pf[nb >> 1][(nb & 1) * 2 + 0] = pack_bf16(p0, p1);
          pf[nb >> 1][(nb & 1) * 2 + 1] = pack_bf16(p2, p3);
        }
        l0 = l0 * corr0 + rs0; l1 = l1 * corr1 + rs1;
        if (c > 0 && __any_sync(0xffffffffu, corr0 != 1.0f || corr1 != 1.0f)) {
#pragma unroll
          for (int i = 0; i < 8; ++i) { o[i][0] *= corr0; o[i][1] *= corr0; o[i][2] *= corr1; o[i][3] *= corr1; }
        }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
          for (int db = 0; db < 4; ++db) {
            uint32_t b0, b1, b2, b3;
            ldmatrix_x4_trans(aV + ks * 2048 + offV[db], b0, b1, b2, b3);
            mma_bf16(o[db * 2], pf[ks], b0, b1);
            mma_bf16(o[db * 2 + 1], pf[ks], b2, b3);
          }
        }
      }
      if (c + NST < nch) {                         // CTA-uniform: recycle the stage for chunk c + NST
        __syncthreads();
        if (tid == 0) {
          mbar_arrive_expect_tx(&bars[1 + st], 2 * KV_BYTES);
          tma_load_2d(smem + Q_BYTES + st * 2 * KV_BYTES, &map_qkv, &bars[1 + st], D + head * DH, lo + (c + NST) * PK_KC);
          tma_load_2d(smem + Q_BYTES + st * 2 * KV_BYTES + KV_BYTES, &map_qkv, &bars[1 + st], 2 * D + head * DH,
                      lo + (c + NST) * PK_KC);
        }
      }
    }
    if (warp_on) {
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
        const int col = head * DH + nb * 8 + 2 * t;
        if (ra < hi) *reinterpret_cast<uint32_t *>(ctx + (size_t)ra * D + col) = pack_bf16(o[nb][0] * inv0, o[nb][1] * inv0);
        if (rb < hi) *reinterpret_cast<uint32_t *>(ctx + (size_t)rb * D + col) = pack_bf16(o[nb][2] * inv1, o[nb][3] * inv1);
      }
    }
  }
}

// unit table from cu_seqlens (psv_attention hook and the dense pass; the skip path gets it from the compaction kernel):
// one CTA, image after image (not a performance path)
__global__ void units_from_cu_kernel(const int32_t *__restrict__ cu, int batch, int4 *__restrict__ units,
                                     int32_t *__restrict__ count) {
  __shared__ int base;
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  for (int b0 = 0; b0 < batch; b0 += blockDim.x) {
    const int b = b0 + threadIdx.x;
    int lo = 0, hi = 0, nu = 0;
    if (b < batch) { lo = cu[b]; hi = cu[b + 1]; nu = (hi - lo + PK_Q - 1) / PK_Q; }
    // inclusive scan of nu over the block (serial over warps is fine here)
    int incl = nu;
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if ((threadIdx.x & 31) >= o) incl += v; }
    __shared__ int wsum[32];
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    int before = base;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += wsum[w];
    const int first = before + incl - nu;
    for (int q = 0; q < nu; ++q) units[first + q] = make_int4(lo + q * PK_Q, lo, hi, 0);
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) base = before + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = base;
}

}  // namespace

cudaError_t configure_attention_pk() {
  return cudaFuncSetAttribute(attention_pk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PK_SMEM);
}

// have_units: h->attn_units / h->attn_unit_count already describe cu_seqlens (the compaction kernel wrote them);
// otherwise they are built here from cu_seqlens (one more small launch).  rows_hint: expected T (-1 unknown); it only
// sizes the grid -- CTAs loop over the units, so any count is handled.
cudaError_t launch_attention_pk(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                int64_t qkv_rows, bool have_units, int rows_hint, cudaStream_t s) {
  CUtensorMap m;
  cudaError_t e = get_tmap_2d(h->tmaps, qkv, (uint64_t)qkv_rows, (uint64_t)3 * h->D, PK_KC, 64, 2, 128, &m);
  if (e != cudaSuccess) return e;
  if (!have_units) {
    units_from_cu_kernel<<<1, 256, 0, s>>>(cu_seqlens, batch, (int4 *)h->attn_units, h->attn_unit_count);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  LaunchScope scope(h, KK_ATTENTION, s);
  const int max_units = batch * ((h->N + PK_Q - 1) / PK_Q);
  int units = rows_hint > 0 ? rows_hint / PK_Q + batch : max_units;     // sum of ceil(n / 32) <= T / 32 + batch
  if (units > max_units) units = max_units;
  dim3 grid(units, h->H);
  return launch_pdl(attention_pk_kernel, grid, dim3(PK_THREADS), (size_t)PK_SMEM, s, m, (bf16 *)ctx,
                    (const int4 *)h->attn_units, (const int32_t *)h->attn_unit_count, h->D);
}

}  // namespace psv
