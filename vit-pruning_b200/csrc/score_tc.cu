// K1/K2 (bf16 mode): the compressor MLP -> sigmoid -> threshold -> skip mask on the tcgen05 tensor
// cores at fp32-class accuracy (reference model_utils.py:62-68).
//
// score[r] = sigmoid(w2 . relu(W1_cls . cls_b + b1 + W1_tok . x_r) + b2) for every row r of the fp32
// residual stream [B*N, D] (CLS rows are computed too and ignored; it keeps the tiling flat).
//   * cls_half_kernel (grid B/4): hc[b] = W1[:, :D] . cls_b + b1 in fp32.  (Folding this GEMV into the score kernel
//     -- two extra warps computing hc for the images of each tile -- was tried and DOUBLED the kernel: every tile
//     then pulls the 196 KB of W1[:, :D] through L2 again, as much as the tile's own share of the stream.)
//   * score_tc_kernel (persistent, 128-row tiles): the token half  X[128 x D] . W1_tok^T[D x 64]  runs
//     as a SPLIT-bf16 product -- x = x_hi + x_lo, w = w_hi + w_lo (bf16 each) and
//     x.w ~= x_hi.w_hi + x_hi.w_lo + x_lo.w_hi into fp32 TMEM accumulators -- so the result carries ~16 mantissa bits
//     (error ~1e-6 on a score) while the kernel stays HBM-bound: it reads the fp32 stream once (B*N*D*4 bytes) and
//     writes B*N mask bytes.
//     Operand path: the fp32 tiles arrive by TMA (128B-swizzled 32-column boxes), converter warps split them into
//     (hi, lo) bf16 pairs and store those straight INTO TENSOR MEMORY (tcgen05.st); the MMAs take A from TMEM
//     (tcgen05.mma TS form) and only the small weight slabs from shared memory.  The first version wrote the hi / lo
//     planes to shared memory as UMMA operand tiles: per 64-column k-block that is 29 KB TMA write + 29 KB converter read
//     + 29 KB converter write + 48 KB of MMA operand reads (+ 40 KB for the weights) = 175 KB through a 128 B/clk port,
//     0.71 us against the 0.76 us the block takes to arrive from HBM -- the kernel ran at 4.0 TB/s because shared
//     memory, not HBM, was saturated.  With A in TMEM the port carries ~100 KB per block.
//     Three N = 64 MMAs per 16-wide k-step into the SAME 64 accumulator columns: x_hi . w_hi, x_hi . w_lo, x_lo . w_hi
//     (round 2; before, x_hi . [w_hi ; w_lo] went to 128 columns and the epilogue added the halves: two TMEM loads per
//     chunk instead of one, 3-18 us per forward slower; the bits are the same).
//     Warp roles: 0 TMA producer (fp32 tiles), 14 TMA producer (W_hi/W_lo k-slabs), 1 MMA issuer, 2-5 epilogue
//     (TMEM -> ReLU, dot w2, sigmoid, >= mt, mask/scores stores, active counts by warp ballot: each tile STORES
//     the counts of its two images, so nothing has to be zeroed between layers and no atomics are needed),
//     6-13 converters (thread <-> tile row = TMEM lane; two warps per lane quadrant, one per 32-column half).
#include <cstdlib>

#include "tc_common.cuh"

namespace psv {
namespace {

using namespace tc;

constexpr int S_ROWS = 128;
constexpr int S_KB = 64;                 // k elements per block
constexpr int S_CH = 64;                 // compressor hidden width
constexpr int NS_F = 5, NS_W = 3, NS_A = 2;
constexpr int F_HALF = S_ROWS * 32 * 4;        // 16 KB: 128 rows x 32 fp32 (one 128-byte swizzle row per tile row)
constexpr int F_BYTES = 2 * F_HALF;            // 32 KB fp32 staging tile = two 32-column halves
constexpr int W_BYTES = S_CH * S_KB * 2;       // 8 KB per bf16 plane
constexpr int S_THREADS = 480;                // stream TMA, MMA, 4 epilogue, 8 converter warps, weight TMA
constexpr int S_ACC_COLS = 2 * S_CH;           // accumulator stage (the sums use its first 64 columns)
constexpr int S_A_COL = 2 * S_ACC_COLS;        // TMEM columns 256..: A stages, each [hi: 32 cols | lo: 32 cols]
constexpr int S_TMEM_COLS = 512;               // 256 accumulator + 128 operand columns, rounded up to a power of two
constexpr int OFF_F = 0;
constexpr int OFF_W = OFF_F + NS_F * F_BYTES;              // hi plane then lo plane per stage (= one 128-row B operand)
constexpr int OFF_BAR = OFF_W + NS_W * 2 * W_BYTES;
constexpr int S_SMEM = OFF_BAR + 1024 + 1024;

// hc[b][j] = b1[j] + W1[j, 0:D] . cls_b.  CLS_IMGS images per CTA so each W1 row that is
// read serves several images; 16 warps x 4 hidden units, all weight loads of a warp issued back to back.
constexpr int CLS_IMGS = 4;
template <int D>
__global__ void __launch_bounds__(512)
cls_half_kernel(const float *__restrict__ hidden, const float *__restrict__ comp, int N, int batch,
                float *__restrict__ hc) {
  __shared__ __align__(16) float cls[CLS_IMGS][D];
  const int b0 = blockIdx.x * CLS_IMGS, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nimg = min(CLS_IMGS, batch - b0);
  pdl_wait();
  pdl_trigger_now();        // after the wait: once the score kernel starts, everything older than this grid is complete
  for (int e = threadIdx.x; e < nimg * (D / 4); e += 512) {
    const int i = e / (D / 4), q = e % (D / 4);
    *reinterpret_cast<float4 *>(&cls[i][q * 4]) =
        *reinterpret_cast<const float4 *>(hidden + (size_t)(b0 + i) * N * D + q * 4);
  }
  const float *b1 = comp + (size_t)S_CH * 2 * D;
  constexpr int V = D / 128;
  float4 w[4][V];
#pragma unroll
  for (int jj = 0; jj < 4; ++jj)
#pragma unroll
    for (int v = 0; v < V; ++v)
      w[jj][v] = *reinterpret_cast<const float4 *>(comp + (size_t)(warp * 4 + jj) * 2 * D + (v * 32 + lane) * 4);
  __syncthreads();
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    float acc[CLS_IMGS];
#pragma unroll
    for (int i = 0; i < CLS_IMGS; ++i) {
      acc[i] = 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float4 x = *reinterpret_cast<const float4 *>(&cls[i][(v * 32 + lane) * 4]);
        acc[i] = fmaf(w[jj][v].x, x.x, acc[i]); acc[i] = fmaf(w[jj][v].y, x.y, acc[i]);
        acc[i] = fmaf(w[jj][v].z, x.z, acc[i]); acc[i] = fmaf(w[jj][v].w, x.w, acc[i]);
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
    }
    if (lane < nimg) {
      float a = acc[0];
#pragma unroll
      for (int i = 1; i < CLS_IMGS; ++i) a = (lane == i) ? acc[i] : a;
      hc[(size_t)(b0 + lane) * S_CH + warp * 4 + jj] = a + b1[warp * 4 + jj];
    }
  }
}

__device__ __forceinline__ uint32_t pack2(bf16 a, bf16 b) {
  __nv_bfloat162 v(a, b);
  return *reinterpret_cast<uint32_t *>(&v);
}

__global__ void __launch_bounds__(S_THREADS, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_whi,
                const __grid_constant__ CUtensorMap map_wlo, const float *__restrict__ comp,
                const float *__restrict__ hc, float mt, const uint8_t *__restrict__ forced, int rows_total, int N,
                int D, uint8_t *__restrict__ mask, float *__restrict__ scores, int2 *__restrict__ n_tile,
                uint8_t *__restrict__ mask_out, float *__restrict__ scores_out, float *__restrict__ preact_out,
                int tile_rows, int debug, int wait_late, int32_t *__restrict__ unit_count) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
  uint64_t *full_f = bars, *empty_f = full_f + NS_F;
  uint64_t *full_w = empty_f + NS_F, *empty_w = full_w + NS_W;
  uint64_t *full_a = empty_w + NS_W, *empty_a = full_a + NS_A;
  uint64_t *tfull = empty_a + NS_A, *tempty = tfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + 2);
  float *w2s = reinterpret_cast<float *>(tmem_slot + 4);        // [64] + b2
  int *cnt_s = reinterpret_cast<int *>(w2s + S_CH + 4);         // [2 stages][4 warps][2 images]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tile_rows <= 128 rows per tile (the TMA box height): chosen by the launcher so that the tiles divide evenly over
  // the CTAs (e.g. 114 rows -> exactly 3 tiles per SM for 50 432 rows instead of 2.66 tiles of 128); the MMA still
  // runs M = 128 and the rows past tile_rows are ignored.
  const int num_tiles = (rows_total + tile_rows - 1) / tile_rows;
  const int num_kb = D / S_KB;
  pdl_launch_dependents();

  if (threadIdx.x < S_CH + 1) w2s[threadIdx.x] = comp[(size_t)S_CH * 2 * D + S_CH + threadIdx.x];   // w2[64], b2
  // the compaction kernel that follows appends this layer's attention work units: zero their counter (everything that
  // read the previous layer's table finished before cls_half_kernel, this grid's only programmatic predecessor, began)
  if (blockIdx.x == 0 && threadIdx.x == 0) *unit_count = 0;
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_whi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_wlo) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < NS_F; ++i) { mbar_init(&full_f[i], 1); mbar_init(&empty_f[i], 8); }
      for (int i = 0; i < NS_W; ++i) { mbar_init(&full_w[i], 1); mbar_init(&empty_w[i], 1); }
      for (int i = 0; i < NS_A; ++i) { mbar_init(&full_a[i], 8); mbar_init(&empty_a[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_slot)), "n"(S_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // wait_late (the normal case): this grid is a programmatic dependent of cls_half_kernel ONLY -- cls_half itself is an
  // ordinary launch, so everything older (the fp32 stream) is complete and visible when this grid starts -- and only
  // the epilogue warps, which read hc, wait for it: the stream, conversion and MMAs of the first tile overlap the
  // CLS-half GEMV.  With PSV_PDL (every kernel a programmatic dependent) all threads must wait here instead.
  if (!wait_late) pdl_wait();

  // Producer and MMA issuer run as whole warps with warp-uniform control flow; one elected lane executes the TMA /
  // tcgen05 instructions, so descriptors stay in uniform registers and the MMAs of a k-block issue back to back
  // (under `if (lane == 0)` each one sits in an ELECT + R2UR waterfall loop of ~150 cycles -- 5x its execution time).
  if (warp == 0) {
    // ===== TMA producer: two 128B-swizzled [tile_rows x 32] fp32 boxes per k-block =====
    int sf = 0; uint32_t phf = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int row0 = tile * tile_rows;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_f[sf], phf ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_f[sf], (uint32_t)tile_rows * S_KB * 4);
          tma_load_2d(smem + OFF_F + sf * F_BYTES, &map_x, &full_f[sf], kb * S_KB, row0);
          tma_load_2d(smem + OFF_F + sf * F_BYTES + F_HALF, &map_x, &full_f[sf], kb * S_KB + 32, row0);
        }
        __syncwarp();
        if (++sf == NS_F) { sf = 0; phf ^= 1; }
      }
    }
  } else if (warp == 14) {
    // ===== TMA producer of the weight slabs (L2 hits).  A warp of its own: in one in-order producer the wait for a
    // free weight stage also held back the NEXT fp32 tile. =====
    int sw = 0; uint32_t phw = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_w[sw], phw ^ 1);
        if (elect_one()) {
          if (debug & 4) mbar_arrive(&full_w[sw]);
          else {
            mbar_arrive_expect_tx(&full_w[sw], 2 * W_BYTES);
            tma_load_2d(smem + OFF_W + sw * 2 * W_BYTES, &map_whi, &full_w[sw], kb * S_KB, 0);
            tma_load_2d(smem + OFF_W + sw * 2 * W_BYTES + W_BYTES, &map_wlo, &full_w[sw], kb * S_KB, 0);
          }
        }
        __syncwarp();
        if (++sw == NS_W) { sw = 0; phw ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: A (x_hi / x_lo) from tensor memory, B (the weight slabs) from shared memory =====
    constexpr uint32_t idesc = make_idesc(S_ROWS, S_CH);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    int sa = 0, sw = 0, acc = 0; uint32_t pha = 0, phw = 0, acc_ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(&tempty[acc], acc_ph ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + acc * S_ACC_COLS;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_a[sa], pha);
        mbar_wait(&full_w[sw], phw);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_hi = tmem_u + S_A_COL + sa * 64, a_lo = a_hi + 32;
          const uint64_t d_hi = make_sw128_desc(smem_u32(smem + OFF_W + sw * 2 * W_BYTES));
          const uint64_t d_lo = make_sw128_desc(smem_u32(smem + OFF_W + sw * 2 * W_BYTES + W_BYTES));
#pragma unroll
          for (int k = 0; k < S_KB / 16; ++k) {
            if (debug & 2) break;
            const uint64_t o = (uint64_t)(k * 2);
            umma_bf16_ts(d_tmem, a_hi + k * 8, d_hi + o, idesc, (kb | k) ? 1u : 0u);   // x_hi . w_hi
            umma_bf16_ts(d_tmem, a_hi + k * 8, d_lo + o, idesc, 1u);                   // x_hi . w_lo
            umma_bf16_ts(d_tmem, a_lo + k * 8, d_hi + o, idesc, 1u);                   // x_lo . w_hi
          }
          umma_commit(&empty_a[sa]);
          umma_commit(&empty_w[sw]);
          if (kb + 1 == num_kb) umma_commit(&tfull[acc]);
        }
        __syncwarp();
        if (++sa == NS_A) { sa = 0; pha ^= 1; }
        if (++sw == NS_W) { sw = 0; phw ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_ph ^= 1; }
    }
  } else if (warp < 6) {
    // ===== epilogue: one thread per row =====
    const int quad = warp & 3;
    int acc = 0; uint32_t acc_ph = 0;
    if (wait_late) pdl_wait();                                  // hc is written by cls_half_kernel
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int r = tile * tile_rows + quad * 32 + lane;
      const bool valid = r < rows_total && quad * 32 + lane < tile_rows;
      const int b = valid ? r / N : 0;
      const int tok = r - b * N;
      mbar_wait(&tfull[acc], acc_ph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * S_ACC_COLS;
      float z = w2s[S_CH];
      const float4 *hcb = reinterpret_cast<const float4 *>(hc + (size_t)b * S_CH);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t v[16];
        tmem_ld16(taddr + q * 16, v);                           // x_hi.w_hi + x_hi.w_lo + x_lo.w_hi
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 h4 = __ldg(hcb + q * 4 + (j >> 2));
          const float4 w4 = *reinterpret_cast<const float4 *>(w2s + q * 16 + j);
          const float4 a4 = make_float4(__uint_as_float(v[j]) + h4.x, __uint_as_float(v[j + 1]) + h4.y,
                                        __uint_as_float(v[j + 2]) + h4.z, __uint_as_float(v[j + 3]) + h4.w);
          z = fmaf(fmaxf(a4.x, 0.f), w4.x, z);
          z = fmaf(fmaxf(a4.y, 0.f), w4.y, z);
          z = fmaf(fmaxf(a4.z, 0.f), w4.z, z);
          z = fmaf(fmaxf(a4.w, 0.f), w4.w, z);
          // training: keep the pre-activations, the backward pass then needs no second 768-wide product
          if (preact_out && valid && tok > 0)
            *reinterpret_cast<float4 *>(preact_out + ((size_t)b * (N - 1) + tok - 1) * S_CH + q * 16 + j) = a4;
        }
      }
      tc_fence_before();
      __syncwarp();
      const int acc_now = acc;
      if (lane == 0) mbar_arrive(&tempty[acc]);                 // accumulator has been read
      if (++acc == 2) { acc = 0; acc_ph ^= 1; }
      const float s = 1.0f / (1.0f + expf(-z));
      uint8_t m = 0;
      if (valid) {
        if (tok == 0) m = 1;                                     // CLS column is always processed (:67-68)
        else {
          m = forced ? (forced[r] != 0) : (s >= mt);
          scores[(size_t)b * (N - 1) + tok - 1] = s;
          if (scores_out) scores_out[(size_t)b * (N - 1) + tok - 1] = s;
        }
        mask[r] = m;
        if (mask_out) mask_out[r] = m;
      }
      // active-token counts of the tile's two images (a 128-row tile touches at most two, N > 128): the four
      // epilogue warps combine their ballots through shared memory and the tile STORES its pair of counts
      const int b_tile = (tile * tile_rows) / N;
      const unsigned in_first = __ballot_sync(0xffffffffu, m && b == b_tile);
      const unsigned in_next = __ballot_sync(0xffffffffu, m && b != b_tile);
      if (lane == 0) { cnt_s[(acc_now * 4 + quad) * 2] = __popc(in_first); cnt_s[(acc_now * 4 + quad) * 2 + 1] = __popc(in_next); }
      asm volatile("bar.sync 1, 128;" ::: "memory");            // the four epilogue warps
      if (warp == 2 && lane == 0) {
        const int *c = cnt_s + acc_now * 8;
        n_tile[tile] = make_int2(c[0] + c[2] + c[4] + c[6], c[1] + c[3] + c[5] + c[7]);
      }
    }
  } else if (warp < 14) {
    // ===== converters (8 warps): fp32 tile -> (hi, lo) bf16 pairs stored into tensor memory =====
    // thread <-> tile row = TMEM lane 32 * (warp % 4) + lane; the two warps of a lane quadrant take the two
    // 32-column halves of the k-block.  A row of a half is one 128-byte swizzle row (16-byte chunk c at c ^ (row & 7)),
    // so the 8 float4 loads of a thread and those of its 7 neighbours cover all banks: no conflicts.
    const int quad = warp & 3, half = (warp - 6) >> 2;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    int sf = 0, sa = 0; uint32_t phf = 0, pha = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_f[sf], phf);
        mbar_wait(&empty_a[sa], pha ^ 1);
        tc_fence_after();
        if (!(debug & 1)) {
          const uint8_t *src = smem + OFF_F + sf * F_BYTES + half * F_HALF + row * 128;
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 f = *reinterpret_cast<const float4 *>(src + ((c ^ (row & 7)) << 4));
            const bf16 h0 = __float2bfloat16_rn(f.x), h1 = __float2bfloat16_rn(f.y);
            const bf16 h2 = __float2bfloat16_rn(f.z), h3 = __float2bfloat16_rn(f.w);
            hi[2 * c] = pack2(h0, h1);
            hi[2 * c + 1] = pack2(h2, h3);
            lo[2 * c] = pack2(__float2bfloat16_rn(f.x - __bfloat162float(h0)), __float2bfloat16_rn(f.y - __bfloat162float(h1)));
            lo[2 * c + 1] = pack2(__float2bfloat16_rn(f.z - __bfloat162float(h2)), __float2bfloat16_rn(f.w - __bfloat162float(h3)));
          }
          const uint32_t ta = lane_addr + S_A_COL + sa * 64 + half * 16;
          tmem_st16(ta, hi);
          tmem_st16(ta + 32, lo);
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { mbar_arrive(&full_a[sa]); mbar_arrive(&empty_f[sf]); }
        if (++sf == NS_F) { sf = 0; phf ^= 1; }
        if (++sa == NS_A) { sa = 0; pha ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(S_TMEM_COLS) : "memory");
  }
}

// hi/lo bf16 split of the token half of W1:  w[j][k] = c1_w[j][D + k]
__global__ void comp_split_kernel(const float *__restrict__ c1, bf16 *__restrict__ hi, bf16 *__restrict__ lo, int D) {
  const int total = S_CH * D;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int j = e / D, k = e % D;
    const float w = c1[(size_t)j * 2 * D + D + k];
    const bf16 h = __float2bfloat16_rn(w);
    hi[e] = h;
    lo[e] = __float2bfloat16_rn(w - __bfloat162float(h));
  }
}

}  // namespace

cudaError_t configure_score_tc() {
  return cudaFuncSetAttribute(score_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, S_SMEM);
}

cudaError_t launch_comp_split(PsvHandle *h, const LayerPack &lp, cudaStream_t s) {
  comp_split_kernel<<<64, 256, 0, s>>>(lp.c1, lp.c1_tok_hi, lp.c1_tok_lo, h->D);
  return cudaGetLastError();
}

cudaError_t launch_score_mask_tc(PsvHandle *h, const LayerPack &lp, const float *hidden, int batch, float mt,
                                 const uint8_t *forced_mask, uint8_t *mask_out, float *scores_out, float *preact_out,
                                 cudaStream_t s) {
  const int rows = batch * h->N;
  CUtensorMap mx, mhi, mlo;
  // rows per tile: the smallest height that keeps the number of rounds per CTA of 128-row tiles
  const int rounds = (rows + S_ROWS * h->sm_count - 1) / (S_ROWS * h->sm_count);
  int tile_rows = (rows + rounds * h->sm_count - 1) / (rounds * h->sm_count);
  tile_rows = tile_rows < 8 ? 8 : (tile_rows > S_ROWS ? S_ROWS : tile_rows);
  h->score_tile_rows = tile_rows;
  cudaError_t e = get_tmap_2d(h->tmaps, hidden, (uint64_t)rows, (uint64_t)h->D, (uint32_t)tile_rows, 32, 4, 128, &mx);
  if (e != cudaSuccess) return e;
  e = get_tmap_2d(h->tmaps, lp.c1_tok_hi, S_CH, (uint64_t)h->D, S_CH, S_KB, 2, 128, &mhi);
  if (e != cudaSuccess) return e;
  e = get_tmap_2d(h->tmaps, lp.c1_tok_lo, S_CH, (uint64_t)h->D, S_CH, S_KB, 2, 128, &mlo);
  if (e != cudaSuccess) return e;
  {
    LaunchScope scope(h, KK_CLS_HALF, s);
    const int cg = (batch + CLS_IMGS - 1) / CLS_IMGS;
    if (h->D == 1024)     e = launch_pdl(cls_half_kernel<1024>, dim3(cg), dim3(512), 0, s, hidden, (const float *)lp.c1, h->N, batch, h->hc);
    else if (h->D == 768) e = launch_pdl(cls_half_kernel<768>, dim3(cg), dim3(512), 0, s, hidden, (const float *)lp.c1, h->N, batch, h->hc);
    else if (h->D == 384) e = launch_pdl(cls_half_kernel<384>, dim3(cg), dim3(512), 0, s, hidden, (const float *)lp.c1, h->N, batch, h->hc);
    else                  e = cudaErrorNotSupported;
    if (e != cudaSuccess) return e;
  }
  LaunchScope scope(h, KK_SCORE, s);
  static const int dbg = getenv("PSV_SCORE_DEBUG") ? atoi(getenv("PSV_SCORE_DEBUG")) : 0;   // timing experiments only
  const int tiles = (rows + tile_rows - 1) / tile_rows;
  const int grid = tiles < h->sm_count ? tiles : h->sm_count;
  static const bool no_overlap = getenv("PSV_SCORE_NO_OVERLAP") != nullptr;     // A/B switch for the measurement
  const int wait_late = (!pdl_enabled() && !no_overlap) ? 1 : 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(S_THREADS); cfg.dynamicSmemBytes = (size_t)S_SMEM; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = (wait_late || pdl_enabled()) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, score_tc_kernel, mx, mhi, mlo, (const float *)lp.c1, (const float *)h->hc, mt, forced_mask,
                            rows, h->N, h->D, h->mask, h->scores, (int2 *)h->n_tile, mask_out, scores_out, preact_out,
                            tile_rows, dbg, wait_late, h->attn_unit_count);
}

}  // namespace psv
