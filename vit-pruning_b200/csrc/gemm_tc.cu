// K5/K7/K9/K10/K0: bf16 GEMM on the 5th-generation tensor cores (tcgen05.mma, accumulators in
// TMEM), operands staged by TMA into 128B-swizzled shared memory, with the fused epilogue of
// GemmArgs:   out[orow(r), :] = act(A[r, :] . W^T + bias) + res[rrow(r), :]
//
// Structure (one CTA per SM, persistent over output tiles, 576 threads):
//   CTAs run as PAIRS (cluster of 2, tcgen05 cta_group::2): a pair owns a 256 x BN output tile.
//   warp 0      TMA producer   : each CTA loads its 128 rows of A and its half of the W tile ([BN/2 x 64]) per
//                                k-block into an NSTAGE ring; all boxes complete on the leader's full barrier
//   warp 1      MMA issuer     : one lane of the LEADER CTA issues 4 x tcgen05.mma.cta_group::2 (256 x BN x 16)
//                                per k-block; tcgen05.commit (multicast to both CTAs) releases the smem slot /
//                                publishes the accumulator, which lands in each CTA's own TMEM (its 128 rows)
//   warps 2..17 epilogue       : tcgen05.ld the fp32 accumulator (2 TMEM stages, so the epilogue of
//                                tile i overlaps the MMAs of tile i+1), bias, erf-GELU, transpose via
//                                shared memory so global traffic is whole 128-byte lines, fp32
//                                residual (optionally gathered by res_idx), store fp32 or bf16
//                                (optionally scattered by out_idx)
// The row count M is data dependent (T = number of active tokens): it is read from device memory
// by every role, the grid is sized for m_max, and tiles past M are never scheduled.
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>

#include "tc_common.cuh"

namespace psv {

// ------------------------------------------------------------------------------------------------
// tensor-map cache (host)
struct TensorMapCache {
  struct Key {
    const void *ptr; uint64_t rows, cols; uint32_t box_rows, box_cols; int elem_bytes; int sw;
    bool operator==(const Key &o) const {
      return ptr == o.ptr && rows == o.rows && cols == o.cols && box_rows == o.box_rows && box_cols == o.box_cols &&
             elem_bytes == o.elem_bytes && sw == o.sw;
    }
  };
  struct Hash {
    size_t operator()(const Key &k) const {
      return std::hash<const void *>()(k.ptr) ^ (k.rows * 0x9E3779B97F4A7C15ull) ^ (k.cols << 20) ^ k.box_rows ^
             ((size_t)k.box_cols << 12) ^ ((size_t)k.elem_bytes << 40) ^ ((size_t)k.sw << 48);
    }
  };
  std::unordered_map<Key, CUtensorMap, Hash> maps;
  std::mutex mu;
};

TensorMapCache *tmap_cache_create() { return new TensorMapCache(); }
void tmap_cache_destroy(TensorMapCache *c) { delete c; }

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

}  // namespace

bool tmap_encode_available() { return get_encode_fn() != nullptr; }

cudaError_t get_tmap_2d(TensorMapCache *cache, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows,
                        uint32_t box_cols, int elem_bytes, int swizzle, CUtensorMap *out) {
  TensorMapCache::Key key{ptr, rows, cols, box_rows, box_cols, elem_bytes, swizzle};
  std::lock_guard<std::mutex> lock(cache->mu);
  auto it = cache->maps.find(key);
  if (it != cache->maps.end()) { *out = it->second; return cudaSuccess; }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return cudaErrorNotSupported;
  CUtensorMap m;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(&m, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
  if (cache->maps.size() > 4096) cache->maps.clear();
  cache->maps.emplace(key, m);
  *out = m;
  return cudaSuccess;
}

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;            // 64 bf16 = 128 bytes = one swizzle row
constexpr int UMMA_K = 16;
constexpr int EPI_WARPS = 16;
constexpr int TC_THREADS = 64 + 32 * EPI_WARPS;    // TMA warp, MMA warp, 16 epilogue warps

using namespace tc;

// erf-GELU for the bf16 outputs.  gelu(v) = v * Phi(v), Phi(v) = erfc(-v / sqrt 2) / 2, and on z = |v| / sqrt 2
// erfc(z) = 2^(z * P5(z)) to 6e-7 absolute (degree-5 fit of log2 erfc, see DESIGN.md) -- far below bf16 rounding --
// so the whole activation is 5 FMAs, ONE MUFU.EX2, a select and two multiplies; the MUFU pipe (16 lanes/clk/SM)
// is what limited the previous rcp+exp formulation.  (The fp32 mode uses exact erff in gemm_simt.cu.)
__device__ __forceinline__ float gelu_erf_fast(float v) {
  const float z = fabsf(v) * 0.70710678118654752440f;
  float p = fmaf(-0.00294979016f, z, 0.0296096159f);
  p = fmaf(p, z, -0.14868762f);
  p = fmaf(p, z, -0.918500394f);
  p = fmaf(p, z, -1.62789f);
  float t;                                                   // t = erfc(z) / 2 = 2^(z * P(z) - 1)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(p, z, -1.0f)));
  return v * (v >= 0.0f ? 1.0f - t : t);
}

// Packed-pair form of the same activation on Blackwell's FFMA2 (fma.rn.f32x2): the Horner chain runs on two
// accumulator columns per instruction, which is what takes the FC1 epilogue's issue load below the MMA time.
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ void add_f32x2(float &o0, float &o1, float a0, float a1, float b0, float b1) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pack_f32x2(a0, a1)), "l"(pack_f32x2(b0, b1)));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(o0), "=f"(o1) : "l"(r));
}
__device__ __forceinline__ void gelu_erf_fast2(float &x0, float &x1) {
  const uint64_t z = pack_f32x2(fabsf(x0) * 0.70710678118654752440f, fabsf(x1) * 0.70710678118654752440f);
  uint64_t p = fma_f32x2(pack_f32x2(-0.00294979016f, -0.00294979016f), z, pack_f32x2(0.0296096159f, 0.0296096159f));
  p = fma_f32x2(p, z, pack_f32x2(-0.14868762f, -0.14868762f));
  p = fma_f32x2(p, z, pack_f32x2(-0.918500394f, -0.918500394f));
  p = fma_f32x2(p, z, pack_f32x2(-1.62789f, -1.62789f));
  p = fma_f32x2(p, z, pack_f32x2(-1.0f, -1.0f));               // z * P(z) - 1
  float e0, e1, t0, t1;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(e0), "=f"(e1) : "l"(p));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(e0));      // t = erfc(z) / 2
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(e1));
  x0 *= (x0 >= 0.0f ? 1.0f - t0 : t0);
  x1 *= (x1 >= 0.0f ? 1.0f - t1 : t1);
}

template <int BN> struct TcCfg {
  static constexpr int NSTAGE = (BN == 256) ? 6 : 8;
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;          // 16 KB : this CTA's 128 rows of the 256-row pair tile
  static constexpr int B_BYTES = (BN / 2) * BLOCK_K * 2;         // 16 KB / 8 KB : this CTA's half of the W tile
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TMEM_COLS = 2 * BN;                       // two accumulator stages (512 / 256)
  static constexpr int BAR_OFF = NSTAGE * STAGE_BYTES;           // barriers + tmem slot (padded to 1 KB)
  static constexpr int PATCH_OFF = BAR_OFF + 1024;               // 16 epilogue patches of 2 KB, 1 KB aligned
  static constexpr int SMEM_BYTES = PATCH_OFF + EPI_WARPS * 2048 + 1024 /*align slack*/;
};

// Epilogue modes (compile-time, so the hot loops carry no runtime branches on them):
//   EPI_BF16   out = bf16(act(acc + bias))             packed rows, written with TMA stores
//   EPI_RED    out[orow] += acc + bias                 fp32 red.global.add.v4 into the residual stream
//   EPI_STORE  out[orow] = acc + bias (+ res[rrow])    fp32 stores, optional gathered fp32 residual
enum { EPI_BF16 = 0, EPI_RED = 1, EPI_STORE = 2 };

// Work iterator shared by the three roles of a CTA pair.  Round-robin over whole pair-tiles, or (stream-K, used
// by the accumulate epilogue whose partial sums can simply be red-added) a contiguous, equal share of the
// (pair-tile, k-block) space per pair -- no wave quantisation, at the price that a tile cut across two pairs
// receives its two fp32 red.adds in either order.
struct WorkIter {
  int u, u_end, num_kb, tile_rr, step, num_tiles;
  bool sk;
  __device__ WorkIter(bool streamk, int pair, int pairs, int num_tiles_, int num_kb_)
      : num_kb(num_kb_), tile_rr(pair), step(pairs), num_tiles(num_tiles_), sk(streamk) {
    const int total = num_tiles_ * num_kb_;
    const int per = (total + pairs - 1) / pairs;
    u = pair * per;
    u_end = min(total, u + per);
  }
  __device__ bool next(int &tile, int &kb0, int &kb1) {
    if (sk) {
      if (u >= u_end) return false;
      tile = u / num_kb; kb0 = u - tile * num_kb; kb1 = min(num_kb, kb0 + (u_end - u));
      u += kb1 - kb0;
      return true;
    }
    if (tile_rr >= num_tiles) return false;
    tile = tile_rr; tile_rr += step; kb0 = 0; kb1 = num_kb;
    return true;
  }
};

struct EpiArgs {
  const float *bias; const float *res; const int32_t *res_idx; const int32_t *out_idx; void *out;
  long long *trace;      // PSV_GEMM_TRACE=1: globaltimer stamps of CTA 0 (debugging aid), else null
};
__device__ __forceinline__ void gemm_stamp(long long *trace, int slot) {
  if (trace && blockIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    trace[slot] = t;
  }
}

// number of work units of the tail-wave schedule (see gemm_tc_kernel) and the first tile that is split into halves
__device__ __forceinline__ int tail_units(int tiles, int pairs, bool enable, int &tail_from) {
  tail_from = tiles;
  if (!enable) return tiles;
  const int full = (tiles / pairs) * pairs, rest = tiles - full;
  if (rest == 0 || 2 * rest > pairs) return tiles;
  tail_from = full;
  return full + 2 * rest;
}

template <int BN, int MODE, bool GELU>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
               const __grid_constant__ CUtensorMap map_out, EpiArgs ep, int m_max, int N, int K,
               const int32_t *__restrict__ m_dev, int streamk, int pdl, const __grid_constant__ CUtensorMap map_w_half,
               int tail) {
  using Cfg = TcCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::BAR_OFF);
  uint64_t *full_bar = bars;                       // [NSTAGE]
  uint64_t *empty_bar = bars + Cfg::NSTAGE;        // [NSTAGE]
  uint64_t *tfull_bar = bars + 2 * Cfg::NSTAGE;    // [2]
  uint64_t *tempty_bar = tfull_bar + 2;            // [2]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) gemm_stamp(ep.trace, 0);
  // the row count is produced by an earlier kernel: without programmatic launch it can be fetched right away, so
  // the global-load latency overlaps the barrier / TMEM set-up instead of preceding the first TMA load
  const int m_early = (!pdl && m_dev) ? min(*m_dev, m_max) : m_max;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    if (MODE == EPI_BF16) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_out) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < Cfg::NSTAGE; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * EPI_WARPS); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"       // warp 1 of BOTH CTAs
                 ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                              // both CTAs' barriers are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) gemm_stamp(ep.trace, 1);
  pdl_wait();                                      // everything above overlapped the previous kernel's tail
  const int M = pdl ? (m_dev ? min(*m_dev, m_max) : m_max) : m_early;
  const int n_tiles = N / BN;
  // Work unit of a CTA pair = a 256 x BN output tile computed by ONE tcgen05.mma.cta_group::2 stream issued by
  // the even CTA: each CTA stages its own 128 rows of A and its own half of the W tile, the pair's tensor cores
  // exchange the W halves, and each CTA's TMEM receives its 128 rows.  Per CTA and k-block that is 32 KB through
  // shared memory instead of 48 KB -- shared-memory bandwidth (TMA writes + MMA operand reads) is what bounds the
  // single-CTA form.  With an odd number of M-tiles the last pair's second half lies past M: it is computed on
  // stale rows and never written.
  const uint32_t cta_rank = cluster_ctarank();
  const int m_pairs = ((M + BLOCK_M - 1) / BLOCK_M + 1) / 2;
  const int num_tiles = m_pairs * n_tiles;         // pairs
  const int first_tile = blockIdx.x >> 1, tile_step = gridDim.x >> 1;
  const int num_kb = K / BLOCK_K;
  const bool sk = (MODE == EPI_RED) && streamk != 0;
  // Tail wave (tail != 0, BN = 256, round-robin order): when the tiles left over after the last FULL wave number at
  // most half the pairs, each of them is computed as two 256 x 128 half tiles by two different pairs, so the last
  // wave costs ~0.62 of a tile instead of a whole one.  Work units: u < tail_from is full tile u, u >= tail_from is
  // half (u - tail_from) & 1 of tile tail_from + ((u - tail_from) >> 1).  Every output element still sums its k
  // products in the same order, so the bits do not depend on the split.
  const bool tail_on = (BN == 256) && tail != 0 && !sk;

  // The producer and the MMA issuer run as WHOLE warps with warp-uniform control flow and operands (the row count
  // goes through a shuffle broadcast), and one elected lane executes the TMA / tcgen05 instructions.  Under
  // `if (lane == 0)` the compiler cannot keep descriptors in uniform registers and wraps every UTMALDG / UTCHMMA
  // in an ELECT + R2UR waterfall loop (~150 cycles each, more than the 128 cycles one 256x256x16 MMA takes).
  if (warp == 0) {
    // ===== TMA producer =====
    {
      const int Mu = __shfl_sync(0xffffffffu, M, 0);
      const int tiles_u = (((Mu + BLOCK_M - 1) / BLOCK_M + 1) / 2) * n_tiles;
      int tail_from;
      const int units_u = tail_units(tiles_u, tile_step, tail_on, tail_from);
      int stage = 0; uint32_t phase = 0;
      WorkIter it(sk, first_tile, tile_step, units_u, num_kb);
      int unit, kb0, kb1;
      while (it.next(unit, kb0, kb1)) {
        const bool half_u = unit >= tail_from;
        const int tile = half_u ? tail_from + ((unit - tail_from) >> 1) : unit;
        const int bn_u = half_u ? 128 : BN;
        const int m0 = ((tile / n_tiles) * 2 + (int)cta_rank) * BLOCK_M;
        const int n0 = (tile % n_tiles) * BN + (half_u ? ((unit - tail_from) & 1) * 128 : 0);
        const CUtensorMap *mw_u = half_u ? &map_w_half : &map_w;
        const uint32_t stage_tx = (uint32_t)(2 * (Cfg::A_BYTES + (bn_u / 2) * BLOCK_K * 2));
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);            // the pair's MMAs have released this stage
          if (elect_one()) {
            uint8_t *sa = smem + stage * Cfg::STAGE_BYTES;
            // all four boxes of the pair (2 x A, 2 x W half) complete on the LEADER's full barrier
            if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], stage_tx);
            tma_load_2d_2sm(sa, &map_a, &full_bar[stage], kb * BLOCK_K, m0);
            tma_load_2d_2sm(sa + Cfg::A_BYTES, mw_u, &full_bar[stage], kb * BLOCK_K, n0 + (int)cta_rank * (bn_u / 2));
          }
          __syncwarp();
          if (++stage == Cfg::NSTAGE) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the leader CTA drives both tensor cores =====
    if (cta_rank == 0) {
      constexpr uint32_t idesc_full = make_idesc(2 * BLOCK_M, BN), idesc_half = make_idesc(2 * BLOCK_M, 128);
      const int Mu = __shfl_sync(0xffffffffu, M, 0);
      const int tiles_u = (((Mu + BLOCK_M - 1) / BLOCK_M + 1) / 2) * n_tiles;
      int tail_from;
      const int units_u = tail_units(tiles_u, tile_step, tail_on, tail_from);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      WorkIter it(sk, first_tile, tile_step, units_u, num_kb);
      int tile, kb0, kb1;                                    // `tile` is the work-unit index here
      while (it.next(tile, kb0, kb1)) {
        const uint32_t idesc = tile >= tail_from ? idesc_half : idesc_full;
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);          // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            if (kb == kb0 && tile == first_tile) gemm_stamp(ep.trace, 2);
            const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
            const uint64_t da = make_sw128_desc(sa), db = make_sw128_desc(sa + Cfg::A_BYTES);
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
              // advance along K inside the 128B swizzle row: +32 bytes = +2 in the (addr >> 4) field
              umma_bf16_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, ((kb - kb0) | k) ? 1u : 0u);
            }
            umma_commit_2sm(&empty_bar[stage]);              // slot free in BOTH CTAs once these MMAs retire
            if (kb + 1 == kb1) umma_commit_2sm(&tfull_bar[acc]);   // accumulator complete, in both CTAs' TMEM
          }
          __syncwarp();
          if (++stage == Cfg::NSTAGE) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===== 16 epilogue warps: TMEM lane quadrant = warp % 4, column quarter = (warp - 2) / 4 =====
    // Each warp drains 32 rows x BN/4 columns of the accumulator through its own 2 KB shared-memory
    // patch ([32 rows][64 bytes], 16-byte chunks XOR-swizzled by (row >> 1) & 3 = TMA SWIZZLE_64B), so
    // global traffic runs along the rows instead of one row per lane.
    const int quad = warp & 3, part = (warp - 2) >> 2;
    uint8_t *patch = smem + Cfg::PATCH_OFF + (warp - 2) * 2048;
    const uint32_t my_off = (uint32_t)(lane * 64), my_sw = (uint32_t)((lane >> 1) & 3);
    int acc = 0; uint32_t acc_phase = 0;
    int tail_from;
    const int num_units = tail_units(num_tiles, tile_step, tail_on, tail_from);
    WorkIter it(sk, first_tile, tile_step, num_units, num_kb);
    int unit, kb0, kb1;
    while (it.next(unit, kb0, kb1)) {
      const bool add_bias = ep.bias != nullptr && kb0 == 0;   // a k-split tile gets its bias from the first part
      const bool half_u = unit >= tail_from;
      const int tile = half_u ? tail_from + ((unit - tail_from) >> 1) : unit;
      const int bn_u = half_u ? 128 : BN;                     // columns of this work unit
      const int m0 = ((tile / n_tiles) * 2 + (int)cta_rank) * BLOCK_M;
      const int n0 = (tile % n_tiles) * BN + (half_u ? ((unit - tail_from) & 1) * 128 : 0) + part * (bn_u / 4);
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + part * (bn_u / 4);

      if (MODE == EPI_BF16) {
        // ---- 32-column chunks: registers -> bias / GELU -> bf16 -> patch -> one TMA store per chunk
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        if (threadIdx.x == 64 && unit == first_tile) gemm_stamp(ep.trace, 3);
#pragma unroll 1
        for (int c = 0; c < bn_u / 128; ++c) {
          const int col = n0 + c * 32;
          uint32_t v[32];
          tmem_ld32(taddr + c * 32, v);
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // patch free again
          __syncwarp();
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            float f[8];
            const float4 b0 = __ldg(reinterpret_cast<const float4 *>(ep.bias + col + j));
            const float4 b1 = __ldg(reinterpret_cast<const float4 *>(ep.bias + col + j + 4));
            add_f32x2(f[0], f[1], __uint_as_float(v[j]), __uint_as_float(v[j + 1]), b0.x, b0.y);
            add_f32x2(f[2], f[3], __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]), b0.z, b0.w);
            add_f32x2(f[4], f[5], __uint_as_float(v[j + 4]), __uint_as_float(v[j + 5]), b1.x, b1.y);
            add_f32x2(f[6], f[7], __uint_as_float(v[j + 6]), __uint_as_float(v[j + 7]), b1.z, b1.w);
            if (GELU) {
#pragma unroll
              for (int e = 0; e < 8; e += 2) gelu_erf_fast2(f[e], f[e + 1]);
            }
            __nv_bfloat162 p0 = __floats2bfloat162_rn(f[0], f[1]), p1 = __floats2bfloat162_rn(f[2], f[3]);
            __nv_bfloat162 p2 = __floats2bfloat162_rn(f[4], f[5]), p3 = __floats2bfloat162_rn(f[6], f[7]);
            uint4 pk;
            pk.x = *reinterpret_cast<uint32_t *>(&p0); pk.y = *reinterpret_cast<uint32_t *>(&p1);
            pk.z = *reinterpret_cast<uint32_t *>(&p2); pk.w = *reinterpret_cast<uint32_t *>(&p3);
            *reinterpret_cast<uint4 *>(patch + my_off + ((((uint32_t)j >> 3) ^ my_sw) << 4)) = pk;
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(&map_out), "r"(smem_u32(patch)), "r"(col), "r"(m0 + quad * 32) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      } else {
        // ---- fp32 output, 16-column chunks transposed through the patch: 4 lanes x 16 B per row
        const int r_own = m0 + quad * 32 + lane;
        int orow_own = -1, rrow_own = 0;                     // -1: row past M, nothing to write
        if (r_own < M) {
          orow_own = ep.out_idx ? ep.out_idx[r_own] : r_own;
          if (MODE == EPI_STORE && ep.res) rrow_own = ep.res_idx ? ep.res_idx[r_own] : r_own;
        }
        const int c4 = lane & 3;
        int orow[4], rrow[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          orow[it] = __shfl_sync(0xffffffffu, orow_own, it * 8 + (lane >> 2));
          rrow[it] = __shfl_sync(0xffffffffu, rrow_own, it * 8 + (lane >> 2));
        }
        float4 rv[4];
        if (MODE == EPI_STORE && ep.res) {                   // residual of chunk 0, before the accumulator wait
#pragma unroll
          for (int it = 0; it < 4; ++it)
            rv[it] = __ldg(reinterpret_cast<const float4 *>(ep.res + (size_t)rrow[it] * N + n0 + c4 * 4));
        }
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        if (threadIdx.x == 64 && unit == first_tile) gemm_stamp(ep.trace, 3);
#pragma unroll 1
        for (int c = 0; c < bn_u / 64; ++c) {
          const int col = n0 + c * 16;
          uint32_t v[16];
          tmem_ld16(taddr + c * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float4 f = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                   __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            if (add_bias) {
              const float4 b4 = __ldg(reinterpret_cast<const float4 *>(ep.bias + col + 4 * j));
              f.x += b4.x; f.y += b4.y; f.z += b4.z; f.w += b4.w;
            }
            *reinterpret_cast<float4 *>(patch + my_off + (((uint32_t)j ^ my_sw) << 4)) = f;
          }
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int row = it * 8 + (lane >> 2);
            float4 o = *reinterpret_cast<const float4 *>(patch + row * 64 + ((c4 ^ ((row >> 1) & 3)) << 4));
            if (MODE == EPI_STORE && ep.res) { o.x += rv[it].x; o.y += rv[it].y; o.z += rv[it].z; o.w += rv[it].w; }
            if (orow[it] >= 0) {
              float *op = reinterpret_cast<float *>(ep.out) + (size_t)orow[it] * N + col + c4 * 4;
              if (MODE == EPI_RED)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};"
                             ::"l"(op), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
              else
                *reinterpret_cast<float4 *>(op) = o;
            }
          }
          if (MODE == EPI_STORE && ep.res && c + 1 < bn_u / 64) {   // residual of the next chunk
#pragma unroll
            for (int it = 0; it < 4; ++it)
              rv[it] = __ldg(reinterpret_cast<const float4 *>(ep.res + (size_t)rrow[it] * N + col + 16 + c4 * 4));
          }
          __syncwarp();                                      // patch is reused by the next chunk
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tempty_bar[acc]);   // 2 x 16 epilogue warps release the pair's accumulator
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (MODE == EPI_BF16 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // patches read; the stores themselves complete with the grid
    if (threadIdx.x == 64) gemm_stamp(ep.trace, 4);
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                              // the peer may still multicast into / arrive on this CTA
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    if (lane == 0) gemm_stamp(ep.trace, 5);
  }
}

template <int BN, int MODE, bool GELU>
cudaError_t launch_one(const CUtensorMap &ma, const CUtensorMap &mw, const CUtensorMap &mo, const EpiArgs &ep,
                       const GemmArgs &g, int grid, cudaStream_t s, const CUtensorMap &mwh, int tail) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = TcCfg<BN>::SMEM_BYTES; cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 2 : 1;
  // Stream-K is OFF by default: it removes the wave quantisation of the accumulate-epilogue GEMMs (FC2 at
  // M=8448: 43.8 -> 39.1 us) but makes the fp32 residual sums order-dependent, and with hard skip thresholds a
  // 1-ulp change flips about one of the 600 k decisions of a batch-256 forward from run to run.  PSV_STREAMK=1.
  static const int streamk = getenv("PSV_STREAMK") ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, MODE, GELU>, ma, mw, mo, ep, g.m_max, g.n, g.k, g.m_dev, streamk,
                            pdl_enabled() ? 1 : 0, mwh, tail);
}

template <int BN>
cudaError_t dispatch(int mode, bool gelu, const CUtensorMap &ma, const CUtensorMap &mw, const CUtensorMap &mo,
                     const EpiArgs &ep, const GemmArgs &g, int grid, cudaStream_t s, const CUtensorMap &mwh, int tail) {
  if (mode == EPI_BF16) return gelu ? launch_one<BN, EPI_BF16, true>(ma, mw, mo, ep, g, grid, s, mwh, tail)
                                    : launch_one<BN, EPI_BF16, false>(ma, mw, mo, ep, g, grid, s, mwh, tail);
  if (mode == EPI_RED) return launch_one<BN, EPI_RED, false>(ma, mw, mo, ep, g, grid, s, mwh, tail);
  return launch_one<BN, EPI_STORE, false>(ma, mw, mo, ep, g, grid, s, mwh, tail);
}

}  // namespace

// All kernel variants get their dynamic-smem attribute here (outside any stream capture).
cudaError_t configure_gemm_tc() {
  if (!tmap_encode_available()) return cudaErrorNotSupported;
  cudaError_t e = cudaSuccess;
#define PSV_CFG(BN, MODE, GELU) \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<BN, MODE, GELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<BN>::SMEM_BYTES)
  PSV_CFG(256, EPI_BF16, true); PSV_CFG(256, EPI_BF16, false); PSV_CFG(256, EPI_RED, false); PSV_CFG(256, EPI_STORE, false);
  PSV_CFG(128, EPI_BF16, true); PSV_CFG(128, EPI_BF16, false); PSV_CFG(128, EPI_RED, false); PSV_CFG(128, EPI_STORE, false);
#undef PSV_CFG
  return e;
}

cudaError_t launch_gemm_tc(PsvHandle *h, const GemmArgs &g, cudaStream_t s) {
  if (g.n % 128 != 0 || g.k % BLOCK_K != 0 || g.m_max <= 0) return cudaErrorInvalidValue;
  if (g.gelu && g.out_fp32) return cudaErrorInvalidValue;          // GELU is fused only into the bf16 output path
  if (g.accumulate && (!g.out_fp32 || g.res)) return cudaErrorInvalidValue;
  if (!g.out_fp32 && (g.res || g.out_idx || !g.bias)) return cudaErrorInvalidValue;
  const int bn = g.n % 256 ? 128 : 256;
  // Tail wave: with 256-column tiles, the tiles left over after the last full wave are computed as 128-column halves
  // (see gemm_tc_kernel).  Measured 3.487 -> 3.418 ms per forward (+2.0 %) against a host-side tile-width choice from
  // a row-count hint, which it replaced: the device knows the exact row count, the host only a hint.
  const int tail = bn == 256 ? 1 : 0;
  const int mode = !g.out_fp32 ? EPI_BF16 : (g.accumulate ? EPI_RED : EPI_STORE);
  CUtensorMap ma, mw, mo, mwh;
  cudaError_t e = get_tmap_2d(h->tmaps, g.a, (uint64_t)g.m_max, (uint64_t)g.k, BLOCK_M, 64, 2, 128, &ma);
  if (e != cudaSuccess) return e;
  e = get_tmap_2d(h->tmaps, g.w, (uint64_t)g.n, (uint64_t)g.k, (uint32_t)bn / 2, 64, 2, 128, &mw);   // half tile per CTA
  if (e != cudaSuccess) return e;
  mwh = mw;
  if (tail) {                                                // 64-row boxes: a CTA's half of a 128-column half tile
    e = get_tmap_2d(h->tmaps, g.w, (uint64_t)g.n, (uint64_t)g.k, 64, 64, 2, 128, &mwh);
    if (e != cudaSuccess) return e;
  }
  if (mode == EPI_BF16) {
    e = get_tmap_2d(h->tmaps, g.out, (uint64_t)g.m_max, (uint64_t)g.n, 32, 32, 2, 64, &mo);
    if (e != cudaSuccess) return e;
  } else {
    mo = ma;
  }
  static const bool want_trace = getenv("PSV_GEMM_TRACE") != nullptr;
  static long long *trace = nullptr;
  if (want_trace && !trace) { cudaMalloc(&trace, 8 * sizeof(long long)); }
  if (want_trace) cudaMemsetAsync(trace, 0, 8 * sizeof(long long), s);
  EpiArgs ep{g.bias, g.res, g.res_idx, g.out_idx, g.out, want_trace ? trace : nullptr};
  const int max_pairs = (((g.m_max + BLOCK_M - 1) / BLOCK_M + 1) / 2) * (g.n / bn);
  const int max_clusters = h->sm_count / 2;
  const int grid = 2 * (max_pairs < max_clusters ? max_pairs : max_clusters);   // whole 2-CTA clusters
  LaunchScope scope(h, KK_GEMM, s);
  e = bn == 256 ? dispatch<256>(mode, g.gelu != 0, ma, mw, mo, ep, g, grid, s, mwh, tail)
                : dispatch<128>(mode, g.gelu != 0, ma, mw, mo, ep, g, grid, s, mwh, 0);
  if (want_trace && e == cudaSuccess) {
    long long t[8];
    cudaStreamSynchronize(s);
    cudaMemcpy(t, trace, sizeof t, cudaMemcpyDeviceToHost);
    fprintf(stderr, "gemm trace m_max=%d n=%d k=%d mode=%d: setup %lld  first-data %lld  first-acc %lld  epilogue-done %lld  end %lld ns\n",
            g.m_max, g.n, g.k, mode, t[1] - t[0], t[2] - t[0], t[3] - t[0], t[4] - t[0], t[5] - t[0]);
  }
  return e;
}

}  // namespace psv
