// K6 (bf16 mode): varlen attention among the ACTIVE tokens of each image on the 5th-generation tensor
// cores (reference model_utils.py:91 -> HF:171-196: softmax(q k^T / 8) v, per image, per head).
//
// An image has n <= 197 active tokens, so the whole key set of one (image, head) problem fits ONE tile:
// S = Q K^T [128 x n] lives in TMEM, each softmax thread owns one row and makes a SINGLE pass over it,
// P goes back into TMEM as bf16 over the dead S columns and O = P V runs with the A operand read from TMEM.
//
// Work unit = one (image, head); u = head * batch + image, round-robin over one persistent CTA per SM.  K and V
// are staged once per unit and shared by its one (n <= 128) or two 128-row query tiles.
//
//   warp 0       TMA producer : Q tile(s) + K box and the V box of the packed [T, 3D] bf16 activations (128B
//                               swizzle) into two rings (2 x 60 KB, 3 x 28 KB); Q/K slots are released as soon as
//                               the unit's last S retires, V slots after its last P V.  Box heights 32..224 rows
//                               (six tensor maps) keep the over-fetch below 32 rows.
//   warp 1       MMA issuer   : S(j) = Q K^T   tcgen05.mma SS (K-major A and B, 4 k-steps of 16)
//                               O(j) = P V     tcgen05.mma TS (A = P in TMEM, B = V MN-major: V rows are keys,
//                                              i.e. the contraction index is the slow dimension, no transpose)
//                               the warp polls (mbarrier.test_wait + vote) and issues whichever of "next S" /
//                               "next P V" is ready; whole-warp uniform control flow, one elected lane issues
//   warps 2..5   softmax warpgroup 0 (TMEM buffer 0: S [0,224) | P [0,112) | O [128,192) of 256 columns)
//   warps 6..9   softmax warpgroup 1 (TMEM buffer 1); tile j of the CTA's sequence belongs to warpgroup j & 1.
//                thread <-> S row (TMEM lane).  Rolling 32-column chunks: tcgen05.ld of chunk c+1 is in flight while
//                chunk c is exponentiated.  Running max with LAZY rescaling: the reference max only moves when a
//                chunk exceeds it by 2^8; then the few P chunks already written are rescaled in TMEM (exact, and
//                practically never taken).  Row sum over the ROUNDED bf16 probabilities, bf16 P via tcgen05.st;
//                then tcgen05.ld O, the TMEM buffer is handed back, scale by 1/sum, 128-byte row stores.
//
// Measured on B200 (tools/attn_probe.py, batch 256, 12 heads; tools/attn_trace-style timelines and the
// PSV_ATTN_DEBUG phase-skipping bits gave the breakdown): 55 us at n = 128 and 149 us at n = 197 against 78 / 217 us
// for the warp-level mma.sync kernel (attention_mma.cu); below ~70 tokens per image a 128-row tile is mostly
// padding and the per-tile dependency chain (TMA -> S -> softmax -> P V -> store) dominates, so launch_attention
// (psv_api.cu) uses the mma.sync kernel there.  At n = 197 the phases are: loads 49 us (the 232 MB of Q/K/V
// exceed L2), MMA issue + latency 26 us, softmax 62 us of which 39 us is the MUFU floor of the exponentials
// (16 ex2 / clk / SM), O epilogue 13 us; with only two 256-column TMEM buffers the phases of the two tiles of
// an image run in lock step instead of overlapping, which is what separates 149 us from the ~60 us floor.
//
// Rows / keys past n are garbage that is either masked (keys: -inf before the max, P = 0) or never stored
// (queries).  V rows past n are multiplied by P = 0, so they must be finite: they are rows of the same
// activation buffer (written by the QKV GEMM, zero-initialised at psv_create) or TMA out-of-bounds zeros.
#include <cstdlib>

#include "tc_common.cuh"

namespace psv {
namespace {

using namespace tc;

constexpr int AT_WG = 2;                          // softmax warpgroups == TMEM buffers
constexpr int AT_THREADS = 64 + AT_WG * 128;      // 320 -> up to 168 registers per thread
constexpr int AT_KV_ROWS = 224;                   // 197 keys rounded up to 32
constexpr int AT_NQK = 2, AT_NV = 3;
constexpr int AT_Q_BYTES = 128 * 128;             // one 128-row query tile
constexpr int AT_KV_BYTES = AT_KV_ROWS * 128;     // 28 KB
constexpr int AT_QK_BYTES = 2 * AT_Q_BYTES + AT_KV_BYTES;      // Q tile 0 | Q tile 1 | K : 60 KB
constexpr int AT_V_BASE = AT_NQK * AT_QK_BYTES;                // 120 KB
constexpr int AT_BAR_OFF = AT_V_BASE + AT_NV * AT_KV_BYTES;    // 204 KB
constexpr int AT_BAR_BYTES = 256;
constexpr int AT_SMEM = AT_BAR_OFF + AT_BAR_BYTES + 1024 /*align slack*/;   // + the cu_seqlens table when it fits
constexpr int AT_SMEM_MAX = 232448;               // 227 KB
constexpr int AT_BUF_COLS = 256;                  // per buffer: S at +0 (<= 224), P at +0 (<= 112), O at +128 (64)
constexpr int AT_O_COL = 128;
constexpr int AT_TMEM_COLS = AT_WG * AT_BUF_COLS; // 512

// Work unit = one (image, head): K and V are staged once and shared by its one or two 128-row query tiles.
struct Unit {
  int row0;    // first packed row of the image
  int n;       // active tokens of the image
  int head;
  int ntiles;  // query tiles: 1 (n <= 128) or 2
  int ncols;   // S columns = MMA N of S = contraction length of P V (n rounded up to 32)
};

__device__ __forceinline__ bool decode_unit(int u, int batch, const int32_t *cu, Unit &U) {
  const int b = u % batch;
  U.head = u / batch;
  U.row0 = cu[b];
  U.n = min(cu[b + 1] - U.row0, AT_KV_ROWS);
  U.ntiles = U.n > 128 ? 2 : 1;
  U.ncols = (U.n + 31) & ~31;
  return U.n > 0;
}

__device__ __forceinline__ uint32_t idesc_rt(int n, uint32_t b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}
// MN-major, 128B-swizzled B operand (V: rows = keys = contraction index, 64 dims = 128 bytes per row): the
// canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units (cute::UMMA make_umma_desc<Major::MN>) --
// 8 key rows of 128 bytes form one swizzle atom, atoms of consecutive 8-key groups are SBO = 1024 bytes apart;
// LBO (stride between 64-element blocks along N) is unused for N = 64.
__device__ __forceinline__ uint64_t make_sw128_mn_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {       // non-blocking
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// one lane polls, the warp then re-converges: 16 softmax warps hammering the same mbarrier with try_wait from all
// 32 lanes each slows the whole SM down (the polling competes with the working warps for issue slots)
__device__ __forceinline__ void mbar_wait_warp(uint64_t *bar, uint32_t parity, int lane) {
  if (lane == 0) mbar_wait(bar, parity);
  __syncwarp();
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}

constexpr float kScaleLog2 = 0.125f * 1.4426950408889634f;     // 1/sqrt(64) * log2(e)
constexpr float kLazyLog2 = 8.0f;                              // rescale only when the max grows by more than 2^8

__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float &lo, float &hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {      // Blackwell FFMA2
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// max over 32 consecutive keys of which the first `r` are real (PARTIAL: r < 32, possibly <= 0); four chains
template <bool PARTIAL>
__device__ __forceinline__ float chunk_max(const uint32_t (&v)[32], int r) {
  float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    m0 = fmaxf(m0, (!PARTIAL || i < r) ? __uint_as_float(v[i]) : -INFINITY);
    m1 = fmaxf(m1, (!PARTIAL || i + 1 < r) ? __uint_as_float(v[i + 1]) : -INFINITY);
    m2 = fmaxf(m2, (!PARTIAL || i + 2 < r) ? __uint_as_float(v[i + 2]) : -INFINITY);
    m3 = fmaxf(m3, (!PARTIAL || i + 3 < r) ? __uint_as_float(v[i + 3]) : -INFINITY);
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}
// p = 2^(s * c - ms) for 32 keys -> 16 packed bf16 pairs (keys past the first r give 0); returns the row-sum share.
// The sum is taken over the ROUNDED probabilities, so P / sum stays normalised: with the lazy reference max the
// dominant term is not exactly 1.0 and its bf16 rounding error would otherwise reach the output.  Scaling and the
// sums run on packed fp32x2 (FFMA2 / FADD2): the phase is issue-bound, not MUFU-bound.
template <bool PARTIAL>
__device__ __forceinline__ float chunk_exp(const uint32_t (&v)[32], int r, float ms, uint32_t (&pk)[16]) {
  const uint64_t c2 = pack_f32x2(kScaleLog2, kScaleLog2), ms2 = pack_f32x2(-ms, -ms);
  uint64_t acc0 = pack_f32x2(0.f, 0.f), acc1 = acc0;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    if (PARTIAL && 2 * i >= r) { pk[i] = 0u; continue; }     // padded keys (warp-uniform): no exponentials at all
    float x0, x1;
    unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), c2, ms2), x0, x1);
    float p0 = ex2f(x0), p1 = ex2f(x1);
    if (PARTIAL) {
      if (2 * i + 1 >= r) p1 = 0.f;
    }
    pk[i] = pack_bf16x2(p0, p1);
    const uint64_t rounded = pack_f32x2(__uint_as_float(pk[i] << 16), __uint_as_float(pk[i] & 0xffff0000u));
    if (i & 1) acc1 = add_f32x2(acc1, rounded); else acc0 = add_f32x2(acc0, rounded);
  }
  float a, b;
  unpack_f32x2(add_f32x2(acc0, acc1), a, b);
  return a + b;
}

__global__ void __launch_bounds__(AT_THREADS, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap map32, const __grid_constant__ CUtensorMap map64,
                    const __grid_constant__ CUtensorMap map128, const __grid_constant__ CUtensorMap map160,
                    const __grid_constant__ CUtensorMap map192, const __grid_constant__ CUtensorMap map224,
                    bf16 *__restrict__ ctx, const int32_t *__restrict__ cu_global, int batch, int H, int D,
                    int cu_in_smem, int dbg, long long *__restrict__ trace) {
  extern __shared__ uint8_t smem_raw[];
  // optional timeline of CTA 0 (PSV_ATTN_TRACE=1): [role][event] = (tag, globaltimer ns)
  int trace_n = 0;
#define TR(role, tag)                                                                     \
  do {                                                                                    \
    if (trace && blockIdx.x == 0 && trace_n < 250) {                                      \
      long long t__;                                                                      \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t__));                             \
      trace[((role) * 256 + trace_n) * 2] = (tag); trace[((role) * 256 + trace_n) * 2 + 1] = t__; ++trace_n; \
    }                                                                                     \
  } while (0)
  if (threadIdx.x == 0) TR(0, 1);
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + AT_BAR_OFF);
  uint64_t *qk_full = bars;                          // [NQK] Q tiles and K landed
  uint64_t *qk_empty = qk_full + AT_NQK;             // [NQK] S of the unit's last tile retired
  uint64_t *v_full = qk_empty + AT_NQK;              // [NV]  V landed
  uint64_t *v_empty = v_full + AT_NV;                // [NV]  P V of the unit's last tile retired
  uint64_t *s_full = v_empty + AT_NV;                // [WG]  S complete in TMEM
  uint64_t *p_full = s_full + AT_WG;                 // [WG]  P written to TMEM by the 4 softmax warps
  uint64_t *o_full = p_full + AT_WG;                 // [WG]  O complete in TMEM
  uint64_t *buf_free = o_full + AT_WG;               // [WG]  O drained by the 4 softmax warps
  uint64_t *sm_done = buf_free + AT_WG;              // [WG]  softmax of a tile finished (ping-pong token)
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(sm_done + AT_WG);
  int *max_n_s = reinterpret_cast<int *>(tmem_slot + 1);
  int32_t *cu_table = reinterpret_cast<int32_t *>(smem + AT_BAR_OFF + AT_BAR_BYTES);
  // every role walks the same static unit list; the row offsets are staged in shared memory so the walk costs a
  // few shared loads per unit instead of two dependent global loads
  const int32_t *cu_seqlens = cu_in_smem ? cu_table : cu_global;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_units = H * batch;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map128) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map224) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < AT_NQK; ++i) { mbar_init(&qk_full[i], 1); mbar_init(&qk_empty[i], 1); }
      for (int i = 0; i < AT_NV; ++i) { mbar_init(&v_full[i], 1); mbar_init(&v_empty[i], 1); }
      for (int i = 0; i < AT_WG; ++i) {
        mbar_init(&s_full[i], 1); mbar_init(&p_full[i], 4); mbar_init(&o_full[i], 1); mbar_init(&buf_free[i], 4);
        mbar_init(&sm_done[i], 4);
      }
      *max_n_s = 0;
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_slot)), "n"(AT_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  pdl_wait();                                       // qkv / cu_seqlens come from earlier kernels
  __syncthreads();
  {
    // stage the row offsets and find the longest image
    int mx = 0;
    for (int e = threadIdx.x; e <= batch; e += AT_THREADS) {
      const int c = cu_global[e];
      if (cu_in_smem) cu_table[e] = c;
      if (e < batch) mx = max(mx, cu_global[e + 1] - c);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0 && mx > 0) atomicMax(max_n_s, mx);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Ping-pong (the two warpgroups take turns in the softmax phase) pays when every image is a single tile: the
  // tiles of consecutive images then alternate between the warpgroups and one runs its softmax at full speed while
  // the other sits in its MMA waits / O epilogue (n = 128: 60 -> 55 us).  With two-tile images both tiles of an
  // image start together and two warps per scheduler fill the MUFU pipe better than one (n = 197: 158 -> 149 us
  // without it).  The mode must be uniform over the launch (a skipped wait would alias the barrier parity).
  const bool pingpong = *max_n_s <= 128 && !(dbg & 64);

  if (warp == 0) {
    // ===== TMA producer (whole warp, one elected lane issues: see the MMA issuer below) =====
    {
      const uint32_t FULL = 0xffffffffu;
      int qs = 0, vs = 0; uint32_t qph = 0, vph = 0;
      for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
        const int b = u % batch, head = u / batch;
        const int row0 = __shfl_sync(FULL, cu_seqlens[b], 0);
        const int n = min(__shfl_sync(FULL, cu_seqlens[b + 1], 0) - row0, AT_KV_ROWS);
        if (n <= 0) continue;
        uint8_t *sq = smem + qs * AT_QK_BYTES, *sk = sq + 2 * AT_Q_BYTES, *sv = smem + AT_V_BASE + vs * AT_KV_BYTES;
        const int nc = (n + 31) & ~31;
        const int kbox = nc <= 32 ? 32 : (nc <= 64 ? 64 : (nc <= 128 ? 128 : nc));
        const CUtensorMap *mk = nc <= 32 ? &map32 : (nc <= 64 ? &map64 : (nc <= 128 ? &map128 :
                                (nc == 160 ? &map160 : (nc == 192 ? &map192 : &map224))));
        const int q0rows = min(128, n);
        const int q0box = q0rows <= 32 ? 32 : (q0rows <= 64 ? 64 : 128);
        const CUtensorMap *mq0 = q0rows <= 32 ? &map32 : (q0rows <= 64 ? &map64 : &map128);
        const int q1rows = n - 128;                    // second query tile (69 rows for 197 tokens)
        const int q1box = n <= 128 ? 0 : (q1rows <= 32 ? 32 : (q1rows <= 64 ? 64 : 128));
        const CUtensorMap *mq1 = q1rows <= 32 ? &map32 : (q1rows <= 64 ? &map64 : &map128);
        const int hd = head * 64;
        mbar_wait(&qk_empty[qs], qph ^ 1);
        if (elect_one()) {
          TR(0, 10);
          mbar_arrive_expect_tx(&qk_full[qs], (uint32_t)(q0box + q1box + kbox) * 128u);
          tma_load_2d(sq, mq0, &qk_full[qs], hd, row0);
          tma_load_2d(sk, mk, &qk_full[qs], D + hd, row0);
          if (q1box) tma_load_2d(sq + AT_Q_BYTES, mq1, &qk_full[qs], hd, row0 + 128);
        }
        __syncwarp();
        mbar_wait(&v_empty[vs], vph ^ 1);
        if (elect_one()) {
          TR(0, 11);
          mbar_arrive_expect_tx(&v_full[vs], (uint32_t)kbox * 128u);
          tma_load_2d(sv, mk, &v_full[vs], 2 * D + hd, row0);
        }
        __syncwarp();
        if (++qs == AT_NQK) { qs = 0; qph ^= 1; }
        if (++vs == AT_NV) { vs = 0; vph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: two cursors over the (unit, tile) list -- next S, next P V -- issue whichever is ready.
    // The WHOLE warp runs this loop with warp-uniform control flow and warp-uniform operands (shuffle broadcasts,
    // votes), and one elected lane executes the tcgen05 instructions: the compiler then keeps descriptors in
    // uniform registers and the MMAs issue back to back.  (Under `if (lane == 0)` every tcgen05.mma is wrapped in
    // an ELECT / R2UR waterfall loop of ~150 cycles, which serialised the 18 MMAs of a tile to ~1.4 us.)
    {
      const uint32_t FULL = 0xffffffffu;
      const uint32_t tmem_u = __shfl_sync(FULL, tmem_base, 0);
      const uint32_t idesc_o = idesc_rt(64, 1u);     // O = P V : N = 64 dims, B (V) MN-major
      // One cursor per softmax warpgroup / TMEM buffer.  Unit i of the CTA's list belongs to warpgroup i & 1 and BOTH of its
      // query tiles run on that warpgroup's buffer, one after the other; the two warpgroups therefore work on different
      // images and drift into different phases, so the S / P V MMAs and the O epilogue of one overlap the softmax of the
      // other.  (Putting the two tiles of one image on the two buffers -- the earlier scheme -- ran every image as
      // S -> softmax -> P V -> O in lock step with nothing of the next image in flight: 7 us per image against ~3.)
      struct Cur { int u, unit, tile, jw, ncols, ntiles, stage; bool ok; };   // list position, unit index, tile, tiles done on this buffer
      auto settle = [&](Cur &c, int wg) {             // move to the next existing unit of warpgroup wg at or after c.u
        c.ok = false;
        for (; c.u < total_units; c.u += gridDim.x) {
          const int b = c.u % batch;
          const int n = min(__shfl_sync(FULL, cu_seqlens[b + 1] - cu_seqlens[b], 0), AT_KV_ROWS);
          if (n <= 0) continue;
          if ((c.unit & 1) == wg) { c.ncols = (n + 31) & ~31; c.ntiles = n > 128 ? 2 : 1; c.ok = true; break; }
          ++c.unit;
        }
      };
      Cur cur[AT_WG];
      for (int w = 0; w < AT_WG; ++w) {
        cur[w] = Cur{(int)blockIdx.x, 0, 0, 0, 0, 0, 0, false};
        settle(cur[w], w);
      }
      while (cur[0].ok || cur[1].ok) {
        bool issued = false;
#pragma unroll
        for (int w = 0; w < AT_WG; ++w) {
          Cur &c = cur[w];
          if (!c.ok) continue;
          if (c.stage == 0) {
            const int qs = c.unit % AT_NQK;
            const bool ready = mbar_test(&qk_full[qs], (uint32_t)(c.unit / AT_NQK) & 1u) &&
                               (c.jw == 0 || mbar_test(&buf_free[w], (uint32_t)(c.jw - 1) & 1u));
            if (__all_sync(FULL, ready)) {
              tc_fence_after();
              if (elect_one()) {
                const uint32_t sq = smem_u32(smem + qs * AT_QK_BYTES);
                const uint64_t da = make_sw128_desc(sq + c.tile * AT_Q_BYTES), db = make_sw128_desc(sq + 2 * AT_Q_BYTES);
                const uint32_t idesc_s = idesc_rt(c.ncols, 0u);
                const uint32_t t_s = tmem_u + w * AT_BUF_COLS;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (!(dbg & 8)) umma_bf16(t_s, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc_s, k ? 1u : 0u);
                if (c.tile + 1 == c.ntiles) umma_commit(&qk_empty[qs]);
                umma_commit(&s_full[w]);
                TR(1, 20 + w);
              }
              __syncwarp();
              c.stage = 1;
              issued = true;
            }
          } else {
            const int vs = c.unit % AT_NV;
            const bool ready = mbar_test(&p_full[w], (uint32_t)c.jw & 1u) &&
                               mbar_test(&v_full[vs], (uint32_t)(c.unit / AT_NV) & 1u);
            if (__all_sync(FULL, ready)) {
              tc_fence_after();
              if (elect_one()) {
                const uint32_t t_p = tmem_u + w * AT_BUF_COLS, t_o = t_p + AT_O_COL;
                const uint64_t dv = make_sw128_mn_desc(smem_u32(smem + AT_V_BASE + vs * AT_KV_BYTES));
                const int ksteps = c.ncols >> 4;        // 16 keys per MMA: 8 packed TMEM columns of P, 2 KB of V rows
#pragma unroll 2
                for (int k = 0; k < ksteps; ++k)
                  if (!(dbg & 4)) umma_bf16_ts(t_o, t_p + k * 8, dv + (uint64_t)(k * 128), idesc_o, k ? 1u : 0u);
                if (c.tile + 1 == c.ntiles) umma_commit(&v_empty[vs]);
                umma_commit(&o_full[w]);
                TR(1, 24 + w);
              }
              __syncwarp();
              c.stage = 0;
              ++c.jw;
              if (++c.tile == c.ntiles) {                // next unit of this warpgroup
                c.tile = 0; ++c.unit; c.u += gridDim.x;
                settle(c, w);
              }
              issued = true;
            }
          }
        }
        if (!issued && !(dbg & 128)) __nanosleep(32);   // nothing ready: do not steal issue slots from the softmax warps
      }
    }
  } else {
    // ===== softmax warpgroups: thread <-> S row (TMEM lane), warp <-> lane quadrant warp % 4 =====
    const int wg = (warp - 2) >> 2, quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t t_buf = tmem_base + ((uint32_t)(quad * 32) << 16) + wg * AT_BUF_COLS;
    int jw = 0, unit = 0;                             // tiles done by this warpgroup; index of the unit in the CTA's list
    Unit U;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
      if (!decode_unit(u, batch, cu_seqlens, U)) continue;
      const bool mine = (unit & 1) == wg;             // unit i and both of its tiles belong to warpgroup i & 1
      const int j = unit++;
      if (!mine) continue;
      for (int tile = 0; tile < U.ntiles; ++tile, ++jw) {
        const uint32_t ph = (uint32_t)jw & 1u;
        const int q = tile * 128 + row;
        const bool warp_on = tile * 128 + quad * 32 < U.n;       // some row of this warp is a real query
        const bool row_ok = q < U.n;
        float l = 0.f;
        mbar_wait_warp(&s_full[wg], ph, lane);
        if (quad == 0 && lane == 0) TR(2 + wg, 30);
        // single-tile images only (pingpong): unit j waits for the softmax of unit j-1 on the other warpgroup
        if (pingpong && j > 0) mbar_wait_warp(&sm_done[wg ^ 1], (uint32_t)((j - 1) >> 1) & 1u, lane);
        tc_fence_after();
        if (quad == 0 && lane == 0) TR(2 + wg, 31);
        if (warp_on && !(dbg & 1)) {
          const uint32_t t_s = t_buf, t_p = t_buf;
          const int nch = U.ncols >> 5, nv = U.n;
          uint32_t va[32], vb[32], pk[16];
          float m = -INFINITY;                         // reference max of the row (moves lazily)
          // one chunk: max -> (lazy reference move) -> exp / sum -> bf16 P chunk.  P chunk cc (16 columns at
          // 16cc) only overwrites S columns of chunks <= cc/2, all consumed by then.
          auto consume = [&](uint32_t (&v)[32], int cc) {
            if (dbg & 16) return;
            const int r = nv - cc * 32;                // real keys in this chunk; only the last chunk is partial
            const float mc = r >= 32 ? chunk_max<false>(v, r) : chunk_max<true>(v, r);
            if (cc == 0) {
              m = mc;
            } else if (__any_sync(0xffffffffu, (mc - m) * kScaleLog2 > kLazyLog2)) {
              // rare: some row's max grew by more than 2^8 -> move its reference and rescale what it wrote
              tmem_st_wait();                          // the P chunks read back below were stored asynchronously
              const bool mv = (mc - m) * kScaleLog2 > kLazyLog2;
              const float f = mv ? ex2f((m - mc) * kScaleLog2) : 1.0f;
              if (mv) m = mc;
              l *= f;
              for (int pc = 0; pc < cc; ++pc) {
                uint32_t w[16];
                tmem_ld16(t_p + pc * 16, w);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&w[e]));
                  w[e] = pack_bf16x2(f2.x * f, f2.y * f);
                }
                tmem_st16(t_p + pc * 16, w);
              }
            }
            if (dbg & 32) {
#pragma unroll
              for (int e = 0; e < 16; ++e) pk[e] = v[e];
            } else {
              l += r >= 32 ? chunk_exp<false>(v, r, m * kScaleLog2, pk) : chunk_exp<true>(v, r, m * kScaleLog2, pk);
            }
            tmem_st16(t_p + cc * 16, pk);
          };
          // rolling double buffer: chunk c is consumed from va (c even) / vb (c odd) while chunk c+1 is in
          // flight; tcgen05.wait::ld waits for ALL outstanding loads, so exactly one is outstanding at each wait
          tmem_ld32(t_s, va);
          tmem_ld_wait();
          if (nch > 1) tmem_ld32(t_s + 32, vb);
          for (int c = 0; c < nch; c += 2) {
            consume(va, c);
            if (c + 1 < nch) {
              tmem_ld_wait();
              if (c + 2 < nch) tmem_ld32(t_s + (c + 2) * 32, va);
              consume(vb, c + 1);
              if (c + 2 < nch) {
                tmem_ld_wait();
                if (c + 3 < nch) tmem_ld32(t_s + (c + 3) * 32, vb);
              }
            }
          }
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { mbar_arrive(&p_full[wg]); mbar_arrive(&sm_done[wg]); }
        if (quad == 0 && lane == 0) TR(2 + wg, 32);
        // ---- O epilogue
        mbar_wait_warp(&o_full[wg], ph, lane);
        tc_fence_after();
        if (quad == 0 && lane == 0) TR(2 + wg, 33);
        if (warp_on && !(dbg & 2)) {
          uint32_t o0[32], o1[32];
          tmem_ld32(t_buf + AT_O_COL, o0);
          tmem_ld32(t_buf + AT_O_COL + 32, o1);
          tmem_ld_wait();
          // O is in registers: hand the TMEM buffer back now, so the next S overlaps the scaling and the stores
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&buf_free[wg]);
          if (row_ok) {
            const float inv = 1.0f / l;
            uint4 *dst = reinterpret_cast<uint4 *>(ctx + (size_t)(U.row0 + q) * D + U.head * 64);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              uint4 w;
              w.x = pack_bf16x2(__uint_as_float(o0[8 * e]) * inv, __uint_as_float(o0[8 * e + 1]) * inv);
              w.y = pack_bf16x2(__uint_as_float(o0[8 * e + 2]) * inv, __uint_as_float(o0[8 * e + 3]) * inv);
              w.z = pack_bf16x2(__uint_as_float(o0[8 * e + 4]) * inv, __uint_as_float(o0[8 * e + 5]) * inv);
              w.w = pack_bf16x2(__uint_as_float(o0[8 * e + 6]) * inv, __uint_as_float(o0[8 * e + 7]) * inv);
              dst[e] = w;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              uint4 w;
              w.x = pack_bf16x2(__uint_as_float(o1[8 * e]) * inv, __uint_as_float(o1[8 * e + 1]) * inv);
              w.y = pack_bf16x2(__uint_as_float(o1[8 * e + 2]) * inv, __uint_as_float(o1[8 * e + 3]) * inv);
              w.z = pack_bf16x2(__uint_as_float(o1[8 * e + 4]) * inv, __uint_as_float(o1[8 * e + 5]) * inv);
              w.w = pack_bf16x2(__uint_as_float(o1[8 * e + 6]) * inv, __uint_as_float(o1[8 * e + 7]) * inv);
              dst[4 + e] = w;
            }
          }
        }
        if (!(warp_on && !(dbg & 2))) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&buf_free[wg]);
        }
        if (quad == 0 && lane == 0) TR(2 + wg, 34);
      }
    }
  }
#undef TR

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(AT_TMEM_COLS) : "memory");
  }
}

}  // namespace

cudaError_t configure_attention_tc() {
  return cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_MAX);
}

// qkv: [qkv_rows, 3D] bf16 packed activations (row = [q | k | v], heads along columns); ctx: [*, D] bf16
cudaError_t launch_attention_tc(PsvHandle *h, const void *qkv, void *ctx, const int32_t *cu_seqlens, int batch,
                                int64_t qkv_rows, cudaStream_t s) {
  if (h->N > AT_KV_ROWS) return cudaErrorInvalidValue;
  CUtensorMap m[6];
  const uint32_t boxes[6] = {32, 64, 128, 160, 192, AT_KV_ROWS};
  for (int i = 0; i < 6; ++i) {
    cudaError_t e = get_tmap_2d(h->tmaps, qkv, (uint64_t)qkv_rows, (uint64_t)3 * h->D, boxes[i], 64, 2, 128, &m[i]);
    if (e != cudaSuccess) return e;
  }
  LaunchScope scope(h, KK_ATTENTION, s);
  const int units = h->H * batch;
  const int grid = units < h->sm_count ? units : h->sm_count;
  const size_t table = ((size_t)(batch + 1) * sizeof(int32_t) + 15) & ~(size_t)15;
  const int cu_in_smem = AT_SMEM + table <= (size_t)AT_SMEM_MAX;
  static const int dbg = getenv("PSV_ATTN_DEBUG") ? atoi(getenv("PSV_ATTN_DEBUG")) : 0;   // timing experiments only
  static const bool want_trace = getenv("PSV_ATTN_TRACE") != nullptr;
  static long long *trace = nullptr;
  if (want_trace) {
    if (!trace) cudaMalloc(&trace, 4 * 256 * 2 * sizeof(long long));
    cudaMemsetAsync(trace, 0, 4 * 256 * 2 * sizeof(long long), s);
  }
  cudaError_t e = launch_pdl(attention_tc_kernel, dim3(grid), dim3(AT_THREADS),
                             (size_t)AT_SMEM + (cu_in_smem ? table : 0), s, m[0], m[1], m[2], m[3], m[4], m[5],
                             (bf16 *)ctx, cu_seqlens, batch, h->H, h->D, cu_in_smem, dbg, trace);
  if (want_trace && e == cudaSuccess) {               // debugging aid: dump the timeline of CTA 0 to stderr
    static long long host[4 * 256 * 2];
    cudaStreamSynchronize(s);
    cudaMemcpy(host, trace, sizeof host, cudaMemcpyDeviceToHost);
    const long long t0 = host[1];
    for (int r = 0; r < 4; ++r) {
      fprintf(stderr, "trace role %d:", r);
      for (int i = 0; i < 256 && host[(r * 256 + i) * 2]; ++i)
        fprintf(stderr, " %lld@%lld", host[(r * 256 + i) * 2], host[(r * 256 + i) * 2 + 1] - t0);
      fprintf(stderr, "\n");
    }
  }
  return e;
}

}  // namespace psv
