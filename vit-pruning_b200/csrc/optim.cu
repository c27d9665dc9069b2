// Optimizer step of backbone fine-tuning on the handle's own fp32 weights: torch.optim.Adam / AdamW (decoupled weight
// decay) from the flat gradient psv_backbone_backward writes, per-tensor step counters (0 = frozen), and a sharded
// data-parallel form over NVLink peer memory (each rank reduces and updates one contiguous slice of the flat vector, then
// the ranks copy each other's updated slices).
//
// The backbone weights stay separate allocations (the inference path reads them as they are), so the kernels walk a
// device table of segments {destination pointer, flat offset}, one per state-dict tensor in the order of the flat layout;
// the tensor index of a flat position is found by binary search over the offsets, kept in shared memory.  The
// per-tensor bias corrections and the decay factors travel as kernel parameters: nothing is uploaded per step, so a step
// only enqueues work and can be captured into a CUDA graph.
//
// Parameter groups: lr and weight decay may differ per tensor (psv_backbone_adam_step_groups); they only change the
// per-tensor kernel parameters below.  Global-norm clipping (torch.nn.utils.clip_grad_norm_) adds a norm pass before the
// update: fp64 partial sums of squares over a fixed block partition, summed in a fixed order (no atomics, so the bits do
// not depend on timing), and a clip coefficient in device memory that the update reads, so nothing waits on the host.
//
// Arithmetic (per element, fp32, in torch's order; the bias corrections are formed on the host in double as torch does):
//   g  = g * grad_scale [* coef]                   (coef = min(max_norm / (norm + 1e-6), 1) when clipping)
//   p *= 1 - lr * wd                               (AdamW; 1 for Adam, an exact no-op)
//   m  = m + (1 - b1) * (g - m)                    (exp_avg.lerp_(g, 1 - b1))
//   v  = v * b2 + (1 - b2) * g * g                 (exp_avg_sq.mul_(b2).addcmul_(g, g, value=1 - b2))
//   p += -(lr / bc1) * (m / (sqrt(v) * (1 / sqrt(bc2)) + eps))
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <vector>

#include "psv_internal.cuh"

namespace psv {

struct BackboneSeg { float *dst; int64_t off; };

struct BackboneOptim {
  int nt = 0;                          // tensors
  int64_t n = 0;                       // floats
  BackboneSeg *segs = nullptr;         // device [nt + 1]; segs[nt].off = n
  std::vector<BackboneSeg> host;       // the same table on the host (psv_get_backbone_params)
  float *m = nullptr, *v = nullptr;    // Adam moments [n] (lazy, zeroed)
  const float *bucket = nullptr;       // param_bucket of the last peer step (its gather must name it as peer_params[rank])
  int world = 0, rank = -1;
  double *partials = nullptr;          // device [2 * kNormBlocks]: per-block sums of squares of the norm pass
  float *coef = nullptr;               // device: clip coefficient of the last clipped step
  bool coef_covers_comp = false;       // that step's norm included the compressor gradient
  const float *reduced = nullptr;      // own gradient bucket of a psv_backbone_peer_reduce_sqnorm not yet consumed
  int reduced_world = 0, reduced_rank = -1;
  bool reduced_comp = false;           // that reduce's partial covered the compressor gradient
};

const float *backbone_clip_coef(const PsvHandle *h) {
  return h->bopt && h->bopt->coef_covers_comp ? h->bopt->coef : nullptr;
}

void backbone_optim_free(PsvHandle *h) {
  BackboneOptim *o = h->bopt;
  if (!o) return;
  cudaFree(o->segs); cudaFree(o->m); cudaFree(o->v); cudaFree(o->partials);
  delete o;
  h->bopt = nullptr;
}

namespace {

constexpr int kMaxTensors = 8 + 16 * 48;     // embeddings 4 + 16 per layer + head 4: up to 48 layers
constexpr int kNormBlocks = 1184;             // fixed grid of the norm pass (8 per SM of a B200), any device

struct AdamCoefs {                 // per tensor; live[t] == 0: frozen
  float step_size[kMaxTensors];    // lr / (1 - b1^step)
  float inv_bc2s[kMaxTensors];     // 1 / sqrt(1 - b2^step)
  float decay[kMaxTensors];        // 1 - lr * weight_decay
  uint8_t live[kMaxTensors];
};

struct PeerPtrs { const float *p[PSV_MAX_PEERS]; };

__device__ __forceinline__ void adam_elem(float &p, float &m, float &v, float g, float w1, float b2, float w2, float eps,
                                          float step_size, float inv_bc2s, float decay) {
  p = __fmul_rn(p, decay);
  m = fmaf(w1, g - m, m);
  v = fmaf(__fmul_rn(w2, g), g, __fmul_rn(v, b2));
  const float denom = __fadd_rn(__fmul_rn(sqrtf(v), inv_bc2s), eps);
  p = fmaf(-step_size, __fdiv_rn(m, denom), p);
}

// segment table into shared memory; returns the table's offsets / destinations
__device__ __forceinline__ void load_table(const BackboneSeg *__restrict__ segs, int nt, int64_t *s_off, float **s_dst) {
  for (int t = threadIdx.x; t <= nt; t += blockDim.x) {
    s_off[t] = segs[t].off;
    s_dst[t] = segs[t].dst;
  }
  __syncthreads();
}

// tensor holding flat position i: the largest t with s_off[t] <= i
__device__ __forceinline__ int find_tensor(const int64_t *s_off, int nt, int64_t i) {
  int lo = 0, hi = nt - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (s_off[mid] <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// The update of the flat range [lo, hi) (lo a multiple of 4).  kPeer: the gradient is the rank-order sum of the `world`
// buckets and the new value is also written to `bucket` (this rank's published shard; frozen tensors publish their
// unchanged value, so the gather never needs to know which tensors trained).
template <bool kPeer>
__global__ void __launch_bounds__(256)
backbone_adam_kernel(const BackboneSeg *__restrict__ segs, int nt, PeerPtrs grads, int world, float *__restrict__ bucket,
                     float *__restrict__ m, float *__restrict__ v, int64_t lo, int64_t hi, float w1, float b2, float w2,
                     float eps, float gscale, AdamCoefs c) {
  extern __shared__ int64_t s_off[];
  float **s_dst = reinterpret_cast<float **>(s_off + nt + 1);
  load_table(segs, nt, s_off, s_dst);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (int64_t i = lo + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < hi; i += stride) {
    const int t = find_tensor(s_off, nt, i);
    float *dst = s_dst[t] + (i - s_off[t]);
    if (i + 4 <= hi && i + 4 <= s_off[t + 1] && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
      if (!c.live[t]) {
        if (kPeer) *reinterpret_cast<float4 *>(bucket + i) = *reinterpret_cast<const float4 *>(dst);
        continue;
      }
      float4 g = reinterpret_cast<const float4 *>(grads.p[0])[i / 4];
      if (kPeer) {
#pragma unroll
        for (int r = 1; r < PSV_MAX_PEERS; ++r)
          if (r < world) {
            const float4 q = reinterpret_cast<const float4 *>(grads.p[r])[i / 4];     // peer loads go over NVLink
            g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
          }
      }
      float4 p = *reinterpret_cast<const float4 *>(dst);
      float4 mi = reinterpret_cast<const float4 *>(m)[i / 4], vi = reinterpret_cast<const float4 *>(v)[i / 4];
      float *ps = &p.x, *ms = &mi.x, *vs = &vi.x;
      const float *gs = &g.x;
#pragma unroll
      for (int e = 0; e < 4; ++e)
        adam_elem(ps[e], ms[e], vs[e], __fmul_rn(gs[e], gscale), w1, b2, w2, eps, c.step_size[t], c.inv_bc2s[t], c.decay[t]);
      *reinterpret_cast<float4 *>(dst) = p;
      reinterpret_cast<float4 *>(m)[i / 4] = mi;
      reinterpret_cast<float4 *>(v)[i / 4] = vi;
      if (kPeer) *reinterpret_cast<float4 *>(bucket + i) = p;
      continue;
    }
    for (int64_t k = i; k < i + 4 && k < hi; ++k) {      // a segment boundary, an unaligned segment or the tail
      const int tk = find_tensor(s_off, nt, k);
      float *d = s_dst[tk] + (k - s_off[tk]);
      if (!c.live[tk]) {
        if (kPeer) bucket[k] = *d;
        continue;
      }
      float g = grads.p[0][k];
      if (kPeer) {
#pragma unroll
        for (int r = 1; r < PSV_MAX_PEERS; ++r)
          if (r < world) g += grads.p[r][k];
      }
      float p = *d, mk = m[k], vk = v[k];
      adam_elem(p, mk, vk, __fmul_rn(g, gscale), w1, b2, w2, eps, c.step_size[tk], c.inv_bc2s[tk], c.decay[tk]);
      *d = p; m[k] = mk; v[k] = vk;
      if (kPeer) bucket[k] = p;
    }
  }
}

// The update with global-norm clipping: the scaled gradient is also multiplied by the coefficient of the norm pass
// (*clip, read once per thread), g = fp32(fp32(g * gscale) * coef) as clip_grad_norm_ before the optimizer.  A separate
// kernel, so that the unclipped steps keep their code.
template <bool kPeer>
__global__ void __launch_bounds__(256)
backbone_adam_clip_kernel(const BackboneSeg *__restrict__ segs, int nt, PeerPtrs grads, int world,
                          float *__restrict__ bucket, float *__restrict__ m, float *__restrict__ v, int64_t lo, int64_t hi,
                          float w1, float b2, float w2, float eps, float gscale, AdamCoefs c,
                          const float *__restrict__ clip) {
  extern __shared__ int64_t s_off[];
  float **s_dst = reinterpret_cast<float **>(s_off + nt + 1);
  load_table(segs, nt, s_off, s_dst);
  const float coef = *clip;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (int64_t i = lo + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < hi; i += stride) {
    const int t = find_tensor(s_off, nt, i);
    float *dst = s_dst[t] + (i - s_off[t]);
    if (i + 4 <= hi && i + 4 <= s_off[t + 1] && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
      if (!c.live[t]) {
        if (kPeer) *reinterpret_cast<float4 *>(bucket + i) = *reinterpret_cast<const float4 *>(dst);
        continue;
      }
      float4 g = reinterpret_cast<const float4 *>(grads.p[0])[i / 4];
      if (kPeer) {
#pragma unroll
        for (int r = 1; r < PSV_MAX_PEERS; ++r)
          if (r < world) {
            const float4 q = reinterpret_cast<const float4 *>(grads.p[r])[i / 4];     // peer loads go over NVLink
            g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
          }
      }
      float4 p = *reinterpret_cast<const float4 *>(dst);
      float4 mi = reinterpret_cast<const float4 *>(m)[i / 4], vi = reinterpret_cast<const float4 *>(v)[i / 4];
      float *ps = &p.x, *ms = &mi.x, *vs = &vi.x;
      const float *gs = &g.x;
#pragma unroll
      for (int e = 0; e < 4; ++e)
        adam_elem(ps[e], ms[e], vs[e], __fmul_rn(__fmul_rn(gs[e], gscale), coef), w1, b2, w2, eps, c.step_size[t],
                  c.inv_bc2s[t], c.decay[t]);
      *reinterpret_cast<float4 *>(dst) = p;
      reinterpret_cast<float4 *>(m)[i / 4] = mi;
      reinterpret_cast<float4 *>(v)[i / 4] = vi;
      if (kPeer) *reinterpret_cast<float4 *>(bucket + i) = p;
      continue;
    }
    for (int64_t k = i; k < i + 4 && k < hi; ++k) {      // a segment boundary, an unaligned segment or the tail
      const int tk = find_tensor(s_off, nt, k);
      float *d = s_dst[tk] + (k - s_off[tk]);
      if (!c.live[tk]) {
        if (kPeer) bucket[k] = *d;
        continue;
      }
      float g = grads.p[0][k];
      if (kPeer) {
#pragma unroll
        for (int r = 1; r < PSV_MAX_PEERS; ++r)
          if (r < world) g += grads.p[r][k];
      }
      float p = *d, mk = m[k], vk = v[k];
      adam_elem(p, mk, vk, __fmul_rn(__fmul_rn(g, gscale), coef), w1, b2, w2, eps, c.step_size[tk], c.inv_bc2s[tk],
                c.decay[tk]);
      *d = p; m[k] = mk; v[k] = vk;
      if (kPeer) bucket[k] = p;
    }
  }
}

struct LiveMask { uint8_t t[kMaxTensors]; };

__device__ __forceinline__ double sq(float g, float gscale) {
  const double x = __fmul_rn(g, gscale);
  return x * x;
}

// Sum of squares, in fp64, of the gradient Adam sees (fp32(g * gscale)) over the live tensors of the flat range
// [lo, hi) (lo a multiple of 4); writes one partial per block.  The grid is fixed (kNormBlocks) and so is every
// thread's share and the order of the block reduction: repeated runs give the same bits.  nt == 0: the flat
// compressor gradient, blocks of cstride floats per layer of which the first cper are parameters (the rest is padding,
// which the backward leaves unwritten and no norm counts).  kPeer: g is the rank-order fp32 sum of the `world` buckets (the same sum
// the fused update forms); kWriteBack: that sum is stored into `own` at the same position (this rank's own bucket,
// whose shard region no other rank reads), for the update pass.
template <bool kPeer, bool kWriteBack>
__global__ void __launch_bounds__(256)
grad_sqnorm_kernel(const BackboneSeg *__restrict__ segs, int nt, LiveMask live, PeerPtrs grads, int world, float *own,
                   int64_t lo, int64_t hi, float gscale, int cper, int cstride, double *__restrict__ partials) {
  extern __shared__ int64_t s_off[];
  if (nt > 0) {
    for (int t = threadIdx.x; t <= nt; t += blockDim.x) s_off[t] = segs[t].off;
    __syncthreads();
  }
  double acc = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (int64_t i = lo + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < hi; i += stride) {
    const int t = nt > 0 ? find_tensor(s_off, nt, i) : 0;
    if (i + 4 <= hi && (nt == 0 || i + 4 <= s_off[t + 1])) {
      if (nt > 0 && !live.t[t]) continue;
      float4 g = reinterpret_cast<const float4 *>(grads.p[0])[i / 4];
      if (kPeer) {
#pragma unroll
        for (int r = 1; r < PSV_MAX_PEERS; ++r)
          if (r < world) {
            const float4 q = reinterpret_cast<const float4 *>(grads.p[r])[i / 4];
            g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
          }
        if (kWriteBack) reinterpret_cast<float4 *>(own)[i / 4] = g;
      }
      if (nt == 0) {              // cstride is a multiple of 4: one layer block; the vector is far below 2^32 floats
        const int c = (int)((uint32_t)i % (uint32_t)cstride);
        if (c + 1 > cper) g.y = 0.0f;
        if (c + 2 > cper) g.z = 0.0f;
        if (c + 3 > cper) g.w = 0.0f;
        if (c >= cper) continue;
      }
      acc += sq(g.x, gscale) + sq(g.y, gscale) + sq(g.z, gscale) + sq(g.w, gscale);
      continue;
    }
    for (int64_t k = i; k < i + 4 && k < hi; ++k) {
      if (nt > 0 ? !live.t[find_tensor(s_off, nt, k)] : (int)((uint32_t)k % (uint32_t)cstride) >= cper) continue;
      float g = grads.p[0][k];
      if (kPeer) {
#pragma unroll
        for (int r = 1; r < PSV_MAX_PEERS; ++r)
          if (r < world) g += grads.p[r][k];
        if (kWriteBack) own[k] = g;
      }
      acc += sq(g, gscale);
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ double warp_sum[8];
  if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double b = 0.0;
    for (int w = 0; w < 8; ++w) b += warp_sum[w];
    partials[blockIdx.x] = b;
  }
}

struct SlotPtrs { const double *p[PSV_MAX_PEERS]; };

// One block: total = the np partials (fixed order) + the nslots slots (rank order).  Writes the total to sum_out, and
// with norm_out / coef the norm sqrt(total) and clip_grad_norm_'s coefficient min(max_norm / (fp32(norm) + 1e-6), 1)
// (a NaN norm gives a NaN coefficient, as torch's clamp does).
__global__ void __launch_bounds__(256)
sqnorm_finish_kernel(const double *__restrict__ partials, int np, SlotPtrs slots, int nslots, double *sum_out,
                     double *norm_out, float max_norm, float *coef) {
  __shared__ double red[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < np; i += blockDim.x) acc += partials[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int w = 128; w; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  double total = red[0];
#pragma unroll
  for (int r = 0; r < PSV_MAX_PEERS; ++r)              // unrolled: slots stays in the parameter bank
    if (r < nslots) total += *slots.p[r];
  if (sum_out) *sum_out = total;
  const double norm = sqrt(total);
  if (norm_out) *norm_out = norm;
  if (coef) {
    const float c = __fdiv_rn(max_norm, __fadd_rn((float)norm, 1e-6f));
    *coef = c > 1.0f ? 1.0f : c;
  }
}

// Copies every other rank's shard of the flat vector from that rank's parameter bucket into the weights.
struct ShardBounds { int64_t lo[PSV_MAX_PEERS + 1]; };
__global__ void __launch_bounds__(256)
backbone_gather_kernel(const BackboneSeg *__restrict__ segs, int nt, PeerPtrs params, ShardBounds sb, int world,
                       int rank) {
  extern __shared__ int64_t s_off[];
  float **s_dst = reinterpret_cast<float **>(s_off + nt + 1);
  load_table(segs, nt, s_off, s_dst);
  const int64_t n = sb.lo[world], stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    int r = 0;
    const float *src = params.p[0];                                  // shard bounds are multiples of 4
#pragma unroll
    for (int q = 1; q < PSV_MAX_PEERS; ++q)                          // unrolled: params stays in the parameter bank
      if (q < world && sb.lo[q] <= i) { r = q; src = params.p[q]; }
    if (r == rank) continue;
    const int t = find_tensor(s_off, nt, i);
    float *dst = s_dst[t] + (i - s_off[t]);
    if (i + 4 <= n && i + 4 <= s_off[t + 1] && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
      *reinterpret_cast<float4 *>(dst) = reinterpret_cast<const float4 *>(src)[i / 4];
      continue;
    }
    for (int64_t k = i; k < i + 4 && k < n; ++k) {
      const int tk = find_tensor(s_off, nt, k);
      s_dst[tk][k - s_off[tk]] = src[k];
    }
  }
}

int ofail(PsvHandle *h, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return code;
}

#define O_CUDA(h, call)                                                                                    \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess) return ofail(h, PSV_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); \
  } while (0)

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

void shard(int64_t n, int world, int rank, int64_t *lo, int64_t *hi) {
  const int64_t q = n / 4;
  *lo = 4 * (q * rank / world);
  *hi = rank == world - 1 ? n : 4 * (q * (rank + 1) / world);
}

int check_handle(PsvHandle *h) {
  if (!h) return PSV_ERR_INVALID;
  if (h->cfg.precision != PSV_FP32)
    return ofail(h, PSV_ERR_UNSUPPORTED, "the backbone optimizer runs on PSV_FP32 handles (fine-tuning runs there)");
  const int nt = 8 + 16 * h->L;
  if (nt > kMaxTensors) return ofail(h, PSV_ERR_UNSUPPORTED, "the backbone optimizer covers up to 48 layers");
  return PSV_OK;
}

// The segment table (built once per handle: the weights never move) and, with `moments`, the zeroed Adam moments.
int ensure_optim(PsvHandle *h, bool moments, cudaStream_t s) {
  if (!h->bopt) {
    BackboneOptim *o = new BackboneOptim();
    const int64_t D = h->D, F = h->F;
    int64_t off = 0;
    auto add = [&](float *dst, int64_t count) { o->host.push_back({dst, off}); off += count; };
    add(h->cls_token, D); add(h->pos_emb, (int64_t)h->N * D); add(h->patch_w, D * h->KP); add(h->patch_b, D);
    for (const LayerPack &lp : h->layers) {
      add(lp.ln1_w, D); add(lp.ln1_b, D);
      add(lp.wqkv, D * D); add(lp.wqkv + D * D, D * D); add(lp.wqkv + 2 * D * D, D * D);
      add(lp.bqkv, D); add(lp.bqkv + D, D); add(lp.bqkv + 2 * D, D);
      add(lp.wo, D * D); add(lp.bo, D);
      add(lp.ln2_w, D); add(lp.ln2_b, D);
      add(lp.w1, F * D); add(lp.b1, F);
      add(lp.w2, D * F); add(lp.b2, D);
    }
    add(h->final_ln_w, D); add(h->final_ln_b, D); add(h->cls_w, (int64_t)h->C * D); add(h->cls_b, h->C);
    o->nt = (int)o->host.size();
    o->n = off;
    o->host.push_back({nullptr, off});
    cudaError_t e = cudaMalloc((void **)&o->segs, o->host.size() * sizeof(BackboneSeg));
    if (e == cudaSuccess)
      e = cudaMemcpy(o->segs, o->host.data(), o->host.size() * sizeof(BackboneSeg), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc((void **)&o->partials, 2 * kNormBlocks * sizeof(double) + 16);
    if (e == cudaSuccess) o->coef = reinterpret_cast<float *>(o->partials + 2 * kNormBlocks);
    if (e != cudaSuccess) {
      cudaFree(o->segs);
      cudaFree(o->partials);
      delete o;
      return ofail(h, PSV_ERR_CUDA, "backbone optimizer table: %s", cudaGetErrorString(e));
    }
    h->bopt = o;
  }
  BackboneOptim *o = h->bopt;
  if (moments && !o->m) {
    const size_t bytes = (size_t)o->n * sizeof(float) + 256;
    O_CUDA(h, cudaMalloc((void **)&o->m, bytes));
    O_CUDA(h, cudaMalloc((void **)&o->v, bytes));
    O_CUDA(h, cudaMemsetAsync(o->m, 0, bytes, s));
    O_CUDA(h, cudaMemsetAsync(o->v, 0, bytes, s));
  }
  return PSV_OK;
}

// lr / weight_decay: host arrays, one entry per tensor
int make_coefs(PsvHandle *h, const int32_t *steps, const float *lr, float beta1, float beta2, const float *weight_decay,
               AdamCoefs *c) {
  if (!steps) return ofail(h, PSV_ERR_INVALID, "steps (host int32 array, one entry per backbone tensor) is required");
  for (int t = 0; t < h->bopt->nt; ++t) {
    if (steps[t] < 0) return ofail(h, PSV_ERR_INVALID, "steps[%d] = %d: steps are 1-based, 0 = frozen", t, steps[t]);
    c->live[t] = steps[t] > 0;
    const double st = steps[t] > 0 ? steps[t] : 1;
    const double bc1 = 1.0 - std::pow((double)beta1, st), bc2 = 1.0 - std::pow((double)beta2, st);
    c->step_size[t] = (float)((double)lr[t] / bc1);
    c->inv_bc2s[t] = 1.0f / (float)std::sqrt(bc2);
    c->decay[t] = (float)(1.0 - (double)lr[t] * (double)weight_decay[t]);
  }
  return PSV_OK;
}

// The scalar lr / weight decay of psv_backbone_adam_step as per-tensor arrays (the same coefficients bit for bit).
int make_coefs(PsvHandle *h, const int32_t *steps, float lr, float beta1, float beta2, float weight_decay,
               AdamCoefs *c) {
  const std::vector<float> lrs(h->bopt->nt, lr), wds(h->bopt->nt, weight_decay);
  return make_coefs(h, steps, lrs.data(), beta1, beta2, wds.data(), c);
}

int check_groups(PsvHandle *h, const float *lr, const float *weight_decay, float max_grad_norm) {
  if (!lr || !weight_decay)
    return ofail(h, PSV_ERR_INVALID, "lr and weight_decay (host float arrays, one entry per backbone tensor) are required");
  for (int t = 0; t < h->bopt->nt; ++t)
    if (!std::isfinite(lr[t]) || lr[t] < 0.0f || !std::isfinite(weight_decay[t]) || weight_decay[t] < 0.0f)
      return ofail(h, PSV_ERR_INVALID, "tensor %d: lr %g, weight_decay %g must be finite and >= 0", t, (double)lr[t],
                   (double)weight_decay[t]);
  if (!std::isfinite(max_grad_norm)) return ofail(h, PSV_ERR_INVALID, "max_grad_norm must be finite (<= 0: no clipping)");
  return PSV_OK;
}

LiveMask live_mask(const AdamCoefs &c, int nt) {
  LiveMask l{};
  for (int t = 0; t < nt; ++t) l.t[t] = c.live[t];
  return l;
}

int check_peers(PsvHandle *h, const float *const *peers, int world, const char *what) {
  if (!peers) return ofail(h, PSV_ERR_INVALID, "%s is required", what);
  for (int r = 0; r < world; ++r)
    if (!peers[r] || !aligned16(peers[r]))
      return ofail(h, PSV_ERR_INVALID, "%s[%d] must be non-null and 16-byte aligned", what, r);
  return PSV_OK;
}

int check_world(PsvHandle *h, int world, int rank) {
  if (world < 1 || world > PSV_MAX_PEERS) return ofail(h, PSV_ERR_INVALID, "world %d outside [1, %d]", world, PSV_MAX_PEERS);
  if (rank < 0 || rank >= world) return ofail(h, PSV_ERR_INVALID, "rank %d outside [0, %d)", rank, world);
  return PSV_OK;
}

// The norm pass over [lo, hi) of the backbone gradient (table) or of a flat vector (nt = 0), into `partials`.
int launch_sqnorm(PsvHandle *h, bool table, const LiveMask &live, const float *const *grads, int world, int rank,
                  bool write_back, int64_t lo, int64_t hi, float grad_scale, double *partials, cudaStream_t s) {
  BackboneOptim *o = h->bopt;
  PeerPtrs g{};
  for (int r = 0; r < world; ++r) g.p[r] = grads[r];
  const int nt = table ? o->nt : 0;
  const size_t smem = table ? (size_t)(o->nt + 1) * sizeof(int64_t) : 0;
  LaunchScope scope(h, KK_TRAIN, s);
  auto kernel = world == 1 && !write_back ? grad_sqnorm_kernel<false, false>
              : write_back ? grad_sqnorm_kernel<true, true> : grad_sqnorm_kernel<true, false>;
  const int cstride = (int)h->comp_per_layer, cper = (int)(2 * h->CH * h->D + 2 * h->CH + 1);
  kernel<<<kNormBlocks, 256, smem, s>>>(table ? o->segs : nullptr, nt, live, g, world, const_cast<float *>(grads[rank]),
                                        lo, hi, grad_scale, cper, cstride, partials);
  O_CUDA(h, cudaGetLastError());
  return PSV_OK;
}

int launch_finish(PsvHandle *h, int np, const double *const *slots, int nslots, double *sum_out, double *norm_out,
                  float max_grad_norm, bool clip, cudaStream_t s) {
  BackboneOptim *o = h->bopt;
  SlotPtrs sp{};
  for (int r = 0; r < nslots; ++r) sp.p[r] = slots[r];
  LaunchScope scope(h, KK_TRAIN, s);
  sqnorm_finish_kernel<<<1, 256, 0, s>>>(o->partials, np, sp, nslots, sum_out, norm_out, max_grad_norm,
                                         clip ? o->coef : nullptr);
  O_CUDA(h, cudaGetLastError());
  return PSV_OK;
}

int launch_update(PsvHandle *h, bool peer, const float *const *grads, int world, float *bucket, int64_t lo, int64_t hi,
                  float beta1, float beta2, float eps, float grad_scale, const AdamCoefs &c, cudaStream_t s,
                  const float *clip = nullptr) {
  BackboneOptim *o = h->bopt;
  PeerPtrs g{};
  for (int r = 0; r < world; ++r) g.p[r] = grads[r];
  const int64_t groups = (hi - lo + 3) / 4;
  int64_t grid = (groups + 255) / 256;
  if (grid > (int64_t)h->sm_count * 4) grid = (int64_t)h->sm_count * 4;
  if (grid < 1) grid = 1;
  const size_t smem = (size_t)(o->nt + 1) * sizeof(int64_t) + (size_t)(o->nt + 1) * sizeof(float *);
  LaunchScope scope(h, KK_TRAIN, s);
  if (clip) {
    auto kernel = peer ? backbone_adam_clip_kernel<true> : backbone_adam_clip_kernel<false>;
    kernel<<<(unsigned)grid, 256, smem, s>>>(o->segs, o->nt, g, world, bucket, o->m, o->v, lo, hi, 1.0f - beta1, beta2,
                                             1.0f - beta2, eps, grad_scale, c, clip);
  } else {
    auto kernel = peer ? backbone_adam_kernel<true> : backbone_adam_kernel<false>;
    kernel<<<(unsigned)grid, 256, smem, s>>>(o->segs, o->nt, g, world, bucket, o->m, o->v, lo, hi, 1.0f - beta1, beta2,
                                             1.0f - beta2, eps, grad_scale, c);
  }
  O_CUDA(h, cudaGetLastError());
  return PSV_OK;
}

}  // namespace
}  // namespace psv

using namespace psv;

extern "C" {
#pragma GCC visibility push(default)

int psv_backbone_shard(int64_t n, int32_t world, int32_t rank, int64_t *lo, int64_t *hi) {
  if (!lo || !hi || n < 0 || world < 1 || world > PSV_MAX_PEERS || rank < 0 || rank >= world) return PSV_ERR_INVALID;
  shard(n, world, rank, lo, hi);
  return PSV_OK;
}

int psv_backbone_adam_step(PsvHandle *h, const float *grads, const int32_t *steps, float lr, float beta1, float beta2,
                           float eps, float weight_decay, float grad_scale, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!grads || !aligned16(grads)) return ofail(h, PSV_ERR_INVALID, "grads must be non-null and 16-byte aligned");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, true, s))) return rc;
  AdamCoefs c;
  if ((rc = make_coefs(h, steps, lr, beta1, beta2, weight_decay, &c))) return rc;
  h->launches = 0;
  return launch_update(h, false, &grads, 1, nullptr, 0, h->bopt->n, beta1, beta2, eps, grad_scale, c, s);
}

int psv_backbone_peer_reduce_adam_step(PsvHandle *h, const float *const *peer_grads, float *param_bucket, int32_t world,
                                       int32_t rank, const int32_t *steps, float lr, float beta1, float beta2, float eps,
                                       float weight_decay, float grad_scale, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (world < 1 || world > PSV_MAX_PEERS) return ofail(h, PSV_ERR_INVALID, "world %d outside [1, %d]", world, PSV_MAX_PEERS);
  if (rank < 0 || rank >= world) return ofail(h, PSV_ERR_INVALID, "rank %d outside [0, %d)", rank, world);
  if (!peer_grads) return ofail(h, PSV_ERR_INVALID, "peer_grads is required");
  for (int r = 0; r < world; ++r)
    if (!peer_grads[r] || !aligned16(peer_grads[r]))
      return ofail(h, PSV_ERR_INVALID, "peer_grads[%d] must be non-null and 16-byte aligned", r);
  if (!param_bucket || !aligned16(param_bucket))
    return ofail(h, PSV_ERR_INVALID, "param_bucket must be non-null and 16-byte aligned");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, true, s))) return rc;
  AdamCoefs c;
  if ((rc = make_coefs(h, steps, lr, beta1, beta2, weight_decay, &c))) return rc;
  int64_t lo, hi;
  shard(h->bopt->n, world, rank, &lo, &hi);
  h->launches = 0;
  if ((rc = launch_update(h, true, peer_grads, world, param_bucket, lo, hi, beta1, beta2, eps, grad_scale, c, s))) return rc;
  h->bopt->bucket = param_bucket;
  h->bopt->world = world;
  h->bopt->rank = rank;
  return PSV_OK;
}

int psv_backbone_adam_step_groups(PsvHandle *h, const float *grads, const int32_t *steps, const float *lr,
                                  const float *weight_decay, float beta1, float beta2, float eps, float grad_scale,
                                  float max_grad_norm, const float *comp_grads, double *grad_norm_out, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!grads || !aligned16(grads)) return ofail(h, PSV_ERR_INVALID, "grads must be non-null and 16-byte aligned");
  if (comp_grads && !aligned16(comp_grads)) return ofail(h, PSV_ERR_INVALID, "comp_grads must be 16-byte aligned");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, true, s))) return rc;
  if ((rc = check_groups(h, lr, weight_decay, max_grad_norm))) return rc;
  AdamCoefs c;
  if ((rc = make_coefs(h, steps, lr, beta1, beta2, weight_decay, &c))) return rc;
  BackboneOptim *o = h->bopt;
  const bool clip = max_grad_norm > 0.0f;
  h->launches = 0;
  o->coef_covers_comp = false;
  if (clip || grad_norm_out) {
    const LiveMask live = live_mask(c, o->nt);
    if ((rc = launch_sqnorm(h, true, live, &grads, 1, 0, false, 0, o->n, grad_scale, o->partials, s))) return rc;
    int np = kNormBlocks;
    if (comp_grads) {
      const int64_t nc = psv_compressor_param_count(h);
      if ((rc = launch_sqnorm(h, false, live, &comp_grads, 1, 0, false, 0, nc, grad_scale, o->partials + kNormBlocks, s)))
        return rc;
      np += kNormBlocks;
    }
    if ((rc = launch_finish(h, np, nullptr, 0, nullptr, grad_norm_out, max_grad_norm, clip, s))) return rc;
    o->coef_covers_comp = clip && comp_grads;
  }
  return launch_update(h, false, &grads, 1, nullptr, 0, o->n, beta1, beta2, eps, grad_scale, c, s,
                       clip ? o->coef : nullptr);
}

int psv_backbone_peer_reduce_sqnorm(PsvHandle *h, const float *const *peer_grads, int32_t world, int32_t rank,
                                    const int32_t *steps, float grad_scale, const float *const *comp_peer_grads,
                                    double *sqnorm_slot, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_world(h, world, rank))) return rc;
  if ((rc = check_peers(h, peer_grads, world, "peer_grads"))) return rc;
  if (comp_peer_grads && (rc = check_peers(h, comp_peer_grads, world, "comp_peer_grads"))) return rc;
  if (!sqnorm_slot || (reinterpret_cast<uintptr_t>(sqnorm_slot) & 7u))
    return ofail(h, PSV_ERR_INVALID, "sqnorm_slot must be non-null and 8-byte aligned");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, true, s))) return rc;
  AdamCoefs c;
  if ((rc = make_coefs(h, steps, 0.0f, 0.9f, 0.999f, 0.0f, &c))) return rc;      // only the live flags are used
  BackboneOptim *o = h->bopt;
  const LiveMask live = live_mask(c, o->nt);
  int64_t lo, hi;
  shard(o->n, world, rank, &lo, &hi);
  h->launches = 0;
  if ((rc = launch_sqnorm(h, true, live, peer_grads, world, rank, true, lo, hi, grad_scale, o->partials, s))) return rc;
  int np = kNormBlocks;
  if (comp_peer_grads) {
    int64_t clo, chi;
    shard(psv_compressor_param_count(h), world, rank, &clo, &chi);
    if ((rc = launch_sqnorm(h, false, live, comp_peer_grads, world, rank, false, clo, chi, grad_scale,
                            o->partials + kNormBlocks, s)))
      return rc;
    np += kNormBlocks;
  }
  if ((rc = launch_finish(h, np, nullptr, 0, sqnorm_slot, nullptr, 0.0f, false, s))) return rc;
  o->reduced = peer_grads[rank];
  o->reduced_world = world;
  o->reduced_rank = rank;
  o->reduced_comp = comp_peer_grads != nullptr;
  return PSV_OK;
}

int psv_backbone_peer_adam_step_groups(PsvHandle *h, const float *const *peer_grads, float *param_bucket, int32_t world,
                                       int32_t rank, const int32_t *steps, const float *lr, const float *weight_decay,
                                       float beta1, float beta2, float eps, float grad_scale, float max_grad_norm,
                                       const double *const *peer_sqnorms, double *grad_norm_out, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_world(h, world, rank))) return rc;
  if ((rc = check_peers(h, peer_grads, world, "peer_grads"))) return rc;
  if (!param_bucket || !aligned16(param_bucket))
    return ofail(h, PSV_ERR_INVALID, "param_bucket must be non-null and 16-byte aligned");
  const bool clip = max_grad_norm > 0.0f;
  if (!peer_sqnorms && (clip || grad_norm_out))
    return ofail(h, PSV_ERR_INVALID, "clipping and the norm need psv_backbone_peer_reduce_sqnorm and peer_sqnorms");
  if (peer_sqnorms)
    for (int r = 0; r < world; ++r)
      if (!peer_sqnorms[r]) return ofail(h, PSV_ERR_INVALID, "peer_sqnorms[%d] is null", r);
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, true, s))) return rc;
  if ((rc = check_groups(h, lr, weight_decay, max_grad_norm))) return rc;
  BackboneOptim *o = h->bopt;
  if (peer_sqnorms && (o->reduced != peer_grads[rank] || o->reduced_world != world || o->reduced_rank != rank))
    return ofail(h, PSV_ERR_STATE, "peer_sqnorms given, but no psv_backbone_peer_reduce_sqnorm with these peer_grads, "
                 "world and rank precedes this step");
  AdamCoefs c;
  if ((rc = make_coefs(h, steps, lr, beta1, beta2, weight_decay, &c))) return rc;
  int64_t lo, hi;
  shard(o->n, world, rank, &lo, &hi);
  h->launches = 0;
  o->coef_covers_comp = false;
  if (peer_sqnorms) {         // the reduced shard is in this rank's own bucket: update from it alone
    if ((rc = launch_finish(h, 0, peer_sqnorms, world, nullptr, grad_norm_out, max_grad_norm, clip, s))) return rc;
    if ((rc = launch_update(h, true, &peer_grads[rank], 1, param_bucket, lo, hi, beta1, beta2, eps, grad_scale, c, s,
                            clip ? o->coef : nullptr)))
      return rc;
    o->coef_covers_comp = clip && o->reduced_comp;
    o->reduced = nullptr;
  } else if ((rc = launch_update(h, true, peer_grads, world, param_bucket, lo, hi, beta1, beta2, eps, grad_scale, c, s))) {
    return rc;
  }
  o->bucket = param_bucket;
  o->world = world;
  o->rank = rank;
  return PSV_OK;
}

int psv_backbone_peer_gather_params(PsvHandle *h, const float *const *peer_params, int32_t world, int32_t rank,
                                    void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (world < 1 || world > PSV_MAX_PEERS) return ofail(h, PSV_ERR_INVALID, "world %d outside [1, %d]", world, PSV_MAX_PEERS);
  if (rank < 0 || rank >= world) return ofail(h, PSV_ERR_INVALID, "rank %d outside [0, %d)", rank, world);
  if (!peer_params) return ofail(h, PSV_ERR_INVALID, "peer_params is required");
  for (int r = 0; r < world; ++r)
    if (!peer_params[r] || !aligned16(peer_params[r]))
      return ofail(h, PSV_ERR_INVALID, "peer_params[%d] must be non-null and 16-byte aligned", r);
  BackboneOptim *o = h->bopt;
  if (!o || !o->bucket) return ofail(h, PSV_ERR_STATE, "no psv_backbone_peer_reduce_adam_step on this handle yet");
  if (peer_params[rank] != o->bucket || world != o->world || rank != o->rank)
    return ofail(h, PSV_ERR_INVALID, "peer_params[rank], world and rank must be the param_bucket, world and rank of the "
                 "last psv_backbone_peer_reduce_adam_step");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  PeerPtrs p{};
  ShardBounds sb{};
  for (int r = 0; r < world; ++r) {
    p.p[r] = peer_params[r];
    int64_t hi;
    shard(o->n, world, r, &sb.lo[r], &hi);
  }
  sb.lo[world] = o->n;
  h->launches = 0;
  if (world == 1) return PSV_OK;
  int64_t grid = (o->n / 4 + 255) / 256;
  if (grid > (int64_t)h->sm_count * 4) grid = (int64_t)h->sm_count * 4;
  const size_t smem = (size_t)(o->nt + 1) * (sizeof(int64_t) + sizeof(float *));
  LaunchScope scope(h, KK_TRAIN, s);
  backbone_gather_kernel<<<(unsigned)(grid < 1 ? 1 : grid), 256, smem, s>>>(o->segs, o->nt, p, sb, world, rank);
  O_CUDA(h, cudaGetLastError());
  return PSV_OK;
}

int psv_get_backbone_params(PsvHandle *h, float *params_out, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (!params_out) return ofail(h, PSV_ERR_INVALID, "params_out is required");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, false, s))) return rc;
  const BackboneOptim *o = h->bopt;
  for (int t = 0; t < o->nt; ++t)
    O_CUDA(h, cudaMemcpyAsync(params_out + o->host[t].off, o->host[t].dst,
                              (size_t)(o->host[t + 1].off - o->host[t].off) * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return PSV_OK;
}

static int check_range(PsvHandle *h, int64_t offset, int64_t count) {
  const int64_t n = psv_backbone_param_count(h);
  if (offset < 0 || count < 0 || offset + count > n)
    return ofail(h, PSV_ERR_INVALID, "range [%lld, %lld) outside [0, %lld)", (long long)offset,
                 (long long)(offset + count), (long long)n);
  return PSV_OK;
}

int psv_get_backbone_adam_state(PsvHandle *h, int64_t offset, int64_t count, float *m_out, float *v_out, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_range(h, offset, count))) return rc;
  if (!m_out || !v_out) return ofail(h, PSV_ERR_INVALID, "m_out and v_out are required");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t bytes = (size_t)count * sizeof(float);
  if (!h->bopt || !h->bopt->m) {                    // no step taken yet: the moments are zero
    O_CUDA(h, cudaMemsetAsync(m_out, 0, bytes, s));
    O_CUDA(h, cudaMemsetAsync(v_out, 0, bytes, s));
    return PSV_OK;
  }
  O_CUDA(h, cudaMemcpyAsync(m_out, h->bopt->m + offset, bytes, cudaMemcpyDeviceToDevice, s));
  O_CUDA(h, cudaMemcpyAsync(v_out, h->bopt->v + offset, bytes, cudaMemcpyDeviceToDevice, s));
  return PSV_OK;
}

int psv_set_backbone_adam_state(PsvHandle *h, int64_t offset, int64_t count, const float *m, const float *v,
                                void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if ((rc = check_range(h, offset, count))) return rc;
  if (!m || !v) return ofail(h, PSV_ERR_INVALID, "m and v are required");
  DeviceGuard guard(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_optim(h, true, s))) return rc;
  const size_t bytes = (size_t)count * sizeof(float);
  O_CUDA(h, cudaMemcpyAsync(h->bopt->m + offset, m, bytes, cudaMemcpyDeviceToDevice, s));
  O_CUDA(h, cudaMemcpyAsync(h->bopt->v + offset, v, bytes, cudaMemcpyDeviceToDevice, s));
  return PSV_OK;
}

#pragma GCC visibility pop
}  // extern "C"
