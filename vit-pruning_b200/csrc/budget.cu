// Per-layer token budget (psv_set_token_budget): keep the k highest-scoring patches of every image.
//
// budget_mask_kernel: one CTA per image, one thread per patch token (N - 1 <= 255).  It reads the image's fp32
// compressor scores (what the score kernel left in h->scores, the values scores_out returns) into shared memory and
// ranks every token against all others:
//   rank(t) = #{u : s_u > s_t, or s_u == s_t and u < t}      (ties go to the lower index; NaN ranks below every number,
//                                                             NaNs among themselves by index)
// so the ranks are a permutation of 0..N-2 and the kept set does not depend on the thread schedule.
//   EXACT: mask[t] = rank(t) < k                  CAP: mask[t] = (s_t >= mt) && rank(t) < k
// CLS is always kept and not counted.  It overwrites the score kernel's mask and per-image count, which is all the
// compaction (gather_ln_kernel with per-image counts) reads.  No atomics: the count is a __syncthreads_count.
#include "psv_internal.cuh"

namespace psv {

namespace {

constexpr int BM_THREADS = 256;

// u outranks t
__device__ __forceinline__ bool outranks(float su, int u, float st, int t) {
  const bool nu = su != su, nt = st != st;
  if (nt) return !nu || u < t;
  return !nu && (su > st || (su == st && u < t));
}

template <bool CAP>
__global__ void __launch_bounds__(BM_THREADS)
budget_mask_kernel(const float *__restrict__ scores,     // [B, N-1]
                   int N, int k, float mt,
                   uint8_t *__restrict__ mask,            // [B, N] workspace
                   int32_t *__restrict__ n_active,        // [B]
                   uint8_t *__restrict__ mask_out) {      // nullable [B, N]
  __shared__ float ss[BM_THREADS];
  const int b = blockIdx.x, t = threadIdx.x, P = N - 1;
  pdl_wait();
  if (t < P) ss[t] = scores[(size_t)b * P + t];
  __syncthreads();
  bool keep = false;
  if (t < P) {
    const float s = ss[t];
    int rank = 0;
    for (int u = 0; u < P; ++u) rank += outranks(ss[u], u, s, t);      // false for u == t
    keep = rank < k && (!CAP || s >= mt);
  }
  const int count = __syncthreads_count(keep);
  if (t < P) {
    mask[(size_t)b * N + 1 + t] = keep;
    if (mask_out) mask_out[(size_t)b * N + 1 + t] = keep;
  }
  if (t == 0) {
    mask[(size_t)b * N] = 1;
    if (mask_out) mask_out[(size_t)b * N] = 1;
    n_active[b] = count + 1;
  }
}

}  // namespace

cudaError_t launch_budget_mask(PsvHandle *h, int layer, int batch, float mt, uint8_t *mask_out, cudaStream_t s) {
  LaunchScope scope(h, KK_BUDGET, s);
  if (h->N - 1 > BM_THREADS) return cudaErrorNotSupported;
  const int k = h->budget_keep[layer];
  if (h->budget_mode == PSV_BUDGET_CAP)
    return launch_pdl(budget_mask_kernel<true>, dim3(batch), dim3(BM_THREADS), 0, s, (const float *)h->scores, h->N, k,
                      mt, h->mask, h->n_active, mask_out);
  return launch_pdl(budget_mask_kernel<false>, dim3(batch), dim3(BM_THREADS), 0, s, (const float *)h->scores, h->N, k, mt,
                    h->mask, h->n_active, mask_out);
}

}  // namespace psv
