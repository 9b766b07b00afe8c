// Bin partition, points-per-bin allocation and per-bin top-k sampling
// (reference utils/ops.py:435-464, 385-432, 476-505; models/downsample.py:205-240, 264-284).
//
// The reference does this with nb full sorts over N, a Python B x nb slicing loop and ~10*nb tiny
// launches with host syncs.  Here one CTA per cloud keeps everything in shared memory:
// z-score -> bin id -> per-bin count / token-logit mean -> sequential fp32 k allocation (kalloc.h)
// -> ONE bitonic sort of 64-bit keys (bin | inverted score bits | index) -> segmented prefix take.
#include "common.cuh"
#include "kalloc.h"

namespace samble {

constexpr int kSampThreads = 1024;

// deterministic block-wide sum of one double per thread; result valid in every thread.
__device__ __forceinline__ double block_sum(double v, double* red /* smem [32] */) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < nw; ++w) s += red[w];
  return s;
}

// mean and population std of x[0..N) in fp64, returned rounded to fp32 (ops.py:450-452).
__device__ __forceinline__ void mean_std(const float* x, int N, double* red, float& mean_f, float& std_f) {
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += (double)x[i];
  const double mean = block_sum(s, red) / N;
  double s2 = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double d = (double)x[i] - mean;
    s2 += d * d;
  }
  const double var = block_sum(s2, red) / N;
  mean_f = (float)mean;
  std_f = (float)sqrt(var);
}

__global__ void __launch_bounds__(kSampThreads) zscore_kernel(const float* __restrict__ score, int N, float* __restrict__ z) {
  __shared__ double red[32];
  const float* x = score + (long long)blockIdx.x * N;
  float m, s;
  mean_std(x, N, red, m, s);
  for (int i = threadIdx.x; i < N; i += blockDim.x) z[(long long)blockIdx.x * N + i] = __fdiv_rn(__fsub_rn(x[i], m), s);
}

__global__ void __launch_bounds__(256) bin_mask_kernel(const float* __restrict__ z, const float* __restrict__ upper,
                                                       const float* __restrict__ lower, long long total, int nb,
                                                       uint8_t* __restrict__ mask) {
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const float v = z[t];
    for (int j = 0; j < nb; ++j) mask[t * nb + j] = (v < upper[j] && v >= lower[j]) ? 1 : 0;
  }
}

__global__ void num_points_kernel(const float* __restrict__ bin_prob, const long long* __restrict__ cnt, int B, int nb,
                                  int total, int* __restrict__ k_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float w[kMaxBins];
  long long c[kMaxBins];
  int k[kMaxBins];
  for (int j = 0; j < nb; ++j) w[j] = bin_prob[b * nb + j], c[j] = cnt[b * nb + j];
  num_points_to_choose(w, c, nb, total, k);
  for (int j = 0; j < nb; ++j) k_out[b * nb + j] = k[j];
}

// in-place ascending bitonic sort of n (power of two) 64-bit keys in shared memory, whole CTA.
__device__ __forceinline__ void bitonic_sort(unsigned long long* key, int n) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const unsigned long long a = key[lo], b = key[hi];
        if ((a > b) == up) key[lo] = b, key[hi] = a;
      }
    }
  }
  __syncthreads();
}

// Sort key of v = score + 1e-8 (ops.py:478) such that ASCENDING key order == DESCENDING v, for any float: the IEEE
// order-preserving map (negative values: all bits flipped, others: sign bit set), inverted.  -0 counts as +0 and NaN as
// the largest value (torch.sort descending puts NaN first).
__device__ __forceinline__ unsigned desc_key(float v) {
  if (v != v) return 0u;
  if (v == 0.f) v = 0.f;                                   // -0 -> +0
  const unsigned b = __float_as_uint(v);
  const unsigned asc = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ~asc;
}
__device__ __forceinline__ unsigned inv_score_bits(float s) { return desc_key(__fadd_rn(s, 1e-8f)); }

static __host__ __device__ int next_pow2(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}

// ops.py:476-505 for an arbitrary 0/1 mask (bins may overlap): one sort per bin.
__global__ void __launch_bounds__(kSampThreads) index_topk_kernel(const float* __restrict__ score,
                                                                  const uint8_t* __restrict__ mask,
                                                                  const int* __restrict__ k, int N, int nb, int M,
                                                                  int npad, long long* __restrict__ idx_out) {
  extern __shared__ __align__(16) unsigned long long keys[];
  const int b = blockIdx.x;
  int off = 0;
  for (int j = 0; j < nb; ++j) {
    __syncthreads();
    for (int i = threadIdx.x; i < npad; i += blockDim.x) {
      unsigned long long key = ~0ull;
      if (i < N) {
        // non-members carry (score + 1e-8) * 0 = 0: after every member with a positive value and before members with a
        // negative one (ops.py:478-486), in index order among themselves
        const unsigned hi = mask[((long long)b * N + i) * nb + j] ? inv_score_bits(score[(long long)b * N + i]) : desc_key(0.f);
        key = ((unsigned long long)hi << 24) | (unsigned)i;
      }
      keys[i] = key;
    }
    bitonic_sort(keys, npad);
    const int kj = k[b * nb + j];
    for (int r = threadIdx.x; r < kj; r += blockDim.x)
      if (off + r < M && r < N) idx_out[(long long)b * M + off + r] = (long long)(keys[r] & 0xffffffu);
    off += kj;
  }
}

// fused DownSample bin stage for one cloud (downsample.py:205-240).
__global__ void __launch_bounds__(kSampThreads) ds_sample_kernel(const float* __restrict__ score,
                                                                 const float* __restrict__ token_logits,
                                                                 const float* __restrict__ cuts, int N, int nb, int M,
                                                                 int npad, long long* __restrict__ idx_out,
                                                                 uint8_t* __restrict__ bin_id, int* __restrict__ counts,
                                                                 int* __restrict__ k_out, float* __restrict__ w_raw,
                                                                 float* __restrict__ z_out) {
  extern __shared__ __align__(16) unsigned long long keys[];
  __shared__ double red[32];
  __shared__ double tok_sum[kMaxBins];
  __shared__ int cnt[kMaxBins], kk[kMaxBins], start[kMaxBins + 1], koff[kMaxBins + 1];
  const int b = blockIdx.x;
  const float* x = score + (long long)b * N;
  float mean, sd;
  mean_std(x, N, red, mean, sd);
  if (threadIdx.x < kMaxBins) cnt[threadIdx.x] = 0;
  __syncthreads();
  // bin id + key
  double tsum[kMaxBins];
#pragma unroll
  for (int j = 0; j < kMaxBins; ++j) tsum[j] = 0.0;
  for (int i = threadIdx.x; i < npad; i += blockDim.x) {
    unsigned long long key = ~0ull;
    if (i < N) {
      const float s = x[i];
      const float z = __fdiv_rn(__fsub_rn(s, mean), sd);
      if (z_out) z_out[(long long)b * N + i] = z;
      int bin = 255;
      for (int j = nb - 1; j >= 0; --j) {
        // upper = [inf, c0, c1, ...], lower = [c0, c1, ..., -inf]  (ops.py:214-233, 460-462)
        const bool lt_up = (j == 0) ? (z < INFINITY) : (z < cuts[j - 1]);
        const bool ge_lo = (j == nb - 1) ? (z >= -INFINITY) : (z >= cuts[j]);
        if (lt_up && ge_lo) bin = j;      // first matching bin wins (cuts are non-increasing => unique)
      }
      bin_id[(long long)b * N + i] = (uint8_t)bin;
      if (bin < nb) {
        atomicAdd(&cnt[bin], 1);
        const float tl = token_logits[((long long)b * N + i) * nb + bin];
#pragma unroll
        for (int j = 0; j < kMaxBins; ++j)
          if (j == bin) tsum[j] += (double)tl;
      }
      key = ((unsigned long long)bin << 56) | ((unsigned long long)inv_score_bits(s) << 24) | (unsigned)i;
    }
    keys[i] = key;
  }
#pragma unroll
  for (int j = 0; j < kMaxBins; ++j) {
    const double t = (j < nb) ? block_sum(tsum[j], red) : 0.0;
    if (threadIdx.x == 0) tok_sum[j] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float w[kMaxBins];
    long long c[kMaxBins];
    for (int j = 0; j < nb; ++j) {
      c[j] = cnt[j];
      // sum / (count_nonzero + 1e-8) in fp32, then relu (downsample.py:268-274)
      const float raw = __fdiv_rn((float)tok_sum[j], __fadd_rn((float)cnt[j], 1e-8f));
      w_raw[b * nb + j] = raw;
      w[j] = raw > 0.f ? raw : 0.f;
    }
    num_points_to_choose(w, c, nb, M, kk);
    start[0] = 0, koff[0] = 0;
    for (int j = 0; j < nb; ++j) {
      start[j + 1] = start[j] + cnt[j];
      koff[j + 1] = koff[j] + kk[j];
      counts[b * nb + j] = cnt[j];
      k_out[b * nb + j] = kk[j];
    }
  }
  bitonic_sort(keys, npad);   // begins and ends with __syncthreads()
  for (int p = threadIdx.x; p < N; p += blockDim.x) {
    const unsigned long long key = keys[p];
    const int bin = (int)(key >> 56);
    if (bin < nb) {
      const int r = p - start[bin];
      if (r < kk[bin] && koff[bin] + r < M) idx_out[(long long)b * M + koff[bin] + r] = (long long)(key & 0xffffffu);
    }
  }
  // A bin that was asked for more points than it holds (the remainder rule of ops.py:427-430 can do that when nearly
  // every bin is saturated): the reference's per-bin sort continues with the non-members, whose masked value is 0,
  // i.e. in index order (ops.py:486-503).  One warp walks the cloud per such bin.
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    for (int j = 0; j < nb; ++j) {
      int need = kk[j] - cnt[j];
      if (need <= 0) continue;
      int filled = 0;
      for (int i0 = 0; i0 < N && filled < need; i0 += 32) {
        const int i = i0 + lane;
        const bool other = i < N && bin_id[(long long)b * N + i] != j;
        const unsigned m = __ballot_sync(kFull, other);
        const int r = filled + __popc(m & ((1u << lane) - 1u));
        if (other && r < need && koff[j] + cnt[j] + r < M) idx_out[(long long)b * M + koff[j] + cnt[j] + r] = i;
        filled += __popc(m);
      }
    }
  }
}

}  // namespace samble

namespace samble {

// ---- stochastic sampling modes (reference utils/ops.py:507-592): the per-(cloud, bin) categorical distribution that
// torch.multinomial draws from, in ONE kernel per cloud instead of ~15 element-wise ATen launches over (B,N,nb).
//   uniform:  p[b,j,n] = mask[b,n,j]; a bin without points draws from all N (ops.py:512-516)
//   random:   z = tanh(zscore(score)); p = exp(z * inv_t[j]) * mask / sum_n(...); NaN -> 1e-8 (ops.py:518-592), with
//             inv_t = count_j / t_div (boltzmann "mode_1" / "mode_3": t_div = 100 / 200) or a constant (modes 2 / 4, number)
// Output layout (B, nb, N) row-major == p.permute(0, 2, 1).reshape(-1, N) of the reference.
__global__ void __launch_bounds__(kSampThreads) sampling_prob_kernel(const float* __restrict__ score, const uint8_t* __restrict__ mask,
                                                                     int N, int nb, int mode, float inv_t_const, float t_div,
                                                                     float* __restrict__ p) {
  __shared__ double red[32];
  __shared__ float s_sum[kMaxBins];
  __shared__ int s_cnt[kMaxBins];
  const int b = blockIdx.x;
  const float* x = score + (long long)b * N;
  const uint8_t* mk = mask + (long long)b * N * nb;
  float* out = p + (long long)b * nb * N;
  if (threadIdx.x < kMaxBins) s_sum[threadIdx.x] = 0.f, s_cnt[threadIdx.x] = 0;
  __syncthreads();
  for (int j = 0; j < nb; ++j) {                          // bin sizes (deterministic block sums)
    double c = 0.0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) c += mk[(long long)i * nb + j] ? 1.0 : 0.0;
    const double tot = block_sum(c, red);
    if (threadIdx.x == 0) s_cnt[j] = (int)tot;
  }
  __syncthreads();
  if (mode == 0) {                                        // uniform
    for (int j = 0; j < nb; ++j) {
      const float fill = s_cnt[j] == 0 ? 1.f : 0.f;
      for (int i = threadIdx.x; i < N; i += blockDim.x) out[(long long)j * N + i] = (mk[(long long)i * nb + j] ? 1.f : 0.f) + fill;
    }
    return;
  }
  float m, sd;
  mean_std(x, N, red, m, sd);
  for (int j = 0; j < nb; ++j) {
    const float inv_t = t_div > 0.f ? __fdiv_rn((float)s_cnt[j], t_div) : inv_t_const;
    double acc = 0.0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const float z = tanhf(__fdiv_rn(__fsub_rn(x[i], m), sd));
      const float e = mk[(long long)i * nb + j] ? expf(z * inv_t) : 0.f;
      out[(long long)j * N + i] = e;
      acc += (double)e;
    }
    const double tot = block_sum(acc, red);
    const float tf = (float)tot;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const float v = __fdiv_rn(out[(long long)j * N + i], tf);
      out[(long long)j * N + i] = (v != v) ? 1e-8f : v;   // empty bin: 0/0 -> 1e-8 everywhere (ops.py:590)
    }
    __syncthreads();
  }
}

// dynamic bin boundaries (utils/ops.py:174-236) after the batch sort: pick the nb-1 batch quantiles ...
__global__ void quantile_pick_kernel(const float* __restrict__ sorted_desc, long long n, int nb, float* __restrict__ cut) {
  const int j = threadIdx.x + 1;
  if (j < nb) {
    const long long pos = (long long)(int)((float)j / (float)nb * (float)n);       // ops.py:182-183 (fp32 product, int truncation)
    cut[j - 1] = sorted_desc[pos < n ? pos : n - 1];
  }
}
// ... and, after the (nb-1)-float all-reduce, average over ranks and blend into the [upper, lower] pair in place
// (or create it with the +-inf sentinels when there is no previous pair): one launch instead of ~10 element-wise ones.
// The roundings are ATen's on CUDA for `cut / world` and `upper * m + (1 - m) * cut` (utils/ops.py:198-213): a tensor divided by
// a Python scalar is multiplied by the fp32 reciprocal, each scalar reaches the kernel rounded to fp32 from the Python
// double (so 1 - m is fp32(1 - m), not 1.f - fp32(m)), and every product / sum is rounded on its own (no FMA).
__global__ void boundary_ema_kernel(const float* __restrict__ cut_sum, float inv_world, float momentum, float one_minus_momentum,
                                    int has_old, int nb, float* __restrict__ upper, float* __restrict__ lower) {
  const int j = threadIdx.x;                              // cut index 0 .. nb-2
  if (j == 0) upper[0] = INFINITY, lower[nb - 1] = -INFINITY;
  if (j < nb - 1) {
    float c = __fmul_rn(cut_sum[j], inv_world);
    if (has_old) c = __fadd_rn(__fmul_rn(upper[j + 1], momentum), __fmul_rn(one_minus_momentum, c));
    upper[j + 1] = c;
    lower[j] = c;
  }
}

}  // namespace samble

using namespace samble;

extern "C" int samble_zscore(const float* score, int rows, int N, float* z, samble_stream_t stream) {
  SAMBLE_REQUIRE(score && z, "samble_zscore: null pointer");
  SAMBLE_REQUIRE(rows > 0 && N > 0, "samble_zscore: bad shape");
  SAMBLE_PRE((cudaStream_t)stream);
  zscore_kernel<<<rows, kSampThreads, 0, (cudaStream_t)stream>>>(score, N, z);
  SAMBLE_LAUNCHED("zscore_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_bin_mask(const float* z, const float* upper, const float* lower, int rows, int N, int nb,
                               uint8_t* mask, samble_stream_t stream) {
  SAMBLE_REQUIRE(z && upper && lower && mask, "samble_bin_mask: null pointer");
  SAMBLE_REQUIRE(rows > 0 && N > 0 && nb > 0, "samble_bin_mask: bad shape");
  const long long total = (long long)rows * N;
  long long g = (total + 255) / 256;
  SAMBLE_PRE((cudaStream_t)stream);
  bin_mask_kernel<<<(int)(g > 148 * 8 ? 148 * 8 : g), 256, 0, (cudaStream_t)stream>>>(z, upper, lower, total, nb, mask);
  SAMBLE_LAUNCHED("bin_mask_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_num_points_to_choose(const float* bin_prob, const long long* max_num_points, int B, int nb,
                                           int total, int* k_out, samble_stream_t stream) {
  SAMBLE_REQUIRE(bin_prob && max_num_points && k_out, "samble_num_points_to_choose: null pointer");
  SAMBLE_REQUIRE(B > 0 && nb > 0 && nb <= kMaxBins, "samble_num_points_to_choose: nb=%d outside [1,%d]", nb, kMaxBins);
  SAMBLE_PRE((cudaStream_t)stream);
  num_points_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(bin_prob, max_num_points, B, nb, total, k_out);
  SAMBLE_LAUNCHED("num_points_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_downsample_index_topk(const float* score, const uint8_t* mask, const int* k, int B, int N, int nb,
                                            int M, long long* idx_out, samble_stream_t stream) {
  SAMBLE_REQUIRE(score && mask && k && idx_out, "samble_downsample_index_topk: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && nb > 0 && M > 0, "samble_downsample_index_topk: bad shape");
  SAMBLE_REQUIRE(N < (1 << 24), "samble_downsample_index_topk: N=%d >= 2^24", N);
  const int npad = next_pow2(N);
  const size_t smem = (size_t)npad * sizeof(unsigned long long);
  SAMBLE_REQUIRE(smem <= 200 * 1024, "samble_downsample_index_topk: N=%d too large for the shared-memory sort", N);
  cudaFuncSetAttribute(index_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  SAMBLE_PRE((cudaStream_t)stream);
  index_topk_kernel<<<B, kSampThreads, smem, (cudaStream_t)stream>>>(score, mask, k, N, nb, M, npad, idx_out);
  SAMBLE_LAUNCHED("index_topk_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_ds_sample(const float* score, const float* token_logits, const float* cuts, int B, int N, int nb,
                                int M, long long* idx_out, uint8_t* bin_id, int* counts, int* k_out, float* w_raw,
                                float* z_out, samble_stream_t stream) {
  SAMBLE_REQUIRE(score && token_logits && cuts && idx_out && bin_id && counts && k_out && w_raw,
                 "samble_ds_sample: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && M > 0 && M <= N, "samble_ds_sample: bad shape (need 0 < M <= N)");
  SAMBLE_REQUIRE(nb >= 1 && nb <= kMaxBins, "samble_ds_sample: nb=%d outside [1,%d]", nb, kMaxBins);
  SAMBLE_REQUIRE(N < (1 << 24), "samble_ds_sample: N=%d >= 2^24", N);
  const int npad = next_pow2(N);
  const size_t smem = (size_t)npad * sizeof(unsigned long long);
  SAMBLE_REQUIRE(smem <= 200 * 1024, "samble_ds_sample: N=%d too large for the shared-memory sort", N);
  cudaFuncSetAttribute(ds_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  SAMBLE_PRE((cudaStream_t)stream);
  ds_sample_kernel<<<B, kSampThreads, smem, (cudaStream_t)stream>>>(score, token_logits, cuts, N, nb, M, npad, idx_out,
                                                                     bin_id, counts, k_out, w_raw, z_out);
  SAMBLE_LAUNCHED("ds_sample_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_sampling_probabilities(const float* score, const uint8_t* mask, int B, int N, int nb, int mode, float inv_t_const,
                                             float t_div, float* p, samble_stream_t stream) {
  SAMBLE_REQUIRE(score && mask && p, "samble_sampling_probabilities: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && nb > 0 && nb <= kMaxBins, "samble_sampling_probabilities: bad shape (nb <= %d)", kMaxBins);
  SAMBLE_REQUIRE(mode == 0 || mode == 1, "samble_sampling_probabilities: mode must be 0 (uniform) or 1 (random)");
  cudaStream_t st = (cudaStream_t)stream;
  SAMBLE_PRE(st);
  sampling_prob_kernel<<<B, kSampThreads, 0, st>>>(score, mask, N, nb, mode, inv_t_const, t_div, p);
  SAMBLE_LAUNCHED("sampling_prob_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_quantile_pick(const float* sorted_desc, long long n, int nb, float* cut, samble_stream_t stream) {
  SAMBLE_REQUIRE(sorted_desc && cut && n > 0 && nb > 1 && nb <= kMaxBins, "samble_quantile_pick: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  SAMBLE_PRE(st);
  quantile_pick_kernel<<<1, 32, 0, st>>>(sorted_desc, n, nb, cut);
  SAMBLE_LAUNCHED("quantile_pick_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_boundary_ema(const float* cut_sum, int world, double momentum, int has_old, int nb, float* upper, float* lower,
                                   samble_stream_t stream) {
  SAMBLE_REQUIRE(cut_sum && upper && lower && world > 0 && nb > 1 && nb <= kMaxBins, "samble_boundary_ema: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  SAMBLE_PRE(st);
  boundary_ema_kernel<<<1, 32, 0, st>>>(cut_sum, 1.f / (float)world, (float)momentum, (float)(1.0 - momentum), has_old, nb, upper,
                                        lower);
  SAMBLE_LAUNCHED("boundary_ema_kernel");
  return SAMBLE_OK;
}
