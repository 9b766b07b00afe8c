// Backward kernels of the differentiable path (SURVEY 8 row f1).  The reference trains through ATen autograd of
//   torch.gather            utils/ops.py:13   (index_points; via select_neighbors / group, :47-112)
//   torch.gather            utils/ops.py:144  (gather_by_idx)
//   softmax(q k^T) v over K models/attention.py:207-250 (Neighbor2Point attention over gathered differences)
// whose backward passes are scatter-adds.  Here they are scatter-adds too, but over the SAME compact operands the
// forward kernels use: the (B,C,N,K) grouped tensors of the reference's attention never exist in either direction.
//
// Accumulation uses fp32 atomics (RED.ADD): summation order, hence the last bits of a gradient, varies run to run,
// as it does in ATen's own gather backward (index_add / scatter_add on CUDA) while torch.use_deterministic_algorithms is
// off.  With it on, ATen switches to ordered algorithms and so does this library: samble_b200/autograd.py then runs the
// atomic-free kernels of backward_ordered.cu instead, which add the same terms in a defined order.
#include "common.cuh"

namespace samble {

// grad_points[b, idx[b,r], :] += grad_out[b, r, :]      (points (B,N,C) point-major; r over the R = M*K gathered rows)
template <class I>
__global__ void __launch_bounds__(256) index_points_bwd_kernel(const float* __restrict__ go, const I* __restrict__ idx, int N,
                                                               int C, long long R, float* __restrict__ gp) {
  const int b = blockIdx.y;
  const long long total = R * C;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long r = t / C;
    const int c = (int)(t % C);
    const int j = ld_idx(idx, (long long)b * R + r);
    atomicAdd(gp + ((long long)b * N + j) * C + c, go[(long long)b * total + t]);
  }
}

// grad_pcd[b, c, idx[b,m]] += grad_out[b, c, m]          (pcd (B,C,N) channel-major)
template <class I>
__global__ void __launch_bounds__(256) gather_by_idx_bwd_kernel(const float* __restrict__ go, const I* __restrict__ idx, int C,
                                                                int N, int M, float* __restrict__ gp) {
  const int b = blockIdx.y;
  const long long total = (long long)C * M;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(t / M), m = (int)(t % M);
    atomicAdd(gp + ((long long)b * C + c) * N + ld_idx(idx, (long long)b * M + m), go[(long long)b * total + t]);
  }
}

// Neighbor2Point attention backward.  Forward (attention.cu): per point i and head h
//   p_ij = softmax_j(q_i . k_j / sqrt(d)),   out_i = sum_j p_ij v_j - v_i        (j over the K neighbours of i)
// (the reference's k_ij = k_j - k_i, v_ij = v_j - v_i: the -q_i.k_i term cancels in the softmax and sum_j ds_ij = 0 makes
// its gradient vanish too, so the compact form has the SAME gradients w.r.t. q, k and v).  With g_i = dL/dout_i:
//   dp_ij = g_i . v_j          ds_ij = p_ij (dp_ij - sum_j' p_ij' dp_ij')
//   dq_i  = sum_j ds_ij k_j / sqrt(d)         dk_j += ds_ij q_i / sqrt(d)          dv_j += p_ij g_i,   dv_i -= g_i
// One warp per point, lanes across channels (float4), heads = groups of lph lanes; the K rows of k and v are gathered
// exactly as in the forward pass, the scatter side goes through float atomics into dk / dv (pre-zeroed by the caller).
template <class I, int KMAX>
__global__ void __launch_bounds__(256) n2p_attend_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                             const float* __restrict__ v, long long ld, const I* __restrict__ idx,
                                                             int N, int C, int K, int lph, float sqrt_d,
                                                             const float* __restrict__ go, long long ld_go, float* __restrict__ gq,
                                                             float* __restrict__ gk, float* __restrict__ gv, long long ld_g) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int n = blockIdx.x * 8 + warp;
  if (n >= N) return;
  const bool on = lane * 4 < C;
  const long long row = (long long)b * N + n;
  const int my = lane < K ? ld_idx(idx, row * K + lane) : 0;
  float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = q4;
  if (on) {
    q4 = *reinterpret_cast<const float4*>(q + row * ld + lane * 4);
    g4 = *reinterpret_cast<const float4*>(go + row * ld_go + lane * 4);
  }
  float lg[KMAX], dp[KMAX];
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    lg[j] = -INFINITY, dp[j] = 0.f;
    if (j < K) {
      const int nj = __shfl_sync(kFull, my, j);
      float a = 0.f, d = 0.f;
      if (on) {
        const float4 k4 = __ldg(reinterpret_cast<const float4*>(k + ((long long)b * N + nj) * ld + lane * 4));
        const float4 v4 = __ldg(reinterpret_cast<const float4*>(v + ((long long)b * N + nj) * ld + lane * 4));
        a = fmaf(q4.w, k4.w, fmaf(q4.z, k4.z, fmaf(q4.y, k4.y, q4.x * k4.x)));
        d = fmaf(g4.w, v4.w, fmaf(g4.z, v4.z, fmaf(g4.y, v4.y, g4.x * v4.x)));
      }
      for (int o = lph >> 1; o > 0; o >>= 1) {
        a += __shfl_xor_sync(kFull, a, o);
        d += __shfl_xor_sync(kFull, d, o);
      }
      lg[j] = a / sqrt_d;
      dp[j] = d;
    }
  }
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < KMAX; ++j) m = fmaxf(m, lg[j]);
  float s = 0.f, pd = 0.f;
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    const float p = j < K ? expf(lg[j] - m) : 0.f;
    lg[j] = p;                                  // lg now holds the unnormalised probabilities
    s += p;
    pd = fmaf(p, dp[j], pd);
  }
  const float inv_s = 1.f / s;
  pd *= inv_s;                                  // sum_j p_ij dp_ij
  float4 dq = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    if (j < K) {
      const int nj = __shfl_sync(kFull, my, j);
      const float p = lg[j] * inv_s;
      const float ds = p * (dp[j] - pd) / sqrt_d;
      if (on) {
        const long long o = ((long long)b * N + nj);
        const float4 k4 = __ldg(reinterpret_cast<const float4*>(k + o * ld + lane * 4));
        dq.x = fmaf(ds, k4.x, dq.x), dq.y = fmaf(ds, k4.y, dq.y), dq.z = fmaf(ds, k4.z, dq.z), dq.w = fmaf(ds, k4.w, dq.w);
        float* pk = gk + o * ld_g + lane * 4;
        float* pv = gv + o * ld_g + lane * 4;
        atomicAdd(pk + 0, ds * q4.x), atomicAdd(pk + 1, ds * q4.y), atomicAdd(pk + 2, ds * q4.z), atomicAdd(pk + 3, ds * q4.w);
        atomicAdd(pv + 0, p * g4.x), atomicAdd(pv + 1, p * g4.y), atomicAdd(pv + 2, p * g4.z), atomicAdd(pv + 3, p * g4.w);
      }
    }
  }
  if (on) {
    *reinterpret_cast<float4*>(gq + row * ld_g + lane * 4) = dq;
    float* pv = gv + row * ld_g + lane * 4;
    atomicAdd(pv + 0, -g4.x), atomicAdd(pv + 1, -g4.y), atomicAdd(pv + 2, -g4.z), atomicAdd(pv + 3, -g4.w);
  }
}

static int bwd_grid(long long work, int per_block) {
  long long g = (work + per_block - 1) / per_block;
  const long long cap = 148 * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace samble

using namespace samble;

extern "C" int samble_index_points_backward(const float* grad_out, const void* idx, int idx_bits, int B, int N, int C, int R,
                                            float* grad_points, samble_stream_t stream) {
  SAMBLE_REQUIRE(grad_out && idx && grad_points, "samble_index_points_backward: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && C > 0 && R > 0, "samble_index_points_backward: bad shape");
  SAMBLE_REQUIRE(idx_bits == 32 || idx_bits == 64, "samble_index_points_backward: idx_bits must be 32 or 64");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(bwd_grid((long long)R * C, 256), B);
  SAMBLE_PRE(st);
  if (idx_bits == 64)
    index_points_bwd_kernel<long long><<<grid, 256, 0, st>>>(grad_out, (const long long*)idx, N, C, R, grad_points);
  else
    index_points_bwd_kernel<int><<<grid, 256, 0, st>>>(grad_out, (const int*)idx, N, C, R, grad_points);
  SAMBLE_LAUNCHED("index_points_bwd_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_gather_by_idx_backward(const float* grad_out, const void* idx, int idx_bits, int B, int C, int N, int M,
                                             float* grad_pcd, samble_stream_t stream) {
  SAMBLE_REQUIRE(grad_out && idx && grad_pcd, "samble_gather_by_idx_backward: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && C > 0 && M > 0, "samble_gather_by_idx_backward: bad shape");
  SAMBLE_REQUIRE(idx_bits == 32 || idx_bits == 64, "samble_gather_by_idx_backward: idx_bits must be 32 or 64");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(bwd_grid((long long)C * M, 256), B);
  SAMBLE_PRE(st);
  if (idx_bits == 64)
    gather_by_idx_bwd_kernel<long long><<<grid, 256, 0, st>>>(grad_out, (const long long*)idx, C, N, M, grad_pcd);
  else
    gather_by_idx_bwd_kernel<int><<<grid, 256, 0, st>>>(grad_out, (const int*)idx, C, N, M, grad_pcd);
  SAMBLE_LAUNCHED("gather_by_idx_bwd_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_n2p_attend_backward(const float* q, const float* k, const float* v, long long ld, const void* idx, int idx_bits,
                                          int B, int N, int C, int K, int heads, const float* grad_out, long long ld_go,
                                          float* grad_q, float* grad_k, float* grad_v, long long ld_g, samble_stream_t stream) {
  SAMBLE_REQUIRE(q && k && v && idx && grad_out && grad_q && grad_k && grad_v, "samble_n2p_attend_backward: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && K > 0 && K <= 32, "samble_n2p_attend_backward: bad shape (K <= 32)");
  SAMBLE_REQUIRE(C > 0 && C % 4 == 0 && C <= 128, "samble_n2p_attend_backward: C=%d must be a multiple of 4, <= 128", C);
  SAMBLE_REQUIRE(heads > 0 && C % heads == 0 && (C / heads) % 4 == 0, "samble_n2p_attend_backward: C/heads must be a multiple of 4");
  const int lph = C / heads / 4;
  SAMBLE_REQUIRE((lph & (lph - 1)) == 0, "samble_n2p_attend_backward: (C/heads)/4 = %d must be a power of two", lph);
  SAMBLE_REQUIRE(ld % 4 == 0 && ld_go % 4 == 0 && ld_g % 4 == 0, "samble_n2p_attend_backward: leading dimensions must be multiples of 4");
  SAMBLE_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)grad_out | (uintptr_t)grad_q | (uintptr_t)grad_k | (uintptr_t)grad_v) % 16 == 0,
                 "samble_n2p_attend_backward: 16-byte alignment required");
  SAMBLE_REQUIRE(idx_bits == 32 || idx_bits == 64, "samble_n2p_attend_backward: idx_bits must be 32 or 64");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(ceil_div(N, 8), B);
  const float sqrt_d = sqrtf((float)(C / heads));
  SAMBLE_PRE(st);
  if (idx_bits == 64)
    n2p_attend_bwd_kernel<long long, 32><<<grid, 256, 0, st>>>(q, k, v, ld, (const long long*)idx, N, C, K, lph, sqrt_d, grad_out, ld_go,
                                                               grad_q, grad_k, grad_v, ld_g);
  else
    n2p_attend_bwd_kernel<int, 32><<<grid, 256, 0, st>>>(q, k, v, ld, (const int*)idx, N, C, K, lph, sqrt_d, grad_out, ld_go, grad_q,
                                                         grad_k, grad_v, ld_g);
  SAMBLE_LAUNCHED("n2p_attend_bwd_kernel");
  return SAMBLE_OK;
}
