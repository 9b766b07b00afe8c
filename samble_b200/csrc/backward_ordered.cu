// Ordered (atomic-free) backward scatters: the kernels the differentiable path takes while
// torch.use_deterministic_algorithms(True) is in force (samble_b200/autograd.py).  backward.cu's kernels add their
// terms with fp32 atomics in whatever order the hardware serves them; these add the same terms in a defined order.
//
// Order contract.  For cloud b, edge e in [0, R) has target t_e = idx[b, e]; L_j lists the edges with target j in
// ascending e.  Every output element is a left fold in fp32, each product and each sum rounded on its own:
//   acc = 0;  for e in L_j:  acc = acc + term_e;   out[b, j, c] = acc (- sub[b, j, c])
//   term_e = x[b, e / src_div, c]  or  w[b, e, c / (C / heads)] * x[b, e / src_div, c]
// Entries of idx outside [0, N) contribute nothing.
//
//   reverse_index_kernel         idx -> CSR (offsets, edges): a stable counting sort per cloud
//   scatter_rows_ordered_kernel  the fold above, one warp per target row, lanes across channels
//   n2p_attend_bwd_edges_kernel  n2p_attend_bwd_kernel's per-edge pass without the scatter: grad_q plus p and ds per edge
//                                and head, the same fp32 expressions, so dk / dv from the fold add the atomic kernel's terms
#include "common.cuh"

namespace samble {

constexpr int kRevWarps = 32;   // reverse_index_kernel: one 1024-thread CTA per cloud, each warp owns a contiguous edge segment

template <class I>
__device__ __forceinline__ int rev_target(const I* p, long long e, int N) {
  const long long t = (long long)p[e];
  return (t >= 0 && t < N) ? (int)t : -1;
}

// Stable counting sort of the edges of one cloud by target.  Warp w owns the edges [w*seg, (w+1)*seg) and counts them
// into its private row cnt[w][:] of the workspace; an exclusive prefix over the warps (per target) and over the targets
// (per cloud) then gives every warp the first slot of each of its buckets, and the warp places its edges 32 at a time in
// ascending e (lanes with the same target are ranked by __match_any_sync).  No float is involved and every count is an
// integer, so the result does not depend on the order in which the atomics land.
template <class I>
__global__ void __launch_bounds__(1024) reverse_index_kernel(const I* __restrict__ idx, int N, int R, int* __restrict__ offsets,
                                                             int* __restrict__ edges, int* __restrict__ cnt_ws) {
  __shared__ int s_part[kRevWarps];
  __shared__ int s_carry;
  const int b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const I* id = idx + (long long)b * R;
  int* off = offsets + (long long)b * (N + 1);
  int* ed = edges + (long long)b * R;
  int* cnt = cnt_ws + (long long)b * kRevWarps * N;
  int* mine = cnt + (long long)warp * N;
  const int seg = (int)(((long long)R + kRevWarps - 1) / kRevWarps);
  const int e0 = (int)min((long long)warp * seg, (long long)R), e1 = (int)min((long long)e0 + seg, (long long)R);

  for (long long t = threadIdx.x; t < (long long)kRevWarps * N; t += blockDim.x) cnt[t] = 0;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = e0; base < e1; base += 32) {                 // per-warp histogram, one add per distinct target
    const int e = base + lane;
    const int t = e < e1 ? rev_target(id, e, N) : -1;
    const unsigned grp = __match_any_sync(kFull, t);
    if (t >= 0 && lane == __ffs(grp) - 1) atomicAdd(mine + t, __popc(grp));
  }
  __syncthreads();
  for (int base = 0; base < N; base += blockDim.x) {           // prefix over warps per target, then over targets
    const int j = base + threadIdx.x;
    int tot = 0;
    if (j < N)
      for (int w = 0; w < kRevWarps; ++w) {
        const int c = cnt[(long long)w * N + j];
        cnt[(long long)w * N + j] = tot;
        tot += c;
      }
    int incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(kFull, incl, o);
      if (lane >= o) incl += y;
    }
    if (lane == 31) s_part[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int v = s_part[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v += y;
      }
      s_part[lane] = v;
    }
    __syncthreads();
    const int excl = s_carry + (warp ? s_part[warp - 1] : 0) + incl - tot;
    if (j < N) off[j] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) s_carry = excl + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) off[N] = s_carry;
  for (int base = e0; base < e1; base += 32) {                 // stable placement
    const int e = base + lane;
    const int t = e < e1 ? rev_target(id, e, N) : -1;
    const unsigned grp = __match_any_sync(kFull, t);
    int pos = 0;
    if (t >= 0) pos = off[t] + mine[t] + __popc(grp & ((1u << lane) - 1u));
    __syncwarp();
    if (t >= 0) {
      ed[pos] = e;
      if (lane == 31 - __clz(grp)) mine[t] += __popc(grp);
    }
    __syncwarp();
  }
  const int valid = s_carry;                                   // slots past the last bucket hold -1
  for (int p = valid + threadIdx.x; p < R; p += blockDim.x) ed[p] = -1;
}

struct ScatterArgs {
  const float* x;
  long long x_batch, x_row, x_ch;
  int src_div;
  const float* w;
  int heads, dh;
  const int* offsets;
  const int* edges;
  const float* sub;
  long long sub_batch, sub_row;
  int N, R, C;
  float* out;
  long long out_batch, out_row, out_ch;
};

// One warp per target row j, lane l folding channels c0 + l + 32 i (i < 4) over the edges of L_j in ascending e.  The
// time of a row is proportional to its in-degree, so a hub target (every edge on one point) runs serially on one warp.
__global__ void __launch_bounds__(256) scatter_rows_ordered_kernel(const ScatterArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int j = blockIdx.x * 8 + warp;
  if (j >= a.N) return;
  const int* off = a.offsets + (long long)b * (a.N + 1);
  const int p0 = off[j], p1 = off[j + 1];
  const int* ed = a.edges + (long long)b * a.R;
  const float* xb = a.x + (long long)b * a.x_batch;
  const float* wb = a.w ? a.w + (long long)b * a.R * a.heads : nullptr;
  for (int c0 = 0; c0 < a.C; c0 += 128) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    int hh[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) hh[i] = wb ? min(c0 + lane + 32 * i, a.C - 1) / a.dh : 0;
    for (int p = p0; p < p1; ++p) {
      const int e = __ldg(ed + p);
      const float* xr = xb + (long long)(e / a.src_div) * a.x_row;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = c0 + lane + 32 * i;
        if (c < a.C) {
          float term = __ldg(xr + (long long)c * a.x_ch);
          if (wb) term = __fmul_rn(__ldg(wb + (long long)e * a.heads + hh[i]), term);
          acc[i] = __fadd_rn(acc[i], term);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = c0 + lane + 32 * i;
      if (c < a.C) {
        float v = acc[i];
        if (a.sub) v = __fsub_rn(v, a.sub[(long long)b * a.sub_batch + (long long)j * a.sub_row + c]);
        a.out[(long long)b * a.out_batch + (long long)j * a.out_row + (long long)c * a.out_ch] = v;
      }
    }
  }
}

// n2p_attend_bwd_kernel (backward.cu) up to the scatter, statement for statement: the probabilities and their
// gradients are recomputed the same way, dq is the same slot-order fmaf chain, and p_ij / ds_ij are written per edge
// and head instead of being multiplied into atomics.  P / DS: (B,N,K,heads).
template <class I, int KMAX>
__global__ void __launch_bounds__(256) n2p_attend_bwd_edges_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                   const float* __restrict__ v, long long ld, const I* __restrict__ idx,
                                                                   int N, int C, int K, int lph, int heads, float sqrt_d,
                                                                   const float* __restrict__ go, long long ld_go, float* __restrict__ gq,
                                                                   long long ld_g, float* __restrict__ P, float* __restrict__ DS) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int n = blockIdx.x * 8 + warp;
  if (n >= N) return;
  const bool on = lane * 4 < C;
  const bool writer = on && (lane & (lph - 1)) == 0;           // first lane of its head
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
    lg[j] = p;
    s += p;
    pd = fmaf(p, dp[j], pd);
  }
  const float inv_s = 1.f / s;
  pd *= inv_s;
  float4 dq = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    if (j < K) {
      const int nj = __shfl_sync(kFull, my, j);
      const float p = lg[j] * inv_s;
      const float ds = p * (dp[j] - pd) / sqrt_d;
      if (on) {
        const float4 k4 = __ldg(reinterpret_cast<const float4*>(k + ((long long)b * N + nj) * ld + lane * 4));
        dq.x = fmaf(ds, k4.x, dq.x), dq.y = fmaf(ds, k4.y, dq.y), dq.z = fmaf(ds, k4.z, dq.z), dq.w = fmaf(ds, k4.w, dq.w);
      }
      if (writer) {
        const long long o = (row * K + j) * heads + lane / lph;
        P[o] = p;
        DS[o] = ds;
      }
    }
  }
  if (on) *reinterpret_cast<float4*>(gq + row * ld_g + lane * 4) = dq;
}

}  // namespace samble

using namespace samble;

extern "C" size_t samble_reverse_index_workspace_bytes(int B, int N) {
  if (B <= 0 || N <= 0) return 0;
  return (size_t)B * kRevWarps * (size_t)N * sizeof(int);
}

extern "C" int samble_reverse_index(const void* idx, int idx_bits, int B, int N, int R, int* offsets, int* edges, void* ws,
                                    size_t ws_bytes, samble_stream_t stream) {
  SAMBLE_REQUIRE(idx && offsets && edges && ws, "samble_reverse_index: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && R > 0, "samble_reverse_index: bad shape");
  SAMBLE_REQUIRE(idx_bits == 32 || idx_bits == 64, "samble_reverse_index: idx_bits must be 32 or 64");
  if (ws_bytes < samble_reverse_index_workspace_bytes(B, N)) {
    set_error("samble_reverse_index: workspace %zu < %zu bytes", ws_bytes, samble_reverse_index_workspace_bytes(B, N));
    return SAMBLE_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  SAMBLE_PRE(st);
  if (idx_bits == 64)
    reverse_index_kernel<long long><<<B, kRevWarps * 32, 0, st>>>((const long long*)idx, N, R, offsets, edges, (int*)ws);
  else
    reverse_index_kernel<int><<<B, kRevWarps * 32, 0, st>>>((const int*)idx, N, R, offsets, edges, (int*)ws);
  SAMBLE_LAUNCHED("reverse_index_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_scatter_rows_ordered(const float* x, long long x_batch, long long x_row, long long x_ch, int src_div,
                                           const float* w, int heads, const int* offsets, const int* edges, const float* sub,
                                           long long sub_batch, long long sub_row, int B, int N, int R, int C, float* out,
                                           long long out_batch, long long out_row, long long out_ch, samble_stream_t stream) {
  SAMBLE_REQUIRE(x && offsets && edges && out, "samble_scatter_rows_ordered: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && R > 0 && C > 0 && src_div > 0, "samble_scatter_rows_ordered: bad shape");
  SAMBLE_REQUIRE(!w || (heads > 0 && C % heads == 0), "samble_scatter_rows_ordered: C=%d must be a multiple of heads=%d", C, heads);
  ScatterArgs a{x, x_batch, x_row, x_ch, src_div, w, w ? heads : 1, w ? C / heads : C, offsets, edges, sub, sub_batch, sub_row,
                N, R, C, out, out_batch, out_row, out_ch};
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(ceil_div(N, 8), B);
  SAMBLE_PRE(st);
  scatter_rows_ordered_kernel<<<grid, 256, 0, st>>>(a);
  SAMBLE_LAUNCHED("scatter_rows_ordered_kernel");
  return SAMBLE_OK;
}

extern "C" int samble_n2p_attend_backward_edges(const float* q, const float* k, const float* v, long long ld, const void* idx,
                                                int idx_bits, int B, int N, int C, int K, int heads, const float* grad_out,
                                                long long ld_go, float* grad_q, long long ld_g, float* p, float* ds,
                                                samble_stream_t stream) {
  SAMBLE_REQUIRE(q && k && v && idx && grad_out && grad_q && p && ds, "samble_n2p_attend_backward_edges: null pointer");
  SAMBLE_REQUIRE(B > 0 && N > 0 && K > 0 && K <= 32, "samble_n2p_attend_backward_edges: bad shape (K <= 32)");
  SAMBLE_REQUIRE(C > 0 && C % 4 == 0 && C <= 128, "samble_n2p_attend_backward_edges: C=%d must be a multiple of 4, <= 128", C);
  SAMBLE_REQUIRE(heads > 0 && C % heads == 0 && (C / heads) % 4 == 0, "samble_n2p_attend_backward_edges: C/heads must be a multiple of 4");
  const int lph = C / heads / 4;
  SAMBLE_REQUIRE((lph & (lph - 1)) == 0, "samble_n2p_attend_backward_edges: (C/heads)/4 = %d must be a power of two", lph);
  SAMBLE_REQUIRE(ld % 4 == 0 && ld_go % 4 == 0 && ld_g % 4 == 0, "samble_n2p_attend_backward_edges: leading dimensions must be multiples of 4");
  SAMBLE_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)grad_out | (uintptr_t)grad_q) % 16 == 0,
                 "samble_n2p_attend_backward_edges: 16-byte alignment required");
  SAMBLE_REQUIRE(idx_bits == 32 || idx_bits == 64, "samble_n2p_attend_backward_edges: idx_bits must be 32 or 64");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(ceil_div(N, 8), B);
  const float sqrt_d = sqrtf((float)(C / heads));
  SAMBLE_PRE(st);
  if (idx_bits == 64)
    n2p_attend_bwd_edges_kernel<long long, 32><<<grid, 256, 0, st>>>(q, k, v, ld, (const long long*)idx, N, C, K, lph, heads, sqrt_d,
                                                                     grad_out, ld_go, grad_q, ld_g, p, ds);
  else
    n2p_attend_bwd_edges_kernel<int, 32><<<grid, 256, 0, st>>>(q, k, v, ld, (const int*)idx, N, C, K, lph, heads, sqrt_d, grad_out,
                                                               ld_go, grad_q, ld_g, p, ds);
  SAMBLE_LAUNCHED("n2p_attend_bwd_edges_kernel");
  return SAMBLE_OK;
}
