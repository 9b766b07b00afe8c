/*
 * samble_b200.h -- C ABI of the B200-native SAMBLE neighbourhood + sampling hot path.
 *
 * The reference (stevenczwu/SAMBLE) has no native code: its hot path is a Python
 * namespace (utils/ops.py) plus four nn.Modules.  Each entry point below replaces the
 * ATen call sequence of ONE reference function; the reference lines it replaces are
 * cited as file:line (paths relative to the upstream repository root).  The Python
 * binding a maintainer would add is shown in INTEGRATION.md (ctypes, no torch types
 * in any signature).
 *
 * Conventions
 *   - All pointers are DEVICE pointers into caller-owned, contiguous buffers unless
 *     a leading dimension (`ld*`, in elements) is given.  fp32 data, row-major.
 *   - "channel-major" = (B, C, N) as the reference's models pass clouds around;
 *     "point-major"   = (B, N, C).
 *   - Index tensors are int64 (the reference's dtype, torch.topk) when idx_bits==64,
 *     or int32 when idx_bits==32 (internal fast path; halves index traffic).
 *   - `ws` is caller-owned scratch of at least the matching *_workspace_bytes();
 *     the library never allocates, never synchronises, never touches the default
 *     stream: every kernel goes to `stream`, so calls are CUDA-graph capturable.
 *   - Return value: 0 on success, <0 on failure (SAMBLE_E_*).  Nothing throws.
 *     samble_last_error() returns a thread-local description of the last failure.
 */
#ifndef SAMBLE_B200_H_
#define SAMBLE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* samble_stream_t; /* cudaStream_t */

enum {
  SAMBLE_OK = 0,
  SAMBLE_E_INVALID = -1,   /* bad argument (shape, k, alignment, null pointer) */
  SAMBLE_E_WORKSPACE = -2, /* ws too small */
  SAMBLE_E_CUDA = -3       /* launch failed; see samble_last_error() */
};

enum { SAMBLE_GROUP_NEIGHBOR = 0, SAMBLE_GROUP_DIFF = 1, SAMBLE_GROUP_CENTER_NEIGHBOR = 2, SAMBLE_GROUP_CENTER_DIFF = 3 };

int samble_abi_version(void);
const char* samble_last_error(void);
/* number of kernel launches issued by this library on the calling thread since the
 * last reset (bench.py's gpu_launches claim is read from here). */
long long samble_launch_count(void);
void samble_reset_launch_count(void);
/* optional per-kernel device timing: while enabled every launch is bracketed by CUDA events on its
 * stream; samble_profile_report() waits for them and writes "kernel,launches,total_ms" lines. */
void samble_profile_enable(int on);
int samble_profile_report(char* buf, size_t cap);

/* hardware self-test of the tcgen05 path (descriptors, 128B swizzle, TMEM mapping): D (128x128) =
 * A (128xK) * B(128xK)^T with kind::tf32, fp32 accumulate.  K % 32 == 0, K <= 192. */
int samble_selftest_tc_gemm(const float* A, const float* B, int K, float* D, const float* Ax /* 128x8 or NULL */,
                            const float* Bx /* 128x8 or NULL: adds Ax*Bx^T from a non-swizzled slice */,
                            samble_stream_t stream);

/* the same product with the A operand read from TENSOR MEMORY (parked there with tcgen05.st): the form csrc/mlp2.cu uses to
 * feed the hidden activations of a two-layer point-wise MLP to its second GEMM.  K % 32 == 0, K <= 256.  iters > 0 repeats
 * the MMA sequence (D = iters * A B^T) on `ctas` CTAs and writes the SM cycles of each to cycles_out (may be NULL). */
int samble_selftest_tc_gemm_ts(const float* A, const float* B, int K, float* D, int iters, int ctas, long long* cycles_out,
                               samble_stream_t stream);

/* ... and with bf16 operands (kind::f16): A, B are rounded to bf16; A sits in tensor memory two K elements per 32-bit column (the form
 * the feature kNN uses for its query tile), or in shared memory when a_in_smem != 0 (for the rate comparison).  K % 64 == 0, K <= 256. */
int samble_selftest_tc_gemm_ts_bf16(const float* A, const float* B, int K, float* D, int iters, int ctas, long long* cycles_out,
                                    int a_in_smem, samble_stream_t stream);

/* issue-rate probe: `ctas` CTAs each issue iters*4 back-to-back kind::tf32 128 x n_tile x 8 MMAs on resident smem tiles;
 * cycles_out[cta] = SM cycles from first issue to completion (DESIGN.md: measured tensor-pipe ceiling of the SS form). */
int samble_selftest_mma_rate(int n_tile, int iters, int ctas, long long* cycles_out, samble_stream_t stream);

/* extended probe: kind 1 = bf16 (kind::f16, K=16 per MMA), 2 = tf32 (K=8); the MMAs rotate over n_acc accumulators of n_tile columns
 * (n_acc * n_tile <= 512) and n_a distinct A tiles -- the issue pattern of the exact-product GEMM. */
int samble_selftest_mma_rate_ex(int kind, int n_tile, int n_acc, int n_a, int iters, int ctas, long long* cycles_out,
                                samble_stream_t stream);

/* ---------------------------------------------------------------- kNN ----------
 * utils/ops.py:17-44  knn(a, b, k) -> (distance, idx).
 * a: queries, b: candidates; element (bi, n, c) lives at base + bi*a_sb + n*a_sn + c*a_sc
 * (strides in elements), so both the (B,N,C) tensors of ops.knn and the (B,C,N)
 * tensors of ops.select_neighbors (:50, a permute view) are passed without a copy.
 * Both clouds are centred/scaled by a's statistics (:23-29).  Distances use the GEMM
 * form of torch.cdist (:35) in fp32; selection is the k smallest, nearest first,
 * ties broken by lower index.  b == a (same pointer+strides) is the self-kNN case.
 * idx_out: (B,Nq,k) int32|int64.  dist_out: (B,Nq,k) fp32 NEGATIVE Euclidean
 * distance in normalised units (what :43 returns), or NULL.
 * Limits: 1 <= k <= 32, k <= Nr, C <= 512.
 *
 * C <= 3 runs the FFMA xyz kernel.  4 <= C <= 128 runs the tcgen05 path (split-bf16 contraction -> candidate set ->
 * exact fp32 re-rank; output identical to the exact kernel); larger C runs the exact FFMA tile kernel.
 * samble_set_knn_mode: 0 = auto (default), 1 = exact FFMA kernels only (used by the tests as the cross-check).
 *
 * flags: 0, or SAMBLE_KNN_ANY_ORDER (dist_out must be NULL): the k indices of each row are the same SET but in no
 * particular order.  Every consumer on the path reduces over the neighbours (max, softmax-weighted sum, scatter),
 * so the blocks ask for this; the tcgen05 path then computes exact distances only for the few candidates whose approximate
 * score is within the error margin of the k-th (knn_select_kernel) instead of for the whole candidate list. */
#define SAMBLE_KNN_ANY_ORDER 1
void samble_set_knn_mode(int mode);
size_t samble_knn_workspace_bytes(int B, int Nq, int Nr, int C);
int samble_knn(const float* a, long long a_sb, long long a_sn, long long a_sc,
               const float* b, long long b_sb, long long b_sn, long long b_sc,
               int B, int Nq, int Nr, int C, int k,
               void* idx_out, int idx_bits, float* dist_out, int flags,
               void* ws, size_t ws_bytes, samble_stream_t stream);

/* ------------------------------------------------------------- gathers ----------
 * utils/ops.py:5-14  index_points(points (B,N,C), idx (B,M,K)) -> (B,M,K,C).
 * R = M*K rows per cloud. */
int samble_index_points(const float* points, const void* idx, int idx_bits, int B, int N, int C, int R,
                        float* out, samble_stream_t stream);
/* 0 (default): rows move through the copy engine (cp.async.bulk loads into a shared-memory tile, one bulk store per tile) when they
 * are 16-byte aligned; 1: the thread-copy kernel only (cross-check). */
void samble_set_gather_mode(int mode);

/* utils/ops.py:47-65,83-112  select_neighbors/group, AFTER the kNN.
 * pcd (B,C,N) channel-major, idx (B,N,K).
 * type NEIGHBOR|DIFF: out is (B,N,K,C) contiguous -- the reference returns exactly this
 *   memory as a permuted (B,C,N,K) view (:57,:60).
 * type CENTER_*: out is (B,2C,N,K) contiguous (torch.cat, :98-107). */
int samble_group(const float* pcd, const void* idx, int idx_bits, int B, int C, int N, int K, int type,
                 float* out, samble_stream_t stream);

/* utils/ops.py:136-145  gather_by_idx(pcd (B,C,N), idx (B,1,M)) -> (B,C,M). */
int samble_gather_by_idx(const float* pcd, const void* idx, int idx_bits, int B, int C, int N, int M,
                         float* out, samble_stream_t stream);

/* (B,R,C) -> contiguous (B,C,R); input rows in_row_stride floats apart (unit inner stride), matrices in_batch_stride
 * floats apart (so a column slice of a wider row-major buffer is accepted): the change between the
 * reference's channel-major (B,C,N) clouds and the point-major rows the kernels consume (x.permute(0,2,1) in
 * utils/ops.py:50, models/attention.py:165-170). */
int samble_transpose(const float* in, long long in_batch_stride, long long in_row_stride, int B, int R, int C, float* out,
                     samble_stream_t stream);

/* ---- backward of the gathers (SURVEY 8 row f1; the reference relies on ATen autograd of torch.gather, utils/ops.py:13,144).
 * grad_points (B,N,C) / grad_pcd (B,C,N) must be zero-initialised (or hold a gradient to accumulate into); fp32 atomics. */
int samble_index_points_backward(const float* grad_out, const void* idx, int idx_bits, int B, int N, int C, int R,
                                 float* grad_points, samble_stream_t stream);
int samble_gather_by_idx_backward(const float* grad_out, const void* idx, int idx_bits, int B, int C, int N, int M,
                                  float* grad_pcd, samble_stream_t stream);

/* utils/ops.py:125-133  neighbor_mask: dense 0/1 (B,N,N) from idx (B,N,K) (zeros + scatter_). */
int samble_neighbor_mask(const void* idx, int idx_bits, int B, int N, int K, float* out, samble_stream_t stream);

/* --------------------------------------------------- point-wise linear layers ----
 * The 1x1 convolutions / Linear layers over the points of a cloud (models/attention.py:171-191,
 * downsample.py:124-137, upsample.py:150-160, seg_model.py:141-160) as one tcgen05 GEMM with fp32-class accuracy
 * (3xTF32 operand split) and a fused epilogue:
 *   acc = X W^T ;  y = [ (acc (+res if residual_first)) * scale[c] + shift[b?][c] ] -> LeakyReLU(0.2) if lrelu -> (+res)
 * X: M x K.  row-major (x_channel_major=0): X[m*ldx + k]; channel-major: X[(b*K + k)*P + n] with m = b*P + n,
 * P = points_per_cloud.  W: Nout x K row-major (the stored conv/linear weight), rows zero-padded to a multiple of 4
 * columns; W_lo = W - tf32_trunc(W) (samble_split_tf32; weights are constants, split once).  scale/shift: [Nout] or NULL;
 * shift_cloud_stride != 0 selects a per-cloud shift row.  residual and out are each row-major (ld) or
 * channel-major (B, Nout, P). */
int samble_split_tf32(const float* x, float* lo, long long n, samble_stream_t stream);
int samble_linear(const float* X, long long ldx, int x_channel_major, const float* W, const float* W_lo, long long ldw,
                  const float* scale, const float* shift, long long shift_cloud_stride, int lrelu,
                  const float* residual, long long ldr, int residual_channel_major, int residual_first,
                  float* out, long long ldo, int out_channel_major, int M, int K, int Nout, int points_per_cloud,
                  samble_stream_t stream);

/* Two such layers back to back in ONE kernel, the hidden activation never written to memory (csrc/mlp2.cu):
 *   h   = LeakyReLU?( (X W1^T) * scale1[c] + shift1[b?][c] )                       M x Hd, lives in tensor memory only
 *   out = [ (h W2^T (+res if residual_first)) * scale2 + shift2[b?] ] -> LeakyReLU? -> (+res)
 * Neighbor2PointAttention's feed-forward with its residual + bn2 (models/attention.py:187-192: K1 = C = 128, Hd = 512,
 * N2 = 128) and the segmentation head's conv2 -> conv3 (models/seg_model.py:205-214: Hd = 1024, N2 = 256).
 * X: M x K1 row-major, K1 <= 128; W1: Hd x K1, W2: N2 x Hd (the stored weights, with their samble_split_tf32 companions);
 * Hd % 128 == 0; N2 = 128 or 256; scale / shift as in samble_linear (16-byte aligned; a *_cloud_stride != 0 selects a per-cloud
 * shift row and needs points_per_cloud % 128 == 0); residual / out row-major.  For N2 = 128 the result equals the two
 * samble_linear calls it replaces bit for bit (same products, same accumulation chains). */
int samble_mlp2(const float* X, long long ldx, int M, int K1, const float* W1, const float* W1_lo, long long ldw1, int Hd,
                const float* scale1, const float* shift1, long long shift1_cloud_stride, int lrelu1, const float* W2,
                const float* W2_lo, long long ldw2, int N2, const float* scale2, const float* shift2,
                long long shift2_cloud_stride, int lrelu2, const float* residual, long long ldr, int residual_first,
                float* out, long long ldo, int points_per_cloud, samble_stream_t stream);
void samble_set_mlp2_debug(int bits);   /* measurement switches, tools/probe_mlp2.py */
/* while non-NULL every samble_mlp2 CTA writes [total, wait weights, wait conversion, wait output drain, wait X] cycles of its
 * MMA-issuing thread to wait_cycles[5 * cta] (device memory, 5 * 148 entries) */
void samble_set_mlp2_probe(long long* wait_cycles);

/* The same layer followed by max and/or mean over the points of each cloud -- conv -> max/avg pool of
 * models/seg_model.py:199-203, cls_model.py:104/133 (res-link max), embedding.py:88-89 (STN) -- without ever storing
 * the (M x Nout) activation: the epilogue reduces each 32-row group in registers, a second tiny kernel combines the
 * groups of a cloud in a fixed order (deterministic).  X row-major; points_per_cloud a multiple of 32.
 * out_max / out_mean: (M / points_per_cloud, Nout), either may be NULL. */
/* Per-cloud products on the same kernel: rows m of cloud b = m / rows_per_cloud are multiplied by THAT cloud's matrix
 * W[b] (Nout x K, row pitch ldw, cloud pitch Nout*ldw; W_lo its samble_split_tf32 companion):  out[m] = X[m] W[b]^T.
 * With row_max/row_sum the epilogue turns the products into softmax rows whose statistics are already known,
 *   out = exp(acc / logit_div - row_max[m]) / row_sum[m],
 * which is how DownSampleToken's attention rows of the M selected points (models/downsample.py:242-252) are formed
 * from the row statistics of samble_ds_row_stats; a second call (X = those rows, W[b] = V[b]^T) applies them to V.
 * rows_per_cloud must be a multiple of 128. */
int samble_cloud_matmul(const float* X, long long ldx, const float* W, const float* W_lo, long long ldw, int M, int K, int Nout,
                        int rows_per_cloud, const float* row_max, const float* row_sum, float logit_div,
                        const float* residual, long long ldr, float* out, long long ldo, samble_stream_t stream);
/* residual (M x Nout, row pitch ldr) or NULL is added to the result (after the softmax transform, if any).
 *
 * samble_ds_select_rows gathers, for the M selected points idx (B,M) int64 of each cloud, what those two products need:
 * q_sel (B,M,D) = q rows, m_sel / s_sel (B,M) = their softmax statistics, and tok_mix (B,M,C) = the nb token columns'
 * share of the output, sum_t softmax(row)[N+t] * v_tok[t] (v_tok: (nb,C)), which the second product takes as residual. */
int samble_ds_select_rows(const float* q, long long ldq, const float* rowmax, const float* rowsum, const float* token_logits,
                          const float* v_tok, const long long* idx, int B, int N, int M, int D, int nb, int C,
                          float* q_sel, float* m_sel, float* s_sel, float* tok_mix, samble_stream_t stream);

size_t samble_linear_pool_workspace_bytes(int M, int Nout);
int samble_linear_pool(const float* X, long long ldx, const float* W, const float* W_lo, long long ldw,
                       const float* scale, const float* shift, long long shift_cloud_stride, int lrelu,
                       int M, int K, int Nout, int points_per_cloud, float* out_max, float* out_mean,
                       void* ws, size_t ws_bytes, samble_stream_t stream);

/* ------------------------------------------------------------ EdgeConv ----------
 * models/embedding.py:29-39 fused (eval mode): group -> conv1+BN+LeakyReLU(0.2) -> conv2+BN+LeakyReLU
 * -> max over K.  conv1 is linear in [x_i ; x_j - x_i], so the caller projects the N points once:
 *   pr (B,N,ld_pr) point-major = [P' | R'],  P'_i = a1*((W1a-W1b) x_i) + b1,  R'_j = a1*(W1b x_j)
 * (a1,b1 = folded BN1), w2 (C2,C1) = diag(a2) W2, b2 (C2) = folded BN2 shift.  idx (B,N,K) from the kNN.
 * out = lrelu(max_k (w2 . lrelu(P'_i + R'_idx[i,k]) + b2)): (B,C2,N) channel-major when out_ld == 0, point-major rows
 * out[(b*N + n)*out_ld + c] when out_ld >= C2 (a column slice of a wider row-major buffer: the concatenation of several
 * EdgeConv outputs, models/seg_model.py:98-102, then costs nothing).
 * Limits: K <= 32, C1 % 4 == 0, C1 <= 128, C2 in {32,64,128}.
 * C1 % 32 == 0 and C2 in {64,128} run on the tensor cores (tcgen05, 3xTF32 split, fp32-class accuracy);
 * samble_set_edge_mode(1) forces the FFMA kernel (used by the tests as the cross-check). */
void samble_set_edge_mode(int mode);
/* measurement only (tools/probe_edge.py): disable phases of edge_mlp_tc_kernel (1 gathers, 8 stage build, 2 MMAs, 4 epilogue). */
void samble_set_edge_debug(int bits);
int samble_edge_mlp_max(const float* pr, long long ld_pr, const void* idx, int idx_bits, const float* w2,
                        const float* b2, int B, int N, int K, int C1, int C2, float* out, long long out_ld, samble_stream_t stream);

/* ------------------------------------------------- Neighbor2Point attention -----
 * models/attention.py:165-185,207-250 (scalar_dot, asm "dot"), with the bias-free
 * k/v convolutions hoisted out of the neighbour dimension:
 *   W(x_j - x_i) = W x_j - W x_i, and softmax over j is invariant to the -q.Wk x_i shift.
 * q,k,v: point-major (B,N,C) with leading dimension ld (elements per point), i.e. the
 * projections of the N points themselves; idx (B,N,K) from the kNN on x.
 * out (B,N,C) point-major: att_i = sum_j softmax_j(q_i.k_j/sqrt(C/H)) v_j - v_i per head;
 * optional fused tail of attention.py:187 (eval): out = (residual_i + att_i) * scale + shift  (BN1 folded). */
int samble_n2p_attend(const float* q, const float* k, const float* v, long long ld,
                      const void* idx, int idx_bits, int B, int N, int C, int K, int heads,
                      const float* residual, long long ld_res, const float* scale, const float* shift,
                      float* out, long long ld_out, samble_stream_t stream);

/* measurement only (tools/probe_knn.py): low byte: disable phases of knn_tc_kernel (1 MMAs, 2 epilogue; results are garbage
 * while set); bits 8..: CTAs per cluster forced to 1, 2 or 4 (0 = automatic). */
void samble_set_knn_debug(int bits);
/* while non-NULL the tensor-core kNN launches write 8 cycle counters per CTA (device memory, 8 * CTAs entries): MMA thread total,
 * its waits for operands / accumulator drain / query tile, the epilogue's wait for accumulators, producer total, its wait for free stages */
void samble_set_knn_probe(long long* cycles);

/* measurement only (tools/probe_linear.py): disable phases of linear_tma_kernel (1 operand split, 2 epilogue, 4 MMAs);
 * results are garbage while any bit is set.  0 = normal. */
void samble_set_linear_debug(int bits);

/* 0 (default): eight-lanes-per-point kernel when the shape allows; 1: the warp-per-point kernel only (cross-check). */
void samble_set_n2p_mode(int mode);

/* backward of samble_n2p_attend without the fused tail (models/attention.py:207-250 under autograd): grad_out (B,N,C) with leading
 * dimension ld_go -> grad_q (written), grad_k / grad_v (ACCUMULATED with fp32 atomics: zero them first), all with leading
 * dimension ld_g.  Recomputes the probabilities from q, k (no (B,N,K) tensor is saved by the forward pass). */
int samble_n2p_attend_backward(const float* q, const float* k, const float* v, long long ld, const void* idx, int idx_bits,
                               int B, int N, int C, int K, int heads, const float* grad_out, long long ld_go,
                               float* grad_q, float* grad_k, float* grad_v, long long ld_g, samble_stream_t stream);

/* ---- ordered backward scatters (csrc/backward_ordered.cu): the same gradients as the atomic entry points above with a
 * defined summation order, so they are bitwise reproducible (what the Python layer runs under
 * torch.use_deterministic_algorithms(True)).  For cloud b, edge e in [0,R) has target t_e = idx[b,e]; L_j lists the edges
 * with target j in ascending e.  Each output element is the fp32 left fold, every product and sum rounded on its own:
 *   acc = 0;  for e in L_j: acc = acc + term_e;   out[b,j,c] = acc  (or acc - sub[b,j,c])
 *   term_e = x[b, e/src_div, c]   or, with a weight,   w[b,e,c/(C/heads)] * x[b, e/src_div, c].
 * Entries of idx outside [0,N) contribute nothing.
 *
 * samble_reverse_index: idx (B,R) int32/int64 -> offsets (B,N+1) int32 and edges (B,R) int32, the edges of target j at
 * edges[b, offsets[b,j] .. offsets[b,j+1]) in ascending e (a stable counting sort, one CTA per cloud); slots past
 * offsets[b,N] (out-of-range entries) are set to -1.  ws: samble_reverse_index_workspace_bytes(B, N). */
size_t samble_reverse_index_workspace_bytes(int B, int N);
int samble_reverse_index(const void* idx, int idx_bits, int B, int N, int R, int* offsets, int* edges, void* ws, size_t ws_bytes,
                         samble_stream_t stream);
/* samble_scatter_rows_ordered: the fold above, WRITING out (every element of out (B,N,C) is written; nothing needs zeroing).
 * x element (b, row, c) at x[b*x_batch + row*x_row + c*x_ch], out likewise with out_*: row-major and channel-major layouts
 * and column slices of wider buffers are all strides.  w (B,R,heads) contiguous or NULL; sub (B,N,C) with unit channel
 * stride at sub[b*sub_batch + j*sub_row + c], or NULL.  One warp per target row: its time is proportional to the largest
 * in-degree, so a hub target that every edge lists runs as one serial fold. */
int samble_scatter_rows_ordered(const float* x, long long x_batch, long long x_row, long long x_ch, int src_div,
                                const float* w, int heads, const int* offsets, const int* edges, const float* sub,
                                long long sub_batch, long long sub_row, int B, int N, int R, int C, float* out,
                                long long out_batch, long long out_row, long long out_ch, samble_stream_t stream);
/* samble_n2p_attend_backward_edges: samble_n2p_attend_backward's per-edge pass without its scatter.  Same arguments and limits;
 * writes grad_q (ld_g) and, per edge e = n*K + slot and head h, p[(b*N*K + e)*heads + h] = p_ij and ds[...] = ds_ij, the very
 * fp32 values the atomic kernel multiplies into its atomics.  Then, with the reverse index of idx (R = N*K):
 *   grad_k = samble_scatter_rows_ordered(x = q,        src_div = K, w = ds)
 *   grad_v = samble_scatter_rows_ordered(x = grad_out, src_div = K, w = p, sub = grad_out). */
int samble_n2p_attend_backward_edges(const float* q, const float* k, const float* v, long long ld, const void* idx, int idx_bits,
                                     int B, int N, int C, int K, int heads, const float* grad_out, long long ld_go,
                                     float* grad_q, long long ld_g, float* p, float* ds, samble_stream_t stream);

/* --------------------------------------------------- DownSampleToken scoring ----
 * models/downsample.py:124-153: energy = q @ [k | k_tok] / sqrt(D), row softmax over
 * N+nb columns.  The N x (N+nb) map is never written: this pass leaves per-row
 * max and sum-of-exp plus the PRE-softmax token columns (:149-152).
 * q,k: point-major (B,N,D) with leading dims; k_tok: (nb,D) (tokens are shared by the
 * batch, :116).  rowmax,rowsum: (B,N).  token_logits: (B,N,nb).
 * D % 32 == 0, D <= 128, nb <= 8 runs on the tensor cores (tcgen05, 3xTF32 split); samble_set_ds_mode(1) forces the
 * exact FFMA tile kernel (cross-check in the tests; bit-consistent logits with samble_ds_edge_score). */
void samble_set_ds_mode(int mode);
int samble_ds_row_stats(const float* q, long long ldq, const float* k, long long ldk, const float* k_tok,
                        int B, int N, int D, int nb, float* rowmax, float* rowsum, float* token_logits,
                        samble_stream_t stream);

/* The same statistics on the TMA-fed linear kernel (linear_tma.cu): the point columns are the per-cloud product
 * q[b] k[b]^T with a row-statistics epilogue, merged with the token columns by a small second kernel.  k_lo is k's
 * samble_split_tf32 companion (same pitch); N must be a multiple of 128.  ~2x faster than the kernel above. */
size_t samble_ds_row_stats_fast_workspace_bytes(int B, int N);
int samble_ds_row_stats_fast(const float* q, long long ldq, const float* k, const float* k_lo, long long ldk,
                             const float* k_tok, int B, int N, int D, int nb, float* rowmax, float* rowsum,
                             float* token_logits, void* ws, size_t ws_bytes, samble_stream_t stream);

/* ------------------------------------------- exact-product tensor-core GEMM -----
 * The two contractions that decide DownSampleToken's sampled indices -- the q/k/v projection and q k^T
 * (models/downsample.py:124-143) -- with an accumulation that is exact on the bf16 tensor cores (csrc/xgemm.cu):
 * every operand is cut, per cloud, into three signed 8-bit digits stored as bf16 integers; the digit products are summed
 * exactly by tcgen05.mma (integers < 2^23) and recombined with two fp32 roundings.  Result: fp32-class accuracy
 * independent of summation order, bit-identical to an int32 restatement (reference != 0 runs that restatement).
 *
 * samble_digits: x (B, R, C) rows (row pitch ld, cloud pitch batch_stride, floats) -> planes: 3 x (B, R, Cp) bf16,
 * Cp = C rounded up to 64, and scale[b].  The per-cloud magnitude comes from amax_in[b * amax_stride] (bits of max|x|,
 * e.g. written by samble_xgemm's amax_out) or, when amax_in is NULL, from a reduction pass using amax_scratch[B]. */
size_t samble_digits_bytes(int B, int R, int C);
int samble_digits(const float* x, long long ld, long long batch_stride, int B, int R, int C, const unsigned* amax_in,
                  int amax_stride, void* planes, float* scale, unsigned* amax_scratch, samble_stream_t stream);
/* out[(b*Ra + i)*ldo + j] = <A[b,i,:], B[b or 0, j, :]>, A: Ba clouds of Ra rows, B: Bb (== Ba, or 1 = shared) sets of Rb
 * rows, C <= 128 channels.  amax_out (or NULL): [Ba][ceil(Rb/amax_group)] bits of max|out| per cloud and column group
 * (amax_group a multiple of 32), zeroed by the call. */
int samble_xgemm(const void* a_planes, const float* a_scale, int Ba, int Ra, const void* b_planes, const float* b_scale,
                 int Bb, int Rb, int C, float* out, long long ldo, unsigned* amax_out, int amax_group, int reference,
                 samble_stream_t stream);
/* DownSampleToken pass 1 (models/downsample.py:139-153) on that GEMM: row max / sum-of-exp of q k^T / sqrt(D) over the N
 * point columns from the digit planes of q and k, merged with the nb token columns (exact fp32 dot products of the fp32
 * q rows with k_tok, written to token_logits).  Any N. */
size_t samble_ds_row_stats_exact_workspace_bytes(int B, int N);
int samble_ds_row_stats_exact(const void* q_planes, const float* q_scale, const void* k_planes, const float* k_scale,
                              const float* q, long long ldq, const float* k_tok, int B, int N, int D, int nb,
                              float* rowmax, float* rowsum, float* token_logits, void* ws, size_t ws_bytes,
                              samble_stream_t stream);

/* models/downsample.py:242-252 fused flash-style (csrc/ds_attend.cu): out[b, m, :] = softmax(q[idx[b,m]] [k | k_tok]^T / sqrt(D)) . [v ; v_tok]
 * for the M selected points, from the digit planes of q and k (samble_digits), the fp32 v rows (B, N, C; row pitch ldv),
 * the row statistics and token logits of samble_ds_row_stats_exact and v_tok (nb, C).  No (B, M, N) tensor is formed:
 * S = Q_sel K^T tiles live in TMEM, P = exp(S/sqrt(D) - max)/sum goes through shared memory as the A operand of the
 * second MMA.  out: (B, M, C) rows.  ws: V^T as bf16 hi/lo planes. */
size_t samble_ds_attend_rows_workspace_bytes(int B, int N, int C);
int samble_ds_attend_rows(const void* q_planes, const float* q_scale, const void* k_planes, const float* k_scale,
                          const float* v, long long ldv, const long long* idx, const float* rowmax, const float* rowsum,
                          const float* token_logits, const float* v_tok, int B, int N, int M, int D, int C, int nb,
                          float* out, void* ws, size_t ws_bytes, samble_stream_t stream);

/* models/downsample.py:300-344 (idx_mode sparse_col_sqr) without the dense mask:
 *   score[j] = sum_{i : j in kNN(i)} softmax_i[j] / indeg(j)^2,  NaN -> 0.
 * Only the N*K edges are evaluated; accumulation order is fixed (deterministic). */
size_t samble_ds_edge_score_workspace_bytes(int B, int N);
int samble_ds_edge_score(const float* q, long long ldq, const float* k, long long ldk,
                         const float* rowmax, const float* rowsum, const void* idx, int idx_bits,
                         int B, int N, int D, int K, float* score, void* ws, size_t ws_bytes,
                         samble_stream_t stream);

/* ------------------------------------------------ bins, k per bin, sampling -----
 * utils/ops.py:450-452  z = (s - mean) / std_population over the N points of each row. */
int samble_zscore(const float* score, int rows, int N, float* z, samble_stream_t stream);

/* utils/ops.py:460-462  mask[r,n,j] = z < upper[j] && z >= lower[j]  (uint8 0/1). */
int samble_bin_mask(const float* z, const float* upper, const float* lower, int rows, int N, int nb,
                    uint8_t* mask, samble_stream_t stream);

/* utils/ops.py:385-432  calculate_num_points_to_choose. bin_prob (B,nb) fp32,
 * max_num_points (B,nb) int64 -> k (B,nb) int32, op-for-op in fp32 (same summation
 * order, truncation and first-argmax remainder rule). nb <= 8. */
int samble_num_points_to_choose(const float* bin_prob, const long long* max_num_points, int B, int nb, int total,
                                int* k_out, samble_stream_t stream);

/* utils/ops.py:476-505  generating_downsampled_index, 'topk' branch.
 * score (B,N), mask (B,N,nb) uint8, k (B,nb) int32 -> idx (B,M) int64:
 * bins in order, inside a bin descending (score+1e-8)*mask, ties by lower index. */
int samble_downsample_index_topk(const float* score, const uint8_t* mask, const int* k, int B, int N, int nb, int M,
                                 long long* idx_out, samble_stream_t stream);

/* models/downsample.py:205-240 fused for the shipped configuration (mean_relu,
 * multi_token, topk): z-score -> bins by `cuts` (nb-1 descending thresholds, device) ->
 * per-bin mean of token logits -> k per bin -> per-bin top-k.
 * Outputs: idx (B,M) int64; bin_id (B,N) uint8 (255 = in no bin); counts (B,nb) int32;
 * k_out (B,nb) int32; w_raw (B,nb) fp32 (bin_weights_beforerelu); z (B,N) or NULL. */
int samble_ds_sample(const float* score, const float* token_logits, const float* cuts,
                     int B, int N, int nb, int M,
                     long long* idx_out, uint8_t* bin_id, int* counts, int* k_out, float* w_raw, float* z_out,
                     samble_stream_t stream);

/* utils/ops.py:507-592: the per-(cloud, bin) categorical distributions of the 'uniform' (mode 0) / 'random' (mode 1) sampling
 * modes, p (B, nb, N) row-major (= p.permute(0,2,1).reshape(-1,N) of the reference), from score (B,N) and the membership mask
 * (B,N,nb) uint8.  random: exp(tanh(zscore(score)) * inv_t) restricted to the bin and normalised, NaN -> 1e-8, with
 * inv_t = count_of_bin / t_div when t_div > 0 (boltzmann modes 1 / 3: 100 / 200) and inv_t_const otherwise. */
int samble_sampling_probabilities(const float* score, const uint8_t* mask, int B, int N, int nb, int mode, float inv_t_const,
                                  float t_div, float* p, samble_stream_t stream);

/* utils/ops.py:174-236 dynamic bin boundaries, the two steps around the rank average (:191-199):
 * samble_quantile_pick: cut[j-1] = sorted_desc[int(j / nb * n)], j = 1..nb-1 (:182-189);
 * samble_boundary_ema: cut = cut_sum / world, blended into upper[1:] / lower[:-1] (nb floats each, +-inf sentinels kept or
 * created) with the momentum factor when has_old (:201-233), rounded as ATen rounds these statements on CUDA: momentum is
 * the Python float (double) the reference multiplies by, and 1 - momentum is formed in double before rounding to fp32. */
int samble_quantile_pick(const float* sorted_desc, long long n, int nb, float* cut, samble_stream_t stream);
int samble_boundary_ema(const float* cut_sum, int world, double momentum, int has_old, int nb, float* upper, float* lower,
                        samble_stream_t stream);

/* ------------------------------------------------------------- UpSample ---------
 * models/upsample.py:194-212 + utils/ops.py:68-80 fused: 3-NN of each of the N "up"
 * points among the M selected points in xyz (normalised by the up cloud's statistics,
 * ops.py:23-29), weights 1/(d+1e-8) normalised, weighted sum of the selected features.
 * xyz_up (B,3,N), xyz_sel (B,3,M), feat (B,C,M) channel-major -> out (B,C,N).
 * idx_out (B,N,3) int64 and dist_out (B,N,3) (positive) are optional (NULL). */
size_t samble_interpolate3_workspace_bytes(int B, int N, int M);
int samble_interpolate3(const float* xyz_up, const float* xyz_sel, const float* feat,
                        int B, int N, int M, int C, float* out, long long* idx_out, float* dist_out,
                        void* ws, size_t ws_bytes, samble_stream_t stream);
/* Same with point-major features: feat (B,M,C) rows ld_feat apart -> out (B,N,C) rows ld_out apart (so the result can be
 * written straight into the right half of the (B,N,2C) buffer that models/upsample.py:158 concatenates). */
int samble_interpolate3_rows(const float* xyz_up, const float* xyz_sel, const float* feat, long long ld_feat,
                             int B, int N, int M, int C, float* out, long long ld_out,
                             void* ws, size_t ws_bytes, samble_stream_t stream);

/* the two halves of samble_interpolate3_rows as separate calls: the 3-NN search needs the xyz sets only (so it can run beside
 * the convolution that produces feat), nn_idx (B,N,3) int32 / nn_w (B,N,3) normalised inverse-distance weights;
 * the gather then forms out[b,n,:] = sum_j nn_w[b,n,j] * feat[b, nn_idx[b,n,j], :]  (models/upsample.py:206-212). */
int samble_interpolate3_search(const float* xyz_up, const float* xyz_sel, int B, int N, int M, int* nn_idx, float* nn_w,
                               void* ws, size_t ws_bytes, samble_stream_t stream);
int samble_interpolate3_gather_rows(const int* nn_idx, const float* nn_w, const float* feat, long long ld_feat, int B, int N,
                                    int M, int C, float* out, long long ld_out, samble_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SAMBLE_B200_H_ */
