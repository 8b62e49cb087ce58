// Kernels of the history-feature / skip branches of RNNFullModel (model.py:354-358 x_to_z, :376-379 x_to_y with the
// OnlyNonZeroDiagonal constraint :48-66, :386-392 y_to_y) and of NoRecurrenceModel (model.py:264-319).  These models
// add per-(token, item) terms to the logits --  z = hs.W + x.B + A[y_{t-1}] (+ biases)  -- and the reference runs them on
// small catalogs only (a (V,V) transition kernel A; V = 17 for MSNBC), so the (N,V) logits ARE materialised here:
//   seqrec_add_rows              Z[n,:] += table[ids[n],:] (+ bias)        one-hot . A == row lookup (SURVEY D2)
//   seqrec_softmax_rows_stats    per-row (max, sum-exp) and target logit of materialised logits
//   seqrec_softmax_rows_dlogit   Z <- (softmax(Z) - onehot(y)) * coef      in place (un-normalised, like K6)
//   seqrec_softmax_rows_probs    (T,B,V) logits -> (B,T,V) probabilities   (model.predict)
//   seqrec_rows_rank             1-based rank of the target in each row    (Recall@k / MRR@k / NDCG@k)
//   seqrec_gemm_nt               C = A . B^T                               dH = dZ . W^T
//   seqrec_colsum                out[c] += sum_r in[r,c]                   bias gradients
//   seqrec_diag_constraint       W[skip + i, j] *= [i == j]                Keras constraint, applied after the update
#include "common.cuh"

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
add_rows_kernel(float* __restrict__ Z, const float* __restrict__ table, const float* __restrict__ bias,
                const int32_t* __restrict__ ids, int64_t n_tokens, int V) {
  const int64_t total = n_tokens * V;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / V;
    const int v = (int)(i - n * V);
    const int32_t id = ids ? ids[n] : -1;
    float add = bias ? __ldg(bias + v) : 0.f;
    if (id >= 0) add += __ldg(table + (size_t)id * V + v);
    Z[i] += add;
  }
}

extern "C" int seqrec_add_rows(float* Z, const float* table, const float* bias, const int32_t* ids, int64_t n_tokens,
                               int V, void* stream) {
  SEQREC_ARG(Z && n_tokens > 0 && V > 0 && (table || bias), 1);
  int64_t blocks = (n_tokens * V + 255) / 256;
  if (blocks > SEQREC_NUM_SMS * 16) blocks = SEQREC_NUM_SMS * 16;
  add_rows_kernel<<<(int)blocks, 256, 0, as_stream(stream)>>>(Z, table, bias, table ? ids : nullptr, n_tokens, V);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// one warp per token row
__global__ void __launch_bounds__(256)
softmax_rows_stats_kernel(const float* __restrict__ Z, const int32_t* __restrict__ tgt, float* __restrict__ m_out,
                          float* __restrict__ s_out, float* __restrict__ zy, int64_t n_tokens, int V) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (n >= n_tokens) return;
  const float* row = Z + n * V;
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, row[v]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s = 0.f;
  for (int v = lane; v < V; v += 32) s += expf(row[v] - mx);
  s = warp_sum(s);
  if (lane == 0) {
    m_out[n] = mx;
    s_out[n] = s;
    if (zy) {
      const int32_t t = tgt ? tgt[n] : -1;
      zy[n] = t >= 0 ? row[t] : 0.f;
    }
  }
}

extern "C" int seqrec_softmax_rows_stats(const float* Z, const int32_t* tgt, float* m, float* s, float* zy,
                                         int64_t n_tokens, int V, void* stream) {
  SEQREC_ARG(Z && m && s && n_tokens > 0 && V > 0, 1);
  softmax_rows_stats_kernel<<<ceil_div(n_tokens * 32, 256), 256, 0, as_stream(stream)>>>(Z, tgt, m, s, zy, n_tokens, V);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

__global__ void __launch_bounds__(256)
softmax_rows_dlogit_kernel(float* __restrict__ Z, const int32_t* __restrict__ tgt, const float* __restrict__ m,
                           const float* __restrict__ s, const float* __restrict__ coef, int64_t n_tokens, int V) {
  const int64_t total = n_tokens * V;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / V;
    const int v = (int)(i - n * V);
    const float cf = coef[n];
    float d = 0.f;
    if (cf != 0.f) d = (expf(Z[i] - m[n]) / s[n] - (tgt[n] == v ? 1.f : 0.f)) * cf;
    Z[i] = d;
  }
}

extern "C" int seqrec_softmax_rows_dlogit(float* Z, const int32_t* tgt, const float* m, const float* s,
                                          const float* coef, int64_t n_tokens, int V, void* stream) {
  SEQREC_ARG(Z && tgt && m && s && coef && n_tokens > 0 && V > 0, 1);
  int64_t blocks = (n_tokens * V + 255) / 256;
  if (blocks > SEQREC_NUM_SMS * 16) blocks = SEQREC_NUM_SMS * 16;
  softmax_rows_dlogit_kernel<<<(int)blocks, 256, 0, as_stream(stream)>>>(Z, tgt, m, s, coef, n_tokens, V);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// time-major logits (T,B,V) -> batch-major probabilities (B,T,V)
__global__ void __launch_bounds__(256)
softmax_rows_probs_kernel(const float* __restrict__ Z, const float* __restrict__ m, const float* __restrict__ s,
                          float* __restrict__ probs_btv, int T, int B, int V) {
  const int64_t total = (int64_t)T * B * V;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / V;
    const int v = (int)(i - n * V);
    const int t = (int)(n / B), b = (int)(n - (int64_t)t * B);
    probs_btv[((int64_t)b * T + t) * V + v] = expf(Z[i] - m[n]) / s[n];
  }
}

extern "C" int seqrec_softmax_rows_probs(const float* Z, const float* m, const float* s, float* probs_btv, int T, int B,
                                         int V, void* stream) {
  SEQREC_ARG(Z && m && s && probs_btv && T > 0 && B > 0 && V > 0, 1);
  int64_t blocks = ((int64_t)T * B * V + 255) / 256;
  if (blocks > SEQREC_NUM_SMS * 16) blocks = SEQREC_NUM_SMS * 16;
  softmax_rows_probs_kernel<<<(int)blocks, 256, 0, as_stream(stream)>>>(Z, m, s, probs_btv, T, B, V);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// one warp per row: rank[n] = 1 + #{v != y : Z[n,v] > Z[n,y]  or  (Z[n,v] == Z[n,y] and v < y)}, 0 for pads (y < 0).
// The reference value is read from the row itself, so ties are exact.
__global__ void __launch_bounds__(256)
rows_rank_kernel(const float* __restrict__ Z, const int32_t* __restrict__ tgt, int32_t* __restrict__ rank,
                 int64_t n_rows, int V) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (n >= n_rows) return;
  const int32_t y = tgt[n];
  if (y < 0 || y >= V) {
    if (lane == 0) rank[n] = 0;
    return;
  }
  const float* row = Z + n * V;
  const float zy = row[y];
  int c = 0;
  for (int v = lane; v < V; v += 32) {
    const float z = row[v];
    c += v != y && (z > zy || (z == zy && v < y));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) rank[n] = 1 + c;
}

extern "C" int seqrec_rows_rank(const float* Z, const int32_t* tgt, int32_t* rank, int64_t n_rows, int V,
                                void* stream) {
  SEQREC_ARG(Z && tgt && rank && n_rows > 0 && V > 0, 1);
  rows_rank_kernel<<<ceil_div(n_rows * 32, 256), 256, 0, as_stream(stream)>>>(Z, tgt, rank, n_rows, V);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// C[M,N] (=|+=) A[M,K] . B[N,K]^T   (64 x 64 tiles, 4 x 4 micro-tiles; fp32 SIMT like gemm.cu)
#define NT_T 64
#define NT_K 16
#define NT_P 68
__global__ void __launch_bounds__(256)
gemm_nt_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Bm, int ldb, float* __restrict__ C,
               int ldc, int M, int N, int K, int accumulate) {
  __shared__ __align__(16) float As[NT_K][NT_P];
  __shared__ __align__(16) float Bs[NT_K][NT_P];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * NT_T, n0 = blockIdx.x * NT_T;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += NT_K) {
    const int r = tid >> 2, kq = (tid & 3) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + kq + i;
      As[kq + i][r] = (m0 + r < M && k < K) ? A[(size_t)(m0 + r) * lda + k] : 0.f;
      Bs[kq + i][r] = (n0 + r < N && k < K) ? Bm[(size_t)(n0 + r) * ldb + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NT_K; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      if (accumulate) v += C[(size_t)m * ldc + n];
      C[(size_t)m * ldc + n] = v;
    }
  }
}

extern "C" int seqrec_gemm_nt(const float* A, const float* Bm, float* C, int M, int N, int K, int lda, int ldb, int ldc,
                              int accumulate, void* stream) {
  SEQREC_ARG(A && Bm && C && M > 0 && N > 0 && K > 0 && lda >= K && ldb >= K && ldc >= N, 1);
  dim3 grid(ceil_div(N, NT_T), ceil_div(M, NT_T));
  gemm_nt_kernel<<<grid, 256, 0, as_stream(stream)>>>(A, lda, Bm, ldb, C, ldc, M, N, K, accumulate);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ in, int ld, float* __restrict__ out, int64_t rows, int cols,
              int64_t rows_per_block) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int64_t r0 = blockIdx.y * rows_per_block;
  const int64_t r1 = min(rows, r0 + rows_per_block);
  float acc = 0.f;
  for (int64_t r = r0; r < r1; ++r) acc += in[r * ld + c];
  atomicAdd(out + c, acc);
}

extern "C" int seqrec_colsum(const float* in, float* out, int64_t rows, int cols, int ld, void* stream) {
  SEQREC_ARG(in && out && rows > 0 && cols > 0 && ld >= cols, 1);
  int64_t rpb = (rows + 63) / 64;
  if (rpb < 64) rpb = 64;
  dim3 grid(ceil_div(cols, 256), ceil_div(rows, rpb));
  colsum_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, ld, out, rows, cols, rpb);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// OnlyNonZeroDiagonal(input_dim, skip_cols) (model.py:48-66): the kernel (skip + dim, dim) keeps its first `skip` rows and
// only the diagonal of the (dim, dim) block below them.  Keras applies constraints to the UPDATED weights.
__global__ void __launch_bounds__(256)
diag_constraint_kernel(float* __restrict__ W, int skip, int dim) {
  const int64_t total = (int64_t)dim * dim;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / dim), c = (int)(i - (int64_t)r * dim);
    if (r != c) W[(size_t)(skip + r) * dim + c] = 0.f;
  }
}

extern "C" int seqrec_diag_constraint(float* W, int skip_rows, int dim, void* stream) {
  SEQREC_ARG(W && skip_rows >= 0 && dim > 0, 1);
  int64_t blocks = ((int64_t)dim * dim + 255) / 256;
  if (blocks > SEQREC_NUM_SMS * 16) blocks = SEQREC_NUM_SMS * 16;
  diag_constraint_kernel<<<(int)blocks, 256, 0, as_stream(stream)>>>(W, skip_rows, dim);
  SEQREC_CHECK_LAUNCH();
  return 0;
}
