// Sampled softmax with log-Q correction (the training objective of HotPath.set_loss("sampled_softmax")).
//
// A step draws S item ids s_1..s_S with replacement from q and scores every token against its target and those S
// shared items.  With log Q(v) = log(S q(v)) and o_v = h . W_out[:, v] + b_out[v]:
//     l_0 = o_y - log Q(y),   l_j = o_{s_j} - log Q(s_j)  (-inf where s_j == y: accidental hit),
//     loss_n = -l_0 + log sum_{j=0..S} exp(l_j)
// (TF sampled_softmax_loss with subtract_log_q and remove_accidental_hits; no probability clip).  The (N, S) logits are
// materialised panel by panel and the three logits-sized products run on the existing GEMMs; the kernels here are the
// sampler, the sub-catalog gather, the per-row softmax, the target column and the scatter back into the catalog.
//   seqrec_sample_items          ids[i] = draw offset+i of the counter stream (alias table or uniform)
//   seqrec_gather_columns        W_S = W_out[:, ids], bias_S = b_out[ids] - logQ[ids]
//   seqrec_sampled_softmax_rows  per row: loss, Z <- p_j * mask, g_tgt = (p_0 - 1) * mask, deterministic loss sum
//   seqrec_target_columns        dh += g_tgt W_out[:, y], dW_out[:, y] += g_tgt hs, db_out[y] += g_tgt
//   seqrec_scatter_add_columns   dW_out[:, ids] += dW_S, db_out[ids] += db_S
#include "common.cuh"

#define SAMPLE_THREADS 256
#define GATHER_THREADS 256
#define SROWS_THREADS 256
#define SROWS_WARPS (SROWS_THREADS / 32)
#define SROWS_ROWS_PER_WARP 4
#define SROWS_MAX_BLOCKS 1184
#define TCOL_THREADS 256

// ---------------------------------------------------------------------------------------------------------------
// Draw i: r = splitmix64(splitmix64(seed) ^ (offset + i)); column ((r >> 32) * V) >> 32; alias table: keep the column
// if (uint32)r < thr[col], else take alias[col].  state[0] = offset of the next draw, state[1] = block ticket (the
// protocol of seqrec_dropout_mask_dev): a launch captured in a CUDA graph draws fresh ids at every replay.
__global__ void __launch_bounds__(SAMPLE_THREADS)
sample_items_kernel(int32_t* __restrict__ ids, int S, const uint32_t* __restrict__ thr,
                    const int32_t* __restrict__ alias, int V, uint64_t seed, unsigned long long* __restrict__ state) {
  const uint64_t offset = *((volatile unsigned long long*)state);
  const uint64_t key = splitmix64(seed);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S; i += gridDim.x * blockDim.x) {
    const uint64_t r = splitmix64(key ^ (offset + (uint64_t)i));
    const int32_t col = (int32_t)(((r >> 32) * (uint64_t)V) >> 32);
    ids[i] = (thr == nullptr || (uint32_t)r < __ldg(thr + col)) ? col : __ldg(alias + col);
  }
  __syncthreads();                             // every thread of the block has read the offset
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(state + 1, 1ull) == (unsigned long long)gridDim.x - 1) {
      state[0] = offset + (uint64_t)S;
      state[1] = 0ull;
    }
  }
}

extern "C" int seqrec_sample_items(int32_t* ids, int S, const uint32_t* thr, const int32_t* alias, int V, uint64_t seed,
                                   uint64_t* state, void* stream) {
  SEQREC_ARG(ids && state && S >= 1 && V >= 1, 1);
  SEQREC_ARG((thr == nullptr) == (alias == nullptr), 2);
  sample_items_kernel<<<ceil_div(S, SAMPLE_THREADS), SAMPLE_THREADS, 0, as_stream(stream)>>>(
      ids, S, thr, alias, V, seed, reinterpret_cast<unsigned long long*>(state));
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Element (h, j) of W_S reads W_out[h, ids[j]]: consecutive threads write consecutive columns of W_S and read scattered
// columns of W_out, one 32-byte sector per element -- S*H*32 bytes of sectors, small next to the logits panels.
__global__ void __launch_bounds__(GATHER_THREADS)
gather_columns_kernel(const float* __restrict__ W_out, int64_t ldw, const float* __restrict__ b_out,
                      const float* __restrict__ logQ, const int32_t* __restrict__ ids, int S, int H,
                      float* __restrict__ W_S, float* __restrict__ bias_S) {
  const int64_t total = (int64_t)S * H;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t h = i / S;
    const int j = (int)(i - h * S);
    const int32_t c = __ldg(ids + j);
    W_S[i] = __ldg(W_out + h * ldw + c);
    if (h == 0) bias_S[j] = (b_out ? __ldg(b_out + c) : 0.f) - __ldg(logQ + c);
  }
}

extern "C" int seqrec_gather_columns(const float* W_out, int64_t ldw, const float* b_out, const float* logQ,
                                     const int32_t* ids, int S, int H, float* W_S, float* bias_S, void* stream) {
  SEQREC_ARG(W_out && logQ && ids && W_S && bias_S && S >= 1 && H >= 1 && ldw >= 1, 1);
  int64_t blocks = ((int64_t)S * H + GATHER_THREADS - 1) / GATHER_THREADS;
  if (blocks > SEQREC_NUM_SMS * 16) blocks = SEQREC_NUM_SMS * 16;
  gather_columns_kernel<<<(int)blocks, GATHER_THREADS, 0, as_stream(stream)>>>(W_out, ldw, b_out, logQ, ids, S, H, W_S,
                                                                               bias_S);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// One warp per row, the S ids in shared memory (the accidental-hit test of column j is sid[j] == y).  Rows are assigned
// to blocks by n_rows alone and every sum runs in a fixed order, so the loss is bit-reproducible: per-block partials,
// the last block to finish adds them in block order (the scheme of seqrec_ce_finalize).
__device__ double g_srows_partials[SROWS_MAX_BLOCKS];
__device__ unsigned int g_srows_counter = 0;

__global__ void __launch_bounds__(SROWS_THREADS)
sampled_rows_kernel(float* __restrict__ Z, int S, const int32_t* __restrict__ ids, const float* __restrict__ zy,
                    const int32_t* __restrict__ tgt, const float* __restrict__ logQ, const uint8_t* __restrict__ mask,
                    float* __restrict__ ce, float* __restrict__ g_tgt, float* __restrict__ loss_part, int64_t n_rows,
                    int64_t rows_per_block) {
  extern __shared__ int32_t sid[];
  __shared__ double red[SROWS_WARPS];
  __shared__ bool is_last;
  for (int j = threadIdx.x; j < S; j += SROWS_THREADS) sid[j] = ids[j];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r_begin = blockIdx.x * rows_per_block;
  const int64_t r_end = min(n_rows, r_begin + rows_per_block);
  double local = 0.0;
  for (int64_t n = r_begin + warp; n < r_end; n += SROWS_WARPS) {
    float* row = Z + n * S;
    const int32_t y = tgt[n];
    if (y < 0 || mask[n] == 0) {               // pads: no loss, no gradient
      for (int j = lane; j < S; j += 32) row[j] = 0.f;
      if (lane == 0) {
        if (ce) ce[n] = 0.f;
        g_tgt[n] = 0.f;
      }
      continue;
    }
    const float l0 = zy[n] - __ldg(logQ + y);
    float mx = l0;
    for (int j = lane; j < S; j += 32)
      if (sid[j] != y) mx = fmaxf(mx, row[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float s = 0.f;
    for (int j = lane; j < S; j += 32)
      if (sid[j] != y) s += expf(row[j] - mx);
    s = warp_sum(s);
    const float e0 = expf(l0 - mx);
    s += e0;
    const float inv = 1.f / s;
    for (int j = lane; j < S; j += 32) row[j] = sid[j] != y ? expf(row[j] - mx) * inv : 0.f;
    if (lane == 0) {
      const float l = logf(s) - (l0 - mx);
      if (ce) ce[n] = l;
      g_tgt[n] = e0 * inv - 1.f;
      local += (double)l;
    }
  }
  if (lane == 0) red[warp] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int i = 0; i < SROWS_WARPS; ++i) v += red[i];
    g_srows_partials[blockIdx.x] = v;
    __threadfence();
    is_last = atomicAdd(&g_srows_counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    double t = 0.0;
    for (unsigned int i = 0; i < gridDim.x; ++i) t += *((volatile double*)&g_srows_partials[i]);
    loss_part[0] = (float)t;
    g_srows_counter = 0;
  }
}

extern "C" int seqrec_sampled_softmax_rows(float* Z, int S, const int32_t* ids, const float* zy, const int32_t* tgt,
                                           const float* logQ, const uint8_t* mask, float* ce, float* g_tgt,
                                           float* loss_part, int64_t n_rows, void* stream) {
  SEQREC_ARG(Z && ids && zy && tgt && logQ && mask && g_tgt && loss_part && n_rows > 0, 1);
  // the ids live in shared memory for the accidental-hit test: that is what bounds S
  SEQREC_ARG(S >= 1 && S <= SEQREC_MAX_SAMPLED, 2);
  const int64_t per_block_min = (int64_t)SROWS_WARPS * SROWS_ROWS_PER_WARP;
  int64_t blocks = (n_rows + per_block_min - 1) / per_block_min;
  if (blocks > SROWS_MAX_BLOCKS) blocks = SROWS_MAX_BLOCKS;
  const int64_t rows_per_block = (n_rows + blocks - 1) / blocks;
  blocks = (n_rows + rows_per_block - 1) / rows_per_block;
  const size_t smem = sizeof(int32_t) * (size_t)S;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(sampled_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return -(int)e;
  }
  sampled_rows_kernel<<<(unsigned)blocks, SROWS_THREADS, smem, as_stream(stream)>>>(Z, S, ids, zy, tgt, logQ, mask, ce,
                                                                                   g_tgt, loss_part, n_rows,
                                                                                   rows_per_block);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// One warp per token: the target column's terms, which the (N, S) panels do not hold.
__global__ void __launch_bounds__(TCOL_THREADS)
target_columns_kernel(const float* __restrict__ hout, const float* __restrict__ hscale,
                      const float* __restrict__ W_out, int64_t ldw, const int32_t* __restrict__ tgt,
                      const float* __restrict__ g_tgt, float* __restrict__ dh, float* __restrict__ dW_out,
                      float* __restrict__ db_out, int64_t n_tokens, int H) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (n >= n_tokens) return;
  const int32_t y = tgt[n];
  const float g = g_tgt[n];
  if (y < 0 || g == 0.f) return;               // pads carry g = 0
  for (int h = lane; h < H; h += 32) {
    if (dh) dh[n * H + h] += g * __ldg(W_out + (int64_t)h * ldw + y);
    if (dW_out) {
      float x = hout[n * H + h];
      if (hscale) x *= hscale[n * H + h];
      atomicAdd(dW_out + (int64_t)h * ldw + y, g * x);
    }
  }
  if (db_out && lane == 0) atomicAdd(db_out + y, g);
}

extern "C" int seqrec_target_columns(const float* hout, const float* hscale, const float* W_out, int64_t ldw,
                                     const int32_t* tgt, const float* g_tgt, float* dh, float* dW_out, float* db_out,
                                     int64_t n_tokens, int H, void* stream) {
  SEQREC_ARG(hout && W_out && tgt && g_tgt && n_tokens > 0 && H >= 1 && ldw >= 1, 1);
  target_columns_kernel<<<ceil_div(n_tokens * 32, TCOL_THREADS), TCOL_THREADS, 0, as_stream(stream)>>>(
      hout, hscale, W_out, ldw, tgt, g_tgt, dh, dW_out, db_out, n_tokens, H);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// dW_out[h, ids[j]] += dW_S[h, j]; a duplicate id receives one atomic addend per occurrence.
__global__ void __launch_bounds__(GATHER_THREADS)
scatter_add_columns_kernel(const float* __restrict__ dW_S, const float* __restrict__ db_S,
                           const int32_t* __restrict__ ids, int S, int H, float* __restrict__ dW_out, int64_t ldw,
                           float* __restrict__ db_out) {
  const int64_t total = (int64_t)S * H;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t h = i / S;
    const int j = (int)(i - h * S);
    const int32_t c = __ldg(ids + j);
    if (dW_out) atomicAdd(dW_out + h * ldw + c, dW_S[i]);
    if (h == 0 && db_out) atomicAdd(db_out + c, db_S[j]);
  }
}

extern "C" int seqrec_scatter_add_columns(const float* dW_S, const float* db_S, const int32_t* ids, int S, int H,
                                          float* dW_out, int64_t ldw, float* db_out, void* stream) {
  SEQREC_ARG(ids && S >= 1 && H >= 1 && ldw >= 1, 1);
  SEQREC_ARG((dW_out == nullptr || dW_S) && (db_out == nullptr || db_S), 2);
  int64_t blocks = ((int64_t)S * H + GATHER_THREADS - 1) / GATHER_THREADS;
  if (blocks > SEQREC_NUM_SMS * 16) blocks = SEQREC_NUM_SMS * 16;
  scatter_add_columns_kernel<<<(int)blocks, GATHER_THREADS, 0, as_stream(stream)>>>(dW_S, db_S, ids, S, H, dW_out, ldw,
                                                                                    db_out);
  SEQREC_CHECK_LAUNCH();
  return 0;
}
