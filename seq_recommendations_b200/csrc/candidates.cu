// Candidate scoring: logits of a given list of items per row, their order and the target's rank among them.
//
// A serving or evaluation call often asks how the model orders C given items (a retrieval stage's output, the items in
// stock, a category page) rather than the whole catalog.  Scoring the list costs C*H per row instead of a logits pass
// over V items.  The logits read the item-major copy Wt (V_local, H) of W_out, so each candidate is one coalesced row.
//
// The logit of candidate c uses the arithmetic of seqrec_target_logit (ce_tc.cu, target_logit_kernel): lane l of a warp
// accumulates h = l, l+32, ... with fmaf in ascending order, the lanes are summed with warp_sum, the bias is added last.
// So the candidate logit of y equals seqrec_target_logit's zy for target y bit for bit.
#include "common.cuh"

#define CAND_THREADS 256
#define CAND_UNROLL 4                    // candidates in flight per warp (independent accumulators, same order each)
#define ORDER_THREADS 256

// One CTA per row: the row's hidden vector in shared memory, the warps take CAND_UNROLL candidates at a time.
__global__ void __launch_bounds__(CAND_THREADS)
candidate_logits_kernel(const float* __restrict__ hout, const float* __restrict__ Wt, const float* __restrict__ b_out,
                        const int32_t* __restrict__ cand, int64_t cand_ld, float* __restrict__ z, int C, int H,
                        int id_offset, int v_local) {
  extern __shared__ float hs[];
  const int64_t n = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int h = threadIdx.x; h < H; h += CAND_THREADS) hs[h] = hout[n * H + h];
  __syncthreads();
  const int32_t* row = cand + n * cand_ld;
  for (int j0 = warp * CAND_UNROLL; j0 < C; j0 += (CAND_THREADS / 32) * CAND_UNROLL) {
    const float* w[CAND_UNROLL];
    int64_t loc[CAND_UNROLL];
    bool ok[CAND_UNROLL];
    float acc[CAND_UNROLL];
#pragma unroll
    for (int q = 0; q < CAND_UNROLL; ++q) {
      const int32_t c = (j0 + q < C) ? row[j0 + q] : -1;
      loc[q] = (int64_t)c - id_offset;
      // pads and ids of other vocabulary shards never index Wt / b_out
      ok[q] = c >= 0 && loc[q] >= 0 && loc[q] < v_local;
      w[q] = Wt + (ok[q] ? loc[q] : 0) * (int64_t)H;
      acc[q] = 0.f;
    }
    for (int h = lane; h < H; h += 32) {
      const float x = hs[h];
#pragma unroll
      for (int q = 0; q < CAND_UNROLL; ++q)
        if (ok[q]) acc[q] = fmaf(x, __ldg(w[q] + h), acc[q]);
    }
#pragma unroll
    for (int q = 0; q < CAND_UNROLL; ++q) {
      acc[q] = warp_sum(acc[q]);
      if (lane == 0 && j0 + q < C) z[n * C + j0 + q] = ok[q] ? acc[q] + (b_out ? b_out[loc[q]] : 0.f) : 0.f;
    }
  }
}

// entry j precedes entry i: valid before pad; score descending, then lower id, then lower list position
__device__ __forceinline__ bool cand_before(float zj, int32_t cj, int j, float zi, int32_t ci, int i) {
  const bool vj = cj >= 0, vi = ci >= 0;
  if (vj != vi) return vj;
  if (!vj) return j < i;
  return zj > zi || (zj == zi && (cj < ci || (cj == ci && j < i)));
}

// One CTA per row: each entry's output position is the number of entries that precede it (O(C^2) compares).
__global__ void __launch_bounds__(ORDER_THREADS)
candidate_order_kernel(const float* __restrict__ z, const int32_t* __restrict__ cand, int C,
                       const float* __restrict__ m, const float* __restrict__ s, int k, int32_t* __restrict__ out_ids,
                       float* __restrict__ out_scores, const float* __restrict__ zy, const int32_t* __restrict__ tgt,
                       int32_t* __restrict__ rank) {
  extern __shared__ float zs[];
  int32_t* cs = reinterpret_cast<int32_t*>(zs + C);
  __shared__ int count;
  const int64_t n = blockIdx.x;
  for (int j = threadIdx.x; j < C; j += ORDER_THREADS) {
    zs[j] = z[n * C + j];
    cs[j] = cand[n * C + j];
  }
  if (threadIdx.x == 0) count = 0;
  __syncthreads();
  if (out_ids) {
    const float mn = m ? m[n] : 0.f, sn = s ? s[n] : 1.f;
    for (int i = threadIdx.x; i < C; i += ORDER_THREADS) {
      const float zi = zs[i];
      const int32_t ci = cs[i];
      int pos = 0;
      for (int j = 0; j < C; ++j) pos += cand_before(zs[j], cs[j], j, zi, ci, i) ? 1 : 0;
      if (pos < k) {
        out_ids[n * k + pos] = ci >= 0 ? ci : -1;
        out_scores[n * k + pos] = ci < 0 ? 0.f : (m && s) ? expf(zi - mn) / sn : zi;
      }
    }
  }
  if (tgt && rank) {
    const int32_t y = tgt[n];
    if (y < 0) {
      if (threadIdx.x == 0) rank[n] = 0;
      return;
    }
    const float zt = zy[n];
    int part = 0;
    for (int j = threadIdx.x; j < C; j += ORDER_THREADS) {
      const int32_t c = cs[j];
      const float zj = zs[j];
      part += (c >= 0 && c != y && (zj > zt || (zj == zt && c < y))) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&count, part);
    __syncthreads();
    if (threadIdx.x == 0) rank[n] = 1 + count;
  }
}

extern "C" int seqrec_candidate_logits(const float* hout, const float* Wt, const float* b_out, const int32_t* cand,
                                       int64_t cand_ld, float* z, int64_t n_rows, int C, int H, int id_offset,
                                       int v_local, void* stream) {
  SEQREC_ARG(hout && Wt && cand && z && n_rows > 0 && H > 0 && v_local > 0, 1);
  // (no bound on C: the engine scores a target as one extra column, [y | candidates])
  SEQREC_ARG(C >= 1 && cand_ld >= C && n_rows < (1LL << 31), 2);
  const size_t smem = sizeof(float) * (size_t)H;
  if (smem > 227 * 1024) return -1010;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(candidate_logits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return -(int)e;
  }
  candidate_logits_kernel<<<(unsigned)n_rows, CAND_THREADS, smem, as_stream(stream)>>>(hout, Wt, b_out, cand, cand_ld, z,
                                                                                        C, H, id_offset, v_local);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_candidate_order(const float* z, const int32_t* cand, int C, int64_t n_rows, const float* m,
                                      const float* s, int k, int32_t* out_ids, float* out_scores, const float* zy,
                                      const int32_t* tgt, int32_t* rank, void* stream) {
  SEQREC_ARG(z && cand && n_rows > 0 && n_rows < (1LL << 31), 1);
  SEQREC_ARG(C >= 1 && C <= SEQREC_MAX_CANDIDATES, 2);
  SEQREC_ARG(!out_ids || (out_scores && k >= 1 && k <= C), 3);
  SEQREC_ARG((m == nullptr) == (s == nullptr), 4);
  SEQREC_ARG(!tgt || (zy && rank), 5);
  const size_t smem = (sizeof(float) + sizeof(int32_t)) * (size_t)C;
  candidate_order_kernel<<<(unsigned)n_rows, ORDER_THREADS, smem, as_stream(stream)>>>(z, cand, C, m, s, k, out_ids,
                                                                                       out_scores, zy, tgt, rank);
  SEQREC_CHECK_LAUNCH();
  return 0;
}
