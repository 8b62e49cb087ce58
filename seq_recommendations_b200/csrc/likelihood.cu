// Scoring metrics of the reference on the device: per-sequence mean negative log-likelihood of p(true next item), plain
// (utils.py:166-178 compute_likelihood) and with the within-sequence 70/30 cut (utils.py:145-163 compute_likelihood_cut,
// consumed by ValLossHistoryCut, model.py:106-112).  Input is the (n, T) matrix of per-step probabilities the scoring
// kernels produce (right-aligned: a sequence of L steps fills the LAST L columns, like the left-padded batches); one
// warp reduces one sequence, logs and sums in double.
// Also the ranking metrics of next-item evaluation (Recall@k, MRR@k, NDCG@k) from the per-token rank of the target.
#include "common.cuh"

// window of row i: the last L columns (lengths given; L <= 0 or L > T means the whole row, like numpy's pred[-0:]),
// minus the first element when skip_first
__device__ __forceinline__ void row_window(const int32_t* lengths, int64_t i, int T, int skip_first, int& start, int& L) {
  L = T;
  if (lengths) {
    const int l = lengths[i];
    if (l > 0 && l < T) L = l;
  }
  start = T - L;
  if (skip_first && L > 0) { ++start; --L; }
}

__device__ __forceinline__ double neg_log_sum(const float* row, int a, int b, int lane, bool clip) {
  double acc = 0.0;
  for (int j = a + lane; j < b; j += 32) {
    double p = (double)row[j];
    if (clip) p = fmin(fmax(p, 1e-07), 1.0 - 1e-07);
    acc -= log(p);
  }
  return warp_sum_d(acc);
}

// out[0] += sum of per-sequence mean NLL, out[1] += sequences counted
__global__ void __launch_bounds__(256)
likelihood_kernel(const float* __restrict__ P, const int32_t* __restrict__ lengths, int64_t n, int T, int skip_first,
                  double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  int start, L;
  row_window(lengths, i, T, skip_first, start, L);
  if (L <= 0) return;
  const double s = neg_log_sum(P + i * T, start, start + L, lane, true);
  if (lane == 0) { atomicAdd(out, s / L); atomicAdd(out + 1, 1.0); }
}

// out[0], out[1]: sum / count of the "train" parts (first ceil(tp*L) steps); out[2], out[3]: of the "val" parts (last
// floor((1-tp)*L) steps)
__global__ void __launch_bounds__(256)
likelihood_cut_kernel(const float* __restrict__ P, const int32_t* __restrict__ lengths, int64_t n, int T,
                      int skip_first, double train_percent, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  int start, L;
  row_window(lengths, i, T, skip_first, start, L);
  const int te = (int)ceil(train_percent * (double)L);
  const int ve = (int)floor((1.0 - train_percent) * (double)L);
  const float* row = P + i * T;
  if (te > 0) {
    const double s = neg_log_sum(row, start, start + te, lane, false);
    if (lane == 0) { atomicAdd(out, s / te); atomicAdd(out + 1, 1.0); }
  }
  if (ve > 0) {
    const double s = neg_log_sum(row, start + L - ve, start + L, lane, false);
    if (lane == 0) { atomicAdd(out + 2, s / ve); atomicAdd(out + 3, 1.0); }
  }
}

extern "C" int seqrec_likelihood(const float* P, const int32_t* lengths, int64_t n_seqs, int T, int skip_first,
                                 double* out2, void* stream) {
  SEQREC_ARG(P && out2 && n_seqs > 0 && T > 0, 1);
  likelihood_kernel<<<ceil_div(n_seqs * 32, 256), 256, 0, as_stream(stream)>>>(P, lengths, n_seqs, T, skip_first, out2);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_likelihood_cut(const float* P, const int32_t* lengths, int64_t n_seqs, int T, int skip_first,
                                     double train_percent, double* out4, void* stream) {
  SEQREC_ARG(P && out4 && n_seqs > 0 && T > 0 && train_percent <= 1.0 && train_percent >= 0.0, 1);
  likelihood_cut_kernel<<<ceil_div(n_seqs * 32, 256), 256, 0, as_stream(stream)>>>(P, lengths, n_seqs, T, skip_first,
                                                                                   train_percent, out4);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ranking metrics: for q < n_ks and k = ks[q], out[3q..3q+2] += {#(rank <= k), sum 1/rank, sum 1/log2(rank + 1)} over
// the tokens with 0 < rank <= k; out[3 n_ks..3 n_ks+2] += the same sums without a cutoff (the first one is the number of
// scored tokens).  rank 0 (pad) never counts.  Doubles throughout; one warp reduction and three atomics per warp and q.
__global__ void __launch_bounds__(256)
rank_metrics_kernel(const int32_t* __restrict__ rank, int64_t n, const int32_t* __restrict__ ks, int n_ks,
                    double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int q = 0; q <= n_ks; ++q) {
    const int k = q < n_ks ? ks[q] : 0x7fffffff;
    double hits = 0.0, rr = 0.0, dg = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
      const int r = rank[i];
      if (r > 0 && r <= k) {
        hits += 1.0;
        rr += 1.0 / (double)r;
        dg += 1.0 / log2((double)r + 1.0);
      }
    }
    hits = warp_sum_d(hits);
    rr = warp_sum_d(rr);
    dg = warp_sum_d(dg);
    if (lane == 0 && hits > 0.0) {
      atomicAdd(out + 3 * q, hits);
      atomicAdd(out + 3 * q + 1, rr);
      atomicAdd(out + 3 * q + 2, dg);
    }
  }
}

extern "C" int seqrec_rank_metrics(const int32_t* rank, int64_t n, const int32_t* ks, int n_ks, double* out,
                                   void* stream) {
  SEQREC_ARG(rank && ks && out && n > 0 && n_ks >= 1, 1);
  int64_t blocks = (n + 255) / 256;
  if (blocks > SEQREC_NUM_SMS * 4) blocks = SEQREC_NUM_SMS * 4;
  rank_metrics_kernel<<<(int)blocks, 256, 0, as_stream(stream)>>>(rank, n, ks, n_ks, out);
  SEQREC_CHECK_LAUNCH();
  return 0;
}
