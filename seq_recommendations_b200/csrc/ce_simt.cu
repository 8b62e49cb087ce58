// K5 / K6 / K9, fp32 SIMT flavour: TimeDistributed(Dense) + softmax + categorical_crossentropy and its backward
// without ever materialising the (N,V) logits (model.py:382-384, :397; experiments_methods.py:42).
//
// This is the exact-fp32 path used for small or oddly shaped problems (cfg1: V=17, H=100) and as the in-library
// cross-check of the tcgen05 path (ce_tc.cu), which takes over when H and V are tensor-core sized.
//
// Tiling: 64 tokens x 64 items per step, 256 threads, 4x4 register micro-tiles.  The token tile (hout, optionally
// times the z->y dropout factors) sits transposed in shared memory as A_s[h][token]; the W_out tile as W_s[h][item].
#include "common.cuh"

#define CT 64    // tile edge (tokens and items)
#define CP 68    // padded smem row
#define CE_THREADS 256

struct CeSmem {
  float* A_s;   // [H][CP]
  float* W_s;   // [H][CP]
  float* D_s;   // [CT][CP]  (backward only)
};

__device__ __forceinline__ CeSmem carve(float* base, int H) {
  CeSmem s;
  s.A_s = base;
  s.W_s = s.A_s + (size_t)H * CP;
  s.D_s = s.W_s + (size_t)H * CP;
  return s;
}

// A_s[h][r] = hout[n0+r][h] * hscale[n0+r][h]
__device__ __forceinline__ void load_token_tile(float* A_s, const float* __restrict__ hout,
                                                const float* __restrict__ hscale, int64_t n0, int64_t n_tokens,
                                                int H) {
  for (int i = threadIdx.x; i < CT * H; i += CE_THREADS) {
    const int r = i / H, h = i - r * H;
    const int64_t n = n0 + r;
    float v = 0.f;
    if (n < n_tokens) {
      v = hout[n * H + h];
      if (hscale) v *= hscale[n * H + h];
    }
    A_s[h * CP + r] = v;
  }
}

// W_s[h][c] = W_out[h][v0+c]
__device__ __forceinline__ void load_item_tile(float* W_s, const float* __restrict__ W_out, int ldw, int v0, int v_end,
                                               int H) {
  for (int i = threadIdx.x; i < CT * H; i += CE_THREADS) {
    const int h = i / CT, c = i - h * CT;
    const int v = v0 + c;
    W_s[h * CP + c] = (v < v_end) ? W_out[(size_t)h * ldw + v] : 0.f;
  }
}

// acc[i][j] = sum_h A_s[h][ty*4+i] * W_s[h][tx*4+j]
__device__ __forceinline__ void logits_tile(float (&acc)[4][4], const float* A_s, const float* W_s, int H, int tx,
                                            int ty) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 4
  for (int h = 0; h < H; ++h) {
    const float4 a = *reinterpret_cast<const float4*>(A_s + h * CP + ty * 4);
    const float4 b = *reinterpret_cast<const float4*>(W_s + h * CP + tx * 4);
    const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }
}

__device__ __forceinline__ void merge_ms(float& m, float& s, float m2, float s2) {
  const float mn = fmaxf(m, m2);
  if (mn == -INFINITY) { m = mn; s = 0.f; return; }
  s = s * expf(m - mn) + s2 * expf(m2 - mn);
  m = mn;
}

static size_t ce_smem_bytes(int H, bool with_d) { return sizeof(float) * ((size_t)2 * H * CP + (with_d ? CT * CP : 0)); }
static size_t ce_smem_bytes_rank(int H) { return sizeof(float) * ((size_t)2 * H * CP + CT); }

// ---------------------------------------------------------------------------------------------------------------
// forward: per-token running (max, sum-exp) over this CTA's item range, and the target logit
__global__ void __launch_bounds__(CE_THREADS)
ce_forward_simt_kernel(const float* __restrict__ hout, const float* __restrict__ hscale,
                       const float* __restrict__ W_out, const float* __restrict__ b_out,
                       const int32_t* __restrict__ tgt, float* __restrict__ ws_m, float* __restrict__ ws_s,
                       float* __restrict__ zy, int64_t n_tokens, int H, int v_begin, int v_end, int ldw,
                       int items_per_split) {
  extern __shared__ __align__(16) float smem[];
  CeSmem sm = carve(smem, H);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t n0 = (int64_t)blockIdx.x * CT;
  const int vb = v_begin + blockIdx.y * items_per_split;
  const int ve = min(v_end, vb + items_per_split);
  load_token_tile(sm.A_s, hout, hscale, n0, n_tokens, H);
  float m[4], s[4];
  int32_t tg[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = -INFINITY; s[i] = 0.f;
    const int64_t n = n0 + ty * 4 + i;
    tg[i] = (tgt && n < n_tokens) ? tgt[n] : -1;
  }
  for (int v0 = vb; v0 < ve; v0 += CT) {
    __syncthreads();
    load_item_tile(sm.W_s, W_out, ldw, v0, ve, H);
    __syncthreads();
    float acc[4][4];
    logits_tile(acc, sm.A_s, sm.W_s, H, tx, ty);
    float bv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = v0 + tx * 4 + j;
      bv[j] = (b_out && v < ve) ? b_out[v] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int v = v0 + tx * 4 + j;
        const float z = acc[i][j] + bv[j];
        acc[i][j] = z;
        if (v < ve) {
          mx = fmaxf(mx, z);
          if (v == tg[i]) zy[n0 + ty * 4 + i] = z;
        }
      }
      if (mx > -INFINITY) {
        const float mn = fmaxf(m[i], mx);
        float add = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (v0 + tx * 4 + j < ve) add += expf(acc[i][j] - mn);
        s[i] = s[i] * expf(m[i] - mn) + add;
        m[i] = mn;
      }
    }
  }
  // merge the 16 column-threads of each row (lanes differ in bits 0..3)
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m[i], o);
      const float s2 = __shfl_xor_sync(0xffffffffu, s[i], o);
      merge_ms(m[i], s[i], m2, s2);
    }
    const int64_t n = n0 + ty * 4 + i;
    if (tx == 0 && n < n_tokens) {
      ws_m[(int64_t)blockIdx.y * n_tokens + n] = m[i];
      ws_s[(int64_t)blockIdx.y * n_tokens + n] = s[i];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// rank of the target: adds #{v in this CTA's item range, id != y : z_v > z_y  or  (z_v == z_y and id < y)} to rank[n]
// (id = id_offset + v, y = tgt[n] a global id; pads, y < 0, add nothing).  The logits are the 4x4 micro-tiles of the
// forward kernel above; without `ref` the reference z_y is the same fmaf chain over h plus the bias, so an item whose
// W_out column equals the target's ties with it EXACTLY and the tie rule (lower id first) decides.
__global__ void __launch_bounds__(CE_THREADS)
target_rank_simt_kernel(const float* __restrict__ hout, const float* __restrict__ W_out,
                        const float* __restrict__ b_out, const float* __restrict__ ref,
                        const int32_t* __restrict__ tgt, int id_offset, int32_t* __restrict__ rank, int64_t n_tokens,
                        int H, int v_begin, int v_end, int ldw, int items_per_split) {
  extern __shared__ __align__(16) float smem[];
  CeSmem sm = carve(smem, H);
  float* zy_s = sm.W_s + (size_t)H * CP;                     // [CT] reference logits of the tile's tokens
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t n0 = (int64_t)blockIdx.x * CT;
  const int vb = v_begin + blockIdx.y * items_per_split;
  const int ve = min(v_end, vb + items_per_split);
  load_token_tile(sm.A_s, hout, nullptr, n0, n_tokens, H);
  __syncthreads();
  if (tid < CT) {
    const int64_t n = n0 + tid;
    const int32_t y = n < n_tokens ? tgt[n] : -1;
    float z = 0.f;
    const int yl = y - id_offset;                          // column of W_out (ref == NULL: the target is local)
    if (ref && y >= 0) {
      z = ref[n];
    } else if (y >= 0 && yl < ldw) {
      for (int h = 0; h < H; ++h) z = fmaf(sm.A_s[h * CP + tid], W_out[(size_t)h * ldw + yl], z);
      z = z + (b_out ? b_out[yl] : 0.f);
    }
    zy_s[tid] = z;
  }
  __syncthreads();
  float rz[4];
  int32_t tg[4], cnt[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t n = n0 + ty * 4 + i;
    tg[i] = n < n_tokens ? tgt[n] : -1;
    rz[i] = zy_s[ty * 4 + i];
    cnt[i] = 0;
  }
  for (int v0 = vb; v0 < ve; v0 += CT) {
    __syncthreads();
    load_item_tile(sm.W_s, W_out, ldw, v0, ve, H);
    __syncthreads();
    float acc[4][4];
    logits_tile(acc, sm.A_s, sm.W_s, H, tx, ty);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = v0 + tx * 4 + j;
      if (v >= ve) continue;
      const float b = b_out ? b_out[v] : 0.f;
      const int id = id_offset + v;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float z = acc[i][j] + b;
        cnt[i] += tg[i] >= 0 && id != tg[i] && (z > rz[i] || (z == rz[i] && id < tg[i]));
      }
    }
  }
  // the 16 column-threads of a row are lanes differing in bits 0..3
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int c = cnt[i];
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (tx == 0 && c > 0) atomicAdd(rank + n0 + ty * 4 + i, c);
  }
}

extern "C" int seqrec_target_rank(const float* hout, const float* W_out, const float* b_out, const float* ref,
                                  const int32_t* tgt, int id_offset, int32_t* rank, int64_t n_tokens, int H, int V,
                                  int v_begin, int v_end, int ldw, void* stream) {
  SEQREC_ARG(hout && W_out && tgt && rank && n_tokens > 0 && H > 0 && V > 0, 1);
  SEQREC_ARG(v_begin >= 0 && v_end <= V && v_begin < v_end && ldw >= v_end && id_offset >= 0, 2);
  const size_t smem = ce_smem_bytes_rank(H);
  if (smem > 227 * 1024) return -1010;
  cudaError_t e = cudaFuncSetAttribute(target_rank_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return -(int)e;
  // enough CTAs to fill the SMs: the item range is split over blockIdx.y (each split adds its own count)
  const int64_t n_tiles = (n_tokens + CT - 1) / CT;
  const int v_tiles = ceil_div(v_end - v_begin, CT);
  int splits = (int)((2 * SEQREC_NUM_SMS + n_tiles - 1) / n_tiles);
  if (splits > v_tiles) splits = v_tiles;
  if (splits < 1) splits = 1;
  const int ips = ceil_div(v_tiles, splits) * CT;
  splits = ceil_div(v_end - v_begin, ips);
  dim3 grid((unsigned)n_tiles, splits);
  target_rank_simt_kernel<<<grid, CE_THREADS, smem, as_stream(stream)>>>(hout, W_out, b_out, ref, tgt, id_offset, rank,
                                                                         n_tokens, H, v_begin, v_end, ldw, ips);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// finalize: merge the per-split stats, CE with Keras' clip, per-token backward coefficient, deterministic loss sum
// (per-block partials in a fixed order; the last block to finish adds them up in block order)
#define FIN_THREADS 256
#define FIN_MAX_BLOCKS 1184
__device__ double g_fin_partials[FIN_MAX_BLOCKS];
__device__ unsigned int g_fin_counter = 0;

__global__ void __launch_bounds__(FIN_THREADS)
ce_finalize_kernel(const float* __restrict__ ws_m, const float* __restrict__ ws_s, const float* __restrict__ zy,
                   const uint8_t* __restrict__ mask, float* __restrict__ m_out, float* __restrict__ s_out,
                   float* __restrict__ ce, float* __restrict__ py, float* __restrict__ coef,
                   float* __restrict__ loss_sum, const int32_t* __restrict__ n_valid, float* __restrict__ n_valid_f,
                   float* __restrict__ loss_mean, int64_t n_tokens, int splits,
                   const int32_t* __restrict__ n_tokens_dev) {
  // compacted token axis (splits == 1 there): the number of tokens is read on the device
  if (n_tokens_dev) n_tokens = min(n_tokens, (int64_t)n_tokens_dev[0]);
  __shared__ double red[FIN_THREADS / 32];
  __shared__ bool is_last;
  double local = 0.0;
  // fixed token -> (block, thread) assignment, so every partial is reproducible
  const int64_t per_block = (n_tokens + gridDim.x - 1) / gridDim.x;
  const int64_t n_begin = blockIdx.x * per_block;
  const int64_t n_end = min(n_tokens, n_begin + per_block);
  for (int64_t n = n_begin + threadIdx.x; n < n_end; n += FIN_THREADS) {
    float m = ws_m[n], s = ws_s[n];
    for (int k = 1; k < splits; ++k) merge_ms(m, s, ws_m[(int64_t)k * n_tokens + n], ws_s[(int64_t)k * n_tokens + n]);
    m_out[n] = m;
    s_out[n] = s;
    const bool on = mask ? (mask[n] != 0) : true;
    float p = 0.f, c = 0.f, l = 0.f;
    if (on && zy) {
      const float praw = expf(zy[n] - m) / s;
      c = (praw >= SEQREC_P_EPS && praw <= SEQREC_P_ONE_MINUS_EPS) ? 1.f : 0.f;  // Theano clip gradient
      p = fminf(fmaxf(praw, SEQREC_P_EPS), SEQREC_P_ONE_MINUS_EPS);
      l = -logf(p);
    } else {
      p = SEQREC_P_EPS;  // model.py:108-110: pad rows are 0 before the clip
    }
    if (ce) ce[n] = l;
    if (py) py[n] = p;
    if (coef) coef[n] = c;
    local += (double)l;
  }
  local = warp_sum_d(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int i = 0; i < FIN_THREADS / 32; ++i) v += red[i];
    g_fin_partials[blockIdx.x] = v;
    __threadfence();
    const unsigned int done = atomicAdd(&g_fin_counter, 1u);
    is_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    // the last block sums the per-block partials: a fixed thread <- partial assignment and a fixed reduction tree, so
    // the loss is bit-reproducible; all threads take part (a serial loop of dependent L2 loads cost ~15 us at cfg2)
    __threadfence();
    double v = 0.0;
    for (unsigned int i = threadIdx.x; i < gridDim.x; i += FIN_THREADS) v += *((volatile double*)&g_fin_partials[i]);
    v = warp_sum_d(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < FIN_THREADS / 32; ++i) t += red[i];
      if (loss_sum) loss_sum[0] = (float)t;
      if (n_valid) {                          // masked mean, and the count as the float the optimiser divides by
        const float nv = (float)n_valid[0];
        if (n_valid_f) n_valid_f[0] = nv;
        if (loss_mean) loss_mean[0] = (float)t / nv;
      }
      g_fin_counter = 0;  // ready for the next (stream-ordered) launch
    }
  }
}

// dlogit for one element
__device__ __forceinline__ float dlogit_of(float z, float m, float s, float cf, bool is_target) {
  const float p = expf(z - m) / s;
  return (p - (is_target ? 1.f : 0.f)) * cf;
}

// ---------------------------------------------------------------------------------------------------------------
// backward, token-stationary: dh[n,:] = sum_v dlogit[n,v] * W_out[:,v]
template <int HQ>
__global__ void __launch_bounds__(CE_THREADS)
ce_backward_dh_simt_kernel(const float* __restrict__ hout, const float* __restrict__ hscale,
                           const float* __restrict__ W_out, const float* __restrict__ b_out,
                           const int32_t* __restrict__ tgt, const float* __restrict__ mrow,
                           const float* __restrict__ srow, const float* __restrict__ coef,
                           const float* __restrict__ inv_nvalid, float* __restrict__ dh, int64_t n_tokens, int H,
                           int v_begin, int v_end, int ldw, int accumulate) {
  extern __shared__ __align__(16) float smem[];
  CeSmem sm = carve(smem, H);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t n0 = (int64_t)blockIdx.x * CT;
  load_token_tile(sm.A_s, hout, hscale, n0, n_tokens, H);
  const float inv = inv_nvalid ? inv_nvalid[0] : 1.0f;   // NULL: un-normalised gradients (the optimiser divides)
  float m[4], s[4], cf[4];
  int32_t tg[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t n = n0 + ty * 4 + i;
    const bool ok = n < n_tokens;
    m[i] = ok ? mrow[n] : 0.f;
    s[i] = ok ? srow[n] : 1.f;
    cf[i] = ok ? coef[n] * inv : 0.f;
    tg[i] = ok ? tgt[n] : -1;
  }
  float dacc[4][HQ];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int q = 0; q < HQ; ++q) dacc[i][q] = 0.f;

  for (int v0 = v_begin; v0 < v_end; v0 += CT) {
    __syncthreads();
    load_item_tile(sm.W_s, W_out, ldw, v0, v_end, H);
    __syncthreads();
    float acc[4][4];
    logits_tile(acc, sm.A_s, sm.W_s, H, tx, ty);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = v0 + tx * 4 + j;
      const float bj = (b_out && v < v_end) ? b_out[v] : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float d = (v < v_end && cf[i] != 0.f) ? dlogit_of(acc[i][j] + bj, m[i], s[i], cf[i], v == tg[i]) : 0.f;
        sm.D_s[(ty * 4 + i) * CP + tx * 4 + j] = d;
      }
    }
    __syncthreads();
    // dacc[i][q] += sum_c D_s[row_i][c] * W_s[h_q][c],  h_q = tx + 16 q
#pragma unroll 2
    for (int c = 0; c < CT; c += 4) {
      float4 d4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) d4[i] = *reinterpret_cast<const float4*>(sm.D_s + (ty * 4 + i) * CP + c);
#pragma unroll
      for (int q = 0; q < HQ; ++q) {
        const int h = tx + 16 * q;
        if (h < H) {
          const float4 w = *reinterpret_cast<const float4*>(sm.W_s + h * CP + c);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            dacc[i][q] = fmaf(d4[i].x, w.x, dacc[i][q]);
            dacc[i][q] = fmaf(d4[i].y, w.y, dacc[i][q]);
            dacc[i][q] = fmaf(d4[i].z, w.z, dacc[i][q]);
            dacc[i][q] = fmaf(d4[i].w, w.w, dacc[i][q]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t n = n0 + ty * 4 + i;
    if (n >= n_tokens) continue;
#pragma unroll
    for (int q = 0; q < HQ; ++q) {
      const int h = tx + 16 * q;
      if (h >= H) continue;
      float v = dacc[i][q];
      if (hscale) v *= hscale[n * H + h];
      if (accumulate) v += dh[n * H + h];
      dh[n * H + h] = v;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// backward, item-stationary: dW_out[:,v] += sum_n hs[n,:] * dlogit[n,v];  db_out[v] += sum_n dlogit[n,v]
template <int HQ>
__global__ void __launch_bounds__(CE_THREADS)
ce_backward_dw_simt_kernel(const float* __restrict__ hout, const float* __restrict__ hscale,
                           const float* __restrict__ W_out, const float* __restrict__ b_out,
                           const int32_t* __restrict__ tgt, const float* __restrict__ mrow,
                           const float* __restrict__ srow, const float* __restrict__ coef,
                           const float* __restrict__ inv_nvalid, float* __restrict__ dW, float* __restrict__ db,
                           int64_t n_tokens, int H, int v_begin, int v_end, int ldw, int tiles_per_split) {
  extern __shared__ __align__(16) float smem[];
  CeSmem sm = carve(smem, H);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int v0 = v_begin + blockIdx.x * CT;
  load_item_tile(sm.W_s, W_out, ldw, v0, v_end, H);
  const float inv = inv_nvalid ? inv_nvalid[0] : 1.0f;   // NULL: un-normalised gradients (the optimiser divides)
  float bj[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int v = v0 + tx * 4 + j;
    bj[j] = (b_out && v < v_end) ? b_out[v] : 0.f;
  }
  float wacc[HQ][4];
#pragma unroll
  for (int q = 0; q < HQ; ++q)
#pragma unroll
    for (int j = 0; j < 4; ++j) wacc[q][j] = 0.f;
  float bacc = 0.f;  // threads 0..63 own one item column each for db

  const int64_t n_tiles = (n_tokens + CT - 1) / CT;
  const int64_t t_begin = (int64_t)blockIdx.y * tiles_per_split;
  const int64_t t_end = min(n_tiles, t_begin + tiles_per_split);
  for (int64_t tt = t_begin; tt < t_end; ++tt) {
    const int64_t n0 = tt * CT;
    __syncthreads();
    load_token_tile(sm.A_s, hout, hscale, n0, n_tokens, H);
    __syncthreads();
    float acc[4][4];
    logits_tile(acc, sm.A_s, sm.W_s, H, tx, ty);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t n = n0 + ty * 4 + i;
      const bool ok = n < n_tokens;
      const float cf = ok ? coef[n] * inv : 0.f;
      const float m = ok ? mrow[n] : 0.f, s = ok ? srow[n] : 1.f;
      const int32_t tg = ok ? tgt[n] : -1;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int v = v0 + tx * 4 + j;
        const float d = (v < v_end && cf != 0.f) ? dlogit_of(acc[i][j] + bj[j], m, s, cf, v == tg) : 0.f;
        sm.D_s[(ty * 4 + i) * CP + tx * 4 + j] = d;
      }
    }
    __syncthreads();
    // wacc[q][j] += sum_r A_s[h_q][r] * D_s[r][tx*4+j],  h_q = ty + 16 q
#pragma unroll 2
    for (int r = 0; r < CT; r += 4) {
      float4 d4[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) d4[rr] = *reinterpret_cast<const float4*>(sm.D_s + (r + rr) * CP + tx * 4);
#pragma unroll
      for (int q = 0; q < HQ; ++q) {
        const int h = ty + 16 * q;
        if (h < H) {
          const float4 a = *reinterpret_cast<const float4*>(sm.A_s + h * CP + r);
          const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
          for (int rr = 0; rr < 4; ++rr) {
            wacc[q][0] = fmaf(av[rr], d4[rr].x, wacc[q][0]);
            wacc[q][1] = fmaf(av[rr], d4[rr].y, wacc[q][1]);
            wacc[q][2] = fmaf(av[rr], d4[rr].z, wacc[q][2]);
            wacc[q][3] = fmaf(av[rr], d4[rr].w, wacc[q][3]);
          }
        }
      }
    }
    if (db && tid < CT) {
      float t = 0.f;
      for (int r = 0; r < CT; ++r) t += sm.D_s[r * CP + tid];
      bacc += t;
    }
  }
#pragma unroll
  for (int q = 0; q < HQ; ++q) {
    const int h = ty + 16 * q;
    if (h >= H) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = v0 + tx * 4 + j;
      if (v < v_end) atomicAdd(dW + (size_t)h * ldw + v, wacc[q][j]);
    }
  }
  if (db && tid < CT && v0 + tid < v_end) atomicAdd(db + v0 + tid, bacc);
}

// ---------------------------------------------------------------------------------------------------------------
// predict: full softmax probabilities, batch-major (B,T,V) like Keras' model.predict
__global__ void __launch_bounds__(CE_THREADS)
predict_probs_simt_kernel(const float* __restrict__ hout, const float* __restrict__ W_out,
                          const float* __restrict__ b_out, const float* __restrict__ mrow,
                          const float* __restrict__ srow, float* __restrict__ probs, int T, int B, int H, int V) {
  extern __shared__ __align__(16) float smem[];
  CeSmem sm = carve(smem, H);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t n_tokens = (int64_t)T * B;
  const int64_t n0 = (int64_t)blockIdx.x * CT;
  const int v0 = blockIdx.y * CT;
  load_token_tile(sm.A_s, hout, nullptr, n0, n_tokens, H);
  load_item_tile(sm.W_s, W_out, V, v0, V, H);
  __syncthreads();
  float acc[4][4];
  logits_tile(acc, sm.A_s, sm.W_s, H, tx, ty);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t n = n0 + ty * 4 + i;
    if (n >= n_tokens) continue;
    const int64_t t = n / B, b = n - t * B;
    const float m = mrow[n], s = srow[n];
    float* dst = probs + (b * T + t) * (int64_t)V;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = v0 + tx * 4 + j;
      if (v < V) dst[v] = expf(acc[i][j] + (b_out ? b_out[v] : 0.f) - m) / s;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side

int ce_forward_simt(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                    const int32_t* tgt, float* ws_m, float* ws_s, float* zy, int64_t n_tokens, int H, int V,
                    int v_begin, int v_end, int ldw, int splits, cudaStream_t st) {
  const size_t smem = ce_smem_bytes(H, false);
  if (smem > 227 * 1024) return -1010;
  cudaError_t e = cudaFuncSetAttribute(ce_forward_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return -(int)e;
  int ips = ceil_div(v_end - v_begin, splits);
  ips = ceil_div(ips, CT) * CT;
  dim3 grid(ceil_div(n_tokens, CT), splits);
  ce_forward_simt_kernel<<<grid, CE_THREADS, smem, st>>>(hout, hscale, W_out, b_out, tgt, ws_m, ws_s, zy, n_tokens, H,
                                                         v_begin, v_end, ldw, ips);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

template <int HQ>
static int ce_backward_simt_t(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                              const int32_t* tgt, const float* m, const float* s, const float* coef,
                              const float* inv_nvalid, float* dh, float* dW_out, float* db_out, int64_t n_tokens,
                              int H, int v_begin, int v_end, int ldw, int accumulate_dh, cudaStream_t st) {
  const size_t smem = ce_smem_bytes(H, true);
  if (smem > 227 * 1024) return -1010;
  cudaError_t e;
  if (dh) {
    auto k = ce_backward_dh_simt_kernel<HQ>;
    e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return -(int)e;
    k<<<ceil_div(n_tokens, CT), CE_THREADS, smem, st>>>(hout, hscale, W_out, b_out, tgt, m, s, coef, inv_nvalid, dh,
                                                        n_tokens, H, v_begin, v_end, ldw, accumulate_dh);
    SEQREC_CHECK_LAUNCH();
  }
  if (dW_out) {
    auto k = ce_backward_dw_simt_kernel<HQ>;
    e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return -(int)e;
    const int v_tiles = ceil_div(v_end - v_begin, CT);
    const int64_t n_tiles = (n_tokens + CT - 1) / CT;
    int splits = ceil_div(2 * SEQREC_NUM_SMS, v_tiles);
    if (splits > n_tiles) splits = (int)n_tiles;
    if (splits < 1) splits = 1;
    const int tps = ceil_div(n_tiles, splits);
    splits = ceil_div(n_tiles, tps);
    dim3 grid(v_tiles, splits);
    k<<<grid, CE_THREADS, smem, st>>>(hout, hscale, W_out, b_out, tgt, m, s, coef, inv_nvalid, dW_out, db_out,
                                      n_tokens, H, v_begin, v_end, ldw, tps);
    SEQREC_CHECK_LAUNCH();
  }
  return 0;
}

int ce_backward_simt(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                     const int32_t* tgt, const float* m, const float* s, const float* coef, const float* inv_nvalid,
                     float* dh, float* dW_out, float* db_out, int64_t n_tokens, int H, int v_begin, int v_end,
                     int ldw, int accumulate_dh, cudaStream_t st) {
#define CE_BWD_ARGS hout, hscale, W_out, b_out, tgt, m, s, coef, inv_nvalid, dh, dW_out, db_out, n_tokens, H, \
                    v_begin, v_end, ldw, accumulate_dh, st
  if (H <= 64) return ce_backward_simt_t<4>(CE_BWD_ARGS);
  if (H <= 128) return ce_backward_simt_t<8>(CE_BWD_ARGS);
  if (H <= 256) return ce_backward_simt_t<16>(CE_BWD_ARGS);
  return -1011;  // hidden sizes above 256 are not a reference configuration
#undef CE_BWD_ARGS
}

static int ce_finalize_launch(const float* ws_m, const float* ws_s, const float* zy, const uint8_t* mask, float* m_out,
                              float* s_out, float* ce, float* py, float* coef, float* loss_sum, const int32_t* n_valid,
                              float* n_valid_f, float* loss_mean, int64_t n_tokens, int splits,
                              const int32_t* n_tokens_dev, void* stream) {
  SEQREC_ARG(n_tokens > 0 && splits > 0, 1);
  int blocks = (int)((n_tokens + FIN_THREADS - 1) / FIN_THREADS);   // one token per thread while the grid allows it
  if (blocks > FIN_MAX_BLOCKS) blocks = FIN_MAX_BLOCKS;
  ce_finalize_kernel<<<blocks, FIN_THREADS, 0, as_stream(stream)>>>(ws_m, ws_s, zy, mask, m_out, s_out, ce, py, coef,
                                                                   loss_sum, n_valid, n_valid_f, loss_mean, n_tokens,
                                                                   splits, n_tokens_dev);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_ce_finalize(const float* ws_m, const float* ws_s, const float* zy, const uint8_t* mask,
                                  float* m_out, float* s_out, float* ce, float* py, float* coef, float* loss_sum,
                                  int64_t n_tokens, int splits, void* stream) {
  return ce_finalize_launch(ws_m, ws_s, zy, mask, m_out, s_out, ce, py, coef, loss_sum, nullptr, nullptr, nullptr,
                            n_tokens, splits, nullptr, stream);
}

extern "C" int seqrec_ce_finalize_mean(const float* ws_m, const float* ws_s, const float* zy, const uint8_t* mask,
                                       float* m_out, float* s_out, float* ce, float* py, float* coef, float* loss_sum,
                                       const int32_t* n_valid, float* n_valid_f, float* loss_mean, int64_t n_tokens,
                                       int splits, const int32_t* n_tokens_dev, void* stream) {
  SEQREC_ARG(n_valid != nullptr, 11);
  SEQREC_ARG(n_tokens_dev == nullptr || splits == 1, 12);
  return ce_finalize_launch(ws_m, ws_s, zy, mask, m_out, s_out, ce, py, coef, loss_sum, n_valid, n_valid_f, loss_mean,
                            n_tokens, splits, n_tokens_dev, stream);
}

extern "C" int seqrec_predict_probs(const float* hout, const float* W_out, const float* b_out, const float* m,
                                    const float* s, float* probs_btv, int T, int B, int H, int V, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && H > 0 && V > 0, 1);
  const size_t smem = ce_smem_bytes(H, false);
  if (smem > 227 * 1024) return -1010;
  cudaError_t e =
      cudaFuncSetAttribute(predict_probs_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return -(int)e;
  dim3 grid(ceil_div((int64_t)T * B, CT), ceil_div(V, CT));
  predict_probs_simt_kernel<<<grid, CE_THREADS, smem, as_stream(stream)>>>(hout, W_out, b_out, m, s, probs_btv, T, B,
                                                                           H, V);
  SEQREC_CHECK_LAUNCH();
  return 0;
}
