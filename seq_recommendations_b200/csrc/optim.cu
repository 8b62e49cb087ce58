// K8: global-norm clip + Adagrad, dense and row-sparse (experiments_methods.py:41:
// Adagrad(lr, epsilon=1e-08, decay=0.0, clipnorm=1.)), clip + Keras Adam (compile_model's default optimizer, dense and
// over a whole embedding table), plus the dropout-factor generator and the bf16 hi/lo splitter
// that stages operands for the tensor-core logits kernels.  All HBM-bound elementwise passes.
#include "common.cuh"

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sumsq_kernel(const float* __restrict__ g, int64_t n, double* __restrict__ out) {
  __shared__ double red[8];
  double acc = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const int64_t n4 = n >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (int64_t i = i0; i < n4; i += stride) {
      const float4 v = __ldg(g4 + i);
      acc += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
    }
    for (int64_t i = (n4 << 2) + i0; i < n; i += stride) acc += (double)(g[i] * g[i]);
  } else {
    for (int64_t i = i0; i < n; i += stride) acc += (double)(g[i] * g[i]);
  }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double v = threadIdx.x < 8 ? red[threadIdx.x] : 0.0;
    v = warp_sum_d(v);
    if (threadIdx.x == 0) atomicAdd(out, v);
  }
}

// one warp per touched row
__global__ void __launch_bounds__(256)
sumsq_rows_kernel(const float* __restrict__ g, const int32_t* __restrict__ rows, const int32_t* __restrict__ n_rows,
                  int GH, double* __restrict__ out) {
  __shared__ double red[8];
  const int lane = threadIdx.x & 31;
  const int nr = n_rows[0];
  double acc = 0.0;
  for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < nr; w += (gridDim.x * blockDim.x) >> 5) {
    const float* row = g + (size_t)rows[w] * GH;
    if ((GH & 3) == 0) {
      const float4* r4 = reinterpret_cast<const float4*>(row);
      for (int c = lane; c < (GH >> 2); c += 32) {
        const float4 v = r4[c];
        acc += (double)(v.x * v.x) + (double)(v.y * v.y) + (double)(v.z * v.z) + (double)(v.w * v.w);
      }
    } else {
      for (int c = lane; c < GH; c += 32) acc += (double)(row[c] * row[c]);
    }
  }
  acc = warp_sum_d(acc);
  if (lane == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double v = threadIdx.x < 8 ? red[threadIdx.x] : 0.0;
    v = warp_sum_d(v);
    if (threadIdx.x == 0 && v != 0.0) atomicAdd(out, v);
  }
}

// factor applied to the stored gradient: 1/gdenom (the backward pass leaves gradients UN-normalised -- sums over tokens;
// gdenom[0] = the global number of unmasked steps the Keras objective divides by) times the clip factor of the
// normalised gradient.  sumsq[0] = sum of squares of the stored (un-normalised) gradient.
__device__ __forceinline__ float clip_scale(const double* sumsq, float clipnorm, const float* gdenom) {
  const float inv = gdenom ? 1.0f / gdenom[0] : 1.0f;
  if (!(clipnorm > 0.f) || sumsq == nullptr) return inv;
  const float norm = (float)sqrt(sumsq[0]) * inv;
  return (norm >= clipnorm) ? inv * (clipnorm / norm) : inv;  // Keras clip_norm: K.switch(n >= c, g*c/n, g)
}

__global__ void __launch_bounds__(256)
adagrad_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ a, int64_t n, float lr,
               float eps, float clipnorm, const double* __restrict__ sumsq, const float* __restrict__ gdenom) {
  const float sc = clip_scale(sumsq, clipnorm, gdenom);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(a)) & 15) == 0;
  const int64_t n4 = vec ? (n >> 2) : 0;
  float4* p4 = reinterpret_cast<float4*>(p);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* a4 = reinterpret_cast<float4*>(a);
  for (int64_t i = tid; i < n4; i += stride) {
    float4 gv = g4[i], av = a4[i], pv = p4[i];
    gv.x *= sc; gv.y *= sc; gv.z *= sc; gv.w *= sc;
    av.x += gv.x * gv.x; av.y += gv.y * gv.y; av.z += gv.z * gv.z; av.w += gv.w * gv.w;
    pv.x -= lr * gv.x / (sqrtf(av.x) + eps);
    pv.y -= lr * gv.y / (sqrtf(av.y) + eps);
    pv.z -= lr * gv.z / (sqrtf(av.z) + eps);
    pv.w -= lr * gv.w / (sqrtf(av.w) + eps);
    a4[i] = av;
    p4[i] = pv;
  }
  for (int64_t i = (n4 << 2) + tid; i < n; i += stride) {
    const float gv = g[i] * sc;
    const float av = a[i] + gv * gv;
    a[i] = av;
    p[i] = p[i] - lr * gv / (sqrtf(av) + eps);
  }
}

__global__ void __launch_bounds__(256)
adagrad_rows_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ a,
                    const int32_t* __restrict__ rows, const int32_t* __restrict__ n_rows,
                    int32_t* __restrict__ touched, int GH, float lr, float eps, float clipnorm,
                    const double* __restrict__ sumsq, const float* __restrict__ gdenom) {
  const float sc = clip_scale(sumsq, clipnorm, gdenom);
  const int lane = threadIdx.x & 31;
  const int nr = n_rows[0];
  for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < nr; w += (gridDim.x * blockDim.x) >> 5) {
    const int32_t row = rows[w];
    const size_t off = (size_t)row * GH;
    if ((GH & 3) == 0) {                         // 128-bit accesses: 3 loads + 3 stores per 4 parameters
      float4* p4 = reinterpret_cast<float4*>(p + off);
      float4* g4 = reinterpret_cast<float4*>(g + off);
      float4* a4 = reinterpret_cast<float4*>(a + off);
      for (int c = lane; c < (GH >> 2); c += 32) {
        float4 gv = g4[c], av = a4[c], pv = p4[c];
        gv.x *= sc; gv.y *= sc; gv.z *= sc; gv.w *= sc;
        av.x += gv.x * gv.x; av.y += gv.y * gv.y; av.z += gv.z * gv.z; av.w += gv.w * gv.w;
        pv.x -= lr * gv.x / (sqrtf(av.x) + eps);
        pv.y -= lr * gv.y / (sqrtf(av.y) + eps);
        pv.z -= lr * gv.z / (sqrtf(av.z) + eps);
        pv.w -= lr * gv.w / (sqrtf(av.w) + eps);
        a4[c] = av;
        p4[c] = pv;
        g4[c] = make_float4(0.f, 0.f, 0.f, 0.f);  // restore the all-zero invariant of the dense gradient buffer
      }
    } else {
      for (int c = lane; c < GH; c += 32) {
        const float gv = g[off + c] * sc;
        const float av = a[off + c] + gv * gv;
        a[off + c] = av;
        p[off + c] = p[off + c] - lr * gv / (sqrtf(av) + eps);
        g[off + c] = 0.f;
      }
    }
    if (lane == 0) touched[row] = 0;
  }
}

static int grid_for(int64_t n, int per_block) {
  int64_t b = (n + per_block - 1) / per_block;
  const int cap = SEQREC_NUM_SMS * 16;
  return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

extern "C" int seqrec_sumsq(const float* g, int64_t n, double* sumsq, void* stream) {
  SEQREC_ARG(n > 0, 1);
  sumsq_kernel<<<grid_for(n, 256 * 8), 256, 0, as_stream(stream)>>>(g, n, sumsq);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_sumsq_rows(const float* g, const int32_t* rows, const int32_t* n_rows, int GH, int max_rows,
                                 double* sumsq, void* stream) {
  SEQREC_ARG(GH > 0 && max_rows > 0, 1);
  sumsq_rows_kernel<<<grid_for(max_rows, 8), 256, 0, as_stream(stream)>>>(g, rows, n_rows, GH, sumsq);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_adagrad(float* p, const float* g, float* a, int64_t n, float lr, float eps, float clipnorm,
                              const double* sumsq, const float* gdenom, void* stream) {
  SEQREC_ARG(n > 0, 1);
  adagrad_kernel<<<grid_for(n, 256 * 4), 256, 0, as_stream(stream)>>>(p, g, a, n, lr, eps, clipnorm, sumsq, gdenom);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_adagrad_rows(float* p, float* g, float* a, const int32_t* rows, const int32_t* n_rows,
                                   int32_t* touched, int GH, int max_rows, float lr, float eps, float clipnorm,
                                   const double* sumsq, const float* gdenom, void* stream) {
  SEQREC_ARG(GH > 0 && max_rows > 0, 1);
  adagrad_rows_kernel<<<grid_for(max_rows, 8), 256, 0, as_stream(stream)>>>(p, g, a, rows, n_rows, touched, GH, lr,
                                                                            eps, clipnorm, sumsq, gdenom);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Keras 2.0.x Adam.  iterations[0] (device int64) = updates applied before this one; it is read here and advanced by
// the caller after the step, so a launch captured in a CUDA graph uses the current t at every replay.  The bias-
// corrected rate is computed in double once per block.
__device__ __forceinline__ float adam_lr_t(float lr, float beta_1, float beta_2, float decay,
                                           const int64_t* __restrict__ iterations) {
  __shared__ float lr_t;
  if (threadIdx.x == 0) {
    const double k = (double)iterations[0];
    const double lr_e = decay > 0.f ? (double)lr / (1.0 + (double)decay * k) : (double)lr;
    lr_t = (float)(lr_e * sqrt(1.0 - pow((double)beta_2, k + 1.0)) / (1.0 - pow((double)beta_1, k + 1.0)));
  }
  __syncthreads();
  return lr_t;
}

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float lr_t, float b1, float b2,
                                         float eps) {
  m = b1 * m + (1.f - b1) * g;
  v = b2 * v + (1.f - b2) * (g * g);
  p -= lr_t * m / (sqrtf(v) + eps);
}

__device__ __forceinline__ void adam_four(float4& p, float4 g, float4& m, float4& v, float lr_t, float b1, float b2,
                                          float eps) {
  adam_one(p.x, g.x, m.x, v.x, lr_t, b1, b2, eps);
  adam_one(p.y, g.y, m.y, v.y, lr_t, b1, b2, eps);
  adam_one(p.z, g.z, m.z, v.z, lr_t, b1, b2, eps);
  adam_one(p.w, g.w, m.w, v.w, lr_t, b1, b2, eps);
}

__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
            float lr, float b1, float b2, float eps, float decay, float clipnorm, const double* __restrict__ sumsq,
            const float* __restrict__ gdenom, const int64_t* __restrict__ iterations) {
  const float lr_t = adam_lr_t(lr, b1, b2, decay, iterations);
  const float sc = clip_scale(sumsq, clipnorm, gdenom);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  const int64_t n4 = vec ? (n >> 2) : 0;
  float4* p4 = reinterpret_cast<float4*>(p);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* m4 = reinterpret_cast<float4*>(m);
  float4* v4 = reinterpret_cast<float4*>(v);
  for (int64_t i = tid; i < n4; i += stride) {
    float4 gv = g4[i], mv = m4[i], vv = v4[i], pv = p4[i];
    gv.x *= sc; gv.y *= sc; gv.z *= sc; gv.w *= sc;
    adam_four(pv, gv, mv, vv, lr_t, b1, b2, eps);
    m4[i] = mv;
    v4[i] = vv;
    p4[i] = pv;
  }
  for (int64_t i = (n4 << 2) + tid; i < n; i += stride) {
    float pv = p[i], mv = m[i], vv = v[i];
    adam_one(pv, g[i] * sc, mv, vv, lr_t, b1, b2, eps);
    m[i] = mv;
    v[i] = vv;
    p[i] = pv;
  }
}

// Every row of the (F, GH) table moves (the reference's one-hot input product has a dense gradient); one warp per row.
// The gradient row is read only where touched[row] != 0 -- it is all zeros elsewhere -- and is then re-zeroed with its
// flag, which keeps the zero invariant of the dense gradient buffer that adagrad_rows_kernel keeps.
__global__ void __launch_bounds__(256)
adam_table_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                  int32_t* __restrict__ touched, int64_t F, int GH, float lr, float b1, float b2, float eps,
                  float decay, float clipnorm, const double* __restrict__ sumsq, const float* __restrict__ gdenom,
                  const int64_t* __restrict__ iterations) {
  const float lr_t = adam_lr_t(lr, b1, b2, decay, iterations);
  const float sc = clip_scale(sumsq, clipnorm, gdenom);
  const int lane = threadIdx.x & 31;
  const bool vec = (GH & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; row < F; row += warps) {
    int hot = lane == 0 ? touched[row] : 0;
    hot = __shfl_sync(0xffffffffu, hot, 0);
    const size_t off = (size_t)row * GH;
    if (vec) {                                   // 128-bit accesses
      float4* p4 = reinterpret_cast<float4*>(p + off);
      float4* g4 = reinterpret_cast<float4*>(g + off);
      float4* m4 = reinterpret_cast<float4*>(m + off);
      float4* v4 = reinterpret_cast<float4*>(v + off);
      for (int c = lane; c < (GH >> 2); c += 32) {
        float4 gv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (hot) {
          gv = g4[c];
          gv.x *= sc; gv.y *= sc; gv.z *= sc; gv.w *= sc;
          g4[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float4 mv = m4[c], vv = v4[c], pv = p4[c];
        adam_four(pv, gv, mv, vv, lr_t, b1, b2, eps);
        m4[c] = mv;
        v4[c] = vv;
        p4[c] = pv;
      }
    } else {
      for (int c = lane; c < GH; c += 32) {
        float gv = 0.f;
        if (hot) {
          gv = g[off + c] * sc;
          g[off + c] = 0.f;
        }
        float pv = p[off + c], mv = m[off + c], vv = v[off + c];
        adam_one(pv, gv, mv, vv, lr_t, b1, b2, eps);
        m[off + c] = mv;
        v[off + c] = vv;
        p[off + c] = pv;
      }
    }
    if (hot && lane == 0) touched[row] = 0;
  }
}

extern "C" int seqrec_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta_1,
                           float beta_2, float eps, float decay, float clipnorm, const double* sumsq,
                           const float* gdenom, const int64_t* iterations, void* stream) {
  SEQREC_ARG(n > 0, 1);
  SEQREC_ARG(iterations != nullptr, 14);
  adam_kernel<<<grid_for(n, 256 * 4), 256, 0, as_stream(stream)>>>(p, g, m, v, n, lr, beta_1, beta_2, eps, decay,
                                                                     clipnorm, sumsq, gdenom, iterations);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_adam_table(float* p, float* g, float* m, float* v, int32_t* touched, int64_t F, int GH,
                                 float lr, float beta_1, float beta_2, float eps, float decay, float clipnorm,
                                 const double* sumsq, const float* gdenom, const int64_t* iterations, void* stream) {
  SEQREC_ARG(F > 0 && GH > 0, 6);
  SEQREC_ARG(touched != nullptr && iterations != nullptr, 5);
  adam_table_kernel<<<grid_for(F, 8), 256, 0, as_stream(stream)>>>(p, g, m, v, touched, F, GH, lr, beta_1, beta_2,
                                                                   eps, decay, clipnorm, sumsq, gdenom, iterations);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Dropout factors.  Theano's MRG31k3p stream cannot be reproduced (SURVEY a5), so only the distribution is kept:
// out = 0 with probability `rate`, else 1/(1-rate).  Counter-based (splitmix64 of seed, offset+i): reproducible and
// independent of the launch geometry (splitmix64: common.cuh).

__global__ void __launch_bounds__(256)
dropout_mask_kernel(float* __restrict__ out, int64_t n, float rate, uint64_t seed, uint64_t offset) {
  const float keep = 1.0f / (1.0f - rate);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t r = splitmix64(splitmix64(seed) ^ (offset + (uint64_t)i));
    const float u = (float)(r >> 40) * (1.0f / 16777216.0f);
    out[i] = (u >= rate) ? keep : 0.f;
  }
}

// Same factors with the stream position held on the device: state[0] = offset of the next draw, state[1] = block ticket.
// Every block reads the offset when it starts and takes a ticket when it is done; the last one advances the offset by n
// and clears the ticket -- so a launch captured in a CUDA graph draws fresh factors at every replay.
__global__ void __launch_bounds__(256)
dropout_mask_dev_kernel(float* __restrict__ out, int64_t n, float rate, uint64_t seed,
                        unsigned long long* __restrict__ state) {
  const uint64_t offset = *((volatile unsigned long long*)state);
  const float keep = 1.0f / (1.0f - rate);
  const uint64_t key = splitmix64(seed);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint64_t r = splitmix64(key ^ (offset + (uint64_t)i));
    const float u = (float)(r >> 40) * (1.0f / 16777216.0f);
    out[i] = (u >= rate) ? keep : 0.f;
  }
  __syncthreads();                             // every thread of the block has read the offset
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(state + 1, 1ull) == (unsigned long long)gridDim.x - 1) {
      state[0] = offset + (uint64_t)n;
      state[1] = 0ull;
    }
  }
}

extern "C" int seqrec_dropout_mask_dev(float* out, int64_t n, float rate, uint64_t seed, uint64_t* state,
                                       void* stream) {
  SEQREC_ARG(n > 0 && rate >= 0.f && rate < 1.f, 1);
  SEQREC_ARG(state != nullptr, 5);
  dropout_mask_dev_kernel<<<grid_for(n, 256 * 4), 256, 0, as_stream(stream)>>>(
      out, n, rate, seed, reinterpret_cast<unsigned long long*>(state));
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_dropout_mask(float* out, int64_t n, float rate, uint64_t seed, uint64_t offset, void* stream) {
  SEQREC_ARG(n > 0 && rate >= 0.f && rate < 1.f, 1);
  dropout_mask_kernel<<<grid_for(n, 256 * 4), 256, 0, as_stream(stream)>>>(out, n, rate, seed, offset);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 -> (hi, lo) bf16 with hi = bf16(x), lo = bf16(x - hi): 16 mantissa bits between them.
__global__ void __launch_bounds__(256)
split_bf16_kernel(const float* __restrict__ src, const float* __restrict__ scale, __nv_bfloat16* __restrict__ hi,
                  __nv_bfloat16* __restrict__ lo, int64_t rows, int64_t cols, int64_t ld_out) {
  const int64_t total = rows * cols;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t r = i / cols, c = i - r * cols;
    float x = src[i];
    if (scale) x *= scale[i];
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    const __nv_bfloat16 l = __float2bfloat16_rn(x - __bfloat162float(h));
    hi[r * ld_out + c] = h;
    if (lo) lo[r * ld_out + c] = l;
  }
}

// transposing variant through a 32x32 shared-memory tile: out is (cols, rows) with leading dimension ld_out
__global__ void split_bf16_t_kernel(const float* __restrict__ src, const float* __restrict__ scale,
                                    __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int64_t rows,
                                    int64_t cols, int64_t ld_out) {
  __shared__ float tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    float x = 0.f;
    if (r < rows && c < cols) {
      x = src[r * cols + c];
      if (scale) x *= scale[r * cols + c];
    }
    tile[i][threadIdx.x] = x;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) {
      const float x = tile[threadIdx.x][i];
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      hi[c * ld_out + r] = h;
      if (lo) lo[c * ld_out + r] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
  }
}

// both layouts from ONE read of the source: out (rows, cols) with leading dimension ld_out AND out_t (cols, rows) with
// leading dimension ld_t (32x32 tiles through shared memory)
__global__ void split_bf16_both_kernel(const float* __restrict__ src, const float* __restrict__ scale,
                                       __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                       __nv_bfloat16* __restrict__ hi_t, __nv_bfloat16* __restrict__ lo_t,
                                       int64_t rows, int64_t cols, int64_t ld_out, int64_t ld_t) {
  __shared__ float tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    float x = 0.f;
    if (r < rows && c < cols) {
      x = src[r * cols + c];
      if (scale) x *= scale[r * cols + c];
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      hi[r * ld_out + c] = h;
      if (lo) lo[r * ld_out + c] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
    tile[i][threadIdx.x] = x;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) {
      const float x = tile[threadIdx.x][i];
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      hi_t[c * ld_t + r] = h;
      if (lo_t) lo_t[c * ld_t + r] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
  }
}

extern "C" int seqrec_split_bf16_both(const float* src, const float* scale, uint16_t* hi, uint16_t* lo, uint16_t* hi_t,
                                      uint16_t* lo_t, int64_t rows, int64_t cols, int64_t ld_out, int64_t ld_t,
                                      void* stream) {
  SEQREC_ARG(src && hi && hi_t && rows > 0 && cols > 0 && ld_out >= cols && ld_t >= rows, 1);
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32)), block(32, 8);
  SEQREC_ARG(grid.y <= 65535, 2);
  split_bf16_both_kernel<<<grid, block, 0, as_stream(stream)>>>(
      src, scale, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo),
      reinterpret_cast<__nv_bfloat16*>(hi_t), reinterpret_cast<__nv_bfloat16*>(lo_t), rows, cols, ld_out, ld_t);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// ---- token compaction --------------------------------------------------------------------------------------------
// Pad tokens carry neither loss nor gradient, so the logits kernels of a training step run on the VALID tokens only:
// orig[c] = time-major index of the c-th valid token IN ASCENDING ORDER (deterministic: every rank of a
// vocabulary-parallel step must number the gathered tokens identically), tgt_c[c] = its target, count[0] = number of
// valid tokens.  Two launches: per-block counts, then every block sums the counts in front of it and scatters.
__global__ void __launch_bounds__(256)
compact_count_kernel(const uint8_t* __restrict__ mask, int64_t n_tokens, int32_t* __restrict__ block_counts) {
  const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int c = __syncthreads_count(n < n_tokens && mask[n] != 0);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(256)
compact_scatter_kernel(const uint8_t* __restrict__ mask, const int32_t* __restrict__ tgt, int64_t n_tokens,
                       const int32_t* __restrict__ block_counts, int32_t* __restrict__ orig,
                       int32_t* __restrict__ tgt_c, int32_t* __restrict__ count) {
  __shared__ int warp_base[8];
  __shared__ int block_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // exclusive prefix of the block counts (a few hundred values)
  int part = 0;
  for (int i = threadIdx.x; i < (int)blockIdx.x; i += blockDim.x) part += block_counts[i];
  part = (int)warp_sum((float)part);            // exact: counts are far below 2^24 per warp partial
  if (lane == 0) warp_base[warp] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int i = 0; i < 8; ++i) t += warp_base[i];
    block_base = t;
  }
  __syncthreads();
  const int base0 = block_base;
  __syncthreads();
  const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const bool on = n < n_tokens && mask[n] != 0;
  const unsigned bal = __ballot_sync(0xffffffffu, on);
  if (lane == 0) warp_base[warp] = __popc(bal);
  __syncthreads();
  int wb = 0;
  for (int i = 0; i < warp; ++i) wb += warp_base[i];
  if (on) {
    const int c = base0 + wb + __popc(bal & ((1u << lane) - 1u));
    orig[c] = (int32_t)n;
    if (tgt_c) tgt_c[c] = tgt[n];
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
    int t = 0;
    for (int i = 0; i < 8; ++i) t += warp_base[i];
    count[0] = base0 + t;
  }
}

extern "C" int seqrec_compact_tokens(const uint8_t* mask, const int32_t* tgt, int64_t n_tokens, int32_t* orig,
                                     int32_t* tgt_c, int32_t* count, int32_t* block_counts, void* stream) {
  SEQREC_ARG(mask && orig && count && block_counts && n_tokens > 0 && n_tokens < (1ll << 30), 1);
  const unsigned blocks = (unsigned)((n_tokens + 255) / 256);
  compact_count_kernel<<<blocks, 256, 0, as_stream(stream)>>>(mask, n_tokens, block_counts);
  SEQREC_CHECK_LAUNCH();
  compact_scatter_kernel<<<blocks, 256, 0, as_stream(stream)>>>(mask, tgt, n_tokens, block_counts, orig, tgt_c, count);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// split_bf16_both over the compacted rows: output row r (r < n_rows[0], read on the device) is source row orig[r]
__global__ void split_bf16_both_rows_kernel(const float* __restrict__ src, const float* __restrict__ scale,
                                            const int32_t* __restrict__ orig, const int32_t* __restrict__ n_rows,
                                            __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                            __nv_bfloat16* __restrict__ hi_t, __nv_bfloat16* __restrict__ lo_t,
                                            int64_t cols, int64_t ld_out, int64_t ld_t) {
  __shared__ float tile[32][33];
  const int64_t rows = n_rows[0];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  if (r0 >= rows) return;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    float x = 0.f;
    if (r < rows && c < cols) {
      const int64_t sr = orig[r];
      x = src[sr * cols + c];
      if (scale) x *= scale[sr * cols + c];
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      hi[r * ld_out + c] = h;
      if (lo) lo[r * ld_out + c] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
    tile[i][threadIdx.x] = x;
  }
  __syncthreads();
  if (!hi_t) return;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) {
      const float x = tile[threadIdx.x][i];
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      hi_t[c * ld_t + r] = h;
      if (lo_t) lo_t[c * ld_t + r] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
  }
}

extern "C" int seqrec_split_bf16_both_rows(const float* src, const float* scale, const int32_t* orig,
                                           const int32_t* n_rows, uint16_t* hi, uint16_t* lo, uint16_t* hi_t,
                                           uint16_t* lo_t, int64_t max_rows, int64_t cols, int64_t ld_out, int64_t ld_t,
                                           void* stream) {
  SEQREC_ARG(src && orig && n_rows && hi && max_rows > 0 && cols > 0 && ld_out >= cols && ld_t >= max_rows, 1);
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((max_rows + 31) / 32)), block(32, 8);
  SEQREC_ARG(grid.y <= 65535, 2);
  split_bf16_both_rows_kernel<<<grid, block, 0, as_stream(stream)>>>(
      src, scale, orig, n_rows, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo),
      reinterpret_cast<__nv_bfloat16*>(hi_t), reinterpret_cast<__nv_bfloat16*>(lo_t), cols, ld_out, ld_t);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// split + column sums in one pass over src (the dU GEMM's dxp operand and db = sum_n dxp[n,:] both come from it):
// thread <-> column, blockIdx.y <-> a chunk of rows; partial column sums leave through atomicAdd
__global__ void __launch_bounds__(256)
split_bf16_colsum_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                         float* __restrict__ colsum, int64_t rows, int cols, int64_t rows_per_block) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int64_t r0 = blockIdx.y * rows_per_block;
  const int64_t r1 = rows < r0 + rows_per_block ? rows : r0 + rows_per_block;
  float acc = 0.f;
#pragma unroll 4
  for (int64_t r = r0; r < r1; ++r) {
    const float x = src[r * cols + c];
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    hi[r * cols + c] = h;
    lo[r * cols + c] = __float2bfloat16_rn(x - __bfloat162float(h));
    acc += x;
  }
  if (colsum) atomicAdd(colsum + c, acc);
}

extern "C" int seqrec_split_bf16_colsum(const float* src, uint16_t* hi, uint16_t* lo, float* colsum, int64_t rows,
                                        int cols, void* stream) {
  SEQREC_ARG(src && hi && lo && rows > 0 && cols > 0, 1);
  const int64_t rpb = 32;
  dim3 grid((unsigned)((cols + 255) / 256), (unsigned)((rows + rpb - 1) / rpb));
  if (grid.y > 65535) return -1003;
  split_bf16_colsum_kernel<<<grid, 256, 0, as_stream(stream)>>>(src, reinterpret_cast<__nv_bfloat16*>(hi),
                                                                reinterpret_cast<__nv_bfloat16*>(lo), colsum, rows, cols,
                                                                rpb);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_split_bf16(const float* src, const float* scale, uint16_t* hi, uint16_t* lo, int64_t rows,
                                 int64_t cols, int64_t ld_out, int transpose, void* stream) {
  SEQREC_ARG(rows > 0 && cols > 0 && ld_out > 0, 1);
  __nv_bfloat16* h = reinterpret_cast<__nv_bfloat16*>(hi);
  __nv_bfloat16* l = reinterpret_cast<__nv_bfloat16*>(lo);
  if (!transpose) {
    split_bf16_kernel<<<grid_for(rows * cols, 256 * 4), 256, 0, as_stream(stream)>>>(src, scale, h, l, rows, cols,
                                                                                     ld_out);
  } else {
    dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32)), block(32, 8);
    SEQREC_ARG(grid.y <= 65535, 2);
    split_bf16_t_kernel<<<grid, block, 0, as_stream(stream)>>>(src, scale, h, l, rows, cols, ld_out);
  }
  SEQREC_CHECK_LAUNCH();
  return 0;
}
