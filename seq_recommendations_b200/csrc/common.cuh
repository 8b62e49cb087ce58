// Shared device/host helpers for the seqrec_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "../../include/seqrec_b200.h"

#define SEQREC_NUM_SMS 148

// every kernel launch of the library is followed by this macro; it also feeds seqrec_launch_count()
void seqrec_note_launch();
#define SEQREC_CHECK_LAUNCH()                        \
  do {                                               \
    cudaError_t e__ = cudaGetLastError();            \
    if (e__ != cudaSuccess) return -(int)e__;        \
    seqrec_note_launch();                            \
  } while (0)

#define SEQREC_ARG(cond, code)  \
  do {                          \
    if (!(cond)) return -1000 - (code); \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Keras `_EPSILON` = 1e-7 cast to float32 on both clip bounds (Theano backend categorical_crossentropy).
#define SEQREC_P_EPS 1.0000000116860974e-07f
#define SEQREC_P_ONE_MINUS_EPS 0.99999988079071045f

__device__ __forceinline__ float hard_sigmoid_f(float a) { return fminf(fmaxf(0.2f * a + 0.5f, 0.0f), 1.0f); }
// derivative from the POST-activation value: 0.2 on the open linear piece
__device__ __forceinline__ float hard_sigmoid_grad_from_y(float y) { return (y > 0.0f && y < 1.0f) ? 0.2f : 0.0f; }

template <int ACT>
__device__ __forceinline__ float act_f(float a) {
  if (ACT == SEQREC_ACT_RELU) return fmaxf(a, 0.0f);
  if (ACT == SEQREC_ACT_TANH) return tanhf(a);
  return a;
}
template <int ACT>
__device__ __forceinline__ float act_grad_from_y(float y) {
  if (ACT == SEQREC_ACT_RELU) return y > 0.0f ? 1.0f : 0.0f;
  if (ACT == SEQREC_ACT_TANH) return 1.0f - y * y;
  return 1.0f;
}

// counter-based random stream of the dropout factors and the sampled-softmax draws: r_i = splitmix64(splitmix64(seed) ^
// (offset + i)) -- reproducible and independent of the launch geometry
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// streaming 128-bit accesses that do not pollute L1 (rows are touched once per kernel)
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
// vector reduction to global memory (sm_90+): one L2 atomic transaction for four floats
__device__ __forceinline__ void red_add_f4(float* p, const float4& v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
