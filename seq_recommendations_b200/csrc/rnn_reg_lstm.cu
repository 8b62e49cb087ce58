// K3 / K4 fast path for LSTM cells with H <= 100 (cfg1: the reference's own LSTM-100, experiments_server.py:40-42):
// the recurrent kernel U (H x 4H fp32; H = 100: 160 KB) lives in REGISTERS for all T timesteps.
//
// The generic scan (rnn_scan.cu) re-reads U from shared memory at every step: with one batch row per CTA (B = 100 on
// 148 SMs) every FFMA needs its own 4-byte shared-memory operand, i.e. 160 KB / (128 B/clk) = 1250 clocks per step
// before any latency -- measured 2.3 us per step.  Here a persistent CTA of KS*CG threads (CG = H rounded up to 4, KS
// K-slices of KPT hidden units; H = 100: 5 x 100 = 500 threads, 80 registers of U each) owns RB batch rows: thread
// (s, c) keeps K-slice s of the four gate columns of unit c (forward) / of row c of U (backward) in registers, a step
// reads only the hidden vector (forward) or the four pre-activation gradients (backward) from shared memory as
// warp-wide broadcasts, and the KS partial sums meet in shared memory.  Thread (s, c) with s < RB OWNS unit c of batch
// row s: it does the gate math and keeps c_t, the carried dL/dh and dL/dc in registers.  Per-step inputs are prefetched
// one step ahead with cp.async (each owner waits only for its own copies).  Two CTA barriers per step.
// Same semantics, inputs and outputs as the generic LSTM kernels (Keras-2.0.x gate order i, f, c, o; hard_sigmoid
// gates; Theano K.rnn mask switch: masked steps hold h and c).
#include "common.cuh"
#include "rnn_reg.cuh"

namespace {
using namespace regscan;

constexpr int G = 4;

template <int KS, int KPT>
struct Shape {
  static constexpr int KP = KS * KPT;                       // padded hidden size of the dot products
  static constexpr int MAXT = (KS * KP + 31) / 32 * 32;     // CG <= KP
};

// ---------------------------------------------------------------------------------------------------------------
// INIT: h_{-1} and c_{-1} are loaded from h0 and c0 (B,H) instead of zeros; a NULL pointer stands for zeros
template <int ACT, int RB, int KS, int KPT, bool INIT>
__global__ void __launch_bounds__(Shape<KS, KPT>::MAXT, 1)
lstm_forward_reg_kernel(float* __restrict__ xg, const float* __restrict__ U, const uint8_t* __restrict__ mask,
                        float* __restrict__ hout, float* __restrict__ cst, int T, int B, int H, int CG,
                        const float* __restrict__ h0, const float* __restrict__ c0) {
  static_assert(RB <= KS, "one owner thread per (row, unit) needs RB <= KS");
  constexpr int KP = Shape<KS, KPT>::KP;
  const int GH = G * H;
  extern __shared__ __align__(16) float smem[];
  float* h_s = smem;                            // [RB][KP]          h_{t-1} (zero beyond H)
  float* part_s = h_s + RB * KP;                // [KS][RB][G][CG]   partial sums
  float* x_s = part_s + KS * RB * G * CG;       // [2][RB][G][CG]    input projection, double buffered (cp.async)
  const int tid = threadIdx.x;
  const int s = tid / CG, c = tid - s * CG;
  const int b0 = blockIdx.x * RB;
  const bool owner = (s < RB) && (c < H) && (b0 + s < B);
  const int r = s;                              // the batch row this thread owns when `owner`

  float u[G][KPT];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
      const int k = s * KPT + i;
      u[g][i] = (k < H && c < H && s < KS) ? U[(size_t)k * GH + g * H + c] : 0.f;
    }
  if constexpr (INIT) {
    for (int i = tid; i < RB * KP; i += blockDim.x) {
      const int q = i / KP, k = i - q * KP;
      h_s[i] = (h0 && k < H && b0 + q < B) ? h0[(size_t)(b0 + q) * H + k] : 0.f;
    }
  } else {
    for (int i = tid; i < RB * KP; i += blockDim.x) h_s[i] = 0.f;
  }

  auto prefetch_x = [&](int t) {
    if (owner && t < T) {
#pragma unroll
      for (int g = 0; g < G; ++g)
        cp_async4(x_s + (((t & 1) * RB + r) * G + g) * CG + c, xg + ((size_t)t * B + b0 + r) * GH + g * H + c);
    }
    cp_async_commit();
  };
  // mask of this / the next step in registers (the load is issued two steps ahead)
  bool m0 = false, m1 = false;
  if (owner) {
    m0 = mask[b0 + r] != 0;
    m1 = (1 < T) ? (mask[(size_t)B + b0 + r] != 0) : false;
  }
  float hp = 0.f, cp = 0.f;                     // owner: h_{t-1}, c_{t-1} of (row r, unit c)
  if (INIT && owner) {
    if (h0) hp = h0[(size_t)(b0 + r) * H + c];
    if (c0) cp = c0[(size_t)(b0 + r) * H + c];
  }
  prefetch_x(0);
  __syncthreads();

  for (int t = 0; t < T; ++t) {
    const float* xc = x_s + (t & 1) * RB * G * CG;
    prefetch_x(t + 1);
    {
      float acc[G][RB];
#pragma unroll
      for (int g = 0; g < G; ++g)
#pragma unroll
        for (int q = 0; q < RB; ++q) acc[g][q] = 0.f;
      if (s < KS) dot_slices<RB, KPT, G, G>(acc, h_s, KP, s * KPT, u, 0);
      if (s < KS && c < CG) {
#pragma unroll
        for (int g = 0; g < G; ++g)
#pragma unroll
          for (int q = 0; q < RB; ++q) part_s[((s * RB + q) * G + g) * CG + c] = acc[g][q];
      }
    }
    cp_async_wait<1>();                         // this step's xp (own elements, issued one step ago) has landed
    __syncthreads();
    if (owner) {
      const size_t tok = (size_t)t * B + b0 + r;
      bool m2 = false;
      if (t + 2 < T) m2 = mask[(size_t)(t + 2) * B + b0 + r] != 0;
      float a[G];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float v = xc[(r * G + g) * CG + c];
#pragma unroll
        for (int q = 0; q < KS; ++q) v += part_s[((q * RB + r) * G + g) * CG + c];
        a[g] = v;
      }
      const float ig = hard_sigmoid_f(a[0]);
      const float fg = hard_sigmoid_f(a[1]);
      const float gg = act_f<ACT>(a[2]);
      const float og = hard_sigmoid_f(a[3]);
      const float cn = fmaf(fg, cp, ig * gg);
      const float hn = og * act_f<ACT>(cn);
      cp = m0 ? cn : cp;
      hp = m0 ? hn : hp;
      cst[tok * H + c] = cp;
      float* gp = xg + tok * GH;
      gp[c] = ig; gp[H + c] = fg; gp[2 * H + c] = gg; gp[3 * H + c] = og;
      hout[tok * H + c] = hp;
      h_s[r * KP + c] = hp;
      m0 = m1;
      m1 = m2;
    }
    __syncthreads();
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------------------------
// backward: thread (s, c) holds U[c][g*H + s*KPT + i] -- row c of U, K-slice s of every gate block:
//   dL/dh_{t-1}[c] = sum_g sum_j da_g[j] * U[c][g*H + j]
template <int ACT, int RB, int KS, int KPT>
__global__ void __launch_bounds__(Shape<KS, KPT>::MAXT, 1)
lstm_backward_reg_kernel(float* __restrict__ xg, const float* __restrict__ U, const uint8_t* __restrict__ mask,
                         const float* __restrict__ cst, const float* __restrict__ dhout, int T, int B, int H, int CG) {
  static_assert(RB <= KS, "one owner thread per (row, unit) needs RB <= KS");
  constexpr int KP = Shape<KS, KPT>::KP;
  constexpr int NI = 7;                         // prefetched per step: dL/dhout, i, f, g, o, c_t, c_{t-1}
  const int GH = G * H;
  extern __shared__ __align__(16) float smem[];
  float* da_s = smem;                           // [G][RB][KP]       pre-activation gradients of this step
  float* part_s = da_s + G * RB * KP;           // [KS][RB][CG]
  float* in_s = part_s + KS * RB * CG;          // [2][RB][NI][CG]   per-step inputs, double buffered (cp.async)
  const int tid = threadIdx.x;
  const int s = tid / CG, c = tid - s * CG;
  const int b0 = blockIdx.x * RB;
  const bool owner = (s < RB) && (c < H) && (b0 + s < B);
  const int r = s;

  // U rows into registers through shared memory, one gate block at a time: the block is read with coalesced rows and
  // each thread then picks ITS row out of a (H+1)-strided tile (reading U[c][...] directly is one cache line per lane)
  float u[G][KPT];
  {
    float* tile = smem;                         // [H][H+1], aliases the step buffers (initialised below)
    const int ld = H + 1;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      for (int i = tid; i < H * H; i += blockDim.x) {
        const int row = i / H, col = i - row * H;
        tile[row * ld + col] = U[(size_t)row * GH + g * H + col];
      }
      __syncthreads();
#pragma unroll
      for (int i = 0; i < KPT; ++i) {
        const int k = s * KPT + i;
        u[g][i] = (k < H && c < H && s < KS) ? tile[c * ld + k] : 0.f;
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < G * RB * KP; i += blockDim.x) da_s[i] = 0.f;

  auto prefetch_in = [&](int t) {
    if (owner && t >= 0) {
      float* dst = in_s + ((size_t)(t & 1) * RB + r) * NI * CG + c;
      const size_t tok = (size_t)t * B + b0 + r;
      cp_async4(dst, dhout + tok * H + c);
#pragma unroll
      for (int g = 0; g < G; ++g) cp_async4(dst + (1 + g) * CG, xg + tok * GH + g * H + c);
      cp_async4(dst + 5 * CG, cst + tok * H + c);
      if (t > 0) cp_async4(dst + 6 * CG, cst + (tok - B) * H + c);
    }
    cp_async_commit();
  };
  bool m0 = false, m1 = false;
  if (owner) {
    m0 = mask[(size_t)(T - 1) * B + b0 + r] != 0;
    m1 = (T - 2 >= 0) ? (mask[(size_t)(T - 2) * B + b0 + r] != 0) : false;
  }
  float dh_carry = 0.f, dc_carry = 0.f;         // owner: dL/dh_t and dL/dc_t arriving from later steps
  prefetch_in(T - 1);
  __syncthreads();

  for (int t = T - 1; t >= 0; --t) {
    prefetch_in(t - 1);
    cp_async_wait<1>();                         // this step's inputs (own elements) have landed
    float dd = 0.f;                             // direct (non-matmul) part of dL/dh_{t-1}
    if (owner) {
      const float* ic = in_s + ((size_t)(t & 1) * RB + r) * NI * CG + c;
      const size_t tok = (size_t)t * B + b0 + r;
      bool m2 = false;
      if (t - 2 >= 0) m2 = mask[(size_t)(t - 2) * B + b0 + r] != 0;
      const float dh = ic[0] + dh_carry;
      float da[G] = {0.f, 0.f, 0.f, 0.f};
      if (!m0) {
        dd = dh;                                // masked step: h_t = h_{t-1}, c_t = c_{t-1}, no gate gradient
      } else {
        const float ig = ic[CG], fg = ic[2 * CG], gg = ic[3 * CG], og = ic[4 * CG];
        const float ct = ic[5 * CG];
        const float cprev = (t > 0) ? ic[6 * CG] : 0.f;
        const float ac = act_f<ACT>(ct);
        const float dc = dc_carry + dh * og * act_grad_from_y<ACT>(ac);
        da[0] = dc * gg * hard_sigmoid_grad_from_y(ig);
        da[1] = dc * cprev * hard_sigmoid_grad_from_y(fg);
        da[2] = dc * ig * act_grad_from_y<ACT>(gg);
        da[3] = dh * ac * hard_sigmoid_grad_from_y(og);
        dc_carry = dc * fg;
      }
      // dxp[t] = da (overwrites the saved gates, already copied to shared memory by the prefetch)
      float* gp = xg + tok * GH;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        da_s[(g * RB + r) * KP + c] = da[g];
        gp[g * H + c] = da[g];
      }
      m0 = m1;
      m1 = m2;
    }
    __syncthreads();
    {
      float acc[1][RB];
#pragma unroll
      for (int q = 0; q < RB; ++q) acc[0][q] = 0.f;
      if (s < KS) {
#pragma unroll
        for (int g = 0; g < G; ++g) dot_slices<RB, KPT, 1, G>(acc, da_s + g * RB * KP, KP, s * KPT, u, g);
      }
      if (s < KS && c < CG) {
#pragma unroll
        for (int q = 0; q < RB; ++q) part_s[(s * RB + q) * CG + c] = acc[0][q];
      }
    }
    __syncthreads();
    if (owner) {
      float v = dd;
#pragma unroll
      for (int q = 0; q < KS; ++q) v += part_s[(q * RB + r) * CG + c];
      dh_carry = v;
    }
    // (no third barrier: the next step's first shared-memory writes -- da_s by the owners -- come after every thread's
    //  reads of da_s above, and part_s is rewritten only behind the next step's first barrier)
  }
  cp_async_wait<0>();
}

template <int ACT, int RB, int KS, int KPT>
int launch_lstm(bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst, const float* dhout,
                int T, int B, int H, cudaStream_t st, const float* h0, const float* c0) {
  constexpr int KP = Shape<KS, KPT>::KP;
  const int CG = (H + 3) / 4 * 4;
  const int threads = (KS * CG + 31) / 32 * 32;
  const int grid = ceil_div(B, RB);
  if (fwd) {
    const size_t smem = sizeof(float) * (size_t)(RB * KP + KS * RB * G * CG + 2 * RB * G * CG);
    auto k = (h0 || c0) ? lstm_forward_reg_kernel<ACT, RB, KS, KPT, true>
                        : lstm_forward_reg_kernel<ACT, RB, KS, KPT, false>;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return -(int)e;
    }
    k<<<grid, threads, smem, st>>>(xg, U, mask, hout, cst, T, B, H, CG, h0, c0);
  } else {
    const size_t smem_step = sizeof(float) * (size_t)(G * RB * KP + KS * RB * CG + 2 * RB * 7 * CG);
    const size_t smem_load = sizeof(float) * (size_t)H * (H + 1);
    const size_t smem = smem_step > smem_load ? smem_step : smem_load;
    auto k = lstm_backward_reg_kernel<ACT, RB, KS, KPT>;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return -(int)e;
    }
    k<<<grid, threads, smem, st>>>(xg, U, mask, cst, dhout, T, B, H, CG);
  }
  SEQREC_CHECK_LAUNCH();
  return 0;
}

template <int ACT, int RB>
int dispatch_shape(bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                   const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0, const float* c0) {
  // (KS, KPT): KS*KPT >= H, KPT a multiple of 4 (float4 reads of the K-slice), 4*KPT registers of U per thread
  if (H <= 32) return launch_lstm<ACT, RB, 4, 8>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
  if (H <= 64) return launch_lstm<ACT, RB, 4, 16>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
  if (H <= 80) return launch_lstm<ACT, RB, 4, 20>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
  return launch_lstm<ACT, RB, 5, 20>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
}

template <int ACT>
int dispatch_rb(int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0, const float* c0) {
  if (rb <= 1) return dispatch_shape<ACT, 1>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
  return dispatch_shape<ACT, 2>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
}

}  // namespace

bool lstm_reg_applicable(int H) { return H <= 100; }

// rb: batch rows per CTA (clamped to 2).  U is the untransposed recurrent kernel (H, 4H) for BOTH directions.
int lstm_reg_launch(int act, int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                    const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0, const float* c0) {
  switch (act) {
    case SEQREC_ACT_RELU:
      return dispatch_rb<SEQREC_ACT_RELU>(rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
    case SEQREC_ACT_TANH:
      return dispatch_rb<SEQREC_ACT_TANH>(rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
    case SEQREC_ACT_LINEAR:
      return dispatch_rb<SEQREC_ACT_LINEAR>(rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
    default: return -1002;
  }
}
