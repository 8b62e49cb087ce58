// K3 / K4 fast path: GRU and SimpleRNN scans with the recurrent kernel held in REGISTERS for all T timesteps.
//
// For H <= 128 the whole recurrent kernel U (H x G*H fp32; cfg2 GRU-128: 192 KB) fits in the 256 KB register file of
// one SM.  A persistent CTA of 4*CG threads (CG = H rounded up to 32) owns RB batch rows for the whole sequence:
// thread (s, c) keeps the K-slice s of the gate columns of hidden unit c (forward) or of row c of U (backward) in
// registers, so a timestep reads only the RB hidden vectors from shared memory (warp-wide broadcasts), does its share
// of the (RB x H).(H x G*H) product as register FFMAs, and the four K-slices are summed through shared memory.
// Everything a step needs from global memory (input projection / saved gates / dL/dh / mask) is prefetched one step
// ahead into shared memory with cp.async, so neither load latency nor staging registers sit on the sequential path:
// 96 of the 128 registers per thread hold U.
// Same semantics, inputs and outputs as the generic kernels in rnn_scan.cu (Keras-2.0.x GRU: reset applied BEFORE the
// recurrent matmul -> two dependent matvec phases per step; Theano K.rnn mask switch).
#include "common.cuh"
#include "rnn_reg.cuh"

namespace {
using namespace regscan;

constexpr int KS = 4;  // K-slices

template <int CELL>
struct Gates { static constexpr int G = (CELL == SEQREC_CELL_GRU) ? 3 : 1; };

// ---------------------------------------------------------------------------------------------------------------
// INIT: h_{-1} is loaded from h0 (B,H) instead of zeros (rh_s is recomputed every step)
template <int CELL, int ACT, int RB, int KPT, bool INIT>
__global__ void __launch_bounds__(KS * 128, 1)
rnn_forward_reg_kernel(float* __restrict__ xg, const float* __restrict__ U, const uint8_t* __restrict__ mask,
                       float* __restrict__ hout, int T, int B, int H, const float* __restrict__ h0) {
  constexpr int G = Gates<CELL>::G;
  constexpr int G1 = (CELL == SEQREC_CELL_GRU) ? 2 : 1;   // gates whose recurrent product uses h_{t-1} itself
  constexpr int KP = KS * KPT;                 // padded hidden size seen by the dot products
  constexpr int CG = KP;                       // blockDim.x / KS: H rounded up to 32 == KS * KPT (dispatch_kpt)
  const int GH = G * H;
  extern __shared__ __align__(16) float smem[];
  float* h_s = smem;                           // [RB][KP]        h_{t-1}
  float* rh_s = h_s + RB * KP;                 // [RB][KP]        GRU: r * h_{t-1}
  float* part_s = rh_s + RB * KP;              // [KS][RB][G][CG] partial sums
  float* x_s = part_s + KS * RB * G * CG;      // [2][RB][G][CG]  input projection, double buffered (cp.async)
  float* zr_s = x_s + 2 * RB * G * CG;         // [RB][2][CG]     GRU: z and r of this step
  int* m_s = reinterpret_cast<int*>(zr_s + RB * 2 * CG);  // [2][RB] mask of this / next step
  const int tid = threadIdx.x;
  const int s = tid / CG, c = tid - s * CG;
  const int b0 = blockIdx.x * RB;
  // elementwise work (gate math, stores, prefetch) of hidden unit c is spread over the K-slice threads: thread (s, c)
  // with s < RB owns batch row s -- with one owner per unit looping over the rows, 12 of the 16 warps sat in the
  // barrier behind 4 (ncu: 45 % of the samples were stall_barrier)
  const bool owner = (s < RB) && (c < H);
  const int orow = s;                          // the row this thread owns when `owner`

  float u[G][KPT];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
      const int k = s * KPT + i;
      u[g][i] = (k < H && c < H) ? U[(size_t)k * GH + g * H + c] : 0.f;
    }
  if constexpr (INIT) {
    for (int i = tid; i < 2 * RB * KP; i += blockDim.x) {
      const int r = i / KP, k = i - r * KP;    // r >= RB: rh_s
      h_s[i] = (r < RB && k < H && b0 + r < B) ? h0[(size_t)(b0 + r) * H + k] : 0.f;
    }
  } else {
    for (int i = tid; i < 2 * RB * KP; i += blockDim.x) h_s[i] = 0.f;   // h_s and rh_s
  }

  auto prefetch_x = [&](int t) {               // owners: xp of step t -> x_s[t & 1]
    if (owner && t < T) {
      const int r = orow;
      if (b0 + r < B) {
#pragma unroll
        for (int g = 0; g < G; ++g)
          cp_async4(x_s + (((t & 1) * RB + r) * G + g) * CG + c, xg + ((size_t)t * B + b0 + r) * GH + g * H + c);
      }
    }
    cp_async_commit();
  };
  // mask: thread tid < RB pipelines it through two registers so the global load is issued two steps ahead
  int m1 = 0, m2 = 0;
  if (tid < RB) {
    const bool ok = b0 + tid < B;
    m_s[tid] = ok ? (mask[b0 + tid] != 0) : 0;
    m1 = (ok && 1 < T) ? (mask[(size_t)1 * B + b0 + tid] != 0) : 0;
    m2 = (ok && 2 < T) ? (mask[(size_t)2 * B + b0 + tid] != 0) : 0;
  }
  prefetch_x(0);
  __syncthreads();

  for (int t = 0; t < T; ++t) {
    const size_t tok0 = (size_t)t * B + b0;
    const float* xc = x_s + (t & 1) * RB * G * CG;
    prefetch_x(t + 1);                         // lands in the other buffer behind this step's matvecs
    // ---- phase 1: partial h.U over this thread's K-slice (all gates that see h_{t-1} share the loads)
    {
      float acc[G1][RB];
#pragma unroll
      for (int g = 0; g < G1; ++g)
#pragma unroll
        for (int r = 0; r < RB; ++r) acc[g][r] = 0.f;
      dot_slices<RB, KPT, G1, G>(acc, h_s, KP, s * KPT, u, 0);
#pragma unroll
      for (int g = 0; g < G1; ++g)
#pragma unroll
        for (int r = 0; r < RB; ++r) part_s[((s * RB + r) * G + g) * CG + c] = acc[g][r];
    }
    cp_async_wait<1>();                        // this step's xp (issued one step ago) has landed (own elements)
    __syncthreads();
    if constexpr (CELL == SEQREC_CELL_GRU) {
      if (owner) {
        const int r = orow;
        float az = xc[(r * G + 0) * CG + c], ar = xc[(r * G + 1) * CG + c];
#pragma unroll
        for (int q = 0; q < KS; ++q) {
          az += part_s[((q * RB + r) * G + 0) * CG + c];
          ar += part_s[((q * RB + r) * G + 1) * CG + c];
        }
        const float z = hard_sigmoid_f(az), rr = hard_sigmoid_f(ar);
        zr_s[(r * 2 + 0) * CG + c] = z;
        zr_s[(r * 2 + 1) * CG + c] = rr;
        rh_s[r * KP + c] = rr * h_s[r * KP + c];
      }
      __syncthreads();
      // ---- phase 2: candidate, (r*h).U_h
      float acc[1][RB];
#pragma unroll
      for (int r = 0; r < RB; ++r) acc[0][r] = 0.f;
      dot_slices<RB, KPT, 1, G>(acc, rh_s, KP, s * KPT, u, G - 1);
#pragma unroll
      for (int r = 0; r < RB; ++r) part_s[((s * RB + r) * G + 2) * CG + c] = acc[0][r];
      __syncthreads();
    }
    // ---- phase 3: gate math, state update under the mask, stores
    if (owner && b0 + orow < B) {
      const int r = orow;
      const size_t tok = tok0 + r;
      const bool m = m_s[(t & 1) * RB + r] != 0;
      const float hp = h_s[r * KP + c];
      float hn;
      float* gp = xg + tok * GH;
      if constexpr (CELL == SEQREC_CELL_GRU) {
        float ah = xc[(r * G + 2) * CG + c];
#pragma unroll
        for (int q = 0; q < KS; ++q) ah += part_s[((q * RB + r) * G + 2) * CG + c];
        const float hh = act_f<ACT>(ah);
        const float z = zr_s[(r * 2 + 0) * CG + c], rr = zr_s[(r * 2 + 1) * CG + c];
        hn = z * hp + (1.0f - z) * hh;
        gp[c] = z; gp[H + c] = rr; gp[2 * H + c] = hh;
      } else {
        float a = xc[(r * G + 0) * CG + c];
#pragma unroll
        for (int q = 0; q < KS; ++q) a += part_s[((q * RB + r) * G + 0) * CG + c];
        hn = act_f<ACT>(a);
        gp[c] = hn;
      }
      const float hv = m ? hn : hp;
      h_s[r * KP + c] = hv;
      hout[tok * H + c] = hv;
    }
    if (tid < RB) {
      m_s[((t + 1) & 1) * RB + tid] = m1;
      m1 = m2;
      m2 = (b0 + tid < B && t + 3 < T) ? (mask[(size_t)(t + 3) * B + b0 + tid] != 0) : 0;
    }
    __syncthreads();
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------------------------
// backward: thread (s, c) holds U[c][g*H + s*KPT + i] -- row c of U, K-slice s of every gate block.
template <int CELL, int ACT, int RB, int KPT>
__global__ void __launch_bounds__(KS * 128, 1)
rnn_backward_reg_kernel(float* __restrict__ xg, const float* __restrict__ U, const uint8_t* __restrict__ mask,
                        const float* __restrict__ hout, float* __restrict__ cst, const float* __restrict__ dhout,
                        int T, int B, int H) {
  constexpr int G = Gates<CELL>::G;
  constexpr int G1 = (CELL == SEQREC_CELL_GRU) ? 2 : 1;
  constexpr int NI = (CELL == SEQREC_CELL_GRU) ? 5 : 2;   // prefetched per-step inputs: dh, gates..., h_{t-1}
  constexpr int KP = KS * KPT;
  constexpr int CG = KP;                       // blockDim.x / KS: H rounded up to 32 == KS * KPT (dispatch_kpt)
  const int GH = G * H;
  extern __shared__ __align__(16) float smem[];
  float* da_s = smem;                          // [G][RB][KP]      pre-activation gradients of this step
  float* part_s = da_s + G * RB * KP;          // [KS][RB][CG]
  float* in_s = part_s + KS * RB * CG;         // [2][RB][NI][CG]  per-step inputs, double buffered (cp.async)
  float* dd_s = in_s + 2 * RB * NI * CG;       // [RB][CG]         direct part of dL/dh_{t-1}
  float* dc_s = dd_s + RB * CG;                // [RB][CG]         dL/dh_t carried from later steps
  int* m_s = reinterpret_cast<int*>(dc_s + RB * CG);   // [2][RB]
  const int tid = threadIdx.x;
  const int s = tid / CG, c = tid - s * CG;
  const int b0 = blockIdx.x * RB;
  const bool owner = (s < RB) && (c < H);      // thread (s, c), s < RB, owns batch row s of unit c (see the forward)
  const int orow = s;

  // U rows into registers through a per-warp 32 x 33 transpose tile: lane l reads element l of the K-slice of one row
  // (one 128-byte line per load), then picks its own row out of shared memory.  Reading U[c][...] directly is one line
  // per LANE -- 96 loads x 32 tags per warp, which ncu showed as 18 % of the kernel (stall_lg_throttle) at cfg2.
  float u[G][KPT];
  {
    float* tile = smem + (size_t)(tid >> 5) * (32 * 33);    // aliases da_s.. (initialised after the barrier below)
    const int lane = tid & 31, c0 = c - lane;              // CG is a multiple of 32: a warp has one s, 32 rows
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int j = s * KPT + lane;
#pragma unroll 8
      for (int rr = 0; rr < 32; ++rr)
        tile[rr * 33 + lane] = (lane < KPT && j < H && c0 + rr < H) ? U[(size_t)(c0 + rr) * GH + g * H + j] : 0.f;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < KPT; ++i) u[g][i] = tile[lane * 33 + i];
      __syncwarp();
    }
  }
  __syncthreads();
  for (int i = tid; i < G * RB * KP; i += blockDim.x) da_s[i] = 0.f;
  for (int i = tid; i < 2 * RB * CG; i += blockDim.x) dd_s[i] = 0.f;   // dd_s and dc_s

  // in_s[buf][r][0] = dL/dhout, [1..3] = saved gates z, r, hh (SimpleRNN: [1] = output y), [4] = h_{t-1}
  auto prefetch_in = [&](int t) {
    if (owner && t >= 0) {
      float* dst = in_s + (size_t)(t & 1) * RB * NI * CG;
      const int r = orow;
      if (b0 + r < B) {
        const size_t tok = (size_t)t * B + b0 + r;
        cp_async4(dst + (r * NI + 0) * CG + c, dhout + tok * H + c);
        if (CELL == SEQREC_CELL_GRU) {
#pragma unroll
          for (int g = 0; g < 3; ++g) cp_async4(dst + (r * NI + 1 + g) * CG + c, xg + tok * GH + g * H + c);
          if (t > 0) cp_async4(dst + (r * NI + 4) * CG + c, hout + (tok - B) * H + c);
        } else {
          cp_async4(dst + (r * NI + 1) * CG + c, hout + tok * H + c);
        }
      }
    }
    cp_async_commit();
  };
  int m1 = 0, m2 = 0;
  if (tid < RB) {
    const bool ok = b0 + tid < B;
    m_s[((T - 1) & 1) * RB + tid] = ok ? (mask[(size_t)(T - 1) * B + b0 + tid] != 0) : 0;
    m1 = (ok && T - 2 >= 0) ? (mask[(size_t)(T - 2) * B + b0 + tid] != 0) : 0;
    m2 = (ok && T - 3 >= 0) ? (mask[(size_t)(T - 3) * B + b0 + tid] != 0) : 0;
  }
  prefetch_in(T - 1);
  __syncthreads();

  for (int t = T - 1; t >= 0; --t) {
    const size_t tok0 = (size_t)t * B + b0;
    const float* ic = in_s + (size_t)(t & 1) * RB * NI * CG;
    prefetch_in(t - 1);
    cp_async_wait<1>();                        // this step's inputs (own elements) have landed
    // ---- phase 1 (owners): elementwise gate gradients
    if (owner && b0 + orow < B) {
      const int r = orow;
      const size_t tok = tok0 + r;
      const bool m = m_s[(t & 1) * RB + r] != 0;
      const float dh = ic[(r * NI + 0) * CG + c] + dc_s[r * CG + c];
      if (!m) {
        dd_s[r * CG + c] = dh;                 // masked step: h_t = h_{t-1}, no gate gradient
#pragma unroll
        for (int g = 0; g < G; ++g) da_s[(g * RB + r) * KP + c] = 0.f;
        if (CELL == SEQREC_CELL_GRU) cst[tok * H + c] = 0.f;
      } else if (CELL == SEQREC_CELL_GRU) {
        const float z = ic[(r * NI + 1) * CG + c], rg = ic[(r * NI + 2) * CG + c], hh = ic[(r * NI + 3) * CG + c];
        const float hprev = (t > 0) ? ic[(r * NI + 4) * CG + c] : 0.f;
        da_s[(0 * RB + r) * KP + c] = dh * (hprev - hh) * hard_sigmoid_grad_from_y(z);
        da_s[(2 * RB + r) * KP + c] = dh * (1.0f - z) * act_grad_from_y<ACT>(hh);
        dd_s[r * CG + c] = dh * z;
        cst[tok * H + c] = rg * hprev;         // operand of dU's candidate block
      } else {
        da_s[(0 * RB + r) * KP + c] = dh * act_grad_from_y<ACT>(ic[(r * NI + 1) * CG + c]);
        dd_s[r * CG + c] = 0.f;
      }
    }
    __syncthreads();
    if constexpr (CELL == SEQREC_CELL_GRU) {
      // ---- phase 2: d(r*h_{t-1})[c] = sum_j da_h[j] * U[c][2H + j]
      {
        float acc[1][RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) acc[0][r] = 0.f;
        dot_slices<RB, KPT, 1, G>(acc, da_s + 2 * RB * KP, KP, s * KPT, u, 2);
#pragma unroll
        for (int r = 0; r < RB; ++r) part_s[(s * RB + r) * CG + c] = acc[0][r];
      }
      __syncthreads();
      if (owner && b0 + orow < B && m_s[(t & 1) * RB + orow] != 0) {
        const int r = orow;
        float d_rh = 0.f;
#pragma unroll
        for (int q = 0; q < KS; ++q) d_rh += part_s[(q * RB + r) * CG + c];
        const float rg = ic[(r * NI + 2) * CG + c];
        const float hprev = (t > 0) ? ic[(r * NI + 4) * CG + c] : 0.f;
        da_s[(1 * RB + r) * KP + c] = d_rh * hprev * hard_sigmoid_grad_from_y(rg);
        dd_s[r * CG + c] += d_rh * rg;
      }
      __syncthreads();
    }
    // ---- phase 3: dh_{t-1}[c] = direct + sum_j da[j] * U[c][j] over the gates that see h_{t-1} directly
    {
      float acc[1][RB];
#pragma unroll
      for (int r = 0; r < RB; ++r) acc[0][r] = 0.f;
#pragma unroll
      for (int g = 0; g < G1; ++g) dot_slices<RB, KPT, 1, G>(acc, da_s + g * RB * KP, KP, s * KPT, u, g);
      // phase 2's partials were consumed before the barrier above, so part_s can be reused
#pragma unroll
      for (int r = 0; r < RB; ++r) part_s[(s * RB + r) * CG + c] = acc[0][r];
    }
    __syncthreads();
    if (owner && b0 + orow < B) {
      const int r = orow;
      float v = dd_s[r * CG + c];
#pragma unroll
      for (int q = 0; q < KS; ++q) v += part_s[(q * RB + r) * CG + c];
      dc_s[r * CG + c] = v;
      // dxp[t] = da (overwrites the saved gates, already copied to shared memory by the prefetch)
      float* gp = xg + (tok0 + r) * GH;
#pragma unroll
      for (int g = 0; g < G; ++g) gp[g * H + c] = da_s[(g * RB + r) * KP + c];
    }
    if (tid < RB) {
      m_s[((t - 1) & 1) * RB + tid] = m1;
      m1 = m2;
      m2 = (b0 + tid < B && t - 3 >= 0) ? (mask[(size_t)(t - 3) * B + b0 + tid] != 0) : 0;
    }
    __syncthreads();
  }
  cp_async_wait<0>();
}

template <int CELL, int ACT, int RB, int KPT>
int launch_pair(bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst, const float* dhout,
                int T, int B, int H, cudaStream_t st, const float* h0) {
  constexpr int G = Gates<CELL>::G;
  constexpr int NI = (CELL == SEQREC_CELL_GRU) ? 5 : 2;
  const int CG = (H + 31) / 32 * 32;
  const int threads = KS * CG;
  const int grid = ceil_div(B, RB);
  constexpr int KP = KS * KPT;
  if (fwd) {
    const size_t smem = sizeof(float) * (size_t)(2 * RB * KP + KS * RB * G * CG + 2 * RB * G * CG + RB * 2 * CG) +
                        sizeof(int) * 2 * RB;
    auto k = h0 ? rnn_forward_reg_kernel<CELL, ACT, RB, KPT, true> : rnn_forward_reg_kernel<CELL, ACT, RB, KPT, false>;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return -(int)e;
    }
    k<<<grid, threads, smem, st>>>(xg, U, mask, hout, T, B, H, h0);
  } else {
    const size_t smem_step = sizeof(float) * (size_t)(G * RB * KP + KS * RB * CG + 2 * RB * NI * CG + 2 * RB * CG) +
                             sizeof(int) * 2 * RB;
    const size_t smem_load = sizeof(float) * (size_t)(threads / 32) * 32 * 33;   // prologue transpose tiles
    const size_t smem = smem_step > smem_load ? smem_step : smem_load;
    auto k = rnn_backward_reg_kernel<CELL, ACT, RB, KPT>;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return -(int)e;
    }
    k<<<grid, threads, smem, st>>>(xg, U, mask, hout, cst, dhout, T, B, H);
  }
  SEQREC_CHECK_LAUNCH();
  return 0;
}

template <int CELL, int ACT, int RB>
int dispatch_kpt(bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                 const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0) {
  const int kpt = (((H + KS - 1) / KS) + 7) / 8 * 8;   // K-slice length, multiple of 8
  switch (kpt) {
    case 8: return launch_pair<CELL, ACT, RB, 8>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    case 16: return launch_pair<CELL, ACT, RB, 16>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    case 24: return launch_pair<CELL, ACT, RB, 24>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    default: return launch_pair<CELL, ACT, RB, 32>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
  }
}

template <int CELL, int ACT>
int dispatch_rb(int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0) {
  switch (rb) {
    case 1: return dispatch_kpt<CELL, ACT, 1>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    case 2: return dispatch_kpt<CELL, ACT, 2>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    default: return dispatch_kpt<CELL, ACT, 4>(fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
  }
}

template <int CELL>
int dispatch_act(int act, int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                 const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0) {
  switch (act) {
    case SEQREC_ACT_RELU:
      return dispatch_rb<CELL, SEQREC_ACT_RELU>(rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    case SEQREC_ACT_TANH:
      return dispatch_rb<CELL, SEQREC_ACT_TANH>(rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    case SEQREC_ACT_LINEAR:
      return dispatch_rb<CELL, SEQREC_ACT_LINEAR>(rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
    default: return -1002;
  }
}

}  // namespace

// LSTM variant (rnn_reg_lstm.cu)
bool lstm_reg_applicable(int H);
int lstm_reg_launch(int act, int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                    const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0, const float* c0);

// Is the register-resident scan applicable?  (GRU / SimpleRNN with H <= 128, LSTM with H <= 100)
bool rnn_reg_applicable(int cell, int H) {
  if (cell == SEQREC_CELL_LSTM) return lstm_reg_applicable(H);
  return (cell == SEQREC_CELL_GRU || cell == SEQREC_CELL_SIMPLE) && H <= 128;
}

// rb: batch rows per CTA (1, 2 or 4).  U is the untransposed recurrent kernel (H, G*H) for BOTH directions.
// h0 / c0 (forward only): initial state, NULL = zeros; c0 is read by the LSTM only.
int rnn_reg_launch(int cell, int act, int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout,
                   float* cst, const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0,
                   const float* c0) {
  if (cell == SEQREC_CELL_LSTM)
    return lstm_reg_launch(act, rb > 2 ? 2 : rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0, c0);
  if (cell == SEQREC_CELL_GRU)
    return dispatch_act<SEQREC_CELL_GRU>(act, rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
  return dispatch_act<SEQREC_CELL_SIMPLE>(act, rb, fwd, xg, U, mask, hout, cst, dhout, T, B, H, st, h0);
}
