// K3 / K4: masked recurrent scan, forward and backward, for SimpleRNN / LSTM / GRU with Keras-2.0.x semantics
// (model.py:345-352; Theano K.rnn mask switch: state held and previous output repeated on masked steps).
//
// One persistent CTA owns RB batch rows for ALL T timesteps, so there is no inter-CTA synchronisation on the
// sequential axis.  The recurrent kernel U (forward) / U^T (backward) is staged ONCE into shared memory when it fits
// (cfg2 GRU-128: 128x384 fp32 = 192 KB) and is then re-read from shared memory every step; larger cells stream it
// from L2.  Arithmetic is plain fp32 FFMA so the scan matches the fp32 reference to rounding; the per-step GEMM is
// (RB x H).(H x G*H), far too small and too latency-bound for the tensor pipe at the batch sizes of the named configs.
#include "common.cuh"

#define RNN_THREADS 512

// acc[r] += sum_{k in [k0,k1)} vec[r*ldv + k] * mat[k*ldm + col]      (vec in shared memory, mat shared or global)
template <int RB>
__device__ __forceinline__ void mv_accum(float (&acc)[RB], const float* __restrict__ vec, int ldv,
                                         const float* __restrict__ mat, int ldm, int col, int k0, int k1) {
  int k = k0;
  // ldv is a multiple of 4 at every call site; peel until k is too, so the float4 loads of vec are aligned
  for (; k < k1 && (k & 3); ++k) {
    const float u = mat[(size_t)k * ldm + col];
#pragma unroll
    for (int r = 0; r < RB; ++r) acc[r] = fmaf(vec[r * ldv + k], u, acc[r]);
  }
  for (; k + 4 <= k1; k += 4) {
    const float u0 = mat[(size_t)(k + 0) * ldm + col];
    const float u1 = mat[(size_t)(k + 1) * ldm + col];
    const float u2 = mat[(size_t)(k + 2) * ldm + col];
    const float u3 = mat[(size_t)(k + 3) * ldm + col];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const float4 h = *reinterpret_cast<const float4*>(vec + r * ldv + k);
      acc[r] = fmaf(h.x, u0, acc[r]);
      acc[r] = fmaf(h.y, u1, acc[r]);
      acc[r] = fmaf(h.z, u2, acc[r]);
      acc[r] = fmaf(h.w, u3, acc[r]);
    }
  }
  for (; k < k1; ++k) {
    const float u = mat[(size_t)k * ldm + col];
#pragma unroll
    for (int r = 0; r < RB; ++r) acc[r] = fmaf(vec[r * ldv + k], u, acc[r]);
  }
}

__host__ __device__ inline int round_up4(int x) { return (x + 3) & ~3; }

// ---------------------------------------------------------------------------------------------------------------
// forward
// RD = recurrent dropout (Keras `recurrent_dropout`, model.py:346,351): G inverted-dropout masks rm[g] (B,H), constant
// over time, multiply h_{t-1} before the recurrent product of gate block g (GRU candidate: r * h_{t-1} * rm[2]).  The
// masked copies hm[g] = h * rm[g] are kept in shared memory next to h.
// INIT: the scan starts from h0 (B,H) and, for LSTM, c0 (B,H) instead of zeros; a NULL pointer stands for zeros.
template <int CELL, int ACT, int RB, bool USMEM, bool RD, bool INIT>
__global__ void __launch_bounds__(RNN_THREADS, 1)
rnn_forward_kernel(float* __restrict__ xg, const float* __restrict__ U, const uint8_t* __restrict__ mask,
                   float* __restrict__ hout, float* __restrict__ cst, int T, int B, int H,
                   const float* __restrict__ rm, const float* __restrict__ h0, const float* __restrict__ c0) {
  static_assert(!(RD && INIT), "recurrent dropout is training only; the carried state is inference only");
  constexpr int G = (CELL == SEQREC_CELL_LSTM) ? 4 : (CELL == SEQREC_CELL_GRU ? 3 : 1);
  const int GH = G * H;
  const int Hp = round_up4(H);
  const int GHp = round_up4(GH);
  extern __shared__ __align__(16) float smem[];
  float* h_s = smem;                 // [RB][Hp]   current hidden state
  float* c_s = h_s + RB * Hp;        // [RB][Hp]   LSTM cell state / GRU r*h
  float* a_s = c_s + RB * Hp;        // [RB][GHp]  pre-activations (GRU: z,r post-activation after phase 1b)
  float* hm_s = a_s + RB * GHp;      // [G][RB][Hp] h * rm[g] (RD only)
  float* U_s = hm_s + (RD ? G * RB * Hp : 0);   // [H][GH]    (USMEM only)
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * RB;

  if constexpr (INIT) {
    // padding columns u >= H and rows past B stay zero; GRU's c_s (r*h) is recomputed every step
    for (int i = tid; i < RB * Hp; i += RNN_THREADS) {
      const int r = i / Hp, u = i - r * Hp;
      const bool ok = b0 + r < B && u < H;
      const size_t e = (size_t)(b0 + r) * H + u;
      h_s[i] = (ok && h0) ? h0[e] : 0.f;
      c_s[i] = (ok && c0 && CELL == SEQREC_CELL_LSTM) ? c0[e] : 0.f;
    }
  } else {
    for (int i = tid; i < RB * Hp; i += RNN_THREADS) { h_s[i] = 0.f; c_s[i] = 0.f; }
  }
  if (RD) {
    for (int i = tid; i < G * RB * Hp; i += RNN_THREADS) hm_s[i] = 0.f;
  }
  if (USMEM) {
    for (int i = tid; i < H * GH; i += RNN_THREADS) U_s[i] = U[i];
  }
  __syncthreads();
  const int J1 = (CELL == SEQREC_CELL_GRU) ? 2 * H : GH;

  for (int t = 0; t < T; ++t) {
    const size_t tok0 = (size_t)t * B + b0;
    // ---- phase 1: a = xp + h.U (GRU: z and r blocks only)
    for (int j = tid; j < J1; j += RNN_THREADS) {
      float acc[RB];
#pragma unroll
      for (int r = 0; r < RB; ++r) acc[r] = (b0 + r < B) ? xg[(tok0 + r) * GH + j] : 0.f;
      const float* hv_s = RD ? hm_s + (j / H) * RB * Hp : h_s;   // gate block of column j
      if (USMEM) mv_accum<RB>(acc, hv_s, Hp, U_s, GH, j, 0, H);
      else       mv_accum<RB>(acc, hv_s, Hp, U, GH, j, 0, H);
#pragma unroll
      for (int r = 0; r < RB; ++r) a_s[r * GHp + j] = acc[r];
    }
    __syncthreads();
    if (CELL == SEQREC_CELL_GRU) {
      // ---- phase 1b: z, r; r*h_{t-1} feeds the candidate's recurrent product (reset BEFORE the matmul)
      for (int i = tid; i < RB * H; i += RNN_THREADS) {
        const int r = i / H, u = i - r * H;
        const float z = hard_sigmoid_f(a_s[r * GHp + u]);
        const float rr = hard_sigmoid_f(a_s[r * GHp + H + u]);
        a_s[r * GHp + u] = z;
        a_s[r * GHp + H + u] = rr;
        c_s[r * Hp + u] = rr * (RD ? hm_s[(2 * RB + r) * Hp + u] : h_s[r * Hp + u]);
      }
      __syncthreads();
      // ---- phase 2: candidate pre-activation
      for (int j = tid; j < H; j += RNN_THREADS) {
        float acc[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) acc[r] = (b0 + r < B) ? xg[(tok0 + r) * GH + 2 * H + j] : 0.f;
        if (USMEM) mv_accum<RB>(acc, c_s, Hp, U_s, GH, 2 * H + j, 0, H);
        else       mv_accum<RB>(acc, c_s, Hp, U, GH, 2 * H + j, 0, H);
#pragma unroll
        for (int r = 0; r < RB; ++r) a_s[r * GHp + 2 * H + j] = acc[r];
      }
      __syncthreads();
    }
    // ---- phase 3: gates, state update under the mask, stores
    for (int i = tid; i < RB * H; i += RNN_THREADS) {
      const int r = i / H, u = i - r * H;
      if (b0 + r >= B) continue;
      const size_t tok = tok0 + r;
      const bool m = mask[tok] != 0;
      const float hp = h_s[r * Hp + u];
      float hn;
      if (CELL == SEQREC_CELL_LSTM) {
        const float ig = hard_sigmoid_f(a_s[r * GHp + u]);
        const float fg = hard_sigmoid_f(a_s[r * GHp + H + u]);
        const float gg = act_f<ACT>(a_s[r * GHp + 2 * H + u]);
        const float og = hard_sigmoid_f(a_s[r * GHp + 3 * H + u]);
        const float cp = c_s[r * Hp + u];
        const float cn = fmaf(fg, cp, ig * gg);
        hn = og * act_f<ACT>(cn);
        const float cv = m ? cn : cp;
        c_s[r * Hp + u] = cv;
        cst[tok * H + u] = cv;
        float* gp = xg + tok * GH;
        gp[u] = ig; gp[H + u] = fg; gp[2 * H + u] = gg; gp[3 * H + u] = og;
      } else if (CELL == SEQREC_CELL_GRU) {
        const float z = a_s[r * GHp + u];
        const float rr = a_s[r * GHp + H + u];
        const float hh = act_f<ACT>(a_s[r * GHp + 2 * H + u]);
        hn = z * hp + (1.0f - z) * hh;
        float* gp = xg + tok * GH;
        gp[u] = z; gp[H + u] = rr; gp[2 * H + u] = hh;
      } else {
        hn = act_f<ACT>(a_s[r * GHp + u]);
        xg[tok * GH + u] = hn;
      }
      const float hv = m ? hn : hp;
      h_s[r * Hp + u] = hv;
      hout[tok * H + u] = hv;
      if (RD) {
#pragma unroll
        for (int g = 0; g < G; ++g) hm_s[(g * RB + r) * Hp + u] = hv * rm[((size_t)g * B + b0 + r) * H + u];
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// backward.  Walks t = T-1 .. 0 carrying dh (and dc).  xg holds the saved post-activation gates on entry and the
// pre-activation gradients dxp on exit.  Ut = U^T (G*H, H).
template <int CELL, int ACT, int RB, bool USMEM, bool RD>
__global__ void __launch_bounds__(RNN_THREADS, 1)
rnn_backward_kernel(float* __restrict__ xg, const float* __restrict__ Ut, const uint8_t* __restrict__ mask,
                    const float* __restrict__ hout, float* __restrict__ cst, const float* __restrict__ dhout,
                    int T, int B, int H, const float* __restrict__ rm) {
  constexpr int G = (CELL == SEQREC_CELL_LSTM) ? 4 : (CELL == SEQREC_CELL_GRU ? 3 : 1);
  const int GH = G * H;
  const int Hp = round_up4(H);
  const int GHp = round_up4(GH);
  extern __shared__ __align__(16) float smem[];
  float* dh_s = smem;                 // [RB][Hp]  dL/dh_t carried from later steps
  float* dc_s = dh_s + RB * Hp;       // [RB][Hp]  LSTM: dL/dc_t carried;  GRU: reset gate r_t
  float* dd_s = dc_s + RB * Hp;       // [RB][Hp]  direct (non-matmul) part of dL/dh_{t-1}
  float* hp_s = dd_s + RB * Hp;       // [RB][Hp]  GRU: h_{t-1}
  float* da_s = hp_s + RB * Hp;       // [RB][GHp] pre-activation gradients of this step
  float* Ut_s = da_s + RB * GHp;      // [GH][H]   (USMEM only)
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * RB;

  for (int i = tid; i < RB * Hp; i += RNN_THREADS) { dh_s[i] = 0.f; dc_s[i] = 0.f; dd_s[i] = 0.f; hp_s[i] = 0.f; }
  for (int i = tid; i < RB * GHp; i += RNN_THREADS) da_s[i] = 0.f;
  if (USMEM) {
    for (int i = tid; i < H * GH; i += RNN_THREADS) Ut_s[i] = Ut[i];
  }
  __syncthreads();

  for (int t = T - 1; t >= 0; --t) {
    const size_t tok0 = (size_t)t * B + b0;
    // ---- phase 1: elementwise gate gradients
    for (int i = tid; i < RB * H; i += RNN_THREADS) {
      const int r = i / H, u = i - r * H;
      if (b0 + r >= B) continue;
      const size_t tok = tok0 + r;
      const bool m = mask[tok] != 0;
      const float dh = dhout[tok * H + u] + dh_s[r * Hp + u];
      float* da = da_s + r * GHp;
      if (!m) {
        // masked step: h_t = h_{t-1}, c_t = c_{t-1}; the candidate is discarded, so no gate gradient
        dd_s[r * Hp + u] = dh;
#pragma unroll
        for (int g = 0; g < G; ++g) da[g * H + u] = 0.f;
        if (CELL == SEQREC_CELL_GRU) { dc_s[r * Hp + u] = 0.f; hp_s[r * Hp + u] = 0.f; cst[tok * H + u] = 0.f; }
        continue;
      }
      const float* gp = xg + tok * GH;
      if (CELL == SEQREC_CELL_LSTM) {
        const float ig = gp[u], fg = gp[H + u], gg = gp[2 * H + u], og = gp[3 * H + u];
        const float ct = cst[tok * H + u];
        const float cp = (t > 0) ? cst[(tok - B) * H + u] : 0.f;
        const float ac = act_f<ACT>(ct);
        const float d_o = dh * ac;
        const float dc = dc_s[r * Hp + u] + dh * og * act_grad_from_y<ACT>(ac);
        da[u] = dc * gg * hard_sigmoid_grad_from_y(ig);
        da[H + u] = dc * cp * hard_sigmoid_grad_from_y(fg);
        da[2 * H + u] = dc * ig * act_grad_from_y<ACT>(gg);
        da[3 * H + u] = d_o * hard_sigmoid_grad_from_y(og);
        dc_s[r * Hp + u] = dc * fg;
        dd_s[r * Hp + u] = 0.f;
      } else if (CELL == SEQREC_CELL_GRU) {
        const float z = gp[u], rr = gp[H + u], hh = gp[2 * H + u];
        const float hp = (t > 0) ? hout[(tok - B) * H + u] : 0.f;
        const float dz = dh * (hp - hh);
        const float dhh = dh * (1.0f - z);
        da[u] = dz * hard_sigmoid_grad_from_y(z);
        da[2 * H + u] = dhh * act_grad_from_y<ACT>(hh);
        dd_s[r * Hp + u] = dh * z;
        dc_s[r * Hp + u] = rr;
        hp_s[r * Hp + u] = hp;
        // operand of dU's candidate block (with recurrent dropout: r * h_{t-1} * rm[2])
        cst[tok * H + u] = rr * hp * (RD ? rm[((size_t)2 * B + b0 + r) * H + u] : 1.0f);
      } else {
        const float y = hout[tok * H + u];
        da[u] = dh * act_grad_from_y<ACT>(y);
        dd_s[r * Hp + u] = 0.f;
      }
    }
    __syncthreads();
    if (CELL == SEQREC_CELL_GRU) {
      // ---- phase 2: d(r*h_{t-1}) = da_h . U_h^T ; then dr, and the r-path into dh_{t-1}
      for (int k = tid; k < H; k += RNN_THREADS) {
        float acc[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) acc[r] = 0.f;
        if (USMEM) mv_accum<RB>(acc, da_s, GHp, Ut_s, H, k, 2 * H, 3 * H);
        else       mv_accum<RB>(acc, da_s, GHp, Ut, H, k, 2 * H, 3 * H);
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const float rr = dc_s[r * Hp + k];
          const float hp = hp_s[r * Hp + k];
          if (RD) acc[r] *= (b0 + r < B) ? rm[((size_t)2 * B + b0 + r) * H + k] : 0.f;   // d(r*h) from d(r*h*rm)
          da_s[r * GHp + H + k] = acc[r] * hp * hard_sigmoid_grad_from_y(rr);
          dd_s[r * Hp + k] += acc[r] * rr;
        }
      }
      __syncthreads();
    }
    // ---- phase 3: dh_{t-1} = direct + da . U^T (GRU: z and r blocks; the candidate block went through phase 2)
    const int J = (CELL == SEQREC_CELL_GRU) ? 2 * H : GH;
    for (int k = tid; k < H; k += RNN_THREADS) {
      float acc[RB];
#pragma unroll
      for (int r = 0; r < RB; ++r) acc[r] = dd_s[r * Hp + k];
      if (!RD) {
        if (USMEM) mv_accum<RB>(acc, da_s, GHp, Ut_s, H, k, 0, J);
        else       mv_accum<RB>(acc, da_s, GHp, Ut, H, k, 0, J);
      } else {
        // dL/dh_{t-1} += rm[g] * (da_g . U_g^T), one gate block at a time
        for (int g = 0; g < J / H; ++g) {
          float part[RB];
#pragma unroll
          for (int r = 0; r < RB; ++r) part[r] = 0.f;
          if (USMEM) mv_accum<RB>(part, da_s, GHp, Ut_s, H, k, g * H, (g + 1) * H);
          else       mv_accum<RB>(part, da_s, GHp, Ut, H, k, g * H, (g + 1) * H);
#pragma unroll
          for (int r = 0; r < RB; ++r)
            if (b0 + r < B) acc[r] = fmaf(part[r], rm[((size_t)g * B + b0 + r) * H + k], acc[r]);
        }
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) dh_s[r * Hp + k] = acc[r];
    }
    // dxp[t] = da (overwrites the saved gates, which phase 1 has already consumed)
    for (int i = tid; i < RB * GH; i += RNN_THREADS) {
      const int r = i / GH, j = i - r * GH;
      if (b0 + r < B) xg[(tok0 + r) * GH + j] = da_s[r * GHp + j];
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// launch plumbing
static int pick_rb(int B) {
  if (B <= SEQREC_NUM_SMS) return 1;
  if (B <= 2 * SEQREC_NUM_SMS) return 2;
  if (B <= 4 * SEQREC_NUM_SMS) return 4;
  return 8;
}

static const size_t kMaxDynSmem = 227 * 1024;

template <int CELL, int ACT, int RB, bool RD, bool INIT>
static int launch_fwd_rd(float* xg, const float* U, const uint8_t* mask, float* hout, float* cst, int T, int B, int H,
                         const float* rm, const float* h0, const float* c0, cudaStream_t st) {
  constexpr int G = (CELL == SEQREC_CELL_LSTM) ? 4 : (CELL == SEQREC_CELL_GRU ? 3 : 1);
  const int GH = G * H, Hp = round_up4(H), GHp = round_up4(GH);
  const size_t base = sizeof(float) * (size_t)(2 * RB * Hp + RB * GHp + (RD ? G * RB * Hp : 0));
  const size_t with_u = base + sizeof(float) * (size_t)H * GH;
  const int grid = ceil_div(B, RB);
  if (with_u <= kMaxDynSmem) {
    auto k = rnn_forward_kernel<CELL, ACT, RB, true, RD, INIT>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)with_u);
    if (e != cudaSuccess) return -(int)e;
    k<<<grid, RNN_THREADS, with_u, st>>>(xg, U, mask, hout, cst, T, B, H, rm, h0, c0);
  } else {
    auto k = rnn_forward_kernel<CELL, ACT, RB, false, RD, INIT>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)base);
    if (e != cudaSuccess) return -(int)e;
    k<<<grid, RNN_THREADS, base, st>>>(xg, U, mask, hout, cst, T, B, H, rm, h0, c0);
  }
  SEQREC_CHECK_LAUNCH();
  return 0;
}
template <int CELL, int ACT, int RB>
static int launch_fwd(float* xg, const float* U, const uint8_t* mask, float* hout, float* cst, int T, int B, int H,
                      const float* rm, const float* h0, const float* c0, cudaStream_t st) {
  if (h0 || c0) return launch_fwd_rd<CELL, ACT, RB, false, true>(xg, U, mask, hout, cst, T, B, H, nullptr, h0, c0, st);
  if (rm) return launch_fwd_rd<CELL, ACT, RB, true, false>(xg, U, mask, hout, cst, T, B, H, rm, nullptr, nullptr, st);
  return launch_fwd_rd<CELL, ACT, RB, false, false>(xg, U, mask, hout, cst, T, B, H, nullptr, nullptr, nullptr, st);
}

template <int CELL, int ACT, int RB, bool RD>
static int launch_bwd_rd(float* xg, const float* Ut, const uint8_t* mask, const float* hout, float* cst,
                         const float* dhout, int T, int B, int H, const float* rm, cudaStream_t st) {
  constexpr int G = (CELL == SEQREC_CELL_LSTM) ? 4 : (CELL == SEQREC_CELL_GRU ? 3 : 1);
  const int GH = G * H, Hp = round_up4(H), GHp = round_up4(GH);
  const size_t base = sizeof(float) * (size_t)(4 * RB * Hp + RB * GHp);
  const size_t with_u = base + sizeof(float) * (size_t)H * GH;
  const int grid = ceil_div(B, RB);
  if (with_u <= kMaxDynSmem) {
    auto k = rnn_backward_kernel<CELL, ACT, RB, true, RD>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)with_u);
    if (e != cudaSuccess) return -(int)e;
    k<<<grid, RNN_THREADS, with_u, st>>>(xg, Ut, mask, hout, cst, dhout, T, B, H, rm);
  } else {
    auto k = rnn_backward_kernel<CELL, ACT, RB, false, RD>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)base);
    if (e != cudaSuccess) return -(int)e;
    k<<<grid, RNN_THREADS, base, st>>>(xg, Ut, mask, hout, cst, dhout, T, B, H, rm);
  }
  SEQREC_CHECK_LAUNCH();
  return 0;
}
template <int CELL, int ACT, int RB>
static int launch_bwd(float* xg, const float* Ut, const uint8_t* mask, const float* hout, float* cst,
                      const float* dhout, int T, int B, int H, const float* rm, cudaStream_t st) {
  return rm ? launch_bwd_rd<CELL, ACT, RB, true>(xg, Ut, mask, hout, cst, dhout, T, B, H, rm, st)
            : launch_bwd_rd<CELL, ACT, RB, false>(xg, Ut, mask, hout, cst, dhout, T, B, H, nullptr, st);
}

#define DISPATCH_RB(FN, CELL, ACT, ...)                                   \
  switch (rb) {                                                           \
    case 1: return FN<CELL, ACT, 1>(__VA_ARGS__);                         \
    case 2: return FN<CELL, ACT, 2>(__VA_ARGS__);                         \
    case 4: return FN<CELL, ACT, 4>(__VA_ARGS__);                         \
    default: return FN<CELL, ACT, 8>(__VA_ARGS__);                        \
  }

#define DISPATCH_ACT(FN, CELL, ...)                                                         \
  switch (act) {                                                                            \
    case SEQREC_ACT_RELU: DISPATCH_RB(FN, CELL, SEQREC_ACT_RELU, __VA_ARGS__)               \
    case SEQREC_ACT_TANH: DISPATCH_RB(FN, CELL, SEQREC_ACT_TANH, __VA_ARGS__)               \
    case SEQREC_ACT_LINEAR: DISPATCH_RB(FN, CELL, SEQREC_ACT_LINEAR, __VA_ARGS__)           \
    default: return -1002;                                                                  \
  }

// register-resident fast path (rnn_reg.cu)
bool rnn_reg_applicable(int cell, int H);
int rnn_reg_launch(int cell, int act, int rb, bool fwd, float* xg, const float* U, const uint8_t* mask, float* hout,
                   float* cst, const float* dhout, int T, int B, int H, cudaStream_t st, const float* h0 = nullptr,
                   const float* c0 = nullptr);

// rows per CTA of the register-resident scan: 96 of the 128 registers hold U when H > 96, leaving room for 2 rows
static int reg_rb(int rb, int H) { return H > 96 ? (rb > 2 ? 2 : rb) : (rb > 4 ? 4 : rb); }

extern "C" int seqrec_rnn_needs_ut(int cell, int H) { return rnn_reg_applicable(cell, H) ? 0 : 1; }

// h0 / c0: initial state (NULL = zeros; never together with rm)
static int rnn_forward_any(int cell, int act, float* xg, const float* U, const uint8_t* mask, float* hout, float* cst,
                           int T, int B, int H, const float* rm, cudaStream_t st, const float* h0 = nullptr,
                           const float* c0 = nullptr) {
  const int rb = pick_rb(B);
  if (!rm && rnn_reg_applicable(cell, H))
    return rnn_reg_launch(cell, act, reg_rb(rb, H), true, xg, U, mask, hout, cst, nullptr, T, B, H, st, h0, c0);
  switch (cell) {
    case SEQREC_CELL_SIMPLE:
      DISPATCH_ACT(launch_fwd, SEQREC_CELL_SIMPLE, xg, U, mask, hout, cst, T, B, H, rm, h0, c0, st)
    case SEQREC_CELL_LSTM: DISPATCH_ACT(launch_fwd, SEQREC_CELL_LSTM, xg, U, mask, hout, cst, T, B, H, rm, h0, c0, st)
    case SEQREC_CELL_GRU: DISPATCH_ACT(launch_fwd, SEQREC_CELL_GRU, xg, U, mask, hout, cst, T, B, H, rm, h0, c0, st)
    default: return -1003;
  }
}

static int rnn_backward_any(int cell, int act, float* xg, const float* U, const float* Ut, const uint8_t* mask,
                            const float* hout, float* cst, const float* dhout, int T, int B, int H, const float* rm,
                            cudaStream_t st) {
  const int rb = pick_rb(B);
  if (!rm && rnn_reg_applicable(cell, H)) {
    SEQREC_ARG(U != nullptr, 2);
    return rnn_reg_launch(cell, act, reg_rb(rb, H), false, xg, U, mask, const_cast<float*>(hout), cst, dhout, T, B,
                          H, st);
  }
  SEQREC_ARG(Ut != nullptr, 3);
  switch (cell) {
    case SEQREC_CELL_SIMPLE:
      DISPATCH_ACT(launch_bwd, SEQREC_CELL_SIMPLE, xg, Ut, mask, hout, cst, dhout, T, B, H, rm, st)
    case SEQREC_CELL_LSTM:
      DISPATCH_ACT(launch_bwd, SEQREC_CELL_LSTM, xg, Ut, mask, hout, cst, dhout, T, B, H, rm, st)
    case SEQREC_CELL_GRU: DISPATCH_ACT(launch_bwd, SEQREC_CELL_GRU, xg, Ut, mask, hout, cst, dhout, T, B, H, rm, st)
    default: return -1003;
  }
}

extern "C" int seqrec_rnn_forward(int cell, int act, float* xg, const float* U, const uint8_t* mask, float* hout,
                                  float* cst, int T, int B, int H, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && H > 0, 1);
  return rnn_forward_any(cell, act, xg, U, mask, hout, cst, T, B, H, nullptr, as_stream(stream));
}

extern "C" int seqrec_rnn_forward_state(int cell, int act, float* xg, const float* U, const float* h0,
                                        const float* c0, const uint8_t* mask, float* hout, float* cst, int T, int B,
                                        int H, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && H > 0, 1);
  SEQREC_ARG(c0 == nullptr || cell == SEQREC_CELL_LSTM, 2);
  return rnn_forward_any(cell, act, xg, U, mask, hout, cst, T, B, H, nullptr, as_stream(stream), h0, c0);
}

extern "C" int seqrec_rnn_backward(int cell, int act, float* xg, const float* U, const float* Ut,
                                   const uint8_t* mask, const float* hout, float* cst, const float* dhout, int T,
                                   int B, int H, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && H > 0, 1);
  return rnn_backward_any(cell, act, xg, U, Ut, mask, hout, cst, dhout, T, B, H, nullptr, as_stream(stream));
}

// Keras `recurrent_dropout` (model.py:346, :351; swept by tune_params.py:83, tune_params_msnbc.py:54,77): rec_mask
// (G, B, H) holds one inverted-dropout mask per gate block, constant over time.  Always the generic fp32 scan: the
// tensor-core and register-resident scans share ONE h operand between the gate blocks.
extern "C" int seqrec_rnn_forward_rd(int cell, int act, float* xg, const float* U, const float* rec_mask,
                                     const uint8_t* mask, float* hout, float* cst, int T, int B, int H, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && H > 0 && rec_mask != nullptr, 1);
  return rnn_forward_any(cell, act, xg, U, mask, hout, cst, T, B, H, rec_mask, as_stream(stream));
}

extern "C" int seqrec_rnn_backward_rd(int cell, int act, float* xg, const float* Ut, const float* rec_mask,
                                      const uint8_t* mask, const float* hout, float* cst, const float* dhout, int T,
                                      int B, int H, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && H > 0 && rec_mask != nullptr, 1);
  return rnn_backward_any(cell, act, xg, nullptr, Ut, mask, hout, cst, dhout, T, B, H, rec_mask, as_stream(stream));
}
