// K3 on the 5th-generation tensor cores: the masked LSTM / GRU scan (forward) for H = 128 / 256 as ONE persistent
// thread-block-cluster kernel that keeps the recurrent kernel on chip for all T timesteps.
// Reference constructs replaced: keras.layers.LSTM / GRU(return_sequences=True) under Theano's K.rnn with a mask
// (model.py:345-352); same semantics, inputs and outputs as rnn_scan.cu (the fp32 SIMT scan).
//
// Decomposition (sm_100a):
//   * a cluster of CS = H/32 CTAs owns 64 batch rows for the whole sequence; CTA c owns hidden units [32c, 32c+32):
//     its slice of U (all gate columns of those units: 256 x 128 for LSTM-256) is loaded ONCE by TMA as a bf16 hi/lo
//     K-major operand (128 KB) and stays in shared memory for all T steps
//   * per step the CTA computes  acc[64 rows, gate cols] = h_{t-1}[64, H] . U_slice  with tcgen05.mma (M = 64, fp32
//     accumulate in TMEM, 3-pass hi/lo split = fp32-grade products), two M=64 atoms interleaved on the two
//     half-subpartitions of TMEM so that all 128 epilogue threads own one batch row x 16 hidden units with every gate
//     of those units in their own TMEM columns -> the gate math needs no shuffles
//   * the new h slice (bf16 hi/lo, already in the 64-byte-swizzled K-major operand layout) is ALL-GATHERED through
//     distributed shared memory: staged once in the CTA's own shared memory, then pushed to every CTA of the cluster
//     with cp.async.bulk (shared::cta -> shared::cluster) that completes on the receiver's mbarrier -- the operand
//     of the next step's MMA is assembled by the copy engines, no thread touches it
//   * the Keras-2.0.x GRU applies the reset gate BEFORE the recurrent matmul, so a GRU step is two such rounds
//     (z,r from h; candidate from r*h), an LSTM step is one
// Flow control per round r: bar_acc (MMA done, tcgen05.commit) -> epilogue; bar_free (every CTA's MMA of round r has
// finished reading its h operand; remote mbarrier arrives) -> the exchange warp may overwrite the peers' operand;
// bar_hfull (all CS slices landed, complete_tx) -> next MMA.  Every wait is bounded (traps instead of hanging).
#include "common.cuh"
#include "ptx_sm100.cuh"
#include "tma_host.cuh"

namespace {

constexpr int BMR = 64;          // batch rows per cluster (UMMA M)
constexpr int UPC = 32;          // hidden units per CTA
constexpr int RT_THREADS = 192;  // warps 0-3 epilogue (TMEM lane quadrants), warp 4 TMA + MMA, warp 5 exchange
constexpr float RT_LOG2E = 1.4426950408889634f;

// optional timeline capture (scripts/time_rnn.py): CTA 0 stores clock64() at the protocol points of the first rounds
long long* g_rnn_tc_dbg = nullptr;
#define RT_DBG(round, slot)                                                                   \
  do {                                                                                        \
    if (dbg && blockIdx.x == 0 && (round) < 64) dbg[(round) * 8 + (slot)] = clock64();        \
  } while (0)

// the activation stays the exact tanhf / relu of the fp32 scans: an ex2.approx-based tanh (absolute error ~2e-7) was
// measured to cost nothing less on the sequential path and its error is amplified by Adagrad's sign-like first updates
// (smoke(): post-update W_out error 2.2e-4 instead of 3.7e-5)
template <int ACT>
__device__ __forceinline__ float act_fast(float a) {
  return act_f<ACT>(a);
}

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void st_shared_u4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// this thread's 16 values (one batch row, 16 consecutive hidden units) -> bf16 hi / lo into the staging image of the
// CTA's K block: rows of 64 B (32 units), 16-byte chunks XOR-swizzled with (row >> 1) & 3 (SWIZZLE_64B)
__device__ __forceinline__ void stage_slice(uint32_t stage_hi, uint32_t stage_lo, int row, int hh, const float (&v)[16]) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float x0 = v[2 * i], x1 = v[2 * i + 1];
    const __nv_bfloat162 hv = __floats2bfloat162_rn(x0, x1);
    hi[i] = *reinterpret_cast<const uint32_t*>(&hv);
    const __nv_bfloat162 lv = __floats2bfloat162_rn(x0 - __low2float(hv), x1 - __high2float(hv));
    lo[i] = *reinterpret_cast<const uint32_t*>(&lv);
  }
  const uint32_t sw = (uint32_t)((row & 7) >> 1);
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const uint32_t off = (uint32_t)row * 64u + ((((uint32_t)(2 * hh + c)) ^ sw) << 4);
    st_shared_u4(stage_hi + off, hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
    st_shared_u4(stage_lo + off, lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
  }
}

__device__ __forceinline__ void load16(float* dst, const float* __restrict__ src, bool ok) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 v = ok ? __ldg(reinterpret_cast<const float4*>(src) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    dst[4 * i] = v.x; dst[4 * i + 1] = v.y; dst[4 * i + 2] = v.z; dst[4 * i + 3] = v.w;
  }
}
__device__ __forceinline__ void store16(float* dst, const float* src) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
    reinterpret_cast<float4*>(dst)[i] = make_float4(src[4 * i], src[4 * i + 1], src[4 * i + 2], src[4 * i + 3]);
}

template <int CELL, int CS>
struct FwdCfg {
  static constexpr int H = CS * UPC;
  static constexpr int G = (CELL == SEQREC_CELL_LSTM) ? 4 : 3;
  static constexpr int RPS = (CELL == SEQREC_CELL_LSTM) ? 1 : 2;       // exchange rounds per timestep
  static constexpr int KB = H / 64;                                    // 64-wide K blocks of the U operand
  static constexpr int GA = (CELL == SEQREC_CELL_LSTM) ? 4 : 2;        // gates of region A (LSTM i,f,c,o | GRU z,r)
  static constexpr int NA = GA * UPC;                                  // rows per K block, region A
  static constexpr int NB = (CELL == SEQREC_CELL_LSTM) ? 0 : UPC;      // region B: GRU candidate
  static constexpr uint32_t UA_BYTES = KB * NA * 128, UB_BYTES = KB * NB * 128;
  static constexpr uint32_t U_PART = UA_BYTES + UB_BYTES;              // one part (hi or lo) of the U slice
  static constexpr uint32_t H_PART = CS * 4096;                        // one part of the h operand: CS K blocks
  static constexpr uint32_t STG = 4096;                                // one part of one staged slice
  static constexpr uint32_t SMEM = 2 * U_PART + 2 * H_PART + 4 * STG + 128 + 1024;
};

// INIT: the scan starts from h0 (B,H) and, for LSTM, c0 (B,H) instead of zeros (a NULL pointer stands for zeros).
// Every CTA builds the whole h_{-1} operand from h0 with the split and swizzle of stage_slice, so a scan continued
// from hout[T-1] (and cst[T-1]) computes bit for bit what one longer scan computes.
template <int CELL, int ACT, int CS, bool INIT>
__global__ void __launch_bounds__(RT_THREADS, 1)
rnn_tc_forward_kernel(const __grid_constant__ CUtensorMap tmU_hi, const __grid_constant__ CUtensorMap tmU_lo,
                      float* __restrict__ xg, const uint8_t* __restrict__ mask, float* __restrict__ hout,
                      float* __restrict__ cst, int T, int B, long long* __restrict__ dbg,
                      const float* __restrict__ h0, const float* __restrict__ c0) {
  using C = FwdCfg<CELL, CS>;
  constexpr int H = C::H, G = C::G, GH = G * H, RPS = C::RPS, KB = C::KB;
  constexpr bool LSTM = CELL == SEQREC_CELL_LSTM;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sU = base;                                  // [2 parts][region A | region B]
  const uint32_t sH = sU + 2 * C::U_PART;                    // [2 parts][CS K blocks][64 rows][64 B]
  const uint32_t sS = sH + 2 * C::H_PART;                    // [2 buffers][2 parts][4096]
  const uint32_t sBar = sS + 4 * C::STG;
  // bar_hfull[p]: the K slice of source CTA p (hi + lo) has landed -- one barrier per source, so the MMA of a round
  // starts with the first slice and runs behind the exchange instead of after it (the exchange is bound by the
  // ~20 B/clk of distributed shared memory: 56 KB per CTA and round)
  const uint32_t bar_u = sBar, bar_acc = sBar + 16, bar_staged = sBar + 24, bar_free = sBar + 32,
                 tmem_slot = sBar + 40, bar_hfull = sBar + 48;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int b0 = (int)(blockIdx.x / CS) * BMR;
  const int R = T * RPS;

  if (threadIdx.x == 0) {
    ptx::mbar_init(bar_u, 1);
    for (int p = 0; p < CS; ++p) ptx::mbar_init(bar_hfull + 8 * p, 1);
    ptx::mbar_init(bar_acc, 1);
    ptx::mbar_init(bar_staged, 4);
    ptx::mbar_init(bar_free, CS);
    ptx::fence_barrier_init();
  }
  if constexpr (INIT) {
    // the epilogue threads' (row, half) layout: each stages its 16 units of every unit slice p (rows past B: zeros)
    if (warp < 4) {
      const int row = 16 * warp + (lane & 15), hh = lane >> 4;
      const bool ok = h0 != nullptr && b0 + row < B;
      for (int p = 0; p < CS; ++p) {
        float v[16];
        load16(v, h0 + (size_t)(ok ? b0 + row : 0) * H + p * UPC + hh * 16, ok);
        stage_slice(sH + (uint32_t)p * 4096u, sH + C::H_PART + (uint32_t)p * 4096u, row, hh, v);
      }
    }
  } else {
    for (uint32_t i = threadIdx.x * 16u; i < 2 * C::H_PART; i += RT_THREADS * 16u) st_shared_u4(sH + i, 0, 0, 0, 0);
  }
  ptx::fence_proxy_async_smem();                             // h_{-1} is read by the tensor core (async proxy)
  if (warp == 4) {
    ptx::tmem_alloc(tmem_slot, 64);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  ptx::cluster_arrive();                                     // every CTA's barriers exist before any remote traffic
  ptx::cluster_wait();

  if (warp == 4) {
    // ------------------------------------------------------------------------------------- TMA (once) + MMA issuer
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx(bar_u, 2 * C::U_PART);
      for (int part = 0; part < 2; ++part) {
        const CUtensorMap* tm = part ? &tmU_lo : &tmU_hi;
        const uint32_t dstp = sU + part * C::U_PART;
        for (int kb = 0; kb < KB; ++kb) {
          // operand row (N index) of region A: hh*(GA*16) + g*16 + j  <->  U^T row g*H + 32*rank + 16*hh + j
          for (int hh = 0; hh < 2; ++hh)
            for (int g = 0; g < C::GA; ++g)
              ptx::tma_load_2d(dstp + (uint32_t)(kb * C::NA + hh * C::GA * 16 + g * 16) * 128u, tm, bar_u, kb * 64,
                               g * H + (int)rank * UPC + hh * 16);
          if (!LSTM)
            for (int hh = 0; hh < 2; ++hh)
              ptx::tma_load_2d(dstp + C::UA_BYTES + (uint32_t)(kb * C::NB + hh * 16) * 128u, tm, bar_u, kb * 64,
                               2 * H + (int)rank * UPC + hh * 16);
        }
      }
      if (R > 1)
        for (int p = 0; p < CS; ++p) ptx::mbar_arrive_expect_tx(bar_hfull + 8 * p, 2 * C::STG);
    }
    __syncwarp();
    ptx::mbar_wait(bar_u, 0);
    for (int r = 0; r < R; ++r) {
      const bool sub_b = (RPS == 2) && (r & 1);
      const int nh = LSTM ? 64 : (sub_b ? 16 : 32);          // accumulator columns per half = MMA N
      const int nr = sub_b ? C::NB : C::NA;                  // operand rows per K block in this region
      const uint32_t ureg = sU + (sub_b ? C::UA_BYTES : 0u);
      const uint32_t idesc = ptx::umma_idesc_bf16(BMR, nh);
      // descriptor bases once per round; every MMA then needs one 32-bit add per operand (the address field never
      // carries out of its 14 bits), so the single issuing thread keeps up with the tensor pipe
      const uint64_t a_hi0 = ptx::umma_desc_k_sw64(sH), a_lo0 = ptx::umma_desc_k_sw64(sH + C::H_PART);
      const uint64_t b_hi0 = ptx::umma_desc_k_sw128(ureg), b_lo0 = ptx::umma_desc_k_sw128(ureg + C::U_PART);
      const uint32_t kstride = (uint32_t)nr * 8u;                      // one K block of the U region, >> 4
      // K slices in the order they arrive: the own one first, then the sources rank-1, rank-2, ... (every sender
      // serves its destinations in the order rank, rank+1, ...)
      // (LSTM: measured SLOWER when the MMAs run behind the exchange -- 1.19 -> 1.35 ms at cfg3: its M64 x N64 MMAs read
      //  4 KB of operands per ~40 clocks, i.e. they already hold the shared-memory port that the incoming and outgoing
      //  bulk copies need, and the two streams slow each other down.  The LSTM therefore waits for all slices first;
      //  the GRU's smaller rounds gain 11 %.)
      constexpr bool PIPE = !LSTM;
      for (int pass = PIPE ? 1 : 0; pass < 2; ++pass)
      for (int i = 0; i < CS; ++i) {
        const uint32_t p = (rank + (uint32_t)(CS - i)) % (uint32_t)CS;
        if (r > 0 && pass == (PIPE ? 1 : 0)) {
          ptx::mbar_wait_cluster(bar_hfull + 8 * p, (uint32_t)(r - 1) & 1u);   // slice p of the operand has landed
          if (i == (PIPE ? 0 : CS - 1) && lane == 0) RT_DBG(r, 0);
          if (r < R - 1 && ptx::elect_one()) ptx::mbar_arrive_expect_tx(bar_hfull + 8 * p, 2 * C::STG);
          __syncwarp();
        }
        if (pass == 0) continue;
        ptx::tc_fence_after_sync();
        if (ptx::elect_one()) {
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const uint32_t d = tmem_base + ((uint32_t)(hh * 16) << 16);  // second M=64 atom on lanes 16..31 of each quadrant
            const uint32_t bh = (uint32_t)(hh * nh) * 8u;                // (hh * nh rows * 128 B) >> 4
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              const uint32_t s = 2u * p + (uint32_t)ks;                  // K = 16 step of the whole operand
              const uint32_t a_off = (s >> 1) * 256u + (s & 1u) * 2u;    // byte offsets >> 4
              const uint32_t b_off = (s >> 2) * kstride + bh + (s & 3u) * 2u;
              ptx::umma_bf16(d, a_hi0 + a_off, b_lo0 + b_off, idesc, (i > 0 || ks > 0) ? 1u : 0u);
              ptx::umma_bf16(d, a_lo0 + a_off, b_hi0 + b_off, idesc, 1u);
              ptx::umma_bf16(d, a_hi0 + a_off, b_hi0 + b_off, idesc, 1u);
            }
          }
          if (i == CS - 1) {
            ptx::umma_commit(bar_acc);
            RT_DBG(r, 1);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 5) {
    // ------------------------------------------------------------------------------------- exchange (all-gather)
    for (int r = 0; r + 1 < R; ++r) {
      ptx::mbar_wait(bar_staged, (uint32_t)r & 1u);          // this CTA's slice of round r is staged
      if (lane == 0) RT_DBG(r, 4);
      ptx::mbar_wait_cluster(bar_free, (uint32_t)r & 1u);    // every CTA's MMA of round r has read its operand
      if (lane == 0) RT_DBG(r, 5);
      if (ptx::elect_one()) {
        const uint32_t src = sS + (uint32_t)(r & 1) * 2u * C::STG;
        for (uint32_t i = 0; i < (uint32_t)CS; ++i) {            // own copy first, then rank+1, rank+2, ...
          const uint32_t p = (rank + i) % (uint32_t)CS;
          const uint32_t dst = ptx::mapa(sH + rank * 4096u, p);
          const uint32_t bar = ptx::mapa(bar_hfull + 8 * rank, p);
          ptx::bulk_copy_to_cluster(dst, src, C::STG, bar);
          ptx::bulk_copy_to_cluster(dst + C::H_PART, src + C::STG, C::STG, bar);
        }
        RT_DBG(r, 6);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------------------------- epilogue: gate math
    const int q = warp;
    const int row = 16 * q + (lane & 15), hh = lane >> 4;
    const int b = b0 + row;
    const bool valid = b < B;
    const int u0 = (int)rank * UPC + hh * 16;                // first of this thread's 16 hidden units
    const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16);
    float hprev[16], cs[16], zg[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { hprev[j] = 0.f; cs[j] = 0.f; zg[j] = 0.f; }
    if constexpr (INIT) {
      load16(hprev, h0 + (size_t)(valid ? b : 0) * H + u0, valid && h0 != nullptr);
      if (LSTM) load16(cs, c0 + (size_t)(valid ? b : 0) * H + u0, valid && c0 != nullptr);
    }

    auto after_acc = [&](int r) {                            // MMA of round r is complete
      ptx::mbar_wait(bar_acc, (uint32_t)r & 1u);
      ptx::tc_fence_after_sync();
      if (threadIdx.x == 0) RT_DBG(r, 2);
      // "my MMA has finished reading my operand": one lane per peer, no data to publish -> relaxed arrives
      if (warp == 0 && lane < CS && r + 1 < R) ptx::mbar_arrive_cluster_relaxed(ptx::mapa(bar_free, (uint32_t)lane));
    };
    auto stage = [&](int r, const float (&v)[16]) {
      if (r + 1 < R) {
        const uint32_t s0 = sS + (uint32_t)(r & 1) * 2u * C::STG;
        stage_slice(s0, s0 + C::STG, row, hh, v);
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar_staged);
        if (threadIdx.x == 0) RT_DBG(r, 3);
      }
    };

    for (int t = 0; t < T; ++t) {
      const size_t tok = (size_t)t * B + (valid ? b : 0);
      const bool m = valid && mask[tok] != 0;
      float* gp = xg + tok * GH + u0;
      if constexpr (LSTM) {
        float x[64];
#pragma unroll
        for (int g = 0; g < 4; ++g) load16(x + 16 * g, gp + g * H, valid);   // issued before the MMA wait
        after_acc(t);
        uint32_t z0[32], z1[32];
        ptx::tmem_ld_32x32(taddr, z0);
        ptx::tmem_ld_32x32(taddr + 32, z1);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before_sync();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float ig = hard_sigmoid_f(x[j] + __uint_as_float(z0[j]));
          const float fg = hard_sigmoid_f(x[16 + j] + __uint_as_float(z0[16 + j]));
          const float gg = act_fast<ACT>(x[32 + j] + __uint_as_float(z1[j]));
          const float og = hard_sigmoid_f(x[48 + j] + __uint_as_float(z1[16 + j]));
          const float cn = fmaf(fg, cs[j], ig * gg);
          const float hn = og * act_fast<ACT>(cn);
          x[j] = ig; x[16 + j] = fg; x[32 + j] = gg; x[48 + j] = og;
          if (m) { cs[j] = cn; hprev[j] = hn; }
        }
        stage(t, hprev);
        if (valid) {
#pragma unroll
          for (int g = 0; g < 4; ++g) store16(gp + g * H, x + 16 * g);
          store16(cst + tok * H + u0, cs);
          store16(hout + tok * H + u0, hprev);
        }
      } else {
        // ---- round A: z, r from h_{t-1}; r*h_{t-1} is the operand of round B
        float x[32], rh[16];
        load16(x, gp, valid);
        load16(x + 16, gp + H, valid);
        after_acc(2 * t);
        {
          uint32_t z0[32];
          ptx::tmem_ld_32x32(taddr, z0);
          ptx::tmem_ld_wait();
          ptx::tc_fence_before_sync();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float z = hard_sigmoid_f(x[j] + __uint_as_float(z0[j]));
            const float rr = hard_sigmoid_f(x[16 + j] + __uint_as_float(z0[16 + j]));
            zg[j] = z; x[j] = z; x[16 + j] = rr;
            rh[j] = rr * hprev[j];
          }
        }
        stage(2 * t, rh);
        if (valid) { store16(gp, x); store16(gp + H, x + 16); }
        // ---- round B: candidate, state update under the mask
        load16(x, gp + 2 * H, valid);
        after_acc(2 * t + 1);
        {
          uint32_t z0[16];
          tmem_ld_32x16(taddr, z0);
          ptx::tmem_ld_wait();
          ptx::tc_fence_before_sync();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float hc = act_fast<ACT>(x[j] + __uint_as_float(z0[j]));
            const float hn = zg[j] * hprev[j] + (1.0f - zg[j]) * hc;
            x[j] = hc;
            if (m) hprev[j] = hn;
          }
        }
        stage(2 * t + 1, hprev);
        if (valid) { store16(gp + 2 * H, x); store16(hout + tok * H + u0, hprev); }
      }
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, 64);
  }
  ptx::cluster_arrive();                                     // no CTA leaves while peers may still address its memory
  ptx::cluster_wait();
}

template <int CELL, int ACT, int CS>
int launch_fwd(float* xg, const uint16_t* Ut_hi, const uint16_t* Ut_lo, const uint8_t* mask, float* hout, float* cst,
               int T, int B, cudaStream_t st, const float* h0, const float* c0) {
  using C = FwdCfg<CELL, CS>;
  CUtensorMap tm_hi, tm_lo;
  int rc;
  // U^T (G*H rows, H columns) bf16; box = 64 hidden units (K) x 16 gate columns of one (gate, half) group
  if ((rc = tma::make_2d_bf16(&tm_hi, Ut_hi, (uint64_t)C::G * C::H, C::H, C::H, 64, 16, CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  if ((rc = tma::make_2d_bf16(&tm_lo, Ut_lo, (uint64_t)C::G * C::H, C::H, C::H, 64, 16, CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  auto k = (h0 || c0) ? rnn_tc_forward_kernel<CELL, ACT, CS, true> : rnn_tc_forward_kernel<CELL, ACT, CS, false>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
  if (e != cudaSuccess) return -(int)e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(ceil_div(B, BMR) * CS));
  cfg.blockDim = dim3(RT_THREADS);
  cfg.dynamicSmemBytes = C::SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, k, tm_hi, tm_lo, xg, mask, hout, cst, T, B, g_rnn_tc_dbg, h0, c0);
  if (e != cudaSuccess) return -(int)e;
  SEQREC_CHECK_LAUNCH();
  return 0;
}

template <int CELL, int CS>
int dispatch_act_fwd(int act, float* xg, const uint16_t* Ut_hi, const uint16_t* Ut_lo, const uint8_t* mask,
                     float* hout, float* cst, int T, int B, cudaStream_t st, const float* h0, const float* c0) {
  switch (act) {
    case SEQREC_ACT_RELU:
      return launch_fwd<CELL, SEQREC_ACT_RELU, CS>(xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
    case SEQREC_ACT_TANH:
      return launch_fwd<CELL, SEQREC_ACT_TANH, CS>(xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
    case SEQREC_ACT_LINEAR:
      return launch_fwd<CELL, SEQREC_ACT_LINEAR, CS>(xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
    default: return -1002;
  }
}


// ================================================================================================================
// K4 on the tensor cores: the scan's backward pass (Theano's scan gradient of the layer above), same cluster layout.
//   CTA c owns hidden units J_c = [32c, 32c+32) of 64 batch rows: it computes the pre-activation gradients da of ITS
//   gate columns locally (elementwise, fp32), writes them as the bf16 hi/lo A operand [64 rows x (gates x 32)], and
//   the tensor core forms the K-SPLIT partial product  P_c[64, H] = da_c . U[:, cols_c]^T  (M = 64, N = H in two
//   interleaved halves, fp32 in TMEM).  dL/dh_{t-1} = sum_c P_c is REDUCE-SCATTERED through distributed shared memory:
//   every thread stores the 32-unit slice that belongs to CTA p straight from its registers into p's receive buffer
//   (st.shared::cluster), p sums the CS partials of its own units in a fixed order (deterministic).
//   U[:, cols_c] (H rows x gates x 32 columns, bf16 hi/lo, 64-byte-swizzled K blocks of one gate each) is loaded once.
//   GRU: two rounds per step (d(r*h) through U_h first, then z,r through U_zr), LSTM: one.
// xg: in = saved gates, out = dxp; cst: LSTM cell states (in), GRU r*h_{t-1} (out, operand of dU) -- as rnn_scan.cu.
template <int CELL, int CS>
struct BwdCfg {
  static constexpr int H = CS * UPC;
  static constexpr int G = (CELL == SEQREC_CELL_LSTM) ? 4 : 3;
  static constexpr int NBLK = G;                                      // K blocks = gates (32 own columns each)
  static constexpr uint32_t UBLK = H * 64;                            // one K block of the U operand: H rows x 64 B
  static constexpr uint32_t U_PART = NBLK * UBLK;
  static constexpr uint32_t A_PART = NBLK * 4096;                     // da operand: 64 rows x 64 B per gate
  static constexpr uint32_t RECV = CS * 8192;                         // [source CTA][64 rows][32 fp32]
  static constexpr uint32_t SMEM = 2 * U_PART + 2 * A_PART + RECV + 64 + 1024;
  static constexpr int TMEM_COLS = H / 2;                             // accumulator columns per interleaved half
};

template <int CELL, int ACT, int CS>
__global__ void __launch_bounds__(RT_THREADS, 1)
rnn_tc_backward_kernel(const __grid_constant__ CUtensorMap tmU_hi, const __grid_constant__ CUtensorMap tmU_lo,
                       float* __restrict__ xg, const uint8_t* __restrict__ mask, const float* __restrict__ hout,
                       float* __restrict__ cst, const float* __restrict__ dhout, int T, int B,
                       long long* __restrict__ dbg) {
  using C = BwdCfg<CELL, CS>;
  constexpr int H = C::H, G = C::G, GH = G * H;
  constexpr bool LSTM = CELL == SEQREC_CELL_LSTM;
  constexpr int NH = H / 2;                                  // MMA N per half
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sU = base;                                  // [2 parts][G blocks][H rows][64 B]
  const uint32_t sA = sU + 2 * C::U_PART;                    // [2 parts][G blocks][64 rows][64 B]
  const uint32_t sR = sA + 2 * C::A_PART;                    // [CS sources][8 chunks of 16 B][64 rows]
  const uint32_t sBar = sR + C::RECV;
  const uint32_t bar_u = sBar, bar_aready = sBar + 8, bar_acc = sBar + 16, bar_rfull = sBar + 24,
                 bar_rfree = sBar + 32, tmem_slot = sBar + 40;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int b0 = (int)(blockIdx.x / CS) * BMR;
  // MMA rounds: LSTM one per step, GRU two; the step t = 0 needs none (dL/dh_{-1} is not used)
  const int RPS = LSTM ? 1 : 2;
  const int R = (T - 1) * RPS;

  if (threadIdx.x == 0) {
    ptx::mbar_init(bar_u, 1);
    ptx::mbar_init(bar_aready, 4);
    ptx::mbar_init(bar_acc, 1);
    ptx::mbar_init(bar_rfull, 4 * CS);
    ptx::mbar_init(bar_rfree, 4 * CS);
    ptx::fence_barrier_init();
  }
  if (warp == 4) {
    ptx::tmem_alloc(tmem_slot, C::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  ptx::cluster_arrive();
  ptx::cluster_wait();

  if (warp == 4) {
    // ------------------------------------------------------------------------------------- TMA (once) + MMA issuer
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx(bar_u, 2 * C::U_PART);
      for (int part = 0; part < 2; ++part)
        for (int g = 0; g < G; ++g)                          // K block g = columns g*H + 32*rank .. +32 of every row of U
          ptx::tma_load_2d(sU + part * C::U_PART + g * C::UBLK, part ? &tmU_lo : &tmU_hi, bar_u,
                           g * H + (int)rank * UPC, 0);
    }
    __syncwarp();
    ptx::mbar_wait(bar_u, 0);
    const uint32_t idesc = ptx::umma_idesc_bf16(BMR, NH);
    for (int r = 0; r < R; ++r) {
      ptx::mbar_wait(bar_aready, (uint32_t)r & 1u);          // da of this round is in shared memory
      ptx::tc_fence_after_sync();
      // K blocks of this round: LSTM all four gates; GRU round A = candidate block, round B = z and r blocks
      const int kb0 = LSTM ? 0 : ((r & 1) ? 0 : 2);
      const int kb1 = LSTM ? 4 : ((r & 1) ? 2 : 3);
      if (ptx::elect_one()) {
        const uint64_t a_hi0 = ptx::umma_desc_k_sw64(sA), a_lo0 = ptx::umma_desc_k_sw64(sA + C::A_PART);
        const uint64_t b_hi0 = ptx::umma_desc_k_sw64(sU), b_lo0 = ptx::umma_desc_k_sw64(sU + C::U_PART);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t d = tmem_base + ((uint32_t)(hh * 16) << 16);
          for (int kb = kb0; kb < kb1; ++kb)
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              const uint32_t a_off = (uint32_t)kb * 256u + (uint32_t)ks * 2u;                       // byte offsets >> 4
              const uint32_t b_off = (uint32_t)kb * (C::UBLK >> 4) + (uint32_t)(hh * NH) * 4u + (uint32_t)ks * 2u;
              ptx::umma_bf16(d, a_hi0 + a_off, b_lo0 + b_off, idesc, (kb > kb0 || ks > 0) ? 1u : 0u);
              ptx::umma_bf16(d, a_lo0 + a_off, b_hi0 + b_off, idesc, 1u);
              ptx::umma_bf16(d, a_hi0 + a_off, b_hi0 + b_off, idesc, 1u);
            }
        }
        ptx::umma_commit(bar_acc);
      }
      __syncwarp();
    }
  } else if (warp < 4) {
    // ------------------------------------------------------------------------------------- elementwise + exchange
    const int q = warp;
    const int row = 16 * q + (lane & 15), hh = lane >> 4;
    const int b = b0 + row;
    const bool valid = b < B;
    const int u0 = (int)rank * UPC + hh * 16;
    const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16);
    float rec[16], dcar[16], dd[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { rec[j] = 0.f; dcar[j] = 0.f; dd[j] = 0.f; }
    int xr = 0;                                              // exchange rounds done

    // A operand block g <- this thread's 16 values; then tell the MMA warp (after every block of the round is in)
    auto put_block = [&](int g, const float (&v)[16]) {
      stage_slice(sA + (uint32_t)g * 4096u, sA + C::A_PART + (uint32_t)g * 4096u, row, hh, v);
    };
    auto a_ready = [&]() {
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar_aready);
    };
    // partial products of this CTA -> the owners of the hidden units (straight from the accumulator registers)
    auto send = [&]() {
      if (threadIdx.x == 0) RT_DBG(xr, 0);
      ptx::mbar_wait(bar_acc, (uint32_t)xr & 1u);
      ptx::tc_fence_after_sync();
      if (threadIdx.x == 0) RT_DBG(xr, 1);
      ptx::mbar_wait_cluster(bar_rfree, ((uint32_t)xr & 1u) ^ 1u);   // every peer has consumed the previous exchange
      if (threadIdx.x == 0) RT_DBG(xr, 2);
#pragma unroll 1
      for (int i = 0; i < CS / 2; ++i) {
        uint32_t v[32];
        ptx::tmem_ld_32x32(taddr + 32 * i, v);
        ptx::tmem_ld_wait();
        const uint32_t p = (uint32_t)(hh * (CS / 2) + i);    // owner of units [hh*H/2 + 32i, +32)
        // chunk-major layout: the 16 lanes that address one peer write 256 contiguous bytes per instruction (with a
        // row-major buffer every lane hit its own 128-byte row: 16-byte pieces, half of every 32-byte sector wasted)
        const uint32_t dst = ptx::mapa(sR + rank * 8192u + (uint32_t)row * 16u, p);
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k)
          ptx::st_cluster_f4(dst + (k << 10),
                             make_float4(__uint_as_float(v[4 * k]), __uint_as_float(v[4 * k + 1]),
                                         __uint_as_float(v[4 * k + 2]), __uint_as_float(v[4 * k + 3])));
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      // one lane per peer: the release (cumulative over the warp's stores through __syncwarp) is paid once, in parallel
      if (lane < CS) ptx::mbar_arrive_cluster(ptx::mapa(bar_rfull, (uint32_t)lane));
      if (threadIdx.x == 0) RT_DBG(xr, 3);
    };
    // receive: sum the CS partials of OUR units in a fixed order (deterministic), then free the buffer for the peers
    auto recv = [&](float (&sum)[16]) {
      ptx::mbar_wait_cluster(bar_rfull, (uint32_t)xr & 1u);
      if (threadIdx.x == 0) RT_DBG(xr, 4);
#pragma unroll
      for (int j = 0; j < 16; ++j) sum[j] = 0.f;
#pragma unroll 2
      for (uint32_t src = 0; src < (uint32_t)CS; ++src) {
        const uint32_t a = sR + src * 8192u + (uint32_t)row * 16u;
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
          float4 t;
          asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                       : "=f"(t.x), "=f"(t.y), "=f"(t.z), "=f"(t.w)
                       : "r"(a + (((uint32_t)hh * 4u + k) << 10)));
          sum[4 * k] += t.x; sum[4 * k + 1] += t.y; sum[4 * k + 2] += t.z; sum[4 * k + 3] += t.w;
        }
      }
      __syncwarp();
      if (lane < CS) ptx::mbar_arrive_cluster_relaxed(ptx::mapa(bar_rfree, (uint32_t)lane));
      if (threadIdx.x == 0) RT_DBG(xr, 5);
      ++xr;
    };

    // per-step inputs live in registers and are PREFETCHED for step t-1 between send() and recv(): the global-load
    // latency hides behind the exchange instead of sitting on the sequential path
    float dh[16], g0[16], g1[16], g2[16], g3[16], c0[16], c1[16];
    bool m = false;
    auto load_step = [&](int t) {
      const size_t tok = (size_t)t * B + (valid ? b : 0);
      m = valid && mask[tok] != 0;
      const float* gp = xg + tok * GH + u0;
      load16(dh, dhout + tok * H + u0, valid);
      load16(g0, gp, m); load16(g1, gp + H, m); load16(g2, gp + 2 * H, m);
      if constexpr (LSTM) {
        load16(g3, gp + 3 * H, m);
        load16(c0, cst + tok * H + u0, m);
        load16(c1, cst + (tok - (size_t)B) * H + u0, m && t > 0);        // c_{t-1}
      } else {
        load16(c1, hout + (tok - (size_t)B) * H + u0, m && t > 0);       // h_{t-1}
      }
    };
    load_step(T - 1);

    for (int t = T - 1; t >= 0; --t) {
      const size_t tok = (size_t)t * B + (valid ? b : 0);
      float* gp = xg + tok * GH + u0;
#pragma unroll
      for (int j = 0; j < 16; ++j) dh[j] += rec[j];
      if constexpr (LSTM) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (m) {
            const float ac = act_fast<ACT>(c0[j]);
            const float d_o = dh[j] * ac;
            const float dc = dcar[j] + dh[j] * g3[j] * act_grad_from_y<ACT>(ac);
            const float ai = dc * g2[j] * hard_sigmoid_grad_from_y(g0[j]);
            const float af = dc * c1[j] * hard_sigmoid_grad_from_y(g1[j]);
            const float ag = dc * g0[j] * act_grad_from_y<ACT>(g2[j]);
            const float ao = d_o * hard_sigmoid_grad_from_y(g3[j]);
            dcar[j] = dc * g1[j];
            dd[j] = 0.f;
            g0[j] = ai; g1[j] = af; g2[j] = ag; g3[j] = ao;
          } else {                                           // masked step: state held, no gate gradient
            dd[j] = dh[j];
            g0[j] = 0.f; g1[j] = 0.f; g2[j] = 0.f; g3[j] = 0.f;
          }
        }
        if (t > 0) {
          put_block(0, g0); put_block(1, g1); put_block(2, g2); put_block(3, g3);
          a_ready();
        }
        if (valid) { store16(gp, g0); store16(gp + H, g1); store16(gp + 2 * H, g2); store16(gp + 3 * H, g3); }
        if (t > 0) {
          send();
          load_step(t - 1);
          float sum[16];
          recv(sum);
#pragma unroll
          for (int j = 0; j < 16; ++j) rec[j] = dd[j] + sum[j];
        }
      } else {
        // g0 = z, g1 = r, g2 = candidate, c1 = h_{t-1}
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          c0[j] = g1[j] * c1[j];                             // operand of dU's candidate block (0 on masked steps)
          if (m) {
            const float az = dh[j] * (c1[j] - g2[j]) * hard_sigmoid_grad_from_y(g0[j]);
            const float ah = dh[j] * (1.0f - g0[j]) * act_grad_from_y<ACT>(g2[j]);
            dd[j] = dh[j] * g0[j];
            g0[j] = az; g2[j] = ah;
          } else {
            dd[j] = dh[j];
            g0[j] = 0.f; g2[j] = 0.f;
          }
        }
        if (t > 0) {
          // ---- round A: d(r*h_{t-1}) = da_h . U_h^T
          put_block(2, g2);
          a_ready();
          if (valid) store16(cst + tok * H + u0, c0);
          float drh[16];
          send();
          recv(drh);
          // ---- round B: da_r, then dL/dh_{t-1} = direct + [da_z, da_r] . U_zr^T
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float ar = m ? drh[j] * c1[j] * hard_sigmoid_grad_from_y(g1[j]) : 0.f;
            if (m) dd[j] += drh[j] * g1[j];
            g1[j] = ar;
          }
          put_block(0, g0); put_block(1, g1);
          a_ready();
          if (valid) { store16(gp, g0); store16(gp + H, g1); store16(gp + 2 * H, g2); }
          send();
          load_step(t - 1);
          float sum[16];
          recv(sum);
#pragma unroll
          for (int j = 0; j < 16; ++j) rec[j] = dd[j] + sum[j];
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) g1[j] = 0.f;          // h_{-1} = 0: the reset gate has no gradient at t = 0
          if (valid) {
            store16(cst + tok * H + u0, c0);
            store16(gp, g0); store16(gp + H, g1); store16(gp + 2 * H, g2);
          }
        }
      }
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
  ptx::cluster_arrive();
  ptx::cluster_wait();
}

template <int CELL, int ACT, int CS>
int launch_bwd(float* xg, const uint16_t* U_hi, const uint16_t* U_lo, const uint8_t* mask, const float* hout,
               float* cst, const float* dhout, int T, int B, cudaStream_t st) {
  using C = BwdCfg<CELL, CS>;
  CUtensorMap tm_hi, tm_lo;
  int rc;
  // U (H rows, G*H columns) bf16; box = 32 gate columns (one K block) x all H rows, 64-byte swizzle
  if ((rc = tma::make_2d_bf16(&tm_hi, U_hi, C::H, (uint64_t)C::G * C::H, (uint64_t)C::G * C::H, 32, C::H,
                              CU_TENSOR_MAP_SWIZZLE_64B)))
    return rc;
  if ((rc = tma::make_2d_bf16(&tm_lo, U_lo, C::H, (uint64_t)C::G * C::H, (uint64_t)C::G * C::H, 32, C::H,
                              CU_TENSOR_MAP_SWIZZLE_64B)))
    return rc;
  auto k = rnn_tc_backward_kernel<CELL, ACT, CS>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
  if (e != cudaSuccess) return -(int)e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(ceil_div(B, BMR) * CS));
  cfg.blockDim = dim3(RT_THREADS);
  cfg.dynamicSmemBytes = C::SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, k, tm_hi, tm_lo, xg, mask, hout, cst, dhout, T, B, g_rnn_tc_dbg);
  if (e != cudaSuccess) return -(int)e;
  SEQREC_CHECK_LAUNCH();
  return 0;
}

template <int CELL, int CS>
int dispatch_act_bwd(int act, float* xg, const uint16_t* U_hi, const uint16_t* U_lo, const uint8_t* mask,
                     const float* hout, float* cst, const float* dhout, int T, int B, cudaStream_t st) {
  switch (act) {
    case SEQREC_ACT_RELU:
      return launch_bwd<CELL, SEQREC_ACT_RELU, CS>(xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
    case SEQREC_ACT_TANH:
      return launch_bwd<CELL, SEQREC_ACT_TANH, CS>(xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
    case SEQREC_ACT_LINEAR:
      return launch_bwd<CELL, SEQREC_ACT_LINEAR, CS>(xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
    default: return -1002;
  }
}

}  // namespace

/* diagnostics only (not in the public header): device buffer of 64 x 8 clock64() stamps written by CTA 0 */
extern "C" int seqrec_rnn_tc_debug_buffer(long long* dev_buf) {
  g_rnn_tc_dbg = dev_buf;
  return 0;
}

namespace {
template <int CELL, int CS>
int max_clusters_fwd() {
  using C = FwdCfg<CELL, CS>;
  auto k = rnn_tc_forward_kernel<CELL, SEQREC_ACT_TANH, CS, false>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM);
  if (e != cudaSuccess) return -(int)e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(CS * 64));
  cfg.blockDim = dim3(RT_THREADS);
  cfg.dynamicSmemBytes = C::SMEM;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  e = cudaOccupancyMaxActiveClusters(&n, k, &cfg);
  return e == cudaSuccess ? n : -(int)e;
}
}  // namespace

/* How many clusters of the tensor-core scan (64 batch rows each) the current device keeps resident at once: a batch of
 * more than 64 x this many rows runs in waves.  The figure depends on how the part's SMs are spread over its GPCs. */
extern "C" int seqrec_rnn_tc_max_clusters(int cell, int H) {
  if (!seqrec_rnn_tc_applicable(cell, H)) return -1001;
  if (cell == SEQREC_CELL_LSTM) return H == 256 ? max_clusters_fwd<SEQREC_CELL_LSTM, 8>() : max_clusters_fwd<SEQREC_CELL_LSTM, 4>();
  return H == 256 ? max_clusters_fwd<SEQREC_CELL_GRU, 8>() : max_clusters_fwd<SEQREC_CELL_GRU, 4>();
}

extern "C" int seqrec_rnn_tc_applicable(int cell, int H) {
  return ((cell == SEQREC_CELL_LSTM || cell == SEQREC_CELL_GRU) && (H == 128 || H == 256)) ? 1 : 0;
}

extern "C" int seqrec_rnn_tc_forward_state(int cell, int act, float* xg, const uint16_t* Ut_hi,
                                           const uint16_t* Ut_lo, const float* h0, const float* c0,
                                           const uint8_t* mask, float* hout, float* cst, int T, int B, int H,
                                           void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && seqrec_rnn_tc_applicable(cell, H), 1);
  SEQREC_ARG(xg && Ut_hi && Ut_lo && mask && hout && (cell != SEQREC_CELL_LSTM || cst), 2);
  SEQREC_ARG(c0 == nullptr || cell == SEQREC_CELL_LSTM, 2);
  SEQREC_ARG(((uintptr_t)h0 & 15) == 0 && ((uintptr_t)c0 & 15) == 0, 2);   // read as float4
  cudaStream_t st = as_stream(stream);
  if (cell == SEQREC_CELL_LSTM) {
    if (H == 256)
      return dispatch_act_fwd<SEQREC_CELL_LSTM, 8>(act, xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
    return dispatch_act_fwd<SEQREC_CELL_LSTM, 4>(act, xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
  }
  if (H == 256) return dispatch_act_fwd<SEQREC_CELL_GRU, 8>(act, xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
  return dispatch_act_fwd<SEQREC_CELL_GRU, 4>(act, xg, Ut_hi, Ut_lo, mask, hout, cst, T, B, st, h0, c0);
}

extern "C" int seqrec_rnn_tc_forward(int cell, int act, float* xg, const uint16_t* Ut_hi, const uint16_t* Ut_lo,
                                     const uint8_t* mask, float* hout, float* cst, int T, int B, int H,
                                     void* stream) {
  return seqrec_rnn_tc_forward_state(cell, act, xg, Ut_hi, Ut_lo, nullptr, nullptr, mask, hout, cst, T, B, H, stream);
}

extern "C" int seqrec_rnn_tc_backward(int cell, int act, float* xg, const uint16_t* U_hi, const uint16_t* U_lo,
                                      const uint8_t* mask, const float* hout, float* cst, const float* dhout, int T,
                                      int B, int H, void* stream) {
  SEQREC_ARG(T > 0 && B > 0 && seqrec_rnn_tc_applicable(cell, H), 1);
  SEQREC_ARG(xg && U_hi && U_lo && mask && hout && cst && dhout, 2);
  cudaStream_t st = as_stream(stream);
  if (cell == SEQREC_CELL_LSTM) {
    if (H == 256) return dispatch_act_bwd<SEQREC_CELL_LSTM, 8>(act, xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
    return dispatch_act_bwd<SEQREC_CELL_LSTM, 4>(act, xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
  }
  if (H == 256) return dispatch_act_bwd<SEQREC_CELL_GRU, 8>(act, xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
  return dispatch_act_bwd<SEQREC_CELL_GRU, 4>(act, xg, U_hi, U_lo, mask, hout, cst, dhout, T, B, st);
}
