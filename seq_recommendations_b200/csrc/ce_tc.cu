// K5 / K6 on the 5th-generation tensor cores: fused logits GEMM + online-softmax statistics (forward) and the
// recompute-based backward (dH and dW_out), never materialising the (N,V) logits.
// Reference constructs replaced: TimeDistributed(Dense(V)) + softmax + categorical_crossentropy and Theano's
// autodiff of them (model.py:382-384, :397; experiments_methods.py:42).
//
// sm_100a design
//   * operands are bf16, K-major, staged by TMA (cp.async.bulk.tensor, 128-byte swizzle) into shared memory
//   * tcgen05.mma (kind::f16, M=128) issued by ONE elected thread, fp32 accumulators in TMEM
//   * "fp32 mode" = 3-pass split products  a_hi.b_hi + a_hi.b_lo + a_lo.b_hi  with hi = bf16(x), lo = bf16(x - hi)
//     (16 mantissa bits per operand, ~2^-16 relative per product -- inside the 1e-4 budget of north_star);
//     "bf16 mode" issues the hi.hi product only
//   * warp-specialised: warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2..9 = epilogue: two warps per
//     TMEM lane quadrant, each owning one 64-column half of the tile (tcgen05.ld 32x32b: one thread owns one token
//     row -> row-wise softmax statistics need no shuffles; the two halves are merged like two vocabulary splits)
//   * the logits tile never leaves the SM: forward keeps a running (max, sum-exp) per row; backward turns the tile
//     into dlogit = (p - onehot)*coef in registers, writes it as a bf16 hi/lo K-major operand into shared memory and
//     feeds it straight back to the tensor core (dH += dS.W^T  /  dW += H^T.dS).
//
// Tiles: 128 tokens x 128 items; K (= hidden, padded to 64) is walked in 64-element blocks (one 128-byte swizzle row).
#include <cstdlib>

#include "common.cuh"
#include "ptx_sm100.cuh"
#include "tma_host.cuh"

namespace {

constexpr int BM = 128;          // tokens per tile (UMMA M)
constexpr int BN = 128;          // items per tile  (UMMA N of the logits GEMM)
constexpr int KBLK = 64;         // bf16 elements per 128-byte swizzled row
constexpr int TILE_B = 128 * 128;  // bytes of one [128 rows x 64 bf16] operand block
constexpr int TC_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quadrant)
constexpr int TCF_THREADS = 352; // forward: warps 1 and 2 issue alternate tiles, warps 3..10 epilogue
constexpr int N_EPI_WARPS = 8;
constexpr float LOG2E = 1.4426950408889634f;

// ---- host: TMA descriptors --------------------------------------------------------------------------------------
// bf16 matrix (rows, cols) with leading dimension ld (elements); box = 64 columns x box_rows rows, 128-byte swizzle.
int make_tmap(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  return tma::make_2d_bf16(m, ptr, rows, cols, ld, KBLK, box_rows, CU_TENSOR_MAP_SWIZZLE_128B);
}

// ---- device helpers ---------------------------------------------------------------------------------------------
struct Pipe {  // ring of NS stages
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance(int ns) {
    if (++stage == ns) { stage = 0; phase ^= 1; }
  }
};

// one 64-wide K block of the split product: acc (+)= a_hi.b_hi [+ a_hi.b_lo + a_lo.b_hi]
template <bool X3>
__device__ __forceinline__ void mma_kblock(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                           uint32_t idesc, bool first) {
  // called by the whole (converged) MMA warp: descriptors are warp-uniform, one elected lane issues
  const uint64_t da_hi = ptx::umma_desc_k_sw128(a_hi), db_hi = ptx::umma_desc_k_sw128(b_hi);
  const uint64_t da_lo = ptx::umma_desc_k_sw128(a_lo), db_lo = ptx::umma_desc_k_sw128(b_lo);
  if (ptx::elect_one()) {
#pragma unroll
    for (int k = 0; k < KBLK / 16; ++k) {
      const int e = k * 16;
      if (X3) {
        // small cross terms first, the dominant hi.hi product last
        ptx::umma_bf16(tmem_d, ptx::umma_desc_advance_k(da_hi, e), ptx::umma_desc_advance_k(db_lo, e), idesc,
                       (first && k == 0) ? 0u : 1u);
        ptx::umma_bf16(tmem_d, ptx::umma_desc_advance_k(da_lo, e), ptx::umma_desc_advance_k(db_hi, e), idesc, 1u);
        ptx::umma_bf16(tmem_d, ptx::umma_desc_advance_k(da_hi, e), ptx::umma_desc_advance_k(db_hi, e), idesc, 1u);
      } else {
        ptx::umma_bf16(tmem_d, ptx::umma_desc_advance_k(da_hi, e), ptx::umma_desc_advance_k(db_hi, e), idesc,
                       (first && k == 0) ? 0u : 1u);
      }
    }
  }
  __syncwarp();
}

// tcgen05.commit by the elected lane of the converged MMA warp (the lane that issued the MMAs)
__device__ __forceinline__ void commit_elect(uint32_t bar) {
  if (ptx::elect_one()) ptx::umma_commit(bar);
  __syncwarp();
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo_elem, float hi_elem) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo_elem, hi_elem);  // .x = lo_elem (low 16 bits)
  return *reinterpret_cast<const uint32_t*>(&v);
}

// ---- epilogue helpers (each epilogue warp owns 32 rows x 64 columns of a 128 x 128 logits tile) -------------------
// load the warp's 64 accumulator columns (two 32-column tcgen05.ld in flight, one wait)
__device__ __forceinline__ void load_half_tile(uint32_t taddr, float (&z)[64]) {
  uint32_t r0[32], r1[32];
  ptx::tmem_ld_32x32(taddr, r0);
  ptx::tmem_ld_32x32(taddr + 32, r1);
  ptx::tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 32; ++j) { z[j] = __uint_as_float(r0[j]); z[32 + j] = __uint_as_float(r1[j]); }
}

// per-row softmax terms of the backward kernels.  Rows without gradient (pad, clip-saturated) get nb = -inf,
// scale = 0: exp2(z*log2e - inf) = 0 exactly, so no branch and no inf*0.
struct RowTerms {
  float nb;      // -m * log2(e)
  float scale;   // coef * inv_nvalid / s
  float cf;      // coef * inv_nvalid
  int32_t tg;    // target item (or -1)
};
__device__ __forceinline__ RowTerms load_row_terms(int64_t n, int64_t n_tokens, const float* __restrict__ mrow,
                                                   const float* __restrict__ srow, const float* __restrict__ coef,
                                                   const int32_t* __restrict__ tgt, float inv) {
  RowTerms rt;
  rt.nb = -INFINITY; rt.scale = 0.f; rt.cf = 0.f; rt.tg = -1;
  if (n < n_tokens) {
    const float cf = coef[n] * inv;
    if (cf != 0.f) {
      rt.cf = cf;
      rt.nb = -mrow[n] * LOG2E;
      rt.scale = cf / srow[n];
      rt.tg = tgt[n];
    }
  }
  return rt;
}

// z (raw logits of 64 consecutive items starting at item vcol0) -> dlogit in place
__device__ __forceinline__ void dlogit_half_tile(float (&z)[64], const RowTerms& rt, int vcol0, int v_end) {
#pragma unroll
  for (int j = 0; j < 64; ++j) z[j] = ptx::ex2_approx(fmaf(z[j], LOG2E, rt.nb)) * rt.scale;
  if (vcol0 + 64 > v_end) {  // ragged last tile (warp-uniform): items beyond the vocabulary carry no gradient
#pragma unroll
    for (int j = 0; j < 64; ++j)
      if (vcol0 + j >= v_end) z[j] = 0.f;
  }
  const int tj = rt.tg - vcol0;
  if (tj >= 0 && tj < 64) {
#pragma unroll
    for (int j = 0; j < 64; ++j)
      if (j == tj) z[j] -= rt.cf;
  }
}

// ---- persistent work partition ------------------------------------------------------------------------------------
// The (outer, inner) tile pairs are numbered w = outer * n_inner + inner; CTA c of G owns the contiguous range
// [total*c/G, total*(c+1)/G) (balanced to +-1 tile, "stream-K" style).  A maximal run of tiles with the same `outer`
// inside a CTA's range is a SEGMENT: the stationary operand is loaded once per segment and the per-segment result
// (softmax partial, dH or dW accumulator) is flushed at its end.
// d / n and d % n for d < 2^31 by multiply-high with M = floor((2^32 - 1) / n): the estimate is short by at most one.
// Four integer instructions instead of the compiler's division sequence, which goes through I2F / F2I on the XU pipe
// -- the pipe the epilogue warps saturate with ex2 -- and cost ~200 dependent cycles per call on the MMA warp's loop
// header: a bubble in the tensor pipe on EVERY tile (clock64 timeline: tile period 2550 -> 2150 cycles once removed).
struct FastDiv {
  uint32_t n, M;
  __device__ __forceinline__ void init(uint32_t n_) { n = n_; M = 0xFFFFFFFFu / n_; }
  __device__ __forceinline__ void divmod(uint32_t d, uint32_t& q, uint32_t& r) const {
    q = __umulhi(d, M);
    r = d - q * n;
    if (r >= n) { ++q; r -= n; }
  }
};

struct Share {
  int64_t w0, w1;
  int n_inner;
  int o0, i0;   // (outer, inner) of w0: computed ONCE with a 64-bit division; everything per tile is 32-bit
  FastDiv fd;
  __device__ __forceinline__ Share(int64_t total, int n_inner_) : n_inner(n_inner_) {
    w0 = total * blockIdx.x / gridDim.x;
    w1 = total * (blockIdx.x + 1) / gridDim.x;
    o0 = (int)(w0 / n_inner);
    i0 = (int)(w0 - (int64_t)o0 * n_inner);
    fd.init((uint32_t)n_inner);
  }
  __device__ __forceinline__ uint32_t rel(int64_t w) const { return (uint32_t)(w - w0) + (uint32_t)i0; }
  __device__ __forceinline__ int outer(int64_t w) const {
    uint32_t q, r;
    fd.divmod(rel(w), q, r);
    return o0 + (int)q;
  }
  __device__ __forceinline__ int inner(int64_t w) const {
    uint32_t q, r;
    fd.divmod(rel(w), q, r);
    return (int)r;
  }
  __device__ __forceinline__ bool seg_first(int64_t w) const { return w == w0 || inner(w) == 0; }
  __device__ __forceinline__ bool seg_last(int64_t w) const { return w + 1 == w1 || inner(w) == n_inner - 1; }
};
// CTA that owns work item w
__device__ __forceinline__ int cta_of(int64_t w, int64_t total) { return (int)(((w + 1) * gridDim.x - 1) / total); }

// Wave-synchronous partition for problems whose streamed operand does not fit the L2 (ce_tc_backward_ts_kernel).
// With the contiguous split above the G CTAs sit at G different positions of the streamed operand at any instant, so
// every streamed tile is fetched from HBM by almost every CTA that needs it (ncu, cfg3: 46 GB of DRAM reads for 0.3 GB
// of operands).  Here CTA c takes the WHOLE outer tiles c, c+G, c+2G, ... and walks the inner (streamed) index from 0
// in each of them: all CTAs stream the same tiles at the same time and the L2 serves G-1 of every G reads.
// The R = n_outer % G outer tiles of the last, partial wave are handled in one of two ways:
//  * streamed operand L2-resident (`stream_fits_l2`: cfg2, 10 MB): contiguous stream-K split of the R*n_inner pairs --
//    perfectly balanced, at most two segments (accumulator flushes) per CTA, and the re-reads are L2 hits anyway;
//  * otherwise: cut into p PARTS of the inner range each and handed out part-major, so the CTAs of a round work on at
//    most two different parts, i.e. they still walk the streamed operand in (two) lock-step fronts.  p minimises
//    rounds * (part length + SEG_OVH), SEG_OVH = the cost of one more segment (stationary-operand load + accumulator
//    flush through red.global) in inner-tile units.  (Round 1 split every partial wave stream-K style, which put every
//    CTA at its own inner position: at cfg3 the item-stationary dW kernel -- 95 of 391 outer tiles in the partial
//    wave -- read 8.2 GB from DRAM per launch for 0.26 GB of operands, ncu r2b.  A first version of the part-major
//    split without the overhead term cut cfg2's single partial wave into one-tile parts: 0.14 -> 0.39 ms.)
// Same interface as Share, over a CTA-local item index w in [w0 = 0, w1).
struct WaveShare {
  static constexpr int SEG_OVH = 4;
  int w0, w1, n_inner;
  int full_items;          // items of the full waves owned by this CTA = rounds * n_inner
  int tail_o0;             // first outer tile of the partial wave
  int R, L, n_units;       // part-major tail: outer tiles, inner tiles per part, work units = R * parts
  int t0;                  // stream-K tail: first (outer, inner) pair of this CTA's contiguous share
  bool sk;
  FastDiv fd, fdR;
  __device__ __forceinline__ int part_len(int part) const { return min(L, n_inner - part * L); }
  __device__ __forceinline__ WaveShare(int n_outer, int n_inner_, bool stream_fits_l2)
      : n_inner(n_inner_), sk(stream_fits_l2) {
    const int G = (int)gridDim.x, c = (int)blockIdx.x;
    const int rounds = n_outer / G;
    full_items = rounds * n_inner;
    tail_o0 = rounds * G;
    R = n_outer - tail_o0;
    L = n_inner;
    n_units = 0;
    t0 = 0;
    w0 = 0;
    w1 = full_items;
    fd.init((uint32_t)n_inner);
    fdR.init((uint32_t)(R > 0 ? R : 1));
    if (R > 0 && sk) {
      const int64_t tail_total = (int64_t)R * n_inner;
      t0 = (int)(tail_total * c / G);
      w1 += (int)(tail_total * (c + 1) / G) - t0;
    } else if (R > 0) {
      int best_p = 1;
      long long best_cost = -1;
      for (int p = 1; p <= 128 && p <= n_inner; ++p) {
        const int len = (n_inner + p - 1) / p;
        const int parts = (n_inner + len - 1) / len;
        const long long cost = (long long)((R * parts + G - 1) / G) * (len + SEG_OVH);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_p = p; }
      }
      L = (n_inner + best_p - 1) / best_p;
      const int parts = (n_inner + L - 1) / L;
      n_units = R * parts;
      for (int u = c; u < n_units; u += G) {
        uint32_t q, r;
        fdR.divmod((uint32_t)u, q, r);
        w1 += part_len((int)q);
      }
    }
  }
  // Position of one work item; every warp role walks its items in order with start() / advance(), which costs a few
  // integer operations per item (no division outside a change of work unit).
  struct Walk {
    int o, in;               // outer (stationary) tile, inner (streamed) tile
    bool first, last;        // first / last item of a segment (= one residency of the stationary operand)
    int w, u, i, len;        // item index; part-major tail: unit, position inside it, its length
  };
  __device__ __forceinline__ void unit_enter(Walk& k) const {
    uint32_t q, r;
    fdR.divmod((uint32_t)k.u, q, r);
    k.len = part_len((int)q);
    k.o = tail_o0 + (int)r;
    k.in = (int)q * L;
    k.i = 0;
  }
  __device__ __forceinline__ void tail_start(Walk& k) const {
    if (sk) {
      uint32_t q, r;
      fd.divmod((uint32_t)t0, q, r);
      k.o = tail_o0 + (int)q;
      k.in = (int)r;
      k.i = 0;                                 // the first segment may start mid-tile
    } else {
      k.u = (int)blockIdx.x;
      unit_enter(k);
    }
  }
  __device__ __forceinline__ void flags(Walk& k) const {
    if (k.w < full_items) { k.first = k.in == 0; k.last = k.in == n_inner - 1; }
    else if (sk)          { k.first = k.i == 0;  k.last = k.in == n_inner - 1; }
    else                  { k.first = k.i == 0;  k.last = k.i == k.len - 1; }
    k.last = k.last || (k.w + 1 == w1);
  }
  __device__ __forceinline__ void start(Walk& k) const {
    k.w = 0; k.u = 0; k.i = 0; k.len = 0; k.o = (int)blockIdx.x; k.in = 0;
    if (full_items == 0 && w1 > 0) tail_start(k);
    flags(k);
  }
  __device__ __forceinline__ void advance(Walk& k) const {
    ++k.w;
    if (k.w >= w1) return;
    if (k.w < full_items) {
      if (++k.in == n_inner) { k.in = 0; k.o += (int)gridDim.x; }
    } else if (k.w == full_items) {
      tail_start(k);
    } else if (sk) {
      ++k.i;
      if (++k.in == n_inner) { k.in = 0; ++k.o; k.i = 0; }
    } else {
      ++k.in;
      if (++k.i == k.len) { k.u += (int)gridDim.x; unit_enter(k); }
    }
    flags(k);
  }
};
using Walk = WaveShare::Walk;

// ================================================================================================================
// forward: per-row (max, sum-exp) partials of logits = A . Bt^T
//   A  = hout (optionally x dropout factors), [N, Hk] bf16 hi/lo     (tmA_*,  box 64 x 128)
//   Bt = W_out^T,                            [V, Hk] bf16 hi/lo     (tmB_*,  box 64 x 128)
// outer = token tile (A resident per segment), inner = item tile (Bt streamed in 64-wide K blocks, NS stages).
// Every segment writes one partial per 64-column half into ws[(slot*2 + half)][n], slot = position of the CTA among
// the CTAs sharing that token tile; slots a token tile does not use are filled with (-inf, 0).
// RANK: the same pass also counts, per token with target y = tgt[n] >= 0 (a GLOBAL item id; item v of this launch is
// id_offset + v), the items that precede y in the stable descending order of the logits against the exact reference
// logit ref[n]:  #{v != y : z_v > ref  or  (z_v == ref and id < y)}, added to rank[n] with one integer atomicAdd per
// (segment, half) -- integer sums, so the result does not depend on the order of the CTAs.
template <int KB, int NS, bool X3, bool BIAS, bool RANK>
__global__ void __launch_bounds__(TCF_THREADS, 1)
ce_tc_forward_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                     const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                     const float* __restrict__ b_out, float* __restrict__ ws_m, float* __restrict__ ws_s,
                     int64_t n_tokens, int v_begin, int v_end, int max_slots, const float* __restrict__ ref,
                     const int32_t* __restrict__ tgt, int id_offset, int32_t* __restrict__ rank) {
  constexpr int NP = X3 ? 2 : 1;  // operand parts (hi, lo)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = base;                                  // [NP][KB][TILE_B]
  const uint32_t sB = sA + NP * KB * TILE_B;                 // [NS][NP][TILE_B]
  const uint32_t sBar = sB + NS * NP * TILE_B;               // barriers
  // Two MMA-issuing warps take alternate tiles (warp 1 the even ones into logits buffer 0, warp 2 the odd ones into
  // buffer 1): while one warp sits in the waits / fences / commits between two of its tiles, the other has MMAs queued,
  // so the tensor pipe no longer drains once per tile (tile period 2330 -> ~1600 cycles for 1536 of MMA at Hk = 128).
  // Each ring slot has one full barrier PER ISSUING WARP (a warp must never take the other's completion for its own:
  // parity aliasing) and one "token tile no longer read" barrier per issuing warp, committed exactly once per segment
  // (tcgen05.commit also when the warp owns no tile of a one-tile segment: commit arrivals of one thread complete in
  // order, a plain arrive could overtake the commit of the previous segment).
  const uint32_t bar_full = sBar, bar_empty = sBar + 16 * NS, bar_tfull = sBar + 24 * NS,
                 bar_tempty = bar_tfull + 16, bar_a = bar_tempty + 16, bar_afree = bar_a + 8,   // afree: one per MMA warp
                 tmem_slot = bar_afree + 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_vtiles = (v_end - v_begin + BN - 1) / BN;
  const int64_t total = ((n_tokens + BM - 1) / BM) * n_vtiles;
  const Share sh(total, n_vtiles);

  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      ptx::mbar_init(bar_full + 8 * i, 1);                   // even tiles (warp 1)
      ptx::mbar_init(bar_full + 8 * (NS + i), 1);            // odd tiles  (warp 2)
      ptx::mbar_init(bar_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(bar_tfull + 8 * i, 1); ptx::mbar_init(bar_tempty + 8 * i, N_EPI_WARPS); }
    ptx::mbar_init(bar_a, 1);
    ptx::mbar_init(bar_afree, 1);
    ptx::mbar_init(bar_afree + 8, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 256);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------- TMA producer
    {
      if (lane == 0) { ptx::prefetch_tmap(&tmA_hi); ptx::prefetch_tmap(&tmB_hi); }
      Pipe p;
      int seg = 0;
      for (int64_t w = sh.w0; w < sh.w1; ++w) {
        if (sh.seg_first(w)) {
          if (seg > 0) {                                           // the previous segment's MMAs have read sA
            ptx::mbar_wait(bar_afree, (seg - 1) & 1);
            ptx::mbar_wait(bar_afree + 8, (seg - 1) & 1);
          }
          const int row0 = sh.outer(w) * BM;
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(bar_a, NP * KB * TILE_B);
            for (int kb = 0; kb < KB; ++kb) {
              ptx::tma_load_2d(sA + kb * TILE_B, &tmA_hi, bar_a, kb * KBLK, row0);
              if (X3) ptx::tma_load_2d(sA + (KB + kb) * TILE_B, &tmA_lo, bar_a, kb * KBLK, row0);
            }
          }
          ++seg;
        }
        const int v0 = v_begin + sh.inner(w) * BN;
        const int owner = (int)(w - sh.w0) & 1;
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(bar_empty + 8 * p.stage, p.phase ^ 1);
          if (ptx::elect_one()) {
            const uint32_t fb = bar_full + 8 * (owner * NS + p.stage);
            ptx::mbar_arrive_expect_tx(fb, NP * TILE_B);
            const uint32_t dst = sB + p.stage * NP * TILE_B;
            ptx::tma_load_2d(dst, &tmB_hi, fb, kb * KBLK, v0);
            if (X3) ptx::tma_load_2d(dst + TILE_B, &tmB_lo, fb, kb * KBLK, v0);
          }
          p.advance(NS);
        }
      }
    }
  } else if (warp <= 2) {
    // ------------------------------------------------------------------------------------------- MMA issuers
    {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(BM, BN);
      const int me = warp - 1;                               // 0: even tiles, 1: odd tiles
      const uint32_t my_full = bar_full + 8 * (me * NS);
      Pipe p;
      uint32_t bits = 0;                                     // parity of MY full barrier, per slot
      int seg = -1, tc = 0;
      for (int64_t w = sh.w0; w < sh.w1; ++w, ++tc) {
        const bool first = sh.seg_first(w), last = sh.seg_last(w);
        if (first) ++seg;
        if ((tc & 1) != me) {                                // the other warp's tile: only keep the ring position
          for (int kb = 0; kb < KB; ++kb) p.advance(NS);
          if (first && last) commit_elect(bar_afree + 8 * me);   // a one-tile segment I have no part in
          continue;
        }
        // my first tile of this segment: the token tile must have landed
        if (first || (w > sh.w0 && sh.seg_first(w - 1))) {
          ptx::mbar_wait(bar_a, seg & 1);
          ptx::tc_fence_after_sync();
        }
        const int buf = me;
        ptx::mbar_wait(bar_tempty + 8 * buf, ((tc >> 1) & 1) ^ 1);
        ptx::tc_fence_after_sync();
        const uint32_t d = tmem_base + buf * BN;
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(my_full + 8 * p.stage, (bits >> p.stage) & 1u);
          bits ^= 1u << p.stage;
          ptx::tc_fence_after_sync();
          const uint32_t b = sB + p.stage * NP * TILE_B;
          mma_kblock<X3>(d, sA + kb * TILE_B, sA + (KB + kb) * TILE_B, b, b + TILE_B, idesc, kb == 0);
          commit_elect(bar_empty + 8 * p.stage);
          p.advance(NS);
        }
        commit_elect(bar_tfull + 8 * buf);
        // my last tile of this segment (the segment's last tile, or the one before it): sA is no longer read by me
        if (last || (w + 1 < sh.w1 && sh.seg_last(w + 1))) commit_elect(bar_afree + 8 * me);
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------- epilogue
    const int q = warp & 3;                      // TMEM lane quadrant this warp may read
    const int half = (warp - 3) >> 2;            // which 64-column half of the tile this warp owns
    const int row = q * 32 + lane;
    float m = -INFINITY, s = 0.f;
    float rz = 0.f, rz_below = 0.f;              // RANK: reference logit and the float just below it
    int32_t ry = -1, cnt = 0;                    // RANK: target (global id, -1 = no rank) and the running count
    int tc = 0;
    for (int64_t w = sh.w0; w < sh.w1; ++w, ++tc) {
      const int buf = tc & 1;
      const int tt = sh.outer(w), vt = sh.inner(w);
      if (sh.seg_first(w)) {
        m = -INFINITY; s = 0.f;
        if (RANK) {
          const int64_t n = (int64_t)tt * BM + row;
          ry = n < n_tokens ? tgt[n] : -1;
          rz = ry >= 0 ? ref[n] : 0.f;
          rz_below = nextafterf(rz, -INFINITY);
          cnt = 0;
        }
      }
      const int vc0 = v_begin + vt * BN + half * 64;             // first item of this warp's columns
      ptx::mbar_wait(bar_tfull + 8 * buf, (tc >> 1) & 1);
      ptx::tc_fence_after_sync();
      float z[64];
      load_half_tile(tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN + half * 64, z);
      ptx::tc_fence_before_sync();               // accumulator read: hand the TMEM buffer back to the MMA warp
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar_tempty + 8 * buf);
      if (BIAS || vc0 + 64 > v_end) {            // warp-uniform slow path: output bias and the ragged last tile
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const int v = vc0 + j;
          if (v < v_end) { if (BIAS) z[j] += __ldg(b_out + v); }
          else z[j] = -INFINITY;
        }
      }
      if (RANK && ry >= 0) {
        // Columns wholly below the target id count z >= ref, i.e. z > (the float below ref); columns wholly above it
        // count z > ref: ONE compare per logit.  Only the 64 columns that hold the target itself (64/V of the column
        // blocks of a row) take the per-column tie rule, which also leaves the target out.  Columns past v_end are
        // -inf and never count.
        const int tl = ry - (id_offset + vc0);   // target column inside this warp's 64 (may lie outside)
        int c4[4] = {0, 0, 0, 0};
        if (tl < 0 || tl >= 64) {
          const float thr = tl >= 64 ? rz_below : rz;
#pragma unroll
          for (int j = 0; j < 64; j += 4) {
            c4[0] += z[j] > thr; c4[1] += z[j + 1] > thr; c4[2] += z[j + 2] > thr; c4[3] += z[j + 3] > thr;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 64; ++j) c4[j & 3] += (j != tl) && (z[j] > rz || (z[j] == rz && j < tl));
        }
        cnt += (c4[0] + c4[1]) + (c4[2] + c4[3]);
      }
      float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int j = 0; j < 64; j += 4) {
        mx[0] = fmaxf(mx[0], z[j]); mx[1] = fmaxf(mx[1], z[j + 1]);
        mx[2] = fmaxf(mx[2], z[j + 2]); mx[3] = fmaxf(mx[3], z[j + 3]);
      }
      const float cmax = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
      if (cmax > -INFINITY) {
        const float mn = fmaxf(m, cmax);
        const float nb = -mn * LOG2E;
        float add[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 64; j += 4) {
          add[0] += ptx::ex2_approx(fmaf(z[j], LOG2E, nb));
          add[1] += ptx::ex2_approx(fmaf(z[j + 1], LOG2E, nb));
          add[2] += ptx::ex2_approx(fmaf(z[j + 2], LOG2E, nb));
          add[3] += ptx::ex2_approx(fmaf(z[j + 3], LOG2E, nb));
        }
        s = s * ptx::ex2_approx(fmaf(m, LOG2E, nb)) + ((add[0] + add[1]) + (add[2] + add[3]));
        m = mn;
      }
      if (sh.seg_last(w)) {
        // one partial of the vocabulary reduction per (slot, half), merged by seqrec_ce_finalize
        const int64_t n = (int64_t)tt * BM + row;
        if (RANK && ry >= 0 && cnt > 0) atomicAdd(rank + n, cnt);
        if (n < n_tokens) {
          const int slot = (int)blockIdx.x - cta_of((int64_t)tt * n_vtiles, total);
          ws_m[((int64_t)slot * 2 + half) * n_tokens + n] = m;
          ws_s[((int64_t)slot * 2 + half) * n_tokens + n] = s;
          if (vt == n_vtiles - 1) {              // last CTA of this token tile: blank the slots nobody writes
            for (int k = slot + 1; k < max_slots; ++k) {
              ws_m[((int64_t)k * 2 + half) * n_tokens + n] = -INFINITY;
              ws_s[((int64_t)k * 2 + half) * n_tokens + n] = 0.f;
            }
          }
        }
      }
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, 256);
  }
}

// 16 consecutive 32-bit columns, registers -> TMEM (thread i writes lane base + i)
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}

// this thread's row of a K-major bf16 matrix (global memory, leading dimension ld elements), K elements
// [k0, k0 + 32*nchunks) -> packed pairs in TMEM columns [tcol, tcol + 16*nchunks): the A-operand image of a TS-mode MMA
__device__ __forceinline__ void row_to_tmem(uint32_t tcol, const uint16_t* __restrict__ src, int64_t row, int ld,
                                            int k0, int nchunks, bool row_ok) {
  for (int c = 0; c < nchunks; ++c) {
    uint32_t v[16];
    if (row_ok) {
      const uint4* g = reinterpret_cast<const uint4*>(src + row * ld + k0 + c * 32);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint4 t = __ldg(g + i);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0u;
    }
    tmem_st_32x16(tcol + 16 * c, v);
  }
}

// ================================================================================================================
// K9 on the tensor cores: top-k next items per token row, never materialising the (N,V) logits.
// Same MMA pipeline as ce_tc_forward_atm_kernel (token tile in TMEM, W_out^T streamed by TMA); the epilogue thread that
// owns (row, 64-column half) keeps a private, descending top-k list in shared memory ([k][thread] -> conflict free)
// and a register threshold = its current k-th value.  A 64-column slab is skipped after ONE comparison of its maximum
// with the threshold; an insertion is rare (k.ln(n/k) per stream).  Items reach a thread in ascending id order and an
// insertion goes BEHIND equal values, so ties are won by the lower item id (the stable-argsort order of the oracle).
// Every (token tile, CTA, half) stream leaves one list; topk_merge_kernel merges the lists of a row.
constexpr int TOPK_MAX = 32;

__device__ __noinline__ float topk_insert(float* lv, int32_t* li, int k, float z, int32_t id) {
  int i = k - 1;
  while (i > 0 && lv[(i - 1) * 256] < z) {
    lv[i * 256] = lv[(i - 1) * 256];
    li[i * 256] = li[(i - 1) * 256];
    --i;
  }
  lv[i * 256] = z;
  li[i * 256] = id;
  return lv[(k - 1) * 256];
}

template <int KB, int NS, bool X3, bool BIAS>
__global__ void __launch_bounds__(TC_THREADS, 1)
ce_tc_topk_kernel(const uint16_t* __restrict__ A_hi, const uint16_t* __restrict__ A_lo,
                  const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                  const float* __restrict__ b_out, float* __restrict__ cand_v, int32_t* __restrict__ cand_i,
                  int64_t n_tokens, int v_begin, int v_end, int max_slots, int k) {
  constexpr int NP = X3 ? 2 : 1;
  constexpr int HK = KB * KBLK;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sB = base;                                  // [NS][NP][TILE_B]
  const uint32_t sL = sB + NS * NP * TILE_B;                 // lists: values [TOPK_MAX][256], ids [TOPK_MAX][256]
  const uint32_t sBar = sL + 2 * TOPK_MAX * 256 * 4;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * NS, bar_tfull = sBar + 16 * NS,
                 bar_tempty = bar_tfull + 16, bar_a = bar_tempty + 16, bar_afree = bar_a + 8,
                 tmem_slot = bar_afree + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_vtiles = (v_end - v_begin + BN - 1) / BN;
  const int64_t total = ((n_tokens + BM - 1) / BM) * n_vtiles;
  const Share sh(total, n_vtiles);

  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) { ptx::mbar_init(bar_full + 8 * i, 1); ptx::mbar_init(bar_empty + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(bar_tfull + 8 * i, 1); ptx::mbar_init(bar_tempty + 8 * i, N_EPI_WARPS); }
    ptx::mbar_init(bar_a, N_EPI_WARPS);
    ptx::mbar_init(bar_afree, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const uint32_t tmem_a = tmem_base + 2 * BN;

  if (warp == 0) {
    if (lane == 0) ptx::prefetch_tmap(&tmB_hi);
    Pipe p;
    for (int64_t w = sh.w0; w < sh.w1; ++w) {
      const int v0 = v_begin + sh.inner(w) * BN;
      for (int kb = 0; kb < KB; ++kb) {
        ptx::mbar_wait(bar_empty + 8 * p.stage, p.phase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(bar_full + 8 * p.stage, NP * TILE_B);
          const uint32_t dst = sB + p.stage * NP * TILE_B;
          ptx::tma_load_2d(dst, &tmB_hi, bar_full + 8 * p.stage, kb * KBLK, v0);
          if (X3) ptx::tma_load_2d(dst + TILE_B, &tmB_lo, bar_full + 8 * p.stage, kb * KBLK, v0);
        }
        p.advance(NS);
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = ptx::umma_idesc_bf16(BM, BN);
    Pipe p;
    int seg = -1, tc = 0;
    for (int64_t w = sh.w0; w < sh.w1; ++w, ++tc) {
      if (sh.seg_first(w)) {
        ++seg;
        ptx::mbar_wait(bar_a, seg & 1);
        ptx::tc_fence_after_sync();
      }
      const int buf = tc & 1;
      ptx::mbar_wait(bar_tempty + 8 * buf, ((tc >> 1) & 1) ^ 1);
      ptx::tc_fence_after_sync();
      const uint32_t d = tmem_base + buf * BN;
      for (int kb = 0; kb < KB; ++kb) {
        ptx::mbar_wait(bar_full + 8 * p.stage, p.phase);
        ptx::tc_fence_after_sync();
        const uint32_t b = sB + p.stage * NP * TILE_B;
        const uint64_t db_hi = ptx::umma_desc_k_sw128(b), db_lo = ptx::umma_desc_k_sw128(b + TILE_B);
        if (ptx::elect_one()) {
#pragma unroll
          for (int kk = 0; kk < KBLK / 16; ++kk) {
            const uint32_t a_hi = tmem_a + kb * (KBLK / 2) + kk * 8, a_lo = a_hi + HK / 2;
            const uint32_t acc = (kb == 0 && kk == 0) ? 0u : 1u;
            if (X3) {
              ptx::umma_bf16_ts(d, a_hi, ptx::umma_desc_advance_k(db_lo, kk * 16), idesc, acc);
              ptx::umma_bf16_ts(d, a_lo, ptx::umma_desc_advance_k(db_hi, kk * 16), idesc, 1u);
              ptx::umma_bf16_ts(d, a_hi, ptx::umma_desc_advance_k(db_hi, kk * 16), idesc, 1u);
            } else {
              ptx::umma_bf16_ts(d, a_hi, ptx::umma_desc_advance_k(db_hi, kk * 16), idesc, acc);
            }
          }
        }
        __syncwarp();
        commit_elect(bar_empty + 8 * p.stage);
        p.advance(NS);
      }
      commit_elect(bar_tfull + 8 * buf);
      if (sh.seg_last(w)) commit_elect(bar_afree);
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const int e = threadIdx.x - 64;                          // 0..255
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    float* lv = reinterpret_cast<float*>(smem_raw + (sL - ptx::smem_u32(smem_raw))) + e;
    int32_t* li = reinterpret_cast<int32_t*>(smem_raw + (sL - ptx::smem_u32(smem_raw))) + TOPK_MAX * 256 + e;
    float thr = -INFINITY;
    int tc = 0, seg = -1;
    for (int64_t w = sh.w0; w < sh.w1; ++w, ++tc) {
      const int buf = tc & 1;
      const int tt = sh.outer(w), vt = sh.inner(w);
      if (sh.seg_first(w)) {
        ++seg;
        for (int j = 0; j < k; ++j) { lv[j * 256] = -INFINITY; li[j * 256] = 0x7fffffff; }
        thr = -INFINITY;
        if (seg > 0) {
          ptx::mbar_wait(bar_afree, (seg - 1) & 1);
          ptx::tc_fence_after_sync();
        }
        const int64_t n = (int64_t)tt * BM + row;
        row_to_tmem(tmem_a + lane_off + half * (HK / 4), A_hi, n, HK, half * (HK / 2), HK / 64, n < n_tokens);
        if (X3)
          row_to_tmem(tmem_a + lane_off + HK / 2 + half * (HK / 4), A_lo, n, HK, half * (HK / 2), HK / 64,
                      n < n_tokens);
        ptx::tmem_st_wait();
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar_a);
      }
      const int vc0 = v_begin + vt * BN + half * 64;
      ptx::mbar_wait(bar_tfull + 8 * buf, (tc >> 1) & 1);
      ptx::tc_fence_after_sync();
      float z[64];
      load_half_tile(tmem_base + lane_off + buf * BN + half * 64, z);
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar_tempty + 8 * buf);
      if (BIAS || vc0 + 64 > v_end) {
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const int v = vc0 + j;
          if (v < v_end) { if (BIAS) z[j] += __ldg(b_out + v); }
          else z[j] = -INFINITY;
        }
      }
      float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int j = 0; j < 64; j += 4) {
        mx[0] = fmaxf(mx[0], z[j]); mx[1] = fmaxf(mx[1], z[j + 1]);
        mx[2] = fmaxf(mx[2], z[j + 2]); mx[3] = fmaxf(mx[3], z[j + 3]);
      }
      if (fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) > thr) {     // rare after the first tiles
#pragma unroll
        for (int j = 0; j < 64; ++j)
          if (z[j] > thr) thr = topk_insert(lv, li, k, z[j], vc0 + j);
      }
      if (sh.seg_last(w)) {
        const int64_t n = (int64_t)tt * BM + row;
        if (n < n_tokens) {
          const int slot = (int)blockIdx.x - cta_of((int64_t)tt * n_vtiles, total);
          const int64_t o = (((int64_t)slot * 2 + half) * n_tokens + n) * k;
          for (int j = 0; j < k; ++j) { cand_v[o + j] = lv[j * 256]; cand_i[o + j] = li[j * 256]; }
          if (vt == n_vtiles - 1) {                          // last CTA of this token tile: blank the unused slots
            for (int sl = slot + 1; sl < max_slots; ++sl) {
              const int64_t ob = (((int64_t)sl * 2 + half) * n_tokens + n) * k;
              for (int j = 0; j < k; ++j) { cand_v[ob + j] = -INFINITY; cand_i[ob + j] = 0x7fffffff; }
            }
          }
        }
      }
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// one warp per row: k rounds of (value descending, id ascending) selection over the row's n_lists * k candidates
__global__ void __launch_bounds__(256)
topk_merge_kernel(const float* __restrict__ cand_v, const int32_t* __restrict__ cand_i, int n_lists,
                  int64_t list_stride, const float* __restrict__ mrow, const float* __restrict__ srow,
                  int32_t* __restrict__ topk_ids, float* __restrict__ topk_p, int64_t n_rows, int k) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (n >= n_rows) return;
  const int total = n_lists * k;
  constexpr int PER = 12;                                    // candidates per lane (n_lists * k <= 384)
  float v[PER];
  int32_t id[PER];
#pragma unroll
  for (int c = 0; c < PER; ++c) {
    const int x = c * 32 + lane;
    v[c] = -INFINITY; id[c] = 0x7fffffff;
    if (x < total) {
      const int64_t o = (int64_t)(x / k) * list_stride + n * k + (x % k);
      v[c] = cand_v[o]; id[c] = cand_i[o];
    }
  }
  for (int j = 0; j < k; ++j) {
    float bv = -INFINITY;
    int32_t bi = 0x7fffffff;
#pragma unroll
    for (int c = 0; c < PER; ++c)
      if (v[c] > bv || (v[c] == bv && id[c] < bi)) { bv = v[c]; bi = id[c]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int32_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
#pragma unroll
    for (int c = 0; c < PER; ++c)
      if (id[c] == bi) { v[c] = -INFINITY; id[c] = 0x7fffffff; }   // ids are unique across the lists
    if (lane == 0) {
      topk_ids[n * k + j] = bi;
      if (topk_p) topk_p[n * k + j] = (mrow && srow) ? expf(bv - mrow[n]) / srow[n] : bv;
    }
  }
}

// flush a [128 x ncols] fp32 TMEM accumulator slice owned by this warp (32 rows x `ncols` columns starting at
// column col0) into global memory with vector reductions: dst_row points at this thread's row, column col0
__device__ __forceinline__ void flush_acc_red(uint32_t taddr, int ncols, float* dst_row, int valid_cols, bool row_ok,
                                              bool vec_ok, const float* scale_row) {
#pragma unroll 1
  for (int c = 0; c < ncols; c += 32) {
    uint32_t r[32];
    ptx::tmem_ld_32x32(taddr + c, r);
    ptx::tmem_ld_wait();
    if (!row_ok) continue;
    const int valid = min(32, valid_cols - c);
    if (scale_row) {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < valid) r[j] = __float_as_uint(__uint_as_float(r[j]) * scale_row[c + j]);
    }
    if (vec_ok && valid == 32) {
#pragma unroll
      for (int g = 0; g < 8; ++g)
        red_add_f4(dst_row + c + 4 * g, make_float4(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1]),
                                                    __uint_as_float(r[4 * g + 2]), __uint_as_float(r[4 * g + 3])));
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < valid) atomicAdd(dst_row + c + j, __uint_as_float(r[j]));
    }
  }
}

// ================================================================================================================
// backward for wide hidden layers (Hk up to 256), ONE kernel template for both gradients.
//   P = the stationary side (128 rows per tile), Q = the streamed side (128 rows per tile):
//     ITEM_ST = false: P = tokens, Q = items   ->  out = dh     [n, h] += sum_v dS[n, v] . W_out[h, v]
//     ITEM_ST = true : P = items,  Q = tokens  ->  out = dW_out [h, v] += sum_n dS^T[v, n] . hs[n, h]
//   X = stationary operand [P_total, Hk] (A | Bt), resident in shared memory for a whole segment
//   Y = streamed operand of the logits GEMM [Q_total, Hk] (Bt | A):    S[P, Q] = X . Y^T   (M=128, N=128, K=Hk)
//   Z = K-major operand of the second GEMM [Hk, Q_total] (W | Ht):     acc[P, Hk] += dS[P, Q] . Z^T
// The epilogue turns S into dS (rows = lanes = P) and tcgen05.st's it as packed bf16 hi/lo into TENSOR MEMORY, where
// it is the A operand of the second GEMM (TS-mode MMA) -- dS never occupies shared memory, which is what makes
// Hk = 256 fit: 128 KB resident X (x3) + 3 stages of 32 KB.  TMEM: S (double buffered only when Hk <= 128) |
// accumulator (128-column chunks of the hidden axis) | dS hi | dS lo = 512 columns.
// In the item-stationary variant the per-token softmax terms vary along the COLUMNS of the tile: the epilogue warps
// stage {-m.log2e, coef/s, coef, target} of the tile's 128 tokens in shared memory and read them as broadcasts.
template <int KB, bool X3>
struct TsCfg {
  static constexpr int NP = X3 ? 2 : 1;
  static constexpr int NS_RAW = (224 * 1024 - NP * KB * TILE_B) / (NP * TILE_B);
  static constexpr int HK = KB * KBLK;
  static constexpr int NC = (HK + 127) / 128;               // 128-wide hidden chunks of the second GEMM
  // Two MMA-issuing warps: logits GEMMs on warp 1, gradient GEMMs on warp 2, both fed from ONE shared-memory ring.
  // Each ring slot has TWO full barriers, one per kind of block (Y block for the logits GEMM, Z block for the gradient
  // GEMM), so that every barrier has a single waiting warp in lock-step with it; a consumer tracks the parity of ITS
  // barrier per slot in a bit mask.  (With one barrier per slot the two warps alias on the phase parity: the warp that
  // runs ahead takes a completion that belonged to the other warp for its own.)
  static constexpr int NS = (KB <= 2) ? (KB + 2 * NC) : (NS_RAW > 8 ? 8 : NS_RAW);   // Hk <= 128: ring length = period
  static constexpr int THREADS = 352;
  static constexpr int EPI0 = 3;                            // first epilogue warp
  static constexpr int ACC_COLS = NC * 128;
  static constexpr int SBUF = (2 * BN + ACC_COLS + BN <= 512) ? 2 : 1;
  static constexpr uint32_t TERMS_B = 128 * 16;             // per-token terms of one streamed tile (ITEM_ST)
  static constexpr uint32_t SMEM_NEED = NP * KB * TILE_B + NS * NP * TILE_B + TERMS_B + 384;
};

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// MODE selects the variant: TS_DH / TS_DW as described above, and
//   TS_FUSED (token-stationary): forward statistics AND dH from ONE logits pass.  The softmax is evaluated against a
//   per-row REFERENCE logit instead of the row maximum: ref[n] = the target logit zy[n] (exact fp32, computed before this
//   kernel).  exp(z - ref) needs no running maximum (ref is one of the row's logits, so max - ref >= 0 and the sum is
//   >= ~1; fp32 -- and the bf16 hi/lo operand -- carry 8 exponent bits, so values up to e^88 lose no relative
//   precision), hence no accumulator rescale and no per-CTA partial states: every CTA that shares a token tile
//   accumulates  acc[n,:] += sum_v exp(z[n,v] - ref[n]) . W_out[:,v]  and  s[n] += sum_v exp(z[n,v] - ref[n])  against
//   the SAME reference, and both leave through reductions.  seqrec_ce_finalize (splits = 1, m = ref) and
//   seqrec_ce_dh_finish then give the loss, the clip coefficient and  dh = coef . (acc / s - W_out[:, target]).
//   Rows whose target sits more than ~88 nats below the maximum overflow to s = inf: p(target) = 0 is then clipped,
//   the clip passes no gradient (coef = 0) and the finish kernel writes zeros -- the reference's result.
enum { TS_DH = 0, TS_DW = 1, TS_FUSED = 2 };

// Front throttle of the full waves.  WaveShare starts all CTAs on the same streamed tile, but nothing keeps them
// together: over the 7813 item tiles of cfg4 the faster SMs run hundreds of tiles ahead -- further than the L2 reaches
// back (ncu: 36 GB of DRAM reads per launch for 1 GB of W_out^T, L2 hit rate 88 %, tensor pipe 75 % active against 86 %
// at cfg3, whose W_out stays L2-resident).  The producer warp therefore counts the CTAs that have STARTED each chunk
// of TS_CHUNK streamed tiles and does not start chunk c before every CTA has started chunk c - TS_AHEAD: the front of
// the grid stays within TS_AHEAD+1 chunks (24 MB at Hk = 256).  It is a throttle, not a barrier: correctness never
// depends on it and every wait is bounded (a CTA that has waited ~100 us goes on alone), so a co-scheduled kernel
// holding an SM cannot hang the grid.  One counter array per variant (cleared by a memset node in front of the launch).
constexpr int TS_CHUNK = 32, TS_AHEAD = 2, TS_SYNC_SLOTS = 8192;
__device__ int g_ts_sync[3][TS_SYNC_SLOTS];
// experiment switch (SEQREC_ZMN = 1: never / 2: always the MN-major form of the second GEMM's operand; 0 = by size)
__device__ int g_ts_zmn_mode = 0;

template <int KB, bool X3, int MODE>
__global__ void __launch_bounds__(352, 1)
ce_tc_backward_ts_kernel(const __grid_constant__ CUtensorMap tmX_hi, const __grid_constant__ CUtensorMap tmX_lo,
                         const __grid_constant__ CUtensorMap tmY_hi, const __grid_constant__ CUtensorMap tmY_lo,
                         const __grid_constant__ CUtensorMap tmZ_hi, const __grid_constant__ CUtensorMap tmZ_lo,
                         const int32_t* __restrict__ tgt, const float* __restrict__ mrow,
                         const float* __restrict__ srow, const float* __restrict__ coef,
                         const float* __restrict__ inv_nvalid, const float* __restrict__ hscale,
                         float* __restrict__ out, int64_t n_tokens, int H, int v_begin, int v_end, int ldw,
                         uint32_t smem_bytes, const float* __restrict__ b_out, float* __restrict__ db_out,
                         const uint8_t* __restrict__ tok_mask, float* __restrict__ s_out,
                         const int32_t* __restrict__ n_tokens_dev) {
  // compacted token axis: the number of (valid) tokens is only known on the device; the argument is then the upper bound
  // the TMA descriptors were built for
  if (n_tokens_dev) n_tokens = min(n_tokens, (int64_t)n_tokens_dev[0]);
  constexpr bool ITEM_ST = MODE == TS_DW;
  constexpr bool FUSED = MODE == TS_FUSED;
  using C = TsCfg<KB, X3>;
  constexpr int NP = C::NP, NS = C::NS, NC = C::NC, SBUF = C::SBUF;
  constexpr int NJ = BN / KBLK;                             // 64-wide K blocks of the second GEMM per tile
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sX = base;                                  // [NP][KB][TILE_B]   stationary operand
  const uint32_t sB = sX + NP * KB * TILE_B;                 // [NS][NP][TILE_B]   Y / Z blocks
  const uint32_t sT = sB + NS * NP * TILE_B;                 // float4[128]        per-token terms (ITEM_ST)
  const uint32_t sBar = sT + C::TERMS_B;
  const uint32_t bar_full = sBar, bar_empty = sBar + 8 * NS, bar_tfull = sBar + 16 * NS,
                 bar_tempty = bar_tfull + 16, bar_a = bar_tempty + 16, bar_afree = bar_a + 8,
                 bar_dfull = bar_afree + 8, bar_dempty = bar_dfull + 8, bar_hfull = bar_dempty + 8,
                 bar_hempty = bar_hfull + 8, tmem_slot = bar_hempty + 8, bar_fullz = tmem_slot + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0 && base - ptx::smem_u32(smem_raw) + C::SMEM_NEED > smem_bytes) {
    printf("seqrec_b200: ce_tc_backward_ts shared-memory layout does not fit (%u needed)\n", C::SMEM_NEED);
    __trap();
  }
  const int n_vtiles = (v_end - v_begin + BN - 1) / BN;
  const int n_ttiles = (int)((n_tokens + BM - 1) / BM);
  // both streamed operands (Y and Z blocks, hi and lo) of one pass over the inner axis: L2-resident below 32 MB
  const int n_inner_tiles = ITEM_ST ? n_ttiles : n_vtiles;
  const bool stream_fits_l2 = (int64_t)n_inner_tiles * (2 * NP * KB * TILE_B) <= (32ll << 20);
  const WaveShare sh(ITEM_ST ? n_vtiles : n_ttiles, n_inner_tiles, stream_fits_l2);
  // Blocks of the second GEMM's streamed operand per tile.  Item-stationary: [128 hidden x 64 tokens] blocks of H^T.
  // Token-stationary, two forms:
  //  * K-major [128 hidden x 64 items] blocks of W_out (Hk x V), N = 128 per MMA -- the faster form while W_out stays
  //    in the L2 (cfg2, cfg3), but its 128 rows lie V*2 bytes apart: at V = 1M that is one 2 MB page and one DRAM row
  //    per 128-byte piece, and the kernel ran 22 % slower per unit of work than at V = 50k;
  //  * z_mn: the SAME [128 items x 64 hidden] blocks of W_out^T that fed the logits GEMM, fetched a second time (an L2
  //    hit on lines loaded microseconds earlier) and read as an MN-MAJOR operand (N = 64 hidden units along the
  //    128-byte rows, K = the 128 items down the rows).  Twice the MMAs at half the width: 11 % slower at cfg3, 8 %
  //    faster at cfg4 -- taken when the streamed operand is far beyond the L2 (> 160 MB).
  const int chunks_per_round = (n_inner_tiles + TS_CHUNK - 1) / TS_CHUNK;
  const bool throttle = !stream_fits_l2 && sh.full_items > 0 &&
                        (int64_t)(sh.full_items / n_inner_tiles) * chunks_per_round <= TS_SYNC_SLOTS;
  const bool z_mn = !ITEM_ST && (g_ts_zmn_mode == 2 ||
                                 (g_ts_zmn_mode == 0 && (int64_t)n_inner_tiles * (2 * NP * KB * TILE_B) > (160ll << 20)));
  const int NZ = z_mn ? KB : NJ * NC;
  // first row of the stationary / streamed operand of work item w
  auto p_row0 = [&](const Walk& k) { return ITEM_ST ? v_begin + k.o * BN : k.o * BM; };
  auto q_row0 = [&](const Walk& k) { return ITEM_ST ? k.in * BM : v_begin + k.in * BN; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      ptx::mbar_init(bar_full + 8 * i, 1);
      ptx::mbar_init(bar_fullz + 8 * i, 1);
      ptx::mbar_init(bar_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(bar_tfull + 8 * i, 1); ptx::mbar_init(bar_tempty + 8 * i, N_EPI_WARPS); }
    ptx::mbar_init(bar_a, 1);
    ptx::mbar_init(bar_afree, 1);
    ptx::mbar_init(bar_dfull, N_EPI_WARPS);
    ptx::mbar_init(bar_dempty, 1);
    ptx::mbar_init(bar_hfull, 1);
    ptx::mbar_init(bar_hempty, N_EPI_WARPS);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const uint32_t tmem_acc = tmem_base + SBUF * BN;
  const uint32_t tmem_ds = tmem_acc + C::ACC_COLS;           // 64 packed columns hi, then 64 lo

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------- TMA producer
    // stage order = the MMA warp's consumption order: Y(w0), then per work item w: Y(w+1), Z(w)
    if (sh.w0 < sh.w1) {
      if (lane == 0) { ptx::prefetch_tmap(&tmX_hi); ptx::prefetch_tmap(&tmY_hi); ptx::prefetch_tmap(&tmZ_hi); }
      Pipe p;
      int seg = 0;
      bool gave_up = false;                                 // front throttle: this CTA has timed out once
      auto load_s_operands = [&](const Walk& k) {
        if (k.first) {
          if (seg > 0) ptx::mbar_wait(bar_afree, (seg - 1) & 1);
          const int row0 = p_row0(k);
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(bar_a, NP * KB * TILE_B);
            for (int kb = 0; kb < KB; ++kb) {
              ptx::tma_load_2d(sX + kb * TILE_B, &tmX_hi, bar_a, kb * KBLK, row0);
              if (X3) ptx::tma_load_2d(sX + (KB + kb) * TILE_B, &tmX_lo, bar_a, kb * KBLK, row0);
            }
          }
          ++seg;
        }
        const int q0 = q_row0(k);
        if (throttle && k.w < sh.full_items && (k.in % TS_CHUNK) == 0) {
          const int chunk = (k.w / sh.n_inner) * chunks_per_round + k.in / TS_CHUNK;
          if (lane == 0) {
            int* cnt = g_ts_sync[MODE];
            atomicAdd(cnt + chunk, 1);
            if (chunk >= TS_AHEAD && !gave_up) {
              const volatile int* behind = cnt + (chunk - TS_AHEAD);
              const long long t0 = clock64();
              while (*behind < (int)gridDim.x) {
                if (clock64() - t0 > 200000ll) { gave_up = true; break; }   // ~100 us: go on alone from here
                __nanosleep(256);
              }
            }
          }
          __syncwarp();
        }
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(bar_empty + 8 * p.stage, p.phase ^ 1);
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(bar_full + 8 * p.stage, NP * TILE_B);
            const uint32_t dst = sB + p.stage * NP * TILE_B;
            ptx::tma_load_2d(dst, &tmY_hi, bar_full + 8 * p.stage, kb * KBLK, q0);
            if (X3) ptx::tma_load_2d(dst + TILE_B, &tmY_lo, bar_full + 8 * p.stage, kb * KBLK, q0);
          }
          p.advance(NS);
        }
      };
      auto load_z = [&](const Walk& k) {
        const int q0 = q_row0(k);
        if (z_mn) {
          for (int n = 0; n < KB; ++n) {
            ptx::mbar_wait(bar_empty + 8 * p.stage, p.phase ^ 1);
            if (ptx::elect_one()) {
              const uint32_t fb = bar_fullz + 8 * p.stage;
              ptx::mbar_arrive_expect_tx(fb, NP * TILE_B);
              const uint32_t dst = sB + p.stage * NP * TILE_B;
              ptx::tma_load_2d(dst, &tmY_hi, fb, n * KBLK, q0);
              if (X3) ptx::tma_load_2d(dst + TILE_B, &tmY_lo, fb, n * KBLK, q0);
            }
            p.advance(NS);
          }
          return;
        }
        for (int j = 0; j < NJ; ++j)
          for (int c = 0; c < NC; ++c) {
            ptx::mbar_wait(bar_empty + 8 * p.stage, p.phase ^ 1);
            if (ptx::elect_one()) {
              const uint32_t fb = bar_fullz + 8 * p.stage;
              ptx::mbar_arrive_expect_tx(fb, NP * TILE_B);   // rows >= Hk arrive as zeros
              const uint32_t dst = sB + p.stage * NP * TILE_B;
              ptx::tma_load_2d(dst, &tmZ_hi, fb, q0 + j * KBLK, c * 128);
              if (X3) ptx::tma_load_2d(dst + TILE_B, &tmZ_lo, fb, q0 + j * KBLK, c * 128);
            }
            p.advance(NS);
          }
      };
      Walk cur, nxt;
      sh.start(cur);
      nxt = cur;
      load_s_operands(cur);
      for (int w = sh.w0; w < sh.w1; ++w) {
        sh.advance(nxt);
        if (w + 1 < sh.w1) load_s_operands(nxt);
        load_z(cur);
        cur = nxt;
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------- MMA issuer, logits
    // ring positions: S(0) | S(1) G(0) | S(2) G(1) | ... | S(n-1) G(n-2) | G(n-1)   (KB stages per S, NZ per G)
    if (sh.w0 < sh.w1) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 128);
      Pipe p;
      uint32_t ybits = 0;                                   // parity of the Y-block barrier, per slot
      int seg_s = -1, tc_s = 0;
      Walk k;
      sh.start(k);
      for (int w = sh.w0; w < sh.w1; ++w, ++tc_s, sh.advance(k)) {
        if (k.first) {
          ++seg_s;
          ptx::mbar_wait(bar_a, seg_s & 1);
          ptx::tc_fence_after_sync();
        }
        const int buf = tc_s % SBUF;
        ptx::mbar_wait(bar_tempty + 8 * buf, ((tc_s / SBUF) & 1) ^ 1);
        ptx::tc_fence_after_sync();
        const uint32_t d = tmem_base + buf * BN;
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(bar_full + 8 * p.stage, (ybits >> p.stage) & 1u);
          ybits ^= 1u << p.stage;
          ptx::tc_fence_after_sync();
          const uint32_t bb = sB + p.stage * NP * TILE_B;
          mma_kblock<X3>(d, sX + kb * TILE_B, sX + (KB + kb) * TILE_B, bb, bb + TILE_B, idesc, kb == 0);
          commit_elect(bar_empty + 8 * p.stage);
          p.advance(NS);
        }
        commit_elect(bar_tfull + 8 * buf);
        if (k.last) commit_elect(bar_afree);
        if (w > sh.w0)                                      // the stages of G(w-1) follow S(w) in the ring
          for (int i = 0; i < NZ; ++i) p.advance(NS);
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------------------------------- MMA issuer, gradient
    if (sh.w0 < sh.w1) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 128);
      Pipe p;
      uint32_t zbits = 0;                                   // parity of the Z-block barrier, per slot
      for (int i = 0; i < KB; ++i) p.advance(NS);           // S(w0)
      int seg_d = -1, tc_d = 0;
      Walk k;
      sh.start(k);
      for (int w = sh.w0; w < sh.w1; ++w, sh.advance(k)) {
        if (w + 1 < sh.w1)
          for (int i = 0; i < KB; ++i) p.advance(NS);       // S(w+1) precedes G(w) in the ring
        const bool first = k.first;
        if (first) {
          if (seg_d >= 0) {                                 // the epilogue has flushed the previous accumulator
            ptx::mbar_wait(bar_hempty, seg_d & 1);
            ptx::tc_fence_after_sync();
          }
          ++seg_d;
        }
        ptx::mbar_wait(bar_dfull, tc_d & 1);                // dS(w) is in tensor memory
        ptx::tc_fence_after_sync();
        if (z_mn) {
          // acc[:, 64n .. 64n+64) += dS[128 tokens x 128 items] . W_out^T block n (MN-major: K = items down the rows)
          constexpr uint32_t idesc_mn = ptx::umma_idesc_bf16_bmn(128, 64);
          for (int n = 0; n < KB; ++n) {
            ptx::mbar_wait(bar_fullz + 8 * p.stage, (zbits >> p.stage) & 1u);
            zbits ^= 1u << p.stage;
            ptx::tc_fence_after_sync();
            const uint32_t bb = sB + p.stage * NP * TILE_B;
            const uint64_t db_hi = ptx::umma_desc_mn_sw128(bb, TILE_B), db_lo = ptx::umma_desc_mn_sw128(bb + TILE_B, TILE_B);
            const uint32_t d = tmem_acc + n * 64;
            if (ptx::elect_one()) {
#pragma unroll
              for (int ks = 0; ks < BN / 16; ++ks) {
                const uint32_t a_hi = tmem_ds + ks * 8, a_lo = a_hi + BN / 2;
                const uint64_t o = (uint64_t)((ks * 16 * 128) >> 4);   // 16 items = 16 rows of 128 B further down
                const uint32_t acc = (first && ks == 0) ? 0u : 1u;
                if (X3) {
                  ptx::umma_bf16_ts(d, a_hi, db_lo + o, idesc_mn, acc);
                  ptx::umma_bf16_ts(d, a_lo, db_hi + o, idesc_mn, 1u);
                  ptx::umma_bf16_ts(d, a_hi, db_hi + o, idesc_mn, 1u);
                } else {
                  ptx::umma_bf16_ts(d, a_hi, db_hi + o, idesc_mn, acc);
                }
              }
            }
            __syncwarp();
            commit_elect(bar_empty + 8 * p.stage);
            p.advance(NS);
          }
        } else
        for (int j = 0; j < NJ; ++j)
          for (int c = 0; c < NC; ++c) {
            ptx::mbar_wait(bar_fullz + 8 * p.stage, (zbits >> p.stage) & 1u);
            zbits ^= 1u << p.stage;
            ptx::tc_fence_after_sync();
            const uint32_t bb = sB + p.stage * NP * TILE_B;
            const uint64_t db_hi = ptx::umma_desc_k_sw128(bb), db_lo = ptx::umma_desc_k_sw128(bb + TILE_B);
            const uint32_t d = tmem_acc + c * 128;
            if (ptx::elect_one()) {
#pragma unroll
              for (int k = 0; k < KBLK / 16; ++k) {
                const uint32_t a_hi = tmem_ds + j * (KBLK / 2) + k * 8, a_lo = a_hi + BN / 2;
                const uint32_t acc = (first && j == 0 && k == 0) ? 0u : 1u;
                if (X3) {
                  ptx::umma_bf16_ts(d, a_hi, ptx::umma_desc_advance_k(db_lo, k * 16), idesc, acc);
                  ptx::umma_bf16_ts(d, a_lo, ptx::umma_desc_advance_k(db_hi, k * 16), idesc, 1u);
                  ptx::umma_bf16_ts(d, a_hi, ptx::umma_desc_advance_k(db_hi, k * 16), idesc, 1u);
                } else {
                  ptx::umma_bf16_ts(d, a_hi, ptx::umma_desc_advance_k(db_hi, k * 16), idesc, acc);
                }
              }
            }
            __syncwarp();
            commit_elect(bar_empty + 8 * p.stage);
            p.advance(NS);
          }
        commit_elect(bar_dempty);                           // the dS columns may be overwritten
        if (k.last) commit_elect(bar_hfull);
        ++tc_d;
      }
    }
  } else if (warp >= C::EPI0) {
    // ------------------------------------------------------------------------------------------- epilogue
    const int q = warp & 3;
    const int half = (warp - C::EPI0) >> 2;
    const int row = q * 32 + lane;
    const int e = threadIdx.x - 32 * C::EPI0;                // 0..255 among the epilogue threads
    const float inv = inv_nvalid ? inv_nvalid[0] : 1.0f;    // NULL: un-normalised gradients (the optimiser divides)
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    float4* sT_gen = reinterpret_cast<float4*>(smem_raw + (sT - ptx::smem_u32(smem_raw)));
    RowTerms rt;                                             // !ITEM_ST: this thread's token row; ITEM_ST: prefetch
    float bias_v = 0.f, db_acc = 0.f;                        // ITEM_ST: b_out of this thread's item, its dL/db partial
    float s_acc = 0.f;                                       // FUSED: this thread's share of sum_v exp(z - ref)
    int tc = 0, seg = -1;
    Walk k, nxt;
    sh.start(k);
    nxt = k;
    if (ITEM_ST && sh.w0 < sh.w1) {
      if (e < 128) {
        rt = load_row_terms((int64_t)k.in * BM + e, n_tokens, mrow, srow, coef, tgt, inv);
        sT_gen[e] = make_float4(rt.nb, rt.scale, rt.cf, __int_as_float(rt.tg));
      }
      epi_bar_sync();
    }
    for (int w = sh.w0; w < sh.w1; ++w, ++tc, k = nxt) {
      const int buf = tc % SBUF;
      sh.advance(nxt);
      if (k.first) {
        ++seg;
        if (MODE == TS_DH) rt = load_row_terms((int64_t)k.o * BM + row, n_tokens, mrow, srow, coef, tgt, inv);
        if (FUSED) {                                         // exp(z - ref) un-normalised, no one-hot term
          const int64_t n = (int64_t)k.o * BM + row;
          rt.nb = -INFINITY; rt.scale = 0.f; rt.cf = 0.f; rt.tg = -1;
          if (n < n_tokens && (tok_mask == nullptr || tok_mask[n])) { rt.nb = -mrow[n] * LOG2E; rt.scale = 1.f; }
          s_acc = 0.f;
        }
        if (ITEM_ST) {
          const int v = v_begin + k.o * BN + row;
          bias_v = (b_out && v < v_end) ? b_out[v] : 0.f;
          db_acc = 0.f;
        }
      }
      if (ITEM_ST && e < 128 && w + 1 < sh.w1)               // next tile's token terms, behind this tile's math
        rt = load_row_terms((int64_t)nxt.in * BM + e, n_tokens, mrow, srow, coef, tgt, inv);
      ptx::mbar_wait(bar_tfull + 8 * buf, (tc / SBUF) & 1);
      ptx::tc_fence_after_sync();
      float z[64];
      load_half_tile(tmem_base + lane_off + buf * BN + half * 64, z);
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar_tempty + 8 * buf);
      if (!ITEM_ST) {
        const int vc0 = v_begin + k.in * BN + half * 64;
        if (b_out) {                                         // warp-uniform: output bias of the items in the columns
#pragma unroll
          for (int j = 0; j < 64; ++j)
            if (vc0 + j < v_end) z[j] += __ldg(b_out + vc0 + j);
        }
        dlogit_half_tile(z, rt, vc0, v_end);
        if (FUSED) {
          float a4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int j = 0; j < 64; j += 4) { a4[0] += z[j]; a4[1] += z[j + 1]; a4[2] += z[j + 2]; a4[3] += z[j + 3]; }
          s_acc += (a4[0] + a4[1]) + (a4[2] + a4[3]);
        }
      } else {
        const int v = v_begin + k.o * BN + row;              // this thread's item
        const bool row_ok = v < v_end;
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const float4 t = sT_gen[half * 64 + j];            // {-m.log2e, coef/s, coef, target} of token column j
          float x = ptx::ex2_approx(fmaf(z[j] + bias_v, LOG2E, t.x)) * t.y;
          if (__float_as_int(t.w) == v) x -= t.z;
          z[j] = row_ok ? x : 0.f;
          db_acc += z[j];                                    // dL/db_out[v] = sum over tokens of dlogit
        }
      }
      ptx::mbar_wait(bar_dempty, (tc & 1) ^ 1);              // the previous tile's second GEMM has consumed dS
      ptx::tc_fence_after_sync();
      {
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float x0 = z[2 * i], x1 = z[2 * i + 1];
          const __nv_bfloat162 hv = __floats2bfloat162_rn(x0, x1);
          hi[i] = *reinterpret_cast<const uint32_t*>(&hv);
          if (X3) lo[i] = pack_bf16x2(x0 - __low2float(hv), x1 - __high2float(hv));
        }
        const uint32_t dst = tmem_ds + lane_off + half * 32;
        ptx::tmem_st_32x32(dst, hi);
        if (X3) ptx::tmem_st_32x32(dst + BN / 2, lo);
        ptx::tmem_st_wait();
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bar_dfull);
      if (ITEM_ST && w + 1 < sh.w1) {
        epi_bar_sync();                                      // every epilogue thread has read this tile's terms
        if (e < 128) sT_gen[e] = make_float4(rt.nb, rt.scale, rt.cf, __int_as_float(rt.tg));
        epi_bar_sync();
      }
      if (k.last) {
        ptx::mbar_wait(bar_hfull, seg & 1);
        ptx::tc_fence_after_sync();
        const int h0 = half * (C::ACC_COLS / 2);             // this warp's hidden columns of its 32 rows
        if (!ITEM_ST) {
          const int64_t n = (int64_t)k.o * BM + row;
          flush_acc_red(tmem_acc + lane_off + h0, C::ACC_COLS / 2, out + n * H + h0, H - h0, n < n_tokens,
                        (H & 3) == 0, (hscale && !FUSED) ? hscale + n * H + h0 : nullptr);
          if (FUSED && n < n_tokens && s_acc != 0.f) atomicAdd(s_out + n, s_acc);
        } else {
          const int v = v_begin + k.o * BN + row;
          const bool row_ok = v < v_end;
          if (db_out && row_ok) atomicAdd(db_out + v, db_acc);
#pragma unroll 1
          for (int c = 0; c < C::ACC_COLS / 2; c += 32) {
            uint32_t r[32];
            ptx::tmem_ld_32x32(tmem_acc + lane_off + h0 + c, r);
            ptx::tmem_ld_wait();
            if (row_ok) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int h = h0 + c + j;                    // lanes = consecutive items: coalesced reductions
                if (h < H) atomicAdd(out + (size_t)h * ldw + v, __uint_as_float(r[j]));
              }
            }
          }
        }
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar_hempty);
      }
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// exact fp32 target logit: zy[n] = sum_h hs[n,h] * W_out[h, tgt[n]] (+ b_out[tgt[n]]); one warp per token
__global__ void __launch_bounds__(256)
target_logit_kernel(const float* __restrict__ hout, const float* __restrict__ hscale,
                    const float* __restrict__ W_out, const float* __restrict__ b_out,
                    const int32_t* __restrict__ tgt, float* __restrict__ zy, int64_t n_tokens, int H, int ldw,
                    const int32_t* __restrict__ orig, const int32_t* __restrict__ n_tokens_dev) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (n_tokens_dev) n_tokens = min(n_tokens, (int64_t)n_tokens_dev[0]);
  if (n >= n_tokens) return;
  const int32_t t = tgt[n];
  if (t < 0) { if (orig && lane == 0) zy[n] = 0.f; return; }
  const int64_t r = orig ? orig[n] : n;                      // compacted token axis: row of hout behind token n
  float acc = 0.f;
  for (int h = lane; h < H; h += 32) {
    float x = hout[r * H + h];
    if (hscale) x *= hscale[r * H + h];
    acc = fmaf(x, __ldg(W_out + (size_t)h * ldw + t), acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) zy[n] = acc + (b_out ? b_out[t] : 0.f);
}

// persistent grid: one CTA per SM, or one per tile pair when there are fewer pairs than SMs
int persistent_grid(int64_t total) { return (int)(total < SEQREC_NUM_SMS ? total : SEQREC_NUM_SMS); }

// partial slots a token tile can need: CTAs sharing one token tile's run of n_inner item tiles
int forward_slots(int64_t n_tokens, int v_begin, int v_end) {
  const int64_t n_inner = ceil_div(v_end - v_begin, BN);
  const int64_t total = ((n_tokens + BM - 1) / BM) * n_inner;
  const int64_t per = total / persistent_grid(total);      // >= 1: every CTA owns at least `per` tile pairs
  return (int)((n_inner + per - 1) / per + 1);
}

template <int KB, int NS, bool X3, bool BIAS, bool RANK>
int launch_fwd(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
               const float* b_out, float* ws_m, float* ws_s, int64_t n_tokens, int v_begin, int v_end,
               const float* ref, const int32_t* tgt, int id_offset, int32_t* rank, cudaStream_t st) {
  constexpr int NP = X3 ? 2 : 1;
  const size_t smem = 1024 + (size_t)NP * KB * TILE_B + (size_t)NS * NP * TILE_B + 256;
  auto k = ce_tc_forward_kernel<KB, NS, X3, BIAS, RANK>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return -(int)e;
  const int64_t total = ((n_tokens + BM - 1) / BM) * ceil_div(v_end - v_begin, BN);
  k<<<persistent_grid(total), TCF_THREADS, smem, st>>>(a_hi, a_lo, b_hi, b_lo, b_out, ws_m, ws_s, n_tokens, v_begin,
                                                       v_end, forward_slots(n_tokens, v_begin, v_end), ref, tgt,
                                                       id_offset, rank);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

template <int KB, bool X3, int MODE>
int launch_ts_one(int grid, const CUtensorMap& x_hi, const CUtensorMap& x_lo, const CUtensorMap& y_hi,
                  const CUtensorMap& y_lo, const CUtensorMap& z_hi, const CUtensorMap& z_lo, const int32_t* tgt,
                  const float* m, const float* s, const float* coef, const float* inv_nvalid, const float* hscale,
                  float* out, int64_t n_tokens, int H, int v_begin, int v_end, int ldw, const float* b_out,
                  float* db_out, const uint8_t* tok_mask, float* s_out, const int32_t* n_tokens_dev, cudaStream_t st) {
  using C = TsCfg<KB, X3>;
  size_t smem = (size_t)C::SMEM_NEED + 1024;                 // slack for the 1024-byte alignment of the tiles
  if (smem > 227 * 1024) smem = 227 * 1024;                  // (the kernel traps if the aligned layout does not fit)
  auto k = ce_tc_backward_ts_kernel<KB, X3, MODE>;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return -(int)e;
  {
    // chunk counters of the front throttle (this variant's row); the symbol address is looked up once per device, on an
    // eager call (the first step of a shape always is), so a captured step only records the memset node
    static void* sync_ws[64] = {};
    int dev = 0;
    e = cudaGetDevice(&dev);
    if (e != cudaSuccess || dev < 0 || dev >= 64) return e != cudaSuccess ? -(int)e : -1090;
    if (!sync_ws[dev]) {
      e = cudaGetSymbolAddress(&sync_ws[dev], g_ts_sync);
      if (e != cudaSuccess) return -(int)e;
      // (experiments only: the default mode 0 is the symbol's initial value, so a production run never issues this
      //  copy -- which would not be allowed if the first call of this variant happened inside a stream capture)
      const char* zm = getenv("SEQREC_ZMN");
      const int mode = zm ? atoi(zm) : 0;
      if (mode != 0) {
        e = cudaMemcpyToSymbol(g_ts_zmn_mode, &mode, sizeof(int));
        if (e != cudaSuccess) return -(int)e;
      }
    }
    // (the kernel throttles only when its streamed operand exceeds 32 MB; n_tokens is the upper bound of the device-side
    //  token count, so "fits" here implies "fits" there and the memset node can be dropped)
    const int64_t inner_ub = (MODE == TS_DW) ? (n_tokens + BM - 1) / BM : (v_end - v_begin + BN - 1) / BN;
    if (inner_ub * (int64_t)(2 * C::NP * KB * TILE_B) > (32ll << 20)) {
      e = cudaMemsetAsync(static_cast<int*>(sync_ws[dev]) + (size_t)MODE * TS_SYNC_SLOTS, 0,
                          sizeof(int) * TS_SYNC_SLOTS, st);
      if (e != cudaSuccess) return -(int)e;
    }
  }
  k<<<grid, C::THREADS, smem, st>>>(x_hi, x_lo, y_hi, y_lo, z_hi, z_lo, tgt, m, s, coef, inv_nvalid, hscale, out,
                                    n_tokens, H, v_begin, v_end, ldw, (uint32_t)smem, b_out, db_out, tok_mask, s_out,
                                    n_tokens_dev);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

int launch_ts(int KB, bool x3, int mode, int grid, const CUtensorMap& x_hi, const CUtensorMap& x_lo,
              const CUtensorMap& y_hi, const CUtensorMap& y_lo, const CUtensorMap& z_hi, const CUtensorMap& z_lo,
              const int32_t* tgt, const float* m, const float* s, const float* coef, const float* inv_nvalid,
              const float* hscale, float* out, int64_t n_tokens, int H, int v_begin, int v_end, int ldw,
              const float* b_out, float* db_out, const uint8_t* tok_mask, float* s_out, const int32_t* n_tokens_dev,
              cudaStream_t st) {
#define TS3(KBV, X3V, MV)                                                                                          \
  return launch_ts_one<KBV, X3V, MV>(grid, x_hi, x_lo, y_hi, y_lo, z_hi, z_lo, tgt, m, s, coef, inv_nvalid, hscale, \
                                     out, n_tokens, H, v_begin, v_end, ldw, b_out, db_out, tok_mask, s_out, n_tokens_dev, st)
#define TS2(KBV)                                                                           \
  {                                                                                        \
    if (x3) {                                                                              \
      if (mode == TS_DW) TS3(KBV, true, TS_DW);                                            \
      else if (mode == TS_FUSED) TS3(KBV, true, TS_FUSED);                                 \
      else TS3(KBV, true, TS_DH);                                                          \
    } else {                                                                               \
      if (mode == TS_DW) TS3(KBV, false, TS_DW);                                           \
      else if (mode == TS_FUSED) TS3(KBV, false, TS_FUSED);                                \
      else TS3(KBV, false, TS_DH);                                                         \
    }                                                                                      \
  }
  switch (KB) {
    case 1: TS2(1)
    case 2: TS2(2)
    case 3: TS2(3)
    default: TS2(4)
  }
#undef TS2
#undef TS3
}

template <int KB, bool X3, bool BIAS>
int launch_topk(const uint16_t* A_hi, const uint16_t* A_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                const float* b_out, float* cand_v, int32_t* cand_i, int64_t n_rows, int V, int k, cudaStream_t st) {
  constexpr int NP = X3 ? 2 : 1;
  constexpr int NS = X3 ? 4 : 8;
  const size_t smem = 1024 + (size_t)NS * NP * TILE_B + 2 * TOPK_MAX * 256 * 4 + 256;
  auto kern = ce_tc_topk_kernel<KB, NS, X3, BIAS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return -(int)e;
  const int64_t total = ((n_rows + BM - 1) / BM) * ceil_div(V, BN);
  kern<<<persistent_grid(total), TC_THREADS, smem, st>>>(A_hi, A_lo, b_hi, b_lo, b_out, cand_v, cand_i, n_rows, 0, V,
                                                         forward_slots(n_rows, 0, V), k);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

}  // namespace

// top-k on the tensor cores: A / Bt operands as for seqrec_ce_tc_forward; ws_v / ws_i hold
// seqrec_ce_tc_partials(n_rows, 0, V) * n_rows * k candidates.  k <= 32 and partials * k <= 384.
extern "C" int seqrec_topk_tc(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                              const float* b_out, const float* m, const float* s, float* ws_v, int32_t* ws_i,
                              int32_t* topk_ids, float* topk_p, int64_t n_rows, int Hk, int V, int k, int x3,
                              void* stream) {
  SEQREC_ARG(n_rows > 0 && V > 0 && k >= 1 && k <= TOPK_MAX && k <= V, 1);
  SEQREC_ARG(Hk == 64 || Hk == 128 || Hk == 192 || Hk == 256, 2);
  SEQREC_ARG(A_hi && Bt_hi && (!x3 || (A_lo && Bt_lo)) && ws_v && ws_i && topk_ids, 3);
  const int n_lists = 2 * forward_slots(n_rows, 0, V);
  SEQREC_ARG(n_lists * k <= 384, 4);
  CUtensorMap b_hi, b_lo;
  int rc;
  if ((rc = make_tmap(&b_hi, Bt_hi, V, Hk, Hk, BN))) return rc;
  if ((rc = make_tmap(&b_lo, x3 ? Bt_lo : Bt_hi, V, Hk, Hk, BN))) return rc;
  cudaStream_t st = as_stream(stream);
#define TK2(KB, X3V, BV) rc = launch_topk<KB, X3V, BV>(A_hi, x3 ? A_lo : A_hi, b_hi, b_lo, b_out, ws_v, ws_i, n_rows, V, k, st)
#define TK(KB)                                                                   \
  {                                                                              \
    if (x3) { if (b_out) TK2(KB, true, true); else TK2(KB, true, false); }       \
    else    { if (b_out) TK2(KB, false, true); else TK2(KB, false, false); }     \
  }
  switch (Hk / KBLK) {
    case 1: TK(1) break;
    case 2: TK(2) break;
    case 3: TK(3) break;
    default: TK(4) break;
  }
#undef TK2
#undef TK
  if (rc) return rc;
  topk_merge_kernel<<<ceil_div(n_rows * 32, 256), 256, 0, st>>>(ws_v, ws_i, n_lists, n_rows * k, m, s, topk_ids, topk_p,
                                                                n_rows, k);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// merge of n_lists candidate lists per row (vocabulary-parallel ranking: one list of k (probability, item id) pairs per
// item shard): value descending, lower item id first on ties -- the same selection the single-GPU ranking ends with
extern "C" int seqrec_topk_merge(const float* cand_v, const int32_t* cand_i, int n_lists, int64_t list_stride,
                                 int32_t* topk_ids, float* topk_p, int64_t n_rows, int k, void* stream) {
  SEQREC_ARG(cand_v && cand_i && topk_ids && n_rows > 0 && k >= 1 && n_lists >= 1, 1);
  SEQREC_ARG(n_lists * k <= 384 && list_stride >= n_rows * k, 2);
  topk_merge_kernel<<<ceil_div(n_rows * 32, 256), 256, 0, as_stream(stream)>>>(cand_v, cand_i, n_lists, list_stride,
                                                                               nullptr, nullptr, topk_ids, topk_p,
                                                                               n_rows, k);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

// -----------------------------------------------------------------------------------------------------------------
extern "C" int seqrec_target_logit(const float* hout, const float* hscale, const float* W_out, const float* b_out,
                                   const int32_t* tgt, float* zy, int64_t n_tokens, int H, int ldw,
                                   const int32_t* orig, const int32_t* n_tokens_dev, void* stream) {
  SEQREC_ARG(n_tokens > 0 && H > 0 && ldw > 0, 1);
  target_logit_kernel<<<ceil_div(n_tokens * 32, 256), 256, 0, as_stream(stream)>>>(hout, hscale, W_out, b_out, tgt, zy,
                                                                                  n_tokens, H, ldw, orig, n_tokens_dev);
  SEQREC_CHECK_LAUNCH();
  return 0;
}

extern "C" int seqrec_ce_tc_partials(int64_t n_tokens, int v_begin, int v_end) {
  if (n_tokens <= 0 || v_end <= v_begin) return -1001;
  return 2 * forward_slots(n_tokens, v_begin, v_end);
}

namespace {
template <bool RANK>
int ce_tc_forward_impl(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                       const float* b_out, float* ws_m, float* ws_s, const float* ref, const int32_t* tgt,
                       int id_offset, int32_t* rank, int64_t n_tokens, int Hk, int V, int v_begin, int v_end, int x3,
                       void* stream) {
  SEQREC_ARG(n_tokens > 0 && V > 0 && v_begin >= 0 && v_begin < v_end && v_end <= V, 1);
  SEQREC_ARG(Hk == 64 || Hk == 128 || Hk == 192 || Hk == 256, 2);
  SEQREC_ARG(A_hi && Bt_hi && (!x3 || (A_lo && Bt_lo)), 3);
  SEQREC_ARG(!RANK || (ref && tgt && rank), 4);
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
  int rc;
  if ((rc = make_tmap(&a_hi, A_hi, n_tokens, Hk, Hk, BM))) return rc;
  if ((rc = make_tmap(&b_hi, Bt_hi, V, Hk, Hk, BN))) return rc;
  if ((rc = make_tmap(&a_lo, x3 ? A_lo : A_hi, n_tokens, Hk, Hk, BM))) return rc;
  if ((rc = make_tmap(&b_lo, x3 ? Bt_lo : Bt_hi, V, Hk, Hk, BN))) return rc;
  cudaStream_t st = as_stream(stream);
#define FWD2(KB, NS, X3V, BV)                                                                                      \
  return launch_fwd<KB, NS, X3V, BV, RANK>(a_hi, a_lo, b_hi, b_lo, b_out, ws_m, ws_s, n_tokens, v_begin, v_end, ref, \
                                           tgt, id_offset, rank, st)
#define FWD(KB, NS)                                                                      \
  {                                                                                      \
    if (x3) { if (b_out) FWD2(KB, NS, true, true); else FWD2(KB, NS, true, false); }     \
    else    { if (b_out) FWD2(KB, NS, false, true); else FWD2(KB, NS, false, false); }   \
  }
  switch (Hk / KBLK) {
    case 1: FWD(1, 4)
    case 2: FWD(2, 4)
    case 3: FWD(3, 3)
    default: FWD(4, 3)
  }
#undef FWD2
#undef FWD
}
}  // namespace

extern "C" int seqrec_ce_tc_forward(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi,
                                    const uint16_t* Bt_lo, const float* b_out, float* ws_m, float* ws_s,
                                    int64_t n_tokens, int Hk, int V, int v_begin, int v_end, int x3, void* stream) {
  return ce_tc_forward_impl<false>(A_hi, A_lo, Bt_hi, Bt_lo, b_out, ws_m, ws_s, nullptr, nullptr, 0, nullptr, n_tokens,
                                   Hk, V, v_begin, v_end, x3, stream);
}

extern "C" int seqrec_ce_tc_forward_rank(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi,
                                         const uint16_t* Bt_lo, const float* b_out, float* ws_m, float* ws_s,
                                         const float* ref, const int32_t* tgt, int id_offset, int32_t* rank,
                                         int64_t n_tokens, int Hk, int V, int v_begin, int v_end, int x3,
                                         void* stream) {
  return ce_tc_forward_impl<true>(A_hi, A_lo, Bt_hi, Bt_lo, b_out, ws_m, ws_s, ref, tgt, id_offset, rank, n_tokens, Hk,
                                  V, v_begin, v_end, x3, stream);
}

extern "C" int seqrec_ce_tc_backward(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Ht_hi,
                                     const uint16_t* Ht_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                                     const uint16_t* W_hi, const uint16_t* W_lo, const int32_t* tgt, const float* m,
                                     const float* s, const float* coef, const float* inv_nvalid, const float* hscale,
                                     float* dh, float* dW_out, int64_t n_tokens, int H, int Hk, int V, int Vp,
                                     int64_t Np, int v_begin, int v_end, int ldw, int accumulate_dh, int x3,
                                     const float* b_out, float* db_out, const int32_t* n_tokens_dev, void* stream) {
  SEQREC_ARG(n_tokens > 0 && V > 0 && v_begin >= 0 && v_begin < v_end && v_end <= V, 1);
  SEQREC_ARG((Hk == 64 || Hk == 128 || Hk == 192 || Hk == 256) && H <= Hk, 2);
  SEQREC_ARG(Vp >= V && Vp % 8 == 0 && Np >= n_tokens && Np % 8 == 0 && ldw >= v_end, 3);
  cudaStream_t st = as_stream(stream);
  CUtensorMap a_hi, a_lo, b_hi, b_lo, w_hi, w_lo, t_hi, t_lo;
  int rc;
  if ((rc = make_tmap(&a_hi, A_hi, n_tokens, Hk, Hk, BM))) return rc;
  if ((rc = make_tmap(&a_lo, x3 ? A_lo : A_hi, n_tokens, Hk, Hk, BM))) return rc;
  if ((rc = make_tmap(&b_hi, Bt_hi, V, Hk, Hk, BN))) return rc;
  if ((rc = make_tmap(&b_lo, x3 ? Bt_lo : Bt_hi, V, Hk, Hk, BN))) return rc;
  const int KB = Hk / KBLK;
  const int64_t total_ts = ((n_tokens + BM - 1) / BM) * ceil_div(v_end - v_begin, BN);
  const int grid_ts = persistent_grid(total_ts);
  if (dh) {
    if (!accumulate_dh) {
      cudaError_t e = cudaMemsetAsync(dh, 0, sizeof(float) * (size_t)n_tokens * H, st);
      if (e != cudaSuccess) return -(int)e;
    }
    if ((rc = make_tmap(&w_hi, W_hi, Hk, V, Vp, 128))) return rc;
    if ((rc = make_tmap(&w_lo, x3 ? W_lo : W_hi, Hk, V, Vp, 128))) return rc;
    if ((rc = launch_ts(KB, x3 != 0, TS_DH, grid_ts, a_hi, a_lo, b_hi, b_lo, w_hi, w_lo, tgt, m, s, coef, inv_nvalid,
                        hscale, dh, n_tokens, H, v_begin, v_end, ldw, b_out, nullptr, nullptr, nullptr, n_tokens_dev, st)))
      return rc;
  }
  if (dW_out) {
    if ((rc = make_tmap(&t_hi, Ht_hi, Hk, n_tokens, Np, 128))) return rc;
    if ((rc = make_tmap(&t_lo, x3 ? Ht_lo : Ht_hi, Hk, n_tokens, Np, 128))) return rc;
    if ((rc = launch_ts(KB, x3 != 0, TS_DW, grid_ts, b_hi, b_lo, a_hi, a_lo, t_hi, t_lo, tgt, m, s, coef, inv_nvalid,
                        nullptr, dW_out, n_tokens, H, v_begin, v_end, ldw, b_out, db_out, nullptr, nullptr, n_tokens_dev, st)))
      return rc;
  }
  return 0;
}


// ================================================================================================================
// Fused forward + dH (TS_FUSED above) and its finish pass.
//   seqrec_ce_tc_fused:   acc (N,H) += sum_v exp(z - ref) . W_out[:,v]   and   s (N) += sum_v exp(z - ref),
//                         ref = zy (target logit); acc and s must be zero on entry (both leave through reductions).
//   seqrec_ce_dh_finish:  dh[n,:] = coef[n] . (acc[n,:] / s[n] - W_out[:, tgt[n]]) (. hscale), in place over acc.
//                         coef comes from seqrec_ce_finalize (splits = 1, ws_m = ref, ws_s = s); rows with coef = 0 (pads,
//                         clip-saturated, overflowed s) are written as zeros.  The target column of W_out is read from the
//                         bf16 hi/lo image of W_out^T (hi + lo: 16 mantissa bits, the precision class of the x3 products).
extern "C" int seqrec_ce_tc_fused(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* Bt_hi, const uint16_t* Bt_lo,
                                  const uint16_t* W_hi, const uint16_t* W_lo, const float* ref, const uint8_t* mask,
                                  const float* b_out, float* acc, float* s, int64_t n_tokens, int H, int Hk, int V,
                                  int Vp, int v_begin, int v_end, int x3, const int32_t* n_tokens_dev, void* stream) {
  SEQREC_ARG(n_tokens > 0 && V > 0 && v_begin >= 0 && v_begin < v_end && v_end <= V, 1);
  SEQREC_ARG((Hk == 64 || Hk == 128 || Hk == 192 || Hk == 256) && H <= Hk, 2);
  SEQREC_ARG(Vp >= V && Vp % 8 == 0 && ref && acc && s, 3);
  SEQREC_ARG(A_hi && Bt_hi && W_hi && (!x3 || (A_lo && Bt_lo && W_lo)), 4);
  cudaStream_t st = as_stream(stream);
  CUtensorMap a_hi, a_lo, b_hi, b_lo, w_hi, w_lo;
  int rc;
  if ((rc = make_tmap(&a_hi, A_hi, n_tokens, Hk, Hk, BM))) return rc;
  if ((rc = make_tmap(&a_lo, x3 ? A_lo : A_hi, n_tokens, Hk, Hk, BM))) return rc;
  if ((rc = make_tmap(&b_hi, Bt_hi, V, Hk, Hk, BN))) return rc;
  if ((rc = make_tmap(&b_lo, x3 ? Bt_lo : Bt_hi, V, Hk, Hk, BN))) return rc;
  if ((rc = make_tmap(&w_hi, W_hi, Hk, V, Vp, 128))) return rc;
  if ((rc = make_tmap(&w_lo, x3 ? W_lo : W_hi, Hk, V, Vp, 128))) return rc;
  const int64_t total = ((n_tokens + BM - 1) / BM) * ceil_div(v_end - v_begin, BN);
  return launch_ts(Hk / KBLK, x3 != 0, TS_FUSED, persistent_grid(total), a_hi, a_lo, b_hi, b_lo, w_hi, w_lo, nullptr, ref,
                   nullptr, nullptr, nullptr, nullptr, acc, n_tokens, H, v_begin, v_end, V, b_out, nullptr, mask, s,
                   n_tokens_dev, st);
}

namespace {
// one warp per token row
__global__ void __launch_bounds__(256)
ce_dh_finish_kernel(const float* __restrict__ acc, float* __restrict__ dh, const float* __restrict__ srow,
                    const float* __restrict__ coef, const int32_t* __restrict__ tgt,
                    const __nv_bfloat16* __restrict__ Bt_hi, const __nv_bfloat16* __restrict__ Bt_lo,
                    const float* __restrict__ hscale, int64_t n_tokens, int H, int Hk,
                    const int32_t* __restrict__ orig, const int32_t* __restrict__ n_tokens_dev) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (n_tokens_dev) n_tokens = min(n_tokens, (int64_t)n_tokens_dev[0]);
  if (n >= n_tokens) return;
  const int64_t r = orig ? orig[n] : n;                      // compacted token axis: dh row behind token n
  const float cf = coef[n];
  const float* src = acc + n * H;
  float* row = dh + r * H;
  if (cf == 0.f) {
    for (int h = lane; h < H; h += 32) row[h] = 0.f;
    return;
  }
  const float inv_s = 1.0f / srow[n];
  const int32_t y = tgt[n];                                  // -1: the target lives on another item shard
  for (int h = lane; h < H; h += 32) {
    float wy = 0.f;
    if (y >= 0) {
      wy = __bfloat162float(Bt_hi[(size_t)y * Hk + h]);
      if (Bt_lo) wy += __bfloat162float(Bt_lo[(size_t)y * Hk + h]);
    }
    float v = cf * (src[h] * inv_s - wy);
    if (hscale) v *= hscale[r * H + h];
    row[h] = v;
  }
}
}  // namespace

extern "C" int seqrec_ce_dh_finish(const float* acc, float* dh, const float* s, const float* coef, const int32_t* tgt,
                                   const uint16_t* Bt_hi, const uint16_t* Bt_lo, const float* hscale, int64_t n_tokens,
                                   int H, int Hk, const int32_t* orig, const int32_t* n_tokens_dev, void* stream) {
  SEQREC_ARG(acc && dh && s && coef && tgt && Bt_hi && n_tokens > 0 && H > 0 && Hk >= H, 1);
  SEQREC_ARG(orig == nullptr || acc != dh, 2);               // a compacted accumulator cannot be finished in place
  ce_dh_finish_kernel<<<ceil_div(n_tokens * 32, 256), 256, 0, as_stream(stream)>>>(
      acc, dh, s, coef, tgt, reinterpret_cast<const __nv_bfloat16*>(Bt_hi),
      reinterpret_cast<const __nv_bfloat16*>(Bt_lo), hscale, n_tokens, H, Hk, orig, n_tokens_dev);
  SEQREC_CHECK_LAUNCH();
  return 0;
}
