// Flash-attention backward on tcgen05 (sm_100a), fp32-accurate: split-fp16 operands ("x3", see lg_x3.cu / lg_x3_attn.cu),
// head_dim 64.  Backward of Attention.forward (lightglue.py:112-129) as autograd would give it for the reference's
// training step (lightglue.py:484-498); nothing N x M is stored, the scores are recomputed tile by tile.
//
// One kernel template, two roles -- "own" rows X, U (128 per CTA) against tiles of 64 "other" rows Y, W:
//
//   role   own X  own U  other Y  other W   sc = X.Y^T   dp = U.W^T    out1 += D.Y          out2 += P.W
//   DQ     Q      dO     K        V         S            dP            dQ  (x ln 2)         --
//   DKV    K      V      Q        dO        S^T          dP^T          dK  (x ln 2)         dV
//
//   P = 2^(sc - lse[query]),  D = P (dp - delta[query]),  delta = <dO, O>   (the query is the row in DQ, the column in DKV)
//
// Every product is three MMAs on fp16 plane pairs (hi.hi + hi.lo + lo.hi, fp32 accumulation in TMEM): the
// operands Q, K, V carry the activation scaling LG_X3_EA, dO a per-call power of two g chosen so that max |g dO| lies in
// [256, 512) (gradients have no fixed range: a fixed scaling would push small ones into the fp16 subnormals), P the
// scaling LG_X3_EP and D the scaling g / 64; all are powers of two and are undone exactly in the epilogue.
// CTA = warp 0 TMA producer, warp 1 MMA issuer, warps 2.. "softmax" warps (NP threads per own row).
// ALL MMAs ARE OF THE TS FORM (A operand from TMEM): tools/micro/umma_rate.cu measures 48 cycles for an SS MMA of
// 128 x 64 x 16 (6 KB of operands per MMA against the SM's 128 B/clk of shared memory) and the nominal 32 for the TS
// form, so the own rows X, U are copied into TMEM once per CTA by the softmax threads (plain global loads +
// tcgen05.st) and never pass through shared memory.  TMEM (512 columns, one CTA per SM): sc x 2 | dp x 2 (double-
// buffered: the score MMAs of tile j+1 run while the warps work on tile j; a thread writes the D / P plane pairs of a
// tile OVER ITS OWN score columns, so the planes are double-buffered too and no thread waits for another) | out1 | out2
// | X hi, lo | U hi, lo.  The DQ role first sweeps the other tiles once for the row statistics (log-sum-exp in the log2
// domain and delta; written to the workspace for the DKV role), then a second time for dQ.
// TWO-LEVEL ACCUMULATION (as in lg_x3_attn.cu): the tensor core rounds its fp32 accumulator toward zero after every MMA,
// so one accumulator over 2048 other rows (384 MMAs) is ~1e-5 low on same-sign sums (measured against float64:
// tools/attn_bwd_accuracy.py, profiles/r2_attn_bwd_tcgen05.txt).  out1 / out2 therefore collect XB_FLUSH tiles (48 MMAs)
// and are then added, round-to-nearest, to fp32 running sums that every softmax thread keeps for its own row in shared
// memory ([column][row]: conflict-free); the first MMA after a flush overwrites the accumulator.
//
// BF16 INSTANTIATION (template parameter BF, lg_bf16_attention_bwd): the backward of the bf16 forward kernels
// (lg_tc_attn.cu) on the operands that forward read -- Q, K, V bf16 as they are, dO converted once to a head-major bf16
// copy.  Every product is ONE kind::f16 MMA with bf16 A / B formats; P and D go to TMEM as one bf16 plane each, X and U
// take 32 TMEM columns each.  No plane scalings (bf16 has the exponent range of fp32): g = 1, D is stored unscaled;
// P keeps the factor 256 of the shared lse - 8 convention.  delta = <dO, O> is taken in fp32 from the fp32 dctx and the
// bf16 ctx of the forward.  The stage / TMEM layout and the two-level accumulation are those of the x3 kernel.
#include "lg_internal.cuh"
#include "lg_tc_common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <type_traits>

namespace {

constexpr int XB_OT = 64;                       // other rows per tile
constexpr int XB_TBY = XB_OT * 64 * 2;          // one plane of an other tile (64 x 64 fp16, 128-byte swizzle): 8 KB
constexpr int XB_NST = 4;                       // stages of (Yh | Yl | Wh | Wl)
constexpr int XB_Y = 0;                         // XB_NST x 32 KB
constexpr int XB_BAR = XB_Y + XB_NST * 4 * XB_TBY;  // 128 KB of tiles
constexpr int XB_NBAR = 1 + 2 * XB_NST + 2 + 2 + 2 + 1;
constexpr int XB_ACC = XB_BAR + 256;            // [128 columns][128 rows] fp32 running sums of out1 | out2 (64 KB)
constexpr int XB_XCH = XB_ACC;                  // [128 rows][NP parts] float4 (max, sum, partial delta): statistics sweep only
constexpr int XB_SMEM = XB_ACC + 128 * 128 * 4;
constexpr int XB_FLUSH = 4;                     // tiles per TMEM accumulator before it is folded into the running sums
static_assert(XB_SMEM <= 227 * 1024, "attention backward: shared memory");
// TMEM: sc x 2 | dp x 2 (the D / P plane pairs are written over the scores they were computed from) | out1 | out2 |
// own rows as A operands: X hi, X lo, U hi, U lo
constexpr uint32_t XT_SC = 0, XT_DP = 128, XT_O1 = 256, XT_O2 = 320, XT_XH = 384, XT_XL = 416, XT_UH = 448, XT_UL = 480;
constexpr float XB_DC = 1.f / 64.f;             // D planes hold (g / 64) D
// The exponentials are taken against lse - 8, i.e. they ARE the P plane values 256 P (LG_X3_EP); the workspace holds
// lse2 - 8 and delta * g * DT so that D = (256 P) * (dp * DPS - delta') needs no further scaling (powers of two).
static_assert(LG_X3_EP == 256.f, "the exponentials are taken against lse - 8 = lse - log2(LG_X3_EP)");
constexpr float XB_LN2 = 0.69314718055994530942f;

__host__ __device__ constexpr uint32_t xb_idesc(int M, int N, int b_mn_major) {  // kind::f16, fp16 x fp16 -> fp32
  return (1u << 4) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// per-instantiation scalings: BF = false is the x3 kernel (planes of 64 Q / K / V, g dO and (g / 64) D), BF = true
// uses unscaled bf16 operands
template <bool BF>
struct XbMode {
  static constexpr int NPL = BF ? 1 : 2;                  // planes per operand
  static constexpr float EA = BF ? 1.f : LG_X3_EA;        // scaling of Q, K, V (and of Y, W)
  static constexpr float DC = BF ? 1.f : XB_DC;           // D planes hold (g DC) D
  static constexpr float DT = DC / LG_X3_EP;              // delta' = delta * g * DT
  static constexpr float DPS = DT / EA;                   // dp arrives as g EA dP
  static constexpr uint32_t idesc(int M, int N, int b_mn_major) {
    return BF ? tc::idesc_bf16(M, N, b_mn_major) : xb_idesc(M, N, b_mn_major);
  }
};
__device__ __forceinline__ float xb_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// (a, b) -> fp16 pair (a in the low half), saturating at +-65504 instead of overflowing to inf
__device__ __forceinline__ uint32_t xb_pack_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// the same split with saturating conversions: a value beyond the fp16 range (possible only for activations far outside
// the |x| < 1023 contract of the x3 planes) yields finite garbage, not inf - inf = NaN
__device__ __forceinline__ void xb_split_sat(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = xb_pack_sat(a, b);
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  lo = xb_pack_sat(a - hf.x, b - hf.y);
}
// (a, b) -> fp16 pair hi and the fp16 pair of the remainders
__device__ __forceinline__ void xb_split(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 hh = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(hh);
  const __half2 ll = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&hh);
  lo = *reinterpret_cast<const uint32_t*>(&ll);
}
// (a, b) -> bf16 pair (a in the low half)
__device__ __forceinline__ uint32_t xb_pack_bf16(float a, float b) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&v);
}

// ----------------------------------------------------------------------------------------------- operand preparation
// max |dO| over the valid rows, as the bit pattern of a non-negative float (ordered like an unsigned integer)
__global__ void __launch_bounds__(256) xb_absmax_kernel(const float* __restrict__ dctx, int S, int Lp,
                                                        const int32_t* __restrict__ lens, unsigned* __restrict__ slot) {
  const size_t n4 = (size_t)S * Lp * (LG_D / 4);
  float m = 0.f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i / (LG_D / 4);
    const int s = (int)(row / Lp), l = (int)(row % Lp);
    if (lens && l >= lens[s]) continue;
    const float4 v = reinterpret_cast<const float4*>(dctx)[i];
    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    if (v.x != v.x || v.y != v.y || v.z != v.z || v.w != v.w) m = INFINITY;  // (fmaxf drops NaN)
  }
  for (int ofs = 16; ofs; ofs >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, ofs));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(slot, __float_as_uint(m));
}
// g = the power of two that brings the maximum into [256, 512); 1 for an all-zero or non-finite gradient
__global__ void xb_scale_kernel(const unsigned* __restrict__ slot, float* __restrict__ g) {
  const float m = __uint_as_float(*slot);
  float r = 1.f;
  if (m > 0.f && m < INFINITY) {
    int e;
    frexpf(m, &e);  // m = f 2^e, f in [0.5, 1)
    e = 9 - e;
    e = e < -100 ? -100 : (e > 100 ? 100 : e);
    r = ldexpf(1.f, e);
  }
  *g = r;
}
// fp32 -> head-major fp16 plane pair [2][S,4,Lp,64]; rows >= lens are zero.  token_major = 0: src is [S,4,Lp,64];
// 1: src is [S,Lp,256] (ctx layout).  scale from *gptr if given, else LG_X3_EA.
__global__ void __launch_bounds__(256) xb_split_kernel(const float* __restrict__ src, int token_major, int S, int Lp,
                                                       const int32_t* __restrict__ lens, const float* __restrict__ gptr,
                                                       __half* __restrict__ out, size_t plane) {
  const size_t n8 = (size_t)S * LG_HEADS * Lp * (LG_DH / 8);
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const int d8 = (int)(i % (LG_DH / 8));
  const size_t row = i / (LG_DH / 8);  // (s, h, l)
  const int l = (int)(row % Lp), h = (int)((row / Lp) % LG_HEADS), s = (int)(row / ((size_t)Lp * LG_HEADS));
  uint4 hi = make_uint4(0, 0, 0, 0), lo = make_uint4(0, 0, 0, 0);
  if (!lens || l < lens[s]) {
    const float sc = gptr ? *gptr : LG_X3_EA;
    const size_t off = token_major ? ((size_t)s * Lp + l) * LG_D + h * LG_DH + d8 * 8 : row * LG_DH + d8 * 8;
    const float4 a = *reinterpret_cast<const float4*>(src + off), b = *reinterpret_cast<const float4*>(src + off + 4);
    xb_split(a.x * sc, a.y * sc, hi.x, lo.x);
    xb_split(a.z * sc, a.w * sc, hi.y, lo.y);
    xb_split(b.x * sc, b.y * sc, hi.z, lo.z);
    xb_split(b.z * sc, b.w * sc, hi.w, lo.w);
  }
  *reinterpret_cast<uint4*>(out + row * LG_DH + d8 * 8) = hi;
  *reinterpret_cast<uint4*>(out + plane + row * LG_DH + d8 * 8) = lo;
}
// bf16 backward: dctx fp32 [S,Lp,256] -> dO bf16 head-major [S,4,Lp,64]; rows >= lens are zero
__global__ void __launch_bounds__(256) xb_bf16_dout_kernel(const float* __restrict__ src, int S, int Lp,
                                                           const int32_t* __restrict__ lens, __nv_bfloat16* __restrict__ out) {
  const size_t n8 = (size_t)S * LG_HEADS * Lp * (LG_DH / 8);
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const int d8 = (int)(i % (LG_DH / 8));
  const size_t row = i / (LG_DH / 8);  // (s, h, l)
  const int l = (int)(row % Lp), h = (int)((row / Lp) % LG_HEADS), s = (int)(row / ((size_t)Lp * LG_HEADS));
  uint4 o = make_uint4(0, 0, 0, 0);
  if (!lens || l < lens[s]) {
    const float* p = src + ((size_t)s * Lp + l) * LG_D + h * LG_DH + d8 * 8;
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    o = make_uint4(xb_pack_bf16(a.x, a.y), xb_pack_bf16(a.z, a.w), xb_pack_bf16(b.x, b.y), xb_pack_bf16(b.z, b.w));
  }
  *reinterpret_cast<uint4*>(out + row * LG_DH + d8 * 8) = o;
}

// ----------------------------------------------------------------------------------------------- the backward kernel
// NP = softmax threads per own row: 2 (8 warps, 32 score columns each) or 4 (16 warps, 16 columns each).
// BF: bf16 operands (Xp / Up are then bf16 rows addressed as 2-byte elements, plane unused, ctx bf16, gptr unused).
template <bool DKV, int NP, bool BF>
__global__ void __launch_bounds__(64 + 128 * NP, 1)
x3_attn_bwd_kernel(const __half* __restrict__ Xp, const __half* __restrict__ Up, size_t plane,
                   const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmW, int Lp,
                   const int32_t* __restrict__ lens, int kv_xor, const void* __restrict__ ctx,
                   const float* __restrict__ dctx, const float* __restrict__ gptr, float* __restrict__ lse2,
                   float* __restrict__ dlt, float* __restrict__ out1, float* __restrict__ out2) {
  using M = XbMode<BF>;
  constexpr int W_OFF = M::NPL * XB_TBY;  // W planes behind the Y planes of a stage
  const int h = blockIdx.y, r0 = blockIdx.x * 128, s = blockIdx.z;
  const int so = s ^ kv_xor;
  const int n_own = lens ? lens[s] : Lp, n_oth = lens ? lens[so] : Lp;
  if (r0 >= n_own || n_oth <= 0) return;  // (outputs are zero-filled by the caller; no keys: every probability is 0)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (n_oth + XB_OT - 1) / XB_OT;
  const int first_main = DKV ? 0 : n_tiles;  // DQ: iterations [0, n_tiles) are the statistics sweep
  const int n_iter = first_main + n_tiles;
  constexpr int COLS = XB_OT / NP, OC = 64 / NP;  // score / output columns per softmax thread
  constexpr int KP = COLS / 16;                   // K steps (16 other rows) inside one thread's score columns

  extern __shared__ __align__(1024) uint8_t smem[];
  if ((tc::smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + XB_BAR);
  uint64_t* xu_ready = bars;
  uint64_t* y_full = bars + 1;
  uint64_t* y_empty = y_full + XB_NST;
  uint64_t* sc_full = y_empty + XB_NST;  // [2]
  uint64_t* sc_free = sc_full + 2;       // [2] statistics sweep only
  // [2], per score buffer: a warp that is done with tile j may already arrive for tile j + 1 (its scores were issued
  // before the issuer waits for tile j's planes) while another warp still works on tile j; on ONE barrier that early
  // arrival would complete tile j's phase without the late warp's planes
  uint64_t* pd_ready = sc_free + 2;
  uint64_t* out_done = pd_ready + 2;     // one phase per flush group
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + XB_NBAR);
  float4* xch = reinterpret_cast<float4*>(smem + XB_XCH);

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&tmY);
    tc::prefetch_tmap(&tmW);
    tc::mbar_init(xu_ready, 4 * NP);
    for (int i = 0; i < XB_NST; ++i) { tc::mbar_init(&y_full[i], 1); tc::mbar_init(&y_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&sc_full[i], 1); tc::mbar_init(&sc_free[i], 4 * NP); }
    for (int i = 0; i < 2; ++i) tc::mbar_init(&pd_ready[i], 4 * NP);
    tc::mbar_init(out_done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_slot, 512);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------- TMA producer
    if (lane == 0) {
      const int oth_row = (so * LG_HEADS + h) * Lp;
      for (int it = 0; it < n_iter; ++it) {
        const int j = it < first_main ? it : it - first_main, st = it % XB_NST;
        tc::mbar_wait_relaxed(&y_empty[st], ((it / XB_NST) & 1) ^ 1);  // (sleeping polls: the issue slots belong to the softmax warps)
        uint8_t* dst = smem + XB_Y + st * 4 * XB_TBY;
        const bool main = it >= first_main;
        tc::mbar_arrive_expect_tx(&y_full[st], (main ? 2 : 1) * W_OFF);
        tc::tma_load_3d(dst, &tmY, &y_full[st], 0, oth_row + j * XB_OT, 0);
        if (!BF) tc::tma_load_3d(dst + XB_TBY, &tmY, &y_full[st], 0, oth_row + j * XB_OT, 1);
        if (main) {
          tc::tma_load_3d(dst + W_OFF, &tmW, &y_full[st], 0, oth_row + j * XB_OT, 0);
          if (!BF) tc::tma_load_3d(dst + 3 * XB_TBY, &tmW, &y_full[st], 0, oth_row + j * XB_OT, 1);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------- MMA issuer
    constexpr uint32_t idesc_sc = M::idesc(128, XB_OT, 0);
    constexpr uint32_t idesc_out = M::idesc(128, 64, 1);
    const uint32_t tXh = tmem + XT_XH, tXl = tmem + XT_XL, tUh = tmem + XT_UH, tUl = tmem + XT_UL;
    // TMEM address of the A operand of K step ks in a plane pair that a softmax thread wrote over ITS score columns:
    // [part][hi: KP steps x 8 columns | lo: KP steps x 8 columns] (BF: the hi half only, lo = 0)
    auto plane_col = [](int lo, int ks) -> uint32_t { return (uint32_t)((ks / KP) * COLS + lo * (COLS / 2) + (ks % KP) * 8); };
    auto issue_sc = [&](int it) {  // sc[it & 1] = X . Y^T and (main sweep) dp[it & 1] = U . W^T, A operands from TMEM
      const int st = it % XB_NST, b = it & 1;
      const bool main = it >= first_main;
      tc::mbar_wait_relaxed(&y_full[st], (it / XB_NST) & 1, 32);
      // The buffer's previous user is iteration it - 2.  Statistics sweep: the warps arrive on sc_free once they hold
      // the scores.  Main sweep: the warps were done with it before their pd_ready arrive, which this warp observed
      // before it issued out(it - 2); those MMAs (reading the planes in the buffer) precede the ones below in this
      // thread's MMA stream, which executes in order.
      if (it - 2 < first_main) tc::mbar_wait_relaxed(&sc_free[b], ((it >> 1) & 1) ^ 1, 32);
      tc::fence_after_sync();
      const uint32_t ybase = tc::smem_u32(smem + XB_Y + st * 4 * XB_TBY);
      const uint64_t dYh = tc::smem_desc_sw128(ybase, 0, 1024), dYl = tc::smem_desc_sw128(ybase + XB_TBY, 0, 1024);
      const uint64_t dWh = tc::smem_desc_sw128(ybase + W_OFF, 0, 1024), dWl = tc::smem_desc_sw128(ybase + 3 * XB_TBY, 0, 1024);
      const uint32_t tS = tmem + XT_SC + b * XB_OT, tP = tmem + XT_DP + b * XB_OT;
      if (tc::elect_one()) {
        if constexpr (BF) {  // one MMA per product
#pragma unroll
          for (int k = 0; k < 4; ++k) tc::umma_ts(tS, tXh + k * 8, dYh + 2 * k, idesc_sc, k != 0);
          if (main) {
#pragma unroll
            for (int k = 0; k < 4; ++k) tc::umma_ts(tP, tUh + k * 8, dWh + 2 * k, idesc_sc, k != 0);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            tc::umma_ts(tS, tXl + k * 8, dYh + 2 * k, idesc_sc, k != 0);
            tc::umma_ts(tS, tXh + k * 8, dYl + 2 * k, idesc_sc, 1);
            tc::umma_ts(tS, tXh + k * 8, dYh + 2 * k, idesc_sc, 1);
          }
          if (main) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              tc::umma_ts(tP, tUl + k * 8, dWh + 2 * k, idesc_sc, k != 0);
              tc::umma_ts(tP, tUh + k * 8, dWl + 2 * k, idesc_sc, 1);
              tc::umma_ts(tP, tUh + k * 8, dWh + 2 * k, idesc_sc, 1);
            }
          }
        }
        tc::umma_commit(&sc_full[b]);
        if (!main) tc::umma_commit(&y_empty[st]);  // the statistics sweep is done with the stage
      }
      __syncwarp();
    };
    tc::mbar_wait(xu_ready, 0);
    tc::fence_after_sync();
    issue_sc(0);
    for (int it = 0; it < n_iter; ++it) {
      if (it + 1 < n_iter) issue_sc(it + 1);
      if (it < first_main) continue;
      const int jm = it - first_main, st = it % XB_NST, b = it & 1;
      tc::mbar_wait_relaxed(&pd_ready[b], (jm >> 1) & 1, 32);
      tc::fence_after_sync();
      const uint32_t ybase = tc::smem_u32(smem + XB_Y + st * 4 * XB_TBY);
      // MN-major B operands: row = other row (the K index of these MMAs), 16 rows = 2048 B per K step
      const uint64_t mYh = tc::smem_desc_sw128(ybase, XB_TBY, 1024), mYl = tc::smem_desc_sw128(ybase + XB_TBY, XB_TBY, 1024);
      const uint64_t mWh = tc::smem_desc_sw128(ybase + W_OFF, XB_TBY, 1024), mWl = tc::smem_desc_sw128(ybase + 3 * XB_TBY, XB_TBY, 1024);
      const uint32_t tD = tmem + XT_DP + b * XB_OT, tPp = tmem + XT_SC + b * XB_OT;  // D planes over dp, P planes over sc
      if (tc::elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t acc = ((jm % XB_FLUSH) | k) != 0;  // fresh accumulators after every flush
          if constexpr (BF) {
            tc::umma_ts(tmem + XT_O1, tD + plane_col(0, k), mYh + k * (2048 >> 4), idesc_out, acc);
            if (DKV) tc::umma_ts(tmem + XT_O2, tPp + plane_col(0, k), mWh + k * (2048 >> 4), idesc_out, acc);
            continue;
          }
          tc::umma_ts(tmem + XT_O1, tD + plane_col(1, k), mYh + k * (2048 >> 4), idesc_out, acc);
          tc::umma_ts(tmem + XT_O1, tD + plane_col(0, k), mYl + k * (2048 >> 4), idesc_out, 1);
          tc::umma_ts(tmem + XT_O1, tD + plane_col(0, k), mYh + k * (2048 >> 4), idesc_out, 1);
          if (DKV) {
            tc::umma_ts(tmem + XT_O2, tPp + plane_col(1, k), mWh + k * (2048 >> 4), idesc_out, acc);
            tc::umma_ts(tmem + XT_O2, tPp + plane_col(0, k), mWl + k * (2048 >> 4), idesc_out, 1);
            tc::umma_ts(tmem + XT_O2, tPp + plane_col(0, k), mWh + k * (2048 >> 4), idesc_out, 1);
          }
        }
        tc::umma_commit(&y_empty[st]);
        if (jm % XB_FLUSH == XB_FLUSH - 1 || jm == n_tiles - 1) tc::umma_commit(out_done);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------------------------------- softmax warps
    const int quarter = warp & 3;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const int part = (warp - 2) >> 2;  // which COLS columns of every score tile / OC columns of the outputs
    auto ld_cols = [&](uint32_t col, uint32_t* dst) {  // COLS (= OC) consecutive TMEM columns of this thread's lane
      if constexpr (COLS == 32) tc::tmem_ld32(tmem + lane_base + col, dst);
      else tc::tmem_ld16(tmem + lane_base + col, dst);
    };
    auto st_plane = [&](uint32_t col, const uint32_t* src) {  // COLS / 2 packed fp16 pairs
      if constexpr (COLS == 32) tc::tmem_st16(tmem + lane_base + col, src);
      else tc::tmem_st8(tmem + lane_base + col, src);
    };
    const int r = quarter * 32 + lane;
    const bool row_ok = r0 + r < n_own;
    constexpr float s_us = 1.f / (M::EA * M::EA);
    const float g = BF ? 1.f : *gptr;
    const size_t own_stat = ((size_t)s * LG_HEADS + h) * Lp + r0 + r;
    const size_t oth_stat = ((size_t)so * LG_HEADS + h) * Lp;
    float lse_own = 0.f, dlt_own = 0.f;  // DQ: this row's log-sum-exp and g * delta

    // ---- own rows into TMEM: the A operand of every score MMA (rows >= n_own are zero planes).  This thread copies
    // words [part * 32 / NP, ...) of its row of X hi, X lo, U hi, U lo (a word = two fp16 = one TMEM column)
    {
      constexpr int NW = 32 / NP;
      const __half* srcs[4] = {Xp + own_stat * LG_DH, Xp + plane + own_stat * LG_DH, Up + own_stat * LG_DH,
                               Up + plane + own_stat * LG_DH};
      const uint32_t cols[4] = {XT_XH, XT_XL, XT_UH, XT_UL};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (BF && (q & 1)) continue;  // (no lo planes)
        uint32_t w[NW];
        const uint4* src = reinterpret_cast<const uint4*>(srcs[q]) + part * (NW / 4);
#pragma unroll
        for (int i = 0; i < NW / 4; ++i) {
          const uint4 v = src[i];
          w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
        }
        if constexpr (NW == 16) tc::tmem_st16(tmem + lane_base + cols[q] + part * NW, w);
        else tc::tmem_st8(tmem + lane_base + cols[q] + part * NW, w);
      }
      tc::tmem_st_wait();
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(xu_ready);
    }

    if (!DKV) {
      // ---- statistics sweep: every thread keeps the online (max, sum) of ITS columns; partial states merge
      // associatively, so the NP threads of a row are combined once, after the sweep
      float m = -INFINITY, l = 0.f;
      for (int it = 0; it < n_tiles; ++it) {
        const int b = it & 1;
        tc::mbar_wait(&sc_full[b], (it >> 1) & 1);
        tc::fence_after_sync();
        uint32_t sv[COLS];
        ld_cols(XT_SC + b * XB_OT + part * COLS, sv);
        tc::tmem_ld_wait();
        tc::fence_before_sync();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&sc_free[b]);
        const int valid = n_oth - it * XB_OT - part * COLS;
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < COLS; ++i) {
          if (i >= valid) sv[i] = 0xff800000u;  // -inf
          mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(sv[i]));
        }
        const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])) * s_us;
        const float mnew = fmaxf(m, mx);
        const float msafe = mnew == -INFINITY ? 0.f : mnew;
        float rs4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < COLS; ++i) rs4[i & 3] += xb_ex2(fmaf(__uint_as_float(sv[i]), s_us, -msafe));
        l = l * xb_ex2(m - msafe) + ((rs4[0] + rs4[1]) + (rs4[2] + rs4[3]));
        m = mnew;
      }
      float dot = 0.f;
      if (row_ok) {
        const size_t off = ((size_t)s * Lp + r0 + r) * LG_D + h * LG_DH + part * OC;
        if constexpr (BF) {
#pragma unroll
          for (int i = 0; i < OC / 8; ++i) {
            const uint4 o = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(ctx) + off + 8 * i);
            const float4 ga = *reinterpret_cast<const float4*>(dctx + off + 8 * i);
            const float4 gb = *reinterpret_cast<const float4*>(dctx + off + 8 * i + 4);
            const float2 o0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o.x));
            const float2 o1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o.y));
            const float2 o2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o.z));
            const float2 o3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o.w));
            dot += (o0.x * ga.x + o0.y * ga.y) + (o1.x * ga.z + o1.y * ga.w);
            dot += (o2.x * gb.x + o2.y * gb.y) + (o3.x * gb.z + o3.y * gb.w);
          }
        } else {
#pragma unroll
          for (int i = 0; i < OC / 4; ++i) {
            const float4 o = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ctx) + off + 4 * i);
            const float4 gr = *reinterpret_cast<const float4*>(dctx + off + 4 * i);
            dot += (o.x * gr.x + o.y * gr.y) + (o.z * gr.z + o.w * gr.w);
          }
        }
      }
      xch[r * NP + part] = make_float4(m, l, dot, 0.f);
      asm volatile("bar.sync %0, %1;" ::"r"(1 + quarter), "n"(32 * NP) : "memory");
      float4 pt[NP];
#pragma unroll
      for (int i = 0; i < NP; ++i) pt[i] = xch[r * NP + i];
      float mnew = pt[0].x;
#pragma unroll
      for (int i = 1; i < NP; ++i) mnew = fmaxf(mnew, pt[i].x);
      const float msafe = mnew == -INFINITY ? 0.f : mnew;
      float lsum = 0.f, delta = 0.f;
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        lsum += pt[i].y * xb_ex2(pt[i].x - msafe);
        delta += pt[i].z;
      }
      lse_own = lsum > 0.f ? mnew + log2f(lsum) - 8.f : INFINITY;  // (2^(s - lse_own) = 256 P)
      dlt_own = delta * g * M::DT;
      if (part == 0 && row_ok) {
        lse2[own_stat] = lse_own;
        dlt[own_stat] = dlt_own;
      }
    }

    // ---- running sums of this thread's OC (+OC) output columns, [column][row] in shared memory
    float* racc = reinterpret_cast<float*>(smem + XB_ACC) + r;
    if (!DKV) asm volatile("bar.sync 5, %0;" ::"n"(128 * NP) : "memory");  // every softmax thread has read xch (aliased with the sums)
#pragma unroll
    for (int i = 0; i < OC; ++i) {
      racc[(part * OC + i) * 128] = 0.f;
      if (DKV) racc[(64 + part * OC + i) * 128] = 0.f;
    }
    auto flush = [&]() {  // TMEM accumulators (complete: out_done observed) -> running sums, round to nearest
      uint32_t o[OC];
      ld_cols(XT_O1 + part * OC, o);
      tc::tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < OC; ++i) racc[(part * OC + i) * 128] += __uint_as_float(o[i]);
      if (DKV) {
        ld_cols(XT_O2 + part * OC, o);
        tc::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < OC; ++i) racc[(64 + part * OC + i) * 128] += __uint_as_float(o[i]);
      }
    };

    // ---- main sweep
    for (int it = first_main; it < n_iter; ++it) {
      const int jm = it - first_main, b = it & 1;
      const int n0 = jm * XB_OT + part * COLS;  // first other row of this thread's columns
      // DKV: per-column statistics of the queries (uniform over the warp: broadcast loads), fetched BEFORE the wait for
      // the score MMAs -- issued at their first use, the ~700-cycle L2 round trip sat on the critical path of every tile
      // (21 % of the role's stall samples, profiles/r2_attn_bwd_tcgen05.txt)
      float4 lq4[DKV ? COLS / 4 : 1], dq4[DKV ? COLS / 4 : 1];
      if (DKV) {
#pragma unroll
        for (int i4 = 0; i4 < COLS / 4; ++i4) {
          lq4[i4] = *reinterpret_cast<const float4*>(lse2 + oth_stat + n0 + 4 * i4);
          dq4[i4] = *reinterpret_cast<const float4*>(dlt + oth_stat + n0 + 4 * i4);
        }
      }
      tc::mbar_wait(&sc_full[b], (it >> 1) & 1);
      tc::fence_after_sync();
      uint32_t sv[COLS], dv[COLS];
      ld_cols(XT_SC + b * XB_OT + part * COLS, sv);
      ld_cols(XT_DP + b * XB_OT + part * COLS, dv);
      tc::tmem_ld_wait();
      uint32_t dh[COLS / 2], dl[COLS / 2], ph[COLS / 2], pl[COLS / 2];
      auto planes = [&](auto full_tile) {  // full_tile: every column of this thread is a valid other row (no masks)
        constexpr bool FULL = decltype(full_tile)::value;
#pragma unroll
        for (int i4 = 0; i4 < COLS / 4; ++i4) {
          float lq[4], dq[4];
          if (DKV) {
            const float4 l4 = lq4[i4], d4 = dq4[i4];
            lq[0] = l4.x; lq[1] = l4.y; lq[2] = l4.z; lq[3] = l4.w;
            dq[0] = d4.x; dq[1] = d4.y; dq[2] = d4.z; dq[3] = d4.w;
          } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) { lq[c] = lse_own; dq[c] = dlt_own; }
          }
          float p[4], d[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int i = 4 * i4 + c;
            const bool ok = FULL || n0 + i < n_oth;  // (statistics of padding rows are undefined: select, not multiply)
            p[c] = ok ? xb_ex2(fmaf(__uint_as_float(sv[i]), s_us, -lq[c])) : 0.f;            // 256 P
            d[c] = ok ? p[c] * fmaf(__uint_as_float(dv[i]), M::DPS, -dq[c]) : 0.f;           // (g DC) P (dP - delta)
          }
          if constexpr (BF) {
            dh[2 * i4] = xb_pack_bf16(d[0], d[1]);
            dh[2 * i4 + 1] = xb_pack_bf16(d[2], d[3]);
            if (DKV) {
              ph[2 * i4] = xb_pack_bf16(p[0], p[1]);
              ph[2 * i4 + 1] = xb_pack_bf16(p[2], p[3]);
            }
            continue;
          }
          xb_split_sat(d[0], d[1], dh[2 * i4], dl[2 * i4]);
          xb_split_sat(d[2], d[3], dh[2 * i4 + 1], dl[2 * i4 + 1]);
          if (DKV) {
            xb_split(p[0], p[1], ph[2 * i4], pl[2 * i4]);
            xb_split(p[2], p[3], ph[2 * i4 + 1], pl[2 * i4 + 1]);
          }
        }
      };
      if (n0 + COLS <= n_oth) planes(std::true_type{});
      else planes(std::false_type{});
      if (jm > 0 && jm % XB_FLUSH == 0) {
        // the group's MMAs have retired; the issuer starts fresh accumulators with tile jm only after this warp's
        // pd_ready arrive below
        tc::mbar_wait(out_done, (jm / XB_FLUSH - 1) & 1);
        tc::fence_after_sync();
        flush();
      }
      // the plane pairs go over this thread's OWN score columns (hi | lo), read above: no other thread touches them
      st_plane(XT_DP + b * XB_OT + part * COLS, dh);
      if (!BF) st_plane(XT_DP + b * XB_OT + part * COLS + COLS / 2, dl);
      if (DKV) {
        st_plane(XT_SC + b * XB_OT + part * COLS, ph);
        if (!BF) st_plane(XT_SC + b * XB_OT + part * COLS + COLS / 2, pl);
      }
      tc::tmem_st_wait();
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&pd_ready[b]);
    }
    // ---- epilogue: this thread's OC output columns of its row
    tc::mbar_wait(out_done, ((n_tiles + XB_FLUSH - 1) / XB_FLUSH - 1) & 1);
    tc::fence_after_sync();
    flush();
    if (row_ok) {
      const float k1 = XB_LN2 / (g * M::DC * M::EA);  // raw = ((g DC) D) . (EA Y)
      float4* dst = reinterpret_cast<float4*>(out1 + own_stat * LG_DH + part * OC);
#pragma unroll
      for (int i = 0; i < OC / 4; ++i)
        dst[i] = make_float4(racc[(part * OC + 4 * i) * 128] * k1, racc[(part * OC + 4 * i + 1) * 128] * k1,
                             racc[(part * OC + 4 * i + 2) * 128] * k1, racc[(part * OC + 4 * i + 3) * 128] * k1);
      if (DKV) {
        const float k2 = 1.f / (g * LG_X3_EP);  // raw = (256 P) . (g dO)
        float4* dst2 = reinterpret_cast<float4*>(out2 + own_stat * LG_DH + part * OC);
#pragma unroll
        for (int i = 0; i < OC / 4; ++i)
          dst2[i] = make_float4(racc[(64 + part * OC + 4 * i) * 128] * k2, racc[(64 + part * OC + 4 * i + 1) * 128] * k2,
                                racc[(64 + part * OC + 4 * i + 2) * 128] * k2, racc[(64 + part * OC + 4 * i + 3) * 128] * k2);
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem, 512);
  }
}

}  // namespace

size_t lg_x3_attention_bwd_ws_floats(int S, int Lp) {
  return 2 * (size_t)S * LG_HEADS * Lp + 16 + 4 * (size_t)S * Lp * LG_D;
}

// Q, K, V fp32 [S,4,Lp,64]; ctx, dctx fp32 [S,Lp,256]; dQ, dK, dV fp32 [S,4,Lp,64] (zero-filled by the caller);
// ws: lg_x3_attention_bwd_ws_floats(S, Lp) floats.
int lg_x3_attention_bwd(const float* Q, const float* K, const float* V, const float* ctx, const float* dctx, int S,
                        int Lp, const int32_t* lens, int kv_xor, float* dQ, float* dK, float* dV, float* ws,
                        cudaStream_t st) {
  const size_t n_stat = (size_t)S * LG_HEADS * Lp, n_el = (size_t)S * Lp * LG_D;
  float* lse2 = ws;
  float* dlt = ws + n_stat;
  unsigned* slot = reinterpret_cast<unsigned*>(ws + 2 * n_stat);
  float* g = ws + 2 * n_stat + 1;
  __half* planes = reinterpret_cast<__half*>(ws + 2 * n_stat + 16);
  __half* Qp = planes;
  __half* Kp = K == Q ? Qp : planes + 2 * n_el;
  __half* Vp = planes + 4 * n_el;
  __half* Gp = planes + 6 * n_el;
  cudaError_t e;
  if ((e = cudaMemsetAsync(slot, 0, sizeof(unsigned), st)) != cudaSuccess) return (int)e;
  xb_absmax_kernel<<<592, 256, 0, st>>>(dctx, S, Lp, lens, slot);
  LG_LAUNCH_CHECK();
  xb_scale_kernel<<<1, 1, 0, st>>>(slot, g);
  LG_LAUNCH_CHECK();
  const unsigned nb = (unsigned)((n_el / 8 + 255) / 256);
  xb_split_kernel<<<nb, 256, 0, st>>>(Q, 0, S, Lp, lens, nullptr, Qp, n_el);
  LG_LAUNCH_CHECK();
  if (Kp != Qp) {
    xb_split_kernel<<<nb, 256, 0, st>>>(K, 0, S, Lp, lens, nullptr, Kp, n_el);
    LG_LAUNCH_CHECK();
  }
  xb_split_kernel<<<nb, 256, 0, st>>>(V, 0, S, Lp, lens, nullptr, Vp, n_el);
  LG_LAUNCH_CHECK();
  xb_split_kernel<<<nb, 256, 0, st>>>(dctx, 1, S, Lp, lens, g, Gp, n_el);
  LG_LAUNCH_CHECK();

  CUtensorMap tq, tk, tv, tg;
  const uint64_t rows = (uint64_t)S * LG_HEADS * Lp;
  const uint64_t d[3] = {64, rows, 2}, sb[2] = {128, rows * 128};
  const uint32_t box[3] = {64, 64, 1};
  int rc;
  if ((rc = lg_make_tmap_bf16(&tq, Qp, 3, d, sb, box))) return rc;
  if ((rc = lg_make_tmap_bf16(&tk, Kp, 3, d, sb, box))) return rc;
  if ((rc = lg_make_tmap_bf16(&tv, Vp, 3, d, sb, box))) return rc;
  if ((rc = lg_make_tmap_bf16(&tg, Gp, 3, d, sb, box))) return rc;
  // softmax threads per own row, per role (LGB200_X3_BWD_NP = "<dq><dkv>", e.g. 24)
  static const int np_cfg = getenv("LGB200_X3_BWD_NP") ? atoi(getenv("LGB200_X3_BWD_NP")) : 44;
  const dim3 grid(Lp / 128, LG_HEADS, S);
  auto launch = [&](auto kern, int np, const __half* xp, const __half* up, const CUtensorMap& ty, const CUtensorMap& tw,
                    float* o1, float* o2) -> int {
    cudaError_t le = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, XB_SMEM);
    if (le != cudaSuccess) return (int)le;
    kern<<<grid, 64 + 128 * np, XB_SMEM, st>>>(xp, up, n_el, ty, tw, Lp, lens, kv_xor, ctx, dctx, g, lse2, dlt, o1, o2);
    LG_LAUNCH_CHECK();
    return LGB200_OK;
  };
  if (np_cfg / 10 == 2) rc = launch(x3_attn_bwd_kernel<false, 2, false>, 2, Qp, Gp, tk, tv, dQ, nullptr);
  else rc = launch(x3_attn_bwd_kernel<false, 4, false>, 4, Qp, Gp, tk, tv, dQ, nullptr);
  if (rc) return rc;
  if (np_cfg % 10 == 2) rc = launch(x3_attn_bwd_kernel<true, 2, false>, 2, Kp, Vp, tq, tg, dK, dV);
  else rc = launch(x3_attn_bwd_kernel<true, 4, false>, 4, Kp, Vp, tq, tg, dK, dV);
  return rc;
}

size_t lg_bf16_attention_bwd_ws_floats(int S, int Lp) {
  return 2 * (size_t)S * LG_HEADS * Lp + 16 + (size_t)S * Lp * LG_D / 2;
}

// Q, K, V bf16 [S,4,Lp,64] as the bf16 forward read them (rows >= lens finite); ctx bf16 [S,Lp,256] (the forward's
// output), dctx fp32 [S,Lp,256]; dQ, dK, dV fp32 [S,4,Lp,64] (zero-filled by the caller);
// ws: lg_bf16_attention_bwd_ws_floats(S, Lp) floats (row statistics | head-major bf16 dO).
int lg_bf16_attention_bwd(const __nv_bfloat16* Q, const __nv_bfloat16* K, const __nv_bfloat16* V,
                          const __nv_bfloat16* ctx, const float* dctx, int S, int Lp, const int32_t* lens, int kv_xor,
                          float* dQ, float* dK, float* dV, float* ws, cudaStream_t st) {
  const size_t n_stat = (size_t)S * LG_HEADS * Lp, n_el = (size_t)S * Lp * LG_D;
  float* lse2 = ws;
  float* dlt = ws + n_stat;
  __nv_bfloat16* Gp = reinterpret_cast<__nv_bfloat16*>(ws + 2 * n_stat + 16);
  xb_bf16_dout_kernel<<<(unsigned)((n_el / 8 + 255) / 256), 256, 0, st>>>(dctx, S, Lp, lens, Gp);
  LG_LAUNCH_CHECK();

  CUtensorMap tq, tk, tv, tg;
  const uint64_t rows = (uint64_t)S * LG_HEADS * Lp;
  const uint64_t d[3] = {64, rows, 1}, sb[2] = {128, rows * 128};
  const uint32_t box[3] = {64, 64, 1};
  int rc;
  if ((rc = lg_make_tmap_bf16(&tq, Q, 3, d, sb, box))) return rc;
  if ((rc = lg_make_tmap_bf16(&tk, K, 3, d, sb, box))) return rc;
  if ((rc = lg_make_tmap_bf16(&tv, V, 3, d, sb, box))) return rc;
  if ((rc = lg_make_tmap_bf16(&tg, Gp, 3, d, sb, box))) return rc;
  // softmax threads per own row, per role (LGB200_BF16_BWD_NP = "<dq><dkv>", e.g. 24)
  static const int np_cfg = getenv("LGB200_BF16_BWD_NP") ? atoi(getenv("LGB200_BF16_BWD_NP")) : 44;
  const dim3 grid(Lp / 128, LG_HEADS, S);
  auto h = [](const __nv_bfloat16* p) { return reinterpret_cast<const __half*>(p); };  // (2-byte rows, see the kernel)
  auto launch = [&](auto kern, int np, const __nv_bfloat16* xp, const __nv_bfloat16* up, const CUtensorMap& ty,
                    const CUtensorMap& tw, float* o1, float* o2) -> int {
    cudaError_t le = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, XB_SMEM);
    if (le != cudaSuccess) return (int)le;
    kern<<<grid, 64 + 128 * np, XB_SMEM, st>>>(h(xp), h(up), 0, ty, tw, Lp, lens, kv_xor, ctx, dctx, nullptr, lse2, dlt,
                                               o1, o2);
    LG_LAUNCH_CHECK();
    return LGB200_OK;
  };
  if (np_cfg / 10 == 2) rc = launch(x3_attn_bwd_kernel<false, 2, true>, 2, Q, Gp, tk, tv, dQ, nullptr);
  else rc = launch(x3_attn_bwd_kernel<false, 4, true>, 4, Q, Gp, tk, tv, dQ, nullptr);
  if (rc) return rc;
  if (np_cfg % 10 == 2) rc = launch(x3_attn_bwd_kernel<true, 2, true>, 2, K, V, tq, tg, dK, dV);
  else rc = launch(x3_attn_bwd_kernel<true, 4, true>, 4, K, V, tq, tg, dK, dV);
  return rc;
}
