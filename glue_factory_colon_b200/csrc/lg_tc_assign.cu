// MatchAssignment on tcgen05 (sm_100a): similarity GEMM fused with the dual log-softmax.
//
// Both passes run the same strip kernel: a CTA owns 128 rows of md[s] (resident in smem, K = 256)
// and sweeps the 128-row tiles of the other image md[s^1] (TMA, 2-stage ring); each 128x128
// similarity tile is produced by 16 tcgen05.mma into one of two TMEM accumulators so the MMAs
// of tile j+1 overlap the epilogue of tile j.
//   pass 1 (SCORES = false): epilogue keeps an online (max, sum-exp) per row -> lse[s, row].
//          Run for every sequence: rows of image 0 give the row normaliser, rows of image 1 the
//          column normaliser.  Nothing N x M is written.
//   pass 2 (SCORES = true):  epilogue forms 2*sim - lse0[i] - lse1[j] + logsigmoid(z0[i]) +
//          logsigmoid(z1[j]) and writes the fp32 score tile ONCE; tiles are transposed through
//          shared memory so that every warp store is a contiguous 128-byte row segment.
// The N x M matrix is therefore never materialised before its final form and never re-read.
#include "lg_internal.cuh"
#include "lg_tc_common.cuh"

namespace {

constexpr int AS_TILE = 128 * 64 * 2;        // one 128-row x 64-col bf16 box (16 KB)
constexpr int AS_OPER = 4 * AS_TILE;         // 128 rows x K=256 (64 KB)
constexpr int AS_STAGE_OFF = AS_OPER;        // the B ring follows A
#ifndef LG_ASSIGN_WARPS
#define LG_ASSIGN_WARPS 16
#endif
// Epilogue warps: (TMEM lane quarter) x (column part of the tile).  r1 had 8 (two 32-column chunks per warp and tile)
// beside two full 64 KB B stages, and pass 2 was latency-bound at one CTA per SM (issue 38 % active, DRAM 24 %).
// r2: 16 warps, one 32-column chunk each; to make room for their transpose tiles the B operand streams through a ring
// of AS_RING K-boxes of 16 KB (a tile's 16 MMAs take ~1 000 tensor cycles of the ~4 000+ its epilogue needs, so the
// shallower prefetch costs nothing).
#ifndef LG_ASSIGN_CL
#define LG_ASSIGN_CL 1
#endif
// Optional (-DLG_ASSIGN_CL=2): the two CTAs of neighbouring strips form a cluster and share every B box (each loads 64
// of its 128 rows and TMA-multicasts them to both), halving the L2->SM stream (2 048 CTAs x 1 MB at 64 x 2048).  Measured
// on B200: pass 1 270 vs 255 us, pass 2 443 vs 433 us -- the L2 stream is not the limiter, so the default stays 1.
constexpr int AS_CL = LG_ASSIGN_CL;          // CTAs (row strips) that share the B stream: 1 or 2
constexpr int AS_EPI_WARPS = LG_ASSIGN_WARPS;
constexpr int AS_PARTS = AS_EPI_WARPS / 4;   // column parts of a 128-column tile (2 or 4)
constexpr int AS_PCOLS = 128 / AS_PARTS;     // columns per warp and tile (64 or 32)
constexpr int AS_RING = AS_EPI_WARPS == 16 ? 5 : 8;  // B ring depth in K-boxes (8 = the two full stages of r1)
constexpr int AS_BAR_OFF = AS_OPER + AS_RING * AS_TILE;
constexpr int AS_XPOSE_OFF = AS_BAR_OFF + 256;
constexpr int AS_THREADS = (2 + AS_EPI_WARPS) * 32;
constexpr int AS_XP = 32 * 33;               // floats of one warp's 32 x 32 transpose tile (padded)
constexpr int AS_SMEM = AS_XPOSE_OFF + AS_EPI_WARPS * (AS_XP + 32) * 4;

__device__ __forceinline__ float ex2a(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// (value, index) update for torch.max semantics: the candidate with the HIGHER index (b) replaces the running one
// only if it is strictly larger, or if it is the first NaN.  (A depth-5 tournament tree over the 32 candidates of
// a chunk was tried against this serial chain: 827 us vs 628 us for pass 2 -- more selects than it saved stalls.)
__device__ __forceinline__ void amax_merge(float& va, int& ia, float vb, int ib) {
  if (vb > va || (vb != vb && va == va)) { va = vb; ia = ib; }
}

// First arg-max of 32 candidates held in registers, torch.max semantics (lowest index among equal maxima; the
// first NaN if there is one).  The serial chain above is 32 dependent compare -> select steps (~300 cycles with two
// warps per scheduler to hide them); here a NaN-propagating maximum tree of depth 5, then 32 independent equality
// tests collected in a bit mask whose lowest set bit is the answer.  `max.NaN` makes the tree return NaN iff a
// candidate is NaN, and only then (inputs that are already garbage) the mask is built from `v != v` instead.
__device__ __forceinline__ float max_nan(float a, float b) {
  float d;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
__device__ __forceinline__ void chunk_argmax(const float (&v)[32], float& best, int& idx) {
  float m[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) m[i] = max_nan(max_nan(v[i], v[i + 8]), max_nan(v[i + 16], v[i + 24]));
  const float mx = max_nan(max_nan(max_nan(m[0], m[1]), max_nan(m[2], m[3])),
                           max_nan(max_nan(m[4], m[5]), max_nan(m[6], m[7])));
  uint32_t mask[4] = {0u, 0u, 0u, 0u};
  if (mx == mx) {
#pragma unroll
    for (int i = 0; i < 32; ++i) mask[i & 3] |= (v[i] == mx) ? (1u << i) : 0u;
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) mask[i & 3] |= (v[i] != v[i]) ? (1u << i) : 0u;
  }
  idx = __ffs((int)((mask[0] | mask[1]) | (mask[2] | mask[3]))) - 1;
  best = mx;
}

// Epilogue history: the first version had 4 epilogue warps and a rolled, dependent LDS -> FADD -> STG loop per
// output row, and fetched z / lse for the column constants on the critical path of every chunk; pass 2 wrote its
// 1.075 GB at 0.88 TB/s (1.30 ms at 64 pairs x 2048).  Now 8 warps, each owning 32 rows x 64 columns of a tile,
// finished values staged transposed in shared memory, an unrolled store loop (32 independent 128-byte row
// segments in flight per warp) and the column constants prefetched one chunk ahead: 0.63 ms (1.9 TB/s).
// LOSS (third mode, SURVEY.md 8(f) rank 2): pass 2 without the store -- the finished values feed, per row, the sums
// sum_j la*gt, sum_j gt and sum_j exp(la) (weight_loss / row_norm of LightGlue.loss) and the two arg-maxima
// (TokenConfidence.loss); the N x M matrix of an intermediate layer is never written at all.
struct AsLoss {
  const uint8_t* gt;  // [B, R-1, C-1] bool
  float* row_pos;     // [B, R-1] each, zero-initialised: the two column halves of a row add into them (a + b is
  float* row_cnt;     // commutative, so the result does not depend on which half arrives first)
  float* row_exp;
};

template <int MODE>
__global__ void __launch_bounds__(AS_THREADS, 1)
tc_assign_kernel(const __grid_constant__ CUtensorMap tmMd, const __grid_constant__ CUtensorMap tmB, int Lp,
                 const int32_t* __restrict__ lens,
                 const float* __restrict__ z, const float* __restrict__ lse_in, float* __restrict__ lse_out,
                 int R, int C, float* __restrict__ scores, unsigned long long* __restrict__ best0,
                 unsigned long long* __restrict__ best1, AsLoss ls) {
  constexpr bool SCORES = MODE != 0;  // passes 2 (scores written) and 3 (loss reductions)
  constexpr bool LOSS = MODE == 2;
  // SCORES: blockIdx.y = pair b, rows from sequence 2b.  LSE: blockIdx.y = sequence s.
  const int s = SCORES ? 2 * blockIdx.y : blockIdx.y;
  const int so = s ^ 1;
  const int m0 = blockIdx.x * 128;
  const int nq = lens ? lens[s] : (SCORES ? R - 1 : Lp);
  const int nk = lens ? lens[so] : (SCORES ? C - 1 : Lp);
  const uint32_t crank = AS_CL > 1 ? tc::cluster_ctarank() : 0;
  constexpr uint16_t MC_MASK = (uint16_t)((1u << AS_CL) - 1);
  if ((int)(blockIdx.x - crank) * 128 >= nq) return;  // the whole cluster is past the valid rows
  // (a CTA whose own strip is past the valid rows but whose partner's is not runs the pipeline for the partner's
  // sake -- its half of every B box -- and stores nothing: every store below is guarded by row < nq)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (nk + 127) / 128;
  if (n_tiles == 0) {
    if (!SCORES && warp >= 2 && warp < 6) {
      const int r = (warp & 3) * 32 + lane;
      if (m0 + r < nq) lse_out[(size_t)s * Lp + m0 + r] = 0.f;
    }
    return;
  }

  extern __shared__ __align__(1024) uint8_t smem[];
  if ((tc::smem_u32(smem) & 1023u) != 0) __trap();  // swizzled tiles need a 1024-byte aligned base
  uint8_t* sA = smem;
  uint8_t* sB = smem + AS_STAGE_OFF;  // ring of AS_RING K-boxes
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + AS_BAR_OFF);
  uint64_t* a_full = bars;
  uint64_t* b_full = bars + 1;              // [AS_RING]
  uint64_t* b_empty = b_full + AS_RING;     // [AS_RING]
  uint64_t* s_full = b_empty + AS_RING;     // [2]
  uint64_t* s_empty = s_full + 2;           // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_empty + 2);
  float* xpose = reinterpret_cast<float*>(smem + AS_XPOSE_OFF);

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&tmMd);
    tc::mbar_init(a_full, 1);
    for (int i = 0; i < AS_RING; ++i) {
      tc::mbar_init(&b_full[i], 1);
      tc::mbar_init(&b_empty[i], AS_CL);  // every CTA that reads the box releases it in every CTA that refills it
    }
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&s_full[i], 1);
      tc::mbar_init(&s_empty[i], AS_EPI_WARPS);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_slot, 256);
  tc::fence_before_sync();
  __syncthreads();
  if (AS_CL > 1) tc::cluster_sync();  // the peer's barriers exist before anyone multicasts into them
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      tc::mbar_arrive_expect_tx(a_full, AS_OPER);
      for (int kb = 0; kb < 4; ++kb) tc::tma_load_2d(sA + kb * AS_TILE, &tmMd, a_full, kb * 64, s * Lp + m0);
      int slot = 0;
      uint32_t ph = 0;
      for (int j = 0; j < n_tiles; ++j) {
        for (int kb = 0; kb < 4; ++kb) {
          tc::mbar_wait(&b_empty[slot], ph ^ 1);
          tc::mbar_arrive_expect_tx(&b_full[slot], AS_TILE);
          if (AS_CL > 1) {
            constexpr int SL = 128 / AS_CL;  // rows of the box this CTA fetches for everybody
            tc::tma_load_2d_mc(sB + slot * AS_TILE + crank * SL * 128, &tmB, &b_full[slot], kb * 64,
                               so * Lp + j * 128 + (int)crank * SL, MC_MASK);
          } else {
            tc::tma_load_2d(sB + slot * AS_TILE, &tmMd, &b_full[slot], kb * 64, so * Lp + j * 128);
          }
          if (++slot == AS_RING) { slot = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // whole warp, warp-uniform control flow, one elected lane issues (descriptors stay in uniform registers)
    constexpr uint32_t idesc = tc::idesc_bf16(128, 128, 0);
    const uint64_t dA = tc::smem_desc_sw128(tc::smem_u32(sA), 0, 1024);
    const uint64_t dB0 = tc::smem_desc_sw128(tc::smem_u32(sB), 0, 1024);
    tc::mbar_wait(a_full, 0);
    int slot = 0;
    uint32_t bph = 0;
    for (int j = 0; j < n_tiles; ++j) {
      const int st = j & 1;
      const uint32_t ph = (j >> 1) & 1;
      tc::mbar_wait(&s_empty[st], ph ^ 1);
      for (int kb = 0; kb < 4; ++kb) {
        tc::mbar_wait(&b_full[slot], bph);
        tc::fence_after_sync();
        const uint64_t dB = dB0 + (uint64_t)(slot * (AS_TILE >> 4));
        if (tc::elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            tc::umma_ss(tmem + st * 128, dA + kb * (AS_TILE >> 4) + 2 * k, dB + 2 * k, idesc, (kb | k) != 0);
          if (AS_CL > 1) tc::umma_commit_mc(&b_empty[slot], MC_MASK);
          else tc::umma_commit(&b_empty[slot]);
          if (kb == 3) tc::umma_commit(&s_full[st]);
        }
        __syncwarp();
        if (++slot == AS_RING) { slot = 0; bph ^= 1; }
      }
    }
  } else {
    const int ew = warp - 2;
    const int quarter = warp & 3;   // TMEM lane quarter this warp may read
    const int half = ew >> 2;       // column part of every tile (AS_PCOLS columns)
    const int r = quarter * 32 + lane;
    const int row = m0 + r;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    float m_run = -INFINITY, l_run = 0.f;
    float rowconst = 0.f;
    if (SCORES && row < nq) rowconst = lg_logsigmoid(z[(size_t)s * Lp + row]) - lse_in[(size_t)s * Lp + row];
    float* xp = xpose + ew * (AS_XP + 32);
    float* xc = xp + AS_XP;      // this chunk's 32 column constants
    float rbest = -INFINITY;     // fused filter_matches: running row argmax over this warp's columns
    int ridx = 0;
    float a_pos = 0.f, a_cnt = 0.f, a_exp = 0.f;  // LOSS: this thread's row, this warp's columns
    const bool gt16 = LOSS && ((C - 1) % 16 == 0) && ((reinterpret_cast<uintptr_t>(ls.gt) & 15) == 0);
    float pf_z = 0.f, pf_lse = 0.f;  // prefetched z / lse of the next 32-column chunk (lane = column)
    if (SCORES && half * AS_PCOLS + lane < nk) {
      pf_z = z[(size_t)so * Lp + half * AS_PCOLS + lane];
      pf_lse = lse_in[(size_t)so * Lp + half * AS_PCOLS + lane];
    }
    for (int j = 0; j < n_tiles; ++j) {
      const int st = j & 1;
      tc::mbar_wait(&s_full[st], (j >> 1) & 1);
      tc::fence_after_sync();
      if constexpr (!SCORES) {
        const int valid = nk - j * 128 - half * AS_PCOLS;  // valid keys among this thread's columns
        uint32_t sv[AS_PCOLS];
#pragma unroll
        for (int c = 0; c < AS_PCOLS; c += 32) tc::tmem_ld32(tmem + lane_base + st * 128 + half * AS_PCOLS + c, sv + c);
        tc::tmem_ld_wait();
        tc::fence_before_sync();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&s_empty[st]);
        if (valid < AS_PCOLS) {
#pragma unroll
          for (int i = 0; i < AS_PCOLS; ++i)
            if (i >= valid) sv[i] = 0xff800000u;
        }
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int i = 0; i < AS_PCOLS; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(sv[i]));
        const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
        if (mx > -INFINITY) {  // (a fully masked half keeps its running state)
          const float m_new = fmaxf(m_run, mx);
          const float ml2 = m_new * 1.4426950408889634f;
          float rs4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int i = 0; i < AS_PCOLS; ++i) rs4[i & 3] += ex2a(fmaf(__uint_as_float(sv[i]), 1.4426950408889634f, -ml2));
          l_run = l_run * ex2a((m_run - m_new) * 1.4426950408889634f) + ((rs4[0] + rs4[1]) + (rs4[2] + rs4[3]));
          m_run = m_new;
        }
      } else {
#pragma unroll 1
        for (int c = 0; c < AS_PCOLS / 32; ++c) {
          uint32_t v[32];
          tc::tmem_ld32(tmem + lane_base + st * 128 + half * AS_PCOLS + c * 32, v);
          const int cb = j * 128 + half * AS_PCOLS + c * 32;  // first column of this chunk
          const int col = cb + lane;                    // this lane's column in the transposed phase
          // column constant of this chunk from the values fetched one chunk ago; fetch the next chunk's now
          // (an un-prefetched global load here cost ~1000 cycles per chunk on the critical path)
          float colconst = -INFINITY;                   // -inf: the column takes no part in the row max
          if (col < nk) colconst = lg_logsigmoid(pf_z) - pf_lse;
          {
            // next chunk of this warp: same tile, or the same part of the next tile
            const int ncol = (c + 1 < AS_PCOLS / 32 ? cb + 32 : cb + 128 - (AS_PCOLS - 32)) + lane;
            if (ncol < nk) { pf_z = z[(size_t)so * Lp + ncol]; pf_lse = lse_in[(size_t)so * Lp + ncol]; }
          }
          tc::tmem_ld_wait();
          if (c == AS_PCOLS / 32 - 1) {
            tc::fence_before_sync();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&s_empty[st]);
          }
          xc[lane] = colconst;
          __syncwarp();
          // row phase (thread = row): final values, running row argmax over exactly what gets written
          float val[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            val[i] = fmaf(2.f, __uint_as_float(v[i]), rowconst) + xc[i];
            xp[lane * 33 + i] = val[i];
          }
          if (best0) {
#ifdef LG_ASSIGN_SERIAL_ARGMAX
#pragma unroll
            for (int i = 0; i < 32; ++i) amax_merge(rbest, ridx, val[i], cb + i);
#else
            float cm;
            int ci;
            chunk_argmax(val, cm, ci);
            amax_merge(rbest, ridx, cm, cb + ci);
#endif
          }
          if constexpr (LOSS) {
            if (row < nq) {
              const uint8_t* g = ls.gt + ((size_t)blockIdx.y * (R - 1) + row) * (C - 1) + cb;
              uint32_t gw[8];  // 32 ground-truth bytes of this row
              if (gt16 && cb + 32 <= nk) {
                const uint4 g0 = reinterpret_cast<const uint4*>(g)[0], g1 = reinterpret_cast<const uint4*>(g)[1];
                gw[0] = g0.x; gw[1] = g0.y; gw[2] = g0.z; gw[3] = g0.w;
                gw[4] = g1.x; gw[5] = g1.y; gw[6] = g1.z; gw[7] = g1.w;
              } else {
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                  gw[w] = 0;
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    if (cb + 4 * w + k < nk) gw[w] |= (uint32_t)g[4 * w + k] << (8 * k);
                }
              }
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                if (cb + i < nk) {  // (columns past the end carry -inf)
                  a_exp += __expf(val[i]);
                  if ((gw[i >> 2] >> (8 * (i & 3))) & 0xffu) { a_pos += val[i]; a_cnt += 1.f; }
                }
              }
            }
          }
          __syncwarp();
          // column phase (thread = column): every warp store is one contiguous 128-byte row segment
          float* out = LOSS ? nullptr : scores + ((size_t)blockIdx.y * R + m0 + quarter * 32) * C + col;
          const int rows_here = max(0, min(32, nq - (m0 + quarter * 32)));
          if (col < nk) {
            float cbest = -INFINITY;
            int cidx = 0;
            if (rows_here == 32) {
              float cv[32];
#pragma unroll
              for (int rr = 0; rr < 32; ++rr) {
                cv[rr] = xp[rr * 33 + lane];
                if constexpr (!LOSS) out[(size_t)rr * C] = cv[rr];
              }
              if (best1) {
#ifdef LG_ASSIGN_SERIAL_ARGMAX
#pragma unroll
                for (int rr = 0; rr < 32; ++rr) amax_merge(cbest, cidx, cv[rr], rr);
#else
                chunk_argmax(cv, cbest, cidx);
#endif
              }
            } else {
              for (int rr = 0; rr < rows_here; ++rr) {
                const float val = xp[rr * 33 + lane];
                if constexpr (!LOSS) out[(size_t)rr * C] = val;
                if (val > cbest || (val != val && cbest == cbest)) { cbest = val; cidx = rr; }
              }
            }
            if (best1 && rows_here > 0)
              atomicMax(best1 + (size_t)blockIdx.y * C + col, fm_pack(cbest, m0 + quarter * 32 + cidx));
          }
          __syncwarp();
        }
      }
    }
    if constexpr (!SCORES) {
      // combine the column parts of a row: parts 1.. publish (m, l), part 0 merges (in part order) and writes
      float* ex = xpose + (ew & 3) * (AS_XP + 32);
      if (half > 0) { ex[(half - 1) * 64 + 2 * lane] = m_run; ex[(half - 1) * 64 + 2 * lane + 1] = l_run; }
      asm volatile("bar.sync %0, %1;" ::"r"(1 + quarter), "n"(32 * AS_PARTS) : "memory");
      if (half == 0 && row < nq) {
        float m = m_run;
#pragma unroll
        for (int pp = 0; pp < AS_PARTS - 1; ++pp) m = fmaxf(m, ex[pp * 64 + 2 * lane]);
        float l = l_run * ex2a((m_run - m) * 1.4426950408889634f);
#pragma unroll
        for (int pp = 0; pp < AS_PARTS - 1; ++pp)
          l += ex[pp * 64 + 2 * lane + 1] * ex2a((ex[pp * 64 + 2 * lane] - m) * 1.4426950408889634f);
        lse_out[(size_t)s * Lp + row] = m + logf(l);
      }
    } else {
      // both column halves of a row race on one packed (value, ~index) word: 64-bit max keeps the larger value
      // and, among equal values, the lower index (best0 is zeroed by the caller)
      if (best0 && row < nq) atomicMax(best0 + (size_t)blockIdx.y * R + row, fm_pack(rbest, ridx));
      if constexpr (LOSS) {
        if (row < nq) {
          const size_t o = (size_t)blockIdx.y * (R - 1) + row;
          atomicAdd(ls.row_pos + o, a_pos);
          atomicAdd(ls.row_cnt + o, a_cnt);
          atomicAdd(ls.row_exp + o, a_exp);
        }
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (AS_CL > 1) tc::cluster_sync();  // nobody retires while the peer may still multicast into its shared memory
  if (warp == 1) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem, 256);
  }
}

// LOSS: arg-maxima including the dustbins from the packed inner maxima, and the dustbin column's share of row_exp.
// torch.max tie rule: the dustbin has the highest index, so it wins only if strictly larger (or the first NaN).
// Rows / columns past pair b's counts (lens) keep row_exp = 0 and get arg-maximum -1, as lgb200_loss_reduce_ragged.
__global__ void assign_loss_finish_kernel(const float* __restrict__ z, int Lp, int R, int C,
                                          const int32_t* __restrict__ lens,
                                          const unsigned long long* __restrict__ best0,
                                          const unsigned long long* __restrict__ best1, float* __restrict__ row_exp,
                                          int32_t* __restrict__ row_arg, int32_t* __restrict__ col_arg) {
  const int b = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  const int n0 = lens ? lens[2 * b] : R - 1, n1 = lens ? lens[2 * b + 1] : C - 1;
  if (t < R - 1 && t >= n0) {
    if (row_arg) row_arg[(size_t)b * (R - 1) + t] = -1;
  } else if (t < R - 1) {
    const float dz = lg_logsigmoid(-z[(size_t)(2 * b) * Lp + t]);
    const unsigned long long p = best0[(size_t)b * R + t];
    const float v = fm_value(p);
    const bool inner = C > 1 && p != 0ull && !(dz > v || (dz != dz && v == v));
    if (row_arg) row_arg[(size_t)b * (R - 1) + t] = inner ? fm_index(p) : C - 1;
    if (row_exp) row_exp[(size_t)b * (R - 1) + t] += __expf(dz);
  }
  if (t < C - 1 && col_arg && t >= n1) {
    col_arg[(size_t)b * (C - 1) + t] = -1;
  } else if (t < C - 1 && col_arg) {
    const float dz = lg_logsigmoid(-z[(size_t)(2 * b + 1) * Lp + t]);
    const unsigned long long p = best1[(size_t)b * C + t];
    const float v = fm_value(p);
    const bool inner = R > 1 && p != 0ull && !(dz > v || (dz != dz && v == v));
    col_arg[(size_t)b * (C - 1) + t] = inner ? fm_index(p) : R - 1;
  }
}

// Dustbin row / column and zero padding of scores [B,R,C].  One WARP per row, 32 rows per CTA: without padding a
// row's share is a single element (its dustbin), and the first version's one-CTA-per-row grid (R x B = 131 136
// CTAs at 64 pairs) spent 78 us on block scheduling alone.  The dustbin ROW (C elements, each behind a load of z)
// is dealt out 32 columns per CTA: written by one warp it is a chain of C/32 dependent-latency iterations (39 us).
constexpr int AB_ROWS = 32;
__global__ void __launch_bounds__(256) assign_border_kernel(const float* __restrict__ z, int Lp,
                                                            const int32_t* __restrict__ lens, int R, int C,
                                                            float* __restrict__ scores) {
  const int b = blockIdx.y;
  const int n0 = lens ? lens[2 * b] : R - 1, n1 = lens ? lens[2 * b + 1] : C - 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_end = min(R - 1, (int)(blockIdx.x + 1) * AB_ROWS);  // rows [0, R-1); the dustbin row is handled below
  for (int r = blockIdx.x * AB_ROWS + warp; r < r_end; r += 8) {
    float* out = scores + ((size_t)b * R + r) * C;
    if (r < n0) {
      for (int c = n1 + lane; c < C - 1; c += 32) out[c] = 0.f;
      if (lane == 0) out[C - 1] = lg_logsigmoid(-z[(size_t)(2 * b) * Lp + r]);
    } else {
      for (int c = lane; c < C; c += 32) out[c] = 0.f;
    }
  }
  if (warp == 7) {  // this CTA's 32 columns of the dustbin row (the grid covers max(R, C) in steps of 32)
    const int c = blockIdx.x * AB_ROWS + lane;
    if (c < C) scores[((size_t)b * R + (R - 1)) * C + c] = c < n1 ? lg_logsigmoid(-z[(size_t)(2 * b + 1) * Lp + c]) : 0.f;
  }
}

int make_md_map(CUtensorMap* tm, const __nv_bfloat16* md, int S, int Lp, int rows = 128) {
  const uint64_t d[2] = {256, (uint64_t)S * Lp}, sb[1] = {512};
  const uint32_t box[2] = {64, (uint32_t)rows};
  return lg_make_tmap_bf16(tm, md, 2, d, sb, box);
}

// strips are launched as clusters of AS_CL along x (the grid is rounded up; a strip past Lp returns with its cluster
// or, next to a valid partner, only fetches its half of the B boxes)
template <typename Kern, typename... Args>
int launch_strips(Kern kern, dim3 grid, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  grid.x = (grid.x + AS_CL - 1) / AS_CL * AS_CL;
  cfg.gridDim = grid;
  cfg.blockDim = dim3(AS_THREADS);
  cfg.dynamicSmemBytes = AS_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = AS_CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
  if (e != cudaSuccess) return (int)e;
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

}  // namespace

int lg_tc_assign_lse(const __nv_bfloat16* md, int S, int Lp, const int32_t* lens, float* lse,
                     cudaStream_t st) {
  CUtensorMap tm;
  int rc = make_md_map(&tm, md, S, Lp);
  if (rc) return rc;
  cudaError_t e = cudaFuncSetAttribute(tc_assign_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, AS_SMEM);
  if (e != cudaSuccess) return (int)e;
  CUtensorMap tb;
  if ((rc = make_md_map(&tb, md, S, Lp, 128 / AS_CL))) return rc;
  return launch_strips(tc_assign_kernel<0>, dim3(Lp / 128, S), st, tm, tb, Lp, lens, (const float*)nullptr,
                       (const float*)nullptr, lse, 0, 0, (float*)nullptr, (unsigned long long*)nullptr,
                       (unsigned long long*)nullptr, AsLoss{});
}

int lg_tc_assign_scores(const __nv_bfloat16* md, const float* z, const float* lse, int B, int Lp,
                        const int32_t* lens, int R, int C, float* scores, void* best_ws, cudaStream_t st) {
  CUtensorMap tm;
  int rc = make_md_map(&tm, md, 2 * B, Lp);
  if (rc) return rc;
  cudaError_t e = cudaFuncSetAttribute(tc_assign_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, AS_SMEM);
  if (e != cudaSuccess) return (int)e;
  assign_border_kernel<<<dim3(((R > C ? R : C) + AB_ROWS - 1) / AB_ROWS, B), 256, 0, st>>>(z, Lp, lens, R, C, scores);
  LG_LAUNCH_CHECK();
  unsigned long long* best0 = reinterpret_cast<unsigned long long*>(best_ws);
  unsigned long long* best1 = best0 ? best0 + (size_t)B * R : nullptr;
  if (best_ws) {
    e = cudaMemsetAsync(best_ws, 0, sizeof(unsigned long long) * (size_t)B * (R + C), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (R > 1 && C > 1) {
    CUtensorMap tb;
    if ((rc = make_md_map(&tb, md, 2 * B, Lp, 128 / AS_CL))) return rc;
    return launch_strips(tc_assign_kernel<1>, dim3((R - 1 + 127) / 128, B), st, tm, tb, Lp, lens, z, lse, (float*)nullptr, R,
                         C, scores, best0, best1, AsLoss{});
  }
  return LGB200_OK;
}

int lg_tc_assign_loss(const __nv_bfloat16* md, const float* z, const float* lse, int B, int Lp, const int32_t* lens,
                      int R, int C, const uint8_t* gt, float* row_pos, float* row_cnt, float* row_exp,
                      int32_t* row_arg, int32_t* col_arg, void* best_ws, cudaStream_t st) {
  CUtensorMap tm;
  int rc = make_md_map(&tm, md, 2 * B, Lp);
  if (rc) return rc;
  cudaError_t e = cudaFuncSetAttribute(tc_assign_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, AS_SMEM);
  if (e != cudaSuccess) return (int)e;
  unsigned long long* best0 = reinterpret_cast<unsigned long long*>(best_ws);
  unsigned long long* best1 = best0 + (size_t)B * R;
  if ((e = cudaMemsetAsync(best_ws, 0, sizeof(unsigned long long) * (size_t)B * (R + C), st)) != cudaSuccess) return (int)e;
  const size_t nrow = sizeof(float) * (size_t)B * (R - 1);
  if ((e = cudaMemsetAsync(row_pos, 0, nrow, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(row_cnt, 0, nrow, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(row_exp, 0, nrow, st)) != cudaSuccess) return (int)e;
  if (R > 1 && C > 1) {
    CUtensorMap tb;
    if ((rc = make_md_map(&tb, md, 2 * B, Lp, 128 / AS_CL))) return rc;
    if ((rc = launch_strips(tc_assign_kernel<2>, dim3((R - 1 + 127) / 128, B), st, tm, tb, Lp, lens, z, lse, (float*)nullptr,
                            R, C, (float*)nullptr, best0, best1, AsLoss{gt, row_pos, row_cnt, row_exp})))
      return rc;
  }
  const int nmax = (R > C ? R : C) - 1;
  if (nmax > 0) {
    assign_loss_finish_kernel<<<dim3((nmax + 255) / 256, B), 256, 0, st>>>(z, Lp, R, C, lens, best0, best1, row_exp,
                                                                          row_arg, col_arg);
    LG_LAUNCH_CHECK();
  }
  return LGB200_OK;
}
