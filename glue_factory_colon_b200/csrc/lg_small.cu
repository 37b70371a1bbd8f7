// HBM-bound helper kernels of the LightGlue hot path: input staging, positional
// encoding, per-token heads, early-exit test, point-pruning compaction and
// filter_matches.  All are streaming kernels: coalesced 16-byte accesses, warp
// shuffles for reductions, no shared-memory tiling needed.
#include "lg_common.cuh"
#include <cuda_fp16.h>
#include <cooperative_groups.h>

unsigned long long lg_launch_counter = 0;

extern "C" int lgb200_abi_version(void) { return LGB200_ABI_VERSION; }
extern "C" unsigned long long lgb200_launch_count(void) { return lg_launch_counter; }

extern "C" int lgb200_device_ok(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return LGB200_ERR_ARCH;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
    return LGB200_ERR_ARCH;
  return major == 10 ? LGB200_OK : LGB200_ERR_ARCH;
}

extern "C" const char* lgb200_error_string(int code) {
  switch (code) {
    case LGB200_OK: return "ok";
    case LGB200_ERR_SHAPE: return "unsupported shape or alignment";
    case LGB200_ERR_NULL: return "required pointer is NULL";
    case LGB200_ERR_PRECISION: return "unknown precision or epilogue";
    case LGB200_ERR_DRIVER: return "cuTensorMapEncodeTiled unavailable or failed";
    case LGB200_ERR_ARCH: return "device is not sm_100";
    case LGB200_ERR_WEIGHTS: return "required weight missing";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
  }
}

// ---------------------------------------------------------------------------
// pack_rows: [B,n,dim] fp32 -> sequence-major rows (+ bf16 shadow), zero padding
// ---------------------------------------------------------------------------
__global__ void pack_rows_kernel(const float* __restrict__ src, int n, int dim4, int img, int Lp,
                                 float* __restrict__ x32, __nv_bfloat16* __restrict__ x16) {
  const int b = blockIdx.y;
  const int s = 2 * b + img;
  const int total = Lp * dim4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int l = i / dim4, c4 = i - l * dim4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (l < n) v = reinterpret_cast<const float4*>(src)[((size_t)b * n + l) * dim4 + c4];
    const size_t o = ((size_t)s * Lp + l) * dim4 + c4;
    if (x32) reinterpret_cast<float4*>(x32)[o] = v;
    if (x16) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      reinterpret_cast<uint2*>(x16)[o] = pk;
    }
  }
}

extern "C" int lgb200_pack_rows(const float* src, int B, int n, int dim, int img, int Lp,
                                float* x32, void* x16, void* stream) {
  if (!src || (!x32 && !x16)) return LGB200_ERR_NULL;
  if (dim % 4 || Lp % 128 || n > Lp || B <= 0 || (img != 0 && img != 1)) return LGB200_ERR_SHAPE;
  const int total = Lp * (dim / 4);
  dim3 grid((total + 255) / 256 > 148 * 4 ? 148 * 4 : (total + 255) / 256, B);
  pack_rows_kernel<<<grid, 256, 0, lg_stream(stream)>>>(src, n, dim / 4, img, Lp, x32,
                                                        reinterpret_cast<__nv_bfloat16*>(x16));
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

// ---------------------------------------------------------------------------
// posenc: keypoint normalisation + Fourier projection + cos/sin table
// ---------------------------------------------------------------------------
// CTA (b, chunk) handles 256 rows of one pair-image: phase 1 finds shift/scale (given size, or the extent
// of the valid points -- recomputed by every chunk's CTA, it is a few KB), phase 2 writes rot[l, 2f] = cos,
// rot[l, 2f+1] = sin.  (One CTA per pair-image left 84 of the 148 SMs idle at 64 pairs: 63 us per launch.)
__global__ void posenc_kernel(const float* __restrict__ kpts, int n, int kdim,
                              const float* __restrict__ size, const float* __restrict__ Wr,
                              const int32_t* __restrict__ lens, int img, int Lp,
                              float* __restrict__ rot, __half2* __restrict__ rot16) {
  const int b = blockIdx.x;
  const int s = 2 * b + img;
  const int nv = lens ? min(lens[s], n) : n;
  const float* kp = kpts + (size_t)b * n * kdim;
  __shared__ float red[4][32];
  __shared__ float sh_shift[2], sh_scale;
  __shared__ float sW[32 * 4];
  for (int i = threadIdx.x; i < 32 * kdim; i += blockDim.x) sW[i] = Wr[i];
  if (size) {
    if (threadIdx.x == 0) {
      const float w = size[b * 2 + 0], h = size[b * 2 + 1];
      sh_shift[0] = w / 2.f;
      sh_shift[1] = h / 2.f;
      sh_scale = fmaxf(w, h) / 2.f;
    }
  } else {
    float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (int l = threadIdx.x; l < nv; l += blockDim.x) {
      const float x = kp[(size_t)l * kdim], y = kp[(size_t)l * kdim + 1];
      mnx = fminf(mnx, x); mxx = fmaxf(mxx, x);
      mny = fminf(mny, y); mxy = fmaxf(mxy, y);
    }
    for (int o = 16; o; o >>= 1) {
      mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
      mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
      mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
      mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { red[0][w] = mnx; red[1][w] = mny; red[2][w] = mxx; red[3][w] = mxy; }
    __syncthreads();
    if (threadIdx.x == 0) {
      const int nw = blockDim.x >> 5;
      for (int i = 1; i < nw; ++i) {
        red[0][0] = fminf(red[0][0], red[0][i]); red[1][0] = fminf(red[1][0], red[1][i]);
        red[2][0] = fmaxf(red[2][0], red[2][i]); red[3][0] = fmaxf(red[3][0], red[3][i]);
      }
      const float sx = 1.f + red[2][0] - red[0][0], sy = 1.f + red[3][0] - red[1][0];
      sh_shift[0] = sx / 2.f;
      sh_shift[1] = sy / 2.f;
      sh_scale = fmaxf(sx, sy) / 2.f;
    }
  }
  __syncthreads();
  const float shx = sh_shift[0], shy = sh_shift[1], sc = sh_scale;
  // thread = (point, frequency); 32 consecutive threads write one 256-byte row
  const int l0 = blockIdx.y * 256, l1 = min(Lp, l0 + 256);
  for (int i = l0 * 32 + threadIdx.x; i < l1 * 32; i += blockDim.x) {
    const int l = i >> 5, f = i & 31;
    float2 cs = make_float2(0.f, 0.f);
    if (l < nv) {
      const float x = (kp[(size_t)l * kdim] - shx) / sc;
      const float y = (kp[(size_t)l * kdim + 1] - shy) / sc;
      float p = x * sW[f * kdim] + y * sW[f * kdim + 1];
      if (kdim == 4) p += kp[(size_t)l * kdim + 2] * sW[f * 4 + 2] + kp[(size_t)l * kdim + 3] * sW[f * 4 + 3];
      sincosf(p, &cs.y, &cs.x);
    }
    if (rot) reinterpret_cast<float2*>(rot)[((size_t)s * Lp + l) * 32 + f] = cs;
    if (rot16) rot16[((size_t)s * Lp + l) * 32 + f] = __floats2half2_rn(cs.x, cs.y);
  }
}

extern "C" int lgb200_posenc(const float* kpts, int B, int n, int kdim, const float* size,
                             const float* Wr, const int32_t* lens, int img, int Lp, float* rot,
                             void* rot16, void* stream) {
  if (!kpts || !Wr || (!rot && !rot16)) return LGB200_ERR_NULL;
  if ((kdim != 2 && kdim != 4) || Lp % 128 || n > Lp || B <= 0) return LGB200_ERR_SHAPE;
  posenc_kernel<<<dim3(B, (Lp + 255) / 256), 1024, 0, lg_stream(stream)>>>(kpts, n, kdim, size, Wr, lens, img, Lp, rot,
                                                   reinterpret_cast<__half2*>(rot16));
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

// ---------------------------------------------------------------------------
// rowdot: Linear(256,1) (+sigmoid) per token.  One warp per row, 2x float4 per lane.
// ---------------------------------------------------------------------------
template <bool BF>
__global__ void rowdot_kernel(const void* __restrict__ xv, const float* __restrict__ w,
                              const float* __restrict__ bias, int S, int Lp,
                              const int32_t* __restrict__ lens, int sig, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= S * Lp) return;
  const int s = row / Lp, l = row - s * Lp;
  if (lens && l >= lens[s]) return;  // rows past the valid prefix are left untouched
  const float4* wr = reinterpret_cast<const float4*>(w);
  float acc;
  if (BF) {  // 8 consecutive bf16 per lane (one 16-byte load)
    const uint4 raw = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(xv) + (size_t)row * LG_D)[lane];
    const float4 w0 = wr[2 * lane], w1 = wr[2 * lane + 1];
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
    acc = __low2float(h[0]) * w0.x + __high2float(h[0]) * w0.y + __low2float(h[1]) * w0.z + __high2float(h[1]) * w0.w +
          __low2float(h[2]) * w1.x + __high2float(h[2]) * w1.y + __low2float(h[3]) * w1.z + __high2float(h[3]) * w1.w;
  } else {
    const float4* xr = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(xv) + (size_t)row * LG_D);
    const float4 a0 = xr[lane], a1 = xr[lane + 32], w0 = wr[lane], w1 = wr[lane + 32];
    acc = a0.x * w0.x + a0.y * w0.y + a0.z * w0.z + a0.w * w0.w + a1.x * w1.x + a1.y * w1.y +
          a1.z * w1.z + a1.w * w1.w;
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    acc += bias[0];
    out[row] = sig ? lg_sigmoid(acc) : acc;
  }
}

extern "C" int lgb200_rowdot(int precision, const void* x, const float* w, const float* b, int S, int Lp,
                             const int32_t* lens, int apply_sigmoid, float* out, void* stream) {
  if (!x || !w || !b || !out) return LGB200_ERR_NULL;
  if (precision != LGB200_F32 && precision != LGB200_BF16) return LGB200_ERR_PRECISION;
  const long rows = (long)S * Lp;
  const int blocks = (int)((rows * 32 + 255) / 256);
  if (precision == LGB200_BF16)
    rowdot_kernel<true><<<blocks, 256, 0, lg_stream(stream)>>>(x, w, b, S, Lp, lens, apply_sigmoid, out);
  else
    rowdot_kernel<false><<<blocks, 256, 0, lg_stream(stream)>>>(x, w, b, S, Lp, lens, apply_sigmoid, out);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

// ---------------------------------------------------------------------------
// exit_check: one CTA per pair
// ---------------------------------------------------------------------------
__global__ void exit_check_kernel(const float* __restrict__ conf, int Lp,
                                  const int32_t* __restrict__ lens,
                                  const int32_t* __restrict__ total, float thr, float depth_conf,
                                  int layer, int32_t* __restrict__ done,
                                  int32_t* __restrict__ lens_active) {
  const int b = blockIdx.x;
  if (done[b] != 0) return;
  int cnt = 0;
  for (int img = 0; img < 2; ++img) {
    const int s = 2 * b + img;
    const int n = lens[s];
    for (int l = threadIdx.x; l < n; l += blockDim.x) cnt += conf[(size_t)s * Lp + l] < thr;
  }
  __shared__ int red[32];
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int c = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) c += red[i];
    // lightglue.py:579-580 in fp32: 1.0 - sum/num_points > depth_confidence
    const float ratio = 1.0f - __fdiv_rn((float)c, (float)total[b]);
    if (ratio > depth_conf) {
      done[b] = layer + 1;
      lens_active[2 * b] = 0;
      lens_active[2 * b + 1] = 0;
    }
  }
}

extern "C" int lgb200_exit_check(const float* conf, int B, int Lp, const int32_t* lens,
                                 const int32_t* total, float thr, float depth_conf, int layer,
                                 int32_t* done, int32_t* lens_active, void* stream) {
  if (!conf || !lens || !total || !done || !lens_active) return LGB200_ERR_NULL;
  exit_check_kernel<<<B, 512, 0, lg_stream(stream)>>>(conf, Lp, lens, total, thr, depth_conf, layer,
                                                      done, lens_active);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

// ---------------------------------------------------------------------------
// prune_compact: stable stream compaction of token rows, one thread-block CLUSTER per sequence
// ---------------------------------------------------------------------------
// Phase 1: keep flags + block-wide exclusive scan (1024 threads, chunks of 1024)
//          -> dst position per row in shared memory (Lp <= 8192).  Every CTA of the cluster does the whole scan
//          (8 KB of flags): cheaper than exchanging it.
// Phase 2: warps copy kept rows (x32 1 KB, x16 512 B, rot 256 B, ind) to the
//          destination buffers with 16-byte accesses; the rows are dealt round-robin to the PC_SPLIT x 32 warps of
//          the cluster.  (Adaptive inference runs at batch 1 in the reference, i.e. two sequences: with one CTA per
//          sequence the copy of 2048 rows was 64 dependent iterations per warp on two SMs, 20-38 us per layer.)
// lens / lens_active are updated in place by rank 0 at the end; the cluster barrier after the first reads is what
// makes that safe (all CTAs of a cluster are co-resident).
#define LG_MAX_LP 8192
#ifndef PC_SPLIT
#define PC_SPLIT 8
#endif
__global__ void __cluster_dims__(PC_SPLIT, 1, 1) __launch_bounds__(1024) prune_compact_kernel(
    const float* __restrict__ match, const float* __restrict__ conf, float thr, float keep_above,
    int Lp, int32_t* __restrict__ lens, int32_t* __restrict__ lens_active,
    const float* __restrict__ x32s, float* __restrict__ x32d, const __nv_bfloat16* __restrict__ x16s,
    __nv_bfloat16* __restrict__ x16d, const float* __restrict__ rots, float* __restrict__ rotd,
    const uint32_t* __restrict__ rot16s, uint32_t* __restrict__ rot16d, const int32_t* __restrict__ inds, int32_t* __restrict__ indd, int32_t* __restrict__ prune_cnt) {
  __shared__ int16_t dst[LG_MAX_LP];
  __shared__ int warp_sum[32];
  __shared__ int running;
  const int s = blockIdx.y, part = blockIdx.x;  // part = rank in the cluster
  const int n = lens[s];
  const bool active = lens_active[s] != 0;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) running = 0;
  cooperative_groups::this_cluster().sync();  // (also a block barrier) every CTA has read the counts
  for (int base = 0; base < n; base += 1024) {
    const int l = base + threadIdx.x;
    int keep = 0;
    if (l < n) {
      if (!active) {
        keep = 1;
      } else {
        keep = match[(size_t)s * Lp + l] > keep_above;
        if (conf) keep |= conf[(size_t)s * Lp + l] <= thr;
      }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    const int pre = __popc(bal & ((1u << lane) - 1u));
    if (lane == 0) warp_sum[wid] = __popc(bal);
    __syncthreads();
    int woff = 0, tot = 0;
    for (int i = 0; i < 32; ++i) {
      const int v = warp_sum[i];
      if (i < wid) woff += v;
      tot += v;
    }
    const int r0 = running;
    if (l < n) dst[l] = keep ? (int16_t)(r0 + woff + pre) : (int16_t)-1;
    __syncthreads();
    if (threadIdx.x == 0) running = r0 + tot;
    __syncthreads();
  }
  const int kept = running;
  // phase 2: one warp per row
  for (int l = part * 32 + wid; l < n; l += 32 * PC_SPLIT) {
    const int d = dst[l];
    if (d < 0) continue;
    const size_t so = (size_t)s * Lp + l, dofs = (size_t)s * Lp + d;
    if (x32s) {
      const float4* a = reinterpret_cast<const float4*>(x32s + so * LG_D);
      float4* o = reinterpret_cast<float4*>(x32d + dofs * LG_D);
      o[lane] = a[lane];
      o[lane + 32] = a[lane + 32];
    }
    if (x16s) {
      reinterpret_cast<uint4*>(x16d + dofs * LG_D)[lane] =
          reinterpret_cast<const uint4*>(x16s + so * LG_D)[lane];
    }
    if (rots) reinterpret_cast<float2*>(rotd + dofs * 64)[lane] = reinterpret_cast<const float2*>(rots + so * 64)[lane];
    if (rot16s) rot16d[dofs * 32 + lane] = rot16s[so * 32 + lane];
    if (lane == 0) {
      const int orig = inds[so];
      indd[dofs] = orig;
      if (active) prune_cnt[(size_t)s * Lp + orig] += 1;
    }
  }
  if (part == 0 && threadIdx.x == 0 && active) {
    lens[s] = kept;
    lens_active[s] = kept;
  }
}

extern "C" int lgb200_prune_compact(const float* match, const float* conf, float thr,
                                    float width_conf, int S, int Lp, int32_t* lens,
                                    int32_t* lens_active, const float* x32_src, float* x32_dst,
                                    const void* x16_src, void* x16_dst, const float* rot_src,
                                    float* rot_dst, const void* rot16_src, void* rot16_dst,
                                    const int32_t* ind_src, int32_t* ind_dst, int32_t* prune_cnt,
                                    void* stream) {
  if (!match || !lens || !lens_active || !ind_src || !ind_dst || !prune_cnt) return LGB200_ERR_NULL;
  if ((x32_src && !x32_dst) || (x16_src && !x16_dst) || (rot_src && !rot_dst) || (rot16_src && !rot16_dst) ||
      (!x32_src && !x16_src))
    return LGB200_ERR_NULL;
  if (Lp > LG_MAX_LP || Lp % 128 || S < 1 || S > 65535) return LGB200_ERR_SHAPE;
  // lightglue.py:564: keep = scores > (1 - width_confidence), evaluated in fp32
  const float keep_above = 1.0f - width_conf;
  prune_compact_kernel<<<dim3(PC_SPLIT, S), 1024, 0, lg_stream(stream)>>>(
      match, conf, thr, keep_above, Lp, lens, lens_active, x32_src, x32_dst,
      reinterpret_cast<const __nv_bfloat16*>(x16_src), reinterpret_cast<__nv_bfloat16*>(x16_dst),
      rot_src, rot_dst, reinterpret_cast<const uint32_t*>(rot16_src), reinterpret_cast<uint32_t*>(rot16_dst),
      ind_src, ind_dst, prune_cnt);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

// ---------------------------------------------------------------------------
// filter_matches
// ---------------------------------------------------------------------------
// Pass A streams the score matrix once (HBM-bound: N*M*4 bytes read, (N+M)*8 written).  A WARP owns FM_WROWS whole rows
// and sweeps them in blocks of 128 columns, lane = column (every load instruction is one contiguous 128-byte row
// segment; the row pitch of (M+1)*4 bytes rules out aligned vector loads), 32 independent loads in flight per lane.
// Values are compared as order-preserving signed keys (NaN above everything, torch.max); with ascending visit order a
// strictly-greater test keeps the LOWEST index among equal values.  Row maxima stay in registers for the whole sweep
// (one shuffle reduction per row at the end, one plain store: no other warp sees the row); column maxima are
// final for the warp's rows after each block and go out as packed 64-bit atomicMax on
// (ordered value << 32 | ~index) -- N / FM_WROWS atomics per column, no shared memory, no block-wide barrier.
// The first version (256-thread CTAs, 64-bit packed compares per element, two __syncthreads per block) read its
// matrix at 1.0 TB/s.
// Pass B does the mutual check, exp, threshold and scatter.

// (fm_pack / fm_value / fm_index live in lg_common.cuh: the bf16 assignment kernel produces the same
// packed maxima in its epilogue so that this pass can be skipped.)

#ifndef FM_WROWS
#define FM_WROWS 16  // rows per warp (row maxima live in 2 x FM_WROWS registers)
#define FM_GROUP 8   // rows loaded together: 32 independent 128-byte loads in flight per warp
#define FM_MINB 8    // CTAs per SM the register allocation is held to (128 registers, 16 warps per SM)
#endif
#define FM_WARPS 2   // warps per CTA (independent of each other)

// float -> signed int whose order is the float order, every NaN on top; key ^ 0x80000000 is fm_pack's key
__device__ __forceinline__ int fm_key(float v) {
  const int u = __float_as_int(v);
  const int k = u ^ ((u >> 31) & 0x7fffffff);
  return v != v ? 0x7fffffff : k;
}
__device__ __forceinline__ unsigned long long fm_pack_key(int key, int idx) {
  return ((unsigned long long)((unsigned)key ^ 0x80000000u) << 32) | (unsigned)(0xffffffffu - (unsigned)idx);
}

// one block of 128 columns x this warp's 32 rows; FULL: no bounds checks
template <bool FULL>
__device__ __forceinline__ void fm_block(const float* __restrict__ p, int C, int rows, int cols, int r0, int c0, int lane,
                                         int (&rk)[FM_WROWS], int (&ri)[FM_WROWS],
                                         unsigned long long* __restrict__ b1) {
  int ck[4], cr[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { ck[j] = (int)0x80000000; cr[j] = 0; }
  const float* q = p + lane;  // walks down the rows group by group (32 hoisted row pointers would cost 64 registers)
#pragma unroll
  for (int g = 0; g < FM_WROWS / FM_GROUP; ++g) {
    float v[FM_GROUP][4];
#pragma unroll
    for (int i = 0; i < FM_GROUP; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = g * FM_GROUP + i, c = lane + 32 * j;
        if (FULL || (r < rows && c < cols)) v[i][j] = __ldcs(q + i * C + 32 * j);
      }
    q += FM_GROUP * C;
#pragma unroll
    for (int i = 0; i < FM_GROUP; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = g * FM_GROUP + i, c = lane + 32 * j;
        int k = (int)0x80000000;  // out of range: never strictly greater than anything
        if (FULL || (r < rows && c < cols)) k = fm_key(v[i][j]);
        if (k > rk[r]) { rk[r] = k; ri[r] = c0 + c; }
        if (k > ck[j]) { ck[j] = k; cr[j] = r0 + r; }
      }
    asm volatile("" ::: "memory");  // keep the next group's loads behind this group's compares (register budget)
  }
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (FULL || lane + 32 * j < cols) atomicMax(b1 + c0 + lane + 32 * j, fm_pack_key(ck[j], cr[j]));
}

__global__ void __launch_bounds__(FM_WARPS * 32, FM_MINB) fm_argmax_kernel(const float* __restrict__ scores, int R, int C,
                                                                  const int32_t* __restrict__ lens,
                                                                  unsigned long long* __restrict__ best0,
                                                                  unsigned long long* __restrict__ best1) {
  const int b = blockIdx.y;
  const int n0 = lens ? lens[2 * b] : R - 1, n1 = lens ? lens[2 * b + 1] : C - 1;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int r0 = (blockIdx.x * FM_WARPS + wid) * FM_WROWS;
  if (r0 >= n0 || n1 <= 0) return;  // (warps are independent: no block-wide barrier below)
  const float* base = scores + ((size_t)b * R + r0) * C;
  unsigned long long* b1 = best1 + (size_t)b * C;
  const int rows = min(FM_WROWS, n0 - r0);
  int rk[FM_WROWS], ri[FM_WROWS];
#pragma unroll
  for (int i = 0; i < FM_WROWS; ++i) { rk[i] = (int)0x80000000; ri[i] = 0; }
  int c0 = 0;
  if (rows == FM_WROWS)
    for (; c0 + 128 <= n1; c0 += 128) fm_block<true>(base + c0, C, rows, 128, r0, c0, lane, rk, ri, b1);
  for (; c0 < n1; c0 += 128) fm_block<false>(base + c0, C, rows, min(128, n1 - c0), r0, c0, lane, rk, ri, b1);
  unsigned long long* b0 = best0 + (size_t)b * R + r0;
#pragma unroll
  for (int i = 0; i < FM_WROWS; ++i) {
    unsigned long long m = fm_pack_key(rk[i], ri[i]);
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
      m = t > m ? t : m;
    }
    if (lane == (i & 31) && i < rows) b0[i] = m;
  }
}

__global__ void fm_fill_kernel(int64_t* m0, int64_t* m1, float* ms0, float* ms1, long n0tot, long n1tot) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n0tot) { m0[i] = -1; ms0[i] = 0.f; }
  if (i < n1tot) { m1[i] = -1; ms1[i] = 0.f; }
}

__global__ void fm_mutual_kernel(int R, int C, const int32_t* __restrict__ lens, float th,
                                 const unsigned long long* __restrict__ best0,
                                 const unsigned long long* __restrict__ best1,
                                 const int32_t* __restrict__ ind0, const int32_t* __restrict__ ind1,
                                 int ind_ld, int N0, int N1, int64_t* __restrict__ m0,
                                 int64_t* __restrict__ m1, float* __restrict__ ms0,
                                 float* __restrict__ ms1) {
  const int b = blockIdx.y;
  const int n0 = lens ? lens[2 * b] : R - 1, n1 = lens ? lens[2 * b + 1] : C - 1;
  if (n0 <= 0 || n1 <= 0) return;  // lightglue.py:298-303: everything stays -1 / 0
  const unsigned long long* b0 = best0 + (size_t)b * R;
  const unsigned long long* b1 = best1 + (size_t)b * C;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n0) {
    const int j = fm_index(b0[i]);
    const bool mutual = fm_index(b1[j]) == i;
    const float sc = mutual ? expf(fm_value(b0[i])) : 0.f;
    const bool valid = mutual && (sc > th);
    const int oi = ind0 ? ind0[(size_t)b * ind_ld + i] : i;
    const int oj = ind1 ? ind1[(size_t)b * ind_ld + j] : j;
    m0[(size_t)b * N0 + oi] = valid ? (int64_t)oj : -1;
    ms0[(size_t)b * N0 + oi] = sc;
  }
  if (i < n1) {
    const int r = fm_index(b1[i]);
    const bool mutual1 = fm_index(b0[r]) == i;
    // mscores1 = mutual1 ? mscores0[m1] : 0 ; valid1 = mutual1 & valid0[m1]
    // (mutual1 implies row r's best column is i, hence mutual0[r])
    const float sc = mutual1 ? expf(fm_value(b0[r])) : 0.f;
    const bool valid = mutual1 && (sc > th);
    const int oi = ind1 ? ind1[(size_t)b * ind_ld + i] : i;
    const int orow = ind0 ? ind0[(size_t)b * ind_ld + r] : r;
    m1[(size_t)b * N1 + oi] = valid ? (int64_t)orow : -1;
    ms1[(size_t)b * N1 + oi] = sc;
  }
}

extern "C" int lgb200_filter_matches(const float* scores, int B, int R, int C, const int32_t* lens,
                                     float threshold, const int32_t* ind0, const int32_t* ind1,
                                     int ind_ld, int N0, int N1, int64_t* m0, int64_t* m1,
                                     float* ms0, float* ms1, void* workspace, int workspace_has_best,
                                     void* stream) {
  if (B <= 0 || R < 1 || C < 1 || N0 < 0 || N1 < 0) return LGB200_ERR_SHAPE;
  if ((N0 > 0 && (!m0 || !ms0)) || (N1 > 0 && (!m1 || !ms1))) return LGB200_ERR_NULL;
  cudaStream_t st = lg_stream(stream);
  const long n0tot = (long)B * N0, n1tot = (long)B * N1;
  const long mx = n0tot > n1tot ? n0tot : n1tot;
  if (mx > 0) {
    fm_fill_kernel<<<(unsigned)((mx + 255) / 256), 256, 0, st>>>(m0, m1, ms0, ms1, n0tot, n1tot);
    LG_LAUNCH_CHECK();
  }
  if (R == 1 || C == 1) return LGB200_OK;  // empty side
  if ((!scores && !workspace_has_best) || !workspace) return LGB200_ERR_NULL;
  unsigned long long* best0 = reinterpret_cast<unsigned long long*>(workspace);
  unsigned long long* best1 = best0 + (size_t)B * R;
  if (!workspace_has_best) {  // otherwise lgb200_assign_scores already left the packed maxima there
    cudaError_t e = cudaMemsetAsync(workspace, 0, sizeof(unsigned long long) * (size_t)B * (R + C), st);
    if (e != cudaSuccess) return (int)e;
    dim3 g1((R - 1 + FM_WARPS * FM_WROWS - 1) / (FM_WARPS * FM_WROWS), B);
    fm_argmax_kernel<<<g1, FM_WARPS * 32, 0, st>>>(scores, R, C, lens, best0, best1);
    LG_LAUNCH_CHECK();
  }
  const int mxn = (R > C ? R : C) - 1;
  dim3 g2((mxn + 255) / 256, B);
  fm_mutual_kernel<<<g2, 256, 0, st>>>(R, C, lens, threshold, best0, best1, ind0, ind1, ind_ld, N0, N1,
                                       m0, m1, ms0, ms1);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}
