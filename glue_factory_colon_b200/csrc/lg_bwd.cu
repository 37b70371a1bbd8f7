// Backward kernels of the training path (SURVEY.md 8(f) rank 2: "training forward + loss", the part the reference
// gets from autograd, lightglue.py:484-498, 588-637).  What counts here is that the fused forward ops have fused
// backward ops (nothing N x M is materialised by the attention backward either) and that gradients agree with the
// reference's autograd.  The attention backward is the tcgen05 kernel of lg_x3_attn_bwd.cu: lgb200_attention_bwd runs
// its fp32-accurate split-fp16 instantiation, lgb200_attention_bwd_bf16 its bf16 one.  Plain GEMMs of the backward
// (dX = dY.W, dW = dY^T.X) are left to cuBLAS on the host side (glue_factory_colon_b200/train.py).
//
//   heads_bwd_kernel        head-major dq/dk/dv -> token-major d(qkv) incl. the transposed rotary embedding and the
//                           gradient of the rotary angles (-> posenc.Wr)                   lightglue.py:43-50, 157-161
//   ln_gelu_bwd_kernel      GELU(erf)' . LayerNorm backward, d gamma / d beta partials     lightglue.py:144-149
//   assign_dsim_kernel      d sim of sigmoid_log_double_softmax (optionally per-pair counts) lightglue.py:257-269
//   abwd_*_kernel           the same for any upstream gradient of log_assignment, plus d z   lightglue.py:257-269
//   posenc_bwd_kernel       d keypoints through normalize_keypoints and posenc.Wr            lightglue.py:28-40, 61-66
#include "lg_common.cuh"
#include "lg_internal.cuh"

namespace {

// One thread per (token, 4 consecutive head dimensions), looping over the 4 heads.
// n_parts == 3 (self block): out [T,768] = [s0 R^T(dq') | s1 R^T(dk') | s2 dv], column part*256 + head*64 + d -- the
//   packed Wqkv order of lgb200_linear(HEADS); R^T = transposed rotation by the token's angles; dtheta [T,32] +=
//   sum over heads and q/k of (dq'_{2f+1} q'_{2f} - dq'_{2f} q'_{2f+1}) (d/dtheta of a rotation is the rotation by
//   90 degrees: the scale of q' cancels).
// n_parts == 2 (cross block): out [T,512] = [s0 (dq + dk) | s1 dv]  (to_qk feeds both the query and the key side).
__global__ void __launch_bounds__(256) heads_bwd_kernel(const float* __restrict__ dq, const float* __restrict__ dk,
                                                        const float* __restrict__ dv, const float* __restrict__ q,
                                                        const float* __restrict__ k, const float* __restrict__ rot,
                                                        int T, int Lp, const int32_t* __restrict__ lens, int n_parts,
                                                        float s0, float s1, float s2, float* __restrict__ out,
                                                        float* __restrict__ dtheta) {
  const int idx = blockIdx.x * 256 + threadIdx.x;
  const int t = idx >> 4, d4 = (idx & 15) * 4;
  if (t >= T) return;
  const int s = t / Lp, l = t - s * Lp;
  const int N = n_parts * 256;
  float* o = out + (size_t)t * N;
  if (lens && l >= lens[s]) {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = 0; p < n_parts; ++p)
      for (int h = 0; h < LG_HEADS; ++h) *reinterpret_cast<float4*>(o + p * 256 + h * LG_DH + d4) = z4;
    return;
  }
  if (n_parts == 3) {
    const float4 cs = *reinterpret_cast<const float4*>(rot + (size_t)t * 64 + d4);  // (cos f, sin f, cos f+1, sin f+1)
    float th0 = 0.f, th1 = 0.f;
#pragma unroll
    for (int h = 0; h < LG_HEADS; ++h) {
      const size_t off = (((size_t)s * LG_HEADS + h) * Lp + l) * LG_DH + d4;
      const float4 gq = *reinterpret_cast<const float4*>(dq + off), aq = *reinterpret_cast<const float4*>(q + off);
      const float4 gk = *reinterpret_cast<const float4*>(dk + off), ak = *reinterpret_cast<const float4*>(k + off);
      const float4 gv = *reinterpret_cast<const float4*>(dv + off);
      th0 += gq.y * aq.x - gq.x * aq.y + gk.y * ak.x - gk.x * ak.y;
      th1 += gq.w * aq.z - gq.z * aq.w + gk.w * ak.z - gk.z * ak.w;
      *reinterpret_cast<float4*>(o + h * LG_DH + d4) =
          make_float4(s0 * (gq.x * cs.x + gq.y * cs.y), s0 * (gq.y * cs.x - gq.x * cs.y),
                      s0 * (gq.z * cs.z + gq.w * cs.w), s0 * (gq.w * cs.z - gq.z * cs.w));
      *reinterpret_cast<float4*>(o + 256 + h * LG_DH + d4) =
          make_float4(s1 * (gk.x * cs.x + gk.y * cs.y), s1 * (gk.y * cs.x - gk.x * cs.y),
                      s1 * (gk.z * cs.z + gk.w * cs.w), s1 * (gk.w * cs.z - gk.z * cs.w));
      *reinterpret_cast<float4*>(o + 512 + h * LG_DH + d4) = make_float4(s2 * gv.x, s2 * gv.y, s2 * gv.z, s2 * gv.w);
    }
    if (dtheta) {
      float2* p = reinterpret_cast<float2*>(dtheta + (size_t)t * 32 + d4 / 2);
      float2 v = *p;
      v.x += th0;
      v.y += th1;
      *p = v;
    }
  } else {
#pragma unroll
    for (int h = 0; h < LG_HEADS; ++h) {
      const size_t off = (((size_t)s * LG_HEADS + h) * Lp + l) * LG_DH + d4;
      const float4 gq = *reinterpret_cast<const float4*>(dq + off), gk = *reinterpret_cast<const float4*>(dk + off);
      const float4 gv = *reinterpret_cast<const float4*>(dv + off);
      *reinterpret_cast<float4*>(o + h * LG_DH + d4) =
          make_float4(s0 * (gq.x + gk.x), s0 * (gq.y + gk.y), s0 * (gq.z + gk.z), s0 * (gq.w + gk.w));
      *reinterpret_cast<float4*>(o + 256 + h * LG_DH + d4) = make_float4(s1 * gv.x, s1 * gv.y, s1 * gv.z, s1 * gv.w);
    }
  }
}

// y = gelu(LN(h) * gamma + beta), rows of 512.  One warp per row, grid-stride; a lane owns columns 4*(lane + 32 i).
// dh = rstd (dhat - mean(dhat) - hhat mean(dhat hhat)), dhat = da gelu'(hn) gamma.  Every CTA writes its column sums
// of (da gelu' hhat | da gelu') to partials[blockIdx.x][1024]; the caller adds them up (fixed order: reproducible).
__global__ void __launch_bounds__(256) ln_gelu_bwd_kernel(const float* __restrict__ h, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, const float* __restrict__ da,
                                                          int T, int Lp, const int32_t* __restrict__ lens,
                                                          float* __restrict__ dh, float* __restrict__ act,
                                                          float* __restrict__ partials) {
  __shared__ float red[8][1024];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 g4[4], b4[4], sg[4], sb[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    g4[i] = reinterpret_cast<const float4*>(gamma)[lane + 32 * i];
    b4[i] = reinterpret_cast<const float4*>(beta)[lane + 32 * i];
    sg[i] = sb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int row = blockIdx.x * 8 + warp; row < T; row += gridDim.x * 8) {
    float4* po = reinterpret_cast<float4*>(dh + (size_t)row * 512);
    float4* pa = act ? reinterpret_cast<float4*>(act + (size_t)row * 512) : nullptr;
    if (lens) {
      const int s = row / Lp;
      if (row - s * Lp >= lens[s]) {  // padded row: no gradient, and a defined activation for the dW GEMM
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          po[lane + 32 * i] = z4;
          if (pa) pa[lane + 32 * i] = z4;
        }
        continue;
      }
    }
    const float4* ph = reinterpret_cast<const float4*>(h + (size_t)row * 512);
    const float4* pg = reinterpret_cast<const float4*>(da + (size_t)row * 512);
    float v[16], g[16];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 a = ph[lane + 32 * i], b = pg[lane + 32 * i];
      v[4 * i] = a.x; v[4 * i + 1] = a.y; v[4 * i + 2] = a.z; v[4 * i + 3] = a.w;
      g[4 * i] = b.x; g[4 * i + 1] = b.y; g[4 * i + 2] = b.z; g[4 * i + 3] = b.w;
      sum += a.x + a.y + a.z + a.w;
    }
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * (1.f / 512.f);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { v[i] -= mean; sq += v[i] * v[i]; }
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = 1.f / sqrtf(sq * (1.f / 512.f) + 1e-5f);
    float m1 = 0.f, m2 = 0.f;
    float a_out[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float gm = reinterpret_cast<const float*>(&g4[i >> 2])[i & 3];
      const float bt = reinterpret_cast<const float*>(&b4[i >> 2])[i & 3];
      const float hh = v[i] * rstd;               // normalised
      const float hn = hh * gm + bt;
      const float cdf = 0.5f * (1.f + erff(hn * 0.70710678118654752440f));
      const float pdf = 0.39894228040143267794f * expf(-0.5f * hn * hn);
      a_out[i] = hn * cdf;
      const float dn = g[i] * (cdf + hn * pdf);   // d / d hn
      reinterpret_cast<float*>(&sg[i >> 2])[i & 3] += dn * hh;
      reinterpret_cast<float*>(&sb[i >> 2])[i & 3] += dn;
      const float dhat = dn * gm;
      g[i] = dhat;
      v[i] = hh;
      m1 += dhat;
      m2 += dhat * hh;
    }
    for (int o = 16; o; o >>= 1) {
      m1 += __shfl_xor_sync(0xffffffffu, m1, o);
      m2 += __shfl_xor_sync(0xffffffffu, m2, o);
    }
    m1 *= (1.f / 512.f);
    m2 *= (1.f / 512.f);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      po[lane + 32 * i] = make_float4(rstd * (g[4 * i] - m1 - v[4 * i] * m2), rstd * (g[4 * i + 1] - m1 - v[4 * i + 1] * m2),
                                      rstd * (g[4 * i + 2] - m1 - v[4 * i + 2] * m2),
                                      rstd * (g[4 * i + 3] - m1 - v[4 * i + 3] * m2));
      if (pa) pa[lane + 32 * i] = make_float4(a_out[4 * i], a_out[4 * i + 1], a_out[4 * i + 2], a_out[4 * i + 3]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    *reinterpret_cast<float4*>(&red[warp][4 * (lane + 32 * i)]) = sg[i];
    *reinterpret_cast<float4*>(&red[warp][512 + 4 * (lane + 32 * i)]) = sb[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 1024; c += 256) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) a += red[w][c];
    partials[(size_t)blockIdx.x * 1024 + c] = a;
  }
}

// sim [B,m,n] -> d sim in place: 2 g gt - r_i exp(sim - lse0_i) - c_j exp(sim - lse1_j)   (g = d loss / d pos_sum[b],
// r / c = g times the row / column sums of gt; lse from lgb200_assign_lse: rows of image 0, columns of image 1)
// lens (nullable): per-pair counts -- entries outside pair b's valid block (i >= lens[2b] or j >= lens[2b+1]) become 0
// and neither gt nor r / c nor lse is read there
__global__ void __launch_bounds__(256) assign_dsim_kernel(float* __restrict__ sim, int m, int n,
                                                          const float* __restrict__ lse, int Lp,
                                                          const int32_t* __restrict__ lens,
                                                          const uint8_t* __restrict__ gt, const float* __restrict__ g_pos,
                                                          const float* __restrict__ r, const float* __restrict__ c) {
  const int b = blockIdx.z, i = blockIdx.y;
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= n) return;
  const size_t off = ((size_t)b * m + i) * n + j;
  if (lens && (i >= lens[2 * b] || j >= lens[2 * b + 1])) {
    sim[off] = 0.f;
    return;
  }
  const float sv = sim[off];
  const float l0 = lse[(size_t)(2 * b) * Lp + i], l1 = lse[(size_t)(2 * b + 1) * Lp + j];
  const float g = gt[off] ? 2.f * g_pos[b] : 0.f;
  sim[off] = g - r[(size_t)b * m + i] * expf(sv - l0) - c[(size_t)b * n + j] * expf(sv - l1);
}

// ---- backward of log_assignment for any upstream gradient G [B, m+1, n+1] ----------------------------------------
// With R_i / C_j the row / column sums of G over pair b's valid block (n0 x n1):
//   d sim_ij = 2 G_ij - R_i exp(sim_ij - lse0_i) - C_j exp(sim_ij - lse1_j)   inside the block, 0 outside;
//   d z0_i   = R_i sigmoid(-z0_i) - G_{i,n} sigmoid(z0_i),   d z1_j = C_j sigmoid(-z1_j) - G_{m,j} sigmoid(z1_j).
// Three launches, no atomics (every sum has a fixed order, results are bit-reproducible):
//   abwd_sums_kernel   reads G once: a warp owns ABWD_ROWS whole rows and sweeps them in blocks of 128 columns, lane =
//                      column (coalesced 128-byte row segments; the (n+1)-float row pitch rules out vector loads).  Row
//                      sums stay in registers for the whole sweep (complete R_i, then d z0); column sums of the block
//                      go out as per-warp partials part[b][p][j].
//   abwd_cols_kernel   C_j = sum of the partials in warp order, then d z1.
//   abwd_dsim_kernel   warp per row, streams sim -> d sim in place, reading G a second time.
constexpr int ABWD_ROWS = 32;  // rows per warp of the sums pass
constexpr int ABWD_GROUP = 8;  // rows loaded together: 32 independent loads in flight per lane

__device__ __forceinline__ int abwd_chunks(int rows) { return (rows + ABWD_ROWS - 1) / ABWD_ROWS; }

__global__ void __launch_bounds__(128) abwd_sums_kernel(const float* __restrict__ G, int m, int n,
                                                        const int32_t* __restrict__ lens, const float* __restrict__ z,
                                                        int Lp, float* __restrict__ rsum, float* __restrict__ part,
                                                        float* __restrict__ dz0) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int P = abwd_chunks(m);
  if (p >= P) return;
  const int n0 = lens ? min(lens[2 * b], m) : m, n1 = lens ? min(lens[2 * b + 1], n) : n;
  const int C = n + 1, r0 = p * ABWD_ROWS;
  const int rows = max(0, min(ABWD_ROWS, n0 - r0));
  const float* g = G + ((size_t)b * (m + 1) + r0) * C;
  float* pp = part + ((size_t)b * P + p) * n;
  float racc[ABWD_ROWS];
#pragma unroll
  for (int i = 0; i < ABWD_ROWS; ++i) racc[i] = 0.f;
  for (int c0 = 0; rows > 0 && c0 < n1; c0 += 128) {
    float cacc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int gi = 0; gi < ABWD_ROWS / ABWD_GROUP; ++gi) {
      float v[ABWD_GROUP][4];
#pragma unroll
      for (int i = 0; i < ABWD_GROUP; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = gi * ABWD_GROUP + i, c = c0 + lane + 32 * j;
          v[i][j] = (r < rows && c < n1) ? __ldg(g + (size_t)r * C + c) : 0.f;
        }
#pragma unroll
      for (int i = 0; i < ABWD_GROUP; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          racc[gi * ABWD_GROUP + i] += v[i][j];
          cacc[j] += v[i][j];
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c0 + lane + 32 * j < n1) pp[c0 + lane + 32 * j] = cacc[j];
  }
#pragma unroll
  for (int i = 0; i < ABWD_ROWS; ++i) {
    float s = racc[i];
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const int r = r0 + i;
    if (lane == (i & 31) && r < m) {
      const bool in = i < rows;
      rsum[(size_t)b * m + r] = in ? s : 0.f;
      if (dz0) {
        float d = 0.f;
        if (in) {
          const float zv = z[(size_t)(2 * b) * Lp + r];
          d = s * lg_sigmoid(-zv) - g[(size_t)i * C + n] * lg_sigmoid(zv);
        }
        dz0[(size_t)b * m + r] = d;
      }
    }
  }
}

__global__ void __launch_bounds__(256) abwd_cols_kernel(const float* __restrict__ G, int m, int n,
                                                        const int32_t* __restrict__ lens, const float* __restrict__ z,
                                                        int Lp, const float* __restrict__ part,
                                                        float* __restrict__ csum, float* __restrict__ dz1) {
  const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int n0 = lens ? min(lens[2 * b], m) : m, n1 = lens ? min(lens[2 * b + 1], n) : n;
  const int P = abwd_chunks(m);
  float s = 0.f, d = 0.f;
  if (j < n1) {
    const float* pp = part + (size_t)b * P * n + j;
    for (int p = 0; p < abwd_chunks(n0); ++p) s += pp[(size_t)p * n];
    if (dz1) {
      const float zv = z[(size_t)(2 * b + 1) * Lp + j];
      d = s * lg_sigmoid(-zv) - G[((size_t)b * (m + 1) + m) * (n + 1) + j] * lg_sigmoid(zv);
    }
  }
  csum[(size_t)b * n + j] = s;
  if (dz1) dz1[(size_t)b * n + j] = d;
}

__global__ void __launch_bounds__(256) abwd_dsim_kernel(const float* __restrict__ G, float* __restrict__ sim, int m,
                                                        int n, const float* __restrict__ lse, int Lp,
                                                        const int32_t* __restrict__ lens,
                                                        const float* __restrict__ rsum,
                                                        const float* __restrict__ csum) {
  const int b = blockIdx.y, i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= m) return;
  const int n0 = lens ? min(lens[2 * b], m) : m, n1 = lens ? min(lens[2 * b + 1], n) : n;
  float* row = sim + ((size_t)b * m + i) * n;
  if (i >= n0) {
    for (int c = lane; c < n; c += 32) row[c] = 0.f;
    return;
  }
  const float* g = G + ((size_t)b * (m + 1) + i) * (n + 1);
  const float l0 = lse[(size_t)(2 * b) * Lp + i], r = rsum[(size_t)b * m + i];
  const float* l1 = lse + (size_t)(2 * b + 1) * Lp;
  const float* cs = csum + (size_t)b * n;
  for (int c0 = lane; c0 < n; c0 += 128) {
    float sv[4], gv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + 32 * u;
      sv[u] = c < n1 ? row[c] : 0.f;
      gv[u] = c < n1 ? __ldg(g + c) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + 32 * u;
      if (c < n) row[c] = c < n1 ? 2.f * gv[u] - r * expf(sv[u] - l0) - cs[c] * expf(sv[u] - l1[c]) : 0.f;
    }
  }
}

// ---- backward of the positional encoding's keypoint normalisation (lightglue.py:28-40, 61-66) ----------------------
// CTA per pair-image.  d kn = d theta . Wr per point; then, with t = max(size) / 2 and kn = (x - size / 2) / t:
//   d x_l = d kn_l / t  (+ scale / orientation: d kn passes through);
//   size == NULL (size = 1 + max - min over the valid points): with A = sum_l d kn_l and Q = sum_l <d kn_l, kn_l>,
//   d size_x = -(A_x + [x extent is the larger] Q) / (2 t), likewise y; it reaches the arg-max point with + and the
//   arg-min point with -, the lowest index among ties in both (torch's rule for max(dim) / min(dim)), and the x extent
//   counts as the larger one when the two are equal.  All sums have a fixed order (bit-reproducible).
__global__ void __launch_bounds__(1024) posenc_bwd_kernel(const float* __restrict__ kpts, int n, int kdim,
                                                          const float* __restrict__ size, const float* __restrict__ Wr,
                                                          const int32_t* __restrict__ lens, int img, int Lp,
                                                          const float* __restrict__ dtheta, float* __restrict__ dkpts) {
  const int b = blockIdx.x, s = 2 * b + img;
  const int nv = lens ? min(lens[s], n) : n;
  const float* kp = kpts + (size_t)b * n * kdim;
  float* dk = dkpts + (size_t)b * n * kdim;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __shared__ float sW[32 * 4];
  __shared__ unsigned long long ext[4][32];  // packed (value, index) of max x, max y, max -x, max -y per warp
  __shared__ float red[3][32];
  __shared__ float sh[3];
  __shared__ int arg[4], sel;
  for (int i = threadIdx.x; i < 32 * kdim; i += blockDim.x) sW[i] = Wr[i];
  if (size) {
    if (threadIdx.x == 0) {
      const float wd = size[b * 2 + 0], ht = size[b * 2 + 1];
      sh[0] = wd / 2.f;
      sh[1] = ht / 2.f;
      sh[2] = fmaxf(wd, ht) / 2.f;
    }
  } else {
    unsigned long long e[4] = {0ull, 0ull, 0ull, 0ull};
    for (int l = threadIdx.x; l < nv; l += blockDim.x) {
      const float x = kp[(size_t)l * kdim], y = kp[(size_t)l * kdim + 1];
      const unsigned long long c[4] = {fm_pack(x, l), fm_pack(y, l), fm_pack(-x, l), fm_pack(-y, l)};
#pragma unroll
      for (int k = 0; k < 4; ++k) e[k] = c[k] > e[k] ? c[k] : e[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      for (int o = 16; o; o >>= 1) {
        const unsigned long long t = __shfl_xor_sync(0xffffffffu, e[k], o);
        e[k] = t > e[k] ? t : e[k];
      }
      if (lane == 0) ext[k][w] = e[k];
    }
    __syncthreads();
    if (threadIdx.x == 0 && nv > 0) {
      for (int i = 1; i < nw; ++i)
        for (int k = 0; k < 4; ++k) ext[k][0] = ext[k][i] > ext[k][0] ? ext[k][i] : ext[k][0];
      // the forward's arithmetic (posenc_kernel): size = 1 + max - min, shift = size / 2, t = max(size) / 2
      const float sx = 1.f + fm_value(ext[0][0]) - (-fm_value(ext[2][0]));
      const float sy = 1.f + fm_value(ext[1][0]) - (-fm_value(ext[3][0]));
      sh[0] = sx / 2.f;
      sh[1] = sy / 2.f;
      sh[2] = fmaxf(sx, sy) / 2.f;
      sel = sx >= sy ? 0 : 1;
      for (int k = 0; k < 4; ++k) arg[k] = fm_index(ext[k][0]);
    }
  }
  __syncthreads();
  const float shx = sh[0], shy = sh[1], t = sh[2];
  float ax = 0.f, ay = 0.f, q = 0.f;
  for (int l = threadIdx.x; l < n; l += blockDim.x) {
    float d[4] = {0.f, 0.f, 0.f, 0.f};
    if (l < nv) {
      const float4* th = reinterpret_cast<const float4*>(dtheta + ((size_t)s * Lp + l) * 32);
#pragma unroll
      for (int f4 = 0; f4 < 8; ++f4) {
        const float4 v = th[f4];
        const float tv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c < kdim) d[c] = fmaf(tv[u], sW[(f4 * 4 + u) * kdim + c], d[c]);
      }
      if (!size) {
        const float knx = (kp[(size_t)l * kdim] - shx) / t, kny = (kp[(size_t)l * kdim + 1] - shy) / t;
        ax += d[0];
        ay += d[1];
        q += d[0] * knx + d[1] * kny;
      }
      d[0] /= t;
      d[1] /= t;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (c < kdim) dk[(size_t)l * kdim + c] = d[c];
  }
  if (size) return;
  for (int o = 16; o; o >>= 1) {
    ax += __shfl_xor_sync(0xffffffffu, ax, o);
    ay += __shfl_xor_sync(0xffffffffu, ay, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  if (lane == 0) { red[0][w] = ax; red[1][w] = ay; red[2][w] = q; }
  __syncthreads();  // (also orders the d x stores above before thread 0's updates below)
  if (threadIdx.x == 0 && nv > 0) {
    float A[3] = {0.f, 0.f, 0.f};
    for (int i = 0; i < nw; ++i)
      for (int k = 0; k < 3; ++k) A[k] += red[k][i];
    const float dsx = -(A[0] + (sel == 0 ? A[2] : 0.f)) / (2.f * t);
    const float dsy = -(A[1] + (sel == 1 ? A[2] : 0.f)) / (2.f * t);
    dk[(size_t)arg[0] * kdim] += dsx;
    dk[(size_t)arg[2] * kdim] -= dsx;
    dk[(size_t)arg[1] * kdim + 1] += dsy;
    dk[(size_t)arg[3] * kdim + 1] -= dsy;
  }
}

}  // namespace

extern "C" int lgb200_attention_bwd(const float* Q, const float* K, const float* V, const float* ctx, const float* dctx,
                                    int S, int Lp, const int32_t* lens, int kv_xor, float* dQ, float* dK, float* dV,
                                    float* workspace, void* stream) {
  if (!Q || !K || !V || !ctx || !dctx || !dQ || !dK || !dV || !workspace) return LGB200_ERR_NULL;
  if (S <= 0 || Lp <= 0 || Lp % 128 || (kv_xor != 0 && kv_xor != 1) || (kv_xor && (S & 1))) return LGB200_ERR_SHAPE;
  cudaStream_t st = lg_stream(stream);
  cudaError_t e;
  const size_t nb = (size_t)S * Lp * LG_D * sizeof(float);
  if ((e = cudaMemsetAsync(dQ, 0, nb, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(dK, 0, nb, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(dV, 0, nb, st)) != cudaSuccess) return (int)e;
  return lg_x3_attention_bwd(Q, K, V, ctx, dctx, S, Lp, lens, kv_xor, dQ, dK, dV, workspace, st);
}

extern "C" int lgb200_attention_bwd_workspace(int S, int Lp, long long* n_floats) {
  if (!n_floats) return LGB200_ERR_NULL;
  if (S <= 0 || Lp <= 0 || Lp % 128) return LGB200_ERR_SHAPE;
  *n_floats = (long long)lg_x3_attention_bwd_ws_floats(S, Lp);
  return LGB200_OK;
}

extern "C" int lgb200_attention_bwd_bf16(const void* Q, const void* K, const void* V, const void* ctx, const float* dctx,
                                         int S, int Lp, const int32_t* lens, int kv_xor, float* dQ, float* dK, float* dV,
                                         float* workspace, void* stream) {
  if (!Q || !K || !V || !ctx || !dctx || !dQ || !dK || !dV || !workspace) return LGB200_ERR_NULL;
  if (S <= 0 || Lp <= 0 || Lp % 128 || (kv_xor != 0 && kv_xor != 1) || (kv_xor && (S & 1))) return LGB200_ERR_SHAPE;
  cudaStream_t st = lg_stream(stream);
  cudaError_t e;
  const size_t nb = (size_t)S * Lp * LG_D * sizeof(float);
  if ((e = cudaMemsetAsync(dQ, 0, nb, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(dK, 0, nb, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(dV, 0, nb, st)) != cudaSuccess) return (int)e;
  using bf = __nv_bfloat16;
  return lg_bf16_attention_bwd((const bf*)Q, (const bf*)K, (const bf*)V, (const bf*)ctx, dctx, S, Lp, lens, kv_xor, dQ,
                               dK, dV, workspace, st);
}

extern "C" int lgb200_attention_bwd_bf16_workspace(int S, int Lp, long long* n_floats) {
  if (!n_floats) return LGB200_ERR_NULL;
  if (S <= 0 || Lp <= 0 || Lp % 128) return LGB200_ERR_SHAPE;
  *n_floats = (long long)lg_bf16_attention_bwd_ws_floats(S, Lp);
  return LGB200_OK;
}

extern "C" int lgb200_heads_bwd(const float* dQ, const float* dK, const float* dV, const float* Q, const float* K,
                                const float* rot, int S, int Lp, const int32_t* lens, int n_parts, float scale0,
                                float scale1, float scale2, float* out, float* dtheta, void* stream) {
  if (!dQ || !dK || !dV || !out) return LGB200_ERR_NULL;
  if (n_parts != 2 && n_parts != 3) return LGB200_ERR_SHAPE;
  if (n_parts == 3 && (!Q || !K || !rot)) return LGB200_ERR_NULL;
  if (S <= 0 || Lp <= 0 || Lp % 128) return LGB200_ERR_SHAPE;
  const int T = S * Lp;
  const long long threads = (long long)T * 16;
  heads_bwd_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, lg_stream(stream)>>>(
      dQ, dK, dV, Q, K, rot, T, Lp, lens, n_parts, scale0, scale1, scale2, out, dtheta);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_ln_gelu_bwd(const float* h, const float* gamma, const float* beta, const float* da, int T, int Lp,
                                  const int32_t* lens, float* dh, float* act, float* partials, int n_partials,
                                  void* stream) {
  if (!h || !gamma || !beta || !da || !dh || !partials) return LGB200_ERR_NULL;
  if (T <= 0 || Lp <= 0 || T % Lp || n_partials <= 0) return LGB200_ERR_SHAPE;
  ln_gelu_bwd_kernel<<<n_partials, 256, 0, lg_stream(stream)>>>(h, gamma, beta, da, T, Lp, lens, dh, act, partials);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_assign_dsim(float* sim, int B, int m, int n, const float* lse, int Lp,
                                  const uint8_t* gt_assignment, const float* g_pos, const float* r, const float* c,
                                  void* stream) {
  if (!sim || !lse || !gt_assignment || !g_pos || !r || !c) return LGB200_ERR_NULL;
  if (B <= 0 || m <= 0 || n <= 0 || m > Lp || n > Lp || m > 65535) return LGB200_ERR_SHAPE;
  dim3 grid((n + 255) / 256, m, B);
  assign_dsim_kernel<<<grid, 256, 0, lg_stream(stream)>>>(sim, m, n, lse, Lp, nullptr, gt_assignment, g_pos, r, c);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_assign_dsim_ragged(float* sim, int B, int m, int n, const float* lse, int Lp,
                                         const int32_t* lens, const uint8_t* gt_assignment, const float* g_pos,
                                         const float* r, const float* c, void* stream) {
  if (!sim || !lse || !lens || !gt_assignment || !g_pos || !r || !c) return LGB200_ERR_NULL;
  if (B <= 0 || m <= 0 || n <= 0 || m > Lp || n > Lp || m > 65535) return LGB200_ERR_SHAPE;
  dim3 grid((n + 255) / 256, m, B);
  assign_dsim_kernel<<<grid, 256, 0, lg_stream(stream)>>>(sim, m, n, lse, Lp, lens, gt_assignment, g_pos, r, c);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_assign_bwd_workspace(int B, int m, int n, long long* n_floats) {
  if (!n_floats) return LGB200_ERR_NULL;
  if (B <= 0 || m <= 0 || n <= 0) return LGB200_ERR_SHAPE;
  const long long P = (m + ABWD_ROWS - 1) / ABWD_ROWS;
  *n_floats = (long long)B * m + (long long)B * n + (long long)B * P * n;
  return LGB200_OK;
}

extern "C" int lgb200_assign_bwd(const float* G, float* sim, int B, int m, int n, const float* lse, int Lp,
                                 const int32_t* lens, const float* z, float* dz0, float* dz1, float* workspace,
                                 void* stream) {
  if (!G || !sim || !lse || !workspace || (z && (!dz0 || !dz1))) return LGB200_ERR_NULL;
  if (B <= 0 || B > 65535 || m <= 0 || n <= 0 || Lp <= 0 || Lp % 128 || m > Lp || n > Lp) return LGB200_ERR_SHAPE;
  cudaStream_t st = lg_stream(stream);
  const int P = (m + ABWD_ROWS - 1) / ABWD_ROWS;
  float* rsum = workspace;                      // [B, m]
  float* csum = rsum + (size_t)B * m;           // [B, n]
  float* part = csum + (size_t)B * n;           // [B, P, n]
  abwd_sums_kernel<<<dim3((P + 3) / 4, B), 128, 0, st>>>(G, m, n, lens, z, Lp, rsum, part, z ? dz0 : nullptr);
  LG_LAUNCH_CHECK();
  abwd_cols_kernel<<<dim3((n + 255) / 256, B), 256, 0, st>>>(G, m, n, lens, z, Lp, part, csum, z ? dz1 : nullptr);
  LG_LAUNCH_CHECK();
  abwd_dsim_kernel<<<dim3((m + 7) / 8, B), 256, 0, st>>>(G, sim, m, n, lse, Lp, lens, rsum, csum);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_posenc_bwd(const float* kpts, int B, int n, int kdim, const float* size, const float* Wr,
                                 const int32_t* lens, int img, int Lp, const float* dtheta, float* dkpts,
                                 void* stream) {
  if (!kpts || !Wr || !dtheta || !dkpts) return LGB200_ERR_NULL;
  if ((kdim != 2 && kdim != 4) || Lp <= 0 || Lp % 128 || n < 0 || n > Lp || B <= 0 || (img != 0 && img != 1))
    return LGB200_ERR_SHAPE;
  posenc_bwd_kernel<<<B, 1024, 0, lg_stream(stream)>>>(kpts, n, kdim, size, Wr, lens, img, Lp, dtheta, dkpts);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}
