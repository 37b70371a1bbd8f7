// Nearest-neighbour matcher (SURVEY.md 8(f) rank 3; gluefactory/models/matchers/nearest_neighbor_matcher.py).
//   lgb200_nn_scores : similarity = d0 . d1^T (:64) and log_assignment = log_softmax rows + log_softmax columns with
//                      zero dustbins (:72-74), from the fp32 similarity kernel of MatchAssignment (z = NULL mode)
//   lgb200_nn_match  : find_nn (:15-31) in both directions (top-2 by value for the ratio test, distance threshold),
//                      mutual_check (:34-43), matching_scores = (match > -1) (:75-76)
//   lgb200_npair_loss: the N_pair loss (:85-109) on the similarity matrix, forward values
//   lgb200_npair_loss_bwd: its gradient w.r.t. the similarity and the temperature
// fp32 CUDA-core kernels (the baseline matcher is not on the headline path; its cost is the N x M write).
#include "lg_internal.cuh"

namespace {

struct Top2 {
  float v1, v2;  // largest and second largest value (v2 = -inf if there is only one candidate)
  int i1;        // index of the largest (lowest index among equal values)
};
__device__ __forceinline__ void top2_push(Top2& t, float v, int i) {
  if (v > t.v1 || (v == t.v1 && i < t.i1)) { t.v2 = t.v1; t.v1 = v; t.i1 = i; }
  else if (v > t.v2) t.v2 = v;
}
__device__ __forceinline__ void top2_merge(Top2& a, const Top2& b) {
  if (b.v1 > a.v1 || (b.v1 == a.v1 && b.i1 < a.i1)) {
    a.v2 = fmaxf(a.v1, b.v2);
    a.v1 = b.v1;
    a.i1 = b.i1;
  } else {
    a.v2 = fmaxf(a.v2, b.v1);
  }
}
// find_nn's decision for one point: nearest_neighbor_matcher.py:21-31
__device__ __forceinline__ long long nn_decide(const Top2& t, int n_cand, float ratio, float dist_thr) {
  if (n_cand == 0) return -1;
  const float d1 = 2.f * (1.f - t.v1);
  bool ok = true;
  if (ratio > 0.f && n_cand > 1) ok = ok && (d1 <= (ratio * ratio) * (2.f * (1.f - t.v2)));
  if (dist_thr > 0.f) ok = ok && (d1 <= dist_thr * dist_thr);
  return ok ? (long long)t.i1 : -1;
}

// one warp per row of sim [B, N, M]
__global__ void nn_rows_kernel(const float* __restrict__ sim, int N, int M, const int32_t* __restrict__ lens,
                               float ratio, float dist_thr, long long* __restrict__ nn0) {
  const int b = blockIdx.y, row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= N) return;
  const int n0 = lens ? lens[2 * b] : N, n1 = lens ? lens[2 * b + 1] : M;
  long long* out = nn0 + (size_t)b * N + row;
  if (row >= n0) { if (lane == 0) *out = -1; return; }
  const float* p = sim + ((size_t)b * N + row) * M;
  Top2 t = {-INFINITY, -INFINITY, 0x7fffffff};
  for (int c = lane; c < n1; c += 32) top2_push(t, p[c], c);
  for (int o = 16; o; o >>= 1) {
    Top2 u;
    u.v1 = __shfl_xor_sync(0xffffffffu, t.v1, o);
    u.v2 = __shfl_xor_sync(0xffffffffu, t.v2, o);
    u.i1 = __shfl_xor_sync(0xffffffffu, t.i1, o);
    top2_merge(t, u);
  }
  if (lane == 0) *out = nn_decide(t, n1, ratio, dist_thr);
}

// CTA (32 columns) x (8 row groups): coalesced 128-byte reads along a row, top-2 per column
__global__ void nn_cols_kernel(const float* __restrict__ sim, int N, int M, const int32_t* __restrict__ lens,
                               float ratio, float dist_thr, long long* __restrict__ nn1) {
  __shared__ Top2 sh[8][33];
  const int b = blockIdx.y, cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  const int n0 = lens ? lens[2 * b] : N, n1 = lens ? lens[2 * b + 1] : M;
  Top2 t = {-INFINITY, -INFINITY, 0x7fffffff};
  if (col < n1) {
    const float* p = sim + (size_t)b * N * M + col;
    for (int r = ry; r < n0; r += 8) top2_push(t, p[(size_t)r * M], r);
  }
  sh[ry][cx] = t;
  __syncthreads();
  if (ry == 0 && col < M) {
    for (int k = 1; k < 8; ++k) top2_merge(t, sh[k][cx]);
    nn1[(size_t)b * M + col] = col < n1 ? nn_decide(t, n0, ratio, dist_thr) : -1;
  }
}

// mutual_check on the UNfiltered nn0 / nn1 (both outputs use the other side's original matches), scores = match > -1
__global__ void nn_mutual_kernel(const long long* __restrict__ nn0, const long long* __restrict__ nn1, int N, int M,
                                 int mutual, long long* __restrict__ m0, long long* __restrict__ m1,
                                 float* __restrict__ ms0, float* __restrict__ ms1) {
  const int b = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) {
    long long a = nn0[(size_t)b * N + i];
    if (mutual && M > 0 && a > -1 && nn1[(size_t)b * M + a] != i) a = -1;
    m0[(size_t)b * N + i] = a;
    ms0[(size_t)b * N + i] = a > -1 ? 1.f : 0.f;
  }
  if (i < M) {
    long long a = nn1[(size_t)b * M + i];
    if (mutual && N > 0 && a > -1 && nn0[(size_t)b * N + a] != i) a = -1;
    m1[(size_t)b * M + i] = a;
    ms1[(size_t)b * M + i] = a > -1 ? 1.f : 0.f;
  }
}

// ---- N_pair loss (nearest_neighbor_matcher.py:85-109), forward values ---------------------------------------------
// scores = T * (2 - sqrt(clamp(2 (1 - sim), 1e-6)));  nll = -(sum a (prob0 + prob1)) / (2 num),  prob0 / prob1 = row /
// column log-softmax of scores.  Three streaming passes over sim [B,N,M]: row LSE (warp per row), column LSE (32 columns
// x 8 row groups per CTA, online max/sum merged through shared memory), then the ground-truth pass (warp per row ->
// per-row partial sums, no atomics: bit-reproducible).
__device__ __forceinline__ float npair_q(float sim) { return sqrtf(fmaxf(2.f * (1.f - sim), 1e-6f)); }
__device__ __forceinline__ float npair_score(float sim, float T) { return T * (2.f - npair_q(sim)); }
__device__ __forceinline__ void lse_push(float& mx, float& sm, float v) {
  if (v > mx) { sm = sm * __expf(mx - v) + 1.f; mx = v; }
  else sm += __expf(v - mx);
}
__device__ __forceinline__ void lse_merge(float& mx, float& sm, float mx2, float sm2) {
  if (mx2 == -INFINITY) return;
  if (mx2 > mx) { sm = sm * __expf(mx - mx2) + sm2; mx = mx2; }
  else sm += sm2 * __expf(mx2 - mx);
}

__global__ void npair_rows_kernel(const float* __restrict__ sim, int N, int M, float T, float* __restrict__ lse_r) {
  const int b = blockIdx.y, row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= N) return;
  const float* p = sim + ((size_t)b * N + row) * M;
  float mx = -INFINITY, sm = 0.f;
  for (int c = lane; c < M; c += 32) lse_push(mx, sm, npair_score(p[c], T));
  for (int o = 16; o; o >>= 1) {
    const float mx2 = __shfl_xor_sync(0xffffffffu, mx, o), sm2 = __shfl_xor_sync(0xffffffffu, sm, o);
    lse_merge(mx, sm, mx2, sm2);
  }
  if (lane == 0) lse_r[(size_t)b * N + row] = mx + logf(sm);
}

__global__ void npair_cols_kernel(const float* __restrict__ sim, int N, int M, float T, float* __restrict__ lse_c) {
  __shared__ float smx[8][33], ssm[8][33];
  const int b = blockIdx.y, cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  float mx = -INFINITY, sm = 0.f;
  if (col < M) {
    const float* p = sim + (size_t)b * N * M + col;
    for (int r = ry; r < N; r += 8) lse_push(mx, sm, npair_score(p[(size_t)r * M], T));
  }
  smx[ry][cx] = mx;
  ssm[ry][cx] = sm;
  __syncthreads();
  if (ry == 0 && col < M) {
    for (int k = 1; k < 8; ++k) lse_merge(mx, sm, smx[k][cx], ssm[k][cx]);
    lse_c[(size_t)b * M + col] = mx + logf(sm);
  }
}

// row_sum[b,row] = sum_j a (2 score - lse_r[row] - lse_c[j]);  row_cnt[b,row] = sum_j a
__global__ void npair_gt_kernel(const float* __restrict__ sim, const uint8_t* __restrict__ gt, int N, int M, float T,
                                const float* __restrict__ lse_r, const float* __restrict__ lse_c,
                                float* __restrict__ row_sum, float* __restrict__ row_cnt) {
  const int b = blockIdx.y, row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= N) return;
  const size_t off = ((size_t)b * N + row) * M;
  const float lr = lse_r[(size_t)b * N + row];
  float acc = 0.f, cnt = 0.f;
  for (int c = lane; c < M; c += 32) {
    if (gt[off + c]) {
      acc += 2.f * npair_score(sim[off + c], T) - lr - lse_c[(size_t)b * M + c];
      cnt += 1.f;
    }
  }
  for (int o = 16; o; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    row_sum[(size_t)b * N + row] = acc;
    row_cnt[(size_t)b * N + row] = cnt;
  }
}

// ---- N_pair loss backward --------------------------------------------------------------------------------------------
// d nll_b / d s_ij = coef_b (2 a_ij - r_i exp(s_ij - lse_r_i) - c_j exp(s_ij - lse_c_j)), coef_b = -g_b / (2 num_b),
// r / c = row / column counts of a.  d s / d sim = T / q where the clamp passes (2 (1 - sim) >= 1e-6, torch's rule for
// clamp(min=)), 0 where it clamps; d s / d T = 2 - q.

// c[b,j] = sum_i a_ij: 128 columns x 32 row groups per CTA; a warp load is one 32-byte segment of a row.  The sums are
// integer-valued floats, exact in any order.
__global__ void __launch_bounds__(1024) npair_colcnt_kernel(const uint8_t* __restrict__ gt, int N, int M,
                                                            float* __restrict__ col_cnt) {
  __shared__ float sh[32][129];
  const int b = blockIdx.y, lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 128 + lane;
  const uint8_t* p = gt + (size_t)b * N * M;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
  for (int r = ry; r < N; r += 32) {
    const uint8_t* q = p + (size_t)r * M;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (c0 + 32 * k < M && q[c0 + 32 * k]) acc[k] += 1.f;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) sh[ry][lane + 32 * k] = acc[k];
  __syncthreads();
  if (threadIdx.x < 128) {
    const int col = blockIdx.x * 128 + threadIdx.x;
    float s = 0.f;
    for (int k = 0; k < 32; ++k) s += sh[k][threadIdx.x];
    if (col < M) col_cnt[(size_t)b * M + col] = s;
  }
}

// warp per row, four coalesced 128-byte column chunks in flight per lane: dsim (nullable) and the row's partial
// sum_j d s_ij (2 - q_ij) of d nll / d T (per-row partials, no atomics: bit-reproducible)
__global__ void npair_bwd_kernel(const float* __restrict__ sim, const uint8_t* __restrict__ gt, int N, int M, float T,
                                 const float* __restrict__ lse_r, const float* __restrict__ lse_c,
                                 const float* __restrict__ row_cnt, const float* __restrict__ col_cnt,
                                 const float* __restrict__ coef, float* __restrict__ dsim,
                                 float* __restrict__ dtemp_rows) {
  const int b = blockIdx.y, row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= N) return;
  const size_t off = ((size_t)b * N + row) * M;
  const float lr = lse_r[(size_t)b * N + row], r = row_cnt[(size_t)b * N + row], k = coef[b];
  const float* lc = lse_c + (size_t)b * M;
  const float* cc = col_cnt + (size_t)b * M;
  float acc = 0.f;
  for (int c0 = lane; c0 < M; c0 += 128) {
    float sv[4];
    bool av[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + 32 * u;
      sv[u] = c < M ? sim[off + c] : 0.f;
      av[u] = c < M && gt[off + c];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = c0 + 32 * u;
      if (c < M) {
        const float q = npair_q(sv[u]), s = npair_score(sv[u], T);
        const float ds = k * ((av[u] ? 2.f : 0.f) - r * __expf(s - lr) - cc[c] * __expf(s - lc[c]));
        if (dsim) dsim[off + c] = 2.f * (1.f - sv[u]) >= 1e-6f ? ds * T / q : 0.f;
        acc += ds * (2.f - q);
      }
    }
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) dtemp_rows[(size_t)b * N + row] = acc;
}

}  // namespace

extern "C" int lgb200_npair_loss(const float* similarity, const uint8_t* gt_assignment, int B, int N, int M,
                                 float temperature, float* workspace, float* row_sum, float* row_cnt, void* stream) {
  if (!similarity || !gt_assignment || !workspace || !row_sum || !row_cnt) return LGB200_ERR_NULL;
  if (B <= 0 || N <= 0 || M <= 0 || B > 65535) return LGB200_ERR_SHAPE;
  cudaStream_t st = lg_stream(stream);
  float* lse_r = workspace;               // [B, N]
  float* lse_c = workspace + (size_t)B * N;  // [B, M]
  npair_rows_kernel<<<dim3((N + 7) / 8, B), 256, 0, st>>>(similarity, N, M, temperature, lse_r);
  LG_LAUNCH_CHECK();
  npair_cols_kernel<<<dim3((M + 31) / 32, B), 256, 0, st>>>(similarity, N, M, temperature, lse_c);
  LG_LAUNCH_CHECK();
  npair_gt_kernel<<<dim3((N + 7) / 8, B), 256, 0, st>>>(similarity, gt_assignment, N, M, temperature, lse_r, lse_c,
                                                        row_sum, row_cnt);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_npair_loss_bwd(const float* similarity, const uint8_t* gt_assignment, int B, int N, int M,
                                     float temperature, const float* workspace, const float* row_cnt, const float* coef,
                                     float* col_cnt, float* dsim, float* dtemp_rows, void* stream) {
  if (!similarity || !gt_assignment || !workspace || !row_cnt || !coef || !col_cnt || !dtemp_rows) return LGB200_ERR_NULL;
  if (B <= 0 || N <= 0 || M <= 0 || B > 65535) return LGB200_ERR_SHAPE;
  cudaStream_t st = lg_stream(stream);
  const float* lse_r = workspace;
  const float* lse_c = workspace + (size_t)B * N;
  npair_colcnt_kernel<<<dim3((M + 127) / 128, B), 1024, 0, st>>>(gt_assignment, N, M, col_cnt);
  LG_LAUNCH_CHECK();
  npair_bwd_kernel<<<dim3((N + 7) / 8, B), 256, 0, st>>>(similarity, gt_assignment, N, M, temperature, lse_r, lse_c,
                                                         row_cnt, col_cnt, coef, dsim, dtemp_rows);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

extern "C" int lgb200_nn_scores(const float* d, const float* lse, int B, int Lp, const int32_t* lens, int R, int C,
                                float* similarity, float* log_assignment, void* stream) {
  if (!d || !lse || !log_assignment) return LGB200_ERR_NULL;
  if (B <= 0 || Lp <= 0 || Lp % 128 || R < 1 || C < 1 || R - 1 > Lp || C - 1 > Lp) return LGB200_ERR_SHAPE;
  return lg_simt_assign_scores(d, nullptr, lse, B, Lp, lens, R, C, log_assignment, similarity, lg_stream(stream));
}

extern "C" int lgb200_nn_match(const float* similarity, int B, int N, int M, const int32_t* lens, float ratio_thresh,
                               float distance_thresh, int mutual, int64_t* workspace, int64_t* m0, int64_t* m1,
                               float* ms0, float* ms1, void* stream) {
  if (!workspace || !m0 || !m1 || !ms0 || !ms1 || (!similarity && N > 0 && M > 0)) return LGB200_ERR_NULL;
  if (B <= 0 || N < 0 || M < 0) return LGB200_ERR_SHAPE;
  cudaStream_t st = lg_stream(stream);
  long long* nn0 = reinterpret_cast<long long*>(workspace);
  long long* nn1 = nn0 + (size_t)B * N;
  if (N > 0) {
    nn_rows_kernel<<<dim3((N + 7) / 8, B), 256, 0, st>>>(similarity, N, M, lens, ratio_thresh, distance_thresh, nn0);
    LG_LAUNCH_CHECK();
  }
  if (M > 0) {
    nn_cols_kernel<<<dim3((M + 31) / 32, B), 256, 0, st>>>(similarity, N, M, lens, ratio_thresh, distance_thresh, nn1);
    LG_LAUNCH_CHECK();
  }
  const int mx = N > M ? N : M;
  if (mx > 0) {
    nn_mutual_kernel<<<dim3((mx + 255) / 256, B), 256, 0, st>>>(nn0, nn1, N, M, mutual, reinterpret_cast<long long*>(m0),
                                                               reinterpret_cast<long long*>(m1), ms0, ms1);
    LG_LAUNCH_CHECK();
  }
  return LGB200_OK;
}
