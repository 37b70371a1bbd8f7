// Loss-side reductions over a log-assignment matrix (SURVEY.md 8(f) rank 2; forward values only).
//   lgb200_loss_reduce: one pass along the rows and one along the columns of log_assignment [B,R,C]:
//     row_pos[b,i] = sum_j la[b,i,j] * gt[b,i,j]   (j < C-1)   -> weight_loss's positive term, models/utils/losses.py:11,17
//     row_cnt[b,i] = sum_j gt[b,i,j]                            -> num_pos (:15)
//     row_exp[b,i] = sum_{j<C} exp(la[b,i,j])                   -> losses["row_norm"], lightglue.py:606
//     row_arg[b,i] = argmax_{j<C} la[b,i,j]   (i < R-1)         -> TokenConfidence.loss, lightglue.py:87
//     col_arg[b,j] = argmax_{i<R} la[b,i,j]   (j < C-1)         -> lightglue.py:90
//   arg-maxima follow torch.max: lowest index among equal values, NaN is the maximum.
//   lgb200_loss_reduce_ragged: the same per pair b on its valid block only -- rows i < lens[2b], columns
//     j < lens[2b+1] of the inner block plus the dustbin column C-1 / row R-1 (the inference layout of a padded
//     batch).  The valid columns are visited in the order an un-padded [lens[2b]+1, lens[2b+1]+1] matrix would be,
//     with the dustbin last.  Rows / columns past the counts get 0 sums and arg-maximum -1.
// Per-row outputs (no atomics): the caller sums R-1 numbers per pair, so the result is bit-reproducible.
// HBM-bound: the matrix is read twice (4 + 4 bytes per element) plus one byte of ground truth.
#include "lg_internal.cuh"

namespace {

__device__ __forceinline__ void amax_take(float& va, int& ia, float vb, int ib) {
  // b replaces a if it is larger, the first NaN, or equal (incl. both NaN) with a lower index
  const bool an = va != va, bn = vb != vb;
  if ((bn && !an) || (!an && !bn && vb > va) || (((bn && an) || vb == va) && ib < ia)) { va = vb; ia = ib; }
}

// one warp per row i < R-1; lens (nullable): per-pair counts, see lgb200_loss_reduce_ragged
__global__ void loss_rows_kernel(const float* __restrict__ la, int R, int C, const int32_t* __restrict__ lens,
                                 const uint8_t* __restrict__ gt, float* __restrict__ row_pos,
                                 float* __restrict__ row_cnt, float* __restrict__ row_exp,
                                 int32_t* __restrict__ row_arg) {
  const int b = blockIdx.y, row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= R - 1) return;
  const int n0 = lens ? min(max(lens[2 * b], 0), R - 1) : R - 1, n1 = lens ? min(max(lens[2 * b + 1], 0), C - 1) : C - 1;
  const float* p = la + ((size_t)b * R + row) * C;
  const uint8_t* g = gt ? gt + ((size_t)b * (R - 1) + row) * (C - 1) : nullptr;
  float pos = 0.f, cnt = 0.f, ex = 0.f, best = -INFINITY;
  int bi = 0x7fffffff;
  if (row >= n0) bi = -1;  // past the count: zero sums, arg-maximum -1
  else
    for (int k = lane; k <= n1; k += 32) {  // valid columns, then the dustbin
      const int c = k < n1 ? k : C - 1;
      const float v = p[c];
      ex += expf(v);
      if (g && c < C - 1 && g[c]) { pos += v; cnt += 1.f; }
      amax_take(best, bi, v, c);
    }
  for (int o = 16; o; o >>= 1) {
    pos += __shfl_xor_sync(0xffffffffu, pos, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    ex += __shfl_xor_sync(0xffffffffu, ex, o);
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    amax_take(best, bi, ov, oi);
  }
  if (lane == 0) {
    const size_t o = (size_t)b * (R - 1) + row;
    if (row_pos) row_pos[o] = pos;
    if (row_cnt) row_cnt[o] = cnt;
    if (row_exp) row_exp[o] = ex;
    if (row_arg) row_arg[o] = bi;
  }
}

// thread per column j < C-1, 8 row groups per CTA merged through shared memory; a warp reads 128 contiguous bytes
__global__ void loss_cols_kernel(const float* __restrict__ la, int R, int C, const int32_t* __restrict__ lens,
                                 int32_t* __restrict__ col_arg) {
  __shared__ float sv[8][32];
  __shared__ int si[8][32];
  const int b = blockIdx.y, lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + lane;
  const int n0 = lens ? min(max(lens[2 * b], 0), R - 1) : R - 1, n1 = lens ? min(max(lens[2 * b + 1], 0), C - 1) : C - 1;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  if (col < n1) {
    const float* p = la + (size_t)b * R * C + col;
    for (int k = grp; k <= n0; k += 8) {  // valid rows, then the dustbin
      const int r = k < n0 ? k : R - 1;
      amax_take(best, bi, p[(size_t)r * C], r);
    }
  }
  sv[grp][lane] = best;
  si[grp][lane] = bi;
  __syncthreads();
  if (grp == 0 && col < C - 1) {
    for (int g2 = 1; g2 < 8; ++g2) amax_take(best, bi, sv[g2][lane], si[g2][lane]);
    col_arg[(size_t)b * (C - 1) + col] = col < n1 ? bi : -1;
  }
}

}  // namespace

static int loss_reduce(const float* la, int B, int R, int C, const int32_t* lens, const uint8_t* gt, float* row_pos,
                       float* row_cnt, float* row_exp, int32_t* row_arg, int32_t* col_arg, void* stream) {
  cudaStream_t st = lg_stream(stream);
  if (R > 1 && (row_pos || row_cnt || row_exp || row_arg)) {
    loss_rows_kernel<<<dim3((R - 1 + 7) / 8, B), 256, 0, st>>>(la, R, C, lens, gt, row_pos, row_cnt, row_exp, row_arg);
    LG_LAUNCH_CHECK();
  }
  if (C > 1 && col_arg) {
    loss_cols_kernel<<<dim3((C - 1 + 31) / 32, B), 256, 0, st>>>(la, R, C, lens, col_arg);
    LG_LAUNCH_CHECK();
  }
  return LGB200_OK;
}

extern "C" int lgb200_loss_reduce(const float* log_assignment, int B, int R, int C, const uint8_t* gt_assignment,
                                  float* row_pos, float* row_cnt, float* row_exp, int32_t* row_arg, int32_t* col_arg,
                                  void* stream) {
  if (!log_assignment) return LGB200_ERR_NULL;
  if (B < 0 || R < 1 || C < 1) return LGB200_ERR_SHAPE;
  if (B == 0) return LGB200_OK;
  return loss_reduce(log_assignment, B, R, C, nullptr, gt_assignment, row_pos, row_cnt, row_exp, row_arg, col_arg,
                     stream);
}

extern "C" int lgb200_loss_reduce_ragged(const float* log_assignment, int B, int R, int C, const int32_t* lens,
                                         const uint8_t* gt_assignment, float* row_pos, float* row_cnt, float* row_exp,
                                         int32_t* row_arg, int32_t* col_arg, void* stream) {
  if (!log_assignment || !lens) return LGB200_ERR_NULL;
  if (B < 0 || R < 1 || C < 1) return LGB200_ERR_SHAPE;
  if (B == 0) return LGB200_OK;
  return loss_reduce(log_assignment, B, R, C, lens, gt_assignment, row_pos, row_cnt, row_exp, row_arg, col_arg,
                     stream);
}
