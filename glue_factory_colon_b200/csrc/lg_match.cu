// The whole matcher behind one call (include/lightglue_b200.h, "whole matcher"): weight packing on the device
// (lgb200_pack_weights, the layouts of LightGlue._pack) and the no-grad forward (lgb200_match, the non-adaptive eval
// path of LightGlue._forward_impl) as a fixed sequence of the library's own entry points.  The per-pair counts are
// read on the device only, so one call can be captured into a CUDA graph at a fixed capacity and replayed for any
// counts.  lgb200_pack_weights_adaptive / lgb200_match_adaptive add adaptive depth and width ("adaptive matcher"):
// the calls of _forward_impl(static=True) with its host-side tail (exit layers, MatchAssignment per exit layer,
// filter_matches at the pruned counts) moved onto the device.
#include "lg_internal.cuh"
#include <cuda_fp16.h>
#include <limits.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <vector>

namespace {

// ---- packed-weight table ---------------------------------------------------------------------------------------
// Per layer, in this order (lightglue.py:_pack names); then the tail.  W = weight matrix in the precision's operand
// format (bf16 [N][K] or fp16 planes [2][N][K] of 256 w), F = fp32.
enum {
  E_QKV_W, E_QKV_B, E_SF0_W, E_SF0_B, E_SLN_G, E_SLN_B, E_SF3_W, E_SF3_B,
  E_CQV_W, E_CQV_B, E_CF0_W, E_CF0_B, E_CLN_G, E_CLN_B, E_CF3_W, E_CF3_B, E_PER_LAYER
};
enum { T_WR, T_FP_W, T_FP_B, T_M_W, T_M_B, T_IN_W, T_IN_B };
// adaptive table: after the entries above, per layer l < n_layers-1 at n_entries + 6 l + j
enum { A_FP_W, A_FP_B, A_M_W, A_M_B, A_TK_W, A_TK_B, A_PER_LAYER };

enum { FMT_F32 = 0, FMT_BF16 = 1, FMT_PLANES = 2 };

struct EntryShape {
  bool weight;  // W (else F)
  int N, K;     // F entries: N * K floats
};

int cfg_check(const lgb200_match_config* cfg) {
  if (!cfg) return LGB200_ERR_NULL;
  if (cfg->n_layers < 1 || (cfg->kdim != 2 && cfg->kdim != 4) || cfg->input_dim <= 0 || cfg->input_dim % 64)
    return LGB200_ERR_SHAPE;
  if (cfg->precision != LGB200_BF16 && cfg->precision != LGB200_F32X3) return LGB200_ERR_PRECISION;
  return LGB200_OK;
}

int n_entries(const lgb200_match_config* cfg) {
  return E_PER_LAYER * cfg->n_layers + 5 + (cfg->input_dim != 256 ? 2 : 0);
}

int n_adaptive_entries(const lgb200_match_config* cfg) { return n_entries(cfg) + A_PER_LAYER * (cfg->n_layers - 1); }

EntryShape entry_shape(const lgb200_match_config* cfg, int e) {
  if (e >= n_entries(cfg)) {
    switch ((e - n_entries(cfg)) % A_PER_LAYER) {
      case A_FP_W: return {true, 256, 256};
      case A_M_B: case A_TK_B: return {false, 1, 1};
      default: return {false, 256, 1};  // fp_b, m_w, tk_w
    }
  }
  if (e < E_PER_LAYER * cfg->n_layers) {
    switch (e % E_PER_LAYER) {
      case E_QKV_W: return {true, 768, 256};
      case E_QKV_B: return {false, 768, 1};
      case E_SF0_W: case E_CF0_W: return {true, 512, 512};
      case E_SF3_W: case E_CF3_W: return {true, 256, 512};
      case E_SF3_B: case E_CF3_B: return {false, 256, 1};
      case E_CQV_W: return {true, 512, 256};
      default: return {false, 512, 1};  // sf0_b, sln_g, sln_b, cqv_b, cf0_b, cln_g, cln_b
    }
  }
  switch (e - E_PER_LAYER * cfg->n_layers) {
    case T_WR: return {false, 32, cfg->kdim};
    case T_FP_W: return {true, 256, 256};
    case T_FP_B: return {false, 256, 1};
    case T_M_W: return {false, 256, 1};
    case T_M_B: return {false, 1, 1};
    case T_IN_W: return {true, 256, cfg->input_dim};
    default: return {false, 256, 1};  // in_b
  }
}

long long align256(long long b) { return (b + 255) & ~255LL; }

long long entry_bytes(const lgb200_match_config* cfg, const EntryShape& s) {
  const long long nk = (long long)s.N * s.K;
  if (!s.weight) return nk * 4;
  return cfg->precision == LGB200_BF16 ? nk * 2 : nk * 4;  // planes: 2 x fp16
}

// ---- packing kernels ---------------------------------------------------------------------------------------------

// One element of a W entry: bf16, or the split planes of weight_planes (lightglue.py): t = 256 w, hi = fp16(t),
// lo = fp16(t - hi), stored [2][N][K].
__device__ __forceinline__ void store_elem(int fmt, void* out, long long idx, long long nk, float v) {
  if (fmt == FMT_F32) {
    reinterpret_cast<float*>(out)[idx] = v;
  } else if (fmt == FMT_BF16) {
    reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v);
  } else {
    const float t = v * LG_X3_EW;
    const __half hi = __float2half_rn(t);
    __half* o = reinterpret_cast<__half*>(out);
    o[idx] = hi;
    o[nk + idx] = __float2half_rn(t - __half2float(hi));
  }
}

// out row r of [N][K] = row r of a (r < na) or row r - na of b (the to_qk | to_v concatenation).  perm_qkv: row r =
// part*256 + head*64 + d is read from the reference's row head*192 + d*3 + part (lightglue.py:158).
__global__ void pack_rows_kernel(const float* a, int na, const float* b, int N, int K, int perm_qkv, int fmt,
                                 void* out) {
  const long long nk = (long long)N * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nk; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / K), c = (int)(i % K);
    const int sr = perm_qkv ? ((r & 255) >> 6) * 192 + (r & 63) * 3 + (r >> 8) : r;
    const float v = sr < na ? a[(long long)sr * K + c] : b[(long long)(sr - na) * K + c];
    store_elem(fmt, out, i, nk, v);
  }
}

// The out_proj / to_out fold of _pack: W1' = [W1x | W1m Wo] [512][512], b1' = b1 + W1m bo, every sum in float64 and
// rounded to fp32 once, then stored in the W format.  Threads 0 .. 512*512-1 form W1', the next 512 form b1'.
__global__ void fold_kernel(const float* w1, const float* b1, const float* wo, const float* bo, int fmt, void* out_w,
                            float* out_b) {
  constexpr int D = 256, N = 512;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N * N) {
    const int r = i / N, c = i % N;
    float v;
    if (c < D) {
      v = w1[r * N + c];
    } else {
      double acc = 0.0;
      for (int k = 0; k < D; ++k) acc = fma((double)w1[r * N + D + k], (double)wo[k * D + (c - D)], acc);
      v = (float)acc;
    }
    store_elem(fmt, out_w, i, (long long)N * N, v);
  } else if (i < N * N + N) {
    const int r = i - N * N;
    double acc = 0.0;
    for (int k = 0; k < D; ++k) acc = fma((double)w1[r * N + D + k], (double)bo[k], acc);
    out_b[r] = (float)((double)b1[r] + acc);
  }
}

// lens[2b] = clamp(counts0[b], 0, m), lens[2b+1] = clamp(counts1[b], 0, n) (m / n where a count array is NULL).
// order_self / order_cross (nullable): the sequences sorted by lens[s] / lens[s ^ 1], longest first, ties by index --
// the permutations np.argsort(-key, kind="stable") of LightGlue._forward_impl.  One block.
__global__ void lens_order_kernel(const int32_t* c0, const int32_t* c1, int B, int m, int n, int32_t* lens,
                                  int32_t* order_self, int32_t* order_cross) {
  const int S = 2 * B;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    const int32_t* c = (s & 1) ? c1 : c0;
    const int cap = (s & 1) ? n : m;
    lens[s] = c ? min(max(c[s >> 1], 0), cap) : cap;
  }
  if (!order_self) return;
  __syncthreads();
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    const int vs = lens[s], vx = lens[s ^ 1];
    int rs = 0, rx = 0;
    for (int t = 0; t < S; ++t) {
      const int ut = lens[t], uxt = lens[t ^ 1];
      rs += ut > vs || (ut == vs && t < s);
      rx += uxt > vx || (uxt == vx && t < s);
    }
    order_self[rs] = s;
    order_cross[rx] = s;
  }
}

// ---- adaptive state kernels ------------------------------------------------------------------------------------------

// The device state of an adaptive forward (the tensors LightGlue._forward_impl creates for it): lens_active = lens,
// total[b] = lens[2b] + lens[2b+1], done = 0 and, with point pruning (ind != NULL), ind[s][l] = l and prune_cnt = 1.
__global__ void adaptive_init_kernel(const int32_t* lens, int B, int Lp, int32_t* done, int32_t* lens_active,
                                     int32_t* total, int32_t* ind, int32_t* prune_cnt) {
  const int S = 2 * B;
  const long long n = ind ? (long long)S * Lp : S;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (i < S) lens_active[i] = lens[i];
    if (i < B) {
      done[i] = 0;
      total[i] = lens[2 * i] + lens[2 * i + 1];
    }
    if (ind) {
      ind[i] = (int32_t)(i % Lp);
      prune_cnt[i] = 1;
    }
  }
}

// The per-exit-layer counts of the tail: lens_g[e][s] = lens[s] if pair s/2 exits at layer e (done - 1, or L-1 if it
// never stopped), else 0 -- a sequence with count 0 is left untouched by every kernel of a MatchAssignment group.
__global__ void exit_groups_kernel(const int32_t* done, const int32_t* lens, int S, int L, int32_t* lens_g) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L * S; i += gridDim.x * blockDim.x) {
    const int e = i / S, s = i % S, d = done[s >> 1];
    lens_g[i] = (d ? d - 1 : L - 1) == e ? lens[s] : 0;
  }
}

// The outputs of lgb200_match_adaptive past those of lgb200_match, one warp per (pair, image, row):
//   desc0/1 (x != NULL): row l < k of sequence s copied from x (rows of 256 elements of es bytes), zeros past k;
//   prune0/1: prune_cnt[s][l], or L where prune_cnt is NULL;
//   exit_layer[b] = done[b] - 1 (L - 1 where done is NULL or 0), final_counts[b] = (k0, k1).
// k = lens[s], or m / n where lens is NULL.
__global__ void adaptive_outputs_kernel(int B, int m, int n, int L, int Lp, const int32_t* lens, const int32_t* done,
                                        const int32_t* prune_cnt, const void* x, int es, void* desc0, void* desc1,
                                        int32_t* prune0, int32_t* prune1, int32_t* exit_layer,
                                        int32_t* final_counts) {
  const int lane = threadIdx.x & 31;
  const long long rows0 = (long long)B * m, rows = rows0 + (long long)B * n;
  const long long warps = (long long)gridDim.x * blockDim.x / 32;
  for (long long r = (blockIdx.x * (long long)blockDim.x + threadIdx.x) / 32; r < rows; r += warps) {
    const int img = r >= rows0;
    const int cap = img ? n : m;
    const long long rr = img ? r - rows0 : r;
    const int b = (int)(rr / cap), l = (int)(rr % cap), s = 2 * b + img;
    const int k = lens ? lens[s] : cap;
    void* d = img ? desc1 : desc0;
    if (x && d) {
      const int vecs = 256 * es / 16;  // 16-byte words per row: 32 (bf16) or 64 (fp32)
      const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(x) + ((long long)s * Lp + l) * 256 * es);
      uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<char*>(d) + ((long long)b * cap + l) * 256 * es);
      for (int w = lane; w < vecs; w += 32) dst[w] = l < k ? src[w] : make_uint4(0, 0, 0, 0);
    }
    int32_t* p = img ? prune1 : prune0;
    if (p && lane == 0) p[(long long)b * cap + l] = prune_cnt ? prune_cnt[(long long)s * Lp + l] : L;
  }
  if (blockIdx.x == 0) {
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
      if (exit_layer) exit_layer[b] = done && done[b] ? done[b] - 1 : L - 1;
      if (final_counts) {
        final_counts[2 * b] = lens ? lens[2 * b] : m;
        final_counts[2 * b + 1] = lens ? lens[2 * b + 1] : n;
      }
    }
  }
}

// ---- forward plan --------------------------------------------------------------------------------------------------

struct Plan {
  int prec, S, Lp, T, R, C;
  bool x3, proj, use_lens, ordered;
  // byte offsets into the workspace; xs .. hid and z .. lse are contiguous (one memset each)
  long long x, xin, xin_s, rot, xs, q, k, v, ctx, msg, hid, hid_end, z, lse, lse_end, sim, fm_ws, lens;
  // lgb200_match_adaptive only (after everything above, so that lgb200_match's layout is a prefix): conf | msig and
  // ind_b | x_b | rot_b are contiguous; ctl = done [B] | lens_active [S] | total [B]; lens_g [n_layers][S]
  long long ind, pcnt, conf, msig, msig_end, ind_b, x_b, rot_b, rot_b_end, ctl, lens_g;
  long long total;
};

int make_plan(const lgb200_match_config* cfg, int B, int m, int n, bool variable, bool adaptive, Plan* p) {
  int rc = cfg_check(cfg);
  if (rc) return rc;
  if (B <= 0 || m < 0 || n < 0) return LGB200_ERR_SHAPE;
  p->prec = cfg->precision;
  p->x3 = cfg->precision == LGB200_F32X3;
  p->proj = cfg->input_dim != 256;
  const int gran = p->x3 ? 256 : 128;  // (the x3 similarity GEMM tiles the keys by 256)
  const long long mx = m > n ? m : n;
  const long long Lp = mx <= gran ? gran : (mx + gran - 1) / gran * gran;
  const long long T = 2LL * B * Lp;
  if (T * 512 > INT_MAX || (long long)B * (m + 1) * (n + 1) > INT_MAX) return LGB200_ERR_SHAPE;
  p->S = 2 * B;
  p->Lp = (int)Lp;
  p->T = (int)T;
  p->R = m + 1;
  p->C = n + 1;
  p->use_lens = variable || m != Lp || n != Lp;
  p->ordered = variable;
  const long long act = p->x3 ? 4 : 2;  // activation element: fp32 master / bf16
  const long long op = p->x3 ? 4 : 2;   // MMA operand element: fp16 plane pair / bf16
  long long off = 0;
  auto take = [&](long long bytes) { const long long o = off; off += align256(bytes); return o; };
  p->x = take(T * 256 * act);
  p->xin = p->proj ? take(T * cfg->input_dim * act) : 0;
  p->xin_s = p->proj && p->x3 ? take(T * cfg->input_dim * op) : 0;
  p->rot = take(p->x3 ? T * 64 * 4 : T * 32 * 4);  // fp32 (cos, sin) / packed fp16 (cos, sin)
  p->xs = p->x3 ? take(T * 256 * op) : off;
  p->q = take(T * 256 * op);
  p->k = take(T * 256 * op);
  p->v = take(T * 256 * op);
  p->ctx = take(T * 256 * op);
  p->msg = take(T * 256 * op);
  p->hid = take(T * 512 * op);
  p->hid_end = off;
  p->z = take(T * 4);
  p->lse = take(T * 4);
  p->lse_end = off;
  p->sim = p->x3 ? take((long long)B * Lp * Lp * 4) : 0;
  p->fm_ws = take(8LL * B * (p->R + p->C));
  p->lens = take(3LL * p->S * 4);
  if (adaptive) {
    p->ind = take(T * 4);
    p->pcnt = take(T * 4);
    p->conf = take(T * 4);
    p->msig = take(T * 4);
    p->msig_end = off;
    p->ind_b = take(T * 4);
    p->x_b = take(T * 256 * act);
    p->rot_b = take(p->x3 ? T * 64 * 4 : T * 32 * 4);
    p->rot_b_end = off;
    p->ctl = take(4LL * (2 * B + p->S));
    p->lens_g = take(4LL * cfg->n_layers * p->S);
  }
  p->total = off;
  return LGB200_OK;
}

// LightGlue.confidence_threshold (lightglue.py:555-558): clip(0.8 + 0.1 exp(-4 l / L), 0, 1) in double, as a float
float confidence_threshold(int layer, int L) {
  const double t = 0.8 + 0.1 * exp(-4.0 * layer / L);
  return (float)(t < 0.0 ? 0.0 : t > 1.0 ? 1.0 : t);
}

#define LG_TRY(call)            \
  do {                          \
    const int rc__ = (call);    \
    if (rc__) return rc__;      \
  } while (0)

// *out = the tensor called `name` among names[0 .. n): LGB200_ERR_WEIGHTS if it is missing, LGB200_ERR_NULL if NULL
int find_weight(int n, const char* const* names, const float* const* tensors, const char* name, const float** out) {
  int i = 0;
  for (; i < n; ++i)
    if (names[i] && strcmp(names[i], name) == 0) break;
  if (i == n) return LGB200_ERR_WEIGHTS;
  if (!tensors[i]) return LGB200_ERR_NULL;
  *out = tensors[i];
  return LGB200_OK;
}

// entry e of the table from rows of a (and b, see pack_rows_kernel) in the entry's format
int pack_entry(const lgb200_match_config* cfg, int e, const float* a, int na, const float* b, int perm, void* dst,
               cudaStream_t st) {
  const EntryShape s = entry_shape(cfg, e);
  const long long nk = (long long)s.N * s.K;
  const int blocks = (int)((nk + 255) / 256 < 1184 ? (nk + 255) / 256 : 1184);
  const int wfmt = cfg->precision == LGB200_BF16 ? FMT_BF16 : FMT_PLANES;
  pack_rows_kernel<<<blocks, 256, 0, st>>>(a, na, b, s.N, s.K, perm, s.weight ? wfmt : FMT_F32, dst);
  LG_LAUNCH_CHECK();
  return LGB200_OK;
}

}  // namespace

extern "C" int lgb200_weight_table_size(const lgb200_match_config* cfg, int* entries, long long* pack_bytes) {
  if (!cfg || !entries || !pack_bytes) return LGB200_ERR_NULL;
  LG_TRY(cfg_check(cfg));
  const int ne = n_entries(cfg);
  long long bytes = 0;
  for (int e = 0; e < ne; ++e) bytes += align256(entry_bytes(cfg, entry_shape(cfg, e)));
  *entries = ne;
  *pack_bytes = bytes;
  return LGB200_OK;
}

extern "C" int lgb200_pack_weights(const lgb200_match_config* cfg, int n, const char* const* names,
                                   const float* const* tensors, void* pack_buf, long long pack_bytes,
                                   const void** table, void* stream) {
  if (!cfg || !pack_buf || !table || (n > 0 && (!names || !tensors))) return LGB200_ERR_NULL;
  LG_TRY(cfg_check(cfg));
  if (n < 0) return LGB200_ERR_SHAPE;
  int ne;
  long long need;
  LG_TRY(lgb200_weight_table_size(cfg, &ne, &need));
  if (pack_bytes < need || reinterpret_cast<uintptr_t>(pack_buf) % 256) return LGB200_ERR_SHAPE;

  // every required tensor is looked up before the first launch: a missing one leaves pack_buf untouched
  const int L = cfg->n_layers;
  const int n_src = 22 * L + 5 + (cfg->input_dim != 256 ? 2 : 0);
  std::vector<const float*> src(n_src);
  static const char* kLayer[22] = {
      "self_attn.Wqkv.weight", "self_attn.Wqkv.bias", "self_attn.out_proj.weight", "self_attn.out_proj.bias",
      "self_attn.ffn.0.weight", "self_attn.ffn.0.bias", "self_attn.ffn.1.weight", "self_attn.ffn.1.bias",
      "self_attn.ffn.3.weight", "self_attn.ffn.3.bias", "cross_attn.to_qk.weight", "cross_attn.to_qk.bias",
      "cross_attn.to_v.weight", "cross_attn.to_v.bias", "cross_attn.to_out.weight", "cross_attn.to_out.bias",
      "cross_attn.ffn.0.weight", "cross_attn.ffn.0.bias", "cross_attn.ffn.1.weight", "cross_attn.ffn.1.bias",
      "cross_attn.ffn.3.weight", "cross_attn.ffn.3.bias"};
  char name[128];
  for (int j = 0; j < n_src; ++j) {
    if (j < 22 * L) {
      snprintf(name, sizeof name, "transformers.%d.%s", j / 22, kLayer[j % 22]);
    } else {
      static const char* kTail[7] = {"posenc.Wr.weight", "final_proj.weight", "final_proj.bias",
                                     "matchability.weight", "matchability.bias", "input_proj.weight",
                                     "input_proj.bias"};
      const int t = j - 22 * L;
      if (t >= 1 && t <= 4)  // only the last layer's MatchAssignment runs in the forward (lightglue.py:523-524)
        snprintf(name, sizeof name, "log_assignment.%d.%s", L - 1, kTail[t]);
      else
        snprintf(name, sizeof name, "%s", kTail[t]);
    }
    LG_TRY(find_weight(n, names, tensors, name, &src[j]));
  }

  char* base = reinterpret_cast<char*>(pack_buf);
  long long off = 0;
  for (int e = 0; e < ne; ++e) {
    table[e] = base + off;
    off += align256(entry_bytes(cfg, entry_shape(cfg, e)));
  }
  const int wfmt = cfg->precision == LGB200_BF16 ? FMT_BF16 : FMT_PLANES;
  cudaStream_t st = lg_stream(stream);
  auto rows = [&](int e, const float* a, int na, const float* b, int perm) -> int {
    return pack_entry(cfg, e, a, na, b, perm, const_cast<void*>(table[e]), st);
  };
  auto fold = [&](int ew, int eb, const float* w1, const float* b1, const float* wo, const float* bo) -> int {
    fold_kernel<<<(512 * 512 + 512 + 255) / 256, 256, 0, st>>>(w1, b1, wo, bo, wfmt, const_cast<void*>(table[ew]),
                                                               (float*)const_cast<void*>(table[eb]));
    LG_LAUNCH_CHECK();
    return LGB200_OK;
  };
  for (int l = 0; l < L; ++l) {
    const float* const* s = src.data() + 22 * l;
    const int e = E_PER_LAYER * l;
    LG_TRY(rows(e + E_QKV_W, s[0], 768, nullptr, 1));
    LG_TRY(rows(e + E_QKV_B, s[1], 768, nullptr, 1));
    LG_TRY(fold(e + E_SF0_W, e + E_SF0_B, s[4], s[5], s[2], s[3]));
    LG_TRY(rows(e + E_SLN_G, s[6], 512, nullptr, 0));
    LG_TRY(rows(e + E_SLN_B, s[7], 512, nullptr, 0));
    LG_TRY(rows(e + E_SF3_W, s[8], 256, nullptr, 0));
    LG_TRY(rows(e + E_SF3_B, s[9], 256, nullptr, 0));
    LG_TRY(rows(e + E_CQV_W, s[10], 256, s[12], 0));
    LG_TRY(rows(e + E_CQV_B, s[11], 256, s[13], 0));
    LG_TRY(fold(e + E_CF0_W, e + E_CF0_B, s[16], s[17], s[14], s[15]));
    LG_TRY(rows(e + E_CLN_G, s[18], 512, nullptr, 0));
    LG_TRY(rows(e + E_CLN_B, s[19], 512, nullptr, 0));
    LG_TRY(rows(e + E_CF3_W, s[20], 256, nullptr, 0));
    LG_TRY(rows(e + E_CF3_B, s[21], 256, nullptr, 0));
  }
  const float* const* t = src.data() + 22 * L;
  const int e = E_PER_LAYER * L;
  LG_TRY(rows(e + T_WR, t[0], 32, nullptr, 0));
  LG_TRY(rows(e + T_FP_W, t[1], 256, nullptr, 0));
  LG_TRY(rows(e + T_FP_B, t[2], 256, nullptr, 0));
  LG_TRY(rows(e + T_M_W, t[3], 256, nullptr, 0));
  LG_TRY(rows(e + T_M_B, t[4], 1, nullptr, 0));
  if (cfg->input_dim != 256) {
    LG_TRY(rows(e + T_IN_W, t[5], 256, nullptr, 0));
    LG_TRY(rows(e + T_IN_B, t[6], 256, nullptr, 0));
  }
  return LGB200_OK;
}

extern "C" int lgb200_adaptive_table_size(const lgb200_match_config* cfg, int* entries, long long* pack_bytes) {
  if (!cfg || !entries || !pack_bytes) return LGB200_ERR_NULL;
  LG_TRY(cfg_check(cfg));
  const int ne = n_adaptive_entries(cfg);
  long long bytes = 0;
  for (int e = 0; e < ne; ++e) bytes += align256(entry_bytes(cfg, entry_shape(cfg, e)));
  *entries = ne;
  *pack_bytes = bytes;
  return LGB200_OK;
}

extern "C" int lgb200_pack_weights_adaptive(const lgb200_match_config* cfg, int n, const char* const* names,
                                            const float* const* tensors, void* pack_buf, long long pack_bytes,
                                            const void** table, void* stream) {
  if (!cfg || !pack_buf || !table || (n > 0 && (!names || !tensors))) return LGB200_ERR_NULL;
  LG_TRY(cfg_check(cfg));
  if (n < 0) return LGB200_ERR_SHAPE;
  int ne_all;
  long long need;
  LG_TRY(lgb200_adaptive_table_size(cfg, &ne_all, &need));
  if (pack_bytes < need || reinterpret_cast<uintptr_t>(pack_buf) % 256) return LGB200_ERR_SHAPE;

  // the adaptive heads are looked up first, lgb200_pack_weights looks up the rest: nothing is launched before every
  // required tensor is found
  const int L = cfg->n_layers;
  std::vector<const float*> src(A_PER_LAYER * (L - 1));
  static const char* kHead[A_PER_LAYER] = {"log_assignment.%d.final_proj.weight",  "log_assignment.%d.final_proj.bias",
                                           "log_assignment.%d.matchability.weight", "log_assignment.%d.matchability.bias",
                                           "token_confidence.%d.token.0.weight",   "token_confidence.%d.token.0.bias"};
  char name[128];
  for (int j = 0; j < (int)src.size(); ++j) {
    snprintf(name, sizeof name, kHead[j % A_PER_LAYER], j / A_PER_LAYER);
    LG_TRY(find_weight(n, names, tensors, name, &src[j]));
  }
  LG_TRY(lgb200_pack_weights(cfg, n, names, tensors, pack_buf, pack_bytes, table, stream));

  const int ne = n_entries(cfg);
  long long off = 0;
  for (int e = 0; e < ne_all; ++e) {
    if (e >= ne) table[e] = reinterpret_cast<char*>(pack_buf) + off;
    off += align256(entry_bytes(cfg, entry_shape(cfg, e)));
  }
  cudaStream_t st = lg_stream(stream);
  for (int j = 0; j < (int)src.size(); ++j) {
    const EntryShape s = entry_shape(cfg, ne + j);
    LG_TRY(pack_entry(cfg, ne + j, src[j], s.N, nullptr, 0, const_cast<void*>(table[ne + j]), st));
  }
  return LGB200_OK;
}

extern "C" int lgb200_match_workspace(const lgb200_match_config* cfg, int B, int m, int n, long long* bytes) {
  if (!cfg || !bytes) return LGB200_ERR_NULL;
  Plan p;
  LG_TRY(make_plan(cfg, B, m, n, true, false, &p));  // (the layout does not depend on the counts)
  *bytes = p.total;
  return LGB200_OK;
}

extern "C" int lgb200_match_adaptive_workspace(const lgb200_match_config* cfg, int B, int m, int n, long long* bytes) {
  if (!cfg || !bytes) return LGB200_ERR_NULL;
  Plan p;
  LG_TRY(make_plan(cfg, B, m, n, true, true, &p));  // (nor on the confidences)
  *bytes = p.total;
  return LGB200_OK;
}

namespace {

// What lgb200_match_adaptive adds to lgb200_match.
struct Adaptive {
  bool depth, width;  // the modes that are on
  float depth_conf, width_conf;
  int32_t *prune0, *prune1, *exit_layer, *final_counts;
};

// The forward of both entry points, after their argument checks.  ad == NULL (lgb200_match), or neither mode on: the
// calls of lgb200_match.  Otherwise the calls of LightGlue._forward_impl(static=True) with its tail on the device.
int forward(const lgb200_match_config* cfg, Plan p, const Adaptive* ad, const void* const* table, int B, int m, int n,
            const float* kpts0, const float* kpts1, const float* desc0, const float* desc1, const float* size0,
            const float* size1, const int32_t* counts0, const int32_t* counts1, int64_t* matches0, int64_t* matches1,
            float* scores0, float* scores1, float* log_assignment, void* desc_out0, void* desc_out1, void* workspace,
            void* stream) {
  const bool early = ad && ad->depth, prune = ad && ad->width, adaptive = early || prune;
  if (adaptive) p.use_lens = true;  // (as in the Python forward: the adaptive kernels shrink lens on the device)
  const int prec = p.prec, S = p.S, Lp = p.Lp, T = p.T, L = cfg->n_layers, din = cfg->input_dim;
  const bool x3 = p.x3;
  char* ws = reinterpret_cast<char*>(workspace);
  void* x = ws + p.x;
  void* xs = x3 ? ws + p.xs : nullptr;
  void *q = ws + p.q, *k = ws + p.k, *v = ws + p.v, *ctx = ws + p.ctx, *md = ws + p.msg, *hid = ws + p.hid;
  float* rot = x3 ? reinterpret_cast<float*>(ws + p.rot) : nullptr;
  void* rot16 = x3 ? nullptr : ws + p.rot;
  float* z = reinterpret_cast<float*>(ws + p.z);
  float* lse = reinterpret_cast<float*>(ws + p.lse);
  float* sim = x3 ? reinterpret_cast<float*>(ws + p.sim) : nullptr;
  void* fm_ws = ws + p.fm_ws;
  int32_t* lens_buf = reinterpret_cast<int32_t*>(ws + p.lens);
  const int32_t* lens = p.use_lens ? lens_buf : nullptr;
  const int32_t* order_self = p.ordered ? lens_buf + S : nullptr;
  const int32_t* order_cross = p.ordered ? lens_buf + 2 * S : nullptr;
  // adaptive state: lens_act = the counts the layers see (0 for pairs that stopped), lens = the pruned counts
  int32_t *done = nullptr, *lens_act = nullptr, *total = nullptr, *ind = nullptr, *ind_b = nullptr, *pcnt = nullptr;
  float *conf = nullptr, *msig = nullptr;
  void* x_b = nullptr;
  float* rot_b = nullptr;
  void* rot16_b = nullptr;
  if (adaptive) {
    done = reinterpret_cast<int32_t*>(ws + p.ctl);
    lens_act = done + B;
    total = lens_act + S;
    conf = reinterpret_cast<float*>(ws + p.conf);
    msig = reinterpret_cast<float*>(ws + p.msig);
    if (prune) {
      ind = reinterpret_cast<int32_t*>(ws + p.ind);
      ind_b = reinterpret_cast<int32_t*>(ws + p.ind_b);
      pcnt = reinterpret_cast<int32_t*>(ws + p.pcnt);
      x_b = ws + p.x_b;
      rot_b = x3 ? reinterpret_cast<float*>(ws + p.rot_b) : nullptr;
      rot16_b = x3 ? nullptr : ws + p.rot_b;
    }
  }
  const int32_t* la = adaptive ? lens_act : lens;
  const float* f32 = nullptr;  // typed NULL
  cudaStream_t st = lg_stream(stream);
  auto W = [&](int e) { return table[e]; };
  auto F = [&](int e) { return reinterpret_cast<const float*>(table[e]); };
  auto memset0 = [&](long long from, long long to) -> int {
    const cudaError_t ce = cudaMemsetAsync(ws + from, 0, to - from, st);
    return ce == cudaSuccess ? LGB200_OK : (int)ce;
  };

  if (p.use_lens) {
    lens_order_kernel<<<1, 256, 0, st>>>(counts0, counts1, B, m, n, lens_buf, p.ordered ? lens_buf + S : nullptr,
                                         p.ordered ? lens_buf + 2 * S : nullptr);
    LG_LAUNCH_CHECK();
    // padded rows must hold finite values (masked keys multiply V rows by exactly 0)
    LG_TRY(memset0(p.xs, p.hid_end));
  }
  LG_TRY(memset0(p.z, p.lse_end));
  if (adaptive) {
    const long long nt = prune ? (long long)T : S;
    const int blocks = (int)((nt + 255) / 256 < 1184 ? (nt + 255) / 256 : 1184);
    adaptive_init_kernel<<<blocks, 256, 0, st>>>(lens_buf, B, Lp, done, lens_act, total, ind, pcnt);
    LG_LAUNCH_CHECK();
    LG_TRY(memset0(p.conf, p.msig_end));
    if (prune) LG_TRY(memset0(p.ind_b, p.rot_b_end));
  }
  // lgb200_linear with the operand conventions of the precision (x3: A / out / outp are split planes, resid and out32
  // the fp32 master; bf16: resid and out are the bf16 residual stream)
  auto linear = [&](int epi, const void* A0, const void* A1, int K0, const void* Wt, const float* bias, int N, int K,
                    const int32_t* ln, float s0, void* resid, void* out, void* out32, int n_rot, void* o0, void* o1,
                    void* o2, const float* gamma, const float* beta) {
    return lgb200_linear(prec, epi, A0, A1, K0, Wt, bias, T, N, K, ln, Lp, s0, 1.f, 1.f,
                         x3 ? (const float*)resid : f32, x3 ? nullptr : resid, x3 ? (float*)out32 : nullptr, out, rot,
                         rot16, n_rot, o0, o1, o2, gamma, beta, stream);
  };
  const int hprec = x3 ? LGB200_F32 : LGB200_BF16;  // the matchability head reads the fp32 master in x3 mode
  const int e_tail = E_PER_LAYER * L;
  const int e_ad = n_entries(cfg);  // adaptive heads of layer l at e_ad + 6 l

  // ---- staging: descriptors (+ input_proj) and positional encoding (lightglue.py:456-465) ----
  if (p.proj) {
    void* xin = ws + p.xin;
    float* xin32 = x3 ? (float*)xin : nullptr;
    void* xin16 = x3 ? nullptr : xin;
    LG_TRY(lgb200_pack_rows(desc0, B, m, din, 0, Lp, xin32, xin16, stream));
    LG_TRY(lgb200_pack_rows(desc1, B, n, din, 1, Lp, xin32, xin16, stream));
    if (x3) {
      void* xin_s = ws + p.xin_s;
      LG_TRY(lgb200_split_rows(xin32, (long long)T * din, xin_s, stream));
      LG_TRY(linear(LGB200_EPI_ROWMAJOR, xin_s, nullptr, din, W(e_tail + T_IN_W), F(e_tail + T_IN_B), 256, din,
                    nullptr, 1.f, nullptr, xs, x, 0, nullptr, nullptr, nullptr, nullptr, nullptr));
    } else {
      LG_TRY(linear(LGB200_EPI_ROWMAJOR, xin, nullptr, din, W(e_tail + T_IN_W), F(e_tail + T_IN_B), 256, din,
                    nullptr, 1.f, nullptr, x, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr));
    }
  } else {
    float* x32 = x3 ? (float*)x : nullptr;
    void* x16 = x3 ? nullptr : x;
    LG_TRY(lgb200_pack_rows(desc0, B, m, 256, 0, Lp, x32, x16, stream));
    LG_TRY(lgb200_pack_rows(desc1, B, n, 256, 1, Lp, x32, x16, stream));
    if (x3) LG_TRY(lgb200_split_rows(x32, (long long)T * 256, xs, stream));
  }
  LG_TRY(lgb200_posenc(kpts0, B, m, cfg->kdim, size0, F(e_tail + T_WR), lens, 0, Lp, rot, rot16, stream));
  LG_TRY(lgb200_posenc(kpts1, B, n, cfg->kdim, size1, F(e_tail + T_WR), lens, 1, Lp, rot, rot16, stream));

  // ---- transformer layers (lightglue.py:151-164, 193-222), out_proj / to_out folded into FFN1 ----
  const float q_scale = (float)(1.4426950408889634 / 8.0);  // log2(e) / sqrt(64)
  const float c_scale = (float)sqrt(1.4426950408889634 / 8.0);
  for (int i = 0; i < L; ++i) {
    const int e = E_PER_LAYER * i;
    void* xa = x3 ? xs : x;  // A operand of the projections
    LG_TRY(linear(LGB200_EPI_HEADS, xa, nullptr, 256, W(e + E_QKV_W), F(e + E_QKV_B), 768, 256, la, q_scale,
                  nullptr, nullptr, nullptr, 2, q, k, v, nullptr, nullptr));
    LG_TRY(lgb200_attention_ordered(prec, q, k, v, S, Lp, la, order_self, 0, ctx, stream));
    LG_TRY(linear(LGB200_EPI_LN_GELU, xa, ctx, 256, W(e + E_SF0_W), F(e + E_SF0_B), 512, 512, la, 1.f, nullptr,
                  hid, nullptr, 0, nullptr, nullptr, nullptr, F(e + E_SLN_G), F(e + E_SLN_B)));
    LG_TRY(linear(LGB200_EPI_ROWMAJOR, hid, nullptr, 512, W(e + E_SF3_W), F(e + E_SF3_B), 256, 512, la, 1.f, x,
                  x3 ? xs : x, x3 ? x : nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr));
    LG_TRY(linear(LGB200_EPI_HEADS, xa, nullptr, 256, W(e + E_CQV_W), F(e + E_CQV_B), 512, 256, la, c_scale,
                  nullptr, nullptr, nullptr, 0, q, v, nullptr, nullptr, nullptr));
    LG_TRY(lgb200_attention_ordered(prec, q, q, v, S, Lp, la, order_cross, 1, ctx, stream));
    LG_TRY(linear(LGB200_EPI_LN_GELU, xa, ctx, 256, W(e + E_CF0_W), F(e + E_CF0_B), 512, 512, la, 1.f, nullptr,
                  hid, nullptr, 0, nullptr, nullptr, nullptr, F(e + E_CLN_G), F(e + E_CLN_B)));
    LG_TRY(linear(LGB200_EPI_ROWMAJOR, hid, nullptr, 512, W(e + E_CF3_W), F(e + E_CF3_B), 256, 512, la, 1.f, x,
                  x3 ? xs : x, x3 ? x : nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr));
    if (!adaptive || i == L - 1) continue;
    // ---- adaptive depth (lightglue.py:501-505) and width (:506-521): every layer is launched, pairs that stopped
    // have lens_act == 0 and cost empty kernels ----
    const int ea = e_ad + A_PER_LAYER * i;
    const float thr = confidence_threshold(i, L);
    if (early) {
      LG_TRY(lgb200_rowdot(hprec, x, F(ea + A_TK_W), F(ea + A_TK_B), S, Lp, la, 1, conf, stream));
      LG_TRY(lgb200_exit_check(conf, B, Lp, lens_buf, total, thr, ad->depth_conf, i, done, lens_act, stream));
    }
    if (prune) {
      LG_TRY(lgb200_rowdot(hprec, x, F(ea + A_M_W), F(ea + A_M_B), S, Lp, la, 1, msig, stream));
      LG_TRY(lgb200_prune_compact(msig, early ? conf : nullptr, thr, ad->width_conf, S, Lp, lens_buf, lens_act,
                                  x3 ? (const float*)x : nullptr, x3 ? (float*)x_b : nullptr, x3 ? nullptr : x,
                                  x3 ? nullptr : x_b, rot, rot_b, rot16, rot16_b, ind, ind_b, pcnt, stream));
      void* tx = x; x = x_b; x_b = tx;
      if (x3) LG_TRY(lgb200_split_rows((const float*)x, (long long)T * 256, xs, stream));  // planes follow the master
      float* tr = rot; rot = rot_b; rot_b = tr;
      void* tr16 = rot16; rot16 = rot16_b; rot16_b = tr16;
      int32_t* ti = ind; ind = ind_b; ind_b = ti;
    }
  }

  // ---- MatchAssignment of the exit layer(s) (lightglue.py:523-524) and filter_matches (:525-536) ----
  // one group per exit layer e: final_proj, matchability and the normalisers of layer e on the sequences in lens_g
  auto group = [&](int e, const int32_t* lens_g) -> int {
    const int ea = e_ad + A_PER_LAYER * e;
    const bool last = e == L - 1;
    LG_TRY(linear(LGB200_EPI_ROWMAJOR, x3 ? xs : x, nullptr, 256, W(last ? e_tail + T_FP_W : ea + A_FP_W),
                  F(last ? e_tail + T_FP_B : ea + A_FP_B), 256, 256, lens_g, 0.25f, nullptr, md, nullptr, 0, nullptr,
                  nullptr, nullptr, nullptr, nullptr));
    LG_TRY(lgb200_rowdot(hprec, x, F(last ? e_tail + T_M_W : ea + A_M_W), F(last ? e_tail + T_M_B : ea + A_M_B), S,
                         Lp, lens_g, 0, z, stream));
    if (x3) {
      LG_TRY(lgb200_x3_similarity(md, B, Lp, lens_g, sim, stream));
      LG_TRY(lgb200_x3_assign_lse(sim, B, Lp, lens_g, m, n, lse, stream));
    } else {
      LG_TRY(lgb200_assign_lse(prec, md, S, Lp, lens_g, lse, stream));
    }
    return LGB200_OK;
  };
  if (!early) {
    LG_TRY(group(L - 1, lens));
  } else {
    int32_t* lens_g = reinterpret_cast<int32_t*>(ws + p.lens_g);
    exit_groups_kernel<<<(L * S + 255) / 256 < 148 ? (L * S + 255) / 256 : 148, 256, 0, st>>>(done, lens_buf, S, L,
                                                                                               lens_g);
    LG_LAUNCH_CHECK();
    for (int e = 0; e < L; ++e) LG_TRY(group(e, lens_g + (long long)e * S));
  }
  if (x3) {
    LG_TRY(lgb200_x3_assign_scores(sim, z, lse, B, Lp, lens, p.R, p.C, log_assignment, stream));
  } else {
    LG_TRY(lgb200_assign_scores(prec, md, z, lse, B, Lp, lens, p.R, p.C, log_assignment, fm_ws, stream));
  }
  LG_TRY(lgb200_filter_matches(log_assignment, B, p.R, p.C, lens, cfg->filter_threshold, ind,
                               ind ? ind + Lp : nullptr, 2 * Lp, m, n, matches0, matches1, scores0, scores1, fm_ws,
                               x3 ? 0 : 1, stream));

  // ---- ref_descriptors of the exit layer (lightglue.py:546-547) ----
  const int es = x3 ? 4 : 2;
  if (!adaptive) {  // rows < m / n of each sequence
    const size_t row = 256 * es;
    void* dst[2] = {desc_out0, desc_out1};
    const int cnt[2] = {m, n};
    for (int img = 0; img < 2; ++img) {
      if (!dst[img] || cnt[img] == 0) continue;
      const cudaError_t ce = cudaMemcpy2DAsync(dst[img], cnt[img] * row, (char*)x + img * Lp * row, 2 * Lp * row,
                                               cnt[img] * row, B, cudaMemcpyDeviceToDevice, st);
      if (ce != cudaSuccess) return (int)ce;
    }
  }
  // ---- lgb200_match_adaptive's further outputs (and, adaptive, the descriptors: rows < the pruned count) ----
  if (ad && ((adaptive && (desc_out0 || desc_out1)) || ad->prune0 || ad->prune1 || ad->exit_layer ||
             ad->final_counts)) {
    const long long threads = 32LL * B * (m + n);
    const int blocks = (int)((threads + 255) / 256 < 4096 ? (threads + 255) / 256 : 4096);
    adaptive_outputs_kernel<<<blocks < 1 ? 1 : blocks, 256, 0, st>>>(
        B, m, n, L, Lp, lens, done, pcnt, adaptive ? x : nullptr, es, desc_out0, desc_out1, ad->prune0, ad->prune1,
        ad->exit_layer, ad->final_counts);
    LG_LAUNCH_CHECK();
  }
  return LGB200_OK;
}

}  // namespace

extern "C" int lgb200_match(const lgb200_match_config* cfg, const void* const* table, int B, int m, int n,
                            const float* kpts0, const float* kpts1, const float* desc0, const float* desc1,
                            const float* size0, const float* size1, const int32_t* counts0, const int32_t* counts1,
                            int64_t* matches0, int64_t* matches1, float* scores0, float* scores1,
                            float* log_assignment, void* desc_out0, void* desc_out1, void* workspace,
                            long long workspace_bytes, void* stream) {
  if (!cfg || !table || !kpts0 || !kpts1 || !desc0 || !desc1 || !matches0 || !matches1 || !scores0 || !scores1 ||
      !log_assignment || !workspace)
    return LGB200_ERR_NULL;
  Plan p;
  LG_TRY(make_plan(cfg, B, m, n, counts0 || counts1, false, &p));
  if (workspace_bytes < p.total || reinterpret_cast<uintptr_t>(workspace) % 256) return LGB200_ERR_SHAPE;
  const int ne = n_entries(cfg);
  for (int e = 0; e < ne; ++e)
    if (!table[e]) return LGB200_ERR_NULL;
  return forward(cfg, p, nullptr, table, B, m, n, kpts0, kpts1, desc0, desc1, size0, size1, counts0, counts1,
                 matches0, matches1, scores0, scores1, log_assignment, desc_out0, desc_out1, workspace, stream);
}

extern "C" int lgb200_match_adaptive(const lgb200_match_config* cfg, const lgb200_adaptive_config* acfg,
                                     const void* const* table, int B, int m, int n, const float* kpts0,
                                     const float* kpts1, const float* desc0, const float* desc1, const float* size0,
                                     const float* size1, const int32_t* counts0, const int32_t* counts1,
                                     int64_t* matches0, int64_t* matches1, float* scores0, float* scores1,
                                     float* log_assignment, void* desc_out0, void* desc_out1, int32_t* prune0,
                                     int32_t* prune1, int32_t* exit_layer, int32_t* final_counts, void* workspace,
                                     long long workspace_bytes, void* stream) {
  if (!cfg || !acfg || !table || !kpts0 || !kpts1 || !desc0 || !desc1 || !matches0 || !matches1 || !scores0 ||
      !scores1 || !log_assignment || !workspace)
    return LGB200_ERR_NULL;
  Plan p;
  LG_TRY(make_plan(cfg, B, m, n, counts0 || counts1, true, &p));
  if (workspace_bytes < p.total || reinterpret_cast<uintptr_t>(workspace) % 256) return LGB200_ERR_SHAPE;
  const Adaptive ad{acfg->depth_confidence > 0.f, acfg->width_confidence > 0.f, acfg->depth_confidence,
                    acfg->width_confidence, prune0, prune1, exit_layer, final_counts};
  if (ad.width && p.Lp > 8192) return LGB200_ERR_SHAPE;  // lgb200_prune_compact's limit
  const int ne = ad.depth || ad.width ? n_adaptive_entries(cfg) : n_entries(cfg);
  for (int e = 0; e < ne; ++e)
    if (!table[e]) return LGB200_ERR_NULL;
  return forward(cfg, p, &ad, table, B, m, n, kpts0, kpts1, desc0, desc1, size0, size1, counts0, counts1, matches0,
                 matches1, scores0, scores1, log_assignment, desc_out0, desc_out1, workspace, stream);
}
