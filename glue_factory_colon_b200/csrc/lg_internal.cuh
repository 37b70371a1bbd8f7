// Internal (non-ABI) entry points shared between translation units.
#pragma once
#include "lg_common.cuh"

// fp32 CUDA-core path (lg_simt.cu)
int lg_simt_linear(int epilogue, const float* A0, const float* A1, int K0, const float* W, int T, int N,
                   int K, const int32_t* lens, LgEpi epi, cudaStream_t st);
int lg_simt_attention(const float* Q, const float* K, const float* V, int S, int Lp, const int32_t* lens,
                      int kv_xor, float* ctx, cudaStream_t st);
int lg_simt_assign_lse(const float* md, int S, int Lp, const int32_t* lens, float* lse, cudaStream_t st);
int lg_simt_assign_scores(const float* md, const float* z, const float* lse, int B, int Lp,
                          const int32_t* lens, int R, int C, float* scores, float* sim_out, cudaStream_t st);

// bf16 tcgen05 path (lg_tc_*.cu)
int lg_tc_linear(int epilogue, const __nv_bfloat16* A0, const __nv_bfloat16* A1, int K0,
                 const __nv_bfloat16* W, int T, int N, int K, const int32_t* lens, LgEpi epi,
                 cudaStream_t st);
int lg_tc_linear_v2(int epilogue, const __nv_bfloat16* A0, const __nv_bfloat16* A1, int K0,
                    const __nv_bfloat16* W, int T, int N, int K, const int32_t* lens, LgEpi epi,
                    const void* rot16, const __nv_bfloat16* resid16, cudaStream_t st);
int lg_tc_attention(const __nv_bfloat16* Q, const __nv_bfloat16* K, const __nv_bfloat16* V, int S, int Lp,
                    const int32_t* lens, int kv_xor, __nv_bfloat16* ctx, const int32_t* order, cudaStream_t st);
int lg_tc_attention2(const __nv_bfloat16* Q, const __nv_bfloat16* K, const __nv_bfloat16* V, int S, int Lp,
                     const int32_t* lens, int kv_xor, __nv_bfloat16* ctx, cudaStream_t st);
int lg_tc_assign_lse(const __nv_bfloat16* md, int S, int Lp, const int32_t* lens, float* lse,
                     cudaStream_t st);
int lg_tc_assign_scores(const __nv_bfloat16* md, const float* z, const float* lse, int B, int Lp,
                        const int32_t* lens, int R, int C, float* scores, void* best_ws, cudaStream_t st);
int lg_tc_assign_loss(const __nv_bfloat16* md, const float* z, const float* lse, int B, int Lp, const int32_t* lens,
                      int R, int C, const uint8_t* gt, float* row_pos, float* row_cnt, float* row_exp,
                      int32_t* row_arg, int32_t* col_arg, void* best_ws, cudaStream_t st);

// fp32-accurate tensor-core path: split-fp16 operands, three MMAs per product (lg_x3.cu, lg_x3_attn.cu)
int lg_x3_linear(int epilogue, const void* A0, const void* A1, int K0, const void* W, int T, int N, int K,
                 const int32_t* lens, LgEpi epi, void* outs, cudaStream_t st);
int lg_x3_attention(const void* Q, const void* K, const void* V, int S, int Lp, const int32_t* lens, int kv_xor,
                    void* ctx, cudaStream_t st);
// attention backward on tcgen05, split-fp16 operands (lg_x3_attn_bwd.cu)
size_t lg_x3_attention_bwd_ws_floats(int S, int Lp);
int lg_x3_attention_bwd(const float* Q, const float* K, const float* V, const float* ctx, const float* dctx, int S,
                        int Lp, const int32_t* lens, int kv_xor, float* dQ, float* dK, float* dV, float* ws,
                        cudaStream_t st);
// the same kernel template on bf16 operands: backward of the bf16 forward (lg_x3_attn_bwd.cu)
size_t lg_bf16_attention_bwd_ws_floats(int S, int Lp);
int lg_bf16_attention_bwd(const __nv_bfloat16* Q, const __nv_bfloat16* K, const __nv_bfloat16* V,
                          const __nv_bfloat16* ctx, const float* dctx, int S, int Lp, const int32_t* lens, int kv_xor,
                          float* dQ, float* dK, float* dV, float* ws, cudaStream_t st);
// x3 plane scaling: a plane pair stores x * 2^e so that the LOW plane stays a normal fp16 number (fp16 normals end at
// 6.1e-5 and lo ~ 2^-11 |x|: unscaled, the low planes of all weights and of every activation below 0.12 are subnormal
// (or flushed) and the pair carries ~12 bits instead of 22).  Powers of two: exact, undone in the consuming epilogue.
#define LG_X3_EA 64.0f    /* activations, q / k / v, md: |x| < 1023, low plane normal for |x| > 2e-3 */
#define LG_X3_EW 256.0f   /* weights (host side, lightglue.py:_pack) */
#define LG_X3_EP 256.0f   /* attention probabilities (<= 16 with the lazy maximum threshold of 4) */
