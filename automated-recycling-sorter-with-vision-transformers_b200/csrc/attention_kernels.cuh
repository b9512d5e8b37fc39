// Per-kernel launchers and fit predicates of the attention kernels.  Only the attention sources
// include this header: everything else goes through attention.cuh, so that the choice between
// these kernels is made in attention.cu alone.  Each launcher checks the shapes its kernel takes.
#pragma once
#include <cuda_bf16.h>

#include "attention.cuh"

namespace vitk {

// ---- packed qkv, head_dim 64 (attention_fwd's operand layout)
// mma.sync flash kernels, whole head in shared memory (attention_flash.cu).
int attention_fwd_hd64(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                       cudaStream_t stream);
int attention_bwd_hd64(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                       void* dqkv, int B, int N, int H, int hd, cudaStream_t stream);
// tcgen05 forwards: one key block, N <= 256 (attention_tc.cu); item-pipelined, N <= 208, with
// dropout (attention_tc2.cu); key blocks with a lazily moved softmax reference, N <= 640
// (attention_tc3.cu).
int attention_fwd_tc(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                     cudaStream_t stream);
int attention_fwd_tc2(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                      cudaStream_t stream, const DropParams* drop = nullptr);
int attention_fwd_tc3(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                      cudaStream_t stream);
// tcgen05 backwards, N <= 256 (attention_bwd_tc.cu), and its software-pipelined form
// (attention_bwd_tc2.cu: 64-query sub-blocks, score tiles double-buffered in TMEM) wherever its
// larger shared-memory footprint fits.  Both accumulate dbias themselves.
struct BwdParams {
  int B, N, H, Nk;
  float scale;
  const __nv_bfloat16* ctx;
  const __nv_bfloat16* dctx;
  const float* lse;
  DropParams drop;  // attention-probability dropout of the forward (same index space / key)
  float* dbias;     // optional [3 D]: += column sums of d_qkv (the qkv bias gradient)
};
int attention_bwd_tc(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                     void* dqkv, int B, int N, int H, int hd, cudaStream_t stream,
                     const DropParams* drop, float* dbias);
bool attention_bwd_tc2_fits(int N, int H, bool with_dbias);
int attention_bwd_tc2(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                      void* dqkv, int B, int N, int H, int hd, cudaStream_t stream,
                      const DropParams* drop, float* dbias);
// CUDA-core kernels for the shapes the tensor-core kernels do not cover (attention_gen.cu):
// head_dim 8 .. 128 in steps of 8, up to 1024 tokens, optional log-sum-exp and dropout.
bool attention_gen_fits(int N, int hd);
int attention_gen_fwd(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                      cudaStream_t stream, const DropParams* drop = nullptr);
int attention_gen_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                      void* dqkv, int B, int N, int H, int hd, cudaStream_t stream,
                      const DropParams* drop, float* dbias);

// ---- separate sources (AttnXSrc); output rows at ctx + b*ctx_img + r*ldc + h*hd
// mma.sync inference kernel, head_dim 32 / 64 / 96 / 128, no log-sum-exp (attention_x.cu).
int attention_x(const void* q, long long q_img, int ldq, const void* k, const void* v,
                long long kv_img, int ldkv, void* ctx, long long ctx_img, int ldc, int B, int Nq,
                int Nk, int H, int hd, cudaStream_t stream);
// tcgen05 kernel for one query tile and one key block (<= 128 queries, <= 256 keys)
// (attention_xtc.cu).
bool attention_xtc_applicable(long long q_img, long long kv_img, int B, int Nq, int Nk, int hd);
int attention_xtc(const void* q, long long q_img, int ldq, const void* k, const void* v,
                  long long kv_img, int ldkv, void* ctx, long long ctx_img, int ldc, int B, int Nq,
                  int Nk, int H, int hd, cudaStream_t stream, float* lse = nullptr);
// mma.sync training forward and backward, head_dim 16 .. 128 in steps of 16, queries and keys of
// one head within shared memory (attention_xmma.cu).
bool attention_xmma_fits(int Nq, int Nk, int hd);
int attention_xmma_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                       int Nq, int Nk, int H, int hd, cudaStream_t stream,
                       const DropParams* drop = nullptr);
int attention_xmma_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                       int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                       void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                       cudaStream_t stream, const DropParams* drop = nullptr);
// CUDA-core training forward and backward, head_dim 8 .. 128 in steps of 8, up to 1024 queries /
// keys (attention_gen.cu).
int attention_xgen_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                       int Nq, int Nk, int H, int hd, cudaStream_t stream,
                       const DropParams* drop = nullptr);
int attention_xgen_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                       int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                       void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                       cudaStream_t stream, const DropParams* drop = nullptr);

}  // namespace vitk
