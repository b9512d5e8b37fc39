// Kernel selection for every attention entry point (attention.cuh).  The rule lives here and
// nowhere else; the kernels and their launchers are in the other attention_*.cu files.
//
// "dropping": drop != nullptr && drop->thresh != 0.  "impl": vitk_attention_set_impl.
//
// packed fwd   hd != 64, with lse or dropping or hd not in {32, 96, 128}:
//                impl != 1 and xmma fits -> attn_xmma_fwd_kernel, else attn_gen_fwd_kernel
//              hd in {32, 96, 128}, no lse, not dropping -> attn_x_kernel
//              hd 64, dropping: N <= 208 on sm_100 -> attn_fwd_tc2_kernel<true>, else attn_gen_fwd
//              hd 64, impl 0: on sm_100 with N <= 640, tc2 up to 208 tokens, attn_fwd_tc_kernel up
//                to 256, attn_fwd_tc3_kernel above; otherwise attn_fwd_hd64_kernel
//              hd 64, impl 1: hd64.  2: tc2 / tc / tc3 by N as for impl 0, without the device
//                check.  3: tc up to 256 tokens, tc3 above.  4: tc3
// packed bwd   hd 64, N <= 256, sm_100, and impl != 1 or dropping: attn_bwd_tc2_kernel where its
//                shared memory fits, else attn_bwd_tc_kernel
//              else hd != 64 or N > 256 or dropping: impl != 1 and xmma fits ->
//                attn_xmma_bwd_kernel + colsum_bf16 (dbias), else attn_gen_bwd_kernel
//              else attn_bwd_hd64_kernel + colsum_bf16 (dbias)
// "ragged": hd not in {32, 64, 96, 128} and attention_src_supported(Nq, Nk, hd) (16 <= hd <= 128,
// Nq <= 128, Nk <= 256): the shapes only the xr kernels (attention_xr.cu, attention_xr_bwd.cu) take.
// src fwd      no lse: impl != 1 and xtc applies -> attn_xtc_kernel; ragged -> attn_xr_fwd_kernel
//                (any impl); else attn_x_kernel
//              lse: impl != 1, not dropping and xtc applies -> xtc; ragged, unless impl 1 and hd
//                is a multiple of 8 -> xr; else impl != 1 and xmma fits -> attn_xmma_fwd_kernel;
//                else attn_xgen_fwd_kernel
// src bwd      ragged, unless impl 1 and hd is a multiple of 8 -> attn_xr_bwd_kernel; else
//                impl != 1 and xmma fits -> attn_xmma_bwd_kernel, else attn_xgen_bwd_kernel
#include "attention_kernels.cuh"
#include "common.h"
#include "train_ops.cuh"

namespace vitk {

namespace {

// Values of vitk_attention_set_impl (tests and A/B timing).
enum AttnImpl : int {
  kImplAuto = 0,
  kImplNoTcgen05 = 1,      // the mma.sync / CUDA-core kernels wherever a choice exists
  kImplTcgen05 = 2,        // head_dim 64 forward: the tcgen05 kernels, chosen by N
  kImplTcUnpipelined = 3,  // ... without the item-pipelined one (attention_tc2.cu)
  kImplTcKeyBlock = 4,     // ... the key-block one (attention_tc3.cu) for every N
};
AttnImpl g_attn_impl = kImplAuto;

bool dropping(const DropParams* drop) { return drop != nullptr && drop->thresh != 0u; }

bool ragged(int Nq, int Nk, int hd) {
  return !(hd == 32 || hd == 64 || hd == 96 || hd == 128) && attention_src_supported(Nq, Nk, hd);
}

// impl 1 keeps the CUDA-core training kernels wherever they take the head_dim
bool xr_for_training(int Nq, int Nk, int hd) {
  return ragged(Nq, Nk, hd) && !(g_attn_impl == kImplNoTcgen05 && hd % 8 == 0);
}

}  // namespace

void attention_force_impl(int impl) { g_attn_impl = static_cast<AttnImpl>(impl); }

// head_dim 64 up to 256 tokens: the tcgen05 backward kernels; every other shape (train.py's own
// Config has head_dim 16; a 384 px fine-tune 577 tokens): the CUDA-core kernels, as far as one
// head's operands fit in shared memory.
bool attention_trainable(int N, int hd) {
  return (hd == 64 && N <= 256) || attention_gen_fits(N, hd);
}

int attention_fwd(const void* qkv, void* ctx, float* lse, int B, int N, int H, int hd,
                  cudaStream_t stream, const DropParams* drop) {
  VITK_REQUIRE(qkv && ctx, "attention: null operand");
  if (hd != 64) {
    const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(qkv);
    const int D = H * hd;
    const long long img = static_cast<long long>(N) * 3 * D;
    if (lse == nullptr && !dropping(drop) && (hd == 32 || hd == 96 || hd == 128))
      return attention_x(p, img, 3 * D, p + D, p + 2 * D, img, 3 * D, ctx,
                         static_cast<long long>(N) * D, D, B, N, N, H, hd, stream);
    if (g_attn_impl != kImplNoTcgen05 && attention_xmma_fits(N, N, hd)) {
      const AttnXSrc src{p, img, 3 * D, p + D, p + 2 * D, img, 3 * D};
      return attention_xmma_fwd(src, ctx, static_cast<long long>(N) * D, D, lse, B, N, N, H, hd,
                                stream, drop);
    }
    return attention_gen_fwd(qkv, ctx, lse, B, N, H, hd, stream, drop);
  }
  if (dropping(drop)) {
    // the pipelined tcgen05 kernel regenerates the masks in its softmax warps up to 208 tokens
    if (N <= 208 && device_cc() >= 100)
      return attention_fwd_tc2(qkv, ctx, lse, B, N, H, hd, stream, drop);
    return attention_gen_fwd(qkv, ctx, lse, B, N, H, hd, stream, drop);
  }
  const AttnImpl impl = g_attn_impl;
  if (impl == kImplNoTcgen05 || (impl == kImplAuto && (N > 640 || device_cc() < 100)))
    return attention_fwd_hd64(qkv, ctx, lse, B, N, H, hd, stream);
  if (impl == kImplTcKeyBlock) return attention_fwd_tc3(qkv, ctx, lse, B, N, H, hd, stream);
  if (impl != kImplTcUnpipelined && N <= 208)
    return attention_fwd_tc2(qkv, ctx, lse, B, N, H, hd, stream);
  if (N <= 256) return attention_fwd_tc(qkv, ctx, lse, B, N, H, hd, stream);
  return attention_fwd_tc3(qkv, ctx, lse, B, N, H, hd, stream);
}

int attention_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse, void* dqkv,
                  int B, int N, int H, int hd, cudaStream_t stream, const DropParams* drop,
                  float* dbias) {
  VITK_REQUIRE(qkv && ctx && dctx && lse && dqkv, "attention_bwd: null operand");
  const bool tcgen05 = g_attn_impl != kImplNoTcgen05;
  if ((tcgen05 || dropping(drop)) && hd == 64 && N <= 256 && device_cc() >= 100) {
    if (attention_bwd_tc2_fits(N, H, dbias != nullptr))
      return attention_bwd_tc2(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream, drop, dbias);
    return attention_bwd_tc(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream, drop, dbias);
  }
  const int D = H * hd;
  if (hd != 64 || N > 256 || dropping(drop)) {
    if (!tcgen05 || !attention_xmma_fits(N, N, hd))
      return attention_gen_bwd(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream, drop, dbias);
    // q, k, v are column blocks of the packed activation
    const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(qkv);
    __nv_bfloat16* dp = static_cast<__nv_bfloat16*>(dqkv);
    const long long img = static_cast<long long>(N) * 3 * D, cimg = static_cast<long long>(N) * D;
    const AttnXSrc src{p, img, 3 * D, p + D, p + 2 * D, img, 3 * D};
    VITK_TRY(attention_xmma_bwd(src, ctx, dctx, cimg, D, lse, dp, img, 3 * D, dp + D, dp + 2 * D,
                                img, 3 * D, B, N, N, H, hd, stream, drop));
  } else {
    VITK_TRY(attention_bwd_hd64(qkv, ctx, dctx, lse, dqkv, B, N, H, hd, stream));
  }
  // neither kernel accumulates the bias gradient itself
  if (dbias != nullptr) return colsum_bf16(dqkv, 3ll * D, B * N, 3 * D, dbias, stream);
  return VITK_OK;
}

int attention_src_fwd(const AttnXSrc& s, void* ctx, long long ctx_img, int ldc, float* lse, int B,
                      int Nq, int Nk, int H, int hd, cudaStream_t stream, const DropParams* drop) {
  const bool tcgen05 = g_attn_impl != kImplNoTcgen05;
  if (lse == nullptr) {
    if (tcgen05 && attention_xtc_applicable(s.q_img, s.kv_img, B, Nq, Nk, hd))
      return attention_xtc(s.q, s.q_img, s.ldq, s.k, s.v, s.kv_img, s.ldkv, ctx, ctx_img, ldc, B,
                           Nq, Nk, H, hd, stream);
    if (ragged(Nq, Nk, hd))
      return attention_xr_fwd(s, ctx, ctx_img, ldc, nullptr, B, Nq, Nk, H, hd, stream);
    return attention_x(s.q, s.q_img, s.ldq, s.k, s.v, s.kv_img, s.ldkv, ctx, ctx_img, ldc, B, Nq,
                       Nk, H, hd, stream);
  }
  if (tcgen05 && !dropping(drop) && attention_xtc_applicable(s.q_img, s.kv_img, B, Nq, Nk, hd))
    return attention_xtc(s.q, s.q_img, s.ldq, s.k, s.v, s.kv_img, s.ldkv, ctx, ctx_img, ldc, B, Nq,
                         Nk, H, hd, stream, lse);
  if (xr_for_training(Nq, Nk, hd))
    return attention_xr_fwd(s, ctx, ctx_img, ldc, lse, B, Nq, Nk, H, hd, stream, drop);
  if (tcgen05 && attention_xmma_fits(Nq, Nk, hd))
    return attention_xmma_fwd(s, ctx, ctx_img, ldc, lse, B, Nq, Nk, H, hd, stream, drop);
  return attention_xgen_fwd(s, ctx, ctx_img, ldc, lse, B, Nq, Nk, H, hd, stream, drop);
}

int attention_src_bwd(const AttnXSrc& s, const void* ctx, const void* dctx, long long ctx_img,
                      int ldc, const float* lse, void* dq, long long dq_img, int lddq, void* dk,
                      void* dv, long long dkv_img, int lddkv, int B, int Nq, int Nk, int H, int hd,
                      cudaStream_t stream, const DropParams* drop) {
  if (xr_for_training(Nq, Nk, hd))
    return attention_xr_bwd(s, ctx, dctx, ctx_img, ldc, lse, dq, dq_img, lddq, dk, dv, dkv_img,
                            lddkv, B, Nq, Nk, H, hd, stream, drop);
  if (g_attn_impl != kImplNoTcgen05 && attention_xmma_fits(Nq, Nk, hd))
    return attention_xmma_bwd(s, ctx, dctx, ctx_img, ldc, lse, dq, dq_img, lddq, dk, dv, dkv_img,
                              lddkv, B, Nq, Nk, H, hd, stream, drop);
  return attention_xgen_bwd(s, ctx, dctx, ctx_img, ldc, lse, dq, dq_img, lddq, dk, dv, dkv_img,
                            lddkv, B, Nq, Nk, H, hd, stream, drop);
}

}  // namespace vitk
