// kernels.h -- host-side launchers of the hand-written sm_100a kernels.
// Activation tensors are NHWC ("[N, P=H*W, C]"), element type fp32 or bf16 (`bf16` flag).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dp {

constexpr int GN_GROUPS = 32;
constexpr int GN_MAX_SPLITS = 16;
// GroupNorm scratch (`partial`): N * GN_WS_FLOATS_PER_SAMPLE + GN_WS_FLOATS_EXTRA floats: the two-pass kernels' split
// partials, and the statistics-only kernel's per-tile partials (it runs while tiles * 64 fits GN_WS_FLOATS_PER_SAMPLE)
constexpr int GN_WS_FLOATS_PER_SAMPLE = 8192;
constexpr int GN_WS_FLOATS_EXTRA = 4096;

// ---- classifier-side kernels (kernels_net.cu) --------------------------------------
// timm StdConv2d standardisation of OIHW fp32 weights -> KRSC (NHWC filter), channel-padded.
void launch_weight_standardize(const float* w_oihw, void* w_krsc, int O, int I, int kh, int kw, int Ipad,
                               bool bf16, bool standardize, cudaStream_t st);
// z [N,3,H,W] fp32 -> [N,H,W,Cp] T (pad channels zero) and back (first 3 channels).
void launch_pack_nchw(const float* z, void* out, int N, int H, int W, int Cp, bool bf16, cudaStream_t st);
void launch_unpack_nhwc(const void* in, float* dz, int N, int H, int W, int Cp, bool bf16, cudaStream_t st);

int gn_splits(int P, int C, bool bf16);
// GroupNorm(32)+ReLU forward: stats partials -> apply.  `stats` [N][32][2] receives (mean, rstd).
void launch_gn_relu_forward(const void* x, void* y, const float* gamma, const float* beta, float* partial,
                            float* stats, int N, int P, int C, bool bf16, cudaStream_t st);
// statistics only (head): fills `stats`.
void launch_gn_stats(const void* x, float* partial, float* stats, int N, int P, int C, bool bf16, cudaStream_t st);
// backward of GroupNorm+ReLU wrt its input: dx = GNbwd(dy * relu'(.)) (+ addend).
// gamma_pos: the caller knows every gamma[c] > 0 (checked once at weight load) -> bf16 may use the packed ReLU gate.
void launch_gn_relu_backward(const void* dy, const void* x, const void* addend, void* dx, const float* gamma,
                             const float* beta, const float* stats, float* partial, int N, int P, int C, bool bf16,
                             cudaStream_t st, bool gamma_pos = false);
// profiling aid (tools/gnbench.cu): device buffer [CTAs][8] that receives clock64 stamps at the v2 forward kernel's phase boundaries
void gn2_set_trace(unsigned long long* dev_ptr);
// ConstantPad2d(1,0)+MaxPool(3,2): x [N,Hs,Ws,C] -> y [N,Hs/2,Ws/2,C]; argmax (int8, 0..8) optional.
void launch_maxpool_forward(const void* x, void* y, int8_t* amax, int N, int Hs, int Ws, int C, bool bf16,
                            cudaStream_t st);
void launch_maxpool_backward(const void* dy, const int8_t* amax, void* dx, int N, int Hs, int Ws, int C, bool bf16,
                             cudaStream_t st);
// head: pooled[n][c] = mean_p relu(gn(x))  (the fc layer itself runs through cublasLt in the engine)
void launch_head_pool(const void* x, const float* gamma, const float* beta, const float* stats, float* pooled,
                      int N, int P, int C, bool bf16, cudaStream_t st);
// dy[n,p,c] = dpooled[n][c] / P
void launch_pool_grad_bcast(const float* dpooled, void* dy, int N, int P, int C, bool bf16, cudaStream_t st);
// strided spatial subsample [N,H,W,C] -> [N,H/2,W/2,C] (rows/cols 0,2,4,..) and its scatter-add adjoint
void launch_subsample2(const void* x, void* y, int N, int H, int W, int C, bool bf16, cudaStream_t st);
void launch_subsample2_adjoint_add(const void* dy, void* dx, int N, int H, int W, int C, bool bf16, cudaStream_t st);

// ---- hand-written bf16 tensor-core stem convolution on the tight C=3 input (kernels_stem.cu)
void launch_stem_pack(const void* w_krsc, void* w_kn, int cin_pad, cudaStream_t st);
void launch_stem_forward(const void* in, const void* w_kn, void* out, int N, int H, int W, cudaStream_t st);
// stem dgrad fused with the masked EOT reduce: G[b] (+)= 2 * sum_s keep_s * dX_s, dX never materialised
void launch_stem_bwd_reduce(const void* dY, const void* w_krsc, int cin_pad, const int16_t* rects, float* G, int B, int S,
                            int n0, int n, int H, int W, cudaStream_t st);

// same, additionally fusing the pad+max-pool backward (reads d_pool + the saved argmax; d_stem never hits HBM)
void launch_stem_bwd_pool_reduce(const void* dpool, const int8_t* amax, const void* w_krsc, int cin_pad, const int16_t* rects,
                                 float* G, int B, int S, int n0, int n, int H, int W, cudaStream_t st);

// ---- opt-in: GroupNorm+ReLU applied in the prologue of a tcgen05 1x1-convolution GEMM (kernels_gemm.cu, bf16)
// out[m,n] = sum_k relu(gn(x))[m,k] * W[n,k] (+ shortcut[m,n]); `stats` from launch_gn_stats on x.
bool gn_gemm_supported(int P, int K, int Nout);
void launch_gn_gemm_pack(const void* w_nk, void* w_packed, int Nout, int K, cudaStream_t st);
bool launch_gn_gemm_forward(const void* x, const void* w_packed, const float* stats, const float* gamma, const float* beta,
                            const void* shortcut, void* out, int N, int P, int K, int Nout, cudaStream_t st);

// ---- patch-side kernels (kernels_patch.cu) -------------------------------------------
// utils.clip + add: adv_x = x + min(eps/||m(p-x)||,1) * m(p-x); l2[b], scale[b] dev outputs.
void launch_paste(const float* x, const float* mask, const float* pattern, float* adv_x, float* l2, float* scale,
                  int B, int H, int W, float eps, cudaStream_t st);
// K1: EOT expansion (paste + normalise + occlude) -> [N,H,W,Cp] T.
// fused==true: reads x/mask/pattern/scale (img ignored); else reads img [B,3,H,W].
// rects [B*S][4][4] int16 dev or nullptr; samples [n0, n0+n) of the b-major ordering are
// written to out + (n - n0) * H*W*Cp.
void set_expand_tuning(int rows, int sg, int mode);
void get_expand_last(int* out4);   // tile rows, sample groups, grid, resident CTAs/SM of the last K1 launch   // K1 launch-shape / store-path overrides (0 = heuristic / default); sweeps only
void launch_expand(const float* img, const float* x, const float* mask, const float* pattern, const float* scale,
                   const int16_t* rects, void* out, int B, int S, int n0, int n, int H, int W, int Cp, bool bf16,
                   bool fused, int num_sms, cudaStream_t st);
// optional affine / colour EOT (gather) and its adjoint (atomic scatter into a zeroed G); xf [N][8] dev
void launch_expand_affine(const float* adv, const float* xf, const int16_t* rects, void* out, int S, int n0, int n,
                          int H, int W, int Cp, bool bf16, cudaStream_t st);
void launch_reduce_affine(const void* dz, const float* adv, const float* xf, const int16_t* rects, float* G, int S, int n0,
                          int n, int H, int W, int Cp, bool bf16, cudaStream_t st);
// K4: CW loss, argmax, dlogits (scaled by inv_s_total).  y/targeted are per-sample dev arrays.
void launch_cw(const float* logits, const int32_t* y, const uint8_t* targeted, float confidence, float inv_s_total,
               float* loss, int32_t* preds, float* dlogits, int N, int K, cudaStream_t st);
void launch_argmax(const float* logits, int32_t* preds, int N, int K, cudaStream_t st);
// K1^T: G[b] (+)= 2 * sum_s keep_s * dz[b,s]  for samples [n0,n0+n).
void launch_reduce(const void* dz, const int16_t* rects, float* G, int B, int S, int n0, int n, int H, int W,
                   int Cp, bool bf16, cudaStream_t st);
// structural loss value [B] + gradient field dLs [B,3,H,W]  (attack.py:33-45,227-228)
void launch_struct(const float* adv_x, const float* x, float* loss_struc, float* dLs, int B, int H, int W,
                   cudaStream_t st);
// density / group-lasso values + per-group statistics for their gradients (attack.py:72-80,235-245)
void launch_maskreg(const float* mask, float* loss_density, float* group_lasso, float* win_dev, float* grp_ss,
                    int B, int H, int W, int unit, cudaStream_t st);
// K3: chain rule + sign step + clip (attack.py:332-342)
void launch_update(const float* x, float* mask, float* pattern, const float* G, const float* dLs,
                   const float* scale, const float* win_dev, const float* grp_ss, const float* lr,
                   const float* structured, const float* coeff_gl, float density, float lo, float hi, int stage,
                   float* gp_out, float* gm_out, const float* gp_bias, int B, int H, int W, int unit, cudaStream_t st);
// failed-mask bitmap update of one step (attack.py:259-267) + popcount per image
void launch_failed_update(uint32_t* bits, int words, const int32_t* idx, const float* loss, const int32_t* nff, const uint8_t* active,
                          int B, int S, float thresh, int32_t* count, cudaStream_t st);
// k x k window sums of [B,1,H,W] (optionally of the squares)
void launch_window_sum(const float* t, float* out, int B, int H, int W, int k, bool square, cudaStream_t st);

}  // namespace dp
