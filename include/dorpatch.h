/* dorpatch.h -- C ABI of libdorpatch.so, the B200-native DorPatch hot-path engine.
 *
 * Plain C: opaque handle, raw pointers, sizes, int error codes.  No torch types.
 * "dev" pointers are CUDA device pointers on the engine's device, "host" pointers
 * are ordinary host memory.  `stream` is a cudaStream_t passed as void* (PyTorch's
 * current stream when driven from Python); all device work of a call is issued on
 * it.  Calls that return host results synchronise that stream before returning.
 * One engine per GPU; an engine is not thread-safe.
 *
 * Every entry point returns 0 on success, non-zero on failure; dp_last_error()
 * then holds a human-readable message (the Python host raises RuntimeError with it).
 *
 * Reference interfaces replaced (CGCL-codes/DorPatch @ 0751fd4, /root/reference):
 *   dp_paste            utils.py:105-110 `clip` + attack.py:185 (adv_x = x + delta)
 *   dp_expand           attack.py:204-220 (mask gather + occlude [+dual]) and
 *                       utils.py:77-78 NormModel's (x-0.5)/0.5, fused       [K1]
 *   dp_predict          `model(adv_x_masked)` forward (attack.py:222,397;
 *                       defenses/PatchCleanser.py:72,86,109; main.py:91,156)  [K1+K2]
 *   dp_attack_grad      attack.py:184-247: paste, EOT expansion, classifier
 *                       fwd + backward-to-input, CW loss (attack.py:16-23),
 *                       structural / density / group-lasso terms (:227-245),
 *                       masked EOT gradient reduce                [K1,K2,K4,K1^T]
 *   dp_attack_update    attack.py:332-342 sign step + clip (+ chain rule through
 *                       utils.clip and the regulariser gradients)            [K3]
 *   dp_window_sum       the all-ones Conv2d of attack.py:72-80,365-368
 *   dp_engine_load_weights   utils.py:57-62 (timm state_dict) + timm StdConv2d
 *                       weight standardisation, folded once
 */
#ifndef DORPATCH_H_
#define DORPATCH_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DP_ABI_VERSION 7

enum dp_precision {
  DP_PREC_FP32 = 0, /* fp32 storage, fp32 FMA math (no tensor cores): parity checks   */
  DP_PREC_TF32 = 1, /* fp32 storage, TF32 tensor-core math (the reference's GPU default) */
  DP_PREC_BF16 = 2  /* bf16 storage between layers, fp32 accumulate / statistics        */
};

typedef struct dp_engine dp_engine;

typedef struct dp_config {
  int32_t device;        /* CUDA device ordinal                                   */
  int32_t img;           /* H == W of the images (multiple of 56; 224 for ImageNet) */
  int32_t n_classes;     /* classifier outputs (1000)                              */
  int32_t precision;     /* enum dp_precision                                      */
  int32_t chunk;         /* samples per classifier pass (workspace capacity), >= 1 */
  int32_t max_images;    /* largest B a call will pass                             */
  int32_t autotune;      /* 1: cudnnFind* / cublasLt heuristics top-k timing at create */
  int32_t reserved;
} dp_config;

/* ---- library ---------------------------------------------------------------- */
int32_t     dp_abi_version(void);
const char* dp_last_error(void);

/* ---- engine lifetime ---------------------------------------------------------- */
int32_t dp_engine_create(const dp_config* cfg, dp_engine** out);
void    dp_engine_destroy(dp_engine* e);

/* timm-named fp32 tensors of resnetv2_50x1_bit (host pointers, OIHW / vectors).
 * Conv weights are standardised (timm StdConv2d, eps 1e-8) once on the device. */
int32_t dp_engine_load_weights(dp_engine* e, int32_t n_tensors, const char* const* names,
                               const float* const* host_ptrs, const int64_t* numels);

/* bytes of device memory the engine holds (workspace + weights) */
int64_t dp_engine_device_bytes(const dp_engine* e);
/* number of CUDA kernels / library launches issued by the engine since create */
int64_t dp_engine_launch_count(const dp_engine* e);
/* number of dp_attack_grad calls served by replaying a captured CUDA graph (the launch count above still counts the
 * kernels each replay executes) */
int64_t dp_engine_graph_replays(const dp_engine* e);
/* empty, or why the last graph capture was abandoned (the call then ran as ordinary launches) */
const char* dp_engine_graph_status(const dp_engine* e);

/* Per-kernel-category profiler: CUDA events around every launch the engine issues.
 * enable: 0 off, 1 on, 2 on + reset counters.  Read returns accumulated device ms, the
 * ALGORITHMIC bytes / flops of the launches (what a perfect kernel must move / compute) and
 * launch counts per category; `names` is a [max_n][name_stride] char array. */
int32_t dp_engine_profile(dp_engine* e, int32_t enable);
int32_t dp_engine_profile_read(dp_engine* e, int32_t max_n, char* names, int32_t name_stride, double* ms,
                               double* bytes, double* flops, int64_t* counts, int32_t* n_out);

/* ---- per-image pieces ----------------------------------------------------------- */
/* adv_x = x + clip(mask, pattern, x, eps)  (utils.py:105-110, attack.py:185).
 * x, pattern, adv_x_out: [B,3,H,W] fp32 NCHW dev; mask [B,1,H,W] dev;
 * l2_host[B] receives ||delta||_2 (before clipping), scale_host[B] min(eps/l2,1);
 * either may be NULL. */
int32_t dp_paste(dp_engine* e, const float* x, const float* mask, const float* pattern, int32_t B,
                 float eps, float* adv_x_out, float* l2_host, float* scale_host, void* stream);

/* Non-overlapping k x k window sums of a [B,1,H,W] dev tensor -> out_host[B,(H/k)*(W/k)]. */
int32_t dp_window_sum(dp_engine* e, const float* t, int32_t B, int32_t k, int32_t square,
                      float* out_host, void* stream);

/* ---- K1: EOT expansion ------------------------------------------------------------ */
/* img [B,3,H,W] fp32 dev in [0,1]; rects_host [B*S][4][4] int16 (r0,r1,c0,c1; empty
 * rect = all zeros) or NULL (no occlusion).  Writes the engine's network-input buffer
 * for samples [0, B*S) when it fits `chunk`, or to `out` (dev, engine layout:
 * [B*S,H,W,Cpad] in the engine's activation dtype) when out != NULL.  Occluded pixels
 * are 0.5 in image space = exactly 0 after normalisation. */
int32_t dp_expand(dp_engine* e, const float* img, int32_t B, int32_t S, const int16_t* rects_host,
                  void* out, void* stream);
/* Same kernel with the rectangles already on the device (int16 [B*S][4][4] dev, or NULL): no host copy, no
 * synchronisation -- exactly one kernel launch on `stream` (what bench.py brackets with CUDA events). */
int32_t dp_expand_dev(dp_engine* e, const float* img, int32_t B, int32_t S, const int16_t* rects_dev,
                      void* out, void* stream);
/* The variant of K1 the hot loop launches (attack.py:184-185 fused in: reads x / mask / pattern [B,...] dev and the
 * engine's per-image clip scale, which only the last dp_attack_grad or dp_paste with adv_x_out == NULL writes; a
 * dp_paste with an output buffer leaves it alone), for samples [n0, n0+n) of the b-major
 * [B*S] ordering -- one classifier chunk.  Rectangles on the device; exactly one kernel launch, no synchronisation
 * (bench.py's roofline leg times this launch). */
int32_t dp_expand_step_dev(dp_engine* e, const float* x, const float* mask, const float* pattern, int32_t B, int32_t S,
                           const int16_t* rects_dev, int32_t n0, int32_t n, void* out, void* stream);
/* How many EOT samples one K1 launch of dp_attack_grad covers when the step holds n_samples: all of them (one launch
 * per step into a step-sized buffer) while that buffer stays under DORPATCH_K1_WHOLE_MB, else one classifier chunk. */
int32_t dp_k1_samples_per_launch(const dp_engine* e, int32_t n_samples);
int32_t dp_input_layout(const dp_engine* e, int32_t* c_pad, int32_t* elem_bytes);

/* ---- forward-only: model(occlude(img)) ---------------------------------------------- */
/* preds_host[B*S] = argmax logits; logits_host[B*S*n_classes] optional (NULL to skip). */
int32_t dp_predict(dp_engine* e, const float* img, int32_t B, int32_t S, const int16_t* rects_host,
                   int32_t* preds_host, float* logits_host, void* stream);

/* ---- hot loop ------------------------------------------------------------------------ */
typedef struct dp_attack_args {
  int32_t B;                 /* images                                              */
  int32_t S;                 /* EOT samples per image processed by THIS call (local shard) */
  int32_t S_total;           /* EOT samples per image across all ranks (loss mean divisor)  */
  int32_t stage;             /* 0: mask+pattern learnable, 1: pattern only           */
  const float* x;            /* [B,3,H,W] dev                                        */
  const float* mask;         /* [B,1,H,W] dev                                        */
  const float* pattern;      /* [B,3,H,W] dev                                        */
  const int16_t* rects_host; /* [B*S][4][4] occluder rectangles of each sample       */
  const int64_t* y_host;     /* [B] labels / targets                                 */
  const uint8_t* targeted_host; /* [B] CW criterion is targeted?                     */
  float confidence;          /* CW kappa (attack.py:52, 0.1)                         */
  float eps;                 /* L2 bound of utils.clip                               */
  /* outputs */
  float* grad_adv;           /* [B,3,H,W] dev: d(mean_s CW)/d adv_x (sum over local S,
                                 divided by S_total) -- the buffer ranks all-reduce  */
  float* loss_adv_host;      /* [B*S] CW loss per sample                             */
  int32_t* preds_host;       /* [B*S] argmax of the logits                           */
  float* loss_struc_host;    /* [B]                                                  */
  float* loss_density_host;  /* [B] (stage 0; else untouched)                        */
  float* group_lasso_host;   /* [B] (stage 0; else untouched)                        */
  float* l2_host;            /* [B] ||delta||_2 before clipping                      */
  /* optional affine / colour EOT (SURVEY 8f N3; not in the reference, NULL = off = reference
   * behaviour): [B*S][8] = {t00,t01,t02,t10,t11,t12 (affine_grid theta, align_corners=False,
   * border padding), contrast, brightness}; applied to adv_x before the occlusion. */
  const float* xform_host;
} dp_attack_args;

/* attack.py:184-247 up to (and including) backward; leaves per-image state
 * (adv_x, clip scale, regulariser gradients) inside the engine for dp_attack_update. */
int32_t dp_attack_grad(dp_engine* e, const dp_attack_args* a, void* stream);

typedef struct dp_update_args {
  int32_t B;
  int32_t stage;
  const float* x;              /* [B,3,H,W] dev                                      */
  float* mask;                 /* [B,1,H,W] dev, updated in place when stage == 0     */
  float* pattern;              /* [B,3,H,W] dev, updated in place                     */
  const float* grad_adv;       /* [B,3,H,W] dev (after the cross-rank all-reduce)     */
  const float* lr_host;        /* [B] step size per image (0 = frozen image)          */
  const float* structured_host;/* [B] coefficient of the structural loss              */
  const float* coeff_gl_host;  /* [B] coefficient of the group lasso (stage 0)        */
  float density;               /* coefficient of the density loss (stage 0)           */
  float clip_min, clip_max;
  float* grad_pattern_out;     /* optional [B,3,H,W] dev: full d loss / d pattern     */
  float* grad_mask_out;        /* optional [B,1,H,W] dev: full d loss / d mask        */
  const float* grad_pattern_bias; /* optional [B,3,H,W] dev, added to d loss / d pattern before the
                                     sign: the stale stage-0 gradient the reference's first stage-1
                                     step accumulates onto (attack.py:310-315 break precedes :342) */
} dp_update_args;

/* attack.py:332-342: theta -= lr * sign(grad theta); clip.  Must follow a
 * dp_attack_grad on the same (x, mask, pattern). */
int32_t dp_attack_update(dp_engine* e, const dp_update_args* a, void* stream);

/* Same step through HOST buffers (bench.py's e2e leg): copies x/mask/pattern in from
 * host memory, runs dp_attack_grad + dp_attack_update, copies mask/pattern back.
 * Pointers named *dev* in dp_attack_args / dp_update_args are HOST pointers here;
 * grad_adv may be NULL. */
int32_t dp_attack_step_host(dp_engine* e, const dp_attack_args* g, const dp_update_args* u, void* stream);

/* ---- debugging / test hooks ------------------------------------------------------------ */
/* Run the classifier forward (and optionally backward from dlogits) on an already
 * normalised NCHW fp32 dev batch z[N,3,H,W]; N <= chunk.  logits_dev [N,n_classes]
 * fp32 dev; if dlogits_dev != NULL also writes dz_dev [N,3,H,W] fp32 (d/dz). */
int32_t dp_net_forward_backward(dp_engine* e, const float* z, int32_t N, float* logits_dev,
                                const float* dlogits_dev, float* dz_dev, void* stream);

/* ---- failed-mask sets on the device (attack.py:96 `failed_idxs`, :187-190 scan, :259-267 per-step update) --------
 * One bitmap over the mask universe per image, owned by the engine.  dp_failed_set_write replaces image b's set (the
 * result of a universe scan); dp_failed_set_update applies one step -- idx_host [B*S] sampled mask indices, the first
 * nff_host[b] of image b drawn from its failed set, loss < thresh = success; loss_host NULL = use the CW losses the last
 * dp_attack_grad left on the device -- and returns the set sizes count_host[B] (all the bookkeeping of attack.py:269-308
 * needs); dp_failed_set_read returns the sorted indices (needed only when the sampler draws from the set, i >= 1000). */
int32_t dp_failed_set_write(dp_engine* e, int32_t b, const int32_t* idx_host, int32_t n, void* stream);
int32_t dp_failed_set_update(dp_engine* e, int32_t B, int32_t S, const int32_t* idx_host, const int32_t* nff_host,
                             const uint8_t* active_host, const float* loss_host, float thresh, int32_t* count_host,
                             void* stream);
int32_t dp_failed_set_read(dp_engine* e, int32_t b, int32_t* idx_host_out, int32_t cap, int32_t* n_out, void* stream);

/* Op-level hooks for the parity tests (tests/test_gpu_ops.py, tests/test_gpu_patch_kernels.py); not part of the
 * reference-facing surface.
 * dp_debug_k1t: the K1^T dp_attack_grad runs for samples [n0, n0+n) of the b-major [B*S] ordering, into the caller's
 *   G [B,3,H,W] fp32 dev: G[b] = 2 * sum_s keep_s * dX_s over the launch's samples of image b, OVERWRITING G[b] when the
 *   launch holds image b's first sample and adding to it otherwise (G is not cleared).  rects_host as in dp_expand.
 *   dz is the chunk's slice (sample n0 first): on the bf16 engine with the fused stem backward dz = dY
 *   [n, H/2, W/2, 64] bf16 and dX_s = conv7x7s2^T(dY_s, W_stem); otherwise dz = dX [n, H, W, Cpd] in the activation
 *   dtype (Cpd = 4 fp32 / 8 bf16; channels >= 3 are ignored).
 * dp_debug_cw: K4 on caller-supplied device buffers: logits [N,K] fp32, y [N] int32, targeted [N] uint8; writes
 *   loss [N], preds [N] int32 and dlogits [N,K] (= w * d loss / d logits) -- each may be NULL (loss NULL: preds only).
 * dp_debug_gn_gemm: the tcgen05 GroupNorm-prologue GEMM on caller-supplied operands: out[m,n] = sum_k
 *   relu(gn(x))[m,k] * W[n,k] (+ shortcut); x [N*P,K] bf16, w_nk [Nout,K] bf16, stats [N,32,2] (mean, rstd), all dev.
 * dp_debug_gn: GroupNorm(32)+ReLU forward (and, with dy, backward-to-input) in the engine's activation dtype on
 *   caller-supplied [N,P,C] tensors; stats [N,32,2] dev out.  y == NULL: statistics pass only (the streaming
 *   kernel in front of the tcgen05 GEMM and the classifier head). */
int32_t dp_debug_k1t(dp_engine* e, const void* dz, const int16_t* rects_host, int32_t B, int32_t S, int32_t n0, int32_t n,
                     float* G, void* stream);
int32_t dp_debug_cw(dp_engine* e, const float* logits, const int32_t* y, const uint8_t* targeted, float confidence, float w,
                    float* loss, int32_t* preds, float* dlogits, int32_t N, int32_t K, void* stream);
/* K1 launch-shape sweep hook (tools/k1_step_sweep.py): tile rows / sample groups (0 = the wave-efficiency heuristic) and the
 * store path (0 = bulk stores + 16-byte stores for occluded rows, 1 = 16-byte stores only).  Process-wide. */
int32_t dp_debug_k1_tuning(int32_t rows, int32_t sg, int32_t mode);
/* launch shape of the last K1 launch: {tile rows, sample groups, grid, resident CTAs per SM}. */
int32_t dp_debug_k1_last(int32_t* out4);
int32_t dp_debug_gn_gemm(dp_engine* e, const void* x, const void* w_nk, const float* stats, const float* gamma,
                         const float* beta, const void* shortcut, void* out, int32_t N, int32_t P, int32_t K,
                         int32_t Nout, void* stream);
int32_t dp_debug_gn(dp_engine* e, const void* x, const void* dy, const void* addend, const float* gamma, const float* beta,
                    int32_t gamma_positive, void* y, void* dx, float* stats, int32_t N, int32_t P, int32_t C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DORPATCH_H_ */
