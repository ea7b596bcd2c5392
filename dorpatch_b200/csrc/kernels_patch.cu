// kernels_patch.cu -- hand-written sm_100a kernels of the patch side of the DorPatch hot loop.
//
//   paste    utils.py:105-110 (clip) + attack.py:185        per image, L2 norm via warp shuffles
//   expand   K1: attack.py:204-220 + utils.py:77-78         paste + normalise + occlude, ONE HBM pass,
//                                                           TMA (cp.async.bulk) staged shared-memory tiles
//   cw       K4: attack.py:16-23,224-225                    CW margin loss + argmax + dlogits
//   reduce   K1^T: adjoint of the occlusion/normalisation   masked EOT gradient reduce over S
//   struct   attack.py:33-45,227-228                        structural loss + its (one-sided) gradient
//   maskreg  attack.py:72-80,235-245                        density + group-lasso values / statistics
//   update   K3: attack.py:332-342                          chain rule through clip + sign step + clip
// (file:line into /root/reference).  Images are NCHW fp32; network input is NHWC(Cp) T.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace dp {

// =====================================================================================
// paste: one CTA per image (deterministic reduction order)
// =====================================================================================
__global__ void __launch_bounds__(1024) paste_kernel(const float* __restrict__ x, const float* __restrict__ mask,
                                                     const float* __restrict__ pattern, float* __restrict__ adv,
                                                     float* __restrict__ l2, float* __restrict__ scale, int HW,
                                                     float eps) {
  __shared__ float red[32];
  const int b = blockIdx.x;
  const float* xb = x + (size_t)b * 3 * HW;
  const float* pb = pattern + (size_t)b * 3 * HW;
  const float* mb = mask + (size_t)b * HW;
  float s = 0.f;
  for (int i = threadIdx.x; i < HW; i += blockDim.x) {
    const float m = mb[i];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float d = __fmul_rn(m, __fsub_rn(pb[c * HW + i], xb[c * HW + i]));
      s = fmaf(d, d, s);
    }
  }
  const float norm = sqrtf(block_sum(s, red));
  const float sc = fminf(__fdiv_rn(eps, norm), 1.0f);   // eps/0 = inf -> 1, as torch .clip(max=1)
  if (threadIdx.x == 0) { l2[b] = norm; scale[b] = sc; }
  if (adv != nullptr) {
    float* ab = adv + (size_t)b * 3 * HW;
    for (int i = threadIdx.x; i < HW; i += blockDim.x) {
      const float m = mb[i];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float xv = xb[c * HW + i];
        const float d = __fmul_rn(__fmul_rn(m, __fsub_rn(pb[c * HW + i], xv)), sc);
        ab[c * HW + i] = __fadd_rn(xv, d);
      }
    }
  }
}
void launch_paste(const float* x, const float* mask, const float* pattern, float* adv_x, float* l2, float* scale,
                  int B, int H, int W, float eps, cudaStream_t st) {
  paste_kernel<<<B, 1024, 0, st>>>(x, mask, pattern, adv_x, l2, scale, H * W, eps);
}

// =====================================================================================
// K1 expand: TMA bulk loads of the image planes -> shared; "clean" normalised NHWC tile
// composed once per (image, row tile); per EOT sample either bulk-stored straight from
// the clean tile (no occluder touches these rows) or from a staging tile with the
// occluded pixels zeroed.  HBM-bound: bytes written = N*H*W*Cp*sizeof(T).
// =====================================================================================
namespace ptx {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
}  // namespace ptx

constexpr int EXP_R_DEFAULT = 8;  // image rows per tile (DORPATCH_K1_ROWS overrides; must divide H)
constexpr int EXP_THREADS = 256;
constexpr int EXP_WARPS = EXP_THREADS / 32;
constexpr int EXP_HDR = 512 + 2048;   // mbarrier + per-item rectangle cache (64 samples x 32 B)
constexpr int EXP_RCACHE = 64;

__device__ __forceinline__ bool rect_hit(const short* r, int row, int col) {
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (row >= r[4 * k] && row < r[4 * k + 1] && col >= r[4 * k + 2] && col < r[4 * k + 3]) return true;
  return false;
}

struct ExpandParams {
  const float* img; const float* x; const float* mask; const float* pattern; const float* scale;
  const int16_t* rects; void* out;
  int B, S, n0, n, H, W, sgroups, R;
  int mode;   // 0: bulk stores (cp.async.bulk) for untouched tiles / rows + 16-byte stores for occluded rows; 1: 16-byte stores only
};

// Shared memory (dynamic): [mbarrier, 512 B][input planes NP*R*W fp32][clean tile R*W*CP T].
// A tile is R full image rows of the output layout = one contiguous run of the output tensor.
// Per EOT sample a warp either bulk-stores the clean tile / clean rows (TMA, cp.async.bulk) when no
// occluder crosses them, or writes an occluded row itself with 16-byte global stores whose keep /
// zero / mixed status comes from <= 4 element intervals (no staging copy, no block barrier).
template <typename T, int CP, bool FUSED>
__global__ void __launch_bounds__(EXP_THREADS) expand_kernel(ExpandParams p) {
  constexpr int NP = FUSED ? 7 : 3;
  constexpr int EPC = 16 / (int)sizeof(T);                 // elements per 16-byte chunk
  extern __shared__ __align__(128) unsigned char smem[];
  const int W = p.W, H = p.H, HW = H * W;
  const int EXP_R = p.R;
  const int tile_px = EXP_R * W;
  const uint32_t plane_bytes = (uint32_t)tile_px * 4u;
  const int row_elems = W * CP;
  const uint32_t row_bytes = (uint32_t)row_elems * (uint32_t)sizeof(T);
  const uint32_t out_bytes = row_bytes * EXP_R;
  const int row_chunks = row_elems / EPC;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  int4* srect = reinterpret_cast<int4*>(smem + 512);
  float* in = reinterpret_cast<float*>(smem + EXP_HDR);
  unsigned char* clean_b = smem + EXP_HDR + NP * plane_bytes;
  T* clean = reinterpret_cast<T*>(clean_b);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) { ptx::mbar_init(bar, 1); ptx::fence_mbar_init(); ptx::fence_proxy_async(); }
  __syncthreads();

  const int b_first = p.n0 / p.S, b_last = (p.n0 + p.n - 1) / p.S;
  const int tiles = H / EXP_R;
  const int items = (b_last - b_first + 1) * tiles * p.sgroups;
  uint32_t phase = 0;

  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int sg = item % p.sgroups;
    const int tile = (item / p.sgroups) % tiles;
    const int b = b_first + item / (p.sgroups * tiles);
    const int lo = max(p.n0, b * p.S), hi = min(p.n0 + p.n, (b + 1) * p.S);
    const int cnt = hi - lo;
    const int s_lo = lo + (int)(((long long)cnt * sg) / p.sgroups), s_hi = lo + (int)(((long long)cnt * (sg + 1)) / p.sgroups);
    if (s_lo >= s_hi) continue;   // uniform across the CTA
    const int r0 = tile * EXP_R;

    // every warp's bulk stores of the previous item have finished READING the clean tile (see loop end)
    __syncthreads();
    if (threadIdx.x == 0) {
      ptx::mbar_expect_tx(bar, NP * plane_bytes);
      if (FUSED) {
        for (int c = 0; c < 3; ++c) ptx::bulk_load(in + c * tile_px, p.x + ((size_t)(b * 3 + c) * H + r0) * W, plane_bytes, bar);
        for (int c = 0; c < 3; ++c) ptx::bulk_load(in + (3 + c) * tile_px, p.pattern + ((size_t)(b * 3 + c) * H + r0) * W, plane_bytes, bar);
        ptx::bulk_load(in + 6 * tile_px, p.mask + ((size_t)b * H + r0) * W, plane_bytes, bar);
      } else {
        for (int c = 0; c < 3; ++c) ptx::bulk_load(in + c * tile_px, p.img + ((size_t)(b * 3 + c) * H + r0) * W, plane_bytes, bar);
      }
    }
    // rectangle cache of this item's samples (hides the per-sample global-load latency)
    const bool cached = p.rects != nullptr && (s_hi - s_lo) <= EXP_RCACHE;
    if (cached)
      for (int i = threadIdx.x; i < 2 * (s_hi - s_lo); i += EXP_THREADS)
        srect[i] = __ldg(reinterpret_cast<const int4*>(p.rects + (size_t)s_lo * 16) + i);
    ptx::mbar_wait(bar, phase);
    phase ^= 1u;

    const float sc = FUSED ? p.scale[b] : 1.0f;
    for (int i = threadIdx.x; i < tile_px; i += EXP_THREADS) {
      float v[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float a = in[c * tile_px + i];
        if (FUSED) {
          const float d = __fmul_rn(__fmul_rn(in[6 * tile_px + i], __fsub_rn(in[(3 + c) * tile_px + i], a)), sc);
          a = __fadd_rn(a, d);
        }
        v[c] = __fmul_rn(__fsub_rn(a, 0.5f), 2.0f);   // (a - 0.5) / 0.5
      }
#pragma unroll
      for (int c = 0; c < CP; ++c) clean[i * CP + c] = from_float<T>(c < 3 ? v[c] : 0.f);
    }
    ptx::fence_proxy_async();
    __syncthreads();

    // ---- one warp per EOT sample (measured: splitting a touched tile's rows across the warps is 1.5x slower --
    //      every warp then decodes every sample's rectangles) -----------------------------------------------
    for (int n = s_lo + warp; n < s_hi; n += EXP_WARPS) {
      unsigned char* dst = reinterpret_cast<unsigned char*>(p.out) + ((size_t)(n - p.n0) * HW + (size_t)r0 * W) * CP * sizeof(T);
      int rr0[4], rr1[4], el[4], eh[4];
      bool any = false;
      if (p.rects != nullptr) {
        int4 q0, q1;
        if (cached) { q0 = srect[2 * (n - s_lo)]; q1 = srect[2 * (n - s_lo) + 1]; }
        else {
          const int4* rp = reinterpret_cast<const int4*>(p.rects + (size_t)n * 16);
          q0 = __ldg(rp); q1 = __ldg(rp + 1);                 // same address in every lane: broadcast
        }
        const int w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          rr0[k] = (short)(w[2 * k] & 0xffff); rr1[k] = (short)(w[2 * k] >> 16);
          el[k] = (short)(w[2 * k + 1] & 0xffff) * CP; eh[k] = (short)(w[2 * k + 1] >> 16) * CP;
          if (eh[k] <= el[k]) { rr0[k] = 0; rr1[k] = 0; }      // empty rectangle
          any = any || (rr0[k] < r0 + EXP_R && rr1[k] > r0);
        }
      }
      const bool use_bulk = p.mode == 0;
      if (!any && use_bulk) {                                   // whole tile untouched: one bulk store
        if (lane == 0) { ptx::bulk_store(dst, clean_b, out_bytes); ptx::bulk_commit(); }
        continue;
      }
      // Row-independent part, once per sample: field j (EPC bits) of zm[k] = which elements of this lane's chunk
      // (cb + lane + 32 j) rectangle k zeroes -- all ones inside, zero outside, a bit range on the <= 2 chunks that
      // straddle an edge.  A row then only ORs the words of the rectangles that cover it.
      constexpr int JB = 32 / EPC;                              // chunks per lane per mask word (4 bf16 / 8 fp32)
      constexpr uint32_t FULL = (1u << EPC) - 1u;
      for (int cb = 0; cb < row_chunks; cb += 32 * JB) {        // one pass for rows up to 2048 B (bf16) / 4096 B (fp32)
        uint32_t zm[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint32_t z = 0u;
#pragma unroll
          for (int j = 0; j < JB; ++j) {
            const int e0 = (cb + lane + 32 * j) * EPC;
            const int lo = min(max(el[k] - e0, 0), EPC), hi = min(max(eh[k] - e0, 0), EPC);
            const uint32_t m = hi > lo ? (((1u << hi) - 1u) & ~((1u << lo) - 1u)) : 0u;
            z |= m << (EPC * j);
          }
          zm[k] = z;
        }
        for (int rr = 0; rr < EXP_R; ++rr) {
          const int row = r0 + rr;
          uint32_t Z = 0u;
          bool rany = false;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const bool cov = row >= rr0[k] && row < rr1[k];
            rany = rany || cov;
            Z |= cov ? zm[k] : 0u;
          }
          if (!rany && use_bulk) {                              // clean row: bulk store
            if (cb == 0 && lane == 0) { ptx::bulk_store(dst + (size_t)rr * row_bytes, clean_b + (size_t)rr * row_bytes, row_bytes); ptx::bulk_commit(); }
            continue;
          }
          const uint4* crow = reinterpret_cast<const uint4*>(clean_b + (size_t)rr * row_bytes);
          uint4* drow = reinterpret_cast<uint4*>(dst + (size_t)rr * row_bytes);
#pragma unroll
          for (int j = 0; j < JB; ++j) {
            const int ch = cb + lane + 32 * j;
            if (ch >= row_chunks) break;
            const uint32_t m = (Z >> (EPC * j)) & FULL;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (m != FULL) {
              v = crow[ch];
              if (m != 0u) {                                    // edge chunk: clear the covered elements
                if (EPC == 8) {                                 // two 16-bit elements per word
                  v.x &= ~(((m & 1u) ? 0xffffu : 0u) | ((m & 2u) ? 0xffff0000u : 0u));
                  v.y &= ~(((m & 4u) ? 0xffffu : 0u) | ((m & 8u) ? 0xffff0000u : 0u));
                  v.z &= ~(((m & 16u) ? 0xffffu : 0u) | ((m & 32u) ? 0xffff0000u : 0u));
                  v.w &= ~(((m & 64u) ? 0xffffu : 0u) | ((m & 128u) ? 0xffff0000u : 0u));
                } else {
                  if (m & 1u) v.x = 0u;
                  if (m & 2u) v.y = 0u;
                  if (m & 4u) v.z = 0u;
                  if (m & 8u) v.w = 0u;
                }
              }
            }
            drow[ch] = v;
          }
        }
      }
    }
    // before the clean tile is overwritten: each issuing lane waits for its bulk stores' reads
    if (lane == 0) ptx::bulk_wait_read<0>();
  }
  // (global visibility of the bulk stores is guaranteed at kernel completion)
}

// Launch shape.  Work items = images x row tiles (R rows) x sample groups, walked grid-stride by the resident CTAs.
// Measured over tile heights x sample groups x launch sizes (tools/k1_step_sweep.py, profiles/r02_k1_sweep.txt): tiles of
// 4-8 rows are equivalent and best (a CTA's load + compose prologue stays short and 3-6 CTAs per SM overlap it with their
// neighbours' stores), 14-16 rows lose 10-30 % (1-2 CTAs per SM, the prologue is exposed), 2 rows lose 15-20 % (per-item
// overhead), and a launch wants >= 4 items per SM.  Rule: R = 8, or 4 when that leaves fewer than 4 items per SM; sample
// groups (each re-loads and re-composes the tile) only when the images alone give fewer than 2 items per SM (B = 1).
// Round 2's first rule maximised "wave efficiency" and picked R = 14 for 512- and 2048-sample launches: 0.29 / 0.65 of
// peak against 0.72 / 0.79 with R = 8.  DORPATCH_K1_ROWS / _K1_SG (or dp_debug_k1_tuning) pin the choice.
static int g_k1_rows = -2, g_k1_sg = -1, g_k1_mode = 0;   // launch-shape overrides (environment, or set_expand_tuning for sweeps)
static int g_k1_last[4] = {0, 0, 0, 0};                    // tile rows, sample groups, grid, resident CTAs per SM of the last launch
void get_expand_last(int* out4) { for (int i = 0; i < 4; ++i) out4[i] = g_k1_last[i]; }
void set_expand_tuning(int rows, int sg, int mode) { g_k1_rows = rows < 0 ? 0 : rows; g_k1_sg = sg < 0 ? 0 : sg; g_k1_mode = mode; }

template <typename T, int CP, bool FUSED>
static void expand_launch(const ExpandParams& p, int num_sms, cudaStream_t st) {
  if (g_k1_rows == -2) {
    const char* e = getenv("DORPATCH_K1_ROWS"); g_k1_rows = e ? atoi(e) : 0;
    const char* g = getenv("DORPATCH_K1_SG"); g_k1_sg = g ? atoi(g) : 0;
    const char* m = getenv("DORPATCH_K1_MODE"); g_k1_mode = m ? atoi(m) : 0;
  }
  const int rows_env = g_k1_rows, sg_env = g_k1_sg;
  constexpr int NP = FUSED ? 7 : 3;
  auto smem_of = [&](int R) { return (size_t)EXP_HDR + (size_t)NP * R * p.W * 4 + (size_t)R * p.W * CP * sizeof(T); };
  static int occ_cache[33];
  static bool occ_init = false;
  if (!occ_init) { for (int& v : occ_cache) v = -1; occ_init = true; }
  auto resident = [&](int R) {
    if (occ_cache[R] < 0) {
      const size_t sm = smem_of(R);
      cudaFuncSetAttribute(expand_kernel<T, CP, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, expand_kernel<T, CP, FUSED>, EXP_THREADS, sm) != cudaSuccess || nb < 1) { cudaGetLastError(); nb = 1; }
      occ_cache[R] = nb;
    }
    return occ_cache[R];
  };
  const int nb_img = (p.n0 + p.n - 1) / p.S - p.n0 / p.S + 1;
  auto usable = [&](int R) { return R >= 1 && R <= 32 && p.H % R == 0 && smem_of(R) <= 200 * 1024; };
  int best_R = 0, best_sg = 1;
  if (rows_env > 0 && usable(rows_env)) best_R = rows_env;
  else {
    const int pref[] = {8, 7, 4, 2, 1};
    for (int R : pref)
      if (usable(R)) { if (best_R == 0) best_R = R; if (nb_img * (p.H / R) >= 4 * num_sms || R <= 4) { best_R = R; break; } }
    if (best_R == 0) best_R = 1;
  }
  if (sg_env > 0) best_sg = sg_env;
  else
    while (nb_img * (p.H / best_R) * best_sg < 2 * num_sms && best_sg * 2 * EXP_WARPS <= p.S && best_sg < 32) best_sg *= 2;
  const int items_total = nb_img * (p.H / best_R) * best_sg;
  const int slots = num_sms * resident(best_R);
  const int best_grid = items_total < slots ? items_total : slots;
  const size_t smem = smem_of(best_R);
  cudaFuncSetAttribute(expand_kernel<T, CP, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  ExpandParams q = p;
  q.R = best_R;
  q.sgroups = best_sg;
  q.mode = g_k1_mode;
  g_k1_last[0] = best_R; g_k1_last[1] = best_sg; g_k1_last[2] = best_grid; g_k1_last[3] = resident(best_R);
  expand_kernel<T, CP, FUSED><<<best_grid, EXP_THREADS, smem, st>>>(q);
}

void launch_expand(const float* img, const float* x, const float* mask, const float* pattern, const float* scale,
                   const int16_t* rects, void* out, int B, int S, int n0, int n, int H, int W, int Cp, bool bf16,
                   bool fused, int num_sms, cudaStream_t st) {
  ExpandParams p{img, x, mask, pattern, scale, rects, out, B, S, n0, n, H, W, 1, EXP_R_DEFAULT, 0};
#define EXP_CASE(TT, CPV)                                                   \
  if (fused) expand_launch<TT, CPV, true>(p, num_sms, st);                 \
  else expand_launch<TT, CPV, false>(p, num_sms, st)
  if (bf16) {
    if (Cp == 8) { EXP_CASE(__nv_bfloat16, 8); }
    else if (Cp == 4) { EXP_CASE(__nv_bfloat16, 4); }
    else { EXP_CASE(__nv_bfloat16, 3); }
  } else {
    if (Cp == 4) { EXP_CASE(float, 4); }
    else if (Cp == 8) { EXP_CASE(float, 8); }
    else { EXP_CASE(float, 3); }
  }
#undef EXP_CASE
}

// =====================================================================================
// Optional affine / colour EOT (SURVEY 8f N3; named by the north-star, absent from the reference --
// default off).  Per sample: bilinear warp of the pasted image by theta (torch affine_grid /
// grid_sample semantics: align_corners=False, padding_mode='border'), then
// v' = clamp(contrast*(v-0.5)+0.5+brightness, 0, 1), then occlusion + normalisation.
// xf[n] = {t00,t01,t02,t10,t11,t12, contrast, brightness}.  Gather kernel (the source rows are
// arbitrary, so no TMA row tiles); its adjoint scatters with fp32 atomics.
// =====================================================================================
struct AffTap { int i00, i01, i10, i11; float w00, w01, w10, w11; };
__device__ __forceinline__ AffTap affine_taps(const float* __restrict__ t, int h, int w, int H, int W) {
  const float xn = (2.f * w + 1.f) / W - 1.f, yn = (2.f * h + 1.f) / H - 1.f;
  float fx = ((t[0] * xn + t[1] * yn + t[2] + 1.f) * W - 1.f) * 0.5f;
  float fy = ((t[3] * xn + t[4] * yn + t[5] + 1.f) * H - 1.f) * 0.5f;
  fx = fminf(fmaxf(fx, 0.f), (float)(W - 1));
  fy = fminf(fmaxf(fy, 0.f), (float)(H - 1));
  const int x0 = (int)floorf(fx), y0 = (int)floorf(fy);
  const float ax = fx - x0, ay = fy - y0;
  const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
  AffTap a;
  a.i00 = y0 * W + x0; a.i01 = y0 * W + x1; a.i10 = y1 * W + x0; a.i11 = y1 * W + x1;
  a.w00 = (1.f - ax) * (1.f - ay); a.w01 = (x0 + 1 < W ? ax : 0.f) * (1.f - ay);
  a.w10 = (1.f - ax) * (y0 + 1 < H ? ay : 0.f); a.w11 = (x0 + 1 < W ? ax : 0.f) * (y0 + 1 < H ? ay : 0.f);
  return a;
}

template <typename T, int CP>
__global__ void __launch_bounds__(256) expand_affine_kernel(const float* __restrict__ adv, const float* __restrict__ xf,
                                                            const int16_t* __restrict__ rects, T* __restrict__ out,
                                                            int S, int n0, int H, int W) {
  const int HW = H * W, n = n0 + blockIdx.y, b = n / S;
  const int px = blockIdx.x * blockDim.x + threadIdx.x;
  if (px >= HW) return;
  const int h = px / W, w = px % W;
  const float* t = xf + (size_t)n * 8;
  const AffTap a = affine_taps(t, h, w, H, W);
  bool occ = false;
  if (rects != nullptr) {
    short r[16];
    const int4* rp = reinterpret_cast<const int4*>(rects + (size_t)n * 16);
    *reinterpret_cast<int4*>(r) = __ldg(rp); *reinterpret_cast<int4*>(r + 8) = __ldg(rp + 1);
    occ = rect_hit(r, h, w);
  }
  T* o = out + ((size_t)blockIdx.y * HW + px) * CP;
#pragma unroll
  for (int c = 0; c < CP; ++c) {
    float z = 0.f;
    if (c < 3 && !occ) {
      const float* pl = adv + ((size_t)b * 3 + c) * HW;
      float v = a.w00 * pl[a.i00] + a.w01 * pl[a.i01] + a.w10 * pl[a.i10] + a.w11 * pl[a.i11];
      v = fminf(fmaxf(t[6] * (v - 0.5f) + 0.5f + t[7], 0.f), 1.f);
      z = (v - 0.5f) * 2.f;
    }
    o[c] = from_float<T>(z);
  }
}

// adjoint: G[b] += scatter( 2 * keep * contrast * [0 < v' < 1] * dz[n] ); G must be zero-initialised
template <typename T, int CP>
__global__ void __launch_bounds__(256) reduce_affine_kernel(const T* __restrict__ dz, const float* __restrict__ adv,
                                                            const float* __restrict__ xf, const int16_t* __restrict__ rects,
                                                            float* __restrict__ G, int S, int n0, int H, int W) {
  const int HW = H * W, n = n0 + blockIdx.y, b = n / S;
  const int px = blockIdx.x * blockDim.x + threadIdx.x;
  if (px >= HW) return;
  const int h = px / W, w = px % W;
  if (rects != nullptr) {
    short r[16];
    const int4* rp = reinterpret_cast<const int4*>(rects + (size_t)n * 16);
    *reinterpret_cast<int4*>(r) = __ldg(rp); *reinterpret_cast<int4*>(r + 8) = __ldg(rp + 1);
    if (rect_hit(r, h, w)) return;
  }
  const float* t = xf + (size_t)n * 8;
  const AffTap a = affine_taps(t, h, w, H, W);
  const T* q = dz + ((size_t)blockIdx.y * HW + px) * CP;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float* pl = adv + ((size_t)b * 3 + c) * HW;
    const float v = a.w00 * pl[a.i00] + a.w01 * pl[a.i01] + a.w10 * pl[a.i10] + a.w11 * pl[a.i11];
    const float vc = t[6] * (v - 0.5f) + 0.5f + t[7];
    if (vc < 0.f || vc > 1.f) continue;                 // torch.clamp passes the gradient on [min, max]
    const float g = 2.f * t[6] * to_float(q[c]);
    float* gp = G + ((size_t)b * 3 + c) * HW;
    if (a.w00 != 0.f) atomicAdd(gp + a.i00, a.w00 * g);
    if (a.w01 != 0.f) atomicAdd(gp + a.i01, a.w01 * g);
    if (a.w10 != 0.f) atomicAdd(gp + a.i10, a.w10 * g);
    if (a.w11 != 0.f) atomicAdd(gp + a.i11, a.w11 * g);
  }
}

void launch_expand_affine(const float* adv, const float* xf, const int16_t* rects, void* out, int S, int n0, int n,
                          int H, int W, int Cp, bool bf16, cudaStream_t st) {
  dim3 grid((H * W + 255) / 256, n);
#define EA(TT, CPV) expand_affine_kernel<TT, CPV><<<grid, 256, 0, st>>>(adv, xf, rects, (TT*)out, S, n0, H, W)
  if (bf16) { if (Cp == 3) EA(__nv_bfloat16, 3); else if (Cp == 4) EA(__nv_bfloat16, 4); else EA(__nv_bfloat16, 8); }
  else { if (Cp == 3) EA(float, 3); else if (Cp == 4) EA(float, 4); else EA(float, 8); }
#undef EA
}
void launch_reduce_affine(const void* dz, const float* adv, const float* xf, const int16_t* rects, float* G, int S, int n0,
                          int n, int H, int W, int Cp, bool bf16, cudaStream_t st) {
  dim3 grid((H * W + 255) / 256, n);
#define RA(TT, CPV) reduce_affine_kernel<TT, CPV><<<grid, 256, 0, st>>>((const TT*)dz, adv, xf, rects, G, S, n0, H, W)
  if (bf16) { if (Cp == 4) RA(__nv_bfloat16, 4); else if (Cp == 3) RA(__nv_bfloat16, 3); else RA(__nv_bfloat16, 8); }
  else { if (Cp == 4) RA(float, 4); else if (Cp == 3) RA(float, 3); else RA(float, 8); }
#undef RA
}

// =====================================================================================
// K4: CW loss / argmax / dlogits -- one warp per sample
// =====================================================================================
// Does logit (v, i) come before the current pick (best, bi)?  torch.argmax / torch.max order: a NaN ranks above every
// number (the first NaN wins), equal values go to the lower index.
__device__ __forceinline__ bool cw_before(float v, int i, float best, int bi) {
  const bool vn = v != v, bn = best != best;
  if (vn != bn) return vn;
  if (!vn && v != best) return v > best;
  return i < bi;
}
__global__ void cw_kernel(const float* __restrict__ logits, const int32_t* __restrict__ y,
                          const uint8_t* __restrict__ targeted, float confidence, float w, float* __restrict__ loss,
                          int32_t* __restrict__ preds, float* __restrict__ dlogits, int N, int K) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (n >= N) return;
  const float* l = logits + (size_t)n * K;
  const int yy = y != nullptr ? y[n] : -1;
  float best = -INFINITY, obest = -INFINITY; int bi = 0x7fffffff, oi = 0x7fffffff;
  bool finite = true;
  for (int k = lane; k < K; k += 32) {
    const float v = l[k];
    finite = finite && isfinite(v);
    if (cw_before(v, k, best, bi)) { best = v; bi = k; }
    if (k != yy && cw_before(v, k, obest, oi)) { obest = v; oi = k; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float v2 = __shfl_xor_sync(0xffffffffu, best, o); const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
    if (cw_before(v2, i2, best, bi)) { best = v2; bi = i2; }
    const float w2 = __shfl_xor_sync(0xffffffffu, obest, o); const int j2 = __shfl_xor_sync(0xffffffffu, oi, o);
    if (cw_before(w2, j2, obest, oi)) { obest = w2; oi = j2; }
  }
  if (lane == 0 && preds != nullptr) preds[n] = bi;
  if (loss == nullptr) return;
  finite = __all_sync(0xffffffffu, finite);
  const float real = l[yy];
  // attack.py:19: the label slot contributes -1e4 to the max (and wins a tie at -1e4 when its index is the lower one)
  const bool other_is_label_slot = obest < -1e4f || (obest == -1e4f && yy < oi);
  const float other = other_is_label_slot ? -1e4f : obest;
  const bool tg = targeted[n] != 0;
  const float margin = tg ? (other - real) : (real - other);
  // attack.py:18-19 multiply the logits by the one-hot label: one non-finite logit (0 * inf = NaN) makes the loss NaN,
  // which torch.clamp passes on (a failed sample) with a zero gradient
  const float pre = finite ? confidence + margin : NAN;
  if (lane == 0) loss[n] = isnan(pre) ? pre : fmaxf(pre, 0.f);
  if (dlogits != nullptr) {
    float* d = dlogits + (size_t)n * K;
    for (int k = lane; k < K; k += 32) d[k] = 0.f;
    __syncwarp();
    if (lane == 0 && pre >= 0.f) {     // clamp(min=0) passes the gradient where input >= 0
      d[yy] = tg ? -w : w;
      if (!other_is_label_slot) d[oi] = tg ? w : -w;
    }
  }
}
void launch_cw(const float* logits, const int32_t* y, const uint8_t* targeted, float confidence, float inv_s_total,
               float* loss, int32_t* preds, float* dlogits, int N, int K, cudaStream_t st) {
  const size_t threads = (size_t)N * 32;
  cw_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(logits, y, targeted, confidence, inv_s_total, loss, preds, dlogits, N, K);
}
void launch_argmax(const float* logits, int32_t* preds, int N, int K, cudaStream_t st) {
  const size_t threads = (size_t)N * 32;
  cw_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(logits, nullptr, nullptr, 0.f, 0.f, nullptr, preds, nullptr, N, K);
}

// =====================================================================================
// K1^T reduce: G[b,c,h,w] (+)= 2 * sum_{samples n of image b in [n0,n0+n)} keep_n(h,w) * dz[n,h,w,c]
// grid (ceil(HW/256), images touched)
// =====================================================================================
constexpr int RED_MAXS = 128;
template <typename T, int CP>
__global__ void __launch_bounds__(256) reduce_kernel(const T* __restrict__ dz, const int16_t* __restrict__ rects,
                                                     float* __restrict__ G, int S, int n0, int n, int H, int W) {
  __shared__ __align__(16) short sr[RED_MAXS * 16];
  const int HW = H * W;
  const int b = n0 / S + blockIdx.y;
  const int lo = max(n0, b * S), hi = min(n0 + n, (b + 1) * S);
  const int px = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = px / W, col = px % W;
  float acc[3] = {0.f, 0.f, 0.f};
  for (int base = lo; base < hi; base += RED_MAXS) {
    const int m = min(RED_MAXS, hi - base);
    __syncthreads();
    for (int i = threadIdx.x; i < m * 16; i += blockDim.x) sr[i] = rects != nullptr ? rects[(size_t)base * 16 + i] : (short)0;
    __syncthreads();
    if (px < HW) {
      for (int j = 0; j < m; ++j) {
        if (rect_hit(sr + j * 16, row, col)) continue;
        const T* q = dz + ((size_t)(base + j - n0) * HW + px) * CP;
        if (CP * sizeof(T) == 16) {
          Vec<T> v; v.load(q);
          float f[Vec<T>::N]; v.unpack(f);
          acc[0] += f[0]; acc[1] += f[1]; acc[2] += f[2];
        } else {
          acc[0] += to_float(q[0]); acc[1] += to_float(q[1]); acc[2] += to_float(q[2]);
        }
      }
    }
  }
  if (px < HW) {
    const bool first = (lo == b * S);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float* g = G + ((size_t)b * 3 + c) * HW + px;
      const float v = 2.0f * acc[c];
      *g = first ? v : (*g + v);
    }
  }
}
void launch_reduce(const void* dz, const int16_t* rects, float* G, int B, int S, int n0, int n, int H, int W,
                   int Cp, bool bf16, cudaStream_t st) {
  const int nb = (n0 + n - 1) / S - n0 / S + 1;
  dim3 grid((H * W + 255) / 256, nb);
#define RED_CASE(TT, CPV) reduce_kernel<TT, CPV><<<grid, 256, 0, st>>>((const TT*)dz, rects, G, S, n0, n, H, W)
  if (bf16) { if (Cp == 8) RED_CASE(__nv_bfloat16, 8); else if (Cp == 4) RED_CASE(__nv_bfloat16, 4); else RED_CASE(__nv_bfloat16, 3); }
  else { if (Cp == 4) RED_CASE(float, 4); else if (Cp == 8) RED_CASE(float, 8); else RED_CASE(float, 3); }
#undef RED_CASE
}

// =====================================================================================
// structural loss (attack.py:33-45,227-228), reproducing the reference's one-sided gradient
// (quirk Q4): lr[h,w] = |a[h,w]-a[h,w+1]| (raw a[h,W-1] in the last column), gradient only
// through the subtracted (right / lower) neighbour.  One CTA per image.
// =====================================================================================
__device__ __forceinline__ void lv_pair(const float* __restrict__ pl, int h, int w, int H, int W, float& A, float& Bv) {
  const float v = pl[h * W + w];
  A = (w < W - 1) ? fabsf(v - pl[h * W + w + 1]) : v;
  Bv = (h < H - 1) ? fabsf(v - pl[(h + 1) * W + w]) : v;
}
__device__ __forceinline__ float lvx_at(const float* __restrict__ xb, int h, int w, int H, int W) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) { float A, Bv; lv_pair(xb + (size_t)c * H * W, h, w, H, W, A, Bv); s += A + Bv; }
  return s / 3.0f;
}
__global__ void __launch_bounds__(1024) struct_kernel(const float* __restrict__ adv, const float* __restrict__ x,
                                                      float* __restrict__ loss, float* __restrict__ dLs, int H, int W) {
  __shared__ float red[32];
  const int b = blockIdx.x, HW = H * W;
  const float* ab = adv + (size_t)b * 3 * HW;
  const float* xb = x + (size_t)b * 3 * HW;
  float* gb = dLs + (size_t)b * 3 * HW;
  const float inv_hw = 1.0f / (float)HW;
  float s = 0.f;
  for (int i = threadIdx.x; i < HW; i += blockDim.x) {
    const int h = i / W, w = i % W;
    // value at (h,w)
    float mvsum = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float A, Bv; lv_pair(ab + (size_t)c * HW, h, w, H, W, A, Bv);
      mvsum += (A + Bv) * (A > Bv ? Bv : A);
    }
    s += (mvsum / 3.0f) / (lvx_at(xb, h, w, H, W) + 1e-5f);
    // gradient wrt adv[c,h,w]: through lr[h,w-1] and ud[h-1,w]
    const float wl = (w >= 1) ? inv_hw / (3.0f * (lvx_at(xb, h, w - 1, H, W) + 1e-5f)) : 0.f;
    const float wu = (h >= 1) ? inv_hw / (3.0f * (lvx_at(xb, h - 1, w, H, W) + 1e-5f)) : 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* pl = ab + (size_t)c * HW;
      const float v = pl[i];
      float g = 0.f;
      if (w >= 1) {
        float A, Bv; lv_pair(pl, h, w - 1, H, W, A, Bv);
        const float dmv_dA = (A > Bv ? Bv : A) + ((A > Bv) ? 0.f : (A + Bv));
        g += wl * dmv_dA * (-sgn(pl[i - 1] - v));
      }
      if (h >= 1) {
        float A, Bv; lv_pair(pl, h - 1, w, H, W, A, Bv);
        const float dmv_dB = (A > Bv ? Bv : A) + ((A > Bv) ? (A + Bv) : 0.f);
        g += wu * dmv_dB * (-sgn(pl[i - W] - v));
      }
      gb[(size_t)c * HW + i] = g;
    }
  }
  const float tot = block_sum(s, red);
  if (threadIdx.x == 0) loss[b] = tot * inv_hw;
}
void launch_struct(const float* adv_x, const float* x, float* loss_struc, float* dLs, int B, int H, int W, cudaStream_t st) {
  struct_kernel<<<B, 1024, 0, st>>>(adv_x, x, loss_struc, dLs, H, W);
}

// =====================================================================================
// density + group lasso (attack.py:72-80,235-245).  One CTA per image.
//   grp_ss[b][g]  = sum of m^2 over the unit x unit group g          (for d GL / d m = unit*m/sqrt(ss))
//   win_dev[b][w] = 2*(ws_w - mean)/(nw-1) for density window w      (d var / d m inside window w)
// =====================================================================================
__global__ void __launch_bounds__(1024) maskreg_kernel(const float* __restrict__ mask, float* __restrict__ loss_density,
                                                       float* __restrict__ group_lasso, float* __restrict__ win_dev,
                                                       float* __restrict__ grp_ss, int H, int W, int unit) {
  extern __shared__ float sh[];
  __shared__ float red[32];
  const int b = blockIdx.x, GH = H / unit, GW = W / unit, NG = GH * GW;
  float* g_s = sh;            // [NG] plain sums
  float* g_q = sh + NG;       // [NG] sums of squares
  const float* mb = mask + (size_t)b * H * W;
  for (int g = threadIdx.x; g < NG; g += blockDim.x) {
    const int gy = g / GW, gx = g % GW;
    float s = 0.f, q = 0.f;
    for (int dy = 0; dy < unit; ++dy)
      for (int dx = 0; dx < unit; ++dx) { const float m = mb[(gy * unit + dy) * W + gx * unit + dx]; s += m; q = fmaf(m, m, q); }
    g_s[g] = s; g_q[g] = q;
    grp_ss[(size_t)b * NG + g] = q;
  }
  __syncthreads();
  float gl = 0.f;
  for (int g = threadIdx.x; g < NG; g += blockDim.x) gl += sqrtf(g_q[g]);
  gl = block_sum(gl, red);
  if (threadIdx.x == 0) group_lasso[b] = (float)unit * gl;
  // density windows: (W/8) x (W/8) pixels = (W/8/unit)^2 groups each, 8 x 8 windows
  const int win = W / 8, gpw = win / unit, NWX = W / win, NWY = H / win, NW = NWX * NWY;
  __shared__ float ws[64];
  if ((int)threadIdx.x < NW) {
    const int wy = threadIdx.x / NWX, wx = threadIdx.x % NWX;
    float s = 0.f;
    for (int a = 0; a < gpw; ++a)
      for (int c = 0; c < gpw; ++c) s += g_s[(wy * gpw + a) * GW + wx * gpw + c];
    ws[threadIdx.x] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mean = 0.f;
    for (int i = 0; i < NW; ++i) mean += ws[i];
    mean /= NW;
    float var = 0.f;
    for (int i = 0; i < NW; ++i) { const float d = ws[i] - mean; var += d * d; }
    loss_density[b] = var / (NW - 1);
    for (int i = 0; i < NW; ++i) win_dev[(size_t)b * 64 + i] = 2.0f * (ws[i] - mean) / (NW - 1);
  }
}
void launch_maskreg(const float* mask, float* loss_density, float* group_lasso, float* win_dev, float* grp_ss,
                    int B, int H, int W, int unit, cudaStream_t st) {
  const int NG = (H / unit) * (W / unit);
  maskreg_kernel<<<B, 1024, 2 * NG * sizeof(float), st>>>(mask, loss_density, group_lasso, win_dev, grp_ss, H, W, unit);
}

// =====================================================================================
// K3 update: d/d pattern = m * c * g,  d/d mask = c * sum_ch (p-x) * g + density*dDen + coeff*dGL,
// with g = G + structured * dLs; then theta -= lr * sign(grad), clip.
// =====================================================================================
__global__ void __launch_bounds__(256) update_kernel(const float* __restrict__ x, float* __restrict__ mask,
                                                     float* __restrict__ pattern, const float* __restrict__ G,
                                                     const float* __restrict__ dLs, const float* __restrict__ scale,
                                                     const float* __restrict__ win_dev, const float* __restrict__ grp_ss,
                                                     const float* __restrict__ lr, const float* __restrict__ structured,
                                                     const float* __restrict__ coeff_gl, float density, float lo, float hi,
                                                     int stage, float* __restrict__ gp_out, float* __restrict__ gm_out,
                                                     const float* __restrict__ gp_bias, int H, int W, int unit) {
  const int b = blockIdx.y, HW = H * W;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= HW) return;
  const float c = scale[b], step = lr[b], st = structured[b];
  const float m = mask[(size_t)b * HW + i];
  float gm = 0.f;
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const size_t o = ((size_t)b * 3 + ch) * HW + i;
    float g = G[o];
    if (st != 0.f) g = fmaf(st, dLs[o], g);
    const float pv = pattern[o], xv = x[o];
    float gp = m * c * g;
    if (gp_bias != nullptr) gp = gp_bias[o] + gp;
    gm = fmaf((pv - xv) * c, g, gm);
    if (gp_out != nullptr) gp_out[o] = gp;
    if (step != 0.f) pattern[o] = fminf(fmaxf(pv - step * sgn(gp), lo), hi);
  }
  if (stage == 0) {
    const int h = i / W, w = i % W;
    const int win = W / 8;
    const float dden = win_dev[(size_t)b * 64 + (h / win) * (W / win) + (w / win)];
    const float ss = grp_ss[(size_t)b * (H / unit) * (W / unit) + (h / unit) * (W / unit) + (w / unit)];
    const float dgl = (float)unit * m / sqrtf(ss);     // 0/0 = NaN for an all-zero group (quirk Q5)
    if (density != 0.f) gm = fmaf(density, dden, gm);
    gm = fmaf(coeff_gl[b], dgl, gm);
    if (gm_out != nullptr) gm_out[(size_t)b * HW + i] = gm;
    if (step != 0.f) mask[(size_t)b * HW + i] = fminf(fmaxf(m - step * sgn(gm), lo), hi);
  }
}
void launch_update(const float* x, float* mask, float* pattern, const float* G, const float* dLs,
                   const float* scale, const float* win_dev, const float* grp_ss, const float* lr,
                   const float* structured, const float* coeff_gl, float density, float lo, float hi, int stage,
                   float* gp_out, float* gm_out, const float* gp_bias, int B, int H, int W, int unit, cudaStream_t st) {
  update_kernel<<<dim3((H * W + 255) / 256, B), 256, 0, st>>>(x, mask, pattern, G, dLs, scale, win_dev, grp_ss, lr,
                                                              structured, coeff_gl, density, lo, hi, stage, gp_out,
                                                              gm_out, gp_bias, H, W, unit);
}

// =====================================================================================
// k x k window sums (patch_selection's group importance, attack.py:365-368)
// =====================================================================================
__global__ void window_sum_kernel(const float* __restrict__ t, float* __restrict__ out, int H, int W, int k, int square) {
  const int b = blockIdx.y, GW = W / k, NG = (H / k) * GW;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= NG) return;
  const float* tb = t + (size_t)b * H * W;
  const int gy = g / GW, gx = g % GW;
  float s = 0.f;
  for (int dy = 0; dy < k; ++dy)
    for (int dx = 0; dx < k; ++dx) { const float v = tb[(gy * k + dy) * W + gx * k + dx]; s += square ? v * v : v; }
  out[(size_t)b * NG + g] = s;
}
void launch_window_sum(const float* t, float* out, int B, int H, int W, int k, bool square, cudaStream_t st) {
  const int NG = (H / k) * (W / k);
  window_sum_kernel<<<dim3((NG + 127) / 128, B), 128, 0, st>>>(t, out, H, W, k, square ? 1 : 0);
}

// =====================================================================================
// Failed-mask set on the device (SURVEY 8f N2; attack.py:259-267): per image a bitmap over the mask universe.
// One step's update: the first nff[b] sampled indices came from the failed set -- those whose sample now succeeds
// (loss < thresh) leave it; the remaining indices came from the whole universe -- those whose sample fails join it.
// Removal is applied before addition (the reference's setdiff1d precedes its unique), then the popcount is returned.
// One CTA per image; words = ceil(n_mask / 32).
// =====================================================================================
__global__ void failed_update_kernel(uint32_t* __restrict__ bits, int words, const int32_t* __restrict__ idx, const float* __restrict__ loss,
                                     const int32_t* __restrict__ nff, const uint8_t* __restrict__ active, int S, float thresh,
                                     int32_t* __restrict__ count) {
  const int b = blockIdx.x;
  uint32_t* w = bits + (size_t)b * words;
  __shared__ int red[32];
  if (active[b]) {
    const int n_ff = nff[b];
    for (int s = threadIdx.x; s < n_ff; s += blockDim.x)
      if (loss[(size_t)b * S + s] < thresh) { const int k = idx[(size_t)b * S + s]; atomicAnd(&w[k >> 5], ~(1u << (k & 31))); }
    __syncthreads();
    for (int s = n_ff + threadIdx.x; s < S; s += blockDim.x)
      if (!(loss[(size_t)b * S + s] < thresh)) { const int k = idx[(size_t)b * S + s]; atomicOr(&w[k >> 5], 1u << (k & 31)); }
    __syncthreads();
  }
  int c = 0;
  for (int i = threadIdx.x; i < words; i += blockDim.x) c += __popc(w[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { int t = 0; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i]; count[b] = t; }
}
void launch_failed_update(uint32_t* bits, int words, const int32_t* idx, const float* loss, const int32_t* nff, const uint8_t* active,
                          int B, int S, float thresh, int32_t* count, cudaStream_t st) {
  failed_update_kernel<<<B, 128, 0, st>>>(bits, words, idx, loss, nff, active, S, thresh, count);
}

}  // namespace dp
