// kernels_net.cu -- hand-written sm_100a kernels around the classifier's tensor-core
// convolutions: weight standardisation, GroupNorm(32)+ReLU forward / backward-to-input,
// pad+maxpool, head (GN+ReLU+avgpool, fc), layout packers.  All activations NHWC.
//
// Restates the third-party classifier the reference uses (timm 0.6.7
// resnetv2_50x1_bit_distilled, /root/reference/utils.py:51-58): StdConv2d eps=1e-8,
// GroupNormAct(32 groups, eps=1e-5, ReLU), stem 'fixed' (ConstantPad2d(1,0)+MaxPool 3x3/2).
// These kernels are HBM-bound; every one is a coalesced 16-byte-vector pass.
#include <cooperative_groups.h>

#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace dp {

#define DISPATCH_T(bf16, ...)                         \
  do {                                                \
    if (bf16) { using T = __nv_bfloat16; __VA_ARGS__; } \
    else { using T = float; __VA_ARGS__; }            \
  } while (0)

// ------------------------------------------------------------------------------------
// weight standardisation: one CTA per output channel
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void ws_kernel(const float* __restrict__ w, T* __restrict__ out, int I, int kh, int kw, int Ipad,
                          int standardize) {
  __shared__ float red[32];
  const int o = blockIdx.x, n = I * kh * kw;
  const float* wo = w + (size_t)o * n;
  float mean = 0.f, rstd = 1.f;
  if (standardize) {
    float s = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += wo[i];
    mean = block_sum(s, red) / n;
    float v = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { float d = wo[i] - mean; v += d * d; }
    const float var = block_sum(v, red) / n;   // biased, as F.batch_norm(training=True)
    rstd = 1.0f / sqrtf(var + 1e-8f);
  }
  T* oo = out + (size_t)o * kh * kw * Ipad;
  for (int i = threadIdx.x; i < kh * kw * Ipad; i += blockDim.x) {
    const int c = i % Ipad, rs = i / Ipad;
    float v = 0.f;
    if (c < I) v = (wo[(size_t)c * kh * kw + rs] - mean) * rstd;
    oo[i] = from_float<T>(v);
  }
}

void launch_weight_standardize(const float* w, void* out, int O, int I, int kh, int kw, int Ipad, bool bf16,
                               bool standardize, cudaStream_t st) {
  DISPATCH_T(bf16, (ws_kernel<T><<<O, 256, 0, st>>>(w, (T*)out, I, kh, kw, Ipad, standardize ? 1 : 0)));
}

// ------------------------------------------------------------------------------------
// NCHW fp32 <-> NHWC(Cp) T
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void pack_kernel(const float* __restrict__ z, T* __restrict__ out, int HW, int Cp, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t n = i / HW, p = i % HW;
  for (int c = 0; c < Cp; ++c) {
    float v = c < 3 ? z[(n * 3 + c) * HW + p] : 0.f;
    out[i * Cp + c] = from_float<T>(v);
  }
}
template <typename T>
__global__ void unpack_kernel(const T* __restrict__ in, float* __restrict__ dz, int HW, int Cp, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t n = i / HW, p = i % HW;
  for (int c = 0; c < 3; ++c) dz[(n * 3 + c) * HW + p] = to_float(in[i * Cp + c]);
}
void launch_pack_nchw(const float* z, void* out, int N, int H, int W, int Cp, bool bf16, cudaStream_t st) {
  size_t total = (size_t)N * H * W;
  DISPATCH_T(bf16, (pack_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(z, (T*)out, H * W, Cp, total)));
}
void launch_unpack_nhwc(const void* in, float* dz, int N, int H, int W, int Cp, bool bf16, cudaStream_t st) {
  size_t total = (size_t)N * H * W;
  DISPATCH_T(bf16, (unpack_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const T*)in, dz, H * W, Cp, total)));
}

// ------------------------------------------------------------------------------------
// GroupNorm machinery.
// A CTA of GN_THREADS threads walks a contiguous pixel slab of ONE sample.  Thread t owns
// vector column (t % cols) [cols = C/V 16-byte vectors per pixel] and pixel rows
// t/cols, t/cols + rpi, ...   When cols > GN_THREADS a thread owns several columns.
// Partial group sums are combined in a fixed order (deterministic, no float atomics).
// ------------------------------------------------------------------------------------
constexpr int GN_THREADS = 256;

int gn_splits(int P, int C, bool bf16) {
  const int V = bf16 ? 8 : 4;
  const int cols = C / V;
  const int rpi = cols >= GN_THREADS ? 1 : GN_THREADS / cols;   // pixel rows per iteration
  int s = P / (rpi * 4);                                        // >= 4 iterations per CTA
  if (s < 1) s = 1;
  if (s > GN_MAX_SPLITS) s = GN_MAX_SPLITS;
  return s;
}

// Per-thread accumulation of two per-channel quantities over the thread's pixels, then a
// deterministic CTA reduction to per-group sums.  F(px, vals_x[V], c0, acc_a[V], acc_b[V]).
template <typename T, typename F>
__device__ __forceinline__ void gn_reduce_slab(int P, int C, int split, int splits, float* __restrict__ out_partial,
                                               F&& body) {
  constexpr int V = Vec<T>::N;
  __shared__ float sm_a[GN_THREADS * V];
  __shared__ float sm_b[GN_THREADS * V];
  __shared__ float ch_a[2048];   // C <= 2048
  __shared__ float ch_b[2048];
  const int cols = C / V;
  const int p0 = (int)(((long long)P * split) / splits), p1 = (int)(((long long)P * (split + 1)) / splits);
  const int ncolblk = (cols + GN_THREADS - 1) / GN_THREADS;      // 1 or 2
  const int cpt = cols < GN_THREADS ? cols : GN_THREADS;         // columns covered per pass
  const int rpi = GN_THREADS / cpt;
  const int tcol = threadIdx.x % cpt, trow = threadIdx.x / cpt;
  for (int cb = 0; cb < ncolblk; ++cb) {
    const int col = cb * GN_THREADS + tcol;
    float a[V], b[V];
#pragma unroll
    for (int i = 0; i < V; ++i) { a[i] = 0.f; b[i] = 0.f; }
    if (col < cols)
      for (int p = p0 + trow; p < p1; p += rpi) body(p, col * V, a, b);
#pragma unroll
    for (int i = 0; i < V; ++i) { sm_a[threadIdx.x * V + i] = a[i]; sm_b[threadIdx.x * V + i] = b[i]; }
    __syncthreads();
    // channel totals: fixed-order sum over the rpi row-threads
    for (int ch = threadIdx.x; ch < cpt * V; ch += GN_THREADS) {
      const int c_col = ch / V, c_i = ch % V;
      float ta = 0.f, tb = 0.f;
      for (int r = 0; r < rpi; ++r) { ta += sm_a[(r * cpt + c_col) * V + c_i]; tb += sm_b[(r * cpt + c_col) * V + c_i]; }
      const int gch = cb * GN_THREADS * V + ch;
      if (gch < C) { ch_a[gch] = ta; ch_b[gch] = tb; }
    }
    __syncthreads();
  }
  const int cpg = C / GN_GROUPS;
  if (threadIdx.x < GN_GROUPS) {
    float ta = 0.f, tb = 0.f;
    for (int i = 0; i < cpg; ++i) { ta += ch_a[threadIdx.x * cpg + i]; tb += ch_b[threadIdx.x * cpg + i]; }
    out_partial[(split * GN_GROUPS + threadIdx.x) * 2 + 0] = ta;
    out_partial[(split * GN_GROUPS + threadIdx.x) * 2 + 1] = tb;
  }
}

template <typename T>
__global__ void __launch_bounds__(GN_THREADS) gn_stats_kernel(const T* __restrict__ x, float* __restrict__ partial,
                                                               int P, int C, int splits) {
  constexpr int V = Vec<T>::N;
  const int n = blockIdx.y, split = blockIdx.x;
  const T* xn = x + (size_t)n * P * C;
  gn_reduce_slab<T>(P, C, split, splits, partial + (size_t)n * splits * GN_GROUPS * 2,
                    [&](int p, int c0, float* a, float* b) {
                      Vec<T> v; v.load(xn + (size_t)p * C + c0);
                      float f[V]; v.unpack(f);
#pragma unroll
                      for (int i = 0; i < V; ++i) { a[i] += f[i]; b[i] += f[i] * f[i]; }
                    });
}

// finalise (mean, rstd) of sample n into shared memory from the split partials
__device__ __forceinline__ void gn_finalize(const float* __restrict__ partial_n, int splits, float count,
                                            float* s_mean, float* s_rstd) {
  if (threadIdx.x < GN_GROUPS) {
    float s = 0.f, q = 0.f;
    for (int k = 0; k < splits; ++k) {
      s += partial_n[(k * GN_GROUPS + threadIdx.x) * 2 + 0];
      q += partial_n[(k * GN_GROUPS + threadIdx.x) * 2 + 1];
    }
    const float mean = s / count;
    float var = q / count - mean * mean;
    var = var < 0.f ? 0.f : var;
    s_mean[threadIdx.x] = mean;
    s_rstd[threadIdx.x] = rsqrtf(var + 1e-5f);
  }
  __syncthreads();
}

template <typename T>
__global__ void gn_finalize_kernel(const float* __restrict__ partial, float* __restrict__ stats, int P, int C,
                                   int splits) {
  __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS];
  const int n = blockIdx.x;
  gn_finalize(partial + (size_t)n * splits * GN_GROUPS * 2, splits, (float)P * (C / GN_GROUPS), s_mean, s_rstd);
  if (threadIdx.x < GN_GROUPS) {
    stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 0] = s_mean[threadIdx.x];
    stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 1] = s_rstd[threadIdx.x];
  }
}

// y = relu(a*x + b), a = rstd*gamma, b = beta - mean*a.  grid (slabs, N).
template <typename T>
__global__ void __launch_bounds__(GN_THREADS) gn_apply_kernel(const T* __restrict__ x, T* __restrict__ y,
                                                               const float* __restrict__ gamma,
                                                               const float* __restrict__ beta,
                                                               const float* __restrict__ partial,
                                                               float* __restrict__ stats, int P, int C, int splits) {
  constexpr int V = Vec<T>::N;
  __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS];
  const int n = blockIdx.y;
  gn_finalize(partial + (size_t)n * splits * GN_GROUPS * 2, splits, (float)P * (C / GN_GROUPS), s_mean, s_rstd);
  if (blockIdx.x == 0 && threadIdx.x < GN_GROUPS) {
    stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 0] = s_mean[threadIdx.x];
    stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 1] = s_rstd[threadIdx.x];
  }
  const int cols = C / V, cpg = C / GN_GROUPS;
  const int p0 = (int)(((long long)P * blockIdx.x) / gridDim.x), p1 = (int)(((long long)P * (blockIdx.x + 1)) / gridDim.x);
  const int cpt = cols < GN_THREADS ? cols : GN_THREADS, rpi = GN_THREADS / cpt;
  const int tcol = threadIdx.x % cpt, trow = threadIdx.x / cpt;
  const T* xn = x + (size_t)n * P * C;
  T* yn = y + (size_t)n * P * C;
  for (int col = tcol; col < cols; col += cpt) {
    float a[V], b[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = col * V + i, g = c / cpg;
      a[i] = s_rstd[g] * gamma[c];
      b[i] = beta[c] - s_mean[g] * a[i];
    }
    for (int p = p0 + trow; p < p1; p += rpi) {
      Vec<T> v; v.load(xn + (size_t)p * C + col * V);
      float f[V]; v.unpack(f);
#pragma unroll
      for (int i = 0; i < V; ++i) f[i] = fmaxf(fmaf(a[i], f[i], b[i]), 0.f);
      v.pack(f); v.store(yn + (size_t)p * C + col * V);
    }
  }
}

static int apply_slabs(int P, int C, int V) {
  const int cols = C / V;
  const int cpt = cols < GN_THREADS ? cols : GN_THREADS, rpi = GN_THREADS / cpt;
  int s = P / (rpi * 4);
  if (s < 1) s = 1;
  if (s > 32) s = 32;
  return s;
}

static void launch_gn_stats_2pass(const void* x, float* partial, float* stats, int N, int P, int C, bool bf16, cudaStream_t st) {
  const int splits = gn_splits(P, C, bf16);
  DISPATCH_T(bf16, (gn_stats_kernel<T><<<dim3(splits, N), GN_THREADS, 0, st>>>((const T*)x, partial, P, C, splits)));
  DISPATCH_T(bf16, (gn_finalize_kernel<T><<<N, 32, 0, st>>>(partial, stats, P, C, splits)));
}

void launch_gn_relu_forward_2pass(const void* x, void* y, const float* gamma, const float* beta, float* partial,
                                  float* stats, int N, int P, int C, bool bf16, cudaStream_t st) {
  const int splits = gn_splits(P, C, bf16);
  DISPATCH_T(bf16, (gn_stats_kernel<T><<<dim3(splits, N), GN_THREADS, 0, st>>>((const T*)x, partial, P, C, splits)));
  DISPATCH_T(bf16, (gn_apply_kernel<T><<<dim3(apply_slabs(P, C, Vec<T>::N), N), GN_THREADS, 0, st>>>(
                       (const T*)x, (T*)y, gamma, beta, partial, stats, P, C, splits)));
}

// ---- backward -----------------------------------------------------------------------
// s1 = sum dyp*gamma, s2 = sum dyp*gamma*xhat over each (sample, group); dyp = dy * [a*x+b > 0]
template <typename T>
__global__ void __launch_bounds__(GN_THREADS) gn_bwd_reduce_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                                    const float* __restrict__ gamma,
                                                                    const float* __restrict__ beta,
                                                                    const float* __restrict__ stats,
                                                                    float* __restrict__ partial, int P, int C,
                                                                    int splits) {
  constexpr int V = Vec<T>::N;
  __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS];
  const int n = blockIdx.y, split = blockIdx.x;
  if (threadIdx.x < GN_GROUPS) {
    s_mean[threadIdx.x] = stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 0];
    s_rstd[threadIdx.x] = stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 1];
  }
  __syncthreads();
  const int cpg = C / GN_GROUPS;
  const T* xn = x + (size_t)n * P * C;
  const T* dyn = dy + (size_t)n * P * C;
  gn_reduce_slab<T>(P, C, split, splits, partial + (size_t)n * splits * GN_GROUPS * 2,
                    [&](int p, int c0, float* a, float* b) {
                      Vec<T> vx, vd; vx.load(xn + (size_t)p * C + c0); vd.load(dyn + (size_t)p * C + c0);
                      float fx[V], fd[V]; vx.unpack(fx); vd.unpack(fd);
#pragma unroll
                      for (int i = 0; i < V; ++i) {
                        const int c = c0 + i, g = c / cpg;
                        const float ga = gamma[c], sa = s_rstd[g] * ga, sb = beta[c] - s_mean[g] * sa;
                        const float pre = fmaf(sa, fx[i], sb);
                        const float dg = pre > 0.f ? fd[i] * ga : 0.f;
                        const float xh = (fx[i] - s_mean[g]) * s_rstd[g];
                        a[i] += dg; b[i] += dg * xh;
                      }
                    });
}

template <typename T>
__global__ void __launch_bounds__(GN_THREADS) gn_bwd_apply_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                                   const T* __restrict__ addend, T* __restrict__ dx,
                                                                   const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta,
                                                                   const float* __restrict__ stats,
                                                                   const float* __restrict__ partial, int P, int C,
                                                                   int splits) {
  constexpr int V = Vec<T>::N;
  __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS], s_1[GN_GROUPS], s_2[GN_GROUPS];
  const int n = blockIdx.y;
  if (threadIdx.x < GN_GROUPS) {
    s_mean[threadIdx.x] = stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 0];
    s_rstd[threadIdx.x] = stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 1];
    const float* pn = partial + (size_t)n * splits * GN_GROUPS * 2;
    float a = 0.f, b = 0.f;
    for (int k = 0; k < splits; ++k) { a += pn[(k * GN_GROUPS + threadIdx.x) * 2]; b += pn[(k * GN_GROUPS + threadIdx.x) * 2 + 1]; }
    const float inv_m = 1.0f / ((float)P * (C / GN_GROUPS));
    s_1[threadIdx.x] = a * inv_m;
    s_2[threadIdx.x] = b * inv_m;
  }
  __syncthreads();
  const int cols = C / V, cpg = C / GN_GROUPS;
  const int p0 = (int)(((long long)P * blockIdx.x) / gridDim.x), p1 = (int)(((long long)P * (blockIdx.x + 1)) / gridDim.x);
  const int cpt = cols < GN_THREADS ? cols : GN_THREADS, rpi = GN_THREADS / cpt;
  const int tcol = threadIdx.x % cpt, trow = threadIdx.x / cpt;
  const size_t base = (size_t)n * P * C;
  for (int col = tcol; col < cols; col += cpt) {
    float ga[V], sa[V], sb[V], mu[V], rs[V], m1[V], m2[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = col * V + i, g = c / cpg;
      ga[i] = gamma[c]; mu[i] = s_mean[g]; rs[i] = s_rstd[g];
      sa[i] = rs[i] * ga[i]; sb[i] = beta[c] - mu[i] * sa[i];
      m1[i] = s_1[g]; m2[i] = s_2[g];
    }
    for (int p = p0 + trow; p < p1; p += rpi) {
      const size_t off = base + (size_t)p * C + col * V;
      Vec<T> vx, vd; vx.load(x + off); vd.load(dy + off);
      float fx[V], fd[V], fo[V]; vx.unpack(fx); vd.unpack(fd);
      if (addend != nullptr) { Vec<T> va; va.load(addend + off); va.unpack(fo); }
      else {
#pragma unroll
        for (int i = 0; i < V; ++i) fo[i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const float pre = fmaf(sa[i], fx[i], sb[i]);
        const float dg = pre > 0.f ? fd[i] * ga[i] : 0.f;
        const float xh = (fx[i] - mu[i]) * rs[i];
        fo[i] += rs[i] * (dg - m1[i] - xh * m2[i]);
      }
      Vec<T> vo; vo.pack(fo); vo.store(dx + off);
    }
  }
}

void launch_gn_relu_backward_2pass(const void* dy, const void* x, const void* addend, void* dx, const float* gamma,
                                   const float* beta, const float* stats, float* partial, int N, int P, int C, bool bf16,
                                   cudaStream_t st) {
  const int splits = gn_splits(P, C, bf16);
  DISPATCH_T(bf16, (gn_bwd_reduce_kernel<T><<<dim3(splits, N), GN_THREADS, 0, st>>>(
                       (const T*)dy, (const T*)x, gamma, beta, stats, partial, P, C, splits)));
  DISPATCH_T(bf16, (gn_bwd_apply_kernel<T><<<dim3(apply_slabs(P, C, Vec<T>::N), N), GN_THREADS, 0, st>>>(
                       (const T*)dy, (const T*)x, (const T*)addend, (T*)dx, gamma, beta, stats, partial, P, C, splits)));
}

template <typename K, typename... Args>
static bool launch_cluster(K kernel, int cl, int nblocks, int threads, size_t smem, cudaStream_t st, Args... args) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (cl > 8) cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(nblocks);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...) == cudaSuccess;
}

// ------------------------------------------------------------------------------------
// ConstantPad2d(1, 0) + MaxPool2d(3, stride 2): first max in row-major window order wins
// (ATen: `val > maxval`), the zero padding is a real candidate.
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void maxpool_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int8_t* __restrict__ amax, int Hs,
                                   int Ws, int C, size_t total_vec) {
  constexpr int V = Vec<T>::N;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_vec) return;
  const int cols = C / V, Ho = Hs / 2, Wo = Ws / 2;
  const int col = (int)(i % cols);
  size_t r = i / cols;
  const int ox = (int)(r % Wo); r /= Wo;
  const int oy = (int)(r % Ho);
  const size_t n = r / Ho;
  float best[V]; int bi[V];
#pragma unroll
  for (int k = 0; k < V; ++k) { best[k] = -INFINITY; bi[k] = 0; }
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int yy = 2 * oy + ky - 1, xx = 2 * ox + kx - 1;   // unpadded coords
      float f[V];
      if (yy >= 0 && yy < Hs && xx >= 0 && xx < Ws) {
        Vec<T> v; v.load(x + ((n * Hs + yy) * Ws + xx) * (size_t)C + col * V); v.unpack(f);
      } else {
#pragma unroll
        for (int k = 0; k < V; ++k) f[k] = 0.f;
      }
#pragma unroll
      for (int k = 0; k < V; ++k)
        if (f[k] > best[k]) { best[k] = f[k]; bi[k] = ky * 3 + kx; }
    }
  Vec<T> o; o.pack(best); o.store(y + i * V);
  if (amax != nullptr) {   // V argmax bytes packed into one 4- / 8-byte store
    if (V == 8) {
      uint2 pk;
      pk.x = (uint32_t)bi[0] | ((uint32_t)bi[1] << 8) | ((uint32_t)bi[2] << 16) | ((uint32_t)bi[3] << 24);
      pk.y = (uint32_t)bi[4] | ((uint32_t)bi[5] << 8) | ((uint32_t)bi[6] << 16) | ((uint32_t)bi[7] << 24);
      *reinterpret_cast<uint2*>(amax + i * V) = pk;
    } else {
      uint32_t pk = 0;
#pragma unroll
      for (int k = 0; k < V; ++k) pk |= (uint32_t)bi[k] << (8 * k);
      *reinterpret_cast<uint32_t*>(amax + i * V) = pk;
    }
  }
}

template <typename T>
__global__ void maxpool_bwd_kernel(const T* __restrict__ dy, const int8_t* __restrict__ amax, T* __restrict__ dx,
                                   int Hs, int Ws, int C, size_t total_vec) {
  constexpr int V = Vec<T>::N;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_vec) return;
  const int cols = C / V, Ho = Hs / 2, Wo = Ws / 2;
  const int col = (int)(i % cols);
  size_t r = i / cols;
  const int xx = (int)(r % Ws); r /= Ws;
  const int yy = (int)(r % Hs);
  const size_t n = r / Hs;
  float acc[V];
#pragma unroll
  for (int k = 0; k < V; ++k) acc[k] = 0.f;
  // windows (oy, ox) with 2*oy - 1 <= yy <= 2*oy + 1
  for (int oy = (yy) / 2; oy <= (yy + 1) / 2; ++oy) {
    if (oy < 0 || oy >= Ho) continue;
    const int ky = yy - 2 * oy + 1;
    if (ky < 0 || ky > 2) continue;
    for (int ox = (xx) / 2; ox <= (xx + 1) / 2; ++ox) {
      if (ox < 0 || ox >= Wo) continue;
      const int kx = xx - 2 * ox + 1;
      if (kx < 0 || kx > 2) continue;
      const size_t o = (((n * Ho + oy) * Wo + ox) * (size_t)cols + col) * V;
      Vec<T> v; v.load(dy + o);
      float f[V]; v.unpack(f);
      const uint32_t want = (uint32_t)(ky * 3 + kx);
      if (V == 4) {                                         // fp32: the window's 4 argmax bytes in one 32-bit load (-10 %, measured)
        const uint32_t aw = __ldg(reinterpret_cast<const uint32_t*>(amax + o));
#pragma unroll
        for (int k = 0; k < V; ++k)
          if (((aw >> (8 * (k % 4))) & 0xffu) == want) acc[k] += f[k];
      } else {                                              // bf16: byte loads (a 64-bit load measured 20 % slower here)
#pragma unroll
        for (int k = 0; k < V; ++k)
          if ((uint32_t)(uint8_t)amax[o + k] == want) acc[k] += f[k];
      }
    }
  }
  Vec<T> out; out.pack(acc); out.store(dx + i * V);
}

void launch_maxpool_forward(const void* x, void* y, int8_t* amax, int N, int Hs, int Ws, int C, bool bf16,
                            cudaStream_t st) {
  DISPATCH_T(bf16, {
    size_t total = (size_t)N * (Hs / 2) * (Ws / 2) * (C / Vec<T>::N);
    maxpool_fwd_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const T*)x, (T*)y, amax, Hs, Ws, C, total);
  });
}
void launch_maxpool_backward(const void* dy, const int8_t* amax, void* dx, int N, int Hs, int Ws, int C, bool bf16,
                             cudaStream_t st) {
  DISPATCH_T(bf16, {
    size_t total = (size_t)N * Hs * Ws * (C / Vec<T>::N);
    maxpool_bwd_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const T*)dy, amax, (T*)dx, Hs, Ws, C, total);
  });
}

// ------------------------------------------------------------------------------------
// head
// ------------------------------------------------------------------------------------
// pooled[n][c] = (1/P) sum_p relu(a*x+b).  grid (C/(V*32), N), 32 column-threads x 8 row-threads
template <typename T>
__global__ void head_pool_kernel(const T* __restrict__ x, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, const float* __restrict__ stats,
                                 float* __restrict__ pooled, int P, int C) {
  constexpr int V = Vec<T>::N;
  __shared__ float sm[8][32][V];
  const int n = blockIdx.y, col = blockIdx.x * 32 + threadIdx.x, cpg = C / GN_GROUPS;
  float a[V], b[V], acc[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = col * V + i, g = c / cpg;
    const float mean = stats[((size_t)n * GN_GROUPS + g) * 2], rstd = stats[((size_t)n * GN_GROUPS + g) * 2 + 1];
    a[i] = rstd * gamma[c]; b[i] = beta[c] - mean * a[i]; acc[i] = 0.f;
  }
  for (int p = threadIdx.y; p < P; p += 8) {
    Vec<T> v; v.load(x + ((size_t)n * P + p) * C + col * V);
    float f[V]; v.unpack(f);
#pragma unroll
    for (int i = 0; i < V; ++i) acc[i] += fmaxf(fmaf(a[i], f[i], b[i]), 0.f);
  }
#pragma unroll
  for (int i = 0; i < V; ++i) sm[threadIdx.y][threadIdx.x][i] = acc[i];
  __syncthreads();
  if (threadIdx.y == 0) {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float t = 0.f;
      for (int r = 0; r < 8; ++r) t += sm[r][threadIdx.x][i];
      pooled[(size_t)n * C + col * V + i] = t / P;
    }
  }
}
void launch_head_pool(const void* x, const float* gamma, const float* beta, const float* stats, float* pooled,
                      int N, int P, int C, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, (head_pool_kernel<T><<<dim3(C / (Vec<T>::N * 32), N), dim3(32, 8), 0, st>>>(
                       (const T*)x, gamma, beta, stats, pooled, P, C)));
}

template <typename T>
__global__ void pool_grad_bcast_kernel(const float* __restrict__ dp, T* __restrict__ dy, int P, int C, size_t total_vec) {
  constexpr int V = Vec<T>::N;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_vec) return;
  const int cols = C / V, col = (int)(i % cols);
  const size_t n = i / cols / P;
  float f[V];
#pragma unroll
  for (int k = 0; k < V; ++k) f[k] = dp[n * C + col * V + k] / P;
  Vec<T> v; v.pack(f); v.store(dy + i * V);
}
void launch_pool_grad_bcast(const float* dpooled, void* dy, int N, int P, int C, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, {
    size_t total = (size_t)N * P * (C / Vec<T>::N);
    pool_grad_bcast_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(dpooled, (T*)dy, P, C, total);
  });
}

// ------------------------------------------------------------------------------------
// stride-2 spatial subsample (1x1 stride-2 shortcut conv = subsample + GEMM) and adjoint
// ------------------------------------------------------------------------------------
template <typename T>
__global__ void subsample2_kernel(const T* __restrict__ x, T* __restrict__ y, int H, int W, int C, size_t total_vec) {
  constexpr int V = Vec<T>::N;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_vec) return;
  const int cols = C / V, Ho = (H + 1) / 2, Wo = (W + 1) / 2, col = (int)(i % cols);
  size_t r = i / cols;
  const int ox = (int)(r % Wo); r /= Wo;
  const int oy = (int)(r % Ho);
  const size_t n = r / Ho;
  Vec<T> v; v.load(x + ((n * H + 2 * oy) * W + 2 * ox) * (size_t)C + col * V);
  v.store(y + i * V);
}
template <typename T>
__global__ void subsample2_adj_kernel(const T* __restrict__ dy, T* __restrict__ dx, int H, int W, int C, size_t total_vec) {
  constexpr int V = Vec<T>::N;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_vec) return;
  const int cols = C / V, Ho = (H + 1) / 2, Wo = (W + 1) / 2, col = (int)(i % cols);
  size_t r = i / cols;
  const int ox = (int)(r % Wo); r /= Wo;
  const int oy = (int)(r % Ho);
  const size_t n = r / Ho;
  T* dst = dx + ((n * H + 2 * oy) * W + 2 * ox) * (size_t)C + col * V;
  Vec<T> a, b; a.load(dy + i * V); b.load(dst);
  float fa[V], fb[V]; a.unpack(fa); b.unpack(fb);
#pragma unroll
  for (int k = 0; k < V; ++k) fb[k] += fa[k];
  b.pack(fb); b.store(dst);
}
void launch_subsample2(const void* x, void* y, int N, int H, int W, int C, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, {
    size_t total = (size_t)N * ((H + 1) / 2) * ((W + 1) / 2) * (C / Vec<T>::N);
    subsample2_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const T*)x, (T*)y, H, W, C, total);
  });
}
void launch_subsample2_adjoint_add(const void* dy, void* dx, int N, int H, int W, int C, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, {
    size_t total = (size_t)N * ((H + 1) / 2) * ((W + 1) / 2) * (C / Vec<T>::N);
    subsample2_adj_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const T*)dy, (T*)dx, H, W, C, total);
  });
}

// ====================================================================================
// GroupNorm v2, cluster per sample: ONE HBM read of the input.  A thread-block cluster of CL CTAs owns one sample;
// each CTA pulls its contiguous pixel slab into shared memory with TMA bulk copies (cp.async.bulk + mbarrier), reduces
// it to per-group partial sums, the cluster combines the partials through distributed shared memory in rank order
// (deterministic), and every CTA normalises its slab straight out of shared memory.  Shapes the plan below cannot
// place (slab too large, C/V > 256) run on the two-pass kernels above.
// Written against the round-1 cluster kernels (ncu: profiles/r02_gn_fwd_v1_ncu.txt, r02_gn_bwd_v1_ncu.txt): DRAM
// traffic = algorithmic, but 330 warp-instructions per 16-byte (x, dy) vector pair at IPC 1.5 -- 64-bit address
// arithmetic, per-row bound / chunk checks and per-element unpack + gate dominate; those kernels were issue-bound, not
// HBM-bound.  v2:
//   * a CTA's slab is a LINEAR array of 16-byte vectors; thread t owns vectors t, t + T, t + 2T, ... (its channel
//     column is fixed because T % (C/V) == 0), so the loops carry one 32-bit offset and no row / column arithmetic;
//   * the TMA load completes on one mbarrier per 32 KB chunk and the loops walk whole chunks (IPC iterations,
//     fully unrolled: IPC independent shared / global loads in flight per thread), tail handled once;
//   * bf16: unpack = 1 shift / 1 mask per element, ReLU folded into cvt.rn.relu.bf16x2.f32, the backward ReLU gate
//     is ONE packed compare (x > thr_c, thr_c = -sb/sa rounded DOWN to bf16 so that the test is exact on bf16
//     inputs) + one AND per element PAIR; channels with sa <= 0 take the generic fp32 gate (whole-kernel variant);
//   * backward statistics as sum(dy*gate) and sum(dy*gate*x) per channel (gamma, mean, rstd applied once per thread
//     after the loop); backward apply as dx = k1_c*dym + k2_g*x + k3_g: 2 FMA per element.
// Statistics and every sum stay fp32.
// ====================================================================================
namespace gn2 {
__device__ unsigned long long* g_trace = nullptr;   // optional phase trace (tools/gnbench.cu): [CTA][8] clock64 stamps
#define GN2_STAMP(i) do { if (g_trace != nullptr && threadIdx.x == 0) g_trace[(size_t)blockIdx.x * 8 + (i)] = clock64(); } while (0)
constexpr uint32_t CHUNK = 32768;
constexpr int MAX_CHUNKS = 7;                      // <= 224 KB per slab
constexpr int OFF_BAR_X = 0, OFF_BAR_D = 64, OFF_PART = 128, OFF_SA = 384, OFF_SB = 512, OFF_FLAG = 640;
constexpr size_t HDR = 1024;                       // the OFF_* fields above; the reduction scratch follows, then the slab(s)
constexpr int MAX_GPT = 4;                         // groups per thread (V / cpg when cpg < V)
__host__ __device__ constexpr size_t tp_bytes(int threads) { return (size_t)threads * MAX_GPT * 2 * sizeof(float); }

__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(uint32_t bar) { asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar)); }
__device__ __forceinline__ void bar_wait(uint32_t bar) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(0u)
        : "memory");
  }
}
// thread 0: one bulk copy + one mbarrier per 32 KB chunk of a contiguous slab
__device__ __forceinline__ void load_slab(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar0) {
  int k = 0;
  for (uint32_t off = 0; off < bytes; off += CHUNK, ++k) {
    const uint32_t nb = bytes - off < CHUNK ? bytes - off : CHUNK;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * k), "r"(nb) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + off),
                 "l"((const char*)src + off), "r"(nb), "r"(bar0 + 8 * k)
                 : "memory");
  }
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 ldg128(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ float blo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bhi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_relu(float lo, float hi) {   // {relu(hi), relu(lo)} -> bf16x2
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ uint32_t gt2_mask(uint32_t a, uint32_t b) {   // 0xffff per half where a > b (bf16x2)
  return __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
}
// largest bf16 <= t (as the high half of a float): x > t  <=>  x > floor_bf16(t) for every bf16 x
__device__ __forceinline__ uint32_t floor_bf16_bits(float t) {
  uint32_t u = __float_as_uint(t);
  if ((u & 0xffffu) != 0u && (u >> 31)) u += 0x10000u;   // negative: truncation rounds towards zero = up -> step one down
  return u >> 16;
}

template <typename T> struct Acc;   // per-vector math on the raw 16 bytes
template <> struct Acc<float> {
  static constexpr int V = 4;
  static __device__ __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y); f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
  }
  static __device__ __forceinline__ uint4 apply_relu(const uint4& v, const float* sa, const float* sb) {
    float f[4]; unpack(v, f);
    uint4 o;
    o.x = __float_as_uint(fmaxf(fmaf(sa[0], f[0], sb[0]), 0.f)); o.y = __float_as_uint(fmaxf(fmaf(sa[1], f[1], sb[1]), 0.f));
    o.z = __float_as_uint(fmaxf(fmaf(sa[2], f[2], sb[2]), 0.f)); o.w = __float_as_uint(fmaxf(fmaf(sa[3], f[3], sb[3]), 0.f));
    return o;
  }
  static __device__ __forceinline__ uint4 pack(const float* f) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
  }
};
template <> struct Acc<__nv_bfloat16> {
  static constexpr int V = 8;
  static __device__ __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = blo(v.x); f[1] = bhi(v.x); f[2] = blo(v.y); f[3] = bhi(v.y); f[4] = blo(v.z); f[5] = bhi(v.z); f[6] = blo(v.w); f[7] = bhi(v.w);
  }
  static __device__ __forceinline__ uint4 apply_relu(const uint4& v, const float* sa, const float* sb) {
    float f[8]; unpack(v, f);
    uint4 o;
    o.x = pack_relu(fmaf(sa[0], f[0], sb[0]), fmaf(sa[1], f[1], sb[1]));
    o.y = pack_relu(fmaf(sa[2], f[2], sb[2]), fmaf(sa[3], f[3], sb[3]));
    o.z = pack_relu(fmaf(sa[4], f[4], sb[4]), fmaf(sa[5], f[5], sb[5]));
    o.w = pack_relu(fmaf(sa[6], f[6], sb[6]), fmaf(sa[7], f[7], sb[7]));
    return o;
  }
  static __device__ __forceinline__ uint4 pack(const float* f) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
  }
};

// Deterministic CTA reduction of per-thread per-channel accumulators (a[V], b[V]) to the 32 per-group sums, for the
// linear thread -> column mapping (column = threadIdx.x % cols): fixed xor-shuffle tree inside each warp, one
// shared-memory exchange, fixed-order sum over the warps.  ~300 cycles; the shared-memory reduction loop of the round-1
// kernels (profiles/r02_gn_*_v1_ncu.txt) took 3-9k cycles per slab (tools/gnbench.cu phase trace).
// red: >= (blockDim/32) * 64 floats.
template <int V>
__device__ __forceinline__ void group_reduce(const float* a, const float* b, int C, float* red, float* part) {
  const int cols = C / V, cpg = C / GN_GROUPS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (int)blockDim.x >> 5;
  if (cpg <= V) {
    // each thread holds gpt = V / cpg whole groups; threads of one column sit `cols` lanes apart (cols <= 32)
    const int gpt = V / cpg;
    float sa[MAX_GPT], sb[MAX_GPT];
#pragma unroll
    for (int j = 0; j < MAX_GPT; ++j) {
      sa[j] = 0.f; sb[j] = 0.f;
#pragma unroll
      for (int i = 0; i < V; ++i)
        if (i / cpg == j) { sa[j] += a[i]; sb[j] += b[i]; }
    }
    for (int o = cols; o < 32; o <<= 1) {
#pragma unroll
      for (int j = 0; j < MAX_GPT; ++j) {
        sa[j] += __shfl_xor_sync(0xffffffffu, sa[j], o);
        sb[j] += __shfl_xor_sync(0xffffffffu, sb[j], o);
      }
    }
    __syncthreads();                                  // `red` may still be read by the previous use
    if (lane < cols) {
#pragma unroll
      for (int j = 0; j < MAX_GPT; ++j)
        if (j < gpt) { red[warp * 64 + (lane * gpt + j) * 2 + 0] = sa[j]; red[warp * 64 + (lane * gpt + j) * 2 + 1] = sb[j]; }
    }
    __syncthreads();
    if (threadIdx.x < 64) {
      float t = 0.f;
      for (int w = 0; w < nw; ++w) t += red[w * 64 + threadIdx.x];
      part[threadIdx.x] = t;
    }
  } else {
    // a group spans L = cpg / V consecutive columns = consecutive lanes; a pixel row spans cols / 32 = L warps
    const int L = cpg / V;
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) { sa += a[i]; sb += b[i]; }
    for (int o = 1; o < L; o <<= 1) {
      sa += __shfl_xor_sync(0xffffffffu, sa, o);
      sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
    __syncthreads();
    const int gpw = 32 / L;                           // groups per warp
    if ((lane & (L - 1)) == 0) { red[warp * 64 + (lane / L) * 2 + 0] = sa; red[warp * 64 + (lane / L) * 2 + 1] = sb; }
    __syncthreads();
    if (threadIdx.x < 64) {
      const int g = threadIdx.x >> 1, comp = threadIdx.x & 1;
      const int cb = (g * L) >> 5, slot = g % gpw;    // column block (warp index mod L) and slot inside the warp's row
      float t = 0.f;
      for (int w = cb; w < nw; w += L) t += red[w * 64 + slot * 2 + comp];
      part[threadIdx.x] = t;
    }
  }
}

// ---- statistics only (the tcgen05 GEMM applies GroupNorm+ReLU in its prologue; the classifier head) -----------------
// Streaming: grid (tiles, N), a CTA reads one contiguous 64 KB tile of one sample with the linear thread -> vector
// mapping (16 independent 16-byte loads per thread, two batches of 8 in flight), reduces to the 32 group sums and
// writes partial[n][tile][group][2]; gn_finalize_kernel adds the tiles in order (deterministic).
constexpr int ST_TH = 256, ST_ITER = 16, ST_TILE = ST_TH * ST_ITER;   // vectors per tile
template <typename T>
__global__ void __launch_bounds__(ST_TH) stats_kernel(const T* __restrict__ x, float* __restrict__ partial, int P, int C, int tiles) {
  using A = Acc<T>;
  constexpr int V = A::V;
  __shared__ float red[(ST_TH / 32) * 64];
  __shared__ float part[64];
  const int n = blockIdx.y, tile = blockIdx.x;
  const uint32_t nvec = (uint32_t)(((size_t)P * C) / V);
  const uint32_t v0 = (uint32_t)tile * ST_TILE;
  const uint4* src = reinterpret_cast<const uint4*>(x + (size_t)n * P * C) + v0 + threadIdx.x;
  const uint32_t left = nvec - v0;                                  // vectors from the tile start to the sample end
  float a[V], bq[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { a[i] = 0.f; bq[i] = 0.f; }
#pragma unroll
  for (int h = 0; h < ST_ITER / 8; ++h) {
    uint4 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t o = (uint32_t)(h * 8 + j) * ST_TH + threadIdx.x;
      v[j] = o < left ? __ldg(src + (h * 8 + j) * ST_TH) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float f[V]; A::unpack(v[j], f);
#pragma unroll
      for (int i = 0; i < V; ++i) { a[i] += f[i]; bq[i] = fmaf(f[i], f[i], bq[i]); }
    }
  }
  group_reduce<V>(a, bq, C, red, part);
  __syncthreads();
  if (threadIdx.x < 64) partial[((size_t)n * tiles + tile) * 64 + threadIdx.x] = part[threadIdx.x];
}

// ---- forward --------------------------------------------------------------------------------------
template <typename T, int TH>
__global__ void __launch_bounds__(TH, TH == 256 ? 2 : 1) fwd_kernel(const T* __restrict__ x, T* __restrict__ y,
                                                                    const float* __restrict__ gamma,
                                                                    const float* __restrict__ beta,
                                                                    float* __restrict__ stats, int P, int C) {
  using A = Acc<T>;
  constexpr int V = A::V;
  constexpr int IPC = (int)(CHUNK / (TH * 16));       // iterations per 32 KB chunk (8 / 4)
  extern __shared__ __align__(128) unsigned char smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const int n = blockIdx.x / CL;
  const uint32_t sb0 = s32(smem);
  float* part = reinterpret_cast<float*>(smem + OFF_PART);
  float* s_mean = reinterpret_cast<float*>(smem + OFF_SA);
  float* s_rstd = reinterpret_cast<float*>(smem + OFF_SB);
  float* tp = reinterpret_cast<float*>(smem + HDR);
  const uint32_t slab = sb0 + (uint32_t)(HDR + tp_bytes(TH));

  const int p0 = (int)(((long long)P * rank) / CL), p1 = (int)(((long long)P * (rank + 1)) / CL);
  const uint32_t slab_bytes = (uint32_t)((size_t)(p1 - p0) * C * sizeof(T));
  const size_t gbase = ((size_t)n * P + p0) * C * sizeof(T);          // byte offset of the slab in x / y
  GN2_STAMP(0);
  if (threadIdx.x == 0) {
    *reinterpret_cast<unsigned long long*>(smem + OFF_FLAG) = 0ull;
    for (int k = 0; k < MAX_CHUNKS; ++k) bar_init(sb0 + OFF_BAR_X + 8 * k);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    load_slab(slab, reinterpret_cast<const char*>(x) + gbase, slab_bytes, sb0 + OFF_BAR_X);
  }
  const int cols = C / V, cpg = C / GN_GROUPS;
  const int tcol = threadIdx.x % cols;
  const uint32_t nvec = slab_bytes >> 4;
  const uint32_t iters = nvec / TH, rem = nvec % TH;                  // thread t: vectors t + j*TH, j < iters (+1 if t < rem)
  const uint32_t full_chunks = iters / IPC;
  const uint32_t n_chunks = (slab_bytes + CHUNK - 1) / CHUNK;
  __syncthreads();                                                    // barrier inits visible before anyone polls

  float a[V], bq[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { a[i] = 0.f; bq[i] = 0.f; }
  uint32_t sp = slab + threadIdx.x * 16;
  for (uint32_t k = 0; k < full_chunks; ++k) {
    bar_wait(sb0 + OFF_BAR_X + 8 * k);
    uint4 v[IPC];
#pragma unroll
    for (int j = 0; j < IPC; ++j) v[j] = lds128(sp + j * TH * 16);
#pragma unroll
    for (int j = 0; j < IPC; ++j) {
      float f[V]; A::unpack(v[j], f);
#pragma unroll
      for (int i = 0; i < V; ++i) { a[i] += f[i]; bq[i] = fmaf(f[i], f[i], bq[i]); }
    }
    sp += IPC * TH * 16;
  }
  for (uint32_t k = full_chunks; k < n_chunks; ++k) bar_wait(sb0 + OFF_BAR_X + 8 * k);   // tail: everything has landed
  for (uint32_t j = full_chunks * IPC; j < iters + (threadIdx.x < rem ? 1u : 0u); ++j) {
    const uint4 v = lds128(slab + (j * TH + threadIdx.x) * 16);
    float f[V]; A::unpack(v, f);
#pragma unroll
    for (int i = 0; i < V; ++i) { a[i] += f[i]; bq[i] = fmaf(f[i], f[i], bq[i]); }
  }
  GN2_STAMP(1);
  if (g_trace != nullptr && (threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned long long*>(smem + OFF_FLAG), (unsigned long long)clock64());
  group_reduce<V>(a, bq, C, tp, part);
  if (g_trace != nullptr && threadIdx.x == 0) g_trace[(size_t)blockIdx.x * 8 + 2] = *reinterpret_cast<unsigned long long*>(smem + OFF_FLAG);   // slowest warp's loop end
  GN2_STAMP(3);
  cluster.sync();
  GN2_STAMP(4);
  if (threadIdx.x < GN_GROUPS) {
    float2 rv[16];                                                    // all ranks' partials in flight at once (DSMEM ~215 cycles each)
#pragma unroll
    for (int r = 0; r < 16; ++r)
      if (r < CL) rv[r] = *reinterpret_cast<const float2*>(cluster.map_shared_rank(part, r) + threadIdx.x * 2);
    float s = 0.f, q = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r)
      if (r < CL) { s += rv[r].x; q += rv[r].y; }
    const float cnt = (float)P * cpg;
    const float mean = s / cnt;
    float var = q / cnt - mean * mean;
    var = var < 0.f ? 0.f : var;
    const float rstd = rsqrtf(var + 1e-5f);
    s_mean[threadIdx.x] = mean;
    s_rstd[threadIdx.x] = rstd;
    if (rank == 0) {
      stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 0] = mean;
      stats[((size_t)n * GN_GROUPS + threadIdx.x) * 2 + 1] = rstd;
    }
  }
  __syncthreads();
  cluster.barrier_arrive();                                           // our remote reads are done
  float sa[V], sb[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = tcol * V + i, g = c / cpg;
    sa[i] = s_rstd[g] * gamma[c];
    sb[i] = beta[c] - s_mean[g] * sa[i];
  }
  GN2_STAMP(5);
  sp = slab + threadIdx.x * 16;
  char* dst = reinterpret_cast<char*>(y) + gbase + (size_t)threadIdx.x * 16;
  const uint32_t full_groups = iters / IPC;
  for (uint32_t k = 0; k < full_groups; ++k) {
    uint4 v[IPC];
#pragma unroll
    for (int j = 0; j < IPC; ++j) v[j] = lds128(sp + j * TH * 16);
#pragma unroll
    for (int j = 0; j < IPC; ++j) *reinterpret_cast<uint4*>(dst + j * TH * 16) = A::apply_relu(v[j], sa, sb);
    sp += IPC * TH * 16; dst += IPC * TH * 16;
  }
  for (uint32_t j = full_groups * IPC; j < iters + (threadIdx.x < rem ? 1u : 0u); ++j, sp += TH * 16, dst += TH * 16)
    *reinterpret_cast<uint4*>(dst) = A::apply_relu(lds128(sp), sa, sb);
  GN2_STAMP(6);
  cluster.barrier_wait();                                             // every peer has read our partials: we may exit
  GN2_STAMP(7);
}

// ---- backward -------------------------------------------------------------------------------------
// DYS: dy slab resident in shared memory (second TMA load) / streamed from global (twice; the second pass hits L2).
// NEG: generic fp32 ReLU gate (some channel has rstd*gamma <= 0); otherwise bf16 uses the packed threshold compare.
template <typename T, int TH, bool DYS, bool NEG>
__global__ void __launch_bounds__(TH, TH == 256 ? 2 : 1) bwd_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                                    const T* __restrict__ addend, T* __restrict__ dx,
                                                                    const float* __restrict__ gamma,
                                                                    const float* __restrict__ beta,
                                                                    const float* __restrict__ stats, int P, int C,
                                                                    uint32_t slab_stride) {
  using A = Acc<T>;
  constexpr int V = A::V;
  constexpr bool BF = sizeof(T) == 2;
  constexpr bool PACKED = BF && !NEG;                 // packed bf16 threshold gate
  constexpr int IPC = (int)(CHUNK / (TH * 16));
  constexpr int U = 4;                                 // vector pairs in flight per thread per trip
  extern __shared__ __align__(128) unsigned char smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const int n = blockIdx.x / CL;
  const uint32_t sb0 = s32(smem);
  float* part = reinterpret_cast<float*>(smem + OFF_PART);
  float* s_1 = reinterpret_cast<float*>(smem + OFF_SA);
  float* s_2 = reinterpret_cast<float*>(smem + OFF_SB);
  float* tp = reinterpret_cast<float*>(smem + HDR);
  const uint32_t xs = sb0 + (uint32_t)(HDR + tp_bytes(TH));
  const uint32_t ds = xs + slab_stride;

  const int p0 = (int)(((long long)P * rank) / CL), p1 = (int)(((long long)P * (rank + 1)) / CL);
  const uint32_t slab_bytes = (uint32_t)((size_t)(p1 - p0) * C * sizeof(T));
  const size_t gbase = ((size_t)n * P + p0) * C * sizeof(T);
  if (threadIdx.x == 0) {
    for (int k = 0; k < MAX_CHUNKS; ++k) { bar_init(sb0 + OFF_BAR_X + 8 * k); bar_init(sb0 + OFF_BAR_D + 8 * k); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    load_slab(xs, reinterpret_cast<const char*>(x) + gbase, slab_bytes, sb0 + OFF_BAR_X);
    if (DYS) load_slab(ds, reinterpret_cast<const char*>(dy) + gbase, slab_bytes, sb0 + OFF_BAR_D);
  }
  const int cols = C / V, cpg = C / GN_GROUPS;
  const int tcol = threadIdx.x % cols;
  const uint32_t nvec = slab_bytes >> 4;
  const uint32_t iters = nvec / TH, rem = nvec % TH;
  const uint32_t n_chunks = (slab_bytes + CHUNK - 1) / CHUNK;
  const uint32_t my_iters = iters + (threadIdx.x < rem ? 1u : 0u);

  // ReLU-gate constants (live through both passes): packed bf16 thresholds, or the fp32 scale / shift
  float sa[PACKED ? 1 : V], sbv[PACKED ? 1 : V];
  uint32_t thr[V / 2 > 0 ? V / 2 : 1];
  {
    float sa_[V], sb_[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = tcol * V + i, g = c / cpg;
      const float mean = stats[((size_t)n * GN_GROUPS + g) * 2 + 0], rstd = stats[((size_t)n * GN_GROUPS + g) * 2 + 1];
      sa_[i] = rstd * gamma[c];
      sb_[i] = beta[c] - mean * sa_[i];
    }
    if (PACKED) {
#pragma unroll
      for (int i = 0; i < V / 2; ++i) {
        // sa > 0 here (NEG variant otherwise): pre > 0  <=>  x > -sb/sa
        const uint32_t lo = floor_bf16_bits(-sb_[2 * i] / sa_[2 * i]), hi = floor_bf16_bits(-sb_[2 * i + 1] / sa_[2 * i + 1]);
        thr[i] = lo | (hi << 16);
      }
    } else {
#pragma unroll
      for (int i = 0; i < V; ++i) { sa[PACKED ? 0 : i] = sa_[i]; sbv[PACKED ? 0 : i] = sb_[i]; }
    }
  }
  __syncthreads();

  // gated dy of one vector: packed (bf16 words with the dead elements zeroed) or fp32
  auto gate = [&](const uint4& vx, const uint4& vd, float* fx, float* fd) {
    A::unpack(vx, fx);
    if (PACKED) {
      uint4 m;
      m.x = vd.x & gt2_mask(vx.x, thr[0]); m.y = vd.y & gt2_mask(vx.y, thr[1]);
      m.z = vd.z & gt2_mask(vx.z, thr[V / 2 > 2 ? 2 : 0]); m.w = vd.w & gt2_mask(vx.w, thr[V / 2 > 3 ? 3 : 0]);
      A::unpack(m, fd);
    } else {
      A::unpack(vd, fd);
#pragma unroll
      for (int i = 0; i < V; ++i) fd[i] = fmaf(sa[PACKED ? 0 : i], fx[i], sbv[PACKED ? 0 : i]) > 0.f ? fd[i] : 0.f;
    }
  };

  float a[V], bq[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { a[i] = 0.f; bq[i] = 0.f; }
  const char* dyg = reinterpret_cast<const char*>(dy) + gbase + (size_t)threadIdx.x * 16;
  {
    uint32_t j = 0;
    uint32_t have = 0;                                               // chunks [0, have) have landed
    for (; j + U <= my_iters; j += U) {
      const uint32_t need = ((j + U) * TH * 16 + CHUNK - 1) / CHUNK;   // chunks covering iterations [j, j+U)
      for (; have < need && have < n_chunks; ++have) { bar_wait(sb0 + OFF_BAR_X + 8 * have); if (DYS) bar_wait(sb0 + OFF_BAR_D + 8 * have); }
      uint4 vx[U], vd[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint32_t off = ((j + u) * TH + threadIdx.x) * 16;
        vd[u] = DYS ? lds128(ds + off) : ldg128(dyg + (size_t)(j + u) * TH * 16);
        vx[u] = lds128(xs + off);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float fx[V], fd[V]; gate(vx[u], vd[u], fx, fd);
#pragma unroll
        for (int i = 0; i < V; ++i) { a[i] += fd[i]; bq[i] = fmaf(fd[i], fx[i], bq[i]); }
      }
    }
    for (; have < n_chunks; ++have) { bar_wait(sb0 + OFF_BAR_X + 8 * have); if (DYS) bar_wait(sb0 + OFF_BAR_D + 8 * have); }
    for (; j < my_iters; ++j) {
      const uint32_t off = (j * TH + threadIdx.x) * 16;
      const uint4 vd = DYS ? lds128(ds + off) : ldg128(dyg + (size_t)j * TH * 16);
      const uint4 vx = lds128(xs + off);
      float fx[V], fd[V]; gate(vx, vd, fx, fd);
#pragma unroll
      for (int i = 0; i < V; ++i) { a[i] += fd[i]; bq[i] = fmaf(fd[i], fx[i], bq[i]); }
    }
  }
  // per channel: sum dg = gamma * A ; sum dg * xhat = gamma * rstd * (B - mean * A)
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = tcol * V + i, g = c / cpg;
    const float mean = stats[((size_t)n * GN_GROUPS + g) * 2 + 0], rstd = stats[((size_t)n * GN_GROUPS + g) * 2 + 1];
    const float ga = gamma[c], A_ = a[i];
    a[i] = ga * A_;
    bq[i] = rstd * ga * (bq[i] - mean * A_);
  }
  group_reduce<V>(a, bq, C, tp, part);
  cluster.sync();
  if (threadIdx.x < GN_GROUPS) {
    float2 rv[16];
#pragma unroll
    for (int r = 0; r < 16; ++r)
      if (r < CL) rv[r] = *reinterpret_cast<const float2*>(cluster.map_shared_rank(part, r) + threadIdx.x * 2);
    float s = 0.f, q = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r)
      if (r < CL) { s += rv[r].x; q += rv[r].y; }
    const float inv_m = 1.0f / ((float)P * cpg);
    s_1[threadIdx.x] = s * inv_m;
    s_2[threadIdx.x] = q * inv_m;
  }
  __syncthreads();
  cluster.barrier_arrive();
  // dx = rs*(dg - m1 - xhat*m2) = k1*dym + k2*x + k3
  float k1[V], k2[V], k3[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = tcol * V + i, g = c / cpg;
    const float mean = stats[((size_t)n * GN_GROUPS + g) * 2 + 0], rstd = stats[((size_t)n * GN_GROUPS + g) * 2 + 1];
    const float m1 = s_1[g], m2 = s_2[g];
    k1[i] = rstd * gamma[c];
    k2[i] = -rstd * rstd * m2;
    k3[i] = -rstd * m1 - k2[i] * mean;
  }
  char* dxg = reinterpret_cast<char*>(dx) + gbase + (size_t)threadIdx.x * 16;
  const char* adg = addend ? reinterpret_cast<const char*>(addend) + gbase + (size_t)threadIdx.x * 16 : nullptr;
  auto apply = [&](const uint4& vx, const uint4& vd, const uint4& va, bool has_add) -> uint4 {
    float fx[V], fd[V], fo[V];
    gate(vx, vd, fx, fd);
    if (has_add) A::unpack(va, fo);
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const float t = fmaf(k1[i], fd[i], fmaf(k2[i], fx[i], k3[i]));
      fo[i] = has_add ? fo[i] + t : t;
    }
    return A::pack(fo);
  };
  {
    constexpr int U2 = 4;
    uint32_t j = 0;
    const bool has_add = adg != nullptr;
    for (; j + U2 <= my_iters; j += U2) {
      uint4 vx[U2], vd[U2], va[U2];
#pragma unroll
      for (int u = 0; u < U2; ++u) {
        const uint32_t off = ((j + u) * TH + threadIdx.x) * 16;
        vd[u] = DYS ? lds128(ds + off) : ldg128(dyg + (size_t)(j + u) * TH * 16);
        if (has_add) va[u] = ldg128(adg + (size_t)(j + u) * TH * 16);
        vx[u] = lds128(xs + off);
      }
#pragma unroll
      for (int u = 0; u < U2; ++u)
        *reinterpret_cast<uint4*>(dxg + (size_t)(j + u) * TH * 16) = apply(vx[u], vd[u], va[u], has_add);
    }
    for (; j < my_iters; ++j) {
      const uint32_t off = (j * TH + threadIdx.x) * 16;
      const uint4 vd = DYS ? lds128(ds + off) : ldg128(dyg + (size_t)j * TH * 16);
      uint4 va = make_uint4(0u, 0u, 0u, 0u);
      if (has_add) va = ldg128(adg + (size_t)j * TH * 16);
      *reinterpret_cast<uint4*>(dxg + (size_t)j * TH * 16) = apply(lds128(xs + off), vd, va, has_add);
    }
  }
  cluster.barrier_wait();
}

// any channel with rstd*gamma <= 0 needs the generic gate; gamma is constant per layer -> cached per pointer
struct Plan { int cl, threads; bool dys; size_t smem; uint32_t stride; };
}  // namespace gn2

void gn2_set_trace(unsigned long long* dev_ptr) { cudaMemcpyToSymbol(gn2::g_trace, &dev_ptr, sizeof(dev_ptr)); }

// v2 plan limits, chosen by the round-2 sweeps (tools/r2_batch2.sh, r2_batch14.sh): the largest cluster (16 needs the
// non-portable size), the shared memory per CTA that still fits two CTAs per SM, the most one CTA may take, and whether a
// backward CTA that has an SM to itself also keeps its dy slab in shared memory
constexpr int GN2_MAX_CLUSTER = 16;
constexpr size_t GN2_SOFT = 111 * 1024, GN2_HARD = 224 * 1024;
constexpr bool GN2_DYS_BIG = true;
// forward: smallest cluster whose slab leaves room for two CTAs per SM (256 threads), else one 512-thread CTA per SM
static bool gn2_plan_fwd(int P, int C, size_t es, gn2::Plan* pl) {
  const int V = (int)(16 / es);
  if (C % (V * 1) != 0 || (C / V) > 256 || 256 % (C / V) != 0) return false;
  const size_t f256 = gn2::HDR + gn2::tp_bytes(256), f512 = gn2::HDR + gn2::tp_bytes(512);
  for (int cl = 1; cl <= GN2_MAX_CLUSTER; cl *= 2) {
    if (cl > P) break;
    const size_t slab = (((size_t)((P + cl - 1) / cl)) * C * es + 127) / 128 * 128;
    if (slab > gn2::MAX_CHUNKS * (size_t)gn2::CHUNK) continue;
    if (f256 + slab <= GN2_SOFT) { *pl = gn2::Plan{cl, 256, false, f256 + slab, (uint32_t)slab}; return true; }
  }
  for (int cl = 1; cl <= GN2_MAX_CLUSTER; cl *= 2) {
    if (cl > P) break;
    const size_t slab = (((size_t)((P + cl - 1) / cl)) * C * es + 127) / 128 * 128;
    if (slab > gn2::MAX_CHUNKS * (size_t)gn2::CHUNK) continue;
    if (f512 + slab <= GN2_HARD && 512 % (C / V) == 0) { *pl = gn2::Plan{cl, 512, false, f512 + slab, (uint32_t)slab}; return true; }
  }
  return false;
}
// backward: both slabs resident when they fit (two CTAs per SM, else one), else x resident + dy streamed
static bool gn2_plan_bwd(int P, int C, size_t es, gn2::Plan* pl) {
  const int V = (int)(16 / es);
  if ((C / V) > 256 || 256 % (C / V) != 0) return false;
  const size_t f256 = gn2::HDR + gn2::tp_bytes(256), f512 = gn2::HDR + gn2::tp_bytes(512);
  for (int cl = 1; cl <= GN2_MAX_CLUSTER; cl *= 2) {
    if (cl > P) break;
    const size_t slab = (((size_t)((P + cl - 1) / cl)) * C * es + 127) / 128 * 128;
    if (f256 + 2 * slab <= GN2_SOFT) { *pl = gn2::Plan{cl, 256, true, f256 + 2 * slab, (uint32_t)slab}; return true; }
  }
  if (GN2_DYS_BIG)
    for (int cl = 1; cl <= GN2_MAX_CLUSTER; cl *= 2) {
      if (cl > P) break;
      const size_t slab = (((size_t)((P + cl - 1) / cl)) * C * es + 127) / 128 * 128;
      if (f512 + 2 * slab <= GN2_HARD && 512 % (C / V) == 0) { *pl = gn2::Plan{cl, 512, true, f512 + 2 * slab, (uint32_t)slab}; return true; }
    }
  gn2::Plan f;
  if (!gn2_plan_fwd(P, C, es, &f)) return false;
  *pl = f;
  pl->dys = false;
  return true;
}

static bool launch_gn2_forward(const void* x, void* y, const float* gamma, const float* beta, float* stats, int N, int P,
                               int C, bool bf16, cudaStream_t st) {
  gn2::Plan pl;
  if (!gn2_plan_fwd(P, C, bf16 ? 2 : 4, &pl)) return false;
#define GN2F(TT, TH) launch_cluster(gn2::fwd_kernel<TT, TH>, pl.cl, pl.cl * N, TH, pl.smem, st, (const TT*)x, (TT*)y, gamma, beta, stats, P, C)
  bool ok;
  if (bf16) ok = pl.threads == 256 ? GN2F(__nv_bfloat16, 256) : GN2F(__nv_bfloat16, 512);
  else ok = pl.threads == 256 ? GN2F(float, 256) : GN2F(float, 512);
#undef GN2F
  if (!ok) cudaGetLastError();
  return ok;
}

static bool launch_gn2_backward(const void* dy, const void* x, const void* addend, void* dx, const float* gamma,
                                const float* beta, const float* stats, int N, int P, int C, bool bf16, bool gamma_pos, cudaStream_t st) {
  gn2::Plan pl;
  if (!gn2_plan_bwd(P, C, bf16 ? 2 : 4, &pl)) return false;
  const bool neg = bf16 ? !gamma_pos : true;   // fp32 always uses the fp32 gate
#define GN2B(TT, TH, DYS, NEG) launch_cluster(gn2::bwd_kernel<TT, TH, DYS, NEG>, pl.cl, pl.cl * N, TH, pl.smem, st, (const TT*)dy, (const TT*)x, (const TT*)addend, (TT*)dx, gamma, beta, stats, P, C, pl.stride)
#define GN2B_T(TT, NEG) (pl.threads == 256 ? (pl.dys ? GN2B(TT, 256, true, NEG) : GN2B(TT, 256, false, NEG)) : (pl.dys ? GN2B(TT, 512, true, NEG) : GN2B(TT, 512, false, NEG)))
  bool ok;
  if (bf16) ok = neg ? GN2B_T(__nv_bfloat16, true) : GN2B_T(__nv_bfloat16, false);
  else ok = GN2B_T(float, true);
#undef GN2B_T
#undef GN2B
  if (!ok) cudaGetLastError();
  return ok;
}

void launch_gn_relu_forward(const void* x, void* y, const float* gamma, const float* beta, float* partial,
                            float* stats, int N, int P, int C, bool bf16, cudaStream_t st) {
  if (launch_gn2_forward(x, y, gamma, beta, stats, N, P, C, bf16, st)) return;
  launch_gn_relu_forward_2pass(x, y, gamma, beta, partial, stats, N, P, C, bf16, st);
}

void launch_gn_relu_backward(const void* dy, const void* x, const void* addend, void* dx, const float* gamma,
                             const float* beta, const float* stats, float* partial, int N, int P, int C, bool bf16,
                             cudaStream_t st, bool gamma_pos) {
  if (launch_gn2_backward(dy, x, addend, dx, gamma, beta, stats, N, P, C, bf16, gamma_pos, st)) return;
  launch_gn_relu_backward_2pass(dy, x, addend, dx, gamma, beta, stats, partial, N, P, C, bf16, st);
}

void launch_gn_stats(const void* x, float* partial, float* stats, int N, int P, int C, bool bf16, cudaStream_t st) {
  const int V = bf16 ? 8 : 4, cols = C / V;
  const size_t nvec = (size_t)P * cols;
  const int tiles = (int)((nvec + gn2::ST_TILE - 1) / gn2::ST_TILE);
  if (cols <= gn2::ST_TH && gn2::ST_TH % cols == 0 && C % V == 0 && tiles * 64 <= GN_WS_FLOATS_PER_SAMPLE) {
    DISPATCH_T(bf16, (gn2::stats_kernel<T><<<dim3(tiles, N), gn2::ST_TH, 0, st>>>((const T*)x, partial, P, C, tiles)));
    DISPATCH_T(bf16, (gn_finalize_kernel<T><<<N, 32, 0, st>>>(partial, stats, P, C, tiles)));
    return;
  }
  launch_gn_stats_2pass(x, partial, stats, N, P, C, bf16, st);
}

}  // namespace dp
