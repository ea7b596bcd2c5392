// gnbench.cu -- correctness + bandwidth of the GroupNorm(32)+ReLU forward / backward launchers of libdorpatch.so on
// every (pixels, channels) shape ResNetV2-50 uses at 224 px, fp32 and bf16, against a double-precision CPU
// restatement of timm's GroupNormAct (torch.nn.functional.group_norm + relu, eps 1e-5) and its input gradient.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o gnbench tools/gnbench.cu \
//        -Ldorpatch_b200/lib -ldorpatch -Xlinker -rpath,$PWD/dorpatch_b200/lib
//   ./gnbench [N] [only_C]
// Buffers rotate over > 300 MB so that no launch finds its operands in the 126 MB L2.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../dorpatch_b200/csrc/kernels.h"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA %s at %d: %s\n", #x, __LINE__, cudaGetErrorString(e_)); exit(1); } } while (0)

static float bf16r(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

struct Lcg { uint64_t s; float next() { s = s * 6364136223846793005ull + 1442695040888963407ull; return (float)((s >> 40) & 0xffffff) / 8388608.0f - 1.0f; } };

template <typename T> static void fill(std::vector<T>& h, size_t n, Lcg& g, float scale, float shift);
template <> void fill<float>(std::vector<float>& h, size_t n, Lcg& g, float scale, float shift) { h.resize(n); for (auto& v : h) v = g.next() * scale + shift; }
template <> void fill<__nv_bfloat16>(std::vector<__nv_bfloat16>& h, size_t n, Lcg& g, float scale, float shift) { h.resize(n); for (auto& v : h) v = __float2bfloat16_rn(g.next() * scale + shift); }
static double tof(float v) { return v; }
static double tof(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
static void run_shape(int N, int P, int C, bool bf16, bool negative_gamma) {
  const size_t per = (size_t)P * C, bytes = (size_t)N * per * sizeof(T);
  int R = (int)((320ull << 20) / bytes) + 1;
  if (R > 24) R = 24;
  Lcg g{(uint64_t)(P * 131 + C)};
  // one sample-pattern repeated (the CPU check only looks at samples 0 and N-1 of copy 0); shift != 0 exercises the mean
  std::vector<T> hx, hdy, had;
  fill<T>(hx, (size_t)N * per, g, 1.5f, 0.7f);
  fill<T>(hdy, (size_t)N * per, g, 1.0f, 0.05f);
  fill<T>(had, (size_t)N * per, g, 0.5f, 0.0f);
  std::vector<float> hga(C), hbe(C);
  for (int c = 0; c < C; ++c) { hga[c] = 1.0f + 0.3f * g.next(); hbe[c] = 0.3f * g.next(); }
  if (negative_gamma) { hga[1] = -0.5f; hga[C - 3] = 0.0f; }
  T *x, *dy, *ad, *y, *dx;
  float *ga, *be, *stats, *partial;
  CK(cudaMalloc(&x, bytes * R)); CK(cudaMalloc(&dy, bytes * R)); CK(cudaMalloc(&ad, bytes * R));
  CK(cudaMalloc(&y, bytes * R)); CK(cudaMalloc(&dx, bytes * R));
  CK(cudaMalloc(&ga, C * 4)); CK(cudaMalloc(&be, C * 4)); CK(cudaMalloc(&stats, (size_t)N * 64 * 4));
  CK(cudaMalloc(&partial, ((size_t)N * dp::GN_WS_FLOATS_PER_SAMPLE + dp::GN_WS_FLOATS_EXTRA) * 4));
  for (int r = 0; r < R; ++r) {
    CK(cudaMemcpy((char*)x + bytes * r, hx.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy((char*)dy + bytes * r, hdy.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy((char*)ad + bytes * r, had.data(), bytes, cudaMemcpyHostToDevice));
  }
  CK(cudaMemcpy(ga, hga.data(), C * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(be, hbe.data(), C * 4, cudaMemcpyHostToDevice));
  cudaStream_t st; CK(cudaStreamCreate(&st));
  auto fwd = [&](int r) { dp::launch_gn_relu_forward((char*)x + bytes * r, (char*)y + bytes * r, ga, be, partial, stats, N, P, C, bf16, st); };
  auto bwd = [&](int r, bool add) {
    dp::launch_gn_relu_backward((char*)dy + bytes * r, (char*)x + bytes * r, add ? (char*)ad + bytes * r : nullptr, (char*)dx + bytes * r, ga, be,
                                stats, partial, N, P, C, bf16, st, !negative_gamma);
  };
  // ---- correctness (copy 0, samples 0 and N-1) ----
  fwd(0); CK(cudaGetLastError());
  bwd(0, true); CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st));
  std::vector<T> hy((size_t)N * per), hdx((size_t)N * per);
  CK(cudaMemcpy(hy.data(), y, bytes, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hdx.data(), dx, bytes, cudaMemcpyDeviceToHost));
  double ey = 0, edx = 0, my = 0, mdx = 0;
  const int cpg = C / 32;
  for (int n : {0, N - 1}) {
    const T* xs = hx.data() + (size_t)n * per; const T* ds = hdy.data() + (size_t)n * per; const T* as = had.data() + (size_t)n * per;
    for (int gq = 0; gq < 32; ++gq) {
      double s = 0, q = 0;
      for (int p = 0; p < P; ++p) for (int c = gq * cpg; c < (gq + 1) * cpg; ++c) { const double v = tof(xs[(size_t)p * C + c]); s += v; q += v * v; }
      const double cnt = (double)P * cpg, mean = s / cnt, var = q / cnt - mean * mean, rstd = 1.0 / sqrt(var + 1e-5);
      double s1 = 0, s2 = 0;
      for (int p = 0; p < P; ++p) for (int c = gq * cpg; c < (gq + 1) * cpg; ++c) {
        const double v = tof(xs[(size_t)p * C + c]), xh = (v - mean) * rstd, pre = xh * hga[c] + hbe[c];
        const double dg = pre > 0 ? tof(ds[(size_t)p * C + c]) * hga[c] : 0.0;
        s1 += dg; s2 += dg * xh;
      }
      s1 /= cnt; s2 /= cnt;
      for (int p = 0; p < P; ++p) for (int c = gq * cpg; c < (gq + 1) * cpg; ++c) {
        const size_t i = (size_t)p * C + c;
        const double v = tof(xs[i]), xh = (v - mean) * rstd, pre = xh * hga[c] + hbe[c];
        const double yr = pre > 0 ? pre : 0.0;
        const double dg = pre > 0 ? tof(ds[i]) * hga[c] : 0.0;
        const double dr = rstd * (dg - s1 - xh * s2) + tof(as[i]);
        const double yg = tof(hy[(size_t)n * per + i]), dgp = tof(hdx[(size_t)n * per + i]);
        // elements whose pre-activation is within rounding of zero may legitimately gate differently
        if (fabs(pre) > 1e-3) { ey = fmax(ey, fabs(yg - yr)); edx = fmax(edx, fabs(dgp - dr)); }
        my = fmax(my, fabs(yr)); mdx = fmax(mdx, fabs(dr));
      }
    }
  }
  const double tol = bf16 ? 1.0 / 128 : 2e-5;
  const bool ok = ey <= tol * my && edx <= tol * mdx;
  // ---- timing ----
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  auto time_it = [&](auto&& f) {
    for (int r = 0; r < R; ++r) f(r);
    CK(cudaStreamSynchronize(st));
    const int reps = 3 * R;
    CK(cudaEventRecord(e0, st));
    for (int i = 0; i < reps; ++i) f(i % R);
    CK(cudaEventRecord(e1, st));
    CK(cudaEventSynchronize(e1));
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    return ms / reps;
  };
  if (getenv("GNBENCH_TRACE")) {   // phase attribution of the v2 forward kernel: mean cycles between the stamps over all CTAs
    const size_t max_ctas = (size_t)N * 16;
    unsigned long long* tr; CK(cudaMalloc(&tr, max_ctas * 8 * 8)); CK(cudaMemset(tr, 0, max_ctas * 8 * 8));
    for (int r = 0; r < R; ++r) fwd(r);
    CK(cudaStreamSynchronize(st));
    dp::gn2_set_trace(tr);
    fwd(0);
    CK(cudaStreamSynchronize(st));
    dp::gn2_set_trace(nullptr);
    std::vector<unsigned long long> h(max_ctas * 8);
    CK(cudaMemcpy(h.data(), tr, max_ctas * 8 * 8, cudaMemcpyDeviceToHost));
    double d[7] = {0, 0, 0, 0, 0, 0, 0}; size_t cnt = 0;
    unsigned long long tmin = ~0ull, tmax = 0;
    for (size_t c = 0; c < max_ctas; ++c) {
      if (h[c * 8 + 7] == 0) continue;
      for (int i = 0; i < 7; ++i) d[i] += (double)((long long)h[c * 8 + i + 1] - (long long)h[c * 8 + i]);
      ++cnt;
    }
    if (cnt) printf("  trace (%zu CTAs, mean cycles): load+stats, thread 0 %.0f | slowest warp later by %.0f | cta-reduce %.0f | cluster.sync %.0f | finalize %.0f | apply+store %.0f | exit-wait %.0f | total %.0f\n",
                    cnt, d[0] / cnt, d[1] / cnt, d[2] / cnt, d[3] / cnt, d[4] / cnt, d[5] / cnt, d[6] / cnt, (d[0] + d[1] + d[2] + d[3] + d[4] + d[5] + d[6]) / cnt);
    cudaFree(tr);
  }
  const float tf = time_it([&](int r) { fwd(r); });
  const float tb = time_it([&](int r) { bwd(r, false); });
  const float tba = time_it([&](int r) { bwd(r, true); });
  CK(cudaGetLastError());
  printf("%s P=%4d C=%4d N=%d %s| fwd %7.3f ms %5.0f GB/s | bwd %7.3f ms %5.0f GB/s | bwd+add %7.3f ms %5.0f GB/s | err y %.2e dx %.2e (rel) %s\n",
         bf16 ? "bf16" : "fp32", P, C, N, negative_gamma ? "NEG " : "", tf, 2.0 * bytes / tf / 1e6, tb, 3.0 * bytes / tb / 1e6, tba, 4.0 * bytes / tba / 1e6,
         ey / my, edx / mdx, ok ? "OK" : "MISMATCH");
  fflush(stdout);
  cudaFree(x); cudaFree(dy); cudaFree(ad); cudaFree(y); cudaFree(dx); cudaFree(ga); cudaFree(be); cudaFree(stats); cudaFree(partial);
  cudaStreamDestroy(st); cudaEventDestroy(e0); cudaEventDestroy(e1);
}

int main(int argc, char** argv) {
  const int N = argc > 1 ? atoi(argv[1]) : 256;
  const int only_c = argc > 2 ? atoi(argv[2]) : 0;
  const int shapes[][2] = {{3136, 64}, {3136, 256}, {3136, 128}, {784, 128}, {784, 512}, {784, 256}, {196, 256}, {196, 1024}, {196, 512}, {49, 512}, {49, 2048}};
  const char* dt = getenv("GNBENCH_DTYPE");
  for (int pass = 0; pass < 2; ++pass) {
    const bool bf16 = pass == 0;
    if (dt && ((bf16 && dt[0] != 'b') || (!bf16 && dt[0] != 'f'))) continue;
    for (auto& s : shapes) {
      if (only_c && s[1] != only_c) continue;
      if (bf16) run_shape<__nv_bfloat16>(N, s[0], s[1], true, false);
      else run_shape<float>(N, s[0], s[1], false, false);
    }
    if (bf16) { run_shape<__nv_bfloat16>(N > 32 ? 32 : N, 784, 128, true, true); run_shape<__nv_bfloat16>(N > 32 ? 32 : N, 3136, 256, true, true); }
  }
  return 0;
}
