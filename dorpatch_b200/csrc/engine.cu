// engine.cu -- the DorPatch hot-path engine behind include/dorpatch.h.
//
// One engine per GPU.  It owns: the standardised classifier weights (ResNetV2-50x1-BiT,
// NHWC/KRSC), a workspace arena sized for `chunk` EOT samples, cuDNN + cublasLt handles.
// The classifier's 3x3 / 7x7 convolutions run on tensor cores through cuDNN, the 1x1
// convolutions (36 of 53) are plain NHWC GEMMs through cublasLt (the residual add is fused
// as the GEMM's C operand); everything else is the hand-written kernels of kernels_*.cu.
// Backward is data-gradient only (the weights are frozen during the attack; the reference's
// unused weight-gradient, SURVEY quirk Q7, is not computed).
#include <cublasLt.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cudnn.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: no-ops unless a profiler injects itself (ncu --nvtx, nsys)

#include "../../include/dorpatch.h"
#include "kernels.h"

namespace {

thread_local std::string g_last_error;

[[noreturn]] void fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  throw std::runtime_error(buf);
}

#define CUDA_OK(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) fail("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__, cudaGetErrorString(_e)); \
  } while (0)
#define CUDNN_OK(expr)                                                                             \
  do {                                                                                             \
    cudnnStatus_t _s = (expr);                                                                     \
    if (_s != CUDNN_STATUS_SUCCESS) fail("cuDNN error %d (%s) at %s:%d [%s]", (int)_s, cudnnGetErrorString(_s), __FILE__, __LINE__, #expr); \
  } while (0)
#define CUBLAS_OK(expr)                                                                            \
  do {                                                                                             \
    cublasStatus_t _s = (expr);                                                                    \
    if (_s != CUBLAS_STATUS_SUCCESS) fail("cuBLASLt error %d at %s:%d [%s]", (int)_s, __FILE__, __LINE__, #expr); \
  } while (0)
#define KERNEL_OK() CUDA_OK(cudaGetLastError())
// PROF(engine, "category", algorithmic bytes, flops, stream, statement)
#define PROF(E, NAME, BYTES, FLOPS, ST, ...) \
  do { (E)->prof_begin(NAME, (double)(BYTES), (double)(FLOPS), ST); __VA_ARGS__; (E)->prof_end(ST); } while (0)

constexpr int DEPTHS[4] = {3, 4, 6, 3};
constexpr int WIDTHS[4] = {256, 512, 1024, 2048};
constexpr int STEM_CH = 64;
constexpr int STEM_SUB = 128;   // samples per cuDNN stem-conv call
// NVTX range around the phases of the hot loop (host side; inside a graph capture they mark the capture, not the replay)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

constexpr int UNIT = 7;   // basic_unit of the group lasso / patch selection (attack.py:52)

struct ConvW {            // one convolution's weights (device, KRSC, activation dtype)
  int cin = 0, cin_pad = 0, cout = 0, k = 1, stride = 1, pad = 0;
  void* w = nullptr;
  cudnnFilterDescriptor_t wdesc = nullptr;
  cudnnConvolutionDescriptor_t cdesc = nullptr;
};
struct GNW { int C = 0; float* gamma = nullptr; float* beta = nullptr; bool pos = false; };   // pos: every gamma > 0 (packed bf16 ReLU gate allowed)
struct Block {
  int cin, mid, cout, stride, hin, hout;
  bool has_ds;
  GNW n1, n2, n3;
  ConvW ds, c1, c2, c3;
  // saved tensors / stats for backward (device, per chunk)
  void* h1 = nullptr; void* h2 = nullptr; void* out = nullptr;
  float* st1 = nullptr; float* st2 = nullptr; float* st3 = nullptr;
  void* c1p = nullptr; void* c3p = nullptr;   // conv1 / conv3 weights as tcgen05 operand tiles (DORPATCH_FUSED_GEMM=1)
};

struct CudnnPlan {
  cudnnTensorDescriptor_t xdesc = nullptr, ydesc = nullptr;
  cudnnConvolutionFwdAlgo_t fwd_algo; cudnnMathType_t fwd_math; size_t fwd_ws = 0; bool fwd_ready = false;
  cudnnConvolutionBwdDataAlgo_t bwd_algo; cudnnMathType_t bwd_math; size_t bwd_ws = 0; bool bwd_ready = false;
};
struct GemmPlan {
  cublasLtMatmulDesc_t op = nullptr;
  cublasLtMatrixLayout_t a = nullptr, b = nullptr, c = nullptr;
  cublasLtMatmulAlgo_t algo;
  std::vector<cublasLtMatmulAlgo_t> candidates;   // heuristic top-k, timed on first use when autotune is on
  bool tuned = false;
};

}  // namespace

struct dp_engine {
  dp_config cfg;
  bool bf16 = false;
  size_t es = 4;            // activation element size
  int Cp = 4;               // channels per pixel of the network INPUT (3 = tight, own stem kernel)
  int Cpd = 4;              // channels per pixel of d(input) produced by the library dgrad (4 fp32 / 8 bf16)
  bool own_stem = false;    // bf16: hand-written tensor-core stem forward on the tight C=3 layout
  bool fused_gemm = false;  // opt-in (DORPATCH_FUSED_GEMM=1, bf16): GN+ReLU applied inside the tcgen05 1x1-conv GEMM of kernels_gemm.cu
  void* stem_w_kn = nullptr;
  int H = 224, K = 1000, chunk = 64;
  int num_sms = 148;
  cudnnHandle_t cudnn = nullptr;
  cublasLtHandle_t lt = nullptr;
  cudnnDataType_t cudnn_dt = CUDNN_DATA_FLOAT;
  cudaDataType_t cuda_dt = CUDA_R_32F;
  cublasComputeType_t lt_compute = CUBLAS_COMPUTE_32F;
  int64_t device_bytes = 0, launches = 0;
  std::vector<void*> allocs;
  bool weights_loaded = false;

  ConvW stem;
  std::vector<Block> blocks;
  GNW head_gn;
  float* fc_w = nullptr; float* fc_b = nullptr;

  // workspace (sized for `chunk` samples)
  void* net_in = nullptr;          // [chunk,H,H,Cp]
  void* act = nullptr;             // scratch activation (stem out / GN outputs)
  void* act2 = nullptr;            // scratch (subsampled shortcut input)
  void* x0 = nullptr;              // pooled stem output (saved)
  int8_t* pool_amax = nullptr;
  void* g[4] = {nullptr, nullptr, nullptr, nullptr};   // gradient scratch
  float* gn_partial = nullptr;
  float* head_stats = nullptr;
  float* pooled = nullptr; float* dpooled = nullptr;
  float* logits = nullptr; float* dlogits = nullptr;
  void* d_input = nullptr;         // result of backward: [n,H,H,Cp]
  void* lib_ws = nullptr; size_t lib_ws_bytes = 0;

  // ---- lanes: complete per-chunk workspaces.  dp_attack_grad alternates its chunks between two lanes on
  // two internal streams so that one chunk's kernel tails / memory-bound GroupNorm passes overlap the other
  // chunk's tensor-core convolutions.  The members above (net_in, act, ..., Block::h1...) always alias the
  // lane selected by use_lane(); launches capture the pointers at enqueue time, so switching between chunks is safe.
  struct LaneBufs {
    void *net_in = nullptr, *act = nullptr, *act2 = nullptr, *x0 = nullptr;
    int8_t* pool_amax = nullptr;
    void* g[4] = {nullptr, nullptr, nullptr, nullptr};
    float *gn_partial = nullptr, *head_stats = nullptr, *pooled = nullptr, *dpooled = nullptr, *logits = nullptr, *dlogits = nullptr;
    void* lib_ws = nullptr;
    std::vector<void*> h1, h2, out;
    std::vector<float*> st1, st2, st3;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    cudnnHandle_t cudnn = nullptr;
  };
  std::vector<LaneBufs> lanes;
  cudaEvent_t ev_prep = nullptr;
  void use_lane(int l) {
    LaneBufs& L = lanes[l];
    net_in = L.net_in; act = L.act; act2 = L.act2; x0 = L.x0; pool_amax = L.pool_amax;
    for (int i = 0; i < 4; ++i) g[i] = L.g[i];
    gn_partial = L.gn_partial; head_stats = L.head_stats; pooled = L.pooled; dpooled = L.dpooled;
    logits = L.logits; dlogits = L.dlogits; lib_ws = L.lib_ws; cudnn = L.cudnn;
    for (size_t i = 0; i < blocks.size(); ++i) {
      blocks[i].h1 = L.h1[i]; blocks[i].h2 = L.h2[i]; blocks[i].out = L.out[i];
      blocks[i].st1 = L.st1[i]; blocks[i].st2 = L.st2[i]; blocks[i].st3 = L.st3[i];
    }
  }

  // per-image buffers (max_images)
  float* adv_x = nullptr; float* dLs = nullptr; float* scale = nullptr; float* l2 = nullptr;
  float* loss_struc = nullptr; float* loss_density = nullptr; float* group_lasso = nullptr;
  float* win_dev = nullptr; float* grp_ss = nullptr;
  // failed-mask sets (N2): one bitmap of FAILED_WORDS words per image, its popcounts, staging for one step's indices
  static constexpr int FAILED_WORDS = 128;        // up to 4096 masks (the reference's universe has 2520)
  uint32_t* failed_bits = nullptr; int32_t* failed_count = nullptr; int32_t* failed_idx = nullptr; int32_t* failed_nff = nullptr;
  uint8_t* failed_active = nullptr; float* failed_loss = nullptr; int failed_cap = 0;
  float* helper_scale = nullptr; float* helper_l2 = nullptr; float* helper_ws = nullptr;   // scratch of dp_paste(out) / dp_window_sum
  float* lr_d = nullptr; float* structured_d = nullptr; float* coeff_d = nullptr;
  float* host_x = nullptr; float* host_mask = nullptr; float* host_pattern = nullptr; float* host_G = nullptr;  // dp_attack_step_host

  // per-sample buffers (grown on demand)
  int cap_samples = 0;
  int16_t* rects_d = nullptr; int32_t* y_d = nullptr; uint8_t* tg_d = nullptr;
  float* loss_d = nullptr; int32_t* preds_d = nullptr; float* xf_d = nullptr;
  // pinned staging
  unsigned char* pin = nullptr; size_t pin_bytes = 0;

  // ---- optional per-category profiler (CUDA events around every launch) --------------
  bool prof_on = false;
  struct ProfRec { int cat; cudaEvent_t a, b; double bytes, flops; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;
  std::vector<std::string> prof_names;
  std::vector<double> prof_ms, prof_bytes, prof_flops;
  std::vector<int64_t> prof_count;
  int prof_cat(const char* name) {
    for (size_t i = 0; i < prof_names.size(); ++i) if (prof_names[i] == name) return (int)i;
    prof_names.push_back(name); prof_ms.push_back(0); prof_bytes.push_back(0); prof_flops.push_back(0); prof_count.push_back(0);
    return (int)prof_names.size() - 1;
  }
  cudaEvent_t prof_event() {
    if (!prof_pool.empty()) { cudaEvent_t e = prof_pool.back(); prof_pool.pop_back(); return e; }
    cudaEvent_t e; CUDA_OK(cudaEventCreate(&e)); return e;
  }
  void prof_begin(const char* name, double bytes, double flops, cudaStream_t st) {
    if (!prof_on) return;
    ProfRec r; r.cat = prof_cat(name); r.bytes = bytes; r.flops = flops; r.a = prof_event(); r.b = prof_event();
    CUDA_OK(cudaEventRecord(r.a, st));
    prof_recs.push_back(r);
  }
  void prof_end(cudaStream_t st) {
    if (!prof_on) return;
    CUDA_OK(cudaEventRecord(prof_recs.back().b, st));
  }
  void prof_collect() {
    for (auto& r : prof_recs) {
      CUDA_OK(cudaEventSynchronize(r.b));
      float ms = 0.f; CUDA_OK(cudaEventElapsedTime(&ms, r.a, r.b));
      prof_ms[r.cat] += ms; prof_bytes[r.cat] += r.bytes; prof_flops[r.cat] += r.flops; prof_count[r.cat] += 1;
      prof_pool.push_back(r.a); prof_pool.push_back(r.b);
    }
    prof_recs.clear();
  }

  // ---- whole-step CUDA graphs (SURVEY 8f N4): dp_attack_grad's launch sequence (staging copies, paste, regularisers,
  // every chunk's K1 -> forward -> CW -> backward -> K1^T on both lanes, result copies) captured once per call
  // signature and replayed; the first call of a signature runs eagerly (it picks cuDNN / cublasLt algorithms, which
  // synchronises and cannot be captured).  DORPATCH_GRAPH=0 disables.
  struct GraphEnt { int calls = 0; bool failed = false; cudaGraphExec_t exec = nullptr; int64_t launches = 0; };
  typedef std::tuple<int, int, int, int, const void*, const void*, const void*, const void*, float, float, int> GraphKey;
  std::map<GraphKey, GraphEnt> graphs;
  bool graphs_on = true;
  cudaStream_t cap_stream = nullptr;   // capture happens here when the caller's stream is the legacy / per-thread default stream (not capturable)
  int64_t graph_replays = 0;
  std::string graph_msg;               // why the last capture attempt was abandoned (diagnostics)
  void drop_graphs() {
    for (auto& kv : graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    graphs.clear();
  }

  std::map<std::pair<int, int>, CudnnPlan> cudnn_plans;                 // (layer id, N)
  std::map<std::tuple<int, int, int, int>, GemmPlan> gemm_plans;        // (rows, n_out, k, mode)

  // ---------------------------------------------------------------------------------
  void* dmalloc(size_t bytes) {
    void* p = nullptr;
    bytes = (bytes + 255) / 256 * 256;
    if (bytes == 0) bytes = 256;
    CUDA_OK(cudaMalloc(&p, bytes));
    allocs.push_back(p);
    device_bytes += (int64_t)bytes;
    return p;
  }
  void ensure_pin(size_t bytes) {
    if (bytes <= pin_bytes) return;
    drop_graphs();                       // captured copies hold the old staging address
    if (pin) cudaFreeHost(pin);
    pin_bytes = std::max(bytes, (size_t)1 << 20);
    CUDA_OK(cudaMallocHost((void**)&pin, pin_bytes));
  }
  // K1 for the WHOLE step in one launch (all B*S samples into one buffer, the chunks then read their slices): the launch
  // shape of one classifier chunk (16 images x 28 row tiles) is too small to fill 148 SMs for more than one ragged wave
  // (in-step 0.49-0.55 of HBM peak against 0.69 for a 512-sample launch, profiles/README.md).  Bounded by
  // DORPATCH_K1_WHOLE_MB (default 4096; 0 = one launch per chunk as in round 1).
  void* net_in_all = nullptr;
  size_t net_in_all_cap = 0, k1_whole_max = (size_t)4096 << 20;
  size_t sample_in_bytes() const { return (size_t)H * H * Cp * es; }
  bool k1_whole_ok(int n) const { return k1_whole_max > 0 && n > chunk && (size_t)n * sample_in_bytes() <= k1_whole_max; }
  bool ensure_net_in_all(int n) {
    if (!k1_whole_ok(n)) return false;
    const size_t bytes = (size_t)n * sample_in_bytes();
    if (bytes > net_in_all_cap) {
      drop_graphs();
      if (net_in_all) { CUDA_OK(cudaFree(net_in_all)); device_bytes -= (int64_t)net_in_all_cap; net_in_all = nullptr; net_in_all_cap = 0; }
      CUDA_OK(cudaMalloc(&net_in_all, bytes));
      net_in_all_cap = bytes;
      device_bytes += (int64_t)bytes;
    }
    return true;
  }
  void ensure_samples(int n) {
    if (n <= cap_samples) return;
    drop_graphs();                       // captured launches hold the old per-sample buffers
    // (old buffers stay in `allocs` and are released at destroy)
    cap_samples = std::max(n, cap_samples * 2);
    rects_d = (int16_t*)dmalloc((size_t)cap_samples * 16 * sizeof(int16_t));
    y_d = (int32_t*)dmalloc((size_t)cap_samples * sizeof(int32_t));
    tg_d = (uint8_t*)dmalloc((size_t)cap_samples);
    loss_d = (float*)dmalloc((size_t)cap_samples * sizeof(float));
    preds_d = (int32_t*)dmalloc((size_t)cap_samples * sizeof(int32_t));
    xf_d = (float*)dmalloc((size_t)cap_samples * 8 * sizeof(float));
  }

  // ---- geometry -----------------------------------------------------------------------
  int Hs() const { return H / 2; }
  int Hp() const { return H / 4; }
  size_t max_act_elems() const {   // per sample
    size_t m = (size_t)Hs() * Hs() * STEM_CH;
    for (auto& b : blocks) {
      m = std::max(m, (size_t)b.hin * b.hin * std::max(b.cin, b.mid));
      m = std::max(m, (size_t)b.hout * b.hout * b.cout);
    }
    m = std::max(m, (size_t)H * H * std::max(Cp, Cpd));
    return m;
  }

  void build_arch() {
    int cin = STEM_CH, h = Hp();
    for (int s = 0; s < 4; ++s) {
      for (int bi = 0; bi < DEPTHS[s]; ++bi) {
        Block b{};
        b.cin = cin; b.cout = WIDTHS[s]; b.mid = b.cout / 4;
        b.stride = (bi == 0 && s > 0) ? 2 : 1;
        b.hin = h; b.hout = (h + b.stride - 1) / b.stride;
        b.has_ds = (bi == 0);
        blocks.push_back(b);
        cin = b.cout; h = b.hout;
      }
    }
  }

  void make_conv(ConvW& c, int cin, int cout, int k, int stride, int pad, int cin_pad) {
    c.cin = cin; c.cin_pad = cin_pad; c.cout = cout; c.k = k; c.stride = stride; c.pad = pad;
    c.w = dmalloc((size_t)cout * k * k * cin_pad * es);
    if (k > 1) {   // cuDNN path
      CUDNN_OK(cudnnCreateFilterDescriptor(&c.wdesc));
      CUDNN_OK(cudnnSetFilter4dDescriptor(c.wdesc, cudnn_dt, CUDNN_TENSOR_NHWC, cout, cin_pad, k, k));
      CUDNN_OK(cudnnCreateConvolutionDescriptor(&c.cdesc));
      CUDNN_OK(cudnnSetConvolution2dDescriptor(c.cdesc, pad, pad, stride, stride, 1, 1, CUDNN_CROSS_CORRELATION, CUDNN_DATA_FLOAT));
      CUDNN_OK(cudnnSetConvolutionMathType(c.cdesc, default_math()));
    }
  }
  cudnnMathType_t default_math() const {
    if (cfg.precision == DP_PREC_FP32) return CUDNN_FMA_MATH;
    if (cfg.precision == DP_PREC_TF32) return CUDNN_DEFAULT_MATH;   // fp32 data -> TF32 tensor cores
    return CUDNN_TENSOR_OP_MATH;
  }
  void make_gn(GNW& g_, int C) {
    g_.C = C;
    g_.gamma = (float*)dmalloc((size_t)C * 4);
    g_.beta = (float*)dmalloc((size_t)C * 4);
  }

  void allocate() {
    const size_t n = (size_t)chunk;
    make_conv(stem, 3, STEM_CH, 7, 2, 3, Cpd);
    if (own_stem) stem_w_kn = dmalloc((size_t)160 * 64 * 2);
    for (auto& b : blocks) {
      make_gn(b.n1, b.cin); make_gn(b.n2, b.mid); make_gn(b.n3, b.mid);
      if (b.has_ds) make_conv(b.ds, b.cin, b.cout, 1, b.stride, 0, b.cin);
      make_conv(b.c1, b.cin, b.mid, 1, 1, 0, b.cin);
      make_conv(b.c2, b.mid, b.mid, 3, b.stride, 1, b.mid);
      make_conv(b.c3, b.mid, b.cout, 1, 1, 0, b.mid);
      if (fused_gemm) {
        b.c1p = dmalloc((size_t)b.mid * b.cin * 2);
        b.c3p = dmalloc((size_t)b.cout * b.mid * 2);
      }
    }
    make_gn(head_gn, WIDTHS[3]);
    fc_w = (float*)dmalloc((size_t)K * WIDTHS[3] * 4);
    fc_b = (float*)dmalloc((size_t)K * 4);
    const size_t ma = max_act_elems();
    lib_ws_bytes = (size_t)512 << 20;
    int n_lanes = 2;
    if (const char* le = getenv("DORPATCH_LANES")) n_lanes = atoi(le);
    if (n_lanes < 1) n_lanes = 1;
    if (n_lanes > 2) n_lanes = 2;
    lanes.resize(n_lanes);
    CUDA_OK(cudaEventCreateWithFlags(&ev_prep, cudaEventDisableTiming));
    CUDA_OK(cudaStreamCreateWithFlags(&cap_stream, cudaStreamNonBlocking));
    for (int l = 0; l < n_lanes; ++l) {
      LaneBufs& L = lanes[l];
      for (auto& b : blocks) {
        L.h1.push_back(dmalloc(n * b.hin * b.hin * b.mid * es));
        L.h2.push_back(dmalloc(n * b.hout * b.hout * b.mid * es));
        L.out.push_back(dmalloc(n * b.hout * b.hout * b.cout * es));
        L.st1.push_back((float*)dmalloc(n * dp::GN_GROUPS * 2 * 4));
        L.st2.push_back((float*)dmalloc(n * dp::GN_GROUPS * 2 * 4));
        L.st3.push_back((float*)dmalloc(n * dp::GN_GROUPS * 2 * 4));
      }
      L.net_in = dmalloc(n * H * H * Cp * es);
      L.act = dmalloc(n * ma * es);
      L.act2 = dmalloc(n * ma * es / 4 + 256);
      L.x0 = dmalloc(n * Hp() * Hp() * STEM_CH * es);
      L.pool_amax = (int8_t*)dmalloc(n * Hp() * Hp() * STEM_CH);
      for (int i = 0; i < 4; ++i) L.g[i] = dmalloc(n * ma * es);
      L.gn_partial = (float*)dmalloc((n * dp::GN_WS_FLOATS_PER_SAMPLE + dp::GN_WS_FLOATS_EXTRA) * 4);
      L.head_stats = (float*)dmalloc(n * dp::GN_GROUPS * 2 * 4);
      L.pooled = (float*)dmalloc(n * WIDTHS[3] * 4);
      L.dpooled = (float*)dmalloc(n * WIDTHS[3] * 4);
      L.logits = (float*)dmalloc(n * K * 4);
      L.dlogits = (float*)dmalloc(n * K * 4);
      L.lib_ws = dmalloc(lib_ws_bytes);
      CUDA_OK(cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
      CUDA_OK(cudaEventCreateWithFlags(&L.done, cudaEventDisableTiming));
      if (l == 0) L.cudnn = cudnn;
      else CUDNN_OK(cudnnCreate(&L.cudnn));
    }
    use_lane(0);
    const size_t B = (size_t)cfg.max_images, HW = (size_t)H * H;
    adv_x = (float*)dmalloc(B * 3 * HW * 4);
    dLs = (float*)dmalloc(B * 3 * HW * 4);
    host_x = (float*)dmalloc(B * 3 * HW * 4);
    host_pattern = (float*)dmalloc(B * 3 * HW * 4);
    host_mask = (float*)dmalloc(B * HW * 4);
    host_G = (float*)dmalloc(B * 3 * HW * 4);
    for (float** p : {&scale, &l2, &loss_struc, &loss_density, &group_lasso, &lr_d, &structured_d, &coeff_d, &helper_scale, &helper_l2})
      *p = (float*)dmalloc(B * 4);
    helper_ws = (float*)dmalloc(B * HW * 4);
    failed_bits = (uint32_t*)dmalloc(B * FAILED_WORDS * 4);
    CUDA_OK(cudaMemset(failed_bits, 0, B * FAILED_WORDS * 4));
    failed_count = (int32_t*)dmalloc(B * 4); failed_nff = (int32_t*)dmalloc(B * 4); failed_active = (uint8_t*)dmalloc(B);
    win_dev = (float*)dmalloc(B * 64 * 4);
    grp_ss = (float*)dmalloc(B * (H / UNIT) * (H / UNIT) * 4);
    ensure_samples(chunk);
    ensure_pin((size_t)4 << 20);
  }

  // ---- weights -------------------------------------------------------------------------
  void upload_conv(ConvW& c, const float* host, int64_t numel, cudaStream_t st, float* tmp) {
    const int64_t want = (int64_t)c.cout * c.cin * c.k * c.k;
    if (numel != want) fail("conv weight numel %lld != expected %lld", (long long)numel, (long long)want);
    CUDA_OK(cudaMemcpyAsync(tmp, host, (size_t)numel * 4, cudaMemcpyHostToDevice, st));
    dp::launch_weight_standardize(tmp, c.w, c.cout, c.cin, c.k, c.k, c.cin_pad, bf16, true, st);
    KERNEL_OK();
    CUDA_OK(cudaStreamSynchronize(st));
  }
  void upload_vec(float* dst, const float* host, int64_t numel, int64_t want) {
    if (numel != want) fail("vector numel %lld != expected %lld", (long long)numel, (long long)want);
    CUDA_OK(cudaMemcpy(dst, host, (size_t)numel * 4, cudaMemcpyHostToDevice));
  }
  void upload_gamma(GNW& g_, const float* host, int64_t numel) {
    upload_vec(g_.gamma, host, numel, g_.C);
    g_.pos = true;
    for (int64_t i = 0; i < numel; ++i) g_.pos = g_.pos && (host[i] > 0.f);
  }
  void load_weights(int n, const char* const* names, const float* const* ptrs, const int64_t* numels) {
    std::map<std::string, int> idx;
    for (int i = 0; i < n; ++i) idx[names[i]] = i;
    auto get = [&](const std::string& k) -> int {
      auto it = idx.find(k);
      if (it == idx.end()) fail("missing weight tensor '%s'", k.c_str());
      return it->second;
    };
    float* tmp = nullptr;
    CUDA_OK(cudaMalloc((void**)&tmp, (size_t)2048 * 2048 * 9 * 4 / 4 + (size_t)K * 2048 * 4));
    cudaStream_t st = 0;
    try {
      int i = get("stem.conv.weight");
      upload_conv(stem, ptrs[i], numels[i], st, tmp);
      if (own_stem) { dp::launch_stem_pack(stem.w, stem_w_kn, stem.cin_pad, st); KERNEL_OK(); CUDA_OK(cudaStreamSynchronize(st)); }
      int s = 0, bi = 0;
      for (auto& b : blocks) {
        char pre[64];
        snprintf(pre, sizeof(pre), "stages.%d.blocks.%d.", s, bi);
        auto P = [&](const char* suffix) { return std::string(pre) + suffix; };
        if (b.has_ds) { i = get(P("downsample.conv.weight")); upload_conv(b.ds, ptrs[i], numels[i], st, tmp); }
        i = get(P("conv1.weight")); upload_conv(b.c1, ptrs[i], numels[i], st, tmp);
        i = get(P("conv2.weight")); upload_conv(b.c2, ptrs[i], numels[i], st, tmp);
        i = get(P("conv3.weight")); upload_conv(b.c3, ptrs[i], numels[i], st, tmp);
        if (fused_gemm) {
          dp::launch_gn_gemm_pack(b.c1.w, b.c1p, b.mid, b.cin, st); KERNEL_OK();
          dp::launch_gn_gemm_pack(b.c3.w, b.c3p, b.cout, b.mid, st); KERNEL_OK();
          CUDA_OK(cudaStreamSynchronize(st));
        }
        i = get(P("norm1.weight")); upload_gamma(b.n1, ptrs[i], numels[i]);
        i = get(P("norm1.bias")); upload_vec(b.n1.beta, ptrs[i], numels[i], b.cin);
        i = get(P("norm2.weight")); upload_gamma(b.n2, ptrs[i], numels[i]);
        i = get(P("norm2.bias")); upload_vec(b.n2.beta, ptrs[i], numels[i], b.mid);
        i = get(P("norm3.weight")); upload_gamma(b.n3, ptrs[i], numels[i]);
        i = get(P("norm3.bias")); upload_vec(b.n3.beta, ptrs[i], numels[i], b.mid);
        if (++bi == DEPTHS[s]) { bi = 0; ++s; }
      }
      i = get("norm.weight"); upload_gamma(head_gn, ptrs[i], numels[i]);
      i = get("norm.bias"); upload_vec(head_gn.beta, ptrs[i], numels[i], WIDTHS[3]);
      i = get("head.fc.weight"); upload_vec(fc_w, ptrs[i], numels[i], (int64_t)K * WIDTHS[3]);
      i = get("head.fc.bias"); upload_vec(fc_b, ptrs[i], numels[i], K);
    } catch (...) {
      cudaFree(tmp);
      throw;
    }
    cudaFree(tmp);
    weights_loaded = true;
  }

  // ---- cuDNN convolution -------------------------------------------------------------
  CudnnPlan& conv_plan(int layer_id, const ConvW& c, int N, int hin, int hout) {
    auto key = std::make_pair(layer_id, N);
    auto it = cudnn_plans.find(key);
    if (it != cudnn_plans.end()) return it->second;
    CudnnPlan p;
    CUDNN_OK(cudnnCreateTensorDescriptor(&p.xdesc));
    CUDNN_OK(cudnnCreateTensorDescriptor(&p.ydesc));
    CUDNN_OK(cudnnSetTensor4dDescriptor(p.xdesc, CUDNN_TENSOR_NHWC, cudnn_dt, N, c.cin_pad, hin, hin));
    CUDNN_OK(cudnnSetTensor4dDescriptor(p.ydesc, CUDNN_TENSOR_NHWC, cudnn_dt, N, c.cout, hout, hout));
    int on, oc, oh, ow;
    CUDNN_OK(cudnnGetConvolution2dForwardOutputDim(c.cdesc, p.xdesc, c.wdesc, &on, &oc, &oh, &ow));
    if (on != N || oc != c.cout || oh != hout || ow != hout)
      fail("conv layer %d: cuDNN output dims (%d,%d,%d,%d) != expected (%d,%d,%d,%d)", layer_id, on, oc, oh, ow, N, c.cout, hout, hout);
    return cudnn_plans.emplace(key, p).first->second;
  }
  bool math_ok(cudnnMathType_t m) const {
    if (cfg.precision == DP_PREC_FP32) return m == CUDNN_FMA_MATH;   // parity mode: no TF32 down-conversion
    return true;
  }
  void pick_fwd(CudnnPlan& p, const ConvW& c, const void* x, void* y) {
    cudnnConvolutionFwdAlgoPerf_t perf[16];
    int got = 0;
    if (cfg.autotune)
      CUDNN_OK(cudnnFindConvolutionForwardAlgorithmEx(cudnn, p.xdesc, x, c.wdesc, c.w, c.cdesc, p.ydesc, y, 16, &got, perf, lib_ws, lib_ws_bytes));
    else
      CUDNN_OK(cudnnGetConvolutionForwardAlgorithm_v7(cudnn, p.xdesc, c.wdesc, c.cdesc, p.ydesc, 16, &got, perf));
    for (int i = 0; i < got; ++i) {
      if (perf[i].status != CUDNN_STATUS_SUCCESS || perf[i].memory > lib_ws_bytes || !math_ok(perf[i].mathType)) continue;
      p.fwd_algo = perf[i].algo; p.fwd_math = perf[i].mathType; p.fwd_ws = perf[i].memory; p.fwd_ready = true;
      return;
    }
    fail("no usable cuDNN forward algorithm (cin=%d cout=%d k=%d stride=%d, %d candidates)", c.cin_pad, c.cout, c.k, c.stride, got);
  }
  void pick_bwd(CudnnPlan& p, const ConvW& c, const void* dy, void* dx) {
    cudnnConvolutionBwdDataAlgoPerf_t perf[16];
    int got = 0;
    if (cfg.autotune)
      CUDNN_OK(cudnnFindConvolutionBackwardDataAlgorithmEx(cudnn, c.wdesc, c.w, p.ydesc, dy, c.cdesc, p.xdesc, dx, 16, &got, perf, lib_ws, lib_ws_bytes));
    else
      CUDNN_OK(cudnnGetConvolutionBackwardDataAlgorithm_v7(cudnn, c.wdesc, p.ydesc, c.cdesc, p.xdesc, 16, &got, perf));
    // results are sorted by time: take the fastest usable one, but prefer a deterministic algorithm
    // when it is within 25 % of it (a slow "deterministic" dgrad once cost 688 ms on the stem).
    int fastest = -1, det = -1;
    for (int i = 0; i < got; ++i) {
      if (perf[i].status != CUDNN_STATUS_SUCCESS || perf[i].memory > lib_ws_bytes || !math_ok(perf[i].mathType)) continue;
      if (fastest < 0) fastest = i;
      if (det < 0 && perf[i].determinism == CUDNN_DETERMINISTIC) det = i;
    }
    if (fastest >= 0) {
      int pick = fastest;
      if (det >= 0 && (!cfg.autotune || perf[det].time <= 1.25f * perf[fastest].time)) pick = det;
      p.bwd_algo = perf[pick].algo; p.bwd_math = perf[pick].mathType; p.bwd_ws = perf[pick].memory; p.bwd_ready = true;
      return;
    }
    fail("no usable cuDNN backward-data algorithm (cin=%d cout=%d k=%d stride=%d, %d candidates)", c.cin_pad, c.cout, c.k, c.stride, got);
  }
  void conv_fwd(int layer_id, const ConvW& c, int N, int hin, int hout, const void* x, void* y, cudaStream_t st) {
    CudnnPlan& p = conv_plan(layer_id, c, N, hin, hout);
    if (!p.fwd_ready) pick_fwd(p, c, x, y);
    CUDNN_OK(cudnnSetConvolutionMathType(c.cdesc, p.fwd_math));
    const float one = 1.f, zero = 0.f;
    const double fl = 2.0 * N * hout * hout * c.cout * c.k * c.k * c.cin;
    const double by = ((double)N * hin * hin * c.cin_pad + (double)N * hout * hout * c.cout + (double)c.cout * c.k * c.k * c.cin_pad) * es;
    PROF(this, c.k == 7 ? "stem_conv_fwd" : "conv3x3_fwd", by, fl, st,
         CUDNN_OK(cudnnConvolutionForward(cudnn, &one, p.xdesc, x, c.wdesc, c.w, c.cdesc, p.fwd_algo, lib_ws, lib_ws_bytes, &zero, p.ydesc, y)));
    ++launches;
  }
  void conv_bwd(int layer_id, const ConvW& c, int N, int hin, int hout, const void* dy, void* dx, cudaStream_t st) {
    CudnnPlan& p = conv_plan(layer_id, c, N, hin, hout);
    if (!p.bwd_ready) pick_bwd(p, c, dy, dx);
    CUDNN_OK(cudnnSetConvolutionMathType(c.cdesc, p.bwd_math));
    const float one = 1.f, zero = 0.f;
    const double fl = 2.0 * N * hout * hout * c.cout * c.k * c.k * c.cin;
    const double by = ((double)N * hin * hin * c.cin_pad + (double)N * hout * hout * c.cout + (double)c.cout * c.k * c.k * c.cin_pad) * es;
    PROF(this, c.k == 7 ? "stem_conv_bwd" : "conv3x3_bwd", by, fl, st,
         CUDNN_OK(cudnnConvolutionBackwardData(cudnn, &one, c.wdesc, c.w, p.ydesc, dy, c.cdesc, p.bwd_algo, lib_ws, lib_ws_bytes, &zero, p.xdesc, dx)));
    ++launches;
  }

  // ---- cublasLt GEMM (1x1 convolutions, NHWC) ---------------------------------------------
  // mode 0: Y[rows,nout] = X[rows,k] * W[nout,k]^T (+ Cres)      (forward)
  // mode 1: dX[rows,nout] = dY[rows,k] * W[k,nout] (+ dX if beta) (backward data)
  GemmPlan& gemm_plan(int rows, int nout, int k, int mode) {
    auto key = std::make_tuple(rows, nout, k, mode);
    auto it = gemm_plans.find(key);
    if (it != gemm_plans.end()) return it->second;
    GemmPlan p;
    // modes 2 / 3: the fp32 classifier head (fc forward with fused bias / fc backward), always fp32 math
    const bool head = mode >= 2;
    const cudaDataType_t cuda_dt = head ? CUDA_R_32F : this->cuda_dt;
    CUBLAS_OK(cublasLtMatmulDescCreate(&p.op, head ? CUBLAS_COMPUTE_32F : lt_compute, CUDA_R_32F));
    const cublasOperation_t ta = (mode == 0 || mode == 2) ? CUBLAS_OP_T : CUBLAS_OP_N, tb = CUBLAS_OP_N;
    if (mode == 2) {
      const cublasLtEpilogue_t epi = CUBLASLT_EPILOGUE_BIAS;
      const void* bias = fc_b;
      CUBLAS_OK(cublasLtMatmulDescSetAttribute(p.op, CUBLASLT_MATMUL_DESC_EPILOGUE, &epi, sizeof(epi)));
      CUBLAS_OK(cublasLtMatmulDescSetAttribute(p.op, CUBLASLT_MATMUL_DESC_BIAS_POINTER, &bias, sizeof(bias)));
    }
    CUBLAS_OK(cublasLtMatmulDescSetAttribute(p.op, CUBLASLT_MATMUL_DESC_TRANSA, &ta, sizeof(ta)));
    CUBLAS_OK(cublasLtMatmulDescSetAttribute(p.op, CUBLASLT_MATMUL_DESC_TRANSB, &tb, sizeof(tb)));
    // column-major view: D[nout x rows] = op(A) * B
    if (mode == 0 || mode == 2) CUBLAS_OK(cublasLtMatrixLayoutCreate(&p.a, cuda_dt, k, nout, k));   // W as col-major [k x nout], ld k
    else CUBLAS_OK(cublasLtMatrixLayoutCreate(&p.a, cuda_dt, nout, k, nout));              // W[k rows][nout] as col-major [nout x k], ld nout
    CUBLAS_OK(cublasLtMatrixLayoutCreate(&p.b, cuda_dt, k, rows, k));                      // X / dY as col-major [k x rows]
    CUBLAS_OK(cublasLtMatrixLayoutCreate(&p.c, cuda_dt, nout, rows, nout));
    cublasLtMatmulPreference_t pref;
    CUBLAS_OK(cublasLtMatmulPreferenceCreate(&pref));
    CUBLAS_OK(cublasLtMatmulPreferenceSetAttribute(pref, CUBLASLT_MATMUL_PREF_MAX_WORKSPACE_BYTES, &lib_ws_bytes, sizeof(lib_ws_bytes)));
    cublasLtMatmulHeuristicResult_t res[8];
    int got = 0;
    cublasStatus_t s = cublasLtMatmulAlgoGetHeuristic(lt, p.op, p.a, p.b, p.c, p.c, pref, 8, res, &got);
    cublasLtMatmulPreferenceDestroy(pref);
    if (s != CUBLAS_STATUS_SUCCESS || got == 0) fail("cublasLt: no algorithm for GEMM rows=%d nout=%d k=%d mode=%d (status %d)", rows, nout, k, mode, (int)s);
    p.algo = res[0].algo;
    for (int i = 0; i < got; ++i)
      if (res[i].state == CUBLAS_STATUS_SUCCESS) p.candidates.push_back(res[i].algo);
    return gemm_plans.emplace(key, p).first->second;
  }
  void gemm(int rows, int nout, int k, int mode, const void* W, const void* X, const void* Cres, float beta, void* D, cudaStream_t st) {
    GemmPlan& p = gemm_plan(rows, nout, k, mode);
    const float one = 1.f;
    // Autotune (once per shape): time the heuristic's top candidates on the real operands.  Skipped
    // for in-place accumulation (C == D), where repeated trial runs would corrupt the addend.
    const bool in_place_acc = (beta != 0.f) && (Cres == nullptr || Cres == D);
    if (!p.tuned && cfg.autotune && !in_place_acc && p.candidates.size() > 1 && !prof_on) {
      cudaEvent_t e0, e1;
      CUDA_OK(cudaEventCreate(&e0)); CUDA_OK(cudaEventCreate(&e1));
      float best = 1e30f;
      for (auto& cand : p.candidates) {
        bool ok = true;
        for (int rep = 0; rep < 3 && ok; ++rep) {
          if (rep == 1) CUDA_OK(cudaEventRecord(e0, st));
          ok = cublasLtMatmul(lt, p.op, &one, W, p.a, X, p.b, &beta, Cres ? Cres : D, p.c, D, p.c, &cand, lib_ws, lib_ws_bytes, st) == CUBLAS_STATUS_SUCCESS;
        }
        if (!ok) continue;
        CUDA_OK(cudaEventRecord(e1, st));
        CUDA_OK(cudaEventSynchronize(e1));
        float ms = 0.f; CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
        if (ms < best) { best = ms; p.algo = cand; }
      }
      cudaEventDestroy(e0); cudaEventDestroy(e1);
      p.tuned = true;
    }
    const double by = ((double)rows * k + (double)rows * nout * (beta != 0.f ? 2 : 1) + (double)nout * k) * (mode >= 2 ? 4 : es);
    PROF(this, mode == 0 ? "gemm1x1_fwd" : (mode == 1 ? "gemm1x1_bwd" : (mode == 2 ? "fc_fwd" : "fc_bwd")), by, 2.0 * rows * nout * k, st,
         CUBLAS_OK(cublasLtMatmul(lt, p.op, &one, W, p.a, X, p.b, &beta, Cres ? Cres : D, p.c, D, p.c, &p.algo, lib_ws, lib_ws_bytes, st)));
    ++launches;
  }

  // ---- classifier forward ------------------------------------------------------------------
  // input: [N,H,H,Cp] T.  train: keep what backward needs.  Leaves logits in `logits`.
  void forward(int N, const void* input, bool train, cudaStream_t st) {
    NvtxRange nvtx_("dorpatch.classifier_forward");
    if (!weights_loaded) fail("dp_engine_load_weights has not been called");
    if (N > chunk) fail("forward: N=%d exceeds chunk=%d", N, chunk);
    CUDNN_OK(cudnnSetStream(cudnn, st));
    const int hs = Hs(), hp = Hp();
    if (own_stem) {
      PROF(this, "stem_conv_fwd", ((double)N * H * H * 3 + (double)N * hs * hs * STEM_CH) * es, 2.0 * N * hs * hs * STEM_CH * 147, st,
           dp::launch_stem_forward(input, stem_w_kn, act, N, H, H, st));
      KERNEL_OK(); ++launches;
    } else {
      for (int n0 = 0; n0 < N; n0 += STEM_SUB) {   // cuDNN's stem kernels degrade badly beyond ~128 samples of 224x224
        const int n = std::min(STEM_SUB, N - n0);
        conv_fwd(0, stem, n, H, hs, (const char*)input + (size_t)n0 * H * H * Cp * es, (char*)act + (size_t)n0 * hs * hs * STEM_CH * es, st);
      }
    }
    PROF(this, "maxpool_fwd", (double)N * (hs * hs + hp * hp) * STEM_CH * es, 0, st,
         dp::launch_maxpool_forward(act, x0, train ? pool_amax : nullptr, N, hs, hs, STEM_CH, bf16, st)); KERNEL_OK(); ++launches;
    const void* cur = x0;
    int lid = 1;
    for (auto& b : blocks) {
      const int pin_ = b.hin * b.hin, pout = b.hout * b.hout;
      // opt-in: statistics pass + tcgen05 GEMM that normalises its A operand on the way into shared memory
      // (the relu(gn(.)) tensors of norm1 / norm3 are never written); blocks with a downsample branch keep norm1.
      const bool fuse1 = fused_gemm && !b.has_ds && dp::gn_gemm_supported(pin_, b.cin, b.mid);
      const bool fuse3 = fused_gemm && dp::gn_gemm_supported(pout, b.mid, b.cout);
      // xp = relu(gn1(cur))
      if (fuse1) {
        PROF(this, "gn_stats", 1.0 * N * pin_ * b.cin * es, 0, st, dp::launch_gn_stats(cur, gn_partial, b.st1, N, pin_, b.cin, bf16, st));
        KERNEL_OK(); launches += 2;
      } else {
        PROF(this, "gn_relu_fwd", 2.0 * N * pin_ * b.cin * es, 0, st,
             dp::launch_gn_relu_forward(cur, act, b.n1.gamma, b.n1.beta, gn_partial, b.st1, N, pin_, b.cin, bf16, st)); KERNEL_OK(); launches += 2;
      }
      const void* shortcut = cur;
      if (b.has_ds) {
        const void* src = act;
        if (b.stride == 2) {
          PROF(this, "subsample", 2.0 * N * pout * b.cin * es, 0, st, dp::launch_subsample2(act, act2, N, b.hin, b.hin, b.cin, bf16, st));
          KERNEL_OK(); ++launches; src = act2;
        }
        gemm(N * pout, b.cout, b.cin, 0, b.ds.w, src, nullptr, 0.f, b.out, st);
        shortcut = b.out;
      }
      if (fuse1) {
        PROF(this, "gn_gemm1x1_fwd", ((double)N * pin_ * (b.cin + b.mid) + (double)b.mid * b.cin) * es, 2.0 * N * pin_ * b.mid * b.cin, st,
             dp::launch_gn_gemm_forward(cur, b.c1p, b.st1, b.n1.gamma, b.n1.beta, nullptr, b.h1, N, pin_, b.cin, b.mid, st));
        KERNEL_OK(); ++launches;
      } else {
        gemm(N * pin_, b.mid, b.cin, 0, b.c1.w, act, nullptr, 0.f, b.h1, st);
      }
      PROF(this, "gn_relu_fwd", 2.0 * N * pin_ * b.mid * es, 0, st,
           dp::launch_gn_relu_forward(b.h1, act, b.n2.gamma, b.n2.beta, gn_partial, b.st2, N, pin_, b.mid, bf16, st)); KERNEL_OK(); launches += 2;
      conv_fwd(lid, b.c2, N, b.hin, b.hout, act, b.h2, st);
      if (fuse3) {
        PROF(this, "gn_stats", 1.0 * N * pout * b.mid * es, 0, st, dp::launch_gn_stats(b.h2, gn_partial, b.st3, N, pout, b.mid, bf16, st));
        KERNEL_OK(); launches += 2;
        PROF(this, "gn_gemm1x1_fwd", ((double)N * pout * (b.mid + 2.0 * b.cout) + (double)b.cout * b.mid) * es, 2.0 * N * pout * b.cout * b.mid, st,
             dp::launch_gn_gemm_forward(b.h2, b.c3p, b.st3, b.n3.gamma, b.n3.beta, shortcut, b.out, N, pout, b.mid, b.cout, st));
        KERNEL_OK(); ++launches;
      } else {
        PROF(this, "gn_relu_fwd", 2.0 * N * pout * b.mid * es, 0, st,
             dp::launch_gn_relu_forward(b.h2, act, b.n3.gamma, b.n3.beta, gn_partial, b.st3, N, pout, b.mid, bf16, st)); KERNEL_OK(); launches += 2;
        gemm(N * pout, b.cout, b.mid, 0, b.c3.w, act, shortcut, 1.f, b.out, st);   // + shortcut fused as C operand
      }
      cur = b.out;
      ++lid;
    }
    const Block& last = blocks.back();
    const int pl = last.hout * last.hout;
    PROF(this, "head_fwd", (double)N * pl * last.cout * es, 2.0 * N * last.cout * K, st, {
      dp::launch_gn_stats(cur, gn_partial, head_stats, N, pl, last.cout, bf16, st);
      dp::launch_head_pool(cur, head_gn.gamma, head_gn.beta, head_stats, pooled, N, pl, last.cout, bf16, st);
    }); KERNEL_OK(); launches += 3;
    gemm(N, K, last.cout, 2, fc_w, pooled, nullptr, 0.f, logits, st);          // logits = pooled * Wfc^T + b (fp32)
  }

  // ---- classifier backward (to the input) -----------------------------------------------------
  // dlog: [N,K] fp32 dev.  Leaves d/d(input) in `d_input` ([N,H,H,Cp] T).
  // `fused`: non-null -> finish with the fused stem-dgrad + masked EOT reduce into fused->G instead of
  // producing d_input (bf16 own-stem path; the per-sample input gradient is never materialised).
  struct FusedReduce { const int16_t* rects; float* G; int B, S, n0; };
  bool fused_stem_bwd = false;     // set at create: own_stem && DORPATCH_STEM_BWD != "cudnn"
  bool fused_pool_bwd = false;     // ... && DORPATCH_POOL_BWD == "fused": max-pool backward fused in as well (slower, off)
  bool stem_bwd_fused_ok() const { return fused_stem_bwd; }
  void backward(int N, const float* dlog, cudaStream_t st, const FusedReduce* fused = nullptr) {
    NvtxRange nvtx_("dorpatch.classifier_backward");
    CUDNN_OK(cudnnSetStream(cudnn, st));
    const Block& last = blocks.back();
    const int pl = last.hout * last.hout;
    void *GA = g[0], *GB = g[1], *GC = g[2], *GD = g[3];
    gemm(N, last.cout, K, 3, fc_w, dlog, nullptr, 0.f, dpooled, st);           // dpooled = dlogits * Wfc (fp32)
    PROF(this, "head_bwd", 2.0 * N * pl * last.cout * es, 0, st, {
      dp::launch_pool_grad_bcast(dpooled, GB, N, pl, last.cout, bf16, st);
      dp::launch_gn_relu_backward(GB, last.out, nullptr, GA, head_gn.gamma, head_gn.beta, head_stats, gn_partial, N, pl, last.cout, bf16, st, head_gn.pos);
    }); KERNEL_OK(); launches += 3;
    for (int bi = (int)blocks.size() - 1; bi >= 0; --bi) {
      Block& b = blocks[bi];
      const int lid = bi + 1;
      const int pin_ = b.hin * b.hin, pout = b.hout * b.hout;
      const void* xin = (bi == 0) ? x0 : blocks[bi - 1].out;
      // d_a3 = d_out * W3
      gemm(N * pout, b.mid, b.cout, 1, b.c3.w, GA, nullptr, 0.f, GB, st);
      PROF(this, "gn_relu_bwd", 3.0 * N * pout * b.mid * es, 0, st,
           dp::launch_gn_relu_backward(GB, b.h2, nullptr, GC, b.n3.gamma, b.n3.beta, b.st3, gn_partial, N, pout, b.mid, bf16, st, b.n3.pos)); KERNEL_OK(); launches += 2;
      conv_bwd(lid, b.c2, N, b.hin, b.hout, GC, GB, st);
      PROF(this, "gn_relu_bwd", 3.0 * N * pin_ * b.mid * es, 0, st,
           dp::launch_gn_relu_backward(GB, b.h1, nullptr, GC, b.n2.gamma, b.n2.beta, b.st2, gn_partial, N, pin_, b.mid, bf16, st, b.n2.pos)); KERNEL_OK(); launches += 2;
      gemm(N * pin_, b.cin, b.mid, 1, b.c1.w, GC, nullptr, 0.f, GB, st);          // d_xp (conv1 path)
      if (b.has_ds) {
        if (b.stride == 2) {
          gemm(N * pout, b.cin, b.cout, 1, b.ds.w, GA, nullptr, 0.f, GC, st);
          PROF(this, "subsample", 3.0 * N * pout * b.cin * es, 0, st, dp::launch_subsample2_adjoint_add(GC, GB, N, b.hin, b.hin, b.cin, bf16, st)); KERNEL_OK(); ++launches;
        } else {
          gemm(N * pout, b.cin, b.cout, 1, b.ds.w, GA, nullptr, 1.f, GB, st);    // accumulate
        }
        PROF(this, "gn_relu_bwd", 3.0 * N * pin_ * b.cin * es, 0, st,
             dp::launch_gn_relu_backward(GB, xin, nullptr, GD, b.n1.gamma, b.n1.beta, b.st1, gn_partial, N, pin_, b.cin, bf16, st, b.n1.pos)); KERNEL_OK(); launches += 2;
      } else {
        PROF(this, "gn_relu_bwd", 4.0 * N * pin_ * b.cin * es, 0, st,
             dp::launch_gn_relu_backward(GB, xin, GA, GD, b.n1.gamma, b.n1.beta, b.st1, gn_partial, N, pin_, b.cin, bf16, st, b.n1.pos)); KERNEL_OK(); launches += 2;
      }
      std::swap(GA, GD);
    }
    const int hs = Hs();
    if (fused != nullptr && fused_pool_bwd) {
      // max-pool backward + stem dgrad + masked EOT reduce in one kernel: neither d_stem nor d_input is written
      PROF(this, "stem_bwd_reduce", (double)N * (hs / 2) * (hs / 2) * STEM_CH * (es + 1) + 3.0 * H * H * 4 * (double)N / fused->S,
           2.0 * N * hs * hs * STEM_CH * 147, st,
           dp::launch_stem_bwd_pool_reduce(GA, pool_amax, stem.w, stem.cin_pad, fused->rects, fused->G, fused->B, fused->S, fused->n0, N, H, H, st));
      KERNEL_OK(); ++launches;
      d_input = nullptr;
      return;
    }
    PROF(this, "maxpool_bwd", (double)N * (hs * hs + (hs / 2) * (hs / 2)) * STEM_CH * es, 0, st,
         dp::launch_maxpool_backward(GA, pool_amax, GB, N, hs, hs, STEM_CH, bf16, st)); KERNEL_OK(); ++launches;
    if (fused != nullptr) {
      PROF(this, "stem_bwd_reduce", (double)N * hs * hs * STEM_CH * es + 3.0 * H * H * 4 * (double)N / fused->S,
           2.0 * N * hs * hs * STEM_CH * 147, st,
           dp::launch_stem_bwd_reduce(GB, stem.w, stem.cin_pad, fused->rects, fused->G, fused->B, fused->S, fused->n0, N, H, H, st));
      KERNEL_OK(); ++launches;
      d_input = nullptr;
      return;
    }
    for (int n0 = 0; n0 < N; n0 += STEM_SUB) {
      const int n = std::min(STEM_SUB, N - n0);
      conv_bwd(0, stem, n, H, hs, (const char*)GB + (size_t)n0 * hs * hs * STEM_CH * es, (char*)GC + (size_t)n0 * H * H * Cpd * es, st);
    }
    d_input = GC;
  }

  // ---- helpers for the attack entry points --------------------------------------------------
  void h2d_samples(const int16_t* rects_host, int N, cudaStream_t st) {
    ensure_samples(N);
    if (rects_host != nullptr) {
      const size_t bytes = (size_t)N * 16 * sizeof(int16_t);
      ensure_pin(bytes);
      memcpy(pin, rects_host, bytes);
      CUDA_OK(cudaMemcpyAsync(rects_d, pin, bytes, cudaMemcpyHostToDevice, st));
      CUDA_OK(cudaStreamSynchronize(st));   // `pin` is reused right after
    }
  }
  void check_B(int B) const {
    if (B < 1 || B > cfg.max_images) fail("B=%d outside [1, max_images=%d]", B, cfg.max_images);
  }
};

// =========================================================================================
// C ABI
// =========================================================================================
#define DP_TRY try {
#define DP_CATCH                                   \
  }                                                \
  catch (const std::exception& ex) {               \
    g_last_error = ex.what();                      \
    return 1;                                      \
  }                                                \
  catch (...) {                                    \
    g_last_error = "unknown C++ exception";        \
    return 1;                                      \
  }                                                \
  return 0;

extern "C" {

int32_t dp_abi_version(void) { return DP_ABI_VERSION; }
const char* dp_last_error(void) { return g_last_error.c_str(); }

int32_t dp_engine_create(const dp_config* cfg, dp_engine** out) {
  DP_TRY
  if (!cfg || !out) fail("null argument");
  if (cfg->img % 56 != 0 || cfg->img < 56) fail("img=%d must be a positive multiple of 56", cfg->img);
  if (cfg->chunk < 1) fail("chunk must be >= 1");
  if (cfg->max_images < 1) fail("max_images must be >= 1");
  if (cfg->precision < 0 || cfg->precision > 2) fail("unknown precision %d", cfg->precision);
  int ndev = 0;
  CUDA_OK(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) fail("device %d not present (%d CUDA devices)", cfg->device, ndev);
  CUDA_OK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major < 10) fail("device %d is sm_%d%d; this engine is built for sm_100a (B200) only", cfg->device, prop.major, prop.minor);
  dp_engine* e = new dp_engine();
  try {
    e->cfg = *cfg;
    e->num_sms = prop.multiProcessorCount;
    e->bf16 = (cfg->precision == DP_PREC_BF16);
    e->es = e->bf16 ? 2 : 4;
    e->Cpd = e->bf16 ? 8 : 4;
    if (const char* s = getenv("DORPATCH_CPAD")) e->Cpd = atoi(s);
    if (e->Cpd != 4 && e->Cpd != 8) fail("DORPATCH_CPAD must be 4 or 8");
    if (const char* gn = getenv("DORPATCH_GN"); gn && strcmp(gn, "v2") != 0)
      fail("DORPATCH_GN=%s is no longer supported: GroupNorm always runs v2 (the two-pass kernels only on shapes v2 cannot "
           "place); unset DORPATCH_GN or set it to v2", gn);
    const char* stem_env = getenv("DORPATCH_STEM");
    e->own_stem = e->bf16 && !(stem_env && strcmp(stem_env, "cudnn") == 0);
    e->Cp = e->own_stem ? 3 : e->Cpd;
    const char* sb_env = getenv("DORPATCH_STEM_BWD");
    e->fused_stem_bwd = e->own_stem && !(sb_env && strcmp(sb_env, "cudnn") == 0);
    const char* fg_env = getenv("DORPATCH_FUSED_GEMM");
    e->fused_gemm = e->bf16 && fg_env && atoi(fg_env) != 0;   // validated on hardware (tests/test_gpu_ops.py, test_gpu_fused_gemm.py) but 2x slower than cublasLt + GroupNorm: off unless asked for
    if (const char* g_env = getenv("DORPATCH_GRAPH")) e->graphs_on = atoi(g_env) != 0;
    if (const char* k_env = getenv("DORPATCH_K1_WHOLE_MB")) e->k1_whole_max = (size_t)std::max(0, atoi(k_env)) << 20;
    const char* pb_env = getenv("DORPATCH_POOL_BWD");
    // measured: rebuilding the d_stem patch in shared memory costs more than the saved HBM round trip
    // (2.25 ms vs 1.33 + 0.71 ms per 512-sample step) -> off unless DORPATCH_POOL_BWD=fused
    e->fused_pool_bwd = e->fused_stem_bwd && (pb_env && strcmp(pb_env, "fused") == 0);
    e->H = cfg->img; e->K = cfg->n_classes; e->chunk = cfg->chunk;
    e->cudnn_dt = e->bf16 ? CUDNN_DATA_BFLOAT16 : CUDNN_DATA_FLOAT;
    e->cuda_dt = e->bf16 ? CUDA_R_16BF : CUDA_R_32F;
    e->lt_compute = (cfg->precision == DP_PREC_TF32) ? CUBLAS_COMPUTE_32F_FAST_TF32 : CUBLAS_COMPUTE_32F;
    CUDNN_OK(cudnnCreate(&e->cudnn));
    CUBLAS_OK(cublasLtCreate(&e->lt));
    e->build_arch();
    e->allocate();
  } catch (...) {
    dp_engine_destroy(e);
    throw;
  }
  *out = e;
  DP_CATCH
}

void dp_engine_destroy(dp_engine* e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  for (auto& kv : e->cudnn_plans) {
    if (kv.second.xdesc) cudnnDestroyTensorDescriptor(kv.second.xdesc);
    if (kv.second.ydesc) cudnnDestroyTensorDescriptor(kv.second.ydesc);
  }
  for (auto& kv : e->gemm_plans) {
    cublasLtMatmulDescDestroy(kv.second.op);
    cublasLtMatrixLayoutDestroy(kv.second.a);
    cublasLtMatrixLayoutDestroy(kv.second.b);
    cublasLtMatrixLayoutDestroy(kv.second.c);
  }
  auto kill = [](ConvW& c) {
    if (c.wdesc) cudnnDestroyFilterDescriptor(c.wdesc);
    if (c.cdesc) cudnnDestroyConvolutionDescriptor(c.cdesc);
  };
  kill(e->stem);
  for (auto& b : e->blocks) { kill(b.ds); kill(b.c1); kill(b.c2); kill(b.c3); }
  e->drop_graphs();
  for (auto& r : e->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto ev : e->prof_pool) cudaEventDestroy(ev);
  for (size_t l = 0; l < e->lanes.size(); ++l) {
    if (e->lanes[l].stream) cudaStreamDestroy(e->lanes[l].stream);
    if (e->lanes[l].done) cudaEventDestroy(e->lanes[l].done);
    if (l > 0 && e->lanes[l].cudnn) cudnnDestroy(e->lanes[l].cudnn);
  }
  if (!e->lanes.empty()) e->cudnn = e->lanes[0].cudnn;
  if (e->ev_prep) cudaEventDestroy(e->ev_prep);
  if (e->cap_stream) cudaStreamDestroy(e->cap_stream);
  if (e->net_in_all) cudaFree(e->net_in_all);
  for (void* p : e->allocs) cudaFree(p);
  if (e->pin) cudaFreeHost(e->pin);
  if (e->cudnn) cudnnDestroy(e->cudnn);
  if (e->lt) cublasLtDestroy(e->lt);
  delete e;
}

int32_t dp_engine_load_weights(dp_engine* e, int32_t n, const char* const* names, const float* const* ptrs, const int64_t* numels) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  e->load_weights(n, names, ptrs, numels);
  DP_CATCH
}

int64_t dp_engine_device_bytes(const dp_engine* e) { return e ? e->device_bytes : 0; }
int64_t dp_engine_launch_count(const dp_engine* e) { return e ? e->launches : 0; }
int64_t dp_engine_graph_replays(const dp_engine* e) { return e ? e->graph_replays : 0; }
const char* dp_engine_graph_status(const dp_engine* e) { return e ? e->graph_msg.c_str() : ""; }

int32_t dp_engine_profile(dp_engine* e, int32_t enable) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  e->prof_collect();
  e->prof_on = enable != 0;
  if (enable == 2) {   // reset
    for (size_t i = 0; i < e->prof_ms.size(); ++i) { e->prof_ms[i] = 0; e->prof_bytes[i] = 0; e->prof_flops[i] = 0; e->prof_count[i] = 0; }
  }
  DP_CATCH
}

int32_t dp_engine_profile_read(dp_engine* e, int32_t max_n, char* names, int32_t name_stride, double* ms, double* bytes,
                               double* flops, int64_t* counts, int32_t* n_out) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  e->prof_collect();
  int n = (int)e->prof_names.size();
  if (n > max_n) n = max_n;
  for (int i = 0; i < n; ++i) {
    snprintf(names + (size_t)i * name_stride, name_stride, "%s", e->prof_names[i].c_str());
    ms[i] = e->prof_ms[i]; bytes[i] = e->prof_bytes[i]; flops[i] = e->prof_flops[i]; counts[i] = e->prof_count[i];
  }
  *n_out = n;
  DP_CATCH
}

int32_t dp_input_layout(const dp_engine* e, int32_t* c_pad, int32_t* elem_bytes) {
  DP_TRY
  if (!e) fail("null engine");
  if (c_pad) *c_pad = e->Cp;
  if (elem_bytes) *elem_bytes = (int32_t)e->es;
  DP_CATCH
}

int32_t dp_paste(dp_engine* e, const float* x, const float* mask, const float* pattern, int32_t B, float eps,
                 float* adv_x_out, float* l2_host, float* scale_host, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  e->check_B(B);
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(cudaSetDevice(e->cfg.device));
  // with an output buffer this is the stand-alone helper (utils.clip, main.py:140): it must not disturb the per-step
  // state (adv_x, clip scale) a dp_attack_grad left behind for dp_attack_update; without one it IS the step's paste
  float* l2d = adv_x_out ? e->helper_l2 : e->l2;
  float* scd = adv_x_out ? e->helper_scale : e->scale;
  dp::launch_paste(x, mask, pattern, adv_x_out ? adv_x_out : e->adv_x, l2d, scd, B, e->H, e->H, eps, st); KERNEL_OK(); ++e->launches;
  if (l2_host) CUDA_OK(cudaMemcpyAsync(l2_host, l2d, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  if (scale_host) CUDA_OK(cudaMemcpyAsync(scale_host, scd, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  if (l2_host || scale_host) CUDA_OK(cudaStreamSynchronize(st));
  DP_CATCH
}

int32_t dp_window_sum(dp_engine* e, const float* t, int32_t B, int32_t k, int32_t square, float* out_host, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  e->check_B(B);
  if (k < 1 || e->H % k != 0) fail("window %d does not divide img %d", k, e->H);
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(cudaSetDevice(e->cfg.device));
  const size_t n = (size_t)B * (e->H / k) * (e->H / k);
  float* tmp = e->helper_ws;   // own scratch (never the structural-loss gradient the sign step reads)
  dp::launch_window_sum(t, tmp, B, e->H, e->H, k, square != 0, st); KERNEL_OK(); ++e->launches;
  CUDA_OK(cudaMemcpyAsync(out_host, tmp, n * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  DP_CATCH
}

int32_t dp_expand(dp_engine* e, const float* img, int32_t B, int32_t S, const int16_t* rects_host, void* out, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(cudaSetDevice(e->cfg.device));
  const int N = B * S;
  if (out == nullptr && N > e->chunk) fail("dp_expand: B*S=%d exceeds chunk=%d and no output buffer was given", N, e->chunk);
  e->h2d_samples(rects_host, N, st);
  PROF(e, "expand_k1", (double)N * e->H * e->H * 3 * e->es + 3.0 * e->H * e->H * 4 * (double)B, 0, st,
       dp::launch_expand(img, nullptr, nullptr, nullptr, nullptr, rects_host ? e->rects_d : nullptr, out ? out : e->net_in,
                         B, S, 0, N, e->H, e->H, e->Cp, e->bf16, false, e->num_sms, st));
  KERNEL_OK(); ++e->launches;
  DP_CATCH
}

int32_t dp_expand_dev(dp_engine* e, const float* img, int32_t B, int32_t S, const int16_t* rects_dev, void* out, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (!out) fail("dp_expand_dev needs an output buffer");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(cudaSetDevice(e->cfg.device));
  const int N = B * S;
  PROF(e, "expand_k1", (double)N * e->H * e->H * 3 * e->es + 3.0 * e->H * e->H * 4 * (double)B, 0, st,
       dp::launch_expand(img, nullptr, nullptr, nullptr, nullptr, rects_dev, out, B, S, 0, N, e->H, e->H, e->Cp, e->bf16, false, e->num_sms, st));
  KERNEL_OK(); ++e->launches;
  DP_CATCH
}

int32_t dp_expand_step_dev(dp_engine* e, const float* x, const float* mask, const float* pattern, int32_t B, int32_t S,
                           const int16_t* rects_dev, int32_t n0, int32_t n, void* out, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (!out || !x || !mask || !pattern) fail("dp_expand_step_dev: null pointer");
  if (n0 < 0 || n < 1 || n0 + n > B * S) fail("dp_expand_step_dev: samples [%d, %d) outside [0, %d)", n0, n0 + n, B * S);
  e->check_B(B);
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(cudaSetDevice(e->cfg.device));
  PROF(e, "expand_k1", (double)n * e->H * e->H * 3 * e->es + 7.0 * e->H * e->H * 4 * (double)n / S, 0, st,
       dp::launch_expand(nullptr, x, mask, pattern, e->scale, rects_dev, out, B, S, n0, n, e->H, e->H, e->Cp, e->bf16, true, e->num_sms, st));
  KERNEL_OK(); ++e->launches;
  DP_CATCH
}

int32_t dp_k1_samples_per_launch(const dp_engine* e, int32_t n_samples) {
  if (!e || n_samples < 1) return 0;
  return e->k1_whole_ok(n_samples) ? n_samples : std::min(n_samples, e->chunk);
}

int32_t dp_predict(dp_engine* e, const float* img, int32_t B, int32_t S, const int16_t* rects_host, int32_t* preds_host,
                   float* logits_host, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  NvtxRange nvtx_("dorpatch.predict");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(cudaSetDevice(e->cfg.device));
  const int N = B * S;
  if (N < 1) fail("dp_predict: empty batch");
  e->h2d_samples(rects_host, N, st);
  // forward-only scan (collect_failure, PatchCleanser): chunks alternate between the two lanes like dp_attack_grad
  cudaStream_t const user_st = st;
  const bool dual = e->lanes.size() == 2 && N > e->chunk && !e->prof_on;
  if (dual) {
    CUDA_OK(cudaEventRecord(e->ev_prep, user_st));
    for (auto& L : e->lanes) CUDA_OK(cudaStreamWaitEvent(L.stream, e->ev_prep, 0));
  }
  int chunk_id = 0;
  for (int n0 = 0; n0 < N; n0 += e->chunk, ++chunk_id) {
    const int n = std::min(e->chunk, N - n0);
    if (dual) { e->use_lane(chunk_id & 1); st = e->lanes[chunk_id & 1].stream; }
    PROF(e, "expand_k1", (double)n * e->H * e->H * 3 * e->es + 3.0 * e->H * e->H * 4 * (double)n / S, 0, st,
         dp::launch_expand(img, nullptr, nullptr, nullptr, nullptr, rects_host ? e->rects_d : nullptr, e->net_in, B, S, n0, n,
                           e->H, e->H, e->Cp, e->bf16, false, e->num_sms, st));
    KERNEL_OK(); ++e->launches;
    e->forward(n, e->net_in, false, st);
    dp::launch_argmax(e->logits, e->preds_d + n0, n, e->K, st); KERNEL_OK(); ++e->launches;
    if (logits_host) CUDA_OK(cudaMemcpyAsync(logits_host + (size_t)n0 * e->K, e->logits, (size_t)n * e->K * 4, cudaMemcpyDeviceToHost, st));
  }
  if (dual) {
    for (auto& L : e->lanes) {
      CUDA_OK(cudaEventRecord(L.done, L.stream));
      CUDA_OK(cudaStreamWaitEvent(user_st, L.done, 0));
    }
    e->use_lane(0);
    st = user_st;
  }
  CUDA_OK(cudaMemcpyAsync(preds_host, e->preds_d, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  DP_CATCH
}

// Everything dp_attack_grad puts on the stream: staging H2D copies, per-image kernels, the chunk loop on one or two
// lanes, result D2H copies into the pinned staging area.  No host synchronisation inside (capturable).
struct GradLayout { size_t rect_bytes, xf_bytes, d2h_off; int32_t* ys; uint8_t* tg; unsigned char* rp; };
static void attack_grad_enqueue(dp_engine* e, const dp_attack_args* a, const GradLayout& L_, cudaStream_t st) {
  const int B = a->B, S = a->S, N = B * S, H = e->H;
  const size_t rect_bytes = L_.rect_bytes, xf_bytes = L_.xf_bytes;
  CUDA_OK(cudaMemcpyAsync(e->y_d, L_.ys, (size_t)N * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->tg_d, L_.tg, (size_t)N, cudaMemcpyHostToDevice, st));
  if (rect_bytes) CUDA_OK(cudaMemcpyAsync(e->rects_d, L_.rp, rect_bytes, cudaMemcpyHostToDevice, st));
  if (xf_bytes) {
    CUDA_OK(cudaMemcpyAsync(e->xf_d, L_.rp + rect_bytes, xf_bytes, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemsetAsync(a->grad_adv, 0, (size_t)B * 3 * H * H * sizeof(float), st));   // the adjoint scatters with atomics
  }
  const int16_t* rects = rect_bytes ? e->rects_d : nullptr;

  const double img_bytes = (double)B * H * H * 4;
  PROF(e, "paste", 10.0 * img_bytes, 0, st, dp::launch_paste(a->x, a->mask, a->pattern, e->adv_x, e->l2, e->scale, B, H, H, a->eps, st)); KERNEL_OK(); ++e->launches;
  PROF(e, "struct", 9.0 * img_bytes, 0, st, dp::launch_struct(e->adv_x, a->x, e->loss_struc, e->dLs, B, H, H, st)); KERNEL_OK(); ++e->launches;
  if (a->stage == 0) {
    PROF(e, "maskreg", img_bytes, 0, st, dp::launch_maskreg(a->mask, e->loss_density, e->group_lasso, e->win_dev, e->grp_ss, B, H, H, UNIT, st)); KERNEL_OK(); ++e->launches;
  }
  const float inv_s = 1.0f / (float)a->S_total;
  // Two lanes: chunks alternate between two workspaces / internal streams (only when every chunk holds whole
  // images, so no two chunks accumulate into the same G[b]).  Everything enqueued so far is on `st`.
  cudaStream_t const user_st = st;
  // K1 once for the whole step when its output fits the budget (see ensure_net_in_all); the chunks read their slices
  const bool k1_whole = !xf_bytes && e->net_in_all != nullptr && e->k1_whole_ok(N) && (size_t)N * e->sample_in_bytes() <= e->net_in_all_cap;
  if (k1_whole) {
    PROF(e, "expand_k1", (double)N * H * H * 3 * e->es + 7.0 * H * H * 4 * (double)B, 0, st,
         dp::launch_expand(nullptr, a->x, a->mask, a->pattern, e->scale, rects, e->net_in_all, B, S, 0, N, H, H, e->Cp, e->bf16, true, e->num_sms, st));
    KERNEL_OK(); ++e->launches;
  }
  // (the per-category profiler serialises on one lane so that category times do not overlap)
  const bool dual = e->lanes.size() == 2 && N > e->chunk && (e->chunk % S == 0) && !e->prof_on;
  if (dual) {
    CUDA_OK(cudaEventRecord(e->ev_prep, user_st));
    for (auto& L : e->lanes) CUDA_OK(cudaStreamWaitEvent(L.stream, e->ev_prep, 0));
  }
  int chunk_id = 0;
  for (int n0 = 0; n0 < N; n0 += e->chunk, ++chunk_id) {
    const int n = std::min(e->chunk, N - n0);
    if (dual) { e->use_lane(chunk_id & 1); st = e->lanes[chunk_id & 1].stream; }
    const void* chunk_in = e->net_in;
    if (k1_whole) {
      chunk_in = (const char*)e->net_in_all + (size_t)n0 * e->sample_in_bytes();
    } else if (xf_bytes) {
      PROF(e, "expand_affine", (double)n * H * H * 3 * e->es + 3.0 * H * H * 4 * (double)n / S, 0, st,
           dp::launch_expand_affine(e->adv_x, e->xf_d, rects, e->net_in, S, n0, n, H, H, e->Cp, e->bf16, st));
      KERNEL_OK(); ++e->launches;
    } else {
      PROF(e, "expand_k1", (double)n * H * H * 3 * e->es + 7.0 * H * H * 4 * (double)n / S, 0, st,
           dp::launch_expand(nullptr, a->x, a->mask, a->pattern, e->scale, rects, e->net_in, B, S, n0, n, H, H, e->Cp, e->bf16, true, e->num_sms, st));
      KERNEL_OK(); ++e->launches;
    }
    e->forward(n, chunk_in, true, st);
    PROF(e, "cw_k4", 2.0 * n * e->K * 4, 0, st,
         dp::launch_cw(e->logits, e->y_d + n0, e->tg_d + n0, a->confidence, inv_s, e->loss_d + n0, e->preds_d + n0, e->dlogits, n, e->K, st));
    KERNEL_OK(); ++e->launches;
    const bool fuse = !xf_bytes && e->stem_bwd_fused_ok();
    dp_engine::FusedReduce fr{rects, a->grad_adv, B, S, n0};
    e->backward(n, e->dlogits, st, fuse ? &fr : nullptr);
    if (fuse) continue;
    if (xf_bytes) {
      PROF(e, "reduce_affine", (double)n * H * H * 3 * e->es + 3.0 * H * H * 4 * (double)n / S, 0, st,
           dp::launch_reduce_affine(e->d_input, e->adv_x, e->xf_d, rects, a->grad_adv, S, n0, n, H, H, e->Cpd, e->bf16, st));
    } else {
      PROF(e, "reduce_k1t", (double)n * H * H * 3 * e->es + 3.0 * H * H * 4 * (double)n / S, 0, st,
           dp::launch_reduce(e->d_input, rects, a->grad_adv, B, S, n0, n, H, H, e->Cpd, e->bf16, st));
    }
    KERNEL_OK(); ++e->launches;
  }
  if (dual) {
    for (auto& L : e->lanes) {
      CUDA_OK(cudaEventRecord(L.done, L.stream));
      CUDA_OK(cudaStreamWaitEvent(user_st, L.done, 0));
    }
    e->use_lane(0);
    st = user_st;
  }
  // results -> host (pinned staging; the caller synchronises once)
  unsigned char* out = e->pin + L_.d2h_off;
  size_t off = 0;
  auto d2h = [&](const void* src, size_t bytes) { CUDA_OK(cudaMemcpyAsync(out + off, src, bytes, cudaMemcpyDeviceToHost, st)); off += (bytes + 15) / 16 * 16; };
  d2h(e->loss_d, (size_t)N * 4);
  d2h(e->preds_d, (size_t)N * 4);
  d2h(e->loss_struc, (size_t)B * 4);
  d2h(e->loss_density, (size_t)B * 4);
  d2h(e->group_lasso, (size_t)B * 4);
  d2h(e->l2, (size_t)B * 4);
}

static void attack_grad_impl(dp_engine* e, const dp_attack_args* a, cudaStream_t st) {
  NvtxRange nvtx_("dorpatch.attack_grad");
  if (!a) fail("null args");
  e->check_B(a->B);
  if (a->S < 1 || a->S_total < a->S) fail("bad S=%d / S_total=%d", a->S, a->S_total);
  if (!a->x || !a->mask || !a->pattern || !a->grad_adv || !a->y_host || !a->targeted_host) fail("null pointer in dp_attack_args");
  const int B = a->B, S = a->S, N = B * S;
  e->ensure_samples(N);
  if (!a->xform_host) e->ensure_net_in_all(N);
  // per-sample labels / criterion flags / rectangles -> pinned staging.  Layout:
  // [H2D region: ys | tg | rects | xforms][D2H region: results]; the regions never overlap.
  GradLayout L_;
  L_.rect_bytes = a->rects_host ? (size_t)N * 16 * sizeof(int16_t) : 0;
  L_.xf_bytes = a->xform_host ? (size_t)N * 8 * sizeof(float) : 0;
  const size_t h2d_bytes = (((size_t)N * 5 + 15) / 16) * 16 + L_.rect_bytes + L_.xf_bytes;
  L_.d2h_off = (h2d_bytes + 255) / 256 * 256;
  e->ensure_pin(L_.d2h_off + (size_t)N * 8 + (size_t)B * 16 + 512);
  L_.ys = (int32_t*)e->pin;
  L_.tg = (uint8_t*)(L_.ys + N);
  L_.rp = (unsigned char*)e->pin + (((size_t)N * 5 + 15) / 16) * 16;
  for (int b = 0; b < B; ++b)
    if (a->y_host[b] < 0 || a->y_host[b] >= e->K) fail("label %lld of image %d outside [0,%d)", (long long)a->y_host[b], b, e->K);
  for (int b = 0; b < B; ++b)
    for (int s = 0; s < S; ++s) { L_.ys[b * S + s] = (int32_t)a->y_host[b]; L_.tg[b * S + s] = a->targeted_host[b]; }
  if (L_.rect_bytes) memcpy(L_.rp, a->rects_host, L_.rect_bytes);
  if (L_.xf_bytes) memcpy(L_.rp + L_.rect_bytes, a->xform_host, L_.xf_bytes);

  bool done = false;
  if (e->graphs_on && !e->prof_on && !L_.xf_bytes) {
    dp_engine::GraphKey key{B, S, a->S_total, a->stage, a->x, a->mask, a->pattern, a->grad_adv, a->eps, a->confidence, L_.rect_bytes ? 1 : 0};
    dp_engine::GraphEnt& ent = e->graphs[key];
    ++ent.calls;
    if (ent.exec != nullptr) {
      CUDA_OK(cudaGraphLaunch(ent.exec, st));
      e->launches += ent.launches; ++e->graph_replays;
      done = true;
    } else if (!ent.failed && ent.calls >= 2) {          // call 1 ran eagerly: every plan / algorithm choice exists now
      const int64_t l0 = e->launches;
      cudaGraph_t graph = nullptr;
      // the legacy / per-thread default streams (PyTorch's default current stream) cannot be captured: record the
      // sequence on an engine-owned stream instead; the instantiated graph launches on the caller's stream either way
      cudaStream_t cs = (st == nullptr || st == cudaStreamLegacy || st == cudaStreamPerThread) ? e->cap_stream : st;
      const cudaError_t cb = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
      bool ok = cb == cudaSuccess;
      if (ok) {
        try { attack_grad_enqueue(e, a, L_, cs); } catch (const std::exception& ex) { ok = false; e->graph_msg = std::string("enqueue: ") + ex.what(); }
        const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
        if (ce != cudaSuccess || graph == nullptr) { if (ok) e->graph_msg = std::string("end capture: ") + cudaGetErrorString(ce); ok = false; }
      } else e->graph_msg = std::string("begin capture: ") + cudaGetErrorString(cb);
      if (ok) {
        const cudaError_t ci = cudaGraphInstantiate(&ent.exec, graph, 0);
        if (ci != cudaSuccess) { ok = false; ent.exec = nullptr; e->graph_msg = std::string("instantiate: ") + cudaGetErrorString(ci); }
      }
      if (graph) cudaGraphDestroy(graph);
      if (ok) {
        ent.launches = e->launches - l0;
        CUDA_OK(cudaGraphLaunch(ent.exec, st));
        ++e->graph_replays;
        done = true;
      } else {
        cudaGetLastError();                                // clear the capture error; fall back to eager launches for this signature
        e->launches = l0;
        e->use_lane(0);
        ent.failed = true;
      }
    }
  }
  if (!done) attack_grad_enqueue(e, a, L_, st);
  CUDA_OK(cudaStreamSynchronize(st));
  unsigned char* out = e->pin + L_.d2h_off;
  size_t off = 0;
  auto take = [&](void* dst, size_t bytes, bool want) { if (want && dst) memcpy(dst, out + off, bytes); off += (bytes + 15) / 16 * 16; };
  take(a->loss_adv_host, (size_t)N * 4, true);
  take(a->preds_host, (size_t)N * 4, true);
  take(a->loss_struc_host, (size_t)B * 4, true);
  take(a->loss_density_host, (size_t)B * 4, a->stage == 0);
  take(a->group_lasso_host, (size_t)B * 4, a->stage == 0);
  take(a->l2_host, (size_t)B * 4, true);
}

static void attack_update_impl(dp_engine* e, const dp_update_args* u, cudaStream_t st) {
  NvtxRange nvtx_("dorpatch.attack_update");
  if (!u) fail("null args");
  e->check_B(u->B);
  if (!u->x || !u->mask || !u->pattern || !u->grad_adv || !u->lr_host || !u->structured_host) fail("null pointer in dp_update_args");
  if (u->stage == 0 && !u->coeff_gl_host) fail("coeff_gl_host is required in stage 0");
  const int B = u->B;
  e->ensure_pin((size_t)B * 12 + 64);
  float* h = (float*)e->pin;
  for (int b = 0; b < B; ++b) { h[b] = u->lr_host[b]; h[B + b] = u->structured_host[b]; h[2 * B + b] = u->coeff_gl_host ? u->coeff_gl_host[b] : 0.f; }
  CUDA_OK(cudaMemcpyAsync(e->lr_d, h, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->structured_d, h + B, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->coeff_d, h + 2 * B, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  PROF(e, "update_k3", (double)B * e->H * e->H * 4 * (u->stage == 0 ? 15.0 : 13.0), 0, st,
       dp::launch_update(u->x, u->mask, u->pattern, u->grad_adv, e->dLs, e->scale, e->win_dev, e->grp_ss, e->lr_d, e->structured_d,
                         e->coeff_d, u->density, u->clip_min, u->clip_max, u->stage, u->grad_pattern_out, u->grad_mask_out, u->grad_pattern_bias, B, e->H, e->H, UNIT, st));
  KERNEL_OK(); ++e->launches;
  CUDA_OK(cudaStreamSynchronize(st));   // `pin` may be reused by the next call
}

int32_t dp_attack_grad(dp_engine* e, const dp_attack_args* a, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  attack_grad_impl(e, a, (cudaStream_t)stream);
  DP_CATCH
}

int32_t dp_attack_update(dp_engine* e, const dp_update_args* u, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  attack_update_impl(e, u, (cudaStream_t)stream);
  DP_CATCH
}

int32_t dp_attack_step_host(dp_engine* e, const dp_attack_args* g, const dp_update_args* u, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (!g || !u) fail("null args");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  e->check_B(g->B);
  const size_t B = (size_t)g->B, HW = (size_t)e->H * e->H;
  CUDA_OK(cudaMemcpyAsync(e->host_x, g->x, B * 3 * HW * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->host_mask, g->mask, B * HW * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->host_pattern, g->pattern, B * 3 * HW * 4, cudaMemcpyHostToDevice, st));
  dp_attack_args ga = *g;
  ga.x = e->host_x; ga.mask = e->host_mask; ga.pattern = e->host_pattern; ga.grad_adv = e->host_G;
  attack_grad_impl(e, &ga, st);
  dp_update_args ua = *u;
  ua.x = e->host_x; ua.mask = e->host_mask; ua.pattern = e->host_pattern; ua.grad_adv = e->host_G;
  ua.grad_pattern_out = nullptr; ua.grad_mask_out = nullptr; ua.grad_pattern_bias = nullptr;
  attack_update_impl(e, &ua, st);
  CUDA_OK(cudaMemcpyAsync(u->mask, e->host_mask, B * HW * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaMemcpyAsync(u->pattern, e->host_pattern, B * 3 * HW * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  DP_CATCH
}

int32_t dp_net_forward_backward(dp_engine* e, const float* z, int32_t N, float* logits_dev, const float* dlogits_dev,
                                float* dz_dev, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (N < 1 || N > e->chunk) fail("N=%d outside [1, chunk=%d]", N, e->chunk);
  dp::launch_pack_nchw(z, e->net_in, N, e->H, e->H, e->Cp, e->bf16, st); KERNEL_OK(); ++e->launches;
  e->forward(N, e->net_in, dlogits_dev != nullptr, st);
  if (logits_dev) CUDA_OK(cudaMemcpyAsync(logits_dev, e->logits, (size_t)N * e->K * 4, cudaMemcpyDeviceToDevice, st));
  if (dlogits_dev) {
    if (!dz_dev) fail("dz_dev is required when dlogits_dev is given");
    e->backward(N, dlogits_dev, st);
    dp::launch_unpack_nhwc(e->d_input, dz_dev, N, e->H, e->H, e->Cpd, e->bf16, st); KERNEL_OK(); ++e->launches;
  }
  DP_CATCH
}

/* ---- failed-mask sets on the device (attack.py:96,187-190,259-267) ------------------------------------- */
int32_t dp_failed_set_write(dp_engine* e, int32_t b, const int32_t* idx_host, int32_t n, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (b < 0 || b >= e->cfg.max_images) fail("image %d outside [0, max_images=%d)", b, e->cfg.max_images);
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<uint32_t> w(dp_engine::FAILED_WORDS, 0u);
  for (int i = 0; i < n; ++i) {
    if (idx_host[i] < 0 || idx_host[i] >= dp_engine::FAILED_WORDS * 32) fail("mask index %d outside [0, %d)", idx_host[i], dp_engine::FAILED_WORDS * 32);
    w[idx_host[i] >> 5] |= 1u << (idx_host[i] & 31);
  }
  CUDA_OK(cudaMemcpyAsync(e->failed_bits + (size_t)b * dp_engine::FAILED_WORDS, w.data(), w.size() * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaStreamSynchronize(st));
  DP_CATCH
}

int32_t dp_failed_set_update(dp_engine* e, int32_t B, int32_t S, const int32_t* idx_host, const int32_t* nff_host, const uint8_t* active_host,
                             const float* loss_host, float thresh, int32_t* count_host, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  e->check_B(B);
  if (S < 1 || !idx_host || !nff_host || !active_host || !count_host) fail("dp_failed_set_update: bad arguments");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const int N = B * S;
  if (N > e->failed_cap) {
    e->failed_cap = std::max(N, e->failed_cap * 2);
    e->failed_idx = (int32_t*)e->dmalloc((size_t)e->failed_cap * 4);
    e->failed_loss = (float*)e->dmalloc((size_t)e->failed_cap * 4);
  }
  for (int i = 0; i < N; ++i)
    if (idx_host[i] < 0 || idx_host[i] >= dp_engine::FAILED_WORDS * 32) fail("mask index %d outside [0, %d)", idx_host[i], dp_engine::FAILED_WORDS * 32);
  CUDA_OK(cudaMemcpyAsync(e->failed_idx, idx_host, (size_t)N * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->failed_nff, nff_host, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->failed_active, active_host, (size_t)B, cudaMemcpyHostToDevice, st));
  const float* loss = e->loss_d;                       // default: the per-sample CW losses the last dp_attack_grad left on the device
  if (loss_host != nullptr) {                          // EOT-sharded runs pass the all-gathered losses
    CUDA_OK(cudaMemcpyAsync(e->failed_loss, loss_host, (size_t)N * 4, cudaMemcpyHostToDevice, st));
    loss = e->failed_loss;
  } else if (N > e->cap_samples) fail("dp_failed_set_update: no device losses for %d samples", N);
  dp::launch_failed_update(e->failed_bits, dp_engine::FAILED_WORDS, e->failed_idx, loss, e->failed_nff, e->failed_active, B, S, thresh,
                           e->failed_count, st);
  KERNEL_OK(); ++e->launches;
  CUDA_OK(cudaMemcpyAsync(count_host, e->failed_count, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  DP_CATCH
}

int32_t dp_failed_set_read(dp_engine* e, int32_t b, int32_t* idx_host_out, int32_t cap, int32_t* n_out, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (b < 0 || b >= e->cfg.max_images) fail("image %d outside [0, max_images=%d)", b, e->cfg.max_images);
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<uint32_t> w(dp_engine::FAILED_WORDS);
  CUDA_OK(cudaMemcpyAsync(w.data(), e->failed_bits + (size_t)b * dp_engine::FAILED_WORDS, w.size() * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  int n = 0;
  for (int i = 0; i < dp_engine::FAILED_WORDS * 32; ++i)
    if (w[i >> 5] & (1u << (i & 31))) { if (n < cap && idx_host_out) idx_host_out[n] = i; ++n; }
  if (n_out) *n_out = n;
  if (n > cap && idx_host_out) fail("dp_failed_set_read: %d indices, buffer holds %d", n, cap);
  DP_CATCH
}

/* ---- op-level test hooks (tests/test_gpu_ops.py, tests/test_gpu_patch_kernels.py) --------------------- */
int32_t dp_debug_k1t(dp_engine* e, const void* dz, const int16_t* rects_host, int32_t B, int32_t S, int32_t n0, int32_t n,
                     float* G, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (!dz || !G) fail("dp_debug_k1t: null pointer");
  if (B < 1 || S < 1 || n0 < 0 || n < 1 || n0 + n > B * S) fail("dp_debug_k1t: samples [%d, %d) outside [0, %d)", n0, n0 + n, B * S);
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  e->h2d_samples(rects_host, B * S, st);
  const int16_t* rects = rects_host ? e->rects_d : nullptr;
  // the K1^T of dp_attack_grad's chunk loop for this engine (G is not cleared: the first launch of an image overwrites it)
  if (e->stem_bwd_fused_ok()) dp::launch_stem_bwd_reduce(dz, e->stem.w, e->stem.cin_pad, rects, G, B, S, n0, n, e->H, e->H, st);
  else dp::launch_reduce(dz, rects, G, B, S, n0, n, e->H, e->H, e->Cpd, e->bf16, st);
  KERNEL_OK(); ++e->launches;
  DP_CATCH
}

int32_t dp_debug_cw(dp_engine* e, const float* logits, const int32_t* y, const uint8_t* targeted, float confidence, float w,
                    float* loss, int32_t* preds, float* dlogits, int32_t N, int32_t K, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  if (!logits || N < 1 || K < 1) fail("dp_debug_cw: bad arguments");
  if (loss && (!y || !targeted)) fail("dp_debug_cw: the loss needs labels and criterion flags");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  dp::launch_cw(logits, y, targeted, confidence, w, loss, preds, dlogits, N, K, st);
  KERNEL_OK(); ++e->launches;
  DP_CATCH
}

int32_t dp_debug_k1_tuning(int32_t rows, int32_t sg, int32_t mode) {
  dp::set_expand_tuning(rows, sg, mode);
  return 0;
}

int32_t dp_debug_k1_last(int32_t* out4) {
  if (!out4) return 1;
  int v[4]; dp::get_expand_last(v);
  for (int i = 0; i < 4; ++i) out4[i] = v[i];
  return 0;
}

int32_t dp_debug_gn_gemm(dp_engine* e, const void* x, const void* w_nk, const float* stats, const float* gamma, const float* beta,
                         const void* shortcut, void* out, int32_t N, int32_t P, int32_t K, int32_t Nout, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (!dp::gn_gemm_supported(P, K, Nout)) fail("dp_debug_gn_gemm: shape P=%d K=%d Nout=%d not supported by the tcgen05 kernel", P, K, Nout);
  void* packed = nullptr;
  CUDA_OK(cudaMalloc(&packed, (size_t)Nout * K * 2));
  dp::launch_gn_gemm_pack(w_nk, packed, Nout, K, st);
  const bool ok = dp::launch_gn_gemm_forward(x, packed, stats, gamma, beta, shortcut, out, N, P, K, Nout, st);
  cudaError_t err = cudaStreamSynchronize(st);
  cudaFree(packed);
  if (!ok) fail("dp_debug_gn_gemm: launch refused");
  CUDA_OK(err);
  KERNEL_OK(); e->launches += 2;
  DP_CATCH
}

int32_t dp_debug_gn(dp_engine* e, const void* x, const void* dy, const void* addend, const float* gamma, const float* beta,
                    int32_t gamma_positive, void* y, void* dx, float* stats, int32_t N, int32_t P, int32_t C, void* stream) {
  DP_TRY
  if (!e) fail("null engine");
  CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (N > e->chunk) fail("dp_debug_gn: N=%d exceeds chunk=%d (statistics scratch)", N, e->chunk);
  if (y == nullptr) {   // statistics only: the pass in front of the tcgen05 GEMM / the classifier head
    dp::launch_gn_stats(x, e->gn_partial, stats, N, P, C, e->bf16, st); KERNEL_OK();
    e->launches += 2;
    return 0;
  }
  dp::launch_gn_relu_forward(x, y, gamma, beta, e->gn_partial, stats, N, P, C, e->bf16, st); KERNEL_OK();
  if (dy != nullptr) { dp::launch_gn_relu_backward(dy, x, addend, dx, gamma, beta, stats, e->gn_partial, N, P, C, e->bf16, st, gamma_positive != 0); KERNEL_OK(); }
  e->launches += 4;
  DP_CATCH
}

}  // extern "C"
