// Library-wide entry points of libmmmot_sm100a.so (see include/mmmot_b200.h).
#include <algorithm>
#include <atomic>

#include "common.cuh"

static std::atomic<unsigned long long> g_launches{0};

void mm_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

extern "C" unsigned long long mmmot_launch_count(void) { return g_launches.load(); }

extern "C" int mmmot_abi_version(void) { return MMMOT_ABI_VERSION; }

int mm_sm_count(int* sms) {
  static std::atomic<int> cache[64];
  int dev = 0;
  MM_CUDA(cudaGetDevice(&dev));
  int v = cache[dev & 63].load(std::memory_order_relaxed);
  if (!v) {
    MM_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    cache[dev & 63].store(v, std::memory_order_relaxed);
  }
  *sms = v;
  return 0;
}

// ---- status block (first MM_STATUS_BYTES of every workspace) ----
extern "C" int mmmot_status_reset(void* workspace, void* stream) {
  if (!workspace) return MMMOT_E_ARG;
  MM_CUDA(cudaMemsetAsync(workspace, 0, MM_STATUS_BYTES, (cudaStream_t)stream));
  return 0;
}

extern "C" int mmmot_status_check(const void* workspace, void* stream) {
  if (!workspace) return MMMOT_E_ARG;
  int word = 0;
  MM_CUDA(cudaMemcpyAsync(&word, workspace, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  MM_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return (word & 1) ? MMMOT_E_RANGE : 0;
}

// ---- pinned-host fetch (see header): zero-copy read over PCIe by a kernel, stream-ordered ----
__global__ void fetch_pinned_i32_kernel(int* __restrict__ dst, const int* __restrict__ src, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) dst[i] = src[i];
}

extern "C" int mmmot_fetch_pinned_i32(int* dst_device, const int* src_pinned_host, long count, void* stream) {
  if (!dst_device || !src_pinned_host || count < 0) return MMMOT_E_ARG;
  if (count == 0) return 0;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, src_pinned_host) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
    (void)cudaGetLastError();
    return MMMOT_E_ARG;     // pageable (unregistered) or device memory
  }
  const void* dsrc = at.devicePointer;
  const int blocks = (int)std::min<long>(mm_cdiv(count, 256), 32);
  fetch_pinned_i32_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(dst_device, (const int*)dsrc, count);
  MM_LAUNCH_CHECK();
  return 0;
}

extern "C" int mmmot_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  MM_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  MM_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Optional per-launch timing of the hot kernels, used by bench.py for the roofline figures: CUDA events recorded on
// the launching stream around every tagged launch while enabled; mmmot_timing_collect*() synchronises on the
// events and returns the totals (per tag = per (stage, layer)).
#include <mutex>
#include <vector>

namespace {
std::mutex g_tmu;
bool g_timing = false;
struct Span { cudaEvent_t a, b; int tag; double flop, bytes; };
std::vector<Span> g_spans;
const char* const kTagNames[MM_T_COUNT] = {
    "vgg.conv0", "vgg.conv1", "vgg.conv2", "vgg.conv3", "vgg.conv4", "vgg.conv5", "vgg.conv6", "vgg.conv7", "vgg.conv8",
    "vgg.conv9", "vgg.conv10", "vgg.conv11", "vgg.conv12", "vgg.pool_mean_heads",
    "pointnet.l1_3to64", "pointnet.l2_64to64", "pointnet.l3_64to64", "pointnet.l4_64to128", "pointnet.norm_split",
    "pointnet.l5_128to1024_stats", "pointnet.l5_128to1024_segsum", "pointnet.head_64to512_stats",
    "pointnet.head_64to512_segsum",
    "affinity.l1_pair_512to1024", "affinity.newend_means", "affinity.l2_512to512", "affinity.l3_512to128",
    "affinity.logit", "lp.assign"};
}  // namespace

bool mm_timing_on() { return g_timing; }

void mm_timing_begin(cudaStream_t st, int tag, double flop, double bytes) {
  std::lock_guard<std::mutex> l(g_tmu);
  Span s;
  cudaEventCreate(&s.a);
  cudaEventCreate(&s.b);
  s.tag = tag; s.flop = flop; s.bytes = bytes;
  cudaEventRecord(s.a, st);
  g_spans.push_back(s);
}

void mm_timing_end(cudaStream_t st) {
  std::lock_guard<std::mutex> l(g_tmu);
  if (!g_spans.empty()) cudaEventRecord(g_spans.back().b, st);
}

extern "C" int mmmot_timing_enable(int on) {
  std::lock_guard<std::mutex> l(g_tmu);
  g_timing = on != 0;
  return 0;
}

extern "C" int mmmot_timing_tag_count(void) { return MM_T_COUNT; }
extern "C" const char* mmmot_timing_tag_name(int tag) { return (tag >= 0 && tag < MM_T_COUNT) ? kTagNames[tag] : ""; }

// ms / flop / bytes / launches: arrays of mmmot_timing_tag_count() entries (any may be null)
extern "C" int mmmot_timing_collect_tags(double* ms, double* flop, double* bytes, long* launches) {
  std::lock_guard<std::mutex> l(g_tmu);
  for (int t = 0; t < MM_T_COUNT; t++) {
    if (ms) ms[t] = 0.0;
    if (flop) flop[t] = 0.0;
    if (bytes) bytes[t] = 0.0;
    if (launches) launches[t] = 0;
  }
  int rc = 0;
  for (auto& s : g_spans) {
    float t = 0.f;
    cudaError_t e = cudaEventSynchronize(s.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, s.a, s.b);
    if (e != cudaSuccess) rc = (int)e;
    else {
      if (ms) ms[s.tag] += t;
      if (flop) flop[s.tag] += s.flop;
      if (bytes) bytes[s.tag] += s.bytes;
      if (launches) launches[s.tag] += 1;
    }
    cudaEventDestroy(s.a);
    cudaEventDestroy(s.b);
  }
  g_spans.clear();
  return rc;
}

// totals over the 3x3-conv contractions of the VGG trunk (layers 1..12), the dominant kernels
extern "C" int mmmot_timing_collect(double* total_ms, double* total_flop, long* launches) {
  double ms[MM_T_COUNT], fl[MM_T_COUNT];
  long n[MM_T_COUNT];
  int rc = mmmot_timing_collect_tags(ms, fl, nullptr, n);
  if (rc) return rc;
  double a = 0.0, b = 0.0;
  long c = 0;
  for (int t = MM_T_VGG0 + 1; t <= MM_T_VGG0 + 12; t++) { a += ms[t]; b += fl[t]; c += n[t]; }
  if (total_ms) *total_ms = a;
  if (total_flop) *total_flop = b;
  if (launches) *launches = c;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Engine selection + single-contraction test hook.
#include "engines.cuh"

namespace { int g_engine = 0; int g_dbg = 0; int g_kseg = 36; }
int mm_kseg_chunks() { return g_kseg; }
extern "C" int mmmot_set_kseg(int chunks) { if (chunks < 0) return MMMOT_E_ARG; g_kseg = chunks; return 0; }
int mm_debug_flags() { return g_dbg; }
extern "C" int mmmot_set_debug(int flags) {
  if (flags & ~15) return MMMOT_E_ARG;
  g_dbg = flags;
  return 0;
}

int mm_engine() { return g_engine; }

extern "C" int mmmot_set_engine(int engine) {
  if (engine < 0 || engine > 2) return MMMOT_E_ARG;
  g_engine = engine;
  return 0;
}

extern "C" int mmmot_debug_linear(const float* Wt, const void* Wp, float wp_scale, const float* bias, const float* X,
                                  float* Y, int M, int K, int S, int engine, void* stream) {
  (void)Wp; (void)wp_scale;
  if (!Wt || !X || !Y || M <= 0 || K <= 0 || S <= 0 || engine != 1) return MMMOT_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  GemmP p = gemm_defaults();
  p.Wt = Wt; p.ldw = M; p.bias = bias; p.M = M; p.K = K;
  p.S = S;
  p.X = X; p.x_ks = S;
  p.Y = Y; p.y_ms = S;
  p.tiles_per_group = mm_cdiv(S, 128); p.num_tiles = p.tiles_per_group;
  return gemm_simt_launch<XM_DIRECT>(p, st);
}

// Generated-operand tcgen05 engine (gemm_gen.cuh, GEN_NORM): Y[S][M] = relu(X[S][K]*sc + sh) W^T + bias with X, Y
// fp32 channels-last, sc/sh [K].
extern "C" int mmmot_debug_linear_gen(const void* Wp, float wp_scale, const float* bias, const float* X, const float* sc,
                                      const float* sh, float* Y, int M, int K, int S, void* stream) {
  if (!Wp || !X || !Y || !sc || !sh || M <= 0 || K <= 0 || S <= 0) return MMMOT_E_ARG;
  GemmP p = gemm_defaults();
  p.bias = bias; p.M = M; p.K = K;
  p.S = S; p.tiles_per_group = mm_cdiv(S, tc::BN); p.num_tiles = p.tiles_per_group;
  p.x_gs = S;
  p.Y = Y; p.y_gs = S; p.y_ms = M;
  return gemm_gen_launch<gen::GEN_NORM>(p, (const uint4*)Wp, wp_scale, X, K, sc, sh, 0, 0, 0, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Test hooks for the TMA-fed tcgen05 engine (planar FP16 hi/lo channels-last operands).
// Y[rows][M] fp32 (channels-last) = X W^T + bias ; X given as planes Xhi[rows][K], Xlo = Xhi + rows*K
extern "C" int mmmot_debug_linear_planar(const void* Wp, float wp_scale, const float* bias, const void* Xhi,
                                         float* Y, int M, int K, long rows, void* stream) {
  if (!Wp || !Xhi || !Y || M <= 0 || K <= 0 || rows <= 0) return MMMOT_E_ARG;
  GemmP p = gemm_defaults();
  p.bias = bias; p.M = M; p.K = K;
  p.S = (int)rows; p.tiles_per_group = mm_cdiv(rows, tc::BN); p.num_tiles = p.tiles_per_group;
  p.Y = Y; p.y_ms = M;
  return gemm_tma_launch_mat(p, (const uint4*)Wp, wp_scale, (const __half*)Xhi, rows * (long)K, rows, K,
                             (cudaStream_t)stream);
}

// 3x3 conv + bias + ReLU on planar FP16 NHWC: X planes [2][n][H][W][C] -> Y planes [2][n][H][W][M]
extern "C" int mmmot_debug_conv_planar(const void* Wp, float wp_scale, const float* bias, const void* Xhi, void* Yhi,
                                       int n_img, int H, int W, int C, int M, float* kseg_scratch, void* stream) {
  if (!Wp || !Xhi || !Yhi) return MMMOT_E_ARG;
  GemmP p = gemm_defaults();
  p.bias = bias; p.M = M; p.relu = 1;
  return gemm_tma_launch_conv(p, (const uint4*)Wp, wp_scale, (const __half*)Xhi, (long)n_img * H * W * C, n_img, H, W, C,
                              (__half*)Yhi, (long)n_img * H * W * M, (cudaStream_t)stream, kseg_scratch);
}
