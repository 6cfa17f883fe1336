// Shared helpers for libmmmot_sm100a.so (sm_100a only; no torch headers).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mmmot_b200.h"

#define MM_CUDA(x)                                    \
  do {                                                \
    cudaError_t _e = (x);                             \
    if (_e != cudaSuccess) return (int)_e;            \
  } while (0)

#define MM_LAUNCH_CHECK()                             \
  do {                                                \
    mm_count_launch();                                \
    cudaError_t _e = cudaGetLastError();              \
    if (_e != cudaSuccess) return (int)_e;            \
  } while (0)

#define MM_TRY(x)                                     \
  do {                                                \
    int _r = (x);                                     \
    if (_r != 0) return _r;                           \
  } while (0)

void mm_count_launch();
int mm_debug_flags();
int mm_kseg_chunks();  // K-segment length (in 32-wide chunks) of the tcgen05 conv engine, 0 = off (mmmot_set_kseg)
int mm_engine();  // 0 auto, 1 FP32 FFMA engine, 2 tcgen05 engine (mmmot_set_engine)
// Per-launch timing hook (mmmot_timing_*): every hot kernel of the path is bracketed by CUDA events on the launching
// stream while timing is enabled, tagged with (stage, layer) and its ALGORITHMIC work (FLOPs, compulsory HBM bytes).
enum {
  MM_T_VGG0 = 0,          // .. +12 : VGG conv i (tag 0 includes its im2col pre-pass)
  MM_T_VGG_POOL = 13,     // 2x2 max-pools + SkipPool plane means + heads
  MM_T_PN_L1 = 14,        // PointNet 3 -> 64 (statistics + apply)
  MM_T_PN_L2 = 15, MM_T_PN_L3 = 16, MM_T_PN_L4 = 17,
  MM_T_PN_NORM = 18,      // GroupNorm+ReLU -> FP16 planes passes between PointNet layers
  MM_T_PN_L5A = 19, MM_T_PN_L5B = 20,        // 128 -> 1024: statistics pass, normalise + segment-sum pass
  MM_T_PN_HEADA = 21, MM_T_PN_HEADB = 22,    // head 64 -> 512, two passes
  MM_T_AFF_L1 = 23, MM_T_AFF_MEAN = 24, MM_T_AFF_L2 = 25, MM_T_AFF_L3 = 26, MM_T_AFF_LOGIT = 27,
  MM_T_LP = 28,
  MM_T_COUNT = 29
};
bool mm_timing_on();
void mm_timing_begin(cudaStream_t st, int tag, double flop, double bytes);
void mm_timing_end(cudaStream_t st);

// SM count of the CURRENT device (cached per device; the library may be used on several GPUs from one process)
int mm_sm_count(int* sms);
// Opt a kernel into > 48 KB of dynamic shared memory, once per (kernel, device): `done` is a per-call-site bit mask
// indexed by device ordinal.  Safe to race: setting the attribute twice is harmless.
#include <atomic>
template <typename K>
static inline int mm_ensure_smem(K kernel, size_t bytes, std::atomic<unsigned long long>& done) {
  int dev = 0;
  MM_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if (!(done.load(std::memory_order_acquire) & bit)) {
    MM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done.fetch_or(bit, std::memory_order_release);
  }
  return 0;
}

static inline size_t mm_align(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
static inline int mm_cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// Bump allocator over the caller-provided workspace.  The first MM_STATUS_BYTES of EVERY workspace are the status
// block (word 0 = range flag, see mmmot_status_reset / mmmot_status_check): all stages carve behind it, so a flag
// raised by one stage survives the stages that reuse the workspace after it.
constexpr size_t MM_STATUS_BYTES = 256;
struct MmArena {
  char* base;
  size_t cap, off;
  bool dry;  // dry run: only measure
  MmArena(void* p, size_t c) : base((char*)p), cap(c), off(MM_STATUS_BYTES), dry(p == nullptr) {}
  int* status() const { return dry ? nullptr : reinterpret_cast<int*>(base); }
  template <typename T>
  T* take(size_t n) {
    size_t bytes = mm_align(n * sizeof(T));
    char* r = dry ? nullptr : base + off;
    off += bytes;
    return (T*)r;
  }
  bool ok() const { return dry || off <= cap; }
};

__device__ __forceinline__ float mm_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

// FP16 range guard.  Activations enter the tensor cores as FP16 hi/lo pairs; cvt.rn.satfinite clamps |x| >= 65504
// silently, so every conversion site tracks the largest magnitude it converted and raises bit 0 of the workspace
// status word once per thread when the clamp was hit.  The host reads it with mmmot_status_check -> MMMOT_E_RANGE.
constexpr float MM_F16_MAX = 65504.f;
__device__ __forceinline__ void mm_range_flag(int* status, float amax) {
  if (status && !(amax < MM_F16_MAX)) atomicOr(status, 1);      // also catches NaN
}
// packed variant: acc = running max of |hi| over f16x2 words (starts at 0)
__device__ __forceinline__ void mm_range_track2(uint32_t& acc, uint32_t hi2) {
  asm("{\n\t.reg .b32 t;\n\tabs.f16x2 t, %1;\n\tmax.NaN.f16x2 %0, %0, t;\n\t}" : "+r"(acc) : "r"(hi2));
}
__device__ __forceinline__ void mm_range_flag2(int* status, uint32_t acc) {
  if (status && ((acc & 0xFFFFu) >= 0x7BFFu || (acc >> 16) >= 0x7BFFu)) atomicOr(status, 1);
}

// x -> FP16 hi/lo pair, x = hi + lo + O(2^-22 |x|), the operand format of the tcgen05 engines
__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
  unsigned short a, b;
  asm("{\n\t.reg .f32 f;\n\t"
      "cvt.rn.satfinite.f16.f32 %0, %2;\n\t"
      "cvt.f32.f16 f, %0;\n\t"
      "sub.f32 f, %2, f;\n\t"
      "cvt.rn.satfinite.f16.f32 %1, f;\n\t}"
      : "=h"(a), "=h"(b)
      : "f"(x));
  hi = __ushort_as_half(a);
  lo = __ushort_as_half(b);
}
__device__ __forceinline__ void split4_store(float4 x, __half* hi, __half* lo, int* status) {
  mm_range_flag(status, fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
  __half h[4], l[4];
  split_f16(x.x, h[0], l[0]); split_f16(x.y, h[1], l[1]);
  split_f16(x.z, h[2], l[2]); split_f16(x.w, h[3], l[3]);
  *reinterpret_cast<uint2*>(hi) = *reinterpret_cast<uint2*>(h);
  *reinterpret_cast<uint2*>(lo) = *reinterpret_cast<uint2*>(l);
}

