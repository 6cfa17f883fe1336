// Small kernels of the tensor-core (channels-last) pipeline: activations between tcgen05 contractions
// are stored [row][channel], fp32 before the GroupNorm statistics are known and packed FP16 (hi|lo)
// after normalisation.
// Compiled in engines.cu only: the launchers below have external linkage (see engines.cuh).
#pragma once
#include "engines.cuh"

// out planes [2][rows][C] (hi, lo) = split(relu(in[row][c]*sc[g][c] + sh[g][c])),
// g = seg ? seg[row] / L : row / rows_per_group.  GroupNorm + ReLU of the producer layer applied once per
// element and emitted as the FP16 hi/lo planes the next contraction's TMA loads read.
static __global__ void norm_split_kernel(const float* __restrict__ in, long ldi, const float* __restrict__ sc,
                                         const float* __restrict__ sh, int C, long rows, int rows_per_group,
                                         const int* __restrict__ seg, int L, __half* __restrict__ out, int* status) {
  const int c4n = C >> 2;
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * c4n) return;
  const long row = idx / c4n;
  const int c = (int)(idx - row * c4n) * 4;
  const int g = seg ? seg[row] / L : (int)(row / rows_per_group);
  const float4 x = *reinterpret_cast<const float4*>(in + row * ldi + c);
  const float4 a = *reinterpret_cast<const float4*>(sc + (long)g * C + c);
  const float4 b = *reinterpret_cast<const float4*>(sh + (long)g * C + c);
  float4 y;
  y.x = fmaxf(fmaf(x.x, a.x, b.x), 0.f); y.y = fmaxf(fmaf(x.y, a.y, b.y), 0.f);
  y.z = fmaxf(fmaf(x.z, a.z, b.z), 0.f); y.w = fmaxf(fmaf(x.w, a.w, b.w), 0.f);
  split4_store(y, out + row * C + c, out + rows * C + row * C + c, status);
}

int norm_split(const float* in, long ldi, const float* sc, const float* sh, int C, long rows, int rows_per_group,
               const int* seg, int L, __half* out, cudaStream_t st, int* status) {
  norm_split_kernel<<<mm_cdiv(rows * (C / 4), 256), 256, 0, st>>>(in, ldi, sc, sh, C, rows, rows_per_group, seg, L, out,
                                                                 status);
  MM_LAUNCH_CHECK();
  return 0;
}

// dst[g][col][row] = src[g][row][col]   (small matrices: feature stacks 512 x L, U 512 x ndet)
static __global__ void transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols,
                                        int groups) {
  __shared__ float tile[32][33];
  const int g = blockIdx.z;
  const float* s = src + (long)g * rows * cols;
  float* d = dst + (long)g * rows * cols;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[i][threadIdx.x] = s[(long)r * cols + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < rows && c < cols) d[(long)c * rows + r] = tile[threadIdx.x][i];
  }
}
int transpose_f32(const float* src, float* dst, int rows, int cols, int groups, cudaStream_t st) {
  dim3 grid(mm_cdiv(cols, 32), mm_cdiv(rows, 32), groups), block(32, 8);
  transpose_kernel<<<grid, block, 0, st>>>(src, dst, rows, cols, groups);
  MM_LAUNCH_CHECK();
  return 0;
}

// Range guard of the pairwise producers (gemm_gen.cuh GEN_PAIR_*), which convert f_i (*|-) f_j to FP16 hi/lo unseen:
// flag the status word when a feature is large enough for the op to reach 65504 (|f| >= 255.9 for the product,
// |f| >= 65504 for the differences).  feats [n] fp32.
static __global__ void feats_range_kernel(const float* __restrict__ f, long n, float limit, int* status) {
  float amax = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    amax = fmaxf(amax, fabsf(f[i]));
  if (status && !(amax < limit)) atomicOr(status, 1);
}
int feats_range_check(const float* f, long n, float limit, int* status, cudaStream_t st) {
  feats_range_kernel<<<148, 256, 0, st>>>(f, n, limit, status);
  MM_LAUNCH_CHECK();
  return 0;
}
