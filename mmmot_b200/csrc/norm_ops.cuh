// GroupNorm statistics -> per-(group, channel) affine, and a few small shared kernels.
// Compiled in engines.cu only: the launchers below have external linkage (see engines.cuh).
#pragma once
#include "engines.cuh"

// stats[G][C][2] (sum, sumsq over the group's columns, fp64) -> sc/sh[G][C] so that
//   GroupNorm(x)[c] = x*sc + sh,   sc = gamma[c]*rstd,  sh = beta[c] - mean*sc.
// The statistics row of group g is stats[g*stats_ld + c_off + c] (lets two GroupNorms share one
// stacked contraction).
// cpg = channels per normalisation group (1: GroupNorm(C,C); C: GroupNorm(1,C); 32: GroupNorm(16,512)).
// count = columns per group: cnt[g] if cnt != null else `uniform`.  Biased variance, eps 1e-5
// (torch.nn.GroupNorm semantics; a 1-element group yields exactly beta, SURVEY F3).
// Fixed-order reduction of the contraction engine's per-tile partials: stats[g][c] = sum over the
// group's tiles (ascending) of part[tile][c].  Group g owns tiles [g*tpg, (g+1)*tpg) (uniform) or
// [gstart[g], gstart[g+1]) (table tiling).
// `mult` = partials per tile (1 for the FP32 engine, 2 for the tcgen05 engines).
// CTA = 32 channels x 8 tile stripes: stripe y sums tiles t0+y, t0+y+8, ... in order, then the 8 stripe sums are
// added in stripe order -> a fixed summation tree, independent of scheduling.
static __global__ void __launch_bounds__(256) stats_reduce_kernel(const double2* __restrict__ part, int M, int G,
                                                                  int tpg, const int* __restrict__ gstart, int mult,
                                                                  double* __restrict__ stats) {
  __shared__ double2 red[8][32];
  const int g = blockIdx.y;
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int t0 = (gstart ? gstart[g] : g * tpg) * mult, t1 = (gstart ? gstart[g + 1] : (g + 1) * tpg) * mult;
  double s1 = 0.0, s2 = 0.0;
  if (c < M) {
    for (int t = t0 + threadIdx.y; t < t1; t += 8) {
      const double2 v = part[(long)t * M + c];
      s1 += v.x;
      s2 += v.y;
    }
  }
  red[threadIdx.y][threadIdx.x] = make_double2(s1, s2);
  __syncthreads();
  if (threadIdx.y == 0 && c < M) {
    double a1 = 0.0, a2 = 0.0;
#pragma unroll
    for (int y = 0; y < 8; y++) { a1 += red[y][threadIdx.x].x; a2 += red[y][threadIdx.x].y; }
    stats[((long)g * M + c) * 2] = a1;
    stats[((long)g * M + c) * 2 + 1] = a2;
  }
}

int stats_reduce(const double2* part, int M, int G, int tpg, const int* gstart, double* stats, cudaStream_t st,
                 int mult) {
  dim3 grid(mm_cdiv(M, 32), G), block(32, 8);
  stats_reduce_kernel<<<grid, block, 0, st>>>(part, M, G, tpg, gstart, mult, stats);
  MM_LAUNCH_CHECK();
  return 0;
}

static __global__ void gn_finalize_kernel(const double* __restrict__ stats, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, const int* __restrict__ cnt,
                                   int uniform, int G, int C, int cpg, int stats_ld, int c_off,
                                   float* __restrict__ sc, float* __restrict__ sh, int* status) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= G * C) return;
  int g = idx / C, c = idx - g * C;
  int c0 = c / cpg * cpg;
  double s1 = 0.0, s2 = 0.0;
  for (int k = 0; k < cpg; k++) {
    s1 += stats[((long)g * stats_ld + c_off + c0 + k) * 2];
    s2 += stats[((long)g * stats_ld + c_off + c0 + k) * 2 + 1];
  }
  double n = (double)(cnt ? cnt[g] : uniform) * cpg;
  double mean = s1 / n;
  double var = s2 / n - mean * mean;
  if (var < 0.0) var = 0.0;
  double rstd = 1.0 / sqrt(var + 1e-5);
  double a = (double)gamma[c] * rstd;
  sc[idx] = (float)a;
  sh[idx] = (float)((double)beta[c] - mean * a);
  // FP16 range guard for consumers that convert relu(x*sc + sh) to FP16 hi/lo without looking at it (gemm_gen.cuh):
  // a value of a group of n elements lies within sqrt(n) standard deviations of the group mean, so
  // |GN(x)| <= sqrt(n)*|gamma| + |beta|.  (Never triggers for sane checkpoints: needs |gamma| > ~250 at n = 65536.)
  if (status && sqrt(n) * fabs((double)gamma[c]) + fabs((double)beta[c]) >= 65504.0) atomicOr(status, 1);
}

int gn_finalize(const double* stats, const float* gamma, const float* beta, const int* cnt, int uniform, int G, int C,
                int cpg, float* sc, float* sh, cudaStream_t st, int stats_ld, int c_off, int* status) {
  gn_finalize_kernel<<<mm_cdiv((long)G * C, 256), 256, 0, st>>>(
      stats, gamma, beta, cnt, uniform, G, C, cpg, stats_ld ? stats_ld : C, c_off, sc, sh, status);
  MM_LAUNCH_CHECK();
  return 0;
}
