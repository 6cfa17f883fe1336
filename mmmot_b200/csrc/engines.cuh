// The contraction engines and their companion kernels as the stages see them: the parameter block, the operand modes
// and the launchers.  Kernels and launchers are defined in gemm_simt.cuh, gemm_tma.cuh, gemm_tma_px.cuh, gemm_gen.cuh,
// norm_ops.cuh and tc_ops.cuh, which only engines.cu includes, so each is compiled once.
#pragma once
#include <cuda_fp16.h>
#include <string.h>

#include "common.cuh"

// Operand generators of the FP32 engine (gemm_simt.cuh)
enum { XM_DIRECT = 0, XM_NORM_RELU = 1, XM_PAIR_MUL = 2, XM_PAIR_ABS = 3, XM_PAIR_SUB = 4, XM_CONV3 = 5 };

struct GemmP {
  // A operand: transposed weights Wt[K][ldw], output channels [m_base, m_base + M)
  const float* Wt;
  int ldw;
  const float* bias;  // [M] or null
  int M, K;
  // column tiling: uniform (tile_tab == null): every group has S columns; else table of
  // {group, first column (absolute), length, 0}
  int S;
  int tiles_per_group;
  const int4* tile_tab;
  int num_tiles;
  // X operand: X + g*x_gs + k*x_ks + col   (col = column inside group for uniform tiling,
  // absolute column for table tiling, where x_gs must be 0)
  const float* X;
  long x_gs, x_ks;
  const float* sc;  // [G][K]
  const float* sh;
  // pair generator: F[g][K][Lf], objs = columns [0,n), dets = columns [n, n+m)
  int n, m, Lf;
  // conv3x3: X = in[img][Cin][H][W], Y = out[img][M][H][W]; S = n_img*H*W in one group
  int H, W, Cin;
  // output: Y + g*y_gs + co*y_ms + col ; null = statistics only
  float* Y;
  long y_gs, y_ms;
  double2* part;        // [num_tiles][M] per-tile (sum, sumsq) partials or null; reduced in fixed
                        // order by stats_reduce (no atomics: results are run-to-run bit-identical)
  const float* addend;  // Y += addend[co*ld_add + seg[col]] or null
  const int* seg;
  int ld_add;
  int relu;
};

static inline GemmP gemm_defaults() {
  GemmP p;
  memset(&p, 0, sizeof(p));
  return p;
}

namespace tc {
constexpr int BN = 256;            // columns per tile of the tcgen05 engines
}
namespace gen {
// operand generators of the tcgen05 generated-operand engine (gemm_gen.cuh)
enum { GEN_PAIR_MUL = 0, GEN_PAIR_ABS = 1, GEN_PAIR_SUB = 2, GEN_NORM = 3, GEN_COPY = 4 };   // GEN_PAIR_* == MMMOT_AFF_*
}

// FP32 engine.  p.M must be a multiple of 64.
template <int MODE>
int gemm_simt_launch(const GemmP& p, cudaStream_t st);

// tcgen05 generated-operand engine.  g: M, K (multiple of 32, <= 512 for GEN_NORM), bias, S / tiles_per_group / num_tiles
// (uniform column tiling, 256 columns per tile) or tile_tab (GEN_NORM: ragged groups, absolute rows), x_gs (NORM: source
// rows per group), Y / y_gs / y_ms = fp32 channels-last output (or null), part = two GroupNorm partials per tile
// (stats_reduce(..., mult = 2)).  Wp = weights packed by weights.py::pack_tc.  PAIR: src = fcl [G][Lf][K]; NORM: src =
// [G*x_gs][ld_src] fp32, gsc/gsh [G][K].
template <int GEN>
int gemm_gen_launch(const GemmP& g, const uint4* Wp, float out_scale, const float* src, int ld_src, const float* gsc,
                    const float* gsh, int n, int m, int Lf, cudaStream_t st);

// tcgen05 TMA-fed engine, 1x1 contraction on planar FP16 (hi, lo) channels-last activations X_hi[rows][ldx], X_lo = X_hi +
// x_plane; output fp32 channels-last.  g: M, K (multiple of 32), bias, tiles, x_gs (rows per group), Y / y_ms / y_gs, part,
// addend...  segsum: if set, nothing is stored; relu(x*sc[g][co] + sh[g][co]) is summed per detection (g.seg) into
// segsum[det][M] as 2^-32 fixed point.  chunk_tab (seg_chunk_tab) is required with g.seg and g.addend or segsum.
int gemm_tma_launch_mat(const GemmP& g, const uint4* Wp, float out_scale, const __half* Xhi, long x_plane, long rows,
                        int ldx, cudaStream_t st, unsigned long long* segsum = nullptr, const int4* chunk_tab = nullptr);

// tcgen05 TMA-fed engine, 3x3 / pad 1 convolution on planar FP16 NHWC activations; output planar FP16 NHWC (ReLU via
// g.relu).  acc_scratch (fp32 [tiles*256][M], tiles = ceil(W/bx)*ceil(H/by)*ceil(n/bi) <= padded pixel count) enables
// K-segmentation: chains longer than mmmot_set_kseg() chunks of 32 are accumulated in several TMEM passes and summed in
// fp32 RN, which bounds the tensor core's round-toward-zero accumulation error (DESIGN.md §4.2).  nullptr = single pass.
// y_plane_pooled > 0 and did_pool: the 2x2 max-pool may be fused into the epilogue (*did_pool = 1 if it was; then the
// output is the pooled map and pool_sum, if set, receives its per-(image, channel) sums as 2^-32 fixed point).  Wpx: the
// compact N = 64 weight tiles (weights.py::pack_px) that let a 64-channel layer run on the pixel-major kernel.
int gemm_tma_launch_conv(const GemmP& g0, const uint4* Wp, float out_scale, const __half* Xhi, long x_plane, int n_img,
                         int H, int W, int C, __half* Yhi, long y_plane, cudaStream_t st, float* acc_scratch = nullptr,
                         long y_plane_pooled = 0, int* did_pool = nullptr, int* status = nullptr,
                         unsigned long long* pool_sum = nullptr, const uint4* Wpx = nullptr);

// Pixel-major kernel, 1x1 contraction with a 64-channel planar FP16 output (Y_lo = Y_hi + y_plane): g as for
// gemm_tma_launch_mat with M = y_ms = 64, Y = Y_hi and no partials, addend, tile table or segment sums.  Wpx = compact
// weights (weights.py::pack_px).
int gemm_tma_px_launch_mat(const GemmP& g, const uint4* Wpx, float out_scale, const __half* Xhi, long x_plane, long rows,
                           int ldx, long y_plane, int* status, cudaStream_t st);
// First VGG layer (3 -> 64 channels, 3x3 / pad 1) straight from the fp32 NCHW crops [n_img][3][H][W] on the pixel-major
// kernel, the taps generated in shared memory.  Crops it takes: gemm_tma_px_gen27_fits(H, W).
bool gemm_tma_px_gen27_fits(int H, int W);
int gemm_tma_px_launch_gen27(const float* crops, int n_img, int H, int W, const uint4* Wpx, float out_scale,
                             const float* bias, __half* Yhi, long y_plane, int* status, cudaStream_t st);

// Per (column tile, half) chunk descriptors of table-tiled contractions over ragged per-detection columns (tab[2 *
// num_tiles]), for gemm_tma_launch_mat's chunk_tab.
int seg_chunk_tab(const int4* tiles, int num_tiles, const int* seg, int4* tab, cudaStream_t st);

// GroupNorm statistics (norm_ops.cuh): fixed-order reduction of the engines' per-tile partials, and the per-(group,
// channel) affine they give.
int stats_reduce(const double2* part, int M, int G, int tpg, const int* gstart, double* stats, cudaStream_t st,
                 int mult = 1);
int gn_finalize(const double* stats, const float* gamma, const float* beta, const int* cnt, int uniform, int G, int C,
                int cpg, float* sc, float* sh, cudaStream_t st, int stats_ld = 0, int c_off = 0, int* status = nullptr);

// Channels-last companions of the tcgen05 engines (tc_ops.cuh)
int norm_split(const float* in, long ldi, const float* sc, const float* sh, int C, long rows, int rows_per_group,
               const int* seg, int L, __half* out, cudaStream_t st, int* status);
int transpose_f32(const float* src, float* dst, int rows, int cols, int groups, cudaStream_t st);
int feats_range_check(const float* f, long n, float limit, int* status, cudaStream_t st);
