// PointNet encoder over ragged per-detection LiDAR point sets.
// Replaces reference modules/point_net.py:25-44 (PointNet_v1.forward) and :115-153
// (PointNetfeatGN.forward).  Uses two identities proven in SURVEY F4 / B-9:
//   * both STN transforms are input-independent constants -> folded into conv1 / conv2 / head
//     weights by the host weight packer (the STN convs are never executed);
//   * the 1088-wide head conv splits into a 64-wide per-point part plus a per-detection
//     addend  Wh[:,64:] * mean_det(x5)  (1088 -> 64 MACs per point per output channel).
// Per-detection pooling is a MEAN (SURVEY F5).  One frame-pair = one GroupNorm domain.
#include <vector>

#include "engines.cuh"

namespace {

__global__ void transpose_points_kernel(const float* __restrict__ pts, float* __restrict__ xt, long P) {
  long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  xt[p] = pts[p * 3];
  xt[P + p] = pts[p * 3 + 1];
  xt[2 * P + p] = pts[p * 3 + 2];
}

// First trunk layer (3 -> 64) on the tensor-core path.  With K = 3 a contraction kernel is all epilogue, so the
// layer is never materialised in fp32: one kernel accumulates its GroupNorm statistics, a second recomputes it,
// applies GroupNorm + ReLU and writes the FP16 hi/lo planes layer 2's TMA loads read.  Both evaluate
//   y = fma(w2, z, fma(w1, y, fma(w0, x, b)))  in this order, so the statistics describe exactly the values normalised.
// pts [P][3], wt [3][64], part[(tile*2 + h)*64 + c] (h = first / second half of the tile's points, fp64 sums).
__global__ void __launch_bounds__(256) pn_l1_stats_kernel(const float* __restrict__ pts, const int4* __restrict__ tiles,
                                                          const float* __restrict__ wt, const float* __restrict__ bias,
                                                          double2* __restrict__ part) {
  __shared__ float sp[256 * 3];
  __shared__ double2 red[4][64];
  const int4 tt = tiles[blockIdx.x];          // (pair, first point, length <= 256, -)
  for (int i = threadIdx.x; i < tt.z * 3; i += 256) sp[i] = pts[(long)tt.y * 3 + i];
  __syncthreads();
  const int c = threadIdx.x & 63, qd = threadIdx.x >> 6;
  const float w0 = wt[c], w1 = wt[64 + c], w2 = wt[128 + c], b = bias[c];
  double s1 = 0.0, s2 = 0.0;
  const int p1 = min(tt.z, (qd + 1) * 64);
  for (int p = qd * 64; p < p1; p++) {
    const float y = fmaf(w2, sp[3 * p + 2], fmaf(w1, sp[3 * p + 1], fmaf(w0, sp[3 * p], b)));
    s1 += (double)y;
    s2 += (double)y * (double)y;
  }
  red[qd][c] = make_double2(s1, s2);
  __syncthreads();
  if (threadIdx.x < 128) {
    const int h = threadIdx.x >> 6;
    const double2 a = red[2 * h][c], d = red[2 * h + 1][c];
    part[((long)blockIdx.x * 2 + h) * 64 + c] = make_double2(a.x + d.x, a.y + d.y);
  }
}
// x1p planes [2][P][64] = split(relu(GN(y)))  ;  thread = (point, 4 channels)
__global__ void __launch_bounds__(256) pn_l1_apply_kernel(const float* __restrict__ pts, const float* __restrict__ wt,
                                                          const float* __restrict__ bias, const float* __restrict__ sc,
                                                          const float* __restrict__ sh, const int* __restrict__ seg,
                                                          int L, long P, __half* __restrict__ out, int* status) {
  const long idx = (long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= P * 16) return;
  const long row = idx >> 4;
  const int c = (int)(idx & 15) * 4;
  const int g = seg[row] / L;
  const float x = __ldg(pts + row * 3), y = __ldg(pts + row * 3 + 1), z = __ldg(pts + row * 3 + 2);
  const float4 w0 = *reinterpret_cast<const float4*>(wt + c), w1 = *reinterpret_cast<const float4*>(wt + 64 + c),
               w2 = *reinterpret_cast<const float4*>(wt + 128 + c), b = *reinterpret_cast<const float4*>(bias + c);
  const float4 a = *reinterpret_cast<const float4*>(sc + (long)g * 64 + c);
  const float4 s = *reinterpret_cast<const float4*>(sh + (long)g * 64 + c);
  float4 r;
  r.x = fmaxf(fmaf(fmaf(w2.x, z, fmaf(w1.x, y, fmaf(w0.x, x, b.x))), a.x, s.x), 0.f);
  r.y = fmaxf(fmaf(fmaf(w2.y, z, fmaf(w1.y, y, fmaf(w0.y, x, b.y))), a.y, s.y), 0.f);
  r.z = fmaxf(fmaf(fmaf(w2.z, z, fmaf(w1.z, y, fmaf(w0.z, x, b.z))), a.z, s.z), 0.f);
  r.w = fmaxf(fmaf(fmaf(w2.w, z, fmaf(w1.w, y, fmaf(w0.w, x, b.w))), a.w, s.w), 0.f);
  split4_store(r, out + row * 64 + c, out + P * 64 + row * 64 + c, status);
}

// seg[p] = detection owning point p (binary search in the CSR offsets)
__global__ void point_segment_kernel(const int* __restrict__ split, int ndet, long P, int* __restrict__ seg) {
  long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  int lo = 0, hi = ndet;  // split[lo] <= p < split[hi]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (split[mid] <= p) lo = mid; else hi = mid;
  }
  seg[p] = lo;
}

// out[c][d] = mean over the detection's points of relu(Y[c][p]*sc[pair][c] + sh[pair][c]).
// One warp per (c, d); lanes stride the segment (coalesced).
__global__ void segment_mean_kernel(const float* __restrict__ Y, long P, const int* __restrict__ split,
                                    const float* __restrict__ sc, const float* __restrict__ sh, int C,
                                    int ndet, int L, float* __restrict__ out, const float* __restrict__ mask = nullptr) {
  long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= (long)C * ndet) return;
  int d = (int)(w % ndet), c = (int)(w / ndet);
  int pair = d / L;
  float a = sc[(long)pair * C + c], b = sh[(long)pair * C + c];
  int s = split[d], e = split[d + 1];
  const float* row = Y + (long)c * P;
  float acc = 0.f;
  if (mask) {   // training-mode Dropout of the head activation (point_net.py:29-30): mask[c][p] in {0, 1/(1-p)}
    const float* mrow = mask + (long)c * P;
    for (int p = s + lane; p < e; p += 32) acc += fmaxf(fmaf(row[p], a, b), 0.f) * mrow[p];
  } else {
    for (int p = s + lane; p < e; p += 32) acc += fmaxf(fmaf(row[p], a, b), 0.f);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[(long)c * ndet + d] = e > s ? acc / (float)(e - s) : 0.f;
}

// feats[pair][1][c][l] = relu(O[c][d]*sc[pair][c] + sh[pair][c])
__global__ void pointnet_out_kernel(const float* __restrict__ O, const float* __restrict__ sc,
                                    const float* __restrict__ sh, int ndet, int L,
                                    float* __restrict__ feats) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 512L * ndet) return;
  int d = (int)(idx % ndet), c = (int)(idx / ndet);
  int pair = d / L, l = d - pair * L;
  float v = fmaxf(fmaf(O[idx], sc[pair * 512 + c], sh[pair * 512 + c]), 0.f);
  feats[(((long)pair * 3 + 1) * 512 + c) * L + l] = v;
}

// out[d][C] = segsum[d][C] * 2^-32 / (points of detection d): the fixed-point sums of the fused segment-sum epilogue, in
// the layout the tensor-core per-detection contractions read as rows
__global__ void segsum_mean_cl_kernel(const unsigned long long* __restrict__ segsum, const int* __restrict__ split,
                                      int C, int ndet, float* __restrict__ out) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)C * ndet) return;
  const int d = (int)(idx / C);
  const int cnt = split[d + 1] - split[d];
  out[idx] = cnt > 0 ? (float)((double)segsum[idx] * (1.0 / 4294967296.0) / (double)cnt) : 0.f;
}
// feats[pair][1][c][l] = relu(O[d][c]*sc[pair][c] + sh[pair][c]) from channels-last O (32 x 32 tiles through smem)
__global__ void pointnet_out_cl_kernel(const float* __restrict__ O, const float* __restrict__ sc, const float* __restrict__ sh,
                                       int L, float* __restrict__ feats) {
  __shared__ float tile[32][33];
  const int pair = blockIdx.z, c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int l = l0 + i, c = c0 + threadIdx.x;
    if (l < L) tile[i][threadIdx.x] = fmaxf(fmaf(O[((long)pair * L + l) * 512 + c], sc[pair * 512 + c], sh[pair * 512 + c]), 0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, l = l0 + threadIdx.x;
    if (l < L) feats[(((long)pair * 3 + 1) * 512 + c) * L + l] = tile[threadIdx.x][i];
  }
}

// Column-tile table of the ragged per-pair point ranges, built ON THE DEVICE from the CSR offsets (the host only
// needs the tile count for its launch geometry): no pageable host->device copy, so the calling thread never blocks on
// the stream and can keep enqueueing.  gstart[p] = first tile of pair p (one thread: pairs is small), then one thread
// per pair fills its tiles {pair, first point, length <= tw}.
__global__ void pn_tiles_kernel(const int* __restrict__ split, int pairs, int L, int tw, int* __restrict__ cnt,
                                int* __restrict__ gstart, int4* __restrict__ tiles) {
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int p = 0; p < pairs; p++) {
      const int n = split[(p + 1) * L] - split[p * L];
      cnt[p] = n;
      gstart[p] = acc;
      acc += (n + tw - 1) / tw;
    }
    gstart[pairs] = acc;
  }
  __syncthreads();   // single CTA: the prefix is visible to all its threads
  for (int p = threadIdx.x; p < pairs; p += blockDim.x) {
    const int s0 = split[p * L], e = split[(p + 1) * L];
    int t = gstart[p];
    for (int c = s0; c < e; c += tw) tiles[t++] = make_int4(p, c, min(tw, e - c), 0);
  }
}

struct PnWs {
  float *xt, *y1, *t0, *t1, *big, *gmean, *u, *ut, *hmean, *o;
  unsigned long long* segsum;   // tensor-core path: [ndet][1024] fixed-point per-detection sums
  __half *x1p, *xp;     // tensor-core path: FP16 hi/lo planes of normalised activations [2][P][64], [2][P][128]
  float *sc1, *sh1, *sc, *sh;
  double* stats;
  double2* part;
  int *seg, *cnt, *gstart;
  int4 *tiles, *ctab;
};

// use_tc: the tensor-core path never materialises the 1024-wide activation (537 MB per frame-pair at cfg4)
PnWs carve(MmArena& a, int pairs, int L, long P, long max_tiles, bool use_tc) {
  PnWs w;
  long nd = (long)pairs * L;
  w.xt = a.take<float>(3 * P);
  w.y1 = a.take<float>(64 * P);
  w.t0 = a.take<float>(128 * P);
  w.t1 = a.take<float>(64 * P);
  w.big = a.take<float>(use_tc ? 0 : 1024 * P);
  w.segsum = a.take<unsigned long long>(1024 * nd);
  w.x1p = a.take<__half>(2 * 64 * P);
  w.xp = a.take<__half>(2 * 128 * P);
  w.gmean = a.take<float>(1024 * nd);
  w.u = a.take<float>(512 * nd);
  w.ut = a.take<float>(512 * nd);
  w.hmean = a.take<float>(512 * nd);
  w.o = a.take<float>(512 * nd);
  w.sc1 = a.take<float>((size_t)pairs * 64);
  w.sh1 = a.take<float>((size_t)pairs * 64);
  w.sc = a.take<float>((size_t)pairs * 1024);
  w.sh = a.take<float>((size_t)pairs * 1024);
  w.stats = a.take<double>((size_t)pairs * 1024 * 2);
  w.part = a.take<double2>((size_t)max_tiles * 1024);
  w.gstart = a.take<int>(pairs + 1);
  w.seg = a.take<int>(P);
  w.cnt = a.take<int>(pairs);
  w.tiles = a.take<int4>(max_tiles);
  w.ctab = a.take<int4>(2 * max_tiles);
  return w;
}

}  // namespace

// engine choice from the per-pair shape only (see appearance.cu)
static bool pointnet_use_tc(int L) { return mm_engine() == 2 || (mm_engine() == 0 && L >= 16); }

extern "C" size_t mmmot_pointnet_workspace(int pairs, int L, long p_total) {
  MmArena a(nullptr, 0);
  carve(a, pairs, L, p_total, p_total / 128 + 2 * pairs + 2, pointnet_use_tc(L));
  return a.off;
}

extern "C" size_t mmmot_pointnet_train_workspace(int pairs, int L, long p_total) {
  MmArena a(nullptr, 0);
  carve(a, pairs, L, p_total, p_total / 128 + 2 * pairs + 2, false);
  return a.off;
}

// train: FP32 engine; head_mask (optional) = the Dropout mask of the head activation, [512][P] with values {0, 1/(1-p)}
static int pointnet_impl(const mmmot_weights* wts, const float* points, const int* det_split, const int* h_det_split,
                         int pairs, int L, float* feats, void* workspace, size_t workspace_bytes, void* stream, bool train,
                         const float* head_mask);

extern "C" int mmmot_pointnet_fwd(const mmmot_weights* wts, const float* points, const int* det_split,
                                  const int* h_det_split, int pairs, int L, float* feats,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  return pointnet_impl(wts, points, det_split, h_det_split, pairs, L, feats, workspace, workspace_bytes, stream, false, nullptr);
}

extern "C" int mmmot_pointnet_train_fwd(const mmmot_weights* wts, const float* points, const int* det_split,
                                        const int* h_det_split, int pairs, int L, const float* head_drop_mask, float* feats,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  return pointnet_impl(wts, points, det_split, h_det_split, pairs, L, feats, workspace, workspace_bytes, stream, true,
                       head_drop_mask);
}

static int pointnet_impl(const mmmot_weights* wts, const float* points, const int* det_split, const int* h_det_split,
                         int pairs, int L, float* feats, void* workspace, size_t workspace_bytes, void* stream, bool train,
                         const float* head_mask) {
  if (!wts || !points || !det_split || !h_det_split || !feats || !workspace || pairs <= 0 || L <= 0)
    return MMMOT_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int ndet = pairs * L;
  const long P = h_det_split[ndet];
  if (h_det_split[0] != 0 || P <= 0) return MMMOT_E_SHAPE;
  for (int d = 0; d < ndet; d++)
    if (h_det_split[d + 1] <= h_det_split[d]) return MMMOT_E_SHAPE;  // every detection owns >= 1 point

  // column tiles never straddle two frame-pairs (one pair = one GroupNorm domain)
  const bool use_tc = !train && pointnet_use_tc(L);
  const int TNW = use_tc ? tc::BN : 128;
  long n_tiles = 0;   // the host needs only the COUNT (launch geometry); the table itself is built on the device
  for (int p = 0; p < pairs; p++) n_tiles += mm_cdiv((long)h_det_split[(p + 1) * L] - h_det_split[p * L], TNW);
  const long max_tiles = P / 128 + 2 * pairs + 2;   // also bounds 2 partials per 256-wide tile
  MmArena ar(workspace, workspace_bytes);
  PnWs w = carve(ar, pairs, L, P, max_tiles, use_tc);
  if (!ar.ok() || n_tiles > max_tiles) return MMMOT_E_WORKSPACE;
  pn_tiles_kernel<<<1, 256, 0, st>>>(det_split, pairs, L, TNW, w.cnt, w.gstart, w.tiles);
  MM_LAUNCH_CHECK();

  transpose_points_kernel<<<mm_cdiv(P, 256), 256, 0, st>>>(points, w.xt, P);
  MM_LAUNCH_CHECK();
  point_segment_kernel<<<mm_cdiv(P, 256), 256, 0, st>>>(det_split, ndet, P, w.seg);
  MM_LAUNCH_CHECK();
  if (use_tc) {
    MM_TRY(seg_chunk_tab(w.tiles, (int)n_tiles, w.seg, w.ctab, st));
  }

  const int cin[5] = {3, 64, 64, 64, 128}, cout[5] = {64, 64, 64, 128, 1024};
  const bool timed = mm_timing_on();
  if (use_tc) {
    // ---------------- tensor-core path: channels-last activations ----------------
    // layer i writes fp32 Y[p][cout] + GroupNorm partials.  Layers 3 and 4 read the previous layer's Y directly;
    // layer 1's and layer 4's outputs become FP16 hi/lo planes (x1p, kept for the head; xp) for the TMA-fed kernel.
    float* ybuf[5] = {w.y1, w.t0, w.t1, w.t0, nullptr};
    for (int i = 0; i < 5; i++) {
      const float* const* q = &wts->w[MMMOT_W_PN_L1 + 4 * i];
      GemmP p = gemm_defaults();
      p.bias = q[1]; p.M = cout[i]; p.K = cin[i];
      p.tile_tab = w.tiles; p.num_tiles = (int)n_tiles;
      p.Y = ybuf[i]; p.y_ms = cout[i];       // layer 5 (1024 wide): statistics only, nothing stored
      p.part = w.part;
      const uint4* wp = (const uint4*)wts->w[MMMOT_W_PN_WP1 + i];
      const float wps = wts->tc_scale[MMMOT_W_PN_WP1 + i];
      const double cols = (double)P;
      if (i == 0) {
        if (timed) mm_timing_begin(st, MM_T_PN_L1, 2.0 * 64 * 3 * cols, 12.0 * cols);
        pn_l1_stats_kernel<<<(int)n_tiles, 256, 0, st>>>(points, w.tiles, q[0], q[1], w.part);
        MM_LAUNCH_CHECK();
        if (timed) mm_timing_end(st);
      } else {
        // compulsory traffic: activation in (4 B per element) + fp32 activation out (none for the statistics pass)
        if (timed) mm_timing_begin(st, i == 4 ? MM_T_PN_L5A : MM_T_PN_L2 + (i - 1), 2.0 * cout[i] * cin[i] * cols,
                                   4.0 * (cin[i] + (i == 4 ? 0 : cout[i])) * cols);
        if (i == 2 || i == 3) {
          // layers 3, 4: GroupNorm + ReLU of the previous layer applied by this contraction's operand producers
          // (gemm_gen.cuh) straight from its fp32 output: no normalised copy is written
          MM_TRY((gemm_gen_launch<gen::GEN_NORM>(p, wp, wps, ybuf[i - 1], cin[i], w.sc, w.sh, 0, 0, 0, st)));
        } else {                                                // FP16 hi/lo planes [2][P][cin] via TMA
          MM_TRY(gemm_tma_launch_mat(p, wp, wps, i == 1 ? w.x1p : w.xp, P * cin[i], P, cin[i], st));
        }
        if (timed) mm_timing_end(st);
      }
      MM_TRY(stats_reduce(w.part, cout[i], pairs, 0, w.gstart, w.stats, st, 2));
      MM_TRY(gn_finalize(w.stats, q[2], q[3], w.cnt, 0, pairs, cout[i], 1, w.sc, w.sh, st, 0, 0, ar.status()));
      if (i == 0) {
        if (timed) mm_timing_begin(st, MM_T_PN_L1, 0.0, (12.0 + 4.0 * 64) * cols);
        pn_l1_apply_kernel<<<mm_cdiv(P * 16, 256), 256, 0, st>>>(points, q[0], q[1], w.sc, w.sh, w.seg, L, P, w.x1p, ar.status());
        MM_LAUNCH_CHECK();
        if (timed) mm_timing_end(st);
      } else if (i == 1 || i == 2) {
        // consumed in place by the next layer's producers
      } else if (i == 3) {
        if (timed) mm_timing_begin(st, MM_T_PN_NORM, 0.0, 8.0 * cout[i] * cols);
        MM_TRY(norm_split(ybuf[i], cout[i], w.sc, w.sh, cout[i], P, 0, w.seg, L, w.xp, st, ar.status()));
        if (timed) mm_timing_end(st);
      } else {
        // second pass of the 1024-wide layer: recompute, GroupNorm + ReLU + per-detection mean in the epilogue
        // (its 1024 x P activation, 537 MB per frame-pair at cfg4, is never written)
        MM_CUDA(cudaMemsetAsync(w.segsum, 0, (size_t)ndet * 1024 * sizeof(unsigned long long), st));
        p.Y = nullptr; p.part = nullptr;
        p.sc = w.sc; p.sh = w.sh; p.seg = w.seg;
        if (timed) mm_timing_begin(st, MM_T_PN_L5B, 2.0 * cout[i] * cin[i] * cols, 4.0 * cin[i] * cols);
        MM_TRY(gemm_tma_launch_mat(p, wp, wps, w.xp, P * cin[i], P, cin[i], st, w.segsum, w.ctab));
        if (timed) mm_timing_end(st);
        segsum_mean_cl_kernel<<<mm_cdiv(1024L * ndet, 256), 256, 0, st>>>(w.segsum, det_split, 1024, ndet, w.gmean);
        MM_LAUNCH_CHECK();
      }
    }
    {
      // U[det][512] = gmean[det][1024] Wh[:, 64:]^T  (the per-detection part of point_net.py:27-28's conv1), on the
      // tensor cores over channels-last rows; its output is directly the [det][512] addend table of the head
      GemmP p = gemm_defaults();
      p.M = 512; p.K = 1024;
      p.S = ndet; p.tiles_per_group = mm_cdiv(ndet, tc::BN); p.num_tiles = p.tiles_per_group;
      p.x_gs = ndet;
      p.Y = w.ut; p.y_gs = ndet; p.y_ms = 512;
      MM_TRY((gemm_gen_launch<gen::GEN_COPY>(p, (const uint4*)wts->w[MMMOT_W_PN_WHGP], wts->tc_scale[MMMOT_W_PN_WHGP], w.gmean, 1024,
                                             nullptr, nullptr, 0, 0, 0, st)));
    }
    {
      GemmP p = gemm_defaults();
      p.bias = wts->w[MMMOT_W_PN_BH]; p.M = 512; p.K = 64;
      p.tile_tab = w.tiles; p.num_tiles = (int)n_tiles;
      p.Y = nullptr; p.y_ms = 512;           // pass 1: statistics only
      p.part = w.part;
      p.addend = w.ut; p.seg = w.seg; p.ld_add = 512;
      const uint4* whp = (const uint4*)wts->w[MMMOT_W_PN_WHAP];
      const float whs = wts->tc_scale[MMMOT_W_PN_WHAP];
      if (timed) mm_timing_begin(st, MM_T_PN_HEADA, 2.0 * 512 * 64 * (double)P, 4.0 * 64 * (double)P);
      MM_TRY(gemm_tma_launch_mat(p, whp, whs, w.x1p, P * 64, P, 64, st, nullptr, w.ctab));
      if (timed) mm_timing_end(st);
      MM_TRY(stats_reduce(w.part, 512, pairs, 0, w.gstart, w.stats, st, 2));
      MM_TRY(gn_finalize(w.stats, wts->w[MMMOT_W_PN_GHW], wts->w[MMMOT_W_PN_GHB], w.cnt, 0, pairs, 512, 1, w.sc, w.sh, st));
      // pass 2: recompute + GroupNorm + ReLU + per-detection mean
      MM_CUDA(cudaMemsetAsync(w.segsum, 0, (size_t)ndet * 512 * sizeof(unsigned long long), st));
      p.part = nullptr; p.sc = w.sc; p.sh = w.sh;
      if (timed) mm_timing_begin(st, MM_T_PN_HEADB, 2.0 * 512 * 64 * (double)P, 4.0 * 64 * (double)P);
      MM_TRY(gemm_tma_launch_mat(p, whp, whs, w.x1p, P * 64, P, 64, st, w.segsum, w.ctab));
      if (timed) mm_timing_end(st);
      segsum_mean_cl_kernel<<<mm_cdiv(512L * ndet, 256), 256, 0, st>>>(w.segsum, det_split, 512, ndet, w.hmean);
      MM_LAUNCH_CHECK();
    }
    {
      // conv2 512 -> 512 over the pair's L detections, GroupNorm(16,512), ReLU (point_net.py:40-41), on the tensor cores
      const int tpg2 = mm_cdiv(L, tc::BN);
      GemmP p = gemm_defaults();
      p.bias = wts->w[MMMOT_W_PN_BO]; p.M = 512; p.K = 512;
      p.S = L; p.tiles_per_group = tpg2; p.num_tiles = tpg2 * pairs;
      p.x_gs = L;
      p.Y = w.o; p.y_gs = L; p.y_ms = 512;
      p.part = w.part;
      MM_TRY((gemm_gen_launch<gen::GEN_COPY>(p, (const uint4*)wts->w[MMMOT_W_PN_WOP], wts->tc_scale[MMMOT_W_PN_WOP], w.hmean, 512,
                                             nullptr, nullptr, 0, 0, 0, st)));
      MM_TRY(stats_reduce(w.part, 512, pairs, tpg2, nullptr, w.stats, st, 2));
      MM_TRY(gn_finalize(w.stats, wts->w[MMMOT_W_PN_GOW], wts->w[MMMOT_W_PN_GOB], nullptr, L, pairs, 512, 32, w.sc, w.sh, st));
      pointnet_out_cl_kernel<<<dim3(mm_cdiv(L, 32), 16, pairs), dim3(32, 8), 0, st>>>(w.o, w.sc, w.sh, L, feats);
      MM_LAUNCH_CHECK();
      return 0;
    }
  } else {
  // trunk: 3 -> 64 -> 64 -> 64 -> 128 -> 1024, each conv + GroupNorm(C,C) over the pair's points + ReLU
  const float* src[5] = {w.xt, w.y1, w.t0, w.t1, w.t0};
  float* dst[5] = {w.y1, w.t0, w.t1, w.t0, w.big};
  for (int i = 0; i < 5; i++) {
    const float* const* q = &wts->w[MMMOT_W_PN_L1 + 4 * i];
    GemmP p = gemm_defaults();
    p.Wt = q[0]; p.bias = q[1]; p.ldw = cout[i]; p.M = cout[i]; p.K = cin[i];
    p.tile_tab = w.tiles; p.num_tiles = (int)n_tiles;
    p.X = src[i]; p.x_ks = P;
    p.Y = dst[i]; p.y_ms = P;
    p.part = w.part;
    if (i == 0) {
      MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
    } else {
      p.sc = (i == 1) ? w.sc1 : w.sc;
      p.sh = (i == 1) ? w.sh1 : w.sh;
      MM_TRY(gemm_simt_launch<XM_NORM_RELU>(p, st));
    }
    MM_TRY(stats_reduce(w.part, cout[i], pairs, 0, w.gstart, w.stats, st));
    MM_TRY(gn_finalize(w.stats, q[2], q[3], w.cnt, 0, pairs, cout[i], 1, i == 0 ? w.sc1 : w.sc,
                       i == 0 ? w.sh1 : w.sh, st));
  }
  // per-detection mean of the 1024-d feature (reference point_net.py:140-146)
  segment_mean_kernel<<<mm_cdiv(1024L * ndet * 32, 256), 256, 0, st>>>(w.big, P, det_split, w.sc, w.sh,
                                                                       1024, ndet, L, w.gmean);
  MM_LAUNCH_CHECK();
  // U = Wh[:,64:] * gmean  (the per-detection part of point_net.py:27-28's conv1)
  {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[MMMOT_W_PN_WHGT]; p.ldw = 512; p.M = 512; p.K = 1024;
    p.S = ndet; p.tiles_per_group = mm_cdiv(ndet, 128); p.num_tiles = p.tiles_per_group;
    p.X = w.gmean; p.x_ks = ndet;
    p.Y = w.u; p.y_ms = ndet;
    MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
  }
  // head: Wh[:, :64] * x_local + U[:, det(p)] + b -> GroupNorm(512,512) -> ReLU -> per-detection mean
  {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[MMMOT_W_PN_WHAT]; p.bias = wts->w[MMMOT_W_PN_BH]; p.ldw = 512; p.M = 512; p.K = 64;
    p.tile_tab = w.tiles; p.num_tiles = (int)n_tiles;
    p.X = w.y1; p.x_ks = P; p.sc = w.sc1; p.sh = w.sh1;
    p.Y = w.big; p.y_ms = P;
    p.part = w.part;
    p.addend = w.u; p.seg = w.seg; p.ld_add = ndet;
    MM_TRY(gemm_simt_launch<XM_NORM_RELU>(p, st));
    MM_TRY(stats_reduce(w.part, 512, pairs, 0, w.gstart, w.stats, st));
    MM_TRY(gn_finalize(w.stats, wts->w[MMMOT_W_PN_GHW], wts->w[MMMOT_W_PN_GHB], w.cnt, 0, pairs, 512, 1,
                       w.sc, w.sh, st));
    segment_mean_kernel<<<mm_cdiv(512L * ndet * 32, 256), 256, 0, st>>>(w.big, P, det_split, w.sc, w.sh,
                                                                        512, ndet, L, w.hmean, head_mask);
    MM_LAUNCH_CHECK();
  }
  }
  // conv2 512 -> 512 over the pair's L detections, GroupNorm(16,512), ReLU (point_net.py:40-41)
  {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[MMMOT_W_PN_WOT]; p.bias = wts->w[MMMOT_W_PN_BO]; p.ldw = 512; p.M = 512; p.K = 512;
    p.S = L; p.tiles_per_group = mm_cdiv(L, 128); p.num_tiles = p.tiles_per_group * pairs;
    p.X = w.hmean; p.x_gs = L; p.x_ks = ndet;
    p.Y = w.o; p.y_gs = L; p.y_ms = ndet;
    p.part = w.part;
    MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
    MM_TRY(stats_reduce(w.part, 512, pairs, p.tiles_per_group, nullptr, w.stats, st));
    MM_TRY(gn_finalize(w.stats, wts->w[MMMOT_W_PN_GOW], wts->w[MMMOT_W_PN_GOB], nullptr, L, pairs, 512, 32,
                       w.sc, w.sh, st));
    pointnet_out_kernel<<<mm_cdiv(512L * ndet, 256), 256, 0, st>>>(w.o, w.sc, w.sh, ndet, L, feats);
    MM_LAUNCH_CHECK();
  }
  return 0;
}
