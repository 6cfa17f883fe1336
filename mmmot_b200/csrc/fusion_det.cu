// Fusion modules A/B/C and the detection-score branch.
// Replaces reference modules/fusion_net.py:31-42 (C), :62-70 (B), :85-92 (A) and
// modules/tracking_net.py:149-163 (determine_det, eval) with w_det from :92-100.
// GroupNorm(D,D) here normalises each channel over the L detections of one frame-pair.
#include "engines.cuh"

namespace {

// ---- tensor-core path: detection-major rows  F3[(pair*L + l)*3 + stack][512]  (channels-last) ----
// F3[pair][l][s][c] = feats[pair][s][c][l] for the stacks s < ns (32 x 32 tiles through shared memory)
__global__ void feats_to_rows_kernel(const float* __restrict__ feats, float* __restrict__ f3, int L, int ns) {
  __shared__ float tile[32][33];
  const int ps = blockIdx.z, pair = ps / ns, sidx = ps - pair * ns;
  const float* src = feats + ((long)pair * 3 + sidx) * 512 * L;
  const int c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, l = l0 + threadIdx.x;
    if (l < L) tile[i][threadIdx.x] = src[(long)c * L + l];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int l = l0 + i, c = c0 + threadIdx.x;
    if (l < L) f3[(((long)pair * L + l) * 3 + sidx) * 512 + c] = tile[threadIdx.x][i];
  }
}
// fused stack from the channels-last pre-norm linear outputs (rows = pair*L + l): writes feats[pair][2][c][l] and
// F3[row][2][c].  One CTA = 32 detections x 32 channels (transposed through shared memory for the channel-major store).
__global__ void fusion_combine_rows_kernel(int arch, const float* __restrict__ yp, const float* __restrict__ yi,
                                           const float* __restrict__ gp, const float* __restrict__ gi,
                                           const float* __restrict__ scp, const float* __restrict__ shp,
                                           const float* __restrict__ sci, const float* __restrict__ shi, int L,
                                           float* __restrict__ feats, float* __restrict__ f3) {
  __shared__ float tile[32][33];
  const int pair = blockIdx.z, c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int l = l0 + i, c = c0 + threadIdx.x;
    if (l < L) {
      const long idx = ((long)pair * L + l) * 512 + c;
      const int gc = pair * 512 + c;
      float v = fmaf(yp[idx], scp[gc], shp[gc]);
      if (arch != MMMOT_FUSION_A) {
        const float u = fmaf(yi[idx], sci[gc], shi[gc]);
        if (arch == MMMOT_FUSION_B) v = v + u;
        else {
          const float a = mm_sigmoid(gp[idx]), b = mm_sigmoid(gi[idx]);
          v = (a * v + b * u) / (a + b);
        }
      }
      f3[(((long)pair * L + l) * 3 + 2) * 512 + c] = v;
      tile[i][threadIdx.x] = v;
    }
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, l = l0 + threadIdx.x;
    if (l < L) feats[(((long)pair * 3 + 2) * 512 + c) * L + l] = tile[threadIdx.x][i];
  }
}
// det_scores[pair][s][l] from h2[(pair*L + l)*3 + s][256] (post-ReLU): one warp per row, 8 channels per lane
__global__ void det_score_rows_kernel(const float* __restrict__ h2, const float* __restrict__ w3,
                                      const float* __restrict__ b3, int flags, float thr, long rows, int L,
                                      float* __restrict__ out) {
  const long row = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4 x0 = *reinterpret_cast<const float4*>(h2 + row * 256 + lane * 8), x1 = *reinterpret_cast<const float4*>(h2 + row * 256 + lane * 8 + 4);
  const float4 w0 = *reinterpret_cast<const float4*>(w3 + lane * 8), w1 = *reinterpret_cast<const float4*>(w3 + lane * 8 + 4);
  float a = x0.x * w0.x;
  a = fmaf(x0.y, w0.y, a); a = fmaf(x0.z, w0.z, a); a = fmaf(x0.w, w0.w, a);
  a = fmaf(x1.x, w1.x, a); a = fmaf(x1.y, w1.y, a); a = fmaf(x1.z, w1.z, a); a = fmaf(x1.w, w1.w, a);
#pragma unroll
  for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (lane == 0) {
    a += b3[0];
    const float sv = (flags & MMMOT_SCORE_SIGMOID) ? mm_sigmoid(a) : a;
    const long dl = row / 3;
    const int st = (int)(row - dl * 3), pair = (int)(dl / L), l = (int)(dl - (long)pair * L);
    out[((long)pair * 3 + st) * L + l] = ((flags & MMMOT_SCORE_THRESHOLD) && sv < thr) ? sv - 1.0f : sv;
  }
}

// stack2[pair][c][l] from the pre-norm linear outputs.
//   A: GN(Yp)                      B: GN(Yp) + GN(Yi)
//   C: (s(Gp)*GN(Yp) + s(Gi)*GN(Yi)) / (s(Gp) + s(Gi))
__global__ void fusion_combine_kernel(int arch, const float* __restrict__ yp, const float* __restrict__ yi,
                                      const float* __restrict__ gp, const float* __restrict__ gi,
                                      const float* __restrict__ scp, const float* __restrict__ shp,
                                      const float* __restrict__ sci, const float* __restrict__ shi, int pairs,
                                      int L, float* __restrict__ feats) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)pairs * 512 * L) return;
  int l = (int)(idx % L);
  long t = idx / L;
  int c = (int)(t % 512), pair = (int)(t / 512);
  int gc = pair * 512 + c;
  float v = fmaf(yp[idx], scp[gc], shp[gc]);
  if (arch != MMMOT_FUSION_A) {
    float u = fmaf(yi[idx], sci[gc], shi[gc]);
    if (arch == MMMOT_FUSION_B) {
      v = v + u;
    } else {
      float a = mm_sigmoid(gp[idx]), b = mm_sigmoid(gi[idx]);
      v = (a * v + b * u) / (a + b);
    }
  }
  feats[(((long)pair * 3 + 2) * 512 + c) * L + l] = v;
}

// det_scores[g][l] = s - [s < thr],  s = sigmoid(a) if 'cls' in score_arch else a,  a = w3 . h2[g][:, l] + b3
// (tracking_net.py:153-162; the threshold step is the eval branch only)
__global__ void det_score_kernel(const float* __restrict__ h2, const float* __restrict__ w3,
                                 const float* __restrict__ b3, int flags, float thr, int G, int L,
                                 float* __restrict__ out) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= G * L) return;
  int g = idx / L, l = idx - g * L;
  const float* col = h2 + (long)g * 256 * L + l;
  float a = b3[0];
  for (int c = 0; c < 256; c++) a = fmaf(w3[c], col[(long)c * L], a);
  float s = (flags & MMMOT_SCORE_SIGMOID) ? mm_sigmoid(a) : a;
  out[idx] = ((flags & MMMOT_SCORE_THRESHOLD) && s < thr) ? s - 1.0f : s;
}

struct FdWs {
  float *yp, *yi, *gp, *gi, *scp, *shp, *sci, *shi, *h1, *h2, *f3;
  double* stats;
  double2* part;
};
FdWs carve(MmArena& a, int pairs, int L) {
  FdWs w;
  size_t n = (size_t)pairs * 512 * L;
  w.f3 = a.take<float>(3 * n);
  w.yp = a.take<float>(n); w.yi = a.take<float>(n); w.gp = a.take<float>(n); w.gi = a.take<float>(n);
  w.scp = a.take<float>((size_t)pairs * 512); w.shp = a.take<float>((size_t)pairs * 512);
  w.sci = a.take<float>((size_t)pairs * 512); w.shi = a.take<float>((size_t)pairs * 512);
  w.h1 = a.take<float>(3 * n);
  w.h2 = a.take<float>(3 * n / 2);
  w.stats = a.take<double>((size_t)pairs * 512 * 2);
  w.part = a.take<double2>((size_t)pairs * 2 * mm_cdiv(L, 128) * 512);   // 1 partial per 128-tile, 2 per 256-tile
  return w;
}

}  // namespace

extern "C" size_t mmmot_fusion_det_workspace(int pairs, int L) {
  MmArena a(nullptr, 0);
  carve(a, pairs, L);
  return a.off;
}

extern "C" int mmmot_fusion_det_fwd(const mmmot_weights* wts, int fusion_arch, int score_flags, float neg_threshold,
                                    int pairs, int L, float* feats, float* det_scores, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!wts || !feats || !det_scores || !workspace || pairs <= 0 || L <= 0) return MMMOT_E_ARG;
  if (fusion_arch < MMMOT_FUSION_A || fusion_arch > MMMOT_FUSION_C) return MMMOT_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  MmArena ar(workspace, workspace_bytes);
  FdWs w = carve(ar, pairs, L);
  if (!ar.ok()) return MMMOT_E_WORKSPACE;
  const long fs = 3L * 512 * L;  // floats per pair in feats

  // engine choice from the per-pair shape only (see appearance.cu)
  if (mm_engine() == 2 || (mm_engine() == 0 && L >= 64)) {
    // ---------------- tensor-core path: every contraction on the generated-operand engine (GEN_COPY) over
    // detection-major channels-last rows F3[(pair*L + l)*3 + stack][512]
    const int tpg2 = mm_cdiv(L, tc::BN);
    const dim3 tb(32, 8), tg(mm_cdiv(L, 32), 16, pairs * 2);
    feats_to_rows_kernel<<<tg, tb, 0, st>>>(feats, w.f3, L, 2);
    MM_LAUNCH_CHECK();
    auto lin_tc = [&](int wp_id, int wb, int K, int stack, float* Y, bool stats, int gw, int gb, float* sc, float* sh) -> int {
      GemmP p = gemm_defaults();
      p.bias = wts->w[wb]; p.M = 512; p.K = K;
      p.S = L; p.tiles_per_group = tpg2; p.num_tiles = tpg2 * pairs;
      p.x_gs = L;                                            // rows per group (= per pair) of the source view below
      p.Y = Y; p.y_gs = L; p.y_ms = 512;
      p.part = stats ? w.part : nullptr;
      MM_TRY((gemm_gen_launch<gen::GEN_COPY>(p, (const uint4*)wts->w[wp_id], wts->tc_scale[wp_id], w.f3 + (long)stack * 512, 1536,
                                             nullptr, nullptr, 0, 0, 0, st)));
      if (stats) MM_TRY(stats_reduce(w.part, 512, pairs, tpg2, nullptr, w.stats, st, 2));
      if (stats) MM_TRY(gn_finalize(w.stats, wts->w[gw], wts->w[gb], nullptr, L, pairs, 512, 1, sc, sh, st));
      return 0;
    };
    if (fusion_arch == MMMOT_FUSION_A) {
      MM_TRY(lin_tc(MMMOT_W_FU_WPP, MMMOT_W_FU_BP, 1024, 0, w.yp, true, MMMOT_W_FU_GPW, MMMOT_W_FU_GPB, w.scp, w.shp));
    } else {
      MM_TRY(lin_tc(MMMOT_W_FU_WPP, MMMOT_W_FU_BP, 512, 0, w.yp, true, MMMOT_W_FU_GPW, MMMOT_W_FU_GPB, w.scp, w.shp));
      MM_TRY(lin_tc(MMMOT_W_FU_WIP, MMMOT_W_FU_BI, 512, 1, w.yi, true, MMMOT_W_FU_GIW, MMMOT_W_FU_GIB, w.sci, w.shi));
      if (fusion_arch == MMMOT_FUSION_C) {
        MM_TRY(lin_tc(MMMOT_W_FU_GATE_PP, MMMOT_W_FU_GATE_PB, 512, 0, w.gp, false, 0, 0, nullptr, nullptr));
        MM_TRY(lin_tc(MMMOT_W_FU_GATE_IP, MMMOT_W_FU_GATE_IB, 512, 1, w.gi, false, 0, 0, nullptr, nullptr));
      }
    }
    fusion_combine_rows_kernel<<<dim3(mm_cdiv(L, 32), 16, pairs), tb, 0, st>>>(fusion_arch, w.yp, w.yi, w.gp, w.gi, w.scp, w.shp,
                                                                              w.sci, w.shi, L, feats, w.f3);
    MM_LAUNCH_CHECK();
    // w_det on all three stacks = one matrix of pairs*L*3 rows x 512 channels; BN(eval) folded, ReLU in the epilogue
    const long rows = (long)pairs * L * 3;
    GemmP p = gemm_defaults();
    p.bias = wts->w[MMMOT_W_WD_B1]; p.M = 512; p.K = 512; p.relu = 1;
    p.S = (int)rows; p.tiles_per_group = mm_cdiv(rows, tc::BN); p.num_tiles = p.tiles_per_group;
    p.x_gs = rows;
    p.Y = w.h1; p.y_gs = rows; p.y_ms = 512;
    MM_TRY((gemm_gen_launch<gen::GEN_COPY>(p, (const uint4*)wts->w[MMMOT_W_WD_W1P], wts->tc_scale[MMMOT_W_WD_W1P], w.f3, 512, nullptr,
                                           nullptr, 0, 0, 0, st)));
    p.bias = wts->w[MMMOT_W_WD_B2]; p.M = 256;
    p.Y = w.h2; p.y_ms = 256;
    MM_TRY((gemm_gen_launch<gen::GEN_COPY>(p, (const uint4*)wts->w[MMMOT_W_WD_W2P], wts->tc_scale[MMMOT_W_WD_W2P], w.h1, 512, nullptr,
                                           nullptr, 0, 0, 0, st)));
    det_score_rows_kernel<<<mm_cdiv(rows * 32, 256), 256, 0, st>>>(w.h2, wts->w[MMMOT_W_WD_W3], wts->w[MMMOT_W_WD_B3], score_flags,
                                                                  neg_threshold, rows, L, det_scores);
    MM_LAUNCH_CHECK();
    return 0;
  }
  const int tpg = mm_cdiv(L, 128);

  // linear (+ optional GroupNorm statistics) on one modality: X = feats[pair][stack]
  auto linear = [&](int wt, int wb, int K, int stack, float* Y, bool stats, int gw, int gb, float* sc,
                    float* sh) -> int {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[wt]; p.bias = wts->w[wb]; p.ldw = 512; p.M = 512; p.K = K;
    p.S = L; p.tiles_per_group = tpg; p.num_tiles = tpg * pairs;
    p.X = feats + (long)stack * 512 * L; p.x_gs = fs; p.x_ks = L;
    p.Y = Y; p.y_gs = 512L * L; p.y_ms = L;
    p.part = stats ? w.part : nullptr;
    MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
    if (stats) MM_TRY(stats_reduce(w.part, 512, pairs, tpg, nullptr, w.stats, st));
    if (stats) MM_TRY(gn_finalize(w.stats, wts->w[gw], wts->w[gb], nullptr, L, pairs, 512, 1, sc, sh, st));
    return 0;
  };

  if (fusion_arch == MMMOT_FUSION_A) {
    // input_w: D x 2D on the concatenation [image; points] = stacks 0 and 1, contiguous in feats
    MM_TRY(linear(MMMOT_W_FU_WPT, MMMOT_W_FU_BP, 1024, 0, w.yp, true, MMMOT_W_FU_GPW, MMMOT_W_FU_GPB, w.scp, w.shp));
  } else {
    // NB the reference applies input_p / gate_p to stack 0 (image): names are swapped there.
    MM_TRY(linear(MMMOT_W_FU_WPT, MMMOT_W_FU_BP, 512, 0, w.yp, true, MMMOT_W_FU_GPW, MMMOT_W_FU_GPB, w.scp, w.shp));
    MM_TRY(linear(MMMOT_W_FU_WIT, MMMOT_W_FU_BI, 512, 1, w.yi, true, MMMOT_W_FU_GIW, MMMOT_W_FU_GIB, w.sci, w.shi));
    if (fusion_arch == MMMOT_FUSION_C) {
      MM_TRY(linear(MMMOT_W_FU_GATE_PT, MMMOT_W_FU_GATE_PB, 512, 0, w.gp, false, 0, 0, nullptr, nullptr));
      MM_TRY(linear(MMMOT_W_FU_GATE_IT, MMMOT_W_FU_GATE_IB, 512, 1, w.gi, false, 0, 0, nullptr, nullptr));
    }
  }
  fusion_combine_kernel<<<mm_cdiv((long)pairs * 512 * L, 256), 256, 0, st>>>(
      fusion_arch, w.yp, w.yi, w.gp, w.gi, w.scp, w.shp, w.sci, w.shi, pairs, L, feats);
  MM_LAUNCH_CHECK();

  // w_det on all three stacks: groups g = pair*3 + stack, BN(eval) folded, ReLU in the epilogue
  const int G = pairs * 3;
  {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[MMMOT_W_WD_W1T]; p.bias = wts->w[MMMOT_W_WD_B1]; p.ldw = 512; p.M = 512; p.K = 512;
    p.S = L; p.tiles_per_group = tpg; p.num_tiles = tpg * G;
    p.X = feats; p.x_gs = 512L * L; p.x_ks = L;
    p.Y = w.h1; p.y_gs = 512L * L; p.y_ms = L;
    p.relu = 1;
    MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
    p.Wt = wts->w[MMMOT_W_WD_W2T]; p.bias = wts->w[MMMOT_W_WD_B2]; p.ldw = 256; p.M = 256;
    p.X = w.h1;
    p.Y = w.h2; p.y_gs = 256L * L;
    MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
  }
  det_score_kernel<<<mm_cdiv((long)G * L, 128), 128, 0, st>>>(w.h2, wts->w[MMMOT_W_WD_W3],
                                                              wts->w[MMMOT_W_WD_B3], score_flags, neg_threshold, G, L,
                                                              det_scores);
  MM_LAUNCH_CHECK();
  return 0;
}
