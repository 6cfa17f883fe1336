// Pairwise affinity + start/end ("new"/"end") indicator + softmax mode.
// Replaces reference modules/gcn.py:68-82 (affinity_module.forward), modules/new_end.py:62-82
// (NewEndIndicator_v2.forward, mode 'avg') and modules/tracking_net.py:106-126 (associate).
//
// Groups g = pair*3 + stack.  The pairwise tensor x[g][c][i][j] (reference gcn.py:13,24-27;
// 100.7 MB per pair at N=M=128) is generated inside the first contraction's operand producers and
// never exists in HBM; affinity conv1.0 and new/end conv0 (both 512->512 on the same x) run as
// ONE 512->1024 contraction.  On the tensor-core path (gemm_gen.cuh) the GroupNorm + ReLU between
// the MLP layers is applied by the next contraction's producers while they build its operand, so
// each layer output crosses HBM once as channels-last fp32 (written by one epilogue, read by the
// next layer's producers).
#include <algorithm>

#include "engines.cuh"

namespace {

// Row/column means of y = relu(GN_{1,512}(conv0 x)):  new_vec = mean_i y (per j), end_vec = mean_j y
// (reference new_end.py:69-71).  One CTA per (g, c); V is channel-major over absolute columns:
// V[c][g*(M+N) + j] (new part), V[c][g*(M+N) + M + i] (end part).
// mx: reduce with max instead of the mean (NewEndIndicator_v2 mode 'max', new_end.py:73-74; values are >= 0 after the ReLU).
__global__ void __launch_bounds__(256) rowcol_mean_kernel(const float* __restrict__ y0, long y_gs,
                                                          const float* __restrict__ sc,
                                                          const float* __restrict__ sh, int N, int M,
                                                          long ldv, float* __restrict__ V, int mx) {
  extern __shared__ float colacc[];  // [warps][M]: per-warp partial column sums, combined in fixed order
  const int g = blockIdx.x / 512, c = blockIdx.x % 512;
  const float a = sc[g * 512 + c], b = sh[g * 512 + c];
  const float* src = y0 + (long)g * y_gs + (long)c * N * M;
  float* vout = V + (long)c * ldv + (long)g * (M + N);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // each warp owns rows i = warp, warp+nw, ...; lanes stride the columns
  for (int j0 = 0; j0 < M; j0 += 32) {
    const int j = j0 + lane;
    float cs = 0.f;
    for (int i = warp; i < N; i += nw) {
      if (j < M) { const float r = fmaxf(fmaf(src[(long)i * M + j], a, b), 0.f); cs = mx ? fmaxf(cs, r) : cs + r; }
    }
    if (j < M) colacc[warp * M + j] = cs;
  }
  for (int i = warp; i < N; i += nw) {
    float rs = 0.f;
    for (int j = lane; j < M; j += 32) { const float r = fmaxf(fmaf(src[(long)i * M + j], a, b), 0.f); rs = mx ? fmaxf(rs, r) : rs + r; }
#pragma unroll
    for (int o = 16; o; o >>= 1) { const float t = __shfl_xor_sync(0xffffffffu, rs, o); rs = mx ? fmaxf(rs, t) : rs + t; }
    if (lane == 0) vout[M + i] = mx ? rs : rs / (float)M;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    float t = 0.f;
    for (int w2 = 0; w2 < nw; w2++) t = mx ? fmaxf(t, colacc[w2 * M + j]) : t + colacc[w2 * M + j];
    vout[j] = mx ? t : t / (float)N;
  }
}

// ---- channels-last (tensor-core path) variants: y[(g*N + i)*M + j][ld] ----
// end_vec[c][i] = mean_j relu(GN(y0)) -> V[c][g*(M+N) + M + i]   (CTA r < N of group g: row i = r, sum over j)
// new_vec[c][j] = mean_i relu(GN(y0)) -> V[c][g*(M+N) + j]       (CTA r >= N: column j = r - N, sum over i)
// One launch, grid = G x (N + M) with a group's CTAs adjacent: the row pass and the column pass of a group run
// together, so the group's 2 KB-per-row slab is read from HBM once and the second use hits L2.  Threads over channels
// (coalesced 1 KB per row), 8 independent loads in flight per thread, fixed summation order.
__global__ void __launch_bounds__(256) newend_mean_cl_kernel(const float* __restrict__ y, long ld, int coff,
                                                             const float* __restrict__ sc, const float* __restrict__ sh,
                                                             int N, int M, long ldv, float* __restrict__ V, int mx) {
  // ldv == 0: V is channels-last [column][512] (the tensor-core new/end MLP reads it as rows); else V[c][ldv]
  const int g = blockIdx.x / (N + M), r = blockIdx.x % (N + M);
  const bool is_end = r < N;
  const int cnt = is_end ? M : N;
  const long step = is_end ? ld : (long)M * ld;
  const float* src = y + (is_end ? (long)(g * N + r) * M : (long)g * N * M + (r - N)) * ld + coff;
  for (int c = threadIdx.x; c < 512; c += blockDim.x) {
    const float a = sc[g * 512 + c], b = sh[g * 512 + c];
    const float* p = src + c;
    float acc = 0.f;
    int k = 0;
    for (; k + 8 <= cnt; k += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; u++) v[u] = __ldg(p + (long)(k + u) * step);
      if (mx) {
#pragma unroll
        for (int u = 0; u < 8; u++) acc = fmaxf(acc, fmaf(v[u], a, b));     // acc starts at 0: max(relu(.))
      } else {
#pragma unroll
        for (int u = 0; u < 8; u++) acc += fmaxf(fmaf(v[u], a, b), 0.f);
      }
    }
    for (; k < cnt; k++) {
      const float r2 = fmaxf(fmaf(__ldg(p + (long)k * step), a, b), 0.f);
      acc = mx ? fmaxf(acc, r2) : acc + r2;
    }
    const long colv = (long)g * (M + N) + (is_end ? M + r : r - N);
    V[ldv ? (long)c * ldv + colv : colv * 512 + c] = mx ? acc : acc / (float)cnt;
  }
}
// z[row] = w4 . relu(GN(y3[row][0..127])) + b4 : one warp per row (a lane owns 4 channels: one coalesced 512-byte
// load per row, its GroupNorm affine and w4 in registers while the group stays the same), fixed-order shuffle tree
__global__ void __launch_bounds__(256) link_logit_cl_kernel(const float* __restrict__ y3, const float* __restrict__ sc,
                                                            const float* __restrict__ sh, const float* __restrict__ w4,
                                                            const float* __restrict__ b4, long rows, int NM,
                                                            float* __restrict__ z) {
  const int lane = threadIdx.x & 31;
  const long warp = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * blockDim.x) >> 5;
  const float4 w = *reinterpret_cast<const float4*>(w4 + lane * 4);
  const float bias = b4[0];
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
  int gcur = -1;
  // each warp takes a contiguous block of rows (the group changes at most a few times per warp)
  const long per = (rows + nwarps - 1) / nwarps;
  const long r0 = warp * per, r1 = min(rows, r0 + per);
  for (long row = r0; row < r1; row += 4) {
    float4 x[4];
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (row + u < r1) x[u] = __ldcs(reinterpret_cast<const float4*>(y3 + (row + u) * 128 + lane * 4));
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (row + u >= r1) break;
      const int g = (int)((row + u) / NM);
      if (g != gcur) {
        gcur = g;
        a = *reinterpret_cast<const float4*>(sc + g * 128 + lane * 4);
        b = *reinterpret_cast<const float4*>(sh + g * 128 + lane * 4);
      }
      float acc = w.x * fmaxf(fmaf(x[u].x, a.x, b.x), 0.f);
      acc = fmaf(w.y, fmaxf(fmaf(x[u].y, a.y, b.y), 0.f), acc);
      acc = fmaf(w.z, fmaxf(fmaf(x[u].z, a.z, b.z), 0.f), acc);
      acc = fmaf(w.w, fmaxf(fmaf(x[u].w, a.w, b.w), 0.f), acc);
#pragma unroll
      for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) z[row + u] = acc + bias;
    }
  }
}

// Tile table for the new/end MLP: group 2g = new columns (len M), 2g+1 = end columns (len N).
__global__ void ne_tiles_kernel(int G, int N, int M, int tn, int tm_, int tw, int4* __restrict__ tiles,
                                int* __restrict__ cnt, int* __restrict__ gstart) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int per = tm_ + tn;  // tiles per g: tm_ for the M new columns, tn for the N end columns
  if (idx < G * 2) { cnt[idx] = (idx & 1) ? N : M; gstart[idx] = (idx >> 1) * per + ((idx & 1) ? tm_ : 0); }
  if (idx == G * 2) gstart[idx] = G * per;
  if (idx >= G * per) return;
  int g = idx / per, t = idx - g * per;
  if (t < tm_) tiles[idx] = make_int4(2 * g, g * (M + N) + t * tw, min(tw, M - t * tw), 0);
  else { t -= tm_; tiles[idx] = make_int4(2 * g + 1, g * (M + N) + M + t * tw, min(tw, N - t * tw), 0); }
}

// out[col] = sigmoid(w3 . relu(GN(h2))[:, col] + b3) for the new/end MLP; scatters into new_s / end_s.
__global__ void ne_final_kernel(const float* __restrict__ h2, long ldv, const float* __restrict__ sc,
                                const float* __restrict__ sh, const float* __restrict__ w3,
                                const float* __restrict__ b3, int G, int N, int M,
                                float* __restrict__ new_s, float* __restrict__ end_s) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= G * (M + N)) return;
  int g = idx / (M + N), r = idx - g * (M + N);
  int grp = 2 * g + (r >= M);
  float a = b3[0];
  for (int c = 0; c < 128; c++)
    a = fmaf(w3[c], fmaxf(fmaf(h2[(long)c * ldv + idx], sc[grp * 128 + c], sh[grp * 128 + c]), 0.f), a);
  float s = mm_sigmoid(a);
  if (r < M) new_s[(long)g * M + r] = s; else end_s[(long)g * N + (r - M)] = s;
}

// channels-last variant: h2[col][128]; one warp per column (a lane owns 4 channels)
__global__ void ne_final_cl_kernel(const float* __restrict__ h2, const float* __restrict__ sc, const float* __restrict__ sh,
                                   const float* __restrict__ w3, const float* __restrict__ b3, int G, int N, int M,
                                   float* __restrict__ new_s, float* __restrict__ end_s) {
  const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (idx >= G * (M + N)) return;
  const int g = idx / (M + N), r = idx - g * (M + N);
  const int grp = 2 * g + (r >= M);
  const float4 x = *reinterpret_cast<const float4*>(h2 + (long)idx * 128 + lane * 4);
  const float4 a = *reinterpret_cast<const float4*>(sc + grp * 128 + lane * 4), b = *reinterpret_cast<const float4*>(sh + grp * 128 + lane * 4);
  const float4 w = *reinterpret_cast<const float4*>(w3 + lane * 4);
  float acc = w.x * fmaxf(fmaf(x.x, a.x, b.x), 0.f);
  acc = fmaf(w.y, fmaxf(fmaf(x.y, a.y, b.y), 0.f), acc);
  acc = fmaf(w.z, fmaxf(fmaf(x.z, a.z, b.z), 0.f), acc);
  acc = fmaf(w.w, fmaxf(fmaf(x.w, a.w, b.w), 0.f), acc);
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    const float sv = mm_sigmoid(acc + b3[0]);
    if (r < M) new_s[(long)g * M + r] = sv; else end_s[(long)g * N + (r - M)] = sv;
  }
}

// z[g][s] = w4 . relu(GN(y3[g]))[:, s] + b4      (reference gcn.py:65-66: last 1x1 conv 128 -> 1)
__global__ void link_logit_kernel(const float* __restrict__ y3, const float* __restrict__ sc,
                                  const float* __restrict__ sh, const float* __restrict__ w4,
                                  const float* __restrict__ b4, int G, int NM, float* __restrict__ z) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)G * NM) return;
  int g = (int)(idx / NM);
  int s = (int)(idx - (long)g * NM);
  const float* col = y3 + (long)g * 128 * NM + s;
  float a = b4[0];
#pragma unroll 8
  for (int c = 0; c < 128; c++)
    a = fmaf(__ldg(w4 + c), fmaxf(fmaf(col[(long)c * NM], __ldg(sc + g * 128 + c), __ldg(sh + g * 128 + c)), 0.f), a);
  z[idx] = a;
}

// softmax statistics: rows (dim=-1, over j) and columns (dim=-2, over i); one warp per row/column.
__global__ void softmax_stats_kernel(const float* __restrict__ z, int G, int N, int M,
                                     float* __restrict__ rmax, float* __restrict__ rsum,
                                     float* __restrict__ cmax, float* __restrict__ csum) {
  long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= (long)G * (N + M)) return;
  int g = (int)(w / (N + M)), r = (int)(w - (long)g * (N + M));
  const float* base = z + (long)g * N * M;
  int cntv, stride;
  const float* p0;
  if (r < N) { p0 = base + (long)r * M; cntv = M; stride = 1; }
  else { p0 = base + (r - N); cntv = N; stride = M; }
  float mx = -INFINITY;
  for (int t = lane; t < cntv; t += 32) mx = fmaxf(mx, p0[(long)t * stride]);
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sm = 0.f;
  for (int t = lane; t < cntv; t += 32) sm += expf(p0[(long)t * stride] - mx);
#pragma unroll
  for (int o = 16; o; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
  if (lane == 0) {
    if (r < N) { rmax[g * N + r] = mx; rsum[g * N + r] = sm; }
    else { cmax[g * M + r - N] = mx; csum[g * M + r - N] = sm; }
  }
}

__global__ void softmax_apply_kernel(const float* __restrict__ z, int mode, int G, int N, int M,
                                     const float* __restrict__ rmax, const float* __restrict__ rsum,
                                     const float* __restrict__ cmax, const float* __restrict__ csum,
                                     float* __restrict__ link) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)G * N * M) return;
  int g = (int)(idx / ((long)N * M));
  int r = (int)(idx - (long)g * N * M);
  int i = r / M, j = r - i * M;
  float v = z[idx];
  float pr = expf(v - rmax[g * N + i]) / rsum[g * N + i];   // softmax over dim=-1
  float out = pr;
  if (mode != MMMOT_SM_SINGLE) {
    float pc = expf(v - cmax[g * M + j]) / csum[g * M + j]; // softmax over dim=-2
    if (mode == MMMOT_SM_DUAL) out = pr * pc;
    else if (mode == MMMOT_SM_DUAL_ADD) out = (pr + pc) / 2.f;
    else out = fmaxf(pr, pc);
  }
  link[idx] = out;
}

struct AfWs {
  float *y01, *y2, *y3, *z;
  float* fcl;     // tensor-core path: channels-last copy of the feature stacks [G][L][512]
  float *sc1, *sh1, *sc0, *sh0, *sc2, *sh2, *sc3, *sh3;
  float *v, *h1, *h2, *nsc1, *nsh1, *nsc2, *nsh2;
  float *rmax, *rsum, *cmax, *csum;
  double *stats, *nstats;
  int4* tiles;
  int *cnt, *gstart;
  double2 *part, *npart;
};
AfWs carve(MmArena& a, int pairs, int n, int m) {
  AfWs w;
  size_t G = (size_t)pairs * 3, NM = (size_t)n * m, ldv = G * (n + m);
  w.y01 = a.take<float>(G * 1024 * NM);
  w.y2 = a.take<float>(G * 512 * NM);
  w.y3 = a.take<float>(G * 128 * NM);
  w.z = a.take<float>(G * NM);
  w.fcl = a.take<float>(G * (n + m) * 512);
  w.sc1 = a.take<float>(G * 512); w.sh1 = a.take<float>(G * 512);
  w.sc0 = a.take<float>(G * 512); w.sh0 = a.take<float>(G * 512);
  w.sc2 = a.take<float>(G * 512); w.sh2 = a.take<float>(G * 512);
  w.sc3 = a.take<float>(G * 128); w.sh3 = a.take<float>(G * 128);
  w.v = a.take<float>(512 * ldv); w.h1 = a.take<float>(512 * ldv); w.h2 = a.take<float>(128 * ldv);
  w.nsc1 = a.take<float>(2 * G * 512); w.nsh1 = a.take<float>(2 * G * 512);
  w.nsc2 = a.take<float>(2 * G * 128); w.nsh2 = a.take<float>(2 * G * 128);
  w.rmax = a.take<float>(G * n); w.rsum = a.take<float>(G * n);
  w.cmax = a.take<float>(G * m); w.csum = a.take<float>(G * m);
  w.stats = a.take<double>(G * 1024 * 2);
  w.nstats = a.take<double>(2 * G * 512 * 2);
  w.tiles = a.take<int4>(G * (mm_cdiv(n, 128) + mm_cdiv(m, 128)));
  w.cnt = a.take<int>(2 * G);
  w.gstart = a.take<int>(2 * G + 1);
  w.part = a.take<double2>(G * 2 * mm_cdiv(NM, 256) * 1024);   // covers 1 partial per 128-tile and 2 per 256-tile
  w.npart = a.take<double2>(G * 2 * (mm_cdiv(n, 128) + mm_cdiv(m, 128)) * 512);   // 1 partial per 128-tile or 2 per 256-tile
  return w;
}

template <int GEN>
int launch_gen(const GemmP& p, const mmmot_weights* wts, int wid, const float* src, int src_m, const float* gsc,
               const float* gsh, int n, int m, int Lf, cudaStream_t st) {
  return gemm_gen_launch<GEN>(p, (const uint4*)wts->w[wid], wts->tc_scale[wid], src, src_m, gsc, gsh, n, m, Lf, st);
}

}  // namespace

extern "C" size_t mmmot_affinity_workspace(int pairs, int n, int m) {
  MmArena a(nullptr, 0);
  carve(a, pairs, n, m);
  return a.off;
}

extern "C" int mmmot_affinity_fwd(const mmmot_weights* wts, int affinity_op, int softmax_mode, int end_mode, int pairs,
                                  int n, int m, const float* feats, float* link, float* new_s,
                                  float* end_s, void* workspace, size_t workspace_bytes, void* stream) {
  if (!wts || !feats || !link || !new_s || !end_s || !workspace || pairs <= 0 || n <= 0 || m <= 0)
    return MMMOT_E_ARG;
  if (affinity_op < 0 || affinity_op > MMMOT_AFF_MINUS || softmax_mode < 0 || softmax_mode > MMMOT_SM_DUAL_MAX ||
      end_mode < MMMOT_END_AVG || end_mode > MMMOT_END_MAX)
    return MMMOT_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  MmArena ar(workspace, workspace_bytes);
  AfWs w = carve(ar, pairs, n, m);
  if (!ar.ok()) return MMMOT_E_WORKSPACE;
  const int G = pairs * 3, NM = n * m, L = n + m;
  const bool use_tc = mm_engine() == 2 || (mm_engine() == 0 && NM >= 64);   // per-pair shape only (see appearance.cu); a
  // quarter-filled 256-column tile on the tensor cores still beats the FP32 engine (N = 8: 31k -> see DESIGN §6)
  const int tpg = mm_cdiv(NM, use_tc ? tc::BN : 128);
  const float* const* W = wts->w;
  const bool timed = mm_timing_on();

  // layer 1: [conv1.0 ; w_new_end.conv0] 512 -> 1024 on the generated pairwise tensor.
  // FP32 engine: y01[g][1024][NM].  Tensor-core engine: channels-last y01[g*NM + s][1024].
  const int pm = use_tc ? 2 : 1;   // GroupNorm partials per column tile
  if (use_tc) {
    MM_TRY(transpose_f32(feats, w.fcl, 512, L, G, st));
    MM_TRY(feats_range_check(feats, (long)G * 512 * L, affinity_op == MMMOT_AFF_MULTIPLY ? 255.9f : 65504.f, ar.status(),
                             st));
    GemmP p = gemm_defaults();
    p.bias = W[MMMOT_W_AF_B01]; p.M = 1024; p.K = 512;
    p.S = NM; p.tiles_per_group = tpg; p.num_tiles = tpg * G;
    p.Y = w.y01; p.y_gs = NM; p.y_ms = 1024;
    p.part = w.part;
    if (timed) mm_timing_begin(st, MM_T_AFF_L1, 2.0 * 1024 * 512 * (double)G * NM, 4.0 * 1024 * (double)G * NM);
    int r = affinity_op == MMMOT_AFF_MULTIPLY
                ? launch_gen<gen::GEN_PAIR_MUL>(p, wts, MMMOT_W_AF_W01P, w.fcl, 0, nullptr, nullptr, n, m, L, st)
            : affinity_op == MMMOT_AFF_MINUS_ABS
                ? launch_gen<gen::GEN_PAIR_ABS>(p, wts, MMMOT_W_AF_W01P, w.fcl, 0, nullptr, nullptr, n, m, L, st)
                : launch_gen<gen::GEN_PAIR_SUB>(p, wts, MMMOT_W_AF_W01P, w.fcl, 0, nullptr, nullptr, n, m, L, st);
    if (r) return r;
    if (timed) mm_timing_end(st);
  } else {
    GemmP p = gemm_defaults();
    p.Wt = W[MMMOT_W_AF_W01T]; p.bias = W[MMMOT_W_AF_B01]; p.ldw = 1024; p.M = 1024; p.K = 512;
    p.S = NM; p.tiles_per_group = tpg; p.num_tiles = tpg * G;
    p.X = feats; p.n = n; p.m = m; p.Lf = L;
    p.Y = w.y01; p.y_gs = 1024L * NM; p.y_ms = NM;
    p.part = w.part;
    int r = affinity_op == MMMOT_AFF_MULTIPLY    ? gemm_simt_launch<XM_PAIR_MUL>(p, st)
            : affinity_op == MMMOT_AFF_MINUS_ABS ? gemm_simt_launch<XM_PAIR_ABS>(p, st)
                                                 : gemm_simt_launch<XM_PAIR_SUB>(p, st);
    if (r) return r;
  }
  // statistics are [G][1024]: channels 0..511 = conv1.0 -> GroupNorm(512,512) (per channel over N x M),
  // 512..1023 = conv0 -> GroupNorm(1,512) (one group over 512 x N x M; new_end.py:50)
  MM_TRY(stats_reduce(w.part, 1024, G, tpg, nullptr, w.stats, st, pm));
  MM_TRY(gn_finalize(w.stats, W[MMMOT_W_AF_G1W], W[MMMOT_W_AF_G1B], nullptr, NM, G, 512, 1, w.sc1, w.sh1, st, 1024, 0, ar.status()));
  MM_TRY(gn_finalize(w.stats, W[MMMOT_W_AF_G0W], W[MMMOT_W_AF_G0B], nullptr, NM, G, 512, 512, w.sc0, w.sh0, st, 1024, 512));

  // ---- new / end indicator on y0 = channels 512..1023 of y01 ----
  const long ldv = (long)G * (n + m);
  if (use_tc) {
    if (timed) mm_timing_begin(st, MM_T_AFF_MEAN, 0.0, 4.0 * 512 * (double)G * NM);
    newend_mean_cl_kernel<<<G * (n + m), 256, 0, st>>>(w.y01, 1024, 512, w.sc0, w.sh0, n, m, 0, w.v, end_mode);
    MM_LAUNCH_CHECK();
    if (timed) mm_timing_end(st);
  } else {
    rowcol_mean_kernel<<<G * 512, 256, 8 * m * sizeof(float), st>>>(w.y01 + 512L * NM, 1024L * NM, w.sc0, w.sh0,
                                                               n, m, ldv, w.v, end_mode);
    MM_LAUNCH_CHECK();
  }
  const int tw = use_tc ? tc::BN : 128;
  const int tn = mm_cdiv(n, tw), tm_ = mm_cdiv(m, tw), ne_tiles = G * (tn + tm_);
  ne_tiles_kernel<<<mm_cdiv(max(ne_tiles, 2 * G + 1), 128), 128, 0, st>>>(G, n, m, tn, tm_, tw, w.tiles, w.cnt, w.gstart);
  MM_LAUNCH_CHECK();
  if (use_tc) {
    // shared Conv1d MLP on the new / end vectors (new_end.py:53-60) on the tensor cores: rows = columns of V
    // (channels-last), groups = (g, new | end) through the tile table
    GemmP p = gemm_defaults();
    p.bias = W[MMMOT_W_NE_B1]; p.M = 512; p.K = 512;
    p.tile_tab = w.tiles; p.num_tiles = ne_tiles;
    p.Y = w.h1; p.y_ms = 512;
    p.part = w.npart;
    MM_TRY(launch_gen<gen::GEN_COPY>(p, wts, MMMOT_W_NE_W1P, w.v, 512, nullptr, nullptr, 0, 0, 0, st));
    MM_TRY(stats_reduce(w.npart, 512, 2 * G, 0, w.gstart, w.nstats, st, 2));
    MM_TRY(gn_finalize(w.nstats, W[MMMOT_W_NE_G1W], W[MMMOT_W_NE_G1B], w.cnt, 0, 2 * G, 512, 512, w.nsc1, w.nsh1, st, 0, 0, ar.status()));
    p.bias = W[MMMOT_W_NE_B2]; p.M = 128;
    p.Y = w.h2; p.y_ms = 128;
    MM_TRY(launch_gen<gen::GEN_NORM>(p, wts, MMMOT_W_NE_W2P, w.h1, 512, w.nsc1, w.nsh1, 0, 0, 0, st));
    MM_TRY(stats_reduce(w.npart, 128, 2 * G, 0, w.gstart, w.nstats, st, 2));
    MM_TRY(gn_finalize(w.nstats, W[MMMOT_W_NE_G2W], W[MMMOT_W_NE_G2B], w.cnt, 0, 2 * G, 128, 128, w.nsc2, w.nsh2, st));
    ne_final_cl_kernel<<<mm_cdiv((long)G * (n + m) * 32, 256), 256, 0, st>>>(w.h2, w.nsc2, w.nsh2, W[MMMOT_W_NE_W3], W[MMMOT_W_NE_B3],
                                                                            G, n, m, new_s, end_s);
    MM_LAUNCH_CHECK();
  } else {
    GemmP p = gemm_defaults();
    p.Wt = W[MMMOT_W_NE_W1T]; p.bias = W[MMMOT_W_NE_B1]; p.ldw = 512; p.M = 512; p.K = 512;
    p.tile_tab = w.tiles; p.num_tiles = ne_tiles;
    p.X = w.v; p.x_ks = ldv;
    p.Y = w.h1; p.y_ms = ldv;
    p.part = w.npart;
    MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
    MM_TRY(stats_reduce(w.npart, 512, 2 * G, 0, w.gstart, w.nstats, st));
    MM_TRY(gn_finalize(w.nstats, W[MMMOT_W_NE_G1W], W[MMMOT_W_NE_G1B], w.cnt, 0, 2 * G, 512, 512, w.nsc1, w.nsh1, st));
    p.Wt = W[MMMOT_W_NE_W2T]; p.bias = W[MMMOT_W_NE_B2]; p.ldw = 128; p.M = 128;
    p.X = w.h1; p.sc = w.nsc1; p.sh = w.nsh1;
    p.Y = w.h2;
    MM_TRY(gemm_simt_launch<XM_NORM_RELU>(p, st));
    MM_TRY(stats_reduce(w.npart, 128, 2 * G, 0, w.gstart, w.nstats, st));
    MM_TRY(gn_finalize(w.nstats, W[MMMOT_W_NE_G2W], W[MMMOT_W_NE_G2B], w.cnt, 0, 2 * G, 128, 128, w.nsc2, w.nsh2, st));
    ne_final_kernel<<<mm_cdiv((long)G * (n + m), 128), 128, 0, st>>>(w.h2, ldv, w.nsc2, w.nsh2, W[MMMOT_W_NE_W3],
                                                                   W[MMMOT_W_NE_B3], G, n, m, new_s, end_s);
    MM_LAUNCH_CHECK();
  }

  // ---- affinity MLP layers 2, 3 on y1 = channels 0..511 of y01 ----
  if (use_tc) {
    // GroupNorm + ReLU of the previous layer is applied by this layer's operand producers (gemm_gen.cuh, GEN_NORM)
    GemmP p = gemm_defaults();
    p.bias = W[MMMOT_W_AF_B2]; p.M = 512; p.K = 512;
    p.S = NM; p.tiles_per_group = tpg; p.num_tiles = tpg * G;
    p.x_gs = NM;
    p.Y = w.y2; p.y_gs = NM; p.y_ms = 512;
    p.part = w.part;
    if (timed) mm_timing_begin(st, MM_T_AFF_L2, 2.0 * 512 * 512 * (double)G * NM, 4.0 * (512 + 512) * (double)G * NM);
    MM_TRY(launch_gen<gen::GEN_NORM>(p, wts, MMMOT_W_AF_W2P, w.y01, 1024, w.sc1, w.sh1, 0, 0, 0, st));
    if (timed) mm_timing_end(st);
    MM_TRY(stats_reduce(w.part, 512, G, tpg, nullptr, w.stats, st, 2));
    MM_TRY(gn_finalize(w.stats, W[MMMOT_W_AF_G2W], W[MMMOT_W_AF_G2B], nullptr, NM, G, 512, 1, w.sc2, w.sh2, st, 0, 0, ar.status()));
    p.bias = W[MMMOT_W_AF_B3]; p.M = 128;
    p.Y = w.y3; p.y_ms = 128;
    if (timed) mm_timing_begin(st, MM_T_AFF_L3, 2.0 * 128 * 512 * (double)G * NM, 4.0 * (512 + 128) * (double)G * NM);
    MM_TRY(launch_gen<gen::GEN_NORM>(p, wts, MMMOT_W_AF_W3P, w.y2, 512, w.sc2, w.sh2, 0, 0, 0, st));
    if (timed) mm_timing_end(st);
    MM_TRY(stats_reduce(w.part, 128, G, tpg, nullptr, w.stats, st, 2));
    MM_TRY(gn_finalize(w.stats, W[MMMOT_W_AF_G3W], W[MMMOT_W_AF_G3B], nullptr, NM, G, 128, 1, w.sc3, w.sh3, st));
  } else {
    GemmP p = gemm_defaults();
    p.Wt = W[MMMOT_W_AF_W2T]; p.bias = W[MMMOT_W_AF_B2]; p.ldw = 512; p.M = 512; p.K = 512;
    p.S = NM; p.tiles_per_group = tpg; p.num_tiles = tpg * G;
    p.X = w.y01; p.x_gs = 1024L * NM; p.x_ks = NM; p.sc = w.sc1; p.sh = w.sh1;
    p.Y = w.y2; p.y_gs = 512L * NM; p.y_ms = NM;
    p.part = w.part;
    MM_TRY(gemm_simt_launch<XM_NORM_RELU>(p, st));
    MM_TRY(stats_reduce(w.part, 512, G, tpg, nullptr, w.stats, st));
    MM_TRY(gn_finalize(w.stats, W[MMMOT_W_AF_G2W], W[MMMOT_W_AF_G2B], nullptr, NM, G, 512, 1, w.sc2, w.sh2, st));
    p.Wt = W[MMMOT_W_AF_W3T]; p.bias = W[MMMOT_W_AF_B3]; p.ldw = 128; p.M = 128;
    p.X = w.y2; p.x_gs = 512L * NM; p.sc = w.sc2; p.sh = w.sh2;
    p.Y = w.y3; p.y_gs = 128L * NM;
    MM_TRY(gemm_simt_launch<XM_NORM_RELU>(p, st));
    MM_TRY(stats_reduce(w.part, 128, G, tpg, nullptr, w.stats, st));
    MM_TRY(gn_finalize(w.stats, W[MMMOT_W_AF_G3W], W[MMMOT_W_AF_G3B], nullptr, NM, G, 128, 1, w.sc3, w.sh3, st));
  }
  float* zdst = softmax_mode == MMMOT_SM_NONE ? link : w.z;
  if (use_tc) {
    if (timed) mm_timing_begin(st, MM_T_AFF_LOGIT, 2.0 * 128 * (double)G * NM, 4.0 * 129 * (double)G * NM);
    const long lrows = (long)G * NM;
    link_logit_cl_kernel<<<(int)std::min<long>(148L * 8, (lrows + 31) / 32), 256, 0, st>>>(w.y3, w.sc3, w.sh3, W[MMMOT_W_AF_W4],
                                                                                      W[MMMOT_W_AF_B4], lrows, NM, zdst);
  } else {
    link_logit_kernel<<<mm_cdiv((long)G * NM, 256), 256, 0, st>>>(w.y3, w.sc3, w.sh3, W[MMMOT_W_AF_W4],
                                                                 W[MMMOT_W_AF_B4], G, NM, zdst);
  }
  MM_LAUNCH_CHECK();
  if (use_tc && timed) mm_timing_end(st);
  if (softmax_mode != MMMOT_SM_NONE) {
    softmax_stats_kernel<<<mm_cdiv((long)G * (n + m) * 32, 256), 256, 0, st>>>(w.z, G, n, m, w.rmax, w.rsum,
                                                                              w.cmax, w.csum);
    MM_LAUNCH_CHECK();
    softmax_apply_kernel<<<mm_cdiv((long)G * NM, 256), 256, 0, st>>>(w.z, softmax_mode, G, n, m, w.rmax, w.rsum,
                                                                    w.cmax, w.csum, link);
    MM_LAUNCH_CHECK();
  }
  return 0;
}
