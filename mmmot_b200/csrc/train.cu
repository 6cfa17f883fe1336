// Training-mode variants of the two stages that contain BatchNorm (SURVEY.md 8f row N4).
// In .train() the reference's BatchNorm2d layers of the VGG trunk (modules/vgg.py:67-80) and the BatchNorm1d layers of
// w_det (modules/tracking_net.py:92-100) normalise with the statistics of the CURRENT batch (biased variance) and the
// detection scores stay raw logits (tracking_net.py:152-162).  Everything else of the forward (GroupNorm layers,
// PointNet, fusion, affinity) is identical to eval mode and runs through the same entry points.
// These variants run on the FP32 FFMA engine (gemm_simt.cuh): convolution with the UNFOLDED weights + per-tile
// (sum, sumsq) partials -> fixed-order reduction -> per-channel affine -> normalise + ReLU in place.  The batch
// statistics are returned so that the host can update the module's running averages like torch does.
#include "engines.cuh"

namespace {

const int kCout[13] = {64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512};
const int kCin[13] = {3, 64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512};
const bool kPool[13] = {false, true, false, true, false, false, true, false, false, true, false, false, true};
const int kSkip[13] = {-1, -1, -1, 0, -1, -1, 1, -1, -1, 2, -1, -1, 3};
const int kSkipCh[4] = {128, 256, 512, 512};

// y[img][c][hw] = relu(y*sc[c] + sh[c]) in place
__global__ void bn_relu_kernel(float* __restrict__ y, const float* __restrict__ sc, const float* __restrict__ sh, int C,
                               int hw, long n) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const int c = (int)((idx / hw) % C);
  y[idx] = fmaxf(fmaf(y[idx], sc[c], sh[c]), 0.f);
}
// stats[c] = (sum, sumsq) over `count` values -> out[c] = batch mean, out[512 + c] = biased batch variance
__global__ void bn_export_kernel(const double* __restrict__ stats, int C, double count, float* __restrict__ out) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = stats[2 * c] / count;
  double var = stats[2 * c + 1] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  out[c] = (float)mean;
  out[512 + c] = (float)var;
}
__global__ void maxpool2_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, long n_out, int Ho, int Wo) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_out) return;
  int xo = (int)(idx % Wo);
  long t = idx / Wo;
  int yo = (int)(t % Ho);
  long plane = t / Ho;
  const float* src = in + (plane * (2 * Ho) + 2 * yo) * (long)(2 * Wo) + 2 * xo;
  out[idx] = fmaxf(fmaxf(src[0], src[1]), fmaxf(src[2 * Wo], src[2 * Wo + 1]));
}
// mask (optional): DropBlock weights [img][hw] = block_mask * numel / sum (modules/dropblock.py:49-53), applied before
// the SkipPool head's average pool (modules/appear_net.py:27-30)
__global__ void plane_mean_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, long planes, int hw,
                                       const float* __restrict__ mask, int C) {
  long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= planes) return;
  const float* src = in + w * hw;
  const float* mk = mask ? mask + (w / C) * hw : nullptr;
  float s = 0.f;
  for (int i = lane; i < hw; i += 32) s += mk ? src[i] * mk[i] : src[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[w] = s / (float)hw;
}
// det_scores[g][l] = w3 . relu(h2[g][:, l]*sc + sh) + b3   (raw logits: tracking_net.py:152, training branch)
__global__ void det_logit_kernel(const float* __restrict__ h2, const float* __restrict__ sc, const float* __restrict__ sh,
                                 const float* __restrict__ w3, const float* __restrict__ b3, int G, int L,
                                 float* __restrict__ out) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= G * L) return;
  int g = idx / L, l = idx - g * L;
  const float* col = h2 + (long)g * 256 * L + l;
  float a = b3[0];
  for (int c = 0; c < 256; c++) a = fmaf(w3[c], fmaxf(fmaf(col[(long)c * L], sc[c], sh[c]), 0.f), a);
  out[idx] = a;
}

struct TrWs {
  float *buf0, *buf1, *pooled[4], *sc, *sh;
  double* stats;
  double2* part;
};
TrWs carve_tr(MmArena& a, int n_img, int H, int W) {
  TrWs w;
  size_t act = (size_t)n_img * 64 * H * W;
  w.buf0 = a.take<float>(act);
  w.buf1 = a.take<float>(act);
  for (int s = 0; s < 4; s++) w.pooled[s] = a.take<float>((size_t)n_img * kSkipCh[s]);
  w.sc = a.take<float>(512);
  w.sh = a.take<float>(512);
  w.stats = a.take<double>(512 * 2);
  w.part = a.take<double2>((size_t)mm_cdiv((long)n_img * H * W, 128) * 64);   // tiles x channels is largest at layer 0/1
  return w;
}

}  // namespace

// skip-head kernel of the eval path (appearance.cu)
int mm_launch_skip_heads(const mmmot_weights* wts, float* const* pooled, int n_img, int L, float* feats, cudaStream_t st);

extern "C" size_t mmmot_appearance_train_workspace(int n_img, int H, int W) {
  MmArena a(nullptr, 0);
  carve_tr(a, n_img, H, W);
  return a.off;
}

extern "C" int mmmot_appearance_train_fwd(const mmmot_weights* wts, const float* crops, int n_img, int H, int W, int L,
                                          float* feats, float* bn_stats, const float* drop_mask2,
                                          const float* drop_mask3, void* workspace, size_t workspace_bytes,
                                          void* stream) {
  if (!wts || !crops || !feats || !bn_stats || !workspace || n_img <= 0 || L <= 0) return MMMOT_E_ARG;
  if (H % 32 || W % 32 || H <= 0 || W <= 0 || n_img % L) return MMMOT_E_SHAPE;
  if (!wts->w[MMMOT_W_VGG_RAWW0]) return MMMOT_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  MmArena ar(workspace, workspace_bytes);
  TrWs w = carve_tr(ar, n_img, H, W);
  if (!ar.ok()) return MMMOT_E_WORKSPACE;
  const float* cur = crops;
  float* buf[2] = {w.buf0, w.buf1};
  int which = 0, h = H, wd = W;
  for (int i = 0; i < 13; i++) {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[MMMOT_W_VGG_RAWW0 + i];
    p.bias = wts->w[MMMOT_W_VGG_RAWB0 + i];
    p.ldw = kCout[i]; p.M = kCout[i]; p.K = 9 * kCin[i]; p.Cin = kCin[i];
    p.H = h; p.W = wd;
    p.S = n_img * h * wd;
    p.X = cur;
    p.Y = buf[which];
    p.tiles_per_group = mm_cdiv(p.S, 128);
    p.num_tiles = p.tiles_per_group;
    p.part = w.part;
    MM_TRY(gemm_simt_launch<XM_CONV3>(p, st));
    // BatchNorm2d, training: per-channel statistics over (batch, H, W), biased variance, eps 1e-5
    MM_TRY(stats_reduce(w.part, p.M, 1, p.num_tiles, nullptr, w.stats, st));
    MM_TRY(gn_finalize(w.stats, wts->w[MMMOT_W_VGG_BNW0 + i], wts->w[MMMOT_W_VGG_BNB0 + i], nullptr, p.S, 1, p.M, 1, w.sc, w.sh, st));
    bn_export_kernel<<<mm_cdiv(p.M, 128), 128, 0, st>>>(w.stats, p.M, (double)p.S, bn_stats + (long)i * 1024);
    MM_LAUNCH_CHECK();
    const long n = (long)p.S * p.M;
    bn_relu_kernel<<<mm_cdiv(n, 256), 256, 0, st>>>(buf[which], w.sc, w.sh, p.M, h * wd, n);
    MM_LAUNCH_CHECK();
    cur = buf[which]; which ^= 1;
    if (kPool[i]) {
      h /= 2; wd /= 2;
      const long n_out = (long)n_img * kCout[i] * h * wd;
      maxpool2_nchw_kernel<<<mm_cdiv(n_out, 256), 256, 0, st>>>(cur, buf[which], n_out, h, wd);
      MM_LAUNCH_CHECK();
      cur = buf[which]; which ^= 1;
      const int s = kSkip[i];
      if (s >= 0) {
        const long planes = (long)n_img * kSkipCh[s];
        const float* mask = s == 2 ? drop_mask2 : s == 3 ? drop_mask3 : nullptr;
        plane_mean_nchw_kernel<<<mm_cdiv(planes * 32, 256), 256, 0, st>>>(cur, w.pooled[s], planes, h * wd, mask, kSkipCh[s]);
        MM_LAUNCH_CHECK();
      }
    }
  }
  return mm_launch_skip_heads(wts, w.pooled, n_img, L, feats, st);
}

// w_det in training mode on the three stacks of ONE frame-pair: conv -> BatchNorm1d(batch statistics over the 3 x L
// values of a channel) -> ReLU, twice, then the last conv; raw logits out (no sigmoid, no threshold).
// bn_stats: [2][2][512] = (layer, mean | biased var, channel)
extern "C" size_t mmmot_w_det_train_workspace(int L) {
  MmArena a(nullptr, 0);
  a.take<float>(3 * 512 * (size_t)L); a.take<float>(3 * 256 * (size_t)L);
  a.take<float>(3 * 512); a.take<float>(3 * 512);
  a.take<double>(512 * 2); a.take<double2>((size_t)3 * mm_cdiv(L, 128) * 512);
  return a.off;
}

extern "C" int mmmot_w_det_train_fwd(const mmmot_weights* wts, int L, const float* feats, float* det_scores, float* bn_stats,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  if (!wts || !feats || !det_scores || !bn_stats || !workspace || L <= 0) return MMMOT_E_ARG;
  if (!wts->w[MMMOT_W_WD_RAW0]) return MMMOT_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  MmArena ar(workspace, workspace_bytes);
  float* h1 = ar.take<float>(3 * 512 * (size_t)L);
  float* h2 = ar.take<float>(3 * 256 * (size_t)L);
  float* sc = ar.take<float>(3 * 512);
  float* sh = ar.take<float>(3 * 512);
  double* stats = ar.take<double>(512 * 2);
  double2* part = ar.take<double2>((size_t)3 * mm_cdiv(L, 128) * 512);
  if (!ar.ok()) return MMMOT_E_WORKSPACE;
  const float* const* R = &wts->w[MMMOT_W_WD_RAW0];   // w1t b1 bn1w bn1b w2t b2 bn2w bn2b
  const int tpg = mm_cdiv(L, 128), G = 3;
  GemmP p = gemm_defaults();
  p.Wt = R[0]; p.bias = R[1]; p.ldw = 512; p.M = 512; p.K = 512;
  p.S = L; p.tiles_per_group = tpg; p.num_tiles = tpg * G;
  p.X = feats; p.x_gs = 512L * L; p.x_ks = L;
  p.Y = h1; p.y_gs = 512L * L; p.y_ms = L;
  p.part = part;
  MM_TRY(gemm_simt_launch<XM_DIRECT>(p, st));
  MM_TRY(stats_reduce(part, 512, 1, tpg * G, nullptr, stats, st));            // one BatchNorm domain: all 3 stacks
  MM_TRY(gn_finalize(stats, R[2], R[3], nullptr, 3 * L, 1, 512, 1, sc, sh, st));
  bn_export_kernel<<<4, 128, 0, st>>>(stats, 512, 3.0 * L, bn_stats);
  MM_LAUNCH_CHECK();
  for (int g = 1; g < G; g++) {   // the operand generator indexes the affine per group
    MM_CUDA(cudaMemcpyAsync(sc + g * 512, sc, 512 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    MM_CUDA(cudaMemcpyAsync(sh + g * 512, sh, 512 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  p.Wt = R[4]; p.bias = R[5]; p.ldw = 256; p.M = 256;
  p.X = h1; p.sc = sc; p.sh = sh;
  p.Y = h2; p.y_gs = 256L * L;
  MM_TRY(gemm_simt_launch<XM_NORM_RELU>(p, st));
  MM_TRY(stats_reduce(part, 256, 1, tpg * G, nullptr, stats, st));
  MM_TRY(gn_finalize(stats, R[6], R[7], nullptr, 3 * L, 1, 256, 1, sc, sh, st));
  bn_export_kernel<<<2, 128, 0, st>>>(stats, 256, 3.0 * L, bn_stats + 1024);
  MM_LAUNCH_CHECK();
  det_logit_kernel<<<mm_cdiv(G * L, 128), 128, 0, st>>>(h2, sc, sh, wts->w[MMMOT_W_WD_W3], wts->w[MMMOT_W_WD_B3], G, L,
                                                       det_scores);
  MM_LAUNCH_CHECK();
  return 0;
}
