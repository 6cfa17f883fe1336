// Appearance branch: VGG16-BN trunk (BN folded) + 4 SkipPool heads.
// Replaces reference modules/appear_net.py:166-190 (vgg_forward + SkipPool.forward :27-32).
#include <cuda_fp16.h>

#include "engines.cuh"

namespace {

// VGG16 "D" (reference modules/vgg.py:87-90): cout per conv, and whether a 2x2 max-pool follows.
const int kVggCout[13] = {64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512};
const int kVggCin[13] = {3, 64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512};
const bool kPoolAfter[13] = {false, true, false, true, false, false, true, false, false, true, false, false, true};
// skip map s is the output of the pool after conv 3, 6, 9, 12 (reference appear_net.py:139-152:
// the first pool does not close a stage)
const int kSkipAfter[13] = {-1, -1, -1, 0, -1, -1, 1, -1, -1, 2, -1, -1, 3};
const int kSkipC[4] = {128, 256, 512, 512};

// 2x2 / stride 2 max-pool, NCHW.  One thread per output pixel pair-row; float2 loads.
__global__ void maxpool2_kernel(const float* __restrict__ in, float* __restrict__ out, long n_out,
                                int Ho, int Wo) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_out) return;
  int xo = (int)(idx % Wo);
  long t = idx / Wo;
  int yo = (int)(t % Ho);
  long plane = t / Ho;
  const float* src = in + (plane * (2 * Ho) + 2 * yo) * (long)(2 * Wo) + 2 * xo;
  float2 a = *reinterpret_cast<const float2*>(src);
  float2 b = *reinterpret_cast<const float2*>(src + 2 * Wo);
  out[idx] = fmaxf(fmaxf(a.x, a.y), fmaxf(b.x, b.y));
}

// Global average pool of every (img, channel) plane: one warp per plane.
__global__ void plane_mean_kernel(const float* __restrict__ in, float* __restrict__ out, long planes,
                                  int hw) {
  long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= planes) return;
  const float* src = in + w * hw;
  float s = 0.f;
  for (int i = lane; i < hw; i += 32) s += src[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[w] = s / (float)hw;
}

// ---- FP16 hi/lo planes, NHWC: activations of the tensor-core trunk ([2][n][H][W][C]) ----
// 2x2 / stride 2 max-pool, 8 channels per thread (128-bit loads).  The max IS one of the four inputs, so its
// (hi, lo) pair is copied, not re-split.
__global__ void maxpool2_planar_kernel(const __half* __restrict__ in, __half* __restrict__ out, long n_out8,
                                       int Ho, int Wo, int C, long plane_in, long plane_out) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_out8) return;
  const int c8n = C >> 3;
  const int c = (int)(idx % c8n) * 8;
  long t = idx / c8n;
  const int xo = (int)(t % Wo);
  t /= Wo;
  const int yo = (int)(t % Ho);
  const long img = t / Ho;
  const long rs = (long)2 * Wo * C;
  const __half* src = in + ((img * 2 * Ho + 2 * yo) * 2 * Wo + 2 * xo) * (long)C + c;
  const long offs[4] = {0, (long)C, rs, rs + C};
  uint4 bh, bl;
  float best[8];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint4 h = *reinterpret_cast<const uint4*>(src + offs[k]);
    const uint4 l = *reinterpret_cast<const uint4*>(src + offs[k] + plane_in);
    const __half* hh = reinterpret_cast<const __half*>(&h);
    const __half* ll = reinterpret_cast<const __half*>(&l);
    __half* oh = reinterpret_cast<__half*>(&bh);
    __half* ol = reinterpret_cast<__half*>(&bl);
#pragma unroll
    for (int e = 0; e < 8; e++) {
      const float f = __half2float(hh[e]) + __half2float(ll[e]);
      if (k == 0 || f > best[e]) { best[e] = f; oh[e] = hh[e]; ol[e] = ll[e]; }
    }
  }
  __half* dst = out + ((img * Ho + yo) * (long)Wo + xo) * C + c;
  *reinterpret_cast<uint4*>(dst) = bh;
  *reinterpret_cast<uint4*>(dst + plane_out) = bl;
}

// global average of every (img, channel) over the hw pixels of a planar NHWC map -> pooled[img][C] fp32
__global__ void plane_mean_planar_kernel(const __half* __restrict__ in, float* __restrict__ out, long n_img,
                                         int hw, int C, long plane) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_img * C) return;
  const int c = (int)(idx % C);
  const long img = idx / C;
  const __half* src = in + img * hw * (long)C + c;
  float s = 0.f;
  for (int i = 0; i < hw; i++) s += __half2float(src[(long)i * C]) + __half2float(src[(long)i * C + plane]);
  out[idx] = s / (float)hw;
}

// pooled[img][c] = sum[img][c] * 2^-32 / hw : the fixed-point per-image sums of the fused pool epilogue -> SkipPool's average
__global__ void pool_sum_mean_kernel(const unsigned long long* __restrict__ sum, float* __restrict__ out, long n, float inv_hw) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n) out[idx] = (float)((double)sum[idx] * (1.0 / 4294967296.0) * (double)inv_hw);
}

// First VGG layer on the tensor cores: the 3-channel fp32 NCHW crop is expanded to the 27 (+5 zero) taps of every
// pixel, k = ci*9 + ky*3 + kx, as FP16 hi/lo planes [2][pixels][32]; the layer is then a K=32 contraction on the TMA
// engine whose epilogue writes the NHWC planes conv 1 reads.  One thread per pixel, 64 B per plane.
__global__ void __launch_bounds__(256) im2col27_kernel(const float* __restrict__ in, long n_pix, int H, int W,
                                                       __half* __restrict__ out, long plane, int* status) {
  const long pix = (long)blockIdx.x * 256 + threadIdx.x;
  if (pix >= n_pix) return;
  const int hw = H * W;
  const long img = pix / hw;
  const int r = (int)(pix - img * hw);
  const int y = r / W, x = r - y * W;
  const float* src = in + img * 3 * hw;
  __align__(16) __half h[32], l[32];
  float amax = 0.f;
#pragma unroll
  for (int ci = 0; ci < 3; ci++)
#pragma unroll
    for (int ky = 0; ky < 3; ky++)
#pragma unroll
      for (int kx = 0; kx < 3; kx++) {
        const int yy = y + ky - 1, xx = x + kx - 1;
        const float v = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(src + (long)ci * hw + yy * W + xx) : 0.f;
        split_f16(v, h[ci * 9 + ky * 3 + kx], l[ci * 9 + ky * 3 + kx]);
        amax = fmaxf(amax, fabsf(v));
      }
  mm_range_flag(status, amax);
#pragma unroll
  for (int k = 27; k < 32; k++) { h[k] = __ushort_as_half(0); l[k] = __ushort_as_half(0); }
  uint4* dh = reinterpret_cast<uint4*>(out + pix * 32);
  uint4* dl = reinterpret_cast<uint4*>(out + plane + pix * 32);
#pragma unroll
  for (int q = 0; q < 4; q++) {
    dh[q] = reinterpret_cast<const uint4*>(h)[q];
    dl[q] = reinterpret_cast<const uint4*>(l)[q];
  }
}

__device__ __forceinline__ float block_sum_128(float v, float* red) {
  // 128 threads (4 warps)
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}

// One CTA (128 threads) per image per head: GN(1,C) -> 1x1 conv -> GN(1,mid) -> ReLU -> 1x1 conv
// -> GN(1,128) -> ReLU.  GN(1,C) on a C x 1 x 1 input is a per-detection layer norm over channels.
__global__ void __launch_bounds__(128) skip_head_kernel(
    const float* __restrict__ pooled,  // [n_img][C]
    const float* __restrict__ g0w, const float* __restrict__ g0b, const float* __restrict__ w1t,
    const float* __restrict__ b1, const float* __restrict__ g1w, const float* __restrict__ g1b,
    const float* __restrict__ w2t, const float* __restrict__ b2, const float* __restrict__ g2w,
    const float* __restrict__ g2b, int C, int mid, int L, int head, float* __restrict__ feats) {
  __shared__ float v[512];
  __shared__ float h[128];
  __shared__ float red[4];
  const int img = blockIdx.x, t = threadIdx.x;
  const float eps = 1e-5f;
  float s = 0.f;
  for (int c = t; c < C; c += 128) { float x = pooled[(long)img * C + c]; v[c] = x; s += x; }
  float mean = block_sum_128(s, red) / C;
  s = 0.f;
  for (int c = t; c < C; c += 128) { float d = v[c] - mean; s += d * d; }
  float rstd = rsqrtf(block_sum_128(s, red) / C + eps);
  for (int c = t; c < C; c += 128) v[c] = (v[c] - mean) * rstd * g0w[c] + g0b[c];
  __syncthreads();
  // conv C -> mid
  float a = 0.f;
  if (t < mid) {
    a = b1[t];
    for (int c = 0; c < C; c++) a = fmaf(w1t[(long)c * mid + t], v[c], a);
  }
  mean = block_sum_128(t < mid ? a : 0.f, red) / mid;
  float d = t < mid ? a - mean : 0.f;
  rstd = rsqrtf(block_sum_128(d * d, red) / mid + eps);
  if (t < mid) h[t] = fmaxf(d * rstd * g1w[t] + g1b[t], 0.f);
  __syncthreads();
  // conv mid -> 128
  a = b2[t];
  for (int c = 0; c < mid; c++) a = fmaf(w2t[c * 128 + t], h[c], a);
  mean = block_sum_128(a, red) / 128.f;
  d = a - mean;
  rstd = rsqrtf(block_sum_128(d * d, red) / 128.f + eps);
  float o = fmaxf(d * rstd * g2w[t] + g2b[t], 0.f);
  const int pair = img / L, l = img - pair * L;
  feats[(((long)pair * 3 + 0) * 512 + head * 128 + t) * L + l] = o;
}

}  // namespace

int mm_launch_skip_heads(const mmmot_weights* wts, float* const* pooled, int n_img, int L, float* feats, cudaStream_t st);

extern "C" size_t mmmot_appearance_workspace(int n_img, int H, int W) {
  MmArena a(nullptr, 0);
  size_t act = (size_t)n_img * 64 * H * W;
  a.take<float>(act);
  a.take<float>(act);
  for (int s = 0; s < 4; s++) a.take<float>((size_t)n_img * kSkipC[s]);
  a.take<float>((size_t)(n_img + 16) * H * W * 16);   // K-segment partial sums, tile order (largest: 256 ch at H/4 x W/4)
  a.take<unsigned long long>((size_t)n_img * 512);     // per-image sums of a pooled skip map (fused pool epilogue)
  return a.off;
}

extern "C" int mmmot_appearance_fwd(const mmmot_weights* wts, const float* crops, int n_img, int H,
                                    int W, int L, float* feats, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!wts || !crops || !feats || !workspace || n_img <= 0 || L <= 0) return MMMOT_E_ARG;
  if (H % 32 || W % 32 || H <= 0 || W <= 0 || n_img % L) return MMMOT_E_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  MmArena ar(workspace, workspace_bytes);
  size_t act = (size_t)n_img * 64 * H * W;
  float* buf[2] = {ar.take<float>(act), ar.take<float>(act)};
  float* pooled[4];
  for (int s = 0; s < 4; s++) pooled[s] = ar.take<float>((size_t)n_img * kSkipC[s]);
  float* kseg_scratch = ar.take<float>((size_t)(n_img + 16) * H * W * 16);
  unsigned long long* pool_sum = ar.take<unsigned long long>((size_t)n_img * 512);
  if (!ar.ok()) return MMMOT_E_WORKSPACE;

  // Tensor-core trunk: activations live as FP16 hi/lo NHWC planes between layers; the epilogue of one conv
  // writes exactly what the next conv's TMA loads read (3x3 taps = shifted boxes, padding = TMA zero fill).
  // engine choice depends on per-pair shapes only (never on the batch size), so batched, looped and sharded runs
  // take the same path and stay bit-identical
  const bool tc_trunk = mm_engine() == 2 || (mm_engine() == 0 && (long)L * H * W >= 32768);
  if (tc_trunk) {
    // the 64-channel layers 0 and 1 run on the pixel-major kernel, which reads the compact weight tiles
    if (!wts->w[MMMOT_W_VGG_WPX0] || !wts->w[MMMOT_W_VGG_WPX0 + 1]) return MMMOT_E_ARG;
    __half* hb[2] = {reinterpret_cast<__half*>(buf[0]), reinterpret_cast<__half*>(buf[1])};
    const __half* cur = nullptr;
    long cur_plane = 0;
    int which = 0, h = H, w = W;
    const bool timed = mm_timing_on();   // roofline hook: every launch tagged (stage, layer)
    int* status = ar.status();
    for (int i = 0; i < 13; i++) {
      const int cout = kVggCout[i], cin = kVggCin[i];
      const long plane_out = (long)n_img * h * w * cout;
      int pooled_in_epilogue = 0;
      // algorithmic FLOPs 2*Cout*9Cin*pixels; compulsory bytes: activation in + activation out at 4 B per element
      // (the pooled map when the 2x2 max-pool is fused into the epilogue)
      if (timed) mm_timing_begin(st, MM_T_VGG0 + i, 2.0 * cout * 9.0 * cin * (double)n_img * h * w,
                                 4.0 * (double)n_img * h * w * (cin + (i == 1 ? cout / 4.0 : cout)));
      if (i == 0) {
        const long n_pix = (long)n_img * h * w;
        if (gemm_tma_px_gen27_fits(h, w)) {
          // taps generated inside the contraction kernel (no im2col matrix in HBM)
          MM_TRY(gemm_tma_px_launch_gen27(crops, n_img, h, w, (const uint4*)wts->w[MMMOT_W_VGG_WPX0],
                                          wts->tc_scale[MMMOT_W_VGG_WP0], wts->w[MMMOT_W_VGG_B0], hb[which], plane_out,
                                          status, st));
        } else {   // crops too wide for the in-kernel staging
          if (n_pix >= (1L << 31)) return MMMOT_E_SHAPE;
          __half* cols = hb[which ^ 1];   // [2][pixels][32] taps, dead once the contraction has run
          im2col27_kernel<<<mm_cdiv(n_pix, 256), 256, 0, st>>>(crops, n_pix, h, w, cols, n_pix * 32, status);
          MM_LAUNCH_CHECK();
          GemmP p = gemm_defaults();
          p.bias = wts->w[MMMOT_W_VGG_B0]; p.M = cout; p.K = 32; p.relu = 1;
          p.S = (int)n_pix; p.tiles_per_group = mm_cdiv(n_pix, tc::BN); p.num_tiles = p.tiles_per_group;
          p.Y = reinterpret_cast<float*>(hb[which]); p.y_ms = cout;
          MM_TRY(gemm_tma_px_launch_mat(p, (const uint4*)wts->w[MMMOT_W_VGG_WPX0], wts->tc_scale[MMMOT_W_VGG_WP0], cols,
                                        n_pix * 32, n_pix, 32, plane_out, status, st));
        }
      } else {
        GemmP p = gemm_defaults();
        p.bias = wts->w[MMMOT_W_VGG_B0 + i];
        p.M = cout;
        p.relu = 1;
        // a pooled layer asks for the 2x2 max-pool to be fused into the epilogue; a skip map's global average (SkipPool)
        // rides along as per-image fixed-point sums
        const bool skip_layer = kPoolAfter[i] && kSkipAfter[i] >= 0;
        if (skip_layer) MM_CUDA(cudaMemsetAsync(pool_sum, 0, (size_t)n_img * cout * sizeof(unsigned long long), st));
        MM_TRY(gemm_tma_launch_conv(p, (const uint4*)wts->w[MMMOT_W_VGG_WP0 + i], wts->tc_scale[MMMOT_W_VGG_WP0 + i], cur,
                                    cur_plane, n_img, h, w, cin, hb[which], plane_out, st, kseg_scratch,
                                    kPoolAfter[i] ? plane_out / 4 : 0, &pooled_in_epilogue, status,
                                    skip_layer ? pool_sum : nullptr, i == 1 ? (const uint4*)wts->w[MMMOT_W_VGG_WPX0 + 1] : nullptr));
      }
      if (timed) mm_timing_end(st);
      cur = hb[which]; cur_plane = plane_out; which ^= 1;
      if (kPoolAfter[i]) {
        h /= 2; w /= 2;
        const long plane_p = (long)n_img * h * w * cout;
        // compulsory bytes: separate pool = read the map + write the pooled one (+ read it again for the mean); fused =
        // the per-image sums only
        if (timed) mm_timing_begin(st, MM_T_VGG_POOL, 0.0, pooled_in_epilogue ? 12.0 * n_img * cout : 4.0 * 6.0 * plane_p);
        if (pooled_in_epilogue) {
          cur_plane = plane_p;
        } else {
          const long n8 = plane_p / 8;
          maxpool2_planar_kernel<<<mm_cdiv(n8, 256), 256, 0, st>>>(cur, hb[which], n8, h, w, cout, cur_plane, plane_p);
          MM_LAUNCH_CHECK();
          cur = hb[which]; cur_plane = plane_p; which ^= 1;
        }
        int s = kSkipAfter[i];
        if (s >= 0 && pooled_in_epilogue && i > 1) {
          const long nn = (long)n_img * kSkipC[s];
          pool_sum_mean_kernel<<<mm_cdiv(nn, 256), 256, 0, st>>>(pool_sum, pooled[s], nn, 1.0f / (float)(h * w));
          MM_LAUNCH_CHECK();
        } else if (s >= 0) {
          plane_mean_planar_kernel<<<mm_cdiv((long)n_img * kSkipC[s], 128), 128, 0, st>>>(cur, pooled[s], n_img, h * w,
                                                                                         kSkipC[s], cur_plane);
          MM_LAUNCH_CHECK();
        }
        if (timed) mm_timing_end(st);
      }
    }
  } else {
  const float* cur = crops;
  int which = 0, h = H, w = W;
  for (int i = 0; i < 13; i++) {
    GemmP p = gemm_defaults();
    p.Wt = wts->w[MMMOT_W_VGG_WT0 + i];
    p.bias = wts->w[MMMOT_W_VGG_B0 + i];
    p.ldw = kVggCout[i];
    p.M = kVggCout[i];
    p.K = 9 * kVggCin[i];
    p.Cin = kVggCin[i];
    p.H = h; p.W = w;
    p.S = n_img * h * w;
    p.X = cur;
    p.Y = buf[which];
    p.relu = 1;
    p.tiles_per_group = mm_cdiv(p.S, 128);
    p.num_tiles = p.tiles_per_group;
    const bool timed = mm_timing_on();
    if (timed) mm_timing_begin(st, MM_T_VGG0 + i, 2.0 * p.M * (double)p.K * (double)p.S, 4.0 * (double)p.S * (p.Cin + p.M));
    MM_TRY(gemm_simt_launch<XM_CONV3>(p, st));
    if (timed) mm_timing_end(st);
    cur = buf[which]; which ^= 1;
    if (kPoolAfter[i]) {
      h /= 2; w /= 2;
      long n_out = (long)n_img * kVggCout[i] * h * w;
      maxpool2_kernel<<<mm_cdiv(n_out, 256), 256, 0, st>>>(cur, buf[which], n_out, h, w);
      MM_LAUNCH_CHECK();
      cur = buf[which]; which ^= 1;
      int s = kSkipAfter[i];
      if (s >= 0) {
        long planes = (long)n_img * kSkipC[s];
        plane_mean_kernel<<<mm_cdiv(planes * 32, 256), 256, 0, st>>>(cur, pooled[s], planes, h * w);
        MM_LAUNCH_CHECK();
      }
    }
  }
  }
  return mm_launch_skip_heads(wts, pooled, n_img, L, feats, st);
}

// the four SkipPool heads on the pooled maps -> stack 0 of feats (shared with the training-mode variant, train.cu)
int mm_launch_skip_heads(const mmmot_weights* wts, float* const* pooled, int n_img, int L, float* feats, cudaStream_t st) {
  for (int s = 0; s < 4; s++) {
    const float* const* q = &wts->w[MMMOT_W_SKIP0 + 10 * s];
    int C = kSkipC[s], mid = C / 4 > 64 ? C / 4 : 64;
    skip_head_kernel<<<n_img, 128, 0, st>>>(pooled[s], q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7],
                                            q[8], q[9], C, mid, L, s, feats);
    MM_LAUNCH_CHECK();
  }
  return 0;
}
