// FP32 tiled contraction engine  Y[g][co][s] = sum_k Wt[k][co] * Xin(g,k,s) + bias[co]
//
// One mainloop, several operand generators (the "B" operand is never required to exist in HBM):
//   XM_DIRECT     Xin = X[g][k][s]
//   XM_NORM_RELU  Xin = relu(X[g][k][s]*sc[g][k] + sh[g][k])     (GroupNorm+ReLU of the producer layer,
//                                                                folded into the consumer's load)
//   XM_PAIR_*     Xin = f[g][k][i] (*|-) f[g][k][n+j], s = i*m + j  (reference modules/gcn.py:6-41;
//                                                                the 3xDxNxM tensor is never stored)
//   XM_CONV3      Xin = im2col of a 3x3 / pad 1 convolution, k = (ky*3+kx)*Cin + ci, s = (img,y,x)
// and a fused epilogue: bias, optional per-(detection) addend, optional ReLU, optional
// per-(tile, channel) sum / sum-of-squares partials for the following GroupNorm (fp64, reduced in a
// fixed order afterwards, so results are bit-reproducible).
//
// This is the accuracy-first engine (plain FP32 FFMA, 128x128x16 tiles, 8x8 register blocking).
// fp32-exact operand arithmetic is what the 1e-4 parity bound needs (SURVEY F8).
#pragma once
#include "engines.cuh"

template <int MODE, int TM>
__global__ void __launch_bounds__(256, 2) gemm_simt_kernel(const GemmP p) {
  constexpr int TN = 128, TK = 16;
  constexpr int RM = TM / 16;  // rows per thread: 8 (TM=128) or 4 (TM=64)
  __shared__ __align__(16) float As[2][TK][TM];
  __shared__ __align__(16) float Bs[2][TK][TN];

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int tx = tid & 15, ty = tid >> 4;
  const int m_tiles = p.M / TM;
  const int mt = blockIdx.x % m_tiles;
  const int nt = blockIdx.x / m_tiles;
  const int m0 = mt * TM;

  int g, c0, len;
  if (p.tile_tab) {
    int4 t = p.tile_tab[nt];
    g = t.x; c0 = t.y; len = t.z;
  } else {
    g = nt / p.tiles_per_group;
    c0 = (nt - g * p.tiles_per_group) * TN;
    len = min(TN, p.S - c0);
  }

  // ---- per-thread column state for the B loader: columns lane + 32 r, r = 0..3 ----
  const float* xb = p.X;
  int colok[4];
  long coff[4];   // DIRECT/NORM: column offset; PAIR: i | j packed; CONV3: pixel base offset
  int aux[4];     // PAIR: j ; CONV3: tap validity mask
#pragma unroll
  for (int r = 0; r < 4; r++) {
    int col = lane + 32 * r;
    colok[r] = col < len;
    coff[r] = 0; aux[r] = 0;
    if (MODE == XM_DIRECT || MODE == XM_NORM_RELU) {
      coff[r] = (long)g * p.x_gs + c0 + col;
    } else if (MODE == XM_CONV3) {
      int s = c0 + col;
      int hw = p.H * p.W;
      int img = s / hw, pix = s - img * hw;
      int y = pix / p.W, x = pix - y * p.W;
      coff[r] = (long)img * p.Cin * hw + pix;
      int mk = 0;
#pragma unroll
      for (int t = 0; t < 9; t++) {
        int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
        if (yy >= 0 && yy < p.H && xx >= 0 && xx < p.W) mk |= 1 << t;
      }
      aux[r] = colok[r] ? mk : 0;
    } else {
      int s = c0 + col;
      int i = s / p.m, j = s - i * p.m;
      coff[r] = i;
      aux[r] = p.n + j;
    }
  }

  float acc[RM][8];
#pragma unroll
  for (int i = 0; i < RM; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;

  const int ktiles = (p.K + TK - 1) / TK;
  // A loader: TK x TM floats = TK*TM/4 float4, 256 threads
  constexpr int A_F4 = TK * TM / 4 / 256;  // 2 (TM=128) or 1 (TM=64)
  float4 ra[A_F4];
  float rb[8];

  auto load_tile = [&](int kt) {
    const int k0 = kt * TK;
#pragma unroll
    for (int q = 0; q < A_F4; q++) {
      int f = tid + q * 256;
      int kr = f / (TM / 4), c4 = f % (TM / 4);
      int k = k0 + kr;
      ra[q] = (k < p.K) ? *reinterpret_cast<const float4*>(p.Wt + (long)k * p.ldw + m0 + c4 * 4)
                        : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int k = k0 + warp * 2 + h;
      const bool kok = k < p.K;
      if (MODE == XM_DIRECT || MODE == XM_NORM_RELU) {
        float s_c = 1.f, s_h = 0.f;
        if (MODE == XM_NORM_RELU && kok) {
          s_c = __ldg(p.sc + (long)g * p.K + k);
          s_h = __ldg(p.sh + (long)g * p.K + k);
        }
#pragma unroll
        for (int r = 0; r < 4; r++) {
          float v = 0.f;
          if (kok && colok[r]) {
            v = __ldg(xb + coff[r] + (long)k * p.x_ks);
            if (MODE == XM_NORM_RELU) v = fmaxf(fmaf(v, s_c, s_h), 0.f);
          }
          rb[h * 4 + r] = v;
        }
      } else if (MODE == XM_CONV3) {
        int tap = 0, ci = 0;
        if (kok) { tap = k / p.Cin; ci = k - tap * p.Cin; }
        const int d = (tap / 3 - 1) * p.W + (tap % 3 - 1);
        const long koff = (long)ci * p.H * p.W + d;
#pragma unroll
        for (int r = 0; r < 4; r++) {
          float v = 0.f;
          if (kok && ((aux[r] >> tap) & 1)) v = __ldg(xb + coff[r] + koff);
          rb[h * 4 + r] = v;
        }
      } else {
        const float* fr = p.X + ((long)g * p.K + (kok ? k : 0)) * p.Lf;
#pragma unroll
        for (int r = 0; r < 4; r++) {
          float v = 0.f;
          if (kok && colok[r]) {
            float a = __ldg(fr + coff[r]), b = __ldg(fr + aux[r]);
            if (MODE == XM_PAIR_MUL) v = a * b;
            else if (MODE == XM_PAIR_ABS) v = fabsf((a - b) * 0.5f);
            else v = (a - b) * 0.5f;
          }
          rb[h * 4 + r] = v;
        }
      }
    }
  };
  auto store_tile = [&](int buf) {
#pragma unroll
    for (int q = 0; q < A_F4; q++) {
      int f = tid + q * 256;
      int kr = f / (TM / 4), c4 = f % (TM / 4);
      *reinterpret_cast<float4*>(&As[buf][kr][c4 * 4]) = ra[q];
    }
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
      for (int r = 0; r < 4; r++) Bs[buf][warp * 2 + h][lane + 32 * r] = rb[h * 4 + r];
  };

  load_tile(0);
  store_tile(0);
  __syncthreads();
  for (int kt = 0; kt < ktiles; kt++) {
    const int buf = kt & 1;
    if (kt + 1 < ktiles) load_tile(kt + 1);
#pragma unroll
    for (int k = 0; k < TK; k++) {
      float a[RM], b[8];
      float4 t = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
      if (RM == 8) {
        t = *reinterpret_cast<const float4*>(&As[buf][k][(TM / 2) + ty * 4]);
        a[RM - 4] = t.x; a[RM - 3] = t.y; a[RM - 2] = t.z; a[RM - 1] = t.w;
      }
      t = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      b[0] = t.x; b[1] = t.y; b[2] = t.z; b[3] = t.w;
      t = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
      b[4] = t.x; b[5] = t.y; b[6] = t.z; b[7] = t.w;
#pragma unroll
      for (int i = 0; i < RM; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kt + 1 < ktiles) {
      store_tile(buf ^ 1);
      __syncthreads();
    }
  }

  // ---------------------------------------------------------------- epilogue
  const int hw = (MODE == XM_CONV3) ? p.H * p.W : 1;
#pragma unroll
  for (int i = 0; i < RM; i++) {
    const int row = (i < 4) ? (ty * 4 + i) : (TM / 2 + ty * 4 + (i - 4));
    const int co = m0 + row;
    const float bv = p.bias ? __ldg(p.bias + co) : 0.f;
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int hhalf = 0; hhalf < 2; hhalf++) {
      const int cb = hhalf * 64 + tx * 4;
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        float x = acc[i][hhalf * 4 + j] + bv;
        const int col = cb + j;
        if (p.addend && col < len) x += __ldg(p.addend + (long)co * p.ld_add + __ldg(p.seg + c0 + col));
        if (p.relu) x = fmaxf(x, 0.f);
        v[j] = x;
        if (col < len) { s1 += x; s2 += x * x; }
      }
      if (p.Y) {
        float* yp;
        bool vec;
        if (MODE == XM_CONV3) {
          const int s = c0 + cb;
          const int img = s / hw, pix = s - img * hw;
          yp = p.Y + ((long)img * p.M + co) * hw + pix;
          vec = ((hw & 3) == 0) && (cb + 3 < len);
          if (!vec) {
            for (int j = 0; j < 4; j++)
              if (cb + j < len) {
                const int s2i = c0 + cb + j;
                const int im2 = s2i / hw, px2 = s2i - im2 * hw;
                p.Y[((long)im2 * p.M + co) * hw + px2] = v[j];
              }
            continue;
          }
        } else {
          yp = p.Y + (long)g * p.y_gs + (long)co * p.y_ms + c0 + cb;
          vec = (cb + 3 < len) && ((reinterpret_cast<uintptr_t>(yp) & 15) == 0);
        }
        if (vec) {
          *reinterpret_cast<float4*>(yp) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; j++)
            if (cb + j < len) yp[j] = v[j];
        }
      }
    }
    if (p.part) {
      double d1 = s1, d2 = s2;
#pragma unroll
      for (int o = 8; o >= 1; o >>= 1) {
        d1 += __shfl_xor_sync(0xffffffffu, d1, o);
        d2 += __shfl_xor_sync(0xffffffffu, d2, o);
      }
      if (tx == 0) p.part[(long)nt * p.M + co] = make_double2(d1, d2);
    }
  }
}

template <int MODE>
int gemm_simt_launch(const GemmP& p, cudaStream_t st) {
  if (p.M % 64 != 0 || p.num_tiles <= 0) return MMMOT_E_SHAPE;
  if (p.M % 128 == 0) {
    gemm_simt_kernel<MODE, 128><<<(unsigned)((long)p.num_tiles * (p.M / 128)), 256, 0, st>>>(p);
  } else {
    gemm_simt_kernel<MODE, 64><<<(unsigned)((long)p.num_tiles * (p.M / 64)), 256, 0, st>>>(p);
  }
  MM_LAUNCH_CHECK();
  return 0;
}
