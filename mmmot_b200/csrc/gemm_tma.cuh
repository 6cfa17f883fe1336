// tcgen05 contraction engine, TMA-fed variant (sm_100a).
//
// Same arithmetic as the generated-operand kernel (gemm_gen.cuh: FP16 hi/lo split operands, 3 MMAs per k-step, FP32
// accumulate in TMEM, fused epilogue) but the activation operand is not produced by threads: activations between
// tensor-core layers live in HBM as two FP16 planes (hi, lo), channels-last, and the TMA engine
// (cp.async.bulk.tensor, tiled mode, 64-byte swizzle) drops each [256 rows x 32 channels] box straight
// into shared memory in the UMMA K-major SWIZZLE_64B layout:
//   * 1x1 contraction: 2-D map [rows][C], box (32, 256)
//   * 3x3 convolution: 4-D map [img][H][W][C], box (32, bx, by, bi) with bx*by*bi = 256; the 9 taps are the
//     same box at shifted (x, y) coordinates and the zero padding is TMA's out-of-bounds fill — no im2col,
//     no boundary code, no index arithmetic on the SMs.
// CTA (320 threads, persistent, one per SM): warps 0-7 epilogue (two per TMEM lane quadrant, one per
// column half), warp 8 MMA issuer, warp 9 loader (weights by cp.async.bulk, operand boxes by TMA).
// When the tile has one 128-row subtile (Cout <= 128) the 512 TMEM columns hold TWO accumulator buffers, so
// the epilogue of tile i overlaps the MMAs of tile i+1.  Conv outputs are transposed through a per-warp smem
// scratch so each lane stores 64 contiguous bytes (32 channels of one pixel) per plane.
// Compiled in engines.cu only: the launchers below have external linkage (see engines.cuh).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace tma {

using namespace tc;

constexpr int T_THREADS = 320;
constexpr int T_EPI_WARPS = 8, T_MMA_WARP = 8, T_LOAD_WARP = 9;
constexpr int T_EPI_SCRATCH = 32 * 80;   // per epilogue warp: 32 pixels x (64 B of channels + 16 B pad)
constexpr size_t T_SMEM_BYTES = tc_smem_bytes(STAGE_BYTES) + T_EPI_WARPS * T_EPI_SCRATCH;

// chunk descriptors of the table-tiled contractions over ragged per-detection columns (PointNet): tab[tile*2 + half]
static __global__ void seg_chunk_tab_kernel(const int4* __restrict__ tiles, int num_tiles, const int* __restrict__ seg,
                                            int4* __restrict__ tab) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_tiles * 2) return;
  const int4 tt = tiles[idx >> 1];
  const int half = idx & 1, c0 = tt.y, len = tt.z;
  int v[4];
#pragma unroll
  for (int c = 0; c < 4; c++) {
    const int col0 = half * 128 + c * 32;
    v[c] = 0;
    if (col0 < len) {
      const int first = seg[c0 + col0], last = seg[c0 + min(col0 + 31, len - 1)];
      v[c] = (first << 1) | ((col0 + 32 <= len && first == last) ? 1 : 0);
    }
  }
  tab[idx] = make_int4(v[0], v[1], v[2], v[3]);
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t mbar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(mbar)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint32_t mbar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], "
      "[%6];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(mbar)
      : "memory");
}
// one 32-byte (whole sector) store; dst 32-byte aligned
__device__ __forceinline__ void st_global_256(void* dst, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(a.x), "r"(a.y), "r"(a.z),
               "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void st_global_256(void* dst, const uint32_t* r) {
  st_global_256(dst, make_uint4(r[0], r[1], r[2], r[3]), make_uint4(r[4], r[5], r[6], r[7]));
}
// 2x2 max-pool of one 32-column chunk held by a thread (one channel): the chunk is 32/BX box rows of BX pixels, so its
// 16/BX row pairs hold BX/2 windows each: o[a*(BX/2) + b] = window (rows 2a, 2a+1; columns 2b, 2b+1).  BX <= 16.
template <int BX>
__device__ __forceinline__ void pool_chunk(const float (&x)[32], float (&o)[8]) {
#pragma unroll
  for (int a = 0; a < 16 / BX; a++)
#pragma unroll
    for (int b = 0; b < BX / 2; b++) {
      const int i = 2 * a * BX + 2 * b;
      o[a * (BX / 2) + b] = fmaxf(fmaxf(x[i], x[i + 1]), fmaxf(x[i + BX], x[i + BX + 1]));
    }
}

static __global__ void __launch_bounds__(T_THREADS, 1)
gemm_tma_kernel(const TmaP P, const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo) {
  const GemmP& p = P.t.g;
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // full: the loader's single expect_tx arrive (weights + 2 operand boxes)
  const TcPipe C = tc_begin<STAGE_BYTES>(smem_raw, 1, T_EPI_WARPS, warp == T_MMA_WARP);
  uint8_t* epi_scratch = C.sm + STAGES * STAGE_BYTES + 256;

  const int MT = P.t.mt_per_cta;
  const int mgroups = (P.t.m_tiles + MT - 1) / MT;
  const long total_tiles = (long)p.num_tiles * mgroups;
  // K chunks: conv = 9 taps x (C / 32) channel chunks, K order k = tap*C + ci ; matrix = K / 32
  const int KC = P.t.k_chunks;
  const int cchunks = P.conv ? P.C / BK : KC;
  const int nbuf = (MT == 1) ? 2 : 1;   // accumulator buffers in TMEM (256 columns each when MT == 1)

  if (warp < T_EPI_WARPS) {
    // =============================== EPILOGUE ===============================
    const int q = warp & 3, half = warp >> 2;
    const int lbx = 31 - __clz(max(P.bx, 1)), lby = 31 - __clz(max(P.by, 1));
    uint32_t wcount = 0;   // (tile, segment) work items processed by this CTA
    float amax = 0.f;      // largest magnitude converted to FP16 by this thread (range guard)
    __half* yh = reinterpret_cast<__half*>(p.Y);
    __half* scr = reinterpret_cast<__half*>(epi_scratch + warp * T_EPI_SCRATCH);
    // final conv values x[j] (pixel column col0+j, channel cb+lane) -> FP16 hi/lo NHWC planes.  The 32x32 block is
    // transposed through smem so that lane p stores the 32 channels (64 contiguous bytes) of pixel col0+p.
    // lane p stores the 32 channels (64 contiguous bytes per plane) of "its" row: x[j] is (row col0+j, channel cb+lane),
    // the 32x32 block is transposed through the warp's smem scratch; o = element offset of this lane's row at channel cb
    auto store_rows = [&](const float (&x)[32], bool ok, long o) {
      __half h[32], l[32];
#pragma unroll
      for (int j = 0; j < 32; j++) { split_f16(x[j], h[j], l[j]); amax = fmaxf(amax, fabsf(x[j])); }
#pragma unroll
      for (int pl = 0; pl < 2; pl++) {
#pragma unroll
        for (int j = 0; j < 32; j++) scr[j * 40 + lane] = pl ? l[j] : h[j];
        __syncwarp();
        if (ok) {
          // 256-bit stores: each instruction writes whole 32-byte sectors (16-byte pieces cost a partial-sector
          // write each and ran the first layers' epilogues at ~1.8 TB/s)
          const uint4* src = reinterpret_cast<const uint4*>(scr + lane * 40);
          __half* dst = yh + o + (pl ? P.plane_elems : 0);
          const uint4 a = src[0], b = src[1], c = src[2], d = src[3];
          st_global_256(dst, a, b);
          st_global_256(dst + 16, c, d);
        }
        __syncwarp();
      }
    };
    // conv tiles: column -> (image, y, x) of the box, NHWC output
    auto store_planar_block = [&](const float (&x)[32], int col0, int cb, int i0, int y0, int x0) {
      const int col = col0 + lane;
      const int xx = col & (P.bx - 1), r = col >> lbx;
      const int yy = r & (P.by - 1), ii = r >> lby;
      const int img = i0 + ii, y = y0 + yy, xg = x0 + xx;
      store_rows(x, img < P.n_img && y < P.H && xg < P.W, (((long)img * P.H + y) * P.W + xg) * p.y_ms + cb);
    };
    // ---- fused 2x2 max-pool (P.pool): the thread owns one channel of the tile's columns, so every pooling window of
    // its chunks is in its own registers.  NP pooled pixels per emission (8 for bx <= 16; 16 for bx == 32, where a
    // chunk is one box row and the previous chunk's horizontal maxima are kept); lane q < NP stores pooled pixel q's
    // 32 channels.  The pooled values are also summed per (image, channel) for SkipPool's global average.
    const int Hp = P.H >> 1, Wp = P.W >> 1;
    float hprev[16];            // bx == 32: horizontal maxima of the even row
    float psum = 0.f;           // running sum of this thread's pooled values of image psum_img
    int psum_img = -1;
    auto pool_flush = [&](int co_) {
      if (P.pool_sum && psum_img >= 0 && psum_img < P.n_img)
        atomicAdd(P.pool_sum + (long)psum_img * p.M + co_, __float2ull_rn(psum * 4294967296.f));
      psum = 0.f; psum_img = -1;
    };
    // o[q], q < NP: pooled pixels of box rows (r0, r0 + 1), columns 2q', in box-row units r = ii*by + yy
    auto pool_emit = [&](const float (&o)[16], int np, int r0, int wq, int cb, int co_, int i0, int y0, int x0) {
      // pooled pixel q: box row r0 + 2*(q / wq), box column 2*(q % wq)      (wq = windows per row pair)
      float xs[32];
#pragma unroll
      for (int j = 0; j < 32; j++) xs[j] = j < 16 ? o[j] : 0.f;
      const int q = lane < np ? lane : 0;
      const int r = r0 + 2 * (q / wq), xx = 2 * (q - (q / wq) * wq);
      const int yy = r & (P.by - 1), ii = r >> lby;
      const int img = i0 + ii, y = y0 + yy, xg = x0 + xx;
      const bool ok = lane < np && img < P.n_img && y < P.H && xg < P.W;
      store_rows(xs, ok, (((long)img * Hp + (y >> 1)) * Wp + (xg >> 1)) * p.y_ms + cb);
      if (P.pool_sum) {
#pragma unroll
        for (int j = 0; j < 16; j++) {
          if (j < np) {
            const int rj = r0 + 2 * (j / wq), xj = 2 * (j - (j / wq) * wq);
            const int imj = i0 + (rj >> lby);
            const bool okj = imj < P.n_img && y0 + (rj & (P.by - 1)) < P.H && x0 + xj < P.W;
            if (imj != psum_img) { pool_flush(co_); psum_img = imj; }
            if (okj) psum += o[j];
          }
        }
      }
    };
    // one finished 32-column chunk (bias + ReLU applied) of channel co_: store it, or pool it and store the pooled map
    auto emit_conv = [&](const float (&x)[32], int cc, int col0, int co_, int i0, int y0, int x0) {
      if (!P.pool) { store_planar_block(x, col0, co_ - lane, i0, y0, x0); return; }
      float o[16];
      const int r0 = col0 >> lbx;
      if (P.bx == 32) {
        if (!(cc & 1)) {
#pragma unroll
          for (int b = 0; b < 16; b++) hprev[b] = fmaxf(x[2 * b], x[2 * b + 1]);
          return;
        }
#pragma unroll
        for (int b = 0; b < 16; b++) o[b] = fmaxf(hprev[b], fmaxf(x[2 * b], x[2 * b + 1]));
        pool_emit(o, 16, r0 - 1, 16, co_ - lane, co_, i0, y0, x0);
        return;
      }
      float o8[8];
      if (P.bx == 16) pool_chunk<16>(x, o8);
      else if (P.bx == 8) pool_chunk<8>(x, o8);
      else if (P.bx == 4) pool_chunk<4>(x, o8);
      else pool_chunk<2>(x, o8);
#pragma unroll
      for (int j = 0; j < 16; j++) o[j] = j < 8 ? o8[j] : 0.f;
      pool_emit(o, 8, r0, P.bx >> 1, co_ - lane, co_, i0, y0, x0);
    };

    for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const int mg = (int)(t % mgroups);
      const int nt = (int)(t / mgroups);
      int g = 0, c0 = 0, len = BN, i0 = 0, y0 = 0, x0 = 0;
      if (P.conv) conv_origin(P, nt, i0, y0, x0); else tile_cols(p, nt, g, c0, len);
      for (int seg = 0; seg < P.ksegs; seg++, wcount++) {
      const int abuf = acc_buf(wcount, nbuf);
      const uint32_t acc_col = (uint32_t)(abuf * 256);
      mbar_wait(C.tfull_bar(abuf), acc_parity(wcount, nbuf));
      tc_fence_after();
      if (P.ksegs > 1) {
        // K-segmented convolution: the tensor core's fp32 accumulator rounds toward zero at every K=16 step,
        // so long K chains are cut into segments whose partial sums are combined here in fp32 round-to-nearest.
        for (int mt = 0; mt < MT; mt++) {
          const int co = (mg * MT + mt) * 128 + q * 32 + lane;
          const bool rowok = co < p.M;
          const float bv = (rowok && p.bias) ? __ldg(p.bias + co) : 0.f;
#pragma unroll 1
          for (int cc = 0; cc < 4; cc++) {
            const int col0 = half * 128 + cc * 32;
            uint32_t v[32];
            tmem_ld32(C.tmem + ((uint32_t)(q * 32) << 16) + acc_col + (uint32_t)(mt * 256 + col0), v);
            if (!rowok) continue;
            // partial sums live in TILE order, scratch[(tile*256 + column)][M]: no pixel arithmetic, and a
            // warp's 32 channels of one column are one 128-byte access
            float* sp = P.acc_scratch + ((long)nt * BN + col0) * p.M + co;
            if (seg < P.ksegs - 1) {
              if (seg == 0) {
#pragma unroll
                for (int j = 0; j < 32; j++) __stcg(sp + (long)j * p.M, __uint_as_float(v[j]) * P.t.out_scale);
              } else {
                float sv[32];
#pragma unroll
                for (int j = 0; j < 32; j++) sv[j] = __ldcg(sp + (long)j * p.M);
#pragma unroll
                for (int j = 0; j < 32; j++) __stcg(sp + (long)j * p.M, fmaf(__uint_as_float(v[j]), P.t.out_scale, sv[j]));
              }
            } else {
              float sv[32];
#pragma unroll
              for (int j = 0; j < 32; j++) sv[j] = __ldcg(sp + (long)j * p.M);
#pragma unroll
              for (int j = 0; j < 32; j++) {
                float a = fmaf(__uint_as_float(v[j]), P.t.out_scale, sv[j]) + bv;
                sv[j] = p.relu ? fmaxf(a, 0.f) : a;
              }
              emit_conv(sv, cc, col0, co, i0, y0, x0);
            }
          }
          if (P.pool && seg == P.ksegs - 1 && rowok) pool_flush(co);
        }
      } else
      for (int mt = 0; mt < MT; mt++) {
        const int co = (mg * MT + mt) * 128 + q * 32 + lane;
        const bool rowok = co < p.M;
        const float bv = (rowok && p.bias) ? __ldg(p.bias + co) : 0.f;
        float f1 = 0.f, f2 = 0.f;   // this thread's (sum, sum of squares) over its 128 columns: four fp32 chunk sums
        const bool pass2 = P.segsum && !p.part && !p.Y && !p.relu;
        // Everything the four 32-column chunks need from global memory is fetched up front, so its latency is paid once
        // per subtile instead of once (or twice, seg -> addend) per chunk: the detection index at both ends of every
        // chunk (one load: lane 2c / 2c+1 holds chunk c's first / last column), the per-detection addend row of every
        // single-detection chunk, and the GroupNorm affine of the recomputing pass.
        const bool use_seg = p.seg && (p.addend || P.segsum);
        int4 ct = make_int4(0, 0, 0, 0);
        if (use_seg) ct = __ldg(P.chunk_tab + (long)nt * 2 + half);   // same address in every lane: one transaction
        const int cdesc[4] = {ct.x, ct.y, ct.z, ct.w};
        float adv[4] = {0.f, 0.f, 0.f, 0.f};
        unsigned one_det = 0;   // bit c: chunk c is complete and lies inside one detection
#pragma unroll
        for (int c = 0; c < 4; c++) {
          if (cdesc[c] & 1) {
            one_det |= 1u << c;
            if (p.addend && rowok) adv[c] = __ldg(p.addend + (long)(cdesc[c] >> 1) * p.ld_add + co);
          }
        }
        float na = 0.f, nb = 0.f;
        if (P.segsum && rowok) { na = __ldg(p.sc + (long)g * p.M + co); nb = __ldg(p.sh + (long)g * p.M + co); }
#pragma unroll 1
        for (int cc = 0; cc < 4; cc++) {
          const int col0 = half * 128 + cc * 32;
          if (col0 >= len) break;   // warp-uniform
          const int da = (cc == 0 ? ct.x : cc == 1 ? ct.y : cc == 2 ? ct.z : ct.w) >> 1;
          const float adc = cc == 0 ? adv[0] : cc == 1 ? adv[1] : cc == 2 ? adv[2] : adv[3];
          const bool single = (one_det >> cc) & 1u;
          uint32_t v[32];
          tmem_ld32(C.tmem + ((uint32_t)(q * 32) << 16) + acc_col + (uint32_t)(mt * 256 + col0), v);
          if (P.t.dbg & 1) continue;
          float s1 = 0.f, s2 = 0.f;
          bool fast = col0 + 32 <= len;
          if (pass2 && fast) {
            // second (recomputing) pass, whole chunk inside one detection: bias, addend and the GroupNorm affine
            // fold into one fma per element; no statistics, nothing stored
            if (single) {
              if (rowok) {
                const float bva = bv + adc;
                const float a2 = P.t.out_scale * na, b2 = fmaf(bva, na, nb);
                float r0 = 0.f, r1 = 0.f;
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                  r0 += fmaxf(fmaf(__uint_as_float(v[j]), a2, b2), 0.f);
                  r1 += fmaxf(fmaf(__uint_as_float(v[j + 1]), a2, b2), 0.f);
                }
                atomicAdd(P.segsum + (long)da * p.M + co, __float2ull_rn((r0 + r1) * 4294967296.f));
              }
              continue;
            }
          }
          float bva = bv;
          if (fast && p.addend) {
            if (single) bva += adc;
            else fast = false;
          }
          if (fast) {
            if (p.relu) epi_fast<true>(v, P.t.out_scale, bva, s1, s2);
            else epi_fast<false>(v, P.t.out_scale, bva, s1, s2);
          } else {
#pragma unroll
            for (int j = 0; j < 32; j++) {
              float x = fmaf(__uint_as_float(v[j]), P.t.out_scale, bv);
              const int col = col0 + j;
              if (p.addend && rowok && col < len)
                x += __ldg(p.addend + (long)__ldg(p.seg + c0 + col) * p.ld_add + co);
              if (p.relu) x = fmaxf(x, 0.f);
              v[j] = __float_as_uint(x);
              if (col < len) { s1 += x; s2 = fmaf(x, x, s2); }
            }
          }
          f1 += s1; f2 += s2;
          if (P.segsum && rowok) {
            // GroupNorm + ReLU + per-detection sum fused into the (recomputing) second pass: the activation never
            // reaches HBM.  Run sums are fp32 in column order; runs are merged with integer atomics, so the result
            // does not depend on the order in which tiles finish.
            const int nvalid = min(32, len - col0);
            int dcur = da;
            float run = 0.f;
            if (single) {
              // common case: the whole 32-column chunk belongs to one detection
#pragma unroll
              for (int j = 0; j < 32; j++) run += fmaxf(fmaf(__uint_as_float(v[j]), na, nb), 0.f);
            } else {
#pragma unroll
              for (int j = 0; j < 32; j++) {
                if (j < nvalid) {
                  const int d = __ldg(p.seg + c0 + col0 + j);
                  if (d != dcur) {
                    atomicAdd(P.segsum + (long)dcur * p.M + co, __float2ull_rn(run * 4294967296.f));
                    run = 0.f; dcur = d;
                  }
                  run += fmaxf(fmaf(__uint_as_float(v[j]), na, nb), 0.f);
                }
              }
            }
            atomicAdd(P.segsum + (long)dcur * p.M + co, __float2ull_rn(run * 4294967296.f));
          }
          if (!p.Y || !rowok) continue;
          if (P.conv) {
            float xv[32];
#pragma unroll
            for (int j = 0; j < 32; j++) xv[j] = __uint_as_float(v[j]);
            emit_conv(xv, cc, col0, co, i0, y0, x0);
          } else {   // fp32 channels-last
            const int nvalid = min(32, len - col0);
            const long row0 = (long)g * p.y_gs + c0 + col0;
            float* dst = p.Y + row0 * p.y_ms + co;
            if (nvalid == 32) {
#pragma unroll
              for (int j = 0; j < 32; j++) { *dst = __uint_as_float(v[j]); dst += p.y_ms; }
            } else {
#pragma unroll
              for (int j = 0; j < 32; j++)
                if (j < nvalid) dst[(long)j * p.y_ms] = __uint_as_float(v[j]);
            }
          }
        }
        if (p.part && rowok) p.part[((long)nt * 2 + half) * p.M + co] = make_double2((double)f1, (double)f2);
        if (P.conv && P.pool && rowok) pool_flush(co);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(C.tempty_bar(abuf));
      }
    }
    mm_range_flag(P.status, amax);
  } else if (warp == T_MMA_WARP) {
    // =============================== MMA ISSUER ===============================
    if (lane == 0) {
      uint32_t it = 0, tcount = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
       for (int seg = 0; seg < P.ksegs; seg++, tcount++) {
        const int abuf = acc_buf(tcount, nbuf);
        mbar_wait(C.tempty_bar(abuf), acc_parity(tcount, nbuf) ^ 1);
        tc_fence_after();
        const int kc_lo = seg * P.kc_per_seg, kc_hi = min(KC, kc_lo + P.kc_per_seg);
        for (int kc = kc_lo; kc < kc_hi; kc++, it++) {
          const int s = ring_stage(it);
          mbar_wait(C.full_bar(s), ring_parity(it));
          tc_fence_after();
          const uint32_t sa = C.base + s * STAGE_BYTES, sb = sa + 2 * A_SUB;
#pragma unroll
          for (int mt = 0; mt < 2; mt++)
            if (mt < MT && !(P.t.dbg & 8))
              umma_hilo_chunk<true>(C.tmem + (uint32_t)(abuf * 256 + mt * 256), sa + mt * A_SUB, sb, kc - kc_lo);
          umma_commit(C.empty_bar(s));
          if (kc == kc_hi - 1) umma_commit(C.tfull_bar(abuf));
        }
       }
      }
    }
    __syncwarp();
  } else {
    // =============================== LOADER (weights + operand boxes) ===============================
    if (lane == 0) {
      uint32_t it = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int mg = (int)(t % mgroups);
        const int nt = (int)(t / mgroups);
        const int mt0 = mg * MT;
        const int nmt = min(MT, P.t.m_tiles - mt0);
        int g = 0, c0 = 0, len = BN, i0 = 0, y0 = 0, x0 = 0;
        if (P.conv) conv_origin(P, nt, i0, y0, x0); else tile_cols(p, nt, g, c0, len);
        const int row0 = (int)((long)g * p.x_gs + c0);
        for (int kc = 0; kc < KC; kc++, it++) {
          const int s = ring_stage(it);
          mbar_wait(C.empty_bar(s), ring_parity(it) ^ 1);
          const uint32_t abytes = (uint32_t)nmt * A_SUB;
          const bool skipA = P.t.dbg & 2, skipB = P.t.dbg & 4;     // profiling experiments only
          mbar_expect_tx(C.full_bar(s), (skipA ? 0u : abytes) + (skipB ? 0u : 2u * B_HALF));
          const uint32_t sa = C.base + s * STAGE_BYTES, sb = sa + 2 * A_SUB;
          const uint8_t* src = reinterpret_cast<const uint8_t*>(P.t.Wp) + ((size_t)kc * P.t.m_tiles + mt0) * A_SUB;
          if (!skipA) bulk_g2s(sa, src, abytes, C.full_bar(s));
          if (skipB) continue;
          if (P.conv) {
            const int tap = kc / cchunks, cc = kc - tap * cchunks;
            const int dx = tap % 3 - 1, dy = tap / 3 - 1;
            tma_load_4d(sb, &map_hi, cc * BK, x0 + dx, y0 + dy, i0, C.full_bar(s));
            tma_load_4d(sb + B_HALF, &map_lo, cc * BK, x0 + dx, y0 + dy, i0, C.full_bar(s));
          } else {
            tma_load_2d(sb, &map_hi, kc * BK, row0, C.full_bar(s));
            tma_load_2d(sb + B_HALF, &map_lo, kc * BK, row0, C.full_bar(s));
          }
        }
      }
    }
    __syncwarp();
  }
  tc_end(*C.tmem_slot(), warp == T_MMA_WARP);
}

// ---- host side: tensor maps through the driver entry point (no libcuda link dependency) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}
// fp16 [rows][C] matrix (row stride ld elements), box 32 x 256, 64-byte swizzle
static inline int make_map_2d(CUtensorMap* m, const void* basep, long rows, int C, long ld) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return MMMOT_E_ARG;
  cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {32, 256}, es[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(basep), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 900 + (int)r;
}
// fp16 NHWC [n_img][H][W][C], box (32, bx, by, bi)
static inline int make_map_4d(CUtensorMap* m, const void* basep, int n_img, int H, int W, int C, int bx, int by,
                              int bi) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return MMMOT_E_ARG;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n_img};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {32, (cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bi}, es[4] = {1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(basep), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 900 + (int)r;
}

}  // namespace tma

#include "gemm_tma_px.cuh"

int seg_chunk_tab(const int4* tiles, int num_tiles, const int* seg, int4* tab, cudaStream_t st) {
  tma::seg_chunk_tab_kernel<<<mm_cdiv((long)num_tiles * 2, 128), 128, 0, st>>>(tiles, num_tiles, seg, tab);
  MM_LAUNCH_CHECK();
  return 0;
}

// P fully prepared by the caller
static int gemm_tma_launch(const tc::TmaP& P, const CUtensorMap& mh, const CUtensorMap& ml, cudaStream_t st) {
  static std::atomic<unsigned long long> attr{0};
  int grid = 0;
  MM_TRY(tc::tc_grid(tma::gemm_tma_kernel, tma::T_SMEM_BYTES, attr, P.t, &grid));
  tma::gemm_tma_kernel<<<grid, tma::T_THREADS, tma::T_SMEM_BYTES, st>>>(P, mh, ml);
  MM_LAUNCH_CHECK();
  return 0;
}
// pixel-major kernel for 64-channel planar outputs (see gemm_tma_px.cuh); P fully prepared by the caller, P.t.Wp = the
// compact N = 64 weight tiles (weights.py::pack_px).  M = 64, so P.t.m_tiles = 1 and tc_grid's work items are the tiles.
static int gemm_tma_px_launch(const tc::TmaP& P, const CUtensorMap& mh, const CUtensorMap& ml, cudaStream_t st) {
  if (P.t.m_tiles != 1) return MMMOT_E_ARG;
  static std::atomic<unsigned long long> attr{0};
  int grid = 0;
  MM_TRY(tc::tc_grid(tma::gemm_tma_px_kernel<false>, tma::PX_SMEM_BYTES, attr, P.t, &grid));
  tma::gemm_tma_px_kernel<false><<<grid, tma::T_THREADS, tma::PX_SMEM_BYTES, st>>>(P, mh, ml);
  MM_LAUNCH_CHECK();
  return 0;
}

// Crop shapes the GEN27 variant takes: a tile = 256 consecutive pixels of one image, and the tile's neighbourhood,
// (256 + 2W + 2) x 3 floats, is staged in two 8 KB weight slots.  Wider crops need the im2col27 pre-pass.  The K = 32
// operand (27 taps + 5 zeros per pixel, FP16 hi/lo) is generated in shared memory by the kernel's producer warps, so the
// im2col matrix (128 B per pixel written and read back) never exists.  Output: planar FP16 NHWC, bias + ReLU applied.
constexpr int PX_GEN27_MAX_W = 512;
static_assert((tc::BN + 2 * PX_GEN27_MAX_W + 2) * 12 <= 2 * tma::PX_W_SLOT, "GEN27 staging buffer");
bool gemm_tma_px_gen27_fits(int H, int W) { return ((long)H * W) % tc::BN == 0 && W <= PX_GEN27_MAX_W; }

int gemm_tma_px_launch_gen27(const float* crops, int n_img, int H, int W, const uint4* Wpx, float out_scale,
                             const float* bias, __half* Yhi, long y_plane, int* status, cudaStream_t st) {
  if (!crops || !Wpx || !Yhi) return MMMOT_E_ARG;
  const long n_pix = (long)n_img * H * W;
  if (n_pix >= (1L << 31) || !gemm_tma_px_gen27_fits(H, W)) return MMMOT_E_SHAPE;
  tc::TmaP P;
  memset(&P, 0, sizeof(P));
  GemmP g = gemm_defaults();
  g.bias = bias; g.M = 64; g.K = 32; g.relu = 1;
  g.S = (int)n_pix; g.tiles_per_group = mm_cdiv(n_pix, tc::BN); g.num_tiles = g.tiles_per_group;
  g.Y = reinterpret_cast<float*>(Yhi); g.y_ms = 64;
  P.t = tc::tc_params(g, Wpx, out_scale, false);
  P.plane_elems = y_plane;
  P.status = status;
  P.gen_src = crops; P.n_img = n_img; P.H = H; P.W = W;
  static std::atomic<unsigned long long> attr{0};
  int grid = 0;
  MM_TRY(tc::tc_grid(tma::gemm_tma_px_kernel<true>, tma::PX_SMEM_BYTES, attr, P.t, &grid));
  alignas(64) CUtensorMap dummy;
  memset(&dummy, 0, sizeof(dummy));
  tma::gemm_tma_px_kernel<true><<<grid, tma::PX_GEN_THREADS, tma::PX_SMEM_BYTES, st>>>(P, dummy, dummy);
  MM_LAUNCH_CHECK();
  return 0;
}

int gemm_tma_px_launch_mat(const GemmP& g, const uint4* Wpx, float out_scale, const __half* Xhi, long x_plane, long rows,
                           int ldx, long y_plane, int* status, cudaStream_t st) {
  if (!Wpx || g.num_tiles <= 0 || g.K % tc::BK || g.M != 64 || g.y_ms != 64) return MMMOT_E_ARG;
  tc::TmaP P;
  memset(&P, 0, sizeof(P));
  P.t = tc::tc_params(g, Wpx, out_scale, false);
  P.plane_elems = y_plane;
  P.status = status;
  alignas(64) CUtensorMap mh, ml;
  MM_TRY(tma::make_map_2d(&mh, Xhi, rows, g.K, ldx));
  MM_TRY(tma::make_map_2d(&ml, Xhi + x_plane, rows, g.K, ldx));
  return gemm_tma_px_launch(P, mh, ml, st);
}

int gemm_tma_launch_mat(const GemmP& g, const uint4* Wp, float out_scale, const __half* Xhi, long x_plane, long rows,
                        int ldx, cudaStream_t st, unsigned long long* segsum, const int4* chunk_tab) {
  if (!Wp || g.num_tiles <= 0 || g.K % tc::BK) return MMMOT_E_ARG;
  if (g.seg && (g.addend || segsum) && !chunk_tab) return MMMOT_E_ARG;
  tc::TmaP P;
  memset(&P, 0, sizeof(P));
  // two 128-row subtiles per CTA share each operand box; short K chains (<= 16 chunks) are epilogue-bound instead,
  // so they run one subtile per tile and double-buffer the accumulator in TMEM (epilogue overlaps the next MMAs).
  // The arithmetic of a subtile does not depend on this choice.
  P.t = tc::tc_params(g, Wp, out_scale, g.K / tc::BK > 16);
  P.ksegs = 1; P.kc_per_seg = P.t.k_chunks;
  P.segsum = segsum;
  P.chunk_tab = chunk_tab;
  alignas(64) CUtensorMap mh, ml;
  MM_TRY(tma::make_map_2d(&mh, Xhi, rows, g.K, ldx));
  MM_TRY(tma::make_map_2d(&ml, Xhi + x_plane, rows, g.K, ldx));
  return gemm_tma_launch(P, mh, ml, st);
}

int gemm_tma_launch_conv(const GemmP& g0, const uint4* Wp, float out_scale, const __half* Xhi, long x_plane, int n_img,
                         int H, int W, int C, __half* Yhi, long y_plane, cudaStream_t st, float* acc_scratch,
                         long y_plane_pooled, int* did_pool, int* status, unsigned long long* pool_sum, const uint4* Wpx) {
  if (did_pool) *did_pool = 0;
  if (!Wp || C % tc::BK) return MMMOT_E_ARG;
  // box of 256 pixels = bx * by * bi (powers of two): the shape with the least padding waste, widest first
  int bx = 1, by = 1, bi = 256;
  {
    double best = 1e30;
    for (int cx = 256; cx >= 1; cx >>= 1)
      for (int cy = 256 / cx; cy >= 1; cy >>= 1) {
        const int ci = 256 / (cx * cy);
        const double waste = (double)mm_cdiv(W, cx) * cx / W * mm_cdiv(H, cy) * cy / H * mm_cdiv(n_img, ci) * ci / n_img;
        if (waste < best - 1e-9) { best = waste; bx = cx; by = cy; bi = ci; }
      }
  }
  // 64-channel outputs with compact weights run on the pixel-major kernel (gemm_tma_px.cuh) when a 16 x 16
  // single-image box (vertical taps from one halo box, 2x2 pooling windows inside a warp) wastes no more than the best
  // box; for H and W multiples of 16 it always does
  const int seg_chunks = mm_kseg_chunks();   // 0 = single pass
  bool px = Wpx && g0.M == 64 && !g0.part && !(acc_scratch && seg_chunks > 0 && 9 * C / tc::BK > seg_chunks);
  if (px) {
    const double best = (double)mm_cdiv(W, bx) * bx / W * mm_cdiv(H, by) * by / H * mm_cdiv(n_img, bi) * bi / n_img;
    const double w16 = (double)mm_cdiv(W, 16) * 16 / W * mm_cdiv(H, 16) * 16 / H;
    px = w16 <= best + 1e-9;
    if (px) { bx = 16; by = 16; bi = 1; }
  }
  tc::TmaP P;
  memset(&P, 0, sizeof(P));
  GemmP g = g0;
  g.K = 9 * C;
  P.conv = 1; P.bx = bx; P.by = by; P.bi = bi;
  if (px && y_plane_pooled > 0 && did_pool && !(H & 1) && !(W & 1)) {
    P.pool = 1;
    *did_pool = 1;
  }
  // channel-major kernel: the 2x2 max-pool (and SkipPool's per-image sums) fused into the epilogue when every pooling
  // window lies inside one thread's chunks: box rows of <= 32 pixels, an even number of box rows per 128-column half
  if (!px && y_plane_pooled > 0 && did_pool && bx >= 2 && bx <= 32 && by >= 2 && !(H & 1) && !(W & 1)) {
    P.pool = 1;
    P.pool_sum = pool_sum;
    *did_pool = 1;
  }
  P.tiles_x = mm_cdiv(W, bx); P.tiles_y = mm_cdiv(H, by);
  P.n_img = n_img; P.H = H; P.W = W; P.C = C;
  g.num_tiles = P.tiles_x * P.tiles_y * mm_cdiv(n_img, bi);
  g.tile_tab = nullptr;
  g.Y = reinterpret_cast<float*>(Yhi);
  g.y_ms = g.M;
  P.t = tc::tc_params(g, Wp, out_scale, true);
  P.plane_elems = P.pool ? y_plane_pooled : y_plane;
  P.status = status;
  P.ksegs = 1; P.kc_per_seg = P.t.k_chunks;
  if (acc_scratch && seg_chunks > 0 && P.t.k_chunks > seg_chunks) {
    P.ksegs = (P.t.k_chunks + seg_chunks - 1) / seg_chunks;
    P.kc_per_seg = (P.t.k_chunks + P.ksegs - 1) / P.ksegs;
    P.acc_scratch = acc_scratch;
  }
  alignas(64) CUtensorMap mh, ml;
  const int box_y = px ? by + 2 : by;   // pixel-major: halo box of the three vertical taps
  MM_TRY(tma::make_map_4d(&mh, Xhi, n_img, H, W, C, bx, box_y, bi));
  MM_TRY(tma::make_map_4d(&ml, Xhi + x_plane, n_img, H, W, C, bx, box_y, bi));
  if (px) {
    P.t.Wp = Wpx;
    return gemm_tma_px_launch(P, mh, ml, st);
  }
  return gemm_tma_launch(P, mh, ml, st);
}
