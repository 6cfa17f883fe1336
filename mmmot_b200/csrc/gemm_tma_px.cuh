// tcgen05 contraction engine, pixel-major variant for 64-channel outputs (the first two VGG layers).
//
// With Cout = 64 the channel-major kernel (gemm_tma.cuh) pads the MMA's M from 64 to 128 — half of every
// tensor-core instruction is zeros and half of the epilogue warps cannot reach any valid TMEM lane.  Here the
// roles are swapped: the 256-pixel activation box is the A operand (two M=128 subtiles, K-major SWIZZLE_64B, as
// TMA writes it) and the compact weight tiles (below) are the B operand.  D[pixel][channel] lives in TMEM lanes =
// pixels, so all eight epilogue warps work, every thread owns 32 consecutive channels of one pixel and stores its 64
// bytes per plane directly — no shared-memory transpose.  Two 256-column accumulator buffers: the epilogue of tile i
// overlaps the MMAs of tile i+1.
// Same arithmetic as the channel-major kernel: FP16 hi/lo split operands, D += Xhi*Whi + Xhi*Wlo + Xlo*Whi.
#pragma once

namespace tma {

// Conv mode (3x3 conv, 16 x 16 single-image box): a stage holds the (by+2)-row halo box of ONE horizontal tap and
// channel chunk; its three vertical taps are the same shared-memory box read at start addresses dy*bx*64 B (whole
// swizzle atoms for bx >= 8), so the activation traffic from L2 — what bounds this layer — drops from 9 to
// 3*(by+2)/by boxes per chunk.  Optional fused 2x2 max-pool: with bx <= 16 a warp's 32 pixels are whole pooling windows
// (lanes l, l^1, l^bx, l^(bx+1)), so the pooled NHWC planes are written directly and the full-resolution activation
// never exists.
constexpr int PX_W_SLOT = 8192;                 // one k chunk of the compact weight tiles (below)
constexpr int PX_X_OFF = 3 * PX_W_SLOT;         // 24 KB: three tap slots
constexpr int PX_X_PLANE = 24576;               // up to 384 box rows x 64 B per plane
constexpr int PX_STAGE = PX_X_OFF + 2 * PX_X_PLANE;   // 72 KB
constexpr size_t PX_SMEM_BYTES = tc_smem_bytes(PX_STAGE);

constexpr uint32_t IDESC_N64 = (1u << 4) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
constexpr uint32_t IDESC_N128 = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
// Compact weight tiles (weights.py::pack_px): [k group 4][hi rows 0-63 | lo rows 0-63][8 rows][8 k], i.e. per k group a
// 128-row K-major block whose first 64 rows are W_hi and last 64 rows W_lo.  With them the three MMAs of a k-step become
// two:  D[:, 0:128] += X_hi * [W_hi ; W_lo]^T  (N = 128: X_hi is read from shared memory once for both products) and
// D[:, 0:64] += X_lo * W_hi^T; the epilogue adds columns 64..127 (the X_hi*W_lo partial) to columns 0..63.  The N = 64
// MMAs are bound by shared-memory operand bandwidth (4 KB of pixels + 2 KB of weights per 32-clock MMA = 192 B/clk
// against 128 B/clk), so reading X_hi once per k-step instead of twice is what this buys.
constexpr int PX_WC_LBO = 2048;

// GEN27 variant (first VGG layer): eight extra producer warps build the K = 32 activation operand of every tile — the 27
// taps of each pixel read from the fp32 NCHW crop, zero padding at the borders, FP16 hi/lo split — directly in the
// SWIZZLE_64B layout TMA would have written (row = pixel, 64 B per plane; 16-byte chunk c of row r lives at chunk
// c ^ ((r >> 1) & 3)).  Four warps (one group) complete a tile's full barrier.
constexpr int PX_GEN_WARPS = 4, PX_GEN_THREADS = T_THREADS + 2 * 32 * PX_GEN_WARPS;

template <bool GEN27>
static __global__ void __launch_bounds__(GEN27 ? PX_GEN_THREADS : T_THREADS, 1)
gemm_tma_px_kernel(const TmaP P, const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo) {
  const GemmP& p = P.t.g;
  extern __shared__ uint8_t smem_raw[];
  __shared__ float s_bias[64];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long total_tiles = p.num_tiles;
  const int cchunks = P.C / BK;                          // conv: channel chunks per tap
  const int ntap = P.conv ? 3 : 1;                       // vertical taps served by one stage
  const int nstage = P.conv ? 3 * cchunks : P.t.k_chunks;   // stages per tile
  const uint32_t xbytes = P.conv ? (uint32_t)(P.bx * (P.by + 2) * 64) : (uint32_t)B_HALF;

  if (tid < 64) s_bias[tid] = p.bias ? p.bias[tid] : 0.f;
  // full: the loader's expect_tx arrive (+ one arrive per GEN27 producer warp of a group)
  const TcPipe C = tc_begin<PX_STAGE>(smem_raw, GEN27 ? 1 + PX_GEN_WARPS : 1, T_EPI_WARPS, warp == T_MMA_WARP);

  if (warp < T_EPI_WARPS) {
    // =============================== EPILOGUE ===============================
    const int q = warp & 3, cb = (warp >> 2) * 32;   // TMEM lane quadrant (pixels), channel half
    const int lbx = 31 - __clz(max(P.bx, 1)), lby = 31 - __clz(max(P.by, 1));
    __half* yh = reinterpret_cast<__half*>(p.Y);
    uint32_t wcount = 0, racc = 0;   // racc: running max of the converted |hi| values (FP16 range guard)
    // an int tile index (tile counts are < 2^31) keeps the GEN27 variant, at its 96-register cap, from spilling wcount
    for (int nt = blockIdx.x; nt < total_tiles; nt += gridDim.x, wcount++) {
      int i0 = 0, y0 = 0, x0 = 0;
      if (P.conv) conv_origin(P, nt, i0, y0, x0);
      const int abuf = acc_buf(wcount, 2);
      mbar_wait(C.tfull_bar(abuf), acc_parity(wcount, 2));
      tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < 2; sub++) {
        const int col = sub * 128 + q * 32 + lane;
        bool ok;
        long o;
        if (P.conv) {
          const int xx = col & (P.bx - 1), r = col >> lbx;
          const int yy = r & (P.by - 1), ii = r >> lby;
          const int img = i0 + ii, y = y0 + yy, xg = x0 + xx;
          ok = img < P.n_img && y < P.H && xg < P.W;
          o = (((long)img * P.H + y) * P.W + xg) * 64 + cb;
        } else {
          const long row = (long)nt * BN + col;
          ok = row < p.S;
          o = row * 64 + cb;
        }
        // accumulator = columns [0, 64) (hi*hi + lo*hi) + columns [64, 128) (hi*lo partial)
        uint32_t v[32], v2[32];
        tmem_ld32(C.tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(abuf * 256 + sub * 128 + cb), v);
        tmem_ld32(C.tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(abuf * 256 + sub * 128 + 64 + cb), v2);
#pragma unroll
        for (int j = 0; j < 32; j++) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v2[j]));
        if (P.t.dbg & 1) continue;
        if (P.pool) {
          // 2x2 max over lanes l, l^1 (x) and l^bx (y); bias + ReLU commute with the max and are applied below
#pragma unroll
          for (int j = 0; j < 32; j++) {
            float a = __uint_as_float(v[j]);
            a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, 1));
            a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, P.bx));
            v[j] = __float_as_uint(a);
          }
          const int xx = col & (P.bx - 1), r = col >> lbx;
          const int yy = r & (P.by - 1);
          const int y = y0 + yy, xg = x0 + xx;
          ok = ok && !(xx & 1) && !(yy & 1);
          o = (((long)(i0 + (r >> lby)) * (P.H >> 1) + (y >> 1)) * (P.W >> 1) + (xg >> 1)) * 64 + cb;
          if (!ok) continue;
        }
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float x0v = fmaf(__uint_as_float(v[j]), P.t.out_scale, s_bias[cb + j]);
          float x1v = fmaf(__uint_as_float(v[j + 1]), P.t.out_scale, s_bias[cb + j + 1]);
          if (p.relu) { x0v = fmaxf(x0v, 0.f); x1v = fmaxf(x1v, 0.f); }
          split_f16x2(x0v, x1v, hi[j >> 1], lo[j >> 1]);
          mm_range_track2(racc, hi[j >> 1]);
        }
        if (GEN27) {
          // Line-coalesced stores.  A thread owns 64 B per plane of ONE pixel, so a warp-wide store of it touches 32
          // different 128-byte lines (32 LSU wavefronts per instruction; this epilogue is what bounds the layer).  The
          // two warps of a TMEM lane quadrant (channel halves 0-31 / 32-63 of the same 32 pixels) exchange through an
          // 8 KB scratch [plane][pixel][128 B] (16-byte chunk c of pixel p at slot c ^ (p & 7): conflict-free both ways)
          // in an unused tail of the stage buffers; then one warp stores the hi plane, the other the lo plane, every
          // instruction writing 8 complete lines.
          const uint32_t scr = C.base + (uint32_t)((q >> 1) * PX_STAGE + PX_X_OFF + (q & 1) * PX_X_PLANE + 16384);
          const uint32_t rowa = scr + (uint32_t)lane * 128u;
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const uint32_t slot = (uint32_t)((((cb >> 3) + k) ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowa + slot), "r"(hi[4 * k]), "r"(hi[4 * k + 1]),
                         "r"(hi[4 * k + 2]), "r"(hi[4 * k + 3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowa + 4096u + slot), "r"(lo[4 * k]),
                         "r"(lo[4 * k + 1]), "r"(lo[4 * k + 2]), "r"(lo[4 * k + 3]) : "memory");
          }
          asm volatile("bar.sync %0, 64;" ::"r"(3 + q) : "memory");
          const int h = warp >> 2;                                   // plane this warp stores
          const long row0 = (long)nt * BN + sub * 128 + q * 32;
          __half* dstp = yh + (long)h * P.plane_elems + row0 * 64;
#pragma unroll
          for (int r = 0; r < 4; r++) {
            const int idx = r * 32 + lane, px = idx >> 2, c = (idx & 3) * 2;
            const uint32_t ra = scr + (uint32_t)h * 4096u + (uint32_t)px * 128u;
            uint32_t w[8];
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3])
                         : "r"(ra + (uint32_t)((c ^ (px & 7)) << 4)));
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                         : "r"(ra + (uint32_t)(((c + 1) ^ (px & 7)) << 4)));
            if (row0 + px < p.S) st_global_256(dstp + (long)px * 64 + c * 8, w);
          }
          asm volatile("bar.sync %0, 64;" ::"r"(3 + q) : "memory");   // scratch free for the next subtile
        } else if (ok) {
          // 256-bit stores: every instruction writes whole 32-byte sectors (two per plane per thread)
          st_global_256(yh + o, hi);
          st_global_256(yh + o + 16, hi + 8);
          st_global_256(yh + o + P.plane_elems, lo);
          st_global_256(yh + o + P.plane_elems + 16, lo + 8);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(C.tempty_bar(abuf));
    }
    mm_range_flag2(P.status, racc);
  } else if (warp == T_MMA_WARP) {
    // =============================== MMA ISSUER ===============================
    if (lane == 0) {
      uint32_t it = 0, tcount = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x, tcount++) {
        const int abuf = acc_buf(tcount, 2);
        mbar_wait(C.tempty_bar(abuf), acc_parity(tcount, 2) ^ 1);
        tc_fence_after();
        for (int si = 0; si < nstage; si++, it++) {
          const int s = ring_stage(it);
          mbar_wait(C.full_bar(s), ring_parity(it));
          tc_fence_after();
          const uint32_t sw = C.base + s * PX_STAGE, sx = sw + PX_X_OFF;
          if (!(P.t.dbg & 8)) {
            for (int ky = 0; ky < ntap; ky++) {
              const uint32_t xo = sx + (uint32_t)(ky * P.bx * 64), wo = sw + (uint32_t)(ky * PX_W_SLOT);
#pragma unroll
              for (int sub = 0; sub < 2; sub++) {
#pragma unroll
                for (int ks = 0; ks < 2; ks++) {
                  const uint64_t x_hi = smem_desc_sw64(xo + sub * (128 * 64) + ks * 32);
                  const uint64_t x_lo = smem_desc_sw64(xo + PX_X_PLANE + sub * (128 * 64) + ks * 32);
                  const uint64_t w_hl = smem_desc(wo + ks * 2 * PX_WC_LBO, PX_WC_LBO, SBO);   // rows 0-63 W_hi, 64-127 W_lo
                  const uint32_t d = C.tmem + (uint32_t)(abuf * 256 + sub * 128);
                  umma_f16(d, x_hi, w_hl, IDESC_N128, (si | ky | ks) ? 1u : 0u);
                  umma_f16(d, x_lo, w_hl, IDESC_N64, 1u);
                }
              }
            }
          }
          umma_commit(C.empty_bar(s));
          if (si == nstage - 1) umma_commit(C.tfull_bar(abuf));
        }
      }
    }
    __syncwarp();
  } else if (GEN27 && warp > T_LOAD_WARP) {
    // =============================== OPERAND PRODUCERS (first VGG layer) ===============================
    // Two groups of four warps take alternate tiles.  A tile is 256 consecutive pixels of ONE image (H*W is a multiple of
    // 256); the group first stages the pixels' 3-channel neighbourhood — the linear range [r0 - W - 1, r0 + 256 + W + 1)
    // of each channel, zero outside the image — in the stage's two unused weight slots with coalesced loads, then every
    // thread gathers the 27 taps of its two pixels from shared memory (left / right image borders by predicate).
    const int pw = warp - (T_LOAD_WARP + 1);
    const int grp = pw >> 2;
    const int pt = (pw & 3) * 32 + lane;        // 0..127: rows pt and pt + 128 of the group's tiles
    const int W = P.W, hw = P.H * P.W;
    const int span = BN + 2 * W + 2;
    float amax = 0.f;
    uint32_t it = (uint32_t)grp;
    for (long t = blockIdx.x + (long)grp * gridDim.x; t < total_tiles; t += 2L * gridDim.x, it += 2) {
      const int s = ring_stage(it);
      const long row0 = t * BN;
      const long img = row0 / hw;
      const int r0 = (int)(row0 - img * hw);
      const float* src = P.gen_src + img * 3 * hw;
      mbar_wait(C.empty_bar(s), ring_parity(it) ^ 1);
      float* stg = reinterpret_cast<float*>(C.sm + s * PX_STAGE + PX_W_SLOT);
      const int lin0 = r0 - W - 1;
      if (P.t.dbg & 4) {                         // profiling: no operand generation (results wrong)
        __syncwarp();
        if (lane == 0) mbar_arrive(C.full_bar(s));
        continue;
      }
#pragma unroll 1
      for (int i0 = pt; i0 < 3 * span; i0 += 8 * 128) {
        float q[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {           // eight independent loads in flight per thread
          const int i = i0 + u * 128;
          const int ci = i / span, lin = lin0 + (i - ci * span);
          q[u] = (i < 3 * span && lin >= 0 && lin < hw) ? __ldg(src + (long)ci * hw + lin) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; u++)
          if (i0 + u * 128 < 3 * span) stg[i0 + u * 128] = q[u];
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
      const uint32_t sx = C.base + s * PX_STAGE + PX_X_OFF;
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const int rr = j * 128 + pt;
        const int x = (r0 + rr) % W;
        const bool xl = x > 0, xr = x < W - 1;
        const float* c = stg + rr + W + 1;
        float v[28];
#pragma unroll
        for (int ci = 0; ci < 3; ci++)
#pragma unroll
          for (int ky = 0; ky < 3; ky++)
#pragma unroll
            for (int kx = 0; kx < 3; kx++) {
              float q = c[ci * span + (ky - 1) * W + (kx - 1)];
              if (kx == 0 && !xl) q = 0.f;
              if (kx == 2 && !xr) q = 0.f;
              v[ci * 9 + ky * 3 + kx] = q;
              amax = fmaxf(amax, fabsf(q));
            }
        v[27] = 0.f;
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int k = 0; k < 28; k += 2) split_f16x2(v[k], v[k + 1], hi[k >> 1], lo[k >> 1]);
        hi[14] = hi[15] = lo[14] = lo[15] = 0u;
        const uint32_t rowaddr = sx + (uint32_t)rr * 64u, sw = (uint32_t)((rr >> 1) & 3);
#pragma unroll
        for (int cch = 0; cch < 4; cch++) {
          const uint32_t a = rowaddr + ((cch ^ sw) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(hi[4 * cch]), "r"(hi[4 * cch + 1]),
                       "r"(hi[4 * cch + 2]), "r"(hi[4 * cch + 3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + PX_X_PLANE), "r"(lo[4 * cch]),
                       "r"(lo[4 * cch + 1]), "r"(lo[4 * cch + 2]), "r"(lo[4 * cch + 3]) : "memory");
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the MMA's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive(C.full_bar(s));
    }
    mm_range_flag(P.status, amax);
  } else {
    // =============================== LOADER ===============================
    if (lane == 0) {
      uint32_t it = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int nt = (int)t;
        int i0 = 0, y0 = 0, x0 = 0;
        if (P.conv) conv_origin(P, nt, i0, y0, x0);
        for (int si = 0; si < nstage; si++, it++) {
          const int s = ring_stage(it);
          mbar_wait(C.empty_bar(s), ring_parity(it) ^ 1);
          mbar_expect_tx(C.full_bar(s), (uint32_t)ntap * PX_W_SLOT + (GEN27 ? 0u : 2u * xbytes));
          const uint32_t sw = C.base + s * PX_STAGE, sx = sw + PX_X_OFF;
          const int kx = P.conv ? si / cchunks : 0, cc = P.conv ? si - kx * cchunks : 0;
          for (int ky = 0; ky < ntap; ky++) {
            // weights pre-packed for N = 64 (weights.py::pack_px): one 8 KB copy per k chunk
            const int kc = P.conv ? (ky * 3 + kx) * cchunks + cc : si;
            bulk_g2s(sw + ky * PX_W_SLOT, reinterpret_cast<const uint8_t*>(P.t.Wp) + (size_t)kc * PX_W_SLOT, PX_W_SLOT, C.full_bar(s));
          }
          if (P.conv) {
            tma_load_4d(sx, &map_hi, cc * BK, x0 + kx - 1, y0 - 1, i0, C.full_bar(s));
            tma_load_4d(sx + PX_X_PLANE, &map_lo, cc * BK, x0 + kx - 1, y0 - 1, i0, C.full_bar(s));
          } else if (!GEN27) {
            tma_load_2d(sx, &map_hi, si * BK, nt * BN, C.full_bar(s));
            tma_load_2d(sx + PX_X_PLANE, &map_lo, si * BK, nt * BN, C.full_bar(s));
          }
        }
      }
    }
    __syncwarp();
  }

  tc_end(*C.tmem_slot(), warp == T_MMA_WARP);
}

}  // namespace tma
