// tcgen05 contraction engine, GENERATED-operand variant (sm_100a): the affinity MLP.
//
// Same arithmetic as gemm_tma.cuh (FP16 hi/lo split operands, 3 MMAs per k-step, FP32 accumulate in TMEM) but the
// activation operand never exists in HBM in operand form: eight producer warps build each [256 columns x 32 k]
// FP16 hi/lo block in shared memory, in the UMMA canonical K-major layout, from
//   GEN_PAIR_*  the two feature slabs of the frame-pair:  x[(i,j)][k] = f[i][k] (*|-) f[N+j][k]   (reference
//               modules/gcn.py:6-41; the 3 x 512 x N x M tensor is never stored), or
//   GEN_NORM    the previous layer's fp32 output:  x[s][k] = relu(y[s][k]*sc[g][k] + sh[g][k])   (GroupNorm + ReLU of
//               the producer layer applied on the fly; no normalised copy of the activation is ever written), or
//   GEN_COPY    an fp32 channels-last activation as it is (the small per-detection contractions: fusion, w_det).
// All activations are channels-last ([row][channel]).  A producer thread owns one 8-wide k group of four columns per
// chunk: one 256-bit load per (column, source) — a quarter warp reads eight rows, the four quarters the four k groups
// of the same 128-byte lines — and one 16-byte shared-memory store per (column, plane); the epilogue writes a warp's
// 32 channels of one column as one 128-byte line.  (Load/store instructions and their L1 wavefronts, not the FP32
// pipe, are what the producers compete for with the epilogue.)
//
// CTA (576 threads, persistent, one per SM): warps 0-7 epilogue (TMEM lane quadrant x column half), warp 8 MMA
// issuer, warp 9 weight loader (cp.async.bulk of pre-tiled FP16 hi/lo blocks), warps 10-17 operand producers.
// One mbarrier per stage collects the loader's expect_tx and the eight producer warps' arrivals.
#pragma once
#include "tc_common.cuh"

namespace gen {

using namespace tc;

constexpr int G_EPI_WARPS = 8, G_MMA_WARP = 8, G_LOAD_WARP = 9, G_PROD_WARP0 = 10, G_PROD_WARPS = 8;
constexpr int G_THREADS = (G_PROD_WARP0 + G_PROD_WARPS) * 32;   // 576
constexpr size_t G_SMEM_BYTES = tc_smem_bytes(STAGE_BYTES);
constexpr int G_MAX_K = 512;   // producer-side GroupNorm affine staged in shared memory

struct GenP {
  TcP t;               // .g: M, K, bias, S (columns per group), tiles_per_group, num_tiles, Y / y_gs / y_ms (fp32
                       // channels-last: row = g*y_gs + column), part
  const float* src;    // PAIR: fcl [G][Lf][K] channels-last feature stacks; NORM: fp32 channels-last [G*S][ld_src]
  int ld_src;          // NORM: floats per source row (its first K channels are read)
  const float* gsc;    // NORM: GroupNorm affine of the SOURCE layer, [G][K]
  const float* gsh;
  int n, m, Lf;        // PAIR: columns s = i*m + j, objs = feature rows [0, n), dets = [n, n + m), Lf = n + m
  // FP16 range: the producers do not track the magnitudes they convert (their instruction stream is the kernel's
  // bottleneck); the callers bound the operand instead — PAIR: feats_range_kernel on the feature stacks, NORM:
  // gn_finalize's bound sqrt(count)*|gamma| + |beta| on the normalised values (both raise the status flag).
};

__device__ __forceinline__ void lds128(uint32_t addr, float4& v) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
}
__device__ __forceinline__ void ld_global_256(const float* p, float (&v)[8]) {
  asm volatile("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}

// PAIRED: software-pipelined producers (the next chunk's source vectors are loaded before the current chunk is
// converted).  GEN_COPY: always.  GEN_PAIR_*: only for m == 128, where a 256-column tile is two whole rows i and the
// thread's four items are {row i0, row i0 + 1} x {j = cb, j = cb + 64}: 2 + 2 source vectors instead of 4 + 4, which
// leaves the registers.  GEN_NORM: never; it holds the chunk's GroupNorm affine in registers instead.
template <int GEN, bool PAIRED>
static __global__ void __launch_bounds__(G_THREADS, 1) gemm_gen_kernel(const GenP P) {
  const GemmP& p = P.t.g;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(16) float s_gsc[GEN == GEN_NORM ? G_MAX_K : 4], s_gsh[GEN == GEN_NORM ? G_MAX_K : 4];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // full: the loader's expect_tx arrive + one arrive per producer warp
  const TcPipe C = tc_begin<STAGE_BYTES>(smem_raw, 1 + G_PROD_WARPS, G_EPI_WARPS, warp == G_MMA_WARP);

  const int MT = P.t.mt_per_cta;
  const int mgroups = (P.t.m_tiles + MT - 1) / MT;
  const long total_tiles = (long)p.num_tiles * mgroups;
  const int KC = P.t.k_chunks;
  const int nbuf = (MT == 1) ? 2 : 1;   // accumulator buffers in TMEM (256 columns each when MT == 1)

  if (warp < G_EPI_WARPS) {
    // =============================== EPILOGUE ===============================
    const int q = warp & 3, half = warp >> 2;
    uint32_t wcount = 0;
    for (long t = blockIdx.x; t < total_tiles; t += gridDim.x, wcount++) {
      const int mg = (int)(t % mgroups);
      const int nt = (int)(t / mgroups);
      int g, c0, len;
      tile_cols(p, nt, g, c0, len);
      const int abuf = acc_buf(wcount, nbuf);
      mbar_wait(C.tfull_bar(abuf), acc_parity(wcount, nbuf));
      tc_fence_after();
      for (int mt = 0; mt < MT; mt++) {
        const int co = (mg * MT + mt) * 128 + q * 32 + lane;
        const bool rowok = co < p.M;
        const float bv = (rowok && p.bias) ? __ldg(p.bias + co) : 0.f;
        float f1 = 0.f, f2 = 0.f;   // (sum, sum of squares) over this thread's 128 columns: four fp32 chunk sums
        // channels-last: a warp's 32 consecutive channels of one column are one 128-byte line
        float* dst = p.Y + ((long)g * p.y_gs + c0 + half * 128) * p.y_ms + co;
#pragma unroll 1
        for (int cc = 0; cc < 4; cc++) {
          const int col0 = half * 128 + cc * 32;
          if (col0 >= len) break;   // warp-uniform
          uint32_t v[32];
          tmem_ld32(C.tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(abuf * 256 + mt * 256 + col0), v);
          if (P.t.dbg & 1) continue;
          float s1 = 0.f, s2 = 0.f;
          if (col0 + 32 <= len) {
            if (p.relu) epi_fast<true>(v, P.t.out_scale, bv, s1, s2);
            else epi_fast<false>(v, P.t.out_scale, bv, s1, s2);
          } else {
#pragma unroll
            for (int j = 0; j < 32; j++) {
              float x = fmaf(__uint_as_float(v[j]), P.t.out_scale, bv);
              if (p.relu) x = fmaxf(x, 0.f);
              if (col0 + j >= len) x = 0.f;          // columns beyond the group are not counted (and not stored)
              v[j] = __float_as_uint(x);
              s1 += x; s2 = fmaf(x, x, s2);
            }
          }
          f1 += s1; f2 += s2;
          if (p.Y && rowok) {
            float* d = dst + (long)cc * 32 * p.y_ms;
            if (col0 + 32 <= len) {
#pragma unroll
              for (int j = 0; j < 32; j++) { *d = __uint_as_float(v[j]); d += p.y_ms; }
            } else {
#pragma unroll
              for (int j = 0; j < 32; j++)
                if (col0 + j < len) d[(long)j * p.y_ms] = __uint_as_float(v[j]);
            }
          }
        }
        if (p.part && rowok) p.part[((long)nt * 2 + half) * p.M + co] = make_double2((double)f1, (double)f2);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(C.tempty_bar(abuf));
    }
  } else if (warp == G_MMA_WARP) {
    // =============================== MMA ISSUER ===============================
    if (lane == 0) {
      uint32_t it = 0, tcount = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x, tcount++) {
        const int abuf = acc_buf(tcount, nbuf);
        mbar_wait(C.tempty_bar(abuf), acc_parity(tcount, nbuf) ^ 1);
        tc_fence_after();
        for (int kc = 0; kc < KC; kc++, it++) {
          const int s = ring_stage(it);
          mbar_wait(C.full_bar(s), ring_parity(it));
          tc_fence_after();
          const uint32_t sa = C.base + s * STAGE_BYTES, sb = sa + 2 * A_SUB;
#pragma unroll
          for (int mt = 0; mt < 2; mt++)
            if (mt < MT && !(P.t.dbg & 8))
              umma_hilo_chunk<false>(C.tmem + (uint32_t)(abuf * 256 + mt * 256), sa + mt * A_SUB, sb, kc);
          umma_commit(C.empty_bar(s));                       // stage free once these MMAs have read it
          if (kc == KC - 1) umma_commit(C.tfull_bar(abuf));  // accumulators complete
        }
      }
    }
    __syncwarp();
  } else if (warp == G_LOAD_WARP) {
    // =============================== WEIGHT LOADER ===============================
    if (lane == 0) {
      uint32_t it = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int mg = (int)(t % mgroups);
        const int mt0 = mg * MT;
        const int nmt = min(MT, P.t.m_tiles - mt0);
        for (int kc = 0; kc < KC; kc++, it++) {
          const int s = ring_stage(it);
          mbar_wait(C.empty_bar(s), ring_parity(it) ^ 1);
          const uint32_t bytes = (uint32_t)nmt * A_SUB;
          if (P.t.dbg & 2) { mbar_arrive(C.full_bar(s)); continue; }
          mbar_expect_tx(C.full_bar(s), bytes);
          const uint8_t* src = reinterpret_cast<const uint8_t*>(P.t.Wp) + ((size_t)kc * P.t.m_tiles + mt0) * A_SUB;
          bulk_g2s(C.base + s * STAGE_BYTES, src, bytes, C.full_bar(s));
        }
      }
    }
    __syncwarp();
  } else {
    // =============================== OPERAND PRODUCERS ===============================
    // thread = (k group kg of 8, four columns cb + 64 r).  Per chunk every item is converted, split into FP16 hi/lo
    // and written as one 16-byte piece per plane of the canonical K-major layout:
    //   byte offset = kg * B_LBO + (column / 8) * 128 + (column % 8) * 16
    // (a quarter warp = one kg, eight consecutive columns -> 128 contiguous bytes: conflict-free).
    // The 256-bit source loads of chunk c+1 are issued before chunk c is converted (two register sets, ping-pong), so
    // the L2 transfer of one chunk overlaps the conversion of the previous one; the generic pairwise variant (8 source
    // vectors per chunk) has no registers for that and only overlaps its loads with the wait for the ring slot.
    constexpr bool PREFETCH = PAIRED;
    constexpr bool ROWS = GEN == GEN_NORM || GEN == GEN_COPY;      // the operand is a function of one fp32 source row
    constexpr int NA = (ROWS || !PAIRED) ? 4 : 2;                  // source vectors of 8 floats per chunk: a / y ...
    constexpr int NB = ROWS ? 0 : (PAIRED ? 2 : 4);                // ... and b
    const int pt = tid - G_PROD_WARP0 * 32;   // 0..255
    const int kg = (pt >> 3) & 3;
    const int cb = (pt & 7) + 8 * (pt >> 5);
    const uint32_t off0 = (uint32_t)kg * B_LBO + (uint32_t)(cb >> 3) * 128u + (uint32_t)(cb & 7) * 16u;   // + r * 1024
    uint32_t it = 0;
    int g_staged = -1;
    struct Raw { float a[NA][8]; float b[NB ? NB : 1][8]; };
    for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const int nt = (int)(t / mgroups);
      int g, c0, len;
      tile_cols(p, nt, g, c0, len);
      unsigned okmask = 0;
      // 32-bit element offsets of the items' rows (this thread's k group) relative to the tile's / group's base
      const float* tbase = ROWS ? P.src + ((long)g * p.x_gs + c0) * P.ld_src : P.src + (long)g * P.Lf * p.K;
      int oa[NA], ob[NB ? NB : 1];
#pragma unroll
      for (int r = 0; r < 4; r++) {
        const int col = cb + 64 * r;
        if (col < len) okmask |= 1u << r;
        const int cc = min(col, len - 1);
        if (ROWS) {
          oa[r] = cc * P.ld_src + kg * 8;
        } else {
          const int s = c0 + cc;
          const int i = s / P.m, j = s - i * P.m;
          if (!PAIRED) {
            oa[r] = i * p.K + kg * 8;
            ob[r] = (P.n + j) * p.K + kg * 8;
          } else {
            if (!(r & 1)) oa[r >> 1] = i * p.K + kg * 8;          // r = 0, 2: the two rows i
            if (r < 2) ob[r] = (P.n + j) * p.K + kg * 8;          // r = 0, 1: the two detections j
          }
        }
      }
      if (GEN == GEN_NORM && g != g_staged) {   // same decision in every producer thread: stage the group's affine
        asm volatile("bar.sync 1, %0;" ::"n"(G_PROD_WARPS * 32) : "memory");   // previous tile's readers are done
        for (int k = pt; k < p.K; k += G_PROD_WARPS * 32) {
          s_gsc[k] = __ldg(P.gsc + (long)g * p.K + k);
          s_gsh[k] = __ldg(P.gsh + (long)g * p.K + k);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(G_PROD_WARPS * 32) : "memory");
        g_staged = g;
      }
      auto load = [&](Raw& R, int kc) {
        if (P.t.dbg & 4) return;
#pragma unroll
        for (int r = 0; r < NA; r++) ld_global_256(tbase + oa[r] + kc * BK, R.a[r]);
#pragma unroll
        for (int r = 0; r < NB; r++) ld_global_256(tbase + ob[r] + kc * BK, R.b[r]);
      };
      // wait for the ring slot, convert + store the chunk, publish it
      auto emit = [&](const Raw& R, int kc) {
        const int s = ring_stage(it);
        mbar_wait(C.empty_bar(s), ring_parity(it) ^ 1u);
        uint8_t* bh = C.sm + s * STAGE_BYTES + 2 * A_SUB + off0;
        if (!(P.t.dbg & 4)) {
          const uint32_t sca = smem_u32(s_gsc + kc * BK + kg * 8), sha = smem_u32(s_gsh + kc * BK + kg * 8);
          float4 sc0, sc1, sh0, sh1;
#pragma unroll
          for (int r = 0; r < 4; r++) {
            float x[8];
            if (GEN == GEN_NORM) {
              const float(&y)[8] = R.a[r];
              if (r == 0) { lds128(sca, sc0); lds128(sca + 16, sc1); lds128(sha, sh0); lds128(sha + 16, sh1); }
              x[0] = fmaxf(fmaf(y[0], sc0.x, sh0.x), 0.f); x[1] = fmaxf(fmaf(y[1], sc0.y, sh0.y), 0.f);
              x[2] = fmaxf(fmaf(y[2], sc0.z, sh0.z), 0.f); x[3] = fmaxf(fmaf(y[3], sc0.w, sh0.w), 0.f);
              x[4] = fmaxf(fmaf(y[4], sc1.x, sh1.x), 0.f); x[5] = fmaxf(fmaf(y[5], sc1.y, sh1.y), 0.f);
              x[6] = fmaxf(fmaf(y[6], sc1.z, sh1.z), 0.f); x[7] = fmaxf(fmaf(y[7], sc1.w, sh1.w), 0.f);
            } else if (GEN == GEN_COPY) {
#pragma unroll
              for (int e = 0; e < 8; e++) x[e] = R.a[r][e];
            } else {
              const float(&av)[8] = R.a[PAIRED ? (r >> 1) : r];
              const float(&bv)[8] = R.b[NB ? (PAIRED ? (r & 1) : r) : 0];
#pragma unroll
              for (int e = 0; e < 8; e++) {
                if (GEN == GEN_PAIR_MUL) x[e] = av[e] * bv[e];
                else if (GEN == GEN_PAIR_ABS) x[e] = fabsf(av[e] - bv[e]) * 0.5f;   // == |(a - b) / 2| exactly; |.| folds into the FMUL
                else x[e] = (av[e] - bv[e]) * 0.5f;
              }
            }
            uint32_t h[4], l[4];
#pragma unroll
            for (int q = 0; q < 4; q++) split_f16x2(x[2 * q], x[2 * q + 1], h[q], l[q]);
            if (!((okmask >> r) & 1u)) { h[0] = h[1] = h[2] = h[3] = 0u; l[0] = l[1] = l[2] = l[3] = 0u; }   // beyond the group
            *reinterpret_cast<uint4*>(bh + r * 1024) = make_uint4(h[0], h[1], h[2], h[3]);
            *reinterpret_cast<uint4*>(bh + B_HALF + r * 1024) = make_uint4(l[0], l[1], l[2], l[3]);
          }
        }
        fence_async_smem();   // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(C.full_bar(s));
        it++;
      };
      if (PREFETCH) {
        Raw R0, R1;
        load(R0, 0);
        for (int kc = 0; kc < KC; kc += 2) {
          if (kc + 1 < KC) load(R1, kc + 1);
          emit(R0, kc);
          if (kc + 1 < KC) {
            if (kc + 2 < KC) load(R0, kc + 2);
            emit(R1, kc + 1);
          }
        }
      } else {
        for (int kc = 0; kc < KC; kc++) {
          Raw R;
          load(R, kc);
          emit(R, kc);
        }
      }
    }
  }

  tc_end(C.tmem, warp == G_MMA_WARP);
}

}  // namespace gen

template <int GEN, bool PAIRED>
static int gemm_gen_launch_t(const GemmP& g, const uint4* Wp, float out_scale, const float* src, int ld_src,
                           const float* gsc, const float* gsh, int n, int m, int Lf, cudaStream_t st) {
  if (!Wp || !src || g.num_tiles <= 0 || g.K % tc::BK) return MMMOT_E_ARG;
  if (g.tile_tab && ((GEN != gen::GEN_NORM && GEN != gen::GEN_COPY) || g.x_gs || g.y_gs)) return MMMOT_E_ARG;
  if (GEN == gen::GEN_NORM && (g.K > gen::G_MAX_K || !gsc || !gsh)) return MMMOT_E_ARG;
  if ((GEN == gen::GEN_NORM || GEN == gen::GEN_COPY) && (ld_src < g.K || (ld_src & 7))) return MMMOT_E_ARG;
  gen::GenP P;
  memset(&P, 0, sizeof(P));
  P.t = tc::tc_params(g, Wp, out_scale, true);   // M = 128: one subtile, two TMEM accumulator buffers
  P.src = src; P.ld_src = ld_src; P.gsc = gsc; P.gsh = gsh;
  P.n = n; P.m = m; P.Lf = Lf;
  static std::atomic<unsigned long long> attr{0};
  int grid = 0;
  MM_TRY(tc::tc_grid(gen::gemm_gen_kernel<GEN, PAIRED>, gen::G_SMEM_BYTES, attr, P.t, &grid));
  gen::gemm_gen_kernel<GEN, PAIRED><<<grid, gen::G_THREADS, gen::G_SMEM_BYTES, st>>>(P);
  MM_LAUNCH_CHECK();
  return 0;
}

template <int GEN>
int gemm_gen_launch(const GemmP& g, const uint4* Wp, float out_scale, const float* src, int ld_src, const float* gsc,
                    const float* gsh, int n, int m, int Lf, cudaStream_t st) {
  // PAIRED as documented at gemm_gen_kernel
  if constexpr (GEN == gen::GEN_NORM)
    return gemm_gen_launch_t<GEN, false>(g, Wp, out_scale, src, ld_src, gsc, gsh, n, m, Lf, st);
  else if constexpr (GEN == gen::GEN_COPY)
    return gemm_gen_launch_t<GEN, true>(g, Wp, out_scale, src, ld_src, gsc, gsh, n, m, Lf, st);
  else if (m == 128)
    return gemm_gen_launch_t<GEN, true>(g, Wp, out_scale, src, ld_src, gsc, gsh, n, m, Lf, st);
  else
    return gemm_gen_launch_t<GEN, false>(g, Wp, out_scale, src, ld_src, gsc, gsh, n, m, Lf, st);
}
