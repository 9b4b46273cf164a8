// Tensor-core evaluation of the leaf value net (Net2: Linear -> LayerNorm -> GELU -> Linear -> LayerNorm -> GELU -> Linear,
// cfvpy/models.py:64-94) for all pseudo-leaf query rows of a wave, generation 3: tcgen05.mma kind::f16 with fp32 accumulation in
// TMEM, weights resident in shared memory, activations fed back to the tensor cores from TMEM, scheduled so that the epilogue
// warps never wait for the tensor pipe, and with every global->shared transfer done by the bulk-copy engine (cp.async.bulk +
// mbarrier complete_tx; SASS: UBLKCP).  Primitives and the weight-blob layout: leaf_mlp_tc.cuh.
//
// What changed against generation 1 (a one-tile kernel, removed after commit 76e7204; measured there: 11 100 cycles per 128-row
// tile = 2 x 4 550 epilogue + 1 340 exposed MMA tails + 500 output; tensor pipe 26 % busy):
//
//  1. TWO TILES IN FLIGHT, ONE ACCUMULATOR REGION.  TMEM = D [0,256) | A0 [256,384) | A1 [384,512): a single fp32 accumulator
//     region shared by both tiles and one fp16 A-operand region per tile.  The 16 epilogue warps run the phases
//         E1(X) E1(Y) E2(X) E2(Y)   E1(X') E1(Y') ...
//     and every phase starts by pulling the accumulators into registers (64 per thread), which frees D at once; the issuer then
//     runs the big MMA of the OTHER tile (layer 2 of X under E1(Y), layer 2 of Y under E2(X), ...) while this phase computes.
//     Layer 3 (N = 16) of a tile is issued into D[0,16) right after the next phase has emptied D and is read by the four
//     column-quarter-0 warps after their first sub-chunk; the next layer-1 MMA follows.  No accumulator is ever waited for
//     except at the very first tile and for a CTA's odd last tile.  (Generation 2 — leaf_mlp_tc2.cuh of round 1, removed —
//     kept two accumulator regions and moved A through shared memory; its SS MMAs then competed with the epilogue for
//     shared-memory bandwidth and it was slower.  Here A stays in TMEM.)
//  2. MEAN-FREE LayerNorm.  The rows of W1 / W2 and the biases are centred over the 256 output features on the host
//     (W'[j][k] = W[j][k] - mean_j W[j][k]), so sum_j y_j = 0 by construction and LayerNorm needs only sum_j y_j^2: the
//     running-sum chain, the mean and the shift disappear from the epilogue (two-pass-quality variance for free).
//  3. HALVED GELU ARGUMENT.  The affine produces hy = y / 2 directly (gamma / 2 and beta / 2 are stored), the tanh polynomial is
//     rescaled to hy, and GELU(y) = hy + hy * tanh(.): one multiply fewer per pair than before.  Evaluated with packed
//     f32x2 FMAs + tanh.approx.f32, rounded to fp16 once (gelu_hy_t32).  A packed-fp16 evaluation (gelu_hy_x2, now only in the
//     GELU table of cfrb_api.cu) was 6 % faster but inherits the truncation of tanh.approx.f16x2; it was removed after 76e7204.
//  4. One mbarrier arrival per WARP (lane 0 after __syncwarp) instead of per thread, one A-operand hand-over per phase instead of
//     four, LayerNorm partial sums exchanged between the four warps of a row quadrant only (named barrier of 128 threads).
//  5. Weights (once per CTA) and query tiles (double-buffered, issued two tiles ahead by the MMA warp) arrive by cp.async.bulk.
#pragma once
#include "leaf_mlp_tc.cuh"

namespace cfrb {
namespace tc {

constexpr uint32_t kColA0 = 256, kColA1 = 384;

struct Tc3Layout {
  BlobLayout L;
  int x_bytes, off_x0, off_x1, off_part, off_bar, smem_bytes;
  __host__ __device__ explicit Tc3Layout(int kp) : L(kp) {
    x_bytes = kTileM * kp * 2;
    off_x0 = L.off_x;
    off_x1 = off_x0 + x_bytes;
    off_part = off_x1 + x_bytes;                // LayerNorm partial sums: [2 buffers][kParts][128 rows] float
    off_bar = off_part + 2 * kParts * kTileM * 4;
    smem_bytes = off_bar + 128;                 // 12 mbarriers + TMEM base slot
  }
};

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bulk copy global -> shared (the TMA engine without a tensor map); completion is signalled on the mbarrier as transaction bytes.
__device__ __forceinline__ void bulk_g2s(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst), "l"(gsrc),
               "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// GELU(y) for a packed pair given hy = y / 2:  hy + hy * tanh(hy (c0 + c1 hy^2 + c2 hy^4)), the fit
// tanh(y (0.797496 + 3.70057e-2 y^2 - 3.5151e-4 y^4)) rescaled to hy (c0 = 2 x, c1 = 8 x, c2 = 32 x) and the clamp y^2 <= 52 as
// hy^2 <= 13.  fp32 arithmetic (packed f32x2 FMAs, tanh.approx.f32) with ONE rounding to fp16 at the end.  Not fp16: measured on
// B200 (profiles/r2_gelu_table.log), tanh.approx.f16x2 truncates towards zero (mean error -2.4e-4 sign(u) on 0.25 <= |u| < 4, one
// fp16 ulp at most), which gives the packed-fp16 evaluation (gelu_hy_x2, cfrb_api.cu) a coherent negative bias of 1.6e-4 ..
// 3.9e-4 on every activation with |y| > 0.5; the data-generation statistics of the self-play loop respond to that bias
// (tests/test_rela_module.py P5), not to the rounding noise.
__device__ __forceinline__ uint32_t gelu_hy_t32(float hy0, float hy1) {
  const f32x2 hy = pack2(hy0, hy1);
  float s0, s1;
  unpack2(mul2(hy, hy), s0, s1);
  const f32x2 s = pack2(fminf(s0, 13.f), fminf(s1, 13.f));
  const f32x2 p = fma2(s, fma2(s, pack2(-1.124832e-2f, -1.124832e-2f), pack2(2.960456e-1f, 2.960456e-1f)), pack2(1.594992f, 1.594992f));
  float u0, u1, t0, t1, g0, g1;
  unpack2(mul2(hy, p), u0, u1);
  asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(u0));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(u1));
  unpack2(fma2(hy, pack2(t0, t1), hy), g0, g1);
  const __half2 g = __floats2half2_rn(g0, g1);
  return *reinterpret_cast<const uint32_t*>(&g);
}

#define CFRB_TRACE3(slot)                                                                 \
  do {                                                                                    \
    if (kDebug && a.trace && blockIdx.x == 0 && (slot) < 2048) a.trace[slot] = clock64(); \
  } while (0)

// kGelu: 0 = fp32 logistic GELU (CFRB_NET_TC_F16; the LayerNorm parameters in the blob are gamma, beta); 2 = fp32 tanh GELU
// (CFRB_NET_TC_F16X2; gamma / 2, beta / 2).
template <bool kDebug, int kGelu>
__global__ void __launch_bounds__(kThreads, 1) leaf_mlp_tc3_kernel(TcArgs a) {
  constexpr int kMmaWarp = kEpiThreads / 32;
  extern __shared__ __align__(1024) uint8_t smem[];
  const Tc3Layout T(a.Kp);
  const BlobLayout& L = T.L;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rows = *a.rows_ptr;
  const int ntiles = (rows + kTileM - 1) / kTileM;
  if ((int)blockIdx.x >= ntiles) return;
  const int J = (ntiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1;      // tiles of this CTA: blockIdx.x + j * gridDim.x
  const int nphases = 2 * J;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + T.off_bar);
  // 0 weights | 1,2 x[buffer] | 3 dready | 4 dfree | 5,6 a[buffer] | 7 d3 | 8 dout
  const uint32_t bar_w = smem_u32(bars + 0), bar_x = smem_u32(bars + 1), bar_dready = smem_u32(bars + 3), bar_dfree = smem_u32(bars + 4),
                 bar_a = smem_u32(bars + 5), bar_d3 = smem_u32(bars + 7), bar_dout = smem_u32(bars + 8);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  if (tid == 0) {
    mbar_init(bar_w, 1); mbar_init(bar_x, 1); mbar_init(bar_x + 8, 1);
    mbar_init(bar_dready, 1); mbar_init(bar_dfree, kEpiThreads / 32);
    mbar_init(bar_a, kEpiThreads / 32); mbar_init(bar_a + 8, kEpiThreads / 32);
    mbar_init(bar_d3, 1); mbar_init(bar_dout, kParts);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // weights: independent of the CFR kernel that precedes this launch -> fetched while that kernel drains (PDL)
  if (warp == kMmaWarp && lane == 0) {
    mbar_expect_tx(bar_w, (uint32_t)L.blob_bytes);
    for (int o = 0; o < L.blob_bytes; o += 32768)
      bulk_g2s(smem_u32(smem + o), a.blob + o, (uint32_t)min(32768, L.blob_bytes - o), bar_w);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;");

  const uint32_t sw1 = smem_u32(smem + L.off_w1), sw2 = smem_u32(smem + L.off_w2), sw3 = smem_u32(smem + L.off_w3),
                 sones = smem_u32(smem + L.off_ones), sbias2 = smem_u32(smem + L.off_bias2);
  const uint32_t sx0 = smem_u32(smem + T.off_x0);
  auto tile_of = [&](int j) { return (int)blockIdx.x + j * (int)gridDim.x; };
  // phase k of this CTA: pair m = k / 4 (two tiles), within the pair E1(X) E1(Y) E2(X) E2(Y); a pair with a single tile has
  // two phases.  phase_tile / phase_layer are the same arithmetic on both sides.
  auto phase_of = [&](int k, int& j, int& layer) {
    const int full = J / 2;                    // pairs with two tiles
    if (k < 4 * full) { const int m = k >> 2, r = k & 3; j = 2 * m + (r & 1); layer = r >> 1; }
    else { j = J - 1; layer = k - 4 * full; }
  };

  if (warp == kMmaWarp) {
    // ===================== MMA issuer + bulk-copy producer (one thread) =====================
    if (lane == 0) {
      const uint32_t idesc256 = make_idesc(kTileM, kHid), idesc16 = make_idesc(kTileM, kNout);
      const uint32_t lbo_x = (kTileM / 8) * 128, lbo_w = (kHid / 8) * 128, lbo_w3 = (kNout / 8) * 128;
      const size_t x_tile_bytes = (size_t)T.x_bytes;
      const uint8_t* xg = reinterpret_cast<const uint8_t*>(a.Xh);
      auto fetch_x = [&](int j) {              // query tile of the CTA's j-th tile -> x buffer j & 1
        const uint32_t b = bar_x + 8 * (j & 1);
        mbar_expect_tx(b, (uint32_t)x_tile_bytes);
        bulk_g2s(sx0 + (j & 1) * (uint32_t)x_tile_bytes, xg + (size_t)tile_of(j) * x_tile_bytes, (uint32_t)x_tile_bytes, b);
      };
      auto layer1 = [&](int j) {
        mbar_wait(bar_x + 8 * (j & 1), (j >> 1) & 1);
        tc_fence_after();
        const uint32_t sx = sx0 + (j & 1) * (uint32_t)x_tile_bytes;
        for (int k = 0; k < a.Kp / 16; ++k)
          mma_ss(tmem_base + kColD, make_desc(sx + k * 2 * lbo_x, lbo_x, 128), make_desc(sw1 + k * 2 * lbo_w, lbo_w, 128), idesc256, k > 0);
        tc_commit(bar_dready);
      };
      fetch_x(0);
      if (J > 1) fetch_x(1);
      mbar_wait(bar_w, 0);
      layer1(0);
      uint32_t a_uses[2] = {0, 0};             // completed hand-overs per A buffer (parity of the next wait)
      int n_out = 0;                           // layer-3 launches so far (parity of dout)
      for (int k = 0; k < nphases; ++k) {
        int j, layer;
        phase_of(k, j, layer);
        mbar_wait(bar_dfree, k & 1);           // phase k holds its accumulators in registers: D is free
        tc_fence_after();
        CFRB_TRACE3(1024 + k * 4 + 0);
        if (layer == 0 && j + 2 < J) fetch_x(j + 2);          // layer 1 of tile j has completed (the epilogue waited for it)
        if (k > 0) {
          int pj, pl;
          phase_of(k - 1, pj, pl);
          if (pl == 1) {                       // the previous phase finished tile pj's A3: layer 3 into D[0,16)
            const uint32_t acol = (pj & 1) ? kColA1 : kColA0;
            mbar_wait(bar_a + 8 * (pj & 1), a_uses[pj & 1] & 1); ++a_uses[pj & 1];
            tc_fence_after();
            for (int kk = 0; kk < kHid / 16; ++kk)
              mma_ts(tmem_base + kColD, tmem_base + acol + kk * 8, make_desc(sw3 + kk * 2 * lbo_w3, lbo_w3, 128), idesc16, kk != 0);
            tc_commit(bar_d3);
            mbar_wait(bar_dout, n_out & 1); ++n_out;           // ... and read back by the epilogue before D is reused
            tc_fence_after();
          }
        }
        CFRB_TRACE3(1024 + k * 4 + 1);
        if (k + 1 < nphases) {                 // accumulators of the next phase
          int nj, nl;
          phase_of(k + 1, nj, nl);
          if (nl == 0) {
            layer1(nj);
          } else {
            const uint32_t acol = (nj & 1) ? kColA1 : kColA0;
            mbar_wait(bar_a + 8 * (nj & 1), a_uses[nj & 1] & 1); ++a_uses[nj & 1];
            tc_fence_after();
            // D2 = ones * bias2^T + A2 * W2^T (A from TMEM: 16 fp16 = 8 columns per K step)
            mma_ss(tmem_base + kColD, make_desc(sones, lbo_x, 128), make_desc(sbias2, lbo_w, 128), idesc256, 0);
            for (int kk = 0; kk < kHid / 16; ++kk)
              mma_ts(tmem_base + kColD, tmem_base + acol + kk * 8, make_desc(sw2 + kk * 2 * lbo_w, lbo_w, 128), idesc256, 1);
            tc_commit(bar_dready);
          }
        }
        CFRB_TRACE3(1024 + k * 4 + 2);
      }
      {   // drain: layer 3 of the last tile (its A3 was finished by the last phase, D was emptied by that phase)
        const int pj = J - 1;
        const uint32_t acol = (pj & 1) ? kColA1 : kColA0;
        mbar_wait(bar_a + 8 * (pj & 1), a_uses[pj & 1] & 1);
        tc_fence_after();
        for (int kk = 0; kk < kHid / 16; ++kk)
          mma_ts(tmem_base + kColD, tmem_base + acol + kk * 8, make_desc(sw3 + kk * 2 * lbo_w3, lbo_w3, 128), idesc16, kk != 0);
        tc_commit(bar_d3);
      }
    }
  } else {
    // ===================== epilogue warps: thread == (row, column quarter) =====================
    const int quad = warp & 3, part_id = warp >> 2;
    const int row_in_tile = quad * 32 + lane;                      // 0..127 == TMEM lane
    const uint32_t tmem_row = tmem_base + ((uint32_t)(quad * 32) << 16);
    const float2* ln1 = reinterpret_cast<const float2*>(smem + L.off_ln1);
    const float2* ln2 = reinterpret_cast<const float2*>(smem + L.off_ln2);
    const float* b3 = reinterpret_cast<const float*>(smem + L.off_b3);
    float* part_base = reinterpret_cast<float*>(smem + T.off_part);
    mbar_wait(bar_w, 0);                                           // LayerNorm parameters / bias 3 are in shared memory
    int n_out = 0;
    auto read_out = [&](int j) {                                   // layer-3 accumulators of tile j -> out rows (+ bias 3)
      mbar_wait(bar_d3, n_out & 1); ++n_out;
      tc_fence_after();
      uint32_t v[16];
      CFRB_TMEM_LD16(tmem_row + kColD, v);
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_dout);
      const int row = tile_of(j) * kTileM + row_in_tile;
      if (row < rows) {                                            // rows are Hout floats apart, Hout a multiple of 4: 16-byte stores
        float4* o = reinterpret_cast<float4*>(a.out + (size_t)row * a.Hout);
#pragma unroll
        for (int h4 = 0; h4 < kNout / 4; ++h4)
          if (4 * h4 < a.Hout)
            o[h4] = make_float4(__uint_as_float(v[4 * h4]) + b3[4 * h4], __uint_as_float(v[4 * h4 + 1]) + b3[4 * h4 + 1],
                                __uint_as_float(v[4 * h4 + 2]) + b3[4 * h4 + 2], __uint_as_float(v[4 * h4 + 3]) + b3[4 * h4 + 3]);
      }
    };
    for (int k = 0; k < nphases; ++k) {
      int j, layer;
      phase_of(k, j, layer);
      const uint32_t acol = (j & 1) ? kColA1 : kColA0;
      const float2* ln = layer ? ln2 : ln1;
      float* part = part_base + (k & 1) * (kParts * kTileM);
      // ---- accumulators -> registers; D is free as soon as every warp has them
      mbar_wait(bar_dready, k & 1);
      tc_fence_after();
      if (tid == 0) CFRB_TRACE3(k * 8 + 0);
      uint32_t xr[kColsPerThread];
      float sumsq;
      {
        uint32_t* lo = xr; uint32_t* hi = xr + 32;
        CFRB_TMEM_LD32(tmem_row + kColD + part_id * kColsPerThread, lo);
        CFRB_TMEM_LD32(tmem_row + kColD + part_id * kColsPerThread + 32, hi);
        tmem_wait_ld();
        if (tid == 0) CFRB_TRACE3(k * 8 + 1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_dfree);
        if (kDebug && tile_of(j) == 0) {
          float* dbg = layer ? a.dbg_d2 : a.dbg_d1;
          if (dbg)
            for (int i = 0; i < kColsPerThread; ++i) dbg[row_in_tile * kHid + part_id * kColsPerThread + i] = __uint_as_float(xr[i]);
        }
        f32x2 q2[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q2[u] = pack2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < kColsPerThread; i += 2) {
          const f32x2 x2 = pack2(__uint_as_float(xr[i]), __uint_as_float(xr[i + 1]));
          q2[(i >> 1) & 3] = fma2(x2, x2, q2[(i >> 1) & 3]);
        }
        const f32x2 qt = add2(add2(q2[0], q2[1]), add2(q2[2], q2[3]));
        float b0, b1;
        unpack2(qt, b0, b1);
        sumsq = b0 + b1;
      }
      part[part_id * kTileM + row_in_tile] = sumsq;
      if (tid == 0) CFRB_TRACE3(k * 8 + 2);
      named_bar_sync(1 + quad, 128);                               // the four warps that share this row quadrant
      if (tid == 0) CFRB_TRACE3(k * 8 + 3);
      sumsq = (part[row_in_tile] + part[kTileM + row_in_tile]) + (part[2 * kTileM + row_in_tile] + part[3 * kTileM + row_in_tile]);
      // rows of W and the biases are centred over the features on the host: the mean of the 256 accumulators is zero
      const float rstd = rsqrtf(sumsq * (1.f / kHid) + 1e-5f);
      const f32x2 rstd2 = pack2(rstd, rstd);
      const bool out_here = k > 0 && part_id == 0 && ([&] { int pj, pl; phase_of(k - 1, pj, pl); return pl == 1; })();
#pragma unroll
      for (int c = 0; c < kSubChunks; ++c) {
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int jj = c * 16 + 2 * i;
          const float4 pp = *reinterpret_cast<const float4*>(ln + part_id * kColsPerThread + jj);   // {g_j, g_j+1, b_j, b_j+1} (x2: halved)
          float y0, y1;
          unpack2(fma2(mul2(pack2(__uint_as_float(xr[jj]), __uint_as_float(xr[jj + 1])), rstd2), pack2(pp.x, pp.y), pack2(pp.z, pp.w)), y0, y1);
          if (kGelu == 2) {
            pk[i] = gelu_hy_t32(y0, y1);
          } else {
            const __half2 h = __floats2half2_rn(gelu_tc(y0), gelu_tc(y1));
            pk[i] = *reinterpret_cast<const uint32_t*>(&h);
          }
        }
        CFRB_TMEM_ST8(tmem_row + acol + part_id * (kColsPerThread / 2) + c * 8, pk);
        if (c == 0 && out_here) {                                  // previous tile's layer 3 (16 K-steps of N = 16, ~1 800 cycles: the
                                                                   // A-operand fetch bounds a K-step, not N) has landed in D[0,16) by now
          int pj, pl;
          phase_of(k - 1, pj, pl);
          read_out(pj);
        }
        if (tid == 0 && (c == 0 || c == 3)) CFRB_TRACE3(k * 8 + (c == 0 ? 4 : 5));
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a + 8 * (j & 1));
      if (tid == 0) CFRB_TRACE3(k * 8 + 6);
    }
    if (part_id == 0) read_out(J - 1);                             // drain: the last tile
  }
  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

}  // namespace tc
}  // namespace cfrb
