// CFR wave kernels (sm_100a): regret matching, strategy averaging, reach / counterfactual-value traversal
// for thousands of concurrent Liar's Dice subgames.  Replaces, per iteration and per subgame, the CPU loops
// of the reference's CFR::step (subgame_solving.cc:577-664), update_regrets (:538-575),
// compute_reach_probabilities (:54-78), write_query_to (:104-123), query_value_net scaling (:253-269) and
// compute_expected_terminal_values / compute_win_probability (:80-98, :765-789).
//
// Execution model: one thread GROUP (a warp for depth-limited subgames, a whole CTA for full-depth trees) owns one
// subgame and walks the tree template level by level.  Every phase is a flat loop over (child node, hand) or
// (node, hand) items with the lanes strided over the items, so all global accesses of a phase are independent,
// unit-stride and coalesced: the per-(node,hand,action) tables live in HBM as compact [edge = child-1][hand] arrays
// (one subgame contiguous), reach / node values / per-edge temporaries in group-private shared memory.
// `real` is the arithmetic type of the tables: double reproduces the reference's fp64 state (default), float halves
// the table traffic.
//
// One launch = backward half of iteration i-1 (leaf values -> regrets, regret matching, discounting,
// average-strategy accumulation) fused with the forward half of iteration i (reach -> value-net query rows,
// scalers, terminal payoffs).  The value-net kernel runs between two launches.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "cfr_types.h"

namespace cfrb {

template <int G>
__device__ __forceinline__ void group_sync() {
  if (G == 32) __syncwarp(); else __syncthreads();
}
__device__ __forceinline__ float rmax0(float x) { return fmaxf(x, 0.f); }
__device__ __forceinline__ double rmax0(double x) { return fmax(x, 0.0); }
__device__ __forceinline__ float rpow(float a, float b) { return powf(a, b); }
__device__ __forceinline__ double rpow(double a, double b) { return pow(a, b); }

// The reference smooths with 1e-80 (kReachSmoothingEps / kRegretSmoothingEps, subgame_solving.h:34-36).  In fp64 these
// are applied literally, which keeps the fp64 path operation-for-operation identical to the reference (this TU is built
// with -fmad=false for the same reason).  1e-80 does not exist in fp32: there the limit behaviour is used instead
// ("no positive regret -> uniform", "all-zero reach -> uniform"), a documented deviation of CFRB_STATE_F32.
template <typename real> struct Eps;
template <> struct Eps<double> { static constexpr bool kLiteral = true;  static constexpr double v = 1e-80; };
template <> struct Eps<float>  { static constexpr bool kLiteral = false; static constexpr float v = 0.f; };

// Value of query column q of a pseudo-leaf row (write_query_to, subgame_solving.cc:104-123).  The reference's eps =
// 1e-80 only matters when a reach vector is all zero (-> uniform); that case is reproduced explicitly.
template <typename real>
__device__ __forceinline__ float query_value(const CfrDev<real>& p, int q, int leaf_player, int trav, int leaf_bid, const real* r0,
                                             const real* r1, real s0, real s1) {
  const int A = p.A, H = p.H;
  if (q == 0) return (float)leaf_player;
  if (q == 1) return (float)trav;
  if (q < 2 + A) return (q - 2 == leaf_bid) ? 1.f : 0.f;
  if (q < 2 + A + H) {
    if (Eps<real>::kLiteral) return (float)((r0[q - 2 - A] + Eps<real>::v) * s0);     // util.h:68-78 (s = 1 / sum)
    return isfinite(s0) ? (float)(r0[q - 2 - A] * s0) : 1.f / H;
  }
  if (q < 2 + A + 2 * H) {
    if (Eps<real>::kLiteral) return (float)((r1[q - 2 - A - H] + Eps<real>::v) * s1);
    return isfinite(s1) ? (float)(r1[q - 2 - A - H] * s1) : 1.f / H;
  }
  // padding: column Q is the constant 1 that multiplies the bias column of W1 in the tensor-core net (leaf_mlp_tc.cuh);
  // the fp32 SIMT net has a zero weight row there
  return q == 2 + A + 2 * H ? 1.f : 0.f;
}

// Correctly rounded x / b given y = RN(1 / b) (a true division): q0 = x y is within 2 ulp; the first residual step makes it
// faithful, the second one correctly rounded (Markstein) — the same bits as `/` at a tenth of the instructions of an fp64
// division; cross-checked against `/` on 4.3e9 operand pairs by tests/test_gpu_parity.py::test_fast_division_is_correctly_rounded.
// Operands here are regrets in [1e-80, ~1e3] and their sums over at most A actions.
__device__ __forceinline__ double div_by_rcp(double x, double b, double y) {
  double q = x * y;
  double r = fma(-q, b, x);
  q = fma(r, y, q);
  r = fma(-q, b, x);
  return fma(r, y, q);
}
__device__ __forceinline__ float div_by_rcp(float x, float b, float y) { (void)y; return x / b; }

// Forward half of iteration `iter`: reach, query rows + scalers for pseudo-leaves, payoffs for terminals.
template <typename real, int G, int HC>
__device__ void cfr_forward(const CfrDev<real>& p, int k, int trav, real* reach0, real* reach1, int have, real* lsum, real* hist, int lane) {
  const TemplateDev t = p.tmpl[p.sg_tmpl[k]];
  const int H = HC > 0 ? HC : p.H;      // compile-time hand count for the common shapes: item index -> (node, hand) without a division
  const int rp = p.sg_player[k];
  const real* __restrict__ Sg = p.Sg + (size_t)k * p.table_stride;
  const real* __restrict__ b = p.beliefs + (size_t)k * 2 * H;
  const int* __restrict__ parent = p.parent + t.node_off;
  // ---- top-down reach under Sg (compute_reach_probabilities, subgame_solving.cc:54-78).  `have` = player whose reach is
  // already in its buffer: the backward half that just ran left the traverser's reach under the new strategy there
  // (same products, same order), so only the other player's table is rebuilt; -1 = build both.
  for (int h = lane; h < H; h += G) {
    if (have != 0) reach0[h] = b[h];
    if (have != 1) reach1[h] = b[H + h];
  }
  group_sync<G>();
  for (int d = 1; d < t.levels; ++d) {
    const int nb = p.level_begin[t.level_off + d], ne = p.level_begin[t.level_off + d + 1];
    const int actor = rp ^ ((d - 1) & 1);              // who moved into level d
    if (have < 0) {
      for (int it = lane; it < (ne - nb) * H; it += G) {
        const int c = nb + it / H, h = it % H;
        const int par = parent[c];
        const real s = Sg[(c - 1) * H + h];
        const real a0 = reach0[par * H + h], a1 = reach1[par * H + h];
        reach0[c * H + h] = actor == 0 ? a0 * s : a0;
        reach1[c * H + h] = actor == 1 ? a1 * s : a1;
      }
    } else {
      real* ro = have == 0 ? reach1 : reach0;          // the table to rebuild belongs to player 1 - have
      const bool acts = actor != have;
      for (int it = lane; it < (ne - nb) * H; it += G) {
        const int c = nb + it / H, h = it % H;
        const real a = ro[parent[c] * H + h];
        ro[c * H + h] = acts ? a * Sg[(c - 1) * H + h] : a;
      }
    }
    group_sync<G>();
  }
  // ---- pseudo-leaves: normalisation sums + scaler (subgame_solving.cc:257-265)
  const int row0 = p.sg_row_off[k];
  for (int r = lane; r < t.L; r += G) {
    const int n = p.pleaf_node[t.pleaf_off + r];
    real s0 = 0, s1 = 0, e0 = 0, e1 = 0;
    for (int h = 0; h < H; ++h) {
      s0 += reach0[n * H + h]; s1 += reach1[n * H + h];                      // vector_sum (:264)
      e0 += reach0[n * H + h] + Eps<real>::v; e1 += reach1[n * H + h] + Eps<real>::v;   // normalize_probabilities_safe
    }
    // reciprocals: the query columns are float-rounded values of (x + eps) / sum; x * (1 / sum) is within one float ulp
    lsum[2 * r] = (real)1 / e0; lsum[2 * r + 1] = (real)1 / e1;
    p.scaler[row0 + r] = trav == 0 ? s1 : s0;
  }
  group_sync<G>();
  // ---- query rows.  All pseudo-leaves sit on the last level, so their acting player is rp ^ ((levels-1)&1).
  const int leaf_player = rp ^ ((t.levels - 1) & 1);
  const int Qp = p.Qpad;
  if (p.Xh != nullptr) {
    // fp16 tile in UMMA K-major core-matrix order (leaf_mlp_tc.cuh umma_kmajor_offset_halves, R = 128): one lane produces
    // the 8 contiguous halves of a (row, k-chunk) and stores them with a single 16-byte write; consecutive lanes ->
    // consecutive rows -> contiguous chunks
    const int kc = Qp >> 3;
    for (int it = lane; it < t.L * kc; it += G) {
      const int k8 = it / t.L, r = it % t.L;
      const int n = p.pleaf_node[t.pleaf_off + r];
      const int bid = p.last_bid[t.node_off + n];
      const real s0 = lsum[2 * r], s1 = lsum[2 * r + 1];
      union { int4 v; __half h[8]; } c;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        c.h[j] = __float2half_rn(query_value(p, k8 * 8 + j, leaf_player, trav, bid, reach0 + n * H, reach1 + n * H, s0, s1));
      const int Rr = row0 + r, rr = Rr & 127;
      *reinterpret_cast<int4*>(p.Xh + (size_t)(Rr >> 7) * 128 * Qp + k8 * 1024 + (rr >> 3) * 64 + (rr & 7) * 8) = c.v;
    }
  } else if (p.X != nullptr) {
    for (int it = lane; it < t.L * Qp; it += G) {
      const int r = it / Qp, q = it % Qp;
      const int n = p.pleaf_node[t.pleaf_off + r];
      p.X[(size_t)(row0 + r) * Qp + q] = query_value(p, q, leaf_player, trav, p.last_bid[t.node_off + n], reach0 + n * H,
                                                     reach1 + n * H, lsum[2 * r], lsum[2 * r + 1]);
    }
  }
  // ---- terminals (compute_expected_terminal_values, subgame_solving.cc:80-98; win probability :765-789)
  // term_node holds three lists of length T: node id, challenged bid (= parent's last_bid, :287), node depth.
  // Pass 1 (one lane per terminal): believed_counts[m] += reach (hand order), suffix sums from the top (:770-779) and the
  // belief sum — the reference's operation order, so the fp64 path is bit-identical.  Pass 2 (one lane per (terminal,
  // hand)) picks cum[max(0, quantity - matches(hand))], float-rounds it like :785 and forms the payoff.
  constexpr int kMaxBins = 9;            // 2 * num_dice + 1 <= 9
  real* __restrict__ vt = p.vterm + (size_t)k * p.vterm_stride;
  const real* ropp = trav == 0 ? reach1 : reach0;
  for (int z = lane; z < t.T; z += G) {
    const int n = p.term_node[t.term_off + z];
    const int face = p.term_node[t.term_off + t.T + z] % p.F;
    const real* ro = ropp + n * H;
    real cnt[kMaxBins];
#pragma unroll
    for (int m = 0; m < kMaxBins; ++m) cnt[m] = 0;
    real tot = 0;
    for (int g = 0; g < H; ++g) {
      const real r = ro[g];
      const int mg = (int)p.matches[g * p.F + face];
      tot += r;
#pragma unroll
      for (int m = 0; m < kMaxBins; ++m) cnt[m] += (m == mg) ? r : (real)0;
    }
#pragma unroll
    for (int m = kMaxBins - 2; m >= 0; --m) cnt[m] += cnt[m + 1];
#pragma unroll
    for (int m = 0; m < kMaxBins; ++m) hist[z * (kMaxBins + 1) + m] = cnt[m];
    hist[z * (kMaxBins + 1) + kMaxBins] = tot;
  }
  group_sync<G>();
  for (int it = lane; it < t.T * H; it += G) {
    const int z = it / H, h = it % H;
    const int pbid = p.term_node[t.term_off + t.T + z];
    const int ndepth = p.term_node[t.term_off + 2 * t.T + z];
    const int quantity = 1 + pbid / p.F, face = pbid % p.F;   // unpack_action, liars_dice.h:74-80
    int left = quantity - (int)p.matches[h * p.F + face];
    left = left < 0 ? 0 : (left > kMaxBins - 1 ? kMaxBins - 1 : left);
    const real win = hist[z * (kMaxBins + 1) + left], tot = hist[z * (kMaxBins + 1) + kMaxBins];
    const real v = (real)(float)win * 2 - tot;
    // state.player_id of a terminal = the bidder; payoff is negated iff that is not the traverser (:290)
    const int pl = rp ^ (ndepth & 1);
    vt[z * H + h] = (pl != trav) ? -v : v;
  }
}

// Backward half of iteration with traverser `trav` (update_regrets :538-575 and step :577-664).
template <typename real, int G, int HC>
__device__ void cfr_backward(const CfrDev<real>& p, int k, int trav, real* val, real* rt, int lane) {
  // Scratch discipline (all indexed [node * H + hand]): `val` holds node values; once a traverser level is processed its
  // children's slots are dead and take the new regrets R(parent, hand, action->child); later the slots of the traverser
  // nodes themselves take the positive-regret sums.  `rt` is free during the bottom-up sweep and carries the value*sigma
  // products there; in the top-down sweep it becomes the traverser's reach under the new strategy.
  const TemplateDev t = p.tmpl[p.sg_tmpl[k]];
  const int H = HC > 0 ? HC : p.H;
  const int rp = p.sg_player[k];
  real* __restrict__ R = p.R + (size_t)k * p.table_stride;
  real* __restrict__ Sg = p.Sg + (size_t)k * p.table_stride;
  real* __restrict__ S = p.S + (size_t)k * p.table_stride;
  const int* __restrict__ parent = p.parent + t.node_off;
  const int* __restrict__ nchild = p.nchild + t.node_off;
  const int* __restrict__ child_begin = p.child_begin + t.node_off;
  const int row0 = p.sg_row_off[k];
  // leaf values = (float)(net(query) * scaler) (subgame_solving.cc:266-282); terminals from the forward half
  for (int it = lane; it < t.L * H; it += G) {
    const int r = it / H, h = it % H;
    const int n = p.pleaf_node[t.pleaf_off + r];
    val[n * H + h] = p.use_net ? (real)(float)((real)p.net_out[(size_t)(row0 + r) * p.Hout + h] * p.scaler[row0 + r]) : (real)0;
  }
  const real* __restrict__ vt = p.vterm + (size_t)k * p.vterm_stride;
  for (int it = lane; it < t.T * H; it += G) {
    const int z = it / H, h = it % H;
    val[p.term_node[t.term_off + z] * H + h] = vt[z * H + h];
  }
  group_sync<G>();
  // ---- bottom-up (reverse BFS order == decreasing level)
  for (int d = t.levels - 2; d >= 0; --d) {
    const int nb = p.level_begin[t.level_off + d], ne = p.level_begin[t.level_off + d + 1];
    const int cb = ne, ce = p.level_begin[t.level_off + d + 2];
    const bool mine = (rp ^ (d & 1)) == trav;
    if (mine) {   // per-edge products value * sigma
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        rt[c * H + h] = val[c * H + h] * Sg[(c - 1) * H + h];
      }
      group_sync<G>();
    }
    for (int it = lane; it < (ne - nb) * H; it += G) {
      const int n = nb + it / H, h = it % H;
      const int nc = nchild[n];
      if (!nc) continue;
      const int c0 = child_begin[n];
      real v = 0;
      if (mine) { for (int j = 0; j < nc; ++j) v += rt[(c0 + j) * H + h]; }
      else      { for (int j = 0; j < nc; ++j) v += val[(c0 + j) * H + h]; }
      val[n * H + h] = v;
    }
    group_sync<G>();
    if (mine) {   // regrets += action value - node value (kept in the child's slot; written back once, discounted, below)
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        val[c * H + h] = (R[(c - 1) * H + h] + val[c * H + h]) - val[parent[c] * H + h];
      }
      group_sync<G>();
    }
  }
  // ---- root value running mean (:579-590) and discounts (:592-617)
  const int s = p.steps[2 * k + trav];
  {
    const real alpha = p.linear ? (real)2 / (s + 2) : (real)1 / (s + 1);
    real* mu = p.mu + ((size_t)k * 2 + trav) * H;
    for (int h = lane; h < H; h += G) mu[h] += (val[h] - mu[h]) * alpha;
  }
  real pos = 1, neg = 1, strat = 1;
  {
    const real ns = (real)(s + 1);
    if (p.linear) {
      pos = neg = strat = ns / (ns + 1);
    } else if (p.dcfr) {
      pos = p.dcfr_alpha >= 5 ? (real)1 : rpow(ns, p.dcfr_alpha) / (rpow(ns, p.dcfr_alpha) + 1);
      neg = p.dcfr_beta <= -5 ? (real)0 : rpow(ns, p.dcfr_beta) / (rpow(ns, p.dcfr_beta) + 1);
      strat = rpow(ns / (ns + 1), p.dcfr_gamma);
    }
  }
  // ---- top-down: regret matching (:619-634), traverser reach under the new strategy (:636-638), regret
  // discount and sum-strategy update (:639-661).  val[] is reused for the per-(node,hand) positive-regret sums.
  const real* __restrict__ b = p.beliefs + ((size_t)k * 2 + trav) * H;
  group_sync<G>();
  for (int h = lane; h < H; h += G) rt[h] = b[h];
  group_sync<G>();
  for (int d = 0; d + 1 < t.levels; ++d) {
    const int nb = p.level_begin[t.level_off + d], ne = p.level_begin[t.level_off + d + 1];
    const int cb = ne, ce = p.level_begin[t.level_off + d + 2];
    const bool mine = (rp ^ (d & 1)) == trav;
    if (mine) {
      for (int it = lane; it < (ne - nb) * H; it += G) {
        const int n = nb + it / H, h = it % H;
        const int nc = nchild[n];
        if (!nc) continue;
        const int c0 = child_begin[n];
        real sum = 0;
        for (int j = 0; j < nc; ++j) {
          const real r = val[(c0 + j) * H + h];
          sum += Eps<real>::kLiteral ? (r > Eps<real>::v ? r : Eps<real>::v) : rmax0(r);   // max(R, 1e-80) (:626-629)
        }
        val[n * H + h] = sum;
      }
      group_sync<G>();
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        const int e = (c - 1) * H + h, par = parent[c];
        const real r = val[c * H + h], sum = val[par * H + h], rn = rt[par * H + h];
        const real sg = Eps<real>::kLiteral ? (r > Eps<real>::v ? r : Eps<real>::v) / sum
                                            : (sum > 0 ? rmax0(r) / sum : (real)1 / nchild[par]);
        Sg[e] = sg;
        R[e] = r * (r > 0 ? pos : neg);
        S[e] = S[e] * strat + rn * sg;
        rt[c * H + h] = rn * sg;
      }
    } else {
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        rt[c * H + h] = rt[parent[c] * H + h];
      }
    }
    group_sync<G>();
  }
  if (lane == 0) p.steps[2 * k + trav] = s + 1;
}

// Backward half of a FICTITIOUS-PLAY iteration with traverser `trav` (FP::step, subgame_solving.cc:423-460): best response
// against the average strategy (BRSolver::compute_br :316-358), root value running mean, update_sum_strat (:391-421), linear
// discount and re-normalisation of the average strategy.  Table roles in FP mode: Sg = average_strategies (the strategy
// the reach / queries / sampling use), S = sum_strategies, R = last_strategies (belief x best response).
template <typename real, int G, int HC>
__device__ void fp_backward(const CfrDev<real>& p, int k, int trav, real* val, real* rt, int lane) {
  const TemplateDev t = p.tmpl[p.sg_tmpl[k]];
  const int H = HC > 0 ? HC : p.H;
  const int rp = p.sg_player[k];
  real* __restrict__ Last = p.R + (size_t)k * p.table_stride;
  real* __restrict__ Avg = p.Sg + (size_t)k * p.table_stride;
  real* __restrict__ S = p.S + (size_t)k * p.table_stride;
  const int* __restrict__ parent = p.parent + t.node_off;
  const int* __restrict__ nchild = p.nchild + t.node_off;
  const int* __restrict__ child_begin = p.child_begin + t.node_off;
  const int row0 = p.sg_row_off[k];
  for (int it = lane; it < t.L * H; it += G) {
    const int r = it / H, h = it % H;
    const int n = p.pleaf_node[t.pleaf_off + r];
    val[n * H + h] = p.use_net ? (real)(float)((real)p.net_out[(size_t)(row0 + r) * p.Hout + h] * p.scaler[row0 + r]) : (real)0;
  }
  const real* __restrict__ vt = p.vterm + (size_t)k * p.vterm_stride;
  for (int it = lane; it < t.T * H; it += G) {
    const int z = it / H, h = it % H;
    val[p.term_node[t.term_off + z] * H + h] = vt[z * H + h];
  }
  group_sync<G>();
  // ---- bottom-up best response: max over the children at the traverser's nodes (first child wins ties, :336-337; the
  // one-hot br_strategies go to rt as 0/1 flags in the children's slots), plain sums at the opponent's
  for (int d = t.levels - 2; d >= 0; --d) {
    const int nb = p.level_begin[t.level_off + d], ne = p.level_begin[t.level_off + d + 1];
    const bool mine = (rp ^ (d & 1)) == trav;
    for (int it = lane; it < (ne - nb) * H; it += G) {
      const int n = nb + it / H, h = it % H;
      const int nc = nchild[n];
      if (!nc) continue;
      const int c0 = child_begin[n];
      real v = 0;
      if (mine) {
        int best = 0;
        v = val[c0 * H + h];
        for (int j = 1; j < nc; ++j) {
          const real nv = val[(c0 + j) * H + h];
          if (nv > v) { v = nv; best = j; }
        }
        for (int j = 0; j < nc; ++j) rt[(c0 + j) * H + h] = (j == best) ? (real)1 : (real)0;
      } else {
        for (int j = 0; j < nc; ++j) v += val[(c0 + j) * H + h];
      }
      val[n * H + h] = v;
    }
    group_sync<G>();
  }
  // ---- root value running mean (:428-440): num_update = num_strategies / 2 + 1 = steps[trav] + 1 for alternating traversers
  const int s = p.steps[2 * k + trav];
  {
    const real alpha = p.linear ? (real)2 / (s + 2) : (real)1 / (s + 1);
    real* mu = p.mu + ((size_t)k * 2 + trav) * H;
    for (int h = lane; h < H; h += G) mu[h] += (val[h] - mu[h]) * alpha;
  }
  const real disc = (real)(s + 2) / (s + 3);        // (num_update + 1) / (num_update + 2), :447-449
  group_sync<G>();
  // ---- top-down update_sum_strat: val now carries the traverser's beliefs (belief x best response along the path)
  const real* __restrict__ b = p.beliefs + ((size_t)k * 2 + trav) * H;
  for (int h = lane; h < H; h += G) val[h] = b[h];
  group_sync<G>();
  for (int d = 0; d + 1 < t.levels; ++d) {
    const int nb = p.level_begin[t.level_off + d], ne = p.level_begin[t.level_off + d + 1];
    const int cb = ne, ce = p.level_begin[t.level_off + d + 2];
    const bool mine = (rp ^ (d & 1)) == trav;
    if (mine) {
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        const int e = (c - 1) * H + h;
        const real x = val[parent[c] * H + h] * rt[c * H + h];     // traverser_beliefs * br_strategies
        real sn = S[e] + x;
        if (p.linear) sn = sn * disc;
        S[e] = sn; Last[e] = x;
        val[c * H + h] = x;                                        // beliefs of the child
        rt[c * H + h] = sn;
      }
      group_sync<G>();
      for (int it = lane; it < (ne - nb) * H; it += G) {           // normalize_probabilities (util.h:20-34 / 52-63)
        const int n = nb + it / H, h = it % H;
        const int nc = nchild[n];
        if (!nc) continue;
        const int c0 = child_begin[n];
        real tot = 0;
        for (int j = 0; j < nc; ++j) tot += rt[(c0 + j) * H + h];
        if (p.optimistic) {
          real tl = 0;
          for (int j = 0; j < nc; ++j) tl += val[(c0 + j) * H + h];
          tot = tot + tl;
        }
        val[n * H + h] = tot;
      }
      group_sync<G>();
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        const real tot = val[parent[c] * H + h];
        Avg[(c - 1) * H + h] = (p.optimistic ? rt[c * H + h] + val[c * H + h] : rt[c * H + h]) / tot;
      }
    } else {
      for (int it = lane; it < (ce - cb) * H; it += G) {
        const int c = cb + it / H, h = it % H;
        val[c * H + h] = val[parent[c] * H + h];
      }
    }
    group_sync<G>();
  }
  if (lane == 0) p.steps[2 * k + trav] = s + 1;
}

// iter: global iteration index of the forward half.  do_b: run backward half of iteration iter-1 first.
template <typename real, int G, int HC>
__global__ void __launch_bounds__(512) cfr_iter_kernel(CfrDev<real> p, int iter, int do_b, int do_f, int scratch_per_group) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  real* smem = reinterpret_cast<real*>(smem_raw);
  const int groups_per_cta = blockDim.x / G;
  const int gid = threadIdx.x / G, lane = threadIdx.x % G;
  const int k = blockIdx.x * groups_per_cta + gid;
  if (k >= *p.wave_n) return;   // uniform per group (and per CTA when G == blockDim.x)
  const TemplateDev t = p.tmpl[p.sg_tmpl[k]];
  real* base = (G == 32) ? smem + (size_t)gid * scratch_per_group : p.scratch + (size_t)k * p.scratch_stride;
  real* bufA = base; real* bufB = base + p.nh_max; real* tmp = base + 2 * p.nh_max; real* lsum = tmp + p.tmp_reals;
  const int tb = (iter - 1) & 1;
  if (do_b) {
    if (p.fp) fp_backward<real, G, HC>(p, k, tb, bufA, bufB, lane);
    else cfr_backward<real, G, HC>(p, k, tb, bufA, bufB, lane);   // leaves the reach of player tb (new strategy) in bufB
    group_sync<G>();
  }
  // sampling-strategy snapshot for RlRunner (recursive_solving.cc:168-174): state after `iter` iterations
  if (p.sg_act_iter[k] == iter) {
    const real* __restrict__ Sg = p.Sg + (size_t)k * p.table_stride;
    real* __restrict__ Sn = p.Snap + (size_t)k * p.table_stride;
    for (int i = lane; i < (t.N - 1) * p.H; i += G) Sn[i] = Sg[i];
  }
  if (do_f) {
    if (do_b && !p.fp) cfr_forward<real, G, HC>(p, k, iter & 1, tb == 0 ? bufB : bufA, tb == 0 ? bufA : bufB, tb, lsum, tmp, lane);
    else      cfr_forward<real, G, HC>(p, k, iter & 1, bufA, bufB, -1, lsum, tmp, lane);
  }
}

// ======================================================================================================================
// Depth <= 2 specialisation (templates with at most three levels: root, level 1, level 2 — every subgame of a max_depth <= 2
// solver, i.e. the self-play configuration).  Each player acts on exactly one level there (the root player P0 = rp at the
// root, P1 at level 1), which removes most of the generic kernel's scratch:
//   * the traverser's reach at the nodes where it acts is just its root belief;
//   * reach_P0 is constant below level 1 and reach_P1 is the root belief down to level 1, so ONE [N*H] buffer holds
//     everything the forward half needs: slot[n] = reach_P0[n] for level-1 nodes, slot[c] = reach_P1[c] for level-2 nodes;
//   * the backward half uses the same buffer for node values / new regrets and leaves the traverser's new reach
//     (belief * new strategy) in the slots of the level where it acts, exactly the products the forward half would form.
// Scratch per subgame: slot[N*H] | bel[2*H] | hist[10*T] | lsum[2*L] — half of the generic layout, so twice as many
// subgames are resident per SM.  All arithmetic is the generic kernel's, operation for operation (bit-identical results).
struct D2Levels {
  int n1b, n1e, n2e;   // level 1 = [n1b, n1e), level 2 = [n1e, n2e) (empty when the template has two levels)
};
// One tree template, packed into bytes (every depth-2 template has at most 255 nodes) so that a warp copies the whole thing into
// shared memory with a single coalesced round trip at kernel entry; every parent / child / leaf-list lookup of the phases is
// then a shared-memory byte load instead of a dependent global load (the "shared-memory staging of the tree's child-index
// arrays").  Layout (cfrb_api.cu builds it): 16-byte header {N, L, T, levels, n1e, n2e, -, -, qconst_off:int32, -}, then
// parent[N] child_begin[N] nchild[N] last_bid+1[N] pleaf[L] term[3][T] matches[H*F].
struct D2Tmpl {
  int N, L, T, levels, qconst_off;
  const unsigned char *parent, *child_begin, *nchild, *bid1, *pleaf, *term, *matches;
};
__device__ __forceinline__ D2Tmpl d2_tmpl_view(const unsigned char* b, int HF) {
  D2Tmpl t;
  t.N = b[0]; t.L = b[1]; t.T = b[2]; t.levels = b[3];
  t.qconst_off = *reinterpret_cast<const int*>(b + 8);
  t.parent = b + 16; t.child_begin = t.parent + t.N; t.nchild = t.child_begin + t.N; t.bid1 = t.nchild + t.N;
  t.pleaf = t.bid1 + t.N; t.term = t.pleaf + t.L; t.matches = t.term + 3 * t.T;
  (void)HF;
  return t;
}
__device__ __forceinline__ D2Levels d2_levels(const unsigned char* b) {
  D2Levels L;
  L.n1b = 1; L.n1e = b[4]; L.n2e = b[5];
  return L;
}
// Row [H] of reach probabilities of `player` at node n (level 1 or 2) in the d2 scratch.
template <typename real, typename PT>
__device__ __forceinline__ const real* d2_reach_row(const real* slot, const real* bel, const PT* parent, int n, int n1e,
                                                    int player, int rp, int H) {
  if (n < n1e) return player == rp ? slot + n * H : bel + player * H;           // level 1
  return player == rp ? slot + parent[n] * H : slot + n * H;                    // level 2
}

template <typename real, int HC>
__device__ void cfr_backward_d2(const CfrDev<real>& p, const D2Tmpl& t, const D2Levels& lv, int k, int trav, real* val, const real* bel, real* rcp, int lane) {
  constexpr int G = 32;
  const int H = HC > 0 ? HC : p.H;
  const int rp = p.sg_player[k];
  real* R = p.R + (size_t)k * p.table_stride;
  real* Sg = p.Sg + (size_t)k * p.table_stride;
  real* S = p.S + (size_t)k * p.table_stride;
  const unsigned char* parent = t.parent; const unsigned char* nchild = t.nchild; const unsigned char* child_begin = t.child_begin;
  const int row0 = p.sg_row_off[k];
  const bool mine0 = rp == trav;          // traverser acts at the root (else at level 1)
  // leaf values = (float)(net(query) * scaler) (subgame_solving.cc:266-282); terminals from the forward half
  // Table / value-net reads go through the read-only path (ld.global.nc): none of these locations is read again after this
  // launch writes it, and without possible aliasing against the stores the unrolled loops keep several loads in flight per lane
  // instead of one dependent L2 / HBM round trip per iteration (the ncu profile of round 1: 7 warps per issue on long_scoreboard).
#pragma unroll 4
  for (int it = lane; it < t.L * H; it += G) {
    const int r = it / H, h = it % H;
    const int n = t.pleaf[r];
    val[n * H + h] = p.use_net ? (real)(float)((real)__ldg(p.net_out + (size_t)(row0 + r) * p.Hout + h) * __ldg(p.scaler + row0 + r)) : (real)0;
  }
  const real* __restrict__ vt = p.vterm + (size_t)k * p.vterm_stride;
#pragma unroll 4
  for (int it = lane; it < t.T * H; it += G) {
    const int z = it / H, h = it % H;
    val[t.term[z] * H + h] = __ldg(vt + z * H + h);
  }
  __syncwarp();
  // ---- bottom-up (update_regrets :538-575): level-1 node values, then the root
  if (lv.n2e > lv.n1e) {
    for (int it = lane; it < (lv.n1e - lv.n1b) * H; it += G) {
      const int n = lv.n1b + it / H, h = it % H;
      const int nc = nchild[n];
      if (!nc) continue;
      const int c0 = child_begin[n];
      real v = 0;
      if (!mine0) { for (int j = 0; j < nc; ++j) v += val[(c0 + j) * H + h] * __ldg(Sg + (c0 + j - 1) * H + h); }
      else        { for (int j = 0; j < nc; ++j) v += val[(c0 + j) * H + h]; }
      val[n * H + h] = v;
    }
    __syncwarp();
    if (!mine0) {   // new regrets of the level-1 actions, kept in the child's slot
#pragma unroll 4
      for (int it = lane; it < (lv.n2e - lv.n1e) * H; it += G) {
        const int c = lv.n1e + it / H, h = it % H;
        val[c * H + h] = (__ldg(R + (c - 1) * H + h) + val[c * H + h]) - val[parent[c] * H + h];
      }
    }
  }
  for (int h = lane; h < H; h += G) {
    real v = 0;
    if (mine0) { for (int n = lv.n1b; n < lv.n1e; ++n) v += val[n * H + h] * __ldg(Sg + (n - 1) * H + h); }
    else       { for (int n = lv.n1b; n < lv.n1e; ++n) v += val[n * H + h]; }
    val[h] = v;
  }
  __syncwarp();
  if (mine0) {
    for (int it = lane; it < (lv.n1e - lv.n1b) * H; it += G) {
      const int n = lv.n1b + it / H, h = it % H;
      val[n * H + h] = (__ldg(R + (n - 1) * H + h) + val[n * H + h]) - val[h];
    }
  }
  // ---- root value running mean (:579-590) and discounts (:592-617)
  const int s = p.steps[2 * k + trav];
  {
    const real alpha = p.linear ? (real)2 / (s + 2) : (real)1 / (s + 1);
    real* mu = p.mu + ((size_t)k * 2 + trav) * H;
    for (int h = lane; h < H; h += G) mu[h] += (val[h] - mu[h]) * alpha;
  }
  real pos = 1, neg = 1, strat = 1;
  {
    const real ns = (real)(s + 1);
    if (p.linear) {
      pos = neg = strat = ns / (ns + 1);
    } else if (p.dcfr) {
      pos = p.dcfr_alpha >= 5 ? (real)1 : rpow(ns, p.dcfr_alpha) / (rpow(ns, p.dcfr_alpha) + 1);
      neg = p.dcfr_beta <= -5 ? (real)0 : rpow(ns, p.dcfr_beta) / (rpow(ns, p.dcfr_beta) + 1);
      strat = rpow(ns / (ns + 1), p.dcfr_gamma);
    }
  }
  __syncwarp();
  // ---- regret matching (:619-634), regret discount and sum-strategy update (:639-661) on the traverser's level.  The
  // traverser has not acted above that level, so its reach there is its root belief; the child's slot receives
  // belief * new strategy = the traverser's reach under the new strategy (:636-638), which the forward half reuses.
  const real* bt = bel + trav * H;
  const int pb = mine0 ? 0 : lv.n1b, pe = mine0 ? 1 : lv.n1e;            // acting nodes
  const int cb = mine0 ? lv.n1b : lv.n1e, ce = mine0 ? lv.n1e : lv.n2e;  // their children
  for (int it = lane; it < (pe - pb) * H; it += G) {
    const int n = pb + it / H, h = it % H;
    const int nc = nchild[n];
    if (!nc) continue;
    const int c0 = child_begin[n];
    real sum = 0;
    for (int j = 0; j < nc; ++j) {
      const real r = val[(c0 + j) * H + h];
      sum += Eps<real>::kLiteral ? (r > Eps<real>::v ? r : Eps<real>::v) : rmax0(r);   // max(R, 1e-80) (:626-629)
    }
    val[n * H + h] = sum;
    rcp[n * H + h] = (real)1 / sum;      // one true division per (node, hand); the per-action quotients below are derived from it
  }
  __syncwarp();
#pragma unroll 4
  for (int it = lane; it < (ce - cb) * H; it += G) {
    const int c = cb + it / H, h = it % H;
    const int e = (c - 1) * H + h, par = parent[c];
    const real s_old = __ldg(S + e);
    const real r = val[c * H + h], sum = val[par * H + h], rn = bt[h];
    const real sg = Eps<real>::kLiteral ? div_by_rcp(r > Eps<real>::v ? r : Eps<real>::v, sum, rcp[par * H + h])
                                        : (sum > 0 ? rmax0(r) / sum : (real)1 / nchild[par]);
    Sg[e] = sg;
    R[e] = r * (r > 0 ? pos : neg);
    S[e] = s_old * strat + rn * sg;
    val[c * H + h] = rn * sg;
  }
  if (lane == 0) p.steps[2 * k + trav] = s + 1;
  __syncwarp();
}

// Fictitious-play backward half for depth <= 2 templates: fp_backward's arithmetic with the one-buffer discipline of
// cfr_backward_d2.  The best-response flags (1 / 0) replace the children's values in place, then give way to the discounted
// sums, and finally to belief x new average strategy = the reach the forward half needs (same `have` protocol as CFR).
template <typename real, int HC>
__device__ void fp_backward_d2(const CfrDev<real>& p, const D2Tmpl& t, const D2Levels& lv, int k, int trav, real* val, const real* bel, int lane) {
  constexpr int G = 32;
  const int H = HC > 0 ? HC : p.H;
  const int rp = p.sg_player[k];
  real* Last = p.R + (size_t)k * p.table_stride;
  real* Avg = p.Sg + (size_t)k * p.table_stride;
  real* S = p.S + (size_t)k * p.table_stride;
  const unsigned char* parent = t.parent; const unsigned char* nchild = t.nchild; const unsigned char* child_begin = t.child_begin;
  const int row0 = p.sg_row_off[k];
  const bool mine0 = rp == trav;
  for (int it = lane; it < t.L * H; it += G) {
    const int r = it / H, h = it % H;
    const int n = t.pleaf[r];
    val[n * H + h] = p.use_net ? (real)(float)((real)p.net_out[(size_t)(row0 + r) * p.Hout + h] * p.scaler[row0 + r]) : (real)0;
  }
  const real* __restrict__ vt = p.vterm + (size_t)k * p.vterm_stride;
  for (int it = lane; it < t.T * H; it += G) {
    const int z = it / H, h = it % H;
    val[t.term[z] * H + h] = vt[z * H + h];
  }
  __syncwarp();
  // ---- bottom-up best response (BRSolver::compute_br :316-358): level 1, then the root
  if (lv.n2e > lv.n1e) {
    for (int it = lane; it < (lv.n1e - lv.n1b) * H; it += G) {
      const int n = lv.n1b + it / H, h = it % H;
      const int nc = nchild[n];
      if (!nc) continue;
      const int c0 = child_begin[n];
      real v = 0;
      if (!mine0) {
        int best = 0;
        v = val[c0 * H + h];
        for (int j = 1; j < nc; ++j) {
          const real nv = val[(c0 + j) * H + h];
          if (nv > v) { v = nv; best = j; }
        }
        for (int j = 0; j < nc; ++j) val[(c0 + j) * H + h] = (j == best) ? (real)1 : (real)0;
      } else {
        for (int j = 0; j < nc; ++j) v += val[(c0 + j) * H + h];
      }
      val[n * H + h] = v;
    }
    __syncwarp();
  }
  for (int h = lane; h < H; h += G) {
    real v = 0;
    if (mine0) {
      int best = lv.n1b;
      v = val[lv.n1b * H + h];
      for (int n = lv.n1b + 1; n < lv.n1e; ++n) {
        const real nv = val[n * H + h];
        if (nv > v) { v = nv; best = n; }
      }
      for (int n = lv.n1b; n < lv.n1e; ++n) val[n * H + h] = (n == best) ? (real)1 : (real)0;
    } else {
      for (int n = lv.n1b; n < lv.n1e; ++n) v += val[n * H + h];
    }
    val[h] = v;
  }
  __syncwarp();
  const int s = p.steps[2 * k + trav];
  {
    const real alpha = p.linear ? (real)2 / (s + 2) : (real)1 / (s + 1);
    real* mu = p.mu + ((size_t)k * 2 + trav) * H;
    for (int h = lane; h < H; h += G) mu[h] += (val[h] - mu[h]) * alpha;
  }
  const real disc = (real)(s + 2) / (s + 3);
  __syncwarp();
  // ---- update_sum_strat (:391-421) on the traverser's level: its beliefs there are its root beliefs
  const real* bt = bel + trav * H;
  const int pb = mine0 ? 0 : lv.n1b, pe = mine0 ? 1 : lv.n1e;
  const int cb = mine0 ? lv.n1b : lv.n1e, ce = mine0 ? lv.n1e : lv.n2e;
  for (int it = lane; it < (ce - cb) * H; it += G) {
    const int c = cb + it / H, h = it % H;
    const int e = (c - 1) * H + h;
    const real x = bt[h] * val[c * H + h];               // traverser_beliefs * br_strategies
    real sn = S[e] + x;
    if (p.linear) sn = sn * disc;
    S[e] = sn; Last[e] = x;
    val[c * H + h] = sn;
  }
  __syncwarp();
  for (int it = lane; it < (pe - pb) * H; it += G) {     // normalize_probabilities (util.h:20-34 / 52-63)
    const int n = pb + it / H, h = it % H;
    const int nc = nchild[n];
    if (!nc) continue;
    const int c0 = child_begin[n];
    real tot = 0;
    for (int j = 0; j < nc; ++j) tot += val[(c0 + j) * H + h];
    if (p.optimistic) {
      real tl = 0;
      for (int j = 0; j < nc; ++j) tl += Last[(c0 + j - 1) * H + h];
      tot = tot + tl;
    }
    val[n * H + h] = tot;
  }
  __syncwarp();
  for (int it = lane; it < (ce - cb) * H; it += G) {
    const int c = cb + it / H, h = it % H;
    const int e = (c - 1) * H + h;
    const real tot = val[parent[c] * H + h];
    const real avg = (p.optimistic ? val[c * H + h] + Last[e] : val[c * H + h]) / tot;
    Avg[e] = avg;
    val[c * H + h] = bt[h] * avg;                        // the traverser's reach under the new average strategy
  }
  if (lane == 0) p.steps[2 * k + trav] = s + 1;
  __syncwarp();
}

// have: level whose slots already hold the reach of the player acting above it (0: level-1 slots = reach_P0 valid,
// 1: level-2 slots = reach_P1 valid, -1: neither).
template <typename real, int HC>
__device__ void cfr_forward_d2(const CfrDev<real>& p, const D2Tmpl& t, const D2Levels& lv, int k, int trav, real* slot, const real* bel, int have,
                               real* aux, real* hist, int lane) {
  constexpr int G = 32;
  const int H = HC > 0 ? HC : p.H;
  const int rp = p.sg_player[k];
  const real* Sg = p.Sg + (size_t)k * p.table_stride;     // not __restrict__/const-cached: written earlier in this launch
  const unsigned char* parent = t.parent;
  // ---- reach under Sg (compute_reach_probabilities, subgame_solving.cc:54-78): belief * strategy of the acting level
  if (have != 0) {
    const real* b0 = bel + rp * H;
#pragma unroll 4
    for (int it = lane; it < (lv.n1e - lv.n1b) * H; it += G) {
      const int n = lv.n1b + it / H, h = it % H;
      slot[n * H + h] = b0[h] * __ldg(Sg + (n - 1) * H + h);      // a level this launch did not write (see `have`)
    }
  }
  if (have != 1) {
    const real* b1 = bel + (1 - rp) * H;
#pragma unroll 4
    for (int it = lane; it < (lv.n2e - lv.n1e) * H; it += G) {
      const int c = lv.n1e + it / H, h = it % H;
      slot[c * H + h] = b1[h] * __ldg(Sg + (c - 1) * H + h);
    }
  }
  __syncwarp();
  // ---- pseudo-leaves (subgame_solving.cc:257-265, write_query_to :104-123).  All pseudo-leaves of a depth-2 tree sit on level 2:
  // the root player's reach there is its parent's level-1 slot — the same row for every leaf under one level-1 node — so it is
  // summed / normalised once per level-1 node; the other player's reach is the leaf's own slot.  The normalised beliefs are kept
  // as fp16 (the precision of the query tiles) and the 16-byte chunks are assembled from them.
  const int row0 = p.sg_row_off[k];
  const int n1 = lv.n1e - lv.n1b;
  real* par_sum = aux;
  real* par_inv = aux + p.n1max;
  __half* qpar = reinterpret_cast<__half*>(reinterpret_cast<unsigned char*>(aux) + ((2 * p.n1max * (int)sizeof(real) + 15) & ~15));
  __half* qown = qpar + p.n1max * H;
  const int opp = 1 - trav;
  const bool have_l2 = lv.n2e > lv.n1e;
  if (have_l2) {
    for (int i = lane; i < n1; i += G) {
      const real* r = slot + (1 + i) * H;
      real s0 = 0, e0 = 0;
      for (int h = 0; h < H; ++h) { s0 += r[h]; e0 += r[h] + Eps<real>::v; }                  // vector_sum (:264) / normalize_probabilities_safe
      const real inv = (real)1 / e0;
      par_sum[i] = s0; par_inv[i] = inv;
      for (int h = 0; h < H; ++h) {
        float f;
        if (Eps<real>::kLiteral) f = (float)((r[h] + Eps<real>::v) * inv);                    // util.h:68-78
        else f = isfinite(inv) ? (float)(r[h] * inv) : 1.f / H;
        qpar[i * H + h] = __float2half_rn(f);
      }
    }
    __syncwarp();
    for (int r = lane; r < t.L; r += G) {
      const int n = t.pleaf[r];
      const real* ro = slot + n * H;
      real s1 = 0, e1 = 0;
      for (int h = 0; h < H; ++h) { s1 += ro[h]; e1 += ro[h] + Eps<real>::v; }
      const real inv = (real)1 / e1;
      p.scaler[row0 + r] = (opp == rp) ? par_sum[parent[n] - 1] : s1;                         // sum of the opponent's reach (:264-268)
      for (int h = 0; h < H; ++h) {
        float f;
        if (Eps<real>::kLiteral) f = (float)((ro[h] + Eps<real>::v) * inv);
        else f = isfinite(inv) ? (float)(ro[h] * inv) : 1.f / H;
        qown[r * H + h] = __float2half_rn(f);
      }
    }
  } else {
    // two-level template (max_depth 1, or a root whose only children are leaves): the pseudo-leaves are level-1 nodes; the root
    // player's reach is the node's slot, the other player's its root belief
    for (int r = lane; r < t.L; r += G) {
      const int n = t.pleaf[r];
      const real* r0 = d2_reach_row(slot, bel, parent, n, lv.n1e, 0, rp, H);
      const real* r1 = d2_reach_row(slot, bel, parent, n, lv.n1e, 1, rp, H);
      real s0 = 0, s1 = 0, e0 = 0, e1 = 0;
      for (int h = 0; h < H; ++h) { s0 += r0[h]; s1 += r1[h]; e0 += r0[h] + Eps<real>::v; e1 += r1[h] + Eps<real>::v; }
      const real i0 = (real)1 / e0, i1 = (real)1 / e1;
      p.scaler[row0 + r] = trav == 0 ? s1 : s0;
      // qpar <- the root player's columns, qown <- the other player's, like on level 2 (one qpar row per leaf here)
      const real* rr = rp == 0 ? r0 : r1; const real* ro = rp == 0 ? r1 : r0;
      const real ir = rp == 0 ? i0 : i1, io_ = rp == 0 ? i1 : i0;
      for (int h = 0; h < H; ++h) {
        float fr, fo;
        if (Eps<real>::kLiteral) { fr = (float)((rr[h] + Eps<real>::v) * ir); fo = (float)((ro[h] + Eps<real>::v) * io_); }
        else { fr = isfinite(ir) ? (float)(rr[h] * ir) : 1.f / H; fo = isfinite(io_) ? (float)(ro[h] * io_) : 1.f / H; }
        qpar[r * H + h] = __float2half_rn(fr);
        qown[r * H + h] = __float2half_rn(fo);
      }
    }
  }
  __syncwarp();
  // ---- query rows; all pseudo-leaves sit on the last level
  const int leaf_player = rp ^ ((t.levels - 1) & 1);
  const int Qp = p.Qpad;
  if (p.Xh != nullptr) {
    // fp16 tile in UMMA K-major core-matrix order, one 16-byte store per (row, 8 columns).  The constant columns (one-hot of
    // the leaf's last bid, the 1 at column Q, zero padding) come from the per-template table qconst, the acting player /
    // traverser flags are set here, the 2H belief columns are copied from the fp16 rows above.
    const int kc = Qp >> 3;
    const int qb0 = 2 + p.A, qb1 = qb0 + H, qb2 = qb1 + H;      // belief columns [qb0, qb1) player 0, [qb1, qb2) player 1
    const __half* __restrict__ qconst = p.qconst + t.qconst_off;
    for (int it = lane; it < t.L * kc; it += G) {
      const int k8 = it / t.L, r = it % t.L;
      union { int4 v; __half h[8]; } c;
      c.v = *reinterpret_cast<const int4*>(qconst + (size_t)r * Qp + k8 * 8);
      const int q0 = k8 * 8;
      if (q0 == 0) { c.h[0] = __float2half_rn((float)leaf_player); c.h[1] = __float2half_rn((float)trav); }
      if (q0 + 8 > qb0 && q0 < qb2) {
        const __half* rootp = have_l2 ? qpar + (parent[t.pleaf[r]] - 1) * H : qpar + r * H;   // player rp
        const __half* other = qown + r * H;                                                                      // player 1 - rp
        const __half* p0 = rp == 0 ? rootp : other;
        const __half* p1 = rp == 0 ? other : rootp;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int q = q0 + j;
          if (q >= qb0 && q < qb1) c.h[j] = p0[q - qb0];
          else if (q >= qb1 && q < qb2) c.h[j] = p1[q - qb1];
        }
      }
      const int Rr = row0 + r, rr = Rr & 127;
      *reinterpret_cast<int4*>(p.Xh + (size_t)(Rr >> 7) * 128 * Qp + k8 * 1024 + (rr >> 3) * 64 + (rr & 7) * 8) = c.v;
    }
  } else if (p.X != nullptr) {
    // fp32 parity net: the same columns in fp32 from the reach rows themselves
    for (int it = lane; it < t.L * Qp; it += G) {
      const int r = it / Qp, q = it % Qp;
      const int n = t.pleaf[r];
      const real* r0 = d2_reach_row(slot, bel, parent, n, lv.n1e, 0, rp, H);
      const real* r1 = d2_reach_row(slot, bel, parent, n, lv.n1e, 1, rp, H);
      real e0 = 0, e1 = 0;
      for (int h = 0; h < H; ++h) { e0 += r0[h] + Eps<real>::v; e1 += r1[h] + Eps<real>::v; }
      p.X[(size_t)(row0 + r) * Qp + q] = query_value(p, q, leaf_player, trav, (int)t.bid1[n] - 1, r0, r1, (real)1 / e0, (real)1 / e1);
    }
  }
  // ---- terminals (compute_expected_terminal_values :80-98; win probability :765-789), as in cfr_forward
  constexpr int kMaxBins = 9;
  real* __restrict__ vt = p.vterm + (size_t)k * p.vterm_stride;
  __syncwarp();      // hist shares the aux region with the fp16 belief columns the query rows were assembled from
  for (int z = lane; z < t.T; z += G) {
    const int n = t.term[z];
    const int face = t.term[t.T + z] % p.F;
    const real* ro = d2_reach_row(slot, bel, parent, n, lv.n1e, 1 - trav, rp, H);
    real cnt[kMaxBins];
#pragma unroll
    for (int m = 0; m < kMaxBins; ++m) cnt[m] = 0;
    real tot = 0;
    for (int g = 0; g < H; ++g) {
      const real r = ro[g];
      const int mg = (int)t.matches[g * p.F + face];
      tot += r;
#pragma unroll
      for (int m = 0; m < kMaxBins; ++m) cnt[m] += (m == mg) ? r : (real)0;
    }
#pragma unroll
    for (int m = kMaxBins - 2; m >= 0; --m) cnt[m] += cnt[m + 1];
#pragma unroll
    for (int m = 0; m < kMaxBins; ++m) hist[z * (kMaxBins + 1) + m] = cnt[m];
    hist[z * (kMaxBins + 1) + kMaxBins] = tot;
  }
  __syncwarp();
  for (int it = lane; it < t.T * H; it += G) {
    const int z = it / H, h = it % H;
    const int pbid = t.term[t.T + z];
    const int ndepth = t.term[2 * t.T + z];
    const int quantity = 1 + pbid / p.F, face = pbid % p.F;
    int left = quantity - (int)t.matches[h * p.F + face];
    left = left < 0 ? 0 : (left > kMaxBins - 1 ? kMaxBins - 1 : left);
    const real win = hist[z * (kMaxBins + 1) + left], tot = hist[z * (kMaxBins + 1) + kMaxBins];
    const real v = (real)(float)win * 2 - tot;
    const int pl = rp ^ (ndepth & 1);
    vt[z * H + h] = (pl != trav) ? -v : v;
  }
}

// Scratch of a d2 group (reals): slot[nh_max] | bel[2*H] | hist[tmp_reals] | aux (cfr_aux_bytes_d2)
template <typename real, int HC>
__global__ void __launch_bounds__(128, 8) cfr_iter_d2_kernel(CfrDev<real> p, int iter, int do_b, int do_f, int scratch_per_group) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // Programmatic dependent launch: the value-net kernel that follows may be scheduled as soon as every CTA of this grid has
  // started (its weight-staging prologue then overlaps this grid's tail) ...
  asm volatile("griddepcontrol.launch_dependents;");
  const int groups_per_cta = blockDim.x / 32;
  const int gid = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int k = blockIdx.x * groups_per_cta + gid;
  if (k >= *p.wave_n) return;
  const int H = HC > 0 ? HC : p.H;
  // per-group shared memory: [ template bytes (p.tpk_stride) | slot[nh_max] | bel[2*H] | aux ] ; the terminal histogram of the
  // forward half aliases aux (the fp16 belief columns are dead once the query rows are written)
  unsigned char* gbase = smem_raw + (size_t)gid * ((size_t)scratch_per_group * sizeof(real) + p.tpk_stride);
  unsigned char* tb_s = gbase;
  real* slot = reinterpret_cast<real*>(gbase + p.tpk_stride);
  real* bel = slot + p.nh_max; real* aux = bel + 2 * H; real* hist = aux;
  {   // the subgame's template: one coalesced 16-byte-per-lane copy
    const int4* src = reinterpret_cast<const int4*>(p.tpk + (size_t)p.sg_tmpl[k] * p.tpk_stride);
    int4* dst = reinterpret_cast<int4*>(tb_s);
    for (int i = lane; i < p.tpk_stride / 16; i += 32) dst[i] = __ldg(src + i);
  }
  for (int i = lane; i < 2 * H; i += 32) bel[i] = p.beliefs[(size_t)k * 2 * H + i];
  __syncwarp();
  const D2Tmpl t = d2_tmpl_view(tb_s, H * p.F);
  const D2Levels lv = d2_levels(tb_s);
  {
    // The wave's tables (3 x K x 4.3 KB at 1x6f) do not fit in L2 next to the query tiles, so every launch streams them from
    // HBM.  Ask for this subgame's lines now: the requests overlap the leaf-value phase instead of stalling the phases
    // that consume them one DRAM round trip at a time.
    const size_t off = (size_t)k * p.table_stride * sizeof(real);
    const int lines = ((t.N - 1) * H * (int)sizeof(real) + 127) >> 7;
    const char* sg = reinterpret_cast<const char*>(p.Sg) + off;
    for (int i = lane; i < lines; i += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(sg + ((size_t)i << 7)));
    if (do_b) {   // regrets and sum strategy: only the edges below the previous traverser's level are touched
      const bool root_acts = p.sg_player[k] == ((iter - 1) & 1);
      const int e0 = (root_acts ? lv.n1b : lv.n1e) - 1, e1 = (root_acts ? lv.n1e : lv.n2e) - 1;
      const size_t b0 = (size_t)e0 * H * sizeof(real) & ~(size_t)127, b1 = (size_t)e1 * H * sizeof(real);
      const char* rr = reinterpret_cast<const char*>(p.R) + off;
      const char* ss = reinterpret_cast<const char*>(p.S) + off;
      for (size_t o = b0 + ((size_t)lane << 7); o < b1; o += (size_t)32 << 7) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(rr + o));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ss + o));
      }
    }
  }
  // ... and this grid, launched the same way behind the previous value-net kernel, must not touch that kernel's outputs (or
  // tables a still earlier CFR launch wrote) before the kernel has completed.  A no-op for ordinary launches.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  __syncwarp();
  const int tb = (iter - 1) & 1;
  const int rp = p.sg_player[k];
  if (do_b) {
    if (p.fp) fp_backward_d2<real, HC>(p, t, lv, k, tb, slot, bel, lane);
    else cfr_backward_d2<real, HC>(p, t, lv, k, tb, slot, bel, aux, lane);
  }
  // sampling-strategy snapshot for RlRunner (recursive_solving.cc:168-174): state after `iter` iterations
  if (p.sg_act_iter[k] == iter) {
    const real* Sg = p.Sg + (size_t)k * p.table_stride;
    real* __restrict__ Sn = p.Snap + (size_t)k * p.table_stride;
    for (int i = lane; i < (t.N - 1) * H; i += 32) Sn[i] = Sg[i];
  }
  if (do_f) cfr_forward_d2<real, HC>(p, t, lv, k, iter & 1, slot, bel, do_b ? (tb == rp ? 0 : 1) : -1, aux, hist, lane);
}

// Wave initialisation == CFR constructor (subgame_solving.cc:509-524): uniform last strategy, zero regrets,
// sum = uniform * reach-under-uniform of the acting player (get_uniform_reach_weigted_strategy :125-149).
template <typename real, int G>
__global__ void __launch_bounds__(512) cfr_init_kernel(CfrDev<real> p, int scratch_per_group) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  real* smem = reinterpret_cast<real*>(smem_raw);
  const int groups_per_cta = blockDim.x / G;
  const int gid = threadIdx.x / G, lane = threadIdx.x % G;
  const int k = blockIdx.x * groups_per_cta + gid;
  if (k >= *p.wave_n) return;
  const TemplateDev t = p.tmpl[p.sg_tmpl[k]];
  const int H = p.H;
  real* base = (G == 32) ? smem + (size_t)gid * scratch_per_group : p.scratch + (size_t)k * p.scratch_stride;
  real* reach0 = base; real* reach1 = base + p.nh_max;
  real* __restrict__ R = p.R + (size_t)k * p.table_stride;
  real* __restrict__ Sg = p.Sg + (size_t)k * p.table_stride;
  real* __restrict__ S = p.S + (size_t)k * p.table_stride;
  const int* __restrict__ parent = p.parent + t.node_off;
  const int* __restrict__ nchild = p.nchild + t.node_off;
  const real* __restrict__ b = p.beliefs + (size_t)k * 2 * H;
  const int rp = p.sg_player[k];
  // act_iteration == 0: the sampling strategy RlRunner / the sampled recursive evaluation read is the INITIAL (uniform) one
  // (recursive_solving.cc:168-174 runs zero steps before sampling), and cfrb_run(0) launches nothing — so the snapshot is
  // taken here
  real* __restrict__ Sn = p.Snap + (size_t)k * p.table_stride;
  const bool snap0 = p.sg_act_iter[k] == 0;
  for (int h = lane; h < H; h += G) { reach0[h] = b[h]; reach1[h] = b[H + h]; }
  group_sync<G>();
  for (int d = 1; d < t.levels; ++d) {
    const int nb = p.level_begin[t.level_off + d], ne = p.level_begin[t.level_off + d + 1];
    const int actor = rp ^ ((d - 1) & 1);
    for (int it = lane; it < (ne - nb) * H; it += G) {
      const int c = nb + it / H, h = it % H;
      const int par = parent[c], e = (c - 1) * H + h;
      const real u = (real)1 / nchild[par];
      const real a0 = reach0[par * H + h], a1 = reach1[par * H + h];
      Sg[e] = u;
      if (snap0) Sn[e] = u;
      R[e] = p.fp ? u : (real)0;       // FP: last_strategies starts as the uniform strategy (subgame_solving.cc:375-377)
      S[e] = u * (actor == 0 ? a0 : a1);
      reach0[c * H + h] = actor == 0 ? a0 * u : a0;
      reach1[c * H + h] = actor == 1 ? a1 * u : a1;
    }
    group_sync<G>();
  }
  for (int i = lane; i < 2 * H; i += G) p.mu[(size_t)k * 2 * H + i] = 0;
  if (lane < 2) p.steps[2 * k + lane] = 0;
}

}  // namespace cfrb
