// Device-visible plain structs shared by the CFR kernels (cfr_kernels.cu) and the C-ABI host code (cfrb_api.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cfrb {

struct TemplateDev {
  int node_off, level_off, pleaf_off, term_off;
  int N, L, T, levels;
  int qconst_off, pad_[3];
};

template <typename real>
struct CfrDev {
  // game
  int A, H, F, Q, Qpad, Hout;
  // templates (read-only)
  const TemplateDev* tmpl;
  const int* parent; const int* child_begin; const int* nchild; const int* last_bid;
  const int* level_begin; const int* pleaf_node; const int* term_node;
  const unsigned char* matches;   // [H][F] num_matches(hand, face), liars_dice.h:83-91
  const unsigned char* tpk; int tpk_stride;   // packed byte templates (cfr_iter_d2_kernel): template i at tpk + i * tpk_stride
  const __half* qconst;           // per template [L][Qpad] fp16: constant part of the query rows (one-hot last bid, 1 at column Q)
  // wave
  const int* wave_n;              // [1] number of live subgames
  const int* sg_tmpl; const int* sg_player; const int* sg_row_off; const int* sg_act_iter;
  const real* beliefs;            // [K][2][H]
  real* mu;                       // [K][2][H] root_values_means
  int* steps;                     // [K][2]
  real* R; real* Sg; real* S; real* Snap;   // [K][table_stride]
  int table_stride;
  real* vterm; int vterm_stride;  // [K][Tmax*H] terminal payoffs of the current iteration
  float* X;                       // [rows][Qpad] fp32 query rows (SIMT net) -- or nullptr
  __half* Xh;                     // fp16 query tiles in UMMA core-matrix order (tensor-core net) -- or nullptr
  const float* net_out;           // [rows][Hout] raw net outputs
  real* scaler;                   // [rows] sum of opponent reach at the pseudo-leaf
  real* scratch; size_t scratch_stride;   // global scratch (CTA groups), reals per subgame
  int nh_max, tmp_reals;                  // scratch layout: bufA[nh_max] | bufB[nh_max] | tmp[tmp_reals] | lsum[2*Lmax]
  int lmax, tmax, n1max;                  // largest pseudo-leaf / terminal / level-1 node count over the templates (depth <= 2 kernels' layouts)
  // params
  int linear, dcfr; real dcfr_alpha, dcfr_beta, dcfr_gamma;
  int use_net;
  int fp, optimistic;             // fictitious play instead of CFR (FP, subgame_solving.cc:364-506)
};

// Scratch of a group (reals): bufA[N*H] | bufB[N*H] | hist[10*T] | lsum[2*L]  (hist: per-terminal match-count histogram,
// 9 bins + belief sum)
__host__ __device__ inline int cfr_tmp_reals(int N, int H, int L, int T) { (void)N; (void)H; (void)L; return 10 * (T > 0 ? T : 1); }
__host__ __device__ inline int cfr_scratch_reals(int N, int H, int L, int T) { return 2 * N * H + cfr_tmp_reals(N, H, L, T) + 2 * (L > 0 ? L : 1); }

// Depth <= 2 kernel (cfr_iter_d2_kernel): slot[N*H] | bel[2*H] | aux.  aux (bytes) serves the backward half as
// rcp[(n1max + 1) * H] reals (reciprocals of the regret-matching sums) and the forward half first as par_sum[n1max] | par_inv[n1max]
// reals followed by the fp16 belief columns qpar[n1max * H] | qown[L * H], then as the terminal histogram hist[10 * T] reals.
__host__ __device__ inline int cfr_aux_bytes_d2(int sz, int H, int L, int T, int n1max) {
  const int fwd = ((2 * n1max * sz + 15) & ~15) + (((n1max + (L > 0 ? L : 1)) * H * 2 + 15) & ~15);
  const int bwd = (n1max + 1) * H * sz;
  const int hist = 10 * (T > 0 ? T : 1) * sz;
  int m = fwd > bwd ? fwd : bwd;
  m = m > hist ? m : hist;
  return (m + 15) & ~15;
}
__host__ __device__ inline int cfr_scratch_reals_d2(int sz, int N, int H, int L, int T, int n1max) {
  const int per16 = 16 / sz;       // every group's region starts 16-byte aligned (its template bytes are copied with 16-byte accesses)
  const int reals = N * H + 2 * H + (cfr_aux_bytes_d2(sz, H, L, T, n1max) + sz - 1) / sz;
  return (reals + per16 - 1) / per16 * per16;
}

// Full-tree best response (br_kernel.cuh).  Arrays describe ONE full-depth tree rooted at the initial state.
struct BrDev {
  int N, T, levels, H, F;
  const int* parent; const int* child_begin; const int* nchild; const int* level_begin;   // level_begin: [levels + 1]
  const int* term_node;           // [3][T]: node id, challenged bid, depth
  const unsigned char* matches;   // [H][F]
  const double* strategy;         // compact [edge = child - 1][H]
  double* scratch; size_t scratch_stride;   // per traverser: reach0[N*H] | reach1[N*H] | val[N*H] | hist[10*T]
  double* out;                    // [2]
};
void br_launch(const BrDev& p, cudaStream_t st);

// Device-resident self-play (selfplay_kernels.cuh): per-game state of K games advanced in lock-step.
constexpr int kSpMaxH = 64;       // per-thread belief copies live in local memory: larger games use the host walk
constexpr int kSpMaxPath = 16;
struct SpDev {
  int K, A, H, Q, iters, sample_leaf;
  float random_action_prob;
  // per-game state
  int* g_last_bid; int* g_player;     // [K]
  double* g_beliefs;                  // [K][2][H]   (fp64 like RlRunner::beliefs_, whatever the table dtype)
  uint32_t* mt; int* mt_idx;          // [624][K], [K]
  // tree templates (read-only; the same arrays the CFR kernels index)
  const TemplateDev* tmpl; const int* child_begin; const int* nchild; const int* last_bid;
  // wave descriptors
  int* wave;                          // [0] = number of subgames, [1] = value-net rows
  int* sg_tmpl; int* sg_player; int* sg_row_off; int* sg_act;
  int table_stride;
};
void sp_launch_seed(const SpDev& p, const uint32_t* dev_seeds, cudaStream_t st);
// act_iteration draw + subgame descriptors + packed row offsets of the next wave
template <typename real> void sp_launch_begin(const SpDev& p, real* wave_beliefs, cudaStream_t st);
// training examples of the finished wave (skipped when ex_q == nullptr) and the sampling step of every game
template <typename real> void sp_launch_finish(const SpDev& p, const real* mu, const real* snap, float* ex_q, float* ex_v, cudaStream_t st);
// rows [ids[i]] of a [*, width] fp32 matrix -> out[i]  (replay sampling)
void rows_launch_gather(const float* src, int width, const int* ids, int n, float* out, cudaStream_t st);

// Development check of div_by_rcp (cfr_kernels.cuh): n pseudo-random (x, b) pairs per call, returns the number of quotients that
// differ from x / b in *mismatches (device pointer).
void div_check_launch(unsigned long long seed, int blocks, unsigned long long* mismatches, cudaStream_t st);

// Launchers implemented in cfr_kernels.cu (explicitly instantiated for float and double).  `group` is 32 (one warp per
// subgame, shared-memory scratch) or 256 (one CTA per subgame, global scratch).
template <typename real> cudaError_t cfr_configure(int group, int smem_bytes);
template <typename real> void cfr_launch_init(const CfrDev<real>& p, int group, int blocks, int threads, size_t smem, cudaStream_t st,
                                              int scratch_per_group);
template <typename real> void cfr_launch_iter(const CfrDev<real>& p, int group, int blocks, int threads, size_t smem, cudaStream_t st,
                                              int iter, int do_b, int do_f, int scratch_per_group);
// Depth <= 2 specialisation (warp per subgame, half the scratch); threads must be a multiple of 32 and <= 256.
template <typename real> cudaError_t cfr_configure_d2(int smem_bytes);
template <typename real> void cfr_launch_iter_d2(const CfrDev<real>& p, int blocks, int threads, size_t smem, cudaStream_t st, int iter,
                                                 int do_b, int do_f, int scratch_per_group);

}  // namespace cfrb
