// libcfrb200.so — C ABI implementation (include/cfrb200.h) of the B200 CFR wave solver.
// Plain CUDA runtime; no torch, no CPU fallback: every entry point that computes needs the device.
#include "../../include/cfrb200.h"

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <array>
#include <cstring>
#include <string>
#include <vector>

#include "cfr_types.h"
#include "cfr_tree.h"
#include "leaf_mlp_simt.cuh"
#include "leaf_mlp_tc.cuh"
#include "leaf_mlp_tc3.cuh"

namespace {
inline bool is_tc(int net_mode) { return net_mode == CFRB_NET_TC_F16 || net_mode == CFRB_NET_TC_F16X2; }

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(CFRB_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__) + " @" + __FILE__ + ":" + \
                                  std::to_string(__LINE__));                                       \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    n = count;
    return cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
  }
  void release() { if (p) cudaFree(p); p = nullptr; }
};

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Typed (fp32 / fp64) part of the solver state.
template <typename real>
struct WaveState {
  DevBuf<real> beliefs, mu, R, Sg, S, Snap, vterm, scaler, scratch;
  cfrb::CfrDev<real> dev{};
  void release() {
    beliefs.release(); mu.release(); R.release(); Sg.release(); S.release(); Snap.release(); vterm.release();
    scaler.release(); scratch.release();
  }
};

}  // namespace

struct cfrb_handle {
  cfrb_config cfg{};
  cfrb::GameShape g;
  std::vector<cfrb::TreeTemplate> tmpl;   // index = root_bid + 1
  int Nmax = 0, Lmax = 0, Tmax = 0;
  int Qpad = 0, Hout = 0;
  bool f64 = true;
  int group = 32;          // threads per subgame group (32 = warp, 256 = CTA with global scratch)
  int groups_per_cta = 8;
  int scratch_per_group = 0;  // reals
  // depth <= 2 kernel (all templates have at most three levels): own scratch layout and CTA shape
  bool d2 = false;
  int max_levels = 0;
  int d2_groups_per_cta = 8;
  int d2_scratch_per_group = 0;
  size_t d2_smem = 0;      // dynamic shared memory of a depth-2 CTA
  int n1max = 0;           // largest level-1 node count over the templates (depth-2 scratch layout)
  int table_stride = 0;
  int num_sms = 0;
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  int profiling = 0;          // 0 off, n: bracket every n-th value-net launch with CUDA events
  int net_launch_idx = 0, net_launches_run = 0;
  std::vector<cudaEvent_t> net_ev;   // pairs around value-net launches (profiling mode)
  int net_ev_used = 0;
  // CUDA graphs of whole cfrb_run calls (2 launches per iteration would otherwise be enqueued one by one by the host)
  struct GraphEntry { int first, count, prof, has_rows; cudaGraphExec_t exec; int launches, net_launches, ev_used; };
  std::vector<GraphEntry> graphs;
  std::vector<std::array<int, 4>> graph_seen;   // keys requested once: a graph is only built for a key that comes back
  bool capturing = false;           // launch geometry independent of the wave size while a graph is being captured / replayed
  // device: templates
  DevBuf<cfrb::TemplateDev> d_tmpl;
  DevBuf<int> d_parent, d_child_begin, d_nchild, d_last_bid, d_level_begin, d_pleaf_node, d_term_node;
  DevBuf<unsigned char> d_matches;
  // full-depth tree for cfrb_exploitability, built on first use
  struct BrState {
    bool ready = false;
    cfrb::TreeTemplate t;
    DevBuf<int> parent, child_begin, nchild, level_begin, term_node;
    DevBuf<double> strategy, scratch, out;
    size_t scratch_stride = 0;
  } br;
  DevBuf<__half> d_qconst;
  DevBuf<unsigned char> d_tpk;   // byte-packed templates for the depth <= 2 kernel
  int tpk_stride = 0;
  // device: wave (untyped part)
  DevBuf<int> d_wave;      // [0] = n, [1] = rows
  DevBuf<int> d_sg_tmpl, d_sg_player, d_sg_row_off, d_sg_act, d_steps;
  DevBuf<float> d_X, d_out, d_dbg;
  long long* dbg_trace = nullptr;   // set only inside cfrb_debug_net_trace
  DevBuf<__half> d_Xh;
  WaveState<float> sf;
  WaveState<double> sd;
  // device: weights
  DevBuf<float> d_w;
  DevBuf<uint8_t> d_blob;
  // weight upload without stalling the generator pipeline: two pinned staging buffers, stream-ordered copies on own_stream
  uint8_t* w_stage[2] = {nullptr, nullptr};
  size_t w_stage_bytes = 0;
  cudaEvent_t w_ev[2] = {nullptr, nullptr};
  int w_slot = 0;
  cudaEvent_t w_last = nullptr;      // completion of the most recent upload (waited for by runs on other streams)
  cfrb::NetDev net{};
  bool have_weights = false;
  uint64_t weights_version = 0;
  // host mirror of the wave
  int n = 0, rows = 0, iters_done = 0;
  std::vector<int> h_tmpl, h_player, h_row_off, h_last_bid;
  std::vector<double> h_beliefs;
  int64_t launches = 0;
  float last_total_ms = 0.f, last_net_ms = 0.f;
  // device-resident self-play (cfrb_selfplay_*): game states, generator streams
  struct SelfPlay {
    bool ready = false, pending = false;    // pending: a wave has been run whose games have not been advanced yet
    int K = 0;
    DevBuf<int> last_bid, player, mt_idx;
    DevBuf<double> beliefs;
    DevBuf<uint32_t> mt, seeds;
    cfrb::SpDev dev{};
    int64_t waves = 0;
    cudaEvent_t ev_examples = nullptr;    // recorded behind the example / advance kernels of the last finished wave
    bool ev_recorded = false;
  } sp;
  cudaEvent_t marks[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // cfrb_mark: timing events
  void* flush_buf = nullptr; size_t flush_bytes = 0;                                                 // cfrb_l2_flush
  bool rows_on_device = false;   // the wave was built on the device: its row count / roots exist only there
  bool mirror_stale = false;     // ... and the host mirror (h_tmpl, h_beliefs, rows) has not been pulled yet
};

template <typename real> static WaveState<real>& state_of(cfrb_handle* h);
template <> WaveState<float>& state_of<float>(cfrb_handle* h) { return h->sf; }
template <> WaveState<double>& state_of<double>(cfrb_handle* h) { return h->sd; }

#define DISPATCH_REAL(h, fn, ...) ((h)->f64 ? fn<double>(__VA_ARGS__) : fn<float>(__VA_ARGS__))

using cfrb::TemplateDev;

// ------------------------------------------------------------------------------------------ typed helpers
template <typename real>
static int alloc_state(cfrb_handle* h, int max_optin) {
  auto& s = state_of<real>(h);
  const auto& g = h->g;
  const int K = h->cfg.max_subgames;
  const size_t tab = (size_t)K * h->table_stride;
  const size_t rows_cap = (size_t)K * std::max(h->Lmax, 1);
  CK(s.beliefs.alloc((size_t)K * 2 * g.H)); CK(s.mu.alloc((size_t)K * 2 * g.H));
  CK(s.R.alloc(tab)); CK(s.Sg.alloc(tab)); CK(s.S.alloc(tab)); CK(s.Snap.alloc(tab));
  const int vterm_stride = round_up(std::max(h->Tmax, 1) * g.H, 4);     // 16-byte aligned rows
  CK(s.vterm.alloc((size_t)K * vterm_stride + 8)); CK(s.scaler.alloc(rows_cap + 8));
  CK(cudaMemset(s.vterm.p, 0, ((size_t)K * vterm_stride + 8) * sizeof(real)));
  CK(cudaMemset(s.scaler.p, 0, (rows_cap + 8) * sizeof(real)));
  CK(cudaMemset(s.Snap.p, 0, tab * sizeof(real)));
  const size_t per_group_bytes = (size_t)h->scratch_per_group * sizeof(real);
  if (per_group_bytes * 2 <= (size_t)max_optin) {
    h->group = 32;
    // 2 CTAs per SM, as many warps per CTA as fit in ~85 % of the shared memory (the rest stays L1 for the read-only
    // template arrays), capped by the register file (64 registers x 32 warps) and the 512-thread block
    const size_t budget = (size_t)max_optin * 85 / 100 / 2;
    h->groups_per_cta = (int)std::max<size_t>(1, std::min<size_t>(16, budget / per_group_bytes));
    const int smem_bytes = (int)(per_group_bytes * h->groups_per_cta);
    CK(cfrb::cfr_configure<real>(32, smem_bytes));
    const char* no_d2 = std::getenv("CFRB_NO_D2");
    if (h->max_levels <= 3 && h->tpk_stride > 0 && !(no_d2 && *no_d2 == '1')) {
      // 32 warps per SM (register file: 64 registers x 32 warps) as 8 CTAs of 4 warps: small CTAs even out the last round
      // (8192 subgames on 4736 warp slots = 1.73 rounds); each CTA has 1 KB of shared memory reserved by the runtime
      h->d2 = true;
      h->d2_scratch_per_group = cfrb::cfr_scratch_reals_d2((int)sizeof(real), h->Nmax, h->g.H, h->Lmax, h->Tmax, h->n1max);
      const size_t d2_bytes = (size_t)h->d2_scratch_per_group * sizeof(real) + h->tpk_stride;
      const size_t cta_budget = ((size_t)228 * 1024 - 8 * 1024) / 8;
      h->d2_groups_per_cta = (int)std::max<size_t>(1, std::min<size_t>(4, cta_budget / d2_bytes));
      if (const char* e = std::getenv("CFRB_D2_GROUPS")) h->d2_groups_per_cta = std::max(1, std::min(h->d2_groups_per_cta, std::atoi(e)));
      h->d2_smem = d2_bytes * h->d2_groups_per_cta;
      // CFRB_D2_CTAS_PER_SM=n: pad the CTA's shared memory so that exactly n CTAs fit an SM (resident warps = n x warps per CTA);
      // e.g. 7 x 4 = 28 warps make 8192 subgames 1.98 rounds on 148 SMs instead of 1.73 rounds of 32 warps executed as 2
      if (const char* e = std::getenv("CFRB_D2_CTAS_PER_SM")) {
        const int n = std::atoi(e);
        if (n >= 1 && n <= 8) h->d2_smem = std::max(h->d2_smem, ((size_t)227 * 1024 - (size_t)n * 1024) / n / 16 * 16);
      }
      CK(cfrb::cfr_configure_d2<real>((int)h->d2_smem));
    }
  } else {
    h->group = 256;
    h->groups_per_cta = 1;
    CK(s.scratch.alloc((size_t)K * h->scratch_per_group));
  }
  cfrb::CfrDev<real>& d = s.dev;
  d.A = g.A; d.H = g.H; d.F = g.F; d.Q = g.Q; d.Qpad = h->Qpad; d.Hout = h->Hout;
  d.tmpl = h->d_tmpl.p; d.parent = h->d_parent.p; d.child_begin = h->d_child_begin.p; d.nchild = h->d_nchild.p;
  d.last_bid = h->d_last_bid.p; d.level_begin = h->d_level_begin.p; d.pleaf_node = h->d_pleaf_node.p;
  d.term_node = h->d_term_node.p; d.matches = h->d_matches.p; d.qconst = h->d_qconst.p;
  d.tpk = h->d_tpk.p; d.tpk_stride = h->tpk_stride;
  d.wave_n = h->d_wave.p; d.sg_tmpl = h->d_sg_tmpl.p; d.sg_player = h->d_sg_player.p; d.sg_row_off = h->d_sg_row_off.p;
  d.sg_act_iter = h->d_sg_act.p; d.beliefs = s.beliefs.p; d.mu = s.mu.p; d.steps = h->d_steps.p;
  d.R = s.R.p; d.Sg = s.Sg.p; d.S = s.S.p; d.Snap = s.Snap.p; d.table_stride = h->table_stride;
  d.vterm = s.vterm.p; d.vterm_stride = vterm_stride;
  d.lmax = std::max(h->Lmax, 1); d.tmax = std::max(h->Tmax, 1); d.n1max = h->n1max;
  d.X = h->cfg.net_mode == CFRB_NET_FP32 ? h->d_X.p : nullptr;
  d.Xh = is_tc(h->cfg.net_mode) ? h->d_Xh.p : nullptr;
  d.net_out = h->d_out.p; d.scaler = s.scaler.p;
  d.scratch = h->group == 32 ? nullptr : s.scratch.p; d.scratch_stride = h->scratch_per_group;
  d.nh_max = h->Nmax * g.H; d.tmp_reals = cfrb::cfr_tmp_reals(h->Nmax, g.H, h->Lmax, h->Tmax);
  d.linear = h->cfg.linear_update; d.dcfr = h->cfg.dcfr;
  d.dcfr_alpha = (real)h->cfg.dcfr_alpha; d.dcfr_beta = (real)h->cfg.dcfr_beta; d.dcfr_gamma = (real)h->cfg.dcfr_gamma;
  d.use_net = h->cfg.net_mode != CFRB_NET_ZERO;
  d.fp = h->cfg.solver == CFRB_SOLVER_FP; d.optimistic = h->cfg.optimistic;
  return CFRB_OK;
}

template <typename real>
static int launch_init_t(cfrb_handle* h, cudaStream_t st) {
  auto& s = state_of<real>(h);
  const int blocks = (h->n + h->groups_per_cta - 1) / h->groups_per_cta;
  const size_t smem = h->group == 32 ? (size_t)h->scratch_per_group * sizeof(real) * h->groups_per_cta : 0;
  cfrb::cfr_launch_init<real>(s.dev, h->group, blocks, 32 * h->groups_per_cta, smem, st, h->scratch_per_group);
  ++h->launches;
  CK(cudaGetLastError());
  return CFRB_OK;
}

template <typename real>
static int launch_iter_t(cfrb_handle* h, cudaStream_t st, int iter, int do_b, int do_f) {
  auto& s = state_of<real>(h);
  const int nsg = h->capturing ? h->cfg.max_subgames : h->n;   // surplus groups return at once (k >= *wave_n)
  if (h->d2) {
    const int blocks = (nsg + h->d2_groups_per_cta - 1) / h->d2_groups_per_cta;
    const size_t smem = h->d2_smem;
    cfrb::cfr_launch_iter_d2<real>(s.dev, blocks, 32 * h->d2_groups_per_cta, smem, st, iter, do_b, do_f, h->d2_scratch_per_group);
  } else {
    const int blocks = (nsg + h->groups_per_cta - 1) / h->groups_per_cta;
    const size_t smem = h->group == 32 ? (size_t)h->scratch_per_group * sizeof(real) * h->groups_per_cta : 0;
    cfrb::cfr_launch_iter<real>(s.dev, h->group, blocks, 32 * h->groups_per_cta, smem, st, iter, do_b, do_f, h->scratch_per_group);
  }
  ++h->launches;
  CK(cudaGetLastError());
  return CFRB_OK;
}

template <typename real>
static int upload_beliefs_t(cfrb_handle* h, cudaStream_t st) {
  auto& s = state_of<real>(h);
  std::vector<real> tmp(h->h_beliefs.begin(), h->h_beliefs.end());
  CK(cudaMemcpyAsync(s.beliefs.p, tmp.data(), tmp.size() * sizeof(real), cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  return CFRB_OK;
}

// compact [E][H] (edge = child-1) <-> dense [Nmax][H][A]
template <typename real>
static void to_dense(const cfrb_handle* h, int k, const real* compact, double* dense) {
  const auto& t = h->tmpl[h->h_tmpl[k]];
  const int H = h->g.H, A = h->g.A;
  std::memset(dense, 0, sizeof(double) * (size_t)h->Nmax * H * A);
  for (int n = 0; n < t.N; ++n)
    for (int j = 0; j < t.nchild[n]; ++j) {
      const int c = t.child_begin[n] + j, a = t.act_lo[n] + j;
      for (int hd = 0; hd < H; ++hd) dense[((size_t)n * H + hd) * A + a] = (double)compact[(size_t)(c - 1) * H + hd];
    }
}
template <typename real>
static void from_dense(const cfrb_handle* h, int k, const double* dense, real* compact) {
  const auto& t = h->tmpl[h->h_tmpl[k]];
  const int H = h->g.H, A = h->g.A;
  for (int n = 0; n < t.N; ++n)
    for (int j = 0; j < t.nchild[n]; ++j) {
      const int c = t.child_begin[n] + j, a = t.act_lo[n] + j;
      for (int hd = 0; hd < H; ++hd) compact[(size_t)(c - 1) * H + hd] = (real)dense[((size_t)n * H + hd) * A + a];
    }
}

template <typename real>
static int fetch_t(cfrb_handle* h, double* root_value_means, double* snapshot_strategy, double* last_strategy, double* avg_strategy,
                   double* sum_strategy, double* regrets) {
  auto& s = state_of<real>(h);
  const int n = h->n, H = h->g.H, A = h->g.A;
  if (root_value_means) {
    std::vector<real> mu((size_t)n * 2 * H);
    CK(cudaMemcpy(mu.data(), s.mu.p, mu.size() * sizeof(real), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < mu.size(); ++i) root_value_means[i] = (double)mu[i];
  }
  const size_t dense_sz = (size_t)h->Nmax * H * A;
  std::vector<real> tmp;
  std::vector<int> steps((size_t)n * 2);
  CK(cudaMemcpy(steps.data(), h->d_steps.p, steps.size() * sizeof(int), cudaMemcpyDeviceToHost));
  auto pull = [&](const real* dsrc, double* out, bool normalise) -> int {
    tmp.resize((size_t)n * h->table_stride);
    CK(cudaMemcpy(tmp.data(), dsrc, tmp.size() * sizeof(real), cudaMemcpyDeviceToHost));
    for (int k = 0; k < n; ++k) {
      double* dk = out + (size_t)k * dense_sz;
      to_dense<real>(h, k, tmp.data() + (size_t)k * h->table_stride, dk);
      if (normalise) {   // average strategy = normalised sum (subgame_solving.cc:659-660)
        const auto& t = h->tmpl[h->h_tmpl[k]];
        for (int nn = 0; nn < t.N; ++nn) {
          if (!t.nchild[nn]) continue;
          // average_strategies of a player stays the uniform initial strategy until that player's first update
          // (CFR ctor, subgame_solving.cc:516-518; the normalised sum is only written in step(), :659-660)
          const bool untouched = steps[2 * k + (h->h_player[k] ^ (t.depth[nn] & 1))] == 0;
          for (int hd = 0; hd < H; ++hd) {
            double* row = dk + ((size_t)nn * H + hd) * A;
            double sum = 0;
            for (int a = 0; a < A; ++a) sum += row[a];
            if (sum > 0 && !untouched) for (int a = 0; a < A; ++a) row[a] /= sum;
            else for (int j = 0; j < t.nchild[nn]; ++j) row[t.act_lo[nn] + j] = 1.0 / t.nchild[nn];
          }
        }
      }
    }
    return CFRB_OK;
  };
  int rc = CFRB_OK;
  if (snapshot_strategy && (rc = pull(s.Snap.p, snapshot_strategy, false))) return rc;
  const bool fp = h->cfg.solver == CFRB_SOLVER_FP;   // FP: Sg = average_strategies, R = last_strategies
  if (last_strategy && (rc = pull(fp ? s.R.p : s.Sg.p, last_strategy, false))) return rc;
  if (avg_strategy && (rc = fp ? pull(s.Sg.p, avg_strategy, false) : pull(s.S.p, avg_strategy, true))) return rc;
  if (sum_strategy && (rc = pull(s.S.p, sum_strategy, false))) return rc;
  if (regrets && fp) std::fill(regrets, regrets + (size_t)n * dense_sz, 0.0);
  if (regrets && !fp && (rc = pull(s.R.p, regrets, false))) return rc;
  return CFRB_OK;
}

template <typename real>
static int fetch_compact_t(cfrb_handle* h, int which, double* out) {
  auto& s = state_of<real>(h);
  const bool fp = h->cfg.solver == CFRB_SOLVER_FP;
  // 4 = average strategy (ISubgameSolver::get_strategy): FP keeps it in the Sg table; CFR's is normalise(sum) (:659-660)
  const bool avg_from_sum = which == 4 && !fp;
  const real* src = which == 0 ? s.Snap.p : which == 1 ? s.Sg.p : which == 2 ? s.S.p : which == 4 ? (fp ? s.Sg.p : s.S.p) : s.R.p;
  const size_t cnt = (size_t)h->n * h->table_stride;
  if (sizeof(real) == sizeof(double)) {
    CK(cudaMemcpy(out, src, cnt * sizeof(double), cudaMemcpyDeviceToHost));
  } else {
    std::vector<real> tmp(cnt);
    CK(cudaMemcpy(tmp.data(), src, cnt * sizeof(real), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < cnt; ++i) out[i] = (double)tmp[i];
  }
  if (avg_from_sum) {
    std::vector<int> steps((size_t)h->n * 2);
    CK(cudaMemcpy(steps.data(), h->d_steps.p, steps.size() * sizeof(int), cudaMemcpyDeviceToHost));
    const int H = h->g.H;
    for (int k = 0; k < h->n; ++k) {
      const auto& t = h->tmpl[h->h_tmpl[k]];
      double* tk = out + (size_t)k * h->table_stride;
      for (int nn = 0; nn < t.N; ++nn) {
        const int nc = t.nchild[nn];
        if (!nc) continue;
        // the average of a player stays the uniform initial strategy until that player's first update (same rule as cfrb_fetch)
        const bool untouched = steps[2 * k + (h->h_player[k] ^ (t.depth[nn] & 1))] == 0;
        for (int hd = 0; hd < H; ++hd) {
          double sum = 0;
          for (int j = 0; j < nc; ++j) sum += tk[(size_t)(t.child_begin[nn] + j - 1) * H + hd];
          for (int j = 0; j < nc; ++j) {
            double& v = tk[(size_t)(t.child_begin[nn] + j - 1) * H + hd];
            v = (sum > 0 && !untouched) ? v / sum : 1.0 / nc;
          }
        }
      }
    }
  }
  return CFRB_OK;
}

template <typename real>
static int load_state_t(cfrb_handle* h, const double* regrets, const double* last_strategy, const double* sum_strategy,
                        const double* root_value_means) {
  auto& s = state_of<real>(h);
  const int n = h->n, H = h->g.H, A = h->g.A;
  const size_t dense_sz = (size_t)h->Nmax * H * A;
  std::vector<real> tmp((size_t)n * h->table_stride);
  auto push = [&](const double* dense, real* ddst) -> int {
    CK(cudaMemcpy(tmp.data(), ddst, tmp.size() * sizeof(real), cudaMemcpyDeviceToHost));
    for (int k = 0; k < n; ++k) from_dense<real>(h, k, dense + (size_t)k * dense_sz, tmp.data() + (size_t)k * h->table_stride);
    CK(cudaMemcpy(ddst, tmp.data(), tmp.size() * sizeof(real), cudaMemcpyHostToDevice));
    return CFRB_OK;
  };
  int rc;
  if (regrets && (rc = push(regrets, s.R.p))) return rc;
  if (last_strategy && (rc = push(last_strategy, s.Sg.p))) return rc;
  if (sum_strategy && (rc = push(sum_strategy, s.S.p))) return rc;
  if (root_value_means) {
    std::vector<real> mu(root_value_means, root_value_means + (size_t)n * 2 * H);
    CK(cudaMemcpy(s.mu.p, mu.data(), mu.size() * sizeof(real), cudaMemcpyHostToDevice));
  }
  return CFRB_OK;
}

template <typename real>
static int examples_values_t(cfrb_handle* h, float* values) {
  auto& s = state_of<real>(h);
  std::vector<real> mu((size_t)h->n * 2 * h->g.H);
  CK(cudaMemcpy(mu.data(), s.mu.p, mu.size() * sizeof(real), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < mu.size(); ++i) values[i] = (float)mu[i];   // std::copy_n into a float tensor, subgame_solving.cc:224
  return CFRB_OK;
}

template <typename real>
static int scalers_t(cfrb_handle* h, double* out, int rows) {
  auto& s = state_of<real>(h);
  std::vector<real> v(rows);
  CK(cudaMemcpy(v.data(), s.scaler.p, (size_t)rows * sizeof(real), cudaMemcpyDeviceToHost));
  for (int i = 0; i < rows; ++i) out[i] = (double)v[i];
  return CFRB_OK;
}

// A wave built on the device (cfrb_selfplay_wave) has no host mirror of its subgame descriptors; the inspection entry points
// (fetch / examples / load_state / reset, used by tests and evaluators, not by the self-play loop) pull it on demand.
template <typename real>
static int pull_beliefs_t(cfrb_handle* h) {
  auto& s = state_of<real>(h);
  std::vector<real> tmp((size_t)h->n * 2 * h->g.H);
  CK(cudaMemcpy(tmp.data(), s.beliefs.p, tmp.size() * sizeof(real), cudaMemcpyDeviceToHost));
  h->h_beliefs.assign(tmp.begin(), tmp.end());
  return CFRB_OK;
}
template <typename real>
static int selfplay_finish_t(cfrb_handle* h, float* ex_q, float* ex_v, cudaStream_t st) {
  auto& s = state_of<real>(h);
  cfrb::sp_launch_finish<real>(h->sp.dev, s.mu.p, s.Snap.p, ex_q, ex_v, st);
  h->launches += ex_q ? 2 : 1;
  CK(cudaGetLastError());
  return CFRB_OK;
}
template <typename real>
static int selfplay_begin_t(cfrb_handle* h, cudaStream_t st) {
  auto& s = state_of<real>(h);
  cfrb::sp_launch_begin<real>(h->sp.dev, s.beliefs.p, st);
  h->launches += 2;
  CK(cudaGetLastError());
  return CFRB_OK;
}

static int sync_mirror(cfrb_handle* h) {
  if (!h->rows_on_device || !h->mirror_stale) return CFRB_OK;
  CK(cudaDeviceSynchronize());
  const int n = h->n;
  int wave[2] = {0, 0};
  CK(cudaMemcpy(wave, h->d_wave.p, sizeof(wave), cudaMemcpyDeviceToHost));
  h->rows = wave[1];
  h->h_tmpl.resize(n); h->h_player.resize(n); h->h_row_off.resize(n); h->h_last_bid.resize(n);
  CK(cudaMemcpy(h->h_tmpl.data(), h->d_sg_tmpl.p, n * sizeof(int), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(h->h_player.data(), h->d_sg_player.p, n * sizeof(int), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(h->h_row_off.data(), h->d_sg_row_off.p, n * sizeof(int), cudaMemcpyDeviceToHost));
  for (int k = 0; k < n; ++k) h->h_last_bid[k] = h->h_tmpl[k] - 1;
  int rc = DISPATCH_REAL(h, pull_beliefs_t, h);
  if (rc) return rc;
  h->mirror_stale = false;
  return CFRB_OK;
}

extern "C" {

const char* cfrb_last_error(void) { return g_err.c_str(); }

int cfrb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int cfrb_destroy(cfrb_handle* h) {
  if (!h) return CFRB_OK;
  cudaSetDevice(h->cfg.device);
  if (h->own_stream) cudaStreamSynchronize(h->own_stream);
  h->d_tmpl.release(); h->d_parent.release(); h->d_child_begin.release(); h->d_nchild.release(); h->d_last_bid.release();
  h->br.parent.release(); h->br.child_begin.release(); h->br.nchild.release(); h->br.level_begin.release(); h->br.term_node.release();
  h->br.strategy.release(); h->br.scratch.release(); h->br.out.release();
  h->d_tpk.release();
  h->d_level_begin.release(); h->d_pleaf_node.release(); h->d_term_node.release(); h->d_matches.release(); h->d_qconst.release();
  h->d_wave.release(); h->d_sg_tmpl.release(); h->d_sg_player.release(); h->d_sg_row_off.release(); h->d_sg_act.release();
  h->d_steps.release(); h->d_X.release(); h->d_out.release(); h->d_dbg.release(); h->d_Xh.release();
  h->sf.release(); h->sd.release(); h->d_w.release(); h->d_blob.release();
  h->sp.last_bid.release(); h->sp.player.release(); h->sp.mt_idx.release(); h->sp.beliefs.release(); h->sp.mt.release();
  h->sp.seeds.release();
  if (h->sp.ev_examples) cudaEventDestroy(h->sp.ev_examples);
  for (auto e : h->marks) if (e) cudaEventDestroy(e);
  for (int i = 0; i < 2; ++i) { if (h->w_stage[i]) cudaFreeHost(h->w_stage[i]); if (h->w_ev[i]) cudaEventDestroy(h->w_ev[i]); }
  if (h->flush_buf) cudaFree(h->flush_buf);
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
  for (auto e : h->net_ev) cudaEventDestroy(e);
  if (h->ev_a) cudaEventDestroy(h->ev_a);
  if (h->ev_b) cudaEventDestroy(h->ev_b);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return CFRB_OK;
}

static int create_impl(const cfrb_config* cfg, cfrb_handle* h) {
  h->cfg = *cfg;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(CFRB_ENODEV, "no CUDA device visible: libcfrb200 has no CPU fallback");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return fail(CFRB_EINVAL, "device ordinal out of range");
  CK(cudaSetDevice(cfg->device));
  if (cfg->num_dice < 1 || cfg->num_faces < 1 || cfg->max_depth < 1 || cfg->max_subgames < 1)
    return fail(CFRB_EINVAL, "num_dice, num_faces, max_depth, max_subgames must be >= 1");
  if (cfg->net_mode < CFRB_NET_ZERO || cfg->net_mode > CFRB_NET_TC_F16X2) return fail(CFRB_EINVAL, "bad net_mode");
  if (cfg->state_dtype != CFRB_STATE_F64 && cfg->state_dtype != CFRB_STATE_F32) return fail(CFRB_EINVAL, "bad state_dtype");
  if (cfg->solver != CFRB_SOLVER_CFR && cfg->solver != CFRB_SOLVER_FP) return fail(CFRB_EINVAL, "bad solver");
  if (cfg->net_mode != CFRB_NET_ZERO && cfg->hidden != 256) return fail(CFRB_EINVAL, "only hidden == 256 is built");
  h->f64 = cfg->state_dtype == CFRB_STATE_F64;
  h->g = cfrb::GameShape(cfg->num_dice, cfg->num_faces);
  const auto& g = h->g;
  if (g.A > 1024 || g.H > 4096) return fail(CFRB_EINVAL, "game too large");
  // ---- templates: root_bid in {-1, 0 .. A-2}
  std::vector<TemplateDev> td;
  std::vector<int> parent, child_begin, nchild, last_bid, level_begin, pleaf_node, term_node;
  std::vector<__half> qconst;
  const int Qpad = round_up(g.Q + 1, 16);
  for (int rb = -1; rb <= g.A - 2; ++rb) {
    h->tmpl.push_back(cfrb::build_template(g, rb, cfg->max_depth));
    const auto& t = h->tmpl.back();
    TemplateDev d;
    d.node_off = (int)child_begin.size(); d.level_off = (int)level_begin.size();
    d.pleaf_off = (int)pleaf_node.size(); d.term_off = (int)term_node.size();
    d.N = t.N; d.L = t.L; d.T = t.T; d.levels = t.levels;
    d.qconst_off = (int)qconst.size();
    for (int n : t.pleaf_node)
      for (int q = 0; q < Qpad; ++q)   // one-hot of the leaf's last bid (subgame_solving.cc:111-113) and the constant 1 at column Q
        qconst.push_back(__float2half_rn((q >= 2 && q < 2 + g.A && q - 2 == t.last_bid[n]) || q == g.Q ? 1.f : 0.f));
    td.push_back(d);
    parent.insert(parent.end(), t.parent.begin(), t.parent.end());
    child_begin.insert(child_begin.end(), t.child_begin.begin(), t.child_begin.end());
    nchild.insert(nchild.end(), t.nchild.begin(), t.nchild.end());
    last_bid.insert(last_bid.end(), t.last_bid.begin(), t.last_bid.end());
    level_begin.insert(level_begin.end(), t.level_begin.begin(), t.level_begin.end());
    level_begin.push_back(t.N);   // sentinel: "children of the last level" is an empty range
    pleaf_node.insert(pleaf_node.end(), t.pleaf_node.begin(), t.pleaf_node.end());
    term_node.insert(term_node.end(), t.term_node.begin(), t.term_node.end());
    for (int n : t.term_node) term_node.push_back(t.last_bid[t.parent[n]]);   // challenged bid
    for (int n : t.term_node) term_node.push_back(t.depth[n]);
    h->max_levels = std::max(h->max_levels, t.levels);
    h->Nmax = std::max(h->Nmax, t.N); h->Lmax = std::max(h->Lmax, t.L); h->Tmax = std::max(h->Tmax, t.T);
  }
  std::vector<unsigned char> matches((size_t)g.H * g.F);
  for (int hd = 0; hd < g.H; ++hd)
    for (int f = 0; f < g.F; ++f) matches[(size_t)hd * g.F + f] = (unsigned char)g.num_matches(hd, f);

  // byte-packed copies of the templates for cfr_iter_d2_kernel (one coalesced copy into shared memory per subgame and launch):
  // header {N, L, T, levels, n1e, n2e, -, -, qconst_off:int32, -} | parent[N] child_begin[N] nchild[N] last_bid+1[N] pleaf[L]
  // term[3][T] matches[H*F]; only built when every count fits a byte (all depth <= 2 trees of the supported games do)
  std::vector<unsigned char> tpk;
  if (h->max_levels <= 3 && h->Nmax <= 255 && g.A <= 254) {
    size_t mx = 0;
    for (const auto& t : h->tmpl) mx = std::max(mx, (size_t)16 + 4 * (size_t)t.N + t.L + 3 * (size_t)t.T + (size_t)g.H * g.F);
    h->tpk_stride = round_up((int)mx, 16);
    tpk.assign((size_t)h->tpk_stride * h->tmpl.size(), 0);
    for (size_t i = 0; i < h->tmpl.size(); ++i) {
      const auto& t = h->tmpl[i];
      unsigned char* b = tpk.data() + i * h->tpk_stride;
      b[0] = (unsigned char)t.N; b[1] = (unsigned char)t.L; b[2] = (unsigned char)t.T; b[3] = (unsigned char)t.levels;
      b[4] = (unsigned char)(t.levels >= 2 ? t.level_begin[2] : t.level_begin[1]);
      b[5] = (unsigned char)(t.levels >= 3 ? t.level_begin[3] : b[4]);
      std::memcpy(b + 8, &td[i].qconst_off, sizeof(int));
      unsigned char* q = b + 16;
      for (int n = 0; n < t.N; ++n) q[n] = (unsigned char)(t.parent[n] < 0 ? 0 : t.parent[n]);
      q += t.N;
      for (int n = 0; n < t.N; ++n) q[n] = (unsigned char)t.child_begin[n];
      q += t.N;
      for (int n = 0; n < t.N; ++n) q[n] = (unsigned char)t.nchild[n];
      q += t.N;
      for (int n = 0; n < t.N; ++n) q[n] = (unsigned char)(t.last_bid[n] + 1);
      q += t.N;
      for (int r = 0; r < t.L; ++r) q[r] = (unsigned char)t.pleaf_node[r];
      q += t.L;
      for (int z = 0; z < t.T; ++z) {
        q[z] = (unsigned char)t.term_node[z];
        q[t.T + z] = (unsigned char)t.last_bid[t.parent[t.term_node[z]]];     // challenged bid (:287); a terminal is never the root
        q[2 * t.T + z] = (unsigned char)t.depth[t.term_node[z]];
      }
      q += 3 * t.T;
      std::memcpy(q, matches.data(), matches.size());
    }
  }
  auto up = [&](auto& buf, const auto& v) -> cudaError_t {
    cudaError_t e = buf.alloc(v.size());
    if (e != cudaSuccess) return e;
    return cudaMemcpy(buf.p, v.data(), v.size() * sizeof(v[0]), cudaMemcpyHostToDevice);
  };
  CK(up(h->d_tpk, tpk));
  CK(up(h->d_tmpl, td)); CK(up(h->d_parent, parent)); CK(up(h->d_child_begin, child_begin)); CK(up(h->d_nchild, nchild));
  CK(up(h->d_last_bid, last_bid)); CK(up(h->d_level_begin, level_begin)); CK(up(h->d_pleaf_node, pleaf_node));
  CK(up(h->d_term_node, term_node)); CK(up(h->d_matches, matches)); CK(up(h->d_qconst, qconst));

  // ---- sizes
  const int K = cfg->max_subgames;
  h->Qpad = round_up(g.Q + 1, 16);   // one spare column carries the constant 1 that feeds bias 1 through the tensor cores
  h->Hout = round_up(g.H, 4);                                     // value-net output rows padded to 16 bytes
  h->table_stride = round_up(std::max(1, (h->Nmax - 1) * g.H), 4);   // every subgame's tables start 16-byte aligned
  h->n1max = g.A;
  h->scratch_per_group = cfrb::cfr_scratch_reals(h->Nmax, g.H, h->Lmax, h->Tmax);
  int max_optin = 0;
  CK(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device));
  CK(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, cfg->device));
  CK(h->d_wave.alloc(2));
  CK(h->d_sg_tmpl.alloc(K)); CK(h->d_sg_player.alloc(K)); CK(h->d_sg_row_off.alloc(K)); CK(h->d_sg_act.alloc(K));
  CK(h->d_steps.alloc((size_t)K * 2));
  const size_t rows_cap = (size_t)K * std::max(h->Lmax, 1);
  CK(h->d_X.alloc(cfg->net_mode == CFRB_NET_FP32 ? rows_cap * h->Qpad : 1));
  CK(h->d_out.alloc(rows_cap * h->Hout));
  CK(cudaMemset(h->d_wave.p, 0, 2 * sizeof(int)));
  CK(cudaMemset(h->d_out.p, 0, rows_cap * h->Hout * sizeof(float)));
  if (is_tc(cfg->net_mode)) {
    if (g.H > cfrb::tc::kNout) return fail(CFRB_EINVAL, "CFRB_NET_TC_F16 supports num_hands <= 16");
    const size_t tiles = (rows_cap + cfrb::tc::kTileM - 1) / cfrb::tc::kTileM;
    CK(h->d_Xh.alloc(tiles * cfrb::tc::kTileM * h->Qpad));
    CK(cudaMemset(h->d_Xh.p, 0, tiles * cfrb::tc::kTileM * h->Qpad * sizeof(__half)));
    CK(h->d_dbg.alloc(2 * cfrb::tc::kTileM * cfrb::tc::kHid));
    const cfrb::tc::Tc3Layout T3(h->Qpad);
    if (T3.smem_bytes > max_optin) return fail(CFRB_EINVAL, "tensor-core value net does not fit shared memory for this game shape");
    CK(cudaFuncSetAttribute(cfrb::tc::leaf_mlp_tc3_kernel<false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, T3.smem_bytes));
    CK(cudaFuncSetAttribute(cfrb::tc::leaf_mlp_tc3_kernel<true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, T3.smem_bytes));
    CK(cudaFuncSetAttribute(cfrb::tc::leaf_mlp_tc3_kernel<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, T3.smem_bytes));
    CK(cudaFuncSetAttribute(cfrb::tc::leaf_mlp_tc3_kernel<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, T3.smem_bytes));
  }
  CK(cudaFuncSetAttribute(cfrb::leaf_mlp_fp32_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)cfrb::leaf_mlp_fp32_smem(256)));
  int rc = DISPATCH_REAL(h, alloc_state, h, max_optin);
  if (rc) return rc;
  CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&h->ev_a)); CK(cudaEventCreate(&h->ev_b));
  return CFRB_OK;
}

int cfrb_create(const cfrb_config* cfg, cfrb_handle** out) {
  if (!cfg || !out) return fail(CFRB_EINVAL, "null argument");
  cfrb_handle* h = new cfrb_handle();
  int rc = create_impl(cfg, h);
  if (rc != CFRB_OK) {
    std::string keep = g_err;
    cfrb_destroy(h);
    g_err = keep;
    *out = nullptr;
    return rc;
  }
  *out = h;
  return CFRB_OK;
}

int cfrb_num_actions(const cfrb_handle* h) { return h->g.A; }
int cfrb_num_hands(const cfrb_handle* h) { return h->g.H; }
int cfrb_query_size(const cfrb_handle* h) { return h->g.Q; }
int cfrb_max_nodes(const cfrb_handle* h) { return h->Nmax; }

static void export_tree(const cfrb::TreeTemplate& t, int player_id, cfrb_node* out, int cap) {
  for (int n = 0; n < t.N && n < cap; ++n) {
    out[n].last_bid = t.last_bid[n];
    out[n].player_id = player_id ^ (t.depth[n] & 1);
    // like the reference, a processed node with an empty bid range (terminal above the depth limit) keeps
    // children_begin == children_end == (tree size at that moment); unprocessed nodes keep 0/0 (tree.h:59-62)
    out[n].children_begin = t.child_begin[n];
    out[n].children_end = t.child_begin[n] + t.nchild[n];
    out[n].parent = t.parent[n];
    out[n].depth = t.depth[n];
  }
}

int cfrb_unroll_tree(int32_t num_dice, int32_t num_faces, int32_t last_bid, int32_t player_id, int32_t max_depth,
                     cfrb_node* out, int32_t cap) {
  if (num_dice < 1 || num_faces < 1 || max_depth < 0) return fail(CFRB_EINVAL, "bad game shape");
  cfrb::GameShape g(num_dice, num_faces);
  if (last_bid < -1 || last_bid >= g.A) return fail(CFRB_EINVAL, "bad root bid");
  const auto t = cfrb::build_template(g, last_bid, max_depth);
  export_tree(t, player_id, out, cap);
  return t.N;
}

int cfrb_tree_template(const cfrb_handle* h, int32_t last_bid, int32_t player_id, cfrb_node* out, int32_t cap) {
  if (!h || last_bid < -1 || last_bid > h->g.A - 2) return fail(CFRB_EINVAL, "bad root bid");
  const auto& t = h->tmpl[last_bid + 1];
  export_tree(t, player_id, out, cap);
  return t.N;
}

int cfrb_set_weights(cfrb_handle* h, const float* flat, size_t n, uint64_t version) {
  if (!h || !flat) return fail(CFRB_EINVAL, "null argument");
  const int hid = h->cfg.hidden, Q = h->g.Q, H = h->g.H, Qp = h->Qpad;
  const size_t expect = (size_t)hid * Q + 3 * hid + (size_t)hid * hid + 3 * hid + (size_t)H * hid + H;
  if (n != expect) return fail(CFRB_EINVAL, "weight count mismatch: expected " + std::to_string(expect) + " got " + std::to_string(n));
  CK(cudaSetDevice(h->cfg.device));
  const float* w1 = flat; const float* b1 = w1 + (size_t)hid * Q; const float* g1 = b1 + hid; const float* be1 = g1 + hid;
  const float* w2 = be1 + hid; const float* b2 = w2 + (size_t)hid * hid; const float* g2 = b2 + hid; const float* be2 = g2 + hid;
  const float* w3 = be2 + hid; const float* b3 = w3 + (size_t)H * hid;
  // Stream-ordered upload: the packed weights are built in a pinned staging buffer and copied on the handle's stream, i.e.
  // after the waves already enqueued there (ModelLocker::updateModel waits for in-flight forwards; here nothing waits — the
  // generator's software pipeline keeps running) and before everything enqueued later.
  const size_t total_fp32 = (size_t)Qp * hid + 3 * hid + (size_t)hid * hid + 3 * hid + (size_t)hid * h->Hout + h->Hout;
  const size_t need = is_tc(h->cfg.net_mode) ? (size_t)cfrb::tc::BlobLayout(Qp).blob_bytes : total_fp32 * sizeof(float);
  if (h->w_stage_bytes < need) {
    CK(cudaStreamSynchronize(h->own_stream));
    for (int i = 0; i < 2; ++i) {
      if (h->w_stage[i]) cudaFreeHost(h->w_stage[i]);
      h->w_stage[i] = nullptr;
      CK(cudaMallocHost((void**)&h->w_stage[i], need));
      if (!h->w_ev[i]) CK(cudaEventCreateWithFlags(&h->w_ev[i], cudaEventDisableTiming));
    }
    h->w_stage_bytes = need;
  }
  const int slot = h->w_slot;
  h->w_slot ^= 1;
  CK(cudaEventSynchronize(h->w_ev[slot]));        // the copy that last used this staging buffer (two uploads ago) is long done
  std::memset(h->w_stage[slot], 0, need);
  if (is_tc(h->cfg.net_mode)) {
    // tensor-core blob: fp16 weights in UMMA K-major core-matrix order + fp32 {bias, gamma, beta} per feature
    const cfrb::tc::BlobLayout L(Qp);
    struct { uint8_t* p; uint8_t* data() { return p; } } blob{h->w_stage[slot]};
    __half* hw1 = reinterpret_cast<__half*>(blob.data() + L.off_w1);
    __half* hw2 = reinterpret_cast<__half*>(blob.data() + L.off_w2);
    __half* hw3 = reinterpret_cast<__half*>(blob.data() + L.off_w3);
    // LayerNorm without the mean (leaf_mlp_tc3.cuh).  Subtracting from every column of W (and from the bias) its mean over the
    // 256 output features makes the features of y = W x + b sum to zero for every x, which is all the mean subtraction of
    // LayerNorm does; the epilogue then only needs sum y^2.  Done in double, before the fp16 rounding.
    std::vector<double> m1(Q + 1, 0.0), m2(hid + 1, 0.0);
    for (int k = 0; k < Q; ++k) { for (int j = 0; j < hid; ++j) m1[k] += w1[(size_t)j * Q + k]; m1[k] /= hid; }
    for (int j = 0; j < hid; ++j) m1[Q] += b1[j];
    m1[Q] /= hid;
    for (int k = 0; k < hid; ++k) { for (int j = 0; j < hid; ++j) m2[k] += w2[(size_t)j * hid + k]; m2[k] /= hid; }
    for (int j = 0; j < hid; ++j) m2[hid] += b2[j];
    m2[hid] /= hid;
    for (int j = 0; j < hid; ++j) for (int k = 0; k < Q; ++k) hw1[cfrb::tc::umma_kmajor_offset_halves(j, k, hid)] = __float2half_rn((float)(w1[(size_t)j * Q + k] - m1[k]));
    for (int j = 0; j < hid; ++j) hw1[cfrb::tc::umma_kmajor_offset_halves(j, Q, hid)] = __float2half_rn((float)(b1[j] - m1[Q]));   // bias 1 x constant-1 column
    __half* hones = reinterpret_cast<__half*>(blob.data() + L.off_ones);
    __half* hb2 = reinterpret_cast<__half*>(blob.data() + L.off_bias2);
    for (int r = 0; r < cfrb::tc::kTileM; ++r) hones[cfrb::tc::umma_kmajor_offset_halves(r, 0, cfrb::tc::kTileM)] = __float2half_rn(1.f);
    for (int j = 0; j < hid; ++j) hb2[cfrb::tc::umma_kmajor_offset_halves(j, 0, hid)] = __float2half_rn((float)(b2[j] - m2[hid]));
    for (int j = 0; j < hid; ++j) for (int k = 0; k < hid; ++k) hw2[cfrb::tc::umma_kmajor_offset_halves(j, k, hid)] = __float2half_rn((float)(w2[(size_t)j * hid + k] - m2[k]));
    for (int j = 0; j < H; ++j) for (int k = 0; k < hid; ++k) hw3[cfrb::tc::umma_kmajor_offset_halves(j, k, cfrb::tc::kNout)] = __float2half_rn(w3[(size_t)j * hid + k]);
    float* ln1 = reinterpret_cast<float*>(blob.data() + L.off_ln1);
    float* ln2 = reinterpret_cast<float*>(blob.data() + L.off_ln2);
    // CFRB_NET_TC_F16X2's GELU evaluates the activation from y / 2: gamma / 2 and beta / 2 are stored
    const float lnscale = h->cfg.net_mode == CFRB_NET_TC_F16X2 ? 0.5f : 1.f;
    for (int j = 0; j < hid; ++j) {
      // per feature pair (j even): {gamma_j, gamma_j+1, beta_j, beta_j+1} — the packed operands of the epilogue's fma.f32x2
      const int o = (j >> 1) * 4 + (j & 1);
      ln1[o] = lnscale * g1[j]; ln1[o + 2] = lnscale * be1[j];
      ln2[o] = lnscale * g2[j]; ln2[o + 2] = lnscale * be2[j];
    }
    std::copy(b3, b3 + H, reinterpret_cast<float*>(blob.data() + L.off_b3));
    if (!h->d_blob.p) CK(h->d_blob.alloc(L.blob_bytes));
    CK(cudaMemcpyAsync(h->d_blob.p, blob.data(), L.blob_bytes, cudaMemcpyHostToDevice, h->own_stream));
  } else {
    // transposed k-major fp32 weights for the SIMT kernel
    const size_t total = (size_t)Qp * hid + 3 * hid + (size_t)hid * hid + 3 * hid + (size_t)hid * h->Hout + h->Hout;
    struct { float* p; float& operator[](size_t i) { return p[i]; } float* begin() { return p; } float* data() { return p; } } pk{reinterpret_cast<float*>(h->w_stage[slot])};
    size_t o = 0;
    const size_t o_w1 = o; for (int k = 0; k < Q; ++k) for (int j = 0; j < hid; ++j) pk[o_w1 + (size_t)k * hid + j] = w1[(size_t)j * Q + k];
    o += (size_t)Qp * hid;
    const size_t o_b1 = o; std::copy(b1, b1 + hid, pk.begin() + o); o += hid;
    const size_t o_g1 = o; std::copy(g1, g1 + hid, pk.begin() + o); o += hid;
    const size_t o_be1 = o; std::copy(be1, be1 + hid, pk.begin() + o); o += hid;
    const size_t o_w2 = o; for (int k = 0; k < hid; ++k) for (int j = 0; j < hid; ++j) pk[o_w2 + (size_t)k * hid + j] = w2[(size_t)j * hid + k];
    o += (size_t)hid * hid;
    const size_t o_b2 = o; std::copy(b2, b2 + hid, pk.begin() + o); o += hid;
    const size_t o_g2 = o; std::copy(g2, g2 + hid, pk.begin() + o); o += hid;
    const size_t o_be2 = o; std::copy(be2, be2 + hid, pk.begin() + o); o += hid;
    const size_t o_w3 = o; for (int k = 0; k < hid; ++k) for (int j = 0; j < H; ++j) pk[o_w3 + (size_t)k * h->Hout + j] = w3[(size_t)j * hid + k];
    o += (size_t)hid * h->Hout;
    const size_t o_b3 = o; std::copy(b3, b3 + H, pk.begin() + o);
    if (!h->d_w.p) CK(h->d_w.alloc(total));
    CK(cudaMemcpyAsync(h->d_w.p, pk.data(), total * sizeof(float), cudaMemcpyHostToDevice, h->own_stream));
    cfrb::NetDev& nd = h->net;
    nd.Qpad = Qp; nd.hidden = hid; nd.Hout = h->Hout;
    nd.w1t = h->d_w.p + o_w1; nd.b1 = h->d_w.p + o_b1; nd.g1 = h->d_w.p + o_g1; nd.be1 = h->d_w.p + o_be1;
    nd.w2t = h->d_w.p + o_w2; nd.b2 = h->d_w.p + o_b2; nd.g2 = h->d_w.p + o_g2; nd.be2 = h->d_w.p + o_be2;
    nd.w3t = h->d_w.p + o_w3; nd.b3 = h->d_w.p + o_b3;
  }
  CK(cudaEventRecord(h->w_ev[slot], h->own_stream));
  h->w_last = h->w_ev[slot];
  h->have_weights = true;
  h->weights_version = version;
  return CFRB_OK;
}

uint64_t cfrb_weights_version(const cfrb_handle* h) { return h ? h->weights_version : 0; }

int cfrb_begin_wave(cfrb_handle* h, int32_t n, const int32_t* last_bid, const int32_t* player_id, const double* beliefs,
                    const int32_t* act_iteration) {
  if (!h || (n > 0 && (!last_bid || !player_id || !beliefs))) return fail(CFRB_EINVAL, "null argument");
  if (n < 0 || n > h->cfg.max_subgames) return fail(CFRB_EINVAL, "n exceeds max_subgames");
  CK(cudaSetDevice(h->cfg.device));
  const int H = h->g.H;
  std::vector<int> tm(n), pl(n), ro(n), act(n, -1);
  int rows = 0;
  for (int k = 0; k < n; ++k) {
    if (last_bid[k] < -1 || last_bid[k] > h->g.A - 2) return fail(CFRB_EINVAL, "subgame root bid out of range (terminal or invalid)");
    if (player_id[k] != 0 && player_id[k] != 1) return fail(CFRB_EINVAL, "player_id must be 0 or 1");
    tm[k] = last_bid[k] + 1;
    pl[k] = player_id[k];
    ro[k] = rows;
    rows += h->tmpl[tm[k]].L;
    if (act_iteration) act[k] = act_iteration[k];
  }
  h->n = n; h->rows = rows; h->iters_done = 0; h->rows_on_device = false; h->sp.pending = false;
  h->h_tmpl = tm; h->h_player = pl; h->h_row_off = ro;
  h->h_last_bid.assign(last_bid, last_bid + n);
  h->h_beliefs.assign(beliefs, beliefs + (size_t)n * 2 * H);
  cudaStream_t st = h->own_stream;
  CK(cudaStreamSynchronize(st));
  const int wave[2] = {n, rows};
  CK(cudaMemcpyAsync(h->d_wave.p, wave, sizeof(wave), cudaMemcpyHostToDevice, st));
  if (n) {
    CK(cudaMemcpyAsync(h->d_sg_tmpl.p, tm.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_sg_player.p, pl.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_sg_row_off.p, ro.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_sg_act.p, act.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    int rc = DISPATCH_REAL(h, upload_beliefs_t, h, st);
    if (rc) return rc;
    rc = DISPATCH_REAL(h, launch_init_t, h, st);
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(st));   // host staging vectors above go out of scope
  return CFRB_OK;
}

// Inside a stream capture a plain cudaEventRecord only marks a dependency; cudaEventRecordExternal makes it an event-record
// NODE, whose timestamps can be synchronised on and read after every launch of the graph.
static cudaError_t record_event(cfrb_handle* h, cudaEvent_t ev, cudaStream_t st) {
  return h->capturing ? cudaEventRecordWithFlags(ev, st, cudaEventRecordExternal) : cudaEventRecord(ev, st);
}

static int launch_net(cfrb_handle* h, cudaStream_t st, float* dbg1, float* dbg2) {
  if (h->cfg.net_mode == CFRB_NET_ZERO || (h->rows == 0 && !h->rows_on_device)) return CFRB_OK;
  const bool sample = h->profiling > 0 && (h->net_launch_idx % h->profiling) == 0;
  ++h->net_launch_idx;
  if (sample) {
    while ((int)h->net_ev.size() < h->net_ev_used + 2) {
      cudaEvent_t e;
      CK(cudaEventCreate(&e));
      h->net_ev.push_back(e);
    }
    CK(record_event(h, h->net_ev[h->net_ev_used], st));
  }
  if (is_tc(h->cfg.net_mode)) {
    cfrb::tc::TcArgs a{h->d_blob.p, h->d_Xh.p, h->d_wave.p + 1, h->d_out.p, h->Qpad, h->g.H, h->Hout, dbg1, dbg2, nullptr};
    const int tiles = (h->rows + cfrb::tc::kTileM - 1) / cfrb::tc::kTileM;
    const int grid = (h->capturing || h->rows_on_device) ? h->num_sms : std::min(tiles, h->num_sms);   // surplus CTAs return at once
    const bool x2 = h->cfg.net_mode == CFRB_NET_TC_F16X2;
    a.trace = h->dbg_trace;
    const cfrb::tc::Tc3Layout T3(h->Qpad);
    const bool dbg = dbg1 || dbg2 || a.trace;
    // programmatic dependent launch: the kernel fetches its weights while the CFR kernel before it drains
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(cfrb::tc::kThreads); lc.stream = st;
    lc.dynamicSmemBytes = T3.smem_bytes;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at; lc.numAttrs = dbg ? 0 : 1;
    if (dbg && x2) CK(cudaLaunchKernelEx(&lc, cfrb::tc::leaf_mlp_tc3_kernel<true, 2>, a));
    else if (dbg) CK(cudaLaunchKernelEx(&lc, cfrb::tc::leaf_mlp_tc3_kernel<true, 0>, a));
    else if (x2) CK(cudaLaunchKernelEx(&lc, cfrb::tc::leaf_mlp_tc3_kernel<false, 2>, a));
    else CK(cudaLaunchKernelEx(&lc, cfrb::tc::leaf_mlp_tc3_kernel<false, 0>, a));
  } else {
    // a wave built on the device: worst-case grid, CTAs beyond the device-side row count return at once
    const int64_t rows_host = h->rows_on_device ? (int64_t)h->n * std::max(h->Lmax, 1) : h->rows;
    const int blocks = (int)((rows_host + cfrb::kMlpRows - 1) / cfrb::kMlpRows);
    cfrb::leaf_mlp_fp32_kernel<256><<<blocks, 256, cfrb::leaf_mlp_fp32_smem(256), st>>>(h->net, h->d_X.p, h->d_wave.p + 1, h->d_out.p);
  }
  ++h->launches;
  CK(cudaGetLastError());
  if (sample) {
    CK(record_event(h, h->net_ev[h->net_ev_used + 1], st));
    h->net_ev_used += 2;
  }
  return CFRB_OK;
}

int cfrb_reset_wave(cfrb_handle* h, void* cuda_stream) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  h->iters_done = 0;
  if (h->n == 0) return CFRB_OK;
  return DISPATCH_REAL(h, launch_init_t, h, cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream);
}

int cfrb_set_profiling(cfrb_handle* h, int32_t on) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  h->profiling = on < 0 ? 0 : on;
  return CFRB_OK;
}

static int enqueue_run(cfrb_handle* h, cudaStream_t st, int first, int last) {
  CK(record_event(h, h->ev_a, st));
  h->net_ev_used = 0;
  h->net_launch_idx = 0;
  for (int i = first; i <= last; ++i) {
    const int do_b = i > first, do_f = i < last;
    int rc = DISPATCH_REAL(h, launch_iter_t, h, st, i, do_b, do_f);
    if (rc) return rc;
    if (do_f) { rc = launch_net(h, st, nullptr, nullptr); if (rc) return rc; }
  }
  CK(record_event(h, h->ev_b, st));
  h->net_launches_run = h->net_launch_idx;
  return CFRB_OK;
}

int cfrb_run(cfrb_handle* h, int32_t iters, void* cuda_stream) {
  if (!h || iters < 0) return fail(CFRB_EINVAL, "bad argument");
  if (h->cfg.net_mode != CFRB_NET_ZERO && !h->have_weights && h->Lmax > 0)
    return fail(CFRB_ESTATE, "value-net weights not set (cfrb_set_weights) but the subgame trees have non-final leaves");
  if (h->n == 0 || iters == 0) return CFRB_OK;
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  if (st != h->own_stream && h->w_last) CK(cudaStreamWaitEvent(st, h->w_last, 0));   // weights are uploaded on the handle's own stream
  const int first = h->iters_done, last = first + iters;
  // Long runs are replayed from a CUDA graph: one host call instead of 2 * iters kernel launches, so a busy or slow host
  // thread cannot starve the GPU.  The graph bakes in the iteration indices and a wave-size-independent launch geometry; it
  // is keyed by (first iteration, count, profiling period, "the wave has value-net rows").  The fp32 parity net sizes its grid
  // by the row count and stays on the eager path, like short runs.
  static const bool no_graph = [] { const char* e = std::getenv("CFRB_NO_GRAPH"); return e && *e == '1'; }();
  const bool graphable = !no_graph && iters >= 64 && h->cfg.net_mode != CFRB_NET_FP32;
  if (graphable) {
    const int has_rows = h->rows > 0 || h->rows_on_device;
    cfrb_handle::GraphEntry* g = nullptr;
    for (auto& e : h->graphs)
      if (e.first == first && e.count == iters && e.prof == h->profiling && e.has_rows == has_rows) { g = &e; break; }
    if (!g) {
      // capture + instantiation of ~2 * iters nodes costs ~0.1 s: only worth it for a key that repeats (waves of a self-play
      // loop, bench steps), not for one-off run lengths (e.g. the evaluator's per-chunk act_iteration maxima)
      const std::array<int, 4> key{first, iters, h->profiling, has_rows};
      bool seen = false;
      for (const auto& k : h->graph_seen) seen |= k == key;
      if (!seen) {
        if (h->graph_seen.size() >= 64) h->graph_seen.erase(h->graph_seen.begin());
        h->graph_seen.push_back(key);
      }
      if (seen) {
      if (h->profiling > 0)   // events are created outside the capture
        while ((int)h->net_ev.size() < 2 * (iters / h->profiling + 2)) {
          cudaEvent_t e;
          CK(cudaEventCreate(&e));
          h->net_ev.push_back(e);
        }
      const int64_t l0 = h->launches;
      cudaGraph_t graph = nullptr;
      cudaGraphExec_t exec = nullptr;
      h->capturing = true;
      cudaError_t ce = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
      int rc = CFRB_OK;
      if (ce == cudaSuccess) {
        rc = enqueue_run(h, st, first, last);
        ce = cudaStreamEndCapture(st, &graph);
        if (rc == CFRB_OK && ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
      }
      h->capturing = false;
      const int captured = (int)(h->launches - l0);
      h->launches = l0;
      if (rc == CFRB_OK && ce == cudaSuccess && exec) {
        if (h->graphs.size() >= 8) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
        h->graphs.push_back({first, iters, h->profiling, has_rows, exec, captured, h->net_launches_run, h->net_ev_used});
        g = &h->graphs.back();
      } else {
        cudaGetLastError();   // the stream could not be captured (e.g. a legacy stream): run eagerly
      }
      }
    }
    if (g) {
      CK(cudaGraphLaunch(g->exec, st));
      h->launches += g->launches;
      h->net_launches_run = g->net_launches;
      h->net_ev_used = g->ev_used;
      h->iters_done = last;
      return CFRB_OK;
    }
  }
  int rc = enqueue_run(h, st, first, last);
  if (rc) return rc;
  h->iters_done = last;
  return CFRB_OK;
}

int cfrb_sync(cfrb_handle* h) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  return CFRB_OK;
}

int cfrb_iterations_done(const cfrb_handle* h) { return h ? h->iters_done : 0; }

int cfrb_fetch(cfrb_handle* h, double* root_value_means, double* snapshot_strategy, double* last_strategy, double* avg_strategy,
               double* sum_strategy, double* regrets) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  { int rc = sync_mirror(h); if (rc) return rc; }
  if (h->n == 0) return CFRB_OK;
  return DISPATCH_REAL(h, fetch_t, h, root_value_means, snapshot_strategy, last_strategy, avg_strategy, sum_strategy, regrets);
}

int cfrb_table_stride(const cfrb_handle* h) { return h ? h->table_stride : 0; }

int cfrb_fetch_compact(cfrb_handle* h, int32_t which, double* out) {
  if (!h || !out || which < 0 || which > 4) return fail(CFRB_EINVAL, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  { int rc = sync_mirror(h); if (rc) return rc; }
  if (h->n == 0) return CFRB_OK;
  return DISPATCH_REAL(h, fetch_compact_t, h, which, out);
}

int cfrb_examples(cfrb_handle* h, float* queries, float* values) {
  if (!h || !queries || !values) return fail(CFRB_EINVAL, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  { int rc = sync_mirror(h); if (rc) return rc; }
  const int n = h->n, H = h->g.H, A = h->g.A, Q = h->g.Q;
  if (n == 0) return CFRB_OK;
  int rc = DISPATCH_REAL(h, examples_values_t, h, values);
  if (rc) return rc;
  // query of node 0 as seen by traverser t (write_query_to, subgame_solving.cc:104-123); root reach == beliefs
  for (int k = 0; k < n; ++k) {
    const double* b = h->h_beliefs.data() + (size_t)k * 2 * H;
    for (int t = 0; t < 2; ++t) {
      float* q = queries + ((size_t)k * 2 + t) * Q;
      q[0] = (float)h->h_player[k];
      q[1] = (float)t;
      for (int a = 0; a < A; ++a) q[2 + a] = (a == h->h_last_bid[k]) ? 1.f : 0.f;
      for (int p = 0; p < 2; ++p) {
        double s = 0;
        for (int hd = 0; hd < H; ++hd) s += b[p * H + hd] + 1e-80;
        for (int hd = 0; hd < H; ++hd) q[2 + A + p * H + hd] = (float)((b[p * H + hd] + 1e-80) / s);
      }
    }
  }
  return CFRB_OK;
}

int cfrb_load_state(cfrb_handle* h, const double* regrets, const double* last_strategy, const double* sum_strategy,
                    const double* root_value_means, const int32_t* num_steps, int32_t iterations_done) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  { int rc = sync_mirror(h); if (rc) return rc; }
  int rc = DISPATCH_REAL(h, load_state_t, h, regrets, last_strategy, sum_strategy, root_value_means);
  if (rc) return rc;
  if (num_steps) CK(cudaMemcpy(h->d_steps.p, num_steps, (size_t)h->n * 2 * sizeof(int), cudaMemcpyHostToDevice));
  h->iters_done = iterations_done;
  return CFRB_OK;
}

int cfrb_debug_leaf_io(cfrb_handle* h, float* queries, float* net_out, double* scalers, int32_t cap_rows) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  { int rc = sync_mirror(h); if (rc) return rc; }
  const int rows = std::min<int>(h->rows, cap_rows), Q = h->g.Q;
  if (rows > 0 && queries && is_tc(h->cfg.net_mode)) {
    const int tiles = (rows + cfrb::tc::kTileM - 1) / cfrb::tc::kTileM;
    std::vector<__half> x((size_t)tiles * cfrb::tc::kTileM * h->Qpad);
    CK(cudaMemcpy(x.data(), h->d_Xh.p, x.size() * sizeof(__half), cudaMemcpyDeviceToHost));
    for (int r = 0; r < rows; ++r)
      for (int q = 0; q < Q; ++q)
        queries[(size_t)r * Q + q] = __half2float(x[(size_t)(r >> 7) * cfrb::tc::kTileM * h->Qpad +
                                                    cfrb::tc::umma_kmajor_offset_halves(r & 127, q, cfrb::tc::kTileM)]);
  } else if (rows > 0 && queries && h->cfg.net_mode == CFRB_NET_FP32) {
    std::vector<float> x((size_t)rows * h->Qpad);
    CK(cudaMemcpy(x.data(), h->d_X.p, x.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int r = 0; r < rows; ++r) std::memcpy(queries + (size_t)r * Q, x.data() + (size_t)r * h->Qpad, Q * sizeof(float));
  }
  if (rows > 0 && net_out) {
    std::vector<float> o((size_t)rows * h->Hout);
    CK(cudaMemcpy(o.data(), h->d_out.p, o.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int r = 0; r < rows; ++r) std::memcpy(net_out + (size_t)r * h->g.H, o.data() + (size_t)r * h->Hout, h->g.H * sizeof(float));
  }
  if (rows > 0 && scalers) {
    int rc = DISPATCH_REAL(h, scalers_t, h, scalers, rows);
    if (rc) return rc;
  }
  return h->rows;
}

int cfrb_debug_net_trace(cfrb_handle* h, long long* out, int n) {
  if (!h || !is_tc(h->cfg.net_mode)) return fail(CFRB_EINVAL, "trace exists only for the tensor-core value net");
  if (!h->have_weights || h->rows == 0) return fail(CFRB_ESTATE, "no weights or no leaf rows");
  if (n < 2048) return fail(CFRB_EINVAL, "trace buffer must hold 2048 stamps");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  long long* d = nullptr;
  CK(cudaMalloc(&d, 2048 * sizeof(long long)));
  CK(cudaMemset(d, 0, 2048 * sizeof(long long)));
  const int prof = h->profiling;
  h->profiling = 0;
  h->dbg_trace = d;
  int rc = launch_net(h, h->own_stream, nullptr, nullptr);
  h->dbg_trace = nullptr;
  h->profiling = prof;
  if (!rc && cudaStreamSynchronize(h->own_stream) != cudaSuccess) rc = fail(CFRB_ECUDA, "trace launch failed");
  if (!rc) cudaMemcpy(out, d, 2048 * sizeof(long long), cudaMemcpyDeviceToHost);
  cudaFree(d);
  return rc;
}

int cfrb_debug_net_taps(cfrb_handle* h, float* d1, float* d2) {
  if (!h || !is_tc(h->cfg.net_mode)) return fail(CFRB_EINVAL, "taps exist only for CFRB_NET_TC_F16");
  if (!h->have_weights || h->rows == 0) return fail(CFRB_ESTATE, "no weights or no leaf rows");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  const size_t n = (size_t)cfrb::tc::kTileM * cfrb::tc::kHid;
  const int prof = h->profiling;
  h->profiling = 0;
  int rc = launch_net(h, h->own_stream, h->d_dbg.p, h->d_dbg.p + n);
  h->profiling = prof;
  if (rc) return rc;
  CK(cudaStreamSynchronize(h->own_stream));
  if (d1) CK(cudaMemcpy(d1, h->d_dbg.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (d2) CK(cudaMemcpy(d2, h->d_dbg.p + n, n * sizeof(float), cudaMemcpyDeviceToHost));
  return CFRB_OK;
}

int cfrb_exploitability(cfrb_handle* h, const double* full_strategy, double* out2) {
  if (!h || !full_strategy || !out2) return fail(CFRB_EINVAL, "cfrb_exploitability: null argument");
  CK(cudaSetDevice(h->cfg.device));
  auto& b = h->br;
  const auto& g = h->g;
  if (!b.ready) {
    if (g.A > 26) return fail(CFRB_EINVAL, "cfrb_exploitability: full tree too large (2^A - 1 nodes)");
    b.t = cfrb::build_template(g, -1, 1 << 30);
    const auto& t = b.t;
    std::vector<int> term(t.term_node.begin(), t.term_node.end());
    for (int n : t.term_node) term.push_back(t.last_bid[t.parent[n]]);   // challenged bid (:287)
    for (int n : t.term_node) term.push_back(t.depth[n]);
    auto up = [&](auto& buf, const auto& v) -> cudaError_t {
      cudaError_t e = buf.alloc(v.size());
      if (e != cudaSuccess) return e;
      return cudaMemcpy(buf.p, v.data(), v.size() * sizeof(v[0]), cudaMemcpyHostToDevice);
    };
    CK(up(b.parent, t.parent)); CK(up(b.child_begin, t.child_begin)); CK(up(b.nchild, t.nchild));
    CK(up(b.level_begin, t.level_begin)); CK(up(b.term_node, term));
    b.scratch_stride = (size_t)3 * t.N * g.H + (size_t)10 * std::max(t.T, 1);
    CK(b.scratch.alloc(2 * b.scratch_stride));
    CK(b.strategy.alloc((size_t)std::max(t.N - 1, 1) * g.H));
    CK(b.out.alloc(2));
    b.ready = true;
  }
  const auto& t = b.t;
  // dense [n][h][a] -> compact [edge = child - 1][h]
  std::vector<double> compact((size_t)std::max(t.N - 1, 1) * g.H, 0.0);
  for (int n = 0; n < t.N; ++n)
    for (int j = 0; j < t.nchild[n]; ++j)
      for (int hd = 0; hd < g.H; ++hd)
        compact[(size_t)(t.child_begin[n] + j - 1) * g.H + hd] = full_strategy[((size_t)n * g.H + hd) * g.A + t.act_lo[n] + j];
  CK(cudaMemcpyAsync(b.strategy.p, compact.data(), compact.size() * sizeof(double), cudaMemcpyHostToDevice, h->own_stream));
  cfrb::BrDev d{};
  d.N = t.N; d.T = t.T; d.levels = t.levels; d.H = g.H; d.F = g.F;
  d.parent = b.parent.p; d.child_begin = b.child_begin.p; d.nchild = b.nchild.p; d.level_begin = b.level_begin.p;
  d.term_node = b.term_node.p; d.matches = h->d_matches.p; d.strategy = b.strategy.p;
  d.scratch = b.scratch.p; d.scratch_stride = b.scratch_stride; d.out = b.out.p;
  cfrb::br_launch(d, h->own_stream);
  ++h->launches;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out2, b.out.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->own_stream));
  CK(cudaStreamSynchronize(h->own_stream));
  return CFRB_OK;
}

int64_t cfrb_kernel_launches(const cfrb_handle* h) { return h ? h->launches : 0; }
int64_t cfrb_wave_leaf_rows(const cfrb_handle* h) {
  if (!h) return 0;
  if (h->rows_on_device && h->mirror_stale) {   // a wave built on the device: the count lives there
    int wave[2] = {0, 0};
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    if (cudaMemcpy(wave, h->d_wave.p, sizeof(wave), cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return -1; }
    return wave[1];
  }
  return h->rows;
}

// Timing marks: CUDA events recorded on the launching stream (NULL = the handle's stream); elapsed device time between two.
int cfrb_mark(cfrb_handle* h, int32_t slot, void* cuda_stream) {
  if (!h || slot < 0 || slot >= 8) return fail(CFRB_EINVAL, "cfrb_mark: slot must be in [0, 8)");
  CK(cudaSetDevice(h->cfg.device));
  if (!h->marks[slot]) CK(cudaEventCreate(&h->marks[slot]));
  CK(cudaEventRecord(h->marks[slot], cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream));
  return CFRB_OK;
}
int cfrb_mark_wait(cfrb_handle* h, int32_t slot) {
  if (!h || slot < 0 || slot >= 8 || !h->marks[slot]) return fail(CFRB_EINVAL, "cfrb_mark_wait: mark not recorded");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->marks[slot]));
  return CFRB_OK;
}
void* cfrb_handle_stream(cfrb_handle* h) { return h ? (void*)h->own_stream : nullptr; }
int cfrb_mark_elapsed_ms(cfrb_handle* h, int32_t a, int32_t b, float* ms) {
  if (!h || !ms || a < 0 || a >= 8 || b < 0 || b >= 8 || !h->marks[a] || !h->marks[b]) return fail(CFRB_EINVAL, "cfrb_mark_elapsed_ms: bad marks");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->marks[b]));
  CK(cudaEventElapsedTime(ms, h->marks[a], h->marks[b]));
  return CFRB_OK;
}
// Evict the L2 cache: overwrite a scratch buffer of `bytes` (> 126 MB) on the stream, for benchmarks' timed loops.
int cfrb_l2_flush(cfrb_handle* h, size_t bytes, void* cuda_stream) {
  if (!h || bytes == 0) return fail(CFRB_EINVAL, "cfrb_l2_flush: bad argument");
  CK(cudaSetDevice(h->cfg.device));
  if (h->flush_bytes < bytes) {
    if (h->flush_buf) cudaFree(h->flush_buf);
    h->flush_buf = nullptr; h->flush_bytes = 0;
    CK(cudaMalloc(&h->flush_buf, bytes));
    h->flush_bytes = bytes;
  }
  CK(cudaMemsetAsync(h->flush_buf, 1, bytes, cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream));
  return CFRB_OK;
}

int cfrb_last_run_ms(cfrb_handle* h, float* total_ms, float* net_ms) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->ev_b));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, h->ev_a, h->ev_b));
  h->last_total_ms = ms;
  float net = 0.f;
  for (int i = 0; i + 1 < h->net_ev_used; i += 2) {
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, h->net_ev[i], h->net_ev[i + 1]));
    net += t;
  }
  // sampled launches -> estimate for all value-net launches of the run
  if (h->net_ev_used > 0) net = net / (h->net_ev_used / 2) * h->net_launches_run;
  h->last_net_ms = net;
  if (total_ms) *total_ms = ms;
  if (net_ms) *net_ms = net;
  return CFRB_OK;
}

// ============================================================================================ device-resident self-play
int cfrb_selfplay_create(cfrb_handle* h, int32_t n_games, const uint32_t* seeds, float random_action_prob, int32_t sample_leaf) {
  if (!h || !seeds) return fail(CFRB_EINVAL, "null argument");
  if (n_games < 1 || n_games > h->cfg.max_subgames) return fail(CFRB_EINVAL, "n_games must be in [1, max_subgames]");
  if (h->g.H > cfrb::kSpMaxH) return fail(CFRB_EINVAL, "device self-play supports num_hands <= 64");
  if (h->cfg.max_depth > cfrb::kSpMaxPath) return fail(CFRB_EINVAL, "device self-play supports max_depth <= 16");
  CK(cudaSetDevice(h->cfg.device));
  auto& sp = h->sp;
  const int K = n_games, H = h->g.H;
  sp.last_bid.release(); sp.player.release(); sp.mt_idx.release(); sp.beliefs.release(); sp.mt.release(); sp.seeds.release();
  CK(sp.last_bid.alloc(K)); CK(sp.player.alloc(K)); CK(sp.mt_idx.alloc(K)); CK(sp.beliefs.alloc((size_t)K * 2 * H));
  CK(sp.mt.alloc((size_t)624 * K)); CK(sp.seeds.alloc(K));
  cfrb::SpDev& d = sp.dev;
  d.K = K; d.A = h->g.A; d.H = H; d.Q = h->g.Q; d.iters = h->cfg.num_iters; d.sample_leaf = sample_leaf;
  d.random_action_prob = random_action_prob;
  d.g_last_bid = sp.last_bid.p; d.g_player = sp.player.p; d.g_beliefs = sp.beliefs.p; d.mt = sp.mt.p; d.mt_idx = sp.mt_idx.p;
  d.tmpl = h->d_tmpl.p; d.child_begin = h->d_child_begin.p; d.nchild = h->d_nchild.p; d.last_bid = h->d_last_bid.p;
  d.wave = h->d_wave.p; d.sg_tmpl = h->d_sg_tmpl.p; d.sg_player = h->d_sg_player.p; d.sg_row_off = h->d_sg_row_off.p;
  d.sg_act = h->d_sg_act.p; d.table_stride = h->table_stride;
  CK(cudaStreamSynchronize(h->own_stream));
  CK(cudaMemcpyAsync(sp.seeds.p, seeds, (size_t)K * sizeof(uint32_t), cudaMemcpyHostToDevice, h->own_stream));
  cfrb::sp_launch_seed(d, sp.seeds.p, h->own_stream);
  ++h->launches;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->own_stream));
  if (!sp.ev_examples) CK(cudaEventCreateWithFlags(&sp.ev_examples, cudaEventDisableTiming));
  sp.K = K; sp.ready = true; sp.pending = false; sp.waves = 0; sp.ev_recorded = false;
  return CFRB_OK;
}

int cfrb_selfplay_wave(cfrb_handle* h, float* dev_ex_q, float* dev_ex_v, int32_t start_next, void* cuda_stream) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  if (!h->sp.ready) return fail(CFRB_ESTATE, "cfrb_selfplay_create has not been called");
  if ((dev_ex_q == nullptr) != (dev_ex_v == nullptr)) return fail(CFRB_EINVAL, "example buffers: both or none");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  int rows_out = 0;
  if (h->sp.pending) {
    if (!h->rows_on_device || h->n != h->sp.K || h->iters_done != h->cfg.num_iters)
      return fail(CFRB_ESTATE, "the pending self-play wave was replaced or not run to num_iters");
    int rc = DISPATCH_REAL(h, selfplay_finish_t, h, dev_ex_q, dev_ex_v, st);
    if (rc) return rc;
    h->sp.pending = false;
    rows_out = dev_ex_q ? 2 * h->sp.K : 0;
    CK(cudaEventRecord(h->sp.ev_examples, st));
    h->sp.ev_recorded = true;
  }
  if (start_next) {
    int rc = DISPATCH_REAL(h, selfplay_begin_t, h, st);
    if (rc) return rc;
    h->n = h->sp.K; h->rows = 0; h->rows_on_device = true; h->mirror_stale = true; h->iters_done = 0;
    rc = DISPATCH_REAL(h, launch_init_t, h, st);
    if (rc) return rc;
    rc = cfrb_run(h, h->cfg.num_iters, st);
    if (rc) return rc;
    h->sp.pending = true;
    ++h->sp.waves;
  }
  return rows_out;
}

int cfrb_selfplay_wait_examples(cfrb_handle* h) {
  if (!h || !h->sp.ready) return fail(CFRB_ESTATE, "no self-play session");
  if (!h->sp.ev_recorded) return CFRB_OK;
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->sp.ev_examples));
  return CFRB_OK;
}

int cfrb_selfplay_state(cfrb_handle* h, int32_t* last_bid, int32_t* player, double* beliefs) {
  if (!h || !h->sp.ready) return fail(CFRB_ESTATE, "no self-play session");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  const int K = h->sp.K;
  if (last_bid) CK(cudaMemcpy(last_bid, h->sp.last_bid.p, K * sizeof(int), cudaMemcpyDeviceToHost));
  if (player) CK(cudaMemcpy(player, h->sp.player.p, K * sizeof(int), cudaMemcpyDeviceToHost));
  if (beliefs) CK(cudaMemcpy(beliefs, h->sp.beliefs.p, (size_t)K * 2 * h->g.H * sizeof(double), cudaMemcpyDeviceToHost));
  return K;
}

// Roots of the current wave (inspection; pulls the descriptors of a device-built wave).  Returns the number of subgames.
int cfrb_wave_roots(cfrb_handle* h, int32_t* last_bid, int32_t* player_id, int32_t cap) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  { int rc = sync_mirror(h); if (rc) return rc; }
  for (int k = 0; k < h->n && k < cap; ++k) {
    if (last_bid) last_bid[k] = h->h_last_bid[k];
    if (player_id) player_id[k] = h->h_player[k];
  }
  return h->n;
}

// Development / test aid: div_by_rcp (reciprocal + two fused-multiply-add corrections, cfr_kernels.cuh) against IEEE division on
// `blocks` x 256 x 4096 pseudo-random operand pairs; *mismatches receives the number of differing quotients.
int cfrb_debug_div_check(cfrb_handle* h, uint64_t seed, int32_t blocks, uint64_t* mismatches) {
  if (!h || !mismatches || blocks < 1) return fail(CFRB_EINVAL, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  unsigned long long* d = nullptr;
  CK(cudaMalloc((void**)&d, sizeof(unsigned long long)));
  CK(cudaMemset(d, 0, sizeof(unsigned long long)));
  cfrb::div_check_launch(seed, blocks, d, h->own_stream);
  cudaError_t e = cudaStreamSynchronize(h->own_stream);
  unsigned long long out = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&out, d, sizeof(out), cudaMemcpyDeviceToHost);
  cudaFree(d);
  CK(e);
  *mismatches = out;
  return CFRB_OK;
}

// Development / test aid: the value-net GELU of CFRB_NET_TC_F16X2 and a packed-fp16 evaluation of the same function, for every
// fp16 input.  what = 0: tanh.approx.f16x2 itself; 1: gelu_hy_x2, 2: gelu_hy_t32 (leaf_mlp_tc3.cuh), each with hy = the input.
// out[i] = fp16 bits of f(fp16 with bits i).
namespace {
// GELU(y) for a packed pair given hy = y / 2, in fp16 arithmetic: hy + hy * tanh(hy (c0 + c1 hy^2 + c2 hy^4)) with HFMA2 and one
// tanh.approx.f16x2 per pair, the coefficients and the clamp of gelu_hy_t32.  Not used by the value net: tanh.approx.f16x2
// truncates towards zero, which biases every activation with |y| > 0.5 by -1.6e-4 .. -3.9e-4 and shifts the self-play
// statistics.  It stays as the reference that the bias test and the arithmetic model of the reference harness compare against.
__device__ __forceinline__ uint32_t gelu_hy_x2(float hy0, float hy1) {
  const __half2 hy = __floats2half2_rn(hy0, hy1);
  const __half2 s = __hmin2(__hmul2(hy, hy), __float2half2_rn(13.f));
  const __half2 p = __hfma2(s, __hfma2(s, __float2half2_rn(-1.124832e-2f), __float2half2_rn(2.960456e-1f)), __float2half2_rn(1.594992f));
  const __half2 u = __hmul2(hy, p);
  uint32_t t;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(t) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
  const __half2 g = __hfma2(hy, *reinterpret_cast<const __half2*>(&t), hy);
  return *reinterpret_cast<const uint32_t*>(&g);
}

__global__ void gelu_table_kernel(int what, unsigned short* out) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 65536u) return;
  const __half x = __ushort_as_half((unsigned short)i);
  unsigned short r;
  if (what == 0) {
    const __half2 u = __halves2half2(x, x);
    uint32_t t;
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(t) : "r"(*reinterpret_cast<const uint32_t*>(&u)));
    r = (unsigned short)(t & 0xffffu);
  } else {
    const float f = __half2float(x);
    r = (unsigned short)((what == 1 ? gelu_hy_x2(f, f) : cfrb::tc::gelu_hy_t32(f, f)) & 0xffffu);
  }
  out[i] = r;
}
}  // namespace
int cfrb_debug_gelu_table(cfrb_handle* h, int32_t what, uint16_t* out) {
  if (!h || !out || what < 0 || what > 2) return fail(CFRB_EINVAL, "bad argument");
  CK(cudaSetDevice(h->cfg.device));
  unsigned short* d = nullptr;
  CK(cudaMalloc((void**)&d, 65536 * sizeof(unsigned short)));
  gelu_table_kernel<<<256, 256, 0, h->own_stream>>>(what, d);
  cudaError_t e = cudaStreamSynchronize(h->own_stream);
  if (e == cudaSuccess) e = cudaMemcpy(out, d, 65536 * sizeof(unsigned short), cudaMemcpyDeviceToHost);
  cudaFree(d);
  CK(e);
  return CFRB_OK;
}

int cfrb_stream_wait(cfrb_handle* h, void* cuda_stream) {
  if (!h) return fail(CFRB_EINVAL, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaStreamSynchronize(cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream));
  return CFRB_OK;
}

// ============================================================================================ device-resident example rows
struct cfrb_rows {
  int device = 0, q_dim = 0, v_dim = 0;
  int64_t cap = 0;
  float* q = nullptr; float* v = nullptr;
  // id staging for gathers (a small ring: a gather on the consumer's stream is not waited for, its staging slot is reused only
  // after its completion event) and the staging area for batches that leave the device
  struct IdSlot { int* dev = nullptr; int* pin = nullptr; int cap = 0; cudaEvent_t done = nullptr; bool used = false; };
  IdSlot ids[4];
  int next_id = 0;
  float* stage_q = nullptr; float* stage_v = nullptr; int64_t stage_rows = 0;
  cudaStream_t st = nullptr;
};

int cfrb_rows_destroy(cfrb_rows* r) {
  if (!r) return CFRB_OK;
  cudaSetDevice(r->device);
  cudaDeviceSynchronize();
  if (r->st) cudaStreamDestroy(r->st);
  if (r->q) cudaFree(r->q);
  if (r->v) cudaFree(r->v);
  for (auto& s : r->ids) {
    if (s.dev) cudaFree(s.dev);
    if (s.pin) cudaFreeHost(s.pin);
    if (s.done) cudaEventDestroy(s.done);
  }
  if (r->stage_q) cudaFree(r->stage_q);
  if (r->stage_v) cudaFree(r->stage_v);
  delete r;
  return CFRB_OK;
}

int cfrb_rows_create(int32_t device, int64_t capacity_rows, int32_t q_dim, int32_t v_dim, cfrb_rows** out) {
  if (!out || capacity_rows < 1 || q_dim < 1 || v_dim < 1) return fail(CFRB_EINVAL, "bad argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(CFRB_ENODEV, "no CUDA device"); }
  if (device < 0 || device >= ndev) return fail(CFRB_EINVAL, "device ordinal out of range");
  CK(cudaSetDevice(device));
  auto* r = new cfrb_rows();
  r->device = device; r->q_dim = q_dim; r->v_dim = v_dim; r->cap = capacity_rows;
  cudaError_t e = cudaMalloc((void**)&r->q, (size_t)capacity_rows * q_dim * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void**)&r->v, (size_t)capacity_rows * v_dim * sizeof(float));
  // Highest stream priority: the store's gathers and copies run next to a generator that keeps every SM busy with back-to-back
  // (programmatically chained) kernels; at equal priority their blocks waited tens of milliseconds for a slot (measured: 47 ms for a
  // 32 768-row sample, whatever its size), at high priority they take the next slot a retiring CTA frees.
  int prio_least = 0, prio_greatest = 0;
  if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&r->st, cudaStreamNonBlocking, prio_greatest);
  // gather scratch (row-id slots, staging rows of host-bound batches) for batches of up to min(capacity, 262 144) rows, allocated
  // HERE: an allocation later, next to a generator that keeps the GPU busy with whole waves, waits for the end of a wave (measured:
  // 47 ms per sample while the four slots were being created one call at a time)
  const int64_t scratch_rows = std::min<int64_t>(capacity_rows, 1 << 18);
  for (auto& s : r->ids) {
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s.dev, (size_t)scratch_rows * sizeof(int));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&s.pin, (size_t)scratch_rows * sizeof(int));
    if (e == cudaSuccess) s.cap = (int)scratch_rows;
  }
  if (e == cudaSuccess) e = cudaMalloc((void**)&r->stage_q, (size_t)scratch_rows * q_dim * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc((void**)&r->stage_v, (size_t)scratch_rows * v_dim * sizeof(float));
  if (e == cudaSuccess) r->stage_rows = (int)scratch_rows;
  if (e != cudaSuccess) {
    cfrb_rows_destroy(r);
    return fail(CFRB_ENOMEM, std::string("cfrb_rows_create: ") + cudaGetErrorString(e));
  }
  *out = r;
  return CFRB_OK;
}

int cfrb_rows_device(const cfrb_rows* r) { return r ? r->device : -1; }

// kind: 0 = host source, 1 = device source on `src_device` (peer copy when that is another GPU).  Ring wrap-around handled
// here.  Ordered after every gather still in flight on a consumer's stream (it may read the slots being replaced); blocks until
// the rows are in place (the caller publishes them right after).
int cfrb_rows_write(cfrb_rows* r, int64_t slot, int32_t n, const float* q, const float* v, int32_t kind, int32_t src_device) {
  if (!r || !q || !v || n < 0 || slot < 0 || slot >= r->cap || n > r->cap) return fail(CFRB_EINVAL, "cfrb_rows_write: bad argument");
  CK(cudaSetDevice(r->device));
  for (auto& s : r->ids)
    if (s.used) CK(cudaStreamWaitEvent(r->st, s.done, 0));
  auto put = [&](float* dst_base, const float* src, int dim) -> cudaError_t {
    const int64_t first = std::min<int64_t>(n, r->cap - slot);
    for (int part = 0; part < 2; ++part) {
      const int64_t cnt = part == 0 ? first : n - first;
      if (cnt <= 0) continue;
      float* dst = dst_base + (size_t)(part == 0 ? slot : 0) * dim;
      const float* s2 = src + (size_t)(part == 0 ? 0 : first) * dim;
      const size_t bytes = (size_t)cnt * dim * sizeof(float);
      cudaError_t e;
      if (kind == 0) e = cudaMemcpyAsync(dst, s2, bytes, cudaMemcpyHostToDevice, r->st);
      else if (src_device == r->device) e = cudaMemcpyAsync(dst, s2, bytes, cudaMemcpyDeviceToDevice, r->st);
      else e = cudaMemcpyPeerAsync(dst, r->device, s2, src_device, bytes, r->st);
      if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
  };
  CK(put(r->q, q, r->q_dim));
  CK(put(r->v, v, r->v_dim));
  CK(cudaStreamSynchronize(r->st));
  return CFRB_OK;
}

int cfrb_rows_read(cfrb_rows* r, int64_t slot, int32_t n, float* q, float* v) {
  if (!r || !q || !v || n < 0 || slot < 0 || slot >= r->cap || n > r->cap) return fail(CFRB_EINVAL, "cfrb_rows_read: bad argument");
  CK(cudaSetDevice(r->device));
  const int64_t first = std::min<int64_t>(n, r->cap - slot);
  CK(cudaMemcpy(q, r->q + (size_t)slot * r->q_dim, (size_t)first * r->q_dim * sizeof(float), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(v, r->v + (size_t)slot * r->v_dim, (size_t)first * r->v_dim * sizeof(float), cudaMemcpyDeviceToHost));
  if (n > first) {
    CK(cudaMemcpy(q + (size_t)first * r->q_dim, r->q, (size_t)(n - first) * r->q_dim * sizeof(float), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(v + (size_t)first * r->v_dim, r->v, (size_t)(n - first) * r->v_dim * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return CFRB_OK;
}

// Rows ids[0..n) -> out_q [n][q_dim], out_v [n][v_dim].  out_device: -1 = host memory, otherwise the CUDA ordinal the output
// buffers live on.  When the output is on the ring's device and a stream is given, the id upload and the two gather kernels are
// enqueued on THAT stream (the consumer's: the batch is ordered like any other work of the trainer) and the call returns
// without waiting; otherwise the batch is staged on the ring's device, copied out and the call waits for it.
int cfrb_rows_gather(cfrb_rows* r, const int32_t* ids, int32_t n, float* out_q, float* out_v, int32_t out_device, void* cuda_stream) {
  if (!r || !ids || !out_q || !out_v || n < 0) return fail(CFRB_EINVAL, "cfrb_rows_gather: bad argument");
  if (n == 0) return CFRB_OK;
  CK(cudaSetDevice(r->device));
  if (n > r->ids[0].cap) {
    // grow ALL id slots at once (cfrb_rows_create sized them for min(capacity, 262 144) rows, so this is rare): allocations
    // synchronise with the device, and next to a generator that keeps the GPU busy with whole waves each one waits for the end of a wave
    const int cap = 2 * n;
    for (auto& s : r->ids) {
      if (s.used) CK(cudaEventSynchronize(s.done));
      if (s.dev) cudaFree(s.dev);
      if (s.pin) cudaFreeHost(s.pin);
      s.dev = nullptr; s.pin = nullptr; s.cap = 0; s.used = false;
      CK(cudaMalloc((void**)&s.dev, (size_t)cap * sizeof(int)));
      CK(cudaMallocHost((void**)&s.pin, (size_t)cap * sizeof(int)));
      s.cap = cap;
    }
  }
  auto& sl = r->ids[r->next_id];
  r->next_id = (r->next_id + 1) % 4;
  if (sl.used) CK(cudaEventSynchronize(sl.done));
  for (int i = 0; i < n; ++i) {
    if (ids[i] < 0 || ids[i] >= r->cap) return fail(CFRB_EINVAL, "cfrb_rows_gather: row id out of range");
    sl.pin[i] = ids[i];
  }
  const bool same = out_device == r->device;
  const bool direct = same && cuda_stream != nullptr;
  cudaStream_t st = direct ? (cudaStream_t)cuda_stream : r->st;
  CK(cudaMemcpyAsync(sl.dev, sl.pin, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st));
  float* tq = out_q; float* tv = out_v;
  if (!same) {
    if (n > r->stage_rows) {
      CK(cudaStreamSynchronize(r->st));
      if (r->stage_q) cudaFree(r->stage_q);
      if (r->stage_v) cudaFree(r->stage_v);
      r->stage_q = r->stage_v = nullptr; r->stage_rows = 0;
      const int rows = 2 * n;
      CK(cudaMalloc((void**)&r->stage_q, (size_t)rows * r->q_dim * sizeof(float)));
      CK(cudaMalloc((void**)&r->stage_v, (size_t)rows * r->v_dim * sizeof(float)));
      r->stage_rows = rows;
    }
    tq = r->stage_q; tv = r->stage_v;
  }
  cfrb::rows_launch_gather(r->q, r->q_dim, sl.dev, n, tq, st);
  cfrb::rows_launch_gather(r->v, r->v_dim, sl.dev, n, tv, st);
  CK(cudaGetLastError());
  if (!same) {
    const size_t bq = (size_t)n * r->q_dim * sizeof(float), bv = (size_t)n * r->v_dim * sizeof(float);
    if (out_device < 0) {
      CK(cudaMemcpyAsync(out_q, tq, bq, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(out_v, tv, bv, cudaMemcpyDeviceToHost, st));
    } else {
      CK(cudaMemcpyPeerAsync(out_q, out_device, tq, r->device, bq, st));
      CK(cudaMemcpyPeerAsync(out_v, out_device, tv, r->device, bv, st));
    }
  }
  CK(cudaEventRecord(sl.done, st));
  sl.used = true;
  if (!direct) CK(cudaStreamSynchronize(st));
  return CFRB_OK;
}

// Scratch device buffers for hand-over between a generator handle and a row store (examples of one wave).
int cfrb_dev_alloc(int32_t device, size_t bytes, void** out) {
  if (!out) return fail(CFRB_EINVAL, "null argument");
  CK(cudaSetDevice(device));
  CK(cudaMalloc(out, std::max<size_t>(bytes, 1)));
  return CFRB_OK;
}
int cfrb_dev_free(int32_t device, void* p) {
  if (!p) return CFRB_OK;
  CK(cudaSetDevice(device));
  CK(cudaFree(p));
  return CFRB_OK;
}
int cfrb_dev_to_host(int32_t device, void* dst, const void* src, size_t bytes) {
  CK(cudaSetDevice(device));
  CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return CFRB_OK;
}

}  // extern "C"

// ============================================================================================ NCCL (one process per GPU)
// The reference is a single process: generator threads share the trainer's model replicas and its host-memory replay.  With
// one process per GPU the two hand-overs become collectives over NVLink, issued from THIS library on device buffers:
//   ModelLocker::updateModel (rela/model_locker.h:69-79)      -> ncclBroadcast of the flat weight buffer from the trainer's rank
//   PrioritizedReplay::add   (rela/prioritized_replay.h:247-261) -> grouped ncclSend / ncclRecv of every rank's example rows
//                                                                   into the trainer rank's device-resident replay rows
//   recursive_eval's accumulation (recursive_eval.cc:343-363) -> ncclReduce(sum) of the float32 accumulators
#include <nccl.h>

struct cfrb_comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1, device = 0;
  cudaStream_t st = nullptr;
  float* scratch = nullptr; size_t scratch_floats = 0;
  float* pin = nullptr; size_t pin_floats = 0;      // pinned staging of the stream-ordered weight broadcast
  int* vote = nullptr;                               // [4] device ints of the vote
  int* pin_vote = nullptr; int* pin_vote_out = nullptr;   // pinned [4] each: contributions / result
};

#define NCK(call)                                                                                                       \
  do {                                                                                                                  \
    ncclResult_t r__ = (call);                                                                                          \
    if (r__ != ncclSuccess) return fail(CFRB_ECUDA, std::string(#call) + ": " + ncclGetErrorString(r__));              \
  } while (0)

extern "C" {

int cfrb_comm_unique_id(uint8_t* out128) {
  if (!out128) return fail(CFRB_EINVAL, "null argument");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  NCK(ncclGetUniqueId(&id));
  std::memcpy(out128, &id, 128);
  return CFRB_OK;
}

int cfrb_comm_create(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, cfrb_comm** out) {
  if (!id128 || !out || world < 1 || rank < 0 || rank >= world) return fail(CFRB_EINVAL, "cfrb_comm_create: bad argument");
  CK(cudaSetDevice(device));
  auto* c = new cfrb_comm();
  c->rank = rank; c->world = world; c->device = device;
  ncclUniqueId id;
  std::memcpy(&id, id128, 128);
  ncclResult_t r = ncclCommInitRank(&c->comm, world, id, rank);
  if (r != ncclSuccess) { delete c; return fail(CFRB_ECUDA, std::string("ncclCommInitRank: ") + ncclGetErrorString(r)); }
  cudaError_t e = cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMallocHost((void**)&c->pin_vote, 8 * sizeof(int));
  if (e != cudaSuccess) { ncclCommDestroy(c->comm); delete c; return fail(CFRB_ECUDA, cudaGetErrorString(e)); }
  c->pin_vote_out = c->pin_vote + 4;
  *out = c;
  return CFRB_OK;
}

int cfrb_comm_destroy(cfrb_comm* c) {
  if (!c) return CFRB_OK;
  cudaSetDevice(c->device);
  if (c->st) { cudaStreamSynchronize(c->st); cudaStreamDestroy(c->st); }
  if (c->scratch) cudaFree(c->scratch);
  if (c->vote) cudaFree(c->vote);
  if (c->pin) cudaFreeHost(c->pin);
  if (c->pin_vote) cudaFreeHost(c->pin_vote);
  if (c->comm) ncclCommDestroy(c->comm);
  delete c;
  return CFRB_OK;
}

int cfrb_comm_rank(const cfrb_comm* c) { return c ? c->rank : -1; }
int cfrb_comm_world(const cfrb_comm* c) { return c ? c->world : 0; }

static int comm_scratch(cfrb_comm* c, size_t floats) {
  if (c->scratch_floats >= floats) return CFRB_OK;
  if (c->scratch) cudaFree(c->scratch);
  c->scratch = nullptr; c->scratch_floats = 0;
  CK(cudaMalloc((void**)&c->scratch, floats * sizeof(float)));
  c->scratch_floats = floats;
  return CFRB_OK;
}

int cfrb_comm_broadcast_weights(cfrb_comm* c, float* flat_host, size_t n, int32_t root, void* cuda_stream) {
  if (!c || n == 0 || (!flat_host && (!cuda_stream || c->rank == root))) return fail(CFRB_EINVAL, "cfrb_comm_broadcast_weights: bad argument");
  CK(cudaSetDevice(c->device));
  int rc = comm_scratch(c, n);
  if (rc) return rc;
  if (!cuda_stream) {
    if (c->rank == root) CK(cudaMemcpyAsync(c->scratch, flat_host, n * sizeof(float), cudaMemcpyHostToDevice, c->st));
    NCK(ncclBroadcast(c->scratch, c->scratch, n, ncclFloat, root, c->comm, c->st));
    if (c->rank != root) CK(cudaMemcpyAsync(flat_host, c->scratch, n * sizeof(float), cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    return CFRB_OK;
  }
  // stream-ordered: staged through pinned memory owned by the communicator; nothing is waited for here.  The root's buffer is
  // copied now (the caller may reuse it); the other ranks read theirs with cfrb_comm_broadcast_fetch once the stream got there.
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (c->pin_floats < n) {
    if (c->pin) cudaFreeHost(c->pin);
    c->pin = nullptr; c->pin_floats = 0;
    CK(cudaMallocHost((void**)&c->pin, n * sizeof(float)));
    c->pin_floats = n;
  }
  if (c->rank == root) {
    std::memcpy(c->pin, flat_host, n * sizeof(float));
    CK(cudaMemcpyAsync(c->scratch, c->pin, n * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  NCK(ncclBroadcast(c->scratch, c->scratch, n, ncclFloat, root, c->comm, st));
  if (c->rank != root) CK(cudaMemcpyAsync(c->pin, c->scratch, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  return CFRB_OK;
}
int cfrb_comm_broadcast_fetch(cfrb_comm* c, float* out_host, size_t n) {
  if (!c || !out_host || !c->pin || n > c->pin_floats) return fail(CFRB_EINVAL, "cfrb_comm_broadcast_fetch: no stream-ordered broadcast of that size");
  std::memcpy(out_host, c->pin, n * sizeof(float));
  return CFRB_OK;
}

int cfrb_comm_gather_rows(cfrb_comm* c, const float* dev_q, const float* dev_v, int32_t n, int32_t q_dim, int32_t v_dim, float* recv_q,
                          float* recv_v, int32_t root, void* cuda_stream) {
  if (!c || !dev_q || !dev_v || n < 0 || q_dim < 1 || v_dim < 1) return fail(CFRB_EINVAL, "cfrb_comm_gather_rows: bad argument");
  if (c->rank == root && (!recv_q || !recv_v)) return fail(CFRB_EINVAL, "cfrb_comm_gather_rows: the root needs receive buffers");
  CK(cudaSetDevice(c->device));
  const size_t nq = (size_t)n * q_dim, nv = (size_t)n * v_dim;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->st;
  NCK(ncclGroupStart());
  if (c->rank == root) {
    for (int r = 0; r < c->world; ++r) {
      if (r == root) continue;
      NCK(ncclRecv(recv_q + (size_t)r * nq, nq, ncclFloat, r, c->comm, st));
      NCK(ncclRecv(recv_v + (size_t)r * nv, nv, ncclFloat, r, c->comm, st));
    }
  } else {
    NCK(ncclSend(dev_q, nq, ncclFloat, root, c->comm, st));
    NCK(ncclSend(dev_v, nv, ncclFloat, root, c->comm, st));
  }
  NCK(ncclGroupEnd());
  if (c->rank == root) {     // the root's own block: a device-to-device copy into its slot
    CK(cudaMemcpyAsync(recv_q + (size_t)root * nq, dev_q, nq * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(recv_v + (size_t)root * nv, dev_v, nv * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  if (!cuda_stream) CK(cudaStreamSynchronize(st));     // on the caller's stream the collective is just enqueued (stream-ordered)
  return CFRB_OK;
}

// Agreement between the ranks' generator loops (they must issue the same number of collectives): every rank contributes a flag,
// all ranks get the maximum.  Enqueued on `cuda_stream` (NULL: the communicator's stream); cfrb_comm_vote_result reads it once the
// stream has passed that point (the caller synchronises, e.g. with cfrb_mark_wait).
int cfrb_comm_vote(cfrb_comm* c, const int32_t* values, int32_t n, void* cuda_stream) {
  if (!c || !values || n < 1 || n > 4) return fail(CFRB_EINVAL, "cfrb_comm_vote: 1..4 values");
  CK(cudaSetDevice(c->device));
  if (!c->vote) CK(cudaMalloc((void**)&c->vote, 4 * sizeof(int)));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : c->st;
  int* pin_i = c->pin_vote;      // contributions from pinned words owned by the communicator (the previous vote has been read)
  for (int i = 0; i < n; ++i) pin_i[i] = values[i];
  CK(cudaMemcpyAsync(c->vote, pin_i, n * sizeof(int), cudaMemcpyHostToDevice, st));
  NCK(ncclAllReduce(c->vote, c->vote, n, ncclInt32, ncclMax, c->comm, st));
  CK(cudaMemcpyAsync(c->pin_vote_out, c->vote, n * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (!cuda_stream) CK(cudaStreamSynchronize(st));
  return CFRB_OK;
}
int cfrb_comm_vote_result(cfrb_comm* c, int32_t* out, int32_t n) {
  if (!c || !out || !c->vote || n < 1 || n > 4) return fail(CFRB_EINVAL, "cfrb_comm_vote_result: no vote");
  for (int i = 0; i < n; ++i) out[i] = c->pin_vote_out[i];
  return CFRB_OK;
}

int cfrb_comm_reduce_sum(cfrb_comm* c, float* dev_buf, size_t n, int32_t root) {
  if (!c || !dev_buf) return fail(CFRB_EINVAL, "cfrb_comm_reduce_sum: bad argument");
  CK(cudaSetDevice(c->device));
  NCK(ncclReduce(dev_buf, dev_buf, n, ncclFloat, ncclSum, root, c->comm, c->st));
  CK(cudaStreamSynchronize(c->st));
  return CFRB_OK;
}

}  // extern "C"
