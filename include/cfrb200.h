/*
 * cfrb200 — C ABI of the B200-native CFR subgame-wave solver (libcfrb200.so).
 *
 * This is the drop-in boundary beneath the reference's pybind11 module `cfvpy.rela`
 * (csrc/liars_dice/rela/pybind.cc:119-213): host orchestration (rebel_b200/csrc/rela/*.cc, the
 * re-implemented `rela` module) calls ONLY these entry points; they replace, on the GPU and for
 * thousands of subgames at a time, what one reference CPU thread does for one subgame at a time:
 *
 *   cfrb_create / cfrb_begin_wave   <-  build_solver + CFR ctor        (subgame_solving.cc:791-800, 509-534)
 *                                       unroll_tree                    (tree.h:51-70)
 *   cfrb_run                        <-  CFR::step / multistep          (subgame_solving.cc:577-670) including
 *                                       the per-iteration value-net call the reference makes through
 *                                       IValueNet::compute_values      (net_interface.h:28-32,
 *                                       rela/data_loop.h:29-48, rela/model_locker.h:85-95)
 *   cfrb_set_weights                <-  ModelLocker::updateModel       (rela/model_locker.h:69-79)
 *   cfrb_fetch                      <-  ISubgameSolver::get_strategy / get_sampling_strategy /
 *                                       get_hand_values                (subgame_solving.h:60-88)
 *   cfrb_examples                   <-  CFR::update_value_network      (subgame_solving.cc:672-676, 220-226)
 *   cfrb_tree_template              <-  unroll_tree, for bit-exact infoset-index checks (tree_test.cc)
 *   cfrb_exploitability             <-  compute_exploitability2        (subgame_solving.cc:802-816)
 *
 * Conventions: plain C, no exceptions across the boundary; every function returns 0 on success or a
 * negative CFRB_E* code (cfrb_last_error() gives the message for the calling thread); all buffers are
 * caller-owned HOST memory (pinned preferred); one handle per GPU; a handle is not thread-safe (one
 * orchestrator thread per handle).  There is NO CPU fallback: without a CUDA device cfrb_create fails.
 *
 * Layouts (all row-major; solver state crosses the boundary as fp64 like the reference's vector<double>, value-net
 * tensors as fp32 like the reference's float tensors):
 *   beliefs            [n][2][H]          root beliefs of player 0 then player 1 (Pair<vector<double>> in the reference)
 *   dense strategy     [n][Nmax][H][A]    the reference's TreeStrategy = [node][hand][action] (subgame_solving.h:39),
 *                                         padded to Nmax = cfrb_max_nodes() nodes per subgame; entries of illegal
 *                                         actions, leaves and padding are 0
 *   root_value_means   [n][2][H]          CFR::root_values_means (subgame_solving.cc:702-703)
 *   queries            [..][Q]            value-net query rows, Q = 2 + A + 2H (subgame_solving.cc:100-123)
 *   weights            flat fp32 in Net2 state_dict order (cfvpy/models.py:64-94):
 *                      body.0.weight[hid,Q] body.0.bias[hid] body.1.weight[hid] body.1.bias[hid]
 *                      body.4.weight[hid,hid] body.4.bias body.5.weight body.5.bias output.weight[H,hid] output.bias[H]
 */
#ifndef CFRB200_H_
#define CFRB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cfrb_handle cfrb_handle;

enum {
  CFRB_OK = 0,
  CFRB_EINVAL = -1,   /* bad argument */
  CFRB_ECUDA = -2,    /* CUDA runtime error (message has the cudaError string) */
  CFRB_ENODEV = -3,   /* no CUDA device / wrong architecture */
  CFRB_ESTATE = -4,   /* call sequence error (e.g. run before begin_wave, net needed but no weights) */
  CFRB_ENOMEM = -5
};

/* How the leaf value net (Net2 forward) is evaluated. */
enum {
  CFRB_NET_ZERO = 0,      /* leaf values are 0 (reference: create_zero_net, real_net.cc:30-55) */
  CFRB_NET_FP32 = 1,      /* fp32 SIMT kernel: parity path, matches libtorch fp32 to ~1e-6 */
  CFRB_NET_TC_F16 = 2,    /* tcgen05 tensor-core kernel: fp16 operands, fp32 accumulate/LayerNorm/GELU
                             (the reference's own `half_inference` option, selfplay.py:42-43,211) */
  CFRB_NET_TC_F16X2 = 3   /* same kernel with the fast GELU: y/2 (1 + tanh(poly)) with packed f32x2 FMAs and tanh.approx.f32, one
                             rounding to fp16 at the end (same accuracy as mode 2, 1 instead of 2 MUFU operations per element) */
};

/* Subgame solver.  In FP mode cfrb_fetch's "last" is FP::last_strategies (belief x best response), "avg" is
 * FP::average_strategies (also the sampling / belief-propagation strategy, subgame_solving.h:76-83) and "regrets" is empty. */
enum {
  CFRB_SOLVER_CFR = 0,    /* CFR (subgame_solving.cc:508-715), params.use_cfr = true */
  CFRB_SOLVER_FP = 1      /* fictitious play (subgame_solving.cc:364-506), params.use_cfr = false */
};

/* Arithmetic type of the per-infoset CFR tables (regrets, strategies, reach, values). */
enum {
  CFRB_STATE_F64 = 0,     /* double, like the reference's TreeStrategy (default) */
  CFRB_STATE_F32 = 1      /* float: half the table traffic; trajectories drift from the fp64 reference sooner */
};

/* SubgameSolvingParams (subgame_solving.h:43-58) + game shape + capacity. */
typedef struct {
  int32_t num_dice;
  int32_t num_faces;
  int32_t max_depth;        /* depth of every subgame tree */
  int32_t num_iters;        /* iterations per subgame (only used for default graphs/snapshots) */
  int32_t linear_update;
  int32_t dcfr;
  double dcfr_alpha, dcfr_beta, dcfr_gamma;
  int32_t max_subgames;     /* wave capacity K */
  int32_t device;           /* CUDA ordinal */
  int32_t net_mode;         /* CFRB_NET_* */
  int32_t hidden;           /* Net2 n_hidden (256); n_layers = 2, LayerNorm on */
  int32_t state_dtype;      /* CFRB_STATE_* */
  int32_t solver;           /* CFRB_SOLVER_*: which ISubgameSolver build_solver would return (subgame_solving.cc:791-800) */
  int32_t optimistic;       /* FP only: SubgameSolvingParams::optimistic (subgame_solving.h:50, util.h:52-63) */
} cfrb_config;

/* One node of an unrolled subgame tree: UnrolledTreeNode (tree.h:31-47). */
typedef struct {
  int32_t last_bid, player_id, children_begin, children_end, parent, depth;
} cfrb_node;

const char* cfrb_last_error(void);
/* Number of CUDA devices visible (0 if none / driver missing). */
int cfrb_device_count(void);

int cfrb_create(const cfrb_config* cfg, cfrb_handle** out);
int cfrb_destroy(cfrb_handle* h);

/* Shape queries. */
int cfrb_num_actions(const cfrb_handle* h);   /* A */
int cfrb_num_hands(const cfrb_handle* h);     /* H */
int cfrb_query_size(const cfrb_handle* h);    /* Q */
int cfrb_max_nodes(const cfrb_handle* h);     /* Nmax over all root templates */

/* Host-only (no device needed): unroll_tree(game, {last_bid, player_id}, max_depth) (tree.h:51-70) through the same
 * template builder the kernels index with.  Returns the node count or a negative error; writes min(count, cap). */
int cfrb_unroll_tree(int32_t num_dice, int32_t num_faces, int32_t last_bid, int32_t player_id, int32_t max_depth,
                     cfrb_node* out, int32_t cap);

/* Tree of the subgame rooted at (last_bid, player_id) with the handle's max_depth, in the reference's BFS
 * node order.  Returns the node count (>0) or a negative error; writes min(count, cap) nodes. */
int cfrb_tree_template(const cfrb_handle* h, int32_t last_bid, int32_t player_id, cfrb_node* out, int32_t cap);

/* Install value-net weights (flat fp32, `n` floats, layout above).  `version` is remembered and returned by
 * cfrb_weights_version.  Takes effect for kernels enqueued after the call. */
int cfrb_set_weights(cfrb_handle* h, const float* flat, size_t n, uint64_t version);
uint64_t cfrb_weights_version(const cfrb_handle* h);

/* Start a wave of n <= max_subgames subgames.  Subgame k is rooted at (last_bid[k], player_id[k]) with
 * root beliefs beliefs[k][2][H]; state is initialised exactly like the CFR constructor
 * (uniform strategies, reach-weighted uniform sum, zero regrets, subgame_solving.cc:509-524,125-149).
 * act_iteration[k] (may be NULL) is the iteration count after which the sampling strategy
 * (CFR::last_strategies) of subgame k is snapshotted for RlRunner's state sampling
 * (recursive_solving.cc:168-174); -1 = no snapshot. */
int cfrb_begin_wave(cfrb_handle* h, int32_t n, const int32_t* last_bid, const int32_t* player_id,
                    const double* beliefs, const int32_t* act_iteration);

/* Re-initialise the solver state of the CURRENT wave on the device (same roots, beliefs and act_iterations; no
 * host->device traffic): what constructing fresh CFR solvers for the same subgames would do. */
int cfrb_reset_wave(cfrb_handle* h, void* cuda_stream);

/* Profiling switch: 0 = off; n > 0 = cfrb_run brackets every n-th value-net launch with a pair of CUDA events on the
 * launching stream, and cfrb_last_run_ms reports the value-net kernel time of the last run estimated from those samples
 * (mean sampled duration x number of launches).  Sampling keeps the event traffic out of the way of the measurement. */
int cfrb_set_profiling(cfrb_handle* h, int32_t on);

/* Advance every subgame of the wave by `iters` CFR iterations (iteration i has traverser i % 2,
 * CFR::multistep subgame_solving.cc:666-670), asynchronously on `cuda_stream` (a cudaStream_t; NULL = the
 * handle's own stream). */
int cfrb_run(cfrb_handle* h, int32_t iters, void* cuda_stream);
/* Block until everything enqueued by this handle has finished. */
int cfrb_sync(cfrb_handle* h);
/* Iterations done so far in the current wave. */
int cfrb_iterations_done(const cfrb_handle* h);

/* Copy results to the host (any pointer may be NULL).  Synchronises.
 *   root_value_means [n][2][H]; snapshot / last / avg / sum / regrets: dense [n][Nmax][H][A]. */
int cfrb_fetch(cfrb_handle* h, double* root_value_means, double* snapshot_strategy, double* last_strategy,
               double* avg_strategy, double* sum_strategy, double* regrets);

/* Compact fetch for host orchestration (BatchedRlRunner, evaluators): table `which` (0 snapshot, 1 last strategy, 2 sum strategy,
 * 3 regrets, 4 average strategy = ISubgameSolver::get_strategy) of every subgame as stored on the device, [n][cfrb_table_stride()] fp64 with entry (child_node - 1) * H + hand
 * holding the value of (parent node, hand, action leading to child_node).  Synchronises. */
int cfrb_table_stride(const cfrb_handle* h);
int cfrb_fetch_compact(cfrb_handle* h, int32_t which, double* out);

/* Training examples of the finished wave: for each subgame and traverser t in {0,1} the query row of the
 * subgame root as seen by t and the target root_value_means[t].  queries [n][2][Q], values [n][2][H]. */
int cfrb_examples(cfrb_handle* h, float* queries, float* values);

/* Teacher forcing (tests): overwrite solver state of the current wave from dense host arrays
 * [n][Nmax][H][A] (NULL = keep), root_value_means [n][2][H], num_steps [n][2], and set the wave's
 * iteration counter. */
int cfrb_load_state(cfrb_handle* h, const double* regrets, const double* last_strategy, const double* sum_strategy,
                    const double* root_value_means, const int32_t* num_steps, int32_t iterations_done);

/* Debug/parity taps of the most recent iteration: query rows [rows][Q] and the (unscaled) net outputs
 * [rows][H] for all pseudo-leaves of the wave in (subgame, leaf) order; returns the number of rows,
 * writes at most cap_rows. */
int cfrb_debug_leaf_io(cfrb_handle* h, float* queries, float* net_out, double* scalers, int32_t cap_rows);

/* Debug taps of the tensor-core value net (CFRB_NET_TC_F16 only): re-runs it on the current query tiles and returns
 * the raw fp32 accumulators of layer 1 and layer 2 for the first 128 rows, each [128][256]. */
int cfrb_debug_net_taps(cfrb_handle* h, float* d1, float* d2);
/* Development aid: re-runs the tensor-core value net once with clock64() stamps of CTA 0 (out[2048]: epilogue thread 0 at
 * [phase*8 + e], MMA-issuing thread at [1024 + phase*4 + m]; see the CFRB_TRACE3 calls in leaf_mlp_tc3.cuh). */
int cfrb_debug_net_trace(cfrb_handle* h, long long* out, int n);

/* Exploitability (best-response values of both players, compute_exploitability2) of a full-tree strategy
 * given as dense [N_full][H][A] fp64, evaluated on the GPU. out2 = {br0, br1}. */
int cfrb_exploitability(cfrb_handle* h, const double* full_strategy, double* out2);

/* Counters for bench.py: kernels launched by this handle since creation, and leaf rows of the wave. */
int64_t cfrb_kernel_launches(const cfrb_handle* h);
int64_t cfrb_wave_leaf_rows(const cfrb_handle* h);
/* Timing marks (benchmarks): record CUDA event `slot` (0..7) on `cuda_stream` (NULL = the handle's stream); device time
 * between two recorded marks (waits for the second). */
int cfrb_mark(cfrb_handle* h, int32_t slot, void* cuda_stream);
int cfrb_mark_elapsed_ms(cfrb_handle* h, int32_t a, int32_t b, float* ms);
int cfrb_mark_wait(cfrb_handle* h, int32_t slot);          /* block until the mark has been reached */
void* cfrb_handle_stream(cfrb_handle* h);                  /* the handle's own cudaStream_t (what NULL stream arguments mean) */
/* Overwrite a scratch buffer of `bytes` on the stream (pass more than the 126 MB of L2 to evict it between timed steps). */
int cfrb_l2_flush(cfrb_handle* h, size_t bytes, void* cuda_stream);
/* Device time in ms of the most recent cfrb_run, and of its value-net kernels only (CUDA events on
 * the launching stream; valid after cfrb_sync). */
int cfrb_last_run_ms(cfrb_handle* h, float* total_ms, float* net_ms);

/* ---- Device-resident self-play: RlRunner::step (recursive_solving.cc:160-275) for n_games games in lock-step, without host
 * round trips.  Replaces, per wave, RlRunner's act_iteration draw (:168-169), sample_state_to_leaf / sample_state_single
 * (:192-275), normalize_beliefs_inplace (:41-44) and CFR::update_value_network (subgame_solving.cc:672-676).  Game g owns a
 * std::mt19937 seeded with seeds[g] on the device and consumes it in the reference's draw order, so it replays
 * RlRunner(seed = seeds[g]) as long as the solver's strategies agree.  random_action_prob / sample_leaf are
 * RecursiveSolvingParams' fields (recursive_solving.h:31-38). */
int cfrb_selfplay_create(cfrb_handle* h, int32_t n_games, const uint32_t* seeds, float random_action_prob, int32_t sample_leaf);
/* One step of the loop, enqueued asynchronously on `cuda_stream` (NULL = the handle's stream):
 *   1. if a wave is pending: its 2 * n_games training examples are written to the DEVICE buffers dev_ex_q [2n][Q] /
 *      dev_ex_v [2n][H] (both NULL = drop them) and every game samples its next public state (a finished game restarts);
 *   2. if start_next != 0: act_iteration draws, subgame descriptors, CFR constructor and num_iters iterations of the next wave.
 * Returns the number of example rows written (0 or 2 * n_games) or a negative error. */
int cfrb_selfplay_wave(cfrb_handle* h, float* dev_ex_q, float* dev_ex_v, int32_t start_next, void* cuda_stream);
/* Block until the examples written by the most recent cfrb_selfplay_wave are complete (the wave it started keeps running). */
int cfrb_selfplay_wait_examples(cfrb_handle* h);
/* Game states (public state and beliefs [n][2][H]) copied to the host; any pointer may be NULL.  Synchronises.  Returns n_games. */
int cfrb_selfplay_state(cfrb_handle* h, int32_t* last_bid, int32_t* player, double* beliefs);
/* Test aid: the division-free quotient of the regret-matching step (reciprocal of the node's sum + two fused multiply-add
 * corrections, csrc/cfr_kernels.cuh) against IEEE division on blocks x 256 x 4096 pseudo-random operand pairs. */
int cfrb_debug_div_check(cfrb_handle* h, uint64_t seed, int32_t blocks, uint64_t* mismatches);
/* Test aid: GELU evaluations on every fp16 input: out[i] = fp16 bits of f(fp16 with bit pattern i), i < 65536;
 * what 0 = tanh.approx.f16x2, 1 / 2 = GELU(2 x) computed from x = y / 2 in packed-half arithmetic (HFMA2 + tanh.approx.f16x2, a
 * biased evaluation the value net does not use) / the way the fp32-tanh epilogue of CFRB_NET_TC_F16X2 does (tests pin the
 * arithmetic model of oracle/ref_harness.cc against it). */
int cfrb_debug_gelu_table(cfrb_handle* h, int32_t what, uint16_t* out);
/* Roots (last_bid, player_id) of the subgames of the current wave — also of a wave built on the device by cfrb_selfplay_wave
 * (synchronises then).  Writes min(n, cap) entries, returns n. */
int cfrb_wave_roots(cfrb_handle* h, int32_t* last_bid, int32_t* player_id, int32_t cap);
/* Block until the work enqueued on `cuda_stream` (NULL = the handle's stream) has finished. */
int cfrb_stream_wait(cfrb_handle* h, void* cuda_stream);

/* ---- Device-resident example rows: storage of the replay buffer (rela/prioritized_replay.h:224-506 keeps one pair of host
 * tensors per example; here the rows of the ring live in HBM as two [capacity][dim] fp32 matrices and never visit the host on
 * their way from the generator kernels to the trainer's batch).  Bookkeeping (head, size, priorities, blocking) stays with the
 * caller. */
typedef struct cfrb_rows cfrb_rows;
int cfrb_rows_create(int32_t device, int64_t capacity_rows, int32_t q_dim, int32_t v_dim, cfrb_rows** out);
int cfrb_rows_destroy(cfrb_rows* r);
int cfrb_rows_device(const cfrb_rows* r);
/* Store n rows at ring position `slot` (wraps around).  kind 0: q / v are host pointers; kind 1: device pointers on CUDA
 * device src_device (peer copy when that is another GPU).  Returns when the rows are in place. */
int cfrb_rows_write(cfrb_rows* r, int64_t slot, int32_t n, const float* q, const float* v, int32_t kind, int32_t src_device);
/* n rows starting at `slot` (wraps around) to host memory (save / extract). */
int cfrb_rows_read(cfrb_rows* r, int64_t slot, int32_t n, float* q, float* v);
/* Batch assembly (PrioritizedReplay::sample -> makeBatch, rela/types.cc:19-41): rows ids[0..n) gathered into out_q [n][q_dim] /
 * out_v [n][v_dim] on out_device (CUDA ordinal, -1 = host memory).  On the ring's own device the gather kernel runs on
 * `cuda_stream` (the consumer's stream). */
int cfrb_rows_gather(cfrb_rows* r, const int32_t* ids, int32_t n, float* out_q, float* out_v, int32_t out_device, void* cuda_stream);
/* Device scratch for the hand-over of one wave's examples from a generator handle to a row store. */
int cfrb_dev_alloc(int32_t device, size_t bytes, void** out);
int cfrb_dev_free(int32_t device, void* p);
int cfrb_dev_to_host(int32_t device, void* dst, const void* src, size_t bytes);

/* ---- One process per GPU: the two hand-overs the reference performs through shared host memory inside ONE process become NCCL
 * collectives over NVLink, issued by this library on device buffers (no torch.distributed, no host bounce):
 *   ModelLocker::updateModel (rela/model_locker.h:69-79)         -> cfrb_comm_broadcast_weights
 *   PrioritizedReplay::add   (rela/prioritized_replay.h:247-261) -> cfrb_comm_gather_rows into the trainer rank's device rows
 *   recursive_eval's float32 accumulation (recursive_eval.cc:343-363) -> cfrb_comm_reduce_sum
 * The 128-byte id is created on one rank (cfrb_comm_unique_id) and handed to the others by the launcher (e.g. through the
 * torchrun store); every function is a collective: all ranks of the communicator call it, in the same order. */
typedef struct cfrb_comm cfrb_comm;
int cfrb_comm_unique_id(uint8_t* out128);
int cfrb_comm_create(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, cfrb_comm** out);
int cfrb_comm_destroy(cfrb_comm* c);
int cfrb_comm_rank(const cfrb_comm* c);
int cfrb_comm_world(const cfrb_comm* c);
/* flat fp32 weights (cfrb_set_weights layout): read from the root's host buffer, delivered to every other rank.  cuda_stream NULL:
 * the communicator's own stream, the call waits and the other ranks' flat_host is filled.  Otherwise the H2D copy (root), the
 * ncclBroadcast and the D2H copy (others) are only ENQUEUED on that stream (a generator loop puts them between two waves); the
 * other ranks pass flat_host = NULL and read the weights with cfrb_comm_broadcast_fetch once the stream has passed that point. */
int cfrb_comm_broadcast_weights(cfrb_comm* c, float* flat_host, size_t n, int32_t root, void* cuda_stream);
int cfrb_comm_broadcast_fetch(cfrb_comm* c, float* out_host, size_t n);
/* every rank contributes n rows from DEVICE buffers dev_q [n][q_dim], dev_v [n][v_dim]; on the root they arrive in rank order in
 * the DEVICE buffers recv_q [world * n][q_dim], recv_v [world * n][v_dim] (ignored elsewhere).  cuda_stream NULL: the communicator's
 * own stream, the call waits; otherwise the send / recv are only ENQUEUED on that stream — a generator loop puts them between two
 * waves on its handle's stream, where the GPU has nothing else to run and they cost microseconds instead of competing with a
 * wave's kernels for SMs. */
int cfrb_comm_gather_rows(cfrb_comm* c, const float* dev_q, const float* dev_v, int32_t n, int32_t q_dim, int32_t v_dim, float* recv_q,
                          float* recv_v, int32_t root, void* cuda_stream);
/* agreement between generator loops that must issue the same collectives in the same order ("stop after this wave", "the trainer
 * rank has weights version v"): every rank contributes n <= 4 ints, all ranks obtain the element-wise maximum; enqueued on
 * cuda_stream like cfrb_comm_gather_rows, read with cfrb_comm_vote_result once that point is reached. */
int cfrb_comm_vote(cfrb_comm* c, const int32_t* values, int32_t n, void* cuda_stream);
int cfrb_comm_vote_result(cfrb_comm* c, int32_t* out, int32_t n);
/* in-place float32 sum over the ranks of a DEVICE buffer, result on the root. */
int cfrb_comm_reduce_sum(cfrb_comm* c, float* dev_buf, size_t n, int32_t root);

#ifdef __cplusplus
}
#endif
#endif /* CFRB200_H_ */
