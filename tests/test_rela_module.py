"""The `rela` drop-in module (rebel_b200/csrc/rela): Python surface of the reference's cfvpy.rela
(csrc/liars_dice/rela/pybind.cc:119-213).  CPU tests exercise everything that does not need a device; the GPU tests replay
`initialize_datagen` (cfvpy/selfplay.py:182-260) and check the batched self-play walk against the reference's RlRunner."""
import os
import threading
import time

import numpy as np
import pytest
import torch

from oracle.oracle import game_dims


@pytest.fixture(scope="module")
def rela():
    import rebel_b200.rela as m
    return m


def make_cfg(rela, D, F, **kw):
    cfg = rela.RecursiveSolvingParams()
    # exactly what create_mdp_config does (selfplay.py:587-610): hasattr check + setattr, recursing into subgame_params
    spec = dict(num_dice=D, num_faces=F, random_action_prob=0.25, sample_leaf=True,
                subgame_params=dict(num_iters=1024, max_depth=2, linear_update=True, use_cfr=True))
    spec.update(kw)

    def rec(obj, d):
        for k, v in d.items():
            assert hasattr(obj, k), k
            if isinstance(v, dict):
                rec(getattr(obj, k), v)
            else:
                setattr(obj, k, v)
    rec(cfg, spec)
    return cfg


def test_surface_matches_reference(rela):
    for name in ("ValueTransition", "ValuePrioritizedReplay", "ThreadLoop", "SubgameSolvingParams", "RecursiveSolvingParams",
                 "DataThreadLoop", "Context", "ModelLocker", "compute_exploitability_fp", "compute_exploitability_with_net",
                 "compute_stats_with_net", "create_cfr_thread"):
        assert hasattr(rela, name), name
    sp = rela.SubgameSolvingParams()
    assert (sp.num_iters, sp.max_depth, sp.linear_update, sp.use_cfr, sp.optimistic, sp.dcfr) == (10, 2, False, False, False, False)
    cfg = make_cfg(rela, 1, 6)
    assert cfg.subgame_params.num_iters == 1024 and cfg.subgame_params.use_cfr        # nested setattr sticks (by reference)
    assert abs(cfg.random_action_prob - 0.25) < 1e-7 and cfg.sample_leaf
    with pytest.raises(RuntimeError):          # no CUDA device here: the evaluation helpers fail loudly, there is no CPU path
        rela.compute_exploitability_fp(cfg)


def test_context_is_subclassable_like_timed_context(rela):
    class Timed(rela.Context):          # cfvpy/utils.py:70-95
        def __init__(self):
            super().__init__()
            self.t0 = None

        def start(self):
            self.t0 = time.time()
            super().start()
    c = Timed()
    c.start()
    assert c.terminated() and c.t0 is not None      # no loops pushed: trivially terminated


def test_replay_buffer_semantics(rela, tmp_path):
    Q, H = 27, 6
    r = rela.ValuePrioritizedReplay(capacity=100, seed=1, alpha=1.0, beta=0.4, prefetch=3, use_priority=False, compressed_values=False)
    assert r.size() == 0 and r.num_add() == 0
    q = torch.arange(40 * Q, dtype=torch.float32).reshape(40, Q)
    v = torch.arange(40 * H, dtype=torch.float32).reshape(40, H)
    r.push([q, v, torch.ones(40)])
    assert r.size() == 40 and r.num_add() == 40
    batch, w = r.sample(16, "cpu")
    assert batch.query.shape == (16, Q) and batch.values.shape == (16, H) and w.shape == (16,)
    rows = (batch.query[:, 0] / Q).long()
    assert torch.equal(batch.values[:, 0], rows.float() * H)            # query/values of a sample belong to the same row
    path = str(tmp_path / "dump.bin")
    r.save(path)
    assert os.path.getsize(path) == 40 * (8 + 4 * (Q + H))              # int32 qsize, int32 vsize, floats (types.cc:87-94)
    r2 = rela.ValuePrioritizedReplay(100, 2, 1.0, 0.4, 0, False, False)
    r2.load(path, 1.0, -1, 2)                                            # stride 2
    assert r2.size() == 20
    ex = r2.extract()
    assert r2.size() == 0 and torch.equal(ex[0], q[::2]) and torch.equal(ex[1], v[::2]) and torch.equal(ex[2], torch.ones(20))
    r.pop_until(10)
    assert r.size() == 10
    # ring of 1.25 x capacity rows: the 126th row blocks until sampling evicts down to `capacity`
    r.pop_until(0)
    r.push([q.repeat(3, 1), v.repeat(3, 1), torch.ones(120)])
    done = threading.Event()

    def producer():
        r.push([q[:10], v[:10], torch.ones(10)])
        done.set()
    th = threading.Thread(target=producer)
    th.start()
    time.sleep(0.3)
    assert not done.is_set() and r.size() == 120
    r.sample(8, "cpu")                                                   # evicts the oldest rows down to capacity = 100
    th.join(timeout=5)
    assert done.is_set() and r.size() == 110 and r.num_add() == 40 + 120 + 10
    with pytest.raises(RuntimeError):
        rela.ValuePrioritizedReplay(10, 0, 1.0, 1.0, 0, False, True)


def test_prioritized_sampling(rela):
    r = rela.ValuePrioritizedReplay(1000, 3, 1.0, 0.5, 0, True, False)
    q = torch.arange(100, dtype=torch.float32).reshape(100, 1)
    pr = torch.ones(100); pr[50:] = 9.0
    r.push([q, q.clone(), pr])
    cnt_hi = 0
    for _ in range(50):
        b, w = r.sample(20, "cpu")
        cnt_hi += int((b.query[:, 0] >= 50).sum())
        assert float(w.max()) == 1.0
        r.update_priority(torch.ones(20) * 1.0 + 8.0 * (b.query[:, 0] >= 50).float())
    assert 0.85 < cnt_hi / 1000 < 0.95                                   # 9:1 odds


def test_model_locker_snapshots_weights(rela):
    from rebel_b200.models import make_selfplay_net
    net = make_selfplay_net(1, 4)
    replica = torch.jit.script(make_selfplay_net(1, 4, seed=1))
    locker = rela.ModelLocker([replica], "cuda:0")
    assert locker.version == 1
    locker.update_model(net)
    assert locker.version == 2
    for a, b in zip(replica.state_dict().values(), net.state_dict().values()):   # replicas refreshed like the reference
        assert torch.equal(a, b)
    with pytest.raises(RuntimeError):
        rela.ModelLocker([torch.nn.Linear(3, 3)], "cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 2), (1, 3), (1, 4)])
def test_exploitability_of_strategy_bit_exact(rela, golden, D, F):
    """exploitability_of_strategy = compute_exploitability2 / BRSolver::compute_br (subgame_solving.cc:316-358,802-816) on the
    GPU best-response kernel: bit-identical to the compiled reference on the golden 16-iteration full-tree strategies."""
    g = golden("fulltree.npz")
    e = rela.exploitability_of_strategy(D, F, torch.from_numpy(g[f"avg16_{D}x{F}"]))
    assert np.array_equal(np.array(e), g[f"expl_{D}x{F}_nofma"][0])


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6), (2, 3)])
def test_exploitability_of_strategy_on_recursive_eval_golden(rela, golden, D, F):
    g = golden("recursive_eval_zero.npz")
    ss, sr = g[f"summed_strategy_{D}x{F}"], g[f"summed_reach_{D}x{F}"]
    e = rela.exploitability_of_strategy(D, F, torch.from_numpy(ss / (sr + np.float32(1e-6))))
    assert np.array_equal(np.array(e), g[f"exploitability_{D}x{F}"][-1])
    with pytest.raises(RuntimeError):
        rela.exploitability_of_strategy(D, F, torch.zeros(3, 2, 2))


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6), (2, 3)])
@pytest.mark.parametrize("batch_repeats,wave_capacity", [(64, 4096), (1, 37)])
def test_recursive_eval_bit_exact_vs_reference(rela, golden, D, F, batch_repeats, wave_capacity):
    """BASELINE config 5 path (recursive_eval.cc:117-191,343-369): sampled recursive strategies of seeds 0..R-1 solved as
    level-batched GPU waves, float32 reach-weighted sums in strategy_id order, exploitability at powers of two.  Zero net,
    fp64 tables: every number is bit-identical to the compiled reference (fixture from oracle/make_golden.py), however the
    repeats are batched and whatever the wave capacity."""
    g = golden("recursive_eval_zero.npz")
    iters, reps = (int(x) for x in g[f"cfg_{D}x{F}"])
    cfg = make_cfg(rela, D, F, net_mode=0, state_dtype=0, subgame_params=dict(num_iters=iters, max_depth=2, linear_update=True, use_cfr=True))
    r = rela.recursive_eval_sampled(cfg, 0, reps, seed=0, batch_repeats=batch_repeats, wave_capacity=wave_capacity)
    assert list(r["checkpoints"]) == list(g[f"checkpoints_{D}x{F}"])
    assert np.array_equal(r["summed_reach"].numpy(), g[f"summed_reach_{D}x{F}"])
    assert np.array_equal(r["summed_strategy"].numpy(), g[f"summed_strategy_{D}x{F}"])
    assert np.array_equal(r["exploitability"].numpy(), g[f"exploitability_{D}x{F}"])
    assert r["subgames_solved"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6), (2, 3)])
@pytest.mark.parametrize("sample_leaf", [True, False])
def test_batched_walk_reproduces_rlrunner_stream(rela, golden, D, F, sample_leaf):
    """One game stream (concurrent_games = 1), zero net, fp64 tables: the training examples are bit-identical to the
    reference's RlRunner(seed=7) (golden fixture generated by oracle/make_golden.py from the compiled reference)."""
    g = golden("selfplay_zero.npz")
    gq, gv = g[f"q_{D}x{F}_{int(sample_leaf)}"], g[f"v_{D}x{F}_{int(sample_leaf)}"]
    cfg = make_cfg(rela, D, F, sample_leaf=sample_leaf, concurrent_games=1, net_mode=0, state_dtype=0,
                   subgame_params=dict(num_iters=32, max_depth=2, linear_update=True, use_cfr=True))
    q, v = rela.run_selfplay_waves(cfg, 0, 7, len(gq) // 2)
    assert np.array_equal(q.numpy(), gq) and np.array_equal(v.numpy(), gv)


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6), (2, 3)])
def test_batched_walk_with_fictitious_play_reproduces_rlrunner_stream(rela, golden, D, F):
    """use_cfr = false (the YAML default, subgame_solving.h:48): build_solver returns FP; the example stream of one game
    stream is bit-identical to the reference's RlRunner(seed=7) with the fictitious-play solver."""
    g = golden("selfplay_zero.npz")
    gq, gv = g[f"q_fp_{D}x{F}"], g[f"v_fp_{D}x{F}"]
    cfg = make_cfg(rela, D, F, sample_leaf=True, concurrent_games=1, net_mode=0, state_dtype=0,
                   subgame_params=dict(num_iters=32, max_depth=2, linear_update=True, use_cfr=False))
    q, v = rela.run_selfplay_waves(cfg, 0, 7, len(gq) // 2)
    assert np.array_equal(q.numpy(), gq) and np.array_equal(v.numpy(), gv)


def _save_eval_model(tmp_path, D, F, netname):
    from rebel_b200.models import make_selfplay_net
    net = make_selfplay_net(D, F, seed=0)
    if netname == "zero_out":
        with torch.no_grad():
            net.output.weight.zero_()
            net.output.bias.zero_()
    path = str(tmp_path / f"net_{D}x{F}_{netname}.pt")
    torch.jit.script(net).save(path)
    return path


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6), (2, 3)])
@pytest.mark.parametrize("use_cfr", [True, False])
def test_evaluation_entry_points_vs_reference(rela, golden, tmp_path, D, F, use_cfr):
    """compute_exploitability_with_net and compute_stats_with_net (rela/pybind.cc:45-84, eval_net stats.cc:44-153) against
    the compiled reference (fixture from oracle/make_golden.py).  With a net whose output layer is zero the solver
    trajectories are bit-identical, so the exploitabilities agree to float rounding and eval_net's MSE to 1e-6 relative;
    with the random-init net (fp32 SIMT kernel vs ATen) the strategies agree until regret matching amplifies 1e-7 differences,
    so the same quantities are compared to a few percent."""
    g = golden("net_evaluation.npz")
    iters = {(1, 4): 32, (1, 6): 16, (2, 3): 8}[(D, F)]
    tag = ("cfr" if use_cfr else "fp")
    for netname, rel in (("zero_out", 1e-6), ("random", 5e-2)):
        want = g[f"values_{tag}_{netname}_{D}x{F}"]
        path = _save_eval_model(tmp_path, D, F, netname)
        cfg = make_cfg(rela, D, F, net_mode=1, state_dtype=0, subgame_params=dict(num_iters=iters, max_depth=2, linear_update=True, use_cfr=use_cfr))
        e_rec = rela.compute_exploitability_with_net(cfg, path)
        e_leaf, mse_net, mse_full = rela.compute_stats_with_net(cfg, path)
        got = np.array([e_rec, e_leaf, mse_net, mse_full])
        assert np.all(np.abs(got - want) <= rel * np.abs(want) + 1e-7), (netname, got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("use_cfr", [True, False])
def test_compute_exploitability_fp_full_tree(rela, port, use_cfr):
    """compute_exploitability_fp (pybind.cc:86-104): full-tree solve without a net; the returned sum of exploitabilities equals
    the oracle's for the same solver, and a depth-limited tree without a net is rejected like the reference does."""
    D, F, iters = 1, 4, 64
    cfg = make_cfg(rela, D, F, subgame_params=dict(num_iters=iters, max_depth=100000, linear_update=True, use_cfr=use_cfr))
    got = rela.compute_exploitability_fp(cfg)
    b = np.full((2, F ** D), 1.0 / F ** D)
    s = (port.cfr_solve if use_cfr else port.fp_solve)(D, F, b, [iters], num_iters=iters, max_depth=100000)
    want = port.exploitability(D, F, s["avg"][0]).sum()
    assert abs(got - want) <= 1e-6 * abs(want)
    with pytest.raises(RuntimeError):
        rela.compute_exploitability_fp(make_cfg(rela, D, F, subgame_params=dict(num_iters=8, max_depth=2, linear_update=True, use_cfr=True)))


@pytest.mark.gpu
def test_drop_in_datagen_flow(rela):
    """initialize_datagen (selfplay.py:182-260) line for line: ModelLocker per device, replay, create_cfr_thread per
    'thread', Context.start; then update_model, pause/resume, terminate."""
    from rebel_b200.models import make_selfplay_net
    D, F = 1, 6
    A, H, Q = game_dims(D, F)
    net = make_selfplay_net(D, F)
    ref_model = [torch.jit.script(make_selfplay_net(D, F))]
    locker = rela.ModelLocker(ref_model, "cuda:0")
    replay = rela.ValuePrioritizedReplay(capacity=1 << 16, seed=10001, alpha=1.0, beta=1.0, prefetch=8, use_priority=False,
                                         compressed_values=False)
    cfg = make_cfg(rela, D, F, concurrent_games=256, subgame_params=dict(num_iters=64, max_depth=2, linear_update=True, use_cfr=True))
    ctx = rela.Context()
    for i in range(2):
        ctx.push_env_thread(rela.create_cfr_thread(locker, replay, cfg, i))
    ctx.start()
    t0 = time.time()
    while replay.num_add() < 4096 and time.time() - t0 < 60:
        time.sleep(0.05)
    assert replay.num_add() >= 4096, ctx.error()
    locker.update_model(net)                                             # trainer pushes fresh weights
    batch, w = replay.sample(512, "cuda:0")
    assert batch.query.shape == (512, Q) and batch.values.shape == (512, H) and batch.query.is_cuda
    qs = batch.query.cpu().numpy()
    assert np.allclose(qs[:, 2 + A:2 + A + H].sum(-1), 1, atol=1e-5) and set(np.unique(qs[:, :2])) <= {0.0, 1.0}
    ctx.pause()
    time.sleep(0.5)
    n0 = replay.num_add()
    time.sleep(0.5)
    assert replay.num_add() == n0                                        # paused between waves
    ctx.resume()
    t0 = time.time()
    while replay.num_add() == n0 and time.time() - t0 < 30:
        time.sleep(0.05)
    assert replay.num_add() > n0
    ctx.terminate()
    t0 = time.time()
    while not ctx.terminated() and time.time() - t0 < 30:
        time.sleep(0.05)
    assert ctx.terminated() and ctx.error() == ""


def test_model_locker_rejects_deeper_net2(rela):
    """A Net2 with n_layers=3 (the reference Net2's own default) contains all ten keys of the 2-layer net plus more: it must be
    rejected, never truncated (ModelLocker, flatten_state_dict)."""
    from rebel_b200.models import Net2, flatten_state_dict
    deep = Net2(num_faces=4, num_dice=1, n_hidden=256, n_layers=3, use_layer_norm=True)
    with pytest.raises(RuntimeError, match="unexpected parameter"):
        rela.ModelLocker([torch.jit.script(deep)], "cuda:0")
    with pytest.raises(ValueError):
        flatten_state_dict(deep.state_dict())
    narrow = Net2(num_faces=4, num_dice=1, n_hidden=128, n_layers=2, use_layer_norm=True)
    with pytest.raises(RuntimeError, match="256"):
        rela.ModelLocker([torch.jit.script(narrow)], "cuda:0")


def test_terminating_a_loop_keeps_the_shared_replay_open(rela):
    """DataThreadLoop::terminate wakes a producer blocked on the full ring but must not close the buffer for other users
    (the reference's buffer stays usable after Context.terminate)."""
    r = rela.ValuePrioritizedReplay(8, 0, 1.0, 1.0, 0, False, False)
    ctx = rela.Context()
    ctx.terminate()
    q = torch.zeros(4, 3)
    r.push([q, q.clone(), torch.ones(4)])
    assert r.size() == 4 and r.num_add() == 4


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6), (2, 3)])
@pytest.mark.parametrize("sample_leaf,use_cfr", [(True, True), (False, True), (True, False)])
def test_device_walk_equals_host_walk(rela, D, F, sample_leaf, use_cfr):
    """The self-play walk on the device (mt19937 streams, libstdc++ distributions, fp64 belief updates in kernels) emits the
    same example stream, bit for bit, as the per-game host walk that uses std::mt19937 itself — 96 concurrent games, 12 waves,
    zero net and fp32 net."""
    from rebel_b200.models import flatten_state_dict, make_selfplay_net
    w = torch.from_numpy(flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict()))
    for net_mode, weights in ((0, None), (1, w)):
        out = []
        for host_walk in (1, 0):
            cfg = make_cfg(rela, D, F, sample_leaf=sample_leaf, concurrent_games=96, net_mode=net_mode, state_dtype=0, host_walk=host_walk,
                           subgame_params=dict(num_iters=16, max_depth=2, linear_update=True, use_cfr=use_cfr))
            out.append(rela.run_selfplay_waves(cfg, 0, 11, 12, weights))
        (qh, vh), (qd, vd) = out
        assert qh.shape == qd.shape == (12 * 2 * 96, game_dims(D, F)[2])
        assert torch.equal(qh, qd) and torch.equal(vh, vd), (net_mode, int((qh != qd).sum()), int((vh != vd).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("D,F", [(1, 4), (2, 3)])
def test_every_game_of_a_wave_replays_a_reference_runner(rela, port, D, F):
    """Game g of a loop seeded with s consumes the generator seed s + 10^6 g in the reference's draw order: its example stream
    equals RlRunner(seed = s + 10^6 g) — checked against the oracle port (itself pinned bit-exact to the compiled reference's
    RlRunner) for several games of one device-side wave loop, zero net."""
    K, waves, iters, s = 8, 10, 24, 5
    cfg = make_cfg(rela, D, F, sample_leaf=True, concurrent_games=K, net_mode=0, state_dtype=0,
                   subgame_params=dict(num_iters=iters, max_depth=2, linear_update=True, use_cfr=True))
    q, v = rela.run_selfplay_waves(cfg, 0, s, waves)
    q = q.numpy().reshape(waves, K, 2, -1); v = v.numpy().reshape(waves, K, 2, -1)
    for g in (0, 3, 7):
        rq, rv = port.rl_runner(D, F, s + 1000000 * g, n_games=waves, num_iters=iters, cap=4 * waves * 2 * 8)
        n = waves * 2
        assert len(rq) >= n
        assert np.array_equal(q[:, g].reshape(n, -1), rq[:n]) and np.array_equal(v[:, g].reshape(n, -1), rv[:n]), g


@pytest.mark.gpu
def test_replay_rows_live_on_the_device(rela, tmp_path):
    """SURVEY 8 f-3: with a CUDA device the rows of the ring are in HBM; batches are gathered on the device into the tensors
    sample() returns; host round trips only for save / extract / cpu batches.  Same ring semantics as on the host."""
    Q, H = 27, 6
    r = rela.ValuePrioritizedReplay(capacity=100, seed=1, alpha=1.0, beta=0.4, prefetch=3, use_priority=False, compressed_values=False)
    assert r.storage_device() == -2
    q = torch.arange(120 * Q, dtype=torch.float32).reshape(120, Q)
    v = torch.arange(120 * H, dtype=torch.float32).reshape(120, H)
    r.push([q, v, torch.ones(120)])
    assert r.storage_device() >= 0 and r.size() == 120
    for dev in ("cuda:0", "cpu"):
        batch, w = r.sample(64, dev)
        assert batch.query.device.type == ("cuda" if dev != "cpu" else "cpu")
        rows = (batch.query[:, 0] / Q).long().cpu()
        assert torch.equal(batch.query.cpu(), q[rows]) and torch.equal(batch.values.cpu(), v[rows])
    assert r.size() == 100                                               # sampling evicted down to capacity
    r.push([q[:25].cuda(), v[:25].cuda(), torch.ones(25)])               # CUDA tensors are appended device to device; the ring wraps
    assert r.size() == 125
    path = str(tmp_path / "dump.bin")
    r.save(path)
    r2 = rela.ValuePrioritizedReplay(1000, 2, 1.0, 0.4, 0, False, False)
    r2.load(path, 1.0, -1, 1)
    ex = r2.extract()
    want_q = torch.cat([q[20:120], q[:25]]); want_v = torch.cat([v[20:120], v[:25]])
    assert torch.equal(ex[0], want_q) and torch.equal(ex[1], want_v)
    # many batches on the consumer's stream without synchronising in between, while a producer keeps overwriting the ring
    r3 = rela.ValuePrioritizedReplay(64, 3, 1.0, 0.4, 0, False, False)
    r3.push([q[:64], v[:64], torch.ones(64)])
    got = []
    for i in range(40):
        b, _ = r3.sample(32, "cuda:0")
        got.append(b)
        r3.push([q[i:i + 8], v[i:i + 8], torch.ones(8)])
    torch.cuda.synchronize()
    for b in got:
        rows = (b.query[:, 0] / Q).long().cpu()
        assert torch.equal(b.query.cpu(), q[rows]) and torch.equal(b.values.cpu(), v[rows])


def _last_action_stats(q, v, A, net):
    """The statistic cfvpy/selfplay.py:158-169 logs: per last action (bucket A = "initial") example count, target sum, loss sum."""
    onehot = q[:, 2:2 + A]
    aid = np.where(onehot.sum(1) > 0, onehot.argmax(1), A)
    cnt = np.bincount(aid, minlength=A + 1).astype(np.float64)
    vsum = np.zeros(A + 1); lsum = np.zeros(A + 1)
    np.add.at(vsum, aid, v.astype(np.float64).sum(1))
    with torch.no_grad():
        pred = net(torch.from_numpy(q)).numpy()
    np.add.at(lsum, aid, ((v - pred).astype(np.float64) ** 2).mean(1))
    return cnt, vsum, lsum


def _chi2(a, b):
    """Two-sample chi-square statistic of two count vectors (different totals)."""
    na, nb = a.sum(), b.sum()
    m = (a + b) > 0
    return float((((a * np.sqrt(nb / na) - b * np.sqrt(na / nb)) ** 2)[m] / (a + b)[m]).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("net_name,net_mode", [("fp32", 1), ("tc", 2), ("tcx2", 3)])
@pytest.mark.parametrize("D,F", [(1, 4), (1, 6)])
def test_datagen_distribution_matches_reference(rela, golden, D, F, net_name, net_mode):
    """P5 (SURVEY appendix B): the data-generation loop on the GPU (device walk, 1024 iterations, seed-0 Net2) against >= 40 k
    examples of the reference's RlRunner loops: the per-last-action example counts (chi-square), mean targets and mean losses —
    the statistic selfplay.py:158-169 logs.  The bands are measured, not chosen (fixture datagen_stats.npz, oracle/make_golden_r2.py):
      * fp32 net: the same statistics between two disjoint seed sets (a, b) of the REFERENCE;
      * tensor-core nets: the comparison set may also be the REFERENCE ITSELF with its own net evaluated in the kernels'
        arithmetic (fp16 operands, GELU rounded to fp16: set m1, ref_set_net_emulation); the allowed distance stays the
        seed-to-seed band.
    (This test is what exposed the bias of tanh.approx.f16x2: with the packed-half GELU the 1x6f chi-square was 1050-1200 against a
    seed-to-seed 37, while the reference with the SAME arithmetic but a correctly rounded tanh stayed at 43-45;
    profiles/r2_gelu_table.log, profiles/r2_gelu_variants.log.)
    Only complete games are counted on the GPU side (a wave loop stops mid-game)."""
    from rebel_b200.models import flatten_state_dict, make_selfplay_net
    from test_gpu_parity import _note
    A, H, Q = game_dims(D, F)
    g = golden("datagen_stats.npz")
    net = make_selfplay_net(D, F, seed=0)
    w = torch.from_numpy(flatten_state_dict(net.state_dict()))
    K, waves = 1024, 64
    cfg = make_cfg(rela, D, F, concurrent_games=K, net_mode=net_mode, state_dtype=0)
    q, v = rela.run_selfplay_waves(cfg, 0, 123, waves, w)
    q = q.numpy().reshape(waves, K, 2, Q); v = v.numpy().reshape(waves, K, 2, H)
    starts = q[:, :, 0, 2:2 + A].sum(-1) == 0                      # [waves][K]: the subgame at the initial state = a game starts
    last_start = waves - 1 - np.argmax(starts[::-1], axis=0)       # per slot: wave of its last game start
    keep = np.arange(waves)[:, None] < last_start[None, :]         # everything before the (possibly unfinished) last game
    qk, vk = q[keep].reshape(-1, Q), v[keep].reshape(-1, H)
    assert len(qk) >= 50000
    cnt, vsum, lsum = _last_action_stats(qk, vk, A, net)
    sets = {n: (g[f"count_{n}_{D}x{F}"].astype(np.float64), g[f"val_sum_{n}_{D}x{F}"], g[f"loss_sum_{n}_{D}x{F}"]) for n in ("a", "b")}
    model = {"tc": "m1", "tcx2": "m1"}.get(net_name)       # m2 models the packed-half GELU (gelu_hy_x2) with an ideally rounded tanh
    if model is not None and f"count_{model}_{D}x{F}" in g.files:
        sets[model] = (g[f"count_{model}_{D}x{F}"].astype(np.float64), g[f"val_sum_{model}_{D}x{F}"], g[f"loss_sum_{model}_{D}x{F}"])
    big = np.ones(A + 1, bool)
    for c, _, _ in sets.values():
        big &= c >= 300
    mean = lambda s, c: s[big] / (c[big] * H)
    loss = lambda s, c: s[big] / c[big]

    def dist(x, y):       # (chi2 of the counts, max |mean target difference|, max relative mean-loss difference)
        return (_chi2(x[0], y[0]), np.abs(mean(x[1], x[0]) - mean(y[1], y[0])).max(),
                (np.abs(loss(x[2], x[0]) - loss(y[2], y[0])) / loss(y[2], y[0])).max())
    seed_band = dist(sets["a"], sets["b"])                                               # seed-to-seed spread of the reference
    mine = (cnt, vsum, lsum)
    names = sorted(sets)
    got = [min(dist(mine, sets[n])[k] for n in names) for k in range(3)]                  # distance to the nearest reference set
    to_fp32 = [max(dist(mine, sets[n])[k] for n in ("a", "b")) for k in range(3)]
    moved = [max(dist(sets[model], sets[n])[k] for n in ("a", "b")) for k in range(3)] if model in sets else [0, 0, 0]
    _note(f"P5 {D}x{F}f net={net_name}: {len(qk)} GPU examples vs reference sets {names} ({[int(sets[n][0].sum()) for n in names]} examples); "
          f"chi2 of the last-action counts ({A + 1} buckets): GPU to the nearest set {got[0]:.1f}, to the fp32 sets at most {to_fp32[0]:.1f}; "
          f"reference seed-to-seed {seed_band[0]:.1f}; the reference under the kernel's arithmetic moves by {moved[0]:.1f}; "
          f"max |mean target diff| {got[1]:.2e} (seed-to-seed {seed_band[1]:.2e}, model {moved[1]:.2e}); "
          f"max relative loss diff {got[2]:.2e} (seed-to-seed {seed_band[2]:.2e}, model {moved[2]:.2e})")
    assert got[0] <= 3 * max(seed_band[0], A + 1), (got[0], seed_band[0])
    assert got[1] <= 3 * seed_band[1] + 1e-4, (got[1], seed_band[1])
    assert got[2] <= 3 * seed_band[2] + 0.02, (got[2], seed_band[2])


@pytest.mark.gpu
def test_config5_with_the_value_net_vs_reference(rela, golden):
    """BASELINE config 5 WITH the value net (round 1 pinned it with the zero net only): recursive_eval's 64 sampled recursive
    strategies on 1x4f, 1024 iterations, seed-0 Net2.  Reference = compute_sampled_strategy_recursive_to_leaf with ATen fp32
    (fixture config5_net.npz).  Zero net: bit-identical.  With the net the trajectories are chaotic (SURVEY appendix B), so the
    exploitability of the averaged strategy is compared: the fp32 SIMT net must agree with the reference like the reference's
    two builds agree with each other (3x their difference, at least 2e-3), the tensor-core nets within 1e-2 of it."""
    from rebel_b200.models import flatten_state_dict, make_selfplay_net
    from test_gpu_parity import _note
    g = golden("config5_net.npz")
    D, F, iters, reps = [int(x) for x in g["cfg"]]
    want = g["exploitability"].mean(1)
    self_noise = np.abs(g["exploitability_fast_build"].mean(1) - want) if "exploitability_fast_build" in g.files else np.zeros_like(want)
    w = torch.from_numpy(flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict()))
    got = {}
    for name, mode, weights in (("zero", 0, None), ("fp32", 1, w), ("tc_f16", 2, w), ("tc_f16x2", 3, w)):
        cfg = make_cfg(rela, D, F, net_mode=mode, state_dtype=0, subgame_params=dict(num_iters=iters, max_depth=2, linear_update=True, use_cfr=True))
        r = rela.recursive_eval_sampled(cfg, 0, reps, 0, 64, 8192, weights)
        assert list(r["checkpoints"]) == list(g["checkpoints"])
        got[name] = r["exploitability"].numpy().mean(1)
    assert np.array_equal(got["zero"], g["exploitability_zero_net"].mean(1))
    for name in ("fp32", "tc_f16", "tc_f16x2"):
        d = np.abs(got[name] - want)
        _note(f"config5 1x4f R=64 with Net2, net={name}: exploitability {got[name][-1]:.5f} vs reference {want[-1]:.5f} (|d| = {d[-1]:.2e}; "
              f"over the checkpoints R>=8 max |d| = {d[3:].max():.2e}); reference -O3 vs -O2 builds differ by {self_noise[-1]:.2e}")
    assert np.abs(got["fp32"] - want)[-1] <= max(3 * self_noise[-1], 2e-3)
    for name in ("tc_f16", "tc_f16x2"):
        assert np.abs(got[name] - want)[-1] <= 1e-2, (name, got[name][-1], want[-1])
