"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every call goes through the C ABI (rebel_b200.capi ->
libcfrb200.so); the CPU oracle (oracle/) is only the checker.

Protocol (SURVEY.md appendix B, DESIGN.md section 2): integers bit-exact (P1); teacher-forced single CFR steps from oracle
state with tolerances set by the arithmetic of the configuration and regret-matching conditioning masks (P2); iterations 1-2
from the initial state against the golden fixtures generated from the compiled reference (P3); 1024-iteration results against
the reference's own self-noise band (P4); size-independent properties at BASELINE sizes.
"""
import os

import numpy as np
import pytest

from oracle.oracle import game_dims

pytestmark = pytest.mark.gpu

SHAPES = [(1, 4), (1, 6), (2, 3)]


@pytest.fixture(scope="module")
def rb():
    import rebel_b200
    assert rebel_b200.capi.lib().cfrb_device_count() > 0, "no CUDA device: the CUDA path cannot be tested"
    return rebel_b200


def _note(msg):
    """Measured parity numbers end up in gpurun_out/parity_notes.log (copied to profiles/ when they are quoted)."""
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "parity_notes.log"), "a") as f:
        f.write(msg + "\n")


def pad_nodes(x, nmax):
    out = np.zeros((1, nmax) + x.shape[1:], np.float64)
    out[0, :x.shape[0]] = x
    return out


def steps_after(c):
    return np.array([[(c + 1) // 2, c // 2]], np.int32)


# value-noise level of a configuration: what one step may differ from the fp64 oracle in a node value
def noise_level(rb, state, net):
    if net == rb.NET_TC_F16:
        return 1e-5          # fp16 operands: ~5e-4 rms relative on net outputs of scale 1e-2
    if net == rb.NET_TC_F16X2:
        return 1.5e-5        # + GELU on packed fp16 pairs: ~8e-4 rms relative (scripts/gelu_probe.py)
    if state == rb.STATE_F32:
        return 4e-7
    if net == rb.NET_FP32:
        return 3e-8          # fp32 net vs the oracle's scalar fp32 net
    return 1e-13             # fp64 tables, no net: only operation order / FMA contraction


# ---------------------------------------------------------------------------------------------- P1
def test_tree_templates_bit_exact(rb, golden, port):
    g = golden("trees.npz")
    for key in g.files:
        _, D, F, lb, pl, md = (int(x) if x.lstrip("-").isdigit() else x for x in key.split("_"))
        if md > 3 or md == 0:
            continue
        s = rb.WaveSolver(D, F, 1, max_depth=md, net_mode=rb.NET_ZERO)
        t = s.tree(lb, pl)
        assert t.shape == g[key].shape and (t == g[key]).all(), key
        s.close()
    for (D, F) in SHAPES:   # every root template of the data-gen configuration vs the oracle
        A, H, Q = game_dims(D, F)
        s = rb.WaveSolver(D, F, 1, max_depth=2, net_mode=rb.NET_ZERO)
        for lb in range(-1, A - 1):
            for pl in (0, 1):
                assert (s.tree(lb, pl) == port.unroll_tree(D, F, lb, pl, 2)).all()
        s.close()


# ---------------------------------------------------------------------------------------------- P2
def conditioning(tree, R_next, trav, noise):
    """Per (node, hand): is the oracle's regret matching well conditioned at this noise level?  Returns tol_sigma [N,H]
    (inf where it is not: near-ties / sign noise, SURVEY appendix B) and path_tol [N,H], the tolerance accumulated
    over the traverser's ancestors (their sigma enters the reach that weights the sum-strategy update)."""
    N, H = R_next.shape[0], R_next.shape[1]
    nchild = tree[:, 3] - tree[:, 2]
    tol = np.zeros((N, H))
    mine = (nchild > 0) & (tree[:, 1] == trav)
    for n in np.nonzero(mine)[0]:
        lo = tree[n, 0] + 1 if tree[n, 0] >= 0 else 0
        r = R_next[n, :, lo:lo + nchild[n]]
        sumpos = np.maximum(r, 0).sum(-1)
        good_pos = (sumpos > 1e3 * noise) & (np.abs(r).min(-1) > 30 * noise)     # no regret sits on the sign boundary
        good_neg = (r.max(-1) < -30 * noise) | (np.abs(r).max(-1) == 0)          # all negative, or exactly untouched: uniform
        tol[n] = np.where(good_pos, 20 * noise / np.maximum(sumpos, 1e-300) + 10 * noise, np.where(good_neg, 10 * noise, np.inf))
    path_tol = np.zeros((N, H))
    for n in range(N):
        if nchild[n] == 0:
            continue
        here = path_tol[n] + (tol[n] if mine[n] else 0.0)
        for c in range(tree[n, 2], tree[n, 3]):
            path_tol[c] = here
    return tol, path_tol


CONFIGS = [("f64", "zero"), ("f64", "fp32"), ("f32", "zero"), ("f32", "fp32"), ("f64", "tc"), ("f64", "tcx2")]
NETS = lambda rb: {"zero": rb.NET_ZERO, "fp32": rb.NET_FP32, "tc": rb.NET_TC_F16, "tcx2": rb.NET_TC_F16X2}


@pytest.mark.parametrize("D,F", SHAPES + [(2, 4)])
@pytest.mark.parametrize("state_name,net_name", CONFIGS)
@pytest.mark.parametrize("max_depth", [2, 3])
def test_teacher_forced_single_step(rb, port, net_weights, monkeypatch, D, F, state_name, net_name, max_depth):
    if net_name in ("tc", "tcx2") and max_depth != 2:
        pytest.skip("tensor-core net is exercised on the data-generation depth")
    if (D, F) == (2, 4):
        # 16 hands on the generic CFR kernel, bit for bit: at depth 3 the scratch needs a CTA per subgame
        # (cfr_iter_kernel<double, 256, 0>), at depth 2 CFRB_NO_D2=1 selects the 16-hand warp kernel (cfr_iter_kernel<double, 32, 16>)
        if (state_name, net_name) != ("f64", "zero"):
            pytest.skip("2x4f covers the generic kernel's 16-hand paths in the bit-exact configuration")
        monkeypatch.setenv("CFRB_NO_D2", "1")
    A, H, Q = game_dims(D, F)
    state = {"f64": rb.STATE_F64, "f32": rb.STATE_F32}[state_name]
    net = NETS(rb)[net_name]
    noise = noise_level(rb, state, net)
    # fp32 tables + value net: the reference's 1e-80 smoothing cannot be represented, so the query of a leaf reached with zero
    # probability carries uniform beliefs instead of the reference's epsilon mixture and the net output there differs at
    # the 1e-3 level (documented deviation of CFRB_STATE_F32, DESIGN.md); CFRB_STATE_F64 (the default) has no such term
    if state == rb.STATE_F32 and net != rb.NET_ZERO:
        noise = 2e-4
    w = net_weights(D, F) if net != rb.NET_ZERO else None
    cps = [0, 1, 2, 3, 4, 5, 16, 17, 18, 101, 102, 103]
    roots = [(-1, 0), (-1, 1), (1, 1), (A - 4, 0)]
    S = rb.WaveSolver(D, F, 1, max_depth=max_depth, net_mode=net, state_dtype=state)
    if w is not None:
        S.set_weights(w)
    compared = skipped = 0
    worst = {"regrets": 0.0, "mu": 0.0, "last": 0.0, "sum": 0.0}
    for ri, (lb, pl) in enumerate(roots):
        b = port.synthetic_beliefs(H, 300 + ri)
        o = port.cfr_solve(D, F, b, cps, lb, pl, num_iters=max(cps), max_depth=max_depth, net_w=w)
        tree, N = o["tree"], o["tree"].shape[0]
        nchild = tree[:, 3] - tree[:, 2]
        for ci, c in enumerate(cps[:-1]):
            if cps[ci + 1] != c + 1:
                continue
            trav = c % 2
            S.begin([lb], [pl], b[None])
            S.load_state(regrets=pad_nodes(o["regrets"][ci], S.Nmax), last=pad_nodes(o["last"][ci], S.Nmax),
                         sum=pad_nodes(o["sum"][ci], S.Nmax), root_means=o["root_means"][ci][None],
                         num_steps=steps_after(c), iterations_done=c)
            S.run(1)
            g = S.fetch(("root_means", "last", "sum", "regrets"))
            tag = f"{D}x{F}f d{max_depth} {state_name}/{net_name} root={lb},{pl} step {c}->{c + 1}"
            if state == rb.STATE_F64 and net == rb.NET_ZERO:
                # fp64 tables without a net: every operation is the reference's, in the reference's order -> bit-identical
                for k_ in ("regrets", "last", "sum"):
                    assert np.array_equal(g[k_][0, :N], o[k_][ci + 1]), (tag, k_, "not bit-exact",
                                                                         np.abs(g[k_][0, :N] - o[k_][ci + 1]).max())
                assert np.array_equal(g["root_means"][0], o["root_means"][ci + 1]), (tag, "mu not bit-exact")
            Rn = o["regrets"][ci + 1]
            dR = np.abs(g["regrets"][0, :N] - Rn)
            worst["regrets"] = max(worst["regrets"], dR.max())
            assert (dR <= 10 * noise * (1 + np.abs(Rn))).all(), (tag, "regrets", dR.max())
            dmu = np.abs(g["root_means"][0] - o["root_means"][ci + 1])
            worst["mu"] = max(worst["mu"], dmu.max())
            assert dmu.max() < 10 * noise, (tag, "mu", dmu.max())
            tol, path_tol = conditioning(tree, Rn, trav, noise)
            mine = (nchild > 0) & (tree[:, 1] == trav)
            keep = 4e-7 if state == rb.STATE_F32 else 1e-15          # representation error of an untouched table entry
            for n in range(N):
                if nchild[n] == 0:
                    continue
                ds = np.abs(g["last"][0, n] - o["last"][ci + 1][n]).max(-1)       # [H]
                dS = np.abs(g["sum"][0, n] - o["sum"][ci + 1][n]).max(-1)
                if not mine[n]:
                    assert ds.max() <= keep and dS.max() <= keep * max(1.0, np.abs(o["sum"][ci + 1][n]).max()), (tag, "untouched node", n)
                    continue
                ok = np.isfinite(tol[n]) & np.isfinite(path_tol[n])
                compared += ok.sum(); skipped += (~ok).sum()
                if ok.any():
                    worst["last"] = max(worst["last"], ds[ok].max()); worst["sum"] = max(worst["sum"], dS[ok].max())
                assert (ds[ok] <= tol[n][ok]).all(), (tag, "last", n, ds, tol[n])
                assert (dS[ok] <= tol[n][ok] + path_tol[n][ok] + 10 * noise).all(), (tag, "sum", n, dS, tol[n], path_tol[n])
            if net != rb.NET_ZERO and o["queries"].shape[1]:
                q, out, sc = S.leaf_io()
                qtol = 1e-3 if net in (rb.NET_TC_F16, rb.NET_TC_F16X2) else 2e-6        # fp16 query rows: 2^-11 relative on values <= 1
                dq = np.abs(q - o["queries"][ci + 1])
                lv = np.abs(out * sc[:, None] - o["leaf_values"][ci + 1])
                if state == rb.STATE_F32:
                    # documented deviation of fp32 tables: the reference's 1e-80 smoothing does not exist in fp32, so a
                    # belief segment with zero reach is uniform instead of the reference's epsilon mixture; such rows
                    # (and the net outputs computed from them) are excluded
                    seg = q[:, 2 + A:].reshape(-1, 2, H)
                    bad = (seg == np.float32(1.0 / H)).all(-1).any(-1)
                    dq, lv = dq[~bad], lv[~bad]
                if dq.size:
                    assert dq.max() < qtol, (tag, "queries", dq.max())
                    assert lv.max() < 10 * noise, (tag, "leaf values", lv.max())
    S.close()
    _note(f"P2 {D}x{F}f d{max_depth} {state_name}/{net_name}: noise {noise:g}; compared {compared} (node,hand) rows, skipped "
          f"{skipped} ill-conditioned; worst abs diff " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    if noise < 1e-5:     # at fp16-operand / epsilon-deviation noise most regrets of an untrained net's tiny values are near-ties
        assert compared > skipped, (compared, skipped)


# ---------------------------------------------------------------------------------------------- P3
@pytest.mark.parametrize("D,F", SHAPES)
def test_short_horizon_vs_golden(rb, golden, net_weights, D, F):
    for fixture, mode, tol in ((f"cfr_zero_{D}x{F}.npz", rb.NET_ZERO, 1e-11), (f"cfr_net_{D}x{F}.npz", rb.NET_FP32, 2e-5)):
        g = golden(fixture)
        cps = list(g["checkpoints"])
        n = len(g["roots"])
        S = rb.WaveSolver(D, F, n, net_mode=mode)
        if mode != rb.NET_ZERO:
            S.set_weights(net_weights(D, F))
        S.begin(g["roots"][:, 0], g["roots"][:, 1], np.stack([g[f"beliefs{i}"] for i in range(n)]))
        done = 0
        for ci, c in enumerate(cps):
            if c > 2:
                break
            S.run(c - done); done = c
            f = S.fetch(("root_means", "last", "sum", "regrets", "avg"))
            for i in range(n):
                N = g[f"regrets{i}"].shape[1]
                for k in ("regrets", "last", "sum", "avg"):
                    d = np.abs(f[k][i, :N] - g[f"{k}{i}"][ci]).max()
                    assert d < tol, (fixture, k, i, c, d)
                assert np.abs(f["root_means"][i] - g[f"root_means{i}"][ci]).max() < tol
        S.close()


@pytest.mark.parametrize("D,F", SHAPES)
def test_zero_net_trajectories_bit_exact_vs_reference(rb, golden, D, F):
    """fp64 tables, zero net: whole trajectories (64 iterations) are bit-identical to the compiled reference
    (-ffp-contract=off build): regrets, last / sum / average strategies and root value means."""
    g = golden(f"cfr_zero_{D}x{F}.npz")
    cps = list(g["checkpoints"])
    n = len(g["roots"])
    S = rb.WaveSolver(D, F, n, net_mode=rb.NET_ZERO)
    S.begin(g["roots"][:, 0], g["roots"][:, 1], np.stack([g[f"beliefs{i}"] for i in range(n)]))
    done = 0
    for ci, c in enumerate(cps):
        S.run(c - done); done = c
        f = S.fetch(("root_means", "last", "sum", "regrets", "avg"))
        for i in range(n):
            N = g[f"regrets{i}"].shape[1]
            for k in ("regrets", "last", "sum", "avg"):
                assert np.array_equal(f[k][i, :N], g[f"{k}{i}"][ci]), (k, i, c, np.abs(f[k][i, :N] - g[f"{k}{i}"][ci]).max())
            assert np.array_equal(f["root_means"][i], g[f"root_means{i}"][ci]), (i, c)
    S.close()


@pytest.mark.parametrize("D,F", SHAPES)
@pytest.mark.parametrize("max_depth", [2, 3])
def test_discount_variants_vs_reference(rb, golden, port, D, F, max_depth):
    """Vanilla CFR (no discounting) is bit-identical to the reference like linear CFR; DCFR evaluates n^alpha with CUDA's pow,
    which may differ from glibc's by an ulp, so its 8-iteration trajectories are compared to 1e-12."""
    from oracle.make_golden import VARIANTS
    g = golden("cfr_variants.npz")
    cps = list(g["checkpoints"])
    b = g[f"beliefs_{D}x{F}"]
    for name, kw in VARIANTS.items():
        S = rb.WaveSolver(D, F, 2, max_depth=max_depth, net_mode=rb.NET_ZERO, **kw)
        S.begin(np.array([1, 1], np.int32), np.array([1, 1], np.int32), np.stack([b, b]))
        ref = port.cfr_solve(D, F, b, cps, 1, 1, num_iters=8, max_depth=max_depth, **kw)
        done = 0
        for ci, c in enumerate(cps):
            S.run(c - done); done = c
            f = S.fetch(("root_means", "last", "sum", "regrets", "avg"))
            for k in ("regrets", "last", "sum", "avg"):
                x, y = f[k][0, :ref[k].shape[1]], ref[k][ci]
                if max_depth == 2:
                    assert np.array_equal(y, g[f"{k}_{name}_{D}x{F}"][ci])     # the port run IS the golden reference run
                if name == "vanilla":
                    assert np.array_equal(x, y), (name, k, c)
                else:
                    assert np.abs(x - y).max() < 1e-12, (name, k, c, np.abs(x - y).max())
            assert np.abs(f["root_means"][0] - ref["root_means"][ci]).max() < 1e-12
            assert np.array_equal(f["regrets"][0], f["regrets"][1])
        S.close()


@pytest.mark.parametrize("D,F", SHAPES)
def test_fictitious_play_bit_exact_vs_reference(rb, golden, port, net_weights, D, F):
    """CFRB_SOLVER_FP (the reference's other ISubgameSolver, build_solver with use_cfr = false): zero net, fp64 tables —
    33-iteration trajectories of last / sum / average strategies and root value means are bit-identical to the compiled
    reference for linear, plain and optimistic averaging at depth 2, 3 and full depth; with the fp32 value net two iterations
    from the initial state agree with the oracle to fp32 accuracy."""
    from oracle.make_golden import FP_CASES, FP_CPS, FP_ROOTS
    g = golden("fp_zero.npz")
    b = g[f"beliefs_{D}x{F}"]
    for (lin, opt, md) in FP_CASES:
        if md > 3 and (D, F) != (1, 4):
            continue
        S = rb.WaveSolver(D, F, len(FP_ROOTS), max_depth=md, net_mode=rb.NET_ZERO, linear_update=lin, solver=rb.SOLVER_FP, optimistic=opt)
        S.begin(np.array([r[0] for r in FP_ROOTS], np.int32), np.array([r[1] for r in FP_ROOTS], np.int32), np.stack([b] * len(FP_ROOTS)))
        done = 0
        for ci, c in enumerate(FP_CPS):
            S.run(c - done); done = c
            f = S.fetch(("root_means", "last", "sum", "avg"))
            for i, (lb, pl) in enumerate(FP_ROOTS):
                for k in ("last", "sum", "avg"):
                    y = g[f"{k}_{int(lin)}{int(opt)}{md}_{lb}_{D}x{F}"][ci]
                    x = f[k][i, :y.shape[0]]
                    assert np.array_equal(x, y), (lin, opt, md, lb, k, c, np.abs(x - y).max())
                assert np.array_equal(f["root_means"][i], g[f"root_means_{int(lin)}{int(opt)}{md}_{lb}_{D}x{F}"][ci]), (lin, opt, md, lb, c)
        S.close()
    w = net_weights(D, F)
    S = rb.WaveSolver(D, F, 1, net_mode=rb.NET_FP32, solver=rb.SOLVER_FP)
    S.set_weights(w)
    S.begin([-1], [0], b[None])
    S.run(2)
    o = port.fp_solve(D, F, b, [2], -1, 0, num_iters=2, net_w=w)
    f = S.fetch(("root_means", "avg", "sum"))
    assert np.abs(f["root_means"][0] - o["root_means"][0]).max() < 3e-6
    assert np.abs(f["sum"][0, :o["sum"].shape[1]] - o["sum"][0]).max() < 1e-5
    S.close()


# ---------------------------------------------------------------------------------------------- P4
@pytest.mark.parametrize("D,F", SHAPES)
@pytest.mark.parametrize("net_name", ["fp32", "tc", "tcx2"])
def test_long_horizon_within_reference_noise(rb, golden, net_weights, D, F, net_name):
    """1024 iterations with the Net2 value net: root value means vs the reference.  fp32 net: the reference moves by mean
    2.1e-4 / max 2.8e-3 under a ONE-ulp fp32 perturbation of its net outputs (SURVEY appendix B, 'pert'); that band, or 3x the
    reference's own FMA/no-FMA self-noise when larger, is the criterion.  Tensor-core nets: the band is DERIVED, not chosen —
    the REFERENCE solver is run with its own net perturbed the way the tcgen05 kernels perturb it (weights rounded to fp16; on top
    of that, independent relative noise on every output at the kernels' measured level, 5.4e-4 — both GELU variants measure
    4.7e-4 .. 5.0e-4 — 8 seeds; tests/golden/net_band.npz from oracle/make_golden_r2.py), and the GPU must stay within 3x the
    mean response of the reference to that perturbation (or 3x its self-noise, or the fp32 band, whichever is larger)."""
    g = golden(f"cfr_net_{D}x{F}.npz")
    nb = golden("net_band.npz")
    n = len(g["roots"])
    S = rb.WaveSolver(D, F, n, net_mode=NETS(rb)[net_name])
    S.set_weights(net_weights(D, F))
    S.begin(g["roots"][:, 0], g["roots"][:, 1], np.stack([g[f"beliefs{i}"] for i in range(n)]))
    S.run(1024)
    mu = S.fetch(("root_means",))["root_means"]
    for i in range(n):
        a, b = g[f"mu1024_nofma{i}"], g[f"mu1024_fast{i}"]
        self_noise = np.abs(a - b).mean()
        d = np.abs(mu[i] - a)
        band_mean, band_max = max(7e-4, 3 * self_noise), 1e-2
        if net_name != "fp32":
            si = 0                                                     # sigma = 5.4e-4 (the 7.7e-4 set belonged to the packed-half GELU)
            pert = np.abs(nb[f"mu_pert{si}_{D}x{F}_{i}"] - a)                      # [seeds][2][H]
            w16 = np.abs(nb[f"mu_w16_{D}x{F}_{i}"] - a)
            response = max(pert.mean(), w16.mean())
            band_mean = max(band_mean, 3 * response)
            band_max = max(band_max, 3 * max(pert.max(), w16.max()))
            _note(f"P4 {D}x{F}f net={net_name} root{i}: mean|dmu|={d.mean():.3e} max={d.max():.3e} | reference under the same perturbation: "
                  f"fp16 weights {w16.mean():.3e}, + output noise {pert.mean():.3e} (max {pert.max():.3e}); self-noise {self_noise:.3e}; band {band_mean:.2e}")
        else:
            _note(f"P4 {D}x{F}f net={net_name} root{i}: mean|dmu|={d.mean():.3e} max={d.max():.3e} ref-self-noise mean={self_noise:.3e}")
        assert d.mean() <= band_mean, (D, F, i, d.mean(), band_mean)
        assert d.max() <= band_max, (D, F, i, d.max(), band_max)
    S.close()


@pytest.mark.parametrize("D,F", [(1, 2), (1, 3), (1, 4), (1, 6), (2, 3)])
def test_gpu_best_response_bit_exact(rb, golden, port, D, F):
    """cfrb_exploitability (SURVEY 8f-1: BRSolver::compute_br + compute_exploitability2 on the GPU) against the golden
    exploitabilities of the compiled reference and, on random strategies over the whole tree, against the oracle."""
    A, H, Q = game_dims(D, F)
    S = rb.WaveSolver(D, F, 1, net_mode=rb.NET_ZERO)
    if (D, F) in ((1, 2), (1, 3), (1, 4)):
        g = golden("fulltree.npz")
        assert np.array_equal(S.exploitability(g[f"avg16_{D}x{F}"]), g[f"expl_{D}x{F}_nofma"][0])
    else:
        g = golden("recursive_eval_zero.npz")
        ss, sr = g[f"summed_strategy_{D}x{F}"], g[f"summed_reach_{D}x{F}"]
        assert np.array_equal(S.exploitability((ss / (sr + np.float32(1e-6))).astype(np.float64)), g[f"exploitability_{D}x{F}"][-1])
    tree = port.unroll_tree(D, F)
    rng = np.random.RandomState(3)
    for rep in range(2):
        s = np.zeros((len(tree), H, A))
        for n, (lb, pl, cb, ce, par, dep) in enumerate(tree):
            if ce > cb:
                lo = 0 if lb < 0 else lb + 1
                x = rng.rand(H, ce - cb) ** 3
                if rep:
                    x[rng.rand(H, ce - cb) < 0.5] = 0        # sparse strategies: zero reach below many nodes
                    x[:, 0] += 1e-3
                s[n, :, lo:lo + ce - cb] = x / x.sum(-1, keepdims=True)
        assert np.array_equal(S.exploitability(s), port.exploitability(D, F, s)), rep
    S.close()


@pytest.mark.parametrize("state_name", ["f64", "f32"])
def test_full_tree_exploitability_1x4f(rb, golden, port, state_name):
    """BASELINE config 0 on the GPU: full-depth 1x4f tree (511 nodes, CTA-per-subgame path), 1024 linear-CFR iterations,
    exploitability of the average strategy evaluated by the oracle's best response."""
    g = golden("fulltree.npz")
    D, F = 1, 4
    A, H, Q = game_dims(D, F)
    S = rb.WaveSolver(D, F, 1, max_depth=100, net_mode=rb.NET_ZERO, state_dtype=rb.STATE_F64 if state_name == "f64" else rb.STATE_F32)
    S.begin([-1], [0], np.full((1, 2, H), 1.0 / H))
    S.run(16)
    avg16 = S.fetch(("avg",))["avg"][0]
    S.run(1008)
    avg = S.fetch(("avg",))["avg"][0]
    e16 = port.exploitability(D, F, avg16).mean()
    e = port.exploitability(D, F, avg).mean()
    # the GPU best response (cfrb_exploitability, K5) is bit-identical to compute_exploitability2
    assert np.array_equal(S.exploitability(avg16), port.exploitability(D, F, avg16))
    assert np.array_equal(S.exploitability(avg), port.exploitability(D, F, avg))
    ref_a, ref_b = g["expl_1x4_nofma"][1].mean(), g["expl_1x4_fast"][1].mean()
    _note(f"full-tree 1x4f {state_name} exploitability: @16 gpu={e16:.4e} ref={g['expl_1x4_nofma'][0].mean():.4e}; "
          f"@1024 gpu={e:.4e} ref_nofma={ref_a:.4e} ref_fast={ref_b:.4e}")
    if state_name == "f64":
        assert 0 <= e < 1e-3                                                # the reference tests' own threshold
        assert np.array_equal(avg16[:g["avg16_1x4"].shape[0]], g["avg16_1x4"]), "average strategy @16 not bit-exact"
        assert abs(e - ref_a) < 1e-15, (e, ref_a, ref_b)                    # same trajectory as the reference, bit for bit
    else:
        # fp32 tables: the same algorithm in fp32 ON THE CPU ends at 8.8e-4 (vs 5.8e-4 in fp64): a precision floor, not
        # a kernel property (DESIGN.md section 2); only convergence is asserted.
        assert 0 <= e < 2.5e-3
    S.close()


# ---------------------------------------------------------------------------------------------- properties at full size
@pytest.mark.parametrize("net_name", ["fp32", "tc", "tcx2"])
def test_full_size_properties_1x6f(rb, port, net_weights, net_name):
    """BASELINE config 2 shape: 8192 concurrent 1x6f subgames (ragged mix of all root templates)."""
    D, F, K = 1, 6, 8192
    A, H, Q = game_dims(D, F)
    net = NETS(rb)[net_name]
    rng = np.random.RandomState(0)
    lb = rng.randint(-1, A - 1, size=K).astype(np.int32)
    lb[:64] = -1
    pl = rng.randint(0, 2, size=K).astype(np.int32)
    b = rng.rand(K, 2, H); b /= b.sum(-1, keepdims=True)
    act = rng.randint(0, 33, size=K).astype(np.int32)
    dup = [(5, 4000), (17, 8191), (63, 64)]                # identical subgames in different slots
    for s, d in dup:
        lb[d], pl[d], b[d], act[d] = lb[s], pl[s], b[s], act[s]
    S = rb.WaveSolver(D, F, K, net_mode=net)
    S.set_weights(net_weights(D, F))
    outs = []
    for rep in range(2):
        S.begin(lb, pl, b, act)
        S.run(2)
        early = S.fetch(("root_means",))["root_means"].copy()
        S.run(30)
        outs.append(S.fetch(("root_means", "last", "avg", "snapshot")))
    for k in outs[0]:                                        # run-to-run determinism
        assert np.array_equal(outs[0][k], outs[1][k]), k
    f = outs[0]
    if net_name == "fp32":
        for s, d in dup:                                     # slot independence (the tensor-core net accumulates per tile
            for k in f:                                      # in hardware order, so this is asserted for the fp32 net)
                assert np.array_equal(f[k][s], f[k][d]), (k, s, d)
    for k in ("last", "avg", "snapshot"):                    # distributions over legal actions
        x = f[k]
        assert (x >= 0).all() and np.isfinite(x).all()
        sums = x.sum(-1)
        inner = sums > 0
        assert np.abs(sums[inner] - 1).max() < 1e-9
    tol = 2e-6 if net_name == "fp32" else 1e-4
    for k in rng.choice(K, 6, replace=False):                # spot check against the oracle after 2 iterations
        o = port.cfr_solve(D, F, b[k], [2], lb[k], pl[k], num_iters=2, net_w=net_weights(D, F))
        assert np.abs(early[k] - o["root_means"][0]).max() < tol
    q, v = S.examples()                                      # training examples (update_value_network)
    assert q.shape == (K, 2, Q) and v.shape == (K, 2, H)
    assert np.array_equal(v, f["root_means"].astype(np.float32))
    assert (q[:, 0, 0] == pl).all() and (q[:, 0, 1] == 0).all() and (q[:, 1, 1] == 1).all()
    onehot = q[:, 0, 2:2 + A]
    assert ((onehot.argmax(-1) == lb) | (lb < 0)).all() and (onehot.sum(-1) == (lb >= 0)).all()
    assert np.abs(q[:, 0, 2 + A:2 + A + H] - b[:, 0]).max() < 1e-6
    S.close()


@pytest.mark.parametrize("net_name", ["tc_f16x2", "tc_f16"])
@pytest.mark.parametrize("D,F", [(1, 6), (2, 3)])
def test_value_net_rows_do_not_depend_on_their_tile(rb, port, net_weights, D, F, net_name):
    """The two-tiles-in-flight tcgen05 kernel (leaf_mlp_tc3.cuh) evaluates every query row on its own: the outputs of a subgame's
    rows are bit-identical whether the wave has 1, 2, 3, 149 or 1300 subgames (CTAs with a single tile, an odd / even number of
    tiles, first and second TMEM A-operand region, partial last tile), and match the fp32 oracle net within fp16 tolerance."""
    A, H, Q = game_dims(D, F)
    Kmax = 1300
    rng = np.random.RandomState(5)
    b = rng.rand(Kmax, 2, H); b /= b.sum(-1, keepdims=True)
    lb = rng.randint(-1, A - 2, size=Kmax).astype(np.int32); lb[:4] = -1
    pl = rng.randint(0, 2, size=Kmax).astype(np.int32)
    w = net_weights(D, F)
    mode = getattr(rb, "NET_" + net_name.upper())
    ref = None
    for K in (Kmax, 1, 2, 3, 149):
        S = rb.WaveSolver(D, F, K, net_mode=mode)
        S.set_weights(w)
        S.begin(lb[:K], pl[:K], b[:K])
        S.run(2)
        q, o, sc = S.leaf_io()
        mu = S.fetch(("root_means",))["root_means"]
        S.close()
        if ref is None:
            ref = (q, o, mu)
            want = port.net2_forward(w, Q, 256, H, q)
            err = np.abs(o - want)
            assert err.max() < 4e-3 * max(1.0, np.abs(want).max()) and err.mean() < 4e-4, (err.max(), err.mean())
        else:
            n = len(q)
            assert np.array_equal(q, ref[0][:n]) and np.array_equal(o, ref[1][:n]) and np.array_equal(mu, ref[2][:K]), K


def test_snapshot_matches_strategy_at_act_iteration(rb, port):
    D, F = 1, 4
    A, H, Q = game_dims(D, F)
    n = 12
    lb = np.array([-1, 0, 2, 5, -1, 1, 3, 6, -1, 4, 0, 2], np.int32)
    pl = (np.arange(n) % 2).astype(np.int32)
    b = np.stack([port.synthetic_beliefs(H, 40 + i) for i in range(n)])
    act = np.array([0, 1, 2, 3, 7, 8, 16, 5, 20, 11, 20, 0], np.int32)
    S = rb.WaveSolver(D, F, n, net_mode=rb.NET_ZERO)
    S.begin(lb, pl, b, act)
    S.run(20)
    snap = S.fetch(("snapshot",))["snapshot"]
    for a in np.unique(act):
        S.begin(lb, pl, b, None)
        S.run(int(a))
        last = S.fetch(("last",))["last"]
        for k in np.nonzero(act == a)[0]:
            assert np.array_equal(snap[k], last[k]), (k, a)
    S.close()


def test_snapshot_of_act_iteration_zero_needs_no_run(rb, port):
    """act_iteration == 0 (probability 1/136 per subgame in the sampled recursive evaluation at 32 iterations; always possible
    in RlRunner): the sampling strategy is the CFR constructor's uniform one and must be in the snapshot even when cfrb_run
    is called with 0 iterations (or not at all) — on a fresh handle and after a previous wave left other data there."""
    D, F = 1, 6
    A, H, Q = game_dims(D, F)
    S = rb.WaveSolver(D, F, 8, net_mode=rb.NET_ZERO)
    lb = np.array([-1, 3, 0], np.int32); pl = np.array([0, 1, 1], np.int32)
    b = np.stack([port.synthetic_beliefs(H, 70 + i) for i in range(3)])
    for rnd in range(2):
        if rnd == 1:      # leave a non-uniform snapshot of another wave behind first
            S.begin(lb, pl, b, np.array([4, 4, 4], np.int32))
            S.run(6)
        S.begin(lb, pl, b, np.array([0, 0, 0], np.int32))
        S.run(0)
        snap = S.fetch(("snapshot",))["snapshot"]
        S.begin(lb, pl, b, None)
        init = S.fetch(("last",))["last"]                   # the constructor's uniform strategy
        assert np.array_equal(snap, init) and snap.max() > 0, rnd
    S.close()


def test_fast_division_is_correctly_rounded(rb):
    """cfr_iter_d2_kernel obtains sigma = max(R, eps) / sum from the reciprocal of the sum (one true division per (node, hand))
    and two fused multiply-add correction steps instead of one IEEE division per action.  The quotients must be the correctly
    rounded ones — the bits `/` gives — or the solver would leave the reference's trajectory: 4.3e9 pseudo-random operand pairs
    (uniform mantissas, denominators next to 1 and 2, quotients within a few ulp of 1, the 1e-80 scale, small-integer multiples)."""
    S = rb.WaveSolver(1, 4, 1, net_mode=rb.NET_ZERO)
    bad = sum(S.div_check(seed, 1024) for seed in (1, 2, 3, 4))
    S.close()
    assert bad == 0, bad


def test_fast_gelu_is_unbiased(rb):
    """The value-net epilogue's fast GELU on EVERY fp16 input (cfrb_debug_gelu_table): the default fp32-tanh evaluation must be
    as good as rounding the exact erf-GELU to fp16 — no systematic error.  The packed-fp16 evaluation of the same formula (an
    earlier epilogue, now only a table of cfrb_debug_gelu_table) is measured next to it: tanh.approx.f16x2 truncates towards zero, which biases every activation with |y| > 0.5 by -1.6e-4 ..
    -3.9e-4; in the self-play loop that coherent bias moved the generated distribution (P5) although its rms error (6.3e-4 of
    the net output against 5.0e-4) looked harmless."""
    from scipy.special import erf
    S = rb.WaveSolver(1, 4, 1, net_mode=rb.NET_ZERO)
    x, _ = S.gelu_table(0)
    _, half = S.gelu_table(1)
    _, t32 = S.gelu_table(2)
    S.close()
    hy = x.astype(np.float64)
    worst32 = worst16 = 0.0
    for lo, hi in ((-4, -2), (-2, -1), (-1, -0.25), (0.25, 1), (1, 2)):
        m = np.isfinite(hy) & (hy >= lo) & (hy < hi)
        y = 2 * hy[m]
        exact = 0.5 * y * (1 + erf(y / np.sqrt(2)))
        rounding = np.sqrt(((exact.astype(np.float16).astype(np.float64) - exact) ** 2).mean())
        e32, e16 = t32.astype(np.float64)[m] - exact, half.astype(np.float64)[m] - exact
        _note(f"fast GELU, y/2 in [{lo},{hi}): fp32 tanh mean {e32.mean():+.2e} rms {np.sqrt((e32 ** 2).mean()):.2e} | packed half mean {e16.mean():+.2e} "
              f"rms {np.sqrt((e16 ** 2).mean()):.2e} | exact GELU rounded to fp16: rms {rounding:.2e}")
        assert np.sqrt((e32 ** 2).mean()) <= 1.05 * rounding + 5e-5, (lo, hi)
        worst32, worst16 = max(worst32, abs(e32.mean())), max(worst16, abs(e16.mean()))
    assert worst32 <= 1e-4, worst32            # measured 7.9e-5 on [1, 2) (where one fp16 ulp is 9.8e-4 .. 2e-3), <= 8e-6 elsewhere
    assert worst16 >= 1.5e-4, worst16          # the documented bias of the packed-half variant (not the default)


def test_edge_cases_and_errors(rb, port):
    D, F = 1, 4
    A, H, Q = game_dims(D, F)
    S = rb.WaveSolver(D, F, 4, net_mode=rb.NET_FP32)
    b = np.full((1, 2, H), 1.0 / H)
    S.begin([-1], [0], b)
    with pytest.raises(rb.CfrbError):                        # non-final leaves but no weights (subgame_solving.cc:181-184)
        S.run(1)
    with pytest.raises(rb.CfrbError):
        S.begin([A - 1], [0], b)                             # terminal root
    with pytest.raises(rb.CfrbError):
        S.begin([-1] * 5, [0] * 5, np.repeat(b, 5, 0))       # over capacity
    S.close()
    Z = rb.WaveSolver(D, F, 4, net_mode=rb.NET_ZERO)
    Z.begin(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 2, H)))   # empty wave
    Z.run(3)
    assert Z.fetch(("root_means",))["root_means"].shape == (0, 2, H)
    # smallest tree: root bid A-2 has the single child `liar`
    Z.begin([A - 2], [1], b)
    Z.run(4)
    o = port.cfr_solve(D, F, b[0], [4], A - 2, 1, num_iters=4)
    f = Z.fetch(("root_means", "avg"))
    assert np.abs(f["root_means"][0] - o["root_means"][0]).max() < 1e-12
    assert np.abs(f["avg"][0, :2] - o["avg"][0]).max() < 1e-12
    # all-zero beliefs for one player: reference normalises to uniform through its 1e-80 epsilon (util.h:68-78)
    bz = b.copy(); bz[0, 1] = 0
    Z.begin([-1], [0], bz)
    Z.run(2)
    assert np.isfinite(Z.fetch(("root_means",))["root_means"]).all()
    Z.close()
