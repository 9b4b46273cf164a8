"""TEST INFRASTRUCTURE — stores what the reference computes for the cross-checks that used to call it live, so that the tests
compare against it on any machine:

    make -C oracle ref REF=<reference checkout> && python oracle/make_golden_crosscheck.py <reference checkout>

tests/golden/reference_crosscheck.npz (oracle/_ref/libref_nofma.so):
  * cfr_solve / rl_runner / synthetic_beliefs of test_port_vs_compiled_reference_live;
  * the leaf values and queries of one CFR iteration with the reference's Net2 evaluated in fp32 and in the two arithmetic
    models of the tcgen05 value-net kernels (test_reference_net_in_the_kernels_arithmetic).
tests/golden/selfplay_dropin.json (the reference's cfvpy/selfplay.py, unmodified, against rebel_b200.rela):
  * the attribute operations create_mdp_config performs on a RecursiveSolvingParams, recorded call by call;
  * parameter names and shapes of the Net2 models _build_model builds from the YAML's model block and from Net2's defaults,
    the outputs of the first one with the seed-0 weights on a few query rows, and get_last_action_index of those rows.
Net weights are not stored: they are re-created from the seed with rebel_b200.models.make_selfplay_net and pinned by a checksum.
"""
import importlib.util
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.oracle import Oracle, game_dims  # noqa: E402
from rebel_b200.models import flatten_state_dict, make_selfplay_net  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SHAPES = [(1, 4), (1, 6), (2, 3)]
LIVE_ROOTS = [(-1, 0), (4, 1)]
LIVE_CPS = [0, 1, 5, 40]
LIVE_KEYS = ("regrets", "last", "sum", "avg", "root_means", "traverser_values")

# create_mdp_config inputs: the liars_sp.yaml env block with two B200 knobs, an unknown key, and no config at all
MDP_CASES = [{"num_dice": 1, "num_faces": 6, "random_action_prob": 0.25, "sample_leaf": True,
              "subgame_params": {"num_iters": 1024, "max_depth": 2, "linear_update": True, "use_cfr": True},
              "concurrent_games": 4096, "net_mode": 3},
             {"no_such_knob": 1},
             None]
# _build_model's model blocks: liars_sp.yaml:28-33, and the same without n_layers (Net2's default of 3 layers)
MODEL_CASES = {"yaml": dict(n_hidden=256, use_layer_norm=True, n_layers=2), "default_layers": dict(n_hidden=256, use_layer_norm=True)}
DROPIN_LAST_BIDS = [-1, 0, 1, 5, 6, 11, 12]


def dropin_query_rows(port):
    """1x6f query rows of the C port for every last bid of DROPIN_LAST_BIDS (12 = liar), both traversers, plus an all-zero row."""
    D, F = 1, 6
    A, H, Q = game_dims(D, F)
    b = port.synthetic_beliefs(H, 17)
    rows = [np.zeros(Q, np.float32)]
    for lb in DROPIN_LAST_BIDS:
        for trav in (0, 1):
            rows.append(port.query(D, F, trav, lb, trav ^ (lb & 1), b[0], b[1]))
    return np.stack(rows)


def crosscheck_arrays():
    R = Oracle("ref_nofma")
    out = {}
    for (D, F) in SHAPES:
        A, H, Q = game_dims(D, F)
        out[f"synthetic_beliefs11_{D}x{F}"] = R.synthetic_beliefs(H, 11)
        b = R.synthetic_beliefs(H, 5)
        for lb, pl in LIVE_ROOTS:
            y = R.cfr_solve(D, F, b, LIVE_CPS, lb, pl, num_iters=40)
            for k in LIVE_KEYS:
                out[f"{k}_{D}x{F}_{lb}"] = y[k]
        q, v = R.rl_runner(D, F, seed=3, n_games=2, num_iters=24)
        out[f"q_{D}x{F}"], out[f"v_{D}x{F}"] = q, v

    D, F = 1, 6
    A, H, Q = game_dims(D, F)
    w = flatten_state_dict(make_selfplay_net(D, F, seed=0).state_dict())
    out["emulation_w_checksum"] = np.array([w.astype(np.float64).sum(), np.abs(w).astype(np.float64).sum()])
    b = R.synthetic_beliefs(H, 3)
    for model in (0, 1, 2):
        R.set_net_emulation(model)
        r = R.cfr_solve(D, F, b, [1], last_bid=-1, player_id=0, num_iters=1, net_w=w, want=("avg",))
        out[f"emulation_leaf_values{model}"] = r["leaf_values"][0]
        out[f"emulation_queries{model}"] = r["queries"][0]
    R.set_net_emulation(0)
    return out


def load_selfplay(ref):
    """The reference's cfvpy/selfplay.py with `cfvpy.rela` = the given module; the hydra-era packages it imports (omegaconf,
    pytorch_lightning, heyhi) are stubbed, none of them is on the paths recorded here."""
    pkg = types.ModuleType("cfvpy"); pkg.__path__ = [os.path.join(ref, "cfvpy")]
    heyhi = types.ModuleType("heyhi"); heyhi.is_on_slurm = lambda: False
    oc = types.ModuleType("omegaconf"); ocd = types.ModuleType("omegaconf.dictconfig")
    ocd.DictConfig = type("DictConfig", (dict,), {}); oc.dictconfig = ocd
    pl = types.ModuleType("pytorch_lightning"); pll = types.ModuleType("pytorch_lightning.logging"); pl.logging = pll
    rela = types.ModuleType("cfvpy.rela")
    sys.modules.update({"cfvpy": pkg, "cfvpy.rela": rela, "heyhi": heyhi, "omegaconf": oc, "omegaconf.dictconfig": ocd,
                        "pytorch_lightning": pl, "pytorch_lightning.logging": pll})
    pkg.rela = rela
    spec = importlib.util.spec_from_file_location("cfvpy.selfplay", os.path.join(ref, "cfvpy", "selfplay.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["cfvpy.selfplay"] = mod
    spec.loader.exec_module(mod)
    return mod, rela


class Recorder:
    """Stands in for rela.RecursiveSolvingParams: forwards every attribute operation to the real object and logs it as
    [op, dotted path, value]; op is "has" (the attribute exists), "missing" or "set"."""

    def __init__(self, target, log, prefix=""):
        object.__setattr__(self, "_t", (target, log, prefix))

    def __getattr__(self, name):
        target, log, prefix = object.__getattribute__(self, "_t")
        if not hasattr(target, name):
            log.append(["missing", prefix + name, None])
            raise AttributeError(name)
        log.append(["has", prefix + name, None])
        value = getattr(target, name)
        return Recorder(value, log, prefix + name + ".") if type(value).__module__ == type(target).__module__ else value

    def __setattr__(self, name, value):
        target, log, prefix = object.__getattribute__(self, "_t")
        setattr(target, name, value)
        log.append(["set", prefix + name, value])


def dropin_record(ref):
    import torch
    import rebel_b200.rela as our_rela
    selfplay, rela = load_selfplay(ref)
    mdp = []
    for env in MDP_CASES:
        log = []
        rela.RecursiveSolvingParams = lambda: Recorder(our_rela.RecursiveSolvingParams(), log)
        try:
            selfplay.create_mdp_config(env)
            raised = None
        except RuntimeError as e:
            raised = str(e).split(" in ")[0]
        mdp.append({"env": env, "ops": log, "raised": raised})

    ns = types.SimpleNamespace
    env = ns(num_faces=6, num_dice=1)
    models = {}
    for name, kw in MODEL_CASES.items():
        m = selfplay._build_model("cpu", env, ns(name="Net2", kwargs=kw), jit=True)
        models[name] = {"kwargs": kw, "parameters": [[k, list(v.shape)] for k, v in m.state_dict().items()]}
    m = selfplay._build_model("cpu", env, ns(name="Net2", kwargs=MODEL_CASES["yaml"]),
                              state_dict=make_selfplay_net(1, 6, seed=0).state_dict(), jit=True)
    rows = dropin_query_rows(Oracle("port"))
    with torch.no_grad():
        x = torch.from_numpy(rows)
        values = m(x).numpy()
        idx = selfplay.get_last_action_index(x, game_dims(1, 6)[0]).tolist()
    return {"create_mdp_config": mdp, "models": models, "query_rows": rows.tolist(),
            "yaml_model_outputs_seed0": values.tolist(), "get_last_action_index": idx}


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden_crosscheck.py <reference checkout>")
    np.savez_compressed(os.path.join(OUT, "reference_crosscheck.npz"), **crosscheck_arrays())
    with open(os.path.join(OUT, "selfplay_dropin.json"), "w") as f:
        json.dump(dropin_record(sys.argv[1]), f, indent=1)
        f.write("\n")
    for name in ("reference_crosscheck.npz", "selfplay_dropin.json"):
        print(name, os.path.getsize(os.path.join(OUT, name)))


if __name__ == "__main__":
    main()
