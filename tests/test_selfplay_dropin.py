"""The reference's UNMODIFIED cfvpy/selfplay.py against the rebel_b200 `rela` module (SURVEY 8b: selfplay.py drops in unchanged).

What selfplay.py does with the module was recorded by running it against rebel_b200.rela (oracle/make_golden_crosscheck.py,
tests/golden/selfplay_dropin.json): the attribute operations of create_mdp_config, the parameters of the Net2 models
_build_model builds, their outputs and get_last_action_index on query rows of the C port.  The tests replay those operations
on the module and compare with the recording; nothing of the reference's code is in the repository."""
import json
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "selfplay_dropin.json")


@pytest.fixture(scope="module")
def selfplay():
    with open(GOLDEN) as f:
        return json.load(f)


def _replay_mdp_config(rela, case):
    """create_mdp_config (selfplay.py:587-610) as recorded: hasattr before every key, getattr to recurse into subgame_params,
    setattr of every leaf value; it raises when hasattr is false."""
    cfg = rela.RecursiveSolvingParams()

    def parent(path):
        obj = cfg
        for name in path.split(".")[:-1]:
            obj = getattr(obj, name)
        return obj, path.split(".")[-1]
    for op, path, value in case["ops"]:
        obj, name = parent(path)
        assert hasattr(obj, name) == (op != "missing"), (op, path)
        if op == "set":
            setattr(obj, name, value)
    if case["raised"]:
        assert case["ops"][-1][0] == "missing"
    return cfg


def test_create_mdp_config_fills_our_params(selfplay):
    """create_mdp_config (selfplay.py:587-610): hasattr / setattr over cfg.env, recursing into subgame_params; B200 knobs are
    ordinary extra keys; unknown keys raise like with the reference module."""
    import rebel_b200.rela as rela
    full, unknown, empty = selfplay["create_mdp_config"]
    assert full["raised"] is None and len(full["ops"]) == 22
    cfg = _replay_mdp_config(rela, full)
    assert isinstance(cfg, rela.RecursiveSolvingParams)
    assert (cfg.num_dice, cfg.num_faces, cfg.sample_leaf, cfg.concurrent_games) == (1, 6, True, 4096)
    assert abs(cfg.random_action_prob - 0.25) < 1e-7
    sp = cfg.subgame_params
    assert (sp.num_iters, sp.max_depth, sp.linear_update, sp.use_cfr) == (1024, 2, True, True)
    assert unknown["env"] == {"no_such_knob": 1} and unknown["raised"] == "Cannot find key no_such_knob"
    _replay_mdp_config(rela, unknown)
    assert empty["env"] is None and empty["ops"] == [] and empty["raised"] is None
    assert isinstance(_replay_mdp_config(rela, empty), rela.RecursiveSolvingParams)


def test_reference_model_builder_feeds_our_model_locker(selfplay, port):
    """_build_model (selfplay.py:31-50) with the YAML's model block (liars_sp.yaml:28-33) produces the TorchScript Net2 our
    ModelLocker accepts; the reference's default Net2 (n_layers=3) is refused instead of being truncated."""
    import rebel_b200.rela as rela
    from oracle.make_golden_crosscheck import DROPIN_LAST_BIDS, dropin_query_rows
    from rebel_b200.models import Net2, make_selfplay_net
    models = selfplay["models"]
    built = {}
    for name, rec in models.items():
        net = Net2(num_faces=6, num_dice=1, **rec["kwargs"])
        assert [[k, list(v.shape)] for k, v in net.state_dict().items()] == rec["parameters"], name
        built[name] = net
    built["yaml"].load_state_dict(make_selfplay_net(1, 6, seed=0).state_dict())
    good = torch.jit.script(built["yaml"])
    locker = rela.ModelLocker([good], "cuda:0")
    assert locker.version == 1
    rows = dropin_query_rows(port)
    assert np.array_equal(rows, np.asarray(selfplay["query_rows"], np.float32))
    with torch.no_grad():
        out = good(torch.from_numpy(rows)).numpy()
    assert out.shape == (len(rows), 6)
    assert np.allclose(out, np.asarray(selfplay["yaml_model_outputs_seed0"], np.float32), rtol=1e-5, atol=1e-7)
    # the last bid of our query rows, as the reference's get_last_action_index decodes it: 13 = "initial" (all-zero one-hot)
    A = 13
    assert selfplay["get_last_action_index"] == [A] + [A if lb < 0 else lb for lb in DROPIN_LAST_BIDS for _ in (0, 1)]
    deep = torch.jit.script(built["default_layers"])
    with pytest.raises(RuntimeError, match="unexpected parameter"):
        rela.ModelLocker([deep], "cuda:0")
