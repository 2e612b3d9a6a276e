"""GPU parity tests (run with -m gpu on the B200 box): the CUDA engine, called through the C ABI,
against the committed outputs of the reference (tests/golden) and against the CPU oracle.

Bars (BASELINE.json north_star): with identical recorded network outputs and RNG draws, visit counts,
selected actions, sampled chance codes — and in fact every node statistic — are BIT-EXACT; the fp32
network step agrees with the reference's torch fp32 within 1e-5.
"""
import numpy as np
import pytest
import torch

import golden_io
from oracle import mcts_oracle as O
from oracle import net_oracle as NO

pytestmark = pytest.mark.gpu

NET_ATOL = 1e-5          # fp32 CUDA-core network step vs reference torch fp32 (north_star tolerance)
# value / reward scalars come out of inverse_transform_with_support (muzero_model.py:575-591), whose
# sqrt(1 + 0.004*(|y|+1.001)) - 1 cancels ~2 decimal digits: ONE ulp of the categorical expectation y
# moves the fp32 result by up to ~2e-5 relative (3e-4 absolute at |value| ~ 30, the trained 450
# checkpoint).  The reference's own fp32 output carries that error, so scalars are compared with
# rtol 5e-5 on top of the 1e-5 absolute bar.
SCALAR_TOL = dict(atol=1e-5, rtol=5e-5)


def _engine_for(z, **kw):
    from stochastic_muzero_b200 import SearchEngine
    c = z["config"]
    return SearchEngine(c, action_dim=c["action_dim"], chance_dim=c["chance_dim"], **kw)


def _replay_tape(z, lanes=0):
    """Drive the tree kernels with the recorded draws and recorded network outputs."""
    c = z["config"]
    B, N = len(z["n_nodes"]), c["num_simulations"]
    eng = _engine_for(z, max_trees=B, net="external", rng="tape", lanes_per_tree=lanes)
    eng.set_uniform_tape(torch.from_numpy(z["uniforms"]))
    eng.root(root_policy=torch.from_numpy(z["root_policy"]), root_to_play=torch.from_numpy(z["exp_root_to_play"]),
             train=z["train"], dirichlet=torch.from_numpy(z["dirichlet"]))
    actions, branches = [], []
    pol, val, rew = (torch.from_numpy(z[k]).cuda() for k in ("sim_policy", "sim_value", "sim_reward"))
    for s in range(N):
        _slot, action, branch = eng.select(s)
        actions.append(action.cpu().numpy())
        branches.append(branch.cpu().numpy())
        eng.expand_backup(s, pol[:, s].contiguous(), val[:, s].contiguous(), rew[:, s].contiguous())
    eng.stats()   # raises if the tape ran dry or a policy was degenerate
    return eng, np.array(actions).T.reshape(B, N), np.array(branches).T.reshape(B, N)


@pytest.mark.parametrize("name", golden_io.tree_cases())
def test_tree_kernels_replay_reference_tapes_bit_exact(name):
    z = golden_io.load_tree_case(name)
    eng, actions, branches = _replay_tape(z)
    B = len(z["n_nodes"])
    if z["config"]["num_simulations"]:
        assert np.array_equal(actions, z["sim_action"]), "selected leaf actions / sampled chance codes differ"
        assert np.array_equal(branches, z["sim_branch"].astype(np.int32)), "afterstate/dynamics branch differs"
    for b in range(B):
        got = eng.export_tree(b)
        assert got["n_uniforms"] == z["n_uniforms"][b], "engine consumed a different number of uniform draws"
        golden_io.assert_dump_equal(got, golden_io.expected_dump(z, b), f"{name}[{b}]")
    # read-out used by game.py:179-204
    out = eng.read_roots()
    A = z["config"]["action_dim"]
    for b in range(B):
        e = golden_io.expected_dump(z, b)
        kids = np.flatnonzero(e["depth"] == 1)
        assert np.array_equal(out["visits"][b].cpu().numpy(), e["visit"][kids])
        assert np.array_equal(out["priors"][b].cpu().numpy(), e["prior"][kids])
        rv = np.float32(0) if e["visit"][0] == 0 else np.float32(e["value_sum"][0] / np.float32(e["visit"][0]))
        assert out["root_values"][b].item() == rv
    eng.close()


@pytest.mark.parametrize("lanes", [2, 4, 8, 16, 32])
def test_lanes_per_tree_do_not_change_results(lanes):
    z = golden_io.load_tree_case("a2c2k2_n50_train")
    eng, actions, _ = _replay_tape(z, lanes=lanes)
    assert np.array_equal(actions, z["sim_action"])
    for b in range(len(z["n_nodes"])):
        golden_io.assert_dump_equal(eng.export_tree(b), golden_io.expected_dump(z, b), f"lanes={lanes}[{b}]")
    eng.close()


def test_wide_policy_with_32_lanes_only():
    z = golden_io.load_tree_case("a4c32k4_n50")
    with pytest.raises(ValueError):
        _engine_for(z, max_trees=2, net="external", rng="tape", lanes_per_tree=8)


# ---------------------------------------------------------------------------------------------------
def _net_engine(z, B=64, **kw):
    from stochastic_muzero_b200 import ModelShape, SearchEngine
    obs, A, C, S, H, L = [int(v) for v in z["dims"]]
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=kw.pop("N", 50),
                  maxium_action_sample=kw.pop("K", 2), number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, A, C, max_trees=B, model_shape=ModelShape(obs, A, C, S, H, L),
                       net=kw.pop("net", "fp32"), **kw)
    eng.set_weights(z["weights"])
    return eng


# the two reference-precision network steps: fp32 on the CUDA cores, and the tcgen05 chain on fp16 hi/lo split operands
# (three products per K-step, fp32 accumulate; SMZ_TC32_POLY=1 adds the polynomial expm1 for small |x|)
REF_PRECISION_NETS = ["fp32", "tc32", "tc32-poly"]


def _ref_precision_engine(z, net, monkeypatch, **kw):
    monkeypatch.delenv("SMZ_TC32_POLY", raising=False)
    if net == "tc32-poly":
        monkeypatch.setenv("SMZ_TC32_POLY", "1")
    return _net_engine(z, net=net.split("-")[0], **kw)


@pytest.mark.parametrize("net", REF_PRECISION_NETS)
@pytest.mark.parametrize("name", golden_io.net_cases())
def test_fp32_network_step_matches_reference_inference(name, net, monkeypatch):
    z = golden_io.load_net_case(name)
    eng = _ref_precision_engine(z, net, monkeypatch)
    tol = dict(atol=NET_ATOL, rtol=1e-5)
    np.testing.assert_allclose(eng.net_eval("repr", z["obs"])["hidden"].cpu().numpy(), z["repr_h"], **tol)
    o = eng.net_eval("pred", z["repr_h"])
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["pred_policy"], **tol)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["pred_value"], **SCALAR_TOL)
    np.testing.assert_allclose(eng.net_eval("adyn", z["repr_h"], z["actions"])["hidden"].cpu().numpy(), z["adyn_h"], **tol)
    o = eng.net_eval("apred", z["adyn_h"])
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["apred_policy"], **tol)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["apred_value"], **SCALAR_TOL)
    o = eng.net_eval("dyn", z["adyn_h"], z["actions"])
    np.testing.assert_allclose(o["hidden"].cpu().numpy(), z["dyn_h"], **tol)
    np.testing.assert_allclose(o["reward"].cpu().numpy(), z["dyn_reward"], **SCALAR_TOL)
    o = eng.net_eval("enc", z["obs"])
    np.testing.assert_allclose(o["probs"].cpu().numpy(), z["enc_probs"], **tol)
    close = np.abs(z["enc_probs"].max(1) - np.sort(z["enc_probs"], 1)[:, -2]) < 1e-5
    assert np.array_equal(o["code"].cpu().numpy()[~close], z["enc_code"][~close])
    eng.close()


# bf16 tensor-core mode: operands rounded to bf16 (8-bit mantissa) at every layer, fp32 accumulate.
# Stated tolerances against the reference's fp32 outputs (measured worst case on these fixtures:
# hidden 2.2e-2 on the [0,1]-scaled states of the trained 450 checkpoint, policy 2.8e-4, value
# 3.5e-2 at |value| = 34).
BF16_HIDDEN_ATOL = 5e-2
BF16_POLICY_ATOL = 5e-3
BF16_SCALAR_TOL = dict(atol=5e-3, rtol=5e-3)


@pytest.mark.parametrize("name", golden_io.net_cases())
def test_bf16_tcgen05_network_step_within_stated_tolerance(name):
    z = golden_io.load_net_case(name)
    eng = _net_engine(z, B=256, net="bf16")
    h = dict(atol=BF16_HIDDEN_ATOL, rtol=0)
    p = dict(atol=BF16_POLICY_ATOL, rtol=0)
    np.testing.assert_allclose(eng.net_eval("repr", z["obs"])["hidden"].cpu().numpy(), z["repr_h"], **h)
    o = eng.net_eval("pred", z["repr_h"])
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["pred_policy"], **p)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["pred_value"], **BF16_SCALAR_TOL)
    np.testing.assert_allclose(eng.net_eval("adyn", z["repr_h"], z["actions"])["hidden"].cpu().numpy(), z["adyn_h"], **h)
    o = eng.net_eval("apred", z["adyn_h"])
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["apred_policy"], **p)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["apred_value"], **BF16_SCALAR_TOL)
    o = eng.net_eval("dyn", z["adyn_h"], z["actions"])
    np.testing.assert_allclose(o["hidden"].cpu().numpy(), z["dyn_h"], **h)
    np.testing.assert_allclose(o["reward"].cpu().numpy(), z["dyn_reward"], **BF16_SCALAR_TOL)
    o = eng.net_eval("enc", z["obs"])
    np.testing.assert_allclose(o["probs"].cpu().numpy(), z["enc_probs"], **p)
    # a tile boundary: 300 rows = 2 full tiles + a ragged one, against the fp32 engine
    g = np.random.default_rng(0)
    obs = g.standard_normal((300, z["obs"].shape[1])).astype(np.float32)
    e32 = _net_engine(z, B=300, net="fp32")
    eng2 = _net_engine(z, B=300, net="bf16")
    h32, h16 = e32.net_eval("repr", obs)["hidden"], eng2.net_eval("repr", obs)["hidden"]
    np.testing.assert_allclose(h16.cpu().numpy(), h32.cpu().numpy(), **h)
    acts = g.integers(0, int(z["dims"][1]), 300).astype(np.int32)
    d32, d16 = e32.net_eval("dyn", h32, acts), eng2.net_eval("dyn", h32, acts)
    np.testing.assert_allclose(d16["hidden"].cpu().numpy(), d32["hidden"].cpu().numpy(), **h)
    np.testing.assert_allclose(d16["reward"].cpu().numpy(), d32["reward"].cpu().numpy(), **BF16_SCALAR_TOL)
    for e in (eng, e32, eng2):
        e.close()


# plain fp16 operands (11-bit significands, fp32 accumulate, fp32 epilogue): measured worst case on these fixtures
# hidden 1.8e-4, policy 5.4e-5, value 4.0e-3 at |value| = 34 (relative 1.2e-4) — about 8x tighter than bf16
F16_HIDDEN_ATOL = 1e-3
F16_POLICY_ATOL = 5e-4
F16_SCALAR_TOL = dict(atol=1e-3, rtol=1e-3)


@pytest.mark.parametrize("name", golden_io.net_cases())
def test_f16_tcgen05_network_step_within_stated_tolerance(name):
    z = golden_io.load_net_case(name)
    eng = _net_engine(z, B=256, net="f16")
    h = dict(atol=F16_HIDDEN_ATOL, rtol=0)
    p = dict(atol=F16_POLICY_ATOL, rtol=0)
    np.testing.assert_allclose(eng.net_eval("repr", z["obs"])["hidden"].cpu().numpy(), z["repr_h"], **h)
    o = eng.net_eval("pred", z["repr_h"])
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["pred_policy"], **p)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["pred_value"], **F16_SCALAR_TOL)
    np.testing.assert_allclose(eng.net_eval("adyn", z["repr_h"], z["actions"])["hidden"].cpu().numpy(), z["adyn_h"], **h)
    o = eng.net_eval("apred", z["adyn_h"])
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["apred_policy"], **p)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["apred_value"], **F16_SCALAR_TOL)
    o = eng.net_eval("dyn", z["adyn_h"], z["actions"])
    np.testing.assert_allclose(o["hidden"].cpu().numpy(), z["dyn_h"], **h)
    np.testing.assert_allclose(o["reward"].cpu().numpy(), z["dyn_reward"], **F16_SCALAR_TOL)
    o = eng.net_eval("enc", z["obs"])
    np.testing.assert_allclose(o["probs"].cpu().numpy(), z["enc_probs"], **p)
    eng.close()


@pytest.mark.parametrize("net", ["bf16", "f16", "tc32"])
def test_tensor_core_search_is_self_consistent_with_the_oracle(net):
    """Every tensor-core mode end to end (device Philox, ragged last tile): the tree statistics are the reference
    algorithm's, bit for bit, on the network outputs the engine actually produced."""
    zn = golden_io.load_net_case("ckpt450")
    B, N, seed = 300, 50, 99
    eng = _net_engine(zn, B=B, N=N, net=net, rng="philox", seed=seed, record=True)
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(1))
    eng.root(obs=obs, train=True)
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    cfg = O.SearchConfig(discount=0.997, num_simulations=N, maxium_action_sample=2)
    for b in (0, 63, 64, 127, 128, 255, 256, 299):
        model = O.TapeModel(rec["root_policy"][b, :2], rec["sim_policy"][b], np.full(N, 2), rec["sim_value"][b],
                            rec["sim_reward"][b])
        tree = O.search(cfg, model, O.PhiloxUniforms(seed, b), train=True, dirichlet=rec["dirichlet"][b])
        golden_io.assert_dump_equal(eng.export_tree(b), tree.dump(), f"{net}[{b}]")
    eng.close()


def test_bf16_search_is_self_consistent_with_the_oracle():
    """Throughput mode end to end: device Philox + bf16 network.  The tree statistics must still be
    the reference algorithm's, bit for bit, on the network outputs the engine actually produced."""
    zn = golden_io.load_net_case("ckpt450")
    B, N, seed = 300, 50, 99
    eng = _net_engine(zn, B=B, N=N, net="bf16", rng="philox", seed=seed, record=True)
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(1))
    eng.root(obs=obs, train=True)
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    cfg = O.SearchConfig(discount=0.997, num_simulations=N, maxium_action_sample=2)
    for b in (0, 127, 128, 255, 256, 299):
        model = O.TapeModel(rec["root_policy"][b, :2], rec["sim_policy"][b], np.full(N, 2), rec["sim_value"][b],
                            rec["sim_reward"][b])
        tree = O.search(cfg, model, O.PhiloxUniforms(seed, b), train=True, dirichlet=rec["dirichlet"][b])
        golden_io.assert_dump_equal(eng.export_tree(b), tree.dump(), f"bf16[{b}]")
    # and the recorded outputs are what the fp32 oracle network gives on the same hidden states
    net = NO.NetOracle(zn["weights"], *[int(v) for v in zn["dims"]])
    h0 = eng.read_hidden(0).cpu().numpy()
    np.testing.assert_allclose(h0, net.representation(obs.numpy()), atol=BF16_HIDDEN_ATOL)
    pol, val = net.prediction(h0)
    np.testing.assert_allclose(rec["root_policy"][:, :2], pol, atol=BF16_POLICY_ATOL)
    eng.close()


def _oracle_cfg(c):
    return O.SearchConfig(**{k: c[k] for k in ("pb_c_base", "pb_c_init", "discount", "root_dirichlet_alpha",
                                                "root_exploration_fraction", "num_simulations",
                                                "maxium_action_sample", "number_of_player", "custom_loop")})


@pytest.mark.parametrize("net", REF_PRECISION_NETS)
@pytest.mark.parametrize("name", ["mlp450_seed0", "ckpt450", "mlp_small", "mlp_l0"])
def test_full_search_with_internal_network_vs_reference(name, net, monkeypatch):
    """Real-MLP recorded searches: obs + recorded draws in, engine runs its own fp32 network.
    (1) every network output the engine produced matches what the reference produced at the same
    simulation within 1e-5 as long as the paths coincide, (2) replaying the engine's OWN recorded
    outputs through the CPU oracle reproduces the engine's tree bit-exactly, (3) root values / visit
    policies agree with the reference within 1e-5 / exactly unless a sub-1e-5 score tie flipped."""
    z = golden_io.load_tree_case(name)
    zn = golden_io.load_net_case(name)
    c = z["config"]
    B, N = len(z["n_nodes"]), c["num_simulations"]
    eng = _ref_precision_engine(zn, net, monkeypatch, B=B, N=N, K=c["maxium_action_sample"], rng="tape", record=True)
    eng.set_uniform_tape(torch.from_numpy(z["uniforms"]))
    eng.root(obs=torch.from_numpy(z["obs"]), train=True, dirichlet=torch.from_numpy(z["dirichlet"]))
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    S = int(zn["dims"][3])
    np.testing.assert_allclose(eng.read_hidden(0).cpu().numpy(), z["root_hidden"], atol=NET_ATOL, rtol=1e-5)
    np.testing.assert_allclose(rec["root_policy"][:, :c["action_dim"]], z["root_policy"], atol=NET_ATOL, rtol=1e-5)
    identical = 0
    for b in range(B):
        got = eng.export_tree(b)
        # (2) oracle replay of the engine's own record
        rng = O.TapeUniforms(z["uniforms"][b])
        model = O.TapeModel(rec["root_policy"][b, :c["action_dim"]], rec["sim_policy"][b],
                            np.where(rec["sim_branch"][b] == 1, c["action_dim"], c["chance_dim"]),
                            rec["sim_value"][b], rec["sim_reward"][b])
        tree = O.search(_oracle_cfg(c), model, rng, train=True, dirichlet=z["dirichlet"][b])
        golden_io.assert_dump_equal(got, tree.dump(), f"{name}[{b}] engine vs oracle on engine record")
        assert rng.cursor == got["n_uniforms"]
        # (1) network outputs along the common prefix of simulations
        same = 0
        while same < N and rec["sim_branch"][b, same] == z["sim_branch"][b, same] and \
                tree.paths[same] == list(z["exp_paths"][b, same][z["exp_paths"][b, same] >= 0]):
            same += 1
        w = z["sim_policy"].shape[2]
        np.testing.assert_allclose(rec["sim_policy"][b, :same, :w], z["sim_policy"][b, :same], atol=NET_ATOL, rtol=1e-5)
        np.testing.assert_allclose(rec["sim_value"][b, :same], z["sim_value"][b, :same], **SCALAR_TOL)
        np.testing.assert_allclose(rec["sim_reward"][b, :same], z["sim_reward"][b, :same], **SCALAR_TOL)
        hid = np.stack([eng.read_hidden(s + 1)[b].cpu().numpy() for s in range(same)]) if same else np.zeros((0, S))
        np.testing.assert_allclose(hid, z["sim_hidden"][b, :same], atol=NET_ATOL, rtol=1e-5)
        # (3) against the reference's tree
        e = golden_io.expected_dump(z, b)
        if same == N:
            identical += 1
            assert np.array_equal(got["visit"], e["visit"]) and np.array_equal(got["key"], e["key"])
            np.testing.assert_allclose(got["value_sum"] / np.maximum(got["visit"], 1),
                                       e["value_sum"] / np.maximum(e["visit"], 1), **SCALAR_TOL)
            np.testing.assert_allclose(got["prior"], e["prior"], atol=1e-5, rtol=1e-5)
    assert identical >= B - 1, f"only {identical}/{B} searches followed the reference's visiting order"
    eng.close()


def test_philox_device_matches_oracle_and_engine_record_replays():
    """Production mode (device Philox + device Dirichlet + fp32 network): the engine's own record,
    replayed by the oracle with the oracle's Philox restatement, gives the same tree bit for bit."""
    zn = golden_io.load_net_case("mlp450_seed0")
    B, N, seed, offset = 96, 50, 1234, 7
    eng = _net_engine(zn, B=B, N=N, rng="philox", seed=seed, tree_id_offset=offset, record=True)
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(0))
    eng.root(obs=obs, train=True)
    eng.simulate(N)
    st = eng.stats()
    assert 1.0 < st["mean_leaf_depth"] < 12.0
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    assert np.allclose(rec["dirichlet"].sum(1), 1.0) and (rec["dirichlet"] >= 0).all()
    cfg = O.SearchConfig(discount=0.997, num_simulations=N, maxium_action_sample=2)
    for b in range(0, B, 7):
        model = O.TapeModel(rec["root_policy"][b, :2], rec["sim_policy"][b], np.full(N, 2), rec["sim_value"][b],
                            rec["sim_reward"][b])
        rng = O.PhiloxUniforms(seed, offset + b)
        tree = O.search(cfg, model, rng, train=True, dirichlet=rec["dirichlet"][b])
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"philox[{b}]")
        assert rng.cursor == got["n_uniforms"]
    # same seed, second search: set_seed makes it reproducible, a new seed makes it different
    v1 = eng.read_roots()["visits"].cpu().numpy().copy()
    eng.set_seed(seed, offset); eng.root(obs=obs, train=True); eng.simulate(N)
    assert np.array_equal(eng.read_roots()["visits"].cpu().numpy(), v1)
    eng.set_seed(seed + 1, offset); eng.root(obs=obs, train=True); eng.simulate(N)
    assert not np.array_equal(eng.read_roots()["visits"].cpu().numpy(), v1)
    eng.close()


def test_dirichlet_device_sampler_statistics():
    zn = golden_io.load_net_case("mlp450_seed0")
    B = 4096
    eng = _net_engine(zn, B=B, N=1, rng="philox", seed=5, record=True)
    eng.root(obs=torch.zeros(B, 4), train=True)
    d = eng.read_record()["dirichlet"].cpu().numpy()
    # Dirichlet(0.25, 0.25): marginal Beta(0.25, 0.25): mean 0.5, var = 0.25/(4*1.5) = 1/6
    assert abs(d[:, 0].mean() - 0.5) < 0.03 and abs(d[:, 0].var() - 1 / 6) < 0.02
    eng.close()


# ---------------------------------------------------------------------------------------------------
def test_dropin_run_with_reference_shaped_mlp():
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    zn = golden_io.load_net_case("mlp450_seed0")
    model = FakeMuzero(zn["weights"], *[int(v) for v in zn["dims"]])
    mcts = Monte_carlo_tree_search(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                                   root_exploration_fraction=0.25, num_simulations=50, maxium_action_sample=2,
                                   number_of_player=1, custom_loop=None, seed=3)
    root = mcts.run(observation=torch.randn(1, 4), model=model, train=True)
    assert sorted(root.children.keys()) == [0, 1]
    assert sum(c.visit_count for c in root.children.values()) == 50 and root.visit_count == 50
    assert isinstance(root.children[0].prior, np.float64) and abs(sum(c.prior for c in root.children.values()) - 1) < 1e-6
    assert np.isfinite(root.value()) and root.hidden_state.shape == (1, 61)
    # batched entry: same model, many observations
    obs = torch.randn(256, 4)
    roots = mcts.run_batch(obs, model, train=True)
    assert roots.visit_counts.shape == (256, 2) and (roots.visit_counts.sum(1) == 50).all()
    one = roots[5]
    assert [c.visit_count for c in one.children.values()] == roots.visit_counts[5].tolist()
    h = NO.NetOracle(zn["weights"], *[int(v) for v in zn["dims"]]).representation(obs[5:6].numpy())
    np.testing.assert_allclose(one.hidden_state.numpy(), h, atol=1e-5)


def test_dropin_run_with_callback_model_matches_oracle_statistics():
    """Host-model mode: the tree kernels drive an arbitrary duck-typed model (here the network oracle
    behind the reference's five inference methods)."""
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    zn = golden_io.load_net_case("mlp_small")
    model = FakeMuzero(zn["weights"], *[int(v) for v in zn["dims"]])
    model.model_structure = "lstm_model"      # not fusable -> callback path
    mcts = Monte_carlo_tree_search(discount=0.997, num_simulations=20, maxium_action_sample=3, seed=11)
    root = mcts.run(observation=np.zeros((1, 5), np.float32), model=model, train=True)
    assert root.visit_count == 20 and sum(c.visit_count for c in root.children.values()) == 20
    assert len(root.children) == 3 and all(not c.is_chance for c in root.children.values())
    deep = [c for c in root.children.values() if c.expanded()][0]
    assert all(g.is_chance for g in deep.children.values())
    assert deep.hidden_state.shape == (1, 11)


def test_shard_invariance_philox_keyed_by_global_tree_id():
    """B trees on one engine == the same trees split over two engines with tree_id_offset (what the
    multi-GPU sharding does): identical per-tree results, bit for bit."""
    zn = golden_io.load_net_case("mlp450_seed0")
    B, N, seed = 256, 50, 4242
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(3))
    whole = _net_engine(zn, B=B, N=N, rng="philox", seed=seed)
    whole.root(obs=obs, train=True); whole.simulate(N)
    full = {k: v.cpu().numpy() for k, v in whole.read_roots().items()}
    parts = []
    for lo, hi in ((0, 100), (100, 256)):
        e = _net_engine(zn, B=hi - lo, N=N, rng="philox", seed=seed, tree_id_offset=lo)
        e.root(obs=obs[lo:hi], train=True); e.simulate(N)
        parts.append({k: v.cpu().numpy() for k, v in e.read_roots().items()})
        e.close()
    for k in full:
        if k != "error":            # one flag per engine, not per tree
            assert np.array_equal(full[k], np.concatenate([p[k] for p in parts])), k
    assert full["error"][0] == 0 and all(p["error"][0] == 0 for p in parts)
    whole.close()


def test_wide_chance_codebook_full_search_config3_shape():
    """BASELINE config 3 shape (4 actions, 32 chance codes, K=32, N=100) with the internal fp32
    network on synthetic 4x4 boards: engine record replayed by the oracle."""
    from stochastic_muzero_b200 import ModelShape, SearchEngine
    from stochastic_muzero_b200.weights import random_blob
    shape = ModelShape(obs_dim=16, action_dim=4, chance_dim=32, state_dim=61, hidden_dim=126, num_hidden_layers=4)
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=100, maxium_action_sample=32,
                  number_of_player=1, custom_loop=None)
    B, seed = 64, 31
    g = np.random.default_rng(0)
    obs = (g.integers(0, 12, (B, 16)) / 16.0).astype(np.float32)
    for net in ("fp32", "bf16", "tc32"):
        eng = SearchEngine(search, 4, 32, max_trees=B, model_shape=shape, net=net, rng="philox", seed=seed, record=True)
        eng.set_weights(random_blob(shape, seed=3))
        eng.root(obs=obs, train=True); eng.simulate(100)
        eng.stats()
        rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
        cfg = O.SearchConfig(**search)
        for b in (0, 31, 63):
            width = np.where(rec["sim_branch"][b] == 1, 4, 32)
            model = O.TapeModel(rec["root_policy"][b, :4], rec["sim_policy"][b], width, rec["sim_value"][b], rec["sim_reward"][b])
            tree = O.search(cfg, model, O.PhiloxUniforms(seed, b), train=True, dirichlet=rec["dirichlet"][b])
            golden_io.assert_dump_equal(eng.export_tree(b), tree.dump(), f"cfg3-{net}[{b}]")
        assert (eng.read_roots()["visits"].sum(1) == 100).all()
        eng.close()


# ---------------------------------------------------------------------------------------------------
# the step after the search (SURVEY.md §8f-1): device read-out + action selection vs game.py:179-235
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_io.tree_cases())
def test_device_action_selection_matches_reference_policy_step(name):
    z = golden_io.load_tree_case(name)
    eng, _, _ = _replay_tape(z)
    for t_i, T in enumerate(z["readout_temperature"]):
        out = eng.select_actions(float(T), uniforms=torch.from_numpy(z["readout_u"][:, t_i].copy()))
        pol = out["policy"].cpu().numpy()
        e = 1.0 / T if T >= 0.3 else 1.0
        if e in (1.0, 2.0, 0.5):          # exact arithmetic on both sides
            assert np.array_equal(pol, z["readout_policy"][:, t_i]), f"T={T}"
        else:                             # pow(): libm vs CUDA, <= 2 ulp
            np.testing.assert_allclose(pol, z["readout_policy"][:, t_i], rtol=1e-14, atol=0)
        assert np.array_equal(out["actions"].cpu().numpy(), z["readout_index"][:, t_i]), f"T={T}: selected actions"
        assert np.array_equal(out["stored_policy"].cpu().numpy(), z["readout_stored"])
    assert np.array_equal(eng.read_roots()["root_values"].cpu().numpy(), z["readout_root_value"])
    eng.close()


def test_full_size_4096_trees_50_simulations_properties_and_sampled_replay():
    """BASELINE configs[1] at full size in throughput mode.  Size-independent properties for all trees,
    and an oracle replay (bit-exact) of a sample of them from the engine's own record."""
    from stochastic_muzero_b200 import ModelShape, SearchEngine
    from stochastic_muzero_b200.weights import random_blob
    shape = ModelShape(4, 2, 2, 61, 126, 4)
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=50, maxium_action_sample=2,
                  number_of_player=1, custom_loop=None)
    B, N, seed = 4096, 50, 2024
    eng = SearchEngine(search, 2, 2, max_trees=B, model_shape=shape, net="bf16", rng="philox", seed=seed, record=True)
    eng.set_weights(random_blob(shape, seed=0))
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(0))
    eng.root(obs=obs, train=True)
    eng.simulate(N)
    st = eng.stats()
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    # properties: every simulation visits the root once and exactly one root child
    assert (roots["visits"].sum(1) == N).all() and (roots["visits"] >= 0).all()
    assert np.allclose(roots["priors"].sum(1), 1.0, atol=1e-6) and (roots["priors"] > 0).all()
    assert np.isfinite(roots["root_values"]).all()
    # root value = mean of N discounted returns, each bounded by sum_k gamma^k max|r| + gamma^d max|v|
    bound = (np.abs(rec["sim_reward"]).max() / (1 - 0.997) + np.abs(rec["sim_value"]).max())
    assert (np.abs(roots["root_values"]) <= bound).all()
    assert np.allclose(rec["sim_policy"].sum(2), 1.0, atol=1e-5)
    assert set(np.unique(rec["sim_branch"])) <= {0, 1} and (rec["sim_branch"][:, 0] == 0).all()
    assert (rec["sim_reward"][rec["sim_branch"] == 0] == 0).all()
    assert 2.0 < st["mean_leaf_depth"] < 10.0
    # same seed twice => identical statistics (graph replay, atomics only order rows)
    eng.set_seed(seed); eng.root(obs=obs, train=True); eng.simulate(N)
    again = eng.read_roots()
    assert np.array_equal(again["visits"].cpu().numpy(), roots["visits"])
    assert np.array_equal(again["root_values"].cpu().numpy(), roots["root_values"])
    # sampled oracle replay
    cfg = O.SearchConfig(**search)
    for b in np.random.default_rng(0).choice(B, 24, replace=False):
        model = O.TapeModel(rec["root_policy"][b, :2], rec["sim_policy"][b], np.full(N, 2), rec["sim_value"][b],
                            rec["sim_reward"][b])
        tree = O.search(cfg, model, O.PhiloxUniforms(seed, int(b)), train=True, dirichlet=rec["dirichlet"][b])
        golden_io.assert_dump_equal(eng.export_tree(int(b)), tree.dump(), f"full-size[{b}]")
    # device action selection on all trees: argmax at T = 0 equals numpy's
    act = eng.select_actions(0.0)["actions"].cpu().numpy()
    flat = roots["visits"][:, 0] == roots["visits"][:, 1]
    assert np.array_equal(act[~flat], roots["visits"].argmax(1)[~flat])
    eng.close()


# ---------------------------------------------------------------------------------------------------
# external batched network back-end (any model family): tree kernels + torch modules
# ---------------------------------------------------------------------------------------------------
class _TorchMLPBackend:
    """The MLP networks of a weight blob as plain batched torch ops on the GPU (what a non-fused model
    family looks like to run_batch)."""

    def __init__(self, blob, obs, A, C, S, H, L):
        from stochastic_muzero_b200.batched_model import support_to_scalar
        self._s2s = support_to_scalar
        self.A, self.C, self.L, self.OH = A, C, L, max(A, C)
        layout, _ = NO.blob_layout(obs, A, C, S, H, L)
        b = torch.from_numpy(np.asarray(blob, np.float32)).cuda()
        self.w = {k: b[o:o + int(np.prod(s))].reshape(s) for k, (o, s) in layout.items()}

    def _lin(self, x, n):
        return x @ self.w[n + ".w"].T + self.w[n + ".b"]

    def _trunk(self, x, p):
        x = torch.nn.functional.elu(self._lin(x, p + ".in"))
        for _ in range(self.L):
            x = torch.nn.functional.elu(self._lin(x, p + ".mid"))
        return x

    @staticmethod
    def _scale(x):
        lo, hi = x.min(1, keepdim=True)[0], x.max(1, keepdim=True)[0]
        sc = hi - lo
        sc = torch.where(sc < 1e-5, sc + 1e-5, sc)
        return (x - lo) / sc

    def representation(self, obs):
        return self._scale(self._lin(self._trunk(obs.cuda().float(), "repr"), "repr.out"))

    def _pred(self, h, p):
        t = self._trunk(h, p)
        return torch.softmax(self._lin(t, p + ".policy"), -1), self._s2s(self._lin(t, p + ".value"))

    def prediction(self, h):
        return self._pred(h, "pred")

    def afterstate_prediction(self, h):
        return self._pred(h, "apred")

    def _cat(self, h, idx):
        return torch.cat([h, torch.nn.functional.one_hot(idx.long(), self.OH).float()], 1)

    def afterstate_dynamics(self, h, a):
        return self._scale(self._lin(self._trunk(self._cat(h, a), "adyn"), "adyn.state"))

    def dynamics(self, h, c):
        t = self._trunk(self._cat(h, c), "dyn")
        return self._s2s(self._lin(t, "dyn.reward")), self._scale(self._lin(t, "dyn.state"))


def test_run_batch_with_external_batched_backend_matches_fused_engine():
    from stochastic_muzero_b200 import Monte_carlo_tree_search, PackedModel, ModelShape
    zn = golden_io.load_net_case("ckpt450")
    dims = [int(v) for v in zn["dims"]]
    backend = _TorchMLPBackend(zn["weights"], *dims)
    kw = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=30, maxium_action_sample=2, seed=5)
    obs = torch.randn(200, 4, generator=torch.Generator().manual_seed(2))
    ext = Monte_carlo_tree_search(**kw).run_batch(obs, backend, train=True)
    fused = Monte_carlo_tree_search(**kw, net="fp32").run_batch(obs, PackedModel(zn["weights"], ModelShape(*dims)), train=True)
    assert (ext.visit_counts.sum(1) == 30).all()
    same = (ext.visit_counts == fused.visit_counts).all(1).float().mean().item()
    assert same >= 0.97, f"only {same:.3f} of the trees agree between torch back-end and fused fp32 step"
    agree = (ext.visit_counts == fused.visit_counts).all(1)
    np.testing.assert_allclose(ext.root_values[agree].cpu().numpy(), fused.root_values[agree].cpu().numpy(),
                               atol=1e-5, rtol=5e-5)
    assert ext.hidden_store.shape == (31, 200, dims[3])


# ---------------------------------------------------------------------------------------------------
# vision (ResNet-v2) family, BASELINE config 5: native fp32 network step
# ---------------------------------------------------------------------------------------------------
VISION_HIDDEN_ATOL = 2e-4     # channel-wise scale_to_bound amplifies fp32 noise where the 3 channels nearly coincide


def _vision_engine(z, B, N=50, **kw):
    from stochastic_muzero_b200 import SearchEngine, VisionShape
    A, S, H, L = [int(v) for v in z["dims"]]
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=kw.pop("K", 2),
                  number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, A, A, max_trees=B, model_shape=VisionShape(A, S, H, L), net="vision", **kw)
    eng.set_weights(z["weights"])
    return eng


@pytest.mark.parametrize("name", golden_io.vision_cases())
def test_vision_network_step_matches_reference_inference(name):
    z = golden_io.load_vision_case(name)
    n = z["obs"].shape[0]
    eng = _vision_engine(z, B=64)
    flat = lambda x: x.reshape(n, -1)                                            # noqa: E731
    h = eng.net_eval("repr", z["obs"])["hidden"].cpu().numpy()
    np.testing.assert_allclose(h, flat(z["repr_h"]), atol=VISION_HIDDEN_ATOL)
    o = eng.net_eval("pred", flat(z["repr_h"]))
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["pred_policy"], atol=1e-5)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["pred_value"], **SCALAR_TOL)
    ah = eng.net_eval("adyn", flat(z["repr_h"]), z["actions"])["hidden"].cpu().numpy()
    np.testing.assert_allclose(ah, flat(z["adyn_h"]), atol=VISION_HIDDEN_ATOL)
    o = eng.net_eval("apred", flat(z["adyn_h"]))
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["apred_policy"], atol=1e-5)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["apred_value"], **SCALAR_TOL)
    o = eng.net_eval("dyn", flat(z["adyn_h"]), z["actions"])
    np.testing.assert_allclose(o["hidden"].cpu().numpy(), flat(z["dyn_h"]), atol=VISION_HIDDEN_ATOL)
    np.testing.assert_allclose(o["reward"].cpu().numpy(), z["dyn_reward"], **SCALAR_TOL)
    o = eng.net_eval("pred", flat(z["dyn_h"]))
    np.testing.assert_allclose(o["policy"].cpu().numpy(), z["dpred_policy"], atol=1e-5)
    np.testing.assert_allclose(o["value"].cpu().numpy(), z["dpred_value"], **SCALAR_TOL)
    eng.close()


def test_vision_full_search_config5_shape():
    """BASELINE config 5 shape: vision model, A = 4, 1024 trees x 50 simulations on synthetic 98x98 RGB
    observations; the engine's record replayed by the oracle, network outputs against the vision oracle."""
    from oracle import vision_oracle as VO
    z = golden_io.load_vision_case("a4")
    A, S, H, L = [int(v) for v in z["dims"]]
    B, N, seed = 1024, 50, 808
    eng = _vision_engine(z, B=B, N=N, rng="philox", seed=seed, record=True)
    obs = torch.rand(B, 3, 98, 98, generator=torch.Generator().manual_seed(4))
    eng.root(obs=obs.reshape(B, -1), train=True)
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    roots = eng.read_roots()
    assert (roots["visits"].sum(1) == N).all()
    cfg = O.SearchConfig(discount=0.997, num_simulations=N, maxium_action_sample=2)
    for b in (0, 31, 32, 500, 1023):
        model = O.TapeModel(rec["root_policy"][b, :A], rec["sim_policy"][b], np.full(N, A), rec["sim_value"][b],
                            rec["sim_reward"][b])
        tree = O.search(cfg, model, O.PhiloxUniforms(seed, b), train=True, dirichlet=rec["dirichlet"][b])
        golden_io.assert_dump_equal(eng.export_tree(b), tree.dump(), f"vision[{b}]")
    net = VO.VisionOracle(z["weights"], A, S, H, L)
    sub = slice(0, 8)
    h0 = net.representation(obs[sub].numpy())
    np.testing.assert_allclose(eng.read_hidden(0)[sub].cpu().numpy(), h0.reshape(8, -1), atol=VISION_HIDDEN_ATOL)
    pol, _ = net.prediction(h0)
    np.testing.assert_allclose(rec["root_policy"][sub, :A], pol, atol=2e-5)
    assert (rec["sim_branch"][:, 0] == 0).all()      # the first simulation always takes the afterstate pair
    eng.close()


# ---------------------------------------------------------------------------------------------------
# randomised configurations: tapes produced by the (reference-pinned) oracle, replayed by the tree kernels
# ---------------------------------------------------------------------------------------------------
def _random_case(g, case_id):
    A = int(g.integers(1, 33))
    C = int(g.integers(1, 33))
    K = int(g.integers(1, 34))
    N = int(g.integers(0, 61))
    players = int(g.integers(1, 4))
    loop = None if g.random() < 0.8 else ">".join(str(int(v)) for v in g.integers(1, 4, int(g.integers(1, 5))))
    cfg = dict(pb_c_base=int(g.integers(1, 30000)), pb_c_init=float(g.random() * 2), discount=float(0.8 + 0.2 * g.random()),
               root_dirichlet_alpha=float(g.random()), root_exploration_fraction=float(g.random()),
               num_simulations=N, maxium_action_sample=K, number_of_player=players, custom_loop=loop)
    return cfg, A, C


@pytest.mark.parametrize("case_id", range(12))
def test_random_configurations_replay_oracle_tapes_bit_exact(case_id):
    from stochastic_muzero_b200 import SearchEngine
    g = np.random.default_rng(1000 + case_id)
    cfg, A, C = _random_case(g, case_id)
    N, B = cfg["num_simulations"], 6
    ocfg = O.SearchConfig(**cfg)
    n_phase = len(ocfg.cycle_map())
    train = bool(g.random() < 0.7)
    scale = float(10 ** g.uniform(-2, 1.5))
    peaky = float(10 ** g.uniform(-1, 0.7))

    class Stub:
        def __init__(self, seed):
            self.g = np.random.default_rng(seed)
            self.rows = []

        def _p(self, n):
            z = self.g.normal(size=n) * peaky
            e = np.exp(z - z.max())
            return (e / e.sum()).astype(np.float32)

        def root(self):
            self.root_policy = self._p(A)
            return None, self.root_policy, np.float32(0)

        def afterstate(self, sim, h, a):
            p, v = self._p(C), np.float32(self.g.normal() * scale)
            self.rows.append((0, p, v, np.float32(0)))
            return None, p, v

        def dynamics(self, sim, h, a):
            p, v, r = self._p(A), np.float32(self.g.normal() * scale), np.float32(self.g.normal() * scale)
            self.rows.append((1, p, v, r))
            return None, p, v, r

    W = max(A, C)
    trees, stubs, rngs, dirs, phases = [], [], [], [], []
    for b in range(B):
        stub, rng = Stub(case_id * 100 + b), O.MTUniforms(case_id * 100 + b)
        d = np.random.default_rng(b).dirichlet([max(cfg["root_dirichlet_alpha"], 1e-3)] * A)
        ph = int(g.integers(0, n_phase))
        trees.append(O.search(ocfg, stub, rng, train=train, dirichlet=d, root_to_play=ph))
        stubs.append(stub); rngs.append(rng); dirs.append(d); phases.append(ph)
    U = max(len(r.log) for r in rngs) + 1
    uni = np.zeros((B, U)); pol = np.zeros((B, max(N, 1), W), np.float32)
    val = np.zeros((B, max(N, 1)), np.float32); rew = np.zeros((B, max(N, 1)), np.float32)
    rootp = np.zeros((B, W), np.float32)
    for b in range(B):
        uni[b, :len(rngs[b].log)] = rngs[b].log
        rootp[b, :A] = stubs[b].root_policy
        for s, (br, p, v, r) in enumerate(stubs[b].rows):
            pol[b, s, :len(p)], val[b, s], rew[b, s] = p, v, r
    eng = SearchEngine(cfg, A, C, max_trees=B, net="external", rng="tape")
    eng.set_uniform_tape(torch.from_numpy(uni))
    eng.root(root_policy=torch.from_numpy(rootp), root_to_play=torch.tensor(phases, dtype=torch.int32), train=train,
             dirichlet=torch.from_numpy(np.stack(dirs)))
    pol_d, val_d, rew_d = (torch.from_numpy(x).cuda() for x in (pol, val, rew))
    for s in range(N):
        eng.select(s)
        eng.expand_backup(s, pol_d[:, s].contiguous(), val_d[:, s].contiguous(), rew_d[:, s].contiguous())
    eng.stats()
    for b in range(B):
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, trees[b].dump(), f"random[{case_id}][{b}] cfg={cfg} A={A} C={C}")
        assert got["n_uniforms"] == len(rngs[b].log)
    eng.close()


# ---------------------------------------------------------------------------------------------------
# boundary behaviour: ragged batches, misuse errors (return codes of the C ABI surface as exceptions)
# ---------------------------------------------------------------------------------------------------
def test_partial_batch_equals_exact_size_engine():
    zn = golden_io.load_net_case("mlp450_seed0")
    obs = torch.randn(77, 4, generator=torch.Generator().manual_seed(9))
    out = []
    for cap in (77, 300):
        for net in ("fp32", "bf16", "tc32", "f16"):
            e = _net_engine(zn, B=cap, N=20, net=net, rng="philox", seed=66)
            e.root(obs=obs, train=True); e.simulate(20)
            r = e.read_roots()
            assert r["visits"].shape == (77, 2)
            out.append((net, r["visits"].cpu().numpy(), r["root_values"].cpu().numpy()))
            e.close()
    for net in ("fp32", "bf16", "tc32", "f16"):
        a, b = [o for o in out if o[0] == net]
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]), f"{net}: capacity changed the result"


def test_api_misuse_is_reported_not_executed():
    from stochastic_muzero_b200 import ModelShape, SearchEngine, SmzError
    zn = golden_io.load_net_case("mlp_small")
    obs_dim, A, C, S, H, L = [int(v) for v in zn["dims"]]
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=5, maxium_action_sample=2,
                  number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, A, C, max_trees=8, model_shape=ModelShape(obs_dim, A, C, S, H, L), net="fp32")
    with pytest.raises(SmzError, match="smz_set_weights has not been called"):
        eng.root(obs=torch.zeros(4, obs_dim))
    with pytest.raises(ValueError, match="blob has"):
        eng.set_weights(np.zeros(10, np.float32))
    eng.set_weights(zn["weights"])
    with pytest.raises(SmzError, match="smz_root has not been called"):
        eng.simulate(5)
    with pytest.raises(ValueError, match="n_trees"):
        eng.root(obs=torch.zeros(9, obs_dim))
    eng.root(obs=torch.zeros(4, obs_dim), train=False)
    with pytest.raises(ValueError, match="exceed num_simulations"):
        eng.simulate(6)
    eng.simulate(5)
    with pytest.raises(ValueError, match="exceed num_simulations"):
        eng.simulate(1)
    with pytest.raises(ValueError, match="not in"):
        eng.export_tree(4)
    ext = SearchEngine(search, A, C, max_trees=8, net="external")
    with pytest.raises(SmzError, match="has no network"):
        ext.root(obs=torch.zeros(4, obs_dim))
    with pytest.raises(SmzError, match="rng_mode is not TAPE"):
        ext.set_uniform_tape(torch.zeros(8, 4, dtype=torch.float64))
    with pytest.raises(ValueError, match="lanes_per_tree"):
        SearchEngine(search, A, C, max_trees=8, net="external", lanes_per_tree=3)
    eng.close(); ext.close()


_VARIANTS = {
    "chain_one_thread_issue": {"SMZ_NO_PIPE": "1"},
    "chain_128_rows_2_rounds": {"SMZ_M64": "0"},
    "chain_128_rows_two_tiles_per_cta": {"SMZ_M64": "0", "SMZ_PIPE2": "1"},
    "chain_64_rows_64_leaves": {"SMZ_M64": "1", "SMZ_M32": "0"},
    "chain_64_rows_32_leaves": {"SMZ_M64": "1", "SMZ_M32": "1"},
    "chain_32_leaves_every_tile_streamed": {"SMZ_M64": "1", "SMZ_M32": "1", "SMZ_STREAM_ALL": "1"},
    "tree_arena_only": {"SMZ_NO_TREE_SMEM": "1"},
}


def _bf16_search_record(monkeypatch, env, B=300, N=50):
    for k in ("SMZ_NO_PIPE", "SMZ_M64", "SMZ_M32", "SMZ_PIPE2", "SMZ_STREAM_ALL", "SMZ_NO_TREE_SMEM"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    zn = golden_io.load_net_case("ckpt450")
    eng = _net_engine(zn, B=B, N=N, net="bf16", rng="philox", seed=5, record=True)
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(11))
    eng.root(obs=obs, train=True)
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    hid = eng.read_hidden(N).cpu().numpy()
    eng.close()
    return rec, roots, hid


@pytest.mark.parametrize("variant", sorted(_VARIANTS))
def test_kernel_variants_give_the_same_search(monkeypatch, variant):
    """The shipped kernel choice (64-row pipelined chain + shared-memory tree step at this size) and every
    fallback / large-batch variant run the same search: identical visit counts, hidden states and tree
    statistics; network scalars identical up to the reduction order of the head layers."""
    ref_rec, ref_roots, ref_hid = _bf16_search_record(monkeypatch, {})
    rec, roots, hid = _bf16_search_record(monkeypatch, _VARIANTS[variant])
    np.testing.assert_array_equal(roots["visits"], ref_roots["visits"])
    np.testing.assert_array_equal(hid, ref_hid)
    np.testing.assert_allclose(rec["sim_policy"], ref_rec["sim_policy"], atol=1e-6)
    np.testing.assert_allclose(rec["sim_value"], ref_rec["sim_value"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(roots["root_values"], ref_roots["root_values"], rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------------------------------------------
# round-2 boundary behaviour: error flag surfaced, root_to_play wrapped, stale views refused
# ---------------------------------------------------------------------------------------------------
def test_degenerate_policy_raises_like_numpy_choice():
    """A NaN policy makes np.random.choice raise inside the reference's expansion (mcts.py:294); the engine
    sets its error flag, delivers it with the root read-out and the drop-in raises ValueError."""
    from stochastic_muzero_b200 import Monte_carlo_tree_search, SearchEngine
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=4, maxium_action_sample=2,
                  number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, 2, 2, max_trees=3, net="external", rng="philox", seed=1)
    eng.root(root_policy=torch.full((3, 2), 0.5), train=False)
    bad = torch.tensor([[0.5, 0.5], [float("nan"), float("nan")], [0.5, 0.5]])
    eng.select(0)
    eng.expand_backup(0, bad, torch.zeros(3), torch.zeros(3))
    assert int(eng.read_roots()["error"].item()) == 2
    with pytest.raises(ValueError, match="degenerate"):
        eng.raise_for_error(2)
    eng.close()

    class NaNBackend:          # batched back-end whose afterstate policy head returns NaN
        A = C = 2

        def representation(self, obs):
            return torch.zeros(obs.shape[0], 3, device="cuda")

        def prediction(self, h):
            return torch.full((h.shape[0], 2), 0.5, device="cuda"), torch.zeros(h.shape[0], device="cuda")

        def afterstate_dynamics(self, h, a):
            return h

        def afterstate_prediction(self, h):
            return torch.full((h.shape[0], 2), float("nan"), device="cuda"), torch.zeros(h.shape[0], device="cuda")

        def dynamics(self, h, c):
            return torch.zeros(h.shape[0], device="cuda"), h
    mcts = Monte_carlo_tree_search(num_simulations=4, discount=0.997, seed=3)
    with pytest.raises(ValueError, match="degenerate"):
        mcts.run_batch(torch.zeros(5, 4), NaNBackend(), train=False)
    roots = mcts.run_batch(torch.zeros(5, 4), NaNBackend(), train=False, check=False)      # asynchronous form
    with pytest.raises(ValueError):
        roots.raise_if_failed()


def test_root_to_play_is_wrapped_into_the_player_cycle():
    """Values outside [0, n_phases) used to index the sign table out of bounds; they are wrapped like
    Player_cycle.global_step() wraps its counter, and the exported tree agrees with what the device did."""
    z = golden_io.load_tree_case("a3c5k3_n30_p2")
    c = z["config"]
    B, N = len(z["n_nodes"]), c["num_simulations"]
    n_ph = 2

    def run(rtp):
        eng = _engine_for(z, max_trees=B, net="external", rng="tape")
        eng.set_uniform_tape(torch.from_numpy(z["uniforms"]))
        eng.root(root_policy=torch.from_numpy(z["root_policy"]), root_to_play=torch.from_numpy(rtp), train=z["train"],
                 dirichlet=torch.from_numpy(z["dirichlet"]))
        pol, val, rew = (torch.from_numpy(z[k]).cuda() for k in ("sim_policy", "sim_value", "sim_reward"))
        for s in range(N):
            eng.select(s)
            eng.expand_backup(s, pol[:, s].contiguous(), val[:, s].contiguous(), rew[:, s].contiguous())
        out = [eng.export_tree(b) for b in range(B)]
        eng.close()
        return out
    base = z["exp_root_to_play"].astype(np.int32)
    ref = run(base)
    for shift in (n_ph * 7, -n_ph * 3):
        got = run(base + shift)
        for b in range(B):
            golden_io.assert_dump_equal(got[b], ref[b], f"root_to_play + {shift} [{b}]")
            golden_io.assert_dump_equal(got[b], golden_io.expected_dump(z, b), f"wrapped vs reference [{b}]")


def test_views_of_an_older_search_are_refused():
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search, StaleSearchError
    zn = golden_io.load_net_case("mlp450_seed0")
    model = FakeMuzero(zn["weights"], *[int(v) for v in zn["dims"]])
    mcts = Monte_carlo_tree_search(discount=0.997, num_simulations=10, seed=3)
    first = mcts.run_batch(torch.randn(8, 4), model, train=True)
    kept = first.visit_counts.clone()
    node = first[2]
    assert node.hidden_state.shape == (1, 61)             # fetched while the search is current
    root1 = mcts.run(observation=torch.randn(1, 4), model=model, train=True)
    assert torch.equal(first.visit_counts, kept)          # plain result tensors stay valid ...
    with pytest.raises(StaleSearchError):                 # ... arena-backed views do not
        first[0]
    with pytest.raises(StaleSearchError):
        first.select_actions(1.0)
    mcts.run(observation=torch.randn(1, 4), model=model, train=True)
    with pytest.raises(StaleSearchError):
        root1.hidden_state
    assert sum(c.visit_count for c in root1.children.values()) == 10      # materialised statistics survive


def test_host_readout_is_one_consistent_copy():
    """BatchedRoots.host(): visit counts, root values and the error flag fetched with one copy equal the device tensors,
    and stay what they were after the arena has been reused by a later search."""
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    zn = golden_io.load_net_case("mlp450_seed0")
    model = FakeMuzero(zn["weights"], *[int(v) for v in zn["dims"]])
    mcts = Monte_carlo_tree_search(discount=0.997, num_simulations=12, seed=9, net="bf16")
    roots = mcts.run_batch(torch.randn(37, 4), model, train=True)
    h = roots.host()
    assert h["error"] == 0 and h["visit_counts"].dtype == np.int32 and h["root_values"].dtype == np.float32
    np.testing.assert_array_equal(h["visit_counts"], roots.visit_counts.cpu().numpy())
    np.testing.assert_array_equal(h["root_values"], roots.root_values.cpu().numpy())
    assert (h["visit_counts"].sum(1) == 12).all()
    kept = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in h.items()}
    mcts.run_batch(torch.randn(37, 4), model, train=True).host()          # reuses the arena and the pinned buffer
    np.testing.assert_array_equal(roots.host()["visit_counts"], kept["visit_counts"])
    np.testing.assert_array_equal(roots.host()["root_values"], kept["root_values"])


def test_launch_counters_and_real_tree_step_hook():
    """smz_stats counts the kernels of the last search and since creation; smz_backup_select runs the fused
    tree step of the captured loop stand-alone and gives the same search as smz_simulate."""
    zn = golden_io.load_net_case("mlp450_seed0")
    B, N = 200, 12
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(5))
    for net in ("fp32", "bf16", "tc32", "f16"):
        a = _net_engine(zn, B=B, N=N, net=net, rng="philox", seed=8)
        a.root(obs=obs, train=True); a.simulate(N)
        st = a.stats()
        assert st["launches"] == 3 + 1 + 2 * N and st["launches_total"] >= st["launches"]
        ref = a.read_roots()
        b = _net_engine(zn, B=B, N=N, net=net, rng="philox", seed=8)
        b.root(obs=obs, train=True)
        b.select(0)
        for s in range(N):
            b.net_step(s)
            if s + 1 < N:
                b.backup_select(s)
            else:
                b.expand_backup(s)
        got = b.read_roots()
        assert torch.equal(got["visits"], ref["visits"]) and torch.equal(got["root_values"], ref["root_values"])
        with pytest.raises(ValueError, match="no successor"):
            b.backup_select(N - 1)
        a.close(); b.close()


def test_tc32_search_agrees_with_the_fp32_cuda_core_search():
    """Both reference-precision network steps drive the same search: same seeds, 512 trees x 50 simulations on
    the trained checkpoint — identical visit vectors for (nearly) all trees (a sub-1e-6 score tie may flip), root
    values within the scalar tolerance, hidden states within 1e-5, and the ragged last tile handled."""
    zn = golden_io.load_net_case("ckpt450")
    B, N = 500, 50
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(21)) * 0.1
    out = {}
    for net in ("fp32", "tc32"):
        e = _net_engine(zn, B=B, N=N, net=net, rng="philox", seed=77)
        e.root(obs=obs, train=True); e.simulate(N)
        r = e.read_roots()
        assert int(r["error"].item()) == 0
        out[net] = (r["visits"].cpu().numpy(), r["root_values"].cpu().numpy(), e.read_hidden(0).cpu().numpy(),
                    e.read_hidden(1).cpu().numpy())
        e.close()
    same = (out["fp32"][0] == out["tc32"][0]).all(1)
    assert same.mean() >= 0.99, f"only {same.mean():.4f} of the trees have identical visit vectors"
    np.testing.assert_allclose(out["tc32"][1][same], out["fp32"][1][same], **SCALAR_TOL)
    np.testing.assert_allclose(out["tc32"][2], out["fp32"][2], atol=NET_ATOL, rtol=1e-5)
    np.testing.assert_allclose(out["tc32"][3], out["fp32"][3], atol=NET_ATOL, rtol=1e-5)


# ---------------------------------------------------------------------------------------------------
# full-size runs of the other BASELINE configs: size-independent properties on every tree + sampled oracle replay
# ---------------------------------------------------------------------------------------------------
def _full_size_case(search, shape, A, C, B, net, seed, obs, sample, what):
    from stochastic_muzero_b200 import SearchEngine
    from stochastic_muzero_b200.weights import random_blob
    N = search["num_simulations"]
    eng = SearchEngine(search, A, C, max_trees=B, model_shape=shape, net=net, rng="philox", seed=seed, record=True)
    eng.set_weights(random_blob(shape, seed=0))
    eng.root(obs=obs, train=True)
    eng.simulate(N)
    st = eng.stats()                                             # raises on a device error flag
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    assert roots["error"][0] == 0
    assert (roots["visits"].sum(1) == N).all() and (roots["visits"] >= 0).all()       # one root child per simulation
    assert np.allclose(roots["priors"].sum(1), 1.0, atol=1e-6) and (roots["priors"] > 0).all()
    assert np.isfinite(roots["root_values"]).all()
    bound = np.abs(rec["sim_reward"]).max() / (1 - search["discount"]) + np.abs(rec["sim_value"]).max()
    assert (np.abs(roots["root_values"]) <= bound).all()
    width = np.where(rec["sim_branch"] == 1, A, C)
    psum = rec["sim_policy"].sum(2)
    assert np.allclose(psum, 1.0, atol=2e-5), "a recorded policy row does not sum to 1"
    cols = np.arange(rec["sim_policy"].shape[2])[None, None, :]
    assert (rec["sim_policy"][cols >= width[:, :, None]] == 0).all(), "policy mass beyond the head's width"
    assert set(np.unique(rec["sim_branch"])) <= {0, 1} and (rec["sim_branch"][:, 0] == 0).all()
    assert (rec["sim_reward"][rec["sim_branch"] == 0] == 0).all()                    # afterstate pair has no reward
    assert 1.5 < st["mean_leaf_depth"] < 12.0
    # idempotence: same seed, same observations => the same statistics (atomics only order the compacted rows)
    eng.set_seed(seed); eng.root(obs=obs, train=True); eng.simulate(N)
    again = eng.read_roots()
    assert np.array_equal(again["visits"].cpu().numpy(), roots["visits"])
    assert np.array_equal(again["root_values"].cpu().numpy(), roots["root_values"])
    cfg = O.SearchConfig(**search)
    for b in sample:
        b = int(b)
        model = O.TapeModel(rec["root_policy"][b, :A], rec["sim_policy"][b], width[b], rec["sim_value"][b], rec["sim_reward"][b])
        tree = O.search(cfg, model, O.PhiloxUniforms(seed, b), train=True, dirichlet=rec["dirichlet"][b])
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"{what}[{net}][{b}]")
    eng.close()


@pytest.mark.parametrize("net", ["bf16", "tc32"])
def test_full_size_config3_8192_trees_100_simulations_wide_codebook(net):
    """BASELINE configs[2] at full size: 8192 trees x 100 simulations, 4 actions, 32 chance codes, K = 32 (random
    subsets never trigger: every head's children are all kept), synthetic 4x4 boards."""
    from stochastic_muzero_b200 import ModelShape
    shape = ModelShape(obs_dim=16, action_dim=4, chance_dim=32, state_dim=61, hidden_dim=126, num_hidden_layers=4)
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=100, maxium_action_sample=32,
                  number_of_player=1, custom_loop=None)
    B = 8192
    obs = (torch.randint(0, 12, (B, 16), generator=torch.Generator().manual_seed(0)).float() / 16.0)
    sample = [0, 63, 64, 4095, 4096, 8191] + list(np.random.default_rng(1).choice(B, 6, replace=False))
    _full_size_case(search, shape, 4, 32, B, net, 303, obs, sample, "cfg3")


def test_full_size_config4_65536_trees_50_simulations():
    """BASELINE configs[3] on one GPU: 65536 trees x 50 simulations (the large-batch kernels: 128-row chain tiles,
    arena-only tree step), bf16 network step."""
    from stochastic_muzero_b200 import ModelShape
    shape = ModelShape(4, 2, 2, 61, 126, 4)
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=50, maxium_action_sample=2,
                  number_of_player=1, custom_loop=None)
    B = 65536
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(0))
    sample = [0, 127, 128, 32767, 32768, 65535] + list(np.random.default_rng(2).choice(B, 10, replace=False))
    _full_size_case(search, shape, 2, 2, B, "bf16", 404, obs, sample, "cfg4")


# ---------------------------------------------------------------------------------------------------
# what the bf16 throughput mode does to the SEARCH RESULT (DESIGN.md §2: stated thresholds)
# ---------------------------------------------------------------------------------------------------
# fraction of trees with an identical root visit vector / the same most-visited action, and the 99th percentile of the
# relative root-value deviation, bf16 vs fp32-grade (tc32) search on the same seeds, 4096 trees x 50 simulations.
# Measured on B200 (tools/diag_bf16_agreement.py): random init 0.9998 / 1.0000 / 0; checkpoint 450 0.908 / 0.993 / 1.5e-2.
BF16_SEARCH_AGREEMENT = {"mlp450_seed0": dict(identical=0.99, same_action=0.999, value_p99=1e-3),
                         "ckpt450": dict(identical=0.85, same_action=0.98, value_p99=3e-2)}
# the plain-fp16 mode: random init 1.0000 / 1.0000 / 0; checkpoint 450 0.9875 / 0.998 / 6.6e-3
F16_SEARCH_AGREEMENT = {"mlp450_seed0": dict(identical=0.995, same_action=0.999, value_p99=1e-3),
                        "ckpt450": dict(identical=0.97, same_action=0.99, value_p99=1.5e-2)}


@pytest.mark.parametrize("name", sorted(BF16_SEARCH_AGREEMENT))
def test_bf16_search_result_fidelity_against_reference_precision(name):
    zn = golden_io.load_net_case(name)
    B, N = 4096, 50
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(0)) * 0.1
    res = {}
    for net in ("fp32", "tc32", "bf16", "f16"):
        eng = _net_engine(zn, B=B, N=N, net=net, rng="philox", seed=11)
        eng.root(obs=obs, train=True); eng.simulate(N)
        r = eng.read_roots()
        assert int(r["error"].item()) == 0
        res[net] = (r["visits"].cpu().numpy(), r["root_values"].cpu().numpy())
        eng.close()

    def agreement(a, b):
        va, vb = res[a][0], res[b][0]
        flat = (va[:, 0] == va[:, 1]) | (vb[:, 0] == vb[:, 1])
        rel = np.abs(res[a][1] - res[b][1]) / np.maximum(np.abs(res[a][1]), 1e-3)
        return (va == vb).all(1).mean(), (va.argmax(1) == vb.argmax(1))[~flat].mean(), np.percentile(rel, 99)
    for mode, table in (("bf16", BF16_SEARCH_AGREEMENT), ("f16", F16_SEARCH_AGREEMENT)):
        thr = table[name]
        ident, action, p99 = agreement("tc32", mode)
        assert ident >= thr["identical"] and action >= thr["same_action"] and p99 <= thr["value_p99"], \
            f"{name}: {mode} vs tc32 identical {ident:.4f}, same action {action:.4f}, root value p99 {p99:.2e}"
    # the two reference-precision modes differ only where a sub-1e-6 score tie flips
    ident, action, p99 = agreement("fp32", "tc32")
    assert ident >= 0.995 and action >= 0.999 and p99 <= 1e-4, \
        f"{name}: tc32 vs fp32 identical {ident:.4f}, same action {action:.4f}, root value p99 {p99:.2e}"


# inverse_transform_with_support in fp32 (muzero_model.py:575-591): sqrt(1 + 0.004 (|y| + 1.001)) - 1 keeps ~14 bits,
# so the scalar moves in steps ("quanta") of ~1.2e-4 near zero — one ulp of the categorical expectation y can move the
# reference's own fp32 output by one quantum (tests/test_host_logic.py shows it against float64)
SCALAR_QUANTUM_TOL = dict(atol=2.5e-4, rtol=1e-4)


def test_vision_tensor_core_heads_match_the_cuda_core_step(monkeypatch):
    """Simulation step of the vision family: convolution stage on the CUDA cores + MLP heads on the fp32-grade tcgen05
    chain (default) against the all-CUDA-core kernel (SMZ_VISION_CC=1), driven step by step.  Wherever both engines
    feed the network the same input (same parent hidden state — itself produced from equal inputs — and same action),
    the outputs must agree: policies within 1e-5, scalars within one quantum of the support transform, the new
    hidden state bit for bit (same convolution code).  Ragged batch: 300 trees = partial 8-, 32- and 64-row tiles."""
    z = golden_io.load_vision_case("a4")
    A = int(z["dims"][0])
    B, N, seed = 300, 24, 5
    obs = torch.rand(B, 3, 98, 98, generator=torch.Generator().manual_seed(8)).reshape(B, -1)
    out = {}
    for mode in ("tc", "cc"):
        monkeypatch.delenv("SMZ_VISION_CC", raising=False)
        if mode == "cc":
            monkeypatch.setenv("SMZ_VISION_CC", "1")
        eng = _vision_engine(z, B=B, N=N, rng="philox", seed=seed, record=True)
        eng.root(obs=obs, train=True)
        sel = []
        for s in range(N):
            sel.append([t.cpu().numpy() for t in eng.select(s)])
            eng.net_step(s)
            eng.expand_backup(s)
        st = eng.stats()
        assert st["launches"] == 4 + (3 if mode == "tc" else 2) * N + N, st       # the tensor-core stage is a kernel of its own
        rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
        hid = np.stack([eng.read_hidden(k).cpu().numpy() for k in range(N + 1)], 1)          # [B, N+1, 147]
        out[mode] = (np.array(sel), rec, hid)
        eng.close()
    (sa, ra, ha), (sb, rb, hb) = out["tc"], out["cc"]
    rows = np.arange(B)
    clean = np.zeros((B, N + 1), bool)            # hidden slot k holds a state both engines derived from equal inputs
    clean[:, 0] = True
    compared = 0
    for s in range(N):
        eq = (sa[s] == sb[s]).all(0) & clean[rows, sa[s][0]]
        clean[:, s + 1] = eq
        compared += int(eq.sum())
        np.testing.assert_array_equal(ha[eq, s + 1], hb[eq, s + 1])
        np.testing.assert_allclose(ra["sim_policy"][eq, s, :A], rb["sim_policy"][eq, s, :A], atol=1e-5)
        np.testing.assert_allclose(ra["sim_value"][eq, s], rb["sim_value"][eq, s], **SCALAR_QUANTUM_TOL)
        np.testing.assert_allclose(ra["sim_reward"][eq, s], rb["sim_reward"][eq, s], **SCALAR_QUANTUM_TOL)
    assert compared >= 0.9 * B * N, f"only {compared} of {B * N} network evaluations had equal inputs"
    both = clean[:, 1:]
    exact = (ra["sim_value"][both] == rb["sim_value"][both]).mean()
    assert exact >= 0.9, f"only {exact:.3f} of the compared values are bit-identical"
