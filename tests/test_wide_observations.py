"""MLP models whose observations are wider than one 128-column K tile (GPU).  The first layer of the representation
and encoder networks streams its K dimension in slices; every later layer and the per-simulation kernels are the
ones narrow models use.  Checked against the float32 network oracle and, for whole searches, the search oracle."""
import numpy as np
import pytest
import torch

from oracle import mcts_oracle as O
from oracle import net_oracle as NO

pytestmark = pytest.mark.gpu

A, C, S, H, L = 4, 4, 61, 126, 2
WIDTHS = [129, 200, 376, 1000, 8192]
SEARCH = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, maxium_action_sample=2, number_of_player=1, custom_loop=None)

# bars of tests/test_gpu_parity.py: fp32 and tc32 at the reference's precision, bf16 and f16 at their stated tolerances
TOL = {"fp32": (1e-5, 1e-5), "tc32": (1e-5, 1e-5), "f16": (1e-3, 5e-4), "bf16": (5e-2, 5e-3)}   # (hidden, policy / probs)


def _shape(obs):
    from stochastic_muzero_b200 import ModelShape
    return ModelShape(obs, A, C, S, H, L)


def _engine(obs, net, B, N=1, **kw):
    from stochastic_muzero_b200 import SearchEngine
    from stochastic_muzero_b200.weights import random_blob
    eng = SearchEngine(dict(SEARCH, num_simulations=N), A, C, max_trees=B, model_shape=_shape(obs), net=net, **kw)
    blob = random_blob(_shape(obs), seed=obs)
    eng.set_weights(blob)
    return eng, NO.NetOracle(blob, obs, A, C, S, H, L)


def _obs(B, obs, seed=0):
    return np.random.default_rng(seed).standard_normal((B, obs)).astype(np.float32)


@pytest.mark.parametrize("net", ["fp32", "tc32", "f16", "bf16"])
@pytest.mark.parametrize("obs", WIDTHS)
def test_repr_and_enc_of_wide_observations_match_the_oracle(obs, net):
    B = 300                                    # two full 128-row tiles and a ragged one (four 64-row tiles and a ragged one)
    eng, ref = _engine(obs, net, B)
    x = _obs(B, obs)
    h_tol, p_tol = TOL[net]
    rtol = 1e-5 if net in ("fp32", "tc32") else 0
    h = eng.net_eval("repr", x)["hidden"].cpu().numpy()
    np.testing.assert_allclose(h, ref.representation(x), atol=h_tol, rtol=rtol, err_msg=f"repr {net} obs={obs}")
    o = eng.net_eval("enc", x)
    probs, code = ref.encoder(x)
    np.testing.assert_allclose(o["probs"].cpu().numpy(), probs, atol=p_tol, rtol=rtol, err_msg=f"enc {net} obs={obs}")
    if net in ("fp32", "tc32"):
        close = np.abs(probs.max(1) - np.sort(probs, 1)[:, -2]) < 1e-5
        assert np.array_equal(o["code"].cpu().numpy()[~close], code[~close])
    eng.close()


@pytest.mark.parametrize("net", ["fp32", "tc32", "f16", "bf16"])
@pytest.mark.parametrize("B", [4096, 1000])
def test_root_step_of_wide_observations_matches_the_oracle(B, net):
    obs = 1000                                 # the last K slice is partial (1000 = 7 x 128 + 104)
    eng, ref = _engine(obs, net, B, rng="philox", seed=5, record=True)
    x = _obs(B, obs, seed=B)
    eng.root(obs=torch.from_numpy(x), train=False)
    h_tol, p_tol = TOL[net]
    rtol = 1e-5 if net in ("fp32", "tc32") else 0
    h_ref = ref.representation(x)
    np.testing.assert_allclose(eng.read_hidden(0).cpu().numpy(), h_ref, atol=h_tol, rtol=rtol)
    pol, _ = ref.prediction(h_ref)
    np.testing.assert_allclose(eng.read_record()["root_policy"].cpu().numpy()[:, :A], pol, atol=p_tol, rtol=rtol)
    eng.close()


def _search(net, obs, B, N, seed):
    from stochastic_muzero_b200 import Monte_carlo_tree_search, PackedModel
    from stochastic_muzero_b200.weights import random_blob
    blob = random_blob(_shape(obs), seed=obs)
    mcts = Monte_carlo_tree_search(**{k: v for k, v in SEARCH.items() if k not in ("number_of_player", "custom_loop")},
                                   num_simulations=N, net=net, seed=seed, tree_id_offset=0)
    x = torch.from_numpy(_obs(B, obs, seed=seed))
    roots = mcts.run_batch(x, PackedModel(blob, _shape(obs)), train=False)
    return roots, blob, x.numpy(), mcts


@pytest.mark.parametrize("net", ["fp32", "tc32"])
def test_search_with_wide_observations_replays_through_the_oracles(net):
    """run_batch at obs = 376 without Dirichlet noise: sampled trees searched again on the CPU by the search oracle
    driving the network oracle, with the engine's Philox stream of each tree (the first run_batch call's seed)."""
    obs, B, N, seed = 376, 512, 16, 3
    roots, blob, x, mcts = _search(net, obs, B, N, seed)
    visits = roots.visit_counts.cpu().numpy()
    assert (visits.sum(1) == N).all()
    net_ref = NO.NetOracle(blob, obs, A, C, S, H, L)
    cfg = O.SearchConfig(**{k: v for k, v in SEARCH.items() if k not in ("number_of_player", "custom_loop")},
                         num_simulations=N)
    run_seed = (seed + 0x9E3779B97F4A7C15 * 1) & 0xFFFFFFFFFFFFFFFF
    same, sample = 0, list(range(0, B, 13))
    for b in sample:
        tree = O.search(cfg, NO.NetModel(net_ref, x[b]), O.PhiloxUniforms(run_seed, b), train=False)
        kids = [n for n in range(len(tree.visit)) if tree.depth[n] == 1]
        same += np.array_equal(np.array([tree.visit[n] for n in kids]), visits[b])
    # numpy fp32 network vs the GPU network: a score tie below 1e-6 may flip a visit in a few trees
    assert same >= 0.9 * len(sample), f"only {same}/{len(sample)} trees match the oracle replay"


def test_bf16_search_with_wide_observations_is_finite():
    obs, B, N = 376, 512, 16
    roots, _, _, _ = _search("bf16", obs, B, N, seed=4)
    assert (roots.visit_counts.cpu().numpy().sum(1) == N).all()
    assert np.isfinite(roots.root_values.cpu().numpy()).all()


def test_reference_shaped_model_with_wide_observations_takes_the_fused_path(monkeypatch):
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    from stochastic_muzero_b200.weights import random_blob, shape_of
    obs = 376
    model = FakeMuzero(random_blob(_shape(obs), seed=1), obs, A, C, S, H, L)
    assert shape_of(model) == _shape(obs)

    def no_host_path(*a, **k):
        raise AssertionError("a fusable MLP model left the fused engine")
    monkeypatch.setattr(Monte_carlo_tree_search, "_run_batch_external", no_host_path)
    monkeypatch.setattr(Monte_carlo_tree_search, "_run_callback", no_host_path)
    mcts = Monte_carlo_tree_search(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                                   root_exploration_fraction=0.25, num_simulations=20, maxium_action_sample=2,
                                   number_of_player=1, custom_loop=None, seed=3)
    x = torch.from_numpy(_obs(64, obs, seed=9))
    root = mcts.run(observation=x[:1], model=model, train=True)
    assert root.visit_count == 20 and sum(c.visit_count for c in root.children.values()) == 20
    np.testing.assert_allclose(root.hidden_state.numpy(), model.net.representation(x[:1].numpy()), atol=1e-5)
    roots = mcts.run_batch(x, model, train=True)
    assert (roots.visit_counts.sum(1) == 20).all()
    np.testing.assert_allclose(roots[7].hidden_state.numpy(), model.net.representation(x[7:8].numpy()), atol=1e-5)
