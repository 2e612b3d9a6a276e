"""Gumbel MuZero search (smz_set_search(SMZ_SEARCH_GUMBEL) in include/smz.h; `gumbel=True` in the drop-in).

The root samples its considered actions by Gumbel-Top-k and spends the budget on them by Sequential Halving; interior
decision nodes choose deterministically from the improved policy of completed Q-values; chance nodes keep the
reference's sampling.  tests/gumbel_oracle.py states the rule; with the rule off it is the reference's search.

No GPU: the Sequential Halving table, the oracle's schedule and coverage, Gumbel-max sampling at N = 0, policy
improvement on a stub model, argument checks.
GPU: the stand-alone tree kernels at every lane width and the fused step of smz_simulate on both tree kernels and every
network mode, each replayed bit for bit by the oracle (given and device Gumbels), a vision search, the device Gumbels'
distribution, the read-out, a pUCT search after a Gumbel search, and the drop-in's paths.
"""
import pickle

import numpy as np
import pytest

import golden_io
import gumbel_oracle as GO
import test_fused_search_configurations as F
import test_legal_actions as LA
import test_node_pattern as NP
from oracle import mcts_oracle as O

f32 = np.float32
P_KIND = {False: GO.reference_is_chance, True: lambda d: bool(d & 1)}      # node kind by depth: reference, paper
SEARCH_KEYS = ("pb_c_base", "pb_c_init", "discount", "root_dirichlet_alpha", "root_exploration_fraction",
               "num_simulations", "maxium_action_sample", "number_of_player", "custom_loop")


class RootValueModel(NP.StubModel):
    """NP.StubModel with a seeded network value at the root."""

    def root(self):
        h, p, _ = super().root()
        return h, p, f32(np.random.default_rng([self.seed, self.tree, 1 << 29]).normal())


class DominantModel:
    """Every subtree under root action `good` evaluates to +1, every other to -1; uniform policies."""

    def __init__(self, A, C, good):
        self.A, self.C, self.good = A, C, good

    def root(self):
        return ("root", None), np.full(self.A, 1.0 / self.A, f32), f32(0)

    def _tag(self, h, a):
        return h[1] if h[0] != "root" else (a == self.good)

    def afterstate(self, sim, h, a):
        t = self._tag(h, a)
        return ("n", t), np.full(self.C, 1.0 / self.C, f32), f32(1 if t else -1)

    def dynamics(self, sim, h, c):
        t = self._tag(h, c)
        return ("n", t), np.full(self.A, 1.0 / self.A, f32), f32(1 if t else -1), f32(0)


# ---------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------
def test_considered_visits_table():
    assert GO.considered_visits(4, 8) == [0, 0, 0, 0, 1, 1, 2, 2]
    assert GO.considered_visits(16, 50) == ([0] * 16 + [1] * 8 + [2] * 4 + [3] * 4 + [4] * 4 +
                                            [5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11])
    assert GO.considered_visits(1, 5) == [0, 1, 2, 3, 4]
    assert GO.considered_visits(0, 3) == [0, 1, 2]
    assert GO.considered_visits(8, 5) == [0] * 5                 # N < n
    assert GO.considered_visits(2, 6) == [0, 0, 1, 1, 2, 2]
    for n in range(33):
        assert GO.considered_visits(n, 0) == []


@pytest.mark.parametrize("name", golden_io.tree_cases())
def test_oracle_with_the_rule_off_replays_the_reference_tapes(name):
    z = golden_io.load_tree_case(name)
    c = z["config"]
    cfg = O.SearchConfig(**{k: c[k] for k in SEARCH_KEYS})
    for b in range(len(z["n_nodes"])):
        rng = O.TapeUniforms(z["uniforms"][b, :z["n_uniforms"][b]])
        model = O.TapeModel(z["root_policy"][b], z["sim_policy"][b], z["sim_width"][b], z["sim_value"][b],
                            z["sim_reward"][b])
        tree = GO.search(cfg, model, rng, train=z["train"], dirichlet=z["dirichlet"][b],
                         root_to_play=int(z["exp_root_to_play"][b]))
        assert rng.cursor == z["n_uniforms"][b]
        golden_io.assert_dump_equal(tree.dump(), golden_io.expected_dump(z, b), f"{name}[{b}]")


def root_schedule_holds(cfg, gcfg, tree, n_legal):
    """Every simulation's root child had, before its visit, the considered count of T[min(m, |L|)][sim]."""
    T = GO.considered_visits(min(gcfg.max_considered_actions, n_legal), cfg.num_simulations)
    counts = {}
    for sim, path in enumerate(tree.paths):
        a = path[0]
        if counts.get(a, 0) != T[sim]:
            return False
        counts[a] = counts.get(a, 0) + 1
    return True


@pytest.mark.parametrize("A,C,K", [(4, 4, 2), (9, 3, 3), (32, 4, 4), (5, 32, 32), (1, 1, 1)])
@pytest.mark.parametrize("paper", [False, True])
def test_oracle_root_follows_sequential_halving(A, C, K, paper):
    kind = P_KIND[paper]
    for m in (1, 2, 3, 5, 16, 32):
        for N in (0, 1, 11, 50):
            for mask in LA.mask_table(A, m).values():
                L = LA.legal_of(mask)
                cfg = O.SearchConfig(num_simulations=N, maxium_action_sample=K, number_of_player=2, discount=0.97)
                gcfg = GO.GumbelConfig(max_considered_actions=m)
                model = RootValueModel(A * 31 + m, A, C)
                g = np.random.default_rng(m + N).gumbel(size=A)
                tree = GO.search(cfg, model, O.MTUniforms(N), legal=L, gumbel=gcfg, gumbels=g, kind=kind)
                assert [tree.key[c] for c in tree.children[0]] == L
                assert root_schedule_holds(cfg, gcfg, tree, len(L)), (m, N, L)
                firsts = {p[0] for p in tree.paths}
                assert len(firsts) == min(m, len(L), N)
                if m >= len(L) and N >= len(L):
                    assert firsts == set(L)
                act, pol = GO.readout(cfg, gcfg, tree, tree.raw_value[0], g, A)
                assert act in L and abs(pol.sum() - 1) < 1e-12 and (pol[~mask] == 0).all()



def test_gumbel_max_sampling_at_zero_simulations():
    """With N = 0 the read-out action is a Gumbel-max sample of the prior: chi-square over 20 000 seeded trees with the
    engine's device Gumbels (Philox stream 3)."""
    from scipy.stats import chisquare
    A, n, seed = 5, 20000, 123
    policy = np.array([0.4, 0.05, 0.3, 0.15, 0.1], f32)
    cfg = O.SearchConfig(num_simulations=0)
    gcfg = GO.GumbelConfig()
    tree = GO.search(cfg, O.TapeModel(policy, np.zeros((0, A)), [], [], []), O.MTUniforms(0), gumbel=gcfg)
    prior = np.array([float(tree.prior[c]) for c in tree.children[0]])
    counts = np.zeros(A)
    for t in range(n):
        g = GO.philox_gumbels(seed, t, range(A), A)
        counts[GO.readout(cfg, gcfg, tree, tree.raw_value[0], g, A)[0]] += 1
    assert chisquare(counts, prior / prior.sum() * n).pvalue > 1e-3


def test_improved_policy_moves_mass_to_the_dominant_action():
    A, C, good = 4, 3, 2
    for paper in (False, True):
        cfg = O.SearchConfig(num_simulations=30, maxium_action_sample=2, discount=0.99)
        gcfg = GO.GumbelConfig()
        g = np.random.default_rng(7).gumbel(size=A)
        tree = GO.search(cfg, DominantModel(A, C, good), O.MTUniforms(3), gumbel=gcfg, gumbels=g, kind=P_KIND[paper])
        act, pol = GO.readout(cfg, gcfg, tree, tree.raw_value[0], g, A)
        assert pol[good] > 0.9 and pol.argmax() == good and act == good


def test_set_search_validates_its_arguments_without_a_gpu():
    from stochastic_muzero_b200 import Monte_carlo_tree_search, _lib
    lib = _lib.load()
    ok = (_lib.SEARCH_GUMBEL, 16, 50.0, 0.1)
    bad = [((2, 16, 50.0, 0.1), "policy"), ((-1, 16, 50.0, 0.1), "policy"), ((1, 0, 50.0, 0.1), "max_considered"),
           ((1, 33, 50.0, 0.1), "max_considered"), ((1, 16, -1.0, 0.1), "c_visit"), ((1, 16, 50.0, -0.5), "c_visit"),
           ((1, 16, float("inf"), 0.1), "c_visit"), ((1, 16, 50.0, float("nan")), "c_visit")]
    for args, what in bad:
        assert lib.smz_set_search(None, *args) == _lib.SMZ_E_INVALID_ARG
        assert what in lib.smz_last_error().decode(), args
    for args in (ok, (_lib.SEARCH_PUCT, 1, 0.0, 0.0), (1, 32, 0.0, 1e3)):
        assert lib.smz_set_search(None, *args) == _lib.SMZ_E_INVALID_ARG
        assert "null engine" in lib.smz_last_error().decode()
    for kw in ({"max_considered_actions": 0}, {"max_considered_actions": 33}, {"c_visit": -1.0},
               {"c_scale": float("inf")}):
        with pytest.raises(ValueError):
            Monte_carlo_tree_search(gumbel=True, **kw)
    m = Monte_carlo_tree_search.from_config({"monte_carlo_tree_search": {"num_simulations": 4, "gumbel": True,
                                                                          "max_considered_actions": 4, "c_scale": 1.0}})
    assert m.gumbel and m.max_considered_actions == 4 and m.c_scale == 1.0 and m.c_visit == 50.0
    clone = pickle.loads(pickle.dumps(m))
    assert clone.gumbel and clone.max_considered_actions == 4 and clone.c_scale == 1.0
    assert not Monte_carlo_tree_search().gumbel


# ---------------------------------------------------------------------------------------------------
# GPU: helpers
# ---------------------------------------------------------------------------------------------------
def check_readout(cfg, gcfg, tree, got_action, got_policy, gumbels, A, what):
    act, pol = GO.readout(cfg, gcfg, tree, tree.raw_value[0], gumbels, A)
    assert got_action == act, f"{what}: action {got_action}, oracle {act}"
    np.testing.assert_allclose(got_policy, pol, rtol=1e-12, atol=1e-300, err_msg=f"{what}: improved policy")


# ---------------------------------------------------------------------------------------------------
# GPU 1: the stand-alone tree kernels with tape uniforms and given Gumbels
# ---------------------------------------------------------------------------------------------------
STANDALONE = [  # A, C, K, N, players, loop, train, m
    (2, 2, 2, 40, 1, None, True, 16), (3, 4, 2, 50, 2, None, True, 2), (4, 6, 3, 50, 3, None, False, 5),
    (5, 3, 7, 11, 1, "1>2>1>3", True, 1), (16, 9, 4, 50, 2, None, True, 5), (4, 32, 32, 50, 1, None, True, 32),
    (4, 32, 3, 200, 2, None, True, 2), (32, 4, 4, 50, 1, None, True, 16), (32, 32, 32, 11, 2, None, True, 32),
    (6, 6, 1, 1, 1, None, True, 16), (7, 5, 2, 0, 1, None, True, 2)]


def _lane_runs():
    for A, C, K, N, players, loop, train, m in STANDALONE:
        need = max(2, 1 << (max(A, C) - 1).bit_length())
        for G in (2, 4, 8, 16, 32):
            if G >= need:
                yield pytest.param(A, C, K, N, players, loop, train, m, G, id=f"a{A}c{C}k{K}_n{N}_m{m}_p{players}_G{G}")


@pytest.mark.gpu
@pytest.mark.parametrize("A,C,K,N,players,loop,train,m,G", list(_lane_runs()))
def test_standalone_kernels_replay_the_gumbel_oracle(A, C, K, N, players, loop, train, m, G):
    import torch
    from stochastic_muzero_b200 import SearchEngine
    B, seed = 9, 3000 + A * 37 + C + N
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.99, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=K,
                  number_of_player=players, custom_loop=loop)
    cfg = O.SearchConfig(**search)
    gcfg = GO.GumbelConfig(max_considered_actions=m)
    n_phase = len(cfg.cycle_map())
    paper = G in (8, 32)
    models = [RootValueModel(seed, A, C, tree=b) for b in range(B)]
    g = np.random.default_rng(seed)
    tape = g.random((B, 20000))
    rtp = np.arange(B, dtype=np.int32) - 4
    legal = np.concatenate([np.stack(list(LA.mask_table(A, seed).values())), LA.random_masks(B, A, seed)])[:B]
    gumbels = g.gumbel(size=(B, A))
    eng = SearchEngine(search, A, C, max_trees=B, net="external", rng="tape", lanes_per_tree=G, paper_alternation=paper)
    eng.set_uniform_tape(torch.from_numpy(tape))
    eng.set_search(True, m)
    roots_in = [mo.root() for mo in models]
    eng.root_gumbel(root_policy=torch.from_numpy(np.stack([r[1] for r in roots_in])),
                    root_value=torch.from_numpy(np.array([r[2] for r in roots_in], f32)),
                    root_to_play=torch.from_numpy(rtp), train=train, gumbels=torch.from_numpy(gumbels),
                    legal=torch.from_numpy(legal))
    W = max(A, C)
    actions, branches = np.zeros((B, N), np.int64), np.zeros((B, N), np.int64)
    for s in range(N):
        _slot, action, branch = (t.cpu().numpy() for t in eng.select(s))
        pol, val, rew = np.zeros((B, W), f32), np.zeros(B, f32), np.zeros(B, f32)
        for b in range(B):
            p, val[b], rew[b] = models[b].outputs(s, int(branch[b]), int(action[b]))
            pol[b, :len(p)] = p
        actions[:, s], branches[:, s] = action, branch
        eng.expand_backup(s, pol, val, rew)
    eng.stats()
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    out = {k: v.cpu().numpy() for k, v in eng.read_gumbel().items()}
    raw = eng.read_raw_values().cpu().numpy()
    for b in range(B):
        model = RootValueModel(seed, A, C, tree=b)
        rng = O.TapeUniforms(tape[b])
        L = LA.legal_of(legal[b])
        tree = GO.search(cfg, model, rng, train=train, root_to_play=int(rtp[b]) % n_phase, legal=L, gumbel=gcfg,
                         gumbels=gumbels[b], kind=P_KIND[paper])
        what = f"G={G}[{b}]"
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), what)
        assert got["n_uniforms"] == rng.cursor, what
        assert [p[-1] for p in tree.paths] == actions[b].tolist(), f"{what}: selected actions / sampled codes"
        assert [br for _, br, _, _ in model.log] == branches[b].tolist(), f"{what}: evaluation branch"
        assert root_schedule_holds(cfg, gcfg, tree, len(L))
        kids = np.flatnonzero(got["depth"] == 1)
        assert np.array_equal(roots["visits"][b][L], got["visit"][kids]) and roots["visits"][b][~legal[b]].sum() == 0
        exp_g = np.where(legal[b], gumbels[b], 0.0) if train else np.zeros(A)
        assert np.array_equal(out["gumbels"][b], exp_g), what
        assert raw[b, 0] == tree.raw_value[0]
        check_readout(cfg, gcfg, tree, out["actions"][b], out["improved_policy"][b], exp_g, A, what)
    assert roots["error"][0] == 0
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 2: the fused step of smz_simulate on both tree kernels, device Gumbels replayed
# ---------------------------------------------------------------------------------------------------
_BY_NAME = {c.name: c for c in F.CASES}
FUSED_CASES = list(NP.FUSED_CASES) + [_BY_NAME["n1_no_fused_step"], _BY_NAME["n0_wide_readout"],
                                      _BY_NAME["discount0"], _BY_NAME["a2c32k32_n31_mirror_limit"]]
M_OF = {"a16c16k4_lanes16": 4, "a32c32k3_peaky": 32, "players3_custom_loop": 2, "cfg3_a4c32k32_n100": 1,
        "a8c8k2_lanes8": 5}
MASKED = {"a16c16k4_lanes16", "cfg3_a4c32k32_n100", "players3_custom_loop", "a32c32k3_bf16_m64_off"}
PAPER = {"a16c16k4_lanes16", "a2c2k1_n40_lanes2", "cfg3_a4c32k32_n100_tc32"}


def run_gumbel_case(case, monkeypatch, no_smem=False, export=(), legal=None, m=16, paper=False, gumbels=None):
    import torch
    from stochastic_muzero_b200 import SearchEngine
    for k in F.ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in case.env:
        monkeypatch.setenv(k, v)
    if no_smem:
        monkeypatch.setenv("SMZ_NO_TREE_SMEM", "1")
    shape, blob = F._model(case)
    obs, rtp, tape = F._inputs(case)
    eng = SearchEngine(case.search(), case.A, case.C, max_trees=case.max_trees or case.n_trees, model_shape=shape,
                       net=case.net, rng=case.rng, seed=case.seed, tree_id_offset=case.offset,
                       lanes_per_tree=case.lanes, record=True, paper_alternation=paper)
    eng.set_weights(blob)
    if tape is not None:
        eng.set_uniform_tape(torch.from_numpy(tape))
    eng.set_search(True, m)
    eng.root_gumbel(obs=torch.from_numpy(obs), root_to_play=None if rtp is None else torch.from_numpy(rtp),
                    train=case.train, legal=None if legal is None else torch.from_numpy(legal),
                    gumbels=None if gumbels is None else torch.from_numpy(gumbels))
    for k in case.chunks or (case.N,):
        eng.simulate(k)
    eng.stats()
    out = {"roots": {k: v.cpu().numpy() for k, v in eng.read_roots().items()},
           "rec": {k: v.cpu().numpy() for k, v in eng.read_record().items()},
           "gumbel": {k: v.cpu().numpy() for k, v in eng.read_gumbel().items()},
           "raw": eng.read_raw_values().cpu().numpy(),
           "trees": {int(b): eng.export_tree(int(b)) for b in export}, "eng": eng, "tape": tape, "rtp": rtp}
    for k in F.ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    return out


class _RecordModel(O.TapeModel):
    def __init__(self, root_value, *a):
        super().__init__(*a)
        self.root_value = f32(root_value)

    def root(self):
        return None, self.root_policy, self.root_value


def replay_gumbel(case, run, b, legal_row, m, paper, gumbels=None):
    rec = run["rec"]
    width = np.where(rec["sim_branch"][b] == 1, case.A, case.C)
    model = _RecordModel(run["raw"][b, 0], rec["root_policy"][b, :case.A], rec["sim_policy"][b], width,
                         rec["sim_value"][b], rec["sim_reward"][b])
    rng = O.TapeUniforms(run["tape"][b]) if case.rng == "tape" else O.PhiloxUniforms(case.seed, case.offset + b)
    cfg = O.SearchConfig(**case.search())
    phase = 0 if run["rtp"] is None else int(run["rtp"][b]) % len(cfg.cycle_map())
    g = run["gumbel"]["gumbels"][b] if gumbels is None else gumbels
    tree = GO.search(cfg, model, rng, train=case.train, root_to_play=phase, legal=LA.legal_of(legal_row),
                     gumbel=GO.GumbelConfig(max_considered_actions=m), gumbels=g, kind=P_KIND[paper])
    return tree, rng.cursor, cfg


def check_gumbel_replay(case, run, legal, m, paper, what):
    for b, got in run["trees"].items():
        tree, cursor, cfg = replay_gumbel(case, run, b, legal[b], m, paper)
        golden_io.assert_dump_equal(got, tree.dump(), f"{what}[{b}]")
        assert got["n_uniforms"] == cursor, f"{what}[{b}]: {got['n_uniforms']} draws consumed, oracle {cursor}"
        check_readout(cfg, GO.GumbelConfig(max_considered_actions=m), tree, run["gumbel"]["actions"][b],
                      run["gumbel"]["improved_policy"][b], run["gumbel"]["gumbels"][b], case.A, f"{what}[{b}]")
        if case.N:
            assert np.array_equal(run["raw"][b, 1:], run["rec"]["sim_value"][b])
    n = case.n_trees
    assert legal[np.arange(n), run["gumbel"]["actions"]].all()
    assert (run["gumbel"]["improved_policy"][~legal] == 0).all()
    assert (run["gumbel"]["gumbels"][~legal] == 0).all()
    if not case.train:
        assert (run["gumbel"]["gumbels"] == 0).all()


def test_gumbel_case_table():
    names = {c.name for c in FUSED_CASES}
    assert set(M_OF) <= names and MASKED <= names and PAPER <= names
    fused = [c for c in FUSED_CASES if c.N >= 2]
    assert {c.G for c in fused if c.kernel(F.B200_SMS) == "mirror"} >= {2, 4, 8, 16, 32}
    assert {c.net for c in FUSED_CASES} == set(F.NETS) and any(c.chunks for c in FUSED_CASES)
    assert any((c.A, c.C, c.K) == (4, 32, 32) for c in FUSED_CASES)


@pytest.mark.gpu
@pytest.mark.parametrize("case", FUSED_CASES, ids=lambda c: c.name)
def test_fused_gumbel_search_replays_bit_exact_on_both_tree_kernels(case, monkeypatch):
    sample = F.replay_sample(case)
    legal = np.ones((case.n_trees, case.A), bool)
    if case.name in MASKED:
        legal = LA.random_masks(case.n_trees, case.A, case.seed % 2 ** 32)
    m = M_OF.get(case.name, 16)
    paper = case.name in PAPER
    label = case.kernel(F._device_sms()) or "no fused step"
    default = run_gumbel_case(case, monkeypatch, export=sample, legal=legal, m=m, paper=paper)
    check_gumbel_replay(case, default, legal, m, paper, f"{case.name} default ({label}, G={case.G})")
    # the device Gumbels are those of the oracle's Philox restatement (CUDA's log against numpy's: 1e-15)
    for b in sample[:4]:
        exp = GO.philox_gumbels(case.seed, case.offset + b, LA.legal_of(legal[b]), case.A)
        if case.train:
            np.testing.assert_allclose(default["gumbel"]["gumbels"][b], exp, rtol=1e-14, atol=1e-14)
    # the arena-only kernel, replaying the recorded Gumbels through smz_root_gumbel
    arena = run_gumbel_case(case, monkeypatch, no_smem=True, export=sample, legal=legal, m=m, paper=paper,
                            gumbels=default["gumbel"]["gumbels"])
    check_gumbel_replay(case, arena, legal, m, paper, f"{case.name} SMZ_NO_TREE_SMEM=1 (arena, G={case.G})")
    F._assert_roots_equal(default["roots"], arena["roots"], f"{case.name}: {label} vs arena")
    for k in ("actions", "improved_policy", "gumbels"):
        assert np.array_equal(default["gumbel"][k], arena["gumbel"][k]), f"{case.name}: read_gumbel {k}"
    assert default["roots"]["error"][0] == 0 and (default["roots"]["visits"].sum(1) == case.N).all()
    default["eng"].close()
    arena["eng"].close()


@pytest.mark.gpu
def test_vision_gumbel_search_replays_bit_exact():
    import torch
    from stochastic_muzero_b200 import SearchEngine, VisionShape
    z = golden_io.load_vision_case("a4")
    A, S, H, L = [int(v) for v in z["dims"]]
    B, N, seed = 256, 40, 921
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=3,
                  number_of_player=2, custom_loop=None)
    eng = SearchEngine(search, A, A, max_trees=B, model_shape=VisionShape(A, S, H, L), net="vision", rng="philox",
                       seed=seed, record=True)
    eng.set_weights(z["weights"])
    eng.set_search(True, 2)
    legal = LA.random_masks(B, A, seed)
    obs = torch.rand(B, 3, 98, 98, generator=torch.Generator().manual_seed(6))
    eng.root_gumbel(obs=obs.reshape(B, -1), train=True, legal=torch.from_numpy(legal).cuda())
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    gout = {k: v.cpu().numpy() for k, v in eng.read_gumbel().items()}
    raw = eng.read_raw_values().cpu().numpy()
    cfg = O.SearchConfig(**search)
    gcfg = GO.GumbelConfig(max_considered_actions=2)
    for b in (0, 1, 63, 64, 200, 255):
        model = _RecordModel(raw[b, 0], rec["root_policy"][b, :A], rec["sim_policy"][b], np.full(N, A),
                             rec["sim_value"][b], rec["sim_reward"][b])
        rng = O.PhiloxUniforms(seed, b)
        tree = GO.search(cfg, model, rng, legal=LA.legal_of(legal[b]), gumbel=gcfg, gumbels=gout["gumbels"][b])
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"vision[{b}]")
        assert got["n_uniforms"] == rng.cursor
        check_readout(cfg, gcfg, tree, gout["actions"][b], gout["improved_policy"][b], gout["gumbels"][b], A,
                      f"vision[{b}]")
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 3-5: device Gumbels, the read-out over many trees, pUCT after Gumbel
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_gumbels_are_standard_gumbel_and_skip_illegal_actions():
    import torch
    from stochastic_muzero_b200 import SearchEngine
    B, A, seed = 65536, 8, 77
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=0, maxium_action_sample=2,
                  number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, A, A, max_trees=B, net="external", rng="philox", seed=seed, tree_id_offset=5)
    eng.set_search(True)
    legal = LA.random_masks(B, A, seed)
    pol = np.random.default_rng(1).dirichlet([1.0] * A, B).astype(f32)
    eng.root_gumbel(root_policy=torch.from_numpy(pol), root_value=torch.zeros(B), train=True,
                    legal=torch.from_numpy(legal))
    out = {k: v.cpu().numpy() for k, v in eng.read_gumbel().items()}
    g = out["gumbels"]
    assert (g[~legal] == 0).all()
    v = g[legal]
    assert abs(v.mean() - 0.5772156649) < 0.01 and abs(v.var() - np.pi ** 2 / 6) < 0.02
    for b in (0, 1, 4095, B - 1):
        np.testing.assert_allclose(g[b], GO.philox_gumbels(seed, 5 + b, LA.legal_of(legal[b]), A), rtol=1e-14,
                                   atol=1e-14)
    assert legal[np.arange(B), out["actions"]].all()
    assert (out["improved_policy"][~legal] == 0).all()
    np.testing.assert_allclose(out["improved_policy"].sum(1), 1.0, rtol=1e-12)
    # N = 0: the improved policy is the prior over the legal actions, the action its Gumbel-max sample
    priors = eng.read_roots()["priors"].cpu().numpy()
    np.testing.assert_allclose(out["improved_policy"], priors / priors.sum(1, keepdims=True), rtol=1e-12)
    logits = np.where(legal, np.log(np.where(legal, priors, 1.0)), -np.inf)
    assert np.array_equal(out["actions"], np.argmax(logits + g, 1))
    eng.close()


@pytest.mark.gpu
def test_puct_search_after_a_gumbel_search_is_a_fresh_search(monkeypatch):
    import torch
    case = _BY_NAME["a16c16k4_lanes16"]
    sample = F.replay_sample(case)
    fresh = F.run_case(case, monkeypatch, export=sample)
    shape, blob = F._model(case)
    obs, rtp, _ = F._inputs(case)
    from stochastic_muzero_b200 import SearchEngine
    eng = SearchEngine(case.search(), case.A, case.C, max_trees=case.n_trees, model_shape=shape, net=case.net,
                       rng=case.rng, seed=case.seed, tree_id_offset=case.offset, lanes_per_tree=case.lanes, record=True)
    eng.set_weights(blob)
    for gumbel in (False, True, False):        # the graph of the first pUCT search is dropped and captured again
        eng.set_search(gumbel)
        with pytest.raises(Exception):
            (eng.root if gumbel else eng.root_gumbel)(obs=torch.from_numpy(obs), train=True)
        (eng.root_gumbel if gumbel else eng.root)(obs=torch.from_numpy(obs), train=case.train)
        eng.simulate()
        eng.stats()
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    F._assert_roots_equal(fresh["roots"], roots, "pUCT after Gumbel")
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    for k, v in fresh["rec"].items():
        assert np.array_equal(v.view(np.uint8), rec[k].view(np.uint8)), f"record {k}"
    for b in sample:
        golden_io.assert_dump_equal(eng.export_tree(b), fresh["trees"][b], f"pUCT after Gumbel [{b}]")
    with pytest.raises(Exception):
        eng.read_gumbel()
    eng.close()
    fresh["eng"].close()


# ---------------------------------------------------------------------------------------------------
# GPU 6: the drop-in
# ---------------------------------------------------------------------------------------------------
def _check_batch(roots, legal, N):
    g = roots.gumbel()
    act, pol = g["actions"].cpu().numpy(), g["improved_policy"].cpu().numpy()
    n = len(act)
    assert legal[np.arange(n), act].all() and (pol[~legal] == 0).all()
    np.testing.assert_allclose(pol.sum(1), 1.0, rtol=1e-12)
    vis = roots.visit_counts.cpu().numpy()
    assert (vis.sum(1) == N).all() and (vis[~legal] == 0).all()


@pytest.mark.gpu
def test_dropin_gumbel_on_every_search_path():
    import torch
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import ModelShape, Monte_carlo_tree_search, PackedModel, batched_model, random_blob
    from stochastic_muzero_b200.selfplay import SelfPlay, VectorCartPole, reanalyse
    zn = golden_io.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    A = dims[1]
    kw = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=11, maxium_action_sample=2, number_of_player=2,
              custom_loop=None)
    batch = np.random.default_rng(0).random((64, A)) < 0.5
    batch[:, 0] = True
    model = FakeMuzero(zn["weights"], *dims)
    for paper in (False, True):
        mcts = Monte_carlo_tree_search(**kw, seed=3, net="fp32", gumbel=True, max_considered_actions=2,
                                       paper_alternation=paper)
        obs = torch.randn(1, dims[0], generator=torch.Generator().manual_seed(1))
        root = mcts.run(observation=obs, model=model, train=True, legal_actions=[A - 1])
        assert sorted(int(k) for k in root.children) == [A - 1] and root.visit_count == 11
        roots = mcts.run_batch(torch.randn(64, dims[0]), model, train=True, legal_actions=torch.from_numpy(batch).cuda())
        _check_batch(roots, batch, 11)
        clone = pickle.loads(pickle.dumps(mcts))
        assert clone.gumbel and clone.max_considered_actions == 2
        _check_batch(clone.run_batch(torch.randn(64, dims[0]), model, train=False), np.ones((64, A), bool), 11)

    cb_model = FakeMuzero(zn["weights"], *dims)
    cb_model.model_structure = "lstm_model"          # not fusable: host-model callback / batched back-end
    mcts = Monte_carlo_tree_search(**kw, seed=5, gumbel=True)
    root = mcts.run(observation=np.random.default_rng(4).standard_normal((1, dims[0])).astype(np.float32),
                    model=cb_model, train=True, legal_actions=[0])
    assert sorted(int(k) for k in root.children) == [0] and root.visit_count == 11
    assert mcts._engines[("external", A, dims[2], None)].read_gumbel()["actions"].item() == 0
    roots = mcts.run_batch(torch.randn(48, dims[0]), cb_model, train=True, legal_actions=batch[:48])
    _check_batch(roots, batch[:48], 11)
    backend = batched_model.ReferenceModuleBackend(cb_model)
    roots = Monte_carlo_tree_search(**kw, seed=6, gumbel=True).run_batch(torch.randn(32, dims[0]), backend)
    _check_batch(roots, np.ones((32, A), bool), 11)

    # self-play acts on the Gumbel action and stores the improved policy; reanalyse returns it as the target
    shape = ModelShape(4, 2, 2, 61, 126, 4)
    cart = PackedModel(random_blob(shape, 0), shape)
    mcts = Monte_carlo_tree_search(discount=0.997, num_simulations=8, maxium_action_sample=2, net="fp32", seed=7,
                                   gumbel=True)
    buf = SelfPlay(mcts, cart, VectorCartPole(64, device="cuda", seed=0), horizon=3).run()
    pol = buf["child_visits"].cpu().numpy()
    np.testing.assert_allclose(pol.sum(-1), 1.0, rtol=1e-12)
    assert (pol[np.arange(3)[:, None], np.arange(64)[None], buf["actions"].cpu().numpy().astype(np.int64)] > 0).all()
    re = reanalyse(mcts, cart, buf["observations"], chunk=100)
    assert re["child_visits"].shape == (3, 64, 2)
    np.testing.assert_allclose(re["child_visits"].sum(-1).cpu().numpy(), 1.0, rtol=1e-12)
