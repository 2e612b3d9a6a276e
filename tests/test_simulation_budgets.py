"""Per-tree simulation budgets and exploration flags (smz_set_root_budgets in include/smz.h; `num_simulations=` and
`explore=` of the drop-in, `playout_cap` of SelfPlay).

A tree with budget n is, bit for bit, the reference's search with num_simulations = n; the oracles take N as a parameter,
so they define every budgeted tree.  A tree's exploration flag replaces `train` for its root noise.

No GPU: the host checks of budgets and flags, the per-budget Sequential Halving tables against the Gumbel oracle, and the
oracles' per-tree rules.
GPU: all-N budgets change nothing (arena bytes, draws, record, read-out); mixed budgets (0, 1, N - 1, N, random) replayed
by the oracle on the stand-alone kernels, on the fused step of both tree kernels in every network mode, in pUCT and Gumbel,
with legal masks and both node patterns; simulation steps without any tree; independence of the other trees' budgets;
exploration flags; statistics and flag 4; a vision search; the drop-in's paths, self-play with playout caps and reanalyse.
"""
import pickle

import numpy as np
import pytest

import golden_io
import gumbel_oracle as GO
import test_fused_search_configurations as F
import test_gumbel_search as TG
import test_legal_actions as LA
import test_node_pattern as NP
from oracle import mcts_oracle as O

f32 = np.float32
P_KIND = TG.P_KIND


def mixed_budgets(n, N, seed):
    """Budgets of n trees in [0, N]: 0, 1, N - 1 and N first, then seeded random values."""
    b = np.random.default_rng(seed).integers(0, N + 1, n)
    b[:4] = [0, min(1, N), max(N - 1, 0), N][:min(4, n)]
    return b.astype(np.int32)


# ---------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------
def test_host_budgets_and_flags_are_checked_before_any_gpu_work():
    import torch
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    from stochastic_muzero_b200.engine import budget_rows, explore_rows
    assert budget_rows(3, 4, 5).tolist() == [3, 3, 3, 3]
    assert budget_rows([0, 5, 2], 3, 5).dtype == torch.int32
    for bad in ([0, 6, 1], [-1, 0, 0], [0, 1], [[0, 1, 2]], [0.0, 1.0, 2.0], np.array([1.5, 0, 0]), [True, False, True],
                True, 6, -1, torch.tensor([0, 1, 2], dtype=torch.float32)):
        with pytest.raises(ValueError):
            budget_rows(bad, 3, 5)
    assert explore_rows([True, False], 2).tolist() == [1, 0]
    assert explore_rows(np.array([0, 1]), 2).tolist() == [0, 1]
    for bad in ([0, 2], [1, 0, 1], np.array([0.5, 1.0]), [[1, 0]]):
        with pytest.raises(ValueError):
            explore_rows(bad, 2)
    mcts = Monte_carlo_tree_search(num_simulations=4)
    obs = np.zeros((3, 4), f32)
    for kw in ({"num_simulations": [0, 5, 1]}, {"num_simulations": 9}, {"num_simulations": [1, 2]},
               {"num_simulations": [1.0, 2.0, 3.0]}, {"explore": [1, 0]}, {"explore": [0, 3, 1]}):
        with pytest.raises(ValueError):
            mcts.run_batch(obs, object(), **kw)      # raises before the model is looked at
    for n in (1.5, 5, -1, True):
        with pytest.raises(ValueError):
            mcts.run(obs[:1], object(), num_simulations=n)


@pytest.mark.parametrize("N", [0, 1, 7, 50, 64])
def test_per_budget_sequential_halving_tables_equal_the_oracle(N):
    import ctypes as C
    from stochastic_muzero_b200 import _lib
    lib = _lib.load()
    Nt = max(N, 1)
    t = np.zeros((N + 1, 33, Nt), np.int32)
    assert lib.smz_sequential_halving_table(N, t.ctypes.data_as(C.c_void_p)) == 0
    for b in range(N + 1):
        for n in range(33):
            assert t[b, n, :b].tolist() == GO.considered_visits(n, b), (b, n)
            assert (t[b, n, b:] == 0).all()
    assert lib.smz_sequential_halving_table(-1, t.ctypes.data_as(C.c_void_p)) == _lib.SMZ_E_INVALID_ARG


@pytest.mark.parametrize("gumbel", [False, True])
def test_oracle_search_with_n_simulations_is_a_prefix_in_puct_and_follows_its_own_schedule_in_gumbel(gumbel):
    """The budgeted trees of a batch are independent searches with N = budget.  pUCT: such a search visits what the
    first n simulations of an N-simulation search visit (without noise); Gumbel: its root follows T_n, not T_N."""
    A, C, K, N = 5, 4, 3, 24
    for tree_id in range(6):
        for n in (0, 1, 2, 11, N - 1, N):
            for m in (2, 16):
                cfg_n = O.SearchConfig(num_simulations=n, maxium_action_sample=K, number_of_player=2, discount=0.97)
                cfg_N = O.SearchConfig(num_simulations=N, maxium_action_sample=K, number_of_player=2, discount=0.97)
                kw = dict(train=False, gumbel=GO.GumbelConfig(max_considered_actions=m) if gumbel else None,
                          gumbels=np.random.default_rng(tree_id).gumbel(size=A) if gumbel else None)
                tn = GO.search(cfg_n, TG.RootValueModel(tree_id, A, C), O.MTUniforms(tree_id), **kw)
                tN = GO.search(cfg_N, TG.RootValueModel(tree_id, A, C), O.MTUniforms(tree_id), **kw)
                assert len(tn.paths) == n
                if gumbel:
                    assert TG.root_schedule_holds(cfg_n, kw["gumbel"], tn, A)
                else:
                    assert tn.paths == tN.paths[:n]


# ---------------------------------------------------------------------------------------------------
# GPU: runner and replay
# ---------------------------------------------------------------------------------------------------
def make_engine(case, monkeypatch, no_smem=False, paper=False, gumbel=False, m=16, record=True):
    import torch
    from stochastic_muzero_b200 import SearchEngine
    for k in F.ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in case.env:
        monkeypatch.setenv(k, v)
    if no_smem:
        monkeypatch.setenv("SMZ_NO_TREE_SMEM", "1")
    shape, blob = F._model(case)
    eng = SearchEngine(case.search(), case.A, case.C, max_trees=case.max_trees or case.n_trees, model_shape=shape,
                       net=case.net, rng=case.rng, seed=case.seed, tree_id_offset=case.offset,
                       lanes_per_tree=case.lanes, record=record, paper_alternation=paper)
    eng.set_weights(blob)
    obs, rtp, tape = F._inputs(case)
    if tape is not None:
        eng.set_uniform_tape(torch.from_numpy(tape))
    if gumbel:
        eng.set_search(True, m)
    return eng, obs, rtp, tape


def search_once(eng, case, obs, rtp, legal=None, budget=None, explore=None, train=None, gumbels=None, chunks=None,
                export=(), arena=False):
    import torch
    kw = dict(obs=torch.from_numpy(obs), root_to_play=None if rtp is None else torch.from_numpy(rtp),
              train=case.train if train is None else train)
    if legal is not None:
        kw["legal"] = torch.from_numpy(legal)
    if budget is not None:
        kw["budget"] = torch.from_numpy(budget).cuda()          # device budgets: the search runs N steps
    if explore is not None:
        kw["explore"] = torch.from_numpy(explore)
    if eng.gumbel:
        eng.root_gumbel(gumbels=None if gumbels is None else torch.from_numpy(gumbels), **kw)
    else:
        eng.root(**kw)
    for k in chunks or case.chunks or (case.N,):
        eng.simulate(k)
    st = eng.stats()
    out = {"roots": {k: v.cpu().numpy() for k, v in eng.read_roots().items()},
           "rec": {k: v.cpu().numpy() for k, v in eng.read_record().items()},
           "trees": {int(b): eng.export_tree(int(b)) for b in export}, "stats": st}
    if arena:
        out["arena"] = {int(b): eng.export_arena(int(b)) for b in export}
    if eng.gumbel:
        out["gumbel"] = {k: v.cpu().numpy() for k, v in eng.read_gumbel().items()}
        out["raw"] = eng.read_raw_values().cpu().numpy()
    else:
        out["readout"] = {T: {k: v.cpu().numpy() for k, v in eng.select_actions(T).items()} for T in (0.0, 1.0)}
    return out


def replay(case, run, b, n, legal_row, explores, tape, rtp, paper, m):
    """The oracle's search of tree b with num_simulations = n, from the engine's record."""
    rec = run["rec"]
    width = np.where(rec["sim_branch"][b, :n] == 1, case.A, case.C)
    rng = O.TapeUniforms(tape[b]) if case.rng == "tape" else O.PhiloxUniforms(case.seed, case.offset + b)
    cfg = O.SearchConfig(**dict(case.search(), num_simulations=int(n)))
    phase = 0 if rtp is None else int(rtp[b]) % len(cfg.cycle_map())
    args = (rec["root_policy"][b, :case.A], rec["sim_policy"][b, :n], width, rec["sim_value"][b, :n],
            rec["sim_reward"][b, :n])
    if "gumbel" in run:
        tree = GO.search(cfg, TG._RecordModel(run["raw"][b, 0], *args), rng, train=explores,
                         root_to_play=phase, legal=LA.legal_of(legal_row), gumbel=GO.GumbelConfig(max_considered_actions=m),
                         gumbels=run["gumbel"]["gumbels"][b], kind=P_KIND[paper])
    else:
        noise = explores and n > 0
        tree = LA.masked_search(cfg, O.TapeModel(*args), rng, LA.legal_of(legal_row), train=explores,
                                dirichlet=rec["dirichlet"][b] if noise else None, root_to_play=phase, paper=paper)
    return tree, rng.cursor, cfg


def check_budget_replay(case, run, budgets, legal, explore, tape, rtp, paper, m, what):
    n_trees = len(budgets)
    vis = run["roots"]["visits"]
    assert run["roots"]["error"][0] == 0, what
    assert (vis.sum(1) == budgets).all(), f"{what}: root visits against the budgets"
    for b, got in run["trees"].items():
        ex = bool(case.train if explore is None else explore[b])
        tree, cursor, cfg = replay(case, run, b, int(budgets[b]), legal[b], ex, tape, rtp, paper, m)
        golden_io.assert_dump_equal(got, tree.dump(), f"{what}[{b}] budget {budgets[b]}")
        assert got["n_uniforms"] == cursor, f"{what}[{b}]: {got['n_uniforms']} draws, oracle {cursor}"
        if "gumbel" in run:
            TG.check_readout(cfg, GO.GumbelConfig(max_considered_actions=m), tree, run["gumbel"]["actions"][b],
                             run["gumbel"]["improved_policy"][b], run["gumbel"]["gumbels"][b], case.A, f"{what}[{b}]")
    if "readout" in run:
        assert legal[np.arange(n_trees), run["readout"][0.0]["actions"]].all(), f"{what}: read-out"
    dsum = run["stats"]["mean_leaf_depth"] * max(int(np.minimum(budgets, case.N).sum()), 1)
    assert abs(dsum - round(dsum)) < 1e-6 * max(dsum, 1), f"{what}: depth sum {dsum} not over the simulations run"


def assert_same_search(a, b, sample, what):
    F._assert_roots_equal(a["roots"], b["roots"], what)
    for k, v in a["rec"].items():
        assert np.array_equal(v.view(np.uint8), b["rec"][k].view(np.uint8)), f"{what}: record {k}"
    for t in sample:
        for k, v in a["arena"][t].items():
            x, y = (np.ascontiguousarray(np.atleast_1d(c)) for c in (v, b["arena"][t][k]))
            assert x.tobytes() == y.tobytes(), f"{what}[{t}]: arena {k}"
    for key in ("readout", "gumbel"):
        if key in a:
            for k, v in a[key].items():
                if isinstance(v, dict):
                    for kk, vv in v.items():
                        assert np.array_equal(vv, b[key][k][kk]), f"{what}: {key} {k} {kk}"
                else:
                    assert np.array_equal(v, b[key][k]), f"{what}: {key} {k}"
    assert a["stats"]["mean_leaf_depth"] == b["stats"]["mean_leaf_depth"], what


# ---------------------------------------------------------------------------------------------------
# GPU 1-4: the fused step of every network mode on both tree kernels
# ---------------------------------------------------------------------------------------------------
CASES = [c for c in NP.FUSED_CASES if c.N >= 2]
MASKED = {"a16c16k4_lanes16", "cfg3_a4c32k32_n100", "players3_custom_loop", "eval_mode", "chain_n100"}
PAPER = {"a16c16k4_lanes16", "a2c2k1_n40_lanes2", "cfg3_a4c32k32_n100_tc32", "simulate_in_two_chunks"}


def test_budget_case_table():
    names = {c.name for c in CASES}
    assert MASKED <= names and PAPER <= names
    assert {c.G for c in CASES if c.kernel(F.B200_SMS) == "mirror"} >= {2, 4, 8, 16, 32}
    assert {c.net for c in CASES} == set(F.NETS) and any(c.chunks for c in CASES)
    assert any((c.A, c.C, c.K) == (4, 32, 32) for c in CASES)


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["puct", "gumbel"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_fused_budgets_on_both_tree_kernels(case, rule, monkeypatch):
    """On one engine and for both tree kernels: (1) no budgets, (2) all-N budgets with flags = train — byte-identical;
    (3) mixed budgets replayed by the oracle with N = budget per tree, the trees with budget N equal to (1)'s;
    (4) every budget below N and (5) every budget 0 with smz_simulate(N): no error flag, visits = budgets."""
    gumbel = rule == "gumbel"
    sample = F.replay_sample(case)
    n, N = case.n_trees, case.N
    legal = LA.random_masks(n, case.A, case.seed % 2 ** 32) if case.name in MASKED else np.ones((n, case.A), bool)
    paper, m = case.name in PAPER, TG.M_OF.get(case.name, 16)
    mixed = mixed_budgets(n, N, case.seed)
    below = np.minimum(mixed, N - 1).astype(np.int32)
    gumbels = None
    for no_smem in (False, True):
        what = f"{case.name} {rule} {'arena' if no_smem else 'default'}"
        eng, obs, rtp, tape = make_engine(case, monkeypatch, no_smem, paper, gumbel, m)
        base = search_once(eng, case, obs, rtp, legal, export=sample, arena=True, gumbels=gumbels)
        if gumbel and gumbels is None:
            gumbels = base["gumbel"]["gumbels"]                       # the arena kernel replays the device Gumbels
        alln = search_once(eng, case, obs, rtp, legal, budget=np.full(n, N, np.int32),
                           explore=np.full(n, case.train), export=sample, arena=True, gumbels=gumbels)
        assert_same_search(base, alln, sample, f"{what}: all-N budgets")
        mix = search_once(eng, case, obs, rtp, legal, budget=mixed, export=sample, gumbels=gumbels)
        check_budget_replay(case, mix, mixed, legal, None, tape, rtp, paper, m, f"{what} mixed")
        if case.rng == "philox":          # a tree does not depend on the other trees' budgets
            for b in sample:
                if mixed[b] == N:
                    golden_io.assert_dump_equal(mix["trees"][b], base["trees"][b], f"{what}[{b}] mixed vs all-N")
        for budgets, label in ((below, "below N"), (np.zeros(n, np.int32), "all 0")):
            run = search_once(eng, case, obs, rtp, legal, budget=budgets, export=sample[:4], gumbels=gumbels,
                              chunks=(N,))
            check_budget_replay(case, run, budgets, legal, None, tape, rtp, paper, m, f"{what} {label}")
        eng.close()
    for k in F.ENV_KEYS:
        monkeypatch.delenv(k, raising=False)


# ---------------------------------------------------------------------------------------------------
# GPU 2: the stand-alone kernels with tape uniforms at every lane width
# ---------------------------------------------------------------------------------------------------
STANDALONE = [  # A, C, K, N, players, loop, train
    (2, 2, 2, 30, 1, None, True), (3, 4, 2, 40, 2, None, True), (4, 6, 3, 30, 3, None, False),
    (5, 3, 7, 11, 1, "1>2>1>3", True), (16, 9, 4, 30, 2, None, True), (32, 4, 4, 20, 1, None, True),
    (4, 32, 32, 20, 2, None, True)]


def _lane_runs():
    for A, C, K, N, players, loop, train in STANDALONE:
        need = max(2, 1 << (max(A, C) - 1).bit_length())
        for G in (2, 4, 8, 16, 32):
            if G >= need:
                for rule in ("puct", "gumbel"):
                    yield pytest.param(A, C, K, N, players, loop, train, G, rule,
                                       id=f"a{A}c{C}k{K}_n{N}_p{players}_G{G}_{rule}")


@pytest.mark.gpu
@pytest.mark.parametrize("A,C,K,N,players,loop,train,G,rule", list(_lane_runs()))
def test_standalone_kernels_replay_budgeted_trees(A, C, K, N, players, loop, train, G, rule):
    import torch
    from stochastic_muzero_b200 import SearchEngine
    B, seed = 12, 5000 + A * 37 + C + N + G
    gumbel, m = rule == "gumbel", 3
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.99, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=K,
                  number_of_player=players, custom_loop=loop)
    paper = G in (4, 32)
    models = [TG.RootValueModel(seed, A, C, tree=b) for b in range(B)]
    g = np.random.default_rng(seed)
    tape = g.random((B, 20000))
    rtp = np.arange(B, dtype=np.int32) - 4
    legal = LA.random_masks(B, A, seed)
    budgets = mixed_budgets(B, N, seed)
    explore = g.random(B) < 0.5
    gumbels = g.gumbel(size=(B, A))
    eng = SearchEngine(search, A, C, max_trees=B, net="external", rng="tape", lanes_per_tree=G, paper_alternation=paper)
    eng.set_uniform_tape(torch.from_numpy(tape))
    roots_in = [mo.root() for mo in models]
    pol = torch.from_numpy(np.stack([r[1] for r in roots_in]))
    kw = dict(root_policy=pol, root_to_play=torch.from_numpy(rtp), train=train, legal=torch.from_numpy(legal),
              budget=budgets, explore=explore)
    dirichlet = np.random.default_rng(seed + 1).dirichlet([0.25] * A, B)
    if gumbel:
        eng.set_search(True, m)
        eng.root_gumbel(root_value=torch.from_numpy(np.array([r[2] for r in roots_in], f32)),
                        gumbels=torch.from_numpy(gumbels), **kw)
    else:
        eng.root(dirichlet=torch.from_numpy(dirichlet), **kw)
    W = max(A, C)
    for s in range(int(budgets.max())):
        slot, action, branch = (t.cpu().numpy() for t in eng.select(s))
        assert ((slot < 0) == (budgets <= s)).all(), f"select({s}): parent slot -1 exactly for the finished trees"
        pol, val, rew = np.zeros((B, W), f32), np.zeros(B, f32), np.zeros(B, f32)
        for b in range(B):
            if slot[b] >= 0:
                p, val[b], rew[b] = models[b].outputs(s, int(branch[b]), int(action[b]))
                pol[b, :len(p)] = p
            else:                       # ignored by smz_expand_backup
                pol[b], val[b], rew[b] = np.nan, np.nan, np.nan
        eng.expand_backup(s, pol, val, rew)
    eng.stats()
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    assert roots["error"][0] == 0 and (roots["visits"].sum(1) == budgets).all()
    gout = {k: v.cpu().numpy() for k, v in eng.read_gumbel().items()} if gumbel else None
    raw = eng.read_raw_values().cpu().numpy() if gumbel else None
    for b in range(B):
        n = int(budgets[b])
        cfg = O.SearchConfig(**dict(search, num_simulations=n))
        rng = O.TapeUniforms(tape[b])
        L = LA.legal_of(legal[b])
        model = TG.RootValueModel(seed, A, C, tree=b)
        if gumbel:
            tree = GO.search(cfg, model, rng, train=bool(explore[b]), root_to_play=int(rtp[b]) % len(cfg.cycle_map()),
                             legal=L, gumbel=GO.GumbelConfig(max_considered_actions=m), gumbels=gumbels[b],
                             kind=P_KIND[paper])
            exp_g = np.where(legal[b], gumbels[b], 0.0) if explore[b] else np.zeros(A)
            assert np.array_equal(gout["gumbels"][b], exp_g)
            assert raw[b, 0] == tree.raw_value[0]
            TG.check_readout(cfg, GO.GumbelConfig(max_considered_actions=m), tree, gout["actions"][b],
                             gout["improved_policy"][b], exp_g, A, f"G={G}[{b}]")
        else:
            tree = LA.masked_search(cfg, NP.StubModel(seed, A, C, tree=b), rng, L, train=bool(explore[b]),
                                    dirichlet=dirichlet[b] if explore[b] and n else None,
                                    root_to_play=int(rtp[b]) % len(cfg.cycle_map()), paper=paper)
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"G={G}[{b}] budget {n}")
        assert got["n_uniforms"] == rng.cursor, f"G={G}[{b}]"
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 5: exploration flags; GPU 6: statistics, flag 4
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["puct", "gumbel"])
def test_exploration_flags_equal_train_and_eval_searches_tree_for_tree(rule, monkeypatch):
    case = F.Case("explore", 6, 5, 3, 30, 200, net="fp32", shape=(5, 20, 40, 1), seed=71, players=2)
    sample = list(range(0, 200, 7))
    eng, obs, rtp, tape = make_engine(case, monkeypatch, gumbel=rule == "gumbel")
    flags = np.random.default_rng(3).random(case.n_trees) < 0.5
    on = search_once(eng, case, obs, rtp, train=True, export=sample)
    off = search_once(eng, case, obs, rtp, train=False, export=sample)
    for train in (True, False):                 # the flags override the call's `train`
        mix = search_once(eng, case, obs, rtp, train=train, explore=flags, export=sample)
        for b in sample:
            ref = on if flags[b] else off
            golden_io.assert_dump_equal(mix["trees"][b], ref["trees"][b], f"{rule}[{b}] flag {flags[b]}")
            assert np.array_equal(mix["roots"]["priors"][b], ref["roots"]["priors"][b])
            if rule == "gumbel":
                assert np.array_equal(mix["gumbel"]["gumbels"][b], ref["gumbel"]["gumbels"][b])
                assert mix["gumbel"]["actions"][b] == ref["gumbel"]["actions"][b]
    eng.close()


@pytest.mark.gpu
def test_statistics_launch_count_and_flag_4(monkeypatch):
    import torch
    case = F.Case("stats", 4, 4, 2, 20, 300, net="bf16", seed=72)
    eng, obs, rtp, _ = make_engine(case, monkeypatch, record=False)
    eng.root(obs=torch.from_numpy(obs))
    eng.simulate()
    full = eng.stats()
    budgets = mixed_budgets(case.n_trees, case.N, 9)
    eng.root(obs=torch.from_numpy(obs), budget=budgets)        # host budgets on the engine: N steps
    eng.simulate()
    st = eng.stats()
    vis = eng.read_roots()["visits"].cpu().numpy()
    assert (vis.sum(1) == budgets).all()
    dsum = st["mean_leaf_depth"] * budgets.sum()
    assert abs(dsum - round(dsum)) < 1e-6 * dsum and st["launches"] == full["launches"]
    # a device budget outside [0, N]: flag 4 at the check, that tree searched with N, the others unchanged
    bad = budgets.copy()
    bad[5], bad[6] = case.N + 1, -3
    eng.root(obs=torch.from_numpy(obs), budget=torch.from_numpy(bad).cuda())
    eng.simulate()
    with pytest.raises(ValueError, match="budget"):
        eng.stats()
    vis = eng.read_roots()["visits"].cpu().numpy()
    exp = budgets.copy()
    exp[5] = exp[6] = case.N
    assert (vis.sum(1) == exp).all()
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 2: one vision search
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vision_search_with_budgets_replays_bit_exact():
    import torch
    from stochastic_muzero_b200 import SearchEngine, VisionShape
    z = golden_io.load_vision_case("a4")
    A, S, H, L = [int(v) for v in z["dims"]]
    B, N, seed = 256, 30, 923
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=3,
                  number_of_player=2, custom_loop=None)
    eng = SearchEngine(search, A, A, max_trees=B, model_shape=VisionShape(A, S, H, L), net="vision", rng="philox",
                       seed=seed, record=True)
    eng.set_weights(z["weights"])
    budgets = mixed_budgets(B, N, seed)
    obs = torch.rand(B, 3, 98, 98, generator=torch.Generator().manual_seed(7))
    eng.root(obs=obs.reshape(B, -1), train=True, budget=budgets)
    eng.simulate(int(budgets.max()))
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    assert (eng.read_roots()["visits"].cpu().numpy().sum(1) == budgets).all()
    for b in (0, 1, 2, 3, 63, 64, 200, 255):
        n = int(budgets[b])
        cfg = O.SearchConfig(**dict(search, num_simulations=n))
        model = O.TapeModel(rec["root_policy"][b, :A], rec["sim_policy"][b, :n], np.full(n, A), rec["sim_value"][b, :n],
                            rec["sim_reward"][b, :n])
        rng = O.PhiloxUniforms(seed, b)
        tree = O.search(cfg, model, rng, train=True, dirichlet=rec["dirichlet"][b] if n else None)
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"vision[{b}] budget {n}")
        assert got["n_uniforms"] == rng.cursor
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 7: the drop-in and the drivers
# ---------------------------------------------------------------------------------------------------
class _CountingBackend:
    def __init__(self, inner):
        self.inner, self.rows, self.A = inner, 0, inner.A

    def __getattr__(self, k):
        f = getattr(self.inner, k)
        if k in ("afterstate_dynamics", "dynamics"):
            def g(h, a):
                self.rows += int(h.shape[0])
                return f(h, a)
            return g
        return f


@pytest.mark.gpu
def test_dropin_budgets_on_every_search_path():
    import torch
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import ModelShape, Monte_carlo_tree_search, PackedModel, batched_model, random_blob
    from stochastic_muzero_b200.selfplay import SelfPlay, VectorCartPole, reanalyse
    zn = golden_io.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    kw = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=11, maxium_action_sample=2, number_of_player=2,
              custom_loop=None)
    model = FakeMuzero(zn["weights"], *dims)
    budgets = [0, 1, 10, 11, 5, 3, 7, 11]
    for gumbel in (False, True):
        mcts = Monte_carlo_tree_search(**kw, seed=3, net="fp32", gumbel=gumbel)
        obs = torch.randn(8, dims[0], generator=torch.Generator().manual_seed(1))
        launches = {}
        for name, nb in (("mixed", budgets), ("all 11", 11), ("max 4", [4] * 8)):
            roots = mcts.run_batch(obs, model, num_simulations=nb)
            launches[name] = roots._engine.stats()["launches"]
            if name == "mixed":
                assert roots.visit_counts.sum(1).tolist() == budgets and roots.budgets.tolist() == budgets
        # host budgets run max(budget) simulation steps: two kernels per step
        assert launches["mixed"] == launches["all 11"] and launches["all 11"] - launches["max 4"] == 2 * (11 - 4)
        dev = mcts.run_batch(obs, model, num_simulations=torch.tensor(budgets).cuda())
        assert dev.visit_counts.sum(1).tolist() == budgets
        root = mcts.run(observation=obs[:1], model=model, num_simulations=4)
        assert root.visit_count == 4
        clone = pickle.loads(pickle.dumps(mcts))
        assert clone.run_batch(obs, model, num_simulations=3).visit_counts.sum().item() == 24

    cb_model = FakeMuzero(zn["weights"], *dims)
    cb_model.model_structure = "lstm_model"          # not fusable: host-model callback / batched back-end
    calls = {"n": 0}
    inner = cb_model.dynamics_function_inference, cb_model.afterstate_dynamics_function_inference

    def counted(f):
        def g(*a):
            calls["n"] += 1
            return f(*a)
        return g
    cb_model.dynamics_function_inference, cb_model.afterstate_dynamics_function_inference = map(counted, inner)
    mcts = Monte_carlo_tree_search(**kw, seed=5)
    root = mcts.run(observation=np.random.default_rng(4).standard_normal((1, dims[0])).astype(f32), model=cb_model,
                    num_simulations=6)
    assert root.visit_count == 6 and calls["n"] == 6
    backend = _CountingBackend(batched_model.ReferenceModuleBackend(cb_model))
    roots = Monte_carlo_tree_search(**kw, seed=6).run_batch(torch.randn(8, dims[0]), backend, num_simulations=budgets)
    assert roots.visit_counts.sum(1).tolist() == budgets and backend.rows == sum(budgets)    # finished trees not sent

    # self-play with playout caps; None keeps today's buffers; reanalyse with per-position budgets
    shape = ModelShape(4, 2, 2, 61, 126, 4)
    cart = PackedModel(random_blob(shape, 0), shape)
    for gumbel in (False, True):
        mcts = Monte_carlo_tree_search(discount=0.997, num_simulations=8, maxium_action_sample=2, net="fp32", seed=7,
                                       gumbel=gumbel)
        plain = SelfPlay(mcts, cart, VectorCartPole(64, device="cuda", seed=0), horizon=3).run()
        assert "full_search" not in plain
        seen = []
        orig = mcts.run_batch

        def spy(*a, **k):
            r = orig(*a, **k)
            seen.append(r.visit_counts.sum(1).cpu())
            return r
        mcts.run_batch = spy
        buf = SelfPlay(mcts, cart, VectorCartPole(64, device="cuda", seed=0), horizon=3, playout_cap=(0.25, 2),
                       seed=1).run()
        full = buf["full_search"].cpu()
        assert full.any() and (~full).any()
        for t in range(3):
            assert (seen[t] == torch.where(full[t], 8, 2)).all()
        del mcts.run_batch
        re = reanalyse(mcts, cart, buf["observations"], chunk=100,
                       num_simulations=torch.where(full, 8, 1).to(torch.int32))
        assert re["child_visits"].shape == (3, 64, 2)
        with pytest.raises(ValueError):
            SelfPlay(mcts, cart, VectorCartPole(4, device="cuda"), horizon=1, playout_cap=(0.5, 9))
