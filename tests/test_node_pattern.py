"""The Stochastic MuZero node alternation (`paper_alternation`, smz_set_node_pattern in include/smz.h).

With the flag on, a node at depth d is a chance node iff d & 1: the root's children are afterstates, afterstate_dynamics
receives states and dynamics receives afterstates, pUCT runs over actions and sampling over chance codes.  The rules
for leaf evaluation, to_play, rewards and the backup are those of the reference pattern; only the node kinds change.

No GPU: the paper-mode oracle on seeded stub models, and the player tables of the binding.
GPU: the stand-alone tree kernels (smz_select / smz_expand_backup) at every lane width, the fused tree step of
smz_simulate on both tree kernels and every network mode, a vision search, the drop-in's three search paths and
switching the pattern on one engine — each replayed bit for bit by the paper-mode oracle.
"""
import pickle

import numpy as np
import pytest

import golden_io
import paper_oracle as P
import test_fused_search_configurations as F
from oracle import mcts_oracle as O

f32 = np.float32


# ---------------------------------------------------------------------------------------------------
# a seeded stub model: outputs depend on (tree, sim, branch, key) only, so any visiting order fits it
# ---------------------------------------------------------------------------------------------------
class StubModel:
    """Network outputs of the oracle's model interface.  Hidden states are tags (kind, depth): "S" for a state (the
    root and every dynamics output), "A" for an afterstate, so the call log shows what each function was fed."""

    def __init__(self, seed, A, C, tree=0):
        self.seed, self.A, self.C, self.tree = seed, A, C, tree
        self.log = []          # (sim, branch, parent hidden tag, key)

    def outputs(self, sim, branch, key):
        g = np.random.default_rng([self.seed, self.tree, sim, branch, int(key)])
        w = self.A if branch else self.C
        p = (g.random(w) ** 4 + 1e-3).astype(f32)
        p = (p / p.sum(dtype=f32)).astype(f32)
        return p, f32(g.normal()), (f32(g.normal()) if branch else f32(0))

    def root_policy(self):
        g = np.random.default_rng([self.seed, self.tree, 1 << 30])
        p = (g.random(self.A) + 0.05).astype(f32)
        return (p / p.sum(dtype=f32)).astype(f32)

    def root(self):
        return ("S", 0), self.root_policy(), f32(0)

    def afterstate(self, sim, h, a):
        self.log.append((sim, 0, h, int(a)))
        p, v, _ = self.outputs(sim, 0, a)
        return ("A", h[1] + 1), p, v

    def dynamics(self, sim, h, c):
        self.log.append((sim, 1, h, int(c)))
        p, v, r = self.outputs(sim, 1, c)
        return ("S", h[1] + 1), p, v, r


def _parents(tree):
    par = [-1] * len(tree.visit)
    for n, kids in enumerate(tree.children):
        for c in kids:
            par[c] = n
    return par


def check_paper_tree(cfg, tree, log, A, C, root_to_play=0):
    """Every rule of the paper alternation on one oracle tree and its model call log."""
    K, cyc = cfg.maxium_action_sample, cfg.cycle_map()
    par = _parents(tree)
    for n in range(len(tree.visit)):
        d, kids = tree.depth[n], tree.children[n]
        assert tree.is_chance[n] == bool(d & 1), f"node {n} at depth {d}"
        keys = [tree.key[c] for c in kids]
        assert keys == sorted(keys) and len(set(keys)) == len(keys)
        if n == 0:
            assert keys == list(range(A)) and tree.to_play[0] == root_to_play
            continue
        if kids:     # a chance node was expanded by the afterstate pair (C-wide), a decision node by dynamics (A-wide)
            width = C if tree.is_chance[n] else A
            assert len(kids) == min(K, width) and max(keys) < width, f"node {n}: children {keys}"
        p = par[n]
        expect = tree.to_play[p] if tree.is_chance[n] else (tree.to_play[p] + 1) % len(cyc)
        assert tree.to_play[n] == expect, f"node {n}: to_play {tree.to_play[n]}, rule gives {expect}"
        dyn_evaluated = bool(kids) and tree.is_chance[p]
        if not dyn_evaluated:
            assert tree.reward[n] == 0, f"node {n}: reward on a node the dynamics pair did not evaluate"
        else:
            assert d % 2 == 0 and d >= 2
    # afterstate_dynamics receives states (under decision parents, even depth), dynamics receives afterstates
    assert len(log) == cfg.num_simulations
    for sim, branch, h, key in log:
        if branch == 0:
            assert h[0] == "S" and h[1] % 2 == 0 and key < A, (sim, branch, h, key)
        else:
            assert h[0] == "A" and h[1] % 2 == 1 and key < C, (sim, branch, h, key)
    assert sum(tree.visit[c] for c in tree.children[0]) == cfg.num_simulations


# (A, C, K): A != C including BASELINE cfg3's A4 / C32 / K32, K above, equal to and below the widths
SHAPES = [(4, 32, 32), (4, 32, 3), (3, 5, 2), (5, 3, 7), (2, 2, 2), (6, 4, 4), (4, 6, 1), (32, 4, 4), (1, 1, 1)]
PLAYERS = [(1, None), (2, None), (3, None), (1, "1>2>1>3")]


@pytest.mark.parametrize("A,C,K", SHAPES)
@pytest.mark.parametrize("players,loop", PLAYERS)
def test_paper_oracle_follows_the_rules(A, C, K, players, loop):
    cfg = O.SearchConfig(num_simulations=60, maxium_action_sample=K, number_of_player=players, custom_loop=loop,
                         discount=0.99)
    n_phase = len(cfg.cycle_map())
    for phase in range(n_phase):
        for train in (True, False):
            model = StubModel(7 + A * 100 + C, A, C, tree=phase)
            g = np.random.default_rng(phase)
            tree = P.search(cfg, model, O.MTUniforms(phase + 3), train=train, dirichlet=g.dirichlet([0.25] * A),
                            root_to_play=phase)
            check_paper_tree(cfg, tree, model.log, A, C, root_to_play=phase)


@pytest.mark.parametrize("name", golden_io.tree_cases())
def test_paper_oracle_with_the_reference_kinds_replays_the_reference_tapes(name):
    """The restatement in paper_oracle.py differs from oracle/mcts_oracle.search only by its kind function: with the
    reference's F,F,T,T,... it must replay every golden tape of the reference bit for bit."""
    z = golden_io.load_tree_case(name)
    c = z["config"]
    cfg = O.SearchConfig(**{k: c[k] for k in ("pb_c_base", "pb_c_init", "discount", "root_dirichlet_alpha",
                                               "root_exploration_fraction", "num_simulations",
                                               "maxium_action_sample", "number_of_player", "custom_loop")})
    for b in range(len(z["n_nodes"])):
        rng = O.TapeUniforms(z["uniforms"][b, :z["n_uniforms"][b]])
        model = O.TapeModel(z["root_policy"][b], z["sim_policy"][b], z["sim_width"][b], z["sim_value"][b],
                            z["sim_reward"][b])
        tree = P.search(cfg, model, rng, train=z["train"], dirichlet=z["dirichlet"][b],
                        root_to_play=int(z["exp_root_to_play"][b]), kind=P.reference_is_chance)
        assert rng.cursor == z["n_uniforms"][b]
        golden_io.assert_dump_equal(tree.dump(), golden_io.expected_dump(z, b), f"{name}[{b}]")


def test_paper_and_reference_oracles_differ_only_where_the_pattern_does():
    """On the same stub: mcts_oracle gives the reference pattern, paper_oracle the alternation, and with the reference
    kinds paper_oracle gives mcts_oracle's tree."""
    cfg = O.SearchConfig(num_simulations=30, maxium_action_sample=3, number_of_player=2)
    same = P.search(cfg, StubModel(5, 3, 5), O.MTUniforms(1), train=False, kind=P.reference_is_chance)
    golden_io.assert_dump_equal(same.dump(), O.search(cfg, StubModel(5, 3, 5), O.MTUniforms(1), train=False).dump())
    for paper in (False, True):
        model = StubModel(5, 3, 5)
        tree = (P.search if paper else O.search)(cfg, model, O.MTUniforms(1), train=False)
        for n in range(len(tree.visit)):
            d = tree.depth[n]
            assert tree.is_chance[n] == bool((d & 1) if paper else ((d >> 1) & 1))
        kids = tree.children[0]
        assert all(tree.to_play[c] == (0 if paper else 1) for c in kids)


@pytest.mark.parametrize("players,loop", PLAYERS)
def test_player_tables_follow_the_paper_oracle(players, loop):
    from stochastic_muzero_b200.engine import _is_chance, player_tables
    N = 24
    sign, to_play = player_tables(players, loop, N + 2, True)
    cfg = O.SearchConfig(num_simulations=N, maxium_action_sample=2, number_of_player=players, custom_loop=loop,
                         discount=0.99)
    cyc = cfg.cycle_map()
    depths = set()
    for phase in range(len(cyc)):
        tree = P.search(cfg, StubModel(phase, 3, 2), O.MTUniforms(phase), train=False, root_to_play=phase)
        for n in range(len(tree.visit)):
            d = tree.depth[n]
            depths.add(d)
            assert tree.to_play[n] == to_play[phase, d]
            assert tree.is_chance[n] == _is_chance(d, True)
            same = cyc[tree.to_play[0] % len(cyc)] == cyc[tree.to_play[n] % len(cyc)]
            assert sign[phase, d] == (1 if same else -1)
    assert max(depths) >= 4
    # the default stays the reference pattern
    ref = player_tables(players, loop, N + 2)
    assert all(np.array_equal(x, y) for x, y in zip(ref, player_tables(players, loop, N + 2, False)))


def test_node_view_takes_rewards_from_the_parent_kind():
    """The drop-in's Node view reads each node's reward by its parent's kind in the dump, in either pattern."""
    from stochastic_muzero_b200.monte_carlo_tree_search import _node_tree
    for paper in (False, True):
        cfg = O.SearchConfig(num_simulations=40, maxium_action_sample=2, number_of_player=2)
        tree = (P.search if paper else O.search)(cfg, StubModel(3, 3, 4), O.MTUniforms(2), train=False)
        dump = tree.dump()
        got = node_dump(_node_tree(dump), dump["minmax"])
        golden_io.assert_dump_equal(got, dump, f"paper={paper}")
        assert (dump["reward"] != 0).any()


def node_dump(root, minmax):
    """A Node tree in the oracle's canonical dump order (depth-first, children by ascending key)."""
    rows, stack = [], [(root, 0, -1)]
    while stack:
        n, d, k = stack.pop()
        rows.append((d, k, n.visit_count, n.value_sum, n.reward, n.prior, n.is_chance, n.to_play, n.expanded()))
        stack.extend((n.children[c], d + 1, int(c)) for c in sorted(n.children, reverse=True))
    dtypes = (np.int32, np.int32, np.int32, np.float32, np.float32, np.float64, np.int8, np.int32, np.int8)
    out = {k: np.array([r[i] for r in rows], dtype=dt) for i, (k, dt) in enumerate(zip(golden_io.DUMP_KEYS, dtypes))}
    out["minmax"] = np.asarray(minmax, np.float32)
    return out


# ---------------------------------------------------------------------------------------------------
# the fused case table (the Case / runner helpers of test_fused_search_configurations)
# ---------------------------------------------------------------------------------------------------
_BY_NAME = {c.name: c for c in F.CASES}
FUSED_CASES = [_BY_NAME[n] for n in (
    "a32c32k3_peaky", "a16c16k4_lanes16", "a8c8k2_lanes8", "discount1_large_values", "a2c2k1_n40_lanes2",
    "a2c32k32_n32_arena_by_size", "a17c5k3_lanes32", "chain_n100", "k_above_both_widths", "players3_custom_loop",
    "players2_modular", "eval_mode", "simulate_in_two_chunks", "blocks_per_sm_at_limit", "blocks_per_sm_above_limit")]
FUSED_CASES += [c for c in F.CHAIN_CASES]
# BASELINE cfg3's search shape: 4 actions, 32 tile codes, K = 32
FUSED_CASES += [F.Case("cfg3_a4c32k32_n100", 4, 32, 32, 100, 200, net="bf16", shape=(16, 61, 126, 4), seed=60),
                F.Case("cfg3_a4c32k32_n100_tc32", 4, 32, 32, 100, 64, net="tc32", shape=(16, 61, 126, 4), seed=61,
                       rng="tape")]


def test_paper_case_table_reaches_both_tree_kernels():
    fused = [c for c in FUSED_CASES if c.N >= 2]
    assert {c.G for c in fused if c.kernel(F.B200_SMS) == "mirror"} >= {2, 4, 8, 16, 32}
    assert any(c.kernel(F.B200_SMS) == "arena" for c in fused)
    assert {c.net for c in fused} == set(F.NETS) and {c.rng for c in fused} == {"tape", "philox"}
    assert any(c.loop for c in fused) and any(c.players == 2 for c in fused) and any(not c.train for c in fused)
    assert any(c.chunks for c in fused) and any((c.A, c.C, c.K) == (4, 32, 32) for c in fused)
    assert {dict(c.env).get("SMZ_NO_PDL") for c in fused} >= {None, "1"}


def run_paper_case(case, monkeypatch, no_smem=False, export=()):
    """F.run_case with the engine built for the paper alternation."""
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
                       lanes_per_tree=case.lanes, record=True, paper_alternation=True)
    eng.set_weights(blob)
    if tape is not None:
        eng.set_uniform_tape(torch.from_numpy(tape))
    eng.root(obs=torch.from_numpy(obs), root_to_play=None if rtp is None else torch.from_numpy(rtp), train=case.train)
    for k in case.chunks or (case.N,):
        eng.simulate(k)
    eng.stats()
    out = {"roots": {k: v.cpu().numpy() for k, v in eng.read_roots().items()},
           "rec": {k: v.cpu().numpy() for k, v in eng.read_record().items()},
           "trees": {int(b): eng.export_tree(int(b)) for b in export}, "eng": eng, "tape": tape, "rtp": rtp}
    for k in F.ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    return out


def replay(A, C, search, rec, b, rng, train, root_to_play=0):
    """The paper-mode oracle on the engine's own record of tree b."""
    width = np.where(rec["sim_branch"][b] == 1, A, C)
    model = O.TapeModel(rec["root_policy"][b, :A], rec["sim_policy"][b], width, rec["sim_value"][b],
                        rec["sim_reward"][b])
    cfg = O.SearchConfig(**search)
    noise = rec["dirichlet"][b] if train and cfg.num_simulations else None
    tree = P.search(cfg, model, rng, train=train, dirichlet=noise, root_to_play=root_to_play)
    return tree.dump(), rng.cursor


def check_paper_replay(case, run, what, cache):
    rec = run["rec"]
    for b, got in run["trees"].items():
        key = (b,) + tuple(rec[k][b].tobytes() for k in ("root_policy", "sim_policy", "sim_value", "sim_reward",
                                                         "sim_branch", "dirichlet"))
        if key not in cache:
            rng = O.TapeUniforms(run["tape"][b]) if case.rng == "tape" else O.PhiloxUniforms(case.seed, case.offset + b)
            phase = 0 if run["rtp"] is None else int(run["rtp"][b]) % len(O.SearchConfig(**case.search()).cycle_map())
            cache[key] = replay(case.A, case.C, case.search(), rec, b, rng, case.train, phase)
        exp, cursor = cache[key]
        golden_io.assert_dump_equal(got, exp, f"{what}[{b}]")
        assert got["n_uniforms"] == cursor, f"{what}[{b}]: {got['n_uniforms']} draws consumed, oracle {cursor}"
        assert np.array_equal(got["is_chance"], got["depth"] & 1)
        kids = np.flatnonzero(exp["depth"] == 1)
        assert np.array_equal(run["roots"]["visits"][b], exp["visit"][kids]), f"{what}[{b}]: root visits"
        assert np.array_equal(run["roots"]["priors"][b], exp["prior"][kids]), f"{what}[{b}]: root priors"
    if case.N:
        assert (rec["sim_branch"][:, 0] == 0).all()      # the root is a decision node: the afterstate pair first


@pytest.mark.gpu
@pytest.mark.parametrize("case", FUSED_CASES, ids=lambda c: c.name)
def test_fused_paper_search_replays_bit_exact_on_both_tree_kernels(case, monkeypatch):
    sample = F.replay_sample(case)
    label = case.kernel(F._device_sms()) or "no fused step"
    cache = {}
    default = run_paper_case(case, monkeypatch, export=sample)
    check_paper_replay(case, default, f"{case.name} default ({label}, G={case.G})", cache)
    arena = run_paper_case(case, monkeypatch, no_smem=True, export=sample)
    check_paper_replay(case, arena, f"{case.name} SMZ_NO_TREE_SMEM=1 (arena, G={case.G})", cache)
    F._assert_roots_equal(default["roots"], arena["roots"], f"{case.name}: {label} vs arena")
    arena["eng"].close()
    assert default["roots"]["error"][0] == 0 and (default["roots"]["visits"].sum(1) == case.N).all()
    F.check_readout(case, default, f"{case.name} read-out")
    default["eng"].close()


# ---------------------------------------------------------------------------------------------------
# GPU: the stand-alone tree kernels with tape uniforms and the stub model as external network
# ---------------------------------------------------------------------------------------------------
STANDALONE = [  # A, C, K, N, players, loop, train
    (2, 2, 2, 40, 1, None, True), (3, 4, 2, 50, 2, None, True), (4, 6, 3, 50, 3, None, False),
    (5, 3, 7, 40, 1, "1>2>1>3", True), (16, 9, 4, 40, 2, None, True), (4, 32, 32, 40, 1, None, True),
    (4, 32, 3, 50, 2, None, False), (32, 4, 4, 30, 1, None, True)]


def _lane_runs():
    for A, C, K, N, players, loop, train in STANDALONE:
        need = max(2, 1 << (max(A, C) - 1).bit_length())
        for G in (2, 4, 8, 16, 32):
            if G >= need:
                yield pytest.param(A, C, K, N, players, loop, train, G, id=f"a{A}c{C}k{K}_p{players}_G{G}")


@pytest.mark.gpu
@pytest.mark.parametrize("A,C,K,N,players,loop,train,G", list(_lane_runs()))
def test_standalone_kernels_replay_the_paper_oracle(A, C, K, N, players, loop, train, G):
    import torch
    from stochastic_muzero_b200 import SearchEngine
    B, seed = 9, 1000 + A * 37 + C
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.99, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=K,
                  number_of_player=players, custom_loop=loop)
    cfg = O.SearchConfig(**search)
    n_phase = len(cfg.cycle_map())
    models = [StubModel(seed, A, C, tree=b) for b in range(B)]
    g = np.random.default_rng(seed)
    tape = g.random((B, 20000))
    dirichlet = g.dirichlet([0.25] * A, B)
    rtp = np.arange(B, dtype=np.int32) - 4
    eng = SearchEngine(search, A, C, max_trees=B, net="external", rng="tape", lanes_per_tree=G, paper_alternation=True)
    eng.set_uniform_tape(torch.from_numpy(tape))
    eng.root(root_policy=torch.from_numpy(np.stack([m.root_policy() for m in models])),
             root_to_play=torch.from_numpy(rtp), train=train, dirichlet=torch.from_numpy(dirichlet))
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
    for b in range(B):
        model = StubModel(seed, A, C, tree=b)
        rng = O.TapeUniforms(tape[b])
        phase = int(rtp[b]) % n_phase
        tree = P.search(cfg, model, rng, train=train, dirichlet=dirichlet[b], root_to_play=phase)
        check_paper_tree(cfg, tree, model.log, A, C, root_to_play=phase)
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"G={G}[{b}]")
        assert got["n_uniforms"] == rng.cursor
        assert [p[-1] for p in tree.paths] == actions[b].tolist(), f"G={G}[{b}]: selected actions / sampled codes"
        assert [br for _, br, _, _ in model.log] == branches[b].tolist(), f"G={G}[{b}]: evaluation branch"
        kids = np.flatnonzero(got["depth"] == 1)
        assert np.array_equal(roots["visits"][b], got["visit"][kids])
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU: vision family, switching, the drop-in
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vision_paper_search_replays_bit_exact():
    import torch
    from stochastic_muzero_b200 import SearchEngine, VisionShape
    z = golden_io.load_vision_case("a4")
    A, S, H, L = [int(v) for v in z["dims"]]
    B, N, seed = 256, 40, 909
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=3,
                  number_of_player=2, custom_loop=None)
    eng = SearchEngine(search, A, A, max_trees=B, model_shape=VisionShape(A, S, H, L), net="vision", rng="philox",
                       seed=seed, record=True, paper_alternation=True)
    eng.set_weights(z["weights"])
    obs = torch.rand(B, 3, 98, 98, generator=torch.Generator().manual_seed(5))
    eng.root(obs=obs.reshape(B, -1), train=True)
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    for b in (0, 1, 63, 64, 200, 255):
        exp, cursor = replay(A, A, search, rec, b, O.PhiloxUniforms(seed, b), True)
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, exp, f"vision[{b}]")
        assert got["n_uniforms"] == cursor
    assert (rec["sim_branch"][:, 0] == 0).all() and (rec["sim_branch"][:, 1:] == 1).any()
    eng.close()


def _mlp_search_engine(paper, players=2, seed=77, B=128, N=30, net="fp32", **kw):
    from stochastic_muzero_b200 import ModelShape, SearchEngine
    zn = golden_io.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=2,
                  number_of_player=players, custom_loop=None)
    eng = SearchEngine(search, dims[1], dims[2], max_trees=B, model_shape=ModelShape(*dims), net=net, rng="philox",
                       seed=seed, paper_alternation=paper, **kw)
    eng.set_weights(zn["weights"])
    return eng


def _search(eng, obs, rtp):
    import torch
    eng.set_seed(77)
    eng.root(obs=obs, root_to_play=torch.from_numpy(rtp), train=True)
    eng.simulate()
    eng.stats()
    return {k: v.cpu().numpy() for k, v in eng.read_roots().items()}, [eng.export_tree(b) for b in range(len(rtp))]


@pytest.mark.gpu
def test_switching_the_pattern_drops_the_captured_graph():
    """A paper search then a reference search on one engine: the second equals a fresh reference engine's search bit
    for bit.  A pattern set after smz_root leaves the search already rooted as it is."""
    import torch
    from stochastic_muzero_b200 import _lib
    B = 128
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(9))
    rtp = (np.arange(B, dtype=np.int32) % 3) - 1
    fresh = _mlp_search_engine(False, B=B)
    ref_roots, ref_trees = _search(fresh, obs, rtp)
    fresh.close()

    eng = _mlp_search_engine(True, B=B, record=True)
    paper_roots, paper_trees = _search(eng, obs, rtp)
    assert all(np.array_equal(t["is_chance"], t["depth"] & 1) for t in paper_trees)
    assert not all(np.array_equal(a["visit"], b["visit"]) and np.array_equal(a["is_chance"], b["is_chance"])
                   for a, b in zip(paper_trees, ref_trees))
    eng.set_node_pattern(False)
    roots, trees = _search(eng, obs, rtp)
    F._assert_roots_equal(roots, ref_roots, "reference search after a paper search")
    for b in range(B):
        golden_io.assert_dump_equal(trees[b], ref_trees[b], f"switched[{b}]")
        assert trees[b]["n_uniforms"] == ref_trees[b]["n_uniforms"]
    # back to paper: equal to the first paper search
    eng.set_node_pattern(True)
    roots, trees = _search(eng, obs, rtp)
    F._assert_roots_equal(roots, paper_roots, "paper search again")
    # the C setting applies from the next smz_root: a search already rooted keeps its pattern
    eng.set_seed(77)
    eng.root(obs=obs, root_to_play=torch.from_numpy(rtp), train=True)
    assert eng.lib.smz_set_node_pattern(eng._h, _lib.PATTERN_REFERENCE) == 0
    eng.simulate()
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    for b in (0, 1, 2, B - 1):
        golden_io.assert_dump_equal(eng.export_tree(b), paper_trees[b], f"rooted before the switch[{b}]")
        exp, _ = replay(2, 2, dict(eng.search, maxium_action_sample=2), rec, b, O.PhiloxUniforms(77, b), True,
                        int(rtp[b]) % 2)
        golden_io.assert_dump_equal(eng.export_tree(b), exp, f"paper oracle[{b}]")
    for bad in (-1, 2, 7):
        with pytest.raises(ValueError):
            eng._check(eng.lib.smz_set_node_pattern(eng._h, bad))
    eng.close()


class _Capture:
    """Records what a search path hands the engine (seed, root policy, branch and network outputs per simulation), so
    that the oracle can replay the same inputs."""

    def __init__(self, monkeypatch):
        from stochastic_muzero_b200 import engine as E
        self.sims, self.branch = {}, {}
        orig = {n: getattr(E.SearchEngine, n) for n in ("set_seed", "root", "select", "expand_backup")}
        cap = self

        def set_seed(self, seed, tree_id_offset=0):
            cap.seed, cap.offset = int(seed) & 0xFFFFFFFFFFFFFFFF, int(tree_id_offset)
            return orig["set_seed"](self, seed, tree_id_offset)

        def root(self, obs=None, root_policy=None, root_to_play=None, train=True, dirichlet=None):
            cap.root_policy = np.asarray(root_policy.detach().cpu() if hasattr(root_policy, "detach") else root_policy,
                                         np.float32).copy()
            cap.sims.clear()
            cap.branch.clear()
            return orig["root"](self, obs, root_policy, root_to_play, train, dirichlet)

        def select(self, sim):
            out = orig["select"](self, sim)
            cap.branch[sim] = out[2].cpu().numpy().copy()
            return out

        def expand_backup(self, sim, policy=None, value=None, reward=None):
            host = [np.asarray(x.detach().cpu() if hasattr(x, "detach") else x, np.float32).copy()
                    for x in (policy, value, reward)]
            cap.sims[sim] = host
            return orig["expand_backup"](self, sim, policy, value, reward)

        for n, fn in (("set_seed", set_seed), ("root", root), ("select", select), ("expand_backup", expand_backup)):
            monkeypatch.setattr(E.SearchEngine, n, fn)

    def oracle(self, A, C, search, b):
        N = len(self.sims)
        W = max(A, C)
        pol = np.zeros((N, W), np.float32)
        for s in range(N):
            p = self.sims[s][0][b]
            pol[s, :len(p)] = p
        rec = {"root_policy": self.root_policy[b:b + 1], "sim_policy": pol[None],
               "sim_value": np.array([[self.sims[s][1][b] for s in range(N)]], np.float32),
               "sim_reward": np.array([[self.sims[s][2][b] for s in range(N)]], np.float32),
               "sim_branch": np.array([[self.branch[s][b] for s in range(N)]]), "dirichlet": None}
        return replay(A, C, search, rec, 0, O.PhiloxUniforms(self.seed, self.offset + b), False)


def _check_node_tree(root, n_players):
    """is_chance / reward / to_play of a Node tree by the paper rules."""
    stack = [(root, 0, None)]
    seen_reward = False
    while stack:
        n, d, parent = stack.pop()
        assert n.is_chance == bool(d & 1)
        if parent is not None:
            expect = parent.to_play if n.is_chance else (parent.to_play + 1) % n_players
            assert n.to_play == expect
            if not (parent.is_chance and n.expanded()):
                assert n.reward == 0
            else:
                assert d % 2 == 0 and isinstance(n.reward, np.float32)
                seen_reward |= n.reward != 0
        stack.extend((c, d + 1, n) for c in n.children.values())
    return seen_reward


@pytest.mark.gpu
def test_dropin_paper_alternation_on_every_search_path(monkeypatch):
    import torch
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    zn = golden_io.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    A = dims[1]
    kw = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=40, maxium_action_sample=2, number_of_player=2,
              custom_loop=None)
    search = dict(kw)

    # fused run / run_batch
    model = FakeMuzero(zn["weights"], *dims)
    mcts = Monte_carlo_tree_search(**kw, seed=3, net="fp32", paper_alternation=True)
    root = mcts.run(observation=torch.randn(1, 4, generator=torch.Generator().manual_seed(1)), model=model, train=True)
    assert root.visit_count == 40 and all(c.is_chance for c in root.children.values())
    assert _check_node_tree(root, 2)
    eng = next(iter(mcts._engines.values()))
    assert eng.paper_alternation is True
    roots = mcts.run_batch(torch.randn(64, 4, generator=torch.Generator().manual_seed(2)), model, train=True)
    assert (roots.visit_counts.sum(1) == 40).all()
    pick = roots.select_actions(1.0)
    acts = pick["actions"].cpu().numpy()
    assert ((acts >= 0) & (acts < A)).all() and np.allclose(pick["stored_policy"].sum(1).cpu().numpy(), 1.0)
    assert _check_node_tree(roots[7], 2)

    # pickled copies and from_config keep the flag
    clone = pickle.loads(pickle.dumps(mcts))
    assert clone._paper is True and clone._engines == {}
    clone_roots = clone.run_batch(torch.randn(8, 4), model, train=False)
    assert next(iter(clone._engines.values())).paper_alternation is True
    assert _check_node_tree(clone_roots[0], 2) is not None
    assert Monte_carlo_tree_search.from_config({"monte_carlo_tree_search": search}, paper_alternation=True)._paper
    assert Monte_carlo_tree_search(**kw)._paper is False

    # host-model callback path
    cb_model = FakeMuzero(zn["weights"], *dims)
    cb_model.model_structure = "lstm_model"          # not fusable: the tree kernels call the model back per simulation
    cap = _Capture(monkeypatch)
    mcts = Monte_carlo_tree_search(**kw, seed=5, paper_alternation=True)
    root = mcts.run(observation=np.random.default_rng(4).standard_normal((1, 4)).astype(np.float32), model=cb_model,
                    train=False)
    exp, cursor = cap.oracle(A, A, search, 0)
    golden_io.assert_dump_equal(node_dump(root, [mcts.min_max_stats.minimum, mcts.min_max_stats.maximum]), exp,
                                "callback run")
    eng = next(iter(mcts._engines.values()))
    golden_io.assert_dump_equal(eng.export_tree(0), exp, "callback arena")
    assert eng.export_tree(0)["n_uniforms"] == cursor
    assert _check_node_tree(root, 2)

    # run_batch through ReferenceModuleBackend (torch modules of the reference-shaped model)
    mcts = Monte_carlo_tree_search(**kw, seed=6, paper_alternation=True)
    obs = torch.randn(48, 4, generator=torch.Generator().manual_seed(3))
    roots = mcts.run_batch(obs, cb_model, train=False)
    assert (roots.visit_counts.sum(1) == 40).all()
    eng = roots._engine
    for b in (0, 5, 47):
        exp, cursor = cap.oracle(A, A, search, b)
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, exp, f"ReferenceModuleBackend[{b}]")
        assert got["n_uniforms"] == cursor
        golden_io.assert_dump_equal(node_dump(roots[b], got["minmax"]), exp, f"ReferenceModuleBackend Node[{b}]")
