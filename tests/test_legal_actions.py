"""Searches whose root is restricted to the legal actions of its position (smz_root_legal in include/smz.h).

A masked root behaves exactly as the reference's root would if its action space were L, the legal actions in ascending
order: root expansion, Dirichlet noise and the root's pUCT work on the compacted vectors, and the i-th action of the
restricted space is L[i].  So the masked search is pinned by the unchanged oracles through a wrapper (`masked_search`):
its model returns policy[L] at the root and maps the action a' -> L[a'] on calls whose parent is the root, recorded
noise is compacted, and the root's child keys and the first key of each path are relabelled afterwards.

No GPU: the wrapper with the full mask replays every golden tape of the reference; masked oracle trees follow the
rules; the compacted read-out; packing and host-side validation of masks.
GPU: an all-ones mask changes nothing, bit for bit; the stand-alone tree kernels, the fused step of smz_simulate on both
tree kernels and every network mode, a vision search and the read-out replay the wrapped oracle; the drop-in's three
search paths; bad masks raise ValueError.
"""
import pickle

import numpy as np
import pytest
import torch

import golden_io
import paper_oracle as P
import test_fused_search_configurations as F
import test_node_pattern as NP
from oracle import mcts_oracle as O
from oracle import readout_oracle as R

f32 = np.float32


# ---------------------------------------------------------------------------------------------------
# the masked search, through the unchanged oracles
# ---------------------------------------------------------------------------------------------------
class _RootHidden:
    """Tags the root's hidden state, so that calls whose parent is the root can be told apart."""

    def __init__(self, h):
        self.h = h


class LegalModel:
    """The oracle's model interface seen by a root whose action space is L."""

    def __init__(self, model, legal):
        self.model, self.L = model, [int(a) for a in legal]

    def root(self):
        h, policy, v = self.model.root()
        return _RootHidden(h), np.asarray(policy, f32)[self.L], v

    def _unwrap(self, h, a):
        return (h.h, self.L[int(a)]) if isinstance(h, _RootHidden) else (h, a)

    def afterstate(self, sim, h, a):
        h, a = self._unwrap(h, a)
        return self.model.afterstate(sim, h, a)

    def dynamics(self, sim, h, c):
        h, c = self._unwrap(h, c)
        return self.model.dynamics(sim, h, c)


def masked_search(cfg, model, rng, legal, train=True, dirichlet=None, root_to_play=0, paper=False):
    """oracle/mcts_oracle.search (tests/paper_oracle.search with `paper`) of a root whose action space is `legal`
    (ascending action indices); `dirichlet` is noise over all A actions, of which the entries at L are used."""
    L = [int(a) for a in legal]
    noise = None if dirichlet is None else np.asarray(dirichlet, np.float64)[L]
    search = P.search if paper else O.search
    tree = search(cfg, LegalModel(model, L), rng, train=train, dirichlet=noise, root_to_play=root_to_play)
    for c in tree.children[0]:
        tree.key[c] = L[tree.key[c]]
    for path in tree.paths:
        if path:
            path[0] = L[path[0]]
    return tree


def legal_of(mask_row):
    return [int(a) for a in np.flatnonzero(mask_row)]


def compact_readout(visits, priors, mask_row, temperature, u):
    """readout_oracle on the legal entries of one root, scattered back: (action, policy[A], stored_policy[A])."""
    L = legal_of(mask_row)
    v, p = np.asarray(visits, np.float64)[L], np.asarray(priors, np.float64)[L]
    pol, stored = np.zeros(len(mask_row)), np.zeros(len(mask_row))
    pol[L] = R.step_policy(v, p, temperature)
    stored[L] = R.stored_policy(v, p)
    pick, _ = R.select_action(pol[L], temperature, u)
    return L[min(pick, len(L) - 1)], pol, stored


def mask_table(A, seed=0):
    """Named masks over A actions: single action, first / last only, alternating, random, all."""
    g = np.random.default_rng(seed + A)
    out = {"all": np.ones(A, bool), "first": np.eye(A, dtype=bool)[0], "last": np.eye(A, dtype=bool)[A - 1],
           "single": np.eye(A, dtype=bool)[int(g.integers(A))], "alternating": np.arange(A) % 2 == 1}
    r = g.random(A) < 0.5
    r[int(g.integers(A))] = True
    out["random"] = r
    if not out["alternating"].any():
        out["alternating"] = out["first"]
    return out


def random_masks(n, A, seed):
    """n masks with about half the actions legal, never empty; bit A - 1 (bit 31 at A = 32) often set."""
    g = np.random.default_rng(seed)
    m = g.random((n, A)) < 0.5
    m[np.arange(n), g.integers(0, A, n)] = True
    return m


# ---------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_io.tree_cases())
def test_masked_oracle_with_the_full_mask_replays_the_reference_tapes(name):
    z = golden_io.load_tree_case(name)
    c = z["config"]
    cfg = O.SearchConfig(**{k: c[k] for k in ("pb_c_base", "pb_c_init", "discount", "root_dirichlet_alpha",
                                               "root_exploration_fraction", "num_simulations",
                                               "maxium_action_sample", "number_of_player", "custom_loop")})
    A = z["root_policy"].shape[1]
    for b in range(len(z["n_nodes"])):
        rng = O.TapeUniforms(z["uniforms"][b, :z["n_uniforms"][b]])
        model = O.TapeModel(z["root_policy"][b], z["sim_policy"][b], z["sim_width"][b], z["sim_value"][b],
                            z["sim_reward"][b])
        tree = masked_search(cfg, model, rng, range(A), train=z["train"], dirichlet=z["dirichlet"][b],
                             root_to_play=int(z["exp_root_to_play"][b]))
        assert rng.cursor == z["n_uniforms"][b]
        golden_io.assert_dump_equal(tree.dump(), golden_io.expected_dump(z, b), f"{name}[{b}]")


def check_masked_tree(tree, legal, train, log=None):
    """The root has exactly L; its priors sum to 1 over L; no illegal action is ever visited or evaluated."""
    L = list(legal)
    kids = tree.children[0]
    assert [tree.key[c] for c in kids] == L
    if not train:
        assert abs(float(np.sum([f32(tree.prior[c]) for c in kids], dtype=np.float64)) - 1.0) < 1e-5
    else:
        assert abs(sum(float(tree.prior[c]) for c in kids) - 1.0) < 1e-5
    assert all(p[0] in L for p in tree.paths if p)
    assert sum(tree.visit[c] for c in kids) == len(tree.paths)
    if log is not None:       # the model saw the real action at the root's children
        firsts = [key for sim, br, h, key in log if h == ("S", 0)]
        assert firsts and all(a in L for a in firsts)


@pytest.mark.parametrize("A", [1, 2, 4, 9, 32])
@pytest.mark.parametrize("paper", [False, True])
def test_masked_oracle_trees_follow_the_rules(A, paper):
    C = 5
    for mname, row in mask_table(A).items():
        L = legal_of(row)
        for train in (False, True):
            cfg = O.SearchConfig(num_simulations=50, maxium_action_sample=3, number_of_player=2, discount=0.99)
            model = NP.StubModel(11 + A, A, C)
            noise = np.zeros(A)          # device-noise semantics: a Dirichlet over L, 0 elsewhere
            noise[L] = np.random.default_rng(A).dirichlet([0.25] * len(L))
            tree = masked_search(cfg, model, O.MTUniforms(A), L, train=train, dirichlet=noise, paper=paper)
            check_masked_tree(tree, L, train, model.log)
            if mname == "all":     # the full mask is the plain search
                plain = (P.search if paper else O.search)(cfg, NP.StubModel(11 + A, A, C), O.MTUniforms(A),
                                                          train=train, dirichlet=noise)
                golden_io.assert_dump_equal(tree.dump(), plain.dump(), f"A={A} full mask")


def test_compacted_readout():
    g = np.random.default_rng(3)
    for A in (1, 2, 5, 32):
        for row in list(mask_table(A).values()) + list(random_masks(20, A, A)):
            L = legal_of(row)
            visits = np.zeros(A, np.int32)
            visits[L] = g.integers(0, 4, len(L))
            priors = np.zeros(A)
            priors[L] = g.dirichlet([1.0] * len(L))
            for T in F.TEMPERATURES:
                u = g.random()
                act, pol, stored = compact_readout(visits, priors, row, T, u)
                assert act in L and (pol[~row] == 0).all() and (stored[~row] == 0).all()
                assert np.array_equal(pol[L], R.step_policy(visits[L], priors[L], T))
                assert np.array_equal(stored[L], R.stored_policy(visits[L], priors[L]))
                if row.all():
                    assert act == R.select_action(R.step_policy(visits, priors, T), T, u)[0]


def test_packing_a_bool_mask_gives_the_expected_words():
    from stochastic_muzero_b200.engine import pack_legal
    for A in (1, 2, 7, 31, 32):
        m = random_masks(64, A, A)
        m[0] = True
        m[1] = False
        m[1, A - 1] = True           # bit A - 1 alone: bit 31 at A = 32
        words = pack_legal(torch.from_numpy(m))
        assert words.dtype == torch.int32
        exp = [sum(1 << int(a) for a in np.flatnonzero(r)) for r in m]
        assert [int(w) & 0xFFFFFFFF for w in words] == exp
    assert int(pack_legal(torch.ones(1, 32, dtype=torch.bool))[0]) == -1


def test_host_masks_are_checked_before_any_gpu_work():
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    from stochastic_muzero_b200.engine import legal_rows
    ok = np.ones((3, 4), bool)
    assert legal_rows(ok, 3, 4).dtype == torch.bool
    assert legal_rows(ok.astype(np.int64), 3, 4).all()
    for bad in (np.ones((3, 5), bool), np.ones((2, 4), bool), np.ones(4, bool), np.ones((3, 33), bool)):
        with pytest.raises(ValueError, match="shape"):
            legal_rows(bad, 3, 4 if bad.shape[-1] != 33 else None)
    empty = ok.copy()
    empty[1] = False
    with pytest.raises(ValueError, match="no legal action"):
        legal_rows(empty, 3, 4)
    with pytest.raises(ValueError):
        legal_rows(np.full((3, 4), 2), 3, 4)
    # the drop-in checks before it builds an engine or touches the model (model=None would fail later)
    mcts = Monte_carlo_tree_search(num_simulations=4)
    with pytest.raises(ValueError, match="no legal action"):
        mcts.run_batch(np.zeros((3, 4), np.float32), None, legal_actions=empty)
    with pytest.raises(ValueError, match="shape"):
        mcts.run_batch(np.zeros((3, 4), np.float32), None, legal_actions=np.ones((2, 4), bool))
    assert mcts._engines == {}


def test_run_turns_legal_actions_into_a_mask_row():
    from stochastic_muzero_b200.monte_carlo_tree_search import _legal_row
    assert _legal_row([3, 0], 5).tolist() == [[True, False, False, True, False]]
    assert _legal_row(np.array([False, True]), 2).tolist() == [[False, True]]
    assert _legal_row(torch.tensor([31]), 32)[0, 31]
    for bad, A in (([], 4), ([4], 4), ([-1], 4), (np.ones(3, bool), 4)):
        with pytest.raises(ValueError):
            _legal_row(bad, A)


# ---------------------------------------------------------------------------------------------------
# GPU: runners
# ---------------------------------------------------------------------------------------------------
def run_masked_case(case, monkeypatch, legal=None, no_smem=False, paper=False, export=(), dirichlet=None,
                    arena=False, then=()):
    """F.run_case with a root mask (bool [n_trees, A] or None), the node pattern and optional caller noise.  `then`:
    masks of further searches on the same engine (its captured graph reused), whose results go to out["then"]."""
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
    def search(mask):
        kw = {} if mask is None else {"legal": torch.from_numpy(mask)}
        eng.root(obs=torch.from_numpy(obs), root_to_play=None if rtp is None else torch.from_numpy(rtp),
                 train=case.train, dirichlet=None if dirichlet is None else torch.from_numpy(dirichlet), **kw)
        for k in case.chunks or (case.N,):
            eng.simulate(k)
        eng.stats()
        res = {"roots": {k: v.cpu().numpy() for k, v in eng.read_roots().items()},
               "rec": {k: v.cpu().numpy() for k, v in eng.read_record().items()},
               "trees": {int(b): eng.export_tree(int(b)) for b in export}}
        if arena:
            res["arena"] = {int(b): eng.export_arena(int(b)) for b in export}
        res["readout"] = {T: {k: v.cpu().numpy() for k, v in eng.select_actions(T).items()} for T in (0.0, 0.5, 1.0)}
        return res
    out = search(legal)
    out.update(eng=eng, tape=tape, rtp=rtp, obs=obs, blob=blob)
    out["then"] = [search(m) for m in then]
    for k in F.ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    return out


def replay_masked(case, run, b, legal_row, paper=False):
    rec = run["rec"]
    width = np.where(rec["sim_branch"][b] == 1, case.A, case.C)
    model = O.TapeModel(rec["root_policy"][b, :case.A], rec["sim_policy"][b], width, rec["sim_value"][b],
                        rec["sim_reward"][b])
    rng = O.TapeUniforms(run["tape"][b]) if case.rng == "tape" else O.PhiloxUniforms(case.seed, case.offset + b)
    cfg = O.SearchConfig(**case.search())
    phase = 0 if run["rtp"] is None else int(run["rtp"][b]) % len(cfg.cycle_map())
    tree = masked_search(cfg, model, rng, legal_of(legal_row), train=case.train,
                         dirichlet=rec["dirichlet"][b] if case.N else None, root_to_play=phase, paper=paper)
    return tree, rng.cursor


def check_masked_replay(case, run, legal, what, paper=False, cache=None):
    rec = run["rec"]
    cache = {} if cache is None else cache
    for b, got in run["trees"].items():
        row = legal[b]
        key = (b, paper) + tuple(rec[k][b].tobytes() for k in ("root_policy", "sim_policy", "sim_value", "sim_reward",
                                                                "sim_branch", "dirichlet"))
        if key not in cache:
            tree, cursor = replay_masked(case, run, b, row, paper)
            cache[key] = (tree.dump(), cursor)
        exp, cursor = cache[key]
        golden_io.assert_dump_equal(got, exp, f"{what}[{b}]")
        assert got["n_uniforms"] == cursor, f"{what}[{b}]: {got['n_uniforms']} draws consumed, oracle {cursor}"
        L = legal_of(row)
        kids = np.flatnonzero(exp["depth"] == 1)
        assert exp["key"][kids].tolist() == L
        visits, priors = run["roots"]["visits"][b], run["roots"]["priors"][b]
        assert np.array_equal(visits[L], exp["visit"][kids]) and (visits[~row] == 0).all(), f"{what}[{b}]: visits"
        assert np.array_equal(priors[L], exp["prior"][kids]) and (priors[~row] == 0).all(), f"{what}[{b}]: priors"
        assert (run["roots"]["rewards"][b][~row] == 0).all()
        if case.train and case.N:
            assert (rec["dirichlet"][b][~row] == 0).all(), f"{what}[{b}]: recorded noise of illegal actions"


def check_masked_readout(eng, roots, legal, seed, offset, what):
    """select_actions(T) against the compacted read-out oracle, recorded and device (Philox stream 2) uniforms."""
    visits, priors = roots["visits"], roots["priors"]
    n = len(visits)
    u_dev = np.array([O.philox_uniform(seed, offset + b, 0, stream=2) for b in range(n)])
    g = np.random.default_rng(seed % 2 ** 32 + 2)
    for T in F.TEMPERATURES:
        u = g.random(n)
        out = {k: v.cpu().numpy() for k, v in eng.select_actions(T, uniforms=torch.from_numpy(u)).items()}
        dev = {k: v.cpu().numpy() for k, v in eng.select_actions(T).items()}
        for b in range(n):
            act, pol, stored = compact_readout(visits[b], priors[b], legal[b], T, u[b])
            e = 1.0 / T if T >= 0.3 else 1.0
            if e in (1.0, 2.0, 0.5):
                assert np.array_equal(out["policy"][b], pol), f"{what}[{b}]: acting policy at T={T}"
            else:
                np.testing.assert_allclose(out["policy"][b], pol, rtol=1e-14, atol=0, err_msg=f"{what}[{b}] T={T}")
            assert np.array_equal(out["stored_policy"][b], stored), f"{what}[{b}]: stored policy at T={T}"
            L = legal_of(legal[b])
            dev_pol = out["policy"][b]
            exp_act = L[min(R.select_action(dev_pol[L], T, u[b])[0], len(L) - 1)]
            exp_dev = L[min(R.select_action(dev_pol[L], T, u_dev[b])[0], len(L) - 1)]
            assert out["actions"][b] == exp_act, f"{what}[{b}]: T={T} action {out['actions'][b]} vs {exp_act}"
            assert dev["actions"][b] == exp_dev, f"{what}[{b}]: T={T} device-Philox action"
        assert legal[np.arange(n), out["actions"]].all() and legal[np.arange(n), dev["actions"]].all()


# ---------------------------------------------------------------------------------------------------
# GPU 1: the default is unchanged
# ---------------------------------------------------------------------------------------------------
DEFAULT_CASES = NP.FUSED_CASES


def test_default_case_table_covers_lanes_kernels_and_modes():
    fused = [c for c in DEFAULT_CASES if c.N >= 2]
    assert {c.G for c in fused if c.kernel(F.B200_SMS) == "mirror"} >= {2, 4, 8, 16, 32}
    assert {c.net for c in DEFAULT_CASES} == set(F.NETS)
    envs = {tuple(sorted(dict(c.env))) for c in DEFAULT_CASES}
    assert {("SMZ_M32", "SMZ_M64"), ("SMZ_M64", "SMZ_PIPE2")} <= envs


@pytest.mark.gpu
@pytest.mark.parametrize("paper", [False, True], ids=["reference", "paper"])
@pytest.mark.parametrize("case", DEFAULT_CASES, ids=lambda c: c.name)
def test_all_ones_mask_changes_nothing(case, paper, monkeypatch):
    """No mask, then an all-ones mask, then no mask again on one engine (the captured graph is reused): the three
    searches agree bit for bit on the arena, the draw counts, the record and the read-out."""
    sample = F.replay_sample(case)
    ones = np.ones((case.n_trees, case.A), bool)
    for no_smem in (False, True):
        run = run_masked_case(case, monkeypatch, None, no_smem, paper, sample, arena=True, then=(ones, None))
        what = f"{case.name} {'arena' if no_smem else 'default'} paper={paper}"
        for i, other in enumerate(run["then"]):
            F._assert_roots_equal(run["roots"], other["roots"], f"{what} search {i + 1}")
            for k, v in run["rec"].items():
                assert np.array_equal(v.view(np.uint8), other["rec"][k].view(np.uint8)), f"{what}: record {k}"
            for b in sample:
                for k, v in run["arena"][b].items():
                    # raw bytes: slots no search writes keep what the allocation held, which may read as NaN
                    x, y = (np.ascontiguousarray(np.atleast_1d(c)) for c in (v, other["arena"][b][k]))
                    assert x.tobytes() == y.tobytes(), \
                        f"{what}[{b}]: arena {k} differs at {np.flatnonzero(x.view(np.uint8) != y.view(np.uint8))[:8]}"
            for T, r in run["readout"].items():
                for k, v in r.items():
                    assert np.array_equal(v, other["readout"][T][k]), f"{what}: select_actions({T})['{k}']"
        run["eng"].close()


# ---------------------------------------------------------------------------------------------------
# GPU 2: the stand-alone tree kernels with tape uniforms
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("A,C,K,N,players,loop,train,G", list(NP._lane_runs()))
def test_standalone_kernels_replay_the_masked_oracle(A, C, K, N, players, loop, train, G):
    from stochastic_muzero_b200 import SearchEngine
    B, seed = 9, 2000 + A * 37 + C
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.99, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=K,
                  number_of_player=players, custom_loop=loop)
    cfg = O.SearchConfig(**search)
    n_phase = len(cfg.cycle_map())
    paper = G == 32              # both node patterns over the table
    models = [NP.StubModel(seed, A, C, tree=b) for b in range(B)]
    g = np.random.default_rng(seed)
    tape = g.random((B, 20000))
    rtp = np.arange(B, dtype=np.int32) - 4
    legal = np.concatenate([np.stack(list(mask_table(A, seed).values())), random_masks(B, A, seed)])[:B]
    dirichlet = np.full((B, A), 7.0)             # caller noise: only the entries at L may be read
    for b in range(B):
        dirichlet[b, legal[b]] = g.dirichlet([0.25] * int(legal[b].sum()))
    eng = SearchEngine(search, A, C, max_trees=B, net="external", rng="tape", lanes_per_tree=G, paper_alternation=paper)
    eng.set_uniform_tape(torch.from_numpy(tape))
    eng.root(root_policy=torch.from_numpy(np.stack([m.root_policy() for m in models])),
             root_to_play=torch.from_numpy(rtp), train=train, dirichlet=torch.from_numpy(dirichlet),
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
    for b in range(B):
        model = NP.StubModel(seed, A, C, tree=b)
        rng = O.TapeUniforms(tape[b])
        phase = int(rtp[b]) % n_phase
        L = legal_of(legal[b])
        tree = masked_search(cfg, model, rng, L, train=train, dirichlet=dirichlet[b], root_to_play=phase, paper=paper)
        check_masked_tree(tree, L, train, model.log)
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"G={G}[{b}]")
        assert got["n_uniforms"] == rng.cursor
        assert [p[-1] for p in tree.paths] == actions[b].tolist(), f"G={G}[{b}]: selected actions / sampled codes"
        assert [br for _, br, _, _ in model.log] == branches[b].tolist(), f"G={G}[{b}]: evaluation branch"
        kids = np.flatnonzero(got["depth"] == 1)
        assert np.array_equal(roots["visits"][b][L], got["visit"][kids]) and roots["visits"][b][~legal[b]].sum() == 0
    assert roots["error"][0] == 0
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 3: the fused step of smz_simulate on both tree kernels
# ---------------------------------------------------------------------------------------------------
_BY_NAME = {c.name: c for c in F.CASES}
MASKED_CASES = list(NP.FUSED_CASES) + [_BY_NAME["n1_no_fused_step"], _BY_NAME["n0_wide_readout"],
                                       _BY_NAME["a16c16k4_lanes32"], _BY_NAME["discount0"]]
CALLER_NOISE = {"a16c16k4_lanes16", "players3_custom_loop", "cfg3_a4c32k32_n100"}


def test_masked_case_table():
    names = {c.name for c in MASKED_CASES}
    assert any(c.N == 0 for c in MASKED_CASES) and any(c.N == 1 for c in MASKED_CASES)
    assert any(c.N >= 200 or c.n_trees >= 200 for c in MASKED_CASES) and any(c.chunks for c in MASKED_CASES)
    assert CALLER_NOISE <= names and any((c.A, c.C, c.K) == (4, 32, 32) for c in MASKED_CASES)


def check_depth1_network(case, run, legal):
    """fp32 / tc32: the network output of simulation 0 (a root child's leaf) is the network oracle's for the real
    action L[a'], not for the compacted index."""
    from oracle import net_oracle as NO
    if case.net not in ("fp32", "tc32") or case.N == 0:
        return
    obs, S, H, L = case.shape
    net = NO.NetOracle(run["blob"], obs, case.A, case.C, S, H, L)
    rec = run["rec"]
    for b in list(run["trees"])[:8]:
        assert rec["sim_branch"][b, 0] == 0          # the root is a decision node: the afterstate pair first
        tree, _ = replay_masked(case, run, b, legal[b])
        a = tree.paths[0][0]                         # the root child simulation 0 chose, as a real action
        assert legal[b][a]
        h0 = net.representation(run["obs"][b:b + 1])
        p, v = net.afterstate_prediction(net.afterstate_dynamics(h0, [a]))
        np.testing.assert_allclose(rec["sim_policy"][b, 0, :case.C], p[0], atol=2e-5, err_msg=f"{case.name}[{b}]")


@pytest.mark.gpu
@pytest.mark.parametrize("case", MASKED_CASES, ids=lambda c: c.name)
def test_fused_masked_search_replays_bit_exact_on_both_tree_kernels(case, monkeypatch):
    sample = F.replay_sample(case)
    legal = random_masks(case.n_trees, case.A, case.seed % 2 ** 32)
    legal[:len(mask_table(case.A))] = np.stack(list(mask_table(case.A).values()))[:case.n_trees]
    noise = None
    if case.name in CALLER_NOISE:
        noise = np.random.default_rng(case.seed % 2 ** 32).dirichlet([0.3] * case.A, case.n_trees)
    label = case.kernel(F._device_sms()) or "no fused step"
    cache = {}
    default = run_masked_case(case, monkeypatch, legal, export=sample, dirichlet=noise)
    check_masked_replay(case, default, legal, f"{case.name} default ({label}, G={case.G})", cache=cache)
    arena = run_masked_case(case, monkeypatch, legal, no_smem=True, export=sample, dirichlet=noise)
    check_masked_replay(case, arena, legal, f"{case.name} SMZ_NO_TREE_SMEM=1 (arena, G={case.G})", cache=cache)
    F._assert_roots_equal(default["roots"], arena["roots"], f"{case.name}: {label} vs arena")
    arena["eng"].close()
    assert default["roots"]["error"][0] == 0 and (default["roots"]["visits"].sum(1) == case.N).all()
    if noise is not None and case.train and case.N:
        assert np.array_equal(default["rec"]["dirichlet"][legal], noise[legal])
    check_depth1_network(case, default, legal)
    check_masked_readout(default["eng"], default["roots"], legal, case.seed, case.offset, f"{case.name} read-out")
    default["eng"].close()
    if case.name in ("a16c16k4_lanes16", "a2c2k1_n40_lanes2", "cfg3_a4c32k32_n100"):     # the paper alternation
        paper = run_masked_case(case, monkeypatch, legal, paper=True, export=sample, dirichlet=noise)
        check_masked_replay(case, paper, legal, f"{case.name} paper", paper=True)
        paper["eng"].close()


# ---------------------------------------------------------------------------------------------------
# GPU 4 / 5: vision, select_actions over many trees
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_masked_vision_search_replays_bit_exact():
    from stochastic_muzero_b200 import SearchEngine, VisionShape
    z = golden_io.load_vision_case("a4")
    A, S, H, L = [int(v) for v in z["dims"]]
    B, N, seed = 256, 40, 919
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=3,
                  number_of_player=2, custom_loop=None)
    eng = SearchEngine(search, A, A, max_trees=B, model_shape=VisionShape(A, S, H, L), net="vision", rng="philox",
                       seed=seed, record=True)
    eng.set_weights(z["weights"])
    legal = random_masks(B, A, seed)
    obs = torch.rand(B, 3, 98, 98, generator=torch.Generator().manual_seed(5))
    eng.root(obs=obs.reshape(B, -1), train=True, legal=torch.from_numpy(legal).cuda())
    eng.simulate(N)
    eng.stats()
    rec = {k: v.cpu().numpy() for k, v in eng.read_record().items()}
    cfg = O.SearchConfig(**search)
    for b in (0, 1, 63, 64, 200, 255):
        model = O.TapeModel(rec["root_policy"][b, :A], rec["sim_policy"][b], np.full(N, A), rec["sim_value"][b],
                            rec["sim_reward"][b])
        rng = O.PhiloxUniforms(seed, b)
        tree = masked_search(cfg, model, rng, legal_of(legal[b]), train=True, dirichlet=rec["dirichlet"][b])
        got = eng.export_tree(b)
        golden_io.assert_dump_equal(got, tree.dump(), f"vision[{b}]")
        assert got["n_uniforms"] == rng.cursor
    eng.close()


@pytest.mark.gpu
def test_select_actions_never_returns_an_illegal_action():
    import golden_io as G
    from stochastic_muzero_b200 import ModelShape, SearchEngine
    zn = G.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    A = dims[1]
    B, N, seed = 4096, 12, 33
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=N, maxium_action_sample=2,
                  number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, A, dims[2], max_trees=B, model_shape=ModelShape(*dims), net="fp32", rng="philox",
                       seed=seed)
    eng.set_weights(zn["weights"])
    legal = random_masks(B, A, seed)
    legal[:A] = np.eye(A, dtype=bool)
    eng.root(obs=torch.randn(B, dims[0], generator=torch.Generator().manual_seed(1)), train=True,
             legal=torch.from_numpy(legal))
    eng.simulate()
    roots = {k: v.cpu().numpy() for k, v in eng.read_roots().items()}
    assert roots["error"][0] == 0
    assert (roots["visits"][~legal] == 0).all() and (roots["priors"][~legal] == 0).all()
    for T in F.TEMPERATURES:
        for u in (None, torch.from_numpy(np.random.default_rng(int(T * 100)).random(B))):
            out = eng.select_actions(T, uniforms=u)
            act = out["actions"].cpu().numpy()
            assert legal[np.arange(B), act].all(), f"T={T}: illegal action returned"
            assert (out["policy"].cpu().numpy()[~legal] == 0).all()
            assert (out["stored_policy"].cpu().numpy()[~legal] == 0).all()
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU 6 / 7: the drop-in, bad masks
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_dropin_legal_actions_on_every_search_path():
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    zn = golden_io.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    A = dims[1]
    assert A >= 2
    kw = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=30, maxium_action_sample=2, number_of_player=2,
              custom_loop=None)
    only = [A - 1]
    mask = np.zeros(A, bool)
    mask[0] = True

    model = FakeMuzero(zn["weights"], *dims)
    mcts = Monte_carlo_tree_search(**kw, seed=3, net="fp32")
    obs = torch.randn(1, dims[0], generator=torch.Generator().manual_seed(1))
    root = mcts.run(observation=obs, model=model, train=True, legal_actions=only)
    assert sorted(int(k) for k in root.children) == only and root.visit_count == 30
    root = mcts.run(observation=obs, model=model, train=True, legal_actions=mask)
    assert sorted(int(k) for k in root.children) == [0]
    batch = np.random.default_rng(0).random((64, A)) < 0.5
    batch[:, 0] = True
    roots = mcts.run_batch(torch.randn(64, dims[0]), model, train=True, legal_actions=torch.from_numpy(batch).cuda())
    for b in (0, 7, 63):
        assert sorted(int(k) for k in roots[b].children) == legal_of(batch[b])
    acts = roots.select_actions(1.0)["actions"].cpu().numpy()
    assert batch[np.arange(64), acts].all()
    clone = pickle.loads(pickle.dumps(mcts))
    root = clone.run(observation=obs, model=model, train=False, legal_actions=only)
    assert sorted(int(k) for k in root.children) == only

    cb_model = FakeMuzero(zn["weights"], *dims)
    cb_model.model_structure = "lstm_model"          # not fusable: host-model callback per simulation
    mcts = Monte_carlo_tree_search(**kw, seed=5)
    root = mcts.run(observation=np.random.default_rng(4).standard_normal((1, dims[0])).astype(np.float32),
                    model=cb_model, train=True, legal_actions=only)
    assert sorted(int(k) for k in root.children) == only and root.visit_count == 30
    clone = pickle.loads(pickle.dumps(mcts))
    root = clone.run(observation=np.zeros((1, dims[0]), np.float32), model=cb_model, train=False, legal_actions=mask)
    assert sorted(int(k) for k in root.children) == [0]

    mcts = Monte_carlo_tree_search(**kw, seed=6)
    roots = mcts.run_batch(torch.randn(48, dims[0]), cb_model, train=True, legal_actions=batch[:48])
    assert (roots.visit_counts.sum(1) == 30).all()
    for b in (0, 5, 47):
        assert sorted(int(k) for k in roots[b].children) == legal_of(batch[b])
    assert (roots.visit_counts.cpu().numpy()[~batch[:48]] == 0).all()


@pytest.mark.gpu
def test_bad_masks_raise_and_leave_the_other_trees_unchanged(monkeypatch):
    from fake_muzero import FakeMuzero
    from stochastic_muzero_b200 import Monte_carlo_tree_search
    from stochastic_muzero_b200 import engine as E
    zn = golden_io.load_net_case("mlp450_seed0")
    dims = [int(v) for v in zn["dims"]]
    A, B = dims[1], 32
    assert A < 31
    kw = dict(num_simulations=20, maxium_action_sample=2)
    model = FakeMuzero(zn["weights"], *dims)
    obs = torch.randn(B, dims[0], generator=torch.Generator().manual_seed(8))
    plain = Monte_carlo_tree_search(**kw, seed=9, net="fp32").run_batch(obs, model, train=True)
    ref = {k: getattr(plain, k).cpu().numpy() for k in ("visit_counts", "priors", "rewards", "root_values")}
    ref_trees = {b: plain._engine.export_tree(b) for b in (0, 3, B - 1)}

    def check(roots, what):
        for k, v in ref.items():
            assert np.array_equal(getattr(roots, k).cpu().numpy().view(np.uint8), v.view(np.uint8)), f"{what}: {k}"
        for b, t in ref_trees.items():
            golden_io.assert_dump_equal(roots._engine.export_tree(b), t, f"{what}[{b}]")

    # an empty row on the device reaches the kernel
    empty = torch.ones(B, A, dtype=torch.bool, device="cuda")
    empty[3] = False
    mcts = Monte_carlo_tree_search(**kw, seed=9, net="fp32")
    with pytest.raises(ValueError, match="mask"):
        mcts.run_batch(obs, model, train=True, legal_actions=empty)
    mcts = Monte_carlo_tree_search(**kw, seed=9, net="fp32")
    roots = mcts.run_batch(obs, model, train=True, legal_actions=empty, check=False)
    with pytest.raises(ValueError, match="mask"):
        roots.raise_if_failed()
    check(roots, "empty row")
    # bit A set through the C ABI
    orig = E.pack_legal

    def with_bit_a(mask):
        w = orig(mask)
        w[0] |= 1 << A
        return w
    monkeypatch.setattr(E, "pack_legal", with_bit_a)
    mcts = Monte_carlo_tree_search(**kw, seed=9, net="fp32")
    roots = mcts.run_batch(obs, model, train=True, legal_actions=np.ones((B, A), bool), check=False)
    with pytest.raises(ValueError, match="mask"):
        roots.raise_if_failed()
    check(roots, "bit A")
    with pytest.raises(ValueError):
        roots._engine.stats()
