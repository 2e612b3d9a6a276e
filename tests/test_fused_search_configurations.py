"""The fused tree step of smz_simulate, replayed bit for bit by the search oracle across search configurations.

Every production search (`run` / `run_batch` with an MLP model) runs its tree step through one of two kernels, chosen
by smz_launch_backup_select (csrc/smz_tree.cu): k_backup_select_sm<G>, which mirrors the node records, root priors,
tables and a window of Philox draws in shared memory, or the arena-only k_backup_select<G>.  Each case below runs a
whole search through smz_simulate twice, under the default choice and with SMZ_NO_TREE_SMEM=1, and replays the
engine's own record of network outputs through oracle/mcts_oracle.search with the same uniforms: every node statistic
must match bit for bit.  The device read-out (k_select_actions) of the final trees is checked against
oracle/readout_oracle, with recorded uniforms and with the engine's own Philox draw.

The case table is built to reach the mirror kernel at every lane width, the arena-only kernel by size and by batch,
Philox windows that run out within one step, and the behaviour only the fused path has (player phases, evaluation
mode, K against the head widths, chain trees, discount edges, chunked `simulate`, programmatic dependent launch off).
`test_case_table_reaches_both_tree_kernels` (no GPU) checks that it still does.
"""
import dataclasses
import math
import os
import re
from typing import Optional, Tuple

import numpy as np
import pytest

import golden_io
from oracle import mcts_oracle as O
from oracle import readout_oracle as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TREE_CU = os.path.join(ROOT, "stochastic-muzero_b200", "csrc", "smz_tree.cu")
B200_SMS = 148

# ---------------------------------------------------------------------------------------------------
# which tree kernel runs: restates csrc/smz_tree.cu (smz_mirror_bytes, rcp_entries, smz_tree_mirror_fits,
# mirror_pays, smz_launch_backup_select) and the default lane count of smz_create (csrc/smz_api.cu)
# ---------------------------------------------------------------------------------------------------
K_THREADS = 128            # kThreads: threads per tree-kernel block
UWIN = 32                  # SMZ_UWIN: Philox draws generated ahead per tree by the mirror prologue
MAX_POLICY = 32            # SMZ_MAX_POLICY
MIRROR_LIMIT = 96 * 1024   # smz_tree_mirror_fits: dynamic shared memory of the mirror kernel
MIRROR_BLOCKS_PER_SM = 2   # mirror_pays: at most this many blocks per SM


def default_lanes(A, C):
    need = max(2, 1 << (max(A, C) - 1).bit_length())
    return max(need, 4)


def mirror_bytes(G, A, C, K, N):
    tpb = K_THREADS // G
    M = 1 + A + N * max(min(K, A), min(K, C))
    n_tab = max(N + 3, MAX_POLICY + 1)
    n_pbc = N + 2
    return tpb * M * (16 + 8) + tpb * (A + UWIN) * 8 + (n_pbc + n_tab) * 8 + n_tab * 4 + 16


def tree_kernel(G, A, C, K, N, n_trees, sms, no_smem=False):
    """'mirror' / 'arena' for the fused tree step; None when the search has no fused step (N < 2)."""
    if N < 2:
        return None
    blocks = (n_trees * G + K_THREADS - 1) // K_THREADS
    fits = not no_smem and mirror_bytes(G, A, C, K, N) <= MIRROR_LIMIT
    return "mirror" if fits and blocks <= MIRROR_BLOCKS_PER_SM * sms else "arena"


# ---------------------------------------------------------------------------------------------------
# the case table
# ---------------------------------------------------------------------------------------------------
NETS = ("fp32", "tc32", "f16", "bf16")
ENV_KEYS = ("SMZ_NO_TREE_SMEM", "SMZ_NO_PDL", "SMZ_M64", "SMZ_M32", "SMZ_PIPE2", "SMZ_NO_PIPE", "SMZ_STREAM_ALL",
            "SMZ_TC32_POLY")


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    A: int
    C: int
    K: int
    N: int
    n_trees: int
    net: str = "bf16"
    shape: Tuple[int, int, int, int] = (4, 61, 126, 4)     # obs, S, H, L
    lanes: int = 0                                         # 0: the engine's default
    max_trees: int = 0                                     # 0: n_trees
    rng: str = "philox"
    seed: int = 1
    offset: int = 0                                        # tree_id_offset
    players: int = 1
    loop: Optional[str] = None
    root_to_play: Optional[Tuple[int, ...]] = None         # cycled over the trees
    train: bool = True
    pb_c_base: int = 19652
    pb_c_init: float = 1.25
    discount: float = 0.997
    alpha: float = 0.25
    frac: float = 0.25
    policy_scale: float = 1.0                              # pred / apred policy output layers
    value_scale: float = 1.0                               # pred / apred value and dyn reward output layers
    chunks: Tuple[int, ...] = ()                           # simulate() calls; () = one call of N
    env: Tuple[Tuple[str, str], ...] = ()

    @property
    def G(self):
        return self.lanes or default_lanes(self.A, self.C)

    def kernel(self, sms, no_smem=False):
        return tree_kernel(self.G, self.A, self.C, self.K, self.N, self.n_trees, sms, no_smem)

    def search(self):
        return dict(pb_c_base=self.pb_c_base, pb_c_init=self.pb_c_init, discount=self.discount,
                    root_dirichlet_alpha=self.alpha, root_exploration_fraction=self.frac, num_simulations=self.N,
                    maxium_action_sample=self.K, number_of_player=self.players, custom_loop=self.loop)


PEAKY = 3000.0      # policy logits of a few units on random-init trunks: one or two entries carry the mass
LARGE = 2000.0      # value / reward supports driven to their ends: |values| in the hundreds

HAND_PICKED = [
    # mirror at G = 32, random subsets (K < A = C), the 32-draw Philox window overrun by every step
    Case("a32c32k3_peaky", 32, 32, 3, 60, 40, net="bf16", shape=(12, 61, 126, 4), policy_scale=PEAKY, seed=11),
    # mirror at G = 32 just under 96 KB, and one simulation more: the arena-only kernel by size
    Case("a2c32k32_n31_mirror_limit", 2, 32, 32, 31, 24, net="tc32", shape=(16, 61, 126, 4), seed=12),
    Case("a2c32k32_n32_arena_by_size", 2, 32, 32, 32, 24, net="f16", shape=(16, 33, 64, 2), seed=13),
    # non-power-of-two widths on 32 lanes, partial block
    Case("a17c5k3_lanes32", 17, 5, 3, 40, 50, net="fp32", shape=(7, 20, 40, 1), lanes=32, seed=14,
         value_scale=LARGE),
    Case("a16c16k4_lanes16", 16, 16, 4, 50, 100, net="bf16", shape=(9, 64, 128, 3), lanes=16, seed=15),
    Case("a16c16k4_lanes32", 16, 16, 4, 50, 30, net="tc32", shape=(9, 64, 128, 3), lanes=32, seed=16,
         policy_scale=PEAKY),
    Case("a16c16k4_n150_lanes16_arena_by_size", 16, 16, 4, 150, 20, net="fp32", shape=(5, 9, 17, 0), lanes=16,
         seed=17),
    Case("a8c8k2_lanes8", 8, 8, 2, 50, 64, net="f16", shape=(3, 8, 8, 5), lanes=8, rng="tape", seed=18,
         value_scale=LARGE),
    Case("a2c2k1_n40_lanes2", 2, 2, 1, 40, 48, net="fp32", shape=(4, 61, 126, 4), lanes=2, rng="tape", seed=19),
    # deep chains: one child per node, a path of N + 1 nodes; N = 100 fits the mirror, N = 200 does not
    Case("chain_n100", 1, 1, 1, 100, 16, net="bf16", shape=(2, 4, 16, 1), seed=20, value_scale=LARGE),
    Case("chain_n200", 1, 1, 1, 200, 8, net="fp32", shape=(2, 4, 16, 1), seed=21, value_scale=LARGE),
    Case("k_above_both_widths", 5, 3, 7, 40, 20, net="tc32", shape=(6, 12, 24, 2), rng="tape", seed=22),
    Case("n1_no_fused_step", 3, 3, 2, 1, 10, net="bf16", seed=23),
    Case("n2_one_fused_step", 3, 3, 2, 2, 10, net="f16", seed=24),
    # three players, custom cycle with a repeated player, root_to_play outside [0, 4)
    Case("players3_custom_loop", 4, 6, 3, 50, 32, net="bf16", shape=(8, 30, 60, 2), players=3, loop="1>2>1>3",
         root_to_play=(-7, 9, 0, 3, 13, -1, 2, 6), seed=25, value_scale=LARGE),
    Case("players2_modular", 3, 5, 2, 40, 20, net="fp32", shape=(8, 30, 60, 2), players=2,
         root_to_play=(1, 0, -3, 4), seed=26),
    Case("eval_mode", 6, 4, 3, 40, 20, net="f16", shape=(10, 16, 32, 1), train=False, seed=27),
    Case("discount1_large_values", 4, 4, 2, 50, 30, net="tc32", discount=1.0, value_scale=LARGE, seed=28),
    Case("discount0", 4, 4, 2, 50, 30, net="bf16", discount=0.0, value_scale=LARGE, seed=29),
    Case("pbc_base1_init0", 5, 5, 3, 40, 20, net="fp32", pb_c_base=1, pb_c_init=0.0, seed=30),
    Case("max_trees_above_n_trees", 9, 9, 3, 40, 77, max_trees=300, net="bf16", shape=(5, 40, 100, 3), seed=31,
         offset=1000),
    Case("simulate_in_two_chunks", 3, 6, 2, 40, 40, net="f16", chunks=(17, 23), seed=32, offset=77),
    Case("n0_wide_readout", 32, 7, 3, 0, 50, net="fp32", shape=(3, 10, 20, 1), seed=33),
    # both sides of the blocks-per-SM switch at G = 32: 296 blocks of 4 trees, then one tree more
    Case("blocks_per_sm_at_limit", 20, 9, 3, 12, 296 * 4, net="bf16", shape=(6, 32, 64, 2), seed=34),
    Case("blocks_per_sm_above_limit", 20, 9, 3, 12, 296 * 4 + 1, net="bf16", shape=(6, 32, 64, 2), seed=34),
]

# one wide case under every bf16 chain choice and with programmatic dependent launch off: each network kernel
# signals its dependents itself, and the mirror prologue relies on that ordering
_CHAIN_ENVS = {
    "m64_off": (("SMZ_M64", "0"),),
    "two_tiles_per_cta": (("SMZ_M64", "0"), ("SMZ_PIPE2", "1")),
    "m64_64_leaves": (("SMZ_M64", "1"), ("SMZ_M32", "0")),
    "m64_32_leaves": (("SMZ_M64", "1"), ("SMZ_M32", "1")),
    "no_pipe": (("SMZ_NO_PIPE", "1"),),
    "no_pdl": (("SMZ_NO_PDL", "1"),),
}
CHAIN_CASES = [Case(f"a32c32k3_bf16_{k}", 32, 32, 3, 40, 300, net="bf16", shape=(12, 61, 126, 4),
                    policy_scale=PEAKY, value_scale=LARGE, seed=40, offset=5, env=v) for k, v in _CHAIN_ENVS.items()]
CHAIN_CASES.append(Case("a16c16k4_tc32_no_pdl", 16, 16, 4, 40, 200, net="tc32", shape=(12, 61, 126, 4), seed=41,
                        env=(("SMZ_NO_PDL", "1"),)))


def _random_cases(n=16):
    """Seeded random configurations, drawn like test_gpu_parity._random_case, with model shapes and lane counts."""
    out = []
    for i in range(n):
        g = np.random.default_rng(5000 + i)
        A, C, K = int(g.integers(1, 33)), int(g.integers(1, 33)), int(g.integers(1, 34))
        N = int(g.integers(0, 61))
        players = int(g.integers(1, 4))
        loop = None if g.random() < 0.8 else ">".join(str(int(v)) for v in g.integers(1, 4, int(g.integers(1, 5))))
        need = max(2, 1 << (max(A, C) - 1).bit_length())
        lanes = int(g.choice([0] + [G for G in (2, 4, 8, 16, 32) if G >= need]))
        n_trees = int(g.integers(1, 200))
        shape = (int(g.integers(1, 200)), int(g.integers(2, 65)), int(g.integers(1, 129)), int(g.integers(0, 11)))
        out.append(Case(
            f"random{i}", A, C, K, N, n_trees, net=NETS[i % 4], shape=shape, lanes=lanes,
            max_trees=n_trees + int(g.integers(0, 3)) * int(g.integers(0, 100)),
            rng="tape" if n_trees <= 16 else "philox", seed=int(g.integers(1, 2 ** 40)),
            offset=int(g.integers(0, 10 ** 6)), players=players, loop=loop,
            root_to_play=tuple(int(v) for v in g.integers(-9, 10, 5)), train=bool(g.random() < 0.7),
            pb_c_base=int(g.integers(1, 30000)), pb_c_init=float(g.random() * 2), discount=float(0.8 + 0.2 * g.random()),
            alpha=float(max(g.random(), 1e-3)), frac=float(g.random()),
            policy_scale=float(10 ** g.uniform(0, 3.5)), value_scale=float(10 ** g.uniform(0, 3.3))))
    return out


CASES = HAND_PICKED + CHAIN_CASES + _random_cases()


# ---------------------------------------------------------------------------------------------------
# no GPU: the table still reaches what it is meant to reach
# ---------------------------------------------------------------------------------------------------
def test_case_table_reaches_both_tree_kernels():
    assert len({c.name for c in CASES}) == len(CASES)
    fused = [c for c in CASES if c.N >= 2]
    mirror_at = {c.G for c in fused if c.kernel(B200_SMS) == "mirror"}
    assert mirror_at >= {2, 4, 8, 16, 32}, f"mirror kernel reached at G = {sorted(mirror_at)} only"
    by_size = {c.G for c in fused if mirror_bytes(c.G, c.A, c.C, c.K, c.N) > MIRROR_LIMIT}
    assert {16, 32} <= by_size, f"arena-only kernel by size reached at G = {sorted(by_size)} only"
    for c in fused:
        assert c.kernel(B200_SMS, no_smem=True) == "arena"
    # both sides of the blocks-per-SM switch, with a mirror that fits
    limit = MIRROR_BLOCKS_PER_SM * B200_SMS
    blocks = {(c.n_trees * c.G + K_THREADS - 1) // K_THREADS: c for c in fused
              if mirror_bytes(c.G, c.A, c.C, c.K, c.N) <= MIRROR_LIMIT}
    assert limit in blocks and blocks[limit].kernel(B200_SMS) == "mirror"
    assert limit + 1 in blocks and blocks[limit + 1].kernel(B200_SMS) == "arena"
    # the Philox window of the mirror is overrun within one step (a decision node of width > UWIN - K draws)
    assert any(c.kernel(B200_SMS) == "mirror" and c.rng == "philox" and c.A + min(c.K, c.C) > UWIN for c in fused)
    # mirror cases that read root priors beyond the first 16, and deep chains on both kernels
    assert any(c.kernel(B200_SMS) == "mirror" and c.A > 16 for c in fused)
    assert {c.kernel(B200_SMS) for c in fused if c.A == c.C == 1} == {"mirror", "arena"}
    # every network mode, tape and Philox, fused-only behaviour
    assert {c.net for c in CASES} == set(NETS) and {c.rng for c in CASES} == {"tape", "philox"}
    assert any(c.loop for c in fused) and any(not c.train for c in fused) and any(c.chunks for c in fused)
    assert any(c.N == 0 for c in CASES) and any(c.N == 1 for c in CASES)
    assert any(c.K == 1 for c in fused) and any(c.K > max(c.A, c.C) for c in fused)
    assert any(c.discount == 1.0 for c in fused) and any(c.discount == 0.0 for c in fused)
    assert any(c.max_trees > c.n_trees for c in fused)


def test_kernel_choice_restatement_matches_the_source():
    """The constants the restatement above depends on, read from csrc/smz_tree.cu: if the C code changes them, the
    coverage claim of the table fails here instead of silently drifting."""
    src = open(TREE_CU).read()
    assert re.search(r"constexpr int SMZ_UWIN = (\d+);", src).group(1) == str(UWIN)
    assert re.search(r"static const int kThreads = (\d+);", src).group(1) == str(K_THREADS)
    assert "mirror_bytes(a, lanes) <= 96 * 1024" in src
    assert re.search(r'atoi\(getenv\("SMZ_MIRROR_BLOCKS_PER_SM"\)\) : (\d+);', src).group(1) == str(MIRROR_BLOCKS_PER_SM)
    assert "smz_mirror_bytes(kThreads / lanes, a.M, a.A, rcp_entries(a), a.N + 2)" in src
    assert "a.N + 3 > SMZ_MAX_POLICY + 1 ? a.N + 3 : SMZ_MAX_POLICY + 1" in src
    body = re.search(r"inline size_t smz_mirror_bytes\(int tpb, int M, int A, int n_tab, int n_pbc\) \{(.*?)\n\}",
                     src, re.S).group(1)
    lines = [ln.split("//")[0].strip() for ln in body.strip().splitlines()]
    assert lines == ["size_t b = (size_t)tpb * M * (sizeof(int4) + sizeof(int2));",
                     "b += (size_t)tpb * (A + SMZ_UWIN) * sizeof(double);",
                     "b += (size_t)(n_pbc + n_tab) * sizeof(double) + (size_t)n_tab * sizeof(float);",
                     "return b + 16;"]
    assert "smz_tree_mirror_fits(a, lanes) && mirror_pays((n_trees * lanes + kThreads - 1) / kThreads)" in src


# ---------------------------------------------------------------------------------------------------
# GPU: case runner, oracle replay, read-out
# ---------------------------------------------------------------------------------------------------
def _device_sms():
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _model(case):
    from stochastic_muzero_b200 import ModelShape
    from stochastic_muzero_b200.weights import blob_layout, random_blob
    obs, S, H, L = case.shape
    shape = ModelShape(obs, case.A, case.C, S, H, L)
    blob = random_blob(shape, seed=case.seed % 2 ** 32)
    layout, _ = blob_layout(shape)
    # only the head output layers are scaled (the trunks stay at their random init), so the activations of the
    # fp16 operands stay far below 65504
    for name, scale in (("pred.policy.w", case.policy_scale), ("apred.policy.w", case.policy_scale),
                        ("pred.value.w", case.value_scale), ("apred.value.w", case.value_scale),
                        ("dyn.reward.w", case.value_scale)):
        off, shp = layout[name]
        blob[off:off + int(np.prod(shp))] *= np.float32(scale)
    return shape, blob


def _inputs(case):
    g = np.random.default_rng(case.seed % 2 ** 32 + 1)
    obs = g.standard_normal((case.n_trees, case.shape[0])).astype(np.float32)
    rtp = None
    if case.root_to_play is not None:
        rtp = np.resize(np.asarray(case.root_to_play, np.int32), case.n_trees)
    # tape long enough for any of these searches (the engine raises if a tree runs past its end)
    tape = g.random((case.n_trees, 100_000)) if case.rng == "tape" else None
    return obs, rtp, tape


def run_case(case, monkeypatch, no_smem=False, record=True, export=()):
    """One fused search: engine built with the case's environment switches (set before the graph is captured),
    root + simulate (in chunks if the case says so); returns the record, the root read-out, the engine and the
    canonical dumps of the trees in `export`."""
    import torch
    from stochastic_muzero_b200 import SearchEngine
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in case.env:
        monkeypatch.setenv(k, v)
    if no_smem:
        monkeypatch.setenv("SMZ_NO_TREE_SMEM", "1")
    shape, blob = _model(case)
    obs, rtp, tape = _inputs(case)
    eng = SearchEngine(case.search(), case.A, case.C, max_trees=case.max_trees or case.n_trees, model_shape=shape,
                       net=case.net, rng=case.rng, seed=case.seed, tree_id_offset=case.offset,
                       lanes_per_tree=case.lanes, record=record)
    eng.set_weights(blob)
    if tape is not None:
        eng.set_uniform_tape(torch.from_numpy(tape))
    eng.root(obs=torch.from_numpy(obs), root_to_play=None if rtp is None else torch.from_numpy(rtp), train=case.train)
    for k in case.chunks or (case.N,):
        eng.simulate(k)
    eng.stats()                                             # raises on the device error flag
    out = {"roots": {k: v.cpu().numpy() for k, v in eng.read_roots().items()},
           "rec": {k: v.cpu().numpy() for k, v in eng.read_record().items()} if record else None,
           "trees": {int(b): eng.export_tree(int(b)) for b in export}, "eng": eng, "tape": tape, "rtp": rtp}
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    return out


def replay_sample(case):
    """Every tree up to 64 trees; else the first and last tree of the first and last block, the last live tree and
    random picks."""
    n = case.n_trees
    if n <= 64:
        return list(range(n))
    tpb = K_THREADS // case.G
    last_block = (n - 1) // tpb * tpb
    pick = {0, min(tpb, n) - 1, last_block, n - 1}
    pick |= set(int(b) for b in np.random.default_rng(case.seed % 2 ** 32).choice(n, 12, replace=False))
    return sorted(pick)


def _oracle_tree(case, run, b):
    rec = run["rec"]
    A, N = case.A, case.N
    width = np.where(rec["sim_branch"][b] == 1, A, case.C)
    model = O.TapeModel(rec["root_policy"][b, :A], rec["sim_policy"][b], width, rec["sim_value"][b], rec["sim_reward"][b])
    rng = O.TapeUniforms(run["tape"][b]) if case.rng == "tape" else O.PhiloxUniforms(case.seed, case.offset + b)
    cfg = O.SearchConfig(**case.search())
    phase = 0 if run["rtp"] is None else int(run["rtp"][b]) % len(cfg.cycle_map())
    tree = O.search(cfg, model, rng, train=case.train, dirichlet=rec["dirichlet"][b] if N else None,
                    root_to_play=phase)
    return tree.dump(), rng.cursor


def check_replay(case, run, what, cache):
    """Each exported tree against the oracle's replay of the engine's own record.  `cache` holds oracle results by
    record row: a second run that recorded the same outputs and draws is compared with the same replay."""
    rec = run["rec"]
    for b, got in run["trees"].items():
        key = (b, rec["root_policy"][b].tobytes(), rec["sim_policy"][b].tobytes(), rec["sim_value"][b].tobytes(),
               rec["sim_reward"][b].tobytes(), rec["sim_branch"][b].tobytes(), rec["dirichlet"][b].tobytes())
        if key not in cache:
            cache[key] = _oracle_tree(case, run, b)
        exp, cursor = cache[key]
        golden_io.assert_dump_equal(got, exp, f"{what}[{b}]")
        assert got["n_uniforms"] == cursor, f"{what}[{b}]: {got['n_uniforms']} draws consumed, oracle {cursor}"
        # the root read-out agrees with the replayed tree
        kids = np.flatnonzero(exp["depth"] == 1)
        assert np.array_equal(run["roots"]["visits"][b], exp["visit"][kids]), f"{what}[{b}]: root visits"
        assert np.array_equal(run["roots"]["priors"][b], exp["prior"][kids]), f"{what}[{b}]: root priors"
        rv = np.float32(0) if exp["visit"][0] == 0 else np.float32(exp["value_sum"][0] / np.float32(exp["visit"][0]))
        assert run["roots"]["root_values"][b] == rv, f"{what}[{b}]: root value"


TEMPERATURES = (0.0, 0.05, 0.1, 0.2, 0.25, 0.3, 1 / 3, 0.5, 1.0, 2.0)


def check_readout(case, run, what):
    """select_actions(T) on every tree against readout_oracle: recorded uniforms, and the device Philox draw
    (stream 2, index 0 of tree tree_id_offset + b)."""
    import torch
    eng = run["eng"]
    visits, priors = run["roots"]["visits"], run["roots"]["priors"]
    n = case.n_trees
    stored = np.array([R.stored_policy(visits[b], priors[b]) for b in range(n)])
    u_dev = np.array([O.philox_uniform(case.seed, case.offset + b, 0, stream=2) for b in range(n)])
    g = np.random.default_rng(case.seed % 2 ** 32 + 2)
    for T in TEMPERATURES:
        u = g.random(n)
        out = {k: v.cpu().numpy() for k, v in eng.select_actions(T, uniforms=torch.from_numpy(u)).items()}
        dev = {k: v.cpu().numpy() for k, v in eng.select_actions(T).items()}
        pol = out["policy"]
        exp = np.array([R.step_policy(visits[b], priors[b], T) for b in range(n)])
        e = 1.0 / T if T >= 0.3 else 1.0
        if e in (1.0, 2.0, 0.5):          # exact arithmetic on both sides
            assert np.array_equal(pol, exp), f"{what}: acting policy at T={T}"
        else:                             # pow(): libm vs CUDA, <= 2 ulp
            np.testing.assert_allclose(pol, exp, rtol=1e-14, atol=0, err_msg=f"{what}: acting policy at T={T}")
        assert np.array_equal(out["stored_policy"], stored), f"{what}: stored policy at T={T}"
        assert np.array_equal(dev["policy"], pol) and np.array_equal(dev["stored_policy"], stored)
        # the sampling / argmax step on the policy the device computed
        act = np.array([R.select_action(pol[b], T, u[b])[0] for b in range(n)])
        act_dev = np.array([R.select_action(pol[b], T, u_dev[b])[0] for b in range(n)])
        bad = np.flatnonzero(out["actions"] != act)
        assert not len(bad), f"{what}: T={T} recorded-uniform actions differ at trees {bad[:5]}"
        bad = np.flatnonzero(dev["actions"] != act_dev)
        assert not len(bad), f"{what}: T={T} device-Philox actions differ at trees {bad[:5]}"


def _assert_roots_equal(a, b, what):
    for k in ("visits", "root_values", "priors", "rewards", "error"):
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), f"{what}: read_roots()['{k}'] differs"


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_fused_search_replays_bit_exact_on_both_tree_kernels(case, monkeypatch):
    sample = replay_sample(case)
    label = case.kernel(_device_sms()) or "no fused step"
    cache = {}
    default = run_case(case, monkeypatch, export=sample)
    check_replay(case, default, f"{case.name} default ({label}, G={case.G})", cache)
    arena = run_case(case, monkeypatch, no_smem=True, export=sample)
    check_replay(case, arena, f"{case.name} SMZ_NO_TREE_SMEM=1 (arena, G={case.G})", cache)
    _assert_roots_equal(default["roots"], arena["roots"], f"{case.name}: {label} vs arena")
    arena["eng"].close()
    assert default["roots"]["error"][0] == 0 and (default["roots"]["visits"].sum(1) == case.N).all()
    check_readout(case, default, f"{case.name} read-out")
    default["eng"].close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["a32c32k3_peaky", "a16c16k4_lanes16", "players3_custom_loop"])
def test_record_off_gives_the_same_search(name, monkeypatch):
    """The record buffers are written by the tree step only when asked for; the search itself must not change."""
    case = next(c for c in CASES if c.name == name)
    every = list(range(case.n_trees))
    on = run_case(case, monkeypatch, record=True, export=every)
    off = run_case(case, monkeypatch, record=False, export=every)
    _assert_roots_equal(on["roots"], off["roots"], f"{name}: record off")
    for b in every:
        golden_io.assert_dump_equal(off["trees"][b], on["trees"][b], f"{name}[{b}] record off vs on")
        assert off["trees"][b]["n_uniforms"] == on["trees"][b]["n_uniforms"]
    for T in (0.0, 0.5, 1.0):
        a, b = on["eng"].select_actions(T), off["eng"].select_actions(T)
        for k in a:
            assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy()), f"{name}: select_actions({T})['{k}']"
    on["eng"].close()
    off["eng"].close()
