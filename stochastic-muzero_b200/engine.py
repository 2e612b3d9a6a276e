"""SearchEngine — thin torch-facing wrapper over the C ABI (include/smz.h).

torch is used for device memory and streams only; every computation happens in libsmz.so.  Tensors
are handed over as raw ``data_ptr()``; the engine owns nothing but its arena.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .weights import VISION_FLAT, ModelShape, VisionShape

SEARCH_KEYS = ("pb_c_base", "pb_c_init", "discount", "root_dirichlet_alpha", "root_exploration_fraction",
               "num_simulations", "maxium_action_sample", "number_of_player", "custom_loop")
_NET = {"external": _lib.NET_EXTERNAL, "fp32": _lib.NET_FP32, "bf16": _lib.NET_BF16, "vision": _lib.NET_VISION,
        "tc32": _lib.NET_TC32, "f16": _lib.NET_F16}
_RNG = {"philox": _lib.RNG_PHILOX, "tape": _lib.RNG_TAPE}


class SmzError(RuntimeError):
    pass


def _is_chance(depth: int, paper_alternation: bool = False) -> bool:
    """Node kind by depth: the reference's F,F,T,T,F,F,... (monte_carlo_tree_search.py:211, :333-345), or with
    ``paper_alternation`` the Stochastic MuZero alternation F,T,F,T,... (smz_set_node_pattern in include/smz.h)."""
    return bool((depth >> (0 if paper_alternation else 1)) & 1)


def player_tables(number_of_player: int, custom_loop: Optional[str], n_depth: int, paper_alternation: bool = False):
    """Player_cycle (monte_carlo_tree_search.py:38-72) flattened per (root_to_play phase, depth):
    to_play of a node and the sign its backed-up value gets (:302-305).  A chance node keeps its parent's
    to_play, a decision node gets the next player, so the tables follow the node pattern."""
    if custom_loop is not None:
        cycle = [float(i) for i in custom_loop.split(">")]
    else:
        cycle = list(range(number_of_player))
    n = len(cycle)
    sign = np.ones((n, n_depth), np.int8)
    to_play = np.zeros((n, n_depth), np.int32)
    for p in range(n):
        tp = p
        for d in range(n_depth):
            if d >= 1:
                tp = tp if _is_chance(d, paper_alternation) else (tp + 1) % n      # :210, :296
            to_play[p, d] = tp
            sign[p, d] = 1 if cycle[p % n] == cycle[tp % n] else -1
    return sign, to_play


class RootStats(dict):
    """read_roots() result: the tensors by name; ``block`` = the device block that holds visits | root values | error."""
    block = None


class SearchEngine:
    """One engine = one arena of ``max_trees`` trees on one GPU, driven on one CUDA stream."""

    def __init__(self, search: Dict, action_dim: int, chance_dim: Optional[int] = None, max_trees: int = 1,
                 model_shape: Optional[ModelShape] = None, net: str = "external", rng: str = "philox",
                 seed: int = 0, tree_id_offset: int = 0, device: Optional[int] = None, lanes_per_tree: int = 0,
                 record: bool = False, paper_alternation: bool = False):
        """``paper_alternation``: search with the Stochastic MuZero node alternation instead of the reference's depth
        pattern (smz_set_node_pattern in include/smz.h); ``set_node_pattern`` changes it for later searches."""
        if not torch.cuda.is_available():
            raise SmzError("SearchEngine needs a CUDA device; the search path has no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.search = {k: search[k] for k in SEARCH_KEYS if k in search}
        self.A = int(action_dim)
        self.Cdim = int(chance_dim if chance_dim is not None else action_dim)
        self.N = int(search["num_simulations"])
        self.K = int(search["maxium_action_sample"])
        self.net, self.rng = net, rng
        cfg = _lib.smz_config()
        cfg.abi_version = _lib.SMZ_ABI_VERSION
        cfg.device = self.device
        cfg.max_trees = int(max_trees)
        cfg.num_simulations = self.N
        cfg.action_dim, cfg.chance_dim = self.A, self.Cdim
        cfg.max_action_sample = self.K
        cfg.pb_c_base = int(search["pb_c_base"])
        cfg.pb_c_init = float(search["pb_c_init"])
        cfg.discount = float(search["discount"])
        cfg.root_dirichlet_alpha = float(search["root_dirichlet_alpha"])
        cfg.root_exploration_fraction = float(search["root_exploration_fraction"])
        if net == "vision":
            if not isinstance(model_shape, VisionShape) or model_shape.action_dim != self.A or self.Cdim != self.A:
                raise ValueError("the vision network needs a VisionShape with action_dim == chance_dim == A")
            cfg.obs_dim, cfg.state_dim = 3 * 98 * 98, model_shape.state_dim
            cfg.hidden_dim, cfg.num_hidden_layers = model_shape.hidden_dim, model_shape.num_hidden_layers
        elif net != "external":
            if model_shape is None:
                raise ValueError("model_shape is required for an internal network")
            if (model_shape.action_dim, model_shape.chance_dim) != (self.A, self.Cdim):
                raise ValueError("model_shape action/chance widths differ from the search's")
            cfg.obs_dim, cfg.state_dim = model_shape.obs_dim, model_shape.state_dim
            cfg.hidden_dim, cfg.num_hidden_layers = model_shape.hidden_dim, model_shape.num_hidden_layers
        self.model_shape = model_shape
        # floats of a hidden-state row that carry data (the rest of the arena row is padding)
        self.hidden_width = VISION_FLAT if net == "vision" else (model_shape.state_dim if model_shape else 0)
        cfg.net_mode, cfg.rng_mode = _NET[net], _RNG[rng]
        cfg.lanes_per_tree = int(lanes_per_tree)
        cfg.record = int(record)
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.tree_id_offset = int(tree_id_offset)
        self._h = C.c_void_p()
        self._check(self.lib.smz_create(C.byref(cfg), C.byref(self._h)))
        self.dims = _lib.smz_dims()
        self._check(self.lib.smz_get_dims(self._h, C.byref(self.dims)))
        self.max_trees = int(max_trees)
        self.n_trees = 0
        self.generation = 0       # bumped by every root(): views of an older search can tell that they are stale
        self._keep = {}           # tensors the engine holds raw pointers to
        self._pinned = {}         # pinned host staging buffers by size (BatchedRoots.host)
        # sqrt(n) * pb_c(n) with numpy's sqrt/log, exactly as monte_carlo_tree_search.py:236-237 evaluates
        # `np.sqrt(parent.visit_count) * pb_c` on this host (the product is then multiplied by the prior)
        base, init = int(search["pb_c_base"]), float(search["pb_c_init"])
        pbc = np.array([np.sqrt(n) * (np.log((n + base + 1) / base) + init) for n in range(self.N + 2)], np.float64)
        self._check(self.lib.smz_set_pbc_table(self._h, pbc.ctypes.data_as(C.POINTER(C.c_double)), len(pbc)))
        self.paper_alternation = None         # pattern of the current search and of the uploaded player tables
        self._next_paper = bool(paper_alternation)
        self._apply_node_pattern()

    def set_node_pattern(self, paper_alternation: bool):
        """Node pattern of the searches started by the following root() calls; a search already rooted keeps its own."""
        self._next_paper = bool(paper_alternation)

    def _apply_node_pattern(self):
        """Engine setting and player tables of the pending pattern, before a root step (the tables follow the pattern)."""
        paper = self._next_paper
        if paper == self.paper_alternation:
            return
        self._check(self.lib.smz_set_node_pattern(self._h, _lib.PATTERN_PAPER if paper else _lib.PATTERN_REFERENCE))
        sign, to_play = player_tables(int(self.search.get("number_of_player", 1)), self.search.get("custom_loop"),
                                      self.N + 2, paper)
        self.to_play_table = to_play
        self.n_phases = sign.shape[0]
        sign, to_play = np.ascontiguousarray(sign), np.ascontiguousarray(to_play)
        self._check(self.lib.smz_set_player_tables(self._h, sign.ctypes.data_as(C.POINTER(C.c_int8)),
                                                   to_play.ctypes.data_as(C.POINTER(C.c_int32)), self.n_phases))
        self.paper_alternation = paper

    # ------------------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            msg = self.lib.smz_last_error().decode()
            exc = ValueError if rc in (_lib.SMZ_E_INVALID_ARG, _lib.SMZ_E_CAPACITY) else SmzError
            raise exc(f"libsmz error {rc}: {msg}")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.smz_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, t, dtype, name):
        if t is None:
            return None
        if not torch.is_tensor(t):
            t = torch.as_tensor(np.asarray(t))
        t = t.to(device=f"cuda:{self.device}", dtype=dtype, non_blocking=True).contiguous()
        self._keep[name] = t
        return t

    def to_device(self, t, dtype):
        """Host or device tensor / array -> contiguous tensor of `dtype` on the engine's device (asynchronous copy)."""
        if not torch.is_tensor(t):
            t = torch.as_tensor(np.asarray(t))
        return t.to(device=f"cuda:{self.device}", dtype=dtype, non_blocking=True).contiguous()

    @staticmethod
    def _ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def _new(self, *shape, dtype):
        return torch.empty(*shape, dtype=dtype, device=f"cuda:{self.device}")

    # ------------------------------------------------------------------------------------------
    def set_weights(self, blob):
        """blob: fp32 tensor/array in the layout of weights.blob_layout (host or device)."""
        if torch.is_tensor(blob) and blob.is_cuda:
            t = blob.to(dtype=torch.float32).contiguous()
            self._check(self.lib.smz_set_weights(self._h, self._ptr(t), t.numel(), 1, self._stream))
            self._keep["blob"] = t
        else:
            arr = np.ascontiguousarray(blob.cpu().numpy() if torch.is_tensor(blob) else blob, dtype=np.float32)
            self._check(self.lib.smz_set_weights(self._h, C.c_void_p(arr.ctypes.data), arr.size, 0, self._stream))
            torch.cuda.current_stream(self.device).synchronize()

    def set_seed(self, seed: int, tree_id_offset: int = 0):
        self._check(self.lib.smz_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(tree_id_offset), self._stream))

    def set_uniform_tape(self, uniforms):
        t = self._dev(uniforms, torch.float64, "tape")
        assert t.dim() == 2
        self._check(self.lib.smz_set_uniform_tape(self._h, self._ptr(t), t.shape[1]))

    def root(self, obs=None, root_policy=None, root_to_play=None, train=True, dirichlet=None):
        src = obs if obs is not None else root_policy
        n = int(src.shape[0])
        obs_t = self._dev(obs, torch.float32, "obs")
        pol_t = None
        if root_policy is not None:
            pol_t = self._pad_policy(self._dev(root_policy, torch.float32, "root_policy"), "root_policy")
        rtp = self._dev(root_to_play, torch.int32, "root_to_play")
        dr = self._dev(dirichlet, torch.float64, "dirichlet")
        self._apply_node_pattern()
        self._check(self.lib.smz_root(self._h, n, self._ptr(obs_t), self._ptr(pol_t), self._ptr(rtp), int(bool(train)),
                                      self._ptr(dr), self._stream))
        self.n_trees = n
        self.generation += 1

    def _pad_policy(self, p, name):
        W = self.dims.policy_stride
        if p.shape[1] != W:
            q = torch.zeros(p.shape[0], W, dtype=torch.float32, device=p.device)
            q[:, :p.shape[1]] = p
            p = q
            self._keep[name] = p
        return p

    def simulate(self, n_sims=None):
        self._check(self.lib.smz_simulate(self._h, self.N if n_sims is None else int(n_sims), self._stream))

    def select(self, sim):
        slot, action, branch = (self._new(self.n_trees, dtype=torch.int32) for _ in range(3))
        self._check(self.lib.smz_select(self._h, int(sim), self._ptr(slot), self._ptr(action), self._ptr(branch),
                                        self._stream))
        return slot, action, branch

    def net_step(self, sim):
        self._check(self.lib.smz_net_step(self._h, int(sim), self._stream))

    def backup_select(self, sim):
        """The fused tree step of the captured loop (expansion + backup of `sim`, descent of `sim + 1`)."""
        self._check(self.lib.smz_backup_select(self._h, int(sim), self._stream))

    def expand_backup(self, sim, policy=None, value=None, reward=None):
        if policy is None:
            self._check(self.lib.smz_expand_backup(self._h, int(sim), None, None, None, self._stream))
            return
        p = self._pad_policy(self._dev(policy, torch.float32, "policy"), "policy")
        v = self._dev(value, torch.float32, "value")
        r = self._dev(reward, torch.float32, "reward")
        self._check(self.lib.smz_expand_backup(self._h, int(sim), self._ptr(p), self._ptr(v), self._ptr(r), self._stream))

    def net_eval(self, which: str, x, idx=None):
        """Stand-alone evaluation of one network: which in repr/pred/adyn/apred/dyn/enc."""
        w = ["repr", "pred", "adyn", "apred", "dyn", "enc"].index(which)
        x = self._dev(x, torch.float32, "eval_in")
        n = x.shape[0]
        x = x.reshape(n, -1)
        if w not in (0, 5) and x.shape[1] != self.dims.hidden_stride:
            xp = torch.zeros(n, self.dims.hidden_stride, dtype=torch.float32, device=x.device)
            xp[:, :x.shape[1]] = x
            x = xp
        idx_t = self._dev(idx, torch.int32, "eval_idx")
        S = self.hidden_width
        hidden = self._new(n, self.dims.hidden_stride, dtype=torch.float32)
        policy = torch.zeros(n, self.dims.policy_stride, dtype=torch.float32, device=x.device)
        value, reward = self._new(n, dtype=torch.float32), self._new(n, dtype=torch.float32)
        code = self._new(n, dtype=torch.int32)
        self._check(self.lib.smz_net_eval(self._h, w, n, self._ptr(x), self._ptr(idx_t), self._ptr(hidden),
                                          self._ptr(policy), self._ptr(value), self._ptr(reward), self._ptr(code),
                                          self._stream))
        out = {}
        if w in (0, 2, 4):
            out["hidden"] = hidden[:, :S]
        if w == 4:
            out["reward"] = reward
        if w in (1, 3):
            out["policy"] = policy[:, :(self.A if w == 1 else self.Cdim)]
            out["value"] = value
        if w == 5:
            out["probs"], out["code"] = policy[:, :self.Cdim], code
        return out

    # ------------------------------------------------------------------------------------------
    def pinned(self, n_int32: int):
        """A pinned host staging buffer of n int32 (kept per size: read-outs of equal shape reuse it)."""
        buf = self._pinned.get(n_int32)
        if buf is None:
            buf = torch.empty(n_int32, dtype=torch.int32).pin_memory()
            self._pinned[n_int32] = buf
        return buf

    def read_roots(self, out=None):
        n, A = self.n_trees, self.A
        if out is None:
            # visit counts, root values and the error flag share ONE device block: a consumer on the host fetches all
            # three with a single copy (BatchedRoots.host)
            blk = self._new(n * A + n + 1, dtype=torch.int32)
            out = {"visits": blk[:n * A].view(n, A), "root_values": blk[n * A:n * A + n].view(torch.float32),
                   "priors": self._new(n, A, dtype=torch.float64), "rewards": self._new(n, A, dtype=torch.float32),
                   "error": blk[n * A + n:]}
            out = RootStats(out)
            out.block = blk
        self._check(self.lib.smz_read_roots(self._h, self._ptr(out.get("visits")), self._ptr(out.get("root_values")),
                                            self._ptr(out.get("priors")), self._ptr(out.get("rewards")),
                                            self._ptr(out.get("error")), self._stream))
        return out

    @staticmethod
    def raise_for_error(code: int):
        """Error flag of a search (smz_read_roots) -> the exception the reference would have raised."""
        if code == 1:
            raise SmzError("uniform tape exhausted during the search")
        if code == 2:       # np.random.choice at monte_carlo_tree_search.py:208 / :294 raises ValueError here
            raise ValueError("probabilities contain NaN or sum to zero: a policy met during expansion was degenerate "
                             "(np.random.choice raises at this point in the reference)")

    def select_actions(self, temperature: float, uniforms=None):
        """game.py:179-235 for every tree: -> dict(actions int32[n], policy f64[n,A], stored_policy f64[n,A])."""
        n, A = self.n_trees, self.A
        u = self._dev(uniforms, torch.float64, "readout_u")
        out = {"actions": self._new(n, dtype=torch.int32), "policy": self._new(n, A, dtype=torch.float64),
               "stored_policy": self._new(n, A, dtype=torch.float64)}
        self._check(self.lib.smz_select_actions(self._h, float(temperature), self._ptr(u), self._ptr(out["actions"]),
                                                self._ptr(out["policy"]), self._ptr(out["stored_policy"]), self._stream))
        return out

    def read_hidden(self, slot):
        out = self._new(self.n_trees, self.dims.hidden_stride, dtype=torch.float32)
        self._check(self.lib.smz_read_hidden(self._h, int(slot), self._ptr(out), self._stream))
        return out[:, :self.hidden_width]

    def read_record(self):
        n, N, W, A = self.n_trees, self.N, self.dims.policy_stride, self.A
        rec = {"sim_policy": self._new(n, N, W, dtype=torch.float32), "sim_value": self._new(n, N, dtype=torch.float32),
               "sim_reward": self._new(n, N, dtype=torch.float32), "sim_branch": self._new(n, N, dtype=torch.int8),
               "dirichlet": self._new(n, A, dtype=torch.float64), "root_policy": self._new(n, W, dtype=torch.float32)}
        self._check(self.lib.smz_read_record(self._h, self._ptr(rec["sim_policy"]), self._ptr(rec["sim_value"]),
                                             self._ptr(rec["sim_reward"]), self._ptr(rec["sim_branch"]),
                                             self._ptr(rec["dirichlet"]), self._ptr(rec["root_policy"]), self._stream))
        return rec

    def stats(self):
        depth, launches, total = C.c_double(), C.c_int64(), C.c_int64()
        self._check(self.lib.smz_stats(self._h, C.byref(depth), C.byref(launches), C.byref(total), self._stream))
        return {"mean_leaf_depth": depth.value, "launches": launches.value, "launches_total": total.value}

    def export_arena(self, tree: int) -> Dict[str, np.ndarray]:
        """One tree in arena order (see smz_tree_host)."""
        M, A = self.dims.nodes_per_tree, self.A
        cols = {"visit": np.zeros(M, np.int32), "value_sum": np.zeros(M, np.float32), "reward": np.zeros(M, np.float32),
                "prior": np.zeros(M, np.float32), "child_base": np.zeros(M, np.int32), "key": np.zeros(M, np.int32),
                "root_prior": np.zeros(A, np.float64)}
        th = _lib.smz_tree_host()
        th.visit = cols["visit"].ctypes.data_as(C.POINTER(C.c_int32))
        th.value_sum = cols["value_sum"].ctypes.data_as(C.POINTER(C.c_float))
        th.reward = cols["reward"].ctypes.data_as(C.POINTER(C.c_float))
        th.prior = cols["prior"].ctypes.data_as(C.POINTER(C.c_float))
        th.child_base = cols["child_base"].ctypes.data_as(C.POINTER(C.c_int32))
        th.key = cols["key"].ctypes.data_as(C.POINTER(C.c_int32))
        th.root_prior = cols["root_prior"].ctypes.data_as(C.POINTER(C.c_double))
        self._check(self.lib.smz_export_tree(self._h, int(tree), C.byref(th), self._stream))
        cols["minmax"] = np.array([th.minmax[0], th.minmax[1]], np.float32)
        cols["n_uniforms"] = int(th.n_uniforms)
        cols["root_to_play"] = int(th.root_to_play)
        return cols

    def n_children(self, depth: int) -> int:
        """Children of an expanded node at `depth`: A at the root, else min(K, width of the head that
        expanded it) — dynamics pair (width A) iff its parent is a chance node (T2), in either node pattern."""
        if depth == 0:
            return self.A
        return min(self.K, self.A) if _is_chance(depth - 1, self.paper_alternation) else min(self.K, self.Cdim)

    def export_tree(self, tree: int) -> Dict[str, np.ndarray]:
        """Canonical dump: depth-first, children in ascending key order (same format as the oracle's
        Tree.dump() and the golden files)."""
        ar = self.export_arena(tree)
        phase = ar["root_to_play"] % self.n_phases
        rows = []
        stack = [(0, 0)]
        while stack:
            n, d = stack.pop()
            cb = int(ar["child_base"][n])
            prior = 0.0 if n == 0 else (ar["root_prior"][n - 1] if d == 1 else np.float64(ar["prior"][n]))
            rows.append((d, -1 if n == 0 else int(ar["key"][n]), int(ar["visit"][n]), ar["value_sum"][n],
                         ar["reward"][n], prior, _is_chance(d, self.paper_alternation), int(self.to_play_table[phase, d]),
                         cb != 0, n))
            if cb:
                k = self.n_children(d)
                stack.extend((cb + i, d + 1) for i in reversed(range(k)))
        names = ("depth", "key", "visit", "value_sum", "reward", "prior", "is_chance", "to_play", "expanded", "node")
        dtypes = (np.int32, np.int32, np.int32, np.float32, np.float32, np.float64, np.int8, np.int32, np.int8, np.int32)
        out = {k: np.array([r[i] for r in rows], dtype=dt) for i, (k, dt) in enumerate(zip(names, dtypes))}
        out["minmax"] = ar["minmax"]
        out["n_uniforms"] = ar["n_uniforms"]
        return out
