"""Drop-in replacement for the reference's ``monte_carlo_tree_search.py`` backed by the CUDA engine.

Same call surface as /root/reference/monte_carlo_tree_search.py — ``Node`` (:6-21), ``MinMaxStats``
(:24-36), ``Player_cycle`` (:38-72), ``Monte_carlo_tree_search.__init__/reset/run`` (:75-349) — as
consumed by self_play.py:46/:85/:419 and muzero_cli.py:131-139, plus the additive batched entry
``run_batch`` (thousands of independent trees per call).  The tree lives in the engine's HBM arena;
``run`` returns a ``Node`` view materialised from it, so ``root.children[a].visit_count``,
``.prior``, ``.reward`` and ``root.value()`` (all that game.py:179-235 touches) behave as before.

Two ways a model can be attached:
  * a reference-style ``Muzero`` with ``model_structure == "mlp_model"``: its six modules are packed
    once (weights.pack_weights) and the whole search, network step included, runs on the GPU;
  * any other object exposing the five ``*_function_inference`` methods (other model families, test
    stubs): the tree kernels run on the GPU and the model is called back on the host once per
    simulation, like the reference does (:271-286).
"""
from __future__ import annotations

import weakref
from typing import Optional

import numpy as np
import torch

from . import batched_model
from .engine import SearchEngine, budget_rows, explore_rows, legal_rows
from .weights import (PackedModel, VisionShape, pack_vision_weights, pack_weights, shape_of, weights_version)


class Node(object):
    """Per-node record, attribute-compatible with the reference's Node (:6-21)."""

    __slots__ = ("visit_count", "prior", "value_sum", "children", "reward", "to_play", "is_chance",
                 "_hidden", "_hidden_fetch")

    def __init__(self, prior: float):
        self.visit_count = 0
        self.prior = prior
        self.value_sum = 0
        self.children = {}
        self.reward = 0
        self.to_play = -1
        self.is_chance = False
        self._hidden = 0
        self._hidden_fetch = None

    @property
    def hidden_state(self):
        if self._hidden_fetch is not None:
            self._hidden, self._hidden_fetch = self._hidden_fetch(), None
        return self._hidden

    @hidden_state.setter
    def hidden_state(self, value):
        self._hidden, self._hidden_fetch = value, None

    def expanded(self):
        return len(self.children) > 0

    def value(self) -> float:
        if self.visit_count == 0:
            return 0
        return self.value_sum / self.visit_count


class MinMaxStats(object):
    """Running bounds of the node values seen during one search (:24-36)."""

    def __init__(self, minimum=float("inf"), maximum=-float("inf")):
        self.maximum = maximum
        self.minimum = minimum

    def update(self, value: float):
        self.maximum = max(self.maximum, value)
        self.minimum = min(self.minimum, value)

    def normalize(self, value: float) -> float:
        if self.maximum > self.minimum:
            return (value - self.minimum) / (self.maximum - self.minimum)
        return value


class Player_cycle:
    """to_play bookkeeping (:38-72): modular cycle over ``number_of_player`` or a custom "1>2>3" loop."""

    def __init__(self, number_of_player: int = None, custom_loop: str = None):
        self.number_of_player = number_of_player
        self.custom_loop = custom_loop
        if isinstance(custom_loop, str):
            self.cycle_map = torch.tensor([float(i) for i in custom_loop.split(">")])
        elif number_of_player is not None and number_of_player >= 1:
            self.cycle_map = torch.arange(0, number_of_player)
        else:
            raise Exception("You have to provide a number of player >= 1 or a custom loop like : \"1>2>3\" ")
        self.loop_cycle = None
        self.global_origin = self.cycle_map[0]
        self.global_count = 0

    def _len(self):
        return self.cycle_map.size()[0]

    def proximate_player_step(self, player_index):
        return (player_index + 1) % self._len()

    def global_step(self):
        player_in_play = self.global_count % self._len()
        self.global_count = (1 + self.global_count) % self._len()
        return player_in_play

    def global_reset(self):
        self.global_count = 0

    def player_in_play(self, player_index):
        return self.cycle_map[player_index % self._len()]


def _node_tree(dump, hidden_fetch=None):
    """Materialise Node objects from a canonical depth-first dump (engine.export_tree)."""
    nodes, stack = [], []
    A_root = None
    for i in range(len(dump["depth"])):
        d = int(dump["depth"][i])
        prior = dump["prior"][i]
        if d == 0:
            node = Node(0)
        else:
            # root children carry float64 priors (Dirichlet mixing, :224), everything below float32
            node = Node(np.float64(prior) if d == 1 else np.float32(prior))
        node.visit_count = int(dump["visit"][i])
        node.value_sum = np.float32(dump["value_sum"][i]) if node.visit_count else 0
        node.to_play = int(dump["to_play"][i])
        node.is_chance = bool(dump["is_chance"][i])
        if dump["expanded"][i] and hidden_fetch is not None:
            node._hidden_fetch = (lambda n=int(dump["node"][i]): hidden_fetch(n))
        while stack and stack[-1][0] >= d:
            stack.pop()
        # only a node evaluated by the dynamics pair, i.e. one whose parent is a chance node, carries a reward (:333-337)
        node.reward = np.float32(dump["reward"][i]) if stack and stack[-1][1].is_chance and dump["expanded"][i] else 0
        if stack:
            stack[-1][1].children[np.int64(dump["key"][i])] = node
        stack.append((d, node))
        nodes.append(node)
    return nodes[0]


def _legal_row(legal_actions, A):
    """``run``'s legal actions (a sequence of action indices, or a bool mask [A]) -> bool mask [1, A] on the host."""
    if torch.is_tensor(legal_actions):
        legal_actions = legal_actions.cpu()
    a = np.asarray(legal_actions)
    if a.dtype == np.bool_:
        if a.shape != (A,):
            raise ValueError(f"a bool legal-action mask has shape [{A}], got {list(a.shape)}")
        return a.reshape(1, A)
    idx = a.astype(np.int64).reshape(-1)
    if idx.size == 0 or (idx < 0).any() or (idx >= A).any():
        raise ValueError(f"legal actions must be a non-empty sequence of indices in [0, {A}), got {idx.tolist()}")
    row = np.zeros((1, A), np.bool_)
    row[0, idx] = True
    return row


def _legal_kw(legal):
    """root() keyword for an optional mask (no keyword at all without one: the unmasked call stays as it was)."""
    return {} if legal is None else {"legal": legal}


def _budget_plan(num_simulations, n, N):
    """``num_simulations`` of run_batch / run -> (budgets for the root step or None, simulation steps to run).  None: every
    tree N; an int or a host sequence: checked here, and the search runs max(budget) steps; a device tensor: N steps, no
    host synchronisation (its range is checked by the root kernel)."""
    if num_simulations is None:
        return None, N
    bud = budget_rows(num_simulations, n, N)
    return bud, N if bud.is_cuda else (int(bud.max()) if bud.numel() else 0)


def _root_kw(legal, budget, explore):
    kw = _legal_kw(legal)
    if budget is not None:
        kw["budget"] = budget
    if explore is not None:
        kw["explore"] = explore
    return kw


class StaleSearchError(RuntimeError):
    """A view of a finished search was used after the engine's arena had been reused by a newer search."""


class BatchedRoots:
    """Result of ``run_batch``: root statistics of B trees as device tensors + lazy ``Node`` views.

    Lifetime: ``visit_counts`` / ``priors`` / ``rewards`` / ``root_values`` are tensors of their own and stay valid.
    ``roots[i]``, ``select_actions()`` and the lazy ``Node.hidden_state`` of a returned tree read the engine's arena,
    which the NEXT ``run`` / ``run_batch`` on the same ``Monte_carlo_tree_search`` reuses: from then on they raise
    ``StaleSearchError`` instead of silently describing the newer search (the reference's roots are
    self-contained; take what you need before searching again, or use a second Monte_carlo_tree_search)."""

    def __init__(self, engine: SearchEngine, stats):
        self._engine = engine
        self._generation = engine.generation
        self.visit_counts = stats["visits"]       # int32 [B, A]
        self.priors = stats["priors"]             # float64 [B, A]
        self.rewards = stats["rewards"]           # float32 [B, A]
        self.root_values = stats["root_values"]   # float32 [B]
        self.error = stats.get("error")           # int32 [1] device: the search's error flag (engine.raise_for_error)
        self.budgets = engine.budgets             # int32 [B] simulations of each tree (host or device), None = N each
        self._block = getattr(stats, "block", None)   # visit counts | root values | error flag in one device block
        self._host = None

    def __len__(self):
        return int(self.visit_counts.shape[0])

    def _live(self):
        if self._engine.generation != self._generation or not self._engine._h.value:
            raise StaleSearchError("this search's arena has been reused by a later run()/run_batch() (or the engine "
                                   "was reset); read roots[i] / select_actions() / hidden_state before searching again")
        return self._engine

    def host(self):
        """Visit counts int32 [B, A], root values float32 [B] and the error flag on the HOST: one device-to-host copy
        into a pinned buffer and one synchronisation for all three (cached: the check of ``run_batch`` already paid it)."""
        if self._host is None:
            B, A = self.visit_counts.shape
            if self._block is not None:
                pin = self._engine.pinned(self._block.numel())
                pin.copy_(self._block, non_blocking=True)
                torch.cuda.current_stream(self._block.device).synchronize()
                buf = pin.numpy().copy()
                self._host = {"visit_counts": buf[:B * A].reshape(B, A), "root_values": buf[B * A:B * A + B].view(np.float32),
                              "error": int(buf[B * A + B])}
            else:
                self._host = {"visit_counts": self.visit_counts.cpu().numpy(), "root_values": self.root_values.cpu().numpy(),
                              "error": int(self.error.item()) if self.error is not None else 0}
        return self._host

    def raise_if_failed(self):
        """Synchronises on the read-out and raises what the reference would have raised inside ``run``
        (np.random.choice's ValueError on a NaN / all-zero policy, monte_carlo_tree_search.py:208/:294)."""
        if self.error is not None:
            self._engine.raise_for_error(self.host()["error"])
        return self

    def gumbel(self):
        """Read-out of a Gumbel search (``Monte_carlo_tree_search(..., gumbel=True)``): dict(actions int32[B] — the
        action to play, improved_policy float64[B, A] — the policy target, 0 for illegal actions)."""
        out = self._live().read_gumbel()
        return {"actions": out["actions"], "improved_policy": out["improved_policy"]}

    def select_actions(self, temperature: float = 0.0, uniforms=None):
        """Batched Game.policy_step / store_search_statistics (game.py:179-235) on the device:
        dict(actions, policy, stored_policy); root values are `self.root_values`."""
        return self._live().select_actions(temperature, uniforms)

    def __getitem__(self, i) -> Node:
        return _node_tree(self._live().export_tree(int(i)), self._hidden_fetcher(int(i)))

    @property
    def roots(self):
        return self

    def _hidden_fetcher(self, tree):
        eng = self._engine
        if eng.net == "external":
            return None
        A, kmax = eng.A, eng.dims.max_children

        def fetch(node_index, _ar={}):
            self._live()
            if "cb" not in _ar:
                _ar["cb"] = eng.export_arena(tree)["child_base"]
            cb = int(_ar["cb"][node_index])
            slot = 0 if cb == 1 else (cb - 1 - A) // kmax + 1
            return eng.read_hidden(slot)[tree:tree + 1].cpu()
        return fetch


class Monte_carlo_tree_search():
    def __init__(self,
                 pb_c_base=19652,
                 pb_c_init=1.25,
                 discount=0.95,
                 root_dirichlet_alpha=0.25,
                 root_exploration_fraction=0.25,
                 num_simulations=10,
                 maxium_action_sample=2,
                 number_of_player=1,
                 custom_loop=None,
                 *, net="tc32", device=None, seed=None, max_batch=None, tree_id_offset=None, paper_alternation=False,
                 gumbel=False, max_considered_actions=16, c_visit=50.0, c_scale=0.1):
        """Same nine arguments as the reference (:76-85).  Keyword-only extras: ``net`` — the fused MLP network step:
        "tc32" (default: the reference's fp32 precision on the tensor cores, fp16 hi/lo split operands, 1e-5 against the
        reference's inference), "fp32" (the same precision on CUDA cores), "bf16" / "f16" (throughput modes with
        stated tolerances); ``device`` (CUDA ordinal), ``seed``
        (Philox key; default drawn from numpy's global RNG so ``np.random.seed`` reproduces runs),
        ``max_batch`` (arena capacity reserved for ``run_batch``), ``tree_id_offset`` (global id of local tree 0:
        the Philox streams are keyed by (seed, global tree id), so ranks of a sharded self-play that seed
        numpy identically still draw different noise; default rank * max_batch when torch.distributed is
        initialised, else 0), ``paper_alternation`` (search with the Stochastic MuZero node alternation — decision,
        chance, decision, ... from the root, so afterstate_dynamics sees states and dynamics sees afterstates —
        instead of the reference's depth pattern F,F,T,T,...; default off: the reference's search), ``gumbel`` (search
        with Gumbel MuZero — Gumbel-Top-k and Sequential Halving at the root, completed-Q selection below — instead of
        pUCT with Dirichlet noise, with ``max_considered_actions`` / ``c_visit`` / ``c_scale``; read its action and
        policy target with ``BatchedRoots.gumbel()``; default off: the reference's search)."""
        self._net, self._device, self._seed, self._max_batch = net, device, seed, max_batch
        self._paper = bool(paper_alternation)
        self.gumbel = bool(gumbel)
        self.max_considered_actions, self.c_visit, self.c_scale = int(max_considered_actions), float(c_visit), float(c_scale)
        if not 1 <= self.max_considered_actions <= 32 or not (0 <= self.c_visit < float("inf")) or \
                not (0 <= self.c_scale < float("inf")):
            raise ValueError("max_considered_actions must be in [1, 32], c_visit and c_scale finite and >= 0")
        self._tree_id_offset = tree_id_offset
        self._engines = {}
        self._weights_seen = {}
        self._per_model, self._pinned = weakref.WeakKeyDictionary(), {}
        self._run_counter = 0
        self.reset(pb_c_base, pb_c_init, discount, root_dirichlet_alpha, root_exploration_fraction,
                   num_simulations, maxium_action_sample, number_of_player, custom_loop)

    def reset(self, pb_c_base=19652, pb_c_init=1.25, discount=0.95, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=10, maxium_action_sample=2, number_of_player=1,
              custom_loop=None):
        # argument checks and messages of the reference (:148-173)
        assert isinstance(pb_c_base, int) and pb_c_base >= 1, "pb_c_base ∈ int | {1 < pb_c_base < +inf)"
        assert isinstance(pb_c_init, float) and pb_c_init >= 0, "pb_c_init ∈ float | {0 < pb_c_init < +inf)"
        assert isinstance(discount, (int, float)) and discount >= 0, "discount ∈ float | {0 < discount < +inf)"
        assert isinstance(root_dirichlet_alpha, float) and 0 <= root_dirichlet_alpha <= 1, \
            "root_dirichlet_alpha ∈ float | {0< root_dirichlet_alpha < 1)"
        assert isinstance(root_exploration_fraction, float) and 0 <= root_exploration_fraction <= 1, \
            "root_exploration_fraction ∈ float | {0 < root_exploration_fraction < 1)"
        assert isinstance(maxium_action_sample, int) and maxium_action_sample >= 1, \
            "maxium_action_sample ∈ int | {1 < maxium_action_sample < +inf)"
        assert isinstance(num_simulations, int) and num_simulations >= 0, \
            "num_simulations ∈ int | {0 < num_simulations < +inf)"
        assert isinstance(number_of_player, int) and number_of_player >= 1, \
            "number_of_player ∈ int | {1 < number_of_player < +inf)"
        assert isinstance(custom_loop, str) or custom_loop is None, "custom_loop ∈ str | 1>2>3>3 "
        self.pb_c_base, self.pb_c_init, self.discount = pb_c_base, pb_c_init, discount
        self.root_dirichlet_alpha, self.root_exploration_fraction = root_dirichlet_alpha, root_exploration_fraction
        self.maxium_action_sample, self.num_simulations = maxium_action_sample, num_simulations
        self.number_of_player, self.custom_loop = number_of_player, custom_loop
        self.node = None
        self.model = None
        self.root = None
        self.min_max_stats = MinMaxStats()
        self.cycle = Player_cycle(number_of_player=number_of_player, custom_loop=custom_loop)
        for eng in self._engines.values():
            eng.close()
        self._engines = {}

    # ------------------------------------------------------------------------------------------
    def search_config(self):
        return dict(pb_c_base=self.pb_c_base, pb_c_init=self.pb_c_init, discount=self.discount,
                    root_dirichlet_alpha=self.root_dirichlet_alpha,
                    root_exploration_fraction=self.root_exploration_fraction,
                    num_simulations=self.num_simulations, maxium_action_sample=self.maxium_action_sample,
                    number_of_player=self.number_of_player, custom_loop=self.custom_loop)

    @classmethod
    def from_config(cls, config: dict, **extras):
        """Build from the JSON section "monte_carlo_tree_search" (self_play.py:639-647), verbatim."""
        section = config.get("monte_carlo_tree_search", config)
        keys = ("pb_c_base", "pb_c_init", "discount", "root_dirichlet_alpha", "root_exploration_fraction",
                "num_simulations", "maxium_action_sample", "number_of_player", "custom_loop")
        opts = {k: section[k] for k in ("gumbel", "max_considered_actions", "c_visit", "c_scale") if k in section}
        return cls(**{k: section[k] for k in keys if k in section}, **{**opts, **extras})

    def _base_seed(self):
        if self._seed is None:
            self._seed = int(np.random.randint(0, 2 ** 31 - 1))
        return self._seed

    def _engine(self, kind, batch, action_dim, chance_dim, shape=None):
        cap = max(batch, self._max_batch or 1)
        key = (kind, action_dim, chance_dim, shape)
        eng = self._engines.get(key)
        if eng is None or eng.max_trees < batch:
            if eng is not None:
                eng.close()
            eng = SearchEngine(self.search_config(), action_dim, chance_dim, max_trees=cap, model_shape=shape,
                               net=kind, rng="philox", seed=self._base_seed(), device=self._device,
                               paper_alternation=self._paper)
            self._engines[key] = eng
            self._weights_seen.pop(key, None)
        if self.gumbel or eng.gumbel:      # host-side setting, applied by the next root step
            eng.set_search(self.gumbel, self.max_considered_actions, self.c_visit, self.c_scale)
        return eng, key

    @staticmethod
    def _is_fusable(model):
        if isinstance(model, PackedModel):
            return True
        return getattr(model, "model_structure", None) in ("mlp_model", "vision_model") and all(
            hasattr(model, f"{n}_function") for n in ("representation", "prediction", "afterstate_prediction",
                                                      "afterstate_dynamics", "dynamics", "encoder"))

    def _model_cache(self, model) -> dict:
        """Per-model scratch (packed vision blob, torch back-end), dropped with the model: keyed by a weak reference,
        not by id() — an id can be reused by another object after garbage collection."""
        try:
            return self._per_model.setdefault(model, {})
        except TypeError:                    # not weak-referenceable / unhashable: pin it, so its id stays its own
            return self._pinned.setdefault(id(model), (model, {}))[1]

    def _next_seed(self):
        self._run_counter += 1
        return (self._base_seed() + 0x9E3779B97F4A7C15 * self._run_counter) & 0xFFFFFFFFFFFFFFFF

    def _offset(self, batch):
        """Global id of local tree 0 (see ``tree_id_offset`` in __init__)."""
        if self._tree_id_offset is not None:
            return int(self._tree_id_offset)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank() * max(int(batch), self._max_batch or 1)
        return 0

    # engines hold ctypes handles and device memory: copies / pickles (the reference ships the search object to ray
    # workers, self_play.py:240-256) carry the configuration only and rebuild their engines lazily
    def __getstate__(self):
        state = dict(self.__dict__)
        state["_engines"], state["_weights_seen"] = {}, {}
        state["_pinned"] = {}
        del state["_per_model"]
        state["root"] = state["node"] = state["model"] = None
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._per_model = weakref.WeakKeyDictionary()

    # ------------------------------------------------------------------------------------------
    def run_batch(self, observations, model=None, train=True, root_to_play=None, check=True, *,
                  legal_actions=None, num_simulations=None, explore=None) -> BatchedRoots:
        """B independent searches in one call.  ``observations``: float tensor/array [B, obs_dim]
        (host or device).  Returns BatchedRoots (device tensors; ``roots[i]`` gives a Node view).
        ``check`` (default): wait for the search and raise if it met a degenerate policy, like the reference's
        np.random.choice does; ``check=False`` returns without synchronising (``roots.raise_if_failed()`` later).
        ``legal_actions``: bool / 0-1 mask [B, A] (host or device): each root searches the legal actions of its
        position only, as the reference's root would with that action space; illegal actions get no child, no visit and
        prior 0, and ``select_actions`` never returns one.  A host mask with an empty row raises ValueError before any
        GPU work; a device mask with an empty row or a bit >= A raises ValueError at the check (that tree is searched
        with every action legal).
        ``num_simulations``: the simulations of each tree — an int <= N, or an int sequence / tensor [B] (host or device)
        — or None for N (the constructor's ``num_simulations``).  A tree with budget n is the search with num_simulations
        = n.  Host budgets run max(budget) simulation steps; a device tensor runs N steps and needs no host
        synchronisation.  ``explore``: bool / 0-1 [B] per-tree root noise (Dirichlet, or Gumbels with ``gumbel``)
        replacing ``train`` for that tree, or None.  Out-of-range host budgets raise ValueError before any GPU work, device
        ones at the check (that tree is searched with N)."""
        if legal_actions is not None:
            legal_actions = legal_rows(legal_actions, len(observations))
        budget, n_sims = _budget_plan(num_simulations, len(observations), self.num_simulations)
        if explore is not None:
            explore = explore_rows(explore, len(observations))
        if not self._is_fusable(model):
            roots = self._run_batch_external(observations, model, train, root_to_play, legal_actions, budget, explore)
            return roots.raise_if_failed() if check else roots
        self.model = model
        vision = getattr(model, "model_structure", None) == "vision_model"
        obs = observations if torch.is_tensor(observations) else torch.as_tensor(np.asarray(observations))
        obs = obs.reshape(obs.shape[0], -1)
        if vision:
            # vision (ResNet-v2) family: fp32 CUDA-core network step, observations [B, 3, 98, 98]
            cache = self._model_cache(model)
            ver = weights_version(model)
            if cache.get("vver") != ver:
                blob, shape = pack_vision_weights(model) if not isinstance(model, PackedModel) else (model.blob, model.shape)
                cache["vshape"], cache["vblob"], cache["vver"] = shape, blob, ver
            shape = cache["vshape"]
            eng, key = self._engine("vision", obs.shape[0], shape.action_dim, shape.action_dim, shape)
            if self._weights_seen.get(key) != ver:
                eng.set_weights(cache["vblob"])
                self._weights_seen[key] = ver
        else:
            shape = shape_of(model)
            eng, key = self._engine(self._net, obs.shape[0], shape.action_dim, shape.chance_dim, shape)
            ver = weights_version(model)
            if self._weights_seen.get(key) != ver:
                blob, _ = pack_weights(model)
                eng.set_weights(blob)
                self._weights_seen[key] = ver
        obs = eng.to_device(obs, torch.float32)      # the observations' host-to-device copy is enqueued first
        eng.set_seed(self._next_seed(), self._offset(obs.shape[0]))
        kw = _root_kw(legal_actions, budget, explore)
        if self.gumbel:
            eng.root_gumbel(obs=obs, root_to_play=root_to_play, train=train, **kw)
        else:
            eng.root(obs=obs, root_to_play=root_to_play, train=train, **kw)
        eng.simulate(n_sims)
        roots = BatchedRoots(eng, eng.read_roots())
        return roots.raise_if_failed() if check else roots

    def _run_batch_external(self, observations, model, train, root_to_play, legal_actions=None, budget=None,
                            explore=None):
        """Any other model family: tree kernels in the engine, network step = five batched device
        functions (batched_model.py) — either supplied directly or built from the six nn.Modules of a
        reference-style Muzero."""
        self.model = model
        if batched_model.is_batched_backend(model):
            backend = model
        elif all(hasattr(model, f"{n}_function") for n in ("representation", "prediction", "afterstate_prediction",
                                                           "afterstate_dynamics", "dynamics")):
            cache = self._model_cache(model)
            ver = weights_version(model)
            if cache.get("backend_ver") != ver:      # the back-end works on its own device copy of the modules
                cache["backend"] = batched_model.ReferenceModuleBackend(
                    model, device=f"cuda:{self._device if self._device is not None else torch.cuda.current_device()}")
                cache["backend_ver"] = ver
            backend = cache["backend"]
        else:
            raise TypeError("run_batch needs a reference-style Muzero or an object with the five batched "
                            "network functions (see batched_model.py)")
        obs = observations if torch.is_tensor(observations) else torch.as_tensor(np.asarray(observations))
        A = int(getattr(backend, "A", 0)) or int(getattr(model, "action_dimension"))
        C = int(getattr(backend, "C", A))
        eng, _ = self._engine("external", obs.shape[0], A, C)
        eng.set_seed(self._next_seed(), self._offset(obs.shape[0]))
        store = batched_model.run_search(eng, backend, obs, self.num_simulations, root_to_play, train, legal_actions,
                                         budget, explore)
        roots = BatchedRoots(eng, eng.read_roots())
        roots.hidden_store = store
        return roots

    def run(self, observation=None, model=None, train=True, *, legal_actions=None, num_simulations=None):
        """One search, reference signature (:311).  Returns the root Node.  ``legal_actions``: the legal actions of the
        position, as a sequence of action indices or a bool mask [A] (see ``run_batch``); ``root.children`` then has
        exactly those keys.  ``num_simulations``: an int <= N, this search's budget (None: N)."""
        if num_simulations is not None:
            if not isinstance(num_simulations, (int, np.integer)) or isinstance(num_simulations, (bool, np.bool_)):
                raise ValueError(f"run's num_simulations is an int, got {num_simulations!r}")
            budget_rows(int(num_simulations), 1, self.num_simulations)
        self.model = model
        to_play = self.cycle.global_step()
        if self._is_fusable(model):
            obs = observation if torch.is_tensor(observation) else torch.as_tensor(np.asarray(observation))
            legal = None
            if legal_actions is not None:
                legal = _legal_row(legal_actions, model.shape.action_dim if isinstance(model, PackedModel)
                                   else int(model.action_dimension))
            batch = self.run_batch(obs.reshape(1, *obs.shape[1:]) if obs.dim() > 1 else obs.reshape(1, -1), model, train,
                                   root_to_play=torch.tensor([to_play], dtype=torch.int32), legal_actions=legal,
                                   num_simulations=num_simulations)
            eng = batch._engine
            dump = eng.export_tree(0)
            self.root = _node_tree(dump, batch._hidden_fetcher(0))
        else:
            self.root = self._run_callback(observation, model, train, to_play, legal_actions, num_simulations)
            return self.root
        self.min_max_stats = MinMaxStats(np.float32(dump["minmax"][0]), np.float32(dump["minmax"][1]))
        self.node = self.root
        return self.root

    def _run_callback(self, observation, model, train, to_play, legal_actions=None, num_simulations=None):
        """Host-model mode: tree kernels on the GPU, the five inference methods called back per
        simulation (:182, :198, :271-286)."""
        h0 = model.representation_function_inference(observation)
        policy, value0 = model.prediction_function_inference(h0)
        policy = np.asarray(policy, dtype=np.float32).reshape(1, -1)
        A = policy.shape[1]
        eng, _ = self._engine("external", 1, A, getattr(model, "chance_dimension", A))
        eng.set_seed(self._next_seed(), self._offset(1))
        legal = None if legal_actions is None else _legal_row(legal_actions, A)
        budget, n_sims = _budget_plan(num_simulations, 1, self.num_simulations)
        kw = _root_kw(legal, budget, None)
        if self.gumbel:
            eng.root_gumbel(root_policy=policy, root_value=np.array([value0], dtype=np.float32).reshape(1),
                            root_to_play=torch.tensor([to_play], dtype=torch.int32), train=train, **kw)
        else:
            eng.root(root_policy=policy, root_to_play=torch.tensor([to_play], dtype=torch.int32), train=train, **kw)
        hidden = {0: h0}
        for sim in range(n_sims):                 # the model is called for the tree's own simulations only
            slot, action, branch = (int(t.item()) for t in eng.select(sim))
            if branch:
                reward, h = model.dynamics_function_inference(hidden[slot], np.int64(action))
                policy, value = model.prediction_function_inference(h)
            else:
                reward = 0.0
                h = model.afterstate_dynamics_function_inference(hidden[slot], np.int64(action))
                policy, value = model.afterstate_prediction_function_inference(h)
            hidden[sim + 1] = h
            eng.expand_backup(sim, np.asarray(policy, dtype=np.float32).reshape(1, -1),
                              np.array([value], dtype=np.float32), np.array([reward], dtype=np.float32))
        eng.raise_for_error(int(eng.read_roots()["error"].item()))
        dump = eng.export_tree(0)
        kmax = eng.dims.max_children
        arena_cb = eng.export_arena(0)["child_base"]

        def fetch(node_index):
            cb = int(arena_cb[node_index])
            return hidden[0 if cb == 1 else (cb - 1 - A) // kmax + 1]
        root = _node_tree(dump, fetch)
        self.min_max_stats = MinMaxStats(np.float32(dump["minmax"][0]), np.float32(dump["minmax"][1]))
        self.node = root
        return root
