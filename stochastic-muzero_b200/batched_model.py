"""Batched model back-ends for `run_batch` when the network step is NOT the fused MLP kernel.

The tree kernels (selection, expansion, backup) always run in the CUDA engine; the network step is then
any object exposing five BATCHED device functions — the batched counterparts of the reference's
`Muzero.*_function_inference` methods (muzero_model.py:802-909):

    representation(obs[B, ...])            -> hidden[B, ...]
    prediction(hidden)                     -> (policy[B, A] softmaxed, value[B])
    afterstate_dynamics(hidden, action[B]) -> hidden
    afterstate_prediction(hidden)          -> (policy[B, C] softmaxed, value[B])
    dynamics(hidden, code[B])              -> (reward[B], hidden)

`ReferenceModuleBackend` builds those five from the six `nn.Module`s of a reference-style `Muzero` of ANY
model family (lstm / transformer / vision ...), evaluated in batch on the GPU by torch, with the facade
arithmetic of muzero_model.py re-stated in torch: one-hot action (:496-523; a constant plane (a+1)/A for
vision models), softmax on the policy head (:837), inverse_transform_with_support (:575-591).
"""
from __future__ import annotations

import copy

import torch


def support_to_scalar(logits: torch.Tensor) -> torch.Tensor:
    """muzero_model.py:575-591 for a batch of rows."""
    S = logits.shape[1]
    half = S // 2
    rem = int(2 * ((S / 2) - half))
    support = torch.arange(-half, half + rem, device=logits.device, dtype=logits.dtype)
    y = (torch.softmax(logits, dim=1) * support).sum(dim=1)
    return torch.sign(y) * (((torch.sqrt(1 + 4 * 0.001 * (torch.abs(y) + 1 + 0.001)) - 1) / (2 * 0.001)) ** 2 - 1)


class ReferenceModuleBackend:
    def __init__(self, model, device="cuda"):
        self.device = torch.device(device)
        self.A = int(model.action_dimension)
        self.is_rgb = bool(getattr(model, "is_RGB", False))
        mods = {}
        for name in ("representation", "prediction", "afterstate_dynamics", "afterstate_prediction", "dynamics"):
            m = getattr(model, f"{name}_function")
            m = m.module if m.__class__.__name__ == "DataParallel" else m
            # a private copy: the caller's modules keep their device, dtype and train/eval mode (the trainer still
            # owns them); the search object rebuilds this back-end whenever weights_version(model) changes
            mods[name] = copy.deepcopy(m).to(self.device).float().eval()
        self.m = mods

    def _onehot(self, idx, like):
        idx = idx.to(self.device).long()
        if self.is_rgb:      # muzero_model.py:511-522: a constant plane (a+1)/A of the state's spatial shape
            plane = ((idx.float() + 1) / self.A).view(-1, 1, 1, 1)
            return plane.expand(-1, 1, like.shape[2], like.shape[3])
        return torch.nn.functional.one_hot(idx, num_classes=self.A).float()

    @torch.no_grad()
    def representation(self, obs):
        return self.m["representation"](obs.to(self.device).float())

    @torch.no_grad()
    def prediction(self, h):
        p, v = self.m["prediction"](h)
        return torch.softmax(p.float(), dim=-1), support_to_scalar(v.float())

    @torch.no_grad()
    def afterstate_prediction(self, h):
        p, v = self.m["afterstate_prediction"](h)
        return torch.softmax(p.float(), dim=-1), support_to_scalar(v.float())

    @torch.no_grad()
    def afterstate_dynamics(self, h, action):
        return self.m["afterstate_dynamics"](h, self._onehot(action, h))

    @torch.no_grad()
    def dynamics(self, h, code):
        r, nh = self.m["dynamics"](h, self._onehot(code, h))
        return support_to_scalar(r.float()), nh


BATCHED_METHODS = ("representation", "prediction", "afterstate_dynamics", "afterstate_prediction", "dynamics")


def is_batched_backend(model) -> bool:
    return all(callable(getattr(model, n, None)) for n in BATCHED_METHODS)


def run_search(engine, backend, observations, n_sims, root_to_play=None, train=True, legal=None, budget=None,
               explore=None):
    """Drive one batched search with an external batched network: the engine's select / expand_backup
    hooks around torch calls.  ``legal``: optional legal-action mask [B, A] of the roots (SearchEngine.root);
    ``budget`` / ``explore``: optional per-tree simulation budgets and exploration flags (SearchEngine.root): the search
    runs max(budget) simulations, and a tree without simulation s (select's parent slot -1) is not sent to the model.
    Returns the hidden-state store [N+1, B, ...] (slot-major like the arena's)."""
    dev = torch.device("cuda", engine.device)
    h0 = backend.representation(observations)
    B = h0.shape[0]
    policy, value = backend.prediction(h0)
    store = torch.zeros((n_sims + 1,) + tuple(h0.shape), dtype=h0.dtype, device=dev)
    store[0] = h0
    kw = {} if legal is None else {"legal": legal}
    if budget is not None:
        kw["budget"] = budget
        n_sims = min(n_sims, int(budget.max()) if budget.numel() else 0)     # one host read per search
    if explore is not None:
        kw["explore"] = explore
    if engine.gumbel:          # the Gumbel search completes Q-values with each node's network value, the root's too
        engine.root_gumbel(root_policy=policy.float(), root_value=value.float().reshape(-1), root_to_play=root_to_play,
                           train=train, **kw)
    else:
        engine.root(root_policy=policy.float(), root_to_play=root_to_play, train=train, **kw)
    W = engine.dims.policy_stride
    rows = torch.arange(B, device=dev)
    for sim in range(n_sims):
        slot, action, branch = engine.select(sim)
        live = slot >= 0                           # trees whose budget is used up take no part in this simulation
        parent = store[slot.long().clamp(min=0), rows]
        is_dyn = branch.bool()
        pol = torch.zeros(B, W, dtype=torch.float32, device=dev)
        val = torch.zeros(B, dtype=torch.float32, device=dev)
        rew = torch.zeros(B, dtype=torch.float32, device=dev)
        i_a, i_d = (live & ~is_dyn).nonzero(as_tuple=True)[0], (live & is_dyn).nonzero(as_tuple=True)[0]
        if i_a.numel():
            h = backend.afterstate_dynamics(parent[i_a], action[i_a])
            p, v = backend.afterstate_prediction(h)
            store[sim + 1, i_a] = h
            pol[i_a, :p.shape[1]], val[i_a] = p.float(), v.float()
        if i_d.numel():
            r, h = backend.dynamics(parent[i_d], action[i_d])
            p, v = backend.prediction(h)
            store[sim + 1, i_d] = h
            pol[i_d, :p.shape[1]], val[i_d], rew[i_d] = p.float(), v.float(), r.float()
        engine.expand_backup(sim, pol, val, rew)
    return store
