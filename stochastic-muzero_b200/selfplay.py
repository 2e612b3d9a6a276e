"""Batched self-play driver: thousands of games advance one move per `run_batch` call with no host
round-trip inside a move (SURVEY.md §8f-2).  It replaces the reference's per-game loop
(self_play.py:63-98: observation -> mcts.run -> Game.policy_step -> Game.store_search_statistics) and its
`ray` fan-out of whole games (self_play.py:240-256) by B concurrent games stepped in lock-step on the device:

    obs[B] -> Monte_carlo_tree_search.run_batch -> BatchedRoots.select_actions(temperature) -> env.step

with done-masking and automatic reset of finished games (every move starts a fresh search, so a finished
game's arena slot is recycled by the next root step).  What the trainer needs (observations, actions,
rewards, stored visit policies, root values — Game.store_search_statistics / make_target inputs,
game.py:179-204, :291-337) is written into preallocated device tensors [T, B, ...].

The environment is any object with `reset(mask) -> obs[B, ...]` and
`step(action[B]) -> (obs, reward[B], done[B])` on the device; one that also has `legal_mask() -> bool[B, A]` gets
each search restricted to the legal actions of its position.  `VectorCartPole` is the synthetic vector
environment used here: CartPole-v1's published equations of motion (Barto, Sutton & Anderson 1983, as used by
gymnasium's cartpole.py: gravity 9.8, cart 1.0 kg, pole 0.1 kg, half-length 0.5 m, force 10 N, tau 0.02 s,
Euler integration, termination at |x| > 2.4 or |theta| > 12 degrees, reward 1 per step, 500-step limit),
restated for B environments as element-wise torch ops.  The reference drives gymnasium environments on the
CPU; gymnasium is not part of this build (parity of the environment itself is not claimed).
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch


class VectorCartPole:
    GRAVITY, MASSCART, MASSPOLE, LENGTH, FORCE, TAU = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02
    X_LIMIT, THETA_LIMIT, STEP_LIMIT = 2.4, 12 * 2 * math.pi / 360, 500

    def __init__(self, n_envs: int, device="cuda", seed: int = 0):
        self.n, self.device = n_envs, torch.device(device)
        self.gen = torch.Generator(device=self.device).manual_seed(seed)
        self.state = torch.zeros(n_envs, 4, device=self.device)
        self.steps = torch.zeros(n_envs, dtype=torch.int32, device=self.device)
        self.reset()

    @property
    def action_dim(self):
        return 2

    def reset(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        fresh = torch.rand(self.n, 4, device=self.device, generator=self.gen) * 0.1 - 0.05
        if mask is None:
            self.state, self.steps = fresh, torch.zeros_like(self.steps)
        else:
            self.state = torch.where(mask[:, None], fresh, self.state)
            self.steps = torch.where(mask, torch.zeros_like(self.steps), self.steps)
        return self.state

    def step(self, action: torch.Tensor):
        x, x_dot, th, th_dot = self.state.unbind(1)
        force = torch.where(action.to(self.device) == 1, self.FORCE, -self.FORCE)
        cos, sin = torch.cos(th), torch.sin(th)
        total_mass, pml = self.MASSCART + self.MASSPOLE, self.MASSPOLE * self.LENGTH
        temp = (force + pml * th_dot ** 2 * sin) / total_mass
        th_acc = (self.GRAVITY * sin - cos * temp) / (self.LENGTH * (4.0 / 3.0 - self.MASSPOLE * cos ** 2 / total_mass))
        x_acc = temp - pml * th_acc * cos / total_mass
        self.state = torch.stack([x + self.TAU * x_dot, x_dot + self.TAU * x_acc,
                                  th + self.TAU * th_dot, th_dot + self.TAU * th_acc], 1)
        self.steps = self.steps + 1
        terminated = (self.state[:, 0].abs() > self.X_LIMIT) | (self.state[:, 2].abs() > self.THETA_LIMIT)
        done = terminated | (self.steps >= self.STEP_LIMIT)
        reward = torch.ones(self.n, device=self.device)
        return self.state, reward, done


class SelfPlay:
    """Lock-step self-play of B games for T moves; trajectories stay on the device.

    ``playout_cap=(p_full, n_fast)``: playout-cap randomisation (Wu 2019, "Accelerating Self-Play Learning in Go"; used
    by KataGo).  Every move of every game draws, from a generator seeded with ``seed``, a full search (the search's N
    simulations, root noise as ``train`` says) with probability p_full, else a fast search of n_fast simulations.  With
    pUCT the fast search has no Dirichlet noise; with Gumbel it keeps its Gumbels, which are how Gumbel picks the move.
    The buffer's ``full_search`` [T, B] marks the full searches, whose policy targets a trainer keeps.  None: every move
    is a full search and the buffer is as without the option."""

    def __init__(self, mcts, model, env, horizon: int, playout_cap=None, seed: int = 0):
        self.mcts, self.model, self.env, self.T = mcts, model, env, horizon
        if playout_cap is not None:
            p_full, n_fast = playout_cap
            if not 0.0 <= float(p_full) <= 1.0:
                raise ValueError(f"playout_cap's p_full must be in [0, 1], got {p_full}")
            if isinstance(n_fast, bool) or not isinstance(n_fast, (int,)) or not 0 <= n_fast <= mcts.num_simulations:
                raise ValueError(f"playout_cap's n_fast must be an int in [0, {mcts.num_simulations}], got {n_fast!r}")
            playout_cap = (float(p_full), int(n_fast))
        self.playout_cap, self.seed = playout_cap, int(seed)

    @torch.no_grad()
    def run(self, temperature: float = 1.0, train: bool = True) -> Dict[str, torch.Tensor]:
        env, T = self.env, self.T
        obs = env.reset()
        B, dev = obs.shape[0], obs.device
        A = env.action_dim
        buf = {"observations": torch.zeros((T, B) + tuple(obs.shape[1:]), device=dev),
               "actions": torch.zeros(T, B, dtype=torch.int32, device=dev),
               "rewards": torch.zeros(T, B, device=dev), "dones": torch.zeros(T, B, dtype=torch.bool, device=dev),
               "child_visits": torch.zeros(T, B, A, dtype=torch.float64, device=dev),
               "root_values": torch.zeros(T, B, device=dev)}
        gumbel = getattr(self.mcts, "gumbel", False)
        if self.playout_cap is not None:
            buf["full_search"] = torch.zeros(T, B, dtype=torch.bool, device=dev)
            gen = torch.Generator(device=dev).manual_seed(self.seed)
            N, (p_full, n_fast) = self.mcts.num_simulations, self.playout_cap
        for t in range(T):
            legal = env.legal_mask() if hasattr(env, "legal_mask") else None
            cap = {}
            if self.playout_cap is not None:       # budgets and flags stay on the device: no host round-trip per move
                full = torch.rand(B, device=dev, generator=gen) < p_full
                buf["full_search"][t] = full
                cap["num_simulations"] = torch.where(full, N, n_fast).to(torch.int32)
                if not gumbel:
                    cap["explore"] = full & bool(train)
            roots = self.mcts.run_batch(obs, self.model, train=train, legal_actions=legal, **cap)   # one move of every game
            if gumbel:                                   # Gumbel search: its action, its improved policy as the target
                g = roots.gumbel()
                pick = {"actions": g["actions"], "stored_policy": g["improved_policy"]}
            else:
                pick = roots.select_actions(temperature)                            # game.py:223-235 on the device
            buf["observations"][t], buf["actions"][t] = obs, pick["actions"]
            buf["child_visits"][t], buf["root_values"][t] = pick["stored_policy"], roots.root_values
            obs, reward, done = env.step(pick["actions"])
            buf["rewards"][t], buf["dones"][t] = reward, done
            obs = env.reset(done)                                                   # finished games restart
        return buf


@torch.no_grad()
def reanalyse(mcts, model, observations: torch.Tensor, chunk: int = 16384, train: bool = True,
              legal_actions: Optional[torch.Tensor] = None, num_simulations=None) -> Dict[str, torch.Tensor]:
    """Reanalyse (self_play.py:30-44, game.py:112-116, replay_buffer.py:229-266): re-run the search over stored
    observations of old games with the current weights.  Every stored position is an independent tree, so
    the [T, B, ...] trajectory block is simply flattened into large batches for the engine.
    ``legal_actions``: optional bool mask [T, B, A] of the stored positions' legal actions.
    ``num_simulations``: an int, or an int [T, B] tensor / array giving each stored position its own budget (older or less
    valuable data may get fewer simulations), or None for the search's N.
    Returns fresh targets: child_visits [T, B, A] (stored visit policy; the improved policy of a Gumbel search) and
    root_values [T, B]."""
    T, B = observations.shape[:2]
    flat = observations.reshape((T * B,) + tuple(observations.shape[2:]))
    legal = None if legal_actions is None else legal_actions.reshape(T * B, -1)
    budget = num_simulations
    if budget is not None and not isinstance(budget, int):
        budget = budget if torch.is_tensor(budget) else torch.as_tensor(budget)
        if tuple(budget.shape) != (T, B):
            raise ValueError(f"reanalyse's num_simulations must be an int or have shape [{T}, {B}], got "
                             f"{list(budget.shape)}")
        budget = budget.reshape(T * B)
    visits, values = [], []
    for lo in range(0, T * B, chunk):
        roots = mcts.run_batch(flat[lo:lo + chunk], model, train=train,
                               legal_actions=None if legal is None else legal[lo:lo + chunk],
                               num_simulations=budget if budget is None or isinstance(budget, int)
                               else budget[lo:lo + chunk])
        if getattr(mcts, "gumbel", False):         # the Gumbel search's policy target
            visits.append(roots.gumbel()["improved_policy"])
        else:
            visits.append(roots.select_actions(0.0)["stored_policy"])
        values.append(roots.root_values.clone())
    child_visits = torch.cat(visits)
    return {"child_visits": child_visits.reshape(T, B, -1), "root_values": torch.cat(values).reshape(T, B)}
