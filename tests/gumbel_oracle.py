"""TEST INFRASTRUCTURE — CPU oracle of the Gumbel MuZero search (smz_set_search(SMZ_SEARCH_GUMBEL) in include/smz.h).

`search` is the search of `oracle/mcts_oracle.search`, through that oracle's primitives (same casts, same draw order),
with three options:
  * `kind`: the node kind by depth (tests/paper_oracle.py), the reference's F,F,T,T,... by default;
  * `legal`: the root's action space L (ascending); the root's policy is compacted to policy[L] before normalisation and
    the draws of root expansion, and its children carry the real actions;
  * `gumbel`: a GumbelConfig.  Decision nodes then choose by the Gumbel MuZero rule (Danihelka et al., ICLR 2022) and
    draw no uniform; the root mixes no Dirichlet noise; chance nodes and expansions keep the reference's draws.
With gumbel=None and every action legal it is mcts_oracle.search, which tests/test_gumbel_search.py pins against every
golden tape of the reference.

The decision rule, float64 in the order written, sums in ascending child order:
  v_mix = (v + sum N * (sum_{N_i>0} p_i q_i) / (sum_{N_i>0} p_i)) / (sum N + 1)   (v when sum N = 0)
  cq_i = q_i if N_i > 0 else v_mix;  r_i = (cq_i - min cq) / max(max cq - min cq, 1e-8)
  sigma_i = (c_visit + max N) * c_scale * r_i
  interior: argmax pi'_i - N_i / (1 + sum N), pi'_i = p_i exp(sigma_i - max sigma) / sum_j p_j exp(sigma_j - max sigma)
  root: argmax over {N_a == T[min(m, |L|)][sum N]} of max(-1e9, g_a + logit_a + sigma_a)
Ties go to the smaller action.  q_i = reward + discount * value() in float32 (mcts_oracle.ucb_score's value term before
normalisation), p_i the float64 root prior at the root and the float32 prior below, v the node's own network value.
"""
import dataclasses
import math
from typing import List, Optional

import numpy as np

from oracle import mcts_oracle as O

f32, f64 = np.float32, np.float64


@dataclasses.dataclass
class GumbelConfig:
    max_considered_actions: int = 16
    c_visit: float = 50.0
    c_scale: float = 0.1


def reference_is_chance(depth: int) -> bool:
    return bool((depth >> 1) & 1)


def considered_visits(n: int, N: int) -> List[int]:
    """Sequential Halving's visit schedule for n considered actions and N simulations (the published implementation's
    table, truncated to N entries)."""
    if n <= 1:
        return list(range(N))
    log2max = int(math.ceil(math.log2(n)))
    visits, seq, k = [0] * n, [], n
    while len(seq) < N:
        extra = max(1, int(N / (log2max * k)))
        for _ in range(extra):
            seq.extend(visits[:k])
            for i in range(k):
                visits[i] += 1
        k = max(2, k // 2)
    return seq[:N]


def philox_gumbels(seed: int, tree_id: int, legal, A: int) -> np.ndarray:
    """The engine's device Gumbels of one tree: -log(-log u) of uniform #rank of Philox stream 3 for the legal actions
    in ascending order (u = 0 taken as 2^-53), 0 for illegal actions."""
    g = np.zeros(A)
    for rank, a in enumerate(legal):
        u = O.philox_uniform(seed, tree_id, rank, stream=3)
        u = u if u > 0 else f64(1.0 / 9007199254740992.0)
        g[a] = -np.log(-np.log(u))
    return g


def q_value(cfg, tree, c) -> np.float64:
    return f64(f32(tree.reward[c] + f32(f32(cfg.discount) * tree.value(c))))


def sigma(cfg, gcfg: GumbelConfig, tree, kids, vhat, priors):
    """sigma_i of the completed Q-values over `kids` (priors: float64 p_i), and sum N."""
    n = [tree.visit[c] for c in kids]
    q = [q_value(cfg, tree, c) if tree.visit[c] > 0 else f64(0) for c in kids]
    sn = sum(n)
    spq, sp = f64(0), f64(0)
    for i in range(len(kids)):
        if n[i] > 0:
            spq = f64(spq + f64(priors[i] * q[i]))
            sp = f64(sp + priors[i])
    vmix = f64(vhat) if sn == 0 else f64(f64(f64(vhat) + f64(f64(f64(sn) * spq) / sp)) / f64(sn + 1))
    cq = [q[i] if n[i] > 0 else vmix for i in range(len(kids))]
    lo, hi = min(cq), max(cq)
    rng_ = max(f64(hi - lo), f64(1e-8))
    scale = f64(f64(f64(gcfg.c_visit) + f64(max(n))) * f64(gcfg.c_scale))
    return [f64(scale * f64(f64(c - lo) / rng_)) for c in cq], sn


def root_logits(priors) -> np.ndarray:
    lp = np.log(np.asarray(priors, np.float64))
    return lp - lp.max()


def readout(cfg, gcfg, tree, vhat, gumbels, A):
    """(action, improved_policy[A]) of a finished Gumbel search: argmax over the most-visited legal actions of
    g + logit + sigma; softmax over the legal actions of logit + sigma."""
    kids = tree.children[0]
    keys = [tree.key[c] for c in kids]
    pri = [f64(tree.prior[c]) for c in kids]
    sig, _ = sigma(cfg, gcfg, tree, kids, vhat, pri)
    lg = root_logits(pri)
    mn = max(tree.visit[c] for c in kids)
    best, bs = None, None
    for i, c in enumerate(kids):
        if tree.visit[c] == mn:
            s = f64(f64(f64(gumbels[keys[i]]) + lg[i]) + sig[i])
            if best is None or s > bs:
                best, bs = i, s
    z = [f64(lg[i] + sig[i]) for i in range(len(kids))]
    zm = max(z)
    e = [f64(np.exp(f64(v - zm))) for v in z]
    se = f64(0)
    for v in e:
        se = f64(se + v)
    pol = np.zeros(A)
    for i, k in enumerate(keys):
        pol[k] = f64(e[i] / se)
    return keys[best], pol


def _pick_gumbel(cfg, gcfg, tree, node, kids, vhat, root, gumbels, logits, n_legal):
    pri = [f64(tree.prior[c]) for c in kids]
    sig, sn = sigma(cfg, gcfg, tree, kids, vhat, pri)
    best, bs = None, None
    if root:
        considered = considered_visits(min(gcfg.max_considered_actions, n_legal), cfg.num_simulations)[sn]
        for i, c in enumerate(kids):
            if tree.visit[c] != considered:
                continue
            s = max(f64(-1e9), f64(f64(f64(gumbels[tree.key[c]]) + logits[i]) + sig[i]))
            if best is None or s > bs:
                best, bs = c, s
        return kids[0] if best is None else best
    ms = max(sig)
    w = [f64(pri[i] * f64(np.exp(f64(sig[i] - ms)))) for i in range(len(kids))]
    sw = f64(0)
    for v in w:
        sw = f64(sw + v)
    for i, c in enumerate(kids):
        s = f64(f64(w[i] / sw) - f64(f64(tree.visit[c]) / f64(1 + sn)))
        if best is None or s > bs:
            best, bs = c, s
    return best


def search(cfg: O.SearchConfig, model, rng, train: bool = True, dirichlet: Optional[np.ndarray] = None,
           root_to_play: int = 0, kind=reference_is_chance, legal=None, gumbel: Optional[GumbelConfig] = None,
           gumbels: Optional[np.ndarray] = None) -> O.Tree:
    """One search.  `dirichlet`: noise over the root's (compacted) action space L, pUCT only.  `gumbels`: float64 [A]
    Gumbels by action (Gumbel only; None = 0, as with train=False).  The result's `raw_value` lists every node's network
    value (root: model.root()'s third output)."""
    cycle = cfg.cycle_map()
    n_cycle = len(cycle)

    def next_player(p):
        return (p + 1) % n_cycle

    def in_play(p):
        return cycle[p % n_cycle]

    def child_to_play(depth, parent_to_play):
        return parent_to_play if kind(depth) else next_player(parent_to_play)

    tree = O.Tree()
    tree.raw_value = {}
    root = tree.add(prior=0, key=-1, depth=0, is_chance=False, to_play=root_to_play)
    hidden, policy, root_value = model.root()
    tree.hidden[root] = hidden
    tree.raw_value[root] = f32(root_value)
    policy = np.asarray(policy, np.float32)
    L = list(range(policy.shape[0])) if legal is None else [int(a) for a in legal]

    p = O.normalise_policy(policy[L])
    n = p.shape[0]
    for i in sorted(O.choice_without_replacement(n, n, p, rng)):
        c = tree.add(prior=p[i], key=L[i], depth=1, is_chance=kind(1), to_play=child_to_play(1, root_to_play))
        tree.children[root].append(c)

    logits = None
    if gumbel is not None:
        A = policy.shape[0]
        gumbels = np.zeros(A) if gumbels is None or not train else np.asarray(gumbels, np.float64)
        logits = root_logits([f64(tree.prior[c]) for c in tree.children[root]])
    else:
        if cfg.num_simulations == 0:
            train = False
        if train:
            noise = np.asarray(dirichlet, dtype=np.float64)
            frac = cfg.root_exploration_fraction
            for c, nz in zip(tree.children[root], noise):
                scaled = f32(f32(tree.prior[c]) * f32(1 - frac))
                tree.prior[c] = f64(f64(scaled) + f64(nz) * f64(frac))

    for sim in range(cfg.num_simulations):
        node = root
        path = [root]
        keys = []
        while tree.children[node]:
            kids = tree.children[node]
            if tree.is_chance[node]:
                probs = O.smoothed_chance_probs(np.array([tree.prior[c] for c in kids], dtype=np.float32))
                cdf = O.choice_cdf(probs)
                pick = kids[int(np.searchsorted(cdf, rng.next(), side="right"))]
            elif gumbel is not None:
                pick = _pick_gumbel(cfg, gumbel, tree, node, kids, tree.raw_value[node], node == root, gumbels,
                                    logits, len(L))
            else:
                best = None
                for c in kids:
                    s = O.ucb_score(cfg, tree, node, c, rng.next())
                    if best is None or (s, tree.key[c]) > best[:2]:
                        best = (s, tree.key[c], c)
                pick = best[2]
            node = pick
            keys.append(tree.key[pick])
            path.append(pick)
        tree.paths.append(keys)
        parent = path[-2]

        if tree.is_chance[parent]:
            h, policy, value, reward = model.dynamics(sim, tree.hidden[parent], keys[-1])
            tree.reward[node] = f32(reward)
        else:
            h, policy, value = model.afterstate(sim, tree.hidden[parent], keys[-1])
        tree.hidden[node] = h
        tree.raw_value[node] = f32(value)

        p = O.normalise_policy(policy)
        n = p.shape[0]
        bound = min(cfg.maxium_action_sample, n)
        d = tree.depth[node] + 1
        for i in sorted(O.choice_without_replacement(n, bound, p, rng)):
            c = tree.add(prior=p[i], key=i, depth=d, is_chance=kind(d), to_play=child_to_play(d, tree.to_play[node]))
            tree.children[node].append(c)

        value = f32(value)
        for b in reversed(path):
            same = in_play(tree.to_play[root]) == in_play(tree.to_play[b])
            tree.value_sum[b] = f32(tree.value_sum[b] + (value if same else f32(-value)))
            tree.visit[b] += 1
            nv = tree.value(b)
            tree.vmax = max(tree.vmax, nv)
            tree.vmin = min(tree.vmin, nv)
            value = f32(tree.reward[b] + f32(f32(cfg.discount) * value))
    return tree
