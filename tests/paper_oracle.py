"""TEST INFRASTRUCTURE — CPU oracle of the search under the Stochastic MuZero node alternation (`paper_alternation`).

`oracle/mcts_oracle.search` restates the reference's search, whose node kinds go F,F,T,T,... by depth (SURVEY.md §8a
T2).  `search` below is the same search with the alternation the Stochastic MuZero recurrence is written for: a node at
depth d is a chance node iff d & 1, so the root's children are afterstates, afterstate_dynamics receives states and
dynamics receives afterstates.  Everything else is the reference's rule, through the primitives of mcts_oracle (same
casts, same draw order):
  * leaf evaluation: afterstate pair iff the leaf's parent is a decision node, else the dynamics pair (which stores the
    leaf's reward); the new children are chosen from that head's policy, min(K, width) of them;
  * selection: pUCT at decision nodes (one uniform per child), smoothed-prior sampling at chance nodes (one uniform);
  * to_play: a chance child keeps its parent's player, a decision child gets the next one — the root's children too;
  * backup: value = reward + discount * value at every node of the path, float32.
"""
from typing import Optional

import numpy as np

from oracle import mcts_oracle as O

f32, f64 = np.float32, np.float64


def is_chance(depth: int) -> bool:
    """The paper alternation: decision, chance, decision, ... from the root."""
    return bool(depth & 1)


def reference_is_chance(depth: int) -> bool:
    """The reference's pattern F,F,T,T,... (T2): with it, `search` must reproduce mcts_oracle.search and the golden
    tapes of the reference, which pins this restatement (tests/test_node_pattern.py)."""
    return bool((depth >> 1) & 1)


def search(cfg: O.SearchConfig, model, rng, train: bool = True, dirichlet: Optional[np.ndarray] = None,
           root_to_play: int = 0, dirichlet_fn=None, kind=is_chance) -> O.Tree:
    """mcts_oracle.search with node kinds by depth from `kind` (default: the paper alternation); same arguments and
    result."""
    cycle = cfg.cycle_map()
    n_cycle = len(cycle)

    def next_player(p):
        return (p + 1) % n_cycle

    def in_play(p):
        return cycle[p % n_cycle]

    def child_to_play(depth, parent_to_play):
        return parent_to_play if kind(depth) else next_player(parent_to_play)

    tree = O.Tree()
    root = tree.add(prior=0, key=-1, depth=0, is_chance=False, to_play=root_to_play)
    hidden, policy, _root_value = model.root()
    tree.hidden[root] = hidden

    p = O.normalise_policy(policy)
    n = p.shape[0]
    for i in sorted(O.choice_without_replacement(n, n, p, rng)):
        c = tree.add(prior=p[i], key=i, depth=1, is_chance=kind(1), to_play=child_to_play(1, root_to_play))
        tree.children[root].append(c)

    if cfg.num_simulations == 0:
        train = False
    if train:
        noise = np.asarray(dirichlet if dirichlet is not None else dirichlet_fn(n), dtype=np.float64)
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
