"""Cost of per-tree simulation budgets (smz_set_root_budgets): whole searches (root step + simulations), bf16 network
step, at BASELINE cfg2 (4096 trees x 50 simulations, A = C = K = 2) and cfg4 (65536 trees, same model), CUDA events
around each search after warm-up searches of the same shape, sides alternated round by round in one process.

  - default path: no budgets, against the same search with all-N budgets (the budgeted tree kernels), and with
    --parent-lib against the default search of a libsmz.so built at an earlier commit;
  - playout-cap mix: 25 % of the trees with 50 simulations, 75 % with 10 (budgets on the device, 50 steps), against
    uniform 50 and uniform 10 (10 steps).  "sims run/s" counts the simulations the trees actually ran (sum of budgets).

Prints one line per measurement and writes them to --out.

    python tools/bench_budgets.py [--reps 10] [--rounds 4] [--parent-lib PARENT/libsmz.so] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_gumbel import SEARCH, load_other  # noqa: E402
from stochastic_muzero_b200 import ModelShape, SearchEngine, _lib  # noqa: E402
from stochastic_muzero_b200.weights import random_blob  # noqa: E402

WORKLOADS = {"cfg2": 4096, "cfg4": 65536}     # trees; 50 simulations, obs 4, A = C = K = 2


class Runner:
    """One engine, one search shape: budgets None (no budgets), or an int32 device tensor; `steps` simulation steps."""

    def __init__(self, B, budgets, steps, lib=None):
        N = 50
        self.B, self.steps = B, steps
        shape = ModelShape(4, 2, 2, 61, 126, 4)
        saved = _lib._lib
        if lib is not None:           # SearchEngine binds _lib.load(): hand it the other library for its lifetime
            _lib._lib = lib
        try:
            self.eng = SearchEngine(dict(SEARCH, num_simulations=N, maxium_action_sample=2), 2, 2, max_trees=B,
                                    model_shape=shape, net="bf16", rng="philox", seed=1)
        finally:
            _lib._lib = saved
        self.eng.set_weights(random_blob(shape, seed=0))
        self.budgets = budgets
        self.sims = B * N if budgets is None else int(budgets.sum())
        self.x = torch.randn(B, 4, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
        for _ in range(2):            # the first searches capture the graph and warm up
            self.search()
        torch.cuda.synchronize()

    def search(self):
        if self.budgets is None:
            self.eng.root(obs=self.x, train=True)
        else:
            self.eng.root(obs=self.x, train=True, budget=self.budgets)
        self.eng.simulate(self.steps)

    def time(self, reps):
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.search()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return np.array(ts)


def line(label, r, t):
    return (f"{label:36s} {r.B:6d} trees {r.steps:3d} steps  {np.median(t):8.3f} ms [{t.min():.3f}, {t.max():.3f}]  "
            f"{r.sims / (np.median(t) * 1e-3) / 1e6:8.2f} M sims run/s")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_budgets.py measures on the GPU"
    gpu = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                          "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    lines = [f"# GPU: {gpu} (name, power limit, max SM clock); median [min, max] of {args.reps} searches per round"]
    print(lines[0], flush=True)
    parent = load_other(args.parent_lib) if args.parent_lib else None
    for wl, B in WORKLOADS.items():
        dev = lambda v: torch.as_tensor(v, dtype=torch.int32, device="cuda")   # noqa: E731
        full = np.random.default_rng(0).random(B) < 0.25
        runners = {"default (no budgets)": Runner(B, None, 50), "all-N budgets": Runner(B, dev(np.full(B, 50)), 50)}
        if parent is not None:
            runners["parent default"] = Runner(B, None, 50, parent)
        runners["uniform 50"] = Runner(B, dev(np.full(B, 50)), 50)
        runners["mix 25% x 50 / 75% x 10"] = Runner(B, dev(np.where(full, 50, 10)), 50)
        runners["uniform 10"] = Runner(B, dev(np.full(B, 10)), 10)
        for rnd in range(args.rounds):        # the order is reversed every other round: no side always runs first
            for name, r in (list(runners.items()) if rnd % 2 == 0 else list(runners.items())[::-1]):
                lines.append(line(f"{wl} {name} round {rnd + 1}", r, r.time(args.reps)))
                print(lines[-1], flush=True)
        for r in runners.values():
            r.eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
