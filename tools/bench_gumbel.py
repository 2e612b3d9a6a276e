"""Cost of the Gumbel MuZero search: whole searches (root step + simulations) with the default pUCT search and with the
Gumbel search (`smz_set_search(SMZ_SEARCH_GUMBEL)`, m = 16, c_visit 50, c_scale 0.1), alternated, at BASELINE cfg2
(4096 trees x 50 simulations, A = C = K = 2), cfg4 (65536 trees x 50 simulations, same model) and the cfg3 shape
(8192 trees x 100 simulations, A 4 / C 32 / K 32), bf16 network step.  CUDA events around each search, after warm-up
searches of the same shape; the mean leaf depth comes from smz_stats.  The two rules visit different trees, so the
rate difference includes the difference in tree shape.

With --parent-lib (a libsmz.so built at an earlier commit), the default search of that library is timed in the same
process, alternated with this tree's default search, at cfg2 and cfg4: an A/B of the default path with its spread.
Prints one line per measurement and writes them to --out.

    python tools/bench_gumbel.py [--reps 10] [--rounds 4] [--parent-lib PARENT/libsmz.so] [--out FILE]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from stochastic_muzero_b200 import ModelShape, SearchEngine, _lib  # noqa: E402
from stochastic_muzero_b200.weights import random_blob  # noqa: E402

SEARCH = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, number_of_player=1, custom_loop=None)
WORKLOADS = {  # name: (trees, simulations, obs, A, C, K)
    "cfg2": (4096, 50, 4, 2, 2, 2),
    "cfg4": (65536, 50, 4, 2, 2, 2),
    "cfg3": (8192, 100, 16, 4, 32, 32),
}


def load_other(path):
    """A second libsmz.so in this process (its own kernels and symbols), bound for the entries it exports."""
    lib = C.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SIGNATURES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    return lib


class Runner:
    def __init__(self, wl, gumbel, lib=None):
        B, N, obs, A, C_, K = WORKLOADS[wl]
        self.B, self.N = B, N
        shape = ModelShape(obs, A, C_, 61, 126, 4)
        if lib is not None:           # SearchEngine binds _lib.load(): hand it the other library for its lifetime
            saved = _lib._lib
            _lib._lib = lib
        try:
            self.eng = SearchEngine(dict(SEARCH, num_simulations=N, maxium_action_sample=K), A, C_, max_trees=B,
                                    model_shape=shape, net="bf16", rng="philox", seed=1)
        finally:
            if lib is not None:
                _lib._lib = saved
        self.eng.set_weights(random_blob(shape, seed=0))
        if gumbel:
            self.eng.set_search(True)
        self.gumbel = gumbel
        self.x = torch.randn(B, obs, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
        for _ in range(2):            # the first searches capture the graph and warm up
            self.search()
        torch.cuda.synchronize()

    def search(self):
        (self.eng.root_gumbel if self.gumbel else self.eng.root)(obs=self.x, train=True)
        self.eng.simulate(self.N)

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
    depth = r.eng.stats()["mean_leaf_depth"]
    return (f"{label:34s} {r.B:6d} trees x {r.N:3d} sims  {np.median(t):8.3f} ms [{t.min():.3f}, {t.max():.3f}]  "
            f"{r.B * r.N / (np.median(t) * 1e-3) / 1e6:8.2f} M sims/s  mean leaf depth {depth:.3f}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_gumbel.py measures on the GPU"
    gpu = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                          "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    lines = [f"# GPU: {gpu} (name, power limit, max SM clock); median [min, max] of {args.reps} searches per round"]
    print(lines[0], flush=True)
    parent = load_other(args.parent_lib) if args.parent_lib else None
    for wl in WORKLOADS:
        runners = {"puct": Runner(wl, False), "gumbel": Runner(wl, True)}
        if parent is not None and wl in ("cfg2", "cfg4"):
            runners = {"parent puct": Runner(wl, False, parent), **runners}
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
