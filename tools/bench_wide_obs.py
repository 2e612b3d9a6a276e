"""Cost of wide observations: the root step (representation + prediction + root expansion) at B = 4096 for several
observation widths in every MLP network mode, and whole searches (4096 trees x 50 simulations, the cfg2 model) at
obs = 376 against obs = 4.  CUDA events around each step; the L2 is overwritten (256 MiB memset) before every timed
step, so the observations and weights come from HBM.  Prints one line per measurement and writes them to --out.

    python tools/bench_wide_obs.py [--reps 20] [--out profiles/wide_obs.txt]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from stochastic_muzero_b200 import ModelShape, SearchEngine  # noqa: E402
from stochastic_muzero_b200.weights import random_blob  # noqa: E402

SEARCH = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, maxium_action_sample=2, number_of_player=1, custom_loop=None)
MODES = ["fp32", "tc32", "f16", "bf16"]
WIDTHS = [4, 128, 376, 1024, 8192]


def timed(fn, reps, flush):
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return np.array(ts)


def engine(net, obs, B, N):
    shape = ModelShape(obs, 2, 2, 61, 126, 4)
    eng = SearchEngine(dict(SEARCH, num_simulations=N), 2, 2, max_trees=B, model_shape=shape, net=net, rng="philox", seed=1)
    eng.set_weights(random_blob(shape, seed=0))
    x = torch.randn(B, obs, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    return eng, x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_wide_obs.py measures on the GPU"
    gpu = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = [f"# GPU: {gpu} (name, power limit, max SM clock); B = {args.B}; median [min, max] of {args.reps} steps"]
    print(lines[0], flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    B = args.B
    lines.append("## root step (representation + prediction + root expansion), microseconds")
    for net in MODES:
        for obs in WIDTHS:
            eng, x = engine(net, obs, B, 50)
            step = lambda: eng.root(obs=x, train=False)        # noqa: E731
            timed(step, 3, flush)                               # warm-up
            t = timed(step, args.reps, flush)
            obs_bytes = B * obs * 4
            lines.append(f"root  net={net:5s} obs={obs:5d}  {np.median(t):9.1f} us  [{t.min():.1f}, {t.max():.1f}]  "
                         f"observation read {obs_bytes / 1e6:7.1f} MB = {obs_bytes / np.median(t) / 1e3:7.1f} GB/s")
            print(lines[-1], flush=True)
            eng.close()
    lines.append("## whole search, 50 simulations (root step included), simulations per second")
    for net in MODES:
        for obs in (4, 376):
            eng, x = engine(net, obs, B, 50)

            def search():
                eng.root(obs=x, train=False)
                eng.simulate(50)
            timed(search, 3, flush)
            t = timed(search, args.reps, flush)
            lines.append(f"search net={net:5s} obs={obs:5d}  {np.median(t) / 1e3:8.3f} ms  [{t.min() / 1e3:.3f}, {t.max() / 1e3:.3f}]  "
                         f"{B * 50 / (np.median(t) * 1e-6) / 1e6:7.1f} M sims/s")
            print(lines[-1], flush=True)
            eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
