"""Cost of the node pattern: whole searches (root step + simulations) under the reference's depth pattern and under the
Stochastic MuZero alternation (`paper_alternation`), on the BASELINE cfg2 shape (4096 trees x 50 simulations,
A = C = K = 2) and the cfg3 shape (8192 trees x 100 simulations, A 4 / C 32 / K 32), in bf16 and tc32.  CUDA events
around each search, after warm-up searches of the same shape; the mean leaf depth comes from smz_stats.  The two
patterns visit different trees (a leaf's branch, and so the width of its children, depends on the pattern), so the
rate difference includes the difference in tree shape.  Prints one line per measurement and writes them to --out.

    python tools/bench_node_pattern.py [--reps 10] [--out profiles/node_pattern.txt]
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
              root_exploration_fraction=0.25, number_of_player=1, custom_loop=None)
WORKLOADS = {  # name: (trees, simulations, obs, A, C, K)
    "cfg2": (4096, 50, 4, 2, 2, 2),
    "cfg3": (8192, 100, 16, 4, 32, 32),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_node_pattern.py measures on the GPU"
    gpu = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = [f"# GPU: {gpu} (name, power limit, max SM clock); median [min, max] of {args.reps} searches"]
    print(lines[0], flush=True)
    for wl, (B, N, obs, A, C, K) in WORKLOADS.items():
        for net in ("bf16", "tc32"):
            for paper in (False, True):
                shape = ModelShape(obs, A, C, 61, 126, 4)
                eng = SearchEngine(dict(SEARCH, num_simulations=N, maxium_action_sample=K), A, C, max_trees=B,
                                   model_shape=shape, net=net, rng="philox", seed=1, paper_alternation=paper)
                eng.set_weights(random_blob(shape, seed=0))
                x = torch.randn(B, obs, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
                ts = []
                for i in range(args.reps + 2):           # the first two searches capture the graph and warm up
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    eng.root(obs=x, train=True)
                    eng.simulate(N)
                    e1.record()
                    torch.cuda.synchronize()
                    if i >= 2:
                        ts.append(e0.elapsed_time(e1))
                depth = eng.stats()["mean_leaf_depth"]
                t = np.array(ts)
                lines.append(f"{wl} net={net:4s} pattern={'paper' if paper else 'reference':9s} {B} trees x {N} sims  "
                             f"{np.median(t):8.3f} ms [{t.min():.3f}, {t.max():.3f}]  "
                             f"{B * N / (np.median(t) * 1e-3) / 1e6:7.2f} M sims/s  mean leaf depth {depth:.3f}")
                print(lines[-1], flush=True)
                eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
