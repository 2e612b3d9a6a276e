#!/usr/bin/env python
"""bench.py — MCTS simulations/sec of the batched Stochastic-MuZero search (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--net auto|bf16|tc32|fp32]
                    [--dump-outputs DIR]

A "step" is one whole batched search: root step (representation + prediction, root expansion,
Dirichlet mixing) + 50 simulations for 4096 concurrent trees (BASELINE.json configs[1]: CartPole MLP
of config/experiment_450_config.json, synthetic observations, random-init weights).  N > 1 shards
independent trees across ranks (4096 per GPU, weak scaling; the only collective is one NCCL weight
broadcast before timing).  One JSON line is printed by rank 0.  Besides the contract keys it carries
  "fp32"            the same workload with the reference-precision network step (1e-5 parity mode)
  "strong_scaling"  BASELINE configs[3]: 65536 trees split over the N ranks (cfg4), weight broadcast timed
  "roofline" / "roofline_tree"   the two kernels of the timed loop, each timed stand-alone with CUDA events
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEARCH = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
              root_exploration_fraction=0.25, num_simulations=50, maxium_action_sample=2,
              number_of_player=1, custom_loop=None)
DIMS = dict(obs_dim=4, action_dim=2, chance_dim=2, state_dim=61, hidden_dim=126, num_hidden_layers=4)
METRIC, UNIT = "mcts_simulations_per_sec", "sims/s"

# BASELINE.json configs.  cfg2 is the bench line (the metric is quoted on it); the others are parity-test
# shapes that can be timed on request (--workload) and are reported with the same JSON contract.
WORKLOADS = {
    "cfg2": dict(name="BASELINE configs[1]: CartPole MLP (obs 4, A 2, S 61, H 126, L 4)", trees=4096, sims=50,
                 dims=DIMS, K=2, net=None),
    "cfg3": dict(name="BASELINE configs[2]: stochastic 2048-like (4x4 board obs 16, 4 actions, 32 chance codes, K 32)",
                 trees=8192, sims=100, dims=dict(DIMS, obs_dim=16, action_dim=4, chance_dim=32), K=32, net=None),
    "cfg4": dict(name="BASELINE configs[3]: CartPole MLP, 65536 trees sharded across the ranks", trees=65536, sims=50,
                 dims=DIMS, K=2, net=None, total=True),
    "cfg5": dict(name="BASELINE configs[4]: vision ResNet-v2 (98x98 RGB, A 4, S 61, H 126, L 4)", trees=1024, sims=50,
                 dims=dict(action_dim=4, state_dim=61, hidden_dim=126, num_hidden_layers=4), K=2, net="vision"),
}
KERNEL_NAMES = {"bf16": "k_bf16_chain_m32 / _m64 / _pipe / _pipeN<2> by batch size, tcgen05 kind::f16 on bf16 operands",
                "f16": "k_tc32_chain_m64<1>, tcgen05 kind::f16 on fp16 operands (one product)",
                "tc32": "k_tc32_chain_m64, tcgen05 kind::f16 on fp16 hi/lo split operands (hi and lo rows stacked along M: 2 MMAs per K-step give all 4 partial products, fp32-grade)",
                "fp32": "k_net_sim, fp32 CUDA cores", "vision": "k_vision_step, fp32 CUDA cores"}
DTYPES = {"bf16": "bf16", "f16": "f16", "tc32": "f32 (fp16 hi+lo split operands, fp32 accumulate)", "fp32": "f32", "vision": "f32"}


def vision_flops_per_sim(d):
    """2*MAC of the vision per-simulation networks: 3x3 convs on 3x7x7 maps + three 147->H->..->S/A MLP heads."""
    H, L, S, A = d["hidden_dim"], d["num_hidden_layers"], d["state_dim"], d["action_dim"]
    conv = lambda ci, co: 2 * ci * co * 9 * 49                                    # noqa: E731
    res = 3 * conv(3, 3)
    mlp = lambda n: 2 * (147 * H + L * H * H + H * n)                             # noqa: E731
    trunk = conv(4, 3) + L * res
    pred = L * res + 2 * 2 * 9 * 49 + mlp(S) + mlp(A)
    after = trunk + pred
    dyn = trunk + 2 * 12 * 49 + mlp(S) + pred
    return after, dyn, 0


def flops_per_sim(d):
    """SURVEY.md §8d: 2*MAC, trunk counted once, one-hot counted as dense S+A input."""
    S, H, L, A, C = d["state_dim"], d["hidden_dim"], d["num_hidden_layers"], d["action_dim"], d["chance_dim"]
    OH = max(A, C)
    after = 2 * ((S + OH) * H + L * H * H + H * S) + 2 * (S * H + L * H * H + H * C + H * S)
    dyn = 2 * ((S + OH) * H + L * H * H + 2 * H * S) + 2 * (S * H + L * H * H + H * A + H * S)
    root = 2 * (d["obs_dim"] * H + L * H * H + H * S) + 2 * (S * H + L * H * H + H * A + H * S)
    return after, dyn, root


def tree_bytes_per_sim(depth, K, S):
    """SURVEY.md §8d algorithmic bytes of the tree kernels per simulation (select + expand + backup)."""
    return depth * (16 * K + 8) + 8 * S + 4 + 12 * K + 20 * (depth + 1) + 8


class ClockSampler(threading.Thread):
    """NVML poller (about 1 kHz) for SM clock, power and clock-event reasons: the timed region of the default
    run is a few tens of milliseconds, far below nvidia-smi's own sampling period."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device):
        super().__init__(daemon=True)
        self.samples, self.stop_flag, self.h, self.max_mhz = [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(device))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    @staticmethod
    def _physical_index(device):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if device < len(ids) and ids[device].isdigit():
                return int(ids[device])
        return device

    def run(self):
        if self.h is None:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append((time.time(), float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                     nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0,
                                     int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:
                pass
            time.sleep(0.0005)

    def window(self, t0, t1, label):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"], "samples": 0, "window": label}
        rows = [r for r in self.samples if t0 <= r[0] <= t1]
        sm = sorted(r[1] for r in rows)
        bits = 0
        for r in rows:
            bits |= r[3]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if bits & b), "samples": len(rows),
                "power_w_max": max((r[2] for r in rows), default=None), "window": label}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, roots):
    """Writes the root statistics of the last timed step (SearchEngine.read_roots: visit counts, root values, root
    priors and rewards of the children, error flag) as <path>/<name>.npy in float32 / float64, so that two builds
    can be compared output for output.  Above DUMP_LIMIT_BYTES a fixed, seeded sample of trees is kept;
    tree_index.npy says which."""
    import numpy as np
    arrays = {"visits": roots["visits"].float(), "root_values": roots["root_values"], "priors": roots["priors"],
              "rewards": roots["rewards"]}
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    n = len(arrays["visits"])
    per_tree = sum(a.nbytes for a in arrays.values()) // n + 8
    idx = np.arange(n)
    if n * per_tree > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // per_tree, replace=False))
    arrays = {k: v[idx] for k, v in arrays.items()}
    arrays["tree_index"] = idx.astype(np.float64)
    arrays["error"] = roots["error"].cpu().numpy().astype(np.float32)
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def run_reference(args):
    """Reference arm: the reference's CPU search path on all host cores (the unmodified reference where a
    checkout is reachable, else the oracle port — see oracle/cpu_baseline.py); each step is a bounded sample of
    configs[0]."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline
    per_step = max(2.0, min(10.0, 60.0 / max(1, args.steps + args.warmup)))
    for _ in range(min(args.warmup, 1)):
        cpu_baseline.measure(seconds=1.0)
    rates, t0 = [], time.perf_counter()
    for _ in range(args.steps):
        rates.append(cpu_baseline.measure(seconds=per_step))
    wall = time.perf_counter() - t0
    value = sum(r["value"] for r in rates) / len(rates)
    base = dict(rates[-1], value=value)
    base.pop("per_core", None)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[0]: CartPole MLP 450 shape, 1 tree per host process, 50 "
                                   "simulations/move, reference CPU algorithm (%s)" % base["kind"], "sims_per_move": 50},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


class Bench:
    """One engine + the measurements taken on it."""

    def __init__(self, torch, dist, args, wl, net, B, N, world, rank, local, blob, obs):
        from stochastic_muzero_b200 import ModelShape, SearchEngine, VisionShape
        self.torch, self.dist, self.args, self.wl, self.net = torch, dist, args, wl, net
        self.B, self.N, self.world, self.rank, self.local = B, N, world, rank, local
        self.dev = torch.device("cuda", local)
        self.vision = net == "vision"
        dims = wl["dims"]
        self.shape = VisionShape(**dims) if self.vision else ModelShape(**dims)
        self.A = self.shape.action_dim
        self.C = self.A if self.vision else self.shape.chance_dim
        self.search = dict(SEARCH, num_simulations=N, maxium_action_sample=wl["K"])
        self.eng = SearchEngine(self.search, self.A, self.C, max_trees=B, model_shape=self.shape, net=net,
                                rng="philox", seed=20240 + rank, tree_id_offset=rank * B, device=local)
        self.eng.set_weights(blob)
        self.blob, self.obs = blob, obs

    def step(self):
        self.eng.root(obs=self.obs, train=True)
        self.eng.simulate(self.N)

    def timed(self, steps, warmup, flush, sampler=None, soak_s=0.0):
        """W warm-up steps, then exactly `steps` timed steps (CUDA events per step, L2 flushed in between,
        barrier + synchronize on both sides, max over ranks); optionally a sampled soak of identical steps."""
        torch, dist, world = self.torch, self.dist, self.world
        for i in range(warmup):
            self.eng.set_seed(1000 + i, self.rank * self.B)
            self.step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = self.eng.stats()["launches_total"]
        wall0 = time.time()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i, (a, b) in enumerate(evs):
            self.eng.set_seed(2000 + i, self.rank * self.B)
            flush.zero_()                      # evict the arena from L2 between timed steps (not timed)
            a.record()
            self.step()
            b.record()
        torch.cuda.synchronize()
        wall1 = time.time()
        if world > 1:
            dist.barrier()
        st = self.eng.stats()
        dev_ms = sum(a.elapsed_time(b) for a, b in evs)
        # what a caller of the timed path receives from its last step (--dump-outputs)
        self.last_roots = self.eng.read_roots()
        # every rank must have finished every tree: sum of root visits over all ranks == world * B * N
        visits = self.last_roots["visits"].sum().to(torch.float64).reshape(1)
        t = torch.tensor([dev_ms], dtype=torch.float64, device=self.dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(visits, op=dist.ReduceOp.SUM)
        assert int(visits.item()) == world * self.B * self.N, "a rank did not finish its trees"
        dev_ms = float(t.item())
        out = {"value": world * self.B * self.N * steps / (dev_ms * 1e-3), "ms_per_step": dev_ms / steps,
               "gpu_launches": st["launches_total"] - l0, "mean_leaf_depth": st["mean_leaf_depth"],
               "visit_checksum": int(visits.item())}
        if sampler is not None:
            out["clocks"] = sampler.window(wall0, wall1, "timed region (%d steps, NVML polled at ~1 kHz)" % steps)
        if soak_s > 0 and sampler is not None:
            # the timed region of the default run is ~25 ms: a soak of identical back-to-back steps (no flush, not part
            # of `value`) gives the clock record a seconds-long window under the same load
            s0, n = time.time(), 0
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            while time.time() - s0 < soak_s:
                for _ in range(20):
                    self.step()
                n += 20
                torch.cuda.synchronize()
            b.record()
            torch.cuda.synchronize()
            soak = sampler.window(s0, time.time(), "soak: %d identical steps back to back after the timed region" % n)
            soak["value"] = self.B * self.N * n / (a.elapsed_time(b) * 1e-3)
            soak["note"] = "per-GPU sims/s over the soak, warm L2 — a cross-check, not the bench value"
            out["clocks"]["soak"] = soak
        return out

    def rooflines(self, dev_ms_per_step, depth, peaks):
        """The two kernels of the timed loop, each timed stand-alone with CUDA events on the launching stream in a
        step-by-step replay of one more search: the network step (8 back-to-back idempotent launches per simulation)
        and the REAL fused tree step (smz_backup_select = k_backup_select_sm / k_backup_select, the kernel the
        captured graph runs between two network steps)."""
        torch, eng, N, B = self.torch, self.eng, self.N, self.B
        eng.set_seed(3000, self.rank * B)
        eng.root(obs=self.obs, train=True)
        torch.cuda.synchronize()
        ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
        marks = []
        NET_REP = 8
        eng.select(0)
        for s in range(N):
            e1, e2, e3 = ev(), ev(), ev()
            e1.record()
            for _ in range(NET_REP):            # the network step is idempotent: back-to-back launches hide the host launch gap
                eng.net_step(s)
            e2.record()
            if s + 1 < N:
                eng.backup_select(s)
            else:
                eng.expand_backup(s)
            e3.record()
            marks.append((e1, e2, e3))
        torch.cuda.synchronize()
        t_net = sum(m[0].elapsed_time(m[1]) for m in marks) / (N * NET_REP)
        t_tree = sum(m[1].elapsed_time(m[2]) for m in marks[:-1]) / max(1, N - 1)
        dims = self.wl["dims"]
        f_after, f_dyn, _ = vision_flops_per_sim(dims) if self.vision else flops_per_sim(dims)
        frac_dyn = self.dyn_fraction()
        flops_launch = B * ((1 - frac_dyn) * f_after + frac_dyn * f_dyn)
        which = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        # the network step is timed in isolation (bursts of 8 launches, idle GPU in between): burst peak
        tensor_peak = peaks.get("bf16_tflops", 1590.0)
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        achieved_tf = flops_launch / (t_net * 1e-3) / 1e12
        roofline = {"kernel": "network step (%s)" % KERNEL_NAMES[self.net], "bound": "tensor", "achieved": achieved_tf,
                    "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved_tf / tensor_peak, "traffic": None,
                    "peak_source": which + ", burst bf16 (kernel timed in isolation)", "avg_launch_us": 1e3 * t_net,
                    "algorithmic_flops_per_launch": flops_launch,
                    "frac_of_sustained_peak": achieved_tf / peaks.get("bf16_tflops_sustained", 1400.0),
                    "how": "CUDA events around %d back-to-back launches of the (idempotent) network step of every "
                           "simulation of one extra search replayed step by step on the launching stream" % NET_REP,
                    # share of the real (graph + PDL) step: launches x per-launch time / measured step time.  Kernels
                    # overlap a little under PDL, so the shares of all kernels add up to slightly more than 1.
                    "share_of_step": min(1.0, N * t_net / dev_ms_per_step)}
        tr = {}
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if self.args.workload == "cfg2" and self.net in tr.get("network_step", {}):
                roofline["traffic"] = tr["network_step"][self.net]
                roofline["traffic_source"] = tr.get("source")
        except Exception:
            pass
        K = min(self.wl["K"], max(self.A, self.C))
        tb = tree_bytes_per_sim(depth, K, 147 if self.vision else dims["state_dim"]) * B
        achieved_gbs = tb / (t_tree * 1e-3) / 1e9
        roofline_tree = {"kernel": "tree step of the timed loop (smz_backup_select: k_backup_select_sm / k_backup_select — "
                                   "expansion + backup of simulation s fused with the descent of s+1)",
                         "bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved_gbs / hbm_peak, "peak_source": which, "avg_launch_us": 1e3 * t_tree,
                         "traffic": tr.get("tree_step", {}).get("k_backup_select_sm") if self.args.workload == "cfg2" else None,
                         "algorithmic_bytes_per_launch": tb, "mean_leaf_depth": depth,
                         "share_of_step": min(1.0, (N - 1) * t_tree / dev_ms_per_step),
                         "how": "CUDA events around the stand-alone launch of the same kernel the captured graph runs "
                                "(its tree-mirroring prologue, hidden under the network step in the real loop, is "
                                "exposed here)"}
        return roofline, roofline_tree

    def dyn_fraction(self):
        """Share of simulations that took the dynamics pair, from the per-simulation branch counters."""
        if not hasattr(self, "_dyn"):
            torch, eng = self.torch, self.eng
            eng.set_seed(3001, self.rank * self.B)
            eng.root(obs=self.obs, train=True)
            n_dyn = torch.zeros((), dtype=torch.int64, device=self.dev)
            for s in range(self.N):
                _, _, br = eng.select(s)
                n_dyn += br.sum()
                eng.net_step(s)
                eng.expand_backup(s)
            self._dyn = float(n_dyn.item()) / (self.B * self.N)
        return self._dyn

    def e2e(self, steps):
        """End to end through the public API: pinned host observations in, host visit counts / root values out."""
        from stochastic_muzero_b200 import Monte_carlo_tree_search, PackedModel
        torch, dist, world = self.torch, self.dist, self.world
        mcts = Monte_carlo_tree_search(**self.search, net=self.net, device=self.local, seed=77 + self.rank,
                                       max_batch=self.B, tree_id_offset=self.rank * self.B)
        model = PackedModel(self.blob.cpu().numpy(), self.shape)
        obs_host = self.obs.cpu().pin_memory()
        for _ in range(3):
            mcts.run_batch(obs_host, model, train=True).host()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            h = mcts.run_batch(obs_host, model, train=True).host()     # one D2H: visits, root values, error flag
            v_host, rv_host = h["visit_counts"], h["root_values"]
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device=self.dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
        assert int(v_host.sum()) == self.B * self.N
        self.model = model
        return {"value": world * self.B * self.N * steps / e2e_s, "unit": UNIT,
                "h2d_bytes_per_step": int(obs_host.numel() * 4),
                "d2h_bytes_per_step": int(v_host.size * 4 + rv_host.size * 4 + 4),
                "ms_per_step": 1e3 * e2e_s / steps,
                "api": "Monte_carlo_tree_search.run_batch(pinned host observations).host() -> visit counts + root values "
                       "(+ the search's error flag) on host"}

    def close(self):
        self.eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--net", default=os.environ.get("SMZ_BENCH_NET", "auto"), choices=["auto", "fp32", "bf16", "tc32", "f16"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--trees", type=int, default=None, help="concurrent trees per GPU (default: the workload's)")
    ap.add_argument("--sims", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the fp32 leg, the strong-scaling leg and the soak")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--soak-seconds", type=float, default=2.5)
    ap.add_argument("--profile-only", action="store_true", help="timed steps only (for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the root statistics of the last timed step to DIR/<name>.npy (rank 0's trees)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist
    from stochastic_muzero_b200 import ModelShape, VisionShape, random_blob, vision_blob_layout

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    wl = WORKLOADS[args.workload]
    dims = wl["dims"]
    N = args.sims or wl["sims"]
    B = args.trees or (wl["trees"] // world if wl.get("total") else wl["trees"])
    vision = wl["net"] == "vision"
    net = "vision" if vision else args.net
    if net == "auto":
        net = os.environ.get("SMZ_DEFAULT_NET", "bf16")
    shape = VisionShape(**dims) if vision else ModelShape(**dims)
    obs_shape = (3 * 98 * 98,) if vision else (shape.obs_dim,)

    # weights: rank 0 draws them, one NCCL broadcast hands them to the other shards
    if vision:      # torch default init is not reproducible here: N(0, 0.05) convs / heads, identity-like BatchNorm
        lay, tot = vision_blob_layout(shape)
        w0 = (np.random.default_rng(0).standard_normal(tot) * 0.05).astype(np.float32)
        for k, (o, shp) in lay.items():
            if k.endswith(".bn"):
                c = shp[1]
                w0[o:o + 4 * c] = np.concatenate([np.ones(c), np.zeros(c), np.zeros(c), np.ones(c)])
    else:
        w0 = random_blob(shape, seed=0)
    blob = torch.from_numpy(w0).to(dev) if rank == 0 else torch.empty(len(w0), dtype=torch.float32, device=dev)
    bcast = {"cold_ms": 0.0, "warm_ms": 0.0, "bytes": int(blob.numel() * 4)}
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    if world > 1:
        dist.all_reduce(torch.zeros(1, device=dev))           # NCCL communicator set-up is not the broadcast
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dist.broadcast(blob, src=0)                            # first broadcast: cold (channel set-up for this size)
        torch.cuda.synchronize()
        bcast["cold_ms"] = 1e3 * (time.perf_counter() - t0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):                                    # the per-weight-update cost: warm, device-timed
            dist.broadcast(blob, src=0)
        e1.record()
        torch.cuda.synchronize()
        bcast["warm_ms"] = e0.elapsed_time(e1) / 10
    gen = torch.Generator().manual_seed(rank)
    if args.workload == "cfg3":      # 4x4 board, log2(tile)/16 with tiles drawn from {0..11} (SURVEY.md 8d)
        obs = (torch.randint(0, 12, (B,) + obs_shape, generator=gen).float() / 16.0).to(dev)
    elif vision:
        obs = torch.rand((B,) + obs_shape, generator=gen).to(dev)
    else:
        obs = torch.randn((B,) + obs_shape, generator=gen).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    main_b = Bench(torch, dist, args, wl, net, B, N, world, rank, local, blob, obs)
    res = main_b.timed(args.steps, args.warmup, flush, sampler,
                       soak_s=0.0 if (args.profile_only or args.no_extras) else args.soak_seconds)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main_b.last_roots)
    if args.profile_only:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": res["value"], "unit": UNIT, "ms_per_step": res["ms_per_step"],
                              "note": "profile-only run; not a bench value if taken under ncu"}), flush=True)
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    roofline, roofline_tree = main_b.rooflines(res["ms_per_step"], res["mean_leaf_depth"], peaks)
    e2e = main_b.e2e(args.steps)

    # ---- the reference-precision leg: same workload, fp32-grade network step (1e-5 parity mode) ----------------
    fp32_leg = None
    if not vision and not args.no_extras and net == "bf16":
        legs = {}
        for mode in ("tc32", "fp32", "f16"):
            try:
                b2 = Bench(torch, dist, args, wl, mode, B, N, world, rank, local, blob, obs)
            except Exception as exc:          # mode not built into this library
                legs[mode] = {"unavailable": str(exc)[:200]}
                continue
            r2 = b2.timed(args.steps, args.warmup, flush)
            rf, _ = b2.rooflines(r2["ms_per_step"], r2["mean_leaf_depth"], peaks)
            legs[mode] = {"value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"], "dtype": DTYPES[mode],
                          "gpu_launches": r2["gpu_launches"], "roofline": rf, "e2e": b2.e2e(args.steps)}
            b2.close()
        best = max((m for m in legs if "value" in legs[m] and m != "f16"), key=lambda m: legs[m]["value"], default=None)
        fp32_leg = dict(legs[best], network_step=best, note="reference precision: network outputs within 1e-5 of the "
                        "reference's torch fp32 (tests/test_gpu_parity.py); modes.f16 = plain fp16 operands, a second "
                        "throughput mode with ~8x tighter network tolerances than bf16", modes=legs) if best else {"modes": legs}

    # ---- BASELINE configs[3]: 65536 trees split over the ranks (strong scaling), every N --------------------------
    strong = None
    if args.workload == "cfg2" and not args.no_extras and not vision:
        wl4 = WORKLOADS["cfg4"]
        B4 = wl4["trees"] // world
        obs4 = torch.randn((B4, shape.obs_dim), generator=torch.Generator().manual_seed(100 + rank)).to(dev)
        b4 = Bench(torch, dist, args, wl4, net, B4, wl4["sims"], world, rank, local, blob, obs4)
        r4 = b4.timed(min(args.steps, 20), 3, flush)
        rf4 = None
        if rank == 0:          # roofline of the large-batch network step (the two-tile kernel above one wave of tiles)
            try:
                rf4, _ = b4.rooflines(r4["ms_per_step"], r4["mean_leaf_depth"], peaks)
            except Exception:
                rf4 = None
        strong = {"workload": wl4["name"], "trees_total": wl4["trees"], "trees_per_gpu": B4, "simulations": wl4["sims"],
                  "value": r4["value"], "unit": UNIT, "ms_per_step": r4["ms_per_step"], "scaling": "strong",
                  "network_step": net, "weight_broadcast": bcast, "visit_checksum": r4["visit_checksum"], "roofline": rf4}
        b4.close()

    # ---- the reference's own call, one tree at a time (BASELINE configs[0] shape through the drop-in run()) ----
    single = None
    if rank == 0 and world == 1 and not vision:
        from stochastic_muzero_b200 import Monte_carlo_tree_search
        one = Monte_carlo_tree_search(**main_b.search, device=local, seed=5)       # default mode: reference precision (tc32)
        for _ in range(3):
            one.run(observation=torch.randn(1, shape.obs_dim), model=main_b.model, train=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        moves = 20
        for _ in range(moves):
            one.run(observation=torch.randn(1, shape.obs_dim), model=main_b.model, train=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        single = {"ms_per_move": 1e3 * dt / moves, "value": moves * N / dt, "unit": UNIT,
                  "api": "Monte_carlo_tree_search.run(observation, model, train) -> Node, default (fp32-grade tcgen05) network step, 1 tree"}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import cpu_baseline
        cpu = cpu_baseline.measure(seconds=args.cpu_seconds)
    if sampler:
        sampler.stop_flag = True
    if rank == 0:
        line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": DTYPES[net], "data": "synthetic",
                "config": {"workload": f"{wl['name']}: {B} concurrent trees x {N} simulations per GPU, synthetic "
                                       f"observations, random-init weights, device Philox RNG",
                           "workload_id": args.workload,
                           "trees_per_gpu": B, "simulations": N, "network_step": net, "tree_arithmetic": "f32/f64 "
                           "(reference numpy semantics)", "l2": "256 MiB flush buffer written between timed steps",
                           "sharding": f"{world} x {B} independent trees, no data-path collective",
                           "weight_broadcast_ms": bcast["warm_ms"], "weight_broadcast": bcast},
                "roofline": roofline, "roofline_tree": roofline_tree, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": res["gpu_launches"], "clocks": res.get("clocks"), "mean_leaf_depth": res["mean_leaf_depth"],
                "visit_checksum": res["visit_checksum"], "fp32": fp32_leg, "strong_scaling": strong,
                "single_tree_dropin": single}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
