"""Vision (ResNet-v2) family, BASELINE config 5: every network output of a search against a float64 reference.

The per-simulation step of the vision family (k_vision_step's convolution stage + the tensor-core MLP heads, or the
all-CUDA-core k_vision_step with SMZ_VISION_CC=1) is checked leaf by leaf: for every simulation of a search the
expanded leaf is found in the exported tree, the float64 reference is fed the ENGINE's own parent state (errors do not
compound along a path) and the new hidden state, policy, value and reward the engine recorded are compared with it.
The stand-alone evaluation (smz_net_eval) is checked at the same shapes, and a degenerate model pins the
`spread < 1e-5` branch of the channel-wise scale_to_bound.

The reference is a float64 restatement of oracle/vision_oracle.py (itself pinned to the reference's inference outputs)
written with torch ops, so the same code runs on the CPU, where it is pinned to the goldens and to the float32 oracle,
and on the GPU, where it evaluates the tens of thousands of leaves of a search.

Tolerances (all quantities from the float64 pass):
* hidden state: scale_to_bound divides by the spread hi - lo of the three channels of a pixel, so an fp32 trunk whose
  pre-normalisation values carry errors of a few ulps of the values it computed produces errors of that size over
  the spread:
      |got - ref| <= C_HIDDEN * 2^-24 * M / max(spread, 1e-5) + 1e-6
  with M the largest |value| of any step of that row's trunk (convolution, BatchNorm, residual sum), not |pre|
  itself: where the last residual sums cancel, the rounding is that of their terms.
  Elements whose spread lies within a relative 1e-6 of the 1e-5 threshold are excluded (the output jumps there);
  they are counted and must stay rare.
* policy: 1e-5 absolute, the suite's fp32-grade bar, for both head paths.
* value / reward: the reference evaluates inverse_transform_with_support in float32 (muzero_model.py:575-591), a
  staircase with steps of ~1.2e-4 near zero (tests/test_host_logic.py).  The float64 reference computes the exact
  categorical expectation y and applies that float32 transform; an fp32 engine whose y is a few ulps away can sit on
  the neighbouring step.  So the engine's scalar must lie within SCALAR_TOL of the transform evaluated over
  [y - dy, y + dy], dy = C_LOGIT * 2^-24 * (m * E|s - y| + E|s|): m = max |W_out| |h| + |b_out| scales the rounding
  of the output logits, E|s - y| turns a logit error into an error of y, E|s| covers the fp32 expectation itself.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import golden_io
from oracle import vision_oracle as VO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCALAR_TOL = dict(atol=1e-5, rtol=5e-5)
POLICY_ATOL = 1e-5
# Worst measured on one B200 (1000 W power limit) over every case of this file, printed with -s:
#   hidden   needed c 5.45 on both head paths (one convolution code)      -> C_HIDDEN = 24, 4.4x above
#   scalars  needed C_LOGIT 2 tensor-core heads, 0.5 CUDA-core heads     -> C_LOGIT = 8, 4x above
#   policy   1.1e-6 tensor-core heads, 5.8e-7 CUDA-core heads            (bar 1e-5)
C_HIDDEN = 24.0
C_LOGIT = 8.0
ULP = 2.0 ** -24
SPREAD_EPS = 1e-5
EXCLUDED_MAX = 1e-3          # share of hidden elements allowed at the scale_to_bound threshold
CONV_STAGE_LEAVES = 8        # leaves per CTA of the convolution stage (RC in csrc/smz_net_vision.cu)
SMS = 148


# ---------------------------------------------------------------------------------------------------
# seeded random vision weights (weights.vision_blob_layout)
# ---------------------------------------------------------------------------------------------------
def vision_blob(A, S, H, L, seed, policy_scale=1.0, value_scale=1.0, reward_scale=1.0, symmetric_trunks=False):
    """Convolutions uniform in +-sqrt(3 / fan_in) (unit-variance preserving, the trunk's channels stay apart),
    linear layers uniform in +-sqrt(2 / fan_in) (with ReLU: the logits of an 18-layer head stay O(1)), BatchNorm with
    gamma ~ 1, var in [0.5, 2] and non-zero mean and beta (the fold at pack time has work to do).  The scale factors
    multiply the output layers of the policy, value and reward heads (peaky policies, values in the hundreds).
    symmetric_trunks: every convolution gives its output channels identical weights and every BatchNorm identical
    parameters, so the three channels of each hidden state coincide (spread exactly 0)."""
    from stochastic_muzero_b200.weights import VisionShape, vision_blob_layout
    layout, total = vision_blob_layout(VisionShape(A, S, H, L))
    g = np.random.default_rng(seed)
    blob = np.zeros(total, np.float64)
    for name, (off, shape) in layout.items():
        n = int(np.prod(shape))
        if name.endswith(".bn"):
            c = shape[1]
            v = np.stack([g.uniform(0.8, 1.25, c), g.uniform(-0.2, 0.2, c), g.uniform(-0.2, 0.2, c), g.uniform(0.5, 2.0, c)])
            if symmetric_trunks:
                v[:] = v[:, :1]
        elif len(shape) == 4 or name.endswith("conv_reward.w") or name.endswith("conv_value.w") or \
                name.endswith("conv_policy.w"):
            fan = n // shape[0]
            v = g.uniform(-1, 1, shape) * np.sqrt(3.0 / fan)
            if symmetric_trunks and len(shape) == 4:
                v[:] = v[:1]
        elif name.endswith(".w"):
            v = g.uniform(-1, 1, shape) * np.sqrt(2.0 / shape[1])
        else:
            v = g.uniform(-0.1, 0.1, shape)
        if name.endswith(".out.w") or name.endswith(".out.b"):
            v = v * (policy_scale if ".policy." in name else reward_scale if name.startswith("dyn.reward") else value_scale)
        blob[off:off + n] = np.ravel(v)
    return blob.astype(np.float32)


# ---------------------------------------------------------------------------------------------------
# float64 reference (the steps of oracle/vision_oracle.py)
# ---------------------------------------------------------------------------------------------------
def transform32(y):
    """inverse_transform_with_support after the expectation, in float32 exactly as the reference (and the kernels)
    evaluate it: sqrt(1 + 4 eps (|y| + 1 + eps)), minus 1, over 2 eps, squared, minus 1, with the sign of y."""
    f32 = np.float32
    y = np.asarray(y, np.float32)
    inner = np.sqrt(f32(1) + f32(4) * f32(0.001) * ((np.abs(y) + f32(1)) + f32(0.001)), dtype=np.float32)
    t = (inner - f32(1)) / (f32(2) * f32(0.001))
    return (np.sign(y) * (t * t - f32(1))).astype(np.float32)


class Ref64:
    def __init__(self, blob, A, S, H, L, device="cpu"):
        from stochastic_muzero_b200.weights import VisionShape, vision_blob_layout
        self.A, self.S, self.H, self.L, self.dev = A, S, H, L, device
        layout, total = vision_blob_layout(VisionShape(A, S, H, L))
        blob = np.asarray(blob, np.float32)
        assert blob.size == total
        self.w = {k: torch.tensor(blob[o:o + int(np.prod(s))].reshape(s), dtype=torch.float64, device=device)
                  for k, (o, s) in layout.items()}
        half = S // 2
        self.support = torch.arange(-half, S - half, dtype=torch.float64, device=device)

    def t(self, x):
        return torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).to(self.dev, torch.float64)

    # Every trunk step maps a pair (x, m): x the value, m [n, 1, 1, 1] the largest |value| the trunk has computed so far
    # for that row.  An fp32 evaluation rounds every step relative to the values it adds, so its error at the end is a
    # modest multiple of ulp(m) whatever cancels in the last sums.
    @staticmethod
    def _track(x, m):
        return torch.maximum(m, x.abs().amax((1, 2, 3), keepdim=True))

    def _bn_relu(self, x, m, bn):
        gamma, beta, mean, var = (v[None, :, None, None] for v in bn)
        y = (x - mean) / torch.sqrt(var + VO.BN_EPS) * gamma + beta
        return torch.relu(y), self._track(y, m)

    def _conv(self, x, m, w, stride=1):
        y = F.conv2d(x, w, stride=stride, padding=1)
        return y, self._track(y, m)

    def _res(self, x, m, p):
        bn, c1, c3 = self.w[p + ".bn"], self.w[p + ".conv1"], self.w[p + ".conv3"]
        y, m = self._conv(*self._bn_relu(x, m, bn), c1)
        y, m = self._conv(*self._bn_relu(y, m, bn), c3)
        y, m = self._conv(*self._bn_relu(y, m, bn), c1)
        return y + x, self._track(y + x, m)

    @staticmethod
    def _scale(pre, m):
        """channel-wise scale_to_bound -> (state, largest |value| of the trunk, per-pixel spread)"""
        lo, hi = pre.amin(1, keepdim=True), pre.amax(1, keepdim=True)
        spread = hi - lo
        sc = torch.where(spread < SPREAD_EPS, spread + SPREAD_EPS, spread)
        return (pre - lo) / sc, m, spread

    def _mlp(self, x, p):
        """-> (output logits, largest magnitude |W_out| |h| + |b_out| of the last layer's sums)"""
        for name in [".in"] + [".mid"] * self.L:
            x = torch.relu(x @ self.w[p + name + ".w"].T + self.w[p + name + ".b"])
        w, b = self.w[p + ".out.w"], self.w[p + ".out.b"]
        return x @ w.T + b, (x.abs() @ w.abs().T + b.abs()).amax(1)

    def _scalar(self, logits, mag):
        """-> (exact expectation y over the support, dy of the tolerance note)"""
        p = torch.softmax(logits, -1)
        y = (p * self.support).sum(1)
        spread = (p * (self.support[None] - y[:, None]).abs()).sum(1)
        return y, mag * spread + (p * self.support.abs()).sum(1)

    @staticmethod
    def _conv1x1(x, w, b):
        return (torch.einsum("bchw,oc->bohw", x, w) + b[None, :, None, None]).flatten(1)

    def representation(self, obs):
        x = self.t(obs).reshape(-1, 3, 98, 98)
        x, m = self._conv(x, x.abs().amax((1, 2, 3), keepdim=True), self.w["repr.conv_in"], stride=2)
        for _ in range(2):
            x, m = self._res(x, m, "repr.res_in")
        x, m = self._conv(x, m, self.w["repr.conv_out"], stride=2)
        for i in range(5):
            x, m = self._res(x, m, "repr.res_out")
            if i in (1, 4):
                x = F.avg_pool2d(x, 3, 2, 1, count_include_pad=True)
        return self._scale(*self._res(x, m, "repr.res_last"))

    def _with_action(self, h, idx):
        h = self.t(h).reshape(-1, 3, 7, 7)
        plane = (self.t(idx) + 1) / self.A
        return torch.cat([h, plane[:, None, None, None].expand(-1, 1, 7, 7)], 1)

    def _trunk(self, x, net):
        y, m = self._bn_relu(*self._conv(x, x.abs().amax((1, 2, 3), keepdim=True), self.w[net + ".conv"]),
                             self.w[net + ".bn"])
        for _ in range(self.L):
            y, m = self._res(y, m, net + ".res")
        return self._scale(torch.relu(y), m)

    def afterstate_dynamics(self, h, action):
        return self._trunk(self._with_action(h, action), "adyn")

    def dynamics(self, h, code):
        """-> ((y, dy) of the reward, trunk triple)"""
        x = self._with_action(h, code)
        r = self._conv1x1(x, self.w["dyn.conv_reward.w"], self.w["dyn.conv_reward.b"])
        return self._scalar(*self._mlp(r, "dyn.reward")), self._trunk(x, "dyn")

    def _pred(self, h, net):
        y = self.t(h).reshape(-1, 3, 7, 7)
        m = y.abs().amax((1, 2, 3), keepdim=True)
        for _ in range(self.L):
            y, m = self._res(y, m, net + ".res")
        v = self._conv1x1(y, self.w[net + ".conv_value.w"], self.w[net + ".conv_value.b"])
        p = self._conv1x1(y, self.w[net + ".conv_policy.w"], self.w[net + ".conv_policy.b"])
        return torch.softmax(self._mlp(p, net + ".policy")[0], -1), self._scalar(*self._mlp(v, net + ".value"))

    def prediction(self, h):
        """-> (policy, (y, dy) of the value)"""
        return self._pred(h, "pred")

    def afterstate_prediction(self, h):
        return self._pred(h, "apred")


# ---------------------------------------------------------------------------------------------------
# checks; each returns the worst measured ratio against its bar
# ---------------------------------------------------------------------------------------------------
def _np(x):
    return x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def check_hidden(got, ref, what):
    """got [n, 147]; ref = (state, magnitude, spread) of the float64 pass.  -> (needed c, excluded elements)"""
    h, mag, spread = (_np(v).astype(np.float64) for v in ref)
    n = h.shape[0]
    got = np.asarray(_np(got), np.float64).reshape(n, 3, 7, 7)
    unit = np.maximum(ULP * mag / np.maximum(spread, SPREAD_EPS), 1e-30)
    edge = np.broadcast_to(np.abs(spread - SPREAD_EPS) <= 1e-6 * SPREAD_EPS, h.shape)
    err = np.where(edge, 0.0, np.abs(got - h))
    bad = err > C_HIDDEN * unit + 1e-6
    if bad.any():
        i = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {int(bad.sum())} hidden elements off, first at {tuple(i)}: got "
                             f"{got[tuple(i)]:.8g}, float64 {h[tuple(i)]:.8g}, bar {C_HIDDEN * unit[i[0], 0, i[2], i[3]] + 1e-6:.3g}")
    assert edge.sum() <= EXCLUDED_MAX * edge.size, f"{what}: {int(edge.sum())} elements at the threshold"
    return float((np.maximum(err - 1e-6, 0) / unit).max()) if n else 0.0, int(edge.sum())


def check_policy(got, ref, what):
    got, ref = np.asarray(_np(got), np.float64), _np(ref)
    err = np.abs(got - ref)
    assert err.max(initial=0) <= POLICY_ATOL, f"{what}: policy off by {err.max():.3g} at row {np.argmax(err.max(1))}"
    return float(err.max(initial=0)) / POLICY_ATOL


def _scalar_err(got, y, dy):
    """distance of got from the float32 transform over [y - dy, y + dy], in units of SCALAR_TOL"""
    pts = [transform32(y - dy), transform32(y + dy)]
    across = (y - dy <= 0) & (y + dy >= 0)
    pts += [np.where(across, transform32(s * 1e-30), pts[0]) for s in (1.0, -1.0)]
    lo, hi = np.minimum.reduce(pts).astype(np.float64), np.maximum.reduce(pts).astype(np.float64)
    err = np.maximum(np.maximum(lo - got, got - hi), 0)
    return err / (SCALAR_TOL["atol"] + SCALAR_TOL["rtol"] * np.abs(transform32(y)))


def check_scalar(got, ref, what):
    """got [n]; ref = (y, dy) of the float64 pass.  -> needed C_LOGIT (the smallest power of two that passes)"""
    got = np.asarray(_np(got), np.float64)
    y, dy = (_np(v) for v in ref)
    ratio = _scalar_err(got, y, C_LOGIT * ULP * dy)
    if (ratio > 1).any():
        i = int(np.argmax(ratio))
        raise AssertionError(f"{what}: {int((ratio > 1).sum())} scalars off, row {i}: got {got[i]:.8g}, float64 "
                             f"expectation {y[i]:.10g} -> {transform32(y[i]):.8g}")
    need = 0.0
    while need < C_LOGIT and (_scalar_err(got, y, need * ULP * dy) > 1).any():
        need = max(2 * need, 1.0 / 64)
    return need


class Worst(dict):
    def add(self, key, v):
        self[key] = max(self.get(key, 0.0), v)


# ---------------------------------------------------------------------------------------------------
# CPU: the float64 reference against the goldens and the float32 oracle
# ---------------------------------------------------------------------------------------------------
GOLDEN_HIDDEN_ATOL = 2e-4        # the suite's bar of the fp32 reference's own hidden states (test_oracle_golden.py)


@pytest.mark.parametrize("name", golden_io.vision_cases())
def test_float64_reference_matches_reference_inference(name):
    z = golden_io.load_vision_case(name)
    A, S, H, L = (int(v) for v in z["dims"])
    ref = Ref64(z["weights"], A, S, H, L)
    flat = lambda x: np.asarray(x, np.float64).reshape(x.shape[0], -1)       # noqa: E731

    def scalar(yd, gold):
        np.testing.assert_allclose(transform32(_np(yd[0])), gold, **SCALAR_TOL)

    np.testing.assert_allclose(flat(_np(ref.representation(z["obs"])[0])), flat(z["repr_h"]), atol=GOLDEN_HIDDEN_ATOL)
    pol, val = ref.prediction(z["repr_h"])
    np.testing.assert_allclose(_np(pol), z["pred_policy"], atol=POLICY_ATOL)
    scalar(val, z["pred_value"])
    np.testing.assert_allclose(flat(_np(ref.afterstate_dynamics(z["repr_h"], z["actions"])[0])), flat(z["adyn_h"]),
                               atol=GOLDEN_HIDDEN_ATOL)
    pol, val = ref.afterstate_prediction(z["adyn_h"])
    np.testing.assert_allclose(_np(pol), z["apred_policy"], atol=POLICY_ATOL)
    scalar(val, z["apred_value"])
    rew, st = ref.dynamics(z["adyn_h"], z["actions"])
    np.testing.assert_allclose(flat(_np(st[0])), flat(z["dyn_h"]), atol=GOLDEN_HIDDEN_ATOL)
    scalar(rew, z["dyn_reward"])
    pol, val = ref.prediction(z["dyn_h"])
    np.testing.assert_allclose(_np(pol), z["dpred_policy"], atol=POLICY_ATOL)
    scalar(val, z["dpred_value"])


# ---------------------------------------------------------------------------------------------------
# the case table
# ---------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, A, S, H, L, n_trees, N, K, max_trees=None, seed=0, policy_scale=1.0, value_scale=1.0,
                 reward_scale=1.0, paper=False, no_pdl=False, stepwise=False):
        self.name, self.A, self.S, self.H, self.L = name, A, S, H, L
        self.n_trees, self.N, self.K, self.max_trees = n_trees, N, K, max_trees or n_trees
        self.seed, self.paper, self.no_pdl, self.stepwise = seed, paper, no_pdl, stepwise
        self.scales = dict(policy_scale=policy_scale, value_scale=value_scale, reward_scale=reward_scale)

    @property
    def dims(self):
        return self.A, self.S, self.H, self.L

    def blob(self):
        return vision_blob(*self.dims, seed=self.seed, **self.scales)

    def __repr__(self):
        return self.name


PEAKY, LARGE = 20.0, 40.0        # output-layer gains: the top policy entry carries ~3/4 of the mass, |values| ~100s
CASES = [
    Case("limits_l16_k32", 32, 64, 128, 16, 65, 10, 32, seed=1),
    Case("limits_l1_partial", 32, 64, 128, 1, 300, 12, 3, max_trees=512, seed=2),
    Case("even_s_h17_k1", 5, 64, 17, 2, 33, 16, 1, seed=3),
    Case("cfg5_1024", 4, 61, 126, 4, 1024, 16, 2, seed=4),
    Case("cfg5_4096", 4, 61, 126, 4, 4096, 8, 2, seed=5),
    Case("golden_small_stepwise", 3, 21, 40, 1, 7, 20, 3, seed=6, stepwise=True),
    Case("a1_chain", 1, 21, 16, 1, 1, 12, 1, seed=7),
    Case("paper_alternation", 6, 31, 64, 3, 300, 16, 2, seed=8, paper=True),
    Case("no_pdl_l5", 8, 40, 96, 5, 129, 12, 8, seed=9, no_pdl=True),
    Case("peaky_large", 9, 51, 72, 2, 65, 20, 3, seed=10, policy_scale=PEAKY, value_scale=LARGE, reward_scale=LARGE),
]
PATHS = ("tc", "cc")             # tensor-core heads (default), all-CUDA-core step (SMZ_VISION_CC=1)
CHECK_ALL_UP_TO = 1024           # trees; larger searches check SAMPLE_TREES of them


def test_case_table_reaches_every_limit():
    """The leaf-by-leaf search cases run on both head paths and together reach every limit smz_vision_create
    accepts, a partial batch, ragged batches, both branch widths and more CTAs than one wave."""
    dims = {c.dims for c in CASES}
    assert {(32, 64, 128, 16), (32, 64, 128, 1), (4, 61, 126, 4), (3, 21, 40, 1)} <= dims
    assert any(c.S % 2 == 0 and c.H % 8 for c in CASES) and any(c.S % 2 for c in CASES)
    assert any(c.A == 1 for c in CASES)
    assert {1, 7, 33, 65, 300} <= {c.n_trees for c in CASES}
    assert any(c.n_trees < c.max_trees for c in CASES)
    assert any(c.K == 1 for c in CASES) and any(c.K >= c.A > 1 for c in CASES)
    cfg5 = {c.n_trees for c in CASES if c.dims == (4, 61, 126, 4)}
    assert {1024, 4096} <= cfg5
    # the convolution stage runs n / 8 + 1 CTAs, the head chains 5 x n / 64: both have more CTAs than the GPU has SMs
    assert any((c.n_trees + CONV_STAGE_LEAVES - 1) // CONV_STAGE_LEAVES + 1 > SMS for c in CASES)
    assert any(5 * ((c.n_trees + 63) // 64) > SMS for c in CASES)
    assert any(c.paper for c in CASES) and any(c.no_pdl for c in CASES) and any(c.stepwise for c in CASES)
    assert any(c.scales["policy_scale"] > 1 and c.scales["value_scale"] > 1 for c in CASES)
    assert set(PATHS) == {"tc", "cc"}
    assert max(c.L for c in CASES) == 16 and max(c.A for c in CASES) == 32 and max(c.S for c in CASES) == 64
    assert max(c.H for c in CASES) == 128


@pytest.mark.parametrize("case", CASES, ids=repr)
def test_float64_reference_matches_the_float32_oracle(case):
    """At every shape of the table (random weights with the case's output gains) the float32 oracle is within fp32
    noise of the float64 reference, by the same bars the kernels are held to."""
    A, S, H, L = case.dims
    blob = case.blob()
    ref, orc = Ref64(blob, A, S, H, L), VO.VisionOracle(blob, A, S, H, L)
    g = np.random.default_rng(case.seed)
    obs = g.random((2, 3, 98, 98), dtype=np.float32)
    h = orc.representation(obs)
    check_hidden(h.reshape(2, -1), ref.representation(obs), f"{case} repr")
    h = np.concatenate([h, g.random((6, 3, 7, 7), dtype=np.float32)])
    act = g.integers(0, A, len(h))
    check_hidden(orc.afterstate_dynamics(h, act).reshape(len(h), -1), ref.afterstate_dynamics(h, act), f"{case} adyn")
    r32, d32 = orc.dynamics(h, act)
    r64, d64 = ref.dynamics(h, act)
    check_hidden(d32.reshape(len(h), -1), d64, f"{case} dyn")
    check_scalar(r32, r64, f"{case} reward")
    for fn in ("prediction", "afterstate_prediction"):
        p32, v32 = getattr(orc, fn)(h)
        p64, v64 = getattr(ref, fn)(h)
        check_policy(p32, p64, f"{case} {fn}")
        check_scalar(v32, v64, f"{case} {fn}")


# ---------------------------------------------------------------------------------------------------
# GPU: every leaf of whole searches
# ---------------------------------------------------------------------------------------------------
def _engine(case, monkeypatch, path, max_trees=None, blob=None, record=True):
    from stochastic_muzero_b200 import SearchEngine, VisionShape
    monkeypatch.delenv("SMZ_VISION_CC", raising=False)
    monkeypatch.delenv("SMZ_NO_PDL", raising=False)
    if path == "cc":
        monkeypatch.setenv("SMZ_VISION_CC", "1")
    if case.no_pdl:
        monkeypatch.setenv("SMZ_NO_PDL", "1")
    search = dict(pb_c_base=19652, pb_c_init=1.25, discount=0.997, root_dirichlet_alpha=0.25,
                  root_exploration_fraction=0.25, num_simulations=case.N, maxium_action_sample=case.K,
                  number_of_player=1, custom_loop=None)
    eng = SearchEngine(search, case.A, case.A, max_trees=max_trees or case.max_trees, model_shape=VisionShape(*case.dims),
                       net="vision", rng="philox", seed=100 + case.seed, record=record, paper_alternation=case.paper)
    eng.set_weights(case.blob() if blob is None else blob)
    return eng


def _sample_trees(n):
    if n <= CHECK_ALL_UP_TO:
        return np.arange(n)
    edges = [t + d for t in range(0, n + 1, 64) for d in (-1, 0, 7, 8)]
    extra = np.random.default_rng(n).choice(n, 256, replace=False)
    return np.unique(np.clip(np.concatenate([edges, extra, [0, n - 1]]), 0, n - 1))


def _expansions(eng, trees, N):
    """For every checked tree and simulation s: (parent hidden slot, action / code) of the leaf s expanded.  The
    leaf is the node whose child_base is 1 + A + s Kmax; its parent's hidden slot is 0 for a child of the root, else
    the simulation that created it, + 1."""
    A, Kmax = eng.A, eng.dims.max_children
    slot = np.zeros((len(trees), N), np.int64)
    key = np.zeros((len(trees), N), np.int64)
    for i, b in enumerate(trees):
        ar = eng.export_arena(int(b))
        node_of = {int(cb): n for n, cb in enumerate(ar["child_base"]) if cb}
        for s in range(N):
            leaf = node_of[1 + A + s * Kmax]
            key[i, s] = ar["key"][leaf]
            slot[i, s] = 0 if leaf <= A else (leaf - 1 - A) // Kmax + 1
    return slot, key


def run_search_and_check(case, path, monkeypatch, worst=None):
    dev = torch.device("cuda")
    A, N, n = case.A, case.N, case.n_trees
    eng = _engine(case, monkeypatch, path)
    obs = torch.rand(n, 3 * 98 * 98, generator=torch.Generator().manual_seed(case.seed))
    eng.root(obs=obs, train=True)
    sel = None
    if case.stepwise:
        sel = []
        for s in range(N):
            sel.append([_np(t) for t in eng.select(s)])
            eng.net_step(s)
            eng.expand_backup(s)
        expect = 4 + (3 if path == "tc" else 2) * N + N        # root (2 + dirichlet + expansion), then per simulation
    else:                                                        # select, network step, expansion/backup
        eng.simulate(N)
        expect = 4 + 1 + (3 if path == "tc" else 2) * N          # + first select; the heads are a kernel of their own
    st = eng.stats()
    assert st["launches"] == expect, f"{case}/{path}: {st} (expected {expect}: wrong head path)"
    roots = eng.read_roots()
    assert int(roots["error"].item()) == 0 and (roots["visits"].sum(1) == N).all()
    rec = {k: _np(v) for k, v in eng.read_record().items()}
    hid = torch.stack([eng.read_hidden(k) for k in range(N + 1)], 1)           # [n, N + 1, 147] on the device
    trees = _sample_trees(n)
    slot, key = _expansions(eng, trees, N)
    branch = rec["sim_branch"][trees].astype(np.int64)
    if sel is not None:     # the derivation from the exported tree is what select() reported
        for s in range(N):
            np.testing.assert_array_equal(sel[s][0][trees], slot[:, s])
            np.testing.assert_array_equal(sel[s][1][trees], key[:, s])
            np.testing.assert_array_equal(sel[s][2][trees], branch[:, s])
    eng.close()

    ref = Ref64(case.blob(), *case.dims, device=dev)
    worst = Worst() if worst is None else worst
    what = f"{case}/{path}"
    # root: representation of the observation, prediction of the engine's own h0
    tt = torch.as_tensor(trees)
    h0 = hid[tt.to(dev), 0]
    c, ex = check_hidden(h0, ref.representation(obs[tt]), f"{what} root hidden")
    worst.add(f"{path} hidden c", c)
    pol, _ = ref.prediction(h0)
    worst.add(f"{path} policy", check_policy(rec["root_policy"][trees, :A], pol, f"{what} root policy"))
    # every leaf: parent state from the engine, new state, its prediction, the reward of the dynamics pair
    ti = tt.to(dev)[:, None].expand(-1, N)
    si = torch.arange(N, device=dev)[None].expand(len(trees), -1)
    parent = hid[ti, torch.as_tensor(slot, device=dev)]
    new = hid[ti, si + 1]
    keys = torch.as_tensor(key, device=dev)
    excluded = 0
    for b in (0, 1):
        m = branch == b
        if not m.any():
            continue
        mt = torch.as_tensor(m, device=dev)
        tag = f"{what} {'dynamics' if b else 'afterstate'} leaves"
        if b:
            rew, st3 = ref.dynamics(parent[mt], keys[mt])
            worst.add(f"{path} scalar C", check_scalar(rec["sim_reward"][trees][m], rew, f"{tag}: reward"))
            pol, val = ref.prediction(new[mt])
        else:
            st3 = ref.afterstate_dynamics(parent[mt], keys[mt])
            assert (rec["sim_reward"][trees][m] == 0).all()
            pol, val = ref.afterstate_prediction(new[mt])
        c, ex = check_hidden(new[mt], st3, f"{tag}: hidden")
        excluded += ex
        worst.add(f"{path} hidden c", c)
        worst.add(f"{path} policy", check_policy(rec["sim_policy"][trees][m][:, :A], pol, f"{tag}: policy"))
        worst.add(f"{path} scalar C", check_scalar(rec["sim_value"][trees][m], val, f"{tag}: value"))
    assert branch[:, 0].tolist() == [0] * len(trees)
    print(f"\n{what}: {len(trees)} trees x {N} simulations, {excluded} hidden elements at the threshold; worst", dict(worst))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("case", CASES, ids=repr)
def test_every_leaf_of_a_vision_search_matches_float64(case, path, monkeypatch):
    run_search_and_check(case, path, monkeypatch)


# ---------------------------------------------------------------------------------------------------
# GPU: stand-alone evaluation (smz_net_eval)
# ---------------------------------------------------------------------------------------------------
EVAL_ROWS = (1, 31, 32, 33, 100)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for i, c in enumerate(CASES) if c.dims not in {d.dims for d in CASES[:i]}], ids=repr)
def test_network_evaluation_matches_float64(case, monkeypatch):
    dev = torch.device("cuda")
    A = case.A
    eng = _engine(case, monkeypatch, "tc", max_trees=max(EVAL_ROWS), record=False)
    ref = Ref64(case.blob(), *case.dims, device=dev)
    g = torch.Generator().manual_seed(case.seed)
    for n in EVAL_ROWS:
        what = f"{case} net_eval n={n}"
        obs = torch.rand(n, 3 * 98 * 98, generator=g)
        h = eng.net_eval("repr", obs)["hidden"].clone()
        check_hidden(h, ref.representation(obs), f"{what} repr")
        idx = torch.randint(0, A, (n,), generator=g)
        o = eng.net_eval("adyn", h, idx)
        check_hidden(o["hidden"], ref.afterstate_dynamics(h, idx), f"{what} adyn")
        o = eng.net_eval("dyn", h, idx)
        rew, st3 = ref.dynamics(h, idx)
        check_hidden(o["hidden"], st3, f"{what} dyn")
        check_scalar(o["reward"], rew, f"{what} dyn reward")
        for which, fn in (("pred", ref.prediction), ("apred", ref.afterstate_prediction)):
            o = eng.net_eval(which, h)
            pol, val = fn(h)
            check_policy(o["policy"], pol, f"{what} {which}")
            check_scalar(o["value"], val, f"{what} {which} value")
    eng.close()


# ---------------------------------------------------------------------------------------------------
# GPU: the spread == 0 branch of scale_to_bound
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
def test_coinciding_channels_give_a_zero_state(path, monkeypatch):
    """Trunks whose convolutions give all three output channels the same weights (and BatchNorms the same parameters):
    every pixel's channels coincide, the spread is exactly 0, scale_to_bound divides 0 by 1e-5 and every hidden state
    of the search, root included, is exactly 0.  Predictions of the zero state against float64."""
    case = Case("symmetric", 5, 21, 40, 2, 33, 8, 2, seed=11)
    blob = vision_blob(*case.dims, seed=case.seed, symmetric_trunks=True)
    eng = _engine(case, monkeypatch, path, blob=blob)
    obs = torch.rand(case.n_trees, 3 * 98 * 98, generator=torch.Generator().manual_seed(3))
    eng.root(obs=obs, train=True)
    eng.simulate(case.N)
    for k in range(case.N + 1):
        assert (eng.read_hidden(k) == 0).all(), f"{path}: hidden slot {k} is not exactly 0"
    rec = {k: _np(v) for k, v in eng.read_record().items()}
    zero = torch.zeros(1, 147, dtype=torch.float64)
    ref = Ref64(blob, *case.dims)
    assert (_np(ref.afterstate_dynamics(zero, [0])[0]) == 0).all() and (_np(ref.dynamics(zero, [0])[1][0]) == 0).all()
    (pol, val), (apol, aval) = ref.prediction(zero), ref.afterstate_prediction(zero)
    br = rec["sim_branch"].astype(bool)
    check_policy(rec["root_policy"][:, :case.A], pol.expand(case.n_trees, -1), "root policy")
    check_policy(rec["sim_policy"][br][:, :case.A], pol.expand(int(br.sum()), -1), "dynamics leaves")
    check_policy(rec["sim_policy"][~br][:, :case.A], apol.expand(int((~br).sum()), -1), "afterstate leaves")
    check_scalar(rec["sim_value"][br], tuple(v.expand(int(br.sum())) for v in val), "dynamics values")
    check_scalar(rec["sim_value"][~br], tuple(v.expand(int((~br).sum())) for v in aval), "afterstate values")
    eng.close()
