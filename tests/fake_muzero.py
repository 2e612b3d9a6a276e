"""Reference-SHAPED models for tests that must run without the reference checkout: six torch modules with
the attribute names and Sequential structure of neural_network_mlp_model.py (tied hidden Linear, separate
heads) and their forward, filled from a weight blob, plus the five ``*_function_inference`` methods of
muzero_model.py:802-909 computed by the network oracle; and the five vision (ResNet-v2) modules as torch
functions of a vision weight blob (the arithmetic of oracle/vision_oracle.py)."""
import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from oracle import net_oracle as NO
from oracle import vision_oracle as VO


def _stack(in_dim, H, L, out_dim, mid=None):
    first = nn.Linear(in_dim, H)
    mid = mid if mid is not None else nn.Linear(H, H)
    seq = [first, nn.ELU()] + [mid, nn.ELU()] * L + [nn.Linear(H, out_dim)]
    return nn.Sequential(*seq)


def _share_trunk(dst: nn.Sequential, src: nn.Sequential):
    for i in range(len(src) - 1):
        dst[i] = src[i]


def _scale_to_bound(x):
    """neural_network_mlp_model.py:349-357 (MLP: over the state) and vision:495-503 (over the 3 channels)."""
    lo, hi = x.min(1, keepdim=True)[0], x.max(1, keepdim=True)[0]
    scale = hi - lo
    scale = torch.where(scale < 1e-5, scale + 1e-5, scale)
    return (x - lo) / scale


class _Holder(nn.Module):
    pass


class _Representation(nn.Module):
    def forward(self, x):
        return _scale_to_bound(self.state_norm(x))


class _TwoHeads(nn.Module):
    """Prediction / Afterstate_prediction: (policy logits, value logits)."""

    def forward(self, x):
        return self.policy(x), self.value(x)


class _AfterstateDynamics(nn.Module):
    def forward(self, h, onehot):
        return _scale_to_bound(self.next_state_normalized(torch.cat([h, onehot], 1)))


class _Dynamics(nn.Module):
    def forward(self, h, onehot):
        x = torch.cat([h, onehot], 1)
        return self.reward(x), _scale_to_bound(self.next_state_normalized(x))


class FakeMuzero:
    model_structure = "mlp_model"

    def __init__(self, blob, obs, A, C, S, H, L):
        self.dims = (obs, A, C, S, H, L)
        self.net = NO.NetOracle(blob, obs, A, C, S, H, L)
        self.action_dimension, self.state_dimension = A, S
        OH = max(A, C)
        layout, _ = NO.blob_layout(obs, A, C, S, H, L)
        blob = np.asarray(blob, np.float32)

        def t(name):
            o, shp = layout[name]
            return torch.from_numpy(blob[o:o + int(np.prod(shp))].reshape(shp).copy())

        def fill(seq, prefix, head):
            lin = [m for m in seq if isinstance(m, nn.Linear)]
            with torch.no_grad():
                lin[0].weight.copy_(t(prefix + ".in.w")); lin[0].bias.copy_(t(prefix + ".in.b"))
                if L > 0:
                    lin[1].weight.copy_(t(prefix + ".mid.w")); lin[1].bias.copy_(t(prefix + ".mid.b"))
                lin[-1].weight.copy_(t(f"{prefix}.{head}.w")); lin[-1].bias.copy_(t(f"{prefix}.{head}.b"))

        def two_heads(cls, prefix, in_dim, h1, w1, attr1, h2, w2, attr2):
            m = cls()
            a = _stack(in_dim, H, L, w1)
            b = _stack(in_dim, H, L, w2)
            _share_trunk(b, a)
            fill(a, prefix, h1); fill(b, prefix, h2)
            setattr(m, attr1, a); setattr(m, attr2, b)
            return m

        rep = _Representation(); rep.state_norm = _stack(obs, H, L, S); fill(rep.state_norm, "repr", "out")
        enc = _Holder(); enc.encoder = _stack(obs, H, L, C); fill(enc.encoder, "enc", "code")
        ady = _AfterstateDynamics(); ady.next_state_normalized = _stack(S + OH, H, L, S)
        fill(ady.next_state_normalized, "adyn", "state")
        self.representation_function = rep
        self.encoder_function = enc
        self.afterstate_dynamics_function = ady
        self.prediction_function = two_heads(_TwoHeads, "pred", S, "policy", A, "policy", "value", S, "value")
        self.afterstate_prediction_function = two_heads(_TwoHeads, "apred", S, "policy", C, "policy", "value", S,
                                                        "value")
        self.dynamics_function = two_heads(_Dynamics, "dyn", S + OH, "reward", S, "reward", "state", S,
                                           "next_state_normalized")

    # the five inference methods (batch 1, numpy/torch on CPU like the reference)
    def representation_function_inference(self, obs):
        return torch.from_numpy(self.net.representation(np.asarray(obs, np.float32).reshape(1, -1)))

    def prediction_function_inference(self, h):
        p, v = self.net.prediction(np.asarray(h, np.float32))
        return p, v[0]

    def afterstate_prediction_function_inference(self, h):
        p, v = self.net.afterstate_prediction(np.asarray(h, np.float32))
        return p, v[0]

    def afterstate_dynamics_function_inference(self, h, a):
        return torch.from_numpy(self.net.afterstate_dynamics(np.asarray(h, np.float32), [int(a)]))

    def dynamics_function_inference(self, h, a):
        r, nh = self.net.dynamics(np.asarray(h, np.float32), [int(a)])
        return r[0], torch.from_numpy(nh)


class _VisionNet(nn.Module):
    """One of the five vision functions, evaluated by torch from the tensors of a vision weight blob."""

    def __init__(self, kind, w, L):
        super().__init__()
        self.kind, self.L, self.names = kind, L, sorted(w)
        for i, k in enumerate(self.names):
            self.register_buffer(f"w{i}", w[k])

    def _w(self, name):
        return getattr(self, f"w{self.names.index(name)}")

    def _bn_relu(self, x, bn):
        return F.relu(F.batch_norm(x, bn[2], bn[3], bn[0], bn[1], training=False, eps=VO.BN_EPS))

    def _res(self, x, p):
        bn, c1, c3 = self._w(p + ".bn"), self._w(p + ".conv1"), self._w(p + ".conv3")
        y = F.conv2d(self._bn_relu(x, bn), c1, padding=1)
        y = F.conv2d(self._bn_relu(y, bn), c3, padding=1)
        return F.conv2d(self._bn_relu(y, bn), c1, padding=1) + x

    def _mlp(self, x, p):
        x = F.relu(F.linear(x, self._w(p + ".in.w"), self._w(p + ".in.b")))
        for _ in range(self.L):
            x = F.relu(F.linear(x, self._w(p + ".mid.w"), self._w(p + ".mid.b")))
        return F.linear(x, self._w(p + ".out.w"), self._w(p + ".out.b"))

    def _conv1x1(self, x, p):
        w = self._w(p + ".w")
        return F.conv2d(x, w.reshape(*w.shape, 1, 1), self._w(p + ".b")).flatten(1)

    def _trunk(self, x, net):
        y = self._bn_relu(F.conv2d(x, self._w(net + ".conv"), padding=1), self._w(net + ".bn"))
        for _ in range(self.L):
            y = self._res(y, net + ".res")
        return _scale_to_bound(F.relu(y))

    def forward(self, x, plane=None):
        if self.kind == "repr":
            x = F.conv2d(x, self._w("repr.conv_in"), stride=2, padding=1)
            x = self._res(self._res(x, "repr.res_in"), "repr.res_in")
            x = F.conv2d(x, self._w("repr.conv_out"), stride=2, padding=1)
            x = self._res(self._res(x, "repr.res_out"), "repr.res_out")
            x = F.avg_pool2d(x, 3, 2, 1)
            for _ in range(3):
                x = self._res(x, "repr.res_out")
            x = F.avg_pool2d(x, 3, 2, 1)
            return _scale_to_bound(self._res(x, "repr.res_last"))
        if self.kind in ("pred", "apred"):
            y = x
            for _ in range(self.L):
                y = self._res(y, self.kind + ".res")
            return (self._mlp(self._conv1x1(y, self.kind + ".conv_policy"), self.kind + ".policy"),
                    self._mlp(self._conv1x1(y, self.kind + ".conv_value"), self.kind + ".value"))
        x = torch.cat([x, plane], 1)
        if self.kind == "adyn":
            return self._trunk(x, "adyn")
        return self._mlp(self._conv1x1(x, "dyn.conv_reward"), "dyn.reward"), self._trunk(x, "dyn")


class FakeVisionMuzero:
    """The five functions the search uses of a reference vision `Muzero` (is_RGB: the action enters as a plane)."""
    is_RGB = True

    def __init__(self, blob, A, S, H, L):
        layout, _ = VO.blob_layout(A, S, H, L)
        blob = np.asarray(blob, np.float32)
        w = {k: torch.from_numpy(blob[o:o + int(np.prod(s))].reshape(s).copy()) for k, (o, s) in layout.items()}
        self.action_dimension, self.state_dimension = A, S
        for name, kind in (("representation", "repr"), ("prediction", "pred"), ("afterstate_prediction", "apred"),
                           ("afterstate_dynamics", "adyn"), ("dynamics", "dyn")):
            setattr(self, f"{name}_function", _VisionNet(kind, w, L))
