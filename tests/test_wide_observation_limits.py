"""The observation-width limit of the MLP family, checked by smz_create before it touches a device."""
import ctypes as C

import pytest


def _mlp_config(obs_dim, net_mode):
    from stochastic_muzero_b200 import _lib
    cfg = _lib.smz_config()
    cfg.abi_version = _lib.SMZ_ABI_VERSION
    cfg.max_trees, cfg.num_simulations, cfg.action_dim, cfg.chance_dim = 4, 5, 2, 2
    cfg.max_action_sample, cfg.pb_c_base, cfg.pb_c_init, cfg.discount = 2, 19652, 1.25, 0.99
    cfg.obs_dim, cfg.state_dim, cfg.hidden_dim, cfg.num_hidden_layers = obs_dim, 61, 126, 2
    cfg.net_mode = net_mode
    return cfg


@pytest.mark.parametrize("mode", ["fp32", "bf16", "tc32", "f16"])
def test_create_rejects_observations_wider_than_8192_without_gpu_work(mode):
    from stochastic_muzero_b200 import _lib
    lib = _lib.load()
    net_mode = {"fp32": _lib.NET_FP32, "bf16": _lib.NET_BF16, "tc32": _lib.NET_TC32, "f16": _lib.NET_F16}[mode]
    h = C.c_void_p()
    assert lib.smz_create(C.byref(_mlp_config(8193, net_mode)), C.byref(h)) == _lib.SMZ_E_CAPACITY
    assert not h.value
    assert b"8192" in lib.smz_last_error()
