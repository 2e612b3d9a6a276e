"""The torch re-statement of the inference facade in batched_model.ReferenceModuleBackend against the
reference's own batch-1 `*_function_inference` outputs stored in tests/golden (net_*.npz for the MLP family,
vision_*.npz for the vision family), evaluated on reference-shaped modules filled with the stored weights."""
import numpy as np
import pytest
import torch

import golden_io
from fake_muzero import FakeMuzero, FakeVisionMuzero


def _cases(family):
    if family == "mlp":
        for name in golden_io.net_cases():
            z = golden_io.load_net_case(name)
            yield name, FakeMuzero(z["weights"], *[int(v) for v in z["dims"]]), z
    else:
        for name in golden_io.vision_cases():
            z = golden_io.load_vision_case(name)
            yield name, FakeVisionMuzero(z["weights"], *[int(v) for v in z["dims"]]), z


@pytest.mark.parametrize("family", ["mlp", "vision"])
def test_reference_module_backend_matches_reference_inference(family):
    from stochastic_muzero_b200.batched_model import ReferenceModuleBackend
    torch.set_num_threads(1)
    # vision: scale_to_bound_action normalises over the 3 CHANNELS of each pixel (vision:495-503); when the
    # three values nearly coincide the division amplifies fp32 noise (batched vs batch-1 conv algorithms)
    hid_tol = 1e-5 if family == "mlp" else 2e-4
    for name, mz, z in _cases(family):
        be = ReferenceModuleBackend(mz, device="cpu")
        t = {k: torch.from_numpy(z[k]) for k in ("obs", "repr_h", "adyn_h", "dyn_h")}
        acts = torch.from_numpy(z["actions"]).long()
        np.testing.assert_allclose(be.representation(t["obs"]).numpy(), z["repr_h"], atol=hid_tol, err_msg=name)
        for h, pol, val, fn in (("repr_h", "pred_policy", "pred_value", be.prediction),
                                ("adyn_h", "apred_policy", "apred_value", be.afterstate_prediction),
                                ("dyn_h", "dpred_policy", "dpred_value", be.prediction)):
            p, v = fn(t[h])
            np.testing.assert_allclose(p.numpy(), z[pol], atol=1e-5, err_msg=f"{name} {pol}")
            np.testing.assert_allclose(v.numpy(), z[val], atol=1e-5, rtol=5e-5, err_msg=f"{name} {val}")
        ah = be.afterstate_dynamics(t["repr_h"], acts)
        np.testing.assert_allclose(ah.numpy(), z["adyn_h"], atol=hid_tol, err_msg=name)
        r, dh = be.dynamics(t["adyn_h"], acts)
        np.testing.assert_allclose(dh.numpy(), z["dyn_h"], atol=hid_tol, err_msg=name)
        np.testing.assert_allclose(r.numpy(), z["dyn_reward"], atol=1e-5, rtol=5e-5, err_msg=name)
