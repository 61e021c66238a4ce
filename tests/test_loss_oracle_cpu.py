"""CPU: oracle/loss_oracle.recon_losses against the unmodified reference's dvr_model static methods
(compute_recon_loss, mask_losses, apply_loss_weights; lab4d/engine/model.py:386-611) on the same synthetic batch.  The
reference's losses on these seeded batches are stored in tests/golden/reference/checks.npz (oracle/gen_golden.py)."""
import os

import numpy as np
import pytest
import torch

import loss_oracle as LO

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "checks.npz")
CONFIG = {"train_res": 256, "mask_wt": 0.1, "rgb_wt": 0.1, "depth_wt": 1e-4, "flow_wt": 0.5, "vis_wt": 1e-2, "feature_wt": 1e-2,
          "feat_reproj_wt": 5e-2, "reg_gauss_mask_wt": 0.01}


def synth_loss_inputs(field_type, M=6, N=16, seed=0, device="cpu", dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.rand(*s, generator=g)
    rn = lambda *s: torch.randn(*s, generator=g)
    rendered = {"mask": r(M, N, 1), "rgb": r(M, N, 3), "depth": 1 + r(M, N, 1), "flow": 3 * rn(M, N, 2)}
    aux = {}
    if field_type in ("fg", "comp"):
        aux["fg"] = {"vis": r(M, N, 1), "feature": torch.nn.functional.normalize(rn(M, N, 16), dim=-1), "xy_reproj": 128 + 30 * rn(M, N, 2),
                     "gauss_mask": r(M, N, 1)}
        rendered["gauss_mask"] = aux["fg"]["gauss_mask"]
    if field_type in ("bg", "comp"):
        aux["bg"] = {"vis": r(M, N, 1)}
    if field_type == "comp":
        rendered["mask_fg"] = r(M, N, 1)
    batch = {"mask": r(M, N, 1) > 0.4, "vis2d": r(M, N, 1) > 0.1, "is_detected": torch.tensor([True] * (M - 1) + [False]),
             "rgb": r(M, N, 3), "depth": 1 + r(M, N, 1), "flow": 3 * rn(M, N, 2), "flow_uct": r(M, N, 1) - 0.3,
             "feature": torch.nn.functional.normalize(rn(M, N, 16), dim=-1), "hxy": torch.cat([128 + 40 * rn(M, N, 2), torch.ones(M, N, 1)], -1)}
    # exact zeros in a few places (the v > 0 selection must treat them like the reference)
    rendered["rgb"][0, :3] = batch["rgb"][0, :3]
    cv = lambda t: t.to(device=device, dtype=dtype) if t.dtype.is_floating_point else t.to(device)
    mv = lambda d: {k: (mv(v) if isinstance(v, dict) else cv(v)) for k, v in d.items()}
    return mv(rendered), mv(aux), mv(batch)


@pytest.mark.parametrize("field_type", ["fg", "bg", "comp"])
def test_recon_loss_oracle_is_the_reference(field_type):
    golden = np.load(GOLDEN)
    rendered, aux, batch = synth_loss_inputs(field_type)
    ours = LO.recon_losses(rendered, aux, batch, field_type, dict(CONFIG, field_type=field_type))
    keys = [str(k) for k in golden[f"loss/{field_type}/keys"]]
    assert list(ours) == keys
    for k in keys:
        ref = torch.from_numpy(golden[f"loss/{field_type}/{k}"])
        assert torch.equal(ours[k], ref), (k, float(ours[k]), float(ref))
