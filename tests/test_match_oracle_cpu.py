"""CPU: the oracle's global_match against the unmodified reference's FeatureNeRF.global_match
(lab4d/nnutils/feature.py:152-205) under the same random draw - the pin of the checker of the match kernels.  The
reference's results on these seeded inputs are stored in tests/golden/reference/checks.npz (oracle/gen_golden.py)."""
import os

import numpy as np
import torch

import lab4d_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "checks.npz")
CANDIDATES = (1024, 128)


def match_inputs():
    g = torch.Generator().manual_seed(3)
    M, N, D = 3, 5, 40
    feat_px = torch.nn.functional.normalize(torch.randn(M, N, 16, generator=g), dim=-1)
    feat_can = torch.nn.functional.normalize(torch.randn(M, N, D, 16, generator=g), dim=-1)
    xyz = 0.2 * torch.randn(M, N, D, 3, generator=g)
    return feat_px, feat_can, xyz, torch.tensor([0.7])


def test_global_match_oracle_is_the_reference():
    golden = np.load(GOLDEN)
    feat_px, feat_can, xyz, logsigma = match_inputs()
    for K in CANDIDATES:
        torch.manual_seed(5)  # the reference draws its candidates with torch.randperm after this seed
        idx = torch.randperm(xyz[..., 0].numel())[:min(K, xyz[..., 0].numel())]
        ours = O.global_match(feat_px, feat_can, xyz, logsigma, idx)
        assert torch.equal(ours, torch.from_numpy(golden[f"match/K{K}"])), K
