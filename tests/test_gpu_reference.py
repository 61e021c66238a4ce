"""GPU: the UNMODIFIED reference (its copy under oracle/_ref/, imported through oracle/ref_shims) with and without
lab4d_b200.nnutils.install(): the patched reference modules run the B200 kernels end to end through the reference's own
entry points (field.get_samples -> field.query_field -> render_pixel -> loss.backward(), and the eval-mode path of
lab4d/render.py), and are compared with the un-patched reference on CUDA.  Skipped where the copy is absent."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_shims"))
import _install  # noqa: E402

from util import rel_l2  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _install.available(), reason="the reference's lab4d package is not present (oracle/_ref/)")]
DEV = "cuda"


def _setup(field_type, motion, M, N, D, seed=0):
    import ref_harness as H
    import synth

    mf = H.build_field(field_type, motion, seed=seed).to(DEV)
    cat = "bg" if field_type == "bg" else "fg"
    field = mf.field_params[cat]
    H.set_n_depth(D)
    rays = synth.synth_rays(M, N, seed=seed + 1)
    Kinv, batch = H.make_batch(field, rays, DEV)
    g = torch.Generator().manual_seed(3)
    batch["feature"] = torch.nn.functional.normalize(torch.randn(M, N, 16, generator=g), dim=-1).to(DEV)
    return mf, field, Kinv, batch


def _run(field, Kinv, batch, train, coeff=None):
    from lab4d.utils.render_utils import render_pixel  # resolved at call time: the patched or the reference function

    torch.manual_seed(11)  # eikonal ray subsampling / feature-match candidates draw from torch's generators
    field.train(train)
    field.zero_grad()
    ctx = torch.enable_grad() if train else torch.no_grad()
    with ctx:
        samples = field.get_samples(Kinv, batch)
        feat, deltas, aux = field.query_field(samples, flow_thresh=None)
        rend = render_pixel(feat, deltas)
        grads = None
        if train:
            if coeff is None:
                g = torch.Generator().manual_seed(5)
                coeff = {k: torch.rand(v.shape, generator=g).to(DEV) / v[..., 0].numel() for k, v in sorted(rend.items()) if k != "eikonal"}
            loss = sum((coeff[k] * rend[k]).sum() for k in coeff)
            loss = loss + rend["eikonal"].mean()  # second-order term: the eikonal kernels in the patched run, autograd.grad(create_graph) in the reference
            if "xy_reproj" in aux:
                loss = loss + 1e-3 * aux["xy_reproj"].mean()
            loss.backward()
            grads = {k: p.grad.clone() for k, p in field.named_parameters() if p.grad is not None}
    return {k: v.detach() for k, v in rend.items()}, {k: v.detach() for k, v in aux.items()}, grads, coeff


@pytest.mark.parametrize("field_type,motion,dq", [("fg", "bob", False), ("bg", "rigid", False), ("fg", "bob", True)])
def test_patched_reference_trains_like_the_reference(field_type, motion, dq):
    """dq: also the reference's quaternion operators (lab4d.utils.quat_transform) on the quaternion kernels."""
    from lab4d_b200 import nnutils

    M, N, D = 4, 16, 32
    mf, field, Kinv, batch = _setup(field_type, motion, M, N, D)
    rend_ref, aux_ref, g_ref, coeff = _run(field, Kinv, batch, train=True)
    undo = nnutils.install(n_depth=D, dqtorch=dq)
    try:
        rend, aux, g, _ = _run(field, Kinv, batch, train=True, coeff=coeff)
    finally:
        undo()
    rows = [f"{k}={rel_l2(rend[k].cpu(), rend_ref[k].cpu()):.1e}" for k in sorted(rend_ref) if k in rend]
    print(f"[reference] {field_type}/{motion} train, rendered: " + " ".join(rows))
    assert set(rend) == set(rend_ref), set(rend) ^ set(rend_ref)
    assert rel_l2(rend["rgb"].cpu(), rend_ref["rgb"].cpu()) <= 1e-4
    for k in ("mask", "depth"):
        assert rel_l2(rend[k].cpu(), rend_ref[k].cpu()) <= 1e-4, k
    # eikonal term: same random ray subset (same generator draws), sdf gradient from the reverse chain on fp16 operands
    assert float((rend["eikonal"] != 0).float().mean()) == float((rend_ref["eikonal"] != 0).float().mean())
    assert rel_l2(rend["eikonal"].cpu(), rend_ref["eikonal"].cpu()) <= 2e-2
    assert set(aux) == set(aux_ref)
    for k in aux_ref:
        assert rel_l2(aux[k].cpu(), aux_ref[k].cpu()) <= 5e-3, k
    # every parameter the reference trains through this path receives the same gradient (ReLU-flip noise floor ~1e-2)
    rows, bad = [], []
    for k, gr in sorted(g_ref.items()):
        if float(gr.abs().max()) == 0.0:
            continue
        assert k in g, f"parameter {k} got no gradient through the patched path"
        e = rel_l2(g[k].cpu(), gr.cpu())
        rows.append(f"{k}={e:.1e}")
        if e > 3e-2:
            bad.append((k, e))
    print(f"[reference] {field_type}/{motion} gradients ({len(rows)} tensors): " + " ".join(rows))
    assert not bad, bad


def test_patched_reference_eval_mode():
    """lab4d/render.py path: dvr_model.evaluate -> query_field in eval mode (importance sampling, aabb masking, normals)."""
    from lab4d_b200 import nnutils

    M, N, D = 2, 32, 32
    mf, field, Kinv, batch = _setup("fg", "bob", M, N, D)
    import lab4d.nnutils.nerf as rnerf

    # the reference's importance_sampling takes n_depth as a keyword default (nerf.py:697): align it with D
    orig = rnerf.NeRF.importance_sampling
    rnerf.NeRF.importance_sampling = lambda self, *a, **k: orig(self, *a, **dict(k, n_depth=D))
    try:
        rend_ref, _, _, _ = _run(field, Kinv, batch, train=False)
        undo = nnutils.install(n_depth=D)
        try:
            rend, _, _, _ = _run(field, Kinv, batch, train=False)
        finally:
            undo()
    finally:
        rnerf.NeRF.importance_sampling = orig
    rows = [f"{k}={rel_l2(rend[k].cpu(), rend_ref[k].cpu()):.1e}" for k in sorted(rend_ref) if k in rend]
    print("[reference] fg/bob eval, rendered: " + " ".join(rows))
    assert set(rend) == set(rend_ref), set(rend) ^ set(rend_ref)
    # importance samples sit on inverse-CDF discontinuities (tests/test_gpu_parity.py): a few rays move by a bin
    assert rel_l2(rend["rgb"].cpu(), rend_ref["rgb"].cpu()) <= 2e-3
    assert rel_l2(rend["mask"].cpu(), rend_ref["mask"].cpu()) <= 2e-3
    assert rel_l2(rend["normal"].cpu(), rend_ref["normal"].cpu()) <= 5e-2
