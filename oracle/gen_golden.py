"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on CPU.

Run in the build container only:  python oracle/gen_golden.py
Each fixture holds the synthetic ray batch, the per-frame tables the reference's small MLPs
produced (inputs of the hot path), the reference's per-sample field outputs, its rendered pixels,
and gradient probes of a fixed scalar loss.  Weights are NOT stored: they are regenerated from
oracle/synth.synth_tensor(name, shape, seed, category).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as H  # noqa: E402
import synth  # noqa: E402

OUT = os.path.join(HERE, "..", "tests", "golden")

# keys whose per-parameter gradient is stored in full (small tensors); the rest get 3 probes
FULL_GRAD = ("sdf.", "rgb.2.", "logibeta", "logscale", "warp.logibeta", "log_gauss", "vis_mlp.basefield.linear_final",
             "delta_field.linear_final", "feature_field.linear_final")


def loss_coeffs(rendered, seed):
    rs = np.random.RandomState(4242 + seed)
    return {k: torch.from_numpy(rs.uniform(0.5, 1.5, tuple(v.shape)).astype(np.float32)) for k, v in sorted(rendered.items())}


def grad_probes(named_grads):
    out = {}
    for k, g in named_grads.items():
        g = g.detach().numpy().astype(np.float64)
        if any(s in k for s in FULL_GRAD) or g.size <= 4096:
            out["gfull/" + k] = g.astype(np.float32)
        r = synth.synth_tensor(k + ".probe", g.shape, 99).astype(np.float64)
        out["gprobe/" + k] = np.array([g.sum(), np.sqrt((g * g).sum()), (g * r).sum()], np.float64)
    return out


def one(name, field_type, motion, M, N, D, seed=0, flow_thresh=None, with_grad=True):
    torch.manual_seed(0)
    mf = H.build_field(field_type, motion, seed=seed)
    rays = synth.synth_rays(M, N, seed=seed)
    cats = list(mf.field_params.keys())
    pack = {"meta/M": M, "meta/N": N, "meta/D": D, "meta/seed": seed, "meta/flow_thresh": -1.0 if flow_thresh is None else flow_thresh}
    for k, v in rays.items():
        pack["rays/" + k] = v
    feats, dls, graphs = {}, {}, {}
    for cat in cats:
        if len(cats) > 1 and cat == "bg":
            # every field has its own near/far in the reference (nnutils/nerf.py near_far parameter); identical planes
            # would put fg and bg samples at exactly tied depths, whose order after argsort is arbitrary
            rays_c = dict(rays, near_far=rays["near_far"] * np.array([[0.93, 1.11]], np.float32))
            pack["bg/rays/near_far"] = rays_c["near_far"]
        else:
            rays_c = rays
        feat, deltas, rend, tabs, graph = H.run_field(mf, cat, rays_c, D, flow_thresh=flow_thresh)
        feats[cat], dls[cat], graphs[cat] = feat, deltas, graph
        for k, v in tabs.items():
            pack[f"{cat}/tab/{k}"] = v
        for k, v in feat.items():
            pack[f"{cat}/feat/{k}"] = v.numpy()
        pack[f"{cat}/deltas"] = deltas.numpy()
        for k, v in rend.items():
            pack[f"{cat}/rend/{k}"] = v.numpy()
        if with_grad:
            field = mf.field_params[cat]
            gfeat, gdel, grend, gsamples = graph
            coeff = loss_coeffs({k: v for k, v in grend.items() if k != "eikonal"}, seed)
            loss = sum((coeff[k] * grend[k]).sum() for k in coeff)
            field.zero_grad()
            loss.backward()
            pack[f"{cat}/loss"] = np.float64(loss.item())
            for k, c in coeff.items():
                pack[f"{cat}/coeff/{k}"] = c.numpy()
            named = {k: p.grad for k, p in field.named_parameters() if p.grad is not None}
            for k, v in grad_probes(named).items():
                pack[f"{cat}/{k}"] = v
    if len(cats) > 1:
        from lab4d.nnutils.multifields import MultiFields
        from lab4d.utils.render_utils import render_pixel

        fd, dl = MultiFields.compose_fields({c: feats[c] for c in cats}, {c: dls[c] for c in cats})
        rend = render_pixel(fd, dl)
        for k, v in fd.items():
            pack[f"comp/feat/{k}"] = v.numpy()
        pack["comp/deltas"] = dl.numpy()
        for k, v in rend.items():
            pack[f"comp/rend/{k}"] = v.numpy()
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **pack)
    print(name, "->", os.path.getsize(path) // 1024, "KiB;",
          {c: (float(pack[f"{c}/rend/mask"].min()), float(pack[f"{c}/rend/mask"].max())) for c in cats})


def one_importance(name, motion, M, N, D, seed=0):
    """Eval-mode NeRF.importance_sampling (nnutils/nerf.py:686-738) of the unmodified reference: merged depths, deltas."""
    torch.manual_seed(0)
    mf = H.build_field("fg", motion, seed=seed)
    rays = synth.synth_rays(M, N, seed=seed)
    field = mf.field_params["fg"]
    _, _, _, tabs, graph = H.run_field(mf, "fg", rays, D)   # training-mode pass: gives the per-frame tables / samples_dict
    samples = graph[3]
    field.eval()
    with torch.no_grad():
        xyz_cam, dir_cam, deltas, depth = field.importance_sampling(
            samples["hxy"], samples["Kinv"], samples["near_far"], samples["field2cam"], samples["frame_id"], samples["inst_id"],
            samples, n_depth=D)
    field.train()
    pack = {"meta/M": M, "meta/N": N, "meta/D": D, "meta/seed": seed}
    for k, v in rays.items():
        pack["rays/" + k] = v
    for k, v in tabs.items():
        pack["fg/tab/" + k] = v
    pack.update({"imp/xyz_cam": xyz_cam.numpy(), "imp/dir": dir_cam.numpy(), "imp/deltas": deltas.numpy(), "imp/depth": depth.numpy()})
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **pack)
    print(name, "->", os.path.getsize(path) // 1024, "KiB; depth range", float(depth.min()), float(depth.max()))


def reference_checks():
    """tests/golden/reference/checks.npz: the reference's own results on the seeded inputs of three tests - dvr_model's
    reconstruction losses (tests/test_loss_oracle_cpu.py), FeatureNeRF.global_match (tests/test_match_oracle_cpu.py) and
    quat_transform.quaternion_apply with its gradients (tests/test_gpu_quat.py).  A subdirectory: the field fixtures are every
    tests/golden/*.npz."""
    import copy

    sys.path.insert(0, os.path.join(HERE, "..", "tests"))
    import types

    import lab4d.utils.quat_transform as qt
    from lab4d.engine.model import dvr_model
    from lab4d.nnutils.feature import FeatureNeRF
    from test_gpu_quat import quat_apply_inputs
    from test_loss_oracle_cpu import CONFIG, synth_loss_inputs
    from test_match_oracle_cpu import CANDIDATES, match_inputs

    pack = {}
    for ft in ("fg", "bg", "comp"):
        rendered, aux, batch = synth_loss_inputs(ft)
        config = dict(CONFIG, field_type=ft)
        results = {"rendered": copy.deepcopy(rendered), "aux_dict": copy.deepcopy(aux)}
        if "fg" in aux:  # the reference reads gauss_mask from aux (render_samples puts every field's rendering there)
            results["aux_dict"]["fg"]["gauss_mask"] = results["rendered"]["gauss_mask"]
        ref = {}
        dvr_model.compute_recon_loss(ref, results, batch, config)
        dvr_model.mask_losses(ref, batch, config)
        dvr_model.apply_loss_weights(ref, config)
        pack[f"loss/{ft}/keys"] = np.array(list(ref))
        for k, v in ref.items():
            pack[f"loss/{ft}/{k}"] = v.detach().numpy()
    feat_px, feat_can, xyz, logsigma = match_inputs()
    for K in CANDIDATES:
        torch.manual_seed(5)
        pack[f"match/K{K}"] = FeatureNeRF.global_match(types.SimpleNamespace(logsigma=logsigma), feat_px, feat_can, xyz, num_candidates=K).numpy()
    q, p = (t.requires_grad_(True) for t in quat_apply_inputs())
    out = qt.quaternion_apply(q.expand(5, 7, 4), p)
    gq, gp = torch.autograd.grad(out.square().sum(), (q, p))
    pack.update({"quat_apply/out": out.detach().numpy(), "quat_apply/gq": gq.numpy(), "quat_apply/gp": gp.numpy()})
    path = os.path.join(OUT, "reference", "checks.npz")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, **pack)
    print(path, "->", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    one("bg_rigid_M2_N16_D16", "bg", "rigid", 2, 16, 16)
    one("fg_rigid_M4_N8_D16", "fg", "rigid", 4, 8, 16)
    one("fg_bob_M4_N8_D16", "fg", "bob", 4, 8, 16)
    one("fg_bob_M2_N4_D128_thresh", "fg", "bob", 2, 4, 128, seed=1, flow_thresh=40.0)
    one("comp_bob_M2_N8_D16", "comp", "bob", 2, 8, 16, seed=0, with_grad=False)
    one("fg_compquad_M4_N8_D16", "fg", "comp_skel-quad_dense", 4, 8, 16, seed=3)
    one("fg_skelhuman_M4_N8_D24", "fg", "skel-human", 4, 8, 24, seed=4)
    one_importance("imp_fg_bob_M2_N8_D32", "bob", 2, 8, 32, seed=5)
    reference_checks()
