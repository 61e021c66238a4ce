"""fp16x3 forward (b200r_field_fwd / b200r_field_fwd_train, SPLIT instantiations): both tile groups' warps share one tile's
epilogues, so the tape and the per-sample outputs are written from two groups of threads.  Checks that the training
forward computes exactly what the inference forward does, that the point-warp entry with a tape gives the points it
gives without one, and that the tape (16-bit operand images and ReLU sign words) is the same on every run."""
import pytest
import torch

import synth
from lab4d_b200 import spec
from test_gpu_parity import synth_tables
from util import synth_params

pytestmark = pytest.mark.gpu
DEV = "cuda"
CFGS = {"fg_bob": spec.FG_BOB, "fg_skelhuman": spec.FG_SKEL_HUMAN, "fg_compquad": spec.FG_COMP_QUAD}
# (M frames, N rays, D samples): a small batch and the default benchmark's 2048 rays x 128 samples
SHAPES = [(2, 8, 16), (8, 256, 128)]


def _setup(name, M, N):
    from lab4d_b200.render import FieldRenderer

    cfg = CFGS[name]
    P = synth_params(cfg, 3, device=DEV)
    rays = {k: torch.from_numpy(v).to(DEV) for k, v in synth.synth_rays(M, N, seed=7).items()}
    tab = synth_tables(cfg, M, DEV, seed=7, rays=rays, P=P)
    r = FieldRenderer(cfg, DEV, operand_dtype="fp16x3")
    r.pack_train(P)
    return r, P, rays, tab


@pytest.mark.parametrize("M,N,D", SHAPES)
@pytest.mark.parametrize("name", sorted(CFGS))
def test_training_forward_equals_inference(name, M, N, D):
    r, P, rays, tab = _setup(name, M, N)
    feat_t, deltas_t, _ = r.query_field_train(P, rays, tab, D)
    feat_t = {k: v.clone() for k, v in feat_t.items()}
    deltas_t = deltas_t.clone()
    feat_i, deltas_i = r.query_field(P, rays, tab, D)
    torch.cuda.synchronize()
    assert torch.equal(deltas_t, deltas_i)
    common = sorted(k for k in feat_t if k in feat_i and k != "eikonal")
    assert {"rgb", "density", "xyz", "flow"} <= set(common), common
    bad = [k for k in common if not torch.equal(feat_t[k], feat_i[k])]
    assert not bad, bad


@pytest.mark.parametrize("M,N,D", SHAPES)
@pytest.mark.parametrize("name", sorted(CFGS))
def test_tape_is_deterministic(name, M, N, D):
    r, P, rays, tab = _setup(name, M, N)
    r.query_field_train(P, rays, tab, D)  # allocates the tape buffers
    tapes = []
    for _ in range(2):
        for b in r._tape_slots["field"]:
            b.zero_()  # bytes a run does not write compare equal
        feat, _, ctx = r.query_field_train(P, rays, tab, D)
        torch.cuda.synchronize()
        t = ctx["tape"]
        a, mask = r._tape_slots["field"][0], r._tape_slots["field"][2]
        off_a, off_m = t.a - a.data_ptr(), t.mask - mask.data_ptr()
        tapes.append((a[off_a:off_a + t.a_bytes].clone(), mask[off_m:off_m + t.mask_bytes].clone(), feat["rgb"].clone()))
    (a0, m0, rgb0), (a1, m1, rgb1) = tapes
    assert int(a0.count_nonzero()) > 0 and int(m0.count_nonzero()) > 0
    assert torch.equal(a0, a1), "operand images differ between runs"
    assert torch.equal(m0, m1), "sign words differ between runs"
    assert torch.equal(rgb0, rgb1)


@pytest.mark.parametrize("Pn", [16, 4096])
@pytest.mark.parametrize("name", sorted(CFGS))
def test_point_warp_with_and_without_tape(name, Pn):
    M = 4
    r, P, rays, tab = _setup(name, M, 4)
    g = torch.Generator().manual_seed(Pn)
    xyz = (0.12 * torch.randn(M, Pn, 3, generator=g)).to(DEV)
    out_t, _ = r.warp_points_train(P, xyz, tab)
    out_t = out_t.clone()
    out_i, _ = r.warp_points(P, xyz, tab, backward=False)
    torch.cuda.synchronize()
    assert torch.equal(out_t, out_i.view(M, Pn, 3))
