"""CPU: the drop-in adapter reads the architecture and the per-frame tables out of live reference modules exactly as the
golden-vector harness does.  Needs the reference's lab4d package (a reference checkout, or its copy under oracle/_ref/)."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "ref_shims"))
import _install  # noqa: E402

pytestmark = pytest.mark.skipif(not _install.available(), reason="the reference's lab4d package is not present (oracle/_ref/)")


def test_adapter_reads_reference_modules():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import ref_harness as H
    import synth
    from lab4d_b200 import nnutils, spec

    mf = H.build_field("fg", "bob")
    field = mf.field_params["fg"]
    cfg = nnutils.config_from_module(field)
    assert cfg == spec.FG_BOB
    assert nnutils.config_from_module(H.build_field("bg", "rigid").field_params["bg"]) == spec.BG
    comp = H.build_field("fg", "comp_skel-quad_dense")
    assert nnutils.config_from_module(comp.field_params["fg"]) == spec.FG_COMP_QUAD
    _, _, _, ctabs, cgraph = H.run_field(comp, "fg", synth.synth_rays(2, 4), 4)
    with torch.no_grad():
        ctab = nnutils.tables_from_module(comp.field_params["fg"], cgraph[3])
    for k in ("dense_t_embed", "inst_dense_fwd", "inst_dense_bwd"):
        assert torch.equal(ctab[k], torch.from_numpy(ctabs[k])), k
    rays = synth.synth_rays(4, 4)
    feat, deltas, rend, tabs, graph = H.run_field(mf, "fg", rays, 8)
    samples = graph[3]
    with torch.no_grad():
        tab = nnutils.tables_from_module(field, samples)
    for k, v in tab.items():
        assert torch.allclose(v, torch.from_numpy(tabs[k]), atol=0, rtol=0), k
    # parameter names the renderer reads exist in the module
    names = dict(field.named_parameters())
    for k in spec.field_param_shapes(cfg):
        assert k in names and tuple(names[k].shape) == tuple(spec.field_param_shapes(cfg)[k]), k
    # no CPU fallback: on a CPU device the patched entry point fails loudly
    field.train()
    with pytest.raises(RuntimeError, match="CUDA"):
        nnutils.query_field(field, samples)


def test_install_rebinds_and_restores_the_reference_symbols():
    """install() / undo bookkeeping (no kernels run): every patched symbol is replaced and restored; with dqtorch=True the
    reference's quaternion operators keep working on CPU tensors (the reference's own functions stay in charge there)."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import ref_harness  # noqa: F401  (imports lab4d through the shims)
    import lab4d.engine.model as rmodel
    import lab4d.nnutils.deformable as rdef
    import lab4d.nnutils.multifields as rmf
    import lab4d.nnutils.nerf as rnerf
    import lab4d.utils.quat_transform as qt
    import lab4d.utils.render_utils as rru
    from lab4d_b200 import nnutils, render

    before = (rnerf.NeRF.query_field, rdef.Deformable.query_field, rru.render_pixel, rmodel.render_pixel, rmf.MultiFields.__dict__["compose_fields"],
              rmodel.dvr_model.compute_loss, qt.quaternion_mul, qt.quaternion_conjugate)
    undo = nnutils.install(dqtorch=True)
    try:
        assert rru.render_pixel is render.render_pixel and rmodel.render_pixel is render.render_pixel
        assert rmodel.dvr_model.compute_loss is nnutils.compute_loss
        assert rnerf.NeRF.query_field is not before[0] and rdef.Deformable.query_field is rnerf.NeRF.query_field
        assert qt.quaternion_mul is not before[6] and qt.quaternion_conjugate is not before[7]
        g = torch.Generator().manual_seed(0)
        q = torch.nn.functional.normalize(torch.randn(5, 4, generator=g), dim=-1)
        p = torch.randn(5, 3, generator=g)
        assert torch.equal(qt.quaternion_mul(q, p), before[6](q, p))           # CPU tensors: the reference's own function
        assert torch.equal(qt.quaternion_conjugate(q), before[7](q))
        assert torch.equal(qt.quaternion_apply(q, p), qt.quaternion_apply(q, p))
    finally:
        undo()
    after = (rnerf.NeRF.query_field, rdef.Deformable.query_field, rru.render_pixel, rmodel.render_pixel, rmf.MultiFields.__dict__["compose_fields"],
             rmodel.dvr_model.compute_loss, qt.quaternion_mul, qt.quaternion_conjugate)
    assert all(a is b for a, b in zip(after, before))
