"""GPU parity of the quaternion operators (lab4d_b200/quaternion.py over csrc/quat.cu: the dqtorch extension of the reference,
lab4d/third_party/quaternion/src/quaternion.cu:29-217) against the pure-torch restatement with the CUDA kernels' semantics
(3-vectors are pure quaternions): product, conjugate, first and second derivatives.  fp32 elementwise: 1e-6."""
import os

import numpy as np
import pytest
import torch

from test_quat_cpu import conj, qmul
from util import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("B,D1,D2", [(1, 4, 4), (1000, 4, 4), (4097, 4, 3), (333, 3, 4), (70001, 3, 3)])
def test_quaternion_mul_and_its_two_derivatives(B, D1, D2):
    from lab4d_b200 import quaternion as Q

    g = torch.Generator().manual_seed(B)
    mk = lambda *s: torch.randn(*s, generator=g).to(DEV).requires_grad_(True)
    a, b, G = mk(B, D1), mk(B, D2), mk(B, 4)
    a2, b2, G2 = (t.detach().clone().requires_grad_(True) for t in (a, b, G))
    out, ref = Q.quaternion_mul(a, b), qmul(a2, b2)
    assert rel_l2(out.cpu(), ref.cpu()) <= 1e-6
    ga, gb = torch.autograd.grad(out, (a, b), G, create_graph=True)
    ra, rb = torch.autograd.grad(ref, (a2, b2), G2, create_graph=True)
    assert rel_l2(ga.cpu(), ra.cpu()) <= 1e-6 and rel_l2(gb.cpu(), rb.cpu()) <= 1e-6
    u1, u2 = torch.randn(B, D1, generator=g).to(DEV), torch.randn(B, D2, generator=g).to(DEV)
    ours = torch.autograd.grad((ga, gb), (G, a, b), (u1, u2))
    theirs = torch.autograd.grad((ra, rb), (G2, a2, b2), (u1, u2))
    for o, t, name in zip(ours, theirs, ("g_G", "g_a", "g_b")):
        assert rel_l2(o.cpu(), t.cpu()) <= 1e-6, name
    q = mk(B, 4)
    c = Q.quaternion_conjugate(q)
    assert torch.equal(c.detach(), conj(q.detach()))
    (gq,) = torch.autograd.grad(c, q, G.detach())
    assert torch.equal(gq, conj(G.detach()))


def quat_apply_inputs():
    g = torch.Generator().manual_seed(2)
    q = torch.nn.functional.normalize(torch.randn(5, 1, 4, generator=g), dim=-1)
    p = torch.randn(5, 7, 3, generator=g)
    return q, p


def test_quat_transform_runs_on_the_kernels():
    """nnutils.install(dqtorch=True): lab4d.utils.quat_transform.quaternion_apply (q p q*, vector part) on CUDA tensors goes
    through nnutils._dq_mul / _dq_conj; on the kernels it equals the reference's own results and gradients, with broadcasting
    operands (stored in tests/golden/reference/checks.npz by oracle/gen_golden.py)."""
    from lab4d_b200 import nnutils

    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "checks.npz"))
    q, p = (t.to(DEV).requires_grad_(True) for t in quat_apply_inputs())
    qe = q.expand(5, 7, 4)
    out = nnutils._dq_mul(nnutils._dq_mul(qe, p), nnutils._dq_conj(qe))[..., 1:]
    (gq, gp) = torch.autograd.grad(out.square().sum(), (q, p))
    for name, o in (("out", out.detach()), ("gq", gq), ("gp", gp)):
        assert rel_l2(o.cpu(), torch.from_numpy(golden[f"quat_apply/{name}"])) <= 1e-6, name
