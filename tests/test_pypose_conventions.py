"""Pins the two pypose conventions the LM restatement depends on to the REFERENCE'S OWN analytic Jacobian.

pypose 0.6.8 is not installable here, so `oracle/pypose_shim` restates it and SURVEY.md §8c calls that part "parity
unpinned". What CAN be pinned without the library: MAC-VO's authors wrote an analytic Jacobian for the two-frame graph
(Module/Optimization/TwoFramePGO/Graphs.py:201-230) and validated it against pypose's autograd with their
`verify_jacobian` (Module/Optimization/PyposeOptimizers.py:60-73). That Jacobian is only correct for ONE parameter-update
rule and ONE tangent ordering:

    d(T^-1 p_w) / d(delta) = [ -R^T | R^T [p_w]x ]    <=>    T <- Exp(delta) * T  (LEFT retraction),  delta = [tau, phi]

(under the right retraction T <- T * Exp(delta) it would be [ -I | [p_c]x ]). tests/golden/pypose_jacobian.pt holds the
reference graph's `forward()` and `build_jacobian()` at a pose far from identity (tests/golden/make_golden_macvo.py). The test
below pins the oracle's restatement of that residual (oracle/pgo.py) to the stored `forward()`, differentiates it numerically
under the shim's `Parameter.add_` and under the opposite (right) rule: the reference's analytic Jacobian must match the
former to 1e-6 and be far from the latter. The same check covers the shim's `Exp`, `Inv`, `rotation().matrix()` and
composition; the LM control flow itself (TrustRegion / StopOnPlateau) is MAC-VO's own `LM_analytic.step` executed verbatim
(tests/golden/make_golden.py)."""
import os
import sys

import numpy as np
import torch

from tests.golden import cases

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_analytic_jacobian_pins_left_retraction_and_tangent_order(golden):
    sys.path.insert(0, os.path.join(REPO, "oracle", "pypose_shim"))
    try:
        import pypose as pp
    finally:
        sys.path.remove(os.path.join(REPO, "oracle", "pypose_shim"))
    from oracle import pgo as opgo
    g = golden("pypose_jacobian.pt")
    K = g["K"]
    c = cases.pgo_inputs(*g["case"])
    graph = cases.pgo_graph(c)
    J = g["jacobian"].double()                                        # the REFERENCE's analytic Jacobian
    assert J.shape == (K, 3, 7) and (J[..., 6] == 0).all()
    base = g["pose"].double().reshape(1, 7)
    np.testing.assert_allclose(base.numpy()[0], g["start"].double().numpy(), rtol=0, atol=0)
    residual_at = lambda pose: torch.from_numpy(opgo.residual(graph, pose.reshape(7).numpy())[0])
    torch.testing.assert_close(residual_at(base), g["residual"].double(), rtol=1e-9, atol=1e-9)   # same residual as forward()

    def fd(rule):
        cols = []
        for k in range(6):
            e = torch.zeros(1, 7, dtype=torch.double)
            e[0, k] = 1e-6
            rp, rm = residual_at(rule(base, e)), residual_at(rule(base, -e))
            cols.append((rp - rm) / 2e-6)
        return torch.stack(cols, dim=-1)

    def left(pose, e):                      # what the shim's Parameter.add_ does (the optimiser's update, PyposeOptimizers.py:181)
        p = pp.Parameter(pp.SE3(pose.clone()))
        p.add_(e)
        return p.detach().as_subclass(torch.Tensor)

    def right(pose, e):                     # the opposite convention
        return (pp.SE3(pose.clone()) @ pp.se3(e[..., :6]).Exp()).as_subclass(torch.Tensor)

    with torch.no_grad():                   # like the optimiser's update
        J_left, J_right = fd(left), fd(right)
    scale = J[..., :6].abs().max().item()
    err_left = (J[..., :6] - J_left).abs().max().item() / scale
    err_right = (J[..., :6] - J_right).abs().max().item() / scale
    assert err_left < 1e-6, err_left
    assert err_right > 1e-2, err_right
    # tangent ordering: columns 0..2 must be the TRANSLATION part (-R^T): perturbing tau_k moves every point by the same camera-frame vector
    Rt = pp.SE3(base).rotation().matrix()[0].T
    pc = (pp.SE3(base).Inv() * c["pos_Tw"].double())
    x = pc[:, 0]
    # d r_disp / d tau = (-bl fx / x^2) * (-R^T)[0, :]
    fx, bl = c["K"][0, 0].double(), float(c["baseline"])
    expect = (-(bl * fx) / x.square()).unsqueeze(-1) * (-Rt[0:1, :])
    assert torch.allclose(J[:, 2, :3], expect, rtol=1e-9, atol=1e-12)
