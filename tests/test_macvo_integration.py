"""The five B200 plugin classes against a recorded run of the REAL, unmodified `Odometry/MACVO.py` with MAC-VO's own
modules: 4 frames of `MACVO.run` (`initialize`, `run_pair`, `get_graph_data` -> `TwoFrame_PGO._optimize(GraphInput)` ->
`write_graph_data`, mapping branch) -> `terminate` (MotionInterpolate), stored per optimiser graph type in
tests/golden/macvo_run_<graph>.pt by tests/golden/make_golden_macvo.py. No GPU here: every C-ABI call is answered by the
CPU oracle (tests/mock_ops.py), so what this pins is the plugin HOST logic:

  (a) every GraphInput MAC-VO handed its optimiser goes through `B200_TwoFrame_PGO` (the GraphInput -> PGOInput adapter
      of graph types disp / icp / reproj) and must give the reference optimiser's motion;
  (b) the plugins driven in MAC-VO's call order (Odometry/MACVO.py:158-378) — the transposed `flow_cov` view of
      MACVO.py:231-232 that the covariance clamps in place and that becomes `pixel2_uv_cov`, (K,1) disparities, the
      `pp.SE3` initial motion, CPU float64 covariances — must rebuild the same optimiser inputs and end in the same map:
      same number of observations, same covariances, same poses."""
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = r'''
import sys, os, torch
sys.path.insert(0, %r)
os.environ["TORCHDYNAMO_DISABLE"] = "1"
from types import SimpleNamespace as NS
import macvo_b200.plugins as P
from macvo_b200 import synthetic
from macvo_b200.pipeline import quat_rotate, se3_act
from tests import mock_ops
mock_ops.install()
g = torch.load(sys.argv[1], weights_only=False)
gt = g["graph_type"]
pgo_args = NS(device="cpu", vectorize=True, parallel=False, graph_type=gt, autodiff=False)

# (a) the recorded GraphInputs through the optimiser plugin
opt = P.B200_TwoFrame_PGO(pgo_args)
for c in g["calls"]:
    gi = NS(observations=NS(data=c["obs"]), points=NS(data=c["pts"]), images_intrinsic=c["K"], baseline=c["baseline"],
            init_motion=c["init_motion"], frame_idx=c["frame_idx"], from_idx=c["from_idx"])
    opt.start_optimize(gi)
    torch.testing.assert_close(opt.get_result().motion.double().reshape(1, 7), c["motion"].double().reshape(1, 7), rtol=1e-4, atol=1e-4)

# (b) the plugins in MAC-VO's call order
def quat_matrix(q):
    return torch.stack([quat_rotate(q, e) for e in torch.eye(3, dtype=q.dtype)], dim=-1)

fe = P.B200_FlowFormerCovFrontend(NS(device="cpu", weight="synthetic:0", enc_dtype="fp32", dec_dtype="fp32",
                                     decoder_depth=g["decoder_depth"], enforce_positive_disparity=False, cuda_graph=False))
sel = P.B200_CovAwareSelector_NoDepth(NS(device="cpu", kernel_size=7, mask_width=32, max_match_cov=100.0))
msel = P.B200_MappingPointSelector(NS(max_depth=5.0, max_depth_cov=0.005, mask_width=32))
cov = P.B200_MatchCovariance(NS(device="cpu", kernel_size=31, match_cov_default=0.25, min_depth_cov=0.05, min_flow_cov=0.25))
filt = P.B200_CovarianceSanityFilter(NS())
post = P.B200_MotionInterpolate(NS(device="cpu"))
opt = P.B200_TwoFrame_PGO(pgo_args)
torch.set_float32_matmul_precision("highest")     # the B200 frontend switches to "medium" like the reference CUDA frontend
torch.manual_seed(5)
ew, mcd = 32, 0.25
frames = synthetic.make_sequence(g["seq"]["n_frames"], g["seq"]["H"], g["seq"]["W"])
poses = [torch.tensor([0., 0., 0., 0., 0., 0., 1.])]
uv_cov_all, obs2_all, n_map, calls = [], [], 0, []
frame0, depth0 = frames[0], fe.estimate_depth(frames[0])
for t, frame1 in enumerate(frames[1:], start=1):
    depth1, match01 = fe.estimate_pair(frame0, frame1)
    if opt.get_result() is not None:                                  # write_map: the previous frame's result
        poses[-1] = opt.get_result().motion.reshape(7).float()
    prev_pose = poses[-1]
    kp0_uv = sel.select_point(frame0, g["num_point"], depth0, depth1, match01)
    kp1_uv = kp0_uv + fe.retrieve_pixels(kp0_uv, match01.flow).T
    inb = (kp1_uv[:, 0] > ew) & (kp1_uv[:, 0] < frame1.width - ew) & (kp1_uv[:, 1] > ew) & (kp1_uv[:, 1] < frame1.height - ew)
    kp0_uv, kp1_uv = kp0_uv[inb], kp1_uv[inb]
    n = kp0_uv.size(0)
    kp0_d = fe.retrieve_pixels(kp0_uv, depth0.depth).squeeze(0)
    kp1_d = fe.retrieve_pixels(kp1_uv, depth1.depth).squeeze(0)
    kp1_disp = fe.retrieve_pixels(kp1_uv, depth1.disparity)
    kp1_sigma_disp = fe.retrieve_pixels(kp1_uv, depth1.disparity_uncertainty)
    kp0_sigma_uv = torch.ones((n, 3)) * mcd
    kp0_sigma_uv[:, 2] = 0.
    kp1_sigma_uv = fe.retrieve_pixels(kp0_uv, match01.cov).T          # a transposed VIEW, clamped in place below
    K = frame0.frame_K
    pos0_Tc = torch.stack([kp0_d, (kp0_uv[:, 0] - K[0, 2]) / K[0, 0] * kp0_d, (kp0_uv[:, 1] - K[1, 2]) / K[1, 1] * kp0_d], -1)
    pos0_cov = cov.estimate(frame0, kp0_uv, depth0, fe.retrieve_pixels(kp0_uv, depth0.cov).squeeze(0), kp0_sigma_uv)
    pos1_cov = cov.estimate(frame1, kp1_uv, depth1, fe.retrieve_pixels(kp1_uv, depth1.cov).squeeze(0), kp1_sigma_uv)
    assert pos1_cov.dtype == torch.float64 and not pos1_cov.is_cuda
    keep = filt.filter(NS(data={"obs1_covTc": pos0_cov, "obs2_covTc": pos1_cov}), torch.device("cpu"))
    R = quat_matrix(prev_pose[3:].float()).double()                   # fp32 rotation of the fp32 map pose, then promoted
    obs = {"pixel2_uv": kp1_uv[keep], "pixel2_d": kp1_d.unsqueeze(-1)[keep], "pixel2_disp": kp1_disp.T[keep],
           "pixel2_uv_cov": kp1_sigma_uv[keep], "pixel2_disp_cov": kp1_sigma_disp.T[keep], "obs2_covTc": pos1_cov[keep]}
    pts = {"pos_Tw": se3_act(prev_pose, pos0_Tc)[keep], "cov_Tw": (R @ pos0_cov @ R.T)[keep]}
    uv_cov_all.append(obs["pixel2_uv_cov"])
    obs2_all.append(obs["obs2_covTc"])
    poses.append(prev_pose.clone())                                   # StaticMotionModel
    gi = NS(observations=NS(data=obs), points=NS(data=pts), images_intrinsic=frame1.frame_K, baseline=frame1.baseline,
            init_motion=prev_pose.reshape(1, 7), frame_idx=torch.tensor([t]), from_idx=torch.tensor([t - 1]))
    calls.append((obs, pts))
    opt.start_optimize(gi)
    map0_uv = msel.select_point(frame0, 2000, depth0, depth1, match01)
    n_map += map0_uv.size(0)
    frame0, depth0 = frame1, depth1
poses[-1] = opt.get_result().motion.reshape(7).float()
fr = NS(data={"pose": torch.stack(poses), "need_interp": torch.zeros(len(poses), dtype=torch.bool)})
post.elaborate_map(fr)
got_poses = fr.data["pose"]

assert len(calls) == len(g["calls"])
for (obs, pts), c in zip(calls, g["calls"]):
    assert obs["pixel2_uv"].shape == c["obs"]["pixel2_uv"].shape, (obs["pixel2_uv"].shape, c["obs"]["pixel2_uv"].shape)
    torch.testing.assert_close(obs["pixel2_uv"].float(), c["obs"]["pixel2_uv"].float(), rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(obs["pixel2_disp"].float(), c["obs"]["pixel2_disp"].float(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(obs["pixel2_d"].float(), c["obs"]["pixel2_d"].float(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(pts["pos_Tw"].float(), c["pts"]["pos_Tw"].float(), rtol=1e-4, atol=1e-4)
    scale = c["pts"]["cov_Tw"].abs().amax(dim=(-1, -2), keepdim=True)              # R Sigma R^T: fp32 rotation, per-block scale
    assert ((pts["cov_Tw"] - c["pts"]["cov_Tw"]).abs() <= 2e-3 * scale).all()
got_uv_cov, got_obs2 = torch.cat(uv_cov_all), torch.cat(obs2_all)
assert got_uv_cov.size(0) == g["num_match"] == g["num_points"] and g["num_match"] > 100, (got_uv_cov.size(0), g["num_match"])
assert n_map == g["num_map_points"], (n_map, g["num_map_points"])
assert torch.isfinite(got_poses).all()
torch.testing.assert_close(got_poses.float(), g["poses"].float(), rtol=1e-4, atol=1e-4)          # poses of all 4 frames
torch.testing.assert_close(got_uv_cov.float(), g["pixel2_uv_cov"].float(), rtol=1e-4, atol=1e-6)   # the in-place clamp reached the map
torch.testing.assert_close(got_obs2.double(), g["obs2_covTc"].double(), rtol=1e-3, atol=1e-9)
assert (got_uv_cov[:, :2] >= 0.0625).all()
print("MACVO-INTEGRATION-OK", got_uv_cov.size(0), n_map)
''' % REPO


@pytest.mark.parametrize("graph_type", ["disp", "icp", "reproj"])
def test_b200_plugins_under_the_real_macvo_run_pair(graph_type):
    """`disp` is MACVO_Performant / Fast, `icp` Paper_Reproduce.yaml:108; a subprocess, because tests/mock_ops.py replaces
    the kernels process-wide"""
    golden = os.path.join(REPO, "tests", "golden", f"macvo_run_{graph_type}.pt")
    r = subprocess.run([sys.executable, "-c", CODE, golden], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, TORCHDYNAMO_DISABLE="1"))
    assert "MACVO-INTEGRATION-OK" in r.stdout, r.stdout[-2500:] + r.stderr[-3500:]
