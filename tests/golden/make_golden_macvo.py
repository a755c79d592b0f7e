"""Generate the fixtures of the tests that compare with MAC-VO as a whole by running the REFERENCE ITSELF on the CPU.

Needs the MAC-VO tree (MACVO_REFERENCE_ROOT):  python tests/golden/make_golden_macvo.py
The tests only read the fixtures, so they run wherever the repository does.

  macvo_run_<graph>.pt   the unmodified Odometry/MACVO.py with MAC-VO's own modules (CovAwareSelector_NoDepth,
                         MatchCovariance, MappingPointSelector, CovarianceSanityFilter, MotionInterpolate,
                         TwoFrame_PGO with graph type disp / icp / reproj) over 4 frames of synthetic.make_sequence(4, 192, 256)
                         with the synthetic:0 weights at decoder depth 4: every GraphInput the optimiser received with its
                         result, and the final map (tests/test_macvo_integration.py)
  macvo_registry.pt      for each module the B200 plugins replace: the interface MAC-VO files it under, its args in
                         Config/Experiment/MACVO/MACVO_Performant.yaml and which of them its `is_valid_config` requires
                         (tests/test_reference_registration.py)
  pypose_jacobian.pt     residual and analytic Jacobian of Analytic_ReprojDisp_TwoFramePGO at a pose far from identity on
                         cases.pgo_inputs(48, 6) (tests/test_pypose_conventions.py)
"""
from __future__ import annotations

import os
import sys
from types import SimpleNamespace as NS

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
os.environ.setdefault("TORCHDYNAMO_DISABLE", "1")

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests.golden import cases, refharness  # noqa: E402

SEQ = dict(n_frames=4, H=192, W=256)
NUM_POINT = 64
DECODER_DEPTH = 4


def save(name: str, obj: dict) -> None:
    path = os.path.join(HERE, name)
    torch.save(obj, path)
    print(f"wrote {name}: {os.path.getsize(path) / 1024:.1f} KiB")


def _t(v):
    v = v.tensor if hasattr(v, "tensor") and not isinstance(v, torch.Tensor) else v
    return torch.as_tensor(v).detach().as_subclass(torch.Tensor).clone()      # pypose LieTensors as plain tensors


def macvo_run(graph_type: str, weight_path: str) -> dict:
    import pypose as pp
    from DataLoader import StereoData, StereoFrame
    from Module.Optimization.TwoFramePGO.Optimizer import TwoFrame_PGO
    from Odometry.MACVO import MACVO
    from macvo_b200 import synthetic

    calls = []
    inner = TwoFrame_PGO.__dict__["_optimize"].__func__

    def recording(context, graph_data):
        context, out = inner(context, graph_data)
        obs, pts = graph_data.observations.data, graph_data.points.data
        calls.append({
            "obs": {k: _t(obs[k]) for k in ("pixel2_uv", "pixel2_d", "pixel2_disp", "pixel2_uv_cov", "pixel2_disp_cov", "obs2_covTc")},
            "pts": {k: _t(pts[k]) for k in ("pos_Tw", "cov_Tw")},
            "K": _t(graph_data.images_intrinsic), "baseline": _t(graph_data.baseline),
            "init_motion": _t(graph_data.init_motion), "frame_idx": _t(graph_data.frame_idx),
            "from_idx": _t(graph_data.from_idx), "motion": _t(out.motion)})
        return context, out

    TwoFrame_PGO._optimize = staticmethod(recording)
    torch.cuda.current_stream = lambda *a, **k: None     # _optimize only hands it to an inactive GPU timer
    try:
        cfg = NS(Odometry=NS(
            name="t", args=NS(device="cpu", edgewidth=32, num_point=NUM_POINT, match_cov_default=0.25, profile=False, mapping=True),
            cov=NS(obs=NS(type="MatchCovariance", args=NS(device="cpu", kernel_size=31, match_cov_default=0.25, min_depth_cov=0.05,
                                                          min_flow_cov=0.25))),
            keypoint=NS(type="CovAwareSelector_NoDepth", args=NS(device="cpu", kernel_size=7, mask_width=32, max_match_cov=100.0)),
            mappoint=NS(type="MappingPointSelector", args=NS(device="cpu", max_depth=5.0, max_depth_cov=0.005, mask_width=32)),
            frontend=NS(type="FlowFormerCovFrontend", args=NS(device="cpu", weight=weight_path, enc_dtype="fp32", dec_dtype="fp32",
                                                               decoder_depth=DECODER_DEPTH, enforce_positive_disparity=False)),
            motion=NS(type="StaticMotionModel", args=NS()), outlier=NS(type="CovarianceSanityFilter", args=NS()),
            postprocess=NS(type="MotionInterpolate", args=NS()), keyframe=NS(type="AllKeyframe", args=NS()),
            optimizer=NS(type="TwoFrame_PGO", args=NS(device="cpu", vectorize=True, parallel=False, graph_type=graph_type,
                                                      autodiff=False))))
        odo = MACVO[StereoFrame].from_config(cfg)
        torch.set_float32_matmul_precision("highest")
        torch.manual_seed(5)
        for i, f in enumerate(synthetic.make_sequence(SEQ["n_frames"], SEQ["H"], SEQ["W"])):
            sd = StereoData(T_BS=pp.identity_SE3(1), K=f.K, baseline=f.baseline, time_ns=f.time_ns, height=f.height,
                            width=f.width, imageL=f.imageL, imageR=f.imageR)
            odo.run(StereoFrame(idx=[i], time_ns=f.time_ns, stereo=sd))
        odo.terminate()
    finally:
        TwoFrame_PGO._optimize = staticmethod(inner)
    m = odo.get_map()
    return {"graph_type": graph_type, "seq": SEQ, "num_point": NUM_POINT, "decoder_depth": DECODER_DEPTH, "calls": calls,
            "poses": _t(m.frames.data["pose"]), "num_match": len(m.match), "num_points": len(m.points),
            "num_map_points": len(m.map_points), "pixel2_uv_cov": _t(m.match.data["pixel2_uv_cov"]),
            "obs2_covTc": _t(m.match.data["obs2_covTc"]), "pixel2_uv": _t(m.match.data["pixel2_uv"]),
            "pos_Tw": _t(m.points.data["pos_Tw"])}


def registry() -> dict:
    import yaml
    from Module import ICovariance2to3, IFrontend, IKeypointSelector, IOptimizer

    class Loader(yaml.SafeLoader):
        pass
    Loader.add_constructor("!include", lambda loader, node: None)
    with open(os.path.join(refharness.REFERENCE_ROOT, "Config", "Experiment", "MACVO", "MACVO_Performant.yaml")) as f:
        odom = yaml.load(f, Loader)["Odometry"]
    modules = {"frontend": odom["frontend"], "keypoint": odom["keypoint"], "mappoint": odom["mappoint"],
               "cov": odom["cov"]["obs"], "optimizer": odom["optimizer"]}
    from Utility.Extensions.Testable import ConfigTestable
    seen = []
    inner = ConfigTestable.__dict__["_enforce_config_spec"].__func__

    def recording(config, spec, allow_excessive_cfg=False):
        if isinstance(spec, dict) and not seen:
            seen.append((list(spec), allow_excessive_cfg))
        return inner(config, spec, allow_excessive_cfg)

    out = {}
    ConfigTestable._enforce_config_spec = staticmethod(recording)
    try:
        for role, m in modules.items():
            name, args = m["type"], dict(m["args"])
            iface = next(i for i in (IFrontend, IKeypointSelector, ICovariance2to3, IOptimizer) if name in i._SubclassRegistry__HIERARCHY)
            cls = iface.get_class(name)
            seen.clear()
            try:
                cls.is_valid_config(NS(**args))
            except KeyError:
                pass                        # MappingPointSelector: the YAML's `device` is not in the class's own spec
            keys, allow_excess = seen[0]
            accepted = {k: v for k, v in args.items() if k in keys}
            cls.is_valid_config(NS(**accepted))
            out[role] = {"type": name, "interface": iface.__name__, "spec_keys": sorted(keys), "args": accepted,
                         "yaml_args": args, "excess_rejected": not allow_excess}
    finally:
        ConfigTestable._enforce_config_spec = staticmethod(inner)
    return out


def pypose_jacobian() -> dict:
    import pypose as pp
    from Module.Map import MatchObs, PointNode
    from Module.Optimization.TwoFramePGO.Graphs import Analytic_ReprojDisp_TwoFramePGO, GraphInput
    from oracle import pgo as opgo
    K = 48
    c = cases.pgo_inputs(K, 6)
    obs = MatchObs.init({
        "pixel1_uv": torch.zeros(K, 2), "pixel2_uv": c["kp2_uv"], "pixel1_d": torch.zeros(K, 1), "pixel2_d": torch.zeros(K, 1),
        "pixel1_disp": torch.zeros(K, 1), "pixel2_disp": c["kp2_disp"].unsqueeze(-1),
        "pixel1_disp_cov": torch.zeros(K, 1), "pixel2_disp_cov": c["disp_cov"].unsqueeze(-1),
        "pixel1_d_cov": torch.zeros(K, 1), "pixel2_d_cov": torch.zeros(K, 1),
        "pixel1_uv_cov": torch.zeros(K, 3), "pixel2_uv_cov": c["uv_cov"],
        "obs1_covTc": torch.zeros(K, 3, 3, dtype=torch.double), "obs2_covTc": torch.zeros(K, 3, 3, dtype=torch.double)})
    pts = PointNode.init({"pos_Tw": c["pos_Tw"], "cov_Tw": torch.zeros(K, 3, 3, dtype=torch.double),
                          "color": torch.zeros(K, 3, dtype=torch.uint8)})
    start = torch.tensor(opgo.se3_exp(np.array([0.3, -0.1, 0.2, 0.25, -0.2, 0.15])), dtype=torch.float32)
    gi = GraphInput(torch.tensor([1]), torch.tensor([0]), pp.SE3(start.unsqueeze(0)), torch.tensor([c["baseline"]]), obs, pts,
                    c["K"], torch.zeros(K, dtype=torch.long), "cpu")
    graph = Analytic_ReprojDisp_TwoFramePGO(gi).to(dtype=torch.double)
    with torch.no_grad():
        r0 = graph.forward().clone()
        J = graph.build_jacobian().reshape(K, 3, 7).clone()
    return {"K": K, "case": (K, 6), "start": start, "pose": graph.pose2opt.detach().clone().as_subclass(torch.Tensor),
            "residual": r0.as_subclass(torch.Tensor).reshape(K, 3), "jacobian": J.as_subclass(torch.Tensor)}


def main() -> None:
    import tempfile
    refharness.install()
    torch.set_num_threads(8)
    import Module  # noqa: F401  (registers every plugin class)
    from macvo_b200.flowformer_cov import synthetic_state_dict
    save("pypose_jacobian.pt", pypose_jacobian())
    save("macvo_registry.pt", registry())
    with tempfile.TemporaryDirectory() as tmp:
        w = os.path.join(tmp, "w.pth")
        torch.save(synthetic_state_dict(0), w)
        for gt in ("disp", "icp", "reproj"):
            save(f"macvo_run_{gt}.pt", macvo_run(gt, w))


if __name__ == "__main__":
    main()
