"""TEST INFRASTRUCTURE: oracle-backed CPU stand-ins for the C-ABI calls in `macvo_b200.ops`.

Purpose: run the HOST logic of the five B200 plugin classes (config handling, adapters, tensor shapes / dtypes / devices,
`GraphInput -> PGOInput`, the in-place side effects MAC-VO relies on) without a GPU, against a recorded run of
`Odometry/MACVO.py` (tests/test_macvo_integration.py). Every kernel call is answered by
the CPU oracle that the GPU parity tests pin the kernels to. Never imported by the product.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import covariance as ocov
from oracle import frontend as ofe
from oracle import keypoint as okp
from oracle import pgo as opgo


class _Cand:
    def __init__(self, h, w, device):
        self.req = None
        self.idx = torch.empty(h * w, dtype=torch.int32, device=device)     # (only its size / device are inspected)
        self.w = w


def install() -> None:
    from macvo_b200 import ops, plugins
    torch.Tensor.pin_memory = lambda self, *a, **k: self          # no CUDA driver here
    plugins._require_cuda = lambda device, who: torch.device(device)

    ops.corr_build = lambda f1, f2, mode=None: ofe.corr_volume(f1.float(), f2.float())
    ops.corr_lookup = lambda cost_maps, coords, rows=False: ofe.window_lookup(cost_maps, coords)

    def dense_postproc(est_flow, est_cov, bl_fx, epd=False, score=None):
        d = ofe.dense_postproc(est_flow, est_cov, bl_fx, 1.0, epd)        # (bl * fx) enters only as a product
        if score is not None:
            score.mock_cov = d["flow_cov"]
        return d
    ops.dense_postproc = dense_postproc

    def score_only(match_cov, score):
        score.mock_cov = match_cov
        score.generation += 1
    ops.score_only = score_only
    ops.CandidateList = _Cand

    def select_candidates(score, mask_width, max_match_cov, extra_mask, out):
        out.req = ("kp", score.mock_cov, score.ksize, mask_width, max_match_cov, extra_mask)
    ops.select_candidates = select_candidates

    def select_mapping_candidates(depth, depth_cov, mask_width, max_depth, max_depth_cov, out):
        out.req = ("map", depth, depth_cov, max_depth, max_depth_cov, mask_width)
    ops.select_mapping_candidates = select_mapping_candidates

    def sample_candidates_many(requests):
        outs = []
        for cand, num in requests:
            kind, *a = cand.req
            if kind == "kp":
                cov, ksize, mw, mc, mask = a
                outs.append(okp.cov_aware_select_nodepth(cov, num, ksize, mw, mc, mask))
            else:
                depth, dcov, md, mdc, mw = a
                outs.append(okp.mapping_select(depth, dcov, num, md, mdc, mw))
        return outs
    ops.sample_candidates_many = sample_candidates_many
    ops.sample_candidates = lambda cand, num: sample_candidates_many([(cand, num)])[0]
    ops.retrieve_pixels = lambda pixel_uv, scalar_map: ofe.retrieve_pixels(pixel_uv, scalar_map)

    def match_covariance(kp, depth_map, flow_cov, fx, fy, cx, cy, kernel_size=31, min_flow_cov=0.25, min_depth_cov=0.05,
                         match_cov_default=0.25, want_point=False, depth_cov=None, out_cov=None):
        cov = ocov.match_covariance(kp, depth_map, flow_cov, fx, fy, cx, cy, kernel_size, min_flow_cov, min_depth_cov,
                                    match_cov_default, depth_cov=depth_cov)
        return cov, None, torch.zeros(1, dtype=torch.int32)
    ops.match_covariance = match_covariance

    def motion_interpolate_(poses, need_interp):
        from oracle import map_processor as omp
        out, idx = omp.motion_interpolate(poses.numpy(), need_interp.numpy().astype(bool))
        poses.copy_(torch.from_numpy(out))
        return torch.tensor([len(idx)], dtype=torch.int32)
    ops.motion_interpolate_ = motion_interpolate_

    def pgo_solve(pos_Tw, kp2_uv, kp2_disp, uv_cov, disp_cov, intr, init_pose, cluster=0, **kw):
        g = opgo.GraphData(pos_Tw=pos_Tw.numpy(), kp2_uv=kp2_uv.numpy(), kp2_disp=kp2_disp.numpy().reshape(-1),
                           uv_cov=uv_cov.numpy(), disp_cov=disp_cov.numpy().reshape(-1), fx=intr[0], fy=intr[1],
                           cx=intr[2], cy=intr[3], baseline=intr[4], init_pose=init_pose.numpy().reshape(7))
        pose = opgo.lm_solve(g)
        return torch.tensor(np.asarray(pose)), torch.zeros(8, dtype=torch.float64)
    ops.pgo_solve = pgo_solve

    def pgo_solve_graph(graph_type, pos_Tw, intr, init_pose, kp2_uv=None, kp2_disp=None, uv_cov=None, disp_cov=None, pc_obs=None,
                        obs_cov=None, pts_cov=None, cluster=0, **kw):
        n = lambda t: None if t is None else t.double().cpu().numpy()
        K = pos_Tw.shape[0]
        z = np.zeros
        g = opgo.GraphData(pos_Tw=n(pos_Tw), kp2_uv=n(kp2_uv) if kp2_uv is not None else z((K, 2)),
                           kp2_disp=n(kp2_disp).reshape(-1) if kp2_disp is not None else z(K),
                           uv_cov=n(uv_cov) if uv_cov is not None else z((K, 3)),
                           disp_cov=n(disp_cov).reshape(-1) if disp_cov is not None else z(K), fx=intr[0], fy=intr[1],
                           cx=intr[2], cy=intr[3], baseline=intr[4], init_pose=n(init_pose).reshape(7), graph_type=graph_type,
                           pc_obs=n(pc_obs), obs_cov=n(obs_cov), pts_cov=n(pts_cov))
        return torch.tensor(np.asarray(opgo.lm_solve(g))), torch.zeros(8, dtype=torch.float64)
    ops.pgo_solve_graph = pgo_solve_graph
