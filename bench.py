"""Benchmark of the MAC-VO per-frame hot path (BASELINE.json metric: stereo frames/sec @640x480; corr-vol
HBM GB/s vs roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config performant|fast]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one stereo frame through the whole hot path: FlowFormerCov frontend (correlation volume +
12 x window lookup on the sm_100a kernels, dense layers through cuDNN/cuBLAS, CUDA graph) -> fused dense
post-processing + keypoint scoring -> candidate selection -> device-side observation building (gathers, 2 x observation
covariance, sanity filter, MatchObs packing) -> two-frame pose-graph LM solve -> mapping points, on a seeded synthetic TartanAir-shape 640x480 sequence with the
MACVO_Performant settings (fp32 network, 200 keypoints, mapping on). `value` keeps the images resident in
HBM; `e2e` goes through the plugin API with pinned HOST images (H2D inside the timed region) and reads the
optimised pose back every frame. N > 1 = N independent streams, one per GPU (BASELINE config 5:
"replicas only", no data-path collective), value = total frames / max-over-ranks time.

`--impl reference` times the reference's own CPU arithmetic (the oracle port, see oracle/) with all host
threads on `--steps` frames of the same workload (about 10 s per frame).

`--dump-outputs DIR` writes what the timed GPU path returned for its last step (bench.dump_outputs); the inputs are
seeded, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
os.environ.setdefault("TORCHDYNAMO_DISABLE", "1")

import torch  # noqa: E402

METRIC = "stereo frames/sec @640x480"
H, W = 480, 640
CONFIGS = {
    "performant": dict(enc_dtype="fp32", dec_dtype="fp32", num_point=200),     # Config/Experiment/MACVO/MACVO_Performant.yaml
    "fast": dict(enc_dtype="fp16", dec_dtype="bf16", num_point=2048),          # MACVO_Fast.yaml dtypes, BASELINE configs[2]: 2048 keypoints
}
SEQ_LEN = 8     # distinct synthetic frames, cycled (forwards / backwards) by the timed loop
SHARDED = dict(H=720, W=1280, num_point=4096)          # BASELINE configs[3]: one 1280x720 stream, GN blocks over N GPUs


def workload_name(cfg: dict) -> str:
    """one name for the workload, shared by both arms' `config`"""
    fast = cfg["enc_dtype"] != "fp32"
    return (f"640x480 synthetic stereo sequence, MACVO_{'Fast' if fast else 'Performant'} settings "
            f"({cfg['num_point']} keypoints, mapping on, decoder_depth 12), BASELINE configs[{2 if fast else 1}]")


def _dist():
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


class ClockSampler:
    """nvidia-smi style clock / throttle sampling during the timed region (pynvml)."""
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
            "hw_power_brake": 0x80}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self) -> dict:
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# --------------------------------------------------------------------------------------------------
# CPU arm (reference arithmetic = oracle port)
# --------------------------------------------------------------------------------------------------
def run_cpu(cfg: dict, frames_to_time: int, warm: int) -> dict:
    from macvo_b200 import synthetic
    from macvo_b200.flowformer_cov import synthetic_state_dict
    from macvo_b200.pipeline import TwoFrameOdometry
    from oracle import pipeline_cpu as pc
    dt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}
    # torch's CPU kernels stop scaling (and collapse from oversubscription) beyond ~16 threads on this workload:
    # 128 threads measured 178 s/frame on the GPU box against ~9 s/frame with 8; use what the path can use
    cores = min(os.cpu_count() or 1, int(os.environ.get("MACVO_BENCH_CPU_THREADS", 16)))
    torch.set_num_threads(cores)
    # the B200 frontend (like the reference's CUDA-graph frontend) sets matmul precision "medium" process-wide; the
    # reference's CPU path never does, and on CPUs with bf16 units "medium" changes fp32 matmuls -> pin "highest"
    prev_prec = torch.get_float32_matmul_precision()
    torch.set_float32_matmul_precision("highest")
    frames = synthetic.make_sequence(SEQ_LEN, H, W)
    torch.manual_seed(5)
    odo = TwoFrameOdometry(pc.CpuFrontend(synthetic_state_dict(0), dt[cfg["enc_dtype"]], dt[cfg["dec_dtype"]]),
                           pc.CpuSelector(), pc.CpuCovariance(), pc.CpuPGO(), num_point=cfg["num_point"],
                           map_selector=pc.CpuMapSelector())
    odo.initialize(frames[0])
    idx = 1
    for _ in range(warm):
        odo.run_pair(frames[idx % SEQ_LEN]); idx += 1
    t0 = time.perf_counter()
    for _ in range(frames_to_time):
        odo.run_pair(frames[idx % SEQ_LEN]); idx += 1
    odo.finish()
    dt_s = time.perf_counter() - t0
    torch.set_float32_matmul_precision(prev_prec)
    return {"value": frames_to_time / dt_s, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{frames_to_time} frame(s) of the same 640x480 workload after {warm} warm-up, "
                      f"{dt_s / frames_to_time:.2f} s/frame, torch CPU kernels with {cores} threads"}


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def build_gpu_pipeline(cfg: dict, device: str, fused: bool = True):
    from types import SimpleNamespace as NS
    from macvo_b200 import plugins
    from macvo_b200.pipeline import FusedTwoFrameOdometry, TwoFrameOdometry
    fe = plugins.B200_FlowFormerCovFrontend(NS(weight="synthetic:0", device=device, enc_dtype=cfg["enc_dtype"],
                                               dec_dtype=cfg["dec_dtype"], decoder_depth=12,
                                               enforce_positive_disparity=False, cuda_graph=True))
    sel = plugins.B200_CovAwareSelector_NoDepth(NS(device=device, kernel_size=7, mask_width=32, max_match_cov=100.0))
    msel = plugins.B200_MappingPointSelector(NS(max_depth=5.0, max_depth_cov=0.005, mask_width=32))
    cov = plugins.B200_MatchCovariance(NS(device=device, kernel_size=31, match_cov_default=0.25, min_depth_cov=0.05,
                                          min_flow_cov=0.25))
    pgo = plugins.B200_TwoFrame_PGO(NS(graph_type="disp", device=device, vectorize=True, parallel=False, autodiff=False))
    # fused: observation building / sanity filter / MatchObs packing / counted LM solve on the device, one host sync per
    # frame (pipeline.FusedTwoFrameOdometry); plugin-API: the call sequence Odometry/MACVO.py:173-337 makes
    cls = FusedTwoFrameOdometry if fused else TwoFrameOdometry
    return cls(fe, sel, cov, pgo, num_point=cfg["num_point"], map_selector=msel)


def time_corr_kernel(device: str, iters: int = 10) -> dict:
    """achieved HBM GB/s of the correlation-volume build at the workload's shape (B=2, D=256, N=4800)."""
    from macvo_b200 import ops
    g = torch.Generator().manual_seed(2)
    # channels_last like the network's `channel_convertor` output (cuDNN NHWC): the operand pre-pass is then elementwise
    f1 = (torch.randn(2, 256, H // 8, W // 8, generator=g) * 0.5).to(device).contiguous(memory_format=torch.channels_last)
    f2 = (torch.randn(2, 256, H // 8, W // 8, generator=g) * 0.5).to(device).contiguous(memory_format=torch.channels_last)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    for _ in range(3):
        ops.corr_build(f1, f2)
    times = []
    for _ in range(iters):
        flush.zero_()                                                      # evict L2 (126 MB) between launches
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.corr_build(f1, f2)                                             # enqueued on torch's current stream
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e) * 1e-3)
    n = (H // 8) * (W // 8)
    algo_bytes = 2 * (4 * n * n + 8 * n * 256)                             # SURVEY.md §8d: 4 N^2 + 2*4*N*D per pair
    mode = ops.default_corr_mode(256, n)
    return {"seconds": sum(times) / len(times), "bytes": algo_bytes, "mode": ops.CORR_MODE_NAMES[mode]}


def dump_outputs(odo, out_dir: str) -> None:
    """What the fused driver hands its caller for the last timed frame — the optimised pose, the frame's packed observations
    and mapping points — plus the whole trajectory, as <name>.npy (float32 / float64, counts as 1-element arrays); well under
    1 MB for every config. An array with no rows is not written: it holds nothing to compare (on the synthetic sequence no
    pixel passes the mapping selector's depth gates, so the mapping points are empty)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"pose": odo.latest_pose(), "trajectory": odo.finish()}
    for k, v in odo.observations().items():
        arrays[k] = torch.as_tensor(v).reshape(-1) if not torch.is_tensor(v) else v
    for k, v in arrays.items():
        v = v.detach().cpu()
        if v.numel() == 0:
            continue
        v = v.double() if v.dtype in (torch.float64, torch.int64, torch.int32) else v.float()
        np.save(os.path.join(out_dir, f"{k}.npy"), v.numpy())


def run_gpu(cfg: dict, steps: int, warmup: int, n_gpus: int, dump_dir: str | None = None) -> dict:
    rank, world, local = _dist()
    assert torch.cuda.is_available(), "bench.py (GPU arm) needs CUDA; use --impl reference for the CPU arm"
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(device))
    from macvo_b200 import build, ops, synthetic
    build.build(verbose=False)
    ops.load_library()

    frames_host = synthetic.make_sequence(SEQ_LEN, H, W, seed=1000 + rank, pin=True)
    frames_dev = []
    for f in frames_host:
        import copy
        fd = copy.copy(f)
        fd.imageL, fd.imageR = f.imageL.to(device), f.imageR.to(device)
        frames_dev.append(fd)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(frames, read_pose: bool, fused: bool = True):
        torch.manual_seed(5)
        odo = build_gpu_pipeline(cfg, device, fused)
        odo.initialize(frames[0])
        period = 2 * SEQ_LEN - 2                                          # ping-pong 0,1,..,7,6,..,1,0,1,...
        pp = lambda i: (i % period) if (i % period) < SEQ_LEN else period - (i % period)
        seq = [frames[pp(i)] for i in range(1, warmup + steps + 1)]
        # fused driver: the next frame is announced so its frontend is launched ahead of this frame's tail (software pipelining
        # across frames: pipeline.FusedTwoFrameOdometry.run_pair); every frame of the timed region is still uploaded, run through
        # the whole path and finished inside it (odo.finish() drains the last tail)
        # (the last warm-up step announces nothing: the first timed frame's frontend must be launched INSIDE the timed region, so
        # that the region holds exactly `steps` frontends and `steps` tails)
        step = (lambda i: odo.run_pair(seq[i], next_frame=seq[i + 1] if i + 1 < len(seq) and i != warmup - 1 else None)) if fused \
            else (lambda i: odo.run_pair(seq[i]))
        for i in range(warmup):
            step(i)
        barrier()
        ops.LAUNCHES[0] = 0
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.cuda.nvtx.range_push("macvo_timed")     # lets `ncu --nvtx --nvtx-include macvo_timed/` list exactly these launches
        last = None
        for i in range(warmup, len(seq)):
            step(i)
            if read_pose and fused:
                last = odo.latest_pose()                                  # D2H of the step's result (waits for this frame)
            elif read_pose and odo.optimizer.get_result() is not None:
                last = odo.optimizer.get_result().motion.cpu()            # D2H of the step's result (synchronises)
        odo.finish()
        torch.cuda.nvtx.range_pop()
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, ops.LAUNCHES[0], odo

    with ClockSampler(local) as clk:
        ms_dev, launches, odo_dev = timed(frames_dev, read_pose=False)
        if dump_dir and rank == 0:
            dump_outputs(odo_dev, dump_dir)
        del odo_dev
        ms_e2e, _, _ = timed(frames_host, read_pose=True)
        ms_api, _, _ = timed(frames_host, read_pose=True, fused=False)
    corr = time_corr_kernel(device)

    peaks_path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"
    traffic, traffic_src = None, None
    tpath = os.path.join(REPO, "profiles", "corr_tc_traffic.json")
    if os.path.exists(tpath):       # NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture
        tj = json.load(open(tpath))
        traffic = tj.get(corr["mode"], tj).get("dram_bytes_per_launch")
        traffic_src = tj.get(corr["mode"], tj).get("source")
    kernel_names = {"tf32": "macvo_corr_build: corr_tc_kernel<2> (tcgen05 kind::tf32, one pass over the fp32 K-major features, no pre-pass)",
                    "tc3": "macvo_corr_build: fp16 hi/lo operand split + corr_tc_kernel<3>",
                    "tc1": "macvo_corr_build: fp16 operand rounding + corr_tc_kernel<1>", "simt": "corr_simt_kernel"}
    achieved = corr["bytes"] / corr["seconds"] / 1e9
    out = {
        "metric": METRIC, "value": world * steps / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32" if cfg["enc_dtype"] == "fp32" else "f32 (MACVO_Fast fp16/bf16 request served by the TF32 pipeline, half_precision=tf32)",
        "data": "synthetic (seeded smoothed-noise TartanAir-shape stereo sequence, synthetic:0 network weights)",
        "config": {"workload": workload_name(cfg),
                   "streams": world, "parallelism": "replicas only (one independent stream per GPU, no collective)",
                   "l2": "per-frame working set (184 MB correlation volume + >1 GB activations) exceeds the 126 MB L2; "
                         "the corr roofline loop flushes L2 with a 256 MB write between launches",
                   "matmul_precision": "TF32 like the reference GPU frontend (Frontend.py:275-277): cuDNN / cuBLAS layers, our attention / "
                                       "PatchEmbed kernels and the correlation volume (kind::tf32); the decoder's SepConvGRU units and 3x3 / 1x1 "
                                       "convolutions on our tcgen05 kernels with fp16 operands (11-bit significand), fp32 accumulation "
                                       "and fp32 recurrent state; token path, LayerNorm, lookup, "
                                       "post-processing, covariance fp32; LM fp64. Parity of this mode at this shape: "
                                       "tests/test_gpu_parity_ladder.py (flow 9e-4 of its scale vs float64 truth; strict-fp32 mode 2.5e-6)"},
        # e2e: pinned HOST images in, optimised pose + the frame's packed observations / mapping points out, through the
        # package's public driver (FusedTwoFrameOdometry over the C ABI); each image crosses PCIe once (2 per frame)
        "e2e": {"value": world * steps / (ms_e2e * 1e-3), "unit": "frames/s",
                "h2d_bytes_per_step": 2 * 3 * H * W * 4 + 2 * 8 * 2200,
                "d2h_bytes_per_step": 7 * 8 + (31 * cfg["num_point"] + 4) * 8 + 2000 * (72 + 12) + 3 * 8},
        # the same frames through the plugin-API call sequence of Odometry/MACVO.py:173-337 (CPU fp64 covariances,
        # boolean indexing on the host's behalf: >= 7 host syncs per frame that the reference's API shape forces)
        "e2e_plugin_api": {"value": world * steps / (ms_api * 1e-3), "unit": "frames/s"},
        "gpu_launches": launches,
        "clocks": clk.summary(),
        "roofline": {"kernel": kernel_names[corr["mode"]] + ", B=2 D=256 N=4800, channels_last features (the mode the frontend "
                               "uses under its allow_tf32 setting)", "bound": "hbm",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": corr["bytes"],
                     "launch_seconds": corr["seconds"]},
    }
    if rank == 0 and world == 1:
        out["cpu_baseline"] = run_cpu(cfg, frames_to_time=1, warm=0)
    if world > 1:
        dist.destroy_process_group()
    return out if rank == 0 else {}


def run_sharded(steps: int, warmup: int, dump_dir: str | None = None) -> dict:
    """BASELINE configs[3]: ONE 1280x720 stream, 4096 keypoints, on N GPUs. Rank 0 owns the frontend, the selection and the
    device-side observation building; per frame it broadcasts the five LM input arrays (NCCL, 80 B per keypoint slot) and
    every rank solves its shard of residual blocks with the all-reduce of the 55-double accumulator fused into the persistent
    LM kernel over NVLink peer memory (sharded_pgo.FusedShardedPGO). Strong scaling of a 0.8 ms solve: reported to show where
    the exchange sits, not because it pays at K = 4096 (DESIGN.md §6 has the crossover table)."""
    import torch.distributed as dist
    rank, world, local = _dist()
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    from types import SimpleNamespace as NS
    from macvo_b200 import build, ops, plugins, synthetic
    from macvo_b200.pipeline import FusedTwoFrameOdometry
    from macvo_b200.sharded_pgo import FusedShardedPGO
    build.build(verbose=False)
    ops.load_library()
    Hs, Ws, KP = SHARDED["H"], SHARDED["W"], SHARDED["num_point"]
    fused = FusedShardedPGO() if world > 1 else None
    solver = (lambda obs, intr, pose_io, stats, min_k: fused.solve_packed(obs, intr, pose_io, stats, min_k)) if fused else None
    frames = synthetic.make_sequence(4, Hs, Ws, pin=True)
    n_total = warmup + steps
    intr = None
    if rank == 0:
        fe = plugins.B200_FlowFormerCovFrontend(NS(weight="synthetic:0", device=device, enc_dtype="fp32", dec_dtype="fp32",
                                                   decoder_depth=12, enforce_positive_disparity=False, cuda_graph=True))
        # NMS window 3 instead of MACVO_Performant's 7: with the random-weight stand-in network the 7x7 non-minimum suppression
        # leaves only ~200 candidates in a 1280x720 frame; 3x3 leaves > 4096, so that the solve really has 4096 residual blocks
        sel = plugins.B200_CovAwareSelector_NoDepth(NS(device=device, kernel_size=3, mask_width=32, max_match_cov=100.0))
        msel = plugins.B200_MappingPointSelector(NS(max_depth=5.0, max_depth_cov=0.005, mask_width=32))
        cov = plugins.B200_MatchCovariance(NS(device=device, kernel_size=31, match_cov_default=0.25, min_depth_cov=0.05, min_flow_cov=0.25))
        pgo = plugins.B200_TwoFrame_PGO(NS(graph_type="disp", device=device, vectorize=True, parallel=False, autodiff=False))
        torch.manual_seed(5)
        odo = FusedTwoFrameOdometry(fe, sel, cov, pgo, num_point=KP, map_selector=msel, solver=solver)
        odo.initialize(frames[0])
    else:
        obs = ops.ObservationBuffers(KP, device)
        pose_io = torch.zeros(7, dtype=torch.float64, device=device)
        stats = torch.zeros(8, dtype=torch.float64, device=device)
        K = frames[0].frame_K
        intr = (float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]),
                float(torch.as_tensor(frames[0].frame_baseline, dtype=torch.float32).double().reshape(-1)[0]))

    def step(i):
        if rank == 0:
            odo.run_pair(frames[1 + (i % 3)])
            return odo.latest_pose()
        fused.solve_packed(obs, intr, pose_io, stats, 10)
        return None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    with ClockSampler(local) as clk:
        for i in range(warmup):
            step(i)
        barrier()
        ops.LAUNCHES[0] = 0
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        last = None
        for i in range(warmup, n_total):
            last = step(i)
        e.record()
        barrier()
    ms = s.elapsed_time(e)
    poses_equal = None
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        mine = odo.pose_dev[-1].clone() if rank == 0 else pose_io.clone()
        gathered = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        poses_equal = all(torch.equal(g, gathered[0]) for g in gathered)
    if dump_dir and rank == 0:
        dump_outputs(odo, dump_dir)
    out = {}
    if rank == 0:
        o = odo.observations()
        out = {"metric": "stereo frames/sec @1280x720, 4096 keypoints, GN residual blocks sharded over the GPUs",
               "value": steps / (ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": warmup,
               "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic (seeded smoothed-noise 1280x720 stereo sequence, synthetic:0 network weights)",
               "config": {"workload": "1280x720 synthetic stereo stream, 4096 keypoints, decoder_depth 12, GN/LM residual blocks "
                                      "sharded over the GPUs, BASELINE configs[3]",
                          "parallelism": ("1 GPU: persistent LM kernel" if world == 1 else
                                          f"rank 0: frontend + observation building; per frame 2 NCCL broadcasts (LM inputs {80 * KP} B, "
                                          f"count+pose 64 B); {world} ranks: fused peer-memory all-reduce inside the LM kernel "
                                          "(no NCCL call inside the solve)"),
                          "num_obs_last_frame": o["num_obs"], "poses_bit_identical_on_all_ranks": poses_equal},
               "e2e": {"value": steps / (ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": 2 * 3 * Hs * Ws * 4,
                       "d2h_bytes_per_step": 7 * 8 + (31 * KP + 4) * 8},
               "gpu_launches": ops.LAUNCHES[0], "clocks": clk.summary()}
    if fused is not None:
        fused.close()
    if world > 1:
        dist.destroy_process_group()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="performant", choices=list(CONFIGS) + ["sharded"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned for its last step as DIR/<name>.npy (GPU arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    rank, world, _ = _dist()
    if a.config == "sharded":
        out = run_sharded(a.steps, a.warmup, a.dump_outputs)
        if rank == 0:
            print(json.dumps(out), flush=True)
        return
    cfg = CONFIGS[a.config]
    if a.impl == "reference":
        if rank != 0:
            return                                   # rank 0 alone runs the CPU arm
        steps = a.steps                              # ~10 s per 640x480 frame on 8 cores
        warm = min(a.warmup, 1)
        r = run_cpu(cfg, frames_to_time=steps, warm=warm)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "frames/s", "n_gpus": a.gpus,
                "steps": steps, "warmup": warm, "ms_per_step": 1e3 / r["value"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_name(cfg),
                           "arm": "CPU arithmetic of the reference (oracle port), "
                                  f"{steps} frame(s) of the same workload"},
                "cpu_baseline": r, "e2e": {"value": r["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return
    out = run_gpu(cfg, a.steps, a.warmup, a.gpus, a.dump_outputs)
    if rank == 0:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
