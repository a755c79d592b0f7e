"""Multi-GPU tests (need >= 2 GPUs of one node: `gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py -m gpu`;
skipped on a single-GPU box). BASELINE config 4: GN / LM residual blocks sharded across ranks, one process per GPU.

  * fused path: `sharded_pgo.FusedShardedPGO` — the whole LM loop is one persistent launch per rank, the all-reduce of
    the 55-double accumulator is fused into the kernel over NVLink peer memory (csrc/pgo.cu::exchange_ranks);
  * NCCL baseline: `sharded_pgo.solve_on_gpus` — host-driven loop, `ops.pgo_accumulate` + `dist.all_reduce` per evaluation.
Asserted: every rank ends with the SAME BITS; both paths reproduce the single-GPU persistent kernel (`ops.pgo_solve`) and
the fp64 oracle to 1e-8 with the same accept / reject sequence (steps / evaluations)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank: int, world: int, port: int, out_q):
    sys.path.insert(0, REPO)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = f"cuda:{rank}"
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(dev))
    from macvo_b200 import ops, sharded_pgo as sp
    from tests.golden import cases
    fused = sp.FusedShardedPGO()
    res = {}
    for K, seed in ((64, 6), (512, 6), (200, 9), (4096, 6)):
        c = cases.pgo_inputs(K, seed)
        f64 = lambda t: t.double().to(dev)
        Kt = c["K"].double()
        intr = (Kt[0, 0].item(), Kt[1, 1].item(), Kt[0, 2].item(), Kt[1, 2].item(), float(torch.tensor([c["baseline"]]).double()))
        full = [f64(c[k]) for k in ("pos_Tw", "kp2_uv", "kp2_disp", "uv_cov", "disp_cov")]
        init = f64(c["init_pose"])
        for rep in range(2):                                   # twice: round numbering persists across launches
            pose_f, st_f = fused.solve(*full, intr, init)
        pose_n, st_n = sp.solve_on_gpus(*full, intr, init)
        pose_1, st_1 = ops.pgo_solve(*full, intr, init)
        torch.cuda.synchronize()
        res[(K, seed)] = dict(fused=pose_f.cpu().numpy(), fused_stats=st_f.cpu().numpy(), nccl=pose_n.cpu().numpy(),
                              nccl_stats=st_n, single=pose_1.cpu().numpy(), single_stats=st_1.cpu().numpy())
    fused.close()
    out_q.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("world", [2, 4])
def test_fused_sharded_pgo_matches_single_gpu_and_oracle(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    from oracle import pgo as opgo
    from tests.golden import cases
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + (os.getpid() % 2000) + world
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for (K, seed), r0 in results[0].items():
        trace = opgo.LMTrace()
        ref = opgo.lm_solve(cases.pgo_graph(cases.pgo_inputs(K, seed)), trace=trace)
        for r in range(1, world):
            np.testing.assert_array_equal(results[r][(K, seed)]["fused"], r0["fused"])     # identical bits on every rank
            np.testing.assert_array_equal(results[r][(K, seed)]["nccl"], r0["nccl"])
        np.testing.assert_allclose(r0["fused"], ref, rtol=1e-8, atol=1e-9)
        np.testing.assert_allclose(r0["nccl"], ref, rtol=1e-8, atol=1e-9)
        np.testing.assert_allclose(r0["fused"], r0["single"], rtol=1e-9, atol=1e-10)
        assert int(r0["fused_stats"][0]) == trace.steps and int(r0["fused_stats"][1]) == trace.evaluations
        assert r0["nccl_stats"]["steps"] == trace.steps and r0["nccl_stats"]["evaluations"] == trace.evaluations
