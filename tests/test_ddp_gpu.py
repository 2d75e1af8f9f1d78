"""Data-parallel correctness on 2 GPUs (NCCL): the overlapped step vs all-reduce-after-backward vs one GPU on the
concatenated batch. Needs >= 2 visible GPUs; skipped on a single-GPU machine."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_overlapped_step_matches_plain_allreduce_and_single_gpu(tmp_path):
    out = tmp_path / "ddp.json"
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ddp_worker.py")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", "29541",
           worker, str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.load(open(out))
    assert res["tiles"] and res["ranks_equal"], res
    # same kernels, same data: only the order of the split-K / bias-gradient atomics differs between the two schedules
    assert res["A_vs_B_0"] < 1e-5 and res["A_vs_B_1"] < 1e-5, res
    # two ranks x B=4 averaged == one GPU with B=8 (different GEMM shapes -> different accumulation order and tile configs)
    assert res["A_vs_C_l2"] < 2e-3 and res["A_vs_C_worst_tensor_l2"] < 1e-2, res
    assert res["loss_mean_of_ranks_vs_global"] < 1e-5, res
