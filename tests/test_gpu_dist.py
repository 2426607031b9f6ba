"""GPU, >= 2 devices: the sharded product path over NCCL (optable_b200.dist.trace_sharded behind
OpticalTable.trace_bundle(group=...)) against the single-GPU trace of the same batch, and the C-ABI monitor merge.
One rank per GPU under torch.distributed.run; skipped on a single-GPU box (the host logic is covered by the gloo tests
in tests/test_dist_cpu.py, and `gpurun --gpus 2` runs this file: profiles/r2_dist_nccl_2gpu.log)."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_sharded_trace_over_nccl_equals_single_gpu():
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU under torch.distributed.run)")
    world = 2 if n < 4 else (4 if n < 8 else 8)
    run = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                          "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
                          os.path.join(ROOT, "tests", "dist_gpu_worker.py")], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert run.returncode == 0, run.stdout[-3000:] + run.stderr[-3000:]
    assert "DIST_OK" in run.stdout and run.stdout.count("DIST_CASE_OK") == 3 and "DIST_CABI_OK" in run.stdout, run.stdout[-3000:]
