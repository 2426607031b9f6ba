"""GPU, >= 2 devices: sweeps sharded over GPUs by configuration over NCCL (`trace_sweep` / `SweepScene.trace` with
`group=`) against the one-GPU sweep, bit for bit, and the C-host recipe with optb_monitor_merge. One rank per GPU under
torch.distributed.run (tests/dist_sweep_gpu_worker.py); skipped on a single-GPU box (the host logic is covered by the
gloo tests in tests/test_dist_sweep_cpu.py)."""
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


def test_sharded_sweeps_over_nccl_equal_single_gpu():
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU under torch.distributed.run)")
    world = 2 if n < 4 else (4 if n < 8 else 8)
    run = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                          "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
                          os.path.join(ROOT, "tests", "dist_sweep_gpu_worker.py")], capture_output=True, text=True,
                         cwd=ROOT, timeout=900)
    print(run.stdout[-3000:])
    assert run.returncode == 0, run.stdout[-3000:] + run.stderr[-3000:]
    assert "SWEEP_DIST_OK" in run.stdout and run.stdout.count("SWEEP_CASE_OK") == 3 and "SWEEP_CABI_OK" in run.stdout, \
        run.stdout[-3000:]
