"""Multi-process coverage of the multi-GPU bank (bench.py --gpus N): gloo/world_size 2 on CPU for the layout arithmetic and the
decomposition it implies, the library bank over NCCL on real GPUs when the box has at least two."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def _free_port() -> int:
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return int(s.getsockname()[1])


def _launch(backend: str, world: int):
    port = _free_port()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "dist_worker.py"), "--backend", backend]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert "dist_worker ok" in proc.stdout, proc.stdout[-2000:]


def test_partition_sharding_decomposition_gloo_world2():
    _launch("gloo", 2)


@pytest.mark.gpu
def test_partition_sharding_nccl(gpu):
    if gpu.device_count() < 2:
        pytest.skip("needs two GPUs")
    _launch("nccl", 2)
