"""GPU, >= 2 devices: sharded train step over NCCL == single-GPU full minibatch (SURVEY 4 multi-GPU
test: same clipped gradient within fp32 reduction-order tolerance; identical parameters on all ranks)."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from helpers import ROOT

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_train_step_matches_single_gpu(tmp_path):
    n = min(torch.cuda.device_count(), 4)
    out = str(tmp_path / "res.json")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mp_train_worker.py"), out]
    proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, start_new_session=True)
    try:
        out_txt, _ = proc.communicate(timeout=420)
    except subprocess.TimeoutExpired:
        import signal
        os.killpg(proc.pid, signal.SIGKILL)                 # exactly the process group this test started
        out_txt, _ = proc.communicate()
        raise AssertionError("multi-GPU worker timed out; output so far:\n" + out_txt[-4000:])
    assert proc.returncode == 0, out_txt[-4000:]
    res = json.load(open(out))
    assert res["world"] == n and res["params_identical"]
    assert res["grad_err"] <= 1e-4 * res["grad_max"] + 1e-8, res
    assert res["stats_err"] <= 1e-3, res
    assert res["captured_step_ok"], res       # CUDA-graph optimizer step with the NCCL all-reduce captured inside
