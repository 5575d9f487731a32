"""parallel.match_dsc_many_sharded on real GPUs over NCCL: launches tests/mgpu_match_dsc_many_worker.py under torchrun on
2, 4 and 8 GPUs; every rank's result must equal its own 1-GPU match_dsc_many bit for bit.  Skipped below the needed GPU
count (NCCL refuses two ranks on one device); tests/test_match_dsc_many_cpu.py covers the gather on CPU and
tests/test_match_dsc_many.py the per-rank steps of simulated worlds on one GPU."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_match_dsc_many_on_n_gpus_equals_one_gpu(world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(29640 + world),
           os.path.join(REPO, "tests", "mgpu_match_dsc_many_worker.py")]
    r = subprocess.run(cmd, cwd=REPO, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and ("MGPU-DSC-MANY-OK %d" % world) in r.stdout, r.stdout[-4000:]
