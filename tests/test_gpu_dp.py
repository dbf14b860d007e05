"""Data-parallel step over NCCL on real GPUs (SURVEY.md 8a a20, 8e row 2): spawns `torchrun --nproc-per-node 2`
of tests/dp_gpu_worker.py when at least two GPUs are visible (skips otherwise) and requires the reduced
gradients, the bound and the post-update parameters to match the fp64 oracle on the FULL minibatch."""
import json
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


@pytest.mark.parametrize("p2p", ["1", "0"])       # 1: the tail kernel is the collective (peer memory); 0: ncclAllReduce
@pytest.mark.parametrize("world", [2])
def test_dp_step_matches_oracle_over_nccl(tmp_path, world, p2p):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    out = tmp_path / "dp.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "dp_gpu_worker.py"), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, VAEB_DP_P2P=p2p))
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    res = json.load(open(out))
    assert res["world"] == world and len(res["cases"]) == 3
    for c in res["cases"]:
        assert c["ranks_bit_identical"]
        assert c["bound_rel_err"] < (1e-2 if c["precision"] == "bf16" else 1e-4)
    print(json.dumps(res))
