"""The library's multi-GPU entry points (include/sourmash_b200.h "multi-GPU", csrc/comm.cu: NCCL inside the library)
against the one-process results and the oracle.  tests/workers/comm_worker.py is one rank; here it is started once
with a world of 1 (any GPU box) and once per GPU with a world of 2 (boxes with at least two GPUs -- NCCL refuses two
ranks on one device)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "workers", "comm_worker.py")


def _run_world(world, tmp_path, no_comm=False):
    id_file = str(tmp_path / ("nccl_id_%d" % world))
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD=str(world), LOCAL_RANK=str(r), COMM_ID_FILE=id_file, NO_COMM="1" if no_comm else "0")
        procs.append(subprocess.Popen([sys.executable, WORKER], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        outs.append((p.returncode, out))
    for r, (rc, out) in enumerate(outs):
        assert rc == 0 and "ok" in out, "rank %d failed:\n%s" % (r, out[-4000:])


def test_collectives_world_1(tmp_path):
    _run_world(1, tmp_path)


def test_collectives_without_a_communicator(tmp_path):
    _run_world(1, tmp_path, no_comm=True)


def test_collectives_world_2(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _run_world(2, tmp_path)


def test_collectives_world_4(tmp_path):
    import torch
    if torch.cuda.device_count() < 4:
        pytest.skip("needs four GPUs")
    _run_world(4, tmp_path)
