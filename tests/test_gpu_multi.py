"""The library's own NCCL communicator (caf_b200_comm_*, caf_b200_surface_sharded_*, caf_b200_peak_allgather_dev).
The 1-rank case runs on any GPU box; the 2-rank case needs two GPUs (it is skipped on a single-GPU box — the
hardware is absent, nothing falls back) and launches one process per GPU, exactly as bench.py is launched."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DATA, FS, ROOT


@pytest.mark.gpu
def test_world1_communicator_and_sharded_call(tmp_path, chirp0):
    from caf_cookoff_b200 import Handle, bench_shifts, surface_arrays
    from caf_cookoff_b200.dist import Comm
    needle, hay = chirp0
    h = Handle(0)
    comm = Comm(h, 1, 0, str(tmp_path / "id"))
    assert comm.shard(400) == (0, 400)
    freqs = bench_shifts()
    surf, pk = comm.surface_sharded(needle, hay, freqs, FS)
    ref, _, _, rpk = surface_arrays(needle, hay, freqs, FS, handle=h)
    assert np.array_equal(surf, ref)
    assert (pk.value, pk.freq_hz, pk.doppler_idx, pk.delay_idx) == (rpk.value, 69.0, 338, 202)
    comm.close()


@pytest.mark.gpu
def test_world2_rows_sharded_over_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "scripts", "mgpu_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    print(res.stdout[-2000:], res.stderr[-3000:])
    assert res.returncode == 0
    assert res.stdout.count("via the library's NCCL communicator") == 2
