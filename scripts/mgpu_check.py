"""N-GPU check of the library's own NCCL path (no torch.distributed on the data path): one process per GPU.
   python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 scripts/mgpu_check.py
torchrun is only the launcher here (RANK / LOCAL_RANK / WORLD_SIZE); the NCCL id travels through a file."""
import os, sys, tempfile
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from caf_cookoff_b200 import Handle, bench_shifts, read_file_c64, surface_arrays
from caf_cookoff_b200.dist import Comm

rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
# the path is unique per launch (torchrun's run id); Comm additionally checks a per-run nonce inside the file
id_path = os.environ.get("CAF_NCCL_ID_FILE") or os.path.join(tempfile.gettempdir(), "caf_nccl_id_%s_%s" % (
    os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", "x")))
import torch
torch.cuda.set_device(local)
h = Handle(local)
D = os.path.join(ROOT, "tests/golden/data/")
needle = read_file_c64(D + "chirp_0_raw.c64"); hay = read_file_c64(D + "chirp_0_T+202samp_F+69.25Hz.c64")[:4096]
freqs = bench_shifts()

def run_checks(comm):
    lib = h._lib
    lo, hi = comm.shard(freqs.size)
    surf, pk = comm.surface_sharded(needle, hay, freqs, 48000)
    assert (pk.freq_hz, pk.delay_idx, pk.doppler_idx) == (69.0, 202, 338), (pk.freq_hz, pk.delay_idx, pk.doppler_idx)
    ref, _, _, _ = surface_arrays(needle, hay, freqs[lo:hi], 48000, handle=h)
    assert np.array_equal(surf, ref), "sharded rows differ from the same rows computed alone"
    # device-resident variant: local peak stays on the device, packed there, all-gathered by NCCL
    nd = torch.from_numpy(needle).cuda(); hd = torch.from_numpy(hay).cuda(); fd = torch.from_numpy(freqs[lo:hi].copy()).cuda()
    rv = torch.empty(hi - lo, dtype=torch.float64, device="cuda"); ri = torch.empty(hi - lo, dtype=torch.int64, device="cuda")
    pkd = torch.zeros(4, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    rc = lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, 4096, fd.data_ptr(), hi - lo, 48000, None, rv.data_ptr(), ri.data_ptr(), pkd.data_ptr())
    assert rc == 0
    g = comm.peak_allgather_dev(pkd.data_ptr(), lo)
    assert (g.freq_hz, g.delay_idx, g.doppler_idx) == (69.0, 202, 338), (g.freq_hz, g.delay_idx, g.doppler_idx)
    # a tie across ranks resolves to the lowest global row: every rank reports the same value from its first row
    tie = torch.zeros(4, dtype=torch.int64, device="cuda")
    tie[0] = torch.tensor(np.float64(5.0).view(np.int64)); tie[1] = torch.tensor(np.float64(1.0).view(np.int64)); tie[2] = 0; tie[3] = 7
    torch.cuda.synchronize()
    t = comm.peak_allgather_dev(tie.data_ptr(), lo)
    assert (t.value, t.doppler_idx, t.delay_idx) == (5.0, 0, 7), (t.value, t.doppler_idx, t.delay_idx)
    # the fully asynchronous device path: local rows, find_peak packed in the kernel, ncclAllGather, device-side resolve
    outp = torch.zeros(4, dtype=torch.int64, device="cuda")
    comm.sharded_dev(nd.data_ptr(), hd.data_ptr(), 4096, fd.data_ptr(), hi - lo, lo, 48000, outp.data_ptr(),
                     row_val_dev=rv.data_ptr(), row_idx_dev=ri.data_ptr())
    h.sync()
    o = outp.cpu().numpy()
    assert (float(o.view(np.float64)[1]), int(o[3]), int(o[2])) == (69.0, 202, 338), o
    assert not comm.remote_error()
    # a rank that cannot compute its shard (fs = 0 is rejected before any launch) must still enter the collective: the
    # healthy ranks get CAF_B200_EREMOTE semantics (remote_error) instead of hanging in ncclAllGather
    from caf_cookoff_b200.api import CafError
    bad = (rank == world - 1) and world > 1
    try:
        comm.sharded_dev(nd.data_ptr(), hd.data_ptr(), 4096, fd.data_ptr(), hi - lo, lo, 0 if bad else 48000, outp.data_ptr())
        failed_here = False
    except CafError:
        failed_here = True
    h.sync()
    assert failed_here == bad
    if world > 1 and not bad:
        assert comm.remote_error(), "the peer's failure mark did not arrive"
    # many exchanges back to back (the mailbox transport alternates between two parities): values change every round
    for k in range(40):
        t2 = torch.zeros(4, dtype=torch.int64, device="cuda")
        val = 1.0 + ((k * 7 + rank * 3) % 11)
        t2[0] = torch.tensor(np.float64(val).view(np.int64)); t2[1] = torch.tensor(np.float64(float(k)).view(np.int64)); t2[2] = 0; t2[3] = k
        torch.cuda.synchronize()
        g2 = comm.peak_allgather_dev(t2.data_ptr(), lo)
        vals = [1.0 + ((k * 7 + r_ * 3) % 11) for r_ in range(world)]
        win = max(range(world), key=lambda r_: (vals[r_], -r_))
        assert (g2.value, g2.delay_idx) == (max(vals), k) and g2.doppler_idx == comm_shard_lo(win), (k, g2.value, g2.doppler_idx)


def comm_shard_lo(r_):
    return freqs.size * r_ // world


transports = []
for forced in (None, "0"):
    if forced is None:
        os.environ.pop("CAF_B200_P2P", None)
    else:
        os.environ["CAF_B200_P2P"] = forced
    comm = Comm(h, world, rank, id_path + ("_nccl" if forced else ""))
    transports.append("p2p mailbox kernel" if comm.uses_p2p() else "ncclAllGather")
    if forced == "0":
        assert not comm.uses_p2p()
    run_checks(comm)
    comm.close()
print(f"rank {rank}/{world}: rows ok, global peak (69.0 Hz, delay 202, row 338) via the library's NCCL communicator; exchange transports exercised: {transports}", flush=True)


# Sharded detection: every rank's merged list must be the list rank 0 gets from detecting the whole surface on one GPU,
# through the library's communicator (Comm.detect_sharded) and through torch.distributed (dist.detect_sharded).
import torch.distributed as tdist
from caf_cookoff_b200 import api
from caf_cookoff_b200.dist import detect_sharded
tdist.init_process_group("nccl", device_id=torch.device("cuda", local))
comm = Comm(h, world, rank, id_path + "_detect")
nd = torch.from_numpy(needle).cuda(); hd = torch.from_numpy(hay).cuda(); fd = torch.from_numpy(freqs.copy()).cuda()
S = torch.empty((freqs.size, 8192), dtype=torch.float64, device="cuda")
torch.cuda.synchronize()
assert h._lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, 4096, fd.data_ptr(), freqs.size, 48000,
                                     S.data_ptr(), None, None, None) == 0
kw = dict(guard_doppler=2, guard_delay=2, train_doppler=4, train_delay=16)
for det in ("detect", "cfar", "cfar_os"):
    out = torch.empty((16, 6 if det == "detect" else 8), dtype=torch.float64, device="cuda")
    cnt = torch.empty(1, dtype=torch.int64, device="cuda")
    N = api.cfar_train_cells(2, 2, 4, 16)
    args = (S.data_ptr(), 1, freqs.size, 8192, fd.data_ptr(), 16, out.data_ptr(), cnt.data_ptr())
    if det == "detect":
        api.detect_dev(*args, guard_doppler=2, guard_delay=2, handle=h)
    elif det == "cfar":
        api.detect_cfar_dev(*args, scale=api.cfar_scale(1e-6, N), handle=h, **kw)
    else:
        rk = (3 * N + 3) // 4
        api.detect_cfar_os_dev(*args, rank=rk, scale=api.cfar_os_scale(1e-6, N, rk), handle=h, **kw)
    h.sync()
    want = torch.cat([out.view(torch.int64).reshape(-1), cnt])
    ref = want.clone()
    tdist.broadcast(ref, 0)                                   # rank 0's whole-surface list
    assert torch.equal(want, ref), "the whole-surface call differs between ranks"
    args = (det, nd, hd, fd, 48000, 16)
    for name, fn in (("Comm", comm.detect_sharded), ("torch.distributed", detect_sharded)):
        res, c = fn(*args, **(kw if det != "detect" else dict(guard_doppler=2, guard_delay=2)))
        got = torch.cat([res.view(torch.int64).reshape(-1), c])
        assert torch.equal(got, ref), (det, name, int(c[0]), int(ref[-1]))
# a rank whose block detection is refused (a window beyond the limits) still enters the exchange; its peers get EREMOTE
# (through the library's communicator and through torch.distributed alike)
from caf_cookoff_b200.api import CafError
bad = world > 1 and rank == world - 1
for fn in (comm.detect_sharded, detect_sharded):
    try:
        fn("cfar", nd, hd, fd, 48000, 16, guard_doppler=2, guard_delay=2, train_doppler=40 if bad else 4,
           train_delay=16)
        status = 0
    except CafError as e:
        status = e.status
    assert status == (-1 if bad else (-7 if world > 1 else 0)), (fn, status)
comm.close()
tdist.destroy_process_group()
print(f"rank {rank}/{world}: sharded detect / CA-CFAR / OS-CFAR equal the whole-surface lists of rank 0", flush=True)
