"""OS-CFAR detection and its noise map on the GPU (caf_b200_surface_detect_cfar_os, caf_b200_detect_cfar_os_*_dev,
caf_b200_cfar_os_noise_*_dev) against oracle/cfar_os.py, bit for bit (include/caf_b200.h, DESIGN.md section 11)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import test_gpu_cfar as G
from caf_cookoff_b200 import _lib, api, bench_shifts
from conftest import FS
from oracle import cfar as F
from oracle import cfar_os as O
from test_cfar_os_reference import margins_db, planted_scene

pytestmark = pytest.mark.gpu

same, key, as_tuples, of_structs, map_equal, bits = G.same, G.key, G.as_tuples, G.of_structs, G.map_equal, G.bits


def default_rank(gr, gd, tr, tc):
    return (3 * F.train_cells(gr, gd, tr, tc) + 3) // 4


def run_dev(S, freqs, k_max, gr, gd, tr, tc, rank, scale, handle=None):
    """S [p][d][n] numpy (float64 or float32) -> (records [p][k_max] as tuples, counts [p]) through detect_cfar_os_*_dev"""
    import torch
    dev = torch.device("cuda", 0)
    p, d, n = S.shape
    ts = torch.from_numpy(np.ascontiguousarray(S)).to(dev)
    tf = torch.from_numpy(np.ascontiguousarray(freqs, dtype=np.float64)).to(dev)
    out = torch.zeros((p, k_max, 8), dtype=torch.float64, device=dev)
    cnt = torch.full((p,), -1, dtype=torch.int64, device=dev)
    api.detect_cfar_os_dev(ts.data_ptr(), p, d, n, tf.data_ptr(), k_max, out.data_ptr(), cnt.data_ptr(), rank=rank,
                           scale=scale, guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc,
                           f32=S.dtype == np.float32, handle=handle)
    torch.cuda.synchronize()
    recs = out.cpu().numpy().view(G.REC).reshape(p, k_max)
    return [as_tuples(recs[i]) for i in range(p)], [int(c) for c in cnt.cpu().numpy()]


def run_map(S, gr, gd, tr, tc, rank, handle=None):
    import torch
    dev = torch.device("cuda", 0)
    p, d, n = S.shape
    ts = torch.from_numpy(np.ascontiguousarray(S)).to(dev)
    out = torch.zeros((p, d, n), dtype=torch.float64, device=dev)
    api.cfar_os_noise_dev(ts.data_ptr(), p, d, n, out.data_ptr(), rank=rank, guard_doppler=gr, guard_delay=gd,
                          train_doppler=tr, train_delay=tc, f32=S.dtype == np.float32, handle=handle)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def check_against_reference(S, freqs, k_max, gr, gd, tr, tc, rank, scale, with_map=True):
    got, cnt = run_dev(S, freqs, k_max, gr, gd, tr, tc, rank, scale)
    noise = run_map(S, gr, gd, tr, tc, rank) if with_map else None
    for i in range(S.shape[0]):
        want = O.detect_cfar_os(S[i], freqs, k_max, gr, gd, tr, tc, rank, scale)
        assert cnt[i] == len(want)
        same(got[i], O.padded(want, k_max))
        if with_map:
            for x in got[i][:cnt[i]]:
                assert bits(x[6]) == bits(noise[i, x[2], x[3]])          # a record's noise is the map's cell
    return got, cnt


MAP_CASES = [  # (p, d, n, gr, gd, tr, tc, rank or None for ceil(3N/4))
    (3, 9, 300, 1, 1, 2, 16, None), (1, 3, 520, 0, 0, 32, 256, None), (1, 5, 9, 0, 1, 1, 3, 1),
    (2, 70, 1000, 2, 2, 4, 16, None), (1, 1, 64, 0, 2, 0, 5, 6), (2, 20, 300, 2, 3, 6, 20, 1),
    (1, 12, 200, 1, 1, 3, 9, 150),
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("case", MAP_CASES)
def test_dense_map_matches_reference_bit_for_bit(case, dtype):
    """Cells of a power law, NaN, -0.0 and +inf: the k_m-th smallest, edge rows and m = 0 cells included."""
    p, d, n, gr, gd, tr, tc, rank = case
    rank = rank or default_rank(gr, gd, tr, tc)
    rng = np.random.default_rng(hash(case) % 1000)
    S = (rng.random((p, d, n)) ** 3 * 1e3).astype(dtype)
    S[rng.random(S.shape) < 0.02] = -0.0
    S[rng.random(S.shape) < 0.01] = np.inf
    S[rng.random(S.shape) < 0.03] = np.nan
    got = run_map(S, gr, gd, tr, tc, rank)
    for i in range(p):
        map_equal(got[i], O.os_noise_map(S[i], gr, gd, tr, tc, rank)[0])


SHAPES = [  # (p, d, n, gr, gd, tr, tc, k_max): d = 1, 2, 3, 5 and 37 give tiles of 1, 2, 4, 8 and 16 rows
    (3, 1, 300, 0, 0, 0, 5, 7), (3, 2, 517, 1, 1, 1, 4, 16), (2, 3, 400, 1, 1, 2, 6, 9), (2, 5, 333, 1, 2, 2, 8, 30),
    (2, 37, 1000, 2, 3, 4, 16, 64), (1, 37, 600, 2, 3, 30, 253, 3), (4, 2, 9, 1, 1, 0, 3, 3), (2, 20, 257, 32, 1, 0, 2, 1),
    (1, 40, 520, 5, 40, 10, 20, 1024), (2, 33, 800, 2, 2, 30, 36, 40), (1, 37, 1000, 1, 1, 0, 1, 1024),
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_tie_heavy_surfaces_match_reference(shape, dtype):
    """Integers 0 ... 4 with NaN: many ties, and scales 1.0 and 2.0 put v == scale * x exactly on many training cells,
    which the counting step must not count as below v.  Every tile height, the largest windows (unstaged), k_max up to
    1024; a batch equals its pairs."""
    p, d, n, gr, gd, tr, tc, k_max = shape
    N = F.train_cells(gr, gd, tr, tc)
    rng = np.random.default_rng(hash(shape) % 1000)
    S = rng.integers(0, 5, size=(p, d, n)).astype(dtype)
    S[rng.random(S.shape) < 0.02] = np.nan
    freqs = np.cumsum(rng.random(d) + 0.05) - 3.0
    for rank, scale in ((default_rank(gr, gd, tr, tc), 1.0), ((N + 1) // 2, 2.0), (1, 2.0), (N, 0.7)):
        got, _ = check_against_reference(S, freqs, k_max, gr, gd, tr, tc, rank, scale, with_map=S.size * N < 4e7)
        one = [run_dev(S[i:i + 1], freqs, k_max, gr, gd, tr, tc, rank, scale)[0][0] for i in range(p)]
        assert [[key(x) for x in g] for g in got] == [[key(x) for x in o] for o in one]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_many_candidates_repeatable_and_handle_independent(dtype):
    """Noise with low scales: many qualifying maxima per tile, so the selection runs often, the per-tile cut and the pair
    floor work at k_max up to 1024; the same bits on every call and from a second handle."""
    rng = np.random.default_rng(5)
    S = (rng.random((2, 100, 4100)) ** 3).astype(dtype)
    freqs = np.linspace(-50.0, 50.0, 100)
    other = api.Handle(0)
    for k_max, gr, gd, tr, tc, scale in ((1024, 1, 1, 2, 16, 1.0), (200, 0, 0, 1, 1, 2.0), (33, 4, 17, 8, 40, 3.0),
                                         (16, 2, 2, 4, 16, 1.5)):
        rank = default_rank(gr, gd, tr, tc)
        got, _ = check_against_reference(S, freqs, k_max, gr, gd, tr, tc, rank, scale, with_map=False)
        for _ in range(2):
            assert run_dev(S, freqs, k_max, gr, gd, tr, tc, rank, scale)[0] == got
        assert run_dev(S, freqs, k_max, gr, gd, tr, tc, rank, scale, handle=other)[0] == got
    other.close()


SCENES = [  # (emitters, seed, the weak emitter's delay cell)
    ([(202, 69.0, 1.0), (230, 69.0, 0.15)], 7, 230),
    ([(202, 69.0, 1.0), (240, 66.0, 0.15)], 11, 240),
]


@pytest.mark.parametrize("variant", [api._Variant, api._Variant32], ids=["f64", "f32"])
@pytest.mark.parametrize("scene", range(len(SCENES)))
def test_os_finds_the_emitter_ca_misses(scene, variant):
    """On the bench grid, with the training region in delay only (guard 32 x 2, training 0 x 64) at Pfa 1e-6: CA-CFAR
    on the same surface misses the weak emitter inside the strong one's training region, OS-CFAR at rank 3N/4 finds it
    by >= 4 dB (5.0 and 5.6 dB in the seeded f64 references).  At the default 4 x 16 window the strong emitter's own Doppler
    lobe caps CA at ~6 dB and OS clears it by > 15 dB.  Lists bit for bit against the reference."""
    ems, seed, weak = SCENES[scene]
    shifts = bench_shifts()
    needle, hay = planted_scene(ems, seed)
    s = api.DeviceSurface(needle, hay, shifts, FS, variant=variant)
    S = s.fetch_rows()
    w = (32, 2, 0, 64)
    N = F.train_cells(*w)
    rank = default_rank(*w)
    a_ca, a_os = api.cfar_scale(1e-6, N), api.cfar_os_scale(1e-6, N, rank)
    ca = s.detect_cfar(16, *w)
    os_ = s.detect_cfar_os(16, *w)                                        # default rank and scale
    if variant is api._Variant:                                           # the reference takes ~15 s at this window
        same(of_structs(os_), O.detect_cfar_os(S, shifts, 16, *w, rank, a_os))
    m_ca, m_os = margins_db(of_structs(ca), a_ca), margins_db(of_structs(os_), a_os)
    assert weak not in m_ca and m_ca[202] > 20.0
    assert m_os[weak] > 4.0 and m_os[202] > 20.0
    w = (2, 2, 4, 16)
    N = F.train_cells(*w)
    rank = default_rank(*w)
    a_ca, a_os = api.cfar_scale(1e-6, N), api.cfar_os_scale(1e-6, N, rank)
    os_ = s.detect_cfar_os(16, *w, rank, a_os)
    same(of_structs(os_), O.detect_cfar_os(S, shifts, 16, *w, rank, a_os))
    assert margins_db(of_structs(os_), a_os)[202] > 15.0
    assert margins_db(of_structs(s.detect_cfar(16, *w)), a_ca)[202] < 7.0
    s.close()


def test_error_codes():
    import torch
    lib = _lib.load()
    h = api.Handle(0)
    needle, hay, _ = G.planted()
    s = api.DeviceSurface(needle[:64], hay[:64], np.linspace(-5, 5, 11), FS, handle=h)   # 11 x 128
    out = (_lib.CfarDetection * 1025)()
    C.memset(out, 0x5a, C.sizeof(out))
    before = bytes(out)
    cnt = C.c_size_t(77)
    N = F.train_cells(1, 1, 2, 16)
    for args in ((0, 1, 1, 2, 16, 10, 10.0), (1025, 1, 1, 2, 16, 10, 10.0), (4, 1, 1, 32, 16, 10, 10.0),
                 (4, 1, 1, 2, 63, 10, 10.0), (4, 1, 1, 0, 0, 1, 10.0), (4, 1, 1, 2, 16, 10, 0.0),
                 (4, 1, 1, 2, 16, 10, float("nan")), (4, 1, 1, 2, 16, 0, 10.0), (4, 1, 1, 2, 16, N + 1, 10.0)):
        assert lib.caf_b200_surface_detect_cfar_os(s.raw, *args, out, C.byref(cnt)) == -1, args
        assert cnt.value == 77 and bytes(out) == before
    assert lib.caf_b200_surface_detect_cfar_os(s.raw, 4, 1, 1, 2, 16, N, 10.0, out, C.byref(cnt)) == 0
    assert lib.caf_b200_surface_detect_cfar_os(s.raw, 4, 1, 1, 2, 16, 1, 10.0, None, C.byref(cnt)) == -1
    dev = torch.device("cuda", 0)
    S = torch.rand((1, 4, 16), dtype=torch.float64, device=dev)
    f = torch.zeros(4, dtype=torch.float64, device=dev)
    o = torch.full((1, 4, 8), 3.0, dtype=torch.float64, device=dev)
    c = torch.full((1,), 9, dtype=torch.int64, device=dev)
    nz = torch.full((1, 4, 16), 3.0, dtype=torch.float64, device=dev)
    P = lambda t: t.data_ptr()
    n2 = F.train_cells(1, 1, 0, 2)                                                      # 3 x 7 - 9 = 12
    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 7, 1, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 2, n2 + 1, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 2, 0, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, None, 1, 4, 16, P(f), 4, 1, 1, 0, 2, 1, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, P(S), 1, 4, 16, None, 4, 1, 1, 0, 2, 1, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_os_f32_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 2, 1, 2.0, None, P(c)) == -1
    assert lib.caf_b200_cfar_os_noise_f64_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 2, n2 + 1, P(nz)) == -1
    assert lib.caf_b200_cfar_os_noise_f64_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 2, 0, P(nz)) == -1
    assert lib.caf_b200_cfar_os_noise_f64_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 7, 1, P(nz)) == -1
    assert lib.caf_b200_cfar_os_noise_f32_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 2, 1, None) == -1
    torch.cuda.synchronize()
    assert bool((o == 3.0).all()) and int(c[0]) == 9 and bool((nz == 3.0).all())
    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, P(S), 1, 0, 16, P(f), 4, 1, 1, 0, 2, 1, 2.0, P(o), P(c)) == 0
    torch.cuda.synchronize()
    assert int(c[0]) == 0 and as_tuples(o.cpu().numpy().view(G.REC).reshape(4)) == [F.NONE] * 4
    h.close()
    assert lib.caf_b200_surface_detect_cfar_os(s.raw, 4, 1, 1, 2, 16, 10, 10.0, out, C.byref(cnt)) == -1
    assert "handle" in lib.caf_b200_last_error().decode()
    s.close()


def test_overlap_detect_cfar_os_between_surface_launches():
    """With overlap mode 4 and rotated outputs, detect_cfar_os calls between surface launches leave every surface and peak
    bit-identical to the serialised run, raise the launch count by two each, and give the reference's list."""
    import torch
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    lib = _lib.load()
    h = api.Handle(0, stream=stream.cuda_stream)
    L = 4096
    needle, hay, _ = G.planted()
    nd = torch.from_numpy(needle).to(dev)
    hd = torch.from_numpy(hay).to(dev)
    shifts = bench_shifts()
    fd = torch.from_numpy(shifts).to(dev)
    K, NB = 12, 9
    rank = default_rank(2, 2, 4, 16)

    def run(overlap, with_detect):
        lib.caf_b200_set_overlap(h.raw, overlap)
        surfs = [torch.zeros((400, 2 * L), dtype=torch.float64, device=dev) for _ in range(NB)]
        rv = torch.zeros((K, 400), dtype=torch.float64, device=dev); ri = torch.zeros((K, 400), dtype=torch.int64, device=dev)
        pk = torch.zeros((K, 4), dtype=torch.int64, device=dev)
        out = torch.zeros((K, 8, 8), dtype=torch.float64, device=dev); cnt = torch.zeros(K, dtype=torch.int64, device=dev)
        with torch.cuda.stream(stream):
            for k in range(K):
                sb = k % NB
                assert lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, L, fd.data_ptr(), 400, FS,
                                                  surfs[sb].data_ptr(), rv[k].data_ptr(), ri[k].data_ptr(), pk[k].data_ptr()) == 0
                if with_detect and k % 3 == 1:
                    before = h.launch_count
                    assert lib.caf_b200_detect_cfar_os_f64_dev(h.raw, surfs[sb].data_ptr(), 1, 400, 2 * L, fd.data_ptr(), 8,
                                                               2, 2, 4, 16, rank, 3.0, out[k].data_ptr(), cnt[k].data_ptr()) == 0
                    assert h.launch_count == before + 2
        torch.cuda.synchronize()
        return [x.cpu().numpy() for x in surfs], rv.cpu().numpy(), ri.cpu().numpy(), pk.cpu().numpy(), out.cpu().numpy(), cnt.cpu().numpy()

    want = run(0, False)
    got = run(4, True)
    for a, b in zip(want[0], got[0]):
        assert np.array_equal(a, b)
    for i in (1, 2, 3):
        assert np.array_equal(want[i], got[i])
    ref = O.detect_cfar_os(want[0][1], shifts, 8, 2, 2, 4, 16, rank, 3.0)
    assert len(ref) >= 1
    for k in range(1, K, 3):
        same(as_tuples(got[4][k].view(G.REC).reshape(8))[:int(got[5][k])], ref)
    lib.caf_b200_set_overlap(h.raw, 0)
    h.close()


def test_two_handles_alternate_large_and_small_windows():
    """The OS tile kernel's shared-memory allowance belongs to the device: a handle that ran small windows must not take
    it away from another handle's one-row tile that stages a ~200 KB training region, nor from the largest windows."""
    rng = np.random.default_rng(21)
    S64 = (rng.random((1, 70, 700)) ** 3)
    S32 = S64.astype(np.float32)
    freqs = np.linspace(-10.0, 10.0, 70)
    a, b = api.Handle(0), api.Handle(0)
    for S in (S64, S32, S64):
        for h, w in ((a, (2, 2, 30, 36)), (b, (1, 1, 0, 1)), (a, (2, 3, 30, 253)), (b, (0, 0, 1, 0)), (a, (2, 2, 30, 36)),
                     (b, (31, 255, 1, 1)), (a, (1, 1, 2, 16))):
            rank = default_rank(*w)
            got, cnt = run_dev(S, freqs, 8, *w, rank, 0.5, handle=h)
            want = O.detect_cfar_os(S[0], freqs, 8, *w, rank, 0.5)
            assert cnt[0] == len(want)
            same(got[0], O.padded(want, 8))
    a.close()
    b.close()


def test_cli_prints_os_lines(tmp_path):
    """--detect 16 --cfar-db X --cfar-rank K: the two main.rs lines, then OS-CFAR's detections, which include the weak
    emitter that the same command without --cfar-rank (CA-CFAR) leaves out."""
    import subprocess
    exe = G._cli(tmp_path)
    gr, gd, tr, tc = 32, 2, 0, 64
    N = F.train_cells(gr, gd, tr, tc)
    rank = default_rank(gr, gd, tr, tc)
    needle, hay = planted_scene(SCENES[0][0], SCENES[0][1])
    a, b = str(tmp_path / "needle.c64"), str(tmp_path / "hay.c64")
    for path, x in ((a, needle), (b, hay)):
        np.stack([x.real, x.imag], axis=1).astype("<f4").tofile(path)
    plain = subprocess.run([exe, a, b], capture_output=True, text=True, timeout=120)
    assert plain.returncode == 0, plain.stderr
    win = ["--detect", "16", "--guard-doppler", str(gr), "--guard-delay", str(gd), "--train-doppler", str(tr),
           "--train-delay", str(tc)]
    cells = {}
    for label, db, extra in (("ca", 10 * np.log10(api.cfar_scale(1e-6, N)), []),
                             ("os", 10 * np.log10(api.cfar_os_scale(1e-6, N, rank)), ["--cfar-rank", str(rank)])):
        res = subprocess.run([exe, a, b] + win + ["--cfar-db", "%.6f" % db] + extra, capture_output=True, text=True,
                             timeout=120)
        assert res.returncode == 0, res.stderr
        assert res.stdout.startswith(plain.stdout)
        cells[label] = []
        for line in res.stdout.splitlines()[2:]:
            m = re.match(r"Detection \d+: (\S+)Hz \(grid (\S+)Hz\), (\S+) samples \(cell (\d+)\), (\S+) dB below the "
                         r"first, (\S+) dB above the noise$", line)
            assert m and float(m.group(6)) > db, line
            cells[label].append(int(m.group(4)))
    assert 202 in cells["ca"] and 230 not in cells["ca"]
    assert 202 in cells["os"] and 230 in cells["os"]


def test_cpp_detect_cfar_os_refuses_other_threads(tmp_path):
    """caf_b200_surface_detect_cfar_os runs on the surface's handle: the C++ mirror refuses other threads."""
    import shutil
    import subprocess
    from conftest import ROOT
    src = tmp_path / "owner.cpp"
    src.write_text(r'''
#include <cmath>
#include <cstdio>
#include <thread>
#include "caf_b200.hpp"
int main() {
    std::vector<caf::Complex64> x(256), y(256);
    for (int i = 0; i < 256; ++i) x[i] = {std::sin(0.37 * i * i), std::cos(1.3 * i + 0.011 * i * i)};
    for (int i = 0; i < 256; ++i) y[i] = x[(i + 250) % 256];      // delayed by 6 samples
    const auto rows = caf::CafB200::caf_surface(x, y, {-1.0, 0.0, 1.0}, 48000);
    const auto here = caf::CafB200::detect_cfar_os(rows, 3, 1, 1, 0, 16, 72, 10.0);
    bool refused = false;
    std::thread t([&] { try { caf::CafB200::detect_cfar_os(rows, 3, 1, 1, 0, 16, 72, 10.0); } catch (const caf::Panic&) { refused = true; } });
    t.join();
    std::printf("%zu %d %llu %llu\n", here.size(), refused ? 1 : 0, (unsigned long long)here[0].delay_idx,
                (unsigned long long)here[0].train_cells);
    return 0;
}
''')
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "owner")
    subprocess.check_call([shutil.which("g++"), "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    n, refused, k, m = res.stdout.split()
    assert int(n) >= 1 and refused == "1" and int(k) == 6 and int(m) == 3 * 32   # 3 rows x (2 x 16) side cells
