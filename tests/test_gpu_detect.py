"""caf_b200_surface_detect / caf_b200_detect_*_dev on the GPU against oracle/detect.py (include/caf_b200.h)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from caf_cookoff_b200 import _lib, api, bench_shifts
from conftest import FS, load_case
from oracle import detect as D

pytestmark = pytest.mark.gpu

REC = np.dtype([("value", "f8"), ("freq_hz", "f8"), ("doppler_idx", "u8"), ("delay_idx", "u8"),
                ("lag_samples", "f8"), ("freq_hz_interp", "f8")])
UMAX = (1 << 64) - 1


def as_tuples(recs):
    return [(float(x["value"]), float(x["freq_hz"]), int(x["doppler_idx"]), int(x["delay_idx"]),
             float(x["lag_samples"]), float(x["freq_hz_interp"])) for x in recs]


def same(got, want):
    """indices and values exactly, refinements to 1e-12 relative"""
    assert len(got) == len(want), (len(got), len(want))
    for i, (g, w) in enumerate(zip(got, want)):
        assert g[:4] == w[:4], (i, g, w)
        for a, b in ((g[4], w[4]), (g[5], w[5])):
            assert abs(a - b) <= 1e-12 * max(1.0, abs(b)), (i, g, w)


def run_dev(S, freqs, k_max, gr, gd, ratio=0.0, handle=None):
    """S [p][d][n] numpy (float64 or float32) -> (records [p][k_max] as tuples, counts [p]) through detect_*_dev"""
    import torch
    dev = torch.device("cuda", 0)
    p, d, n = S.shape
    ts = torch.from_numpy(np.ascontiguousarray(S)).to(dev)
    tf = torch.from_numpy(np.ascontiguousarray(freqs, dtype=np.float64)).to(dev)
    out = torch.zeros((p, k_max, 6), dtype=torch.float64, device=dev)
    cnt = torch.full((p,), -1, dtype=torch.int64, device=dev)
    h = handle or api.default_handle()
    api.detect_dev(ts.data_ptr(), p, d, n, tf.data_ptr(), k_max, out.data_ptr(), cnt.data_ptr(), guard_doppler=gr,
                   guard_delay=gd, min_ratio=ratio, f32=S.dtype == np.float32, handle=h)
    torch.cuda.synchronize()
    recs = out.cpu().numpy().view(REC).reshape(p, k_max)
    return [as_tuples(recs[i]) for i in range(p)], [int(c) for c in cnt.cpu().numpy()]


def check_against_reference(S, freqs, k_max, gr, gd, ratio=0.0):
    got, cnt = run_dev(S, freqs, k_max, gr, gd, ratio)
    for i in range(S.shape[0]):
        want = D.detect(S[i], freqs, k_max, gr, gd, ratio)
        assert cnt[i] == len(want)
        same(got[i], D.padded(want, k_max))
    return got, cnt


SHAPES = [  # (p, d, n, gr, gd, k_max)
    (3, 1, 300, 0, 0, 7), (3, 2, 517, 1, 1, 16), (2, 37, 1000, 2, 3, 64), (1, 37, 513, 32, 256, 3),
    (1, 37, 1000, 0, 0, 1024), (4, 2, 9, 1, 4, 3), (1, 37, 520, 5, 40, 1024), (2, 20, 257, 32, 1, 1),
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_tie_heavy_surfaces_match_reference(shape, dtype):
    p, d, n, gr, gd, k_max = shape
    rng = np.random.default_rng(hash(shape) % 1000)
    S = rng.integers(0, 5, size=(p, d, n)).astype(dtype)
    S[rng.random(S.shape) < 0.02] = np.nan
    freqs = np.cumsum(rng.random(d) + 0.05) - 3.0
    got, _ = check_against_reference(S, freqs, k_max, gr, gd)
    one = [run_dev(S[i:i + 1], freqs, k_max, gr, gd)[0][0] for i in range(p)]
    assert got == one                                       # a batch equals its pairs run one at a time
    check_against_reference(S, freqs, k_max, gr, gd, ratio=0.5)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_distinct_values_large_k_and_repeatability(dtype):
    """Many local maxima per tile (noise), k_max up to the cap: the per-tile cut and the pair floor must keep exactly the
    reference's answer, bit for bit on every call."""
    rng = np.random.default_rng(5)
    S = (rng.random((2, 100, 4100)) ** 3).astype(dtype)
    freqs = np.linspace(-50.0, 50.0, 100)
    for k_max, gr, gd in ((1024, 1, 1), (200, 0, 0), (33, 4, 17)):
        got, _ = check_against_reference(S, freqs, k_max, gr, gd)
        for _ in range(3):
            assert run_dev(S, freqs, k_max, gr, gd)[0] == got


def surface_of(case, variant, handle=None):
    needle, hay, shifts = load_case(case)
    return api.DeviceSurface(needle, hay, shifts, FS, variant=variant, handle=handle), shifts


@pytest.mark.parametrize("variant", [api._Variant, api._Variant32], ids=["f64", "f32"])
def test_known_answer_surfaces(known_answers, variant):
    """Detection 0 is find_peak's cell; the whole list is the reference's on the fetched surface; guard 1 x 1 refines the
    ten fixtures to within 0.01 Hz and 0.01 sample of what their file names say."""
    seen = set()
    for case in known_answers:
        if case["haystack"] in seen:
            continue
        seen.add(case["haystack"])
        s, shifts = surface_of(case, variant)
        dets = s.detect(32, 1, 1)
        pk = s.find_peak()
        d0 = dets[0]
        assert (d0.value, d0.freq_hz, d0.doppler_idx, d0.delay_idx) == (pk.value, pk.freq_hz, pk.doppler_idx, pk.delay_idx)
        S = s.fetch_rows()
        same([(x.value, x.freq_hz, x.doppler_idx, x.delay_idx, x.lag_samples, x.freq_hz_interp) for x in dets],
             D.detect(S, shifts, 32, 1, 1))
        same([(x.value, x.freq_hz, x.doppler_idx, x.delay_idx, x.lag_samples, x.freq_hz_interp) for x in s.detect(8, 3, 20, 0.01)],
             D.detect(S, shifts, 8, 3, 20, 0.01))
        if variant is api._Variant:
            m = re.search(r"T\+(\d+)samp_F([+-][\d.]+)Hz", case["haystack"])
            assert abs(d0.lag_samples - int(m.group(1))) <= 0.01, case["haystack"]
            assert abs(d0.freq_hz_interp - float(m.group(2))) <= 0.01, case["haystack"]
        s.close()
    assert len(seen) == 10


def planted():
    rng = np.random.default_rng(7)
    N = 4096
    needle = np.hanning(N) * (rng.standard_normal(N) + 1j * rng.standard_normal(N)) / np.sqrt(2)
    hay = np.zeros(N, dtype=np.complex128)
    emitters = [(202, 69.0, 1.0), (57, -31.5, 0.5), (140, 12.0, 0.25), (90, -80.25, 0.15)]
    for lag, f, a in emitters:
        x = np.concatenate([np.zeros(lag), needle])[:N]
        hay += a * x * np.exp(2j * np.pi * f * np.arange(N) / FS)
    hay += 1e-3 * (rng.standard_normal(N) + 1j * rng.standard_normal(N))
    return needle, hay, emitters


def test_four_planted_emitters():
    needle, hay, emitters = planted()
    s = api.DeviceSurface(needle, hay, bench_shifts(), FS)
    dets = s.detect(5, 2, 2)
    for x, (lag, f, _) in zip(dets[:4], emitters):
        assert x.lag_samples == pytest.approx(lag, abs=0.5) and int(x.delay_idx) == lag
        assert abs(x.freq_hz - f) <= 2.5 and abs(x.freq_hz_interp - f) <= 2.5
    assert dets[4].value < dets[3].value / 2
    same([(x.value, x.freq_hz, x.doppler_idx, x.delay_idx, x.lag_samples, x.freq_hz_interp) for x in dets],
         D.detect(s.fetch_rows(), bench_shifts(), 5, 2, 2))


@pytest.mark.parametrize("variant", [api._Variant, api._Variant32], ids=["f64", "f32"])
def test_long_rows(variant):
    rng = np.random.default_rng(11)
    L = 8192
    needle = rng.standard_normal(L) + 1j * rng.standard_normal(L)
    hay = np.roll(needle, 300) * np.exp(2j * np.pi * 20.0 * np.arange(L) / FS) + 0.5 * (rng.standard_normal(L) + 1j * rng.standard_normal(L))
    freqs = np.linspace(0.0, 40.0, 16)
    s = api.DeviceSurface(needle, hay, freqs, FS, variant=variant)
    assert s.shape == (16, 2 * L)
    dets = s.detect(100, 1, 2)
    same([(x.value, x.freq_hz, x.doppler_idx, x.delay_idx, x.lag_samples, x.freq_hz_interp) for x in dets],
         D.detect(s.fetch_rows(), freqs, 100, 1, 2))
    assert dets[0].delay_idx == 300


def test_error_codes():
    import torch
    lib = _lib.load()
    h = api.Handle(0)
    needle, hay, _ = planted()
    shifts = np.linspace(-5, 5, 11)
    s = api.DeviceSurface(needle[:64], hay[:64], shifts, FS, handle=h)           # 11 x 128
    out = (_lib.Detection * 1025)()
    cnt = C.c_size_t(77)
    for args in ((0, 1, 1, 0.0), (1025, 1, 1, 0.0), (4, 33, 1, 0.0), (4, 1, 257, 0.0), (4, 1, 64, 0.0),
                 (4, 1, 1, -0.1), (4, 1, 1, 1.5), (4, 1, 1, float("nan"))):
        assert lib.caf_b200_surface_detect(s.raw, *args, out, C.byref(cnt)) == -1, args
        assert cnt.value == 77
    assert lib.caf_b200_surface_detect(s.raw, 4, 1, 63, 1.0, out, C.byref(cnt)) == 0       # 2 * 63 + 1 <= 128
    assert lib.caf_b200_surface_detect(s.raw, 4, 1, 1, 0.0, None, C.byref(cnt)) == -1
    dev = torch.device("cuda", 0)
    S = torch.rand((1, 4, 16), dtype=torch.float64, device=dev)
    f = torch.zeros(4, dtype=torch.float64, device=dev)
    o = torch.zeros((1, 4, 6), dtype=torch.float64, device=dev)
    c = torch.zeros(1, dtype=torch.int64, device=dev)
    assert lib.caf_b200_detect_f64_dev(h.raw, S.data_ptr(), 1, 4, 16, f.data_ptr(), 4, 1, 8, 0.0, o.data_ptr(), c.data_ptr()) == -1
    assert lib.caf_b200_detect_f64_dev(h.raw, None, 1, 4, 16, f.data_ptr(), 4, 1, 1, 0.0, o.data_ptr(), c.data_ptr()) == -1
    assert lib.caf_b200_detect_f64_dev(h.raw, S.data_ptr(), 1, 4, 16, f.data_ptr(), 4, 1, 1, 0.0, None, c.data_ptr()) == -1
    # empty shapes: count 0, every slot "none"
    o.fill_(1.0)
    c.fill_(5)
    assert lib.caf_b200_detect_f64_dev(h.raw, S.data_ptr(), 1, 0, 16, f.data_ptr(), 4, 1, 1, 0.0, o.data_ptr(), c.data_ptr()) == 0
    torch.cuda.synchronize()
    assert int(c[0]) == 0 and as_tuples(o.cpu().numpy().view(REC).reshape(4)) == [D.NONE] * 4
    # a surface whose handle is gone
    h.close()
    assert lib.caf_b200_surface_detect(s.raw, 4, 1, 1, 0.0, out, C.byref(cnt)) == -1
    assert "handle" in lib.caf_b200_last_error().decode()
    s.close()


def test_overlap_detect_between_surface_launches():
    """With overlap mode 4 and rotated outputs, detect calls placed between surface launches leave every surface and
    every peak bit-identical to the serialised run, raise the launch count by two each, and detect what the reference
    detects on the finished surface."""
    import torch
    from oracle import oracle as O
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    lib = _lib.load()
    h = api.Handle(0, stream=stream.cuda_stream)
    L = 4096
    needle, hay, _ = planted()
    nd = torch.from_numpy(needle).to(dev)
    hd = torch.from_numpy(hay).to(dev)
    shifts = bench_shifts()
    fd = torch.from_numpy(shifts).to(dev)
    K, NB = 12, 9

    def run(overlap, with_detect):
        lib.caf_b200_set_overlap(h.raw, overlap)
        surfs = [torch.zeros((400, 2 * L), dtype=torch.float64, device=dev) for _ in range(NB)]
        rv = torch.zeros((K, 400), dtype=torch.float64, device=dev); ri = torch.zeros((K, 400), dtype=torch.int64, device=dev)
        pk = torch.zeros((K, 4), dtype=torch.int64, device=dev)
        out = torch.zeros((K, 8, 6), dtype=torch.float64, device=dev); cnt = torch.zeros(K, dtype=torch.int64, device=dev)
        with torch.cuda.stream(stream):
            for k in range(K):
                sb = k % NB
                assert lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, L, fd.data_ptr(), 400, FS,
                                                  surfs[sb].data_ptr(), rv[k].data_ptr(), ri[k].data_ptr(), pk[k].data_ptr()) == 0
                if with_detect and k % 3 == 1:
                    before = h.launch_count
                    assert lib.caf_b200_detect_f64_dev(h.raw, surfs[sb].data_ptr(), 1, 400, 2 * L, fd.data_ptr(), 8, 2, 2,
                                                       0.0, out[k].data_ptr(), cnt[k].data_ptr()) == 0
                    assert h.launch_count == before + 2
        torch.cuda.synchronize()
        return [x.cpu().numpy() for x in surfs], rv.cpu().numpy(), ri.cpu().numpy(), pk.cpu().numpy(), out.cpu().numpy(), cnt.cpu().numpy()

    want = run(0, False)
    got = run(4, True)
    for a, b in zip(want[0], got[0]):
        assert np.array_equal(a, b)
    for i in (1, 2, 3):
        assert np.array_equal(want[i], got[i])
    ref = D.detect(want[0][1], shifts, 8, 2, 2)
    for k in range(1, K, 3):
        same(as_tuples(got[4][k].view(REC).reshape(8))[:int(got[5][k])], ref)
    lib.caf_b200_set_overlap(h.raw, 0)
    h.close()


def test_cli_detect_prints_the_four_emitters(tmp_path):
    """tools/caf_cli --detect 4 on the planted pair: the two main.rs lines, then the four emitters in amplitude order.
    Without the flag the output is byte-identical to the plain report."""
    import shutil
    import subprocess
    from conftest import ROOT
    gxx = shutil.which("g++")
    assert gxx, "g++ is required for the CLI"
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "caf_cli")
    subprocess.check_call([gxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "caf_cli.cpp"),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    needle, hay, emitters = planted()
    a, b = str(tmp_path / "needle.c64"), str(tmp_path / "hay.c64")
    for path, x in ((a, needle), (b, hay)):
        np.stack([x.real, x.imag], axis=1).astype("<f4").tofile(path)
    plain = subprocess.run([exe, a, b], capture_output=True, text=True, timeout=120)
    assert plain.returncode == 0, plain.stderr
    assert plain.stdout == "Frequency offset: 69.0Hz\nTime offset: 202 samples (4.208ms)\n"
    res = subprocess.run([exe, a, b, "--detect", "4", "--guard-doppler", "2", "--guard-delay", "2"], capture_output=True,
                         text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    lines = res.stdout.splitlines()
    assert res.stdout.startswith(plain.stdout) and len(lines) == 6
    for line, (lag, f, _) in zip(lines[2:], emitters):
        m = re.match(r"Detection \d: (\S+)Hz \(grid (\S+)Hz\), (\S+) samples \(cell (\d+)\)", line)
        assert m and int(m.group(4)) == lag and abs(float(m.group(1)) - f) <= 2.5, line
    res = subprocess.run([exe, a, b, "--detect", "4", "--min-db", "7"], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and len(res.stdout.splitlines()) == 4      # 0.25 and 0.15 of the amplitude: -12 and -16 dB


def test_two_handles_alternate_large_and_small_guards():
    """The tile kernel's shared-memory allowance belongs to the device: a handle that ran small guards must not take it
    away from another handle's large-guard search (32 x 256 needs 186 KB in f64)."""
    rng = np.random.default_rng(21)
    S64 = (rng.random((1, 40, 600)) ** 3)
    S32 = S64.astype(np.float32)
    freqs = np.linspace(-10.0, 10.0, 40)
    a, b = api.Handle(0), api.Handle(0)
    for S in (S64, S32, S64):
        for h, gr, gd in ((a, 32, 256), (b, 1, 1), (a, 32, 256), (b, 0, 0), (a, 32, 256), (b, 32, 256), (a, 1, 1)):
            got, cnt = run_dev(S, freqs, 8, gr, gd, handle=h)
            want = D.detect(S[0], freqs, 8, gr, gd)
            assert cnt[0] == len(want)
            same(got[0], D.padded(want, 8))
    a.close()
    b.close()


def test_cpp_detect_refuses_other_threads(tmp_path):
    """caf_b200_surface_detect runs on the surface's handle, which is not thread-safe: the C++ mirror's detect refuses
    to run off the thread that made the surface (the Rust shim asserts the same)."""
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
    const auto here = caf::CafB200::detect(rows, 3);
    bool refused = false;
    std::thread t([&] { try { caf::CafB200::detect(rows, 3); } catch (const caf::Panic&) { refused = true; } });
    t.join();
    std::printf("%zu %d %llu\n", here.size(), refused ? 1 : 0, (unsigned long long)here[0].delay_idx);
    return 0;
}
''')
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "owner")
    subprocess.check_call([shutil.which("g++"), "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    n, refused, k = res.stdout.split()
    assert int(n) >= 1 and refused == "1" and int(k) == 6
