//! The reference's `caf` module surface (caf_rust/src/caf/mod.rs:13-462) on the B200 library:
//! `CafSurfaceRow`, `trait CafSurface { caf_surface, find_peak, apply_freq_shift }` and the seven strategy
//! structs the tests and benches name (caf_bench.rs:12-19).  Every strategy is the same GPU path.
use std::os::raw::c_void;
use std::sync::Arc;

use num_complex::Complex64;
use once_cell::sync::OnceCell;

use crate::ffi;

/// One surface on the GPU (caf_b200_surface_*), shared by its rows.  The reference's `CafSurfaceRow` owns a `Vec<f64>` per
/// row but keeps every field private (mod.rs:17-22), so no caller of the crate can read it: `tests/test.rs` and
/// `benches/caf_bench.rs` hand the rows to `find_peak` and look at nothing else.  Here a row is (surface, row number) and
/// the 2L doubles of `xcor_mag` cross PCIe only if `xcor_mag()` is called.
pub struct DeviceSurface {
    raw: ffi::caf_b200_surface,
    rows: usize,
    cells: usize,
    peaks: OnceCell<(Vec<f64>, Vec<f64>, Vec<u64>)>,      // (freq, xcor_peak_val, xcor_peak_idx), 24 bytes per row, on demand
    owner: std::thread::ThreadId,                          // the thread whose HANDLE made it: detection runs on that handle
}
// the object is immutable after creation and caf_b200_surface_fetch_rows / _row_peaks do not touch the handle's stream;
// caf_b200_surface_detect does, so detect() checks that it runs on the owner thread (a handle is not thread-safe)
unsafe impl Send for DeviceSurface {}
unsafe impl Sync for DeviceSurface {}
impl DeviceSurface {
    fn peaks(&self) -> &(Vec<f64>, Vec<f64>, Vec<u64>) {
        self.peaks.get_or_init(|| {
            let (mut f, mut v, mut i) = (vec![0f64; self.rows], vec![0f64; self.rows], vec![0u64; self.rows]);
            ffi::check(unsafe { ffi::caf_b200_surface_row_peaks(self.raw, f.as_mut_ptr(), v.as_mut_ptr(), i.as_mut_ptr()) });
            (f, v, i)
        })
    }
    fn detect(&self, k_max: usize, guard_doppler: u32, guard_delay: u32, min_ratio: f64) -> Vec<ffi::caf_b200_detection> {
        assert!(std::thread::current().id() == self.owner, "detect: a surface is searched on the thread that created it");
        let mut out = vec![ffi::caf_b200_detection::default(); k_max];
        let mut count = 0usize;
        ffi::check(unsafe {
            ffi::caf_b200_surface_detect(self.raw, k_max, guard_doppler, guard_delay, min_ratio, out.as_mut_ptr(), &mut count)
        });
        out.truncate(count);
        out
    }
    fn detect_cfar(&self, k_max: usize, guard_doppler: u32, guard_delay: u32, train_doppler: u32, train_delay: u32,
                   scale: f64) -> Vec<ffi::caf_b200_cfar_detection> {
        assert!(std::thread::current().id() == self.owner, "detect_cfar: a surface is searched on the thread that created it");
        let mut out = vec![ffi::caf_b200_cfar_detection::default(); k_max];
        let mut count = 0usize;
        ffi::check(unsafe {
            ffi::caf_b200_surface_detect_cfar(self.raw, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale,
                                              out.as_mut_ptr(), &mut count)
        });
        out.truncate(count);
        out
    }
    fn fused_peak(&self) -> ffi::caf_b200_peak {
        let mut pk = ffi::caf_b200_peak::default();
        ffi::check(unsafe { ffi::caf_b200_surface_find_peak(self.raw, &mut pk) });
        pk
    }
}
impl Drop for DeviceSurface {
    fn drop(&mut self) { unsafe { ffi::caf_b200_surface_destroy(self.raw); } }
}

#[allow(dead_code)]
pub struct CafSurfaceRow {
    surface: Arc<DeviceSurface>,
    row: usize,
}

impl CafSurfaceRow {
    // accessors are an addition: the reference keeps the fields private (mod.rs:18-21)
    pub fn freq(&self) -> f64 { self.surface.peaks().0[self.row] }
    pub fn xcor_peak_val(&self) -> f64 { self.surface.peaks().1[self.row] }
    pub fn xcor_peak_idx(&self) -> usize { self.surface.peaks().2[self.row] as usize }
    /// lazy: this row's 2L cells come over PCIe now (one cudaMemcpy), not when the surface was computed
    pub fn xcor_mag(&self) -> Vec<f64> {
        let mut out = vec![0f64; self.surface.cells];
        ffi::check(unsafe { ffi::caf_b200_surface_fetch_rows(self.surface.raw, self.row, 1, out.as_mut_ptr() as *mut c_void) });
        out
    }
}

/// inputs up (one pinned block, one H2D), ONE fused launch, the 32-byte find_peak result down: the cost of a peak-only call
fn surface_on_gpu(needle: &[Complex64], haystack: &[Complex64], freqs_hz: &[f64], fs: u32) -> Vec<CafSurfaceRow> {
    assert!(needle.len() == haystack.len());            // xcor_rustfft.rs:54-55
    let mut raw: ffi::caf_b200_surface = std::ptr::null_mut();
    ffi::HANDLE.with(|h| ffi::check(unsafe {
        ffi::caf_b200_surface_create_f64(h.0, needle.as_ptr(), haystack.as_ptr(), needle.len(), freqs_hz.as_ptr(),
                                         freqs_hz.len(), fs, &mut raw)
    }));
    let surface = Arc::new(DeviceSurface { raw, rows: freqs_hz.len(), cells: 2 * needle.len(), peaks: OnceCell::new(),
                                           owner: std::thread::current().id() });
    (0..freqs_hz.len()).map(|row| CafSurfaceRow { surface: surface.clone(), row }).collect()
}

pub trait CafSurface {
    fn caf_surface(needle: &[Complex64], haystack: &[Complex64], freqs_hz: &[f64], fs: u32) -> Vec<CafSurfaceRow> {
        surface_on_gpu(needle, haystack, freqs_hz, fs)
    }

    // mod.rs:31-42, unchanged semantics: strict > from a dummy row, in VECTOR order.  When `arr` is what caf_surface
    // returned, untouched (every row of one surface, in order), that scan is what the kernel's fused find_peak already
    // did; any other vector (reordered, truncated, rows of several surfaces) is scanned here from the rows' peaks.
    fn find_peak(arr: Vec<CafSurfaceRow>) -> (f64, usize) {
        if let Some(first) = arr.first() {
            let whole = arr.len() == first.surface.rows
                && arr.iter().enumerate().all(|(i, r)| r.row == i && Arc::ptr_eq(&r.surface, &first.surface));
            if whole {
                let pk = first.surface.fused_peak();
                return (pk.freq_hz, pk.delay_idx as usize);
            }
        }
        let (mut best, mut out) = (0.0f64, (0.0f64, 0usize));
        for row in arr.iter() {
            if row.xcor_peak_val() > best { best = row.xcor_peak_val(); out = (row.freq(), row.xcor_peak_idx()); }
        }
        out
    }

    // mod.rs:46-65
    fn apply_freq_shift(samples: &[Complex64], freq_shift: f64, fs: u32) -> Vec<Complex64> {
        let mut out = vec![Complex64::new(0.0, 0.0); samples.len()];
        ffi::HANDLE.with(|h| ffi::check(unsafe {
            ffi::caf_b200_apply_freq_shift_f64(h.0, samples.as_ptr(), samples.len(), freq_shift, fs, out.as_mut_ptr())
        }));
        out
    }

    // README.md:124 calls it apply_shift
    fn apply_shift(samples: &[Complex64], freq_shift: f64, fs: u32) -> Vec<Complex64> {
        Self::apply_freq_shift(samples, freq_shift, fs)
    }
}

macro_rules! strategy { ($($name:ident),*) => { $(pub struct $name {} impl CafSurface for $name {})* } }
strategy!(CafB200, CafFFTW, CafRustFFT, CafRustFFTRayon, CafRustFFTIter, CafRustFFTIterRayon, CafRustFFTThreads,
          CafRustFFTThreadpool);

impl CafB200 {
    /// The `k_max` strongest local maxima of the surface behind `arr`, best first, each refined below the grid
    /// (include/caf_b200.h, caf_b200_surface_detect).  `arr` must be what `caf_surface` returned, untouched: a reordered or
    /// partial vector no longer names one surface, so it panics.  It also panics off the thread that called `caf_surface`:
    /// the search runs on that thread's handle.
    pub fn detect(arr: &[CafSurfaceRow], k_max: usize, guard_doppler: u32, guard_delay: u32, min_ratio: f64)
                  -> Vec<ffi::caf_b200_detection> {
        let first = arr.first().expect("detect needs the untouched rows of one caf_surface call");
        let whole = arr.len() == first.surface.rows
            && arr.iter().enumerate().all(|(i, r)| r.row == i && Arc::ptr_eq(&r.surface, &first.surface));
        assert!(whole, "detect needs the untouched rows of one caf_surface call");
        first.surface.detect(k_max, guard_doppler, guard_delay, min_ratio)
    }
    /// The local maxima of the surface behind `arr` that exceed `scale` x their local noise estimate (cell-averaging
    /// CFAR, include/caf_b200.h, caf_b200_surface_detect_cfar), best first, at most `k_max` and possibly none.  Same rules
    /// for `arr` and the calling thread as `detect`.
    pub fn detect_cfar(arr: &[CafSurfaceRow], k_max: usize, guard_doppler: u32, guard_delay: u32, train_doppler: u32,
                       train_delay: u32, scale: f64) -> Vec<ffi::caf_b200_cfar_detection> {
        let first = arr.first().expect("detect_cfar needs the untouched rows of one caf_surface call");
        let whole = arr.len() == first.surface.rows
            && arr.iter().enumerate().all(|(i, r)| r.row == i && Arc::ptr_eq(&r.surface, &first.surface));
        assert!(whole, "detect_cfar needs the untouched rows of one caf_surface call");
        first.surface.detect_cfar(k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale)
    }
}

/// caf_surface + find_peak fused on the GPU; the surface never leaves the chip.
pub fn caf_peak(needle: &[Complex64], haystack: &[Complex64], freqs_hz: &[f64], fs: u32) -> (f64, usize) {
    assert!(needle.len() == haystack.len());
    let mut pk = ffi::caf_b200_peak::default();
    ffi::HANDLE.with(|h| ffi::check(unsafe {
        ffi::caf_b200_peak_f64(h.0, needle.as_ptr(), haystack.as_ptr(), needle.len(), freqs_hz.as_ptr(),
                               freqs_hz.len(), fs, &mut pk)
    }));
    (pk.freq_hz, pk.delay_idx as usize)
}

/// xcor_rustfft.rs:14-93 (crate-private there; public here so parity can be checked from outside)
#[derive(Clone)]
pub struct Xcor { n: usize }
impl Xcor {
    pub fn new(n: usize) -> Self { Xcor { n } }
    pub fn run(&mut self, a: &[Complex64], b: &[Complex64]) -> Vec<Complex64> {
        assert!(a.len() == self.n);
        assert!(b.len() == self.n);
        let mut out = vec![Complex64::new(0.0, 0.0); self.n];
        ffi::HANDLE.with(|h| ffi::check(unsafe { ffi::caf_b200_xcor_f64(h.0, a.as_ptr(), b.as_ptr(), self.n, out.as_mut_ptr()) }));
        out
    }
}

/// One process per GPU: rank `rank` of `world` computes its block of doppler rows and every rank gets the global
/// `find_peak` answer (one 32-byte NCCL all-gather inside the library).  `id` is the 128-byte NCCL id rank 0 made with
/// `nccl_unique_id()` and handed to the other ranks out of band.  This is mod.rs:185's `par_iter` over rows with GPUs
/// in place of rayon workers.
pub struct ShardedCaf { comm: ffi::caf_b200_comm }
pub fn nccl_unique_id() -> [u8; ffi::CAF_B200_NCCL_ID_BYTES] {
    let mut id = [0u8; ffi::CAF_B200_NCCL_ID_BYTES];
    ffi::check(unsafe { ffi::caf_b200_comm_unique_id(id.as_mut_ptr()) });
    id
}
impl ShardedCaf {
    pub fn new(world: usize, rank: usize, id: &[u8; ffi::CAF_B200_NCCL_ID_BYTES]) -> Self {
        let mut comm: ffi::caf_b200_comm = std::ptr::null_mut();
        ffi::HANDLE.with(|h| ffi::check(unsafe { ffi::caf_b200_comm_create(h.0, world as i32, rank as i32, id.as_ptr(), &mut comm) }));
        ShardedCaf { comm }
    }
    /// (rows [lo, hi) of the surface owned by this rank, global (freq, delay) peak)
    pub fn caf_surface_peak(&self, needle: &[Complex64], haystack: &[Complex64], freqs_hz: &[f64], fs: u32)
                            -> (Vec<f64>, (usize, usize), (f64, usize)) {
        assert!(needle.len() == haystack.len());
        let (mut lo, mut hi) = (0usize, 0usize);
        ffi::check(unsafe { ffi::caf_b200_comm_shard(self.comm, freqs_hz.len(), &mut lo, &mut hi) });
        let mut local = vec![0f64; (hi - lo) * 2 * needle.len()];
        let mut pk = ffi::caf_b200_peak::default();
        ffi::HANDLE.with(|h| ffi::check(unsafe {
            ffi::caf_b200_surface_sharded_f64(h.0, self.comm, needle.as_ptr(), haystack.as_ptr(), needle.len(),
                                              freqs_hz.as_ptr(), freqs_hz.len(), fs, local.as_mut_ptr(), &mut pk)
        }));
        (local, (lo, hi), (pk.freq_hz, pk.delay_idx as usize))
    }
}
impl Drop for ShardedCaf {
    fn drop(&mut self) { unsafe { ffi::caf_b200_comm_destroy(self.comm); } }
}

/// The Go program's surface (caf_go/caf.go:162-173): [d][2l] of |xcor|, column k = lag l - k.
pub fn go_amb_surf(needle: &[Complex64], haystack: &[Complex64], freqs_hz: &[f64], samp_rate: f64) -> Vec<Vec<f64>> {
    assert!(needle.len() == haystack.len());
    // caf.go:118 takes a float64 rate, the library the crate's u32 (mod.rs:46): refuse what the u32 cannot hold exactly
    assert!(samp_rate >= 1.0 && samp_rate <= u32::MAX as f64 && samp_rate.fract() == 0.0, "samp_rate must be a whole number of Hz");
    let (l, d) = (needle.len(), freqs_hz.len());
    let mut flat = vec![0f64; d * 2 * l];
    ffi::HANDLE.with(|h| ffi::check(unsafe {
        ffi::caf_b200_surface_layout_f64(h.0, needle.as_ptr(), haystack.as_ptr(), l, freqs_hz.as_ptr(), d,
                                         samp_rate as u32, 2, flat.as_mut_ptr(), std::ptr::null_mut())
    }));
    flat.chunks(2 * l).map(|r| r.to_vec()).collect()
}
