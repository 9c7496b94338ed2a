//! Hand-written extern "C" block for include/caf_b200.h (only what the crate API needs).
#![allow(non_camel_case_types, dead_code)]
use num_complex::{Complex32, Complex64};
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct caf_b200_handle_s { _private: [u8; 0] }
pub type caf_b200_handle = *mut caf_b200_handle_s;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct caf_b200_peak {
    pub value: f64,
    pub freq_hz: f64,
    pub doppler_idx: u64,
    pub delay_idx: u64,
}

/// caf_b200_detection: a local maximum of a surface, refined below the grid (the first four fields are caf_b200_peak's)
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct caf_b200_detection {
    pub value: f64,
    pub freq_hz: f64,
    pub doppler_idx: u64,
    pub delay_idx: u64,
    pub lag_samples: f64,
    pub freq_hz_interp: f64,
}

/// caf_b200_cfar_detection: caf_b200_detection's six fields, then the cell's local noise estimate and its training cells
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct caf_b200_cfar_detection {
    pub value: f64,
    pub freq_hz: f64,
    pub doppler_idx: u64,
    pub delay_idx: u64,
    pub lag_samples: f64,
    pub freq_hz_interp: f64,
    pub noise: f64,
    pub train_cells: u64,
}

extern "C" {
    pub fn caf_b200_create(device: c_int, out: *mut caf_b200_handle) -> c_int;
    pub fn caf_b200_destroy(h: caf_b200_handle) -> c_int;
    pub fn caf_b200_last_error() -> *const c_char;
    pub fn caf_b200_set_overlap(h: caf_b200_handle, on: c_int) -> c_int;
    pub fn caf_b200_apply_freq_shift_f64(h: caf_b200_handle, input: *const Complex64, n: usize, freq_hz: f64,
                                         fs: u32, out: *mut Complex64) -> c_int;
    pub fn caf_b200_xcor_f64(h: caf_b200_handle, a: *const Complex64, b: *const Complex64, n: usize,
                             out: *mut Complex64) -> c_int;
    pub fn caf_b200_surface_f64(h: caf_b200_handle, needle: *const Complex64, haystack: *const Complex64, l: usize,
                                freqs_hz: *const f64, d: usize, fs: u32, surface: *mut f64,
                                row_peak_val: *mut f64, row_peak_idx: *mut u64, peak: *mut caf_b200_peak) -> c_int;
    pub fn caf_b200_peak_f64(h: caf_b200_handle, needle: *const Complex64, haystack: *const Complex64, l: usize,
                             freqs_hz: *const f64, d: usize, fs: u32, peak: *mut caf_b200_peak) -> c_int;
    // device-resident surface objects: what CafSurfaceRow holds (fields are private upstream, mod.rs:17-22)
    pub fn caf_b200_surface_create_f64(h: caf_b200_handle, needle: *const Complex64, haystack: *const Complex64, l: usize,
                                       freqs_hz: *const f64, d: usize, fs: u32, out: *mut caf_b200_surface) -> c_int;
    pub fn caf_b200_surface_shape(s: caf_b200_surface, rows: *mut usize, cells_per_row: *mut usize) -> c_int;
    pub fn caf_b200_surface_row_peaks(s: caf_b200_surface, freq_hz: *mut f64, peak_val: *mut f64, peak_idx: *mut u64) -> c_int;
    pub fn caf_b200_surface_find_peak(s: caf_b200_surface, out: *mut caf_b200_peak) -> c_int;
    pub fn caf_b200_surface_fetch_rows(s: caf_b200_surface, row0: usize, count: usize, out: *mut c_void) -> c_int;
    pub fn caf_b200_surface_destroy(s: caf_b200_surface) -> c_int;
    // non-coherent integration: the surfaces of k segment pairs [k][l] summed cell by cell into one f64 surface
    pub fn caf_b200_surface_create_integrated_f64(h: caf_b200_handle, needles: *const Complex64, haystacks: *const Complex64,
                                                  k: usize, l: usize, freqs_hz: *const f64, d: usize, fs: u32,
                                                  out: *mut caf_b200_surface) -> c_int;
    pub fn caf_b200_surface_create_integrated_f32(h: caf_b200_handle, needles: *const Complex32, haystacks: *const Complex32,
                                                  k: usize, l: usize, freqs_hz: *const f64, d: usize, fs: u32,
                                                  out: *mut caf_b200_surface) -> c_int;
    pub fn caf_b200_integrate_f64_dev(h: caf_b200_handle, needles: *const Complex64, haystacks: *const Complex64, k: usize,
                                      l: usize, freqs_hz: *const f64, d: usize, fs: u32, surface: *mut f64,
                                      row_peak_val: *mut f64, row_peak_idx: *mut u64, peak: *mut caf_b200_peak) -> c_int;
    pub fn caf_b200_integrate_f32_dev(h: caf_b200_handle, needles: *const Complex32, haystacks: *const Complex32, k: usize,
                                      l: usize, freqs_hz: *const f64, d: usize, fs: u32, surface: *mut f64,
                                      row_peak_val: *mut f64, row_peak_idx: *mut u64, peak: *mut caf_b200_peak) -> c_int;
    // detection: the strongest local maxima of a stored surface (host records), or of device surfaces [p][d][n]
    pub fn caf_b200_surface_detect(s: caf_b200_surface, k_max: usize, guard_doppler: u32, guard_delay: u32, min_ratio: f64,
                                   out: *mut caf_b200_detection, count: *mut usize) -> c_int;
    pub fn caf_b200_detect_f64_dev(h: caf_b200_handle, surface: *const f64, p: usize, d: usize, n: usize,
                                   freqs_hz: *const f64, k_max: usize, guard_doppler: u32, guard_delay: u32, min_ratio: f64,
                                   out: *mut caf_b200_detection, counts: *mut u64) -> c_int;
    pub fn caf_b200_detect_f32_dev(h: caf_b200_handle, surface: *const f32, p: usize, d: usize, n: usize,
                                   freqs_hz: *const f64, k_max: usize, guard_doppler: u32, guard_delay: u32, min_ratio: f64,
                                   out: *mut caf_b200_detection, counts: *mut u64) -> c_int;
    // CFAR detection: local maxima above scale x their local noise estimate, and the dense noise map
    pub fn caf_b200_surface_detect_cfar(s: caf_b200_surface, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                        train_doppler: u32, train_delay: u32, scale: f64,
                                        out: *mut caf_b200_cfar_detection, count: *mut usize) -> c_int;
    pub fn caf_b200_detect_cfar_f64_dev(h: caf_b200_handle, surface: *const f64, p: usize, d: usize, n: usize,
                                        freqs_hz: *const f64, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                        train_doppler: u32, train_delay: u32, scale: f64,
                                        out: *mut caf_b200_cfar_detection, counts: *mut u64) -> c_int;
    pub fn caf_b200_detect_cfar_f32_dev(h: caf_b200_handle, surface: *const f32, p: usize, d: usize, n: usize,
                                        freqs_hz: *const f64, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                        train_doppler: u32, train_delay: u32, scale: f64,
                                        out: *mut caf_b200_cfar_detection, counts: *mut u64) -> c_int;
    pub fn caf_b200_cfar_noise_f64_dev(h: caf_b200_handle, surface: *const f64, p: usize, d: usize, n: usize,
                                       guard_doppler: u32, guard_delay: u32, train_doppler: u32, train_delay: u32,
                                       noise_out: *mut f64) -> c_int;
    pub fn caf_b200_cfar_noise_f32_dev(h: caf_b200_handle, surface: *const f32, p: usize, d: usize, n: usize,
                                       guard_doppler: u32, guard_delay: u32, train_doppler: u32, train_delay: u32,
                                       noise_out: *mut f64) -> c_int;
    // OS-CFAR detection: the same against the rank-th smallest training cell, and its dense noise map
    pub fn caf_b200_surface_detect_cfar_os(s: caf_b200_surface, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                           train_doppler: u32, train_delay: u32, rank: u32, scale: f64,
                                           out: *mut caf_b200_cfar_detection, count: *mut usize) -> c_int;
    pub fn caf_b200_detect_cfar_os_f64_dev(h: caf_b200_handle, surface: *const f64, p: usize, d: usize, n: usize,
                                           freqs_hz: *const f64, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                           train_doppler: u32, train_delay: u32, rank: u32, scale: f64,
                                           out: *mut caf_b200_cfar_detection, counts: *mut u64) -> c_int;
    pub fn caf_b200_detect_cfar_os_f32_dev(h: caf_b200_handle, surface: *const f32, p: usize, d: usize, n: usize,
                                           freqs_hz: *const f64, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                           train_doppler: u32, train_delay: u32, rank: u32, scale: f64,
                                           out: *mut caf_b200_cfar_detection, counts: *mut u64) -> c_int;
    pub fn caf_b200_cfar_os_noise_f64_dev(h: caf_b200_handle, surface: *const f64, p: usize, d: usize, n: usize,
                                          guard_doppler: u32, guard_delay: u32, train_doppler: u32, train_delay: u32,
                                          rank: u32, noise_out: *mut f64) -> c_int;
    pub fn caf_b200_cfar_os_noise_f32_dev(h: caf_b200_handle, surface: *const f32, p: usize, d: usize, n: usize,
                                          guard_doppler: u32, guard_delay: u32, train_doppler: u32, train_delay: u32,
                                          rank: u32, noise_out: *mut f64) -> c_int;
    // detection on the owned rows of a row block of a sharded surface (records carry global rows), and the merge of
    // the ranks' lists (device memory)
    pub fn caf_b200_detect_rows_f64_dev(h: caf_b200_handle, surface: *const f64, d_buf: usize, n: usize,
                                        freqs_hz: *const f64, row_lo: usize, row_hi: usize, row_offset: u64,
                                        d_global: usize, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                        min_ratio: f64, out: *mut caf_b200_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_detect_rows_f32_dev(h: caf_b200_handle, surface: *const f32, d_buf: usize, n: usize,
                                        freqs_hz: *const f64, row_lo: usize, row_hi: usize, row_offset: u64,
                                        d_global: usize, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                        min_ratio: f64, out: *mut caf_b200_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_detect_cfar_rows_f64_dev(h: caf_b200_handle, surface: *const f64, d_buf: usize, n: usize,
                                             freqs_hz: *const f64, row_lo: usize, row_hi: usize, row_offset: u64,
                                             d_global: usize, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                             train_doppler: u32, train_delay: u32, scale: f64,
                                             out: *mut caf_b200_cfar_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_detect_cfar_rows_f32_dev(h: caf_b200_handle, surface: *const f32, d_buf: usize, n: usize,
                                             freqs_hz: *const f64, row_lo: usize, row_hi: usize, row_offset: u64,
                                             d_global: usize, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                             train_doppler: u32, train_delay: u32, scale: f64,
                                             out: *mut caf_b200_cfar_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_detect_cfar_os_rows_f64_dev(h: caf_b200_handle, surface: *const f64, d_buf: usize, n: usize,
                                                freqs_hz: *const f64, row_lo: usize, row_hi: usize, row_offset: u64,
                                                d_global: usize, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                                train_doppler: u32, train_delay: u32, rank: u32, scale: f64,
                                                out: *mut caf_b200_cfar_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_detect_cfar_os_rows_f32_dev(h: caf_b200_handle, surface: *const f32, d_buf: usize, n: usize,
                                                freqs_hz: *const f64, row_lo: usize, row_hi: usize, row_offset: u64,
                                                d_global: usize, k_max: usize, guard_doppler: u32, guard_delay: u32,
                                                train_doppler: u32, train_delay: u32, rank: u32, scale: f64,
                                                out: *mut caf_b200_cfar_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_detect_merge_dev(h: caf_b200_handle, lists: *const caf_b200_detection, counts: *const u64,
                                     world: usize, k_max: usize, min_ratio: f64, out: *mut caf_b200_detection,
                                     count: *mut u64) -> c_int;
    pub fn caf_b200_cfar_merge_dev(h: caf_b200_handle, lists: *const caf_b200_cfar_detection, counts: *const u64,
                                   world: usize, k_max: usize, out: *mut caf_b200_cfar_detection, count: *mut u64) -> c_int;
    // read_file_c64 straight onto the device, and device memory for callers without a CUDA runtime of their own
    pub fn caf_b200_load_c64_dev_f64(h: caf_b200_handle, path: *const c_char, first_sample: usize, max_samples: usize,
                                     dev_out: *mut *mut Complex64, n_out: *mut usize) -> c_int;
    pub fn caf_b200_dev_free(p: *mut c_void) -> c_int;
    pub fn caf_b200_dev_alloc(h: caf_b200_handle, bytes: usize, dev_out: *mut *mut c_void) -> c_int;
    pub fn caf_b200_dev_upload(h: caf_b200_handle, dev_dst: *mut c_void, host_src: *const c_void, bytes: usize) -> c_int;
    pub fn caf_b200_dev_download(h: caf_b200_handle, host_dst: *mut c_void, dev_src: *const c_void, bytes: usize) -> c_int;
    pub fn caf_b200_batch_f64_dev(h: caf_b200_handle, needles: *const Complex64, haystacks: *const Complex64, p: usize, l: usize,
                                  freqs_hz: *const f64, d: usize, fs: u32, surface: *mut f64, row_peak_val: *mut f64,
                                  row_peak_idx: *mut u64, peaks: *mut caf_b200_peak) -> c_int;
    pub fn caf_b200_host_alloc(out: *mut *mut c_void, bytes: usize) -> c_int;
    pub fn caf_b200_host_free(p: *mut c_void) -> c_int;
    // sibling layouts (caf_go / caf_python conventions): layout 1 = Python [d][l], 2 = Go [d][2l], |xcor|
    pub fn caf_b200_surface_layout_f64(h: caf_b200_handle, needle: *const Complex64, haystack: *const Complex64, l: usize,
                                       freqs_hz: *const f64, d: usize, fs: u32, layout: c_int, out: *mut f64,
                                       peak: *mut caf_b200_peak) -> c_int;
    // multi-GPU: the library's own NCCL communicator (libnccl is dlopen()ed by the library, nothing to link here)
    pub fn caf_b200_comm_unique_id(id: *mut u8) -> c_int;
    pub fn caf_b200_comm_create(h: caf_b200_handle, world: c_int, rank: c_int, id: *const u8, out: *mut caf_b200_comm) -> c_int;
    pub fn caf_b200_comm_destroy(c: caf_b200_comm) -> c_int;
    pub fn caf_b200_comm_shard(c: caf_b200_comm, n: usize, lo: *mut usize, hi: *mut usize) -> c_int;
    pub fn caf_b200_surface_sharded_f64(h: caf_b200_handle, c: caf_b200_comm, needle: *const Complex64,
                                        haystack: *const Complex64, l: usize, freqs_hz: *const f64, d: usize, fs: u32,
                                        surface_local: *mut f64, peak: *mut caf_b200_peak) -> c_int;
    pub fn caf_b200_detect_allgather_dev(h: caf_b200_handle, c: caf_b200_comm, local: *const caf_b200_detection,
                                         local_count: *const u64, k_max: usize, min_ratio: f64,
                                         out: *mut caf_b200_detection, count: *mut u64) -> c_int;
    pub fn caf_b200_cfar_allgather_dev(h: caf_b200_handle, c: caf_b200_comm, local: *const caf_b200_cfar_detection,
                                       local_count: *const u64, k_max: usize, out: *mut caf_b200_cfar_detection,
                                       count: *mut u64) -> c_int;
}

#[repr(C)]
pub struct caf_b200_surface_s { _private: [u8; 0] }
pub type caf_b200_surface = *mut caf_b200_surface_s;

#[repr(C)]
pub struct caf_b200_comm_s { _private: [u8; 0] }
pub type caf_b200_comm = *mut caf_b200_comm_s;
pub const CAF_B200_NCCL_ID_BYTES: usize = 128;

/// One lazily created handle per thread: the trait functions are associated functions without `self`, callable
/// from any thread (rayon workers included), and a handle is not thread-safe.
pub struct ThreadHandle(pub caf_b200_handle);
impl Drop for ThreadHandle {
    fn drop(&mut self) { unsafe { caf_b200_destroy(self.0); } }
}
thread_local! {
    pub static HANDLE: ThreadHandle = {
        let mut h: caf_b200_handle = std::ptr::null_mut();
        let rc = unsafe { caf_b200_create(0, &mut h) };
        if rc != 0 { panic!("caf_b200_create failed ({}): {}", rc, last_error()); }
        ThreadHandle(h)
    };
}

pub fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(caf_b200_last_error()).to_string_lossy().into_owned() }
}

/// The reference panics where this library returns a status (xcor_rustfft.rs:54-55 assert!, unwrap()s).
pub fn check(rc: c_int) {
    if rc != 0 { panic!("caf_b200 status {}: {}", rc, last_error()); }
}
