//! Drop-in replacement for `aprilgrid::detector::TagDetector` backed by the B200 CUDA library.
//!
//! Same signatures as the reference (aprilgrid 0.8.0, src/detector.rs):
//!   * `TagDetector::new(&TagFamily, Option<DetectorParams>) -> TagDetector`        (:364)
//!   * `detect(&self, &DynamicImage) -> HashMap<u32, [(f32, f32); 4]>`              (:505)
//!   * `detect_kornia<const N: usize>(&self, &kornia::image::Image<u8, N>)`         (:479)
//!   * `refined_saddle_points(&self, &DynamicImage) -> Vec<Saddle>`                 (:408)
//! plus the added `detect_batch(&self, &[DynamicImage]) -> Vec<HashMap<..>>` (one GPU) and
//! `MultiTagDetector::detect_batch` (every GPU of the box, frames sharded image-wise).  A slice of
//! images of mixed sizes or pixel formats goes through the frame-list entry points
//! (`ag_detect_frames`, ...), each image from its own buffer.
//!
//! NOT a full drop-in: the lower-level public functions the reference's `examples/develop.rs`
//! uses (`decode_positions`, `bit_code`, `best_tag`, `rochade_refine`, `init_quads`,
//! `try_find_best_board`, `Board`, `is_valid_quad`) are not re-exported -- they are internal
//! stages of the CUDA pipeline here (INTEGRATION.md lists what replaces them).
//!
//! `new` is infallible in the reference, so a failure to reach the GPU panics here (there is
//! no CPU fallback by design).  This file is shipped as source: the build image has no cargo.
use image::DynamicImage;
use std::collections::HashMap;
use std::os::raw::{c_char, c_int, c_long, c_void};
use std::sync::Mutex;

#[derive(Debug, Clone, Copy)]
pub enum TagFamily {
    T16H5 = 0,
    T25H7 = 1,
    T25H9 = 2,
    T36H11 = 3,
    /// 1 bit border
    T36H11B1 = 4,
}

impl std::str::FromStr for TagFamily {
    type Err = std::fmt::Error;
    fn from_str(s: &str) -> Result<Self, Self::Err> {
        let c = std::ffi::CString::new(s).map_err(|_| std::fmt::Error)?;
        let mut fam: c_int = 0;
        if unsafe { ffi::ag_family_from_str(c.as_ptr(), &mut fam) } != 0 {
            return Err(std::fmt::Error);
        }
        Ok(match fam {
            0 => TagFamily::T16H5,
            1 => TagFamily::T25H7,
            2 => TagFamily::T25H9,
            3 => TagFamily::T36H11,
            _ => TagFamily::T36H11B1,
        })
    }
}

#[repr(C)]
#[derive(Debug, Clone, Copy)]
pub struct DetectorParams {
    pub tag_spacing_ratio: f32,
    pub min_saddle_angle: f32,
    pub max_saddle_angle: f32,
    pub max_num_of_boards: u8,
}

impl DetectorParams {
    pub fn default_params() -> DetectorParams {
        DetectorParams { tag_spacing_ratio: 0.3, min_saddle_angle: 30.0, max_saddle_angle: 60.0, max_num_of_boards: 2 }
    }
}

/// `aprilgrid::saddle::Saddle` (src/saddle.rs:3-9).
#[derive(Debug, Clone, Copy, Default)]
pub struct Saddle {
    pub p: (f32, f32),
    pub k: f32,
    pub theta: f32,
    pub phi: f32,
}

/// `ag_saddle` of include/aprilgrid_b200.h: five plain floats (a Rust tuple has no defined
/// layout, so the public `Saddle` is never handed to C).
#[repr(C)]
#[derive(Clone, Copy, Default)]
struct AgSaddle {
    x: f32,
    y: f32,
    k: f32,
    theta: f32,
    phi: f32,
}

#[repr(C)]
#[derive(Clone, Copy)]
struct AgTag {
    id: u32,
    xy: [f32; 8],
}

/// `ag_frame` of include/aprilgrid_b200.h: one image of a frame list.
#[repr(C)]
#[derive(Clone, Copy)]
struct AgFrame {
    pixels: *const c_void,
    width: c_int,
    height: c_int,
    row_stride: usize,
    format: c_int,
}

mod ffi {
    use super::*;
    #[repr(C)]
    pub struct AgDetector {
        _private: [u8; 0],
    }
    #[repr(C)]
    pub struct AgMulti {
        _private: [u8; 0],
    }
    extern "C" {
        pub fn ag_family_from_str(name: *const c_char, family_out: *mut c_int) -> c_int;
        pub fn ag_create(family: c_int, params: *const DetectorParams, device: c_int, out: *mut *mut AgDetector) -> c_int;
        pub fn ag_destroy(det: *mut AgDetector);
        pub fn ag_last_error(det: *const AgDetector) -> *const c_char;
        pub fn ag_detect(det: *mut AgDetector, pixels: *const c_void, width: c_int, height: c_int, row_stride: usize,
                         format: c_int, out: *mut AgTag, cap: c_int, n: *mut c_int) -> c_int;
        pub fn ag_detect_planes(det: *mut AgDetector, luma32f: *const f32, f32_row_stride: usize, luma8: *const u8,
                                u8_row_stride: usize, width: c_int, height: c_int, out: *mut AgTag, cap: c_int,
                                n: *mut c_int) -> c_int;
        pub fn ag_detect_batch(det: *mut AgDetector, frames: *const c_void, frame_stride: usize, n_frames: c_int,
                               width: c_int, height: c_int, row_stride: usize, format: c_int, out: *mut AgTag,
                               cap_per_frame: c_int, n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
        pub fn ag_set_option(det: *mut AgDetector, key: *const c_char, value: c_long) -> c_int;
        pub fn ag_detect_batch_wait(det: *mut AgDetector, keep_in_flight: c_int) -> c_int;
        pub fn ag_refined_saddle_points(det: *mut AgDetector, pixels: *const c_void, width: c_int, height: c_int,
                                        row_stride: usize, format: c_int, out: *mut AgSaddle, cap: c_int, n: *mut c_int) -> c_int;
        pub fn ag_refined_saddle_points_batch(det: *mut AgDetector, frames: *const c_void, frame_stride: usize,
                                              n_frames: c_int, width: c_int, height: c_int, row_stride: usize,
                                              format: c_int, out: *mut AgSaddle, cap_per_frame: c_int,
                                              n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
        pub fn ag_detect_frames(det: *mut AgDetector, frames: *const AgFrame, n_frames: c_int, out: *mut AgTag,
                                cap_per_frame: c_int, n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
        pub fn ag_refined_saddle_points_frames(det: *mut AgDetector, frames: *const AgFrame, n_frames: c_int,
                                               out: *mut AgSaddle, cap_per_frame: c_int, n_per_frame: *mut c_int,
                                               frame_status: *mut u32) -> c_int;
        pub fn ag_multi_detect_frames(m: *mut AgMulti, frames: *const AgFrame, n_frames: c_int, out: *mut AgTag,
                                      cap_per_frame: c_int, n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
        pub fn ag_multi_refined_saddle_points_frames(m: *mut AgMulti, frames: *const AgFrame, n_frames: c_int,
                                                     out: *mut AgSaddle, cap_per_frame: c_int,
                                                     n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
        pub fn ag_host_alloc(bytes: usize) -> *mut c_void;
        pub fn ag_host_free(p: *mut c_void);
        pub fn ag_multi_create(family: c_int, params: *const DetectorParams, devices: *const c_int, n_devices: c_int,
                               out: *mut *mut AgMulti) -> c_int;
        pub fn ag_multi_destroy(m: *mut AgMulti);
        pub fn ag_multi_last_error(m: *const AgMulti) -> *const c_char;
        pub fn ag_multi_detect_batch(m: *mut AgMulti, frames: *const c_void, frame_stride: usize, n_frames: c_int,
                                     width: c_int, height: c_int, row_stride: usize, format: c_int, out: *mut AgTag,
                                     cap_per_frame: c_int, n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
        pub fn ag_multi_refined_saddle_points_batch(m: *mut AgMulti, frames: *const c_void, frame_stride: usize,
                                                    n_frames: c_int, width: c_int, height: c_int, row_stride: usize,
                                                    format: c_int, out: *mut AgSaddle, cap_per_frame: c_int,
                                                    n_per_frame: *mut c_int, frame_status: *mut u32) -> c_int;
    }
}

const AG_L8: c_int = 0;
const AG_L16: c_int = 1;
const AG_RGB8: c_int = 2;
const AG_LA8: c_int = 4;
const AG_RGBA8: c_int = 5;
const AG_LA16: c_int = 6;
const AG_RGB16: c_int = 7;
const AG_RGBA16: c_int = 8;
const AG_RGB32F: c_int = 9;
const AG_RGBA32F: c_int = 10;
const AG_ERR_CAPACITY: c_int = 4;
const TAG_CAP: usize = 1024; // >= the largest family (587 codes)
const SADDLE_CAP: usize = 16384; // the library's hard limit per frame

/// Page-locked host buffer (ag_host_alloc): frames packed here upload at the PCIe rate.
struct Pinned {
    ptr: *mut u8,
    len: usize,
}
impl Pinned {
    fn new(len: usize) -> Pinned {
        let ptr = unsafe { ffi::ag_host_alloc(len.max(1)) } as *mut u8;
        if ptr.is_null() {
            panic!("aprilgrid_b200: ag_host_alloc({len}) failed");
        }
        Pinned { ptr, len }
    }
    fn as_mut_slice(&mut self) -> &mut [u8] {
        unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) }
    }
}
impl Drop for Pinned {
    fn drop(&mut self) {
        unsafe { ffi::ag_host_free(self.ptr as *mut c_void) }
    }
}
unsafe impl Send for Pinned {}

/// One C handle serialises the calls made on it.  The reference's `TagDetector` is `Send + Sync`
/// and `detect(&self)` runs concurrently from many threads, so this type keeps a POOL of handles:
/// a call checks one out (creating another if all are busy) and returns it afterwards.
pub struct TagDetector {
    family: TagFamily,
    params: DetectorParams,
    device: c_int,
    pool: Mutex<Vec<*mut ffi::AgDetector>>,
}
unsafe impl Send for TagDetector {}
unsafe impl Sync for TagDetector {}

impl Drop for TagDetector {
    fn drop(&mut self) {
        for h in self.pool.lock().unwrap().drain(..) {
            unsafe { ffi::ag_destroy(h) }
        }
    }
}

fn last_error(h: *const ffi::AgDetector) -> String {
    unsafe { std::ffi::CStr::from_ptr(ffi::ag_last_error(h)).to_string_lossy().into_owned() }
}

fn u16_bytes(raw: &[u16]) -> &[u8] {
    unsafe { std::slice::from_raw_parts(raw.as_ptr() as *const u8, raw.len() * 2) }
}
fn f32_bytes(raw: &[f32]) -> &[u8] {
    unsafe { std::slice::from_raw_parts(raw.as_ptr() as *const u8, raw.len() * 4) }
}

/// Raw pixel view of a DynamicImage: (bytes, pixel format, row stride in bytes, width, height).  All ten
/// variants are passed through untouched and converted to gray on the GPU as `image` 0.25 does it.
fn pixels_of(img: &DynamicImage) -> (&[u8], c_int, usize, u32, u32) {
    let (w, h) = (img.width(), img.height());
    let (bytes, fmt, bpp) = match img {
        DynamicImage::ImageLuma8(b) => (b.as_raw().as_slice(), AG_L8, 1),
        DynamicImage::ImageRgb8(b) => (b.as_raw().as_slice(), AG_RGB8, 3),
        DynamicImage::ImageLuma16(b) => (u16_bytes(b.as_raw()), AG_L16, 2),
        DynamicImage::ImageLumaA8(b) => (b.as_raw().as_slice(), AG_LA8, 2),
        DynamicImage::ImageRgba8(b) => (b.as_raw().as_slice(), AG_RGBA8, 4),
        DynamicImage::ImageLumaA16(b) => (u16_bytes(b.as_raw()), AG_LA16, 4),
        DynamicImage::ImageRgb16(b) => (u16_bytes(b.as_raw()), AG_RGB16, 6),
        DynamicImage::ImageRgba16(b) => (u16_bytes(b.as_raw()), AG_RGBA16, 8),
        DynamicImage::ImageRgb32F(b) => (f32_bytes(b.as_raw()), AG_RGB32F, 12),
        DynamicImage::ImageRgba32F(b) => (f32_bytes(b.as_raw()), AG_RGBA32F, 16),
        _ => panic!("aprilgrid_b200: unsupported DynamicImage variant"),
    };
    (bytes, fmt, bpp * w as usize, w, h)
}

fn corners(t: &AgTag) -> [(f32, f32); 4] {
    [(t.xy[0], t.xy[1]), (t.xy[2], t.xy[3]), (t.xy[4], t.xy[5]), (t.xy[6], t.xy[7])]
}

fn saddle_lists_of(out: &[AgSaddle], counts: &[c_int], cap: usize) -> Vec<Vec<Saddle>> {
    (0..counts.len())
        .map(|i| {
            out[i * cap..i * cap + (counts[i] as usize).min(cap)]
                .iter()
                .map(|s| Saddle { p: (s.x, s.y), k: s.k, theta: s.theta, phi: s.phi })
                .collect()
        })
        .collect()
}

fn maps_of(out: &[AgTag], counts: &[c_int], cap: usize) -> Vec<HashMap<u32, [(f32, f32); 4]>> {
    (0..counts.len())
        .map(|i| out[i * cap..i * cap + (counts[i] as usize).min(cap)].iter().map(|t| (t.id, corners(t))).collect())
        .collect()
}

/// Whether every image of a slice has the size and pixel format of the first.
fn uniform(imgs: &[DynamicImage]) -> bool {
    let (_, fmt, _, w, h) = pixels_of(&imgs[0]);
    imgs.iter().all(|im| {
        let (_, f, _, ww, hh) = pixels_of(im);
        ww == w && hh == h && f == fmt
    })
}

/// Frame-list descriptors of a slice: each image read from its own buffer (valid while `imgs` is borrowed).
fn frames_of(imgs: &[DynamicImage]) -> Vec<AgFrame> {
    imgs.iter()
        .map(|im| {
            let (bytes, fmt, stride, w, h) = pixels_of(im);
            AgFrame { pixels: bytes.as_ptr() as *const c_void, width: w as c_int, height: h as c_int, row_stride: stride,
                      format: fmt }
        })
        .collect()
}

/// Pack equally sized images of one pixel format into one pinned buffer.
fn pack(imgs: &[DynamicImage]) -> (Pinned, u32, u32, c_int, usize) {
    let (_, fmt, stride, w, h) = pixels_of(&imgs[0]);
    let frame_bytes = stride * h as usize;
    let mut packed = Pinned::new(frame_bytes * imgs.len());
    for (i, im) in imgs.iter().enumerate() {
        let (bytes, f, _, ww, hh) = pixels_of(im);
        assert!(ww == w && hh == h && f == fmt, "detect_batch: all frames must have the same size and pixel format");
        packed.as_mut_slice()[i * frame_bytes..(i + 1) * frame_bytes].copy_from_slice(&bytes[..frame_bytes]);
    }
    (packed, w, h, fmt, stride)
}

impl TagDetector {
    pub fn new(tag_family: &TagFamily, optional_detector_params: Option<DetectorParams>) -> TagDetector {
        let params = optional_detector_params.unwrap_or(DetectorParams::default_params());
        let device: c_int = std::env::var("APRILGRID_B200_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        let det = TagDetector { family: *tag_family, params, device, pool: Mutex::new(Vec::new()) };
        let h = det.checkout(); // fail here, loudly, if the GPU cannot be reached
        det.checkin(h);
        det
    }

    fn checkout(&self) -> *mut ffi::AgDetector {
        if let Some(h) = self.pool.lock().unwrap().pop() {
            return h;
        }
        let mut h: *mut ffi::AgDetector = std::ptr::null_mut();
        let rc = unsafe { ffi::ag_create(self.family as c_int, &self.params, self.device, &mut h) };
        if rc != 0 {
            panic!("aprilgrid_b200: ag_create failed ({rc}): {}", last_error(std::ptr::null()));
        }
        h
    }
    fn checkin(&self, h: *mut ffi::AgDetector) {
        self.pool.lock().unwrap().push(h);
    }

    pub fn detect(&self, img: &DynamicImage) -> HashMap<u32, [(f32, f32); 4]> {
        match img {
            // exact by construction: the reference's own conversions
            DynamicImage::ImageRgb32F(_) | DynamicImage::ImageRgba32F(_) => self.detect_planes(img),
            _ => {
                let (bytes, fmt, stride, w, h) = pixels_of(img);
                self.detect_raw(bytes.as_ptr(), w, h, stride, fmt)
            }
        }
    }

    /// The float variants: the reference's own conversions (`to_luma32f`, `to_luma8`), both planes to the GPU.
    fn detect_planes(&self, img: &DynamicImage) -> HashMap<u32, [(f32, f32); 4]> {
        let luma32f = img.to_luma32f();
        let luma8 = img.to_luma8();
        let (w, h) = (img.width(), img.height());
        let mut out = vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP];
        let mut n: c_int = 0;
        let det = self.checkout();
        let rc = unsafe {
            ffi::ag_detect_planes(det, luma32f.as_raw().as_ptr(), 0, luma8.as_raw().as_ptr(), 0, w as c_int, h as c_int,
                                  out.as_mut_ptr(), TAG_CAP as c_int, &mut n)
        };
        if rc != 0 {
            let msg = last_error(det);
            self.checkin(det);
            panic!("aprilgrid_b200: ag_detect_planes failed ({rc}): {msg}");
        }
        self.checkin(det);
        out[..n as usize].iter().map(|t| (t.id, corners(t))).collect()
    }

    fn detect_raw(&self, ptr: *const u8, w: u32, h: u32, stride: usize, fmt: c_int) -> HashMap<u32, [(f32, f32); 4]> {
        let mut out = vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP];
        let mut n: c_int = 0;
        let det = self.checkout();
        let rc = unsafe {
            ffi::ag_detect(det, ptr as *const c_void, w as c_int, h as c_int, stride, fmt, out.as_mut_ptr(),
                           TAG_CAP as c_int, &mut n)
        };
        // the reference's detect has no error path: anything but success is a bug or a frame beyond the
        // library's hard limits (AG_ERR_CAPACITY: > 16384 saddles) -- never a silently truncated map
        if rc != 0 {
            let msg = last_error(det);
            self.checkin(det);
            panic!("aprilgrid_b200: ag_detect failed ({rc}): {msg}");
        }
        self.checkin(det);
        out[..n as usize].iter().map(|t| (t.id, corners(t))).collect()
    }

    /// New: one call for a batch of images.  Equally sized images of one pixel format are packed into
    /// one pinned buffer; a slice of mixed sizes or formats goes through `ag_detect_frames` unpacked.
    pub fn detect_batch(&self, imgs: &[DynamicImage]) -> Vec<HashMap<u32, [(f32, f32); 4]>> {
        if imgs.is_empty() {
            return Vec::new();
        }
        if !uniform(imgs) {
            let frames = frames_of(imgs);
            let mut out = vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP * imgs.len()];
            let mut counts = vec![0 as c_int; imgs.len()];
            let det = self.checkout();
            let rc = unsafe {
                ffi::ag_detect_frames(det, frames.as_ptr(), imgs.len() as c_int, out.as_mut_ptr(), TAG_CAP as c_int,
                                      counts.as_mut_ptr(), std::ptr::null_mut())
            };
            if rc != 0 {
                let msg = last_error(det);
                self.checkin(det);
                panic!("aprilgrid_b200: ag_detect_frames failed ({rc}): {msg}");
            }
            self.checkin(det);
            return maps_of(&out, &counts, TAG_CAP);
        }
        let (packed, w, h, fmt, stride) = pack(imgs);
        let mut out = vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP * imgs.len()];
        let mut counts = vec![0 as c_int; imgs.len()];
        let det = self.checkout();
        let rc = unsafe {
            ffi::ag_detect_batch(det, packed.ptr as *const c_void, stride * h as usize, imgs.len() as c_int, w as c_int,
                                 h as c_int, stride, fmt, out.as_mut_ptr(), TAG_CAP as c_int, counts.as_mut_ptr(),
                                 std::ptr::null_mut())
        };
        if rc != 0 {
            let msg = last_error(det);
            self.checkin(det);
            panic!("aprilgrid_b200: ag_detect_batch failed ({rc}): {msg}");
        }
        self.checkin(det);
        maps_of(&out, &counts, TAG_CAP)
    }

    /// New: a stream of batches over host frames (`BatchStream::submit` / `wait`): the uploads of one
    /// batch overlap the board searches of the one before.  The stream owns its own handle, so the
    /// synchronous methods of the detector stay usable meanwhile.
    pub fn stream(&self) -> BatchStream {
        let det = self.checkout();
        let key = std::ffi::CString::new("host_async").unwrap();
        unsafe { ffi::ag_set_option(det, key.as_ptr(), 1) };
        BatchStream { det, pending: std::collections::VecDeque::new() }
    }

    pub fn refined_saddle_points(&self, img: &DynamicImage) -> Vec<Saddle> {
        let (bytes, fmt, stride, w, h) = pixels_of(img);
        let mut out = vec![AgSaddle::default(); 16384];
        let mut n: c_int = 0;
        let det = self.checkout();
        let rc = unsafe {
            ffi::ag_refined_saddle_points(det, bytes.as_ptr() as *const c_void, w as c_int, h as c_int, stride, fmt,
                                          out.as_mut_ptr(), out.len() as c_int, &mut n)
        };
        if rc != 0 {
            let msg = last_error(det);
            self.checkin(det);
            panic!("aprilgrid_b200: ag_refined_saddle_points failed ({rc}): {msg}");
        }
        self.checkin(det);
        out[..n as usize].iter().map(|s| Saddle { p: (s.x, s.y), k: s.k, theta: s.theta, phi: s.phi }).collect()
    }

    /// New: `refined_saddle_points` of every image of a batch (mixed sizes and formats as in `detect_batch`).
    pub fn refined_saddle_points_batch(&self, imgs: &[DynamicImage]) -> Vec<Vec<Saddle>> {
        if imgs.is_empty() {
            return Vec::new();
        }
        if !uniform(imgs) {
            let frames = frames_of(imgs);
            let mut out = vec![AgSaddle::default(); SADDLE_CAP * imgs.len()];
            let mut counts = vec![0 as c_int; imgs.len()];
            let det = self.checkout();
            let rc = unsafe {
                ffi::ag_refined_saddle_points_frames(det, frames.as_ptr(), imgs.len() as c_int, out.as_mut_ptr(),
                                                     SADDLE_CAP as c_int, counts.as_mut_ptr(), std::ptr::null_mut())
            };
            if rc != 0 {
                let msg = last_error(det);
                self.checkin(det);
                panic!("aprilgrid_b200: ag_refined_saddle_points_frames failed ({rc}): {msg}");
            }
            self.checkin(det);
            return saddle_lists_of(&out, &counts, SADDLE_CAP);
        }
        let (packed, w, h, fmt, stride) = pack(imgs);
        let mut out = vec![AgSaddle::default(); SADDLE_CAP * imgs.len()];
        let mut counts = vec![0 as c_int; imgs.len()];
        let det = self.checkout();
        let rc = unsafe {
            ffi::ag_refined_saddle_points_batch(det, packed.ptr as *const c_void, stride * h as usize, imgs.len() as c_int,
                                                w as c_int, h as c_int, stride, fmt, out.as_mut_ptr(), SADDLE_CAP as c_int,
                                                counts.as_mut_ptr(), std::ptr::null_mut())
        };
        if rc != 0 {
            let msg = last_error(det);
            self.checkin(det);
            panic!("aprilgrid_b200: ag_refined_saddle_points_batch failed ({rc}): {msg}");
        }
        self.checkin(det);
        saddle_lists_of(&out, &counts, SADDLE_CAP)
    }

    #[cfg(feature = "kornia")]
    pub fn detect_kornia<const N: usize>(&self, img: &kornia::image::Image<u8, N>) -> HashMap<u32, [(f32, f32); 4]> {
        let (fmt, stride) = match img.num_channels() {
            1 => (AG_L8, img.width()),
            3 => (AG_RGB8, 3 * img.width()),
            _ => panic!("Only support u8c1 and u8c3"), // as the reference (src/detector.rs:500)
        };
        self.detect_raw(img.as_slice().as_ptr(), img.width() as u32, img.height() as u32, stride, fmt)
    }
}

/// A batch in flight on a `BatchStream`: it owns the packed (pinned) frames and the output arrays
/// the library fills until `wait` has covered it.
struct InFlight {
    _frames: Pinned,
    out: Vec<AgTag>,
    counts: Vec<c_int>,
}

/// Streaming use of `detect_batch` (ag_detect_batch with "host_async" + ag_detect_batch_wait).
pub struct BatchStream {
    det: *mut ffi::AgDetector,
    pending: std::collections::VecDeque<InFlight>,
}
unsafe impl Send for BatchStream {}

impl BatchStream {
    /// Enqueue one batch and return at once.
    pub fn submit(&mut self, imgs: &[DynamicImage]) {
        if imgs.is_empty() {
            return;
        }
        let (packed, w, h, fmt, stride) = pack(imgs);
        let mut b = InFlight { _frames: packed, out: vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP * imgs.len()],
                               counts: vec![0 as c_int; imgs.len()] };
        let rc = unsafe {
            ffi::ag_detect_batch(self.det, b._frames.ptr as *const c_void, stride * h as usize, imgs.len() as c_int,
                                 w as c_int, h as c_int, stride, fmt, b.out.as_mut_ptr(), TAG_CAP as c_int,
                                 b.counts.as_mut_ptr(), std::ptr::null_mut())
        };
        if rc != 0 {
            panic!("aprilgrid_b200: ag_detect_batch failed ({rc}): {}", last_error(self.det));
        }
        self.pending.push_back(b); // the heap buffers of `b` do not move when the struct does
    }

    /// Block until all but the newest `keep_in_flight` batches are complete; returns their results,
    /// oldest batch first.
    pub fn wait(&mut self, keep_in_flight: usize) -> Vec<Vec<HashMap<u32, [(f32, f32); 4]>>> {
        let rc = unsafe { ffi::ag_detect_batch_wait(self.det, keep_in_flight as c_int) };
        if rc != 0 && rc != AG_ERR_CAPACITY {
            panic!("aprilgrid_b200: ag_detect_batch_wait failed ({rc}): {}", last_error(self.det));
        }
        let mut done = Vec::new();
        while self.pending.len() > keep_in_flight {
            let b = self.pending.pop_front().unwrap();
            done.push(maps_of(&b.out, &b.counts, TAG_CAP));
        }
        done
    }
}

impl Drop for BatchStream {
    fn drop(&mut self) {
        unsafe {
            ffi::ag_detect_batch_wait(self.det, 0); // nothing may still write into `pending`
            ffi::ag_destroy(self.det);
        }
    }
}

/// `detect_batch` over every GPU of the box (ag_multi_*): the batch is cut into contiguous frame
/// ranges, one per device, each on its own host thread; results come back in frame order.
pub struct MultiTagDetector {
    m: *mut ffi::AgMulti,
}
unsafe impl Send for MultiTagDetector {}

impl MultiTagDetector {
    /// `devices`: CUDA ordinals; empty = every visible device.
    pub fn new(tag_family: &TagFamily, optional_detector_params: Option<DetectorParams>, devices: &[i32]) -> MultiTagDetector {
        let params = optional_detector_params.unwrap_or(DetectorParams::default_params());
        let mut m: *mut ffi::AgMulti = std::ptr::null_mut();
        let rc = unsafe {
            ffi::ag_multi_create(*tag_family as c_int, &params, if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() },
                                 devices.len() as c_int, &mut m)
        };
        if rc != 0 {
            let msg = unsafe { std::ffi::CStr::from_ptr(ffi::ag_multi_last_error(std::ptr::null())).to_string_lossy().into_owned() };
            panic!("aprilgrid_b200: ag_multi_create failed ({rc}): {msg}");
        }
        MultiTagDetector { m }
    }

    pub fn detect_batch(&mut self, imgs: &[DynamicImage]) -> Vec<HashMap<u32, [(f32, f32); 4]>> {
        if imgs.is_empty() {
            return Vec::new();
        }
        if !uniform(imgs) {
            let frames = frames_of(imgs);
            let mut out = vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP * imgs.len()];
            let mut counts = vec![0 as c_int; imgs.len()];
            let rc = unsafe {
                ffi::ag_multi_detect_frames(self.m, frames.as_ptr(), imgs.len() as c_int, out.as_mut_ptr(),
                                            TAG_CAP as c_int, counts.as_mut_ptr(), std::ptr::null_mut())
            };
            if rc != 0 {
                let msg = unsafe { std::ffi::CStr::from_ptr(ffi::ag_multi_last_error(self.m)).to_string_lossy().into_owned() };
                panic!("aprilgrid_b200: ag_multi_detect_frames failed ({rc}): {msg}");
            }
            return maps_of(&out, &counts, TAG_CAP);
        }
        let (packed, w, h, fmt, stride) = pack(imgs);
        let mut out = vec![AgTag { id: 0, xy: [0.0; 8] }; TAG_CAP * imgs.len()];
        let mut counts = vec![0 as c_int; imgs.len()];
        let rc = unsafe {
            ffi::ag_multi_detect_batch(self.m, packed.ptr as *const c_void, stride * h as usize, imgs.len() as c_int,
                                       w as c_int, h as c_int, stride, fmt, out.as_mut_ptr(), TAG_CAP as c_int,
                                       counts.as_mut_ptr(), std::ptr::null_mut())
        };
        if rc != 0 {
            let msg = unsafe { std::ffi::CStr::from_ptr(ffi::ag_multi_last_error(self.m)).to_string_lossy().into_owned() };
            panic!("aprilgrid_b200: ag_multi_detect_batch failed ({rc}): {msg}");
        }
        maps_of(&out, &counts, TAG_CAP)
    }

    pub fn refined_saddle_points_batch(&mut self, imgs: &[DynamicImage]) -> Vec<Vec<Saddle>> {
        if imgs.is_empty() {
            return Vec::new();
        }
        if !uniform(imgs) {
            let frames = frames_of(imgs);
            let mut out = vec![AgSaddle::default(); SADDLE_CAP * imgs.len()];
            let mut counts = vec![0 as c_int; imgs.len()];
            let rc = unsafe {
                ffi::ag_multi_refined_saddle_points_frames(self.m, frames.as_ptr(), imgs.len() as c_int,
                                                           out.as_mut_ptr(), SADDLE_CAP as c_int, counts.as_mut_ptr(),
                                                           std::ptr::null_mut())
            };
            if rc != 0 {
                let msg = unsafe { std::ffi::CStr::from_ptr(ffi::ag_multi_last_error(self.m)).to_string_lossy().into_owned() };
                panic!("aprilgrid_b200: ag_multi_refined_saddle_points_frames failed ({rc}): {msg}");
            }
            return saddle_lists_of(&out, &counts, SADDLE_CAP);
        }
        let (packed, w, h, fmt, stride) = pack(imgs);
        let mut out = vec![AgSaddle::default(); SADDLE_CAP * imgs.len()];
        let mut counts = vec![0 as c_int; imgs.len()];
        let rc = unsafe {
            ffi::ag_multi_refined_saddle_points_batch(self.m, packed.ptr as *const c_void, stride * h as usize,
                                                      imgs.len() as c_int, w as c_int, h as c_int, stride, fmt,
                                                      out.as_mut_ptr(), SADDLE_CAP as c_int, counts.as_mut_ptr(),
                                                      std::ptr::null_mut())
        };
        if rc != 0 {
            let msg = unsafe { std::ffi::CStr::from_ptr(ffi::ag_multi_last_error(self.m)).to_string_lossy().into_owned() };
            panic!("aprilgrid_b200: ag_multi_refined_saddle_points_batch failed ({rc}): {msg}");
        }
        saddle_lists_of(&out, &counts, SADDLE_CAP)
    }
}

impl Drop for MultiTagDetector {
    fn drop(&mut self) {
        unsafe { ffi::ag_multi_destroy(self.m) }
    }
}
