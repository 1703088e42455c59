//! ns_gpu.rs -- drop-in for `nnnoiseless::{DenoiseState, FRAME_SIZE}` as sleep3r/crispy uses it
//! (src-tauri/src/audio.rs:4, :203, :229, :268), backed by libcrispy_ns.so (include/crispy_ns.h).
//!
//! Place in src-tauri/src/, add `mod ns_gpu;` to main.rs, and change audio.rs:4 from
//!     use nnnoiseless::{DenoiseState, FRAME_SIZE as RNNOISE_FRAME_SIZE};
//! to
//!     use crate::ns_gpu::{DenoiseState, FRAME_SIZE as RNNOISE_FRAME_SIZE};
//! Nothing else in audio.rs changes: the field `denoise: Box<DenoiseState<'static>>` (audio.rs:203), the
//! constructor call `DenoiseState::new()` (:229) and `self.denoise.process_frame(&mut out_buf[..], &in_buf[..])`
//! (:268) type-check against the items below -- `DenoiseState` carries the same lifetime parameter as the crate's
//! (there it borrows the model; here it is a marker).
//! One behavioural difference: nnnoiseless' `new()` cannot fail; this one needs a CUDA device (the library has no
//! CPU fallback) and panics with the library's message if there is none -- under the reference's
//! `panic = "abort"` (Cargo.toml:10-20) that ends the process.  `DenoiseState::try_new()` returns the error instead.
//! NOT COMPILED IN THIS REPOSITORY: the build image has no Rust toolchain (DESIGN.md section 0).  The C entry
//! points it binds are compiled against the header by a C consumer (tests/c_abi/abi_smoke.c) and exercised through
//! ctypes by the test-suite.
use std::marker::PhantomData;
use std::os::raw::{c_char, c_float, c_int, c_void};

#[repr(C)]
pub struct CrispyNsModel {
    _p: [u8; 0],
}
#[repr(C)]
pub struct CrispyNsState {
    _p: [u8; 0],
}
#[repr(C)]
pub struct CrispyNsBatch {
    _p: [u8; 0],
}
#[repr(C)]
pub struct CrispyNsMulti {
    _p: [u8; 0],
}

pub const CRISPY_NS_IN_I16: u32 = 1 << 0;
pub const CRISPY_NS_OUT_I16: u32 = 1 << 1;
pub const CRISPY_NS_UNIT_SCALE: u32 = 1 << 2;
pub const CRISPY_NS_MIX_STEREO_I16: u32 = 1 << 3;
pub const CRISPY_NS_DROP_FIRST_FRAME: u32 = 1 << 8;

/// numerics of a model (crispy_ns_model_set_numerics): the sum order of the pitch path's inner products | the biquad's
/// arithmetic.  0 is xiph's C; every handle created from the model copies the setting.
pub const CRISPY_NS_SUM_SEQUENTIAL: u32 = 0;
pub const CRISPY_NS_SUM_DOT4: u32 = 1;
pub const CRISPY_NS_SUM_DOT4_XCORR: u32 = 2;
pub const CRISPY_NS_SUM_MASK: u32 = 3;
pub const CRISPY_NS_BIQUAD_F32: u32 = 1 << 4;

extern "C" {
    fn crispy_ns_last_error() -> *const c_char;
    fn crispy_ns_device_count() -> c_int;
    pub fn crispy_ns_model_set_numerics(m: *mut CrispyNsModel, numerics: u32) -> c_int;
    pub fn crispy_ns_model_numerics(m: *const CrispyNsModel) -> u32;
    fn crispy_ns_create(model: *const CrispyNsModel, device: c_int, out: *mut *mut CrispyNsState) -> c_int;
    fn crispy_ns_process_frame(st: *mut CrispyNsState, out480: *mut c_float, in480: *const c_float, vad: *mut c_float) -> c_int;
    fn crispy_ns_reset(st: *mut CrispyNsState) -> c_int;
    fn crispy_ns_destroy(st: *mut CrispyNsState);
    fn crispy_ns_batch_create(model: *const CrispyNsModel, device: c_int, n_streams: c_int, out: *mut *mut CrispyNsBatch) -> c_int;
    fn crispy_ns_process_streams_host(
        b: *mut CrispyNsBatch, h_in: *const c_void, h_out: *mut c_void, h_vad: *mut c_float, h_app: *const c_float,
        n_frames: c_int, in_stride: i64, out_stride: i64, vad_stride: i64, app_stride: i64, flags: u32, volume: c_float,
    ) -> c_int;
    fn crispy_ns_batch_state_size(b: *const CrispyNsBatch) -> usize;
    fn crispy_ns_batch_save_state(b: *mut CrispyNsBatch, buf: *mut c_void, len: usize) -> c_int;
    fn crispy_ns_batch_load_state(b: *mut CrispyNsBatch, buf: *const c_void, len: usize) -> c_int;
    fn crispy_ns_process_streams_subset_host(
        b: *mut CrispyNsBatch, streams: *const c_int, n_active: c_int, h_in: *const c_void, h_out: *mut c_void,
        h_vad: *mut c_float, h_app: *const c_float, n_frames: c_int, in_stride: i64, out_stride: i64, vad_stride: i64,
        app_stride: i64, flags: u32, volume: c_float,
    ) -> c_int;
    fn crispy_ns_batch_reset_streams(b: *mut CrispyNsBatch, streams: *const c_int, n: c_int, cuda_stream: *mut c_void) -> c_int;
    fn crispy_ns_stream_state_size() -> usize;
    fn crispy_ns_batch_save_streams(b: *mut CrispyNsBatch, streams: *const c_int, n: c_int, buf: *mut c_void, len: usize) -> c_int;
    fn crispy_ns_batch_load_streams(b: *mut CrispyNsBatch, streams: *const c_int, n: c_int, buf: *const c_void, len: usize)
                                    -> c_int;
    fn crispy_ns_batch_destroy(b: *mut CrispyNsBatch);
    fn crispy_ns_multi_create(model: *const CrispyNsModel, devices: *const c_int, n_devices: c_int, n_streams: c_int,
                              out: *mut *mut CrispyNsMulti) -> c_int;
    fn crispy_ns_multi_process_streams_host(
        m: *mut CrispyNsMulti, h_in: *const c_void, h_out: *mut c_void, h_vad: *mut c_float, h_app: *const c_float,
        n_frames: c_int, in_stride: i64, out_stride: i64, vad_stride: i64, app_stride: i64, flags: u32, volume: c_float,
    ) -> c_int;
    fn crispy_ns_multi_destroy(m: *mut CrispyNsMulti);
    fn crispy_ns_denoise_wav_files(model: *const CrispyNsModel, device: c_int, paths_in: *const *const c_char,
                                   paths_out: *const *const c_char, n_files: c_int, flags: u32, volume: c_float,
                                   mean_vad: *mut c_float) -> c_int;
    fn crispy_ns_linear_resample_count(input_rate: c_float, output_rate: c_float, n_in: i64) -> i64;
    fn crispy_ns_sinc_resample_count(input_rate: c_int, output_rate: c_int, n_in: i64) -> i64;
    fn crispy_ns_resample_audio_count(n_in: i64, from_rate: c_int, to_rate: c_int) -> i64;
    fn crispy_ns_resample_host(device: c_int, h_in: *const c_float, h_out: *mut c_float, n_streams: c_int, n_in: i64,
                               in_stride: i64, out_stride: i64, input_rate: c_int, output_rate: c_int, kind: c_int) -> c_int;
}

/// == nnnoiseless::FRAME_SIZE (audio.rs:4)
pub const FRAME_SIZE: usize = 480;

fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(crispy_ns_last_error()).to_string_lossy().into_owned() }
}

/// Same surface as `nnnoiseless::DenoiseState<'model>` as audio.rs uses it: `Box<DenoiseState<'static>>`
/// (audio.rs:203), `DenoiseState::new()` (:229), `process_frame(&mut [f32], &[f32]) -> f32` (:268).
pub struct DenoiseState<'model> {
    h: *mut CrispyNsState,
    _model: PhantomData<&'model ()>,
}
// guarded by Mutex<NsState> exactly like today (audio.rs:693); the handle itself is not thread-safe
unsafe impl<'model> Send for DenoiseState<'model> {}

impl DenoiseState<'static> {
    /// audio.rs:229 `DenoiseState::new()`: the built-in model ($CRISPY_NS_WEIGHTS, else synthetic seed 0) on device 0
    pub fn new() -> Box<DenoiseState<'static>> {
        match Self::try_new() {
            Ok(b) => b,
            Err(e) => panic!("crispy_ns_create failed: {}", e),
        }
    }
    pub fn try_new() -> Result<Box<DenoiseState<'static>>, String> {
        let mut h = std::ptr::null_mut();
        let rc = unsafe { crispy_ns_create(std::ptr::null(), 0, &mut h) };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(Box::new(DenoiseState { h, _model: PhantomData }))
    }
}

impl<'model> DenoiseState<'model> {
    /// audio.rs:268 `process_frame(&mut out[..], &in[..])`: 480 f32 in 16-bit scale in and out; returns
    /// the VAD probability (the reference discards it).
    pub fn process_frame(&mut self, output: &mut [f32], input: &[f32]) -> f32 {
        assert_eq!(input.len(), FRAME_SIZE); // upstream asserts too
        assert_eq!(output.len(), FRAME_SIZE);
        let mut vad = 0f32;
        let rc = unsafe { crispy_ns_process_frame(self.h, output.as_mut_ptr(), input.as_ptr(), &mut vad) };
        assert!(rc == 0, "crispy_ns_process_frame failed: {}", last_error());
        vad
    }
    /// a fresh state, as the model switch at audio.rs:955-965 builds
    pub fn reset(&mut self) {
        let rc = unsafe { crispy_ns_reset(self.h) };
        assert!(rc == 0, "crispy_ns_reset failed: {}", last_error());
    }
}
impl<'model> Drop for DenoiseState<'model> {
    fn drop(&mut self) {
        unsafe { crispy_ns_destroy(self.h) }
    }
}

/// Many independent recordings at once (north_star `process_streams`): `n_streams` rows of
/// `n_frames * 480` unit-scale f32 samples, `stride` samples apart; arithmetic of
/// RnnNoiseProcessor::push_sample (audio.rs:261-278) fused into the kernels' load/store.
pub struct BatchDenoiser {
    h: *mut CrispyNsBatch,
    n_streams: usize,
}
unsafe impl Send for BatchDenoiser {}

impl BatchDenoiser {
    pub fn new(n_streams: usize, device: i32) -> Result<BatchDenoiser, String> {
        if unsafe { crispy_ns_device_count() } == 0 {
            return Err("no CUDA device: libcrispy_ns has no CPU fallback".into());
        }
        let mut h = std::ptr::null_mut();
        let rc = unsafe { crispy_ns_batch_create(std::ptr::null(), device, n_streams as c_int, &mut h) };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(BatchDenoiser { h, n_streams })
    }
    /// State persists across calls, so a long recording can be fed in pieces.
    pub fn process_streams(&mut self, input: &[f32], output: &mut [f32], vad: Option<&mut [f32]>, n_frames: usize,
                           stride: usize, volume: f32, drop_first_frame: bool) -> Result<(), String> {
        assert!(input.len() >= (self.n_streams - 1) * stride + n_frames * FRAME_SIZE);
        assert!(output.len() >= (self.n_streams - 1) * stride + n_frames * FRAME_SIZE);
        let mut flags = CRISPY_NS_UNIT_SCALE;
        if drop_first_frame {
            flags |= CRISPY_NS_DROP_FIRST_FRAME;
        }
        let (vad_ptr, vad_stride) = match vad {
            Some(v) => {
                assert!(v.len() >= self.n_streams * n_frames);
                (v.as_mut_ptr(), n_frames as i64)
            }
            None => (std::ptr::null_mut(), 0),
        };
        let rc = unsafe {
            crispy_ns_process_streams_host(self.h, input.as_ptr() as *const c_void, output.as_mut_ptr() as *mut c_void, vad_ptr,
                                           std::ptr::null(), n_frames as c_int, stride as i64, stride as i64, vad_stride, 0,
                                           flags, volume)
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(())
    }
    /// recorder path (commands/recording.rs:260-264 + recording.rs:108-110): mic denoised + app raw ->
    /// clamp -> interleaved dual-mono PCM16
    pub fn process_and_mix(&mut self, mic: &[f32], app: &[f32], out_pcm16: &mut [i16], n_frames: usize, stride: usize)
                           -> Result<(), String> {
        assert!(out_pcm16.len() >= 2 * ((self.n_streams - 1) * stride + n_frames * FRAME_SIZE));
        let rc = unsafe {
            crispy_ns_process_streams_host(self.h, mic.as_ptr() as *const c_void, out_pcm16.as_mut_ptr() as *mut c_void,
                                           std::ptr::null_mut(), app.as_ptr(), n_frames as c_int, stride as i64, stride as i64,
                                           0, stride as i64, CRISPY_NS_UNIT_SCALE | CRISPY_NS_MIX_STEREO_I16, 1.0)
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(())
    }
    pub fn save_state(&mut self) -> Result<Vec<u8>, String> {
        let n = unsafe { crispy_ns_batch_state_size(self.h) };
        let mut buf = vec![0u8; n];
        let rc = unsafe { crispy_ns_batch_save_state(self.h, buf.as_mut_ptr() as *mut c_void, n) };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(buf)
    }
    pub fn load_state(&mut self, buf: &[u8]) -> Result<(), String> {
        let rc = unsafe { crispy_ns_batch_load_state(self.h, buf.as_ptr() as *const c_void, buf.len()) };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(())
    }
    /// Streams that advance independently: row i of `input` / `output` (`n_frames * 480` unit-scale samples,
    /// `stride` apart) is batch stream `streams[i]`; every other stream is left as it was.
    pub fn process_streams_subset(&mut self, streams: &[i32], input: &[f32], output: &mut [f32], n_frames: usize,
                                  stride: usize, volume: f32) -> Result<(), String> {
        if let Some(rows) = streams.len().checked_sub(1) {
            assert!(input.len() >= rows * stride + n_frames * FRAME_SIZE);
            assert!(output.len() >= rows * stride + n_frames * FRAME_SIZE);
        }
        let rc = unsafe {
            crispy_ns_process_streams_subset_host(self.h, streams.as_ptr(), streams.len() as c_int,
                                                  input.as_ptr() as *const c_void, output.as_mut_ptr() as *mut c_void,
                                                  std::ptr::null_mut(), std::ptr::null(), n_frames as c_int, stride as i64,
                                                  stride as i64, 0, 0, CRISPY_NS_UNIT_SCALE, volume)
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(())
    }
    /// fresh DenoiseStates for the listed streams, ordered before the next call
    pub fn reset_streams(&mut self, streams: &[i32]) -> Result<(), String> {
        let rc = unsafe { crispy_ns_batch_reset_streams(self.h, streams.as_ptr(), streams.len() as c_int, std::ptr::null_mut()) };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(())
    }
    /// one self-describing record per listed stream; it loads into any stream of any batch of this build
    pub fn save_streams(&mut self, streams: &[i32]) -> Result<Vec<u8>, String> {
        let n = streams.len() * unsafe { crispy_ns_stream_state_size() };
        let mut buf = vec![0u8; n];
        let rc = unsafe {
            crispy_ns_batch_save_streams(self.h, streams.as_ptr(), streams.len() as c_int, buf.as_mut_ptr() as *mut c_void, n)
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(buf)
    }
    pub fn load_streams(&mut self, streams: &[i32], buf: &[u8]) -> Result<(), String> {
        let rc = unsafe {
            crispy_ns_batch_load_streams(self.h, streams.as_ptr(), streams.len() as c_int, buf.as_ptr() as *const c_void,
                                         buf.len())
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(())
    }
}
impl Drop for BatchDenoiser {
    fn drop(&mut self) {
        unsafe { crispy_ns_batch_destroy(self.h) }
    }
}

/// The same batch over every GPU of the box from this one process (crispy_ns_multi_*: contiguous blocks of streams
/// per device, one host thread per device inside the library, nothing exchanged between devices).
pub struct MultiDenoiser {
    h: *mut CrispyNsMulti,
    n_streams: usize,
}
unsafe impl Send for MultiDenoiser {}

impl MultiDenoiser {
    pub fn new(n_streams: usize, devices: &[i32]) -> Result<MultiDenoiser, String> {
        let mut h = std::ptr::null_mut();
        let rc = unsafe { crispy_ns_multi_create(std::ptr::null(), devices.as_ptr(), devices.len() as c_int, n_streams as c_int, &mut h) };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(MultiDenoiser { h, n_streams })
    }
    /// PCM16 in and out (what the recorder stores, recording.rs:101-121): half the bytes on the host link.
    pub fn process_streams_pcm16(&mut self, input: &[i16], output: &mut [i16], n_frames: usize, stride: usize) -> Result<(), String> {
        assert!(input.len() >= (self.n_streams - 1) * stride + n_frames * FRAME_SIZE);
        assert!(output.len() >= (self.n_streams - 1) * stride + n_frames * FRAME_SIZE);
        let rc = unsafe {
            crispy_ns_multi_process_streams_host(self.h, input.as_ptr() as *const c_void, output.as_mut_ptr() as *mut c_void,
                                                 std::ptr::null_mut(), std::ptr::null(), n_frames as c_int, stride as i64,
                                                 stride as i64, 0, 0, CRISPY_NS_IN_I16 | CRISPY_NS_OUT_I16, 1.0)
        };
        if rc == 0 { Ok(()) } else { Err(last_error()) }
    }
}
impl Drop for MultiDenoiser {
    fn drop(&mut self) {
        unsafe { crispy_ns_multi_destroy(self.h) }
    }
}

/// Finished recordings (recording.rs:83-99 WAVs) in, denoised dual-mono WAVs out; returns each file's mean VAD.
pub fn denoise_wav_files(paths_in: &[std::path::PathBuf], paths_out: &[std::path::PathBuf]) -> Result<Vec<f32>, String> {
    use std::ffi::CString;
    assert_eq!(paths_in.len(), paths_out.len());
    let cin: Vec<CString> = paths_in.iter().map(|p| CString::new(p.to_string_lossy().as_bytes()).unwrap()).collect();
    let cout: Vec<CString> = paths_out.iter().map(|p| CString::new(p.to_string_lossy().as_bytes()).unwrap()).collect();
    let pin: Vec<*const c_char> = cin.iter().map(|c| c.as_ptr()).collect();
    let pout: Vec<*const c_char> = cout.iter().map(|c| c.as_ptr()).collect();
    let mut vad = vec![0f32; paths_in.len()];
    let rc = unsafe {
        crispy_ns_denoise_wav_files(std::ptr::null(), 0, pin.as_ptr(), pout.as_ptr(), pin.len() as c_int, 0, 1.0, vad.as_mut_ptr())
    };
    if rc == 0 { Ok(vad) } else { Err(last_error()) }
}

/// Front end for recordings that are not at 48 kHz (audio.rs:217-221 uses the linear interpolator; `sinc` selects the
/// windowed-sinc kernel, the rubato-style alternative).  `input` holds `n_streams` rows of `n_in` samples.
pub fn resample_to_48k(input: &[f32], n_streams: usize, n_in: usize, input_rate: u32, sinc: bool) -> Result<Vec<f32>, String> {
    let n_out = unsafe {
        if sinc { crispy_ns_sinc_resample_count(input_rate as c_int, 48000, n_in as i64) }
        else { crispy_ns_linear_resample_count(input_rate as c_float, 48000.0, n_in as i64) }
    } as usize;
    let mut out = vec![0f32; n_streams * n_out];
    let rc = unsafe {
        crispy_ns_resample_host(0, input.as_ptr(), out.as_mut_ptr(), n_streams as c_int, n_in as i64, n_in as i64,
                                n_out.max(1) as i64, input_rate as c_int, 48000, if sinc { 1 } else { 0 })
    };
    if rc == 0 { Ok(out) } else { Err(last_error()) }
}

/// recording.rs:13-39 `resample_audio(samples, from_rate, to_rate)` for many buffers of one length at once
/// (row-major `[n_streams][n_in]` in, `[n_streams][n_out]` out): bit-identical to the recorder's own loop.
pub fn resample_audio_batch(input: &[f32], n_streams: usize, from_rate: usize, to_rate: usize) -> Result<Vec<f32>, String> {
    assert!(n_streams > 0 && input.len() % n_streams == 0);
    let n_in = input.len() / n_streams;
    let n_out = unsafe { crispy_ns_resample_audio_count(n_in as i64, from_rate as c_int, to_rate as c_int) } as usize;
    let mut out = vec![0f32; n_streams * n_out];
    let rc = unsafe {
        crispy_ns_resample_host(0, input.as_ptr(), out.as_mut_ptr(), n_streams as c_int, n_in as i64, n_in as i64,
                                n_out.max(1) as i64, from_rate as c_int, to_rate as c_int, 2)
    };
    if rc == 0 { Ok(out) } else { Err(last_error()) }
}
