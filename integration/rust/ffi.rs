//! src/ffi.rs — binding of include/wafer_b200.h.  UNTESTED here (no Rust toolchain in the build image).
//!
//! `Array3<R64>` created by `zeros` / `from_elem` / `from_shape_fn` is a standard-layout C-order array and `R64`
//! is a transparent wrapper around `f64`, so `as_ptr() as *const f64` is the padded buffer the library expects.
#![allow(dead_code)]
use errors::*;
use ndarray::Array3;
use noisy_float::prelude::*;
use std::ffi::{CStr, CString};
use std::os::raw::{c_char, c_int, c_void};
use std::ptr;

#[repr(C)]
pub struct WaferParams {
    pub nx: u64,
    pub ny: u64,
    pub nz: u64,
    pub ext: u32,
    pub dn: f64,
    pub dt: f64,
    pub mass: f64,
    pub device: i32,
    pub rank: u32,
    pub world: u32,
    pub nccl_id: *const u8,
    pub max_lower: u32,
    pub flags: u32,
}

#[repr(C)]
#[derive(Default, Debug, Clone, Copy)]
pub struct WaferObservables {
    pub energy: f64,
    pub norm2: f64,
    pub v_infinity: f64,
    pub r2: f64,
}

#[repr(C)]
#[derive(Default, Debug, Clone, Copy)]
pub struct WaferWriteStats {
    pub bytes: u64,
    pub file_bytes: u64,
    pub host_formatted: u64,
}

#[repr(C)]
#[derive(Default, Debug, Clone, Copy)]
pub struct WaferLoadStats {
    pub sx: u64,
    pub sy: u64,
    pub sz: u64,
    pub bytes_read: u64,
    pub sites_converted: u64,
    pub host_converted: u64,
}

/// `WAFER_ERR_FORMAT`: the file is not in a layout the device decoder reads; nothing changed.
pub const WAFER_ERR_FORMAT: c_int = 10;

pub enum WaferCtx {}

extern "C" {
    fn wafer_create(p: *const WaferParams, out: *mut *mut WaferCtx) -> c_int;
    fn wafer_destroy(ctx: *mut WaferCtx) -> c_int;
    fn wafer_last_error(ctx: *const WaferCtx) -> *const c_char;
    fn wafer_set_potential(ctx: *mut WaferCtx, v_padded: *const f64) -> c_int;
    fn wafer_set_pot_sub_scalar(ctx: *mut WaferCtx, c: f64) -> c_int;
    fn wafer_set_pot_sub_array(ctx: *mut WaferCtx, work: *const f64) -> c_int;
    fn wafer_set_phi(ctx: *mut WaferCtx, phi_padded: *const f64) -> c_int;
    fn wafer_get_phi(ctx: *mut WaferCtx, phi_padded: *mut f64) -> c_int;
    fn wafer_push_lower(ctx: *mut WaferCtx, q_padded: *const f64) -> c_int;
    fn wafer_push_lower_from_phi(ctx: *mut WaferCtx) -> c_int;
    fn wafer_phi_from_lower(ctx: *mut WaferCtx, idx: u32) -> c_int;
    fn wafer_phi_seed_from_lower(ctx: *mut WaferCtx, idx: u32) -> c_int;
    fn wafer_generate_gaussian(ctx: *mut WaferCtx, sig: f64, seed: u64) -> c_int;
    fn wafer_symmetrise(ctx: *mut WaferCtx, kind: i32) -> c_int;
    fn wafer_set_phi_resampled(ctx: *mut WaferCtx, src: *const f64, sx: u64, sy: u64, sz: u64, from_csv: u32) -> c_int;
    fn wafer_set_potential_resampled(ctx: *mut WaferCtx, src: *const f64, sx: u64, sy: u64, sz: u64, from_csv: u32) -> c_int;
    fn wafer_push_lower_resampled(ctx: *mut WaferCtx, src: *const f64, sx: u64, sy: u64, sz: u64, from_csv: u32) -> c_int;
    fn wafer_check(ctx: *mut WaferCtx, wnum: u8, out: *mut WaferObservables) -> c_int;
    fn wafer_normalise(ctx: *mut WaferCtx, norm2: f64) -> c_int;
    fn wafer_evolve(ctx: *mut WaferCtx, wnum: u8, steps: u64) -> c_int;
    fn wafer_write_array(ctx: *mut WaferCtx, what: i32, file_type: i32, path: *const c_char, stats: *mut WaferWriteStats) -> c_int;
    fn wafer_load_array(ctx: *mut WaferCtx, what: i32, file_type: i32, path: *const c_char, stats: *mut WaferLoadStats) -> c_int;
    fn wafer_synchronize(ctx: *mut WaferCtx) -> c_int;
    fn wafer_host_register(ptr: *mut c_void, bytes: usize) -> c_int;
    fn wafer_host_unregister(ptr: *mut c_void) -> c_int;
}

/// Owns one `wafer_ctx` (one GPU).  Used from the single thread that runs `grid::solve`.
pub struct Gpu {
    ctx: *mut WaferCtx,
}

impl Gpu {
    fn check(&self, rc: c_int) -> Result<()> {
        if rc == 0 {
            return Ok(());
        }
        let msg = unsafe { CStr::from_ptr(wafer_last_error(self.ctx)).to_string_lossy().into_owned() };
        if rc == 7 {
            Err(ErrorKind::MaxStep.into())
        } else {
            Err(format!("GPU hot path failed (status {}): {}", rc, msg).into())
        }
    }

    pub fn new(size: (usize, usize, usize), ext: usize, dn: R64, dt: R64, mass: R64, wavemax: u8) -> Result<Gpu> {
        let p = WaferParams {
            nx: size.0 as u64,
            ny: size.1 as u64,
            nz: size.2 as u64,
            ext: ext as u32,
            dn: dn.raw(),
            dt: dt.raw(),
            mass: mass.raw(),
            device: -1,
            rank: 0,
            world: 1,
            nccl_id: ptr::null(),
            max_lower: wavemax as u32,
            flags: 0,
        };
        let mut ctx: *mut WaferCtx = ptr::null_mut();
        let rc = unsafe { wafer_create(&p, &mut ctx) };
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(wafer_last_error(ptr::null())).to_string_lossy().into_owned() };
            return Err(format!("wafer_create failed (status {}): {}", rc, msg).into());
        }
        Ok(Gpu { ctx })
    }

    pub fn set_potential(&self, v: &Array3<R64>) -> Result<()> {
        self.check(unsafe { wafer_set_potential(self.ctx, v.as_ptr() as *const f64) })
    }
    pub fn set_pot_sub(&self, pot_sub: &(Option<Array3<R64>>, Option<R64>)) -> Result<()> {
        match *pot_sub {
            (Some(ref arr), None) => self.check(unsafe { wafer_set_pot_sub_array(self.ctx, arr.as_ptr() as *const f64) }),
            (None, Some(c)) => self.check(unsafe { wafer_set_pot_sub_scalar(self.ctx, c.raw()) }),
            _ => self.check(unsafe { wafer_set_pot_sub_scalar(self.ctx, 0.0) }),
        }
    }
    pub fn set_phi(&self, phi: &Array3<R64>) -> Result<()> {
        self.check(unsafe { wafer_set_phi(self.ctx, phi.as_ptr() as *const f64) })
    }
    pub fn get_phi(&self, phi: &mut Array3<R64>) -> Result<()> {
        self.check(unsafe { wafer_get_phi(self.ctx, phi.as_mut_ptr() as *mut f64) })
    }
    pub fn push_lower(&self, q: &Array3<R64>) -> Result<()> {
        self.check(unsafe { wafer_push_lower(self.ctx, q.as_ptr() as *const f64) })
    }
    pub fn push_lower_from_phi(&self) -> Result<()> {
        self.check(unsafe { wafer_push_lower_from_phi(self.ctx) })
    }
    pub fn phi_seed_from_lower(&self, idx: u32) -> Result<()> {
        self.check(unsafe { wafer_phi_seed_from_lower(self.ctx, idx) })
    }
    /// config.rs:636-642 on the device, keyed by `seed` instead of thread_rng: the same seed gives the same start.
    pub fn generate_gaussian(&self, sig: R64, seed: u64) -> Result<()> {
        self.check(unsafe { wafer_generate_gaussian(self.ctx, sig.raw(), seed) })
    }
    /// symmetrise_wavefunction (config.rs:691-728) for every ext: `kind` = `SymmetryConstraint as i32`.
    pub fn symmetrise(&self, kind: i32) -> Result<()> {
        self.check(unsafe { wafer_symmetrise(self.ctx, kind) })
    }
    /// fill_data / read_csv (input.rs:149-176, 641-657) on the device: `src` is the array of an input file as read (work
    /// area data, any shape with every axis >= 2, or the work shape for a Csv file), `from_csv` whether it came from a
    /// Csv file.  Only this rank's source planes are copied.
    pub fn set_phi_resampled(&self, src: &Array3<R64>, from_csv: bool) -> Result<()> {
        let (p, x, y, z) = resample_args(src)?;
        self.check(unsafe { wafer_set_phi_resampled(self.ctx, p, x, y, z, from_csv as u32) })
    }
    pub fn set_potential_resampled(&self, src: &Array3<R64>, from_csv: bool) -> Result<()> {
        let (p, x, y, z) = resample_args(src)?;
        self.check(unsafe { wafer_set_potential_resampled(self.ctx, p, x, y, z, from_csv as u32) })
    }
    pub fn push_lower_resampled(&self, src: &Array3<R64>, from_csv: bool) -> Result<()> {
        let (p, x, y, z) = resample_args(src)?;
        self.check(unsafe { wafer_push_lower_resampled(self.ctx, p, x, y, z, from_csv as u32) })
    }
    pub fn check_state(&self, wnum: u8) -> Result<WaferObservables> {
        let mut o = WaferObservables::default();
        self.check(unsafe { wafer_check(self.ctx, wnum, &mut o) })?;
        Ok(o)
    }
    pub fn normalise(&self, norm2: f64) -> Result<()> {
        self.check(unsafe { wafer_normalise(self.ctx, norm2) })
    }
    pub fn evolve(&self, wnum: u8, steps: u64) -> Result<()> {
        self.check(unsafe { wafer_evolve(self.ctx, wnum, steps) })
    }
    /// output::wavefunction / output::potential (output.rs:79-216) encoded on the device: the work area of psi
    /// (`what` 0) or V (1) to `path` as `file_type` 0 Messagepack, 1 Csv, 2 Json (`FileType as i32`; Yaml / Ron are
    /// refused).  Collective when world > 1: every rank passes the same path and writes its planes into the one file.
    pub fn write_array(&self, what: i32, file_type: i32, path: &str) -> Result<WaferWriteStats> {
        let c = CString::new(path).map_err(|_| Error::from("output path contains a NUL byte"))?;
        let mut st = WaferWriteStats::default();
        self.check(unsafe { wafer_write_array(self.ctx, what, file_type, c.as_ptr(), &mut st) })?;
        Ok(st)
    }
    /// input::load_wavefunctions / fill_data / read_csv (input.rs:113-176, 487-505, 607-662) decoded on the device: the
    /// file `path` of `file_type` 0 Messagepack, 1 Csv, 2 Json into psi (`what` 0), V (1) or a new lower state (2), as
    /// the `*_resampled` entries would set it from the parsed array.  Only the host writers' layouts are read: any other
    /// file returns `Err` with status 10 (`WAFER_ERR_FORMAT`) in the message and leaves everything as it was, so the caller parses it
    /// with `input.rs` and calls the `*_resampled` entry instead.  No communication when world > 1.
    pub fn load_array(&self, what: i32, file_type: i32, path: &str) -> Result<WaferLoadStats> {
        let c = CString::new(path).map_err(|_| Error::from("input path contains a NUL byte"))?;
        let mut st = WaferLoadStats::default();
        self.check(unsafe { wafer_load_array(self.ctx, what, file_type, c.as_ptr(), &mut st) })?;
        Ok(st)
    }
    /// Page-lock the buffer behind `arr` so that set_phi / get_phi run at PCIe speed (54 GB/s measured instead of the
    /// driver's 14 GB/s pageable path).  Call once after allocating the array; `unpin` before it is dropped.
    pub fn pin(&self, arr: &mut Array3<R64>) -> Result<()> {
        let bytes = arr.len() * ::std::mem::size_of::<f64>();
        self.check(unsafe { wafer_host_register(arr.as_mut_ptr() as *mut c_void, bytes) })
    }
    pub fn unpin(&self, arr: &mut Array3<R64>) {
        unsafe { wafer_host_unregister(arr.as_mut_ptr() as *mut c_void) };
    }
}

impl Drop for Gpu {
    fn drop(&mut self) {
        unsafe {
            wafer_synchronize(self.ctx);
            wafer_destroy(self.ctx);
        }
    }
}

/// pointer and shape of a C-order array for the wafer_*_resampled entries
fn resample_args(src: &Array3<R64>) -> Result<(*const f64, u64, u64, u64)> {
    if !src.is_standard_layout() {
        return Err("input array is not in standard (C) layout".into());
    }
    let (x, y, z) = src.dim();
    Ok((src.as_ptr() as *const f64, x as u64, y as u64, z as u64))
}
