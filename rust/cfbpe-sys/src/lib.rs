//! `cfbpe-sys`: raw bindings of `include/cfbpe.h` (ABI version 1) and [`Ctx`], a safe owner of one device context.
//!
//! NOT COMPILED in the repository this file lives in (no Rust toolchain there); kept in step with `include/cfbpe.h` by review.
//! Every entry point returns 0 or a negative `CFBPE_*` code; no panic or exception crosses the boundary; the caller owns every
//! buffer and the library never keeps a caller pointer past return (header, "Conventions").
#![allow(non_camel_case_types)]

use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr::NonNull;

pub const CFBPE_OK: c_int = 0;
pub const CFBPE_ENOENT: c_int = -2;
pub const CFBPE_EIO: c_int = -5;
pub const CFBPE_ENOMEM: c_int = -12;
pub const CFBPE_ENODEV: c_int = -19;
pub const CFBPE_EINVAL: c_int = -22;
pub const CFBPE_ENOSPC: c_int = -28;
pub const CFBPE_EILSEQ: c_int = -84;

pub const CFBPE_FORMAT_TIKTOKEN: u32 = 0;
pub const CFBPE_FORMAT_TEKKEN_JSON: u32 = 1;
pub const CFBPE_MAX_VOCABS: u32 = 8;
pub const CFBPE_KEEP_HEAD: u32 = 0;
pub const CFBPE_KEEP_TAIL: u32 = 1;
pub const CFBPE_MAX_DEVICES: usize = 8;

#[repr(C)]
pub struct cfbpe_ctx {
    _opaque: [u8; 0],
}

/// `cfbpe_config` (header): `struct_size` versions the struct; trailing fields a library does not know are ignored.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct cfbpe_config {
    pub struct_size: u32,
    pub device: i32,
    pub max_batch_bytes: u64,
    pub max_prompts: u32,
    pub flags: u32,
    /// CUDA device ordinals of a multi-device context (`n_devices` > 1: the batch is sharded by bytes across them)
    pub devices: [i32; CFBPE_MAX_DEVICES],
    pub n_devices: u32,
    /// independent workspaces per device: that many host calls run concurrently on one context
    pub n_workspaces: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct cfbpe_vocab_info {
    pub n_ranks: u32,
    pub pattern_id: u32,
    pub max_token_len: u32,
    pub n_pair_entries: u32,
    pub table_bytes: u64,
}

extern "C" {
    pub fn cfbpe_abi_version() -> c_int;
    pub fn cfbpe_build_id() -> *const c_char;
    pub fn cfbpe_create(cfg: *const cfbpe_config, out: *mut *mut cfbpe_ctx) -> c_int;
    pub fn cfbpe_destroy(ctx: *mut cfbpe_ctx);
    pub fn cfbpe_last_error(ctx: *const cfbpe_ctx) -> *const c_char;
    pub fn cfbpe_vocab_load(ctx: *mut cfbpe_ctx, vocab_id: u32, ranks_file: *const u8, len: usize, format: u32,
                            pattern_id: u32, max_ranks: u32) -> c_int;
    pub fn cfbpe_vocab_get_info(ctx: *const cfbpe_ctx, vocab_id: u32, out: *mut cfbpe_vocab_info) -> c_int;
    pub fn cfbpe_vocab_export(ctx: *const cfbpe_ctx, vocab_id: u32, buf: *mut u8, cap: u64, size: *mut u64) -> c_int;
    pub fn cfbpe_vocab_import(ctx: *mut cfbpe_ctx, vocab_id: u32, buf: *const u8, size: u64) -> c_int;
    pub fn cfbpe_encode_batch(ctx: *mut cfbpe_ctx, n_prompts: u32, bytes: *const u8, offsets: *const u64,
                              vocab_ids: *const u8, out_ids: *mut u32, out_cap: u64, out_offsets: *mut u64,
                              out_counts: *mut u32) -> c_int;
    pub fn cfbpe_count_batch(ctx: *mut cfbpe_ctx, n_prompts: u32, bytes: *const u8, offsets: *const u64,
                             vocab_ids: *const u8, out_counts: *mut u32) -> c_int;
    pub fn cfbpe_decode_batch(ctx: *mut cfbpe_ctx, n_seqs: u32, ids: *const u32, id_offsets: *const u64,
                              vocab_ids: *const u8, out_bytes: *mut u8, out_cap: u64, out_offsets: *mut u64) -> c_int;
    pub fn cfbpe_encode_batch_device(ctx: *mut cfbpe_ctx, n_prompts: u32, d_bytes: *const u8, total_bytes: u64,
                                     d_offsets: *const u64, d_vocab_ids: *const u8, d_out_ids: *mut u32, out_cap: u64,
                                     d_out_offsets: *mut u64, d_out_counts: *mut u32, n_tokens: *mut u64,
                                     stream: *mut c_void) -> c_int;
    pub fn cfbpe_encode_truncated(ctx: *mut cfbpe_ctx, n_prompts: u32, bytes: *const u8, offsets: *const u64, vocab_ids: *const u8,
                                  max_tokens: u32, keep: u32, pad_id: u32, budgets: *const u32, out_rows: *mut u32,
                                  out_kept: *mut u32, out_counts: *mut u32, out_cut: *mut u64) -> c_int;
    pub fn cfbpe_encode_truncated_device(ctx: *mut cfbpe_ctx, n_prompts: u32, d_bytes: *const u8, total_bytes: u64,
                                         d_offsets: *const u64, d_vocab_ids: *const u8, max_tokens: u32, keep: u32, pad_id: u32,
                                         d_budgets: *const u32, d_out_rows: *mut u32, d_out_kept: *mut u32, d_out_counts: *mut u32,
                                         d_out_cut: *mut u64, stream: *mut c_void) -> c_int;
    pub fn cfbpe_device_status(ctx: *mut cfbpe_ctx, stream: *mut c_void) -> c_int;
    pub fn cfbpe_host_alloc(ctx: *mut cfbpe_ctx, size: usize) -> *mut c_void;
    pub fn cfbpe_host_free(ctx: *mut cfbpe_ctx, ptr: *mut c_void);
}

/// Error of a native call: the C code and the library's message for it.
#[derive(Debug, thiserror::Error)]
#[error("cfbpe error {code}: {message}")]
pub struct NativeError {
    pub code: c_int,
    pub message: String,
}

/// Result of [`Ctx::encode_batch`]: a dense id stream, `n + 1` offsets into it, `n` counts.
#[derive(Debug, Default)]
pub struct Encoded {
    pub ids: Vec<u32>,
    pub offsets: Vec<u64>,
    pub counts: Vec<u32>,
}

/// Result of [`Ctx::encode_truncated`]: `n x max_tokens` rows (kept ids left-aligned, then `pad_id`; empty without ids),
/// the kept and untruncated counts, and the byte offset of the cut inside each prompt.
#[derive(Debug, Default)]
pub struct Truncated {
    pub rows: Vec<u32>,
    pub kept: Vec<u32>,
    pub counts: Vec<u32>,
    pub cut: Vec<u64>,
}

/// Safe owner of one `cfbpe_ctx`.  The context is internally synchronised (header: "safe to call concurrently from several
/// host threads"), so the wrapper is `Send + Sync` and plugin code shares it behind an `Arc`.
pub struct Ctx(NonNull<cfbpe_ctx>);

// SAFETY: the library serialises / pools access to the context's device state internally (include/cfbpe.h, threading note).
unsafe impl Send for Ctx {}
unsafe impl Sync for Ctx {}

impl Drop for Ctx {
    fn drop(&mut self) {
        // SAFETY: the pointer came from cfbpe_create and is destroyed exactly once.
        unsafe { cfbpe_destroy(self.0.as_ptr()) }
    }
}

impl Ctx {
    /// `devices`: CUDA ordinals (one = single-device context).  Fails with `CFBPE_ENODEV` when no sm_100 device is visible:
    /// there is no CPU fallback.
    pub fn create(devices: &[i32], max_batch_bytes: u64, max_prompts: u32, n_workspaces: u32) -> Result<Self, NativeError> {
        let mut cfg = cfbpe_config {
            struct_size: std::mem::size_of::<cfbpe_config>() as u32,
            device: devices.first().copied().unwrap_or(0),
            max_batch_bytes,
            max_prompts,
            flags: 0,
            devices: [0; CFBPE_MAX_DEVICES],
            n_devices: devices.len().min(CFBPE_MAX_DEVICES) as u32,
            n_workspaces,
        };
        for (slot, d) in cfg.devices.iter_mut().zip(devices) {
            *slot = *d;
        }
        let mut raw: *mut cfbpe_ctx = std::ptr::null_mut();
        // SAFETY: cfg and raw are valid for the call; the library writes raw only on success.
        let rc = unsafe { cfbpe_create(&cfg, &mut raw) };
        match NonNull::new(raw) {
            Some(p) if rc == CFBPE_OK => Ok(Self(p)),
            _ => Err(NativeError { code: rc, message: "cfbpe_create failed (no sm_100 device visible?)".to_owned() }),
        }
    }

    fn check(&self, rc: c_int) -> Result<(), NativeError> {
        if rc == CFBPE_OK {
            return Ok(());
        }
        // SAFETY: cfbpe_last_error returns a NUL-terminated string owned by the context (valid until the next call on this thread).
        let message = unsafe { CStr::from_ptr(cfbpe_last_error(self.0.as_ptr())) }.to_string_lossy().into_owned();
        Err(NativeError { code: rc, message })
    }

    /// What the C ABI cannot check (it takes pointers, not slices): `offsets` has n + 1 entries starting at 0, stays inside
    /// `bytes`, and `vocab_ids` names one vocabulary per prompt.
    fn check_inputs(bytes_len: usize, offsets: &[u64], vocab_ids: Option<&[u8]>) -> Result<u32, NativeError> {
        let bad = |m: &str| NativeError { code: CFBPE_EINVAL, message: m.to_owned() };
        let n = offsets.len().checked_sub(1).ok_or_else(|| bad("offsets needs n + 1 entries"))?;
        if offsets[0] != 0 || offsets[n] > bytes_len as u64 {
            return Err(bad("offsets[0] must be 0 and offsets[n] must not exceed bytes.len()"));
        }
        if vocab_ids.is_some_and(|v| v.len() < n) {
            return Err(bad("vocab_ids needs one entry per prompt"));
        }
        u32::try_from(n).map_err(|_| bad("too many prompts"))
    }

    pub fn vocab_load(&self, vocab_id: u32, ranks_file: &[u8], format: u32, pattern_id: u32, max_ranks: u32) -> Result<(), NativeError> {
        // SAFETY: the slice is valid for the call and is not retained.
        self.check(unsafe { cfbpe_vocab_load(self.0.as_ptr(), vocab_id, ranks_file.as_ptr(), ranks_file.len(), format, pattern_id, max_ranks) })
    }

    pub fn vocab_info(&self, vocab_id: u32) -> Result<cfbpe_vocab_info, NativeError> {
        let mut out = cfbpe_vocab_info::default();
        // SAFETY: out is a valid destination.
        self.check(unsafe { cfbpe_vocab_get_info(self.0.as_ptr(), vocab_id, &mut out) })?;
        Ok(out)
    }

    /// Token ids of every prompt of a packed batch (tiktoken `encode_ordinary` semantics).
    pub fn encode_batch(&self, bytes: &[u8], offsets: &[u64], vocab_ids: Option<&[u8]>) -> Result<Encoded, NativeError> {
        let n = Self::check_inputs(bytes.len(), offsets, vocab_ids)?;
        let total = offsets[n as usize] as usize;
        let mut out = Encoded { ids: vec![0; total.max(1)], offsets: vec![0; n as usize + 1], counts: vec![0; (n as usize).max(1)] };
        // SAFETY: all buffers are valid for the sizes passed; ids never outnumber bytes, so `total` ids always suffice.
        let rc = unsafe {
            cfbpe_encode_batch(self.0.as_ptr(), n, bytes.as_ptr(), offsets.as_ptr(), vocab_ids.map_or(std::ptr::null(), <[u8]>::as_ptr),
                               out.ids.as_mut_ptr(), out.ids.len() as u64, out.offsets.as_mut_ptr(), out.counts.as_mut_ptr())
        };
        self.check(rc)?;
        out.ids.truncate(out.offsets[n as usize] as usize);
        out.counts.truncate(n as usize);
        Ok(out)
    }

    /// `usage::count_tokens`: only the per-prompt counts leave the device.
    pub fn count_batch(&self, bytes: &[u8], offsets: &[u64], vocab_ids: Option<&[u8]>) -> Result<Vec<u32>, NativeError> {
        let n = Self::check_inputs(bytes.len(), offsets, vocab_ids)?;
        let mut counts = vec![0u32; (n as usize).max(1)];
        // SAFETY: as above.
        let rc = unsafe {
            cfbpe_count_batch(self.0.as_ptr(), n, bytes.as_ptr(), offsets.as_ptr(), vocab_ids.map_or(std::ptr::null(), <[u8]>::as_ptr), counts.as_mut_ptr())
        };
        self.check(rc)?;
        counts.truncate(n as usize);
        Ok(counts)
    }

    /// Every prompt cut to `min(count, budgets[i], max_tokens)` tokens, its first ones (`CFBPE_KEEP_HEAD`) or its last ones
    /// (`CFBPE_KEEP_TAIL`); `want_ids == false`: kept counts and cuts only, no id leaves the device.
    #[allow(clippy::too_many_arguments)]
    pub fn encode_truncated(&self, bytes: &[u8], offsets: &[u64], vocab_ids: Option<&[u8]>, max_tokens: u32, keep: u32, pad_id: u32,
                            budgets: Option<&[u32]>, want_ids: bool) -> Result<Truncated, NativeError> {
        let n = Self::check_inputs(bytes.len(), offsets, vocab_ids)?;
        if budgets.is_some_and(|b| b.len() != n as usize) {
            return Err(NativeError { code: CFBPE_EINVAL, message: "budgets needs one entry per prompt".to_owned() });
        }
        let m = (n as usize).max(1);
        let mut out = Truncated {
            rows: if want_ids { vec![0; n as usize * max_tokens as usize] } else { Vec::new() },
            kept: vec![0; m],
            counts: vec![0; m],
            cut: vec![0; m],
        };
        // SAFETY: all buffers are valid for the sizes passed (rows: n x max_tokens); the library checks max_tokens, keep and the
        // row budget of the context before it writes anything.
        let rc = unsafe {
            cfbpe_encode_truncated(self.0.as_ptr(), n, bytes.as_ptr(), offsets.as_ptr(), vocab_ids.map_or(std::ptr::null(), <[u8]>::as_ptr),
                                   max_tokens, keep, pad_id, budgets.map_or(std::ptr::null(), <[u32]>::as_ptr),
                                   if want_ids { out.rows.as_mut_ptr() } else { std::ptr::null_mut() }, out.kept.as_mut_ptr(),
                                   out.counts.as_mut_ptr(), out.cut.as_mut_ptr())
        };
        self.check(rc)?;
        out.kept.truncate(n as usize);
        out.counts.truncate(n as usize);
        out.cut.truncate(n as usize);
        Ok(out)
    }

    /// ids -> bytes (tiktoken `decode_bytes`); grows the output once when the library reports `CFBPE_ENOSPC`.
    pub fn decode_batch(&self, ids: &[u32], id_offsets: &[u64], vocab_ids: Option<&[u8]>) -> Result<(Vec<u8>, Vec<u64>), NativeError> {
        let n = Self::check_inputs(ids.len(), id_offsets, vocab_ids)?;
        let mut out_off = vec![0u64; n as usize + 1];
        let mut out = vec![0u8; ids.len() * 8 + 64];
        for _ in 0..2 {
            // SAFETY: as above.
            let rc = unsafe {
                cfbpe_decode_batch(self.0.as_ptr(), n, ids.as_ptr(), id_offsets.as_ptr(), vocab_ids.map_or(std::ptr::null(), <[u8]>::as_ptr),
                                   out.as_mut_ptr(), out.len() as u64, out_off.as_mut_ptr())
            };
            if rc == CFBPE_ENOSPC {
                out.resize(out_off[n as usize] as usize, 0);
                continue;
            }
            self.check(rc)?;
            out.truncate(out_off[n as usize] as usize);
            return Ok((out, out_off));
        }
        Err(NativeError { code: CFBPE_ENOSPC, message: "decode output kept growing".to_owned() })
    }

    /// The packed device tables of a vocabulary (what one rank broadcasts to the others at init).
    pub fn vocab_export(&self, vocab_id: u32) -> Result<Vec<u8>, NativeError> {
        let mut size = 0u64;
        // SAFETY: a NULL buffer asks for the size only.
        self.check(unsafe { cfbpe_vocab_export(self.0.as_ptr(), vocab_id, std::ptr::null_mut(), 0, &mut size) })?;
        let mut buf = vec![0u8; size as usize];
        // SAFETY: buf holds `size` bytes.
        self.check(unsafe { cfbpe_vocab_export(self.0.as_ptr(), vocab_id, buf.as_mut_ptr(), size, &mut size) })?;
        Ok(buf)
    }

    pub fn vocab_import(&self, vocab_id: u32, blob: &[u8]) -> Result<(), NativeError> {
        // SAFETY: the slice is valid for the call; the library validates the blob before installing it.
        self.check(unsafe { cfbpe_vocab_import(self.0.as_ptr(), vocab_id, blob.as_ptr(), blob.len() as u64) })
    }
}
