/*!
Drop-in replacement for the body of `src/saca.rs` of kvark/dark: same public items
(`Symbol`, `Suffix`, `Constructor::{new, capacity, compute, reuse}`), backed by the
B200-native library through `dark-bwt-sys`, plus `Constructor::bwt` for the two call
sites.  UNCOMPILED in this image (no Rust toolchain) — deliberately thin.

Errors panic, which is the reference's convention (assert!s at saca.rs:272,300,369).
*/
extern crate dark_bwt_sys as sys;

use std::ffi::CStr;
use std::{ptr, slice};

/// Symbol type
pub type Symbol = u8;
/// Suffix type = index of the original sub-string
pub type Suffix = u32;

/// Suffix Array Constructor (GPU)
pub struct Constructor {
    ctx: *mut sys::dark_bwt_ctx,
    n: usize,
    sa: Vec<Suffix>,   // host copy handed out by compute()
    out: Vec<Symbol>,  // the BWT bytes of the block compute() saw last (kept: the transform produces them anyway)
    origin: usize,
}

fn check(ctx: *const sys::dark_bwt_ctx, rc: i32, what: &str) {
    if rc != sys::DARK_BWT_OK {
        let msg = unsafe { CStr::from_ptr(sys::dark_bwt_strerror(rc)) }.to_string_lossy().into_owned();
        let detail = if ctx.is_null() { String::new() } else {
            unsafe { CStr::from_ptr(sys::dark_bwt_last_error(ctx)) }.to_string_lossy().into_owned()
        };
        panic!("{}: {} {}", what, msg, detail);
    }
}

impl Constructor {
    /// Create a new instance for a given maximum input size (on the CUDA device named by the environment variable
    /// `DARK_BWT_DEVICE`, default 0 — the reference's signature has no room for a device argument)
    pub fn new(max_n: usize) -> Constructor {
        let device = std::env::var("DARK_BWT_DEVICE").ok().and_then(|v| v.parse::<i32>().ok()).unwrap_or(0);
        Constructor::with_device(max_n, device)
    }

    /// Same, on an explicit CUDA device: one `Constructor` (one context) per GPU and host thread is how independent
    /// blocks are spread over the GPUs of a box (SURVEY.md 8e)
    pub fn with_device(max_n: usize, device: i32) -> Constructor {
        let mut ctx = ptr::null_mut();
        let rc = unsafe { sys::dark_bwt_create(max_n as u64, device, &mut ctx) };
        check(ctx, rc, "saca::Constructor::new");
        Constructor { ctx: ctx, n: max_n, sa: Vec::new(), out: Vec::new(), origin: 0 }
    }

    /// Device bytes `Constructor::new(max_n)` allocates (0 if max_n is out of range): whether a block fits a card can be
    /// checked before creating a context.  Touches no device.
    pub fn arena_bytes(max_n: usize) -> u64 {
        unsafe { sys::dark_bwt_arena_bytes(max_n as u64, 0) }
    }

    /// Return maximum block size
    pub fn capacity(&self) -> usize {
        unsafe { sys::dark_bwt_capacity(self.ctx) as usize }
    }

    /// Compute the suffix array for a given input
    pub fn compute<'a>(&'a mut self, input: &[Symbol]) -> &'a [Suffix] {
        assert_eq!(input.len(), self.n);
        self.sa.resize(input.len(), 0);
        self.out.resize(input.len(), 0);
        let mut origin = 0u64;
        let rc = unsafe { sys::dark_bwt_forward(self.ctx, input.as_ptr(), input.len() as u64,
            self.out.as_mut_ptr(), &mut origin, self.sa.as_mut_ptr(), ptr::null_mut()) };
        check(self.ctx, rc, "saca::Constructor::compute");
        self.origin = origin as usize;
        &self.sa[..]
    }

    /// BWT bytes and origin of the block `compute` was last called on (what `TransformIterator::new(input, suf)`
    /// would yield), without a second transform
    pub fn last_bwt(&self) -> (&[Symbol], usize) {
        (&self.out[..], self.origin)
    }

    /// BWT bytes and origin of a block: what `compute` + `bwt::TransformIterator` produced
    pub fn bwt(&mut self, input: &[Symbol]) -> (Vec<Symbol>, usize) {
        let mut out = vec![0u8; input.len()];
        let mut origin = 0u64;
        let rc = unsafe { sys::dark_bwt_forward(self.ctx, input.as_ptr(), input.len() as u64,
            out.as_mut_ptr(), &mut origin, ptr::null_mut(), ptr::null_mut()) };
        check(self.ctx, rc, "saca::Constructor::bwt");
        (out, origin as usize)
    }

    /// Many small blocks in one pass over the GPU (`dark_bwt_forward_many`): `(bwt, origin)` per block, each
    /// identical to `self.bwt(block)`.  The blocks share the arena: their lengths must sum to <= capacity.
    pub fn bwt_many(&mut self, blocks: &[&[Symbol]]) -> Vec<(Vec<Symbol>, usize)> {
        let mut outs: Vec<Vec<u8>> = blocks.iter().map(|b| vec![0u8; b.len()]).collect();
        let texts: Vec<*const u8> = blocks.iter().map(|b| b.as_ptr()).collect();
        let ns: Vec<u64> = blocks.iter().map(|b| b.len() as u64).collect();
        let bwts: Vec<*mut u8> = outs.iter_mut().map(|o| o.as_mut_ptr()).collect();
        let mut origins = vec![0u64; blocks.len()];
        let rc = unsafe { sys::dark_bwt_forward_many(self.ctx, texts.as_ptr(), ns.as_ptr(), bwts.as_ptr(),
            origins.as_mut_ptr(), blocks.len() as u64, ptr::null_mut()) };
        check(self.ctx, rc, "saca::Constructor::bwt_many");
        outs.into_iter().zip(origins.into_iter().map(|o| o as usize)).collect()
    }

    /// `compute` + `TransformIterator` + `bwt::dc::encode(&output, suf, &mut mtf)` (block/dc.rs:45-52) in one call: the
    /// distance coder reads the BWT while it is still in HBM.  Returns (BWT bytes, origin, init = `get_init()`); the
    /// distances land in the first n words of `reuse()`, exactly where the reference passes `suf` to `dc::encode`, so
    /// `bwt::dc::EncodeIterator::new(&output, &suf[..n], init)` continues as before.  PARITY UNPINNED for the DC part:
    /// the `compress` crate's source is not in the reference tree (see include/dark_bwt.h).
    pub fn bwt_dc(&mut self, input: &[Symbol]) -> (Vec<Symbol>, usize, [usize; 0x100]) {
        let n = input.len();
        let mut out = vec![0u8; n];
        let mut origin = 0u64;
        let mut info: sys::dark_bwt_dc_info = unsafe { std::mem::zeroed() };
        let dist = self.reuse().as_mut_ptr();
        let rc = unsafe { sys::dark_bwt_forward_dc(self.ctx, input.as_ptr(), n as u64, out.as_mut_ptr(), &mut origin, dist,
            ptr::null_mut(), ptr::null_mut(), ptr::null_mut(), ptr::null_mut(), &mut info, ptr::null_mut()) };
        check(self.ctx, rc, "saca::Constructor::bwt_dc");
        let mut init = [0usize; 0x100];
        for (d, s) in init.iter_mut().zip(info.init.iter()) { *d = *s as usize; }
        (out, origin as usize, init)
    }

    /// Temporarily provide the storage for outside needs
    pub fn reuse<'a>(&'a mut self) -> &'a mut [Suffix] {
        let (mut p, mut cnt) = (ptr::null_mut(), 0u64);
        let rc = unsafe { sys::dark_bwt_reuse(self.ctx, &mut p, &mut cnt) };
        check(self.ctx, rc, "saca::Constructor::reuse");
        unsafe { slice::from_raw_parts_mut(p, cnt as usize) }
    }
}

impl Drop for Constructor {
    fn drop(&mut self) {
        unsafe { sys::dark_bwt_destroy(self.ctx) }
    }
}
