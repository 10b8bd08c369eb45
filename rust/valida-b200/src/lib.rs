//! Safe wrapper over `valida-b200-sys`.
//!
//! * [`Context`] — one per device: `StarkConfigImpl::new(pcs, challenger)` of the reference (`machine/src/config.rs:33-49`)
//!   becomes `Context::new(device)` + [`Context::set_challenger`] with the Poseidon round constants the caller drew
//!   (`basic/src/bin/valida.rs:360-365`).
//! * [`Context::prove_bytes`] — the body of `Machine::prove` (`derive/src/lib.rs:275-446`) from the 14 main and 2
//!   preprocessed traces to the CBOR image of `MachineProof` (`ciborium::into_writer`, `valida.rs:425-426`).
//! * [`Context::verify_bytes`] — `Machine::verify` (`derive/src/lib.rs:492-650`) on the same bytes.
//! * [`LocalGroup`] — ONE proof split across several GPUs, a worker thread per GPU inside this process.
//! * `--features valida`: [`glue::prove`] / [`glue::verify`] with the reference's own types.
//!
//! NOT COMPILED in the container this repository is developed in (no Rust toolchain there); the C caller
//! `tests/c/c_abi_smoke.c` exercises the same ABI and is built and run by the test suite.

use std::ffi::{c_void, CStr};
use std::fmt;
use std::ptr;

pub use valida_b200_sys as sys;
use sys::{vgpu_ctx, vgpu_matrix};

/// An error reported by the library (status code + `vgpu_last_error` text).  The reference's prover panics on failure
/// (`derive/src/lib.rs:319,364,396`); callers that want that behaviour `unwrap()`.
#[derive(Debug, Clone)]
pub struct Error {
    pub code: i32,
    pub message: String,
}

impl fmt::Display for Error {
    fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result {
        write!(f, "valida_b200 error {}: {}", self.code, self.message)
    }
}
impl std::error::Error for Error {}

pub type Result<T> = std::result::Result<T, Error>;

/// Word representation of the BabyBear elements that cross the boundary.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum Repr {
    /// `0 <= x < p`
    Canonical,
    /// `x * 2^32 mod p` — the `value` field of `p3_baby_bear::BabyBear`, so `RowMajorMatrix<BabyBear>.values` crosses zero-copy.
    MontyR32,
}

impl Repr {
    fn raw(self) -> i32 {
        match self {
            Repr::Canonical => sys::VGPU_REPR_CANONICAL,
            Repr::MontyR32 => sys::VGPU_REPR_MONTY_R32,
        }
    }
}

/// A borrowed row-major matrix of field words (`RowMajorMatrix<Val>`).
#[derive(Clone, Copy)]
pub struct MatrixView<'a> {
    pub values: &'a [u32],
    pub width: usize,
}

impl<'a> MatrixView<'a> {
    pub fn new(values: &'a [u32], width: usize) -> Self {
        assert!(width > 0 && values.len() % width == 0, "values.len() must be a multiple of the width");
        Self { values, width }
    }
    pub fn height(&self) -> usize {
        self.values.len() / self.width
    }
    fn raw(&self) -> vgpu_matrix {
        vgpu_matrix { data: self.values.as_ptr(), height: self.height() as u64, width: self.width as u64 }
    }
}

/// Outcome of [`Context::verify_bytes`]: `Machine::verify` returns `Result<(), ()>`; the code says which check failed.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum Verdict {
    Accept,
    /// `VGPU_REJECT_*` of `include/valida_b200.h`; `-100 - chip` is the reference's `OodEvaluationMismatch` of that chip.
    Reject(i32),
}

/// One context per device and stream.  Not `Sync`: a context is single-threaded (a thread per GPU uses a context each).
pub struct Context {
    raw: *mut vgpu_ctx,
}

// A context may move to the worker thread that drives its GPU.
unsafe impl Send for Context {}

impl Context {
    /// `device`: CUDA ordinal.  The library owns its stream; fails when no CUDA device is present (there is no CPU fallback).
    pub fn new(device: i32) -> Result<Self> {
        let mut raw: *mut vgpu_ctx = ptr::null_mut();
        let code = unsafe { sys::vgpu_ctx_create(device, ptr::null_mut(), &mut raw) };
        if raw.is_null() {
            return Err(Error { code, message: "vgpu_ctx_create returned no context".into() });
        }
        let ctx = Context { raw };
        if code != 0 {
            return Err(ctx.error(code));      // dropping `ctx` destroys the half-made context
        }
        Ok(ctx)
    }

    pub fn as_ptr(&self) -> *mut vgpu_ctx {
        self.raw
    }

    fn error(&self, code: i32) -> Error {
        let message = unsafe {
            let p = sys::vgpu_last_error(self.raw);
            if p.is_null() { String::new() } else { CStr::from_ptr(p).to_string_lossy().into_owned() }
        };
        Error { code, message }
    }

    fn check(&self, code: i32) -> Result<()> {
        if code == 0 { Ok(()) } else { Err(self.error(code)) }
    }

    /// The Poseidon instance of the `DuplexChallenger`: 480 round constants (canonical words, `perm16.constants()` order) and
    /// the 16 x 16 MDS matrix row-major, or `None` for `CosetMds<_, 16>::default()`.
    pub fn set_challenger(&mut self, round_constants: &[u32; 480], mds: Option<&[u32; 256]>) -> Result<()> {
        let mds_ptr = mds.map_or(ptr::null(), |m| m.as_ptr());
        self.check(unsafe { sys::vgpu_set_challenger(self.raw, round_constants.as_ptr(), mds_ptr) })
    }

    /// Page-locks a caller buffer in place so that the uploads of [`Context::prove_bytes`] overlap its commits.
    pub fn host_register(&mut self, words: &[u32]) -> Result<()> {
        self.check(unsafe { sys::vgpu_host_register(self.raw, words.as_ptr() as *const c_void, (words.len() * 4) as u64) })
    }
    pub fn host_unregister(&mut self, words: &[u32]) -> Result<()> {
        self.check(unsafe { sys::vgpu_host_unregister(self.raw, words.as_ptr() as *const c_void) })
    }

    /// `Machine::prove`: `main` are the 14 chip traces in BasicMachine order (`basic/src/lib.rs:151-166`), `prep` the
    /// preprocessed traces (program: 7 columns, range: 1 column).  Returns the CBOR image of `MachineProof`.
    pub fn prove_bytes(&mut self, main: &[MatrixView<'_>; sys::VGPU_NUM_CHIPS], prep: &[MatrixView<'_>; 2], repr: Repr) -> Result<Vec<u8>> {
        let main_raw: Vec<vgpu_matrix> = main.iter().map(MatrixView::raw).collect();
        let prep_raw: Vec<vgpu_matrix> = prep.iter().map(MatrixView::raw).collect();
        let (mut bytes, mut len) = (ptr::null_mut::<u8>(), 0u64);
        let code = unsafe { sys::vgpu_prove(self.raw, main_raw.as_ptr(), prep_raw.as_ptr(), repr.raw(), &mut bytes, &mut len) };
        self.check(code)?;
        let proof = unsafe { std::slice::from_raw_parts(bytes, len as usize) }.to_vec();
        unsafe { sys::vgpu_free_bytes(bytes) };
        Ok(proof)
    }

    /// `Machine::verify` on CBOR proof bytes (this library's or the reference's).
    pub fn verify_bytes(&mut self, proof: &[u8], prep: &[MatrixView<'_>; 2], repr: Repr) -> Result<Verdict> {
        let prep_raw: Vec<vgpu_matrix> = prep.iter().map(MatrixView::raw).collect();
        let mut verdict = -1i32;
        let code = unsafe { sys::vgpu_verify(self.raw, proof.as_ptr(), proof.len() as u64, prep_raw.as_ptr(), repr.raw(), &mut verdict) };
        self.check(code)?;
        Ok(if verdict == sys::VGPU_ACCEPT { Verdict::Accept } else { Verdict::Reject(verdict) })
    }

    /// `Machine::verify` for many proofs in one call, checked on the device: proof `i` against the preprocessed traces
    /// `preps[program_of[i]]`.  One verdict per proof, each exactly what `verify_bytes` returns for that proof alone.
    pub fn verify_batch_bytes(&mut self, proofs: &[&[u8]], preps: &[[MatrixView<'_>; 2]], program_of: &[u32], repr: Repr) -> Result<Vec<Verdict>> {
        assert_eq!(proofs.len(), program_of.len(), "one program index per proof");
        let prep_raw: Vec<vgpu_matrix> = preps.iter().flat_map(|p| p.iter().map(MatrixView::raw)).collect();
        let ptrs: Vec<*const u8> = proofs.iter().map(|p| p.as_ptr()).collect();
        let lens: Vec<u64> = proofs.iter().map(|p| p.len() as u64).collect();
        let mut verdicts = vec![-1i32; proofs.len()];
        let code = unsafe {
            sys::vgpu_verify_batch(self.raw, ptrs.as_ptr(), lens.as_ptr(), proofs.len() as u32, prep_raw.as_ptr(), preps.len() as u32,
                                   program_of.as_ptr(), repr.raw(), verdicts.as_mut_ptr())
        };
        self.check(code)?;
        Ok(verdicts.into_iter().map(|v| if v == sys::VGPU_ACCEPT { Verdict::Accept } else { Verdict::Reject(v) }).collect())
    }

    /// Kernels launched by this context so far.
    pub fn launch_count(&self) -> u64 {
        unsafe { sys::vgpu_ctx_launch_count(self.raw) }
    }
}

impl Drop for Context {
    fn drop(&mut self) {
        unsafe { sys::vgpu_ctx_destroy(self.raw) }
    }
}

/// ONE proof split across the GPUs of a box: a context per device, a worker thread per context.  Every rank makes the same
/// call with the same traces and copies only its rows of the tall ones; the proof bytes are identical on all ranks and
/// identical to the single-GPU proof.  The number of ranks must be a power of two (<= 16).
pub struct LocalGroup {
    ranks: Vec<Context>,
}

impl LocalGroup {
    /// `contexts[i]` becomes rank `i`; `set_challenger` must already have been called on each.
    pub fn new(contexts: Vec<Context>) -> Result<Self> {
        assert!(!contexts.is_empty());
        let raws: Vec<*mut vgpu_ctx> = contexts.iter().map(Context::as_ptr).collect();
        let code = unsafe { sys::vgpu_comm_init_local(raws.as_ptr(), raws.len() as i32) };
        contexts[0].check(code)?;
        Ok(LocalGroup { ranks: contexts })
    }

    pub fn len(&self) -> usize {
        self.ranks.len()
    }
    pub fn is_empty(&self) -> bool {
        self.ranks.is_empty()
    }

    /// One proof on all ranks; returns rank 0's bytes after checking that every rank produced the same ones.
    pub fn prove_bytes(&mut self, main: &[MatrixView<'_>; sys::VGPU_NUM_CHIPS], prep: &[MatrixView<'_>; 2], repr: Repr) -> Result<Vec<u8>> {
        let proofs: Vec<Result<Vec<u8>>> = std::thread::scope(|s| {
            let handles: Vec<_> = self.ranks.iter_mut().map(|ctx| s.spawn(move || ctx.prove_bytes(main, prep, repr))).collect();
            handles.into_iter().map(|h| h.join().expect("a rank's worker thread panicked")).collect()
        });
        let mut out: Option<Vec<u8>> = None;
        for p in proofs {
            let p = p?;
            match &out {
                None => out = Some(p),
                Some(first) => assert!(*first == p, "ranks disagree on the proof bytes"),
            }
        }
        Ok(out.unwrap())
    }
}

/// The reference's own types on top of the byte-level calls (`--features valida`).
#[cfg(feature = "valida")]
pub mod glue {
    use super::*;
    use p3_baby_bear::BabyBear;
    use p3_matrix::dense::RowMajorMatrix;
    use p3_matrix::Matrix;
    use valida_machine::{MachineProof, StarkConfig};

    /// `BabyBear` is `#[repr(transparent)]` over its Montgomery `u32` in the pinned fork, so the values slice is viewed in place.
    fn view(m: &RowMajorMatrix<BabyBear>) -> MatrixView<'_> {
        let words = unsafe { std::slice::from_raw_parts(m.values.as_ptr() as *const u32, m.values.len()) };
        MatrixView::new(words, m.width())
    }

    /// Replacement for the body of `Machine::prove` after witness generation (`derive/src/lib.rs:321-446`): the caller keeps
    /// steps 1-7 (`chips.par_iter().map(|c| c.generate_trace(self))`, `preprocessed_trace()`) and hands the traces over.
    pub fn prove<SC>(ctx: &mut Context, main_traces: &[RowMajorMatrix<BabyBear>; 14], preprocessed_traces: &[RowMajorMatrix<BabyBear>; 2]) -> MachineProof<SC>
    where
        SC: StarkConfig<Val = BabyBear>,
        MachineProof<SC>: serde::de::DeserializeOwned,
    {
        let main: Vec<MatrixView<'_>> = main_traces.iter().map(view).collect();
        let prep: Vec<MatrixView<'_>> = preprocessed_traces.iter().map(view).collect();
        let main: [MatrixView<'_>; 14] = main.try_into().ok().unwrap();
        let prep: [MatrixView<'_>; 2] = prep.try_into().ok().unwrap();
        let bytes = ctx.prove_bytes(&main, &prep, Repr::MontyR32).expect("vgpu_prove");   // the reference panics on failure too
        ciborium::from_reader(bytes.as_slice()).expect("proof decoding")
    }

    /// `Machine::verify` (`machine/src/machine.rs:26-31`): `Result<(), ()>` like the reference.
    pub fn verify<SC>(ctx: &mut Context, proof: &MachineProof<SC>, preprocessed_traces: &[RowMajorMatrix<BabyBear>; 2]) -> core::result::Result<(), ()>
    where
        SC: StarkConfig<Val = BabyBear>,
        MachineProof<SC>: serde::Serialize,
    {
        let mut bytes = Vec::new();
        ciborium::into_writer(proof, &mut bytes).map_err(|_| ())?;
        let prep: Vec<MatrixView<'_>> = preprocessed_traces.iter().map(view).collect();
        let prep: [MatrixView<'_>; 2] = prep.try_into().ok().unwrap();
        match ctx.verify_bytes(&bytes, &prep, Repr::MontyR32) {
            Ok(Verdict::Accept) => Ok(()),
            _ => Err(()),
        }
    }
}
