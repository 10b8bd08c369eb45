//! Raw bindings of `include/valida_b200.h` — one declaration per exported symbol, in the header's order.
//!
//! Written by hand (no bindgen in the build) and kept in step with the header by
//! `tests/test_rust_bindings.py`, which parses both files and compares names, arity and every
//! parameter / return type.  NOT COMPILED in the container this repository is developed in (no Rust
//! toolchain there): `tests/c/c_abi_smoke.c` is the caller of the same ABI that is built and run.
#![no_std]
#![allow(non_camel_case_types)]

use core::ffi::{c_char, c_void};

pub const VGPU_REPR_CANONICAL: i32 = 0;
/// `p3_baby_bear::BabyBear { value }` — the Montgomery word `x * 2^32 mod p`.
pub const VGPU_REPR_MONTY_R32: i32 = 1;
/// basic/src/lib.rs:151-166: cpu, program, mem, add, sub, mul, div, shift, lt, com, bitwise, output, range, static_data
pub const VGPU_NUM_CHIPS: usize = 14;
pub const VGPU_MAX_TERMS: usize = 4;
pub const VGPU_MAX_FIELDS: usize = 14;
pub const VGPU_MAX_INTERACTIONS: usize = 5;
pub const VGPU_COMM_ID_BYTES: usize = 128;

pub const VGPU_ACCEPT: i32 = 0;
pub const VGPU_REJECT_MALFORMED: i32 = -1;
pub const VGPU_REJECT_SHAPE: i32 = -2;
pub const VGPU_REJECT_POW: i32 = -3;
pub const VGPU_REJECT_INPUT_MERKLE: i32 = -4;
pub const VGPU_REJECT_FRI_MERKLE: i32 = -5;
pub const VGPU_REJECT_FRI_FINAL: i32 = -6;
pub const VGPU_REJECT_CUMULATIVE_SUM: i32 = -7;
/// chip i's constraints at zeta: `-100 - i` (the reference's `OodEvaluationMismatch`)
pub const VGPU_REJECT_CONSTRAINTS_CHIP0: i32 = -100;

#[repr(C)] pub struct vgpu_ctx { _opaque: [u8; 0] }
#[repr(C)] pub struct vgpu_dmat { _opaque: [u8; 0] }
#[repr(C)] pub struct vgpu_prover_data { _opaque: [u8; 0] }
#[repr(C)] pub struct vgpu_traces { _opaque: [u8; 0] }
#[repr(C)] pub struct vgpu_vmlog { _opaque: [u8; 0] }

/// `RowMajorMatrix<Val>` view over caller-owned host memory.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct vgpu_matrix {
    pub data: *const u32,
    pub height: u64,
    pub width: u64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct vgpu_pair_term {
    pub is_preprocessed: u32,
    pub column: u32,
    pub weight: u32,
}

/// `p3_air::VirtualPairCol`: constant + sum_k weight_k * column_k
#[repr(C)]
#[derive(Clone, Copy)]
pub struct vgpu_pair_col {
    pub constant: u32,
    pub n_terms: u32,
    pub terms: [vgpu_pair_term; VGPU_MAX_TERMS],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct vgpu_interaction {
    pub n_fields: u32,
    pub fields: [vgpu_pair_col; VGPU_MAX_FIELDS],
    pub count: vgpu_pair_col,
    pub bus: u32,
    pub is_send: u32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct vgpu_chip_desc {
    pub chip_id: u32,
    pub width: u32,
    pub preprocessed_width: u32,
    pub n_interactions: u32,
    pub interactions: [vgpu_interaction; VGPU_MAX_INTERACTIONS],
}

extern "C" {
    // ---- context ----
    pub fn vgpu_ctx_create(device: i32, cuda_stream: *mut c_void, out: *mut *mut vgpu_ctx) -> i32;
    pub fn vgpu_ctx_destroy(ctx: *mut vgpu_ctx);
    pub fn vgpu_last_error(ctx: *const vgpu_ctx) -> *const c_char;
    pub fn vgpu_ctx_synchronize(ctx: *mut vgpu_ctx) -> i32;
    pub fn vgpu_ctx_launch_count(ctx: *const vgpu_ctx) -> u64;
    pub fn vgpu_ctx_set_kernel_timing(ctx: *mut vgpu_ctx, on: i32) -> i32;
    pub fn vgpu_ctx_kernel_stats(ctx: *mut vgpu_ctx, names: *mut *const c_char, launches: *mut u32, ms: *mut f32, bytes: *mut f64, cap: u32) -> u32;
    pub fn vgpu_set_challenger(ctx: *mut vgpu_ctx, round_constants: *const u32, mds_16x16_or_null: *const u32) -> i32;

    // ---- caller memory ----
    pub fn vgpu_host_register(ctx: *mut vgpu_ctx, p: *const c_void, bytes: u64) -> i32;
    pub fn vgpu_host_unregister(ctx: *mut vgpu_ctx, p: *const c_void) -> i32;

    // ---- device matrices ----
    pub fn vgpu_dmat_upload(ctx: *mut vgpu_ctx, host: *const vgpu_matrix, repr: i32, out: *mut *mut vgpu_dmat) -> i32;
    pub fn vgpu_dmat_upload_rows(ctx: *mut vgpu_ctx, host: *const vgpu_matrix, repr: i32, out: *mut *mut vgpu_dmat) -> i32;
    pub fn vgpu_dmat_download(ctx: *mut vgpu_ctx, m: *const vgpu_dmat, repr: i32, host_row_major_out: *mut u32) -> i32;
    pub fn vgpu_dmat_dims(m: *const vgpu_dmat, height: *mut u64, width: *mut u64) -> i32;
    pub fn vgpu_dmat_local_rows(m: *const vgpu_dmat, row0: *mut u64, rows: *mut u64) -> i32;
    pub fn vgpu_dmat_free(m: *mut vgpu_dmat);

    // ---- p3-dft ----
    pub fn vgpu_ntt_batch(ctx: *mut vgpu_ctx, m: *mut vgpu_dmat, inverse: i32) -> i32;
    pub fn vgpu_coset_lde_batch(ctx: *mut vgpu_ctx, input: *const vgpu_dmat, log_blowup: u32, shift_canonical: u32, bit_reversed: i32, out: *mut *mut vgpu_dmat) -> i32;
    pub fn vgpu_ntt_batch_host(ctx: *mut vgpu_ctx, row_major: *mut u32, height: u64, width: u64, repr: i32, inverse: i32) -> i32;

    // ---- Pcs::commit_batches / commit_shifted_batches / get_ldes ----
    pub fn vgpu_commit_batches(ctx: *mut vgpu_ctx, mats: *const *const vgpu_dmat, n: u32, coset_shifts_or_null: *const u32, digest_out: *mut u32, out: *mut *mut vgpu_prover_data) -> i32;
    pub fn vgpu_commit_batches_host(ctx: *mut vgpu_ctx, mats: *const vgpu_matrix, n: u32, repr: i32, coset_shifts_or_null: *const u32, digest_out: *mut u32, out: *mut *mut vgpu_prover_data) -> i32;
    pub fn vgpu_prover_data_lde(pd: *const vgpu_prover_data, i: u32, view: *mut *const vgpu_dmat) -> i32;
    pub fn vgpu_prover_data_free(pd: *mut vgpu_prover_data);

    // ---- chips, LogUp, quotient ----
    pub fn vgpu_basic_machine_chip(chip_id: u32) -> *const vgpu_chip_desc;
    pub fn vgpu_perm_trace(ctx: *mut vgpu_ctx, chip: *const vgpu_chip_desc, main: *const vgpu_dmat, prep_or_null: *const vgpu_dmat, challenges: *const u32, out_perm: *mut *mut vgpu_dmat, cumulative_sum_out: *mut u32) -> i32;
    pub fn vgpu_quotient(ctx: *mut vgpu_ctx, chip: *const vgpu_chip_desc, log_degree: u32, prep_lde_or_null: *const vgpu_dmat, main_lde: *const vgpu_dmat, perm_lde: *const vgpu_dmat, cumulative_sum: *const u32, perm_challenges: *const u32, alpha: *const u32, out_chunks: *mut *mut vgpu_dmat) -> i32;

    // ---- transcript ----
    pub fn vgpu_challenger_reset(ctx: *mut vgpu_ctx) -> i32;
    pub fn vgpu_challenger_observe(ctx: *mut vgpu_ctx, values: *const u32, n: u32) -> i32;
    pub fn vgpu_challenger_sample_ext(ctx: *mut vgpu_ctx, out: *mut u32) -> i32;

    // ---- pcs.open_multi_batches ----
    pub fn vgpu_open(ctx: *mut vgpu_ctx, rounds: *const *const vgpu_prover_data, n_rounds: u32, n_points: *const u32, points: *const u32, out_cbor: *mut *mut u8, out_len: *mut u64) -> i32;

    // ---- Machine::prove ----
    pub fn vgpu_prove(ctx: *mut vgpu_ctx, main: *const vgpu_matrix, prep: *const vgpu_matrix, repr: i32, proof_out: *mut *mut u8, proof_len: *mut u64) -> i32;
    pub fn vgpu_prove_device(ctx: *mut vgpu_ctx, main: *const *const vgpu_dmat, prep: *const *const vgpu_dmat, proof_out: *mut *mut u8, proof_len: *mut u64) -> i32;
    pub fn vgpu_free_bytes(p: *mut u8);
    pub fn vgpu_last_prove_phases(ctx: *const vgpu_ctx, names: *mut *const c_char, ms: *mut f32, cap: u32) -> u32;

    // ---- one proof on several GPUs ----
    pub fn vgpu_comm_unique_id(out: *mut u8) -> i32;
    pub fn vgpu_comm_init(ctx: *mut vgpu_ctx, nranks: i32, rank: i32, unique_id: *const u8) -> i32;
    pub fn vgpu_comm_init_local(ctxs: *const *mut vgpu_ctx, nranks: i32) -> i32;
    pub fn vgpu_comm_set_sharding(ctx: *mut vgpu_ctx, on: i32) -> i32;
    pub fn vgpu_comm_stats(ctx: *mut vgpu_ctx, calls: *mut u32, bytes: *mut f64, reset: i32);
    pub fn vgpu_shard_range(total: u64, nranks: i32, rank: i32, begin: *mut u64, end: *mut u64);
    pub fn vgpu_split_column_plan(nranks: i32, n: u32, heights: *const u64, widths: *const u64, begin_out: *mut u32);
    pub fn vgpu_tree_share(len: u64, nranks: i32, rank: i32, begin: *mut u64, count: *mut u64, split: *mut i32);

    // ---- Machine::verify ----
    pub fn vgpu_verify(ctx: *mut vgpu_ctx, proof: *const u8, proof_len: u64, prep: *const vgpu_matrix, repr: i32, verdict: *mut i32) -> i32;
    pub fn vgpu_verify_batch(ctx: *mut vgpu_ctx, proofs: *const *const u8, proof_lens: *const u64, n: u32, prep: *const vgpu_matrix, n_programs: u32, program_of: *const u32, repr: i32, verdicts: *mut i32) -> i32;
    pub fn vgpu_last_verify_batch_phases(ctx: *const vgpu_ctx, names: *mut *const c_char, ms: *mut f32, cap: u32) -> u32;

    // ---- witness generation (host and device) ----
    pub fn vgpu_machine_run(program_words: *const i32, n_instr: u64, initial_pc: u32, initial_fp: u32, max_cycles: u64, out: *mut *mut vgpu_traces, err: *mut c_char, err_len: u64) -> i32;
    pub fn vgpu_machine_run_static(program_words: *const i32, n_instr: u64, initial_pc: u32, initial_fp: u32, max_cycles: u64, static_addrs: *const u32, static_values: *const u32, n_static: u64, out: *mut *mut vgpu_traces, err: *mut c_char, err_len: u64) -> i32;
    pub fn vgpu_traces_main(t: *const vgpu_traces, chip: u32) -> *const vgpu_matrix;
    pub fn vgpu_traces_preprocessed(t: *const vgpu_traces, which: u32) -> *const vgpu_matrix;
    pub fn vgpu_traces_stats(t: *const vgpu_traces, clock: *mut u32, mem_ops: *mut u32, add_ops: *mut u32);
    pub fn vgpu_traces_mem_cell(t: *const vgpu_traces, addr: u32, value: *mut u32) -> i32;
    pub fn vgpu_traces_free(t: *mut vgpu_traces);
    pub fn vgpu_vm_run(program_words: *const i32, n_instr: u64, initial_pc: u32, initial_fp: u32, max_cycles: u64, static_addrs: *const u32, static_values: *const u32, n_static: u64, out: *mut *mut vgpu_vmlog, err: *mut c_char, err_len: u64) -> i32;
    pub fn vgpu_vmlog_stats(log: *const vgpu_vmlog, clock: *mut u32, mem_ops: *mut u32, add_ops: *mut u32);
    pub fn vgpu_vmlog_traces(log: *mut vgpu_vmlog, out: *mut *mut vgpu_traces, err: *mut c_char, err_len: u64) -> i32;
    pub fn vgpu_witness_device(ctx: *mut vgpu_ctx, log: *const vgpu_vmlog, main_out: *mut *mut vgpu_dmat, prep_out: *mut *mut vgpu_dmat) -> i32;
    pub fn vgpu_vmlog_free(log: *mut vgpu_vmlog);
    pub fn vgpu_fib_program(n: u32, out_words: *mut i32) -> u64;
}
