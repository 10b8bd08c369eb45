/* valida_b200 — C ABI of the B200-native STARK prover backend for Valida's Machine::prove().
 *
 * The reference (valida-xyz/valida @ 5058de85) has NO FFI boundary (SURVEY.md §0-D8): its only seam
 * is the Rust generic `StarkConfig::Pcs: UnivariatePcsWithLde<..>` (machine/src/config.rs:7-31) plus
 * the free functions `generate_permutation_trace` (machine/src/chip.rs:121) and `quotient`
 * (machine/src/quotient.rs:18) that `Machine::prove` (machine/src/machine.rs:22-24; body
 * derive/src/lib.rs:275-446) calls directly.  Each entry point below names the reference interface
 * it replaces; INTEGRATION.md shows the Rust `extern "C"` binding a maintainer would add.
 *
 * Conventions: every function returns int32_t status (0 = OK, <0 = error; text via
 * vgpu_last_error).  No exceptions/panics cross the boundary.  A context is single-threaded: one
 * context per device/stream.  BabyBear words cross as uint32_t in the representation named by a
 * `repr` argument so that a Rust caller can pass `RowMajorMatrix<BabyBear>.values` zero-copy
 * (p3-baby-bear stores Montgomery form, R = 2^32).  Host matrices are ROW-major
 * (p3_matrix::dense::RowMajorMatrix); device matrices are column-major Montgomery words.
 */
#ifndef VALIDA_B200_H
#define VALIDA_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define VGPU_REPR_CANONICAL 0 /* 0 <= x < p */
#define VGPU_REPR_MONTY_R32 1 /* x * 2^32 mod p  (p3_baby_bear::BabyBear { value }) */

#define VGPU_NUM_CHIPS 14 /* basic/src/lib.rs:151-166: cpu, program, mem, add, sub, mul, div, shift, lt, com, bitwise, output, range, static_data */

typedef struct vgpu_ctx vgpu_ctx;
typedef struct vgpu_dmat vgpu_dmat;               /* device matrix (column-major, Montgomery) */
typedef struct vgpu_prover_data vgpu_prover_data; /* <ValMmcs as Mmcs>::ProverData: LDEs + digest layers, device resident */
typedef struct vgpu_traces vgpu_traces;           /* host witness of one machine run */

/* RowMajorMatrix<Val> view (caller-owned host memory). */
typedef struct vgpu_matrix {
    const uint32_t* data;
    uint64_t height;
    uint64_t width;
} vgpu_matrix;

/* ---- context ------------------------------------------------------------------------------- */
/* `cuda_stream` may be NULL (library-owned stream) or a cudaStream_t to enqueue on (e.g. torch's). */
int32_t vgpu_ctx_create(int32_t device, void* cuda_stream, vgpu_ctx** out);
void vgpu_ctx_destroy(vgpu_ctx* ctx);
const char* vgpu_last_error(const vgpu_ctx* ctx);
int32_t vgpu_ctx_synchronize(vgpu_ctx* ctx);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
uint64_t vgpu_ctx_launch_count(const vgpu_ctx* ctx);
/* Optional per-kernel-class CUDA-event timing (event pairs on the context's stream around every launch).
 * vgpu_ctx_kernel_stats synchronises, drains the records and returns the number of classes written:
 * names[i] (static strings), launches, summed milliseconds and summed algorithmic bytes (DESIGN.md). */
int32_t vgpu_ctx_set_kernel_timing(vgpu_ctx* ctx, int32_t on);
uint32_t vgpu_ctx_kernel_stats(vgpu_ctx* ctx, const char** names, uint32_t* launches, float* ms, double* bytes, uint32_t cap);
/* Poseidon instance of the DuplexChallenger, as the Rust side builds it
 * (basic/src/bin/valida.rs:360-365,382,397): 480 round constants (canonical), 16x16 MDS matrix
 * row-major or NULL for CosetMds<_,16>::default(). */
int32_t vgpu_set_challenger(vgpu_ctx* ctx, const uint32_t round_constants[480], const uint32_t* mds_16x16_or_null);

/* ---- caller memory: page-lock the buffers that vgpu_prove / vgpu_commit_batches_host read (RowMajorMatrix<Val>.values of the traces), so
 * that their host-to-device copies run asynchronously and overlap the commits; without it the CUDA runtime stages each copy and the call
 * blocks.  Registration costs about as much as one copy of the buffer: register once per buffer that is proven from repeatedly. ------------ */
int32_t vgpu_host_register(vgpu_ctx* ctx, const void* p, uint64_t bytes);
int32_t vgpu_host_unregister(vgpu_ctx* ctx, const void* p);

/* ---- device matrices (K12 staging: H2D + row-major -> column-major + repr conversion) ---------- */
int32_t vgpu_dmat_upload(vgpu_ctx* ctx, const vgpu_matrix* host, int32_t repr, vgpu_dmat** out);
/* Split proof (multi-GPU section below): of a trace tall enough to be split a rank keeps ITS contiguous run of rows only;
 * every rank passes the same host matrix.  Shorter traces, and any trace on a lone GPU, are uploaded whole. */
int32_t vgpu_dmat_upload_rows(vgpu_ctx* ctx, const vgpu_matrix* host, int32_t repr, vgpu_dmat** out);
/* Writes the rows this rank holds at their place in the caller's height x width row-major buffer. */
int32_t vgpu_dmat_download(vgpu_ctx* ctx, const vgpu_dmat* m, int32_t repr, uint32_t* host_row_major_out);
/* Logical dimensions (of the whole matrix, also for a shard). */
int32_t vgpu_dmat_dims(const vgpu_dmat* m, uint64_t* height, uint64_t* width);
/* The rows held here; returns 0 = whole matrix, 1 = row shard, 2 = column share. */
int32_t vgpu_dmat_local_rows(const vgpu_dmat* m, uint64_t* row0, uint64_t* rows);
void vgpu_dmat_free(vgpu_dmat* m);

/* ---- p3-dft: TwoAdicSubgroupDft::dft_batch / idft_batch / coset_lde_batch ------------------------
 * (reached via pcs.commit_batches, derive/src/lib.rs:309,330,355).  In place, natural order in and out. */
int32_t vgpu_ntt_batch(vgpu_ctx* ctx, vgpu_dmat* m, int32_t inverse);
/* out = evaluations over shift*K, |K| = height << log_blowup; bit_reversed != 0 stores row r at reverse_bits(r).
 * Sizes: vgpu_ntt_batch takes every power-of-two height up to 2^27 (BabyBear's two-adicity; heights up to 2^24 run on the fast tiles the
 * prover uses, taller ones on generic tile movement).  vgpu_coset_lde_batch takes log_blowup 1..4 with natural-order output and
 * log_blowup = 1 (the FriConfig of basic/src/bin/valida.rs:385-390, what every commit uses) with bit-reversed output; anything else
 * returns an error naming the limit. */
int32_t vgpu_coset_lde_batch(vgpu_ctx* ctx, const vgpu_dmat* in, uint32_t log_blowup, uint32_t shift_canonical,
                             int32_t bit_reversed, vgpu_dmat** out);
/* Host-buffer variants (row-major, `repr` words; H2D/D2H inside): the e2e path of bench.py. */
int32_t vgpu_ntt_batch_host(vgpu_ctx* ctx, uint32_t* row_major, uint64_t height, uint64_t width, int32_t repr, int32_t inverse);

/* ---- Pcs::commit_batches / UnivariatePcsWithLde::commit_shifted_batches ---------------------------
 * (derive/src/lib.rs:309,330,355,372).  coset_shifts_or_null: per-matrix shift (canonical), NULL = 1.
 * Writes the [BabyBear;8] commitment (canonical words) and returns the prover data handle. */
int32_t vgpu_commit_batches(vgpu_ctx* ctx, const vgpu_dmat* const* mats, uint32_t n, const uint32_t* coset_shifts_or_null,
                            uint32_t digest_out[8], vgpu_prover_data** out);
int32_t vgpu_commit_batches_host(vgpu_ctx* ctx, const vgpu_matrix* mats, uint32_t n, int32_t repr, const uint32_t* coset_shifts_or_null,
                                 uint32_t digest_out[8], vgpu_prover_data** out);
/* pcs.get_ldes (derive/src/lib.rs:311,332,358): borrowed view of committed LDE i (bit-reversed rows). */
int32_t vgpu_prover_data_lde(const vgpu_prover_data* pd, uint32_t i, const vgpu_dmat** view);
void vgpu_prover_data_free(vgpu_prover_data* pd);


/* ---- chip description: Chip::all_interactions (machine/src/chip.rs:40-63) ---------------------------
 * The data-driven half of a chip: its bus interactions as affine combinations of trace columns
 * (p3_air::VirtualPairCol; machine/src/chip.rs:76-80).  The AIR half (Air::eval) is compiled into the
 * library per chip id (BasicMachine order, basic/src/lib.rs:151-166). */
#define VGPU_MAX_TERMS 4
#define VGPU_MAX_FIELDS 14
#define VGPU_MAX_INTERACTIONS 5
typedef struct vgpu_pair_col {      /* VirtualPairCol: constant + sum_k weight_k * column_k */
    uint32_t constant;              /* canonical */
    uint32_t n_terms;
    struct { uint32_t is_preprocessed, column, weight; } terms[VGPU_MAX_TERMS];
} vgpu_pair_col;
typedef struct vgpu_interaction {
    uint32_t n_fields;
    vgpu_pair_col fields[VGPU_MAX_FIELDS];
    vgpu_pair_col count;
    uint32_t bus;                   /* BusArgument::Global(bus) */
    uint32_t is_send;               /* InteractionType::{GlobalSend, GlobalReceive} */
} vgpu_interaction;
typedef struct vgpu_chip_desc {
    uint32_t chip_id;               /* selects the compiled Air::eval */
    uint32_t width, preprocessed_width;
    uint32_t n_interactions;
    vgpu_interaction interactions[VGPU_MAX_INTERACTIONS];
} vgpu_chip_desc;
/* Built-in BasicMachine chips (0..13). */
const vgpu_chip_desc* vgpu_basic_machine_chip(uint32_t chip_id);

/* ---- generate_permutation_trace (machine/src/chip.rs:121-208) ---------------------------------------
 * main (h x width), prep (h x preprocessed_width or NULL); challenges = 3 ext elements (15 canonical
 * words: local alpha base, global alpha base, beta).  Returns the flattened perm trace
 * (h x 5*(k+1), RowMajorMatrix<Challenge>::flatten_to_base) and the cumulative sum (last row, last column). */
int32_t vgpu_perm_trace(vgpu_ctx* ctx, const vgpu_chip_desc* chip, const vgpu_dmat* main, const vgpu_dmat* prep_or_null,
                        const uint32_t challenges[15], vgpu_dmat** out_perm, uint32_t cumulative_sum_out[5]);

/* ---- quotient (machine/src/quotient.rs:18-68) -------------------------------------------------------
 * LDE arguments are committed LDEs (bit-reversed rows, 2h x w) as returned by vgpu_prover_data_lde.
 * Output: the h x 10 quotient-chunk matrix (decompose_and_flatten with log_quotient_degree = 1). */
int32_t vgpu_quotient(vgpu_ctx* ctx, const vgpu_chip_desc* chip, uint32_t log_degree, const vgpu_dmat* prep_lde_or_null,
                      const vgpu_dmat* main_lde, const vgpu_dmat* perm_lde, const uint32_t cumulative_sum[5],
                      const uint32_t perm_challenges[15], const uint32_t alpha[5], vgpu_dmat** out_chunks);

/* ---- Fiat-Shamir transcript owned by the context (DuplexChallenger; config.challenger() clone) ------
 * reset() restores the initial sponge of vgpu_set_challenger; values are canonical words. */
int32_t vgpu_challenger_reset(vgpu_ctx* ctx);
int32_t vgpu_challenger_observe(vgpu_ctx* ctx, const uint32_t* values, uint32_t n);
int32_t vgpu_challenger_sample_ext(vgpu_ctx* ctx, uint32_t out[5]);

/* ---- pcs.open_multi_batches (derive/src/lib.rs:384-392) -------------------------------------------------
 * rounds[r] = prover data of one commitment; for every matrix of every round (in order) n_points[.] opening points
 * (1 or 2), each 5 canonical words in `points`.  Samples / observes on the context's challenger
 * (vgpu_challenger_*), i.e. the caller has already observed the commitments.  Output: CBOR of the Rust tuple
 * (opened_values: Vec<Vec<Vec<Vec<Challenge>>>>, proof: TwoAdicFriPcsProof) = a 2-element array; free with
 * vgpu_free_bytes. */
int32_t vgpu_open(vgpu_ctx* ctx, const vgpu_prover_data* const* rounds, uint32_t n_rounds, const uint32_t* n_points, const uint32_t* points,
                  uint8_t** out_cbor, uint64_t* out_len);

/* ---- Machine::prove (machine/src/machine.rs:22-24; body derive/src/lib.rs:275-446) -------------------
 * main: the 14 chip traces in BasicMachine order; prep: preprocessed traces (program 7 cols, range 1 col).
 * Runs steps 3-23 of the reference's prove() on the device (transcript on the host) and returns the
 * CBOR image of MachineProof (ciborium::into_writer, basic/src/bin/valida.rs:425-426) in a buffer
 * released with vgpu_free_bytes.  vgpu_set_challenger must have been called. */
int32_t vgpu_prove(vgpu_ctx* ctx, const vgpu_matrix main[VGPU_NUM_CHIPS], const vgpu_matrix prep[2], int32_t repr,
                   uint8_t** proof_out, uint64_t* proof_len);
/* Same with the traces already resident in HBM (bench.py's device-resident timing). */
int32_t vgpu_prove_device(vgpu_ctx* ctx, const vgpu_dmat* const main[VGPU_NUM_CHIPS], const vgpu_dmat* const prep[2],
                          uint8_t** proof_out, uint64_t* proof_len);
void vgpu_free_bytes(uint8_t* p);
/* Per-phase device time of the last vgpu_prove* call: names[i] (static strings) / ms[i]; returns the count. */
uint32_t vgpu_last_prove_phases(const vgpu_ctx* ctx, const char** names, float* ms, uint32_t cap);

/* ---- multi-GPU: ONE proof split across the GPUs of one box (SURVEY.md §8(e)) ------------------------------------
 * One rank per GPU, either a process per rank (vgpu_comm_init: NCCL for the small all-gathers, CUDA IPC for the peer
 * pointers; what a torchrun launch uses) or a thread per rank inside one process (vgpu_comm_init_local; what a Rust host
 * with a worker thread per GPU uses; several ranks may share a device).  After either, every rank must make the SAME
 * sequence of library calls with the same arguments, each rank from its own thread / process.
 * Data path with sharding on (the default after init): a trace tall enough (LDE height >= 4096 * nranks) is held as
 * contiguous ROW shards (vgpu_dmat_upload_rows, vgpu_prove); a commit (1) hands every column to the rank that extends it,
 * (2) extends the column shares (coset LDE) and stores each rank's contiguous run of the committed (bit-reversed) rows into
 * that rank's shard — kernels storing through peer pointers over NVLink, the ONE bulk exchange of a commit — and (3) hashes
 * leaves and builds the sub-tree of its own rows; the nranks x 32-byte sub-roots are all-gathered and the top log2(nranks)
 * layers computed by every rank.  LogUp traces, the quotient sweep (its "next" rows are one peer's shard, read over
 * NVLink), inverse denominators, reduced openings and the FRI folds / layer trees work on a rank's own rows; what crosses
 * ranks afterwards are per-rank partial sums, sub-roots and the 40 opened rows.  Shorter matrices are computed whole by
 * every rank.  Roots and proof bytes are identical on all ranks and identical to the single-GPU ones.
 * nranks must be a power of two (<= 16). */
#define VGPU_COMM_ID_BYTES 128
int32_t vgpu_comm_unique_id(uint8_t out[VGPU_COMM_ID_BYTES]);                 /* rank 0 creates, the caller distributes */
int32_t vgpu_comm_init(vgpu_ctx* ctx, int32_t nranks, int32_t rank, const uint8_t unique_id[VGPU_COMM_ID_BYTES]);
int32_t vgpu_comm_init_local(vgpu_ctx* const* ctxs, int32_t nranks);          /* ctxs[i] becomes rank i; call once, before the rank threads start */
int32_t vgpu_comm_set_sharding(vgpu_ctx* ctx, int32_t on);                    /* 0: behave as a lone GPU (independent replicas) */
/* Collectives since the last reset: [0] barriers, [1] all-gathers, [2] peer-store exchanges (calls; bytes sent to peers). */
void vgpu_comm_stats(vgpu_ctx* ctx, uint32_t calls[3], double bytes[3], int32_t reset);
void vgpu_shard_range(uint64_t total, int32_t nranks, int32_t rank, uint64_t* begin, uint64_t* end);   /* contiguous balanced split (rows of a shard) */
/* Which rank extends which columns in one commit of n tall matrices (heights[i] x widths[i]): contiguous ranges per rank, sized by
 * water-filling over the whole commit (tallest first, a column of height h weighs h).  begin_out: n rows of nranks + 1 first-column indices. */
void vgpu_split_column_plan(int32_t nranks, uint32_t n, const uint64_t* heights, const uint64_t* widths, uint32_t* begin_out);
void vgpu_tree_share(uint64_t len, int32_t nranks, int32_t rank, uint64_t* begin, uint64_t* count, int32_t* split); /* ... for tree layers */

/* ---- Machine::verify (machine/src/machine.rs:26-31; body derive/src/lib.rs:492-650) ------------------
 * Checks a CBOR MachineProof (this library's or the reference's) against the preprocessed traces: the
 * preprocessed commitment is recomputed on the device, the transcript replayed, the FRI opening proof and
 * every chip's constraints at zeta checked on the host (machine/src/verify.rs:11-107), and the cumulative
 * sums must cancel.  Returns 0 when the check RAN; *verdict then holds VGPU_ACCEPT or the first failed
 * check.  A non-zero return is an API / device error (vgpu_ctx_last_error). */
#define VGPU_ACCEPT 0
#define VGPU_REJECT_MALFORMED (-1)        /* not the CBOR shape of MachineProof, or a field element >= p */
#define VGPU_REJECT_SHAPE (-2)            /* counts / widths / degrees inconsistent with BasicMachine */
#define VGPU_REJECT_POW (-3)              /* proof-of-work witness */
#define VGPU_REJECT_INPUT_MERKLE (-4)     /* a query's opening of the main / permutation / quotient commitment */
#define VGPU_REJECT_FRI_MERKLE (-5)       /* a query's opening of a FRI commit-phase layer */
#define VGPU_REJECT_FRI_FINAL (-6)        /* folded value != final_poly */
#define VGPU_REJECT_CUMULATIVE_SUM (-7)   /* LogUp sums over all chips do not cancel (derive/src/lib.rs:640-647) */
#define VGPU_REJECT_CONSTRAINTS_CHIP0 (-100) /* chip i's constraints at zeta: -100 - i (OodEvaluationMismatch) */
int32_t vgpu_verify(vgpu_ctx* ctx, const uint8_t* proof, uint64_t proof_len, const vgpu_matrix prep[2], int32_t repr, int32_t* verdict);
/* Machine::verify for n proofs in one call, checked on the device.  Proof i is checked against the preprocessed traces
 * prep[2*program_of[i]] (program ROM) and prep[2*program_of[i]+1] (range table); n_programs pairs are given and each
 * preprocessed commitment is computed once per call.  verdicts[i] is exactly what vgpu_verify returns for proof i alone
 * (VGPU_ACCEPT or the FIRST failed check, in vgpu_verify's order).  Decoding and the transcript replay run on host threads;
 * the Merkle paths, reduced openings, FRI folds and constraints at zeta of all proofs run as a few kernels.  Proofs of
 * different programs and trace heights may be mixed.  Returns 0 when the checks ran; non-zero = API / device error
 * (vgpu_last_error).  n = 0 is valid and writes nothing. */
int32_t vgpu_verify_batch(vgpu_ctx* ctx, const uint8_t* const* proofs, const uint64_t* proof_lens, uint32_t n,
                          const vgpu_matrix* prep, uint32_t n_programs, const uint32_t* program_of, int32_t repr,
                          int32_t* verdicts);
/* Wall-clock stretches of the last vgpu_verify_batch on this context (decode, preprocessed commitments, transcripts, packing,
 * device checks); returns the number of stretches, writes at most cap. */
uint32_t vgpu_last_verify_batch_phases(const vgpu_ctx* ctx, const char** names, float* ms, uint32_t cap);

/* ---- host witness generation (Chip::generate_trace x14; machine/src/chip.rs:22) -------------------
 * program_words: n_instr x 6 int32 (opcode, a, b, c, d, e) as ProgramROM<i32> (machine/src/program.rs:165-185). */
int32_t vgpu_machine_run(const int32_t* program_words, uint64_t n_instr, uint32_t initial_pc, uint32_t initial_fp, uint64_t max_cycles,
                         vgpu_traces** out, char* err, uint64_t err_len);
/* The same with static data preloaded: StaticDataChip::write + MachineWithStaticDataChip::initialize_memory
 * (static_data/src/lib.rs:26-57; the reference's prove_static_data, basic/tests/test_static_data.rs:30-113).
 * static_values[i] is the 32-bit cell at static_addrs[i] (Word bytes big-endian, as Word<u8> -> u32). */
int32_t vgpu_machine_run_static(const int32_t* program_words, uint64_t n_instr, uint32_t initial_pc, uint32_t initial_fp, uint64_t max_cycles,
                                const uint32_t* static_addrs, const uint32_t* static_values, uint64_t n_static,
                                vgpu_traces** out, char* err, uint64_t err_len);
const vgpu_matrix* vgpu_traces_main(const vgpu_traces* t, uint32_t chip);           /* canonical words */
const vgpu_matrix* vgpu_traces_preprocessed(const vgpu_traces* t, uint32_t which);  /* 0 = program (7 cols), 1 = range (1 col) */
void vgpu_traces_stats(const vgpu_traces* t, uint32_t* clock, uint32_t* mem_ops, uint32_t* add_ops);
int32_t vgpu_traces_mem_cell(const vgpu_traces* t, uint32_t addr, uint32_t* value);
void vgpu_traces_free(vgpu_traces* t);
/* ---- witness generation on the device (SURVEY.md 8(f)1) ------------------------------------------------------------------
 * Machine::run alone (the interpreter is a serial host loop): what it leaves behind are its LOGS — one record per cycle, per
 * memory operation, per ALU operation.  vgpu_witness_device expands them into the 14 main and 2 preprocessed traces ON THE
 * GPU (cpu/src/lib.rs:79-97,163-373; memory/src/lib.rs:143-194 with the (addr, clk) sort; alu_u32 op_to_row), column-major
 * Montgomery words ready for vgpu_prove_device: no host row fill, no 2 GB upload, no transpose.  vgpu_vmlog_traces builds the
 * same traces on the host from the same logs (equal word for word; the parity tests compare the two). */
typedef struct vgpu_vmlog vgpu_vmlog;
int32_t vgpu_vm_run(const int32_t* program_words, uint64_t n_instr, uint32_t initial_pc, uint32_t initial_fp, uint64_t max_cycles,
                    const uint32_t* static_addrs, const uint32_t* static_values, uint64_t n_static, vgpu_vmlog** out, char* err, uint64_t err_len);
void vgpu_vmlog_stats(const vgpu_vmlog* log, uint32_t* clock, uint32_t* mem_ops, uint32_t* add_ops);
int32_t vgpu_vmlog_traces(vgpu_vmlog* log, vgpu_traces** out, char* err, uint64_t err_len);
int32_t vgpu_witness_device(vgpu_ctx* ctx, const vgpu_vmlog* log, vgpu_dmat* main_out[VGPU_NUM_CHIPS], vgpu_dmat* prep_out[2]);
void vgpu_vmlog_free(vgpu_vmlog* log);

/* fib_program of basic/tests/test_prover.rs:35-188 with `imm32 -8(fp)` = n; returns the instruction count (23). */
uint64_t vgpu_fib_program(uint32_t n, int32_t* out_words /* >= 23*6 */);

#ifdef __cplusplus
}
#endif
#endif /* VALIDA_B200_H */
