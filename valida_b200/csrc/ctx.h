// Internal context / device-matrix definitions shared by the kernels' host wrappers.
#pragma once
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>
#include <map>
#include <type_traits>
#include <cuda_runtime.h>
#include "../../include/valida_b200.h"
#include "bb.cuh"

constexpr int VG_LOG_NMAX = 27;                    // BabyBear two-adicity: largest transform/LDE size
constexpr int VG_POW_LO_BITS = 12;                 // two-level power tables: base^e = lo[e & 4095] * hi[e >> 12]
constexpr uint32_t VG_POW_LO = 1u << VG_POW_LO_BITS;

struct PowTable {            // device tables of Montgomery words
    uint32_t* lo = nullptr;  // base^j, j < 4096
    uint32_t* hi = nullptr;  // scale * base^(4096 j), j < hi_len
    uint32_t hi_len = 0;
    uint32_t base = 0;       // the base itself (Montgomery), without the scale
};

// kernel classes for the optional per-launch CUDA-event timing (bench.py's roofline line)
enum KClass { KC_NTT = 0, KC_LEAF_HASH, KC_COMPRESS, KC_FRI_LEAF, KC_TRANSPOSE, KC_PERM, KC_QUOTIENT, KC_INVDEN, KC_BARY, KC_REDUCED_OPENING, KC_FRI_FOLD, KC_EXCHANGE, KC_COLLECTIVE, KC_OTHER,
             KC_VERIFY_MERKLE, KC_VERIFY_OPEN, KC_VERIFY_FOLD, KC_VERIFY_CONSTRAINTS, KC_COUNT };
struct KTimer { cudaEvent_t a, b; int cls; double bytes; };

struct vgpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    uint64_t launches = 0;
    int sm_count = 148;
    PowTable root_table;                                        // base = two_adic_generator(27)
    uint32_t* root3 = nullptr;                                   // 3 x 512 words: w^(i), w^(512 i), w^(2^18 i) — a 6 KB, L1-resident form of the same table
    std::map<std::pair<uint32_t, uint32_t>, PowTable> shift_tables;  // (shift, scale) canonical -> table
    std::vector<void*> owned;                                   // freed at destroy
    // Poseidon challenger instance (host side; the transcript is sequential and tiny)
    uint32_t poseidon_rc[480];
    uint32_t poseidon_mds[256];
    bool challenger_set = false;
    bool poseidon_has_mds = false;
    void* challenger = nullptr;                                  // vgh::Challenger* (host/challenger.h)
    void* poseidon = nullptr;                                    // vgh::Poseidon16*
    uint32_t* d_poseidon = nullptr;                              // device copy of the round constants + MDS (pow.cu), dropped when they change
    std::vector<std::pair<const char*, float>> phases;          // last prove: per-phase milliseconds
    struct PhaseMark { const char* name; cudaEvent_t a, b; };
    std::vector<PhaseMark> phase_marks;                         // event pairs of the last prove (read by vgpu_last_prove_phases)
    std::vector<std::pair<const char*, float>> host_phases;     // host-side stretches of the last prove (wall clock)
    bool in_host_prove = false;
    std::vector<std::pair<const char*, float>> verify_phases;   // host / device stretches of the last vgpu_verify_batch (wall clock)
    // size-keyed cache of device buffers: a proof repeats the same allocation sizes every step, so after the
    // first step no driver allocator call is made (single stream => reuse in enqueue order is safe)
    std::multimap<size_t, void*> free_bufs;
    std::map<void*, size_t> live_bufs;
    size_t cached_bytes = 0, live_bytes = 0, peak_bytes = 0;
    // multi-GPU (host/comm.cc): one rank per GPU.  Two transports with one interface: NCCL + CUDA IPC between processes
    // (torchrun ranks), or a thread per GPU inside one process (vgpu_comm_init_local: host barrier + direct peer pointers).
    void* nccl = nullptr;                                        // ncclComm_t
    void* local_group = nullptr;                                 // VgLocalGroup* (in-process ranks)
    int comm_rank = 0, comm_size = 1;
    bool sharding = false;                                       // ONE proof split across the ranks (row shards after one exchange)
    // symmetric heap: one allocation per rank, identical allocation sequence on every rank => identical offsets, so a
    // peer's copy of a buffer is peer_base[d] + (p - symm_base).  Kernels store / load through those pointers over NVLink.
    uint8_t* symm_base = nullptr; size_t symm_bytes = 0;
    std::vector<uint8_t*> peer_base;                             // [comm_size]; peer_base[comm_rank] == symm_base
    std::map<size_t, size_t> symm_free;                          // offset -> length of the free runs
    std::map<void*, size_t> symm_live;
    size_t symm_live_bytes = 0, symm_peak_bytes = 0;
    uint32_t* comm_scratch = nullptr;                            // small device buffer for barriers / handle exchange
    cudaEvent_t bar_ev[2] = {nullptr, nullptr}; uint32_t bar_slot = 0;   // in-process stream-ordered barrier
    struct CommStat { uint32_t calls = 0; double bytes = 0; };
    CommStat stat_barrier, stat_allgather, stat_exchange;        // per-proof collective counters (bench.py)
    cudaStream_t copy_stream = nullptr;                         // H2D copies of a pipelined vgpu_prove (staging.cu)
    void* stager = nullptr;                                     // VgStager*: host threads staging pageable traces through pinned chunks
    cudaStream_t xfer_stream = nullptr;                         // split proof: peer-store exchange of matrix i behind the LDE of matrix i+1
    cudaEvent_t xfer_ev[3] = {nullptr, nullptr, nullptr};       // [0], [1]: exchange out of buffer 0 / 1 done; [2]: LDE done
    bool ntt_attrs_set = false, bary_attrs_set = false;          // cudaFuncSetAttribute is per device: tracked per context, not per process
    bool ktiming = false;
    std::vector<KTimer> ktimers;
    std::vector<cudaEvent_t> event_pool;
};

// Distribution of a matrix over the ranks of a split proof.  FULL: every rank holds all of it (also the only kind on a lone
// GPU).  ROWS: this rank holds the contiguous run [row0, row0 + h) of the STORED row order (natural rows for traces,
// bit-reversed rows for committed LDEs / quotient chunks) of a gh x gw matrix.  COLS: columns [col0, col0 + w), all rows.
enum VgDist { VG_FULL = 0, VG_ROWS = 1, VG_COLS = 2 };
struct vgpu_dmat {
    vgpu_ctx* ctx = nullptr;
    uint32_t* d = nullptr;       // column-major: LOCAL element (r, c) at d[c * col_stride + r], Montgomery form
    uint64_t h = 0, w = 0, col_stride = 0;     // local extent
    uint64_t gh = 0, gw = 0, row0 = 0, col0 = 0;   // logical extent and the position of the local part in it
    int dist = VG_FULL;
    bool symm = false;           // d lives in the symmetric heap
    bool owns = true;
    bool bitrev_rows = false;    // row r of the logical matrix is stored at reverse_bits(r) (quotient-chunk output order)
    // pipelined upload: the row-major image is (being) copied into pend_stage on the copy stream; the transpose into
    // `d` runs on the context's stream at first use (vg_dmat_materialize)
    uint32_t* pend_stage = nullptr;
    cudaEvent_t pend_ev = nullptr;
    int32_t pend_repr = 0;
    void* pend_job = nullptr;    // StageJob* when the source is pageable memory copied by the context's staging threads
};

#define VG_FAIL(ctx, ...) do { char _b[512]; snprintf(_b, sizeof _b, __VA_ARGS__); (ctx)->err = _b; return -1; } while (0)
#define VG_CUDA(ctx, expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { VG_FAIL(ctx, "%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); } } while (0)
#define VG_TRY(expr) do { int32_t _r = (expr); if (_r != 0) return _r; } while (0)
#define VG_LAUNCH_CHECK(ctx) do { (ctx)->launches++; cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { VG_FAIL(ctx, "kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); } } while (0)

// RAII scope: when ctx->ktiming is on, brackets the launches inside it with a CUDA event pair on ctx->stream.
struct KScope {
    vgpu_ctx* ctx; bool on; size_t idx = 0;      // scopes nest (a collective inside a sweep): each closes ITS pair
    KScope(vgpu_ctx* c, int cls, double bytes) : ctx(c), on(c->ktiming) {
        if (!on) return;
        KTimer t; t.cls = cls; t.bytes = bytes;
        for (cudaEvent_t* e : {&t.a, &t.b}) {
            if (!c->event_pool.empty()) { *e = c->event_pool.back(); c->event_pool.pop_back(); }
            else cudaEventCreate(e);
        }
        cudaEventRecord(t.a, c->stream);
        c->ktimers.push_back(t);
        idx = c->ktimers.size() - 1;
    }
    ~KScope() { if (on) cudaEventRecord(ctx->ktimers[idx].b, ctx->stream); }
};

int32_t vg_enter(vgpu_ctx* ctx);                          // make ctx->device current on the calling thread
int32_t vg_alloc(vgpu_ctx* ctx, void** p, size_t bytes);
void vg_free(vgpu_ctx* ctx, void* p);
int32_t vg_dmat_alloc(vgpu_ctx* ctx, uint64_t h, uint64_t w, vgpu_dmat** out);
int32_t vg_get_shift_table(vgpu_ctx* ctx, uint32_t shift_canonical, uint32_t scale_canonical, uint64_t max_exp, const PowTable** out);

// host/comm.cc — every rank calls these in the same order with the same sizes
inline bool vg_sharded(const vgpu_ctx* ctx) { return ctx->sharding && ctx->comm_size > 1; }
// A matrix / vector of `n` stored rows is cut into comm_size contiguous row shards when every shard keeps >= 4096 rows;
// shorter ones are replicated (every rank computes and holds all of them).
inline bool vg_split_rows(const vgpu_ctx* ctx, uint64_t n) { return vg_sharded(ctx) && n >= (uint64_t)ctx->comm_size * 4096; }
void vg_shard_range(uint64_t total, int nranks, int rank, uint64_t* begin, uint64_t* end);   // contiguous, balanced
// buf holds comm_size consecutive blocks of `words_per_rank` u32; this rank's block is already filled
int32_t vg_comm_allgather_inplace(vgpu_ctx* ctx, uint32_t* buf, uint64_t words_per_rank);
// stream-ordered barrier: everything enqueued before it on ANY rank's stream completes before anything enqueued after it
// on any rank's stream starts (peer stores become visible, peer buffers may be reused)
int32_t vg_comm_barrier(vgpu_ctx* ctx);
int32_t vg_comm_group_begin(vgpu_ctx* ctx);   // NCCL group around several all-gathers (no-ops for in-process ranks)
int32_t vg_comm_group_end(vgpu_ctx* ctx);
void vg_comm_free(vgpu_ctx* ctx);
// symmetric heap (collective: same calls, same sizes, same order on every rank)
int32_t vg_symm_reserve(vgpu_ctx* ctx, size_t extra_bytes);     // make room for `extra_bytes` more (grows the heap when nothing is live)
int32_t vg_symm_alloc(vgpu_ctx* ctx, void** p, size_t bytes);
void vg_symm_free(vgpu_ctx* ctx, void* p);
inline size_t vg_symm_round(size_t bytes) { return (bytes + 1023) & ~(size_t)1023; }
template <class T> inline T* vg_peer_ptr(const vgpu_ctx* ctx, T* mine, int peer) {
    return reinterpret_cast<T*>(ctx->peer_base[peer] + (reinterpret_cast<uint8_t*>(const_cast<typename std::remove_const<T>::type*>(mine)) - ctx->symm_base));
}
// exchange.cu — the two transposing exchanges of a split commit, as kernels storing through peer pointers
int32_t vg_exchange_rows_to_cols(vgpu_ctx* ctx, const vgpu_dmat* rows, uint32_t* cols_symm, const uint32_t* col_begin);
int32_t vg_exchange_cols_to_rows(vgpu_ctx* ctx, const uint32_t* lde_cols, uint64_t H, uint64_t c0, uint64_t c1, vgpu_dmat* shard, cudaStream_t on = nullptr);
size_t vg_commit_symm_need(const vgpu_ctx* ctx, const std::vector<std::pair<uint64_t, uint64_t>>& dims_all);
int32_t vg_dmat_alloc_dist(vgpu_ctx* ctx, int dist, uint64_t gh, uint64_t gw, bool symm, vgpu_dmat** out);

// ntt.cu
int32_t vg_ntt_nat2nat(vgpu_ctx* ctx, const uint32_t* src, uint64_t src_cs, uint32_t* dst, uint64_t dst_cs, int log_n, uint64_t w,
                       bool inverse, const PowTable* coset_or_null, uint32_t* tmp, uint64_t tmp_cs);
int32_t vg_coset_lde(vgpu_ctx* ctx, const uint32_t* src, uint64_t src_cs, uint64_t h, uint64_t w, uint32_t shift_canonical,
                     uint32_t* dst, uint64_t dst_cs, bool bit_reversed, bool src_bitrev = false, uint32_t log_blowup = 1);
// staging.cu
int32_t vg_upload_begin(vgpu_ctx* ctx, const uint32_t* host, uint64_t h, uint64_t w, int32_t repr, vgpu_dmat* dst);   // async copy only
int32_t vg_stager_start(vgpu_ctx* ctx);                       // after the last vg_upload_begin of a proof
int32_t vg_stager_finish(vgpu_ctx* ctx);                      // before the caller's buffers may change again
void vg_stager_free(vgpu_ctx* ctx);
int32_t vg_dmat_materialize(vgpu_ctx* ctx, const vgpu_dmat* m);                                                       // no-op unless an upload is pending
int32_t vg_upload_rowmajor(vgpu_ctx* ctx, const uint32_t* host, uint64_t h, uint64_t w, int32_t repr, vgpu_dmat* dst);
int32_t vg_download_rowmajor(vgpu_ctx* ctx, const vgpu_dmat* src, int32_t repr, uint32_t* host);
