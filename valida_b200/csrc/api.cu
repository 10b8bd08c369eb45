// C ABI entry points (include/valida_b200.h): context, device matrices, NTT/LDE, commit.
#include "ctx.h"
#include "merkle.h"
#include <algorithm>
#include <cstring>
#include <new>
#include <utility>

// ---- memory ------------------------------------------------------------------------------------
int32_t vg_alloc(vgpu_ctx* ctx, void** p, size_t bytes) {
    bytes = (bytes + 511) & ~(size_t)511;
    if (bytes == 0) bytes = 512;
    auto it = ctx->free_bufs.find(bytes);
    if (it != ctx->free_bufs.end()) {
        *p = it->second;
        ctx->free_bufs.erase(it);
        ctx->cached_bytes -= bytes;
    } else {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e != cudaSuccess && !ctx->free_bufs.empty()) {   // out of memory: drop the cache and retry once
            cudaGetLastError();
            cudaStreamSynchronize(ctx->stream);
            for (auto& kv : ctx->free_bufs) cudaFree(kv.second);
            ctx->free_bufs.clear(); ctx->cached_bytes = 0;
            e = cudaMalloc(p, bytes);
        }
        if (e != cudaSuccess) VG_FAIL(ctx, "cudaMalloc(%zu bytes) failed: %s (live %zu MB)", bytes, cudaGetErrorString(e), ctx->live_bytes >> 20);
    }
    ctx->live_bufs[*p] = bytes;
    ctx->live_bytes += bytes;
    if (ctx->live_bytes > ctx->peak_bytes) ctx->peak_bytes = ctx->live_bytes;
    return 0;
}
void vg_free(vgpu_ctx* ctx, void* p) {
    if (!p) return;
    auto it = ctx->live_bufs.find(p);
    if (it == ctx->live_bufs.end()) return;
    size_t bytes = it->second;
    ctx->live_bufs.erase(it);
    ctx->live_bytes -= bytes;
    ctx->free_bufs.emplace(bytes, p);
    ctx->cached_bytes += bytes;
}

int32_t vg_dmat_alloc(vgpu_ctx* ctx, uint64_t h, uint64_t w, vgpu_dmat** out) {
    vgpu_dmat* m = new (std::nothrow) vgpu_dmat();
    if (!m) VG_FAIL(ctx, "out of host memory");
    m->ctx = ctx; m->h = h; m->w = w; m->col_stride = h; m->owns = true;
    m->gh = h; m->gw = w;
    int32_t rc = vg_alloc(ctx, (void**)&m->d, h * w * 4);
    if (rc) { delete m; return rc; }
    *out = m;
    return 0;
}

// The local part of a gh x gw matrix: VG_FULL = all of it; VG_ROWS = this rank's run of gh / comm_size stored rows;
// VG_COLS = this rank's column share (vg_shard_range of gw).  symm: taken from the symmetric heap (peers store into it).
int32_t vg_dmat_alloc_dist(vgpu_ctx* ctx, int dist, uint64_t gh, uint64_t gw, bool symm, vgpu_dmat** out) {
    vgpu_dmat* m = new (std::nothrow) vgpu_dmat();
    if (!m) VG_FAIL(ctx, "out of host memory");
    const uint64_t G = (uint64_t)ctx->comm_size, r = (uint64_t)ctx->comm_rank;
    m->ctx = ctx; m->gh = gh; m->gw = gw; m->dist = dist; m->owns = true; m->symm = symm;
    m->h = gh; m->w = gw;
    if (dist == VG_ROWS) { m->h = gh / G; m->row0 = r * m->h; }
    else if (dist == VG_COLS) { uint64_t a, b; vg_shard_range(gw, (int)G, (int)r, &a, &b); m->col0 = a; m->w = b - a; }
    m->col_stride = m->h;
    size_t words = m->h * m->w;
    if (dist == VG_COLS) words = m->h * ((gw + G - 1) / G);       // the same size on every rank
    int32_t rc = symm ? vg_symm_alloc(ctx, (void**)&m->d, words * 4) : vg_alloc(ctx, (void**)&m->d, words * 4);
    if (rc) { delete m; return rc; }
    *out = m;
    return 0;
}

static int32_t build_pow_table(vgpu_ctx* ctx, uint32_t base_monty, uint32_t scale_monty, uint64_t max_exp, PowTable* t) {
    uint64_t hi_len = (max_exp >> VG_POW_LO_BITS) + 1;
    std::vector<uint32_t> lo(VG_POW_LO), hi(hi_len);
    uint32_t a = bb::R1;
    for (uint32_t j = 0; j < VG_POW_LO; j++) { lo[j] = a; a = bb::mul(a, base_monty); }
    uint32_t step = a;  // base^4096
    a = scale_monty;
    for (uint64_t j = 0; j < hi_len; j++) { hi[j] = a; a = bb::mul(a, step); }
    VG_TRY(vg_alloc(ctx, (void**)&t->lo, lo.size() * 4));
    VG_TRY(vg_alloc(ctx, (void**)&t->hi, hi.size() * 4));
    VG_CUDA(ctx, cudaMemcpyAsync(t->lo, lo.data(), lo.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    VG_CUDA(ctx, cudaMemcpyAsync(t->hi, hi.data(), hi.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    VG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // host vectors go out of scope
    t->hi_len = (uint32_t)hi_len;
    t->base = base_monty;
    return 0;
}

int32_t vg_get_shift_table(vgpu_ctx* ctx, uint32_t shift_canonical, uint32_t scale_canonical, uint64_t max_exp, const PowTable** out) {
    auto key = std::make_pair(shift_canonical, scale_canonical);
    auto it = ctx->shift_tables.find(key);
    if (it == ctx->shift_tables.end() || (uint64_t)it->second.hi_len * VG_POW_LO <= max_exp) {
        PowTable t;
        VG_TRY(build_pow_table(ctx, bb::to_monty(shift_canonical), bb::to_monty(scale_canonical), max_exp, &t));
        if (it != ctx->shift_tables.end()) { vg_free(ctx, it->second.lo); vg_free(ctx, it->second.hi); }
        ctx->shift_tables[key] = t;
        it = ctx->shift_tables.find(key);
    }
    *out = &it->second;
    return 0;
}

void vg_host_state_free(vgpu_ctx* ctx);

// Every entry point runs on the context's device whatever the calling thread's current device is (a thread per GPU in
// one process, or torch having switched devices).
int32_t vg_enter(vgpu_ctx* ctx) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != ctx->device) VG_CUDA(ctx, cudaSetDevice(ctx->device));
    return 0;
}

extern "C" {

int32_t vgpu_ctx_create(int32_t device, void* cuda_stream, vgpu_ctx** out) {
    if (!out) return -1;
    *out = nullptr;
    vgpu_ctx* ctx = new (std::nothrow) vgpu_ctx();
    if (!ctx) return -1;
    ctx->device = device;
    *out = ctx;   // returned even on failure so the caller can read vgpu_last_error
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { ctx->err = "no CUDA device available: valida_b200 has no CPU fallback"; return -2; }
    VG_CUDA(ctx, cudaSetDevice(device));
    if (cuda_stream) { ctx->stream = (cudaStream_t)cuda_stream; ctx->own_stream = false; }
    else { VG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)); ctx->own_stream = true; }
    cudaDeviceProp prop;
    VG_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    VG_TRY(build_pow_table(ctx, bb::two_adic_generator_monty(VG_LOG_NMAX), bb::R1, (1ull << VG_LOG_NMAX) - 1, &ctx->root_table));
    {   // three-level table (9 + 9 + 9 exponent bits)
        std::vector<uint32_t> t(3 * 512);
        uint32_t base = bb::two_adic_generator_monty(VG_LOG_NMAX);
        for (int lvl = 0; lvl < 3; lvl++) {
            uint32_t a = bb::R1;
            for (int i = 0; i < 512; i++) { t[lvl * 512 + i] = a; a = bb::mul(a, base); }
            base = a;   // base^512
        }
        VG_TRY(vg_alloc(ctx, (void**)&ctx->root3, t.size() * 4));
        VG_CUDA(ctx, cudaMemcpy(ctx->root3, t.data(), t.size() * 4, cudaMemcpyHostToDevice));
    }
    return 0;
}

void vgpu_ctx_destroy(vgpu_ctx* ctx) {
    if (!ctx) return;
    vg_host_state_free(ctx);
    vg_stager_free(ctx);
    vg_comm_free(ctx);
    if (ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        vg_free(ctx, ctx->root_table.lo); vg_free(ctx, ctx->root_table.hi);
        for (auto& kv : ctx->shift_tables) { vg_free(ctx, kv.second.lo); vg_free(ctx, kv.second.hi); }
        cudaStreamSynchronize(ctx->stream);
        for (auto& kv : ctx->free_bufs) cudaFree(kv.second);
        for (auto& kv : ctx->live_bufs) cudaFree(kv.first);
        for (auto e : ctx->event_pool) cudaEventDestroy(e);
        if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
        if (ctx->xfer_stream) { cudaStreamDestroy(ctx->xfer_stream); for (auto e : ctx->xfer_ev) if (e) cudaEventDestroy(e); }
        if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    }
    delete ctx;
}

const char* vgpu_last_error(const vgpu_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
int32_t vgpu_ctx_synchronize(vgpu_ctx* ctx) { VG_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); return 0; }
uint64_t vgpu_ctx_launch_count(const vgpu_ctx* ctx) { return ctx->launches; }

int32_t vgpu_ctx_set_kernel_timing(vgpu_ctx* ctx, int32_t on) { ctx->ktiming = on != 0; return 0; }
static const char* KCLASS_NAMES[KC_COUNT] = {"ntt_pass_kernel", "leaf_hash_kernel", "compress_layer_kernel", "fri_leaf_hash_kernel", "transpose (rm<->cm)",
                                             "perm trace kernels", "quotient_kernel", "inverse denominators", "bary_kernel", "reduced_opening_kernel", "fri_fold_kernel", "peer-store exchange", "all-gathers + barriers (incl. waiting for the slowest rank)", "other",
                                             "verify_merkle_kernel", "verify_open_kernel", "verify_fold_kernel", "verify_constraints_kernel"};
uint32_t vgpu_ctx_kernel_stats(vgpu_ctx* ctx, const char** names, uint32_t* launches, float* ms, double* bytes, uint32_t cap) {
    cudaStreamSynchronize(ctx->stream);
    uint32_t n[KC_COUNT] = {0}; float t[KC_COUNT] = {0}; double b[KC_COUNT] = {0};
    for (auto& k : ctx->ktimers) {
        float e = 0;
        if (cudaEventElapsedTime(&e, k.a, k.b) == cudaSuccess) { n[k.cls]++; t[k.cls] += e; b[k.cls] += k.bytes; }
        else cudaGetLastError();   // do not leave the error for the caller's next CUDA call
        ctx->event_pool.push_back(k.a); ctx->event_pool.push_back(k.b);
    }
    ctx->ktimers.clear();
    uint32_t out = 0;
    for (int c = 0; c < KC_COUNT && out < cap; c++) if (n[c]) { names[out] = KCLASS_NAMES[c]; launches[out] = n[c]; ms[out] = t[c]; bytes[out] = b[c]; out++; }
    return out;
}

// ---- caller memory ---------------------------------------------------------------------------------
// vgpu_prove copies the traces out of the caller's buffers on a copy stream while the commits of earlier matrices run.  From
// PAGEABLE memory (a Rust Vec, a numpy array) the CUDA runtime stages every copy through its own bounce buffer and the copy call
// blocks the host; page-locking the buffers once lets the same call overlap for real.
int32_t vgpu_host_register(vgpu_ctx* ctx, const void* p, uint64_t bytes) {
    VG_TRY(vg_enter(ctx));
    cudaError_t e = cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterDefault);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return 0; }
    if (e != cudaSuccess) VG_FAIL(ctx, "cudaHostRegister(%llu bytes) failed: %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return 0;
}
int32_t vgpu_host_unregister(vgpu_ctx* ctx, const void* p) {
    VG_TRY(vg_enter(ctx));
    cudaError_t e = cudaHostUnregister(const_cast<void*>(p));
    if (e != cudaSuccess) { cudaGetLastError(); VG_FAIL(ctx, "cudaHostUnregister failed: %s", cudaGetErrorString(e)); }
    return 0;
}

// ---- device matrices -----------------------------------------------------------------------------
int32_t vgpu_dmat_upload(vgpu_ctx* ctx, const vgpu_matrix* host, int32_t repr, vgpu_dmat** out) {
    if (!host || !out) VG_FAIL(ctx, "dmat_upload: null argument");
    VG_TRY(vg_enter(ctx));
    vgpu_dmat* m = nullptr;
    VG_TRY(vg_dmat_alloc(ctx, host->height, host->width, &m));
    int32_t rc = vg_upload_rowmajor(ctx, host->data, host->height, host->width, repr, m);
    if (rc) { vgpu_dmat_free(m); return rc; }
    *out = m;
    return 0;
}
// Split proof: a rank keeps only ITS run of rows of a trace tall enough to be split (every rank passes the same host
// matrix, or at least its own rows of it); shorter traces are uploaded whole.  The handle reports the logical dimensions.
int32_t vgpu_dmat_upload_rows(vgpu_ctx* ctx, const vgpu_matrix* host, int32_t repr, vgpu_dmat** out) {
    if (!host || !out) VG_FAIL(ctx, "dmat_upload_rows: null argument");
    if (!vg_split_rows(ctx, 2 * host->height)) return vgpu_dmat_upload(ctx, host, repr, out);
    VG_TRY(vg_enter(ctx));
    vgpu_dmat* m = nullptr;
    VG_TRY(vg_dmat_alloc_dist(ctx, VG_ROWS, host->height, host->width, false, &m));
    int32_t rc = vg_upload_rowmajor(ctx, host->data + m->row0 * host->width, m->h, m->w, repr, m);
    if (rc) { vgpu_dmat_free(m); return rc; }
    *out = m;
    return 0;
}
// Writes the rows this rank holds (all of them unless the matrix is a row shard) at their place in the caller's
// gh x gw row-major buffer.
int32_t vgpu_dmat_download(vgpu_ctx* ctx, const vgpu_dmat* m, int32_t repr, uint32_t* host_row_major_out) {
    VG_TRY(vg_enter(ctx));
    VG_TRY(vg_dmat_materialize(ctx, m));
    if (m->dist == VG_COLS) VG_FAIL(ctx, "dmat_download: column shares are internal to a commit");
    if (m->dist == VG_ROWS && m->bitrev_rows) VG_FAIL(ctx, "dmat_download: a bit-reversed row shard has no contiguous natural-order image");
    VG_TRY(vg_download_rowmajor(ctx, m, repr, host_row_major_out + m->row0 * m->gw));
    if (m->bitrev_rows && m->h > 1) {   // present the logical (natural) row order to the caller
        int lg = 0; while ((1ull << lg) < m->h) lg++;
        std::vector<uint32_t> tmp(m->w);
        for (uint64_t i = 0; i < m->h; i++) {
            uint64_t j = bb::reverse_bits((uint32_t)i, lg);
            if (i < j) {
                uint32_t* a = host_row_major_out + i * m->w; uint32_t* b = host_row_major_out + j * m->w;
                std::memcpy(tmp.data(), a, m->w * 4); std::memcpy(a, b, m->w * 4); std::memcpy(b, tmp.data(), m->w * 4);
            }
        }
    }
    return 0;
}
int32_t vgpu_dmat_dims(const vgpu_dmat* m, uint64_t* height, uint64_t* width) { *height = m->gh; *width = m->gw; return 0; }
int32_t vgpu_dmat_local_rows(const vgpu_dmat* m, uint64_t* row0, uint64_t* rows) { *row0 = m->row0; *rows = m->h; return m->dist; }
void vgpu_dmat_free(vgpu_dmat* m) {
    if (!m) return;
    if (m->pend_stage) {   // an upload that was never consumed: let the copy finish, then release
        if (m->pend_job) vg_stager_finish(m->ctx);       // joins the staging threads: every chunk is enqueued
        if (m->pend_ev) cudaEventSynchronize(m->pend_ev);
        else if (m->ctx->copy_stream) cudaStreamSynchronize(m->ctx->copy_stream);
        vg_free(m->ctx, m->pend_stage);
        if (m->pend_ev) m->ctx->event_pool.push_back(m->pend_ev);
    }
    if (m->owns) { if (m->symm) vg_symm_free(m->ctx, m->d); else vg_free(m->ctx, m->d); }
    delete m;
}

// ---- NTT / LDE -------------------------------------------------------------------------------------
int32_t vgpu_ntt_batch(vgpu_ctx* ctx, vgpu_dmat* m, int32_t inverse) {
    VG_TRY(vg_enter(ctx));
    if (m->dist != VG_FULL) VG_FAIL(ctx, "ntt_batch: the matrix is a shard of a split proof");
    int log_n = 0;
    while ((1ull << log_n) < m->h) log_n++;
    if ((1ull << log_n) != m->h) VG_FAIL(ctx, "ntt_batch: height %llu is not a power of two", (unsigned long long)m->h);
    if (log_n > VG_LOG_NMAX) VG_FAIL(ctx, "ntt_batch: height exceeds two-adicity");
    if (m->bitrev_rows) VG_FAIL(ctx, "ntt_batch: matrix rows are stored bit-reversed");
    VG_TRY(vg_dmat_materialize(ctx, m));
    uint32_t* tmp = nullptr;
    VG_TRY(vg_alloc(ctx, (void**)&tmp, m->h * m->w * 4));
    int32_t rc = vg_ntt_nat2nat(ctx, m->d, m->col_stride, m->d, m->col_stride, log_n, m->w, inverse != 0, nullptr, tmp, m->h);
    vg_free(ctx, tmp);
    return rc;
}

int32_t vgpu_coset_lde_batch(vgpu_ctx* ctx, const vgpu_dmat* in, uint32_t log_blowup, uint32_t shift_canonical, int32_t bit_reversed, vgpu_dmat** out) {
    if (log_blowup < 1 || log_blowup > 4) VG_FAIL(ctx, "coset_lde: log_blowup must be 1..4");
    VG_TRY(vg_enter(ctx));
    if (in->dist != VG_FULL) VG_FAIL(ctx, "coset_lde: the matrix is a shard of a split proof");
    VG_TRY(vg_dmat_materialize(ctx, in));
    vgpu_dmat* o = nullptr;
    VG_TRY(vg_dmat_alloc(ctx, in->h << log_blowup, in->w, &o));
    int32_t rc = vg_coset_lde(ctx, in->d, in->col_stride, in->h, in->w, shift_canonical, o->d, o->col_stride, bit_reversed != 0, in->bitrev_rows, log_blowup);
    if (rc) { vgpu_dmat_free(o); return rc; }
    *out = o;
    return 0;
}

int32_t vgpu_ntt_batch_host(vgpu_ctx* ctx, uint32_t* row_major, uint64_t height, uint64_t width, int32_t repr, int32_t inverse) {
    vgpu_matrix hm{row_major, height, width};
    vgpu_dmat* m = nullptr;
    VG_TRY(vgpu_dmat_upload(ctx, &hm, repr, &m));
    int32_t rc = vgpu_ntt_batch(ctx, m, inverse);
    if (rc == 0) rc = vgpu_dmat_download(ctx, m, repr, row_major);
    vgpu_dmat_free(m);
    return rc;
}

// ---- commit ------------------------------------------------------------------------------------------
// TwoAdicFriPcs::commit_shifted_batches per matrix: shift = generator / coset_shift_i; LDE; bit-reversed rows.
static uint32_t lde_shift_of(const uint32_t* coset_shifts_or_null, uint32_t i) {
    const uint32_t cs = coset_shifts_or_null ? coset_shifts_or_null[i] : 1;
    return bb::from_monty(bb::mul(bb::to_monty(bb::GEN_CANON), bb::inv(bb::to_monty(cs))));
}

// Which rank extends which columns of the tall matrices of one commit: contiguous column ranges per rank, sized by water-filling
// over the whole commit — tallest matrix first, every column goes to the rank with the least work so far (a column of height h
// weighs h) — so that a rank that had to take two of the ten columns of a 2^24-row matrix takes fewer columns of the others.
// (An even split of every matrix on its own leaves the first ranks with up to 60 % more LDE work than the mean at 8 ranks.)
struct ColPlan { uint32_t begin[17]; uint32_t widest; };
static std::vector<ColPlan> plan_columns(const int G, const std::vector<std::pair<uint64_t, uint64_t>>& dims /* (height, width) of the tall matrices */) {
    std::vector<size_t> order(dims.size());
    for (size_t k = 0; k < dims.size(); k++) order[k] = k;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return dims[a].first > dims[b].first; });
    std::vector<uint64_t> load(G, 0);
    std::vector<ColPlan> plan(dims.size());
    for (size_t k : order) {
        uint32_t count[16] = {0};
        for (uint64_t c = 0; c < dims[k].second; c++) {
            int best = 0;
            for (int r = 1; r < G; r++) if (load[r] < load[best]) best = r;
            count[best]++; load[best] += dims[k].first;
        }
        ColPlan& p = plan[k];
        p.begin[0] = 0; p.widest = 0;
        for (int r = 0; r < G; r++) { p.begin[r + 1] = p.begin[r] + count[r]; p.widest = std::max(p.widest, count[r]); }
    }
    return plan;
}

// Symmetric-heap bytes one commit of matrices with these (height, width) puts there when they arrive as row shards (prover.cc sizes
// the heap for a whole proof with it).
extern "C++" size_t vg_commit_symm_need(const vgpu_ctx* ctx, const std::vector<std::pair<uint64_t, uint64_t>>& dims_all) {
    std::vector<std::pair<uint64_t, uint64_t>> dims;
    for (auto& d : dims_all) if (vg_split_rows(ctx, 2 * d.first)) dims.push_back(d);
    const std::vector<ColPlan> plan = plan_columns(ctx->comm_size, dims);
    size_t need = 0;
    for (size_t k = 0; k < dims.size(); k++)
        need += vg_symm_round((2 * dims[k].first / (uint64_t)ctx->comm_size) * dims[k].second * 4) + vg_symm_round(dims[k].first * plan[k].widest * 4);
    return need;
}

// The column plan of a commit as data (tests; a host program that wants to know which rank extends what): matrices i = 0..n-1 of
// heights[i] x widths[i], all tall enough to be split; begin_out[i * (nranks + 1) + r] = first column of rank r, ... + nranks] = width.
void vgpu_split_column_plan(int32_t nranks, uint32_t n, const uint64_t* heights, const uint64_t* widths, uint32_t* begin_out) {
    std::vector<std::pair<uint64_t, uint64_t>> dims;
    for (uint32_t i = 0; i < n; i++) dims.push_back({heights[i], widths[i]});
    const std::vector<ColPlan> plan = plan_columns(nranks, dims);
    for (uint32_t i = 0; i < n; i++) for (int r = 0; r <= nranks; r++) begin_out[(size_t)i * (nranks + 1) + r] = plan[i].begin[r];
}

// Split proof: the tall matrices of a commit.  (1) a matrix that arrives as row shards is handed to the ranks that extend
// its columns; (2) every rank extends its column share and stores, through peer pointers, each rank's run of the committed
// rows into that rank's shard.  After the closing barrier pd->ldes[i] holds rows [rank * H/G, (rank+1) * H/G) of all columns.
static int32_t extend_split(vgpu_ctx* ctx, vgpu_prover_data* pd, const vgpu_dmat* const* mats, const std::vector<size_t>& tall, const uint32_t* coset_shifts_or_null) {
    const uint64_t G = (uint64_t)ctx->comm_size;
    std::vector<std::pair<uint64_t, uint64_t>> dims;
    for (size_t i : tall) dims.push_back({mats[i]->gh, mats[i]->gw});
    const std::vector<ColPlan> plan = plan_columns(ctx->comm_size, dims);
    size_t need = 0;
    for (size_t k = 0; k < tall.size(); k++) {
        const vgpu_dmat* m = mats[tall[k]];
        need += vg_symm_round((2 * m->gh / G) * m->gw * 4);
        if (m->dist == VG_ROWS) need += vg_symm_round(m->gh * plan[k].widest * 4);
    }
    VG_TRY(vg_symm_reserve(ctx, need));
    std::vector<uint32_t*> cols(tall.size(), nullptr);      // column buffers of the matrices that arrive as row shards (symmetric heap)
    struct Guard { vgpu_ctx* c; std::vector<uint32_t*>& v; ~Guard() { for (auto* p : v) vg_symm_free(c, p); } } guard{ctx, cols};
    bool moved = false;
    for (size_t k = 0; k < tall.size(); k++) {
        const vgpu_dmat* m = mats[tall[k]];
        VG_TRY(vg_dmat_materialize(ctx, m));
        if (m->dist == VG_COLS) VG_FAIL(ctx, "commit: column shares are internal to a commit");
        if (m->dist != VG_ROWS) continue;
        VG_TRY(vg_symm_alloc(ctx, (void**)&cols[k], m->gh * plan[k].widest * 4));
        VG_TRY(vg_exchange_rows_to_cols(ctx, m, cols[k], plan[k].begin));
        moved = true;
    }
    if (moved) VG_TRY(vg_comm_barrier(ctx));
    // (2) extend the column share of matrix k on the context's stream while the exchange of matrix k-1 runs on a second
    // stream: the LDE kernels are issue bound, the exchange is NVLink bound.  Two extension buffers alternate; a buffer is
    // rewritten only after its exchange has finished.  (With per-kernel timing on everything stays on one stream.)
    const bool overlap = !ctx->ktiming;
    if (overlap && !ctx->xfer_stream) {
        VG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->xfer_stream, cudaStreamNonBlocking));
        for (auto& e : ctx->xfer_ev) VG_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    size_t ext_words = 0;
    for (size_t k = 0; k < tall.size(); k++)
        ext_words = std::max<size_t>(ext_words, 2 * mats[tall[k]]->gh * (plan[k].begin[ctx->comm_rank + 1] - plan[k].begin[ctx->comm_rank]));
    uint32_t* ext[2] = {nullptr, nullptr};
    struct ExtGuard { vgpu_ctx* c; uint32_t** e; ~ExtGuard() { vg_free(c, e[0]); vg_free(c, e[1]); } } eg{ctx, ext};
    if (ext_words) { VG_TRY(vg_alloc(ctx, (void**)&ext[0], ext_words * 4)); if (overlap) VG_TRY(vg_alloc(ctx, (void**)&ext[1], ext_words * 4)); }
    bool used[2] = {false, false};
    for (size_t k = 0; k < tall.size(); k++) {
        const size_t i = tall[k];
        const vgpu_dmat* m = mats[i];
        const uint64_t h = m->gh, H = 2 * h;
        const uint64_t c0 = plan[k].begin[ctx->comm_rank], c1 = plan[k].begin[ctx->comm_rank + 1];
        VG_TRY(vg_dmat_alloc_dist(ctx, VG_ROWS, H, m->gw, true, &pd->ldes[i]));
        pd->ldes[i]->bitrev_rows = false;        // committed order IS the stored order of an LDE (rows at reverse_bits)
        if (c1 <= c0) continue;
        const uint32_t* src; uint64_t scs;
        if (m->dist == VG_ROWS) { src = cols[k]; scs = h; }
        else { src = m->d + c0 * m->col_stride; scs = m->col_stride; }
        const int b = overlap ? (int)(k & 1) : 0;
        if (overlap && used[b]) VG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->xfer_ev[b], 0));
        VG_TRY(vg_coset_lde(ctx, src, scs, h, c1 - c0, lde_shift_of(coset_shifts_or_null, (uint32_t)i), ext[b], H, true, m->bitrev_rows));
        if (overlap) {
            VG_CUDA(ctx, cudaEventRecord(ctx->xfer_ev[2], ctx->stream));
            VG_CUDA(ctx, cudaStreamWaitEvent(ctx->xfer_stream, ctx->xfer_ev[2], 0));
            VG_TRY(vg_exchange_cols_to_rows(ctx, ext[b], H, c0, c1, pd->ldes[i], ctx->xfer_stream));
            VG_CUDA(ctx, cudaEventRecord(ctx->xfer_ev[b], ctx->xfer_stream));
            used[b] = true;
        } else {
            VG_TRY(vg_exchange_cols_to_rows(ctx, ext[0], H, c0, c1, pd->ldes[i]));
        }
    }
    if (overlap) for (int b = 0; b < 2; b++) if (used[b]) VG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->xfer_ev[b], 0));
    return vg_comm_barrier(ctx);   // also orders the release of the column buffers (guard) behind every peer's stores
}

int32_t vgpu_commit_batches(vgpu_ctx* ctx, const vgpu_dmat* const* mats, uint32_t n, const uint32_t* coset_shifts_or_null,
                            uint32_t digest_out[8], vgpu_prover_data** out) {
    VG_TRY(vg_enter(ctx));
    vgpu_prover_data* pd = new (std::nothrow) vgpu_prover_data();
    if (!pd) VG_FAIL(ctx, "out of host memory");
    pd->ctx = ctx;
    pd->ldes.assign(n, nullptr);
    std::vector<uint64_t> heights(n);
    std::vector<size_t> tall;
    for (uint32_t i = 0; i < n; i++) {
        if (!mats[i]) { vgpu_prover_data_free(pd); VG_FAIL(ctx, "commit: matrix %u is null", i); }
        heights[i] = mats[i]->gh * 2;
        if (vg_split_rows(ctx, heights[i])) tall.push_back(i);
        else if (mats[i]->dist != VG_FULL) { vgpu_prover_data_free(pd); VG_FAIL(ctx, "commit: matrix %u is a shard but too short to be split", i); }
    }
    int32_t rc = tall.empty() ? 0 : extend_split(ctx, pd, mats, tall, coset_shifts_or_null);
    // The other matrices one height group at a time, when the tree reaches that height; a matrix whose upload is still in
    // flight is waited for here, not earlier.  (Split proof: short matrices are extended, whole, by every rank.)
    auto extend_group = [&](const std::vector<size_t>& group) -> int32_t {
        for (size_t i : group) {
            if (pd->ldes[i]) continue;
            VG_TRY(vg_dmat_materialize(ctx, mats[i]));
            VG_TRY(vgpu_coset_lde_batch(ctx, mats[i], 1, lde_shift_of(coset_shifts_or_null, (uint32_t)i), 1, &pd->ldes[i]));
        }
        return 0;
    };
    if (rc == 0) rc = vg_merkle_build(ctx, pd, heights, extend_group);
    if (rc) { vgpu_prover_data_free(pd); return rc; }
    if (digest_out) std::memcpy(digest_out, pd->root, 32);
    *out = pd;
    return 0;
}

int32_t vgpu_commit_batches_host(vgpu_ctx* ctx, const vgpu_matrix* mats, uint32_t n, int32_t repr, const uint32_t* coset_shifts_or_null,
                                 uint32_t digest_out[8], vgpu_prover_data** out) {
    std::vector<vgpu_dmat*> dm(n, nullptr);
    int32_t rc = 0;
    for (uint32_t i = 0; i < n && rc == 0; i++) rc = vgpu_dmat_upload_rows(ctx, &mats[i], repr, &dm[i]);   // a split proof uploads each rank's rows only
    if (rc == 0) rc = vgpu_commit_batches(ctx, dm.data(), n, coset_shifts_or_null, digest_out, out);
    for (auto* m : dm) vgpu_dmat_free(m);
    return rc;
}

int32_t vgpu_prover_data_lde(const vgpu_prover_data* pd, uint32_t i, const vgpu_dmat** view) {
    if (i >= pd->ldes.size()) return -1;
    *view = pd->ldes[i];
    return 0;
}
void vgpu_prover_data_free(vgpu_prover_data* pd) {
    if (!pd) return;
    for (auto* m : pd->ldes) vgpu_dmat_free(m);
    vg_tree_free(pd->ctx, &pd->tree);
    delete pd;
}

}  // extern "C"
