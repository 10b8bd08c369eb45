// Device side of vgpu_verify_batch: the query-phase checks of many proofs at once (sm_100a).  The host (host/verifier.cc) has
// decoded every proof, replayed its transcript, checked every count, width and path length, and packed the batch (verify_batch.h).
//   verify_merkle_kernel       one thread per opening: (proof, query, input round) and, after the folds, (proof, query, FRI step).
//                              SerializingHasher32<Keccak256> over the opened rows of each height group, the path walked with the
//                              64-byte compression, shorter groups injected where the level reaches them (FieldMerkleTreeMmcs::verify_batch).
//   verify_open_kernel         one thread per (proof, query, matrix, point): alpha^off (p(x) - p(z)) / (x - z) summed over the columns,
//                              one ext5 inversion each; a zero denominator is a SHAPE failure at its key.
//   verify_fold_kernel         one thread per (proof, query): the p3-fri fold chain; each step's 10-word leaf row goes to global memory
//                              for the FRI paths; ro[LOG_BLOWUP] == 0 and the final value against final_poly.
//   verify_constraints_kernel  one thread per (proof, chip): verify_chip.cuh, the text vgpu_verify runs on the host.
// A failing check lowers its proof's slot with atomicMin on (key << 32 | code): the verdict is the FIRST failure in vgpu_verify's
// order however the threads are scheduled.  No field value is accumulated with atomics: ro[lh] is a fixed-order sum of partials.
#include "ctx.h"
#include "keccak.cuh"
#include "verify_batch.h"
#include "verify_chip.cuh"

namespace {

using bb::E5;
using vb::MerkleJob;

constexpr int LOG_BLOWUP = 1;

__device__ __forceinline__ void fail(unsigned long long* best, uint32_t proof, uint32_t key, int32_t code) {
    atomicMin(best + proof, (unsigned long long)vb::slot(key, code));
}

__device__ __forceinline__ void load8(const uint32_t* __restrict__ p, uint32_t o[8]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}

__device__ __forceinline__ void hash_group(const uint32_t* __restrict__ w, uint32_t nwords, uint32_t out[8]) {
    uint32_t d[8];
    kk::keccak256_words(nwords, [&](uint32_t i) { return w[i]; }, d);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = kk::wrap_mod_p(d[i]);
}

// vb::fri_row words are written by verify_fold_kernel earlier on the same stream: plain loads, not the read-only path
__global__ void __launch_bounds__(128) verify_merkle_kernel(const MerkleJob* __restrict__ jobs, uint32_t n, const uint32_t* words,
                                                            const uint32_t* __restrict__ digests, const vb::Group* __restrict__ groups,
                                                            unsigned long long* best) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const MerkleJob& j = jobs[t];
    const vb::Group* g = groups + j.groups;
    const uint32_t* w = words + j.words;
    uint32_t node[8];
    hash_group(w, g[0].nwords, node);
    w += g[0].nwords;
    uint32_t gi = 1, level = g[0].level, index = j.index;
    for (uint32_t s = 0; s < j.path_len; s++) {
        uint32_t sib[8], l[8], r[8];
        load8(digests + (j.path + s) * 8, sib);
        const bool odd = index & 1;
#pragma unroll
        for (int i = 0; i < 8; i++) { l[i] = odd ? sib[i] : node[i]; r[i] = odd ? node[i] : sib[i]; }
        kk::compress_pair(l, r, node);
        index >>= 1; level--;
        if (gi < j.n_groups && g[gi].level == level) {
            uint32_t h[8], c[8];
            hash_group(w, g[gi].nwords, h);
            w += g[gi].nwords; gi++;
#pragma unroll
            for (int i = 0; i < 8; i++) c[i] = node[i];
            kk::compress_pair(c, h, node);
        }
    }
    bool same = gi == j.n_groups;
#pragma unroll
    for (int i = 0; i < 8; i++) same = same && node[i] == j.commit[i];
    if (!same) fail(best, j.proof, j.key, (int32_t)j.code);
}

__global__ void __launch_bounds__(128) verify_open_kernel(const vb::QueryJob* __restrict__ queries, uint32_t nq, const vb::OpenItem* __restrict__ items,
                                                          const vb::ProofHdr* __restrict__ hdrs, const uint32_t* __restrict__ words,
                                                          const E5* __restrict__ exts, E5* __restrict__ partials, unsigned long long* best) {
    const uint32_t qi = blockIdx.x;
    if (qi >= nq) return;
    const vb::QueryJob& job = queries[qi];
    const vb::ProofHdr& hdr = hdrs[job.proof];
    for (uint32_t t = threadIdx.x; t < job.n_items; t += blockDim.x) {
        const vb::OpenItem& it = items[job.items + t];
        const uint32_t rev = bb::reverse_bits(job.index >> (hdr.log_max_height - it.lh), (int)it.lh);
        const uint32_t x = bb::mul(bb::to_monty(bb::GEN_CANON), bb::pow(bb::two_adic_generator_monty((int)it.lh), rev));
        const E5 den = bb::e5_add_base(bb::e5_neg(it.z), x);   // x - z
        E5 part = bb::e5_zero();
        if (bb::e5_is_zero(den)) {
            fail(best, job.proof, vb::key_q(job.q, it.key), VGPU_REJECT_SHAPE);
        } else {
            // sum_c alpha^c (p_c(x) - p_c(z)), Horner from the last column
            const uint32_t* row = words + job.words + it.row_off;
            const E5* at_z = exts + it.vals;
            E5 acc = bb::e5_zero();
            for (uint32_t c = it.width; c-- > 0;)
                acc = bb::e5_add(bb::e5_mul(acc, hdr.fri_alpha), bb::e5_add_base(bb::e5_neg(at_z[c]), bb::to_monty(row[c])));
            part = bb::e5_mul(bb::e5_mul(acc, it.alpha_pow), bb::e5_inv(den));
        }
        partials[job.partials + t] = part;
    }
}

__device__ __forceinline__ E5 reduced_opening(const vb::QueryJob& job, const uint32_t* __restrict__ bk, const E5* __restrict__ partials, uint32_t lh) {
    E5 s = bb::e5_zero();
    for (uint32_t k = bk[lh]; k < bk[lh + 1]; k++) s = bb::e5_add(s, partials[job.partials + bk[33 + k]]);
    return s;
}

__global__ void __launch_bounds__(128) verify_fold_kernel(const vb::QueryJob* __restrict__ queries, uint32_t nq, const vb::ProofHdr* __restrict__ hdrs,
                                                          const uint32_t* __restrict__ buckets, const E5* __restrict__ exts, const E5* __restrict__ partials,
                                                          uint32_t* __restrict__ words, unsigned long long* best) {
    const uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    const vb::QueryJob& job = queries[qi];
    if (!job.fold_steps && !job.check_final) return;
    const vb::ProofHdr& hdr = hdrs[job.proof];
    const uint32_t* bk = buckets + hdr.buckets;
    const int L = (int)hdr.log_max_height;
    uint32_t index = job.index;
    E5 folded = bb::e5_zero();
    uint32_t x = bb::pow(bb::two_adic_generator_monty(L), bb::reverse_bits(index, L));
    const uint32_t minus_one = bb::two_adic_generator_monty(1);
    for (uint32_t s = 0; s < job.fold_steps; s++) {
        const uint32_t lfh = (uint32_t)L - 1 - s;
        folded = bb::e5_add(folded, reduced_opening(job, bk, partials, lfh + 1));
        const bool sib_hi = ((index ^ 1) & 1) != 0;   // the sibling is evals[1]
        const E5 sib = exts[job.sibs + s];
        const E5 e0 = sib_hi ? folded : sib, e1 = sib_hi ? sib : folded;
        uint32_t* row = words + job.rows + 10 * s;
#pragma unroll
        for (int l = 0; l < 5; l++) { row[l] = bb::from_monty(e0.c[l]); row[5 + l] = bb::from_monty(e1.c[l]); }
        const uint32_t x0 = sib_hi ? x : bb::mul(x, minus_one), x1 = sib_hi ? bb::mul(x, minus_one) : x;
        const uint32_t slope_den = bb::inv(bb::sub(x1, x0));
        const E5 slope = bb::e5_mul_base(bb::e5_sub(e1, e0), slope_den);
        folded = bb::e5_add(e0, bb::e5_mul(bb::e5_sub_base(exts[hdr.betas + s], x0), slope));
        index >>= 1;
        x = bb::sqr(x);
    }
    if (!job.check_final) return;
    bool ok = bb::e5_is_zero(reduced_opening(job, bk, partials, LOG_BLOWUP));
    for (int l = 0; l < 5; l++) ok = ok && folded.c[l] == hdr.final_poly.c[l];
    if (!ok) fail(best, job.proof, vb::key_q(job.q, vb::K_FRI_FINAL), VGPU_REJECT_FRI_FINAL);
}

template <int CHIP>
__global__ void __launch_bounds__(64, 1) verify_constraints_kernel(const vb::ChipJob* __restrict__ jobs, uint32_t n, const DevChip* __restrict__ devchips,
                                                               const E5* __restrict__ exts, unsigned long long* best) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const vb::ChipJob& j = jobs[t];
    const vchip::ChipOpenedView ov{exts + j.tl, exts + j.tn, exts + j.pl, exts + j.pn, exts + j.qc};
    if (vchip::chip_constraints<CHIP>(devchips[j.devchip], j.log_degree, ov, j.cumulative_sum, j.zeta, j.alpha) != vchip::CHIP_ACCEPT)
        fail(best, j.proof, j.key, VGPU_REJECT_CONSTRAINTS_CHIP0 - CHIP);
}

// device buffers of one call, released on every path out
struct Bufs {
    vgpu_ctx* ctx; std::vector<void*> p;
    explicit Bufs(vgpu_ctx* c) : ctx(c) {}
    ~Bufs() { for (void* q : p) vg_free(ctx, q); }
    template <class T> int32_t up(const T* host, size_t n, T** out, size_t extra = 0) {
        *out = nullptr;
        const size_t bytes = (n + extra) * sizeof(T);
        if (!bytes) return 0;
        VG_TRY(vg_alloc(ctx, (void**)out, bytes));
        p.push_back(*out);
        if (n) VG_CUDA(ctx, cudaMemcpyAsync(*out, host, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        return 0;
    }
    template <class T> int32_t up(const std::vector<T>& v, T** out, size_t extra = 0) { return up(v.data(), v.size(), out, extra); }
};

template <int CHIP>
int32_t launch_chip(vgpu_ctx* ctx, const vb::ChipJob* jobs, uint32_t n, const DevChip* devchips, const E5* exts, unsigned long long* best) {
    if (!n) return 0;
    {
        KScope ks(ctx, KC_VERIFY_CONSTRAINTS, (double)n * 2048.0);
        verify_constraints_kernel<CHIP><<<(n + 63) / 64, 64, 0, ctx->stream>>>(jobs, n, devchips, exts, best);
    }
    VG_LAUNCH_CHECK(ctx);
    return 0;
}

}  // namespace

namespace vb {

int32_t run_batch(vgpu_ctx* ctx, const Batch& b, std::vector<uint64_t>* best) {
    Bufs bufs(ctx);
    uint32_t *words, *digests, *buckets;
    Group* groups; MerkleJob *input_jobs, *fri_jobs; OpenItem* items; QueryJob* queries; ProofHdr* hdrs;
    E5* exts; E5* partials; DevChip* devchips; unsigned long long* d_best;
    VG_TRY(bufs.up(b.words, &words, b.fri_row_words));
    VG_TRY(bufs.up(b.digests, &digests));
    VG_TRY(bufs.up(b.groups, &groups));
    VG_TRY(bufs.up(b.input_jobs, &input_jobs));
    VG_TRY(bufs.up(b.fri_jobs, &fri_jobs));
    VG_TRY(bufs.up(b.items, &items));
    VG_TRY(bufs.up(b.queries, &queries));
    VG_TRY(bufs.up(b.buckets, &buckets));
    VG_TRY(bufs.up(b.exts, &exts));
    VG_TRY(bufs.up(b.hdrs, &hdrs));
    VG_TRY(bufs.up(b.devchips, &devchips));
    VG_TRY(bufs.up((const E5*)nullptr, 0, &partials, b.n_partials));
    VG_TRY(bufs.up((const unsigned long long*)best->data(), best->size(), &d_best));
    std::vector<ChipJob> chip_flat;
    uint32_t chip_at[VGPU_NUM_CHIPS + 1] = {0};
    for (int c = 0; c < VGPU_NUM_CHIPS; c++) { chip_at[c] = (uint32_t)chip_flat.size(); chip_flat.insert(chip_flat.end(), b.chips[c].begin(), b.chips[c].end()); }
    chip_at[VGPU_NUM_CHIPS] = (uint32_t)chip_flat.size();
    ChipJob* chips;
    VG_TRY(bufs.up(chip_flat, &chips));

    const uint32_t n_in = (uint32_t)b.input_jobs.size(), n_fri = (uint32_t)b.fri_jobs.size(), nq = (uint32_t)b.queries.size();
    if (n_in) {
        {
            KScope ks(ctx, KC_VERIFY_MERKLE, (double)b.words.size() * 4.0 + (double)b.digests.size() * 4.0);
            verify_merkle_kernel<<<(n_in + 127) / 128, 128, 0, ctx->stream>>>(input_jobs, n_in, words, digests, groups, d_best);
        }
        VG_LAUNCH_CHECK(ctx);
    }
    if (nq) {
        {
            KScope ks(ctx, KC_VERIFY_OPEN, (double)b.n_partials * 80.0);
            verify_open_kernel<<<nq, 64, 0, ctx->stream>>>(queries, nq, items, hdrs, words, exts, partials, d_best);
        }
        VG_LAUNCH_CHECK(ctx);
        {
            KScope ks(ctx, KC_VERIFY_FOLD, (double)b.fri_row_words * 4.0);
            verify_fold_kernel<<<(nq + 127) / 128, 128, 0, ctx->stream>>>(queries, nq, hdrs, buckets, exts, partials, words, d_best);
        }
        VG_LAUNCH_CHECK(ctx);
    }
    if (n_fri) {
        {
            KScope ks(ctx, KC_VERIFY_MERKLE, (double)n_fri * 40.0);
            verify_merkle_kernel<<<(n_fri + 127) / 128, 128, 0, ctx->stream>>>(fri_jobs, n_fri, words, digests, groups, d_best);
        }
        VG_LAUNCH_CHECK(ctx);
    }
#define VB_CHIP(c) VG_TRY(launch_chip<c>(ctx, chips + chip_at[c], chip_at[c + 1] - chip_at[c], devchips, exts, d_best));
    VB_CHIP(0) VB_CHIP(1) VB_CHIP(2) VB_CHIP(3) VB_CHIP(4) VB_CHIP(5) VB_CHIP(6)
    VB_CHIP(7) VB_CHIP(8) VB_CHIP(9) VB_CHIP(10) VB_CHIP(11) VB_CHIP(12) VB_CHIP(13)
#undef VB_CHIP
    VG_CUDA(ctx, cudaMemcpyAsync(best->data(), d_best, best->size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    VG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // namespace vb
