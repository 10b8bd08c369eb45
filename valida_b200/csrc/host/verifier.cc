// Machine::verify for proofs in the reference's wire format — the acceptance side of the boundary.
// Follows verify() (derive/src/lib.rs:492-650; hand copy basic/src/lib.rs:677-840):
//   re-commit the preprocessed traces (device, same kernels as the prover) -> replay the transcript ->
//   TwoAdicFriPcs::verify_multi_batches + p3-fri verify_query [P3-UNVERIFIED; SURVEY App. A items 14, 15]
//   -> per-chip verify_constraints (verify.cu) -> the cumulative sums of all chips add to zero.
// Everything except the preprocessed commit is host arithmetic on a ~2 MB proof (40 queries x ~25 Merkle
// paths); it exists so that a caller of this library can check what it produced without the Rust
// verifier, and so that the tests can cross-check prover and verifier against the oracle in both directions.
#include "../ctx.h"
#include "../verify.h"
#include "../verify_batch.h"
#include "challenger.h"
#include <algorithm>
#include <array>
#include <chrono>
#include <cstring>
#include <string>

using bb::E5;

namespace {

constexpr int LOG_BLOWUP = 1, NUM_QUERIES = 40, POW_BITS = 8;   // basic/src/bin/valida.rs:385-390
constexpr int MAX_LOG_DEGREE = 26;

using Digest = std::array<uint32_t, 8>;   // canonical words

// ---- Keccak-256 on the host (original 0x01 padding: p3-keccak wraps tiny-keccak's Keccak::v256) -------
const uint64_t RC[24] = {0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull, 0x000000000000808bull,
                         0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull, 0x000000000000008aull, 0x0000000000000088ull,
                         0x0000000080008009ull, 0x000000008000000aull, 0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull,
                         0x8000000000008003ull, 0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull,
                         0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull};
inline uint64_t rotl(uint64_t x, int n) { return n ? (x << n) | (x >> (64 - n)) : x; }
void keccak_f(uint64_t a[25]) {
    for (int round = 0; round < 24; round++) {
        uint64_t c[5], d[5], b[25];
        for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
        for (int x = 0; x < 5; x++) d[x] = c[(x + 4) % 5] ^ rotl(c[(x + 1) % 5], 1);
        for (int i = 0; i < 25; i++) a[i] ^= d[i % 5];
        // rho + pi walk: lane (x, y) moves to (y, 2x + 3y) with rotation (t+1)(t+2)/2
        int x = 1, y = 0;
        b[0] = a[0];
        for (int t = 0; t < 24; t++) {
            const int nx = y, ny = (2 * x + 3 * y) % 5;
            b[nx + 5 * ny] = rotl(a[x + 5 * y], ((t + 1) * (t + 2) / 2) % 64);
            x = nx; y = ny;
        }
        for (int yy = 0; yy < 25; yy += 5)
            for (int xx = 0; xx < 5; xx++) a[yy + xx] = b[yy + xx] ^ (~b[yy + (xx + 1) % 5] & b[yy + (xx + 2) % 5]);
        a[0] ^= RC[round];
    }
}
// SerializingHasher32<Keccak256Hash>: little-endian canonical words in, 32 bytes out -> 8 words, each reduced mod p
Digest hash_canonical_words(const std::vector<uint32_t>& w) {
    uint64_t st[25] = {0};
    const size_t rate_words = 34;   // 136 bytes
    size_t i = 0;
    while (w.size() - i >= rate_words) {
        for (size_t k = 0; k < 17; k++) st[k] ^= (uint64_t)w[i + 2 * k] | ((uint64_t)w[i + 2 * k + 1] << 32);
        keccak_f(st);
        i += rate_words;
    }
    uint8_t block[136] = {0};
    size_t rem = w.size() - i;
    for (size_t k = 0; k < rem; k++) for (int b = 0; b < 4; b++) block[4 * k + b] = (uint8_t)(w[i + k] >> (8 * b));
    block[4 * rem] ^= 0x01;
    block[135] ^= 0x80;
    for (size_t k = 0; k < 17; k++) { uint64_t v = 0; for (int b = 7; b >= 0; b--) v = (v << 8) | block[8 * k + b]; st[k] ^= v; }
    keccak_f(st);
    Digest d;
    for (int k = 0; k < 4; k++) { d[2 * k] = (uint32_t)st[k] % bb::P; d[2 * k + 1] = (uint32_t)(st[k] >> 32) % bb::P; }
    return d;
}
Digest compress2(const Digest& l, const Digest& r) {
    std::vector<uint32_t> w(16);
    std::memcpy(w.data(), l.data(), 32); std::memcpy(w.data() + 8, r.data(), 32);
    return hash_canonical_words(w);
}

int log2_ceil(uint64_t n) { int l = 0; while ((1ull << l) < n) l++; return l; }

// FieldMerkleTreeMmcs::verify_batch [P3-UNVERIFIED; SURVEY App. A item 8]: matrices sorted by height (stable, tallest
// first); rows of equal padded height are hashed together; a shorter group is injected when the running height reaches it.
struct Dim { uint64_t w, h; };
bool merkle_verify_batch(const Digest& commit, const std::vector<Dim>& dims, uint64_t index,
                         const std::vector<std::vector<uint32_t>>& opened_canonical, const std::vector<Digest>& path) {
    if (dims.empty() || dims.size() != opened_canonical.size()) return false;
    std::vector<size_t> order;
    for (size_t i = 0; i < dims.size(); i++) { if (opened_canonical[i].size() != dims[i].w) return false; order.push_back(i); }
    for (size_t i = 1; i < order.size(); i++)   // stable insertion sort, descending height
        for (size_t j = i; j > 0 && dims[order[j - 1]].h < dims[order[j]].h; j--) std::swap(order[j - 1], order[j]);
    size_t pos = 0;
    int level = log2_ceil(dims[order[0]].h);
    if (path.size() != (size_t)level) return false;
    auto group = [&](int lvl) {
        std::vector<uint32_t> cat;
        while (pos < order.size() && log2_ceil(dims[order[pos]].h) == lvl) { auto& r = opened_canonical[order[pos]]; cat.insert(cat.end(), r.begin(), r.end()); pos++; }
        return hash_canonical_words(cat);
    };
    Digest node = group(level);
    for (const Digest& sib : path) {
        node = (index & 1) ? compress2(sib, node) : compress2(node, sib);
        index >>= 1; level--;
        if (pos < order.size() && log2_ceil(dims[order[pos]].h) == level) node = compress2(node, group(level));
    }
    return pos == order.size() && node == commit;
}

// ---- CBOR reader for exactly the shape vgpu_prove / the reference's ciborium writer emit ----------------
struct Reader {
    const uint8_t* p; const uint8_t* end; bool ok = true;
    uint64_t head(int major) {
        if (!ok || p >= end) { ok = false; return 0; }
        uint8_t b = *p++;
        if ((b >> 5) != major) { ok = false; return 0; }
        uint8_t info = b & 31;
        if (info < 24) return info;
        int n = info == 24 ? 1 : info == 25 ? 2 : info == 26 ? 4 : info == 27 ? 8 : -1;
        if (n < 0 || end - p < n) { ok = false; return 0; }
        uint64_t v = 0;
        for (int i = 0; i < n; i++) v = (v << 8) | *p++;
        return v;
    }
    void key(const char* s) {
        uint64_t n = head(3), want = std::strlen(s);
        if (!ok || n != want || (uint64_t)(end - p) < n || std::memcmp(p, s, n) != 0) { ok = false; return; }
        p += n;
    }
    void map(uint64_t n) { if (head(5) != n) ok = false; }
    // bounded array length: every element costs at least one byte, so a hostile length cannot make us allocate
    uint64_t arr() { uint64_t n = head(4); if (n > (uint64_t)(end - p)) { ok = false; return 0; } return n; }
    uint32_t felt() {   // BabyBear { value: Montgomery word }
        map(1); key("value");
        uint64_t v = head(0);
        if (v >= bb::P) ok = false;
        return (uint32_t)v;
    }
    E5 ext() { E5 e = bb::e5_zero(); map(1); key("value"); if (arr() != 5) ok = false; for (int i = 0; i < 5 && ok; i++) e.c[i] = felt(); return e; }
    Digest digest() { Digest d{}; if (arr() != 8) ok = false; for (int i = 0; i < 8 && ok; i++) d[i] = bb::from_monty(felt()); return d; }
    std::vector<Digest> digests() { std::vector<Digest> v; uint64_t n = arr(); for (uint64_t i = 0; i < n && ok; i++) v.push_back(digest()); return v; }
    std::vector<E5> exts() { std::vector<E5> v; uint64_t n = arr(); for (uint64_t i = 0; i < n && ok; i++) v.push_back(ext()); return v; }
};

struct BatchOpeningV { std::vector<std::vector<uint32_t>> rows_monty; std::vector<Digest> path; };
struct FriStepV { E5 sibling; std::vector<Digest> path; };
struct ProofV {
    Digest main_commit, perm_commit, quot_commit;
    std::vector<Digest> fri_commits;
    std::vector<std::vector<FriStepV>> fri_queries;
    E5 final_poly; uint32_t pow_witness_monty = 0;
    std::vector<std::vector<BatchOpeningV>> query_openings;   // [query][round]
    struct Chip { uint32_t log_degree = 0; VgChipOpening ov; size_t n_prep_local = 0, n_prep_next = 0; E5 cumulative_sum; };
    std::vector<Chip> chips;
};

bool decode(const uint8_t* data, uint64_t len, ProofV* out) {
    Reader r{data, data + len};
    r.map(3);
    r.key("commitments"); r.map(3);
    r.key("main_trace"); out->main_commit = r.digest();
    r.key("perm_trace"); out->perm_commit = r.digest();
    r.key("quotient_chunks"); out->quot_commit = r.digest();
    r.key("opening_proof"); r.map(2);
    r.key("fri_proof"); r.map(4);
    r.key("commit_phase_commits"); out->fri_commits = r.digests();
    r.key("query_proofs");
    for (uint64_t q = 0, nq = r.arr(); q < nq && r.ok; q++) {
        r.map(1); r.key("commit_phase_openings");
        std::vector<FriStepV> steps;
        for (uint64_t s = 0, ns = r.arr(); s < ns && r.ok; s++) {
            FriStepV st;
            r.map(2); r.key("sibling_value"); st.sibling = r.ext(); r.key("opening_proof"); st.path = r.digests();
            steps.push_back(std::move(st));
        }
        out->fri_queries.push_back(std::move(steps));
    }
    r.key("final_poly"); out->final_poly = r.ext();
    r.key("pow_witness"); out->pow_witness_monty = r.felt();
    r.key("query_openings");
    for (uint64_t q = 0, nq = r.arr(); q < nq && r.ok; q++) {
        std::vector<BatchOpeningV> per_round;
        for (uint64_t b = 0, nb = r.arr(); b < nb && r.ok; b++) {
            BatchOpeningV bo;
            r.map(2); r.key("opened_values");
            for (uint64_t m = 0, nm = r.arr(); m < nm && r.ok; m++) {
                std::vector<uint32_t> row;
                for (uint64_t c = 0, nc = r.arr(); c < nc && r.ok; c++) row.push_back(r.felt());
                bo.rows_monty.push_back(std::move(row));
            }
            r.key("opening_proof"); bo.path = r.digests();
            per_round.push_back(std::move(bo));
        }
        out->query_openings.push_back(std::move(per_round));
    }
    r.key("chip_proofs");
    for (uint64_t i = 0, n = r.arr(); i < n && r.ok; i++) {
        ProofV::Chip c;
        r.map(3);
        r.key("log_degree"); c.log_degree = (uint32_t)r.head(0);
        r.key("opened_values"); r.map(7);
        r.key("preprocessed_local"); c.n_prep_local = r.exts().size();
        r.key("preprocessed_next"); c.n_prep_next = r.exts().size();
        r.key("trace_local"); c.ov.trace_local = r.exts();
        r.key("trace_next"); c.ov.trace_next = r.exts();
        r.key("permutation_local"); c.ov.perm_local = r.exts();
        r.key("permutation_next"); c.ov.perm_next = r.exts();
        r.key("quotient_chunks"); c.ov.quotient_chunks = r.exts();
        r.key("cumulative_sum"); c.cumulative_sum = r.ext();
        out->chips.push_back(std::move(c));
    }
    return r.ok && r.p == r.end;
}


struct RoundV { Digest commit; std::vector<Dim> dims; std::vector<std::vector<E5>> points; std::vector<std::vector<const std::vector<E5>*>> values; };

// What the transcript gives a verifier before it opens the first query.
struct Challenges {
    uint32_t perm_challenges[15];   // canonical
    E5 alpha, zeta, fri_alpha;
    std::vector<E5> betas;
    std::vector<uint32_t> indices;
    int log_max_height = 0;
};

// decode + the up-front shape checks of vgpu_verify; VGPU_ACCEPT = go on
int32_t decode_and_check_shape(const uint8_t* proof, uint64_t proof_len, const vgpu_matrix prep[2], ProofV* pf) {
    if (!decode(proof, proof_len, pf)) return VGPU_REJECT_MALFORMED;
    if (pf->chips.size() != (size_t)VGPU_NUM_CHIPS) return VGPU_REJECT_SHAPE;
    for (auto& c : pf->chips) if (c.log_degree > (uint32_t)MAX_LOG_DEGREE || c.n_prep_local || c.n_prep_next) return VGPU_REJECT_SHAPE;
    // the two chips with preprocessed columns have the height of those columns (program ROM, range table): a proof may not
    // shrink them (an all-one-row proof has no FRI layers at all)
    if ((1ull << pf->chips[1].log_degree) != prep[0].height || (1ull << pf->chips[12].log_degree) != prep[1].height) return VGPU_REJECT_SHAPE;
    return VGPU_ACCEPT;
}

// preprocessed commitment, recomputed (derive/src/lib.rs:505-517)
int32_t commit_preprocessed(vgpu_ctx* ctx, const vgpu_matrix prep[2], int32_t repr, uint32_t digest[8]) {
    vgpu_prover_data* pd = nullptr;
    // a verifier checks alone: no collective here even when the context is a rank of a split prover
    const bool was_sharding = ctx->sharding;
    ctx->sharding = false;
    const int32_t rc = vgpu_commit_batches_host(ctx, prep, 2, repr, nullptr, digest, &pd);
    ctx->sharding = was_sharding;
    if (rc) return rc;
    vgpu_prover_data_free(pd);
    return 0;
}

// The whole transcript of Machine::verify and TwoAdicFriPcs::verify_multi_batches up to the query indices, with the checks that
// come before the first query (counts, proof of work, heights).  Also lays out the three opened rounds.  VGPU_ACCEPT = go on.
int32_t replay_transcript(const vgh::Poseidon16& perm, const uint32_t prep_digest[8], const ProofV& pf, std::vector<RoundV>* rounds_out, Challenges* c) {
    vgh::Challenger ch;
    ch.perm = &perm;
    ch.observe_digest_canonical(prep_digest);
    ch.observe_digest_canonical(pf.main_commit.data());
    for (int i = 0; i < 3; i++) { E5 e = ch.sample_ext(); for (int l = 0; l < 5; l++) c->perm_challenges[5 * i + l] = bb::from_monty(e.c[l]); }
    ch.observe_digest_canonical(pf.perm_commit.data());
    c->alpha = ch.sample_ext();
    ch.observe_digest_canonical(pf.quot_commit.data());
    c->zeta = ch.sample_ext();
    const E5 zeta = c->zeta;

    std::vector<RoundV>& rounds = *rounds_out;
    rounds.assign(3, RoundV{});
    rounds[0].commit = pf.main_commit; rounds[1].commit = pf.perm_commit; rounds[2].commit = pf.quot_commit;
    for (int i = 0; i < VGPU_NUM_CHIPS; i++) {
        const vgpu_chip_desc* chip = vgpu_basic_machine_chip(i);
        const ProofV::Chip& cp = pf.chips[i];
        const uint64_t h = 1ull << cp.log_degree;
        const E5 zg = bb::e5_mul_base(zeta, bb::two_adic_generator_monty((int)cp.log_degree));
        rounds[0].dims.push_back({chip->width, h});
        rounds[1].dims.push_back({5ull * (chip->n_interactions + 1), h});
        rounds[2].dims.push_back({10, h});
        rounds[0].points.push_back({zeta, zg}); rounds[0].values.push_back({&cp.ov.trace_local, &cp.ov.trace_next});
        rounds[1].points.push_back({zeta, zg}); rounds[1].values.push_back({&cp.ov.perm_local, &cp.ov.perm_next});
        rounds[2].points.push_back({bb::e5_sqr(zeta)}); rounds[2].values.push_back({&cp.ov.quotient_chunks});
    }

    // TwoAdicFriPcs::verify_multi_batches + p3-fri verifier, up to the queries
    c->fri_alpha = ch.sample_ext();
    c->betas.clear();
    for (const Digest& d : pf.fri_commits) { ch.observe_digest_canonical(d.data()); c->betas.push_back(ch.sample_ext()); }
    if (pf.fri_queries.size() != (size_t)NUM_QUERIES || pf.query_openings.size() != (size_t)NUM_QUERIES) return VGPU_REJECT_SHAPE;
    if (!ch.check_witness(POW_BITS, pf.pow_witness_monty)) return VGPU_REJECT_POW;
    c->log_max_height = (int)pf.fri_commits.size() + LOG_BLOWUP;
    if (c->log_max_height > MAX_LOG_DEGREE + LOG_BLOWUP) return VGPU_REJECT_SHAPE;
    for (auto& rd : rounds)
        for (auto& d : rd.dims) if (log2_ceil(d.h) + LOG_BLOWUP > c->log_max_height) return VGPU_REJECT_SHAPE;
    c->indices.clear();
    for (int q = 0; q < NUM_QUERIES; q++) c->indices.push_back(ch.sample_bits(c->log_max_height));
    return VGPU_ACCEPT;
}

// The queries of the FRI opening proof, on the host; 0 = accept, otherwise the verdict code of include/valida_b200.h
int32_t verify_queries(const std::vector<RoundV>& rounds, const ProofV& pf, const Challenges& chal) {
    const int log_max_height = chal.log_max_height;
    const E5 alpha = chal.fri_alpha;
    const uint32_t gen = bb::to_monty(bb::GEN_CANON);
    for (int q = 0; q < NUM_QUERIES; q++) {
        uint64_t index = chal.indices[q];
        E5 ro[32], apw[32];
        for (int i = 0; i < 32; i++) { ro[i] = bb::e5_zero(); apw[i] = bb::e5_one(); }
        if (pf.query_openings[q].size() != rounds.size()) return VGPU_REJECT_SHAPE;
        for (size_t r = 0; r < rounds.size(); r++) {
            const RoundV& rd = rounds[r];
            const BatchOpeningV& bo = pf.query_openings[q][r];
            if (bo.rows_monty.size() != rd.dims.size()) return VGPU_REJECT_SHAPE;
            std::vector<Dim> lde_dims;
            uint64_t max_h = 0;
            for (auto& d : rd.dims) { lde_dims.push_back({d.w, d.h << LOG_BLOWUP}); max_h = std::max(max_h, d.h << LOG_BLOWUP); }
            std::vector<std::vector<uint32_t>> canon_rows;
            for (auto& row : bo.rows_monty) { std::vector<uint32_t> c; for (uint32_t x : row) c.push_back(bb::from_monty(x)); canon_rows.push_back(std::move(c)); }
            const uint64_t batch_index = index >> (log_max_height - log2_ceil(max_h));
            if (!merkle_verify_batch(rd.commit, lde_dims, batch_index, canon_rows, bo.path)) return VGPU_REJECT_INPUT_MERKLE;
            for (size_t mi = 0; mi < rd.dims.size(); mi++) {
                const int lh = log2_ceil(rd.dims[mi].h) + LOG_BLOWUP;
                const uint32_t rev = bb::reverse_bits((uint32_t)(index >> (log_max_height - lh)), lh);
                const uint32_t x = bb::mul(gen, bb::pow(bb::two_adic_generator_monty(lh), rev));
                for (size_t pi = 0; pi < rd.points[mi].size(); pi++) {
                    const std::vector<E5>& at_z = *rd.values[mi][pi];
                    if (at_z.size() != bo.rows_monty[mi].size()) return VGPU_REJECT_SHAPE;
                    const E5 den = bb::e5_add_base(bb::e5_neg(rd.points[mi][pi]), x);   // x - z
                    if (bb::e5_is_zero(den)) return VGPU_REJECT_SHAPE;
                    const E5 dinv = bb::e5_inv(den);
                    for (size_t c = 0; c < at_z.size(); c++) {
                        const E5 quotient = bb::e5_mul(bb::e5_add_base(bb::e5_neg(at_z[c]), bo.rows_monty[mi][c]), dinv);   // (p(x) - p(z)) / (x - z)
                        ro[lh] = bb::e5_add(ro[lh], bb::e5_mul(apw[lh], quotient));
                        apw[lh] = bb::e5_mul(apw[lh], alpha);
                    }
                }
            }
        }
        // p3-fri verify_query
        const std::vector<FriStepV>& steps = pf.fri_queries[q];
        if (steps.size() != pf.fri_commits.size()) return VGPU_REJECT_SHAPE;
        E5 folded = bb::e5_zero();
        uint32_t x = bb::pow(bb::two_adic_generator_monty(log_max_height), bb::reverse_bits((uint32_t)index, log_max_height));
        const uint32_t minus_one = bb::two_adic_generator_monty(1);
        size_t si = 0;
        for (int lfh = log_max_height - 1; lfh >= LOG_BLOWUP; lfh--, si++) {
            folded = bb::e5_add(folded, ro[lfh + 1]);
            const uint64_t sib = (index ^ 1) & 1, pair = index >> 1;
            E5 evals[2] = {folded, folded};
            evals[sib] = steps[si].sibling;
            std::vector<uint32_t> row(10);
            for (int e = 0; e < 2; e++) for (int l = 0; l < 5; l++) row[5 * e + l] = bb::from_monty(evals[e].c[l]);
            if (!merkle_verify_batch(pf.fri_commits[si], {{10, 1ull << lfh}}, pair, {row}, steps[si].path)) return VGPU_REJECT_FRI_MERKLE;
            uint32_t xs[2] = {x, x};
            xs[sib] = bb::mul(xs[sib], minus_one);
            // line through (xs[0], evals[0]), (xs[1], evals[1]) evaluated at beta; xs[1] - xs[0] = -2 xs[0]
            const uint32_t slope_den = bb::inv(bb::sub(xs[1], xs[0]));
            const E5 slope = bb::e5_mul_base(bb::e5_sub(evals[1], evals[0]), slope_den);
            folded = bb::e5_add(evals[0], bb::e5_mul(bb::e5_sub_base(chal.betas[si], xs[0]), slope));
            index = pair;
            x = bb::sqr(x);
        }
        // The prover's last fold also adds the reduced openings of the height-2 LDEs (traces of ONE row: constant polynomials,
        // for which (p(x) - p(z)) / (x - z) is exactly 0).  The loop above never reaches them, so they are checked here: without
        // this the opened values of every one-row chip — and with them its cumulative sum — would be bound by nothing.
        if (!bb::e5_is_zero(ro[LOG_BLOWUP])) return VGPU_REJECT_FRI_FINAL;
        for (int l = 0; l < 5; l++) if (folded.c[l] != pf.final_poly.c[l]) return VGPU_REJECT_FRI_FINAL;
    }
    return VGPU_ACCEPT;
}

void set_poseidon(const vgpu_ctx* ctx, vgh::Poseidon16* perm) { perm->set(ctx->poseidon_rc, ctx->poseidon_has_mds ? ctx->poseidon_mds : nullptr); }

// ---- batch verification: packing one proof for the device (verify_batch.h) ----------------------------------------------------
// Walks the queries in vgpu_verify's order and packs every check the device has to run, up to the first failure that the packing
// itself finds (a count, a width, a path length): that failure goes into the proof's slot, and nothing after it is packed.
void pack_proof(vb::Batch& b, uint32_t p, const ProofV& pf, const std::vector<RoundV>& rounds, const Challenges& chal, uint32_t devchip0) {
    using namespace vb;
    uint64_t& best = b.best[p];
    auto note = [&](uint32_t key, int32_t code) { best = std::min(best, slot(key, code)); };
    const int L = chal.log_max_height;
    ProofHdr hdr{};
    hdr.log_max_height = (uint32_t)L; hdr.fri_alpha = chal.fri_alpha; hdr.final_poly = pf.final_poly;
    hdr.betas = (uint32_t)b.exts.size();
    b.exts.insert(b.exts.end(), chal.betas.begin(), chal.betas.end());

    // layout of a query's opened rows: per round, the matrices tallest first (stable), rows of one height contiguous
    const size_t NR = rounds.size();
    std::vector<std::vector<uint32_t>> row_off(NR);
    std::vector<uint32_t> round_off(NR), round_groups(NR), round_ngroups(NR), round_top(NR);
    uint32_t block = 0;
    for (size_t r = 0; r < NR; r++) {
        const std::vector<Dim>& dims = rounds[r].dims;
        std::vector<size_t> order(dims.size());
        for (size_t i = 0; i < order.size(); i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t c) { return dims[a].h > dims[c].h; });
        row_off[r].assign(dims.size(), 0);
        round_off[r] = block;
        round_groups[r] = (uint32_t)b.groups.size();
        for (size_t k = 0; k < order.size(); k++) {
            const uint32_t level = (uint32_t)log2_ceil(dims[order[k]].h << LOG_BLOWUP);
            if (k == 0 || b.groups.back().level != level) b.groups.push_back({level, 0});
            b.groups.back().nwords += (uint32_t)dims[order[k]].w;
            row_off[r][order[k]] = block;
            block += (uint32_t)dims[order[k]].w;
        }
        round_ngroups[r] = (uint32_t)b.groups.size() - round_groups[r];
        round_top[r] = (uint32_t)log2_ceil(dims[order[0]].h << LOG_BLOWUP);
    }

    // the reduced-opening items, in vgpu_verify's order; alpha^(columns before it in its log-height bucket) computed here once
    const uint32_t items0 = (uint32_t)b.items.size();
    uint32_t width_fail = UINT32_MAX, width_fail_round = UINT32_MAX;
    {
        uint32_t before[32] = {0};
        for (size_t r = 0; r < NR && width_fail == UINT32_MAX; r++)
            for (size_t mi = 0; mi < rounds[r].dims.size() && width_fail == UINT32_MAX; mi++)
                for (size_t pi = 0; pi < rounds[r].points[mi].size(); pi++) {
                    const std::vector<E5>& at_z = *rounds[r].values[mi][pi];
                    const Dim& d = rounds[r].dims[mi];
                    if (at_z.size() != d.w) { width_fail = k_point((uint32_t)r, (uint32_t)mi, (uint32_t)pi); width_fail_round = (uint32_t)r; break; }
                    OpenItem it{};
                    it.lh = (uint32_t)log2_ceil(d.h) + LOG_BLOWUP;
                    it.width = (uint32_t)d.w; it.row_off = row_off[r][mi]; it.vals = (uint32_t)b.exts.size();
                    it.key = k_point((uint32_t)r, (uint32_t)mi, (uint32_t)pi);
                    it.z = rounds[r].points[mi][pi];
                    it.alpha_pow = bb::e5_pow(chal.fri_alpha, before[it.lh]);
                    before[it.lh] += it.width;
                    b.exts.insert(b.exts.end(), at_z.begin(), at_z.end());
                    b.items.push_back(it);
                }
    }
    const uint32_t n_items = (uint32_t)b.items.size() - items0;
    hdr.buckets = (uint32_t)b.buckets.size();
    {   // 33 begin offsets by lh, then the item indices sorted by lh (stable)
        std::vector<uint32_t> sorted;
        std::vector<uint32_t> begin(33, 0);
        for (uint32_t lh = 0; lh < 32; lh++) {
            begin[lh] = (uint32_t)sorted.size();
            for (uint32_t i = 0; i < n_items; i++) if (b.items[items0 + i].lh == lh) sorted.push_back(i);
        }
        begin[32] = (uint32_t)sorted.size();
        b.buckets.insert(b.buckets.end(), begin.begin(), begin.end());
        b.buckets.insert(b.buckets.end(), sorted.begin(), sorted.end());
    }
    b.hdrs.push_back(hdr);

    for (uint32_t q = 0; q < (uint32_t)NUM_QUERIES; q++) {
        const uint32_t index = chal.indices[q];
        QueryJob job{};
        job.proof = p; job.q = q; job.index = index; job.items = items0; job.partials = b.n_partials;
        job.words = b.words.size();
        uint32_t stop = UINT32_MAX;   // query-local key where the packing found a failure
        const auto& qo = pf.query_openings[q];
        if (qo.size() != NR) { stop = K_QUERY_ROUNDS; note(key_q(q, stop), VGPU_REJECT_SHAPE); }
        for (size_t r = 0; r < NR && stop == UINT32_MAX; r++) {
            const BatchOpeningV& bo = qo[r];
            const std::vector<Dim>& dims = rounds[r].dims;
            if (bo.rows_monty.size() != dims.size()) { stop = k_round((uint32_t)r); note(key_q(q, stop), VGPU_REJECT_SHAPE); break; }
            bool shape_ok = bo.path.size() == round_top[r];
            for (size_t mi = 0; mi < dims.size() && shape_ok; mi++) shape_ok = bo.rows_monty[mi].size() == dims[mi].w;
            if (!shape_ok) { stop = k_round((uint32_t)r) + 1; note(key_q(q, stop), VGPU_REJECT_INPUT_MERKLE); break; }
            const uint64_t at = b.words.size();
            b.words.resize(at + (r + 1 < NR ? round_off[r + 1] : block) - round_off[r]);
            for (size_t mi = 0; mi < dims.size(); mi++)
                for (size_t c = 0; c < dims[mi].w; c++) b.words[job.words + row_off[r][mi] + c] = bb::from_monty(bo.rows_monty[mi][c]);
            MerkleJob mj{};
            mj.proof = p; mj.key = key_q(q, k_round((uint32_t)r) + 1); mj.code = (uint32_t)VGPU_REJECT_INPUT_MERKLE;
            mj.groups = round_groups[r]; mj.n_groups = round_ngroups[r]; mj.path_len = round_top[r];
            mj.index = index >> (L - (int)round_top[r]);
            mj.words = at; mj.path = b.digests.size() / 8;
            for (const Digest& d : bo.path) b.digests.insert(b.digests.end(), d.begin(), d.end());
            std::memcpy(mj.commit, rounds[r].commit.data(), 32);
            b.input_jobs.push_back(mj);
            if (width_fail_round == r) { stop = width_fail; note(key_q(q, stop), VGPU_REJECT_SHAPE); }
        }
        while (job.n_items < n_items && b.items[items0 + job.n_items].key < stop) job.n_items++;
        if (stop == UINT32_MAX) {
            const std::vector<FriStepV>& steps = pf.fri_queries[q];
            if (steps.size() != pf.fri_commits.size()) {
                stop = K_FRI_STEPS; note(key_q(q, stop), VGPU_REJECT_SHAPE);
            } else {
                job.sibs = (uint32_t)b.exts.size();
                job.rows = b.fri_row_words;   // relative to the end of the host words: fixed up once the batch is complete
                for (uint32_t s = 0; s < (uint32_t)steps.size(); s++) {
                    const uint32_t lfh = (uint32_t)L - 1 - s;
                    if (steps[s].path.size() != lfh) { stop = k_fri_step(s); note(key_q(q, stop), VGPU_REJECT_FRI_MERKLE); break; }
                    b.exts.push_back(steps[s].sibling);
                    MerkleJob mj{};
                    mj.proof = p; mj.key = key_q(q, k_fri_step(s)); mj.code = (uint32_t)VGPU_REJECT_FRI_MERKLE;
                    mj.groups = (uint32_t)b.groups.size(); mj.n_groups = 1; mj.path_len = lfh;
                    b.groups.push_back({lfh, 10});
                    mj.index = index >> (s + 1);
                    mj.words = job.rows + 10ull * s; mj.path = b.digests.size() / 8;
                    for (const Digest& d : steps[s].path) b.digests.insert(b.digests.end(), d.begin(), d.end());
                    std::memcpy(mj.commit, pf.fri_commits[s].data(), 32);
                    b.fri_jobs.push_back(mj);
                    job.fold_steps++;
                }
                b.fri_row_words += 10ull * job.fold_steps;
                job.check_final = stop == UINT32_MAX;
            }
        }
        b.n_partials += job.n_items;
        b.queries.push_back(job);
        if (stop != UINT32_MAX) break;   // every later check has a larger key
    }

    // chips at zeta, then the cumulative sum
    E5 sum = bb::e5_zero();
    for (uint32_t i = 0; i < (uint32_t)VGPU_NUM_CHIPS; i++) {
        const vgpu_chip_desc* chip = vgpu_basic_machine_chip(i);
        const ProofV::Chip& cp = pf.chips[i];
        const VgChipOpening& ov = cp.ov;
        sum = bb::e5_add(sum, cp.cumulative_sum);
        const size_t pw = chip->n_interactions + 1;
        if (ov.trace_local.size() != chip->width || ov.trace_next.size() != chip->width || ov.perm_local.size() != 5 * pw ||
            ov.perm_next.size() != 5 * pw || ov.quotient_chunks.size() != 10) { note(key_chip(i), VGPU_REJECT_CONSTRAINTS_CHIP0 - (int32_t)i); continue; }
        ChipJob cj{};
        cj.proof = p; cj.key = key_chip(i); cj.log_degree = cp.log_degree; cj.devchip = devchip0 + i;
        cj.cumulative_sum = cp.cumulative_sum; cj.zeta = chal.zeta; cj.alpha = chal.alpha;
        auto put = [&](const std::vector<E5>& v) { const uint32_t o = (uint32_t)b.exts.size(); b.exts.insert(b.exts.end(), v.begin(), v.end()); return o; };
        cj.tl = put(ov.trace_local); cj.tn = put(ov.trace_next); cj.pl = put(ov.perm_local); cj.pn = put(ov.perm_next); cj.qc = put(ov.quotient_chunks);
        b.chips[i].push_back(cj);
    }
    if (!bb::e5_is_zero(sum)) note(key_cumulative_sum(), VGPU_REJECT_CUMULATIVE_SUM);
}

bool reads_preprocessed(const vgpu_pair_col& pc) {
    for (uint32_t t = 0; t < pc.n_terms && t < VGPU_MAX_TERMS; t++) if (pc.terms[t].is_preprocessed) return true;
    return false;
}

using Clock = std::chrono::steady_clock;
float ms_since(Clock::time_point t0) { return std::chrono::duration<float, std::milli>(Clock::now() - t0).count(); }

}  // namespace

extern "C" int32_t vgpu_verify(vgpu_ctx* ctx, const uint8_t* proof, uint64_t proof_len, const vgpu_matrix prep[2], int32_t repr, int32_t* verdict) {
    if (!ctx) return -1;
    if (!proof || !prep || !verdict) VG_FAIL(ctx, "verify: null argument");
    if (!ctx->challenger_set) VG_FAIL(ctx, "verify: vgpu_set_challenger has not been called");
    VG_TRY(vg_enter(ctx));
    *verdict = VGPU_REJECT_MALFORMED;
    ProofV pf;
    const int32_t shape = decode_and_check_shape(proof, proof_len, prep, &pf);
    if (shape != VGPU_ACCEPT) { *verdict = shape; return 0; }

    vgh::Poseidon16 perm;
    set_poseidon(ctx, &perm);
    uint32_t digest[8];
    VG_TRY(commit_preprocessed(ctx, prep, repr, digest));
    std::vector<RoundV> rounds;
    Challenges chal;
    int32_t v = replay_transcript(perm, digest, pf, &rounds, &chal);
    if (v == VGPU_ACCEPT) v = verify_queries(rounds, pf, chal);
    if (v != VGPU_ACCEPT) { *verdict = v; return 0; }
    for (int i = 0; i < VGPU_NUM_CHIPS; i++) {
        bool ok = false;
        VG_TRY(vg_verify_chip_constraints(ctx, vgpu_basic_machine_chip(i), pf.chips[i].log_degree, pf.chips[i].ov, pf.chips[i].cumulative_sum,
                                          chal.zeta, chal.alpha, chal.perm_challenges, &ok));
        if (!ok) { *verdict = VGPU_REJECT_CONSTRAINTS_CHIP0 - i; return 0; }
    }
    E5 sum = bb::e5_zero();
    for (auto& c : pf.chips) sum = bb::e5_add(sum, c.cumulative_sum);
    if (!bb::e5_is_zero(sum)) { *verdict = VGPU_REJECT_CUMULATIVE_SUM; return 0; }
    *verdict = VGPU_ACCEPT;
    return 0;
}

// Host threads for the per-proof decode and transcript replay of vgpu_verify_batch (independent across proofs)
constexpr int VERIFY_BATCH_THREADS = 8;

extern "C" int32_t vgpu_verify_batch(vgpu_ctx* ctx, const uint8_t* const* proofs, const uint64_t* proof_lens, uint32_t n,
                                     const vgpu_matrix* prep, uint32_t n_programs, const uint32_t* program_of, int32_t repr, int32_t* verdicts) {
    if (!ctx) return -1;
    if (!ctx->challenger_set) VG_FAIL(ctx, "verify_batch: vgpu_set_challenger has not been called");
    if (n == 0) return 0;
    if (!proofs || !proof_lens || !prep || !program_of || !verdicts) VG_FAIL(ctx, "verify_batch: null argument");
    for (uint32_t i = 0; i < n; i++) {
        if (program_of[i] >= n_programs) VG_FAIL(ctx, "verify_batch: program_of[%u] = %u, but only %u programs are given", i, program_of[i], n_programs);
        if (!proofs[i] && proof_lens[i]) VG_FAIL(ctx, "verify_batch: proof %u is null", i);
    }
    for (uint32_t c = 0; c < (uint32_t)VGPU_NUM_CHIPS; c++) {
        const vgpu_chip_desc* chip = vgpu_basic_machine_chip(c);
        for (uint32_t m = 0; m < chip->n_interactions && m < VGPU_MAX_INTERACTIONS; m++) {
            bool prep_col = reads_preprocessed(chip->interactions[m].count);
            for (uint32_t j = 0; j < chip->interactions[m].n_fields && j < VGPU_MAX_FIELDS; j++) prep_col = prep_col || reads_preprocessed(chip->interactions[m].fields[j]);
            if (prep_col) VG_FAIL(ctx, "verify_batch: an interaction reads a preprocessed column, which the proof does not open");
        }
    }
    VG_TRY(vg_enter(ctx));
    ctx->verify_phases.clear();

    // 1. decode + shape (host threads)
    auto t0 = Clock::now();
    std::vector<ProofV> pfs(n);
    std::vector<int32_t> early(n, VGPU_ACCEPT);
#pragma omp parallel for schedule(dynamic) num_threads(VERIFY_BATCH_THREADS)
    for (int64_t i = 0; i < (int64_t)n; i++) early[i] = decode_and_check_shape(proofs[i], proof_lens[i], prep + 2 * program_of[i], &pfs[i]);
    ctx->verify_phases.push_back({"decode + shape checks (host)", ms_since(t0)});

    // 2. the preprocessed commitment of every program a well-formed proof refers to, once
    t0 = Clock::now();
    std::vector<Digest> prep_digest(n_programs);
    std::vector<char> need(n_programs, 0);
    for (uint32_t i = 0; i < n; i++) if (early[i] == VGPU_ACCEPT) need[program_of[i]] = 1;
    for (uint32_t g = 0; g < n_programs; g++) if (need[g]) VG_TRY(commit_preprocessed(ctx, prep + 2 * g, repr, prep_digest[g].data()));
    ctx->verify_phases.push_back({"preprocessed commitments (device)", ms_since(t0)});

    // 3. transcripts (host threads)
    t0 = Clock::now();
    vgh::Poseidon16 perm;
    set_poseidon(ctx, &perm);
    std::vector<std::vector<RoundV>> rounds(n);
    std::vector<Challenges> chal(n);
#pragma omp parallel for schedule(dynamic) num_threads(VERIFY_BATCH_THREADS)
    for (int64_t i = 0; i < (int64_t)n; i++)
        if (early[i] == VGPU_ACCEPT) early[i] = replay_transcript(perm, prep_digest[program_of[i]].data(), pfs[i], &rounds[i], &chal[i]);
    ctx->verify_phases.push_back({"transcript replay (host)", ms_since(t0)});

    // 4. pack the proofs that reach their queries
    t0 = Clock::now();
    vb::Batch b;
    std::vector<uint32_t> slot_of(n, UINT32_MAX);
    for (uint32_t i = 0; i < n; i++) {
        if (early[i] != VGPU_ACCEPT) continue;
        const uint32_t p = b.n_proofs++;
        slot_of[i] = p;
        b.best.push_back(vb::SLOT_NONE);
        const uint32_t devchip0 = (uint32_t)b.devchips.size();
        b.devchips.resize(devchip0 + VGPU_NUM_CHIPS);
        for (int c = 0; c < VGPU_NUM_CHIPS; c++) VG_TRY(vg_build_devchip(ctx, vgpu_basic_machine_chip(c), chal[i].perm_challenges, &b.devchips[devchip0 + c]));
        pack_proof(b, p, pfs[i], rounds[i], chal[i], devchip0);
    }
    // the FRI rows the fold kernel writes follow the opened rows
    const uint64_t host_words = b.words.size();
    for (auto& q : b.queries) q.rows += host_words;
    for (auto& j : b.fri_jobs) j.words += host_words;
    if (b.exts.size() >= UINT32_MAX || b.n_partials >= UINT32_MAX / 2) VG_FAIL(ctx, "verify_batch: batch too large, split it");
    ctx->verify_phases.push_back({"packing (host)", ms_since(t0)});

    // 5. the device checks
    t0 = Clock::now();
    std::vector<uint64_t> best = b.best;
    if (b.n_proofs) VG_TRY(vb::run_batch(ctx, b, &best));
    ctx->verify_phases.push_back({"device checks (wall)", ms_since(t0)});
    for (uint32_t i = 0; i < n; i++) {
        if (slot_of[i] == UINT32_MAX) { verdicts[i] = early[i]; continue; }
        const uint64_t s = best[slot_of[i]];
        verdicts[i] = s == vb::SLOT_NONE ? VGPU_ACCEPT : (int32_t)(uint32_t)s;
    }
    return 0;
}

extern "C" uint32_t vgpu_last_verify_batch_phases(const vgpu_ctx* ctx, const char** names, float* ms, uint32_t cap) {
    if (!ctx) return 0;
    uint32_t k = 0;
    for (; k < ctx->verify_phases.size() && k < cap; k++) { names[k] = ctx->verify_phases[k].first; ms[k] = ctx->verify_phases[k].second; }
    return (uint32_t)ctx->verify_phases.size();
}
