// Internal interface between the batch verifier's host side (host/verifier.cc: decode, transcript, shape checks, packing) and its
// device side (verify_batch.cu: Merkle paths, reduced openings, FRI folds, constraints at zeta).
//
// Every check of vgpu_verify has an ordinal KEY in the order vgpu_verify runs them; a proof's verdict is the code of its smallest
// failing key.  Failures found while packing (counts, widths, path lengths) and on the device land in the same per-proof slot,
// (key << 32) | (uint32_t)code, which only ever decreases (atomicMin on the device).
#pragma once
#include "ctx.h"
#include "devchip.h"
#include <vector>

namespace vb {

constexpr uint32_t NUM_QUERIES = 40;
constexpr uint32_t QSTRIDE = 256;                          // keys per query
constexpr uint32_t K_QUERY_ROUNDS = 0;                     // the query opens a different number of rounds (SHAPE)
BB_HD uint32_t k_round(uint32_t r) { return 1 + 32 * r; } // + 0 opened-row count (SHAPE), + 1 Merkle path (INPUT_MERKLE)
BB_HD uint32_t k_point(uint32_t r, uint32_t mi, uint32_t pi) { return k_round(r) + 2 + 2 * mi + pi; }   // width / zero denominator (SHAPE)
constexpr uint32_t K_FRI_STEPS = 100;                      // FRI step count (SHAPE)
BB_HD uint32_t k_fri_step(uint32_t s) { return 101 + s; } // FRI layer path (FRI_MERKLE)
constexpr uint32_t K_FRI_FINAL = 160;
BB_HD uint32_t key_q(uint32_t q, uint32_t local) { return q * QSTRIDE + local; }
BB_HD uint32_t key_chip(uint32_t i) { return NUM_QUERIES * QSTRIDE + i; }   // -100 - i
BB_HD uint32_t key_cumulative_sum() { return NUM_QUERIES * QSTRIDE + VGPU_NUM_CHIPS; }
BB_HD uint64_t slot(uint32_t key, int32_t code) { return ((uint64_t)key << 32) | (uint32_t)code; }
constexpr uint64_t SLOT_NONE = ~0ull;

struct Group { uint32_t level, nwords; };                  // rows of one padded height, hashed together
// One Merkle opening: the leaf groups (tallest first) at words[words ..], the path at digests[8 * path ..]
struct MerkleJob {
    uint32_t proof, key, code, groups, n_groups, path_len, index;
    uint64_t words, path;
    uint32_t commit[8];
};
// One (round, matrix, point) of a proof's reduced openings; the same for all its queries.
struct OpenItem {
    uint32_t lh, width, row_off, vals, key;                // row_off: into the query's row block; vals: into exts; key: query-local
    bb::E5 z, alpha_pow;                                   // alpha_pow = alpha^(columns before it in the same log-height bucket)
};
struct QueryJob {
    uint32_t proof, q, index;
    uint32_t items, n_items;                               // the first n_items items of the proof are checked (fewer when packing stopped)
    uint32_t partials;                                     // partials[partials + i]: item i's share of ro[lh]
    uint32_t fold_steps, check_final;                      // FRI steps to fold (rows written to words[rows + 10 s]); final check
    uint32_t sibs;                                         // exts[sibs + s]: the sibling value of FRI step s
    uint64_t words, rows;
};
struct ProofHdr {
    uint32_t log_max_height, betas, buckets;               // buckets: 33 begin offsets (by lh), then item indices sorted by lh
    bb::E5 fri_alpha, final_poly;
};
struct ChipJob {
    uint32_t proof, key, log_degree, devchip;
    uint32_t tl, tn, pl, pn, qc;                           // opened values in exts
    bb::E5 cumulative_sum, zeta, alpha;
};

struct Batch {
    uint32_t n_proofs = 0;
    std::vector<uint32_t> words;                           // canonical: opened rows; FRI rows are appended on the device
    uint64_t fri_row_words = 0;
    std::vector<uint32_t> digests;                         // path siblings, 8 canonical words each
    std::vector<Group> groups;
    std::vector<MerkleJob> input_jobs, fri_jobs;
    std::vector<OpenItem> items;
    std::vector<QueryJob> queries;
    uint32_t n_partials = 0;
    std::vector<uint32_t> buckets;
    std::vector<bb::E5> exts;
    std::vector<ProofHdr> hdrs;
    std::vector<ChipJob> chips[VGPU_NUM_CHIPS];            // by chip
    std::vector<DevChip> devchips;
    std::vector<uint64_t> best;                            // per proof: smallest failing slot found on the host
};

// Runs the device checks and lowers best[] to the smallest failing slot of every proof.
int32_t run_batch(vgpu_ctx* ctx, const Batch& b, std::vector<uint64_t>* best);

}  // namespace vb
