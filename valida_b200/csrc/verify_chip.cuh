// Out-of-domain constraint check of ONE chip as a single host/device function: the text behind both vgpu_verify (verify.cu, host)
// and the batch verifier (verify_batch.cu, one thread per (proof, chip)).
// Replaces verify_constraints (machine/src/verify.rs:11-107) with its VerifierConstraintFolder
// (machine/src/folding_builder.rs:127-220): the opened trace / permutation / quotient values at zeta are pushed through the SAME
// Air::eval text the device quotient sweep uses (airs.cuh, value type X = degree-5 extension) and through
// eval_permutation_constraints (machine/src/chip.rs:210-289); the folded sum must equal Z_H(zeta) * quotient(zeta).
// Every opened value is read through a pointer (host vectors or global memory) and no per-thread array is indexed at run time,
// so the device instantiation keeps no local-memory frame.
#pragma once
#include "airs.cuh"
#include "devchip.h"

namespace vchip {

using bb::E5;
using air::X;

struct VerifierFolder {
    using V = X;
    const E5* lrow; const E5* nrow;
    X first, last, trans;
    E5 alpha, acc;
    BB_HD X L(int c) const { return X{lrow[c]}; }
    BB_HD X N(int c) const { return X{nrow[c]}; }
    BB_HD void z(const X& x) { acc = bb::e5_add(bb::e5_mul(acc, alpha), x.e); }   // Horner, folding_builder.rs:196-200
    BB_HD void z_ext(const E5& x) { acc = bb::e5_add(bb::e5_mul(acc, alpha), x); }
};

// VirtualPairCol::apply over extension-valued rows (p3_air::VirtualPairCol; machine/src/chip.rs:76-80)
BB_HD bool pair_col_ext(const DevPairCol& pc, const E5* main_row, E5* out) {
    E5 v = bb::e5_from_base(pc.constant);
    for (uint32_t t = 0; t < pc.n_terms; t++) {
        if (pc.is_prep[t]) return false;   // the reference never opens the preprocessed commitment (derive/src/lib.rs:379-392)
        v = bb::e5_add(v, bb::e5_mul_base(main_row[pc.column[t]], pc.weight[t]));
    }
    *out = v;
    return true;
}

// sum_l v[5m + l] * X^l : the opened flattened columns of one extension column back to one extension value
BB_HD E5 unflatten(const E5* v, uint32_t m) {
    E5 s = bb::e5_zero();
    for (int l = 0; l < 5; l++) {
        E5 mono = bb::e5_zero();
        mono.c[l] = bb::R1;
        s = bb::e5_add(s, bb::e5_mul(v[5 * m + l], mono));
    }
    return s;
}

// The opened values of one ChipProof (machine/src/proof.rs:27-37), Montgomery limbs: trace_local / trace_next hold chip width
// values, perm_local / perm_next 5 (n_interactions + 1), quotient_chunks 10.  The caller checks those counts.
struct ChipOpenedView { const E5 *trace_local, *trace_next, *perm_local, *perm_next, *quotient_chunks; };

enum { CHIP_REJECT = 0, CHIP_ACCEPT = 1, CHIP_READS_PREPROCESSED = -1 };

// CHIP_ACCEPT when the folded constraints at zeta equal Z_H(zeta) * quotient(zeta), CHIP_REJECT when they do not (or when zeta is
// a point of the trace domain's selectors), CHIP_READS_PREPROCESSED when an interaction reads a preprocessed column (never for
// BasicMachine; the proof does not open that commitment).
template <int CHIP>
BB_HD int chip_constraints(const DevChip& dc, uint32_t log_degree, const ChipOpenedView& ov, const E5& cumulative_sum, const E5& zeta, const E5& alpha) {
    const uint32_t k = dc.n_interactions;
    const uint32_t g_inv = bb::inv(bb::two_adic_generator_monty((int)log_degree));
    const E5 z_h = bb::e5_sub_base(bb::e5_exp_pow2(zeta, (int)log_degree), bb::R1);
    const E5 zm1 = bb::e5_sub_base(zeta, bb::R1), zmg = bb::e5_sub_base(zeta, g_inv);
    if (bb::e5_is_zero(zm1) || bb::e5_is_zero(zmg)) return CHIP_REJECT;
    VerifierFolder f;
    f.lrow = ov.trace_local; f.nrow = ov.trace_next;
    f.first = X{bb::e5_mul(z_h, bb::e5_inv(zm1))};
    f.last = X{bb::e5_mul(z_h, bb::e5_inv(zmg))};
    f.trans = X{zmg};
    f.alpha = alpha; f.acc = bb::e5_zero();
    air::eval_chip<CHIP>(f);
    {   // eval_permutation_constraints
        E5 rhs = bb::e5_zero(), phi0 = bb::e5_zero();
        for (uint32_t m = 0; m < k; m++) {
            const DevInteraction& it = dc.interactions[m];
            const E5 pl = unflatten(ov.perm_local, m), pn = unflatten(ov.perm_next, m);
            E5 rlc = it.alpha;
            for (uint32_t j = 0; j < it.n_fields; j++) {
                E5 e;
                if (!pair_col_ext(it.fields[j], f.lrow, &e)) return CHIP_READS_PREPROCESSED;
                rlc = bb::e5_add(rlc, bb::e5_mul(dc.betas[j], e));
            }
            f.z_ext(bb::e5_sub_base(bb::e5_mul(rlc, pl), bb::R1));
            E5 mult_l, mult_n;
            if (!pair_col_ext(it.count, f.lrow, &mult_l) || !pair_col_ext(it.count, f.nrow, &mult_n)) return CHIP_READS_PREPROCESSED;
            const E5 tl = bb::e5_mul(pl, mult_l), tn = bb::e5_mul(pn, mult_n);
            if (it.is_send) { phi0 = bb::e5_add(phi0, tl); rhs = bb::e5_add(rhs, tn); }
            else { phi0 = bb::e5_sub(phi0, tl); rhs = bb::e5_sub(rhs, tn); }
        }
        const E5 plk = unflatten(ov.perm_local, k), pnk = unflatten(ov.perm_next, k);
        f.z_ext(bb::e5_mul(f.trans.e, bb::e5_sub(bb::e5_sub(pnk, plk), rhs)));
        f.z_ext(bb::e5_mul(f.first.e, bb::e5_sub(plk, phi0)));
        f.z_ext(bb::e5_mul(f.last.e, bb::e5_sub(plk, cumulative_sum)));
    }
    // quotient(zeta) = chunk_0(zeta^2) + zeta * chunk_1(zeta^2)   (log_quotient_degree = 1)
    const E5 quot = bb::e5_add(unflatten(ov.quotient_chunks, 0), bb::e5_mul(unflatten(ov.quotient_chunks, 1), zeta));
    const E5 want = bb::e5_mul(z_h, quot);
    bool same = true;
    for (int l = 0; l < 5; l++) same = same && (want.c[l] == f.acc.c[l]);
    return same ? CHIP_ACCEPT : CHIP_REJECT;
}

// chip_constraints for a chip id known only at run time (host)
inline int chip_constraints_any(const DevChip& dc, uint32_t log_degree, const ChipOpenedView& ov, const E5& cumulative_sum, const E5& zeta, const E5& alpha) {
    switch (dc.chip_id) {
#define VCHIP_CASE(c) case c: return chip_constraints<c>(dc, log_degree, ov, cumulative_sum, zeta, alpha);
        VCHIP_CASE(0) VCHIP_CASE(1) VCHIP_CASE(2) VCHIP_CASE(3) VCHIP_CASE(4) VCHIP_CASE(5) VCHIP_CASE(6)
        VCHIP_CASE(7) VCHIP_CASE(8) VCHIP_CASE(9) VCHIP_CASE(10) VCHIP_CASE(11) VCHIP_CASE(12) VCHIP_CASE(13)
#undef VCHIP_CASE
        default: return chip_constraints<1>(dc, log_degree, ov, cumulative_sum, zeta, alpha);   // empty eval, as before
    }
}

}  // namespace vchip
