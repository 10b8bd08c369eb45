// Out-of-domain constraint check of ONE chip — the verifier's half of the AIR — for vgpu_verify.
// The folding itself is verify_chip.cuh (shared with the batch verifier's constraint kernel); this wrapper checks the counts of
// the opened values and folds the LogUp randomness into the chip description.  Host code (a few hundred extension
// multiplications per chip); it lives in a .cu file only because it instantiates the BB_HD templates of airs.cuh.
#include "ctx.h"
#include "devchip.h"
#include "verify_chip.cuh"
#include "verify.h"

int32_t vg_verify_chip_constraints(vgpu_ctx* ctx, const vgpu_chip_desc* chip, uint32_t log_degree, const VgChipOpening& ov,
                                   const bb::E5& cumulative_sum, const bb::E5& zeta, const bb::E5& alpha, const uint32_t perm_challenges[15], bool* ok) {
    *ok = false;
    const uint32_t pw = chip->n_interactions + 1;
    if (ov.trace_local.size() != chip->width || ov.trace_next.size() != chip->width) return 0;
    if (ov.perm_local.size() != 5 * pw || ov.perm_next.size() != 5 * pw || ov.quotient_chunks.size() != 10) return 0;
    DevChip dc;
    VG_TRY(vg_build_devchip(ctx, chip, perm_challenges, &dc));
    const vchip::ChipOpenedView view{ov.trace_local.data(), ov.trace_next.data(), ov.perm_local.data(), ov.perm_next.data(), ov.quotient_chunks.data()};
    const int r = vchip::chip_constraints_any(dc, log_degree, view, cumulative_sum, zeta, alpha);
    if (r == vchip::CHIP_READS_PREPROCESSED) VG_FAIL(ctx, "verify: an interaction reads a preprocessed column, which the proof does not open");
    *ok = r == vchip::CHIP_ACCEPT;
    return 0;
}
