// Keccak-f[1600] on 32-bit register pairs for sm_100a (LOP3 for theta/chi with D folded into a 3-input
// xor, SHF funnel shifts for rho; optional multiply-add rotations on the FMA pipe).
// Replaces tiny-keccak's keccakf as used by p3-keccak::Keccak256Hash inside
// SerializingHasher32 / CompressionFunctionFromHasher (basic/src/bin/valida.rs:367-371).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "bb.cuh"

namespace kk {

__constant__ uint2 RC[24] = {
    {0x00000001u, 0x00000000u}, {0x00008082u, 0x00000000u}, {0x0000808au, 0x80000000u}, {0x80008000u, 0x80000000u},
    {0x0000808bu, 0x00000000u}, {0x80000001u, 0x00000000u}, {0x80008081u, 0x80000000u}, {0x00008009u, 0x80000000u},
    {0x0000008au, 0x00000000u}, {0x00000088u, 0x00000000u}, {0x80008009u, 0x00000000u}, {0x8000000au, 0x00000000u},
    {0x8000808bu, 0x00000000u}, {0x0000008bu, 0x80000000u}, {0x00008089u, 0x80000000u}, {0x00008003u, 0x80000000u},
    {0x00008002u, 0x80000000u}, {0x00000080u, 0x80000000u}, {0x0000800au, 0x00000000u}, {0x8000000au, 0x80000000u},
    {0x80008081u, 0x80000000u}, {0x00008080u, 0x80000000u}, {0x80000001u, 0x00000000u}, {0x80008008u, 0x80000000u}};

// Powers of two as opaque constant-bank operands: rotations are issued as integer multiply-adds so
// that they run on the FMA pipe (idle in Keccak) instead of competing with LOP3 on the INT ALU pipe.
__constant__ uint32_t POW2[32] = {1u << 0, 1u << 1, 1u << 2, 1u << 3, 1u << 4, 1u << 5, 1u << 6, 1u << 7, 1u << 8, 1u << 9, 1u << 10, 1u << 11,
                                  1u << 12, 1u << 13, 1u << 14, 1u << 15, 1u << 16, 1u << 17, 1u << 18, 1u << 19, 1u << 20, 1u << 21, 1u << 22,
                                  1u << 23, 1u << 24, 1u << 25, 1u << 26, 1u << 27, 1u << 28, 1u << 29, 1u << 30, 1u << 31};

// 64-bit rotate-left of (lo = a.x, hi = a.y) by M in 1..31 with three multiply-adds:
//   W      = lo * 2^M                (W.lo = lo << M, W.hi = lo >> (32-M))
//   new_hi = hi * 2^M + W.hi         (disjoint bit ranges: + == |)
//   new_lo = hi32(hi * 2^M) + W.lo
template <int M> __device__ __forceinline__ uint2 rol_small(uint2 a) {
    const uint32_t p = POW2[M];
    uint32_t wlo, whi, nlo, nhi;
    asm("{\n\t.reg .u64 w;\n\tmul.wide.u32 w, %4, %6;\n\tmov.b64 {%0, %1}, w;\n\tmad.lo.u32 %3, %5, %6, %1;\n\tmad.hi.u32 %2, %5, %6, %0;\n\t}"
        : "=&r"(wlo), "=&r"(whi), "=r"(nlo), "=r"(nhi) : "r"(a.x), "r"(a.y), "r"(p));
    return make_uint2(nlo, nhi);
}
// x = lo, y = hi
// Rotation amounts listed in KK_FMA_ROT_MASK (bit n set = rotate-by-n uses the multiply-add form) go to the
// FMA pipe, the rest are SHF funnel shifts on the INT ALU pipe next to the LOP3s.  Measured on B200
// (profiles/r01_keccak_rot.md): the all-IMAD variant is 19% SLOWER than all-SHF, so the default mask is 0.
#ifndef KK_FMA_ROT_MASK
#define KK_FMA_ROT_MASK 0ull
#endif
template <int M> __device__ __forceinline__ uint2 rol_shf(uint2 a) {
    return make_uint2(__funnelshift_l(a.y, a.x, M), __funnelshift_l(a.x, a.y, M));
}
template <int N> __device__ __forceinline__ uint2 rol(uint2 a) {
    if (N == 0) return a;
    if (N == 32) return make_uint2(a.y, a.x);
    constexpr int M = (N & 31) ? (N & 31) : 1;
    const uint2 b = N < 32 ? a : make_uint2(a.y, a.x);
    if ((KK_FMA_ROT_MASK >> N) & 1ull) return rol_small<M>(b);
    return rol_shf<M>(b);
}
__device__ __forceinline__ uint2 x2(uint2 a, uint2 b) { return make_uint2(a.x ^ b.x, a.y ^ b.y); }
__device__ __forceinline__ uint2 x3(uint2 a, uint2 b, uint2 c) { return make_uint2(a.x ^ b.x ^ c.x, a.y ^ b.y ^ c.y); }
__device__ __forceinline__ uint2 x5(uint2 a, uint2 b, uint2 c, uint2 d, uint2 e) { return make_uint2(a.x ^ b.x ^ c.x ^ d.x ^ e.x, a.y ^ b.y ^ c.y ^ d.y ^ e.y); }
__device__ __forceinline__ uint2 chi(uint2 a, uint2 b, uint2 c) { return make_uint2(a.x ^ (~b.x & c.x), a.y ^ (~b.y & c.y)); }

// State lane (x, y) lives in A[x + 5 y].
__device__ __forceinline__ void keccak_round(uint2 A[25], const uint2 rc) {
    uint2 C0 = x5(A[0], A[5], A[10], A[15], A[20]);
    uint2 C1 = x5(A[1], A[6], A[11], A[16], A[21]);
    uint2 C2 = x5(A[2], A[7], A[12], A[17], A[22]);
    uint2 C3 = x5(A[3], A[8], A[13], A[18], A[23]);
    uint2 C4 = x5(A[4], A[9], A[14], A[19], A[24]);
    const uint2 R0 = rol<1>(C1), R1 = rol<1>(C2), R2 = rol<1>(C3), R3 = rol<1>(C4), R4 = rol<1>(C0);
    // D[x] = C[x-1] ^ rol(C[x+1], 1) is folded into the 3-input xor with the lane (one LOP3 per half)
    // theta + rho + pi:  B[y, 2x+3y] = rol(A[x,y] ^ D[x], r[x,y])
    uint2 B0 = x3(A[0], C4, R0);
    uint2 B10 = rol<1>(x3(A[1], C0, R1));
    uint2 B20 = rol<62>(x3(A[2], C1, R2));
    uint2 B5 = rol<28>(x3(A[3], C2, R3));
    uint2 B15 = rol<27>(x3(A[4], C3, R4));
    uint2 B16 = rol<36>(x3(A[5], C4, R0));
    uint2 B1 = rol<44>(x3(A[6], C0, R1));
    uint2 B11 = rol<6>(x3(A[7], C1, R2));
    uint2 B21 = rol<55>(x3(A[8], C2, R3));
    uint2 B6 = rol<20>(x3(A[9], C3, R4));
    uint2 B7 = rol<3>(x3(A[10], C4, R0));
    uint2 B17 = rol<10>(x3(A[11], C0, R1));
    uint2 B2 = rol<43>(x3(A[12], C1, R2));
    uint2 B12 = rol<25>(x3(A[13], C2, R3));
    uint2 B22 = rol<39>(x3(A[14], C3, R4));
    uint2 B23 = rol<41>(x3(A[15], C4, R0));
    uint2 B8 = rol<45>(x3(A[16], C0, R1));
    uint2 B18 = rol<15>(x3(A[17], C1, R2));
    uint2 B3 = rol<21>(x3(A[18], C2, R3));
    uint2 B13 = rol<8>(x3(A[19], C3, R4));
    uint2 B14 = rol<18>(x3(A[20], C4, R0));
    uint2 B24 = rol<2>(x3(A[21], C0, R1));
    uint2 B9 = rol<61>(x3(A[22], C1, R2));
    uint2 B19 = rol<56>(x3(A[23], C2, R3));
    uint2 B4 = rol<14>(x3(A[24], C3, R4));
    // chi
    A[0] = chi(B0, B1, B2); A[1] = chi(B1, B2, B3); A[2] = chi(B2, B3, B4); A[3] = chi(B3, B4, B0); A[4] = chi(B4, B0, B1);
    A[5] = chi(B5, B6, B7); A[6] = chi(B6, B7, B8); A[7] = chi(B7, B8, B9); A[8] = chi(B8, B9, B5); A[9] = chi(B9, B5, B6);
    A[10] = chi(B10, B11, B12); A[11] = chi(B11, B12, B13); A[12] = chi(B12, B13, B14); A[13] = chi(B13, B14, B10); A[14] = chi(B14, B10, B11);
    A[15] = chi(B15, B16, B17); A[16] = chi(B16, B17, B18); A[17] = chi(B17, B18, B19); A[18] = chi(B18, B19, B15); A[19] = chi(B19, B15, B16);
    A[20] = chi(B20, B21, B22); A[21] = chi(B21, B22, B23); A[22] = chi(B22, B23, B24); A[23] = chi(B23, B24, B20); A[24] = chi(B24, B20, B21);
    // iota
    A[0].x ^= rc.x; A[0].y ^= rc.y;
}

// FIRST: round 0 stands outside the loop, so lanes the caller set to literal zeros (the capacity, and most of the rate of a
// 64-byte compression) are folded away by the compiler.  LAST: round 23 stands outside the loop and the caller reads only
// A[0..3] (a 256-bit digest): chi / rho / pi of the other 21 lanes are dead code there.  Both leave the permutation's
// value unchanged — they only expose what the generic loop hides from the optimiser.
template <bool FIRST, bool LAST>
__device__ __forceinline__ void keccak_f_peeled(uint2 A[25]) {
    if (FIRST) keccak_round(A, make_uint2(0x00000001u, 0x00000000u));
#pragma unroll 1
    for (int round = FIRST ? 1 : 0; round < (LAST ? 23 : 24); round++) keccak_round(A, RC[round]);
    if (LAST) keccak_round(A, make_uint2(0x80008008u, 0x80000000u));
}
__device__ __forceinline__ void keccak_f(uint2 A[25]) { keccak_f_peeled<false, false>(A); }

// ---- SerializingHasher32<Keccak256Hash> and CompressionFunctionFromHasher<_, _, 2, 8> over canonical words (the Merkle trees of
// merkle.cu and the paths the batch verifier walks in verify_batch.cu) ------------------------------------------------------------------
constexpr int RATE_WORDS = 34;   // 136-byte rate

// Sponge over `nwords` canonical words fetched by `fetch(i)`; Keccak pad 0x01 .. 0x80.
template <bool SHORT = false, class Fetch>
__device__ __forceinline__ void keccak256_words(const uint32_t nwords, Fetch fetch, uint32_t out[8]) {
    uint2 A[25];
#pragma unroll
    for (int i = 0; i < 25; i++) A[i] = make_uint2(0, 0);
    uint32_t nblocks = nwords / RATE_WORDS + 1;
    if (SHORT) {   // a single block whose length the compiler sees (64-byte compression, FRI leaf): zero lanes fold away in round 0
#pragma unroll
        for (int i = 0; i < RATE_WORDS / 2; i++) {
            const uint32_t g0 = 2 * i, g1 = g0 + 1;
            uint32_t w0 = g0 < nwords ? fetch(g0) : (g0 == nwords ? 1u : 0u);
            uint32_t w1 = g1 < nwords ? fetch(g1) : (g1 == nwords ? 1u : 0u);
            if (i == RATE_WORDS / 2 - 1) w1 ^= 0x80000000u;
            A[i] = make_uint2(w0, w1);
        }
        kk::keccak_f_peeled<true, true>(A);
        out[0] = A[0].x; out[1] = A[0].y; out[2] = A[1].x; out[3] = A[1].y;
        out[4] = A[2].x; out[5] = A[2].y; out[6] = A[3].x; out[7] = A[3].y;
        return;
    }
    for (uint32_t b = 0; b < nblocks; b++) {
        uint32_t base = b * RATE_WORDS;
#pragma unroll
        for (int i = 0; i < RATE_WORDS / 2; i++) {
            uint32_t g0 = base + 2 * i, g1 = g0 + 1;
            uint32_t w0 = g0 < nwords ? fetch(g0) : (g0 == nwords ? 1u : 0u);
            uint32_t w1 = g1 < nwords ? fetch(g1) : (g1 == nwords ? 1u : 0u);
            if (i == RATE_WORDS / 2 - 1 && b == nblocks - 1) w1 ^= 0x80000000u;
            A[i].x ^= w0; A[i].y ^= w1;
        }
        if (b == nblocks - 1) kk::keccak_f_peeled<false, true>(A); else kk::keccak_f(A);
    }
    out[0] = A[0].x; out[1] = A[0].y; out[2] = A[1].x; out[3] = A[1].y;
    out[4] = A[2].x; out[5] = A[2].y; out[6] = A[3].x; out[7] = A[3].y;
}

__device__ __forceinline__ uint32_t wrap_mod_p(uint32_t w) {   // F::from_wrapped_u32
    w = bb::umin32(w, w - bb::P);
    return bb::umin32(w, w - bb::P);
}

__device__ __forceinline__ void compress_pair(const uint32_t l[8], const uint32_t r[8], uint32_t out[8]) {
    uint32_t d[8];
    keccak256_words<true>(16, [&](uint32_t i) { return i < 8 ? l[i] : r[i - 8]; }, d);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = wrap_mod_p(d[i]);
}

}  // namespace kk
