// K3/K4 — Keccak-256 Merkle commitment over mixed-height column-major LDE matrices (sm_100a).
// Replaces FieldMerkleTreeMmcs<BabyBear, SerializingHasher32<Keccak256Hash>,
// CompressionFunctionFromHasher<_,_,2,8>, 8>::commit (basic/src/bin/valida.rs:367-374) as reached
// from TwoAdicFriPcs::commit_shifted_batches (derive/src/lib.rs:309,330,355,372).
//  * leaf kernel: one thread per LDE row; the row of every matrix of that height is streamed from
//    the column-major store (coalesced across the warp), converted Montgomery -> canonical, absorbed
//    little-endian into a register-resident 1600-bit state; digest words are reduced mod p;
//  * node kernel: one thread per parent, 64-byte compression (one permutation), with the
//    "inject shorter matrices" rule: node = compress(compress(l, r), hash(rows at that height)).
//  * short layers (<= 2^15 nodes): tree_tail_kernel reduces a sub-tree per CTA in shared memory, a thread per node while a level is
//    wide, a warp per node (the Keccak state spread over 25 lanes) on the last levels, where only the dependent chain is left.
// Digests are stored canonical, 8 words (32 B) per node, all layers kept for the opening phase.  Split proof (merkle.h): a rank
// computes and keeps its run of every layer — the sub-tree over its rows — and only the layer of comm_size sub-roots is all-gathered.
#include "ctx.h"
#include "keccak.cuh"
#include "merkle.h"
#include <algorithm>
#include <cstdlib>
#include <numeric>

namespace {

using kk::keccak256_words;
using kk::wrap_mod_p;
using kk::compress_pair;

// colptr[i] = device pointer to column i of the concatenated row (all matrices of this height).
// rows [row0, row0 + nrows) of the layer (a rank's share when the tree is split across GPUs)
__global__ void __launch_bounds__(128) leaf_hash_kernel(const uint32_t* const* __restrict__ colptr, uint32_t nwords, uint64_t row0, uint64_t nrows, uint32_t* __restrict__ digests) {
    uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    r += row0;
    uint32_t d[8];
    keccak256_words(nwords, [&](uint32_t i) { return bb::from_monty(__ldg(colptr[i] + r)); }, d);
    uint4* o = reinterpret_cast<uint4*>(digests + r * 8);
    o[0] = make_uint4(wrap_mod_p(d[0]), wrap_mod_p(d[1]), wrap_mod_p(d[2]), wrap_mod_p(d[3]));
    o[1] = make_uint4(wrap_mod_p(d[4]), wrap_mod_p(d[5]), wrap_mod_p(d[6]), wrap_mod_p(d[7]));
}

// next[i] = compress(prev[2i], prev[2i+1]) ; if inject != null: next[i] = compress(next[i], inject[i])
// parents [i0, i0 + n_next) of the layer
__global__ void __launch_bounds__(128) compress_layer_kernel(const uint32_t* __restrict__ prev, const uint32_t* __restrict__ inject, uint64_t i0, uint64_t n_next, uint32_t* __restrict__ next) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_next) return;
    i += i0;
    uint32_t l[8], r[8], o[8];
    const uint4* p = reinterpret_cast<const uint4*>(prev + i * 16);
    uint4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), d = __ldg(p + 3);
    l[0] = a.x; l[1] = a.y; l[2] = a.z; l[3] = a.w; l[4] = b.x; l[5] = b.y; l[6] = b.z; l[7] = b.w;
    r[0] = c.x; r[1] = c.y; r[2] = c.z; r[3] = c.w; r[4] = d.x; r[5] = d.y; r[6] = d.z; r[7] = d.w;
    compress_pair(l, r, o);
    if (inject) {
        const uint4* q = reinterpret_cast<const uint4*>(inject + i * 8);
        uint4 e = __ldg(q), f = __ldg(q + 1);
        uint32_t t[8] = {e.x, e.y, e.z, e.w, f.x, f.y, f.z, f.w};
        uint32_t o2[8];
        compress_pair(o, t, o2);
#pragma unroll
        for (int k = 0; k < 8; k++) o[k] = o2[k];
    }
    uint4* w = reinterpret_cast<uint4*>(next + i * 8);
    w[0] = make_uint4(o[0], o[1], o[2], o[3]);
    w[1] = make_uint4(o[4], o[5], o[6], o[7]);
}

// ---- Keccak-f[1600] spread over the lanes of a warp ------------------------------------------------------------------------------
// For the last few layers of a tree there is nothing to run in parallel: a layer of n <= 32 nodes is n chains of 24 dependent rounds,
// and a lone thread needs ~5.5 us for one (4166 instructions, one warp per scheduler).  Here lane t = x + 5y of a warp holds lane
// A[x, y] of ONE state: a round is 18 shuffles and ~25 ALU instructions per lane (theta: column parity by four shuffles, D by two;
// rho: a per-lane rotation amount; pi: one shuffle; chi: two), ~140 cycles of latency — about a third of the lone thread's chain.
__constant__ uint8_t WK_ROT[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};   // r[x + 5y]
struct WarpKeccak {
    uint32_t rot, col[4], dm, dp, pi, c1, c2, lane;
    __device__ __forceinline__ void init(uint32_t lane_) {
        lane = lane_;
        const uint32_t t = lane < 25 ? lane : 0, x = t % 5, y = t / 5;
        rot = WK_ROT[t];
#pragma unroll
        for (int k = 0; k < 4; k++) col[k] = (t + 5 * (k + 1)) % 25;
        dm = (x + 4) % 5 + 5 * y; dp = (x + 1) % 5 + 5 * y;
        pi = (x + 3 * y) % 5 + 5 * x;                 // B[x, y] comes from A[(x + 3y) mod 5, x]
        c1 = (x + 1) % 5 + 5 * y; c2 = (x + 2) % 5 + 5 * y;
    }
    static __device__ __forceinline__ uint2 sh(uint2 v, uint32_t src) { return make_uint2(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src)); }
    __device__ __forceinline__ void permute(uint2& a) const {
#pragma unroll 1
        for (int round = 0; round < 24; round++) {
            uint2 p = a;
#pragma unroll
            for (int k = 0; k < 4; k++) { const uint2 o = sh(a, col[k]); p.x ^= o.x; p.y ^= o.y; }
            const uint2 pm = sh(p, dm), pp = sh(p, dp);
            a.x ^= pm.x ^ __funnelshift_l(pp.y, pp.x, 1); a.y ^= pm.y ^ __funnelshift_l(pp.x, pp.y, 1);
            uint32_t lo = a.x, hi = a.y;
            if (rot & 32) { const uint32_t tmp = lo; lo = hi; hi = tmp; }
            uint2 b = make_uint2(__funnelshift_l(hi, lo, rot & 31), __funnelshift_l(lo, hi, rot & 31));
            b = sh(b, pi);
            const uint2 b1 = sh(b, c1), b2 = sh(b, c2);
            a.x = b.x ^ (~b1.x & b2.x); a.y = b.y ^ (~b1.y & b2.y);
            if (lane == 0) { const uint2 rc = kk::RC[round]; a.x ^= rc.x; a.y ^= rc.y; }
            if (lane >= 25) a = make_uint2(0, 0);
        }
    }
    // 64-byte compression: lanes 0..7 hold the sixteen input words (2 each); on return lanes 0..3 hold the digest words, reduced mod p
    __device__ __forceinline__ uint2 compress(uint2 words) const {
        uint2 a = lane < 8 ? words : lane == 8 ? make_uint2(1u, 0u) : lane == 16 ? make_uint2(0u, 0x80000000u) : make_uint2(0u, 0u);
        permute(a);
        return make_uint2(wrap_mod_p(a.x), wrap_mod_p(a.y));
    }
};

// The short layers of a tree in ONE launch: a CTA owns `sub` consecutive nodes of the first fused layer and reduces that sub-tree
// level by level in shared memory (each level is written to its place in global memory as well), so the 10 - 16 launches of a tree's
// tail — each a handful of warps waiting on a single Keccak-f — become one or two.  Levels of more than 32 nodes take a thread per
// node; the narrower ones a WARP per node (WarpKeccak), which shortens the dependent chain that is all that is left there.
// Bases are virtual (+ global node index), as in compress_layer_kernel; inj_v[k] = digests of the rows a shorter matrix group
// contributes at fused level k, or null.
constexpr int TAIL_SUB = 256, TAIL_THREADS = 512, TAIL_MAX_LEVELS = 9, TAIL_WARP_NODES = 32;
struct TailParams {
    const uint32_t* prev_v;
    uint32_t* next_v[TAIL_MAX_LEVELS];
    const uint32_t* inj_v[TAIL_MAX_LEVELS];
    uint64_t first_begin;     // first node of the first fused layer computed by this launch
    uint32_t sub;             // nodes of the first fused layer per CTA (power of two <= TAIL_SUB)
    uint32_t levels;          // fused levels: level k has sub >> k nodes per CTA
};
__global__ void __launch_bounds__(TAIL_THREADS) tree_tail_kernel(const __grid_constant__ TailParams p) {
    __shared__ uint4 buf_a[2 * TAIL_SUB * 2];     // children of the current level: 2 * sub digests (two uint4 each)
    __shared__ uint4 buf_b[TAIL_SUB * 2];
    const uint64_t node0 = p.first_begin + (uint64_t)blockIdx.x * p.sub;
    {
        const uint4* src = reinterpret_cast<const uint4*>(p.prev_v + 2 * node0 * 8);
        for (uint32_t i = threadIdx.x; i < 4 * p.sub; i += TAIL_THREADS) buf_a[i] = __ldg(src + i);
    }
    __syncthreads();
    WarpKeccak wk;
    wk.init(threadIdx.x & 31);
    uint4* cur = buf_a; uint4* nxt = buf_b;
    for (uint32_t k = 0; k < p.levels; k++) {
        const uint32_t n = p.sub >> k;
        const uint64_t base = node0 >> k;
        if (n > TAIL_WARP_NODES) {
            for (uint32_t t = threadIdx.x; t < n; t += TAIL_THREADS) {
                const uint4 a = cur[4 * t], b = cur[4 * t + 1], c = cur[4 * t + 2], d = cur[4 * t + 3];
                uint32_t l[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}, r[8] = {c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w}, o[8];
                compress_pair(l, r, o);
                if (p.inj_v[k]) {
                    const uint4* q = reinterpret_cast<const uint4*>(p.inj_v[k] + (base + t) * 8);
                    const uint4 e = __ldg(q), f = __ldg(q + 1);
                    uint32_t tt[8] = {e.x, e.y, e.z, e.w, f.x, f.y, f.z, f.w}, o2[8];
                    compress_pair(o, tt, o2);
#pragma unroll
                    for (int i = 0; i < 8; i++) o[i] = o2[i];
                }
                const uint4 w0 = make_uint4(o[0], o[1], o[2], o[3]), w1 = make_uint4(o[4], o[5], o[6], o[7]);
                nxt[2 * t] = w0; nxt[2 * t + 1] = w1;
                uint4* g = reinterpret_cast<uint4*>(p.next_v[k] + (base + t) * 8);
                g[0] = w0; g[1] = w1;
            }
        } else {
            const uint32_t lane = threadIdx.x & 31;
            for (uint32_t t = threadIdx.x >> 5; t < n; t += TAIL_THREADS / 32) {      // a warp per node
                const uint2* in = reinterpret_cast<const uint2*>(cur + 4 * t);         // 16 words = 8 uint2
                uint2 dg = wk.compress(lane < 8 ? in[lane] : make_uint2(0, 0));        // lanes 0..3: the digest
                if (p.inj_v[k]) {
                    const uint2* q = reinterpret_cast<const uint2*>(p.inj_v[k] + (base + t) * 8);
                    const uint2 w = lane < 4 ? dg : (lane < 8 ? __ldg(q + (lane - 4)) : make_uint2(0, 0));
                    dg = wk.compress(w);
                }
                if (lane < 4) {
                    reinterpret_cast<uint2*>(nxt + 2 * t)[lane] = dg;
                    reinterpret_cast<uint2*>(p.next_v[k] + (base + t) * 8)[lane] = dg;
                }
            }
        }
        __syncthreads();
        uint4* tmp = cur; cur = nxt; nxt = tmp;
    }
}

// FRI commit-phase leaf: the pair (v[2i], v[2i+1]) of ext5 values flattened to 10 base words
// (ExtensionMmcs over a width-2 matrix); v is limb-major: limb l of element e at v[l * cs + e].
__global__ void __launch_bounds__(128) fri_leaf_hash_kernel(const uint32_t* __restrict__ v, uint64_t cs, uint64_t i0, uint64_t npairs, uint32_t* __restrict__ digests) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs) return;
    i += i0;
    uint32_t w[10];
#pragma unroll
    for (int l = 0; l < 5; l++) {
        uint2 t = __ldg(reinterpret_cast<const uint2*>(v + (uint64_t)l * cs + 2 * i));
        w[l] = bb::from_monty(t.x); w[5 + l] = bb::from_monty(t.y);
    }
    uint32_t d[8];
    keccak256_words<true>(10, [&](uint32_t k) { return w[k]; }, d);
    uint4* o = reinterpret_cast<uint4*>(digests + i * 8);
    o[0] = make_uint4(wrap_mod_p(d[0]), wrap_mod_p(d[1]), wrap_mod_p(d[2]), wrap_mod_p(d[3]));
    o[1] = make_uint4(wrap_mod_p(d[4]), wrap_mod_p(d[5]), wrap_mod_p(d[6]), wrap_mod_p(d[7]));
}

}  // namespace

// ---- host side: layer plan, launches --------------------------------------------------------------------------
// Layer plan of a tree over `leaves` leaves (merkle.h): which run of every layer this rank computes and which it keeps.
struct LayerPlan { uint64_t len, cbegin, ccount, sbegin, scount; bool gather; };
static std::vector<LayerPlan> plan_tree(const vgpu_ctx* ctx, uint64_t leaves, bool split) {
    const uint64_t G = split ? (uint64_t)ctx->comm_size : 1, r = split ? (uint64_t)ctx->comm_rank : 0;
    std::vector<LayerPlan> plan;
    for (uint64_t len = leaves; len >= 1; len >>= 1) {
        LayerPlan p{};
        p.len = len;
        if (G > 1 && len >= G) { p.ccount = len / G; p.cbegin = r * p.ccount; } else { p.cbegin = 0; p.ccount = len; }
        if (G > 1 && len > G) { p.sbegin = p.cbegin; p.scount = p.ccount; } else { p.sbegin = 0; p.scount = len; }
        p.gather = G > 1 && len == G;          // the sub-roots: one node per rank, completed by the all-gather
        plan.push_back(p);
        if (len == 1) break;
    }
    return plan;
}
static int32_t alloc_tree(vgpu_ctx* ctx, const std::vector<LayerPlan>& plan, VgTree* t) {
    uint64_t total = 0;
    for (auto& p : plan) total += p.scount;
    VG_TRY(vg_alloc(ctx, (void**)&t->digests, total * 32));
    t->layer_ptr.clear(); t->layer_len.clear(); t->layer_begin.clear(); t->layer_count.clear();
    uint32_t* at = t->digests;
    for (auto& p : plan) { t->layer_ptr.push_back(at); t->layer_len.push_back(p.len); t->layer_begin.push_back(p.sbegin); t->layer_count.push_back(p.scount); at += p.scount * 8; }
    return 0;
}
void vg_tree_free(vgpu_ctx* ctx, VgTree* t) { vg_free(ctx, t->digests); t->digests = nullptr; }

// digest of rows [row0, row0 + nrows) of the concatenated matrices, written to digests_v[row * 8] (digests_v is a VIRTUAL
// base: the stored run starts at its first row).  A row shard contributes its local rows through a base shifted likewise.
static int32_t hash_rows(vgpu_ctx* ctx, const std::vector<const vgpu_dmat*>& mats, uint64_t row0, uint64_t nrows, uint32_t* digests_v) {
    std::vector<const uint32_t*> cols;
    for (auto* m : mats) {
        if (m->dist == VG_ROWS && (row0 < m->row0 || row0 + nrows > m->row0 + m->h)) VG_FAIL(ctx, "commit: rows [%llu, +%llu) are not in this rank's shard", (unsigned long long)row0, (unsigned long long)nrows);
        for (uint64_t c = 0; c < m->w; c++) cols.push_back(m->d + c * m->col_stride - m->row0);
    }
    const uint32_t** dcols = nullptr;
    VG_TRY(vg_alloc(ctx, (void**)&dcols, cols.size() * sizeof(void*)));
    // cudaMemcpyAsync from pageable memory stages synchronously: `cols` may go once the call returns
    VG_CUDA(ctx, cudaMemcpyAsync(dcols, cols.data(), cols.size() * sizeof(void*), cudaMemcpyHostToDevice, ctx->stream));
    {
        KScope ks(ctx, KC_LEAF_HASH, (double)nrows * (4.0 * cols.size() + 32.0));
        leaf_hash_kernel<<<(unsigned)((nrows + 127) / 128), 128, 0, ctx->stream>>>(dcols, (uint32_t)cols.size(), row0, nrows, digests_v);
    }
    VG_LAUNCH_CHECK(ctx);
    vg_free(ctx, dcols);
    return 0;
}

// layers 1.. of a planned tree whose leaf layer is already hashed; inject(lvl, plan, inj_v, &have) fills the digests of the rows a
// shorter matrix group contributes at layer lvl.  Long layers take one launch each; from the first layer of at most TAIL_FUSE nodes
// (computed here) on, runs of up to 9 layers go into ONE launch of tree_tail_kernel; a run ends at the sub-root layer of a split tree
// (its all-gather comes next) and at the root.
constexpr uint64_t TAIL_FUSE = 1u << 15;
template <class Inject>
static int32_t build_upper_layers(vgpu_ctx* ctx, const std::vector<LayerPlan>& plan, VgTree* t, uint32_t* inject_buf, Inject inject) {
    if (plan[0].gather) VG_TRY(vg_comm_allgather_inplace(ctx, t->layer_ptr[0], 8));
    static const bool fuse = [] { const char* e = getenv("VGPU_TREE_TAIL"); return !e || atoi(e) != 0; }();   // tuning knob (profiles/)
    size_t lvl = 1;
    while (lvl < plan.size()) {
        const LayerPlan& p = plan[lvl];
        const uint32_t* prev_v = t->layer_ptr[lvl - 1] - plan[lvl - 1].sbegin * 8;
        if (fuse && p.ccount <= TAIL_FUSE) {
            // one launch: levels lvl .. lvl + n - 1, each half the one below; stop after a gather layer and at the root
            TailParams tp{};
            tp.prev_v = prev_v; tp.first_begin = p.cbegin;
            tp.sub = (uint32_t)std::min<uint64_t>(TAIL_SUB, p.ccount);
            uint32_t n = 0;
            uint32_t* inj_at = inject_buf;
            double bytes = 0;
            while (n < TAIL_MAX_LEVELS && lvl + n < plan.size() && (tp.sub >> n) >= 1) {
                const LayerPlan& q = plan[lvl + n];
                if (q.ccount != (p.ccount >> n) || q.cbegin != (p.cbegin >> n)) break;      // the run of halving layers ends (past a gather layer)
                tp.next_v[n] = t->layer_ptr[lvl + n] - q.sbegin * 8;
                tp.inj_v[n] = nullptr;
                if (inject_buf) {
                    uint32_t* buf_v = inj_at - q.cbegin * 8;
                    bool have = false;
                    VG_TRY(inject(lvl + n, q, buf_v, &have));
                    if (have) { tp.inj_v[n] = buf_v; inj_at += q.ccount * 8; }
                }
                bytes += (double)q.ccount * (tp.inj_v[n] ? 128.0 : 96.0);
                n++;
                if (q.gather) break;
            }
            tp.levels = n;
            {
                KScope ks(ctx, KC_COMPRESS, bytes);
                tree_tail_kernel<<<(unsigned)(p.ccount / tp.sub), TAIL_THREADS, 0, ctx->stream>>>(tp);
            }
            VG_LAUNCH_CHECK(ctx);
            lvl += n;
            if (plan[lvl - 1].gather) VG_TRY(vg_comm_allgather_inplace(ctx, t->layer_ptr[lvl - 1], 8));
            continue;
        }
        uint32_t* next_v = t->layer_ptr[lvl] - p.sbegin * 8;
        const uint32_t* inj_v = nullptr;
        if (inject_buf) {
            uint32_t* buf_v = inject_buf - p.cbegin * 8;
            bool have = false;
            VG_TRY(inject(lvl, p, buf_v, &have));
            if (have) inj_v = buf_v;
        }
        {
            KScope ks(ctx, KC_COMPRESS, (double)p.ccount * (inj_v ? 128.0 : 96.0));
            compress_layer_kernel<<<(unsigned)((p.ccount + 127) / 128), 128, 0, ctx->stream>>>(prev_v, inj_v, p.cbegin, p.ccount, next_v);
        }
        VG_LAUNCH_CHECK(ctx);
        if (p.gather) VG_TRY(vg_comm_allgather_inplace(ctx, t->layer_ptr[lvl], 8));
        lvl++;
    }
    return 0;
}

// Single-matrix tree over ext5 pairs (p3-fri commit phase).
int32_t vg_fri_layer_commit(vgpu_ctx* ctx, const uint32_t* v, uint64_t cs, uint64_t npairs, bool v_is_shard, VgTree* tree, uint32_t root_out[8]) {
    const std::vector<LayerPlan> plan = plan_tree(ctx, npairs, v_is_shard);
    VG_TRY(alloc_tree(ctx, plan, tree));
    const LayerPlan& l0 = plan[0];
    {
        // v holds the pairs of this rank's run when it is a shard (the run IS the computed run), all pairs otherwise
        const uint32_t* v_v = v_is_shard ? v - 2 * l0.cbegin : v;
        KScope ks(ctx, KC_FRI_LEAF, (double)l0.ccount * 72.0);
        fri_leaf_hash_kernel<<<(unsigned)((l0.ccount + 127) / 128), 128, 0, ctx->stream>>>(v_v, cs, l0.cbegin, l0.ccount, tree->layer_ptr[0] - l0.sbegin * 8);
    }
    VG_LAUNCH_CHECK(ctx);
    VG_TRY(build_upper_layers(ctx, plan, tree, nullptr, [](size_t, const LayerPlan&, uint32_t*, bool*) { return 0; }));
    VG_CUDA(ctx, cudaMemcpyAsync(root_out, tree->layer_ptr.back(), 32, cudaMemcpyDeviceToHost, ctx->stream));
    VG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// Build the mixed-height tree over the bit-reversed LDE matrices of `pd` (see merkle.h for `need`).
int32_t vg_merkle_build(vgpu_ctx* ctx, vgpu_prover_data* pd, const std::vector<uint64_t>& heights,
                        const std::function<int32_t(const std::vector<size_t>&)>& need) {
    size_t n = heights.size();
    if (!n) VG_FAIL(ctx, "commit: no matrices");
    std::vector<size_t> order(n);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return heights[a] > heights[b]; });
    uint64_t max_h = heights[order[0]];
    if (max_h & (max_h - 1)) VG_FAIL(ctx, "commit: heights must be powers of two");
    pd->max_height = max_h;
    const std::vector<LayerPlan> plan = plan_tree(ctx, max_h, vg_split_rows(ctx, max_h));
    VG_TRY(alloc_tree(ctx, plan, &pd->tree));
    size_t pos = 0;
    std::vector<size_t> idx;
    std::vector<const vgpu_dmat*> group;
    auto take = [&](uint64_t height) -> int32_t {   // the matrices of that height, extended on demand
        idx.clear(); group.clear();
        while (pos < n && heights[order[pos]] == height) idx.push_back(order[pos++]);
        if (idx.empty()) return 0;
        if (need) VG_TRY(need(idx));
        for (size_t i : idx) {
            if (!pd->ldes[i] || pd->ldes[i]->gh != height) VG_FAIL(ctx, "commit: matrix %zu was not extended to height %llu", i, (unsigned long long)height);
            group.push_back(pd->ldes[i]);
        }
        return 0;
    };
    VG_TRY(take(max_h));
    VG_TRY(hash_rows(ctx, group, plan[0].cbegin, plan[0].ccount, pd->tree.layer_ptr[0] - plan[0].sbegin * 8));
    uint32_t* inject_buf = nullptr;
    if (pos < n) {
        // one layer's row digests at a time — except inside a fused run of short layers, where the digests of every injecting
        // layer of the run (at most 2 * TAIL_FUSE in all) must coexist
        const uint64_t c1 = plan.size() > 1 ? plan[1].ccount : 1;
        VG_TRY(vg_alloc(ctx, (void**)&inject_buf, (c1 <= 2 * TAIL_FUSE ? 2 * c1 : c1) * 32));
    }
    int32_t rc = build_upper_layers(ctx, plan, &pd->tree, inject_buf, [&](size_t, const LayerPlan& p, uint32_t* buf_v, bool* have) -> int32_t {
        VG_TRY(take(p.len));
        *have = !group.empty();
        if (*have) VG_TRY(hash_rows(ctx, group, p.cbegin, p.ccount, buf_v));
        return 0;
    });
    if (inject_buf) vg_free(ctx, inject_buf);
    if (rc) return rc;
    if (pos != n) VG_FAIL(ctx, "commit: a matrix height does not match any tree layer");
    VG_CUDA(ctx, cudaMemcpyAsync(pd->root, pd->tree.layer_ptr.back(), 32, cudaMemcpyDeviceToHost, ctx->stream));
    VG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
