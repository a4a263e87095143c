// bigclam_tile.cuh — the sparse-row step kernel: small nodes in TILES, the rest on the general path, and the
// deterministic reduction that follows every launch.
//
// Why tiles: com-amazon has a mean degree of 5.5 and rows of ~10 non-zeros — a warp that owns ONE such node
// spends most of its issue slots with 5 of 32 lanes busy (the one-warp-per-node kernels execute 2,900 warp
// instructions per node, see profiles/r2_sparse_warp_per_node_ncu.txt).  A tile is a run of up to 8 consecutive
// nodes of the degree-sorted processing order with at most 32 edges in total, handled by one warp; every phase
// maps its work items flat onto the 32 lanes:
//   stage   one bulk copy (cp.async.bulk.shared::cluster.global + mbarrier) per neighbour row and per own row;
//   PRE     lane = edge: x_e = fu . fv_e with fu looked up through the node's bitmask of non-zero components
//           (rank = popcount below the bit), exp/log once for 32 edges of up to 8 nodes;
//   slots   the components a node touches (its own and its neighbours' non-zeros) get consecutive slots in
//           ascending component order (bitmask + prefix popcounts): slot s holds (fu_c, grad_c);
//   axpy    lane groups of 32/nn lanes per node add w_e * fv_e into the slots, edge by edge (CSR order);
//   bounds  which (node, trial) pairs can pass the Armijo test at all (phase H2: a concavity bound on the node's objective
//           from the PRE quantities); on the bench workload 9 of 10 nodes have no such pair and keep their row;
//   LS      for the other nodes, two at a time, lane = (node, trial): dots over the ACTIVE entries only; (edge, trial)
//           pairs whose x is outside (x_lo, x_hi) are constants after the clamp (:166), the others are compacted and
//           exp/log runs on full warps of them;
//   decide  lane = (node, trial); swap: rows written by the node's lane group, one pool allocation per tile.
// A tile whose rows or touched components do not fit the warp's shared memory is processed node by node on the
// general path (SpGen) by the same warp; nodes above 32 edges always are.
#pragma once
#include "bigclam_sparse.cuh"

namespace bigclam {

constexpr int kTlMaxNodes = 8;
constexpr int kTlMaxEdges = 32;
#ifndef BIGCLAM_TL_STAGE16          // neighbour-row staging buffer of a tile, in 16-byte chunks (>= 256: it becomes xs[512])
#define BIGCLAM_TL_STAGE16 288
#endif
#ifndef BIGCLAM_TL_OWN16            // own-row staging buffer, in 16-byte chunks
#define BIGCLAM_TL_OWN16 80
#endif
#ifndef BIGCLAM_TL_SLOTS            // touched components of all nodes of a tile (>= 1.5 * BIGCLAM_TL_ACT)
#define BIGCLAM_TL_SLOTS 384
#endif
#ifndef BIGCLAM_TL_ACT              // active components of all nodes of a tile
#define BIGCLAM_TL_ACT 160
#endif
#ifndef BIGCLAM_TL_ENT              // neighbour entries on active components (>= 128: the pair list lives there later)
#define BIGCLAM_TL_ENT 224
#endif
#ifndef BIGCLAM_TL_EROW             // neighbour entries of a tile (flat entry -> row map)
#define BIGCLAM_TL_EROW 416
#endif
#ifndef BIGCLAM_TL_BULK             // 1: cp.async.bulk + mbarrier; 0: each lane copies its rows with 16-byte loads
#define BIGCLAM_TL_BULK 1
#endif
#ifndef BIGCLAM_TL_ILP2             // 1: the exp/log pass of the line search evaluates two pairs per lane (two independent chains)
#define BIGCLAM_TL_ILP2 1
#endif
#ifndef BIGCLAM_TL_UF               // unroll factor of the flat (lane-strided, uniform) loops over entries / slots / pairs
#define BIGCLAM_TL_UF 1
#endif
#ifndef BIGCLAM_TL_UJ               // unroll factor of the merged dot / decide loops
#define BIGCLAM_TL_UJ 1
#endif
#define BIGCLAM_PRAGMA(x) _Pragma(#x)
#define BIGCLAM_UNROLL(n) BIGCLAM_PRAGMA(unroll n)
#ifndef BIGCLAM_TL_WARPS
#define BIGCLAM_TL_WARPS 6
#endif
#ifndef BIGCLAM_TL_BLOCKS
#define BIGCLAM_TL_BLOCKS 2
#endif
constexpr int kTlStage16 = BIGCLAM_TL_STAGE16;
constexpr int kTlOwn16 = BIGCLAM_TL_OWN16;
constexpr int kTlSlots = BIGCLAM_TL_SLOTS;
constexpr int kTlAct = BIGCLAM_TL_ACT;
constexpr int kTlEnt = BIGCLAM_TL_ENT;
constexpr int kTlErow = BIGCLAM_TL_EROW;
constexpr int kTlWarps = BIGCLAM_TL_WARPS;
constexpr int kTlBlocksPerSM = BIGCLAM_TL_BLOCKS;
constexpr int kTlThreads = kTlWarps * 32;
static_assert(kTlStage16 >= 264, "the neighbour staging buffer doubles as xs[32 edges + 1 scratch row][16 trials]");
static_assert(2 * kTlSlots >= 3 * kTlAct, "fg must hold (f, g) and sumF - f of the active components after compaction");
static_assert(kTlEnt >= 128 && kTlEnt <= 256, "entry lists: the pair list (512 uint16) overlays ent_val; edge ids are bytes");
static_assert(kTlAct <= 255, "active-component ids of the entry lists are bytes");
static_assert(16 * kTlSlots >= 24 * kTlAct + 2 * 16 * kTlMaxEdges, "fg also holds sumF - f of the active components and the pair list of a line-search round");

// per-warp shared memory of the tile path (W = ldp / 32 mask words per node)
__host__ __device__ inline size_t tl_warp_bytes(int ld) {
    const size_t W = (size_t)sp_ldp(ld) / 32;
    size_t b = 16 * (size_t)kTlStage16;                 // stageN (later xs)
    b += 16 * (size_t)kTlOwn16;                         // stageO
    b += 16 * (size_t)kTlSlots;                         // fg (later fa | asfm)
    b += 8 * (size_t)kTlEnt;                            // ent_val
    b += 8 * 32 + 8 * 8 + 8 * 8;                        // we, n_llh, n_G2
    b += 4 * 2 * kTlMaxNodes * W + 4 * kTlMaxNodes;     // tmask, fmask, n_u
    b += 4 * (size_t)kTlAct;                            // lcnt
    b += 2 * 2 * (size_t)kTlSlots;                      // slot_c (later ac), amap
    b += 2 * ((size_t)kTlAct + 2);                      // loff
    b += 2 * 2 * kTlMaxNodes * W;                       // pref_t, pref_f
    b += 2 * (40 + 40 + 12 + 12 + 12 + 8 + 8);          // e_soff, e_cnt, n_es, n_sb, n_ab, n_m, n_tot
    b += 2 * 32;                                        // e_io2
    b += 2 * (size_t)kTlEnt + 8 + 8;                    // ent_e, ent_a, n_js, n_want
    b += (size_t)kTlErow + 2 * 34 + 32;                 // erow, epos, e_ni
    b += 2 * 8 + 8;                                     // n_sv, n_sl (line search by bounds)
    return (b + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t tl_region_bytes(int ld) {
    const size_t t = tl_warp_bytes(ld), g = (sp_gen_warp_bytes(ld) + 15) & ~(size_t)15;
    return t > g ? t : g;
}
// block: steps[kMaxSteps] | sumF[ldp] | mbar[kTlWarps] | wpb x warp region
__host__ __device__ inline size_t tl_block_smem_bytes(int ld, int wpb) {
    return sizeof(double) * (kMaxSteps + (size_t)sp_ldp(ld) + kTlWarps + 8) + (size_t)wpb * tl_region_bytes(ld);
}
// warps per block: as many resident warps per SM as the shared memory (227 KB, 1 KB reserved per block) allows, in
// at most kTlMaxBlocks blocks (wide rows run more blocks of fewer warps)
constexpr int kTlMaxBlocks = 4;
inline int tl_blocks_that_fit(int ld, int wpb) {
    const size_t bytes = tl_block_smem_bytes(ld, wpb) + 1024 + 256;
    const int blocks = (int)((size_t)233472 / bytes);
    const int cap = (wpb == kTlWarps) ? kTlBlocksPerSM : kTlMaxBlocks;      // the full-size block is built for kTlBlocksPerSM
    return blocks > cap ? cap : blocks;
}
inline int tl_warps_per_block(int ld) {
    int best = 1, best_warps = 0;
    for (int wpb = kTlWarps; wpb >= 1; --wpb) {
        const int warps = tl_blocks_that_fit(ld, wpb) * wpb;
        if (warps > best_warps) { best_warps = warps; best = wpb; }
    }
    return best;
}

// ---- mbarrier / bulk-copy primitives (host emulation: the copy happens at once) ----
#if defined(BIGCLAM_EMU)
__device__ __forceinline__ void mbar_init(unsigned long long *) {}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *, unsigned) {}
__device__ __forceinline__ void mbar_wait(unsigned long long *, unsigned) {}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *) { memcpy(dst, src, bytes); }
__device__ __forceinline__ void fence_proxy_async() {}
#else
__device__ __forceinline__ void mbar_init(unsigned long long *bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"((unsigned)__cvta_generic_to_shared(dst)),
                 "l"(src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#endif

struct TlWarp {
    const StepArgs *a;
    const SparseArgs *sp;
    const double *s_steps;
    const double *s_sumF;
    const float *s_lns;              // upper bounds of ln(step size) (line search by bounds)
    double S2_all;                   // sum_c sumF_c^2 (fixed order)
    EdgeConst ec;
    unsigned char *stageN, *stageO;
    double2 *fg;
    double *xs, *ent_val, *we, *n_llh, *n_G2;
    unsigned short *n_sv;
    unsigned char *n_sl;
    int last_ns, last_nw;            // nodes of the last tile that were line-searched / that wanted a line search
    unsigned long long *mbar;
    unsigned int *tmask, *fmask, *lcnt;
    int *n_u;
    unsigned short *slot_c, *amap, *loff, *plist, *pref_t, *pref_f, *e_soff, *e_cnt, *e_io2, *n_es, *n_sb, *n_ab, *n_m, *n_tot;
    unsigned char *ent_e, *ent_a, *erow, *e_ni, *n_want;
    unsigned short *epos;
    signed char *n_js;
    int lane, ld, W;
    unsigned parity;

    __device__ __forceinline__ void carve(unsigned char *p, int ld_, int lane_) {
        ld = ld_;
        lane = lane_;
        W = sp_ldp(ld_) / 32;
        parity = 0;
        stageN = p;                                       p += 16 * (size_t)kTlStage16;
        xs = reinterpret_cast<double *>(stageN);          // (after the rows have been turned into per-component lists)
        stageO = p;                                       p += 16 * (size_t)kTlOwn16;
        fg = reinterpret_cast<double2 *>(p);
        plist = reinterpret_cast<unsigned short *>(p + 24 * (size_t)kTlAct);   // (behind fa | asfm, after the compaction of the active components)
        p += 16 * (size_t)kTlSlots;
        ent_val = reinterpret_cast<double *>(p);          p += 8 * (size_t)kTlEnt;
        we = reinterpret_cast<double *>(p);               p += 8 * 32;
        n_llh = reinterpret_cast<double *>(p);            p += 8 * 8;
        n_G2 = reinterpret_cast<double *>(p);             p += 8 * 8;
        tmask = reinterpret_cast<unsigned int *>(p);      p += 4 * (size_t)kTlMaxNodes * W;
        fmask = reinterpret_cast<unsigned int *>(p);      p += 4 * (size_t)kTlMaxNodes * W;
        n_u = reinterpret_cast<int *>(p);                 p += 4 * kTlMaxNodes;
        lcnt = reinterpret_cast<unsigned int *>(p);       p += 4 * (size_t)kTlAct;
        slot_c = reinterpret_cast<unsigned short *>(p);   p += 2 * (size_t)kTlSlots;
        amap = reinterpret_cast<unsigned short *>(p);     p += 2 * (size_t)kTlSlots;
        loff = reinterpret_cast<unsigned short *>(p);     p += 2 * ((size_t)kTlAct + 2);
        pref_t = reinterpret_cast<unsigned short *>(p);   p += 2 * (size_t)kTlMaxNodes * W;
        pref_f = reinterpret_cast<unsigned short *>(p);   p += 2 * (size_t)kTlMaxNodes * W;
        e_soff = reinterpret_cast<unsigned short *>(p);   p += 2 * 40;
        e_cnt = reinterpret_cast<unsigned short *>(p);    p += 2 * 40;
        e_io2 = reinterpret_cast<unsigned short *>(p);    p += 2 * 32;     // flat entry t of row e: its index is stageN (as uint16) [(e_io2[e] + t) mod 2^16]
        n_es = reinterpret_cast<unsigned short *>(p);     p += 2 * 12;
        n_sb = reinterpret_cast<unsigned short *>(p);     p += 2 * 12;
        n_ab = reinterpret_cast<unsigned short *>(p);     p += 2 * 12;
        n_m = reinterpret_cast<unsigned short *>(p);      p += 2 * 8;
        n_tot = reinterpret_cast<unsigned short *>(p);    p += 2 * 8;
        epos = reinterpret_cast<unsigned short *>(p);     p += 2 * 34;
        ent_e = p;                                        p += (size_t)kTlEnt;
        ent_a = p;                                        p += (size_t)kTlEnt;
        erow = p;                                         p += (size_t)kTlErow;
        e_ni = p;                                         p += 32;
        n_js = reinterpret_cast<signed char *>(p);        p += 8;
        n_want = p;                                       p += 8;
        n_sl = p;                                         p += 8;
        n_sv = reinterpret_cast<unsigned short *>(p);
        last_ns = 0;
        last_nw = 0;
    }

    // inclusive scan over the lanes of a group of gs lanes (sub = lane within the group)
    __device__ __forceinline__ int group_scan(int v, int gs, int sub) const {
#pragma unroll 1
        for (int o = 1; o < gs; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, o);
            if (sub >= o) v += t;
        }
        return v;
    }
    template <class T>
    __device__ __forceinline__ T group_sum(T v, int gs) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            if (o < gs) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    }

    // One tile.  Returns false (nothing written) when the tile does not fit the warp's buffers.
    template <bool kPush>
    __device__ __forceinline__ bool run(const TileMeta tm) {
        const int nn = tm.nn, ne = tm.ne;
        const unsigned lt_mask = (1u << lane) - 1u;
        const uint64_t *__restrict__ hdr_in = sp->hdr_in;
        const double *__restrict__ pool_in = sp->pool_in;
        const bool do_ls = a->do_linesearch != 0;
        const int nsteps = a->nsteps;
        const double max_f = a->max_f;

        // ---------------- A. metadata, row headers, staging ----------------
        int ni = 0;
        uint64_t hv = 0ull, hu = 0ull;
        NodeMeta nm = {0, 0, 0};
        if (lane < ne) {
            const int t = sp->tcol[tm.ecol0 + lane];
            ni = (int)((unsigned)t >> 28);
            hv = __ldg(hdr_in + (t & 0x0fffffff));
        }
        if (lane < nn) {
            nm = a->meta[tm.pos0 + lane];
            hu = __ldg(hdr_in + nm.u);
        }
        const int ce = (int)sp_cnt(hv), cu = (int)sp_cnt(hu);
        const int qe = (int)(sp_words((uint32_t)ce) >> 1), qu = (int)(sp_words((uint32_t)cu) >> 1);     // 16-byte chunks
        // one scan for four counts: chunks of the neighbour rows (bits 0-11) and of the own rows (12-21), degrees (22-31
        // would overflow: separate), entries of the neighbour rows
        int incl_q = qe | (qu << 16), incl_d = nm.deg | (ce << 16), maxdeg = nm.deg;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t1 = __shfl_up_sync(0xffffffffu, incl_q, o);
            const int t3 = __shfl_up_sync(0xffffffffu, incl_d, o);
            const int t4 = __shfl_xor_sync(0xffffffffu, maxdeg, o);
            if (lane >= o) { incl_q += t1; incl_d += t3; }
            maxdeg = max(maxdeg, t4);
        }
        const int incl_e = incl_q & 0xffff, incl_u = incl_q >> 16, incl_c = incl_d >> 16;
        incl_d &= 0xffff;
        const int total_q = __shfl_sync(0xffffffffu, incl_q, 31);
        const int total_e = total_q & 0xffff, total_u = total_q >> 16;
        const int T = __shfl_sync(0xffffffffu, incl_c, 31);                 // neighbour entries of the tile
        if (total_e > kTlStage16 || total_u > kTlOwn16 || T > kTlErow) return false;
        const int soff_e = incl_e - qe, soff_u = incl_u - qu;
        if (lane < ne) {
            e_soff[lane] = (unsigned short)soff_e;
            e_cnt[lane] = (unsigned short)ce;
            e_io2[lane] = (unsigned short)(8 * soff_e + 4 * (int)sp_vpad((uint32_t)ce) - (incl_c - ce));
            epos[lane] = (unsigned short)(incl_c - ce);
            e_ni[lane] = (unsigned char)ni;
            if (lane == 0) epos[ne] = (unsigned short)T;
        }
        if (lane < nn) {
            e_soff[32 + lane] = (unsigned short)soff_u;
            e_cnt[32 + lane] = (unsigned short)cu;
            n_u[lane] = nm.u;
            n_es[lane] = (unsigned short)(incl_d - nm.deg);
            if (lane == nn - 1) n_es[nn] = (unsigned short)incl_d;
            const bool in_uset = (a->node_mask == nullptr) || (a->node_mask[nm.u] != 0);
            n_want[lane] = (unsigned char)(do_ls && in_uset && nm.deg > 0);
        }
#pragma unroll 1
        for (int i = lane; i < nn * W; i += 32) { tmask[i] = 0u; fmask[i] = 0u; }
#if BIGCLAM_TL_BULK
        if (total_e + total_u > 0) {
            fence_proxy_async();                         // this warp's earlier accesses to the buffers come first
            __syncwarp();
            if (lane == 0) mbar_expect_tx(mbar, 16u * (unsigned)(total_e + total_u));
            __syncwarp();
            if (qe > 0) bulk_g2s(stageN + 16 * (size_t)soff_e, pool_in + sp_off8(hv), 16u * (unsigned)qe, mbar);
            if (qu > 0) bulk_g2s(stageO + 16 * (size_t)soff_u, pool_in + sp_off8(hu), 16u * (unsigned)qu, mbar);
            mbar_wait(mbar, parity);
            parity ^= 1u;
        }
#else
        {
            const uint4 *se = reinterpret_cast<const uint4 *>(pool_in + sp_off8(hv));
            uint4 *de = reinterpret_cast<uint4 *>(stageN) + soff_e;
#pragma unroll 1
            for (int q = 0; q < qe; ++q) de[q] = __ldg(se + q);
            const uint4 *su = reinterpret_cast<const uint4 *>(pool_in + sp_off8(hu));
            uint4 *du = reinterpret_cast<uint4 *>(stageO) + soff_u;
#pragma unroll 1
            for (int q = 0; q < qu; ++q) du[q] = __ldg(su + q);
        }
#endif
        __syncwarp();

        // ---------------- B. own rows: masks of the non-zero components, fu.sumF, fu.fu ----------------
        const int lgs = nn <= 1 ? 5 : nn <= 2 ? 4 : nn <= 4 ? 3 : 2;          // lanes per node: 32 / pow2(nn)
        const int gs = 1 << lgs;
        const int g = lane >> lgs, sub = lane & (gs - 1);
        const bool gv = g < nn;
        const unsigned gmask = gs == 32 ? 0xffffffffu : ((1u << gs) - 1u);
        const unsigned below = (1u << sub) - 1u;
        const int gsh = g << lgs;
        const int gW = g * W;
        const int cu_g = gv ? (int)e_cnt[32 + g] : 0;
        double *ov = reinterpret_cast<double *>(stageO + 16 * (size_t)(gv ? e_soff[32 + g] : 0));
        unsigned short *oi = sp_idx(ov, (uint32_t)cu_g);
        double fusf = 0.0, fufu = 0.0;
#pragma unroll 1
        for (int i = sub; i < cu_g; i += gs) {
            const int c = oi[i];
            const double val = ov[i];
            atomicOr(fmask + gW + (c >> 5), 1u << (c & 31));
            fusf = fma(val, s_sumF[c], fusf);
            fufu = fma(val, val, fufu);
        }
        fusf = group_sum(fusf, gs);
        fufu = group_sum(fufu, gs);
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < nn * W; i += 32) tmask[i] = fmask[i];
        __syncwarp();
        // ---------------- C1. components the neighbours' rows touch ----------------
        double *rv = reinterpret_cast<double *>(stageN + 16 * (size_t)soff_e);
        unsigned short *ri = sp_idx(rv, (uint32_t)ce);
        if (lane < ne) {
            unsigned char *er = erow + (incl_c - ce);
#pragma unroll 1
            for (int i = 0; i < ce; ++i) er[i] = (unsigned char)lane;         // flat entry -> row
        }
        __syncwarp();
        unsigned short *stN16 = reinterpret_cast<unsigned short *>(stageN);
        // (from here on the loops over the neighbours' entries are FLAT: entry t of the tile = entry t - epos[row] of row erow[t])
BIGCLAM_UNROLL(BIGCLAM_TL_UF)
        for (int t = lane; t < T; t += 32) {
            const int row = erow[t];
            const int c = stN16[(unsigned short)(e_io2[row] + t)];
            atomicOr(tmask + (int)e_ni[row] * W + (c >> 5), 1u << (c & 31));
        }
        __syncwarp();
        // ---------------- E. slots of the touched components (ascending component order per node) ----------------
        int tot_g = 0;
        {
            int carry = 0;
#pragma unroll 1
            for (int w0 = 0; w0 < W; w0 += gs) {
                const int w = w0 + sub;
                const bool ok = gv && w < W;
                const int pc = ok ? __popc(tmask[gW + w]) : 0;
                const int incl = group_scan(pc, gs, sub);
                if (ok) pref_t[gW + w] = (unsigned short)(carry + incl - pc);
                carry += __shfl_sync(0xffffffffu, incl, gsh + gs - 1);
            }
            tot_g = gv ? carry : 0;
        }
        int base_g = 0, total_slots = 0;
#pragma unroll 1
        for (int q = 0; q < nn; ++q) {
            const int t = __shfl_sync(0xffffffffu, tot_g, q << lgs);
            if (q < g) base_g += t;
            total_slots += t;
        }
        if (total_slots > kTlSlots) return false;
        if (gv && sub == 0) { n_sb[g] = (unsigned short)base_g; n_tot[g] = (unsigned short)tot_g; }
#pragma unroll 1
        for (int i = lane; i < total_slots; i += 32) fg[i] = make_double2(0.0, 0.0);
        __syncwarp();
        // ---------------- C2. every entry learns its slot (kept in place of the component index) ----------------
#pragma unroll 1
        for (int i = sub; i < cu_g; i += gs) {
            const int c = oi[i];
            const int w = c >> 5;
            const unsigned bit = 1u << (c & 31);
            const int slot = base_g + pref_t[gW + w] + __popc(tmask[gW + w] & (bit - 1u));
            fg[slot].x = ov[i];
            slot_c[slot] = (unsigned short)c;
        }
BIGCLAM_UNROLL(BIGCLAM_TL_UF)
        for (int t = lane; t < T; t += 32) {
            const int row = erow[t];
            unsigned short *pc = stN16 + (unsigned short)(e_io2[row] + t);
            const int c = *pc;
            const int node = e_ni[row];
            const int w = c >> 5;
            const unsigned bit = 1u << (c & 31);
            const int slot = (int)n_sb[node] + pref_t[node * W + w] + __popc(tmask[node * W + w] & (bit - 1u));
            slot_c[slot] = (unsigned short)c;
            *pc = (unsigned short)slot;
        }
        __syncwarp();
        // ---------------- C3. PRE dots (:162-165), lane = edge ----------------
        double x = 0.0;
        if (lane < ne) {
#pragma unroll 1
            for (int i = 0; i < ce; ++i) x = fma(rv[i], fg[ri[i]].x, x);
        }
        // ---------------- D. edge terms (:166-167), llh_u (:168) ----------------
        double wgt;
        const double term = edge_term<true>(x, ec, wgt);
        we[lane] = wgt;
        // [bounds, see H2] an edge that is NOT clamped at MAX_P_ is bounded by its tangent (the clamped edge term is
        // concave from x_lo on) plus what the two clamps can add to it: below x_lo the term stops falling with the
        // tangent (at most S_lo - tangent(0)); above x_hi the coded slope w - 1 is not the slope of the flat term
        const bool prune_on = sp->ls_prune != 0;
        const bool e_low = x <= ec.x_lo;
        const float xf = (lane < ne) ? __double2float_ru(x) : 0.0f;
        float violf = 0.0f;              // above x_hi: a constant of the node's bound
        float vnear = 0.0f;              // in range, next to x_lo: only for candidates that can bring x' below x_lo (see H2)
        if (prune_on && !e_low && lane < ne) {
            const double m = wgt - 1.0;
            if (x < ec.x_hi) {
                const double v = fma(m, x, ec.t_lo - (term - x));
                vnear = (v > 0.0) ? __double2float_ru(v) * 1.000001f : 0.0f;
            } else {
                violf = __double2float_ru(m * (x - ec.x_hi)) * 1.000001f;
            }
        }
        const int es_g = gv ? (int)n_es[g] : 0;
        const int deg_g = gv ? (int)n_es[g + 1] - es_g : 0;
        double llh_g = 0.0;
        {
            double S1 = 0.0;
#pragma unroll 1
            for (int r = 0; r < maxdeg; ++r) {            // CSR order, like the reference's fold
                const double t = __shfl_sync(0xffffffffu, term, (es_g + r) & 31);
                if (r < deg_g) S1 += t;
            }
            llh_g = (S1 - fusf) + fufu;
        }
        if (!do_ls) {
            if (gv && sub == 0) sp->node_llh[n_u[g]] = llh_g;
            __syncwarp();
            return true;
        }
        if (gv && sub == 0) n_llh[g] = llh_g;
        __syncwarp();
        // ---------------- G. sum_v fv / (1 - p) (:167-168), edge by edge in CSR order ----------------
#pragma unroll 1
        for (int r = 0; r < maxdeg; ++r) {
            if (r < deg_g) {
                const int e = es_g + r;
                const double wv = we[e];
                const int cn = e_cnt[e];
                const double *vv = reinterpret_cast<const double *>(stageN + 16 * (size_t)e_soff[e]);
                const unsigned short *vi = sp_idx(vv, (uint32_t)cn);
#pragma unroll 1
                for (int i = sub; i < cn; i += gs) {
                    const int slot = vi[i];
                    fg[slot].y = fma(wv, vv[i], fg[slot].y);
                }
            }
            __syncwarp();
        }
        // ---------------- H. gradient (:168), |g|^2, active components ----------------
        int m_g = 0;
        bool hi_lane = false;
        double G2n = 0.0, G2p = 0.0;     // [bounds] |g|^2 over the active components with g < 0 / g > 0
        float r3 = 0.0f, r4 = 0.0f;      // [bounds] R3 >= sum fu_c |gt_c|; magnitudes behind the rounding allowance
        float gmx = 0.0f, g1p = 0.0f;    // [bounds] largest positive gradient component, sum of the positive ones
        double G2node = 0.0;             // |g|^2 of the node (all K components)
        {
            double G2 = 0.0, SF2 = 0.0;
            int maxtot = tot_g;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) maxtot = max(maxtot, __shfl_xor_sync(0xffffffffu, maxtot, o));
#pragma unroll 1
            for (int k0 = 0; k0 < maxtot; k0 += gs) {
                const int k = k0 + sub;
                bool act = false;
                if (k < tot_g) {
                    const int slot = base_g + k;
                    const double2 v = fg[slot];
                    const double sf = s_sumF[slot_c[slot]];
                    const double gr = (v.y - sf) + v.x;
                    fg[slot].y = gr;
                    G2 = fma(gr, gr, G2);
                    SF2 = fma(sf, sf, SF2);
                    act = (v.x > 0.0 || gr > 0.0);
                    hi_lane |= act && (v.x + gr > max_f);
                    if (act && prune_on) {
                        const float ga = __double2float_ru(fabs(gr)), ff = __double2float_ru(v.x);
                        r3 = fmaf(ff, fmaf(2.0f, ga, __double2float_ru(fabs(sf))) + 3.0f * ff, r3);
                        if (gr > 0.0) {
                            G2p = fma(gr, gr, G2p);
                            gmx = fmaxf(gmx, ga);
                            g1p += ga;
                        } else {
                            G2n = fma(gr, gr, G2n);
                        }
                    }
                }
                m_g += __popc((__ballot_sync(0xffffffffu, act) >> gsh) & gmask);
            }
            G2 = group_sum(G2, gs);
            SF2 = group_sum(SF2, gs);
            if (prune_on) {
                G2n = group_sum(G2n, gs);
                G2p = group_sum(G2p, gs);
                r3 = group_sum(r3, gs);
                g1p = group_sum(g1p, gs);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
                    if (o < gs) gmx = fmaxf(gmx, __shfl_xor_sync(0xffffffffu, gmx, o));
                // sum_act |g_c| (2|g_c| + sumF_c + 3 fu_c) <= 2 |g|^2 + |g| sqrt(2 sum sumF_c^2 + 18 fu.fu) over the touched components
                const float g2f = __double2float_ru(G2);
                r4 = fmaf(2.0f, g2f, sqrtf(g2f) * sqrtf(fmaf(2.0f, __double2float_ru(SF2), 18.0f * __double2float_ru(fufu))) * 1.0001f);
            }
            // an untouched component has fu = 0 and gradient -sumF_c: its square is part of S2_all
            G2node = (S2_all - SF2) + G2;
            if (gv && sub == 0) n_G2[g] = G2node;
        }
        if (!gv) m_g = 0;
        int ab_g = 0, maxm = 0;
#pragma unroll 1
        for (int q = 0; q < nn; ++q) {
            const int t = __shfl_sync(0xffffffffu, m_g, q << lgs);
            if (q < g) ab_g += t;
            maxm = max(maxm, t);
        }
        if (gv && sub == 0) { n_ab[g] = (unsigned short)ab_g; n_m[g] = (unsigned short)m_g; }
        // no candidate of any node of the tile can reach MAX_F_ (the largest step is 1): the upper clamp is dropped
        const bool need_hi = __any_sync(0xffffffffu, hi_lane);
        __syncwarp();
        // [bounds, see H2] of the edges that are clamped flat: Dp_e = sum_c max(g_c, 0) fv_c and En_e = sum_{c active} min(g_c, 0) fv_c
        // (a component with g_c < 0 is active iff fu_c > 0)
        double Dp = 0.0, En = 0.0;
        if (prune_on && (e_low || vnear > 0.0f) && lane < ne) {
#pragma unroll 1
            for (int i = 0; i < ce; ++i) {
                const double2 v = fg[ri[i]];
                const double val = rv[i];
                Dp = fma(val, v.y > 0.0 ? v.y : 0.0, Dp);
                En = fma(val, (v.y < 0.0 && v.x > 0.0) ? v.y : 0.0, En);
            }
        }
        // the active components move to the front, in slot order: fg[a] = (fu_c, grad_c), slot_c[a] = c; amap: slot -> a
        int A = 0;
#pragma unroll 1
        for (int p0 = 0; p0 < total_slots; p0 += 32) {
            const int p = p0 + lane;
            const bool ok = p < total_slots;
            double2 v = make_double2(0.0, 0.0);
            int c = 0;
            if (ok) { v = fg[p]; c = slot_c[p]; }
            const bool act = ok && (v.x > 0.0 || v.y > 0.0);
            const unsigned bal = __ballot_sync(0xffffffffu, act);
            __syncwarp();                        // every lane has read its slot; the writes land at or below them
            const int an = A + __popc(bal & lt_mask);
            if (act && an < kTlSlots) { fg[an] = v; slot_c[an] = (unsigned short)c; }
            if (ok) amap[p] = act ? (unsigned short)an : (unsigned short)0xffffu;
            A += __popc(bal);
            __syncwarp();
        }
        if (A > kTlAct - 1) return false;                      // (one spare: the padding component below)
        double *asfm = reinterpret_cast<double *>(fg + kTlAct);            // sumF_c - fu_c of the active components
#pragma unroll 1
        for (int t = lane; t < A; t += 32) asfm[t] = s_sumF[slot_c[t]] - fg[t].x;
        // padding component A: fu = grad = 0, so every candidate is 0 there and adds exactly nothing — the lockstep loops
        // of the line search read it instead of predicating their bodies
        if (lane == 0) { fg[A] = make_double2(0.0, 0.0); asfm[A] = 0.0; }
        __syncwarp();
        // ---------------- H2. bounds: which (node, candidate) pairs can pass the Armijo test at all ----------------
        // Most candidates can be PROVEN to fail (:181) from what the PRE block already has.  Write the node's objective
        // as phi(nf) = sum_v T(nf.fv) - nf.(sumF - fu), T(x) = S(x) + x, S(x) = log(1 - clamp(exp(-x))) (:166,:179): S is
        // the constant S_lo up to x_lo (clamp at MAX_P_), concave and increasing up to x_hi, constant from there.  With
        // D = nf - fu, D_c = min(max(s g_c, -fu_c), MAX_F_ - fu_c) (:110-113, MIN_F_ = 0) and fv >= 0:
        //   * an edge with x_v >  x_lo:  S(x') - S(x_v) <= (w_v - 1) (x' - x_v) + viol_v               (tangent, see D.)
        //   * an edge with x_v <= x_lo:  S(x') - S(x_v) <= H(x_v + s Dp_v),  Dp_v = sum_c max(g_c, 0) fv_c >= (x' - x_v) / s,
        //                                H(y) = S(y) - S_lo <= min(log(y / (1 - MAX_P_)), cap), and 0 for y <= x_lo
        //   * the linear part and the tangents add up to sum_c D_c gt_c, gt_c = g_c - (w_lo - 1) sum_{v low} fv_c: the coded
        //     gradient (:168) minus the slope it books for edges that are clamped flat; gt_c <= g_c, |gt_c| <= 2|g_c| + sumF_c
        //       g_c < 0:  D_c gt_c = min(s |g_c|, fu_c) |gt_c|      -> in total <= min(s Qn, R3),
        //                 Qn = sum_{g<0} g_c^2 - (w_lo - 1) sum_{v low} En_v,  En_v = sum_{g_c<0} g_c fv_c,  R3 >= sum fu_c |gt_c|
        //       g_c > 0:  D_c in [kappa s g_c, min(s g_c, MAX_F_)], kappa = min(1, (MAX_F_ - max fu) / (s max g))
        //                 -> in total <= min(s Qp, MAX_F_ G1) - kappa s Mp,  Qp = sum_{g>0} g_c^2,  G1 = sum_{g>0} g_c,
        //                    Mp = (w_lo - 1) sum_{v low} Dp_v
        // Hence  phi(nf_j) - phi(fu) <= min(s_j Qn, R3) + min(s_j Qp, MAX_F_ G1) - kappa_j s_j Mp + V_j + sum_{v low} H(x_v + s_j Dp_v),
        // V_j = the viol_v of the edges above x_hi and of those edges next to x_lo that candidate j can bring below it
        // (x_v + s_j En_v < x_lo).
        // A pair (node, j) whose bound stays below alpha s_j |g|^2 by more than the rounding allowance — twice the worst-case
        // rounding error of a sum of 4 deg + 3 m + 16 operations on the magnitudes that enter the candidate's sums
        // (c0 + s c1) plus 1e-9 relative — cannot pass and is not
        // evaluated; a node without a surviving pair keeps its row.  Everything else is evaluated exactly as before:
        // the results are the same bits as those of the exhaustive search (BIGCLAM_F_LS_EXHAUSTIVE, tests/test_gpu_prune.py).
        // Mapping: lane = edge for the per-edge terms, then the lanes of a node's group share its candidates.
        const bool prune = prune_on;
        float2 *we2 = reinterpret_cast<float2 *>(we);          // (the weights w_e are not needed any more)
        if (prune) {
            float lnthr = 3.0e38f, Lp = 0.0f;                  // H_e(s) = 0 up to ln s = lnthr, <= min(cap, ln s + Lp) beyond
            if (vnear > 0.0f) {
                // an edge in range next to x_lo: its tangent only fails for x' < x_lo, and x' >= x + s En: from ln s = lnthr on
                // the candidate is charged viol (kept as Lp = -1000 - viol)
                if (En < 0.0) {
                    const float sthr = __double2float_rd((x - ec.x_lo) / (-En)) * 0.99999f;
                    if (sthr > 0.0f) {
                        const float t1 = __log2f(sthr);
                        lnthr = t1 * 0.69314718f - fmaf(1.0e-6f, fabsf(t1), 1.0e-4f);
                    } else {
                        lnthr = -3.0e38f;
                    }
                    Lp = -1000.0f - vnear;
                }
            } else if (Dp > 0.0) {
                const float Df = __double2float_ru(Dp) * 1.000001f;
                const float sthr = (sp->pr_xlo - xf) / Df * 0.99999f;           // x + s Dp stays below x_lo up to here
                if (sthr > 0.0f) {
                    const float t1 = __log2f(sthr), t2 = __log2f(sp->pr_kinv * (Df + xf / sthr));
                    lnthr = t1 * 0.69314718f - fmaf(1.0e-6f, fabsf(t1), 1.0e-4f);
                    Lp = t2 * 0.69314718f + fmaf(1.0e-6f, fabsf(t2), 1.0e-4f);
                } else {
                    lnthr = -3.0e38f;                                           // (always at the cap)
                    Lp = 3.0e38f;
                }
            }
            we2[lane] = make_float2(lnthr, Lp);
            if (!e_low) { Dp = 0.0; En = 0.0; }                // (the node's sums below are over the flat edges only)
        }
        unsigned svbits = 0u;
        {
            const bool want_g = gv && (n_want[gv ? g : 0] != 0);
            const int jn = nsteps < 16 ? nsteps : 16;
            if (prune) {
                double sDp = 0.0, sEn = 0.0;
                float sV = 0.0f;
#pragma unroll 1
                for (int r = 0; r < maxdeg; ++r) {
                    const int src = (es_g + r) & 31;
                    const double tD = __shfl_sync(0xffffffffu, Dp, src);
                    const double tE = __shfl_sync(0xffffffffu, En, src);
                    const float tV = __shfl_sync(0xffffffffu, violf, src);
                    if (r < deg_g) { sDp += tD; sEn += tE; sV += tV; }
                }
                __syncwarp();                                                   // (we2 is complete)
                if (want_g) {
                    const double Mp = (ec.w_lo - 1.0) * sDp, Qn = G2n - (ec.w_lo - 1.0) * sEn;
                    const float cap_f = sp->pr_cap;
                    const float fuf = __double2float_ru(fabs(fusf)), fff = __double2float_ru(fufu);
                    const float base = fmaf(2.0f * cap_f, (float)deg_g, __double2float_ru(fabs(llh_g))) + 2.0f * (fuf + fff) + r3;
                    // rounding allowance: twice the worst case of a sum of (4 deg + 3 m + 16) rounded operations on these magnitudes
#ifdef BIGCLAM_PR_OLDNOPS
                    const float nops = 1.0e-13f;
#else
                    const float nops = 2.3e-16f * (float)(4 * deg_g + 3 * m_g + 16);
#endif
                    const float c0 = fmaf(nops, base, sV) * 1.0001f;
                    const float c1 = nops * fmaf(2.0f, r4, __double2float_ru(sDp)) * 1.0001f;
#ifdef BIGCLAM_PR_NOG1
                    const double G1 = 1.0e300;
#else
                    const double G1 = (double)(__double2float_ru(max_f) * g1p * 1.0001f);   // >= sum_{g>0} min(s g_c, MAX_F_) g_c
#endif
                    const double R3 = (double)(r3 * 1.0001f);
                    const float fmx = sqrtf(fff) * 1.000001f;                   // >= every fu_c
                    const float kap0 = (gmx > 0.0f) ? __fdividef(fmaxf(__double2float_rd(max_f) - fmx, 0.0f), gmx) * 0.9999f : 3.0e38f;
                    // this lane's candidates: sub, sub + gs, sub + 2 gs, sub + 3 gs (gs >= 4); the edge terms of all four in one walk
                    float lns[4], Hs[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int jj = sub + k * gs;
                        lns[k] = (jj < jn) ? s_lns[jj] : -3.0e38f;
                        Hs[k] = 0.0f;
                    }
#pragma unroll 1
                    for (int r = 0; r < deg_g; ++r) {
                        const float2 tl = we2[es_g + r];
                        const bool isv = tl.y < -500.0f;
                        const float vv = -1000.0f - tl.y;
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (lns[k] > tl.x) Hs[k] += isv ? vv : fminf(cap_f, fmaxf(lns[k] + tl.y, 0.0f));
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int jj = sub + k * gs;
                        if (jj < jn) {
                            const double sj = s_steps[jj];
                            const float sfu = __double2float_ru(sj);
                            const float kap = fminf(1.0f, __fdividef(kap0, sfu) * 0.9999f);
                            const double negp = fmin(sj * Qn, R3);
                            const double bound = negp + fmin(sj * G2p, G1) - sj * ((double)kap * Mp) + (double)(fmaf(Hs[k], 1.00001f, c0) + sfu * c1);
                            const double rhs = (a->alpha * sj) * G2node;
                            if (!(bound < rhs * (1.0 - 1.0e-9))) svbits |= 1u << jj;
                        }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
                    if (o < gs) svbits |= __shfl_xor_sync(0xffffffffu, svbits, o);
            } else if (want_g) {
                svbits = (1u << jn) - 1u;
            }
            if (gv && sub == 0) n_sv[g] = (unsigned short)svbits;
        }
        __syncwarp();
        // the nodes that are line-searched at all, in tile order
        const unsigned svmask = __ballot_sync(0xffffffffu, lane < nn && n_sv[lane < nn ? lane : 0] != 0);
        const int ns = __popc(svmask);
        last_ns = ns;
        last_nw = __popc(__ballot_sync(0xffffffffu, lane < nn && n_want[lane < nn ? lane : 0] != 0));
        if (lane < nn) {
            n_js[lane] = -1;
            if ((svmask >> lane) & 1u) n_sl[__popc(svmask & lt_mask)] = (unsigned char)lane;
        }
        __syncwarp();
        if (ns > 0) {
            // ---------------- I. the neighbours' entries on active components, listed per component ----------------
            // (only for the nodes that are line-searched: flat loops over runs of consecutive such nodes — their edges,
            // entries and active components are contiguous)
            unsigned rem = svmask;
#pragma unroll 1
            while (rem) {
                const int na = __ffs(rem) - 1, len = __ffs(~(rem >> na)) - 1;
                rem &= ~(((1u << len) - 1u) << na);
                const int ahi = (int)n_ab[na + len - 1] + (int)n_m[na + len - 1];
#pragma unroll 1
                for (int t = (int)n_ab[na] + lane; t < ahi; t += 32) lcnt[t] = 0u;
            }
            __syncwarp();
            rem = svmask;
#pragma unroll 1
            while (rem) {
                const int na = __ffs(rem) - 1, len = __ffs(~(rem >> na)) - 1;
                rem &= ~(((1u << len) - 1u) << na);
                const int thi = epos[n_es[na + len]];
BIGCLAM_UNROLL(BIGCLAM_TL_UF)
                for (int t = (int)epos[n_es[na]] + lane; t < thi; t += 32) {
                    const unsigned an = amap[stN16[(unsigned short)(e_io2[erow[t]] + t)]];
                    if (an != 0xffffu) atomicAdd(lcnt + an, 1u);
                }
            }
            __syncwarp();
            int TE = 0;
            rem = svmask;
#pragma unroll 1
            while (rem) {
                const int na = __ffs(rem) - 1, len = __ffs(~(rem >> na)) - 1;
                rem &= ~(((1u << len) - 1u) << na);
                const int ahi = (int)n_ab[na + len - 1] + (int)n_m[na + len - 1];
#pragma unroll 1
                for (int t0 = n_ab[na]; t0 < ahi; t0 += 32) {
                    const int t = t0 + lane;
                    const int c = (t < ahi) ? (int)lcnt[t] : 0;
                    int incl = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int v = __shfl_up_sync(0xffffffffu, incl, o);
                        if (lane >= o) incl += v;
                    }
                    if (t < ahi) { loff[t] = (unsigned short)(TE + incl - c); lcnt[t] = (unsigned int)(TE + incl - c); }
                    TE += __shfl_sync(0xffffffffu, incl, 31);
                }
                if (lane == 0) loff[ahi] = (unsigned short)TE;          // end of the run's last list (a following run starts there or later)
            }
            if (TE > kTlEnt - 1) return false;
            if (lane == 0) {
                ent_val[TE] = 0.0;                 // padding entry: component A, a scratch cell behind the 32 edges' cells
                ent_e[TE] = 32;
                ent_a[TE] = (unsigned char)A;
            }
            __syncwarp();
            rem = svmask;
#pragma unroll 1
            while (rem) {
                const int na = __ffs(rem) - 1, len = __ffs(~(rem >> na)) - 1;
                rem &= ~(((1u << len) - 1u) << na);
                const int thi = epos[n_es[na + len]];
BIGCLAM_UNROLL(BIGCLAM_TL_UF)
                for (int t = (int)epos[n_es[na]] + lane; t < thi; t += 32) {
                    const int row = erow[t];
                    const double *vv = reinterpret_cast<const double *>(stageN + 16 * (size_t)e_soff[row]);
                    const int i = t - (int)epos[row];
                    const unsigned an = amap[stN16[(unsigned short)(e_io2[row] + t)]];
                    if (an != 0xffffu) {
                        const unsigned q = atomicAdd(lcnt + an, 1u);
                        ent_val[q] = vv[i];
                        ent_e[q] = (unsigned char)row;
                        ent_a[q] = (unsigned char)an;
                    }
                }
            }
            __syncwarp();
            // ---------------- J. line search (:172-180), two line-searched nodes at a time: lane = (node, trial j) ----------------
            // One loop over the node's active components gives, per candidate: newfu.sfT and newfu.newfu (:176,:180) and,
            // through the components' entry lists, newfu.fv of every edge (xs[edge][trial], component order ascending).
            const int h = lane >> 4, j = lane & 15;
            const double s = s_steps[j < nsteps ? j : 0];
            if (lane < 16) xs[32 * 16 + lane] = 0.0;                          // scratch row of the padding entry (the staged rows are not needed any more)
            __syncwarp();
#pragma unroll 1
            for (int k0 = 0; k0 < ns; k0 += 2) {
                const bool nv = k0 + h < ns;
                const int node = nv ? (int)n_sl[k0 + h] : 0;
                const bool mine = nv && (((unsigned)n_sv[node] >> j) & 1u);     // (a pair that cannot pass is not evaluated)
                const int e0 = nv ? (int)n_es[node] : 0, dn = nv ? (int)n_es[node + 1] - e0 : 0;
                const int t0 = nv ? (int)n_ab[node] : 0, mm = nv ? (int)n_m[node] : 0;
                const int q0 = nv ? (int)loff[t0] : 0, nq = nv ? (int)loff[t0 + mm] - q0 : 0;
#pragma unroll 1
                for (int r = 0; r < dn; ++r) xs[(e0 + r) * 16 + j] = 0.0;       // (each cell belongs to one lane)
                // the two half-warps (two nodes) walk in lockstep: common trip counts, padded with a component / an entry that add nothing
                const int mmax = max(mm, __shfl_xor_sync(0xffffffffu, mm, 16));
                const int qmax = max(nq, __shfl_xor_sync(0xffffffffu, nq, 16));
                const int dmax = max(dn, __shfl_xor_sync(0xffffffffu, dn, 16));
                double a1 = 0.0, b1 = 0.0;
BIGCLAM_UNROLL(BIGCLAM_TL_UJ)
                for (int t = 0; t < mmax; ++t) {
                    const int ti = (t < mm) ? t0 + t : A;                   // (A: the padding component, adds +0.0)
                    const double2 v = fg[ti];
                    const double nf = need_hi ? clamp_step0(v.x, s, v.y, max_f) : clamp_step0_lo(v.x, s, v.y);
                    const double sf = asfm[ti] + nf;                        // sfT = (sumF - fu) + newfu   (:176)
                    a1 = fma(nf, sf, a1);
                    b1 = fma(nf, nf, b1);
                }
BIGCLAM_UNROLL(BIGCLAM_TL_UJ)
                for (int k = 0; k < qmax; ++k) {
                    const int qq = (k < nq) ? q0 + k : TE;                  // (TE: the padding entry, scratch cell, value 0)
                    const double2 v = fg[ent_a[qq]];
                    const double nf = need_hi ? clamp_step0(v.x, s, v.y, max_f) : clamp_step0_lo(v.x, s, v.y);
                    double *cell = xs + (int)ent_e[qq] * 16 + j;
                    *cell = fma(nf, ent_val[qq], *cell);
                }
                // pairs whose x is outside (x_lo, x_hi) are constants after the clamp (:166); the others are listed and exp/log
                // runs on full warps of them
                int np = 0;
#pragma unroll 1
                for (int r = 0; r < dmax; ++r) {
                    const int p = (e0 + r) * 16 + j;
                    const bool valid = mine && r < dn;
                    const double D = valid ? xs[p] : 0.0;
                    const bool low = D <= ec.x_lo;
                    const bool inr = valid && !low && (D < ec.x_hi);
                    if (valid && !inr) xs[p] = (low ? ec.t_lo : ec.t_hi) + D;
                    const unsigned bal = __ballot_sync(0xffffffffu, inr);
                    if (inr) plist[np + __popc(bal & lt_mask)] = (unsigned short)p;
                    np += __popc(bal);
                }
                __syncwarp();
#if BIGCLAM_TL_ILP2
#pragma unroll 1
                for (int b = 0; b < np; b += 64) {
                    const int k1 = b + lane, k2 = b + 32 + lane;
                    const bool ok1 = k1 < np, ok2 = k2 < np;
                    const int pid1 = ok1 ? (int)plist[k1] : 0, pid2 = ok2 ? (int)plist[k2] : 0;
                    const double x1 = ok1 ? xs[pid1] : 1.0, x2 = ok2 ? xs[pid2] : 1.0;
                    const double o1 = 1.0 - exp_neg(x1), o2 = 1.0 - exp_neg(x2);
                    const double t1 = log_pos(o1) + x1, t2 = log_pos(o2) + x2;
                    if (ok1) xs[pid1] = t1;
                    if (ok2) xs[pid2] = t2;
                }
#else
#pragma unroll 1
                for (int b = 0; b < np; b += 32) {
                    const int k = b + lane;
                    const bool ok = k < np;
                    const int pid = ok ? (int)plist[k] : 0;
                    const double xv = ok ? xs[pid] : 1.0;
                    const double omp = 1.0 - exp_neg(xv);
                    const double t = log_pos(omp) + xv;
                    if (ok) xs[pid] = t;
                }
#endif
                __syncwarp();
                // ---------------- K. Armijo test (:181), largest passing step (:182) ----------------
                bool pass = false;
                if (mine) {
                    double acc = 0.0;
#pragma unroll 1
                    for (int r = 0; r < dn; ++r) acc += xs[(e0 + r) * 16 + j];          // the node's edges, in CSR order
                    const double result = (acc - a1) + b1;
                    const double rhs = n_llh[node] + (a->alpha * s) * n_G2[node];
                    pass = result >= rhs;
                }
                const unsigned won = (__ballot_sync(0xffffffffu, pass) >> (16 * h)) & 0xffffu;
                if (nv && j == 0) n_js[node] = (signed char)(won ? __ffs(won) - 1 : -1);
                __syncwarp();
            }
        }
        __syncwarp();
        // ---------------- L. new rows (:183-190) and delta blocks (:191-192) ----------------
        const int js = gv ? (int)n_js[g] : -1;
        const double sstar = s_steps[js >= 0 ? js : 0];
        int nz = 0, nd = 0;
#pragma unroll 1
        for (int t0 = 0; t0 < maxm; t0 += gs) {
            const int t = t0 + sub;
            bool isnz = false, ch = false;
            if (js >= 0 && t < m_g) {
                const double2 v = fg[ab_g + t];
                const double nr = clamp_step(v.x, sstar, v.y, a->min_f, max_f);
                isnz = nr != 0.0;
                ch = v.x != nr;
            }
            nz += __popc((__ballot_sync(0xffffffffu, isnz) >> gsh) & gmask);
            nd += __popc((__ballot_sync(0xffffffffu, ch) >> gsh) & gmask);
        }
        if (js < 0) { nz = cu_g; nd = 0; }
        const int wrow = gv ? (int)sp_words((uint32_t)nz) : 0;
        const int words_g = gv ? wrow + (nd > 0 ? (int)sp_words((uint32_t)nd) : 0) : 0;
        int woff = 0, wtotal = 0;
#pragma unroll 1
        for (int q = 0; q < nn; ++q) {
            const int t = __shfl_sync(0xffffffffu, words_g, q << lgs);
            if (q < g) woff += t;
            wtotal += t;
        }
        unsigned long long rel = 0;
        if (lane == 0 && wtotal > 0) rel = atomicAdd(sp->pool_top, (unsigned long long)wtotal);
        rel = __shfl_sync(0xffffffffu, rel, 0);
        if (rel + (unsigned long long)wtotal > sp->pool_cap8) {
            if (gv && sub == 0) { *sp->overflow = 1; sp->hdr_out[n_u[g]] = sp_pack(0, 0); sp->dcnt[n_u[g]] = 0; }
            __syncwarp();
            return true;
        }
        const unsigned long long off = sp->region_base8 + rel + (unsigned long long)woff;
        double *outv = sp->pool_out + off;
        {
            // accepted nodes: the candidate's non-zeros, ascending, and the delta block right behind the row
            unsigned short *outi = sp_idx(outv, (uint32_t)nz);
            double *dv = outv + wrow;
            unsigned short *di = sp_idx(dv, (uint32_t)nd);
            int pz = 0, pd = 0;
#pragma unroll 1
            for (int t0 = 0; t0 < maxm; t0 += gs) {
                const int t = t0 + sub;
                bool isnz = false, ch = false;
                double nr = 0.0, f = 0.0;
                int c = 0;
                if (js >= 0 && t < m_g) {
                    const double2 v = fg[ab_g + t];
                    c = slot_c[ab_g + t];
                    f = v.x;
                    nr = clamp_step(f, sstar, v.y, a->min_f, max_f);
                    isnz = nr != 0.0;
                    ch = f != nr;
                }
                const unsigned bz = (__ballot_sync(0xffffffffu, isnz) >> gsh) & gmask;
                const unsigned bd = (__ballot_sync(0xffffffffu, ch) >> gsh) & gmask;
                if (isnz) {
                    const int p = pz + __popc(bz & below);
                    outv[p] = nr;
                    outi[p] = (unsigned short)c;
                    if (kPush)
                        for (int pr = 0; pr < sp->n_peers; ++pr) {
                            double *pv = sp->peer_pool[pr] + off;
                            pv[p] = nr;
                            sp_idx(pv, (uint32_t)nz)[p] = (unsigned short)c;
                        }
                }
                if (ch) {
                    const int p = pd + __popc(bd & below);
                    dv[p] = f - nr;
                    di[p] = (unsigned short)c;
                }
                pz += __popc(bz);
                pd += __popc(bd);
            }
        }
        if (gv && js < 0) {
            // row kept: block copy of the staged own row
            const uint4 *src = reinterpret_cast<const uint4 *>(ov);
            uint4 *dst = reinterpret_cast<uint4 *>(outv);
            const int q16 = wrow >> 1;
#pragma unroll 1
            for (int q = sub; q < q16; q += gs) {
                const uint4 blk = src[q];
                dst[q] = blk;
                if (kPush)
                    for (int pr = 0; pr < sp->n_peers; ++pr) reinterpret_cast<uint4 *>(sp->peer_pool[pr] + off)[q] = blk;
            }
        }
        if (gv && sub == 0) {
            const int64_t u = n_u[g];
            const uint64_t hnew = sp_pack(off, (uint32_t)nz);
            sp->hdr_out[u] = hnew;
            sp->dcnt[u] = (unsigned short)nd;
            sp->accepted[u] = (int8_t)js;
            sp->node_llh[u] = llh_g;
            if (kPush)
                for (int pr = 0; pr < sp->n_peers; ++pr) sp->peer_hdr[pr][u] = hnew;
        }
        __syncwarp();
        return true;
    }
};

// kPush: multi-GPU launch, the peers' replicas are written too; kHub: the launch has split hubs.  Both are
// compile-time so that the plain single-GPU kernel carries none of that code.  kHO: the masked objective of a context
// with held-out pairs (bigclam_set_holdout): every node goes through the general path (no tiles, no split hubs).
template <bool kPush, bool kHub, bool kHO = false>
__global__ void __launch_bounds__(kTlThreads, kTlBlocksPerSM) tile_step_kernel(const __grid_constant__ StepArgs a, const __grid_constant__ SparseArgs sp) {
    if (a.done_flag != nullptr && *a.done_flag != 0) return;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int ld = a.ld;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nthreads = (int)blockDim.x;
    const int ldp = sp_ldp(ld);
    double *s_steps = reinterpret_cast<double *>(smem_raw);
    double *s_sumF = s_steps + kMaxSteps;
    unsigned long long *s_mbar = reinterpret_cast<unsigned long long *>(s_sumF + ldp);
    float *s_lns = reinterpret_cast<float *>(s_mbar + kTlWarps);          // 16 floats
    unsigned char *wbase = reinterpret_cast<unsigned char *>(s_mbar + kTlWarps + 8) + (size_t)wib * tl_region_bytes(ld);

#pragma unroll 1
    for (int i = threadIdx.x; i < ldp; i += nthreads) s_sumF[i] = (i < ld) ? a.sumF[i] : 0.0;
#pragma unroll 1
    for (int i = threadIdx.x; i < kMaxSteps; i += nthreads) s_steps[i] = a.steps[i];
    if (threadIdx.x < 16) {
        const float sfu = __double2float_ru(a.steps[threadIdx.x]);
        const float t = (sfu > 0.0f) ? __log2f(sfu) : -3.0e38f;
        s_lns[threadIdx.x] = (sfu > 0.0f) ? t * 0.69314718f + fmaf(1.0e-6f, fabsf(t), 1.0e-4f) : -3.0e38f;
    }
    __syncthreads();
    // S2_all = sum_c sumF_c^2 in a fixed order (every warp computes the same bits)
    double S2 = 0.0;
    for (int c = lane; c < ldp; c += 32) S2 = fma(s_sumF[c], s_sumF[c], S2);
    S2 = warp_sum(S2);

    SpGen G;
    G.a = &a;
    G.sp = &sp;
    G.s_steps = s_steps;
    G.s_sumF = s_sumF;
    G.s_lns = s_lns;
    G.ec = {a.x_lo, a.x_hi, a.t_lo, a.t_hi, a.w_lo, a.w_hi};
    G.carve(wbase, ld, lane);
    TlWarp T;
    T.a = &a;
    T.sp = &sp;
    T.s_steps = s_steps;
    T.s_sumF = s_sumF;
    T.s_lns = s_lns;
    T.S2_all = S2;
    T.ec = G.ec;
    T.carve(wbase, ld, lane);
    T.mbar = s_mbar + wib;
    if (lane == 0) mbar_init(T.mbar);
    G.clear_dense();
    bool dense_clean = true;      // the two paths share the warp's region: the general path needs its dense vectors zeroed
    __syncwarp();

    if constexpr (kHub) {
        for (;;) {
            unsigned int it = 0;
            if (lane == 0) it = atomicAdd(sp.hub_work, 1u);
            it = __shfl_sync(0xffffffffu, it, 0);
            if (it >= (unsigned int)a.n_hub_items) break;
            G.template hub_item<kPush>(a.hub_items[it]);
        }
    }

    const unsigned int n_items = (unsigned int)sp.n_gen + (kHO ? 0u : (unsigned int)sp.ntiles);
    unsigned int item = 0;
    if (lane == 0) item = atomicAdd(a.work_counter, 1u);
    item = __shfl_sync(0xffffffffu, item, 0);
    while (item < n_items) {
        unsigned int nxt = 0;
        if (lane == 0) nxt = atomicAdd(a.work_counter, 1u);
        // nodes for the general path: the item itself, or the nodes of a tile that did not fit (one call site)
        int gen_cnt = 1;
        int64_t gen_pos = (int64_t)a.n_hubs + item;
        const int32_t *gen_col = nullptr;
        if (!kHO && item >= (unsigned int)sp.n_gen) {
            const TileMeta tm = sp.tiles[item - (unsigned int)sp.n_gen];
            dense_clean = false;
            const bool done = T.template run<kPush>(tm);
            if (sp.stats != nullptr && lane == 0) {
                atomicAdd(sp.stats + (done ? 0 : 1), 1u);
                if (done && a.do_linesearch) { atomicAdd(sp.stats + 2, (unsigned)T.last_ns); atomicAdd(sp.stats + 3, (unsigned)T.last_nw); }
            }
            gen_cnt = done ? 0 : tm.nn;
            gen_pos = tm.pos0;
            gen_col = sp.tcol + tm.ecol0;           // the tile's entries of tcol are its nodes' neighbour lists (tagged ids)
        }
#pragma unroll 1
        for (int i = 0; i < gen_cnt; ++i) {
            const NodeMeta nm = a.meta[gen_pos + i];
            if (!dense_clean) { G.clear_dense(); dense_clean = true; }
            G.template node<kPush, kHO>(nm.u, nm.deg, gen_col != nullptr ? gen_col : a.col + nm.e0);
            if (gen_col != nullptr) gen_col += nm.deg;
        }
        item = __shfl_sync(0xffffffffu, nxt, 0);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The sums over nodes, in a fixed order: partials = [D(ld) = sum over accepted nodes of (old - new) | unused(ld) |
// sum_u llh_u | number of accepted nodes].  Warp w of the grid owns a contiguous range of the processing order and
// walks it front to back (delta blocks land in a per-warp dense vector, entries of one node never collide), the
// warps of a block are added in warp order, the blocks in block order by the last block to finish.  No
// floating-point atomics: two runs give the same bits.
struct ReduceArgs {
    const NodeMeta *meta;
    int64_t order_n;
    const uint64_t *hdr_out;
    const double *pool_out;
    const double *node_llh;
    const unsigned short *dcnt;
    const int8_t *accepted;
    int32_t ld;
    int32_t do_linesearch;
    double *block_part;       // gridDim.x x (ld + 2)
    unsigned int *ticket;
    double *partials;         // 2 * ld + 2
    const int32_t *done_flag;
    unsigned int *work_counter;          // reset to work_init for the next launch (no separate memcpy node per step)
    unsigned int work_init;
    unsigned long long *pool_top_in;     // zeroed: this step's input pool is the next step's output pool
    // node-partitioned multi-GPU (fused collective, no NCCL on the data path): the last block also stores this
    // rank's sums into its slot of every rank's exchange buffer (peer memory over NVLink) and then raises its
    // flag there to `seq`; xreduce_kernel on every rank adds the slots up in rank order once all flags are up.
    int32_t world;
    double *xslot[8];                    // this rank's slot (ld + 2 doubles) in rank p's buffer, p = 0 .. world-1
    unsigned long long *xflag[8];        // this rank's flag in rank p's flag array
    unsigned long long seq;
};
constexpr int kRedWarps = 32;      // at most; every warp keeps a dense vector of ldp doubles in shared memory: wide rows run fewer warps
inline int red_warps(int ld) { const int ldp = sp_ldp(ld); return ldp <= 384 ? 32 : ldp <= 768 ? 16 : 8; }

__global__ void __launch_bounds__(kRedWarps * 32) reduce_kernel(const ReduceArgs r) {
    if (r.done_flag != nullptr && *r.done_flag != 0) return;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int ld = r.ld, ldp = sp_ldp(ld);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double *Dw = reinterpret_cast<double *>(smem_raw) + (size_t)wib * ldp;
    __shared__ double s_llh[kRedWarps];
    __shared__ unsigned int s_nupd[kRedWarps];
    __shared__ double s_cnt[kRedWarps];
    __shared__ unsigned int s_last;
    for (int c = lane; c < ldp; c += 32) Dw[c] = 0.0;
    __syncwarp();
    // group q = 32 positions of the processing order, one per lane: q, q + G, q + 2 G, ... (G groups in all).  The order is
    // sorted by degree and the nodes that keep moving (and their long delta blocks) cluster in it: taking every G-th position
    // gives every warp the same mix.  Warp gw takes the groups gw, gw + #warps, ...; a fixed assignment: reproducible sums.
    const int nw = (int)(blockDim.x >> 5);               // warps of this block (red_warps(ld) <= kRedWarps)
    const int64_t nwarps = (int64_t)gridDim.x * nw;
    const int64_t gw = (int64_t)blockIdx.x * nw + wib;
    const int64_t G = (r.order_n + 31) / 32;
    double llh = 0.0;
    unsigned int nupd = 0;
    for (int64_t q = gw; q < G; q += nwarps) {
        const int64_t p = (int64_t)lane * G + q;
        const bool ok = p < r.order_n;
        const int32_t u = ok ? r.meta[p].u : 0;
        if (ok) llh += r.node_llh[u];
        // (header and delta count are loaded together with the accepted flag, not after it: one dependent load less)
        int8_t af = -1;
        uint64_t h = 0;
        int dc = 0;
        if (ok && r.do_linesearch) { af = r.accepted[u]; h = r.hdr_out[u]; dc = r.dcnt[u]; }
        const bool acc = af >= 0;
        unsigned bal = __ballot_sync(0xffffffffu, acc);
        nupd += __popc(bal);
        // the delta blocks of the accepted nodes, four at a time: their first 32 entries are loaded together (independent
        // loads in flight), then added node by node in position order (entries of one node never collide)
        while (bal) {
            int c4[4], d4[4];
            double v4[4];
            const double *dv4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int src = bal ? __ffs(bal) - 1 : 0;
                const bool live = bal != 0u;
                bal &= bal - 1u;
                const uint64_t hs = __shfl_sync(0xffffffffu, h, src);
                const int d = __shfl_sync(0xffffffffu, dc, src);
                d4[k] = live ? d : 0;
                dv4[k] = r.pool_out + sp_off8(hs) + sp_words(sp_cnt(hs));
                const unsigned short *di = sp_idx(dv4[k], (uint32_t)d);
                c4[k] = 0;
                v4[k] = 0.0;
                if (lane < d4[k]) { c4[k] = di[lane]; v4[k] = dv4[k][lane]; }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (lane < d4[k]) Dw[c4[k]] += v4[k];
                if (d4[k] > 32) {                                  // (long delta blocks: the rest of the entries)
                    const unsigned short *di = sp_idx(dv4[k], (uint32_t)d4[k]);
                    for (int i = 32 + lane; i < d4[k]; i += 32) Dw[di[i]] += dv4[k][i];
                }
                __syncwarp();
            }
        }
    }
    llh = warp_sum(llh);
    if (lane == 0) { s_llh[wib] = llh; s_nupd[wib] = nupd; }
    __syncthreads();
    const double *D0 = reinterpret_cast<const double *>(smem_raw);
    double *mine = r.block_part + (size_t)blockIdx.x * (ld + 2);
    for (int c = threadIdx.x; c < ld; c += blockDim.x) {
        double v = 0.0;
        for (int w = 0; w < nw; ++w) v += D0[(size_t)w * ldp + c];
        mine[c] = v;
    }
    if (threadIdx.x == 0) {
        double l = 0.0;
        unsigned int nu = 0;
        for (int w = 0; w < nw; ++w) { l += s_llh[w]; nu += s_nupd[w]; }
        mine[ld] = l;
        mine[ld + 1] = (double)nu;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(r.ticket, 1u) == gridDim.x - 1u) ? 1u : 0u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // block partials: warp w adds a contiguous range of blocks, in block order, for all components (lane-strided, every
    // component's load of a round in flight together); the 16 warp sums are then added in warp order.  A fixed
    // association: the same bits from run to run.
    {
        const unsigned int nb = gridDim.x;
        const unsigned int per = (nb + nw - 1) / nw;
        const unsigned int b0 = min(nb, (unsigned int)wib * per), b1 = min(nb, b0 + per);
        double *Wp = reinterpret_cast<double *>(smem_raw) + (size_t)wib * ldp;          // (ld + 2 <= ldp + 2: the two scalars go to s_llh / s_nupd2)
        double accl = 0.0, accn = 0.0;
        for (int c0 = 0; c0 < ld; c0 += 32 * 4) {
            double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
            const int ca = c0 + lane, cb = ca + 32, cc = ca + 64, cd = ca + 96;
            for (unsigned int b = b0; b < b1; ++b) {
                const double *bp = r.block_part + (size_t)b * (ld + 2);
                if (ca < ld) v0 += __ldcg(bp + ca);
                if (cb < ld) v1 += __ldcg(bp + cb);
                if (cc < ld) v2 += __ldcg(bp + cc);
                if (cd < ld) v3 += __ldcg(bp + cd);
            }
            if (ca < ld) Wp[ca] = v0;
            if (cb < ld) Wp[cb] = v1;
            if (cc < ld) Wp[cc] = v2;
            if (cd < ld) Wp[cd] = v3;
        }
        if (lane < 2) {
            double v = 0.0;
            for (unsigned int b = b0; b < b1; ++b) v += __ldcg(r.block_part + (size_t)b * (ld + 2) + ld + lane);
            if (lane == 0) accl = v; else accn = v;
        }
        accn = __shfl_sync(0xffffffffu, accn, 1);
        __syncthreads();                       // (every warp is done with s_llh / s_nupd of the first phase)
        if (lane == 0) { s_llh[wib] = accl; s_cnt[wib] = accn; }
        __syncthreads();
        for (int c = threadIdx.x; c < ld + 2; c += blockDim.x) {
            double v = 0.0;
            if (c < ld) {
                for (int w = 0; w < nw; ++w) v += D0[(size_t)w * ldp + c];
                r.partials[c] = v;
            } else {
                for (int w = 0; w < nw; ++w) v += (c == ld) ? s_llh[w] : s_cnt[w];
                r.partials[2 * ld + (c - ld)] = v;
            }
            for (int p = 0; p < r.world; ++p) r.xslot[p][c] = v;
        }
    }
    // the next launch starts from a fresh work counter, and the buffer this step read becomes the next output pool
    if (threadIdx.x == 0) {
        if (r.work_counter != nullptr) *r.work_counter = r.work_init;
        if (r.pool_top_in != nullptr) *r.pool_top_in = 0ull;
    }
    if (threadIdx.x == 0) *r.ticket = 0u;
    if (r.world > 0) {
        // the step kernel's rows went to the peers before this kernel started; the slots above follow; only then
        // the flags (system-scope fence in between)
        __threadfence_system();
        __syncthreads();
        if ((int)threadIdx.x < r.world) {
            *reinterpret_cast<volatile unsigned long long *>(r.xflag[threadIdx.x]) = r.seq;
            __threadfence_system();
        }
    }
}

// Multi-GPU: waits until every rank's sums of this step have arrived (flags >= seq), then adds the slots up in rank
// order — every rank gets the same bits — into the partials the finish kernel reads.  One block.
struct XReduceArgs {
    const double *xbuf;                        // world x (ld + 2), this step's half of the local exchange buffer
    const unsigned long long *flags;           // world flags (local memory, written by the peers)
    unsigned long long seq;
    int32_t world, ld;
    double *partials;
    const int32_t *done_flag;
};
__global__ void xreduce_kernel(const XReduceArgs x) {
    if (x.done_flag != nullptr && *x.done_flag != 0) return;
    if ((int)threadIdx.x < x.world) {
        const volatile unsigned long long *f = x.flags + threadIdx.x;
        while (*f < x.seq) __nanosleep(100);
        __threadfence_system();
    }
    __syncthreads();
    const int ld = x.ld;
    for (int c = threadIdx.x; c < ld + 2; c += blockDim.x) {
        double v = 0.0;
        for (int p = 0; p < x.world; ++p) v += __ldcg(x.xbuf + (size_t)p * (ld + 2) + c);
        if (c < ld) x.partials[c] = v;
        else x.partials[2 * ld + (c - ld)] = v;
    }
}

}  // namespace bigclam
