// bigclam_sparse.cuh — the step (codes/bigclam4-7.scala:152-223) over SPARSE rows of F: layout, the general
// one-warp-per-node path (any degree, any row length, K <= 1024) and the split-hub phases.  The tile path for
// small nodes and the kernels themselves are in bigclam_tile.cuh.
//
// Why: the reference keeps F as Breeze sparse vectors (`BSV[Double]`, bigclam4-7.scala:97-104) because the rows
// ARE sparse: on the bench workload (com-amazon, K = 200) a row holds ~9 non-zeros of 200 through the whole
// run and ~17 components are "active" in a line search.  A row is (count, ascending component indices, values)
// in a per-step pool, every neighbour row is read once per step (~112 bytes instead of 1.6 KB), and all
// per-edge work is proportional to the row's non-zeros.
//
// Layout (per F buffer; double-buffered like the dense F):
//   hdr[u]      uint64: (offset in 8-byte words << 24) | count
//   pool        row block at `offset` (16-byte aligned, a multiple of 16 bytes — one bulk copy moves it):
//               vpad(count) doubles, then ipad(count) uint16 indices (ascending);  vpad = count rounded up to 2,
//               ipad = count rounded up to 8.  A node whose step was accepted is followed by its DELTA block in
//               the same format: the non-zero (old - new) components (:191-192), dcnt[u] of them.
//   pool_top    bump allocator of the OUTPUT pool (words), zeroed before every step.  The input pool is only
//               read (Jacobi), so a step whose pool overflowed can simply be repeated with a larger pool.
//
// Per-node results (no floating-point atomics anywhere: the sums over nodes are taken afterwards, in a fixed
// order, by reduce_kernel — bit-identical from run to run):
//   node_llh[u]  llh_u of the PRE block (:168)          accepted[u]  accepted step index, -1 = row kept
//   dcnt[u]      entries of the delta block
//
// General path, per node (one warp), with fu scattered into a dense shared-memory vector fu_d[ld]:
//   PRE   the entries of up to 32 neighbour rows are staged in shared memory; lane e walks row e:
//         x_e = sum_i val_i * fu_d[idx_i]; the gradient sum g_d[idx] += w_e * val goes neighbour by neighbour;
//   scan  one pass over the ld components turns g_d into the gradient (:168), sums |g|^2 and lists the
//         active components (fu > 0 or g > 0);
//   LS    lane (trial j, edge parity h) walks the staged entries of its edges:
//         D = sum_i clamp(fu_d[idx_i] + s_j * g_d[idx_i]) * val_i — an inactive component clamps to 0 and adds
//         exactly nothing; two edges per lane in flight;
//   SWAP  the accepted candidate's non-zeros are compacted (ascending) into the staging buffer, a block is
//         taken from the output pool, the row, its delta block and its header are written.
//
// Limits: ld <= 1024, MIN_F_ == 0.
#pragma once
#include "bigclam_kernels.cuh"

namespace bigclam {

#ifndef BIGCLAM_GEN_BOUNDS          // 1: the line-search bounds of the general path are compiled in (used when SparseArgs::ls_prune > 1)
#define BIGCLAM_GEN_BOUNDS 1
#endif
#ifndef BIGCLAM_GEN_INLINE          // how the general path (one node / one hub item per call, a single call site each) is compiled into the kernel
#define BIGCLAM_GEN_INLINE __forceinline__
#endif

constexpr int kSpBlocksPerSM = 2;
constexpr int kSpWarps = 8;            // warps per block at most; wide rows run fewer (sp_warps_per_block)
constexpr int kSpThreads = kSpWarps * 32;
// staged neighbour entries per chunk of the general path: at least one full row always fits
__host__ __device__ inline int sp_entries(int ld) { return ld > 512 ? ld : 512; }

__host__ __device__ inline uint64_t sp_pack(uint64_t off8, uint32_t cnt) { return (off8 << 24) | (uint64_t)cnt; }
__host__ __device__ inline uint32_t sp_cnt(uint64_t h) { return (uint32_t)(h & 0xffffffull); }
__host__ __device__ inline uint64_t sp_off8(uint64_t h) { return h >> 24; }
__host__ __device__ inline uint32_t sp_vpad(uint32_t cnt) { return (cnt + 1u) & ~1u; }
__host__ __device__ inline uint32_t sp_ipad(uint32_t cnt) { return (cnt + 7u) & ~7u; }
__host__ __device__ inline uint64_t sp_words(uint32_t cnt) { return (uint64_t)sp_vpad(cnt) + sp_ipad(cnt) / 4u; }   // 8-byte words of a block
__host__ __device__ inline const unsigned short *sp_idx(const double *vals, uint32_t cnt) {
    return reinterpret_cast<const unsigned short *>(vals + sp_vpad(cnt));
}
__host__ __device__ inline unsigned short *sp_idx(double *vals, uint32_t cnt) {
    return reinterpret_cast<unsigned short *>(vals + sp_vpad(cnt));
}

struct TileMeta {   // a group of consecutive small nodes of the processing order handled together by one warp
    int32_t pos0;   // first position (index into StepArgs::meta)
    int32_t ecol0;  // first entry of the tile in SparseArgs::tcol
    int32_t nn;     // nodes (<= kTlMaxNodes)
    int32_t ne;     // edges (<= kTlMaxEdges)
};

struct SparseArgs {
    const uint64_t *hdr_in;
    const double *pool_in;
    uint64_t *hdr_out;
    double *pool_out;
    unsigned long long *pool_top;      // words used of this rank's region of pool_out
    uint64_t pool_cap8;                // capacity of that region in words
    uint64_t region_base8;             // where the region starts in pool_out (0 on a single GPU)
    int32_t *overflow;                 // set when a row did not fit (the step must be repeated with a larger pool)
    // per-node results (see the header comment)
    double *node_llh;
    unsigned short *dcnt;
    int8_t *accepted;                  // always written by a line-search launch
    // node-partitioned multi-GPU: the owners' new rows go to the same offsets of every replica's output pool
    // (plain stores to IPC-mapped peer memory over NVLink); each rank allocates only inside its own region, so
    // all replicas end up with the same layout and no remote atomics are needed.
    int32_t n_peers;
    uint64_t *peer_hdr[7];
    double *peer_pool[7];
    unsigned int *hub_work;            // next hub item to hand out (zeroed per launch); items: StepArgs::hub_items
    // work list after the hubs: n_gen nodes for the general path (positions n_hubs ..), then the tiles
    int32_t n_gen;
    int32_t ntiles;
    const TileMeta *tiles;
    const int32_t *tcol;               // per tile edge: neighbour id | (node index within the tile << 28)
    unsigned int *stats;               // optional [tiles done on the tile path, tiles that fell back, nodes line-searched, nodes that asked for it]
    // line search by bounds (bigclam_tile.cuh, H2): 0 = every candidate of every node is evaluated (BIGCLAM_F_LS_EXHAUSTIVE),
    // 1 = bounds on the tile path only, 2 = on the general path too
    int32_t ls_prune;
    float pr_xlo, pr_kinv, pr_cap;     // x_lo rounded down, 1 / (1 - MAX_P_) and S_hi - S_lo rounded up
    // held-out pairs (bigclam_set_holdout): node u's partners ho_col[ho_rowptr[u] .. ho_rowptr[u + 1]); read only by the
    // masked (kHO) instantiation of the step kernel
    const int64_t *ho_rowptr;
    const int32_t *ho_col;
};

// The dense per-warp vectors are padded to a multiple of 32 components (zeros: a padding component has
// fu = sumF = 0, hence gradient 0, never active), so that the loops over components need no bounds checks.
__host__ __device__ inline int sp_ldp(int ld) { return (ld + 31) & ~31; }
// general path, per-warp shared memory:
//   fu_d[ldp] | g_d[ldp] | ent_val[E] | ent_idx[E] u16 | aidx[max(ld, 256)] u16 | poff[40] u16 | cbal[32] u32 | ccum[32] u16
__host__ __device__ inline size_t sp_gen_warp_bytes(int ld) {
    return sizeof(double) * 2 * (size_t)sp_ldp(ld) + (size_t)sp_entries(ld) * 10 + 2 * (size_t)(ld > 256 ? ld : 256) + 2 * 40 + 4 * 32 + 2 * 32;
}

// Split hubs.  A node whose neighbour list is long enough to dominate a launch when one warp walks it is split
// into segments of kSpHubSeg edges that different warps work on; the pieces meet in a global scratch row per
// hub (G[ld] | S1 | ST[16], stride ld + 32 doubles, two counters per hub):
//   phase 1  PRE of one segment: its share of sum_v w_v fv and of S1 into the segment's own slot of the scratch
//            (no atomics: the hub's warps add the slots up in slot order, so the result is reproducible);
//   phase 2  line search of one segment, once all phase-1 segments of the hub are in;
//   phase 3  once per hub, after its phase-2 segments: gradient, active set, Armijo decision, new row.
// Items are handed out in that order by one counter and every warp holds one item at a time on a grid whose
// warps are all resident, so a waiting warp only waits for items that are being processed: no deadlock.
constexpr int kSpHubSeg = 96;
constexpr int kSpHubMaxSlices = 192;      // very large hubs get longer segments: the slot sums are taken by one warp per hub
// scratch of one hub: (nslices + 1) x (ld + 32) doubles: slice sl holds  G_sl[ld] | S1_sl | ST_sl[16], the last
// slot the sums over the slices (G | S1)
__host__ __device__ inline size_t sp_hub_stride(int ld) { return (size_t)ld + 32; }

// ---------------------------------------------------------------------------------------------------------------
// Line search by bounds (derivation: bigclam_tile.cuh, phase H2): the per-node terms of the bound
//   phi(nf_j) - phi(fu) <= min(s Qn, R3) + min(s Qp, G1) - kappa s Mp + c0 + s c1 + Hs_j
// and the test that excludes candidate j.  Shared by the tile path and the general path.
struct LsBound {
    double Qn, Qp, Mp, G1, R3;
    float c0, c1, kap0;
    __device__ __forceinline__ bool cannot_pass(double sj, float Hs, double alpha, double G2node) const {
        const float sfu = __double2float_ru(sj);
        const float kap = fminf(1.0f, __fdividef(kap0, sfu) * 0.9999f);
        const double bound = fmin(sj * Qn, R3) + fmin(sj * Qp, G1) - sj * ((double)kap * Mp) + (double)(fmaf(Hs, 1.00001f, c0) + sfu * c1);
        return bound < (alpha * sj) * G2node * (1.0 - 1.0e-9);
    }
};
// One edge's share Hs of candidate ln(s) = lns given the edge's code (lnthr, Lp): 0 up to lnthr; beyond it
// min(cap, lns + Lp) for an edge that is clamped flat, or the constant -1000 - Lp (an edge next to x_lo, Lp < -500).
__device__ __forceinline__ float ls_edge_share(float lns, float lnthr, float Lp, float cap) {
    if (!(lns > lnthr)) return 0.0f;
    return (Lp < -500.0f) ? (-1000.0f - Lp) : fminf(cap, fmaxf(lns + Lp, 0.0f));
}
// The code of an edge that is clamped flat (x <= x_lo): Dp = sum_c max(g_c, 0) fv_c > 0.
__device__ __forceinline__ void ls_code_flat(float xf, double Dp, float xlo_f, float kinv_f, float &lnthr, float &Lp) {
    const float Df = __double2float_ru(Dp) * 1.000001f;
    const float sthr = (xlo_f - xf) / Df * 0.99999f;                    // x + s Dp stays below x_lo up to here
    if (sthr > 0.0f) {
        const float t1 = __log2f(sthr), t2 = __log2f(kinv_f * (Df + xf / sthr));
        lnthr = t1 * 0.69314718f - fmaf(1.0e-6f, fabsf(t1), 1.0e-4f);
        Lp = t2 * 0.69314718f + fmaf(1.0e-6f, fabsf(t2), 1.0e-4f);
    } else {
        lnthr = -3.0e38f;                                               // (always at the cap)
        Lp = 3.0e38f;
    }
}
// The code of an edge in range next to x_lo with violation `vnear`: charged from x + s En < x_lo on (En < 0).
__device__ __forceinline__ void ls_code_near(double x, double x_lo, double En, float vnear, float &lnthr, float &Lp) {
    const float sthr = __double2float_rd((x - x_lo) / (-En)) * 0.99999f;
    if (sthr > 0.0f) {
        const float t1 = __log2f(sthr);
        lnthr = t1 * 0.69314718f - fmaf(1.0e-6f, fabsf(t1), 1.0e-4f);
    } else {
        lnthr = -3.0e38f;
    }
    Lp = -1000.0f - vnear;
}

// ---------------------------------------------------------------------------------------------------------------
// The general path: everything one warp needs to process one node (or one hub item).
struct SpGen {
    // launch-wide
    const StepArgs *a;
    const SparseArgs *sp;
    const double *s_steps;
    const double *s_sumF;
    const float *s_lns;              // upper bounds of ln(step size), 16 values (line search by bounds)
    EdgeConst ec;
    // per warp
    double *fu_d, *g_d, *ent_val;
    unsigned short *ent_idx, *aidx, *poff, *ccum;
    unsigned int *cbal;
    int lane, ld, ldp, ecap;
    unsigned lt_mask;

    __device__ __forceinline__ void carve(unsigned char *wbase, int ld_, int lane_) {
        ld = ld_;
        ldp = sp_ldp(ld_);
        ecap = sp_entries(ld_);
        lane = lane_;
        lt_mask = (1u << lane_) - 1u;
        fu_d = reinterpret_cast<double *>(wbase);
        g_d = fu_d + ldp;
        ent_val = g_d + ldp;
        ent_idx = reinterpret_cast<unsigned short *>(ent_val + ecap);
        aidx = ent_idx + ecap;
        poff = aidx + (ld > 256 ? ld : 256);
        cbal = reinterpret_cast<unsigned int *>(poff + 40);
        ccum = reinterpret_cast<unsigned short *>(cbal + 32);
    }
    // the tile path uses the same bytes: the dense vectors must be zero whenever the general path starts
    __device__ __forceinline__ void clear_dense() {
#pragma unroll 1
        for (int i = lane; i < ldp; i += 32) { fu_d[i] = 0.0; g_d[i] = 0.0; }
        __syncwarp();
    }

    // Stages the rows of up to 32 neighbours (ids colp[0 .. cnt32), the low 28 bits when `tagged`) of one node
    // into the entry buffer: the longest prefix of them whose entries fit (at least one: a row has at most
    // ld <= ecap entries).  Returns the number ne of staged neighbours; poff[e] .. poff[e + 1] is row e's range.
    __device__ __forceinline__ int stage_chunk(const int32_t *__restrict__ colp, int cnt32) {
        const uint64_t *__restrict__ hdr_in = sp->hdr_in;
        const double *__restrict__ pool_in = sp->pool_in;
        const int v = (lane < cnt32) ? (colp[lane] & 0x0fffffff) : 0;
        const uint64_t hv = (lane < cnt32) ? __ldg(hdr_in + v) : 0ull;
        const int cv = (int)sp_cnt(hv);
        int incl = cv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const unsigned fit = __ballot_sync(0xffffffffu, (lane < cnt32) && (incl <= ecap));
        const int ne = __popc(fit);                     // incl is monotone: the fitting lanes are 0 .. ne-1
        if (lane == 0) poff[0] = 0;
        if (lane < ne) poff[lane + 1] = (unsigned short)incl;
        __syncwarp();
        // the T entries of the ne rows, 32 at a time, one per lane: all loads of a round are in flight together
        const int T = (ne > 0) ? __shfl_sync(0xffffffffu, incl, ne - 1) : 0;
#pragma unroll 1
        for (int base = 0; base < T; base += 32) {
            const int j = base + lane;
            int lo = 0, hi = ne;                                   // row of entry j: the largest e with poff[e] <= j
#pragma unroll
            for (int s = 0; s < 5; ++s) {
                const int mid = (lo + hi) >> 1;
                const bool le = (int)poff[mid] <= j;
                if (hi - lo > 1) { if (le) lo = mid; else hi = mid; }
            }
            const uint64_t he = __shfl_sync(0xffffffffu, hv, lo);
            if (j < T) {
                const int ce = (int)sp_cnt(he);
                const double *vals = pool_in + sp_off8(he);
                const int i = j - (int)poff[lo];
                ent_val[j] = __ldg(vals + i);
                ent_idx[j] = __ldg(sp_idx(vals, (uint32_t)ce) + i);
            }
        }
        __syncwarp();
        return ne;
    }

    // PRE over the edges [eb, ee) of a node whose fu is in fu_d: returns this lane's share of S1 (lane e holds the
    // terms of the chunks' e-th rows); with `axpy` the weighted neighbour rows are added into g_d.  kLin: the pairs are
    // held-out pairs, whose term in the masked objective is x itself with weight 1.
    template <bool kLin = false>
    __device__ __forceinline__ double pre_range(const int32_t *colbase, int eb, int ee, bool axpy, int &nchunks, int &ne_last) {
        double S1 = 0.0;
        nchunks = 0;
        ne_last = 0;
#pragma unroll 1
        for (int cb = eb; cb < ee;) {
            const int ne = stage_chunk(colbase + cb, min(32, ee - cb));
            double x = 0.0;
            if (lane < ne) {
                const int end = poff[lane + 1];
#pragma unroll 1
                for (int i = poff[lane]; i < end; ++i) x = fma(ent_val[i], fu_d[ent_idx[i]], x);
            }
            double w, t;
            if constexpr (kLin) {
                t = x;
                w = 1.0;
            } else {
                t = edge_term<true>(x, ec, w);
            }
            S1 += (lane < ne) ? t : 0.0;
            if (axpy) {
#pragma unroll 1
                for (int e = 0; e < ne; ++e) {
                    const double we = __shfl_sync(0xffffffffu, w, e);
                    const int pe = poff[e], pn = poff[e + 1];
#pragma unroll 1
                    for (int i = pe + lane; i < pn; i += 32) {
                        const int c = ent_idx[i];
                        g_d[c] = fma(we, ent_val[i], g_d[c]);
                    }
                    __syncwarp();
                }
            }
            cb += ne;
            ne_last = ne;
            ++nchunks;
        }
        return S1;
    }
    // g_d (sum of weighted neighbour rows) -> gradient (:168) in place; returns |g|^2, lists the active
    // components in aidx (m of them) and tells whether any candidate can reach MAX_F_.
    __device__ __forceinline__ double scan_gradient(int &m, bool &need_hi) {
        double G2 = 0.0;
        bool hi_lane = false;
        m = 0;
        const double max_f = a->max_f;
#pragma unroll 1
        for (int c0 = 0; c0 < ldp; c0 += 32) {          // (padding components: f = g = 0, inactive)
            const int c = c0 + lane;
            const double f = fu_d[c];
            const double g = (g_d[c] - s_sumF[c]) + f;
            g_d[c] = g;
            G2 = fma(g, g, G2);
            const bool act = (f > 0.0 || g > 0.0);
            const unsigned bal = __ballot_sync(0xffffffffu, act);
            if (act) {
                aidx[m + __popc(bal & lt_mask)] = (unsigned short)c;
                hi_lane |= (f + g > max_f);
            }
            m += __popc(bal);
        }
        G2 = warp_sum(G2);
        need_hi = __any_sync(0xffffffffu, hi_lane);
        __syncwarp();
        return G2;
    }
    // The staged entries of `ne` rows shrink, in place, to those on ACTIVE components (fu > 0 or grad > 0): only
    // they can contribute to a candidate's dot.  Order inside a row is kept, poff is rewritten.
    __device__ __forceinline__ void compact_active(int ne) {
        const int T = poff[ne];
        int total = 0;
#pragma unroll 1
        for (int base = 0; base < T; base += 32) {
            const int j = base + lane;
            const bool in = j < T;
            const int c = in ? (int)ent_idx[j] : 0;
            const double v = in ? ent_val[j] : 0.0;
            const bool act = in && (fu_d[c] > 0.0 || g_d[c] > 0.0);
            const unsigned bal = __ballot_sync(0xffffffffu, act);
            if (lane == 0) { cbal[base >> 5] = bal; ccum[base >> 5] = (unsigned short)total; }
            __syncwarp();                       // this block's reads are done; writes land at or below them
            if (act) {
                const int p = total + __popc(bal & lt_mask);
                ent_idx[p] = (unsigned short)c;
                ent_val[p] = v;
            }
            total += __popc(bal);
        }
        __syncwarp();
        int newp = 0;
        if (lane < ne) {
            const int p = poff[lane];
            newp = (p >= T) ? total : (int)ccum[p >> 5] + __popc(cbal[p >> 5] & ((1u << (p & 31)) - 1u));
        }
        __syncwarp();
        if (lane < ne) poff[lane] = (unsigned short)newp;
        if (lane == 0) poff[ne] = (unsigned short)total;
        __syncwarp();
    }
    // Line search over the edges [eb, ee): lane (j, h) returns the sum over its edges of the clamped edge term
    // for candidate step s; `staged` rows of a single chunk may still be in the buffer from PRE.  kLin: held-out
    // pairs, the term is the dot nf_j.fv itself.
    template <bool kLin = false>
    __device__ __forceinline__ double ls_range(const int32_t *colbase, int eb, int ee, double s, bool need_hi, int staged) {
        const int h = lane >> 4;
        const double max_f = a->max_f;
        double sumterms = 0.0;
#pragma unroll 1
        for (int cb = eb; cb < ee;) {
            const int ne = (staged > 0) ? staged : stage_chunk(colbase + cb, min(32, ee - cb));
            compact_active(ne);
#pragma unroll 1
            for (int e2 = 0; e2 < ne; e2 += 4) {
                const int eA = e2 + h, eB = e2 + 2 + h;
                const bool vA = eA < ne, vB = eB < ne;
                const int iA = vA ? (int)poff[eA] : 0, nA = vA ? (int)poff[eA + 1] - iA : 0;
                const int iB = vB ? (int)poff[eB] : 0, nB = vB ? (int)poff[eB + 1] - iB : 0;
                const int nmax = max(nA, nB);
                double DA = 0.0, DB = 0.0;
#pragma unroll 1
                for (int k = 0; k < nmax; ++k) {
                    const bool ka = k < nA, kb = k < nB;
                    const int ca = ka ? (int)ent_idx[iA + k] : 0, cb2 = kb ? (int)ent_idx[iB + k] : 0;
                    const double pa = ka ? ent_val[iA + k] : 0.0, pb = kb ? ent_val[iB + k] : 0.0;
                    const double fa = fu_d[ca], ga = g_d[ca], fb = fu_d[cb2], gb = g_d[cb2];
                    if (need_hi) {
                        DA = fma(clamp_step0(fa, s, ga, max_f), pa, DA);
                        DB = fma(clamp_step0(fb, s, gb, max_f), pb, DB);
                    } else {
                        DA = fma(clamp_step0_lo(fa, s, ga), pa, DA);
                        DB = fma(clamp_step0_lo(fb, s, gb), pb, DB);
                    }
                }
                double tA, tB;
                if constexpr (kLin) {
                    tA = DA;
                    tB = DB;
                } else {
                    edge_term2(DA, DB, ec, tA, tB);
                }
                sumterms += vA ? tA : 0.0;
                sumterms += vB ? tB : 0.0;
            }
            __syncwarp();
            cb += ne;
        }
        return sumterms;
    }
    // Armijo decision for the 16 candidates tg .. tg+15 given each lane's edge-term sum (already summed over h).
    __device__ __forceinline__ int decide(int tg, double s, bool jok, double sumterms, int m, bool need_hi, double llh_u, double G2, unsigned surv = 0xffffu) {
        const int h = lane >> 4;
        const double max_f = a->max_f;
        // - newfu.sfT + newfu.newfu with sfT = (sumF - fu) + newfu   (:176,:180)
        double oa = 0.0, ob = 0.0;
#pragma unroll 1
        for (int t = h; t < m; t += 2) {
            const int c = aidx[t];
            const double f = fu_d[c], g = g_d[c];
            const double nf = need_hi ? clamp_step0(f, s, g, max_f) : clamp_step0_lo(f, s, g);
            const double sf = (s_sumF[c] - f) + nf;
            oa = fma(nf, sf, oa);
            ob = fma(nf, nf, ob);
        }
        oa += __shfl_xor_sync(0xffffffffu, oa, 16);
        ob += __shfl_xor_sync(0xffffffffu, ob, 16);
        const double result = (sumterms - oa) + ob;
        const double rhs = llh_u + (a->alpha * s) * G2;
        const unsigned pass = __ballot_sync(0xffffffffu, jok && (result >= rhs)) & 0xffffu & surv;
        return pass ? tg + __ffs(pass) - 1 : -1;          // lowest j == largest step (:182 max)
    }
    // SWAP (:183-190): the accepted candidate's non-zeros (or the old row) go to the output pool(s), followed by
    // the delta block (old - new, :191-192) of an accepted node.
    template <bool kPush>
    __device__ __forceinline__ void swap_row(int64_t u, int jstar, int m, int cu, const double *uval, const unsigned short *uidx) {
        const double max_f = a->max_f;
        int cnt_new = 0, nd = 0;
        double s = 0.0;
        __syncwarp();                     // the entry buffers are reused: every lane is done reading the staged rows (PRE, bounds, LS)
        if (jstar >= 0) {
            s = s_steps[jstar];
#pragma unroll 1
            for (int t0 = 0; t0 < m; t0 += 32) {
                const int t = t0 + lane;
                const bool ok = t < m;
                const int c = ok ? (int)aidx[t] : 0;
                const double f = fu_d[c], g = g_d[c];
                const double nr = clamp_step(f, s, g, a->min_f, max_f);
                const bool nz = ok && (nr != 0.0);
                const unsigned bal = __ballot_sync(0xffffffffu, nz);
                if (nz) {
                    const int p = cnt_new + __popc(bal & lt_mask);
                    ent_val[p] = nr;
                    ent_idx[p] = (unsigned short)c;
                }
                cnt_new += __popc(bal);
                nd += __popc(__ballot_sync(0xffffffffu, ok && (f != nr)));
            }
        } else {
#pragma unroll 1
            for (int i = lane; i < cu; i += 32) {
                ent_val[i] = __ldg(uval + i);
                ent_idx[i] = __ldg(uidx + i);
            }
            cnt_new = cu;
        }
        __syncwarp();
        const unsigned long long wrow = sp_words((uint32_t)cnt_new);
        const unsigned long long words = wrow + (nd > 0 ? sp_words((uint32_t)nd) : 0ull);
        unsigned long long rel = 0;
        if (lane == 0 && words > 0) rel = atomicAdd(sp->pool_top, words);
        rel = __shfl_sync(0xffffffffu, rel, 0);
        if (rel + words > sp->pool_cap8) {
            if (lane == 0) { *sp->overflow = 1; sp->hdr_out[u] = sp_pack(0, 0); sp->dcnt[u] = 0; }
            return;
        }
        const unsigned long long off = sp->region_base8 + rel;
        const uint64_t hnew = sp_pack(off, (uint32_t)cnt_new);
        double *ov = sp->pool_out + off;
        unsigned short *oi = sp_idx(ov, (uint32_t)cnt_new);
#pragma unroll 1
        for (int i = lane; i < cnt_new; i += 32) {
            ov[i] = ent_val[i];
            oi[i] = ent_idx[i];
        }
        if (lane == 0) { sp->hdr_out[u] = hnew; sp->dcnt[u] = (unsigned short)nd; }
        if (kPush) {
#pragma unroll 1
            for (int pr = 0; pr < sp->n_peers; ++pr) {
                double *pv = sp->peer_pool[pr] + off;
                unsigned short *pi = sp_idx(pv, (uint32_t)cnt_new);
#pragma unroll 1
                for (int i = lane; i < cnt_new; i += 32) {
                    pv[i] = ent_val[i];
                    pi[i] = ent_idx[i];
                }
                if (lane == 0) sp->peer_hdr[pr][u] = hnew;
            }
        }
        if (nd > 0) {                                    // delta block (local only: the owner reduces it)
            double *dv = ov + wrow;
            unsigned short *di = sp_idx(dv, (uint32_t)nd);
            int q = 0;
#pragma unroll 1
            for (int t0 = 0; t0 < m; t0 += 32) {
                const int t = t0 + lane;
                const bool ok = t < m;
                const int c = ok ? (int)aidx[t] : 0;
                const double f = fu_d[c], g = g_d[c];
                const double nr = clamp_step(f, s, g, a->min_f, max_f);
                const bool ch = ok && (f != nr);
                const unsigned bal = __ballot_sync(0xffffffffu, ch);
                if (ch) {
                    const int p = q + __popc(bal & lt_mask);
                    dv[p] = f - nr;
                    di[p] = (unsigned short)c;
                }
                q += __popc(bal);
            }
        }
    }

    // own row -> fu_d; returns fu.sumF and fu.fu through the references
    __device__ __forceinline__ void scatter_own(int cu, const double *uval, const unsigned short *uidx, double &fusf, double &fufu) {
        fusf = 0.0;
        fufu = 0.0;
#pragma unroll 1
        for (int i = lane; i < cu; i += 32) {
            const double v = __ldg(uval + i);
            const int c = __ldg(uidx + i);
            fu_d[c] = v;
            fusf = fma(v, s_sumF[c], fusf);
            fufu = fma(v, v, fufu);
        }
        fusf = warp_sum(fusf);
        fufu = warp_sum(fufu);
        __syncwarp();
    }

    // Line search by bounds for a node on the general path (gradient in g_d, m active components in aidx): the mask of
    // the candidates 0 .. 15 that the bound cannot exclude.  `staged`: rows of the node's only chunk that are still
    // staged from PRE (0: the chunks are staged again).  Next to x_lo the violation is taken at its cap (w_lo - 1) x.
    __device__ __forceinline__ unsigned bound_mask(const int32_t *colp, int deg, int m, double G2node, double llh_u, double fusf, double fufu, int staged) {
        const int nsteps = a->nsteps;
        const int j = lane & 15, h = lane >> 4;
        // active components: |g|^2 split by sign, R3, G1, max g, sum sumF^2
        float g2n = 0.0f, g2p = 0.0f, r3 = 0.0f, g1p = 0.0f, gmx = 0.0f, sf2 = 0.0f;
#pragma unroll 1
        for (int t = lane; t < m; t += 32) {
            const int c = aidx[t];
            const double f = fu_d[c], g = g_d[c];
            const float ga = __double2float_ru(fabs(g)), ff = __double2float_ru(f), sff = __double2float_ru(fabs(s_sumF[c]));
            r3 = fmaf(ff, fmaf(2.0f, ga, sff) + 3.0f * ff, r3);
            sf2 = fmaf(sff, sff, sf2);
            if (g > 0.0) {
                g2p = fmaf(ga, ga, g2p);
                g1p += ga;
                gmx = fmaxf(gmx, ga);
            } else {
                g2n = fmaf(ga, ga, g2n);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            g2n += __shfl_xor_sync(0xffffffffu, g2n, o);
            g2p += __shfl_xor_sync(0xffffffffu, g2p, o);
            r3 += __shfl_xor_sync(0xffffffffu, r3, o);
            g1p += __shfl_xor_sync(0xffffffffu, g1p, o);
            sf2 += __shfl_xor_sync(0xffffffffu, sf2, o);
            gmx = fmaxf(gmx, __shfl_xor_sync(0xffffffffu, gmx, o));
        }
        // edges, chunk by chunk: x, Dp, En per edge (lane = edge), then every candidate lane (j, h) collects its share
        const float lns = (j < nsteps) ? s_lns[j] : -3.0e38f;
        const float cap_f = sp->pr_cap;
        double sDp = 0.0, sEn = 0.0;
        float sV = 0.0f, Hs = 0.0f;
#pragma unroll 1
        for (int cb = 0; cb < deg;) {
            const int ne = (staged > 0) ? staged : stage_chunk(colp + cb, min(32, deg - cb));
            double x = 0.0, Dp = 0.0, En = 0.0;
            if (lane < ne) {
                const int end = poff[lane + 1];
#pragma unroll 1
                for (int i = poff[lane]; i < end; ++i) {
                    const int c = ent_idx[i];
                    const double v = ent_val[i], f = fu_d[c], g = g_d[c];
                    x = fma(v, f, x);
                    Dp = fma(v, g > 0.0 ? g : 0.0, Dp);
                    En = fma(v, (g < 0.0 && f > 0.0) ? g : 0.0, En);
                }
            }
            float lnthr = 3.0e38f, Lp = 0.0f, violf = 0.0f;
            if (lane < ne) {
                if (x <= ec.x_lo) {
                    if (Dp > 0.0) ls_code_flat(__double2float_ru(x), Dp, sp->pr_xlo, sp->pr_kinv, lnthr, Lp);
                } else {
                    if (x >= ec.x_hi) violf = __double2float_ru((ec.w_hi - 1.0) * (x - ec.x_hi)) * 1.000001f;
                    else if (x < 4.0 * ec.x_lo && En < 0.0)             // (beyond e * x_lo the tangent never fails)
                        ls_code_near(x, ec.x_lo, En, __double2float_ru((ec.w_lo - 1.0) * x) * 1.000001f, lnthr, Lp);
                    Dp = 0.0;
                    En = 0.0;
                }
            }
            sDp += Dp;
            sEn += En;
            sV += violf;
#pragma unroll 1
            for (int r0 = 0; r0 < ne; r0 += 2) {                     // (the two half-warps take alternate edges)
                const int r = r0 + h;
                const float tx = __shfl_sync(0xffffffffu, lnthr, r & 31), ty = __shfl_sync(0xffffffffu, Lp, r & 31);
                if (r < ne) Hs += ls_edge_share(lns, tx, ty, cap_f);
            }
            cb += ne;
        }
        sDp = warp_sum(sDp);
        sEn = warp_sum(sEn);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sV += __shfl_xor_sync(0xffffffffu, sV, o);
        Hs += __shfl_xor_sync(0xffffffffu, Hs, 16);
        LsBound B;
        const double m_lo = ec.w_lo - 1.0;
        B.Qn = (double)(g2n * 1.000001f) - m_lo * sEn;
        B.Qp = (double)(g2p * 1.000001f);
        B.Mp = m_lo * sDp;
        B.G1 = (double)(__double2float_ru(a->max_f) * g1p * 1.0001f);
        B.R3 = (double)(r3 * 1.0001f);
        const float fuf = __double2float_ru(fabs(fusf)), fff = __double2float_ru(fufu), g2f = __double2float_ru(G2node);
        const float r4 = fmaf(2.0f, g2f, sqrtf(g2f) * sqrtf(fmaf(2.0f, sf2, 18.0f * fff)) * 1.0001f);
        const float base = fmaf(2.0f * cap_f, (float)deg, __double2float_ru(fabs(llh_u))) + 2.0f * (fuf + fff) + r3;
        const float nops = 2.3e-16f * (float)(4 * deg + 3 * m + 16);
        B.c0 = fmaf(nops, base, sV) * 1.0001f;
        B.c1 = nops * fmaf(2.0f, r4, __double2float_ru(sDp)) * 1.0001f;
        B.kap0 = (gmx > 0.0f) ? __fdividef(fmaxf(__double2float_rd(a->max_f) - sqrtf(fff) * 1.000001f, 0.0f), gmx) * 0.9999f : 3.0e38f;
        const bool keep = (j < nsteps) && !B.cannot_pass(s_steps[j < nsteps ? j : 0], Hs, a->alpha, G2node);
        return __ballot_sync(0xffffffffu, keep) & 0xffffu;
    }

    // One node, start to finish.  colp: the node's neighbour list (ids in the low 28 bits when it comes from tcol).
    // kHO (masked objective, bigclam_set_holdout): the node's held-out list is walked after its neighbour list, each
    // pair with the linear term x_uv (PRE: S1 += x, g += fv; line search: sumterms += nf_j.fv); the bounds stay off,
    // they were derived for the unmasked objective.
    template <bool kPush, bool kHO = false>
    __device__ BIGCLAM_GEN_INLINE void node(int64_t u, int deg, const int32_t *colp) {
        const uint64_t hu = __ldg(sp->hdr_in + u);
        const int cu = (int)sp_cnt(hu);
        const double *uval = sp->pool_in + sp_off8(hu);
        const unsigned short *uidx = sp_idx(uval, (uint32_t)cu);
        double fusf, fufu;
        scatter_own(cu, uval, uidx, fusf, fufu);
        const bool in_uset = (a->node_mask == nullptr) || (a->node_mask[u] != 0);
        const bool want_ls = a->do_linesearch && in_uset && deg > 0;
        const int nsteps = a->nsteps;
        const int j16 = lane & 15;

        // ---------------- PRE (:157-169) ----------------
        int nchunks, ne_last;
        double S1 = pre_range(colp, 0, deg, want_ls, nchunks, ne_last);
        int hdeg = 0;                                   // held-out pairs of the node (kHO)
        const int32_t *hcol = nullptr;
        if constexpr (kHO) {
            const int64_t h0 = __ldg(sp->ho_rowptr + u);
            hdeg = (int)(__ldg(sp->ho_rowptr + u + 1) - h0);
            hcol = sp->ho_col + h0;
            int hch, hnl;
            S1 += pre_range<true>(hcol, 0, hdeg, want_ls, hch, hnl);
        }
        S1 = warp_sum(S1);
        const double llh_u = (S1 - fusf) + fufu;
        int jstar = -1, m = 0;
        if (want_ls) {
            bool need_hi;
            const double G2 = scan_gradient(m, need_hi);
            // ---------------- LS (:172-182): only if the bounds leave a candidate that can pass ----------------
            unsigned surv = 0xffffu;
            if (!kHO && BIGCLAM_GEN_BOUNDS && sp->ls_prune > 1 && nsteps <= 16) surv = bound_mask(colp, deg, m, G2, llh_u, fusf, fufu, nchunks == 1 ? ne_last : 0);
            if (sp->stats != nullptr && lane == 0) {
                atomicAdd(sp->stats + 3, 1u);
                if (surv != 0u) atomicAdd(sp->stats + 2, 1u);
            }
#pragma unroll 1
            for (int tg = 0; tg < nsteps && jstar < 0 && surv != 0u; tg += 16) {
                const int j = tg + j16;
                const bool jok = j < nsteps;
                const double s = s_steps[jok ? j : 0];
                // a node whose neighbours fitted one chunk still has them staged from PRE (unless held-out pairs
                // were staged after them)
                double sumterms = ls_range(colp, 0, deg, s, need_hi, (nchunks == 1 && tg == 0 && hdeg == 0) ? ne_last : 0);
                if constexpr (kHO) sumterms += ls_range<true>(hcol, 0, hdeg, s, need_hi, 0);
                sumterms += __shfl_xor_sync(0xffffffffu, sumterms, 16);
                jstar = decide(tg, s, jok, sumterms, m, need_hi, llh_u, G2, surv);
            }
        }
        if (lane == 0) sp->node_llh[u] = llh_u;
        if (a->do_linesearch) {
            swap_row<kPush>(u, jstar, m, cu, uval, uidx);
            if (lane == 0) sp->accepted[u] = (int8_t)jstar;
        }
        // ---- leave the dense vectors at zero for the next node ----
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < cu; i += 32) fu_d[__ldg(uidx + i)] = 0.0;
        if (want_ls)
#pragma unroll 1
            for (int c = lane; c < ldp; c += 32) g_d[c] = 0.0;
        __syncwarp();
    }

    // One item of a split hub (see above).
    template <bool kPush>
    __device__ BIGCLAM_GEN_INLINE void hub_item(const HubItem item) {
        const NodeMeta nm = a->meta[item.hub];
        const int64_t u = nm.u, e0 = nm.e0;
        const int deg = nm.deg;
        const size_t hstride = sp_hub_stride(ld);
        double *scr0 = a->hub_scratch + (size_t)item.mslot * hstride;            // mslot: first scratch slot of the hub
        unsigned int *cnt = a->hub_counters + 2 * (size_t)item.hub;
        const int sb = item.slice * item.seg, se = min(deg, sb + item.seg);
        const uint64_t hu = __ldg(sp->hdr_in + u);
        const int cu = (int)sp_cnt(hu);
        const double *uval = sp->pool_in + sp_off8(hu);
        const unsigned short *uidx = sp_idx(uval, (uint32_t)cu);
        double fusf, fufu;
        scatter_own(cu, uval, uidx, fusf, fufu);
        const bool in_uset = (a->node_mask == nullptr) || (a->node_mask[u] != 0);
        const bool want_ls = a->do_linesearch && in_uset;
        const int j16 = lane & 15;
        const int32_t *colp = a->col + e0;
        double *tot = scr0 + (size_t)item.nslices * hstride;                      // the hub's combined slot
        if (item.phase == 1) {
            int nch, nel;
            const double S1 = warp_sum(pre_range(colp, sb, se, want_ls, nch, nel));
            double *scr = scr0 + (size_t)item.slice * hstride;
            if (want_ls) {
#pragma unroll 1
                for (int c = lane; c < ld; c += 32) { scr[c] = g_d[c]; g_d[c] = 0.0; }
            }
            if (lane == 0) scr[ld] = S1;
            __threadfence();
            __syncwarp();
            unsigned int old = 0;
            if (lane == 0) old = atomicAdd(cnt, 1u);
            old = __shfl_sync(0xffffffffu, old, 0);
            if (old == (unsigned int)item.nslices - 1u) {
                // the last segment to arrive adds the slots up, in slot order: whichever warp does it, the sums
                // are the same bits
                __threadfence();
                if (want_ls) {
#pragma unroll 1
                    for (int c = lane; c < ld; c += 32) {
                        double v = 0.0;
#pragma unroll 1
                        for (int sl = 0; sl < item.nslices; ++sl) v += __ldcg(scr0 + (size_t)sl * hstride + c);
                        tot[c] = v;
                    }
                }
                if (lane == 0) {
                    double v = 0.0;
#pragma unroll 1
                    for (int sl = 0; sl < item.nslices; ++sl) v += __ldcg(scr0 + (size_t)sl * hstride + ld);
                    tot[ld] = v;
                }
                __threadfence();
                __syncwarp();
                if (lane == 0) atomicAdd(cnt, 1u);
            }
        } else {
            if (lane == 0) {
                const unsigned int *c = cnt + (item.phase == 2 ? 0 : 1);
                const unsigned int target = (unsigned int)item.nslices + (item.phase == 2 ? 1u : 0u);
                while (*reinterpret_cast<const volatile unsigned int *>(c) < target) __nanosleep(200);
                __threadfence();
            }
            __syncwarp();
            const double llh_u = (__ldcg(tot + ld) - fusf) + fufu;
            int m = 0, jstar = -1;
            bool need_hi = false;
            double G2 = 0.0;
            if (want_ls) {
#pragma unroll 1
                for (int c = lane; c < ldp; c += 32) g_d[c] = (c < ld) ? __ldcg(tot + c) : 0.0;
                __syncwarp();
                G2 = scan_gradient(m, need_hi);
            }
            const int nsteps = a->nsteps;
            const double s = s_steps[j16 < nsteps ? j16 : 0];       // hubs are only split when nsteps <= 16
            if (item.phase == 2) {
                if (want_ls) {
                    double st = ls_range(colp, sb, se, s, need_hi, 0);
                    st += __shfl_xor_sync(0xffffffffu, st, 16);
                    if (lane < 16) scr0[(size_t)item.slice * hstride + ld + 1 + lane] = st;
                }
                __threadfence();
                __syncwarp();
                if (lane == 0) atomicAdd(cnt + 1, 1u);
            } else {
                if (want_ls) {
                    double st = 0.0;
#pragma unroll 1
                    for (int sl = 0; sl < item.nslices; ++sl) st += __ldcg(scr0 + (size_t)sl * hstride + ld + 1 + j16);
                    jstar = decide(0, s, j16 < nsteps, st, m, need_hi, llh_u, G2);
                }
                if (lane == 0) sp->node_llh[u] = llh_u;
                if (a->do_linesearch) {
                    swap_row<kPush>(u, jstar, m, cu, uval, uidx);
                    if (lane == 0) sp->accepted[u] = (int8_t)jstar;
                }
            }
            __syncwarp();
            if (want_ls)
#pragma unroll 1
                for (int c = lane; c < ldp; c += 32) g_d[c] = 0.0;
        }
        __syncwarp();
#pragma unroll 1
        for (int i = lane; i < cu; i += 32) fu_d[__ldg(uidx + i)] = 0.0;
        __syncwarp();
    }
};

// ---------------------------------------------------------------------------------------------------------------
// Held-out log-likelihood of the current F (bigclam_holdout_loglikelihood), every held-out pair once (u < v):
//   L_HO = sum over held-out edges of log(1 - p) + sum over held-out non-edges of log(p),  p = clamp(exp(-Fu.Fv)) (:166).
// One warp per node u scatters u's row into its dense shared-memory vector; lane l scores the pairs (u, v), v > u, at
// positions l, l + 32, ... of u's list by gathering v's entries as PRE does.  Per-node partials (each lane's terms in
// list order, then a fixed butterfly) go to part[u]; holdout_sum_kernel adds them up in node order: reruns give the
// same bits.  The list is here sorted-or-not, symmetric and free of self pairs (bigclam_set_holdout checks).
struct HoLlhArgs {
    const uint64_t *hdr;
    const double *pool;
    const int64_t *ho_rowptr;
    const int32_t *ho_col;
    const uint8_t *ho_edge;
    int64_t n;
    int32_t ld;
    double min_p, max_p;
    double x_lo, x_hi;        // as StepArgs: exp(-x) is only evaluated in between, the clamp decides outside
    double *part;             // n
};
constexpr int kHoWarps = 8;

__global__ void __launch_bounds__(kHoWarps * 32) holdout_llh_kernel(const HoLlhArgs h) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t u = (int64_t)blockIdx.x * kHoWarps + wib;
    if (u >= h.n) return;                                   // (warp-uniform)
    const int ldp = sp_ldp(h.ld);
    double *fu_d = reinterpret_cast<double *>(smem_raw) + (size_t)wib * ldp;
    const int64_t b = h.ho_rowptr[u], e = h.ho_rowptr[u + 1];
    double acc = 0.0;
    if (e > b) {
        for (int i = lane; i < ldp; i += 32) fu_d[i] = 0.0;
        __syncwarp();
        const uint64_t hu = h.hdr[u];
        const int cu = (int)sp_cnt(hu);
        const double *uval = h.pool + sp_off8(hu);
        const unsigned short *uidx = sp_idx(uval, (uint32_t)cu);
        for (int i = lane; i < cu; i += 32) fu_d[uidx[i]] = uval[i];
        __syncwarp();
        for (int64_t q = b + lane; q < e; q += 32) {
            const int v = h.ho_col[q];
            if (v <= u) continue;
            const uint64_t hv = __ldg(h.hdr + v);
            const int cv = (int)sp_cnt(hv);
            const double *vval = h.pool + sp_off8(hv);
            const unsigned short *vidx = sp_idx(vval, (uint32_t)cv);
            double x = 0.0;
            for (int i = 0; i < cv; ++i) x = fma(__ldg(vval + i), fu_d[__ldg(vidx + i)], x);
            const bool inside = (x > h.x_lo) && (x < h.x_hi);
            double p = inside ? exp_neg(x) : (x <= h.x_lo ? h.max_p : h.min_p);
            p = fmin(fmax(p, h.min_p), h.max_p);
            acc += log_pos(h.ho_edge[q] ? 1.0 - p : p);
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) h.part[u] = acc;
}

// sum_u part[u] in a fixed order: thread t adds a contiguous range front to back, the threads' sums meet in a fixed tree.
constexpr int kHoSumThreads = 256;
__global__ void __launch_bounds__(kHoSumThreads) holdout_sum_kernel(const double *part, int64_t n, double *out) {
    __shared__ double s_sum[kHoSumThreads];
    const int t = threadIdx.x;
    const int64_t per = (n + kHoSumThreads - 1) / kHoSumThreads;
    const int64_t b = (int64_t)t * per, e = (b + per < n) ? b + per : n;
    double v = 0.0;
    for (int64_t i = b; i < e; ++i) v += part[i];
    s_sum[t] = v;
    __syncthreads();
    for (int o = kHoSumThreads / 2; o > 0; o >>= 1) {
        if (t < o) s_sum[t] += s_sum[t + o];
        __syncthreads();
    }
    if (t == 0) *out = s_sum[0];
}

// Dense n x ld rows -> sparse rows (one warp per row; non-zeros in ascending component order).
__global__ void dense_to_sparse_kernel(const double *F, int64_t n, int ld, uint64_t *hdr, double *pool,
                                       unsigned long long *pool_top, uint64_t pool_cap8, int32_t *overflow) {
    const int lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= n) return;
    const unsigned lt_mask = (1u << lane) - 1u;
    const double *row = F + (size_t)u * ld;
    int cnt = 0;
    for (int c0 = 0; c0 < ld; c0 += 32) {
        const int c = c0 + lane;
        cnt += __popc(__ballot_sync(0xffffffffu, c < ld && row[c] != 0.0));
    }
    const unsigned long long words = sp_words((uint32_t)cnt);
    unsigned long long off = 0;
    if (lane == 0 && cnt > 0) off = atomicAdd(pool_top, words);
    off = __shfl_sync(0xffffffffu, off, 0);
    if (off + words > pool_cap8) {
        if (lane == 0) { *overflow = 1; hdr[u] = sp_pack(0, 0); }
        return;
    }
    double *ov = pool + off;
    unsigned short *oi = sp_idx(ov, (uint32_t)cnt);
    int p = 0;
    for (int c0 = 0; c0 < ld; c0 += 32) {
        const int c = c0 + lane;
        const double v = (c < ld) ? row[c] : 0.0;
        const unsigned bal = __ballot_sync(0xffffffffu, v != 0.0);
        if (v != 0.0) {
            const int q = p + __popc(bal & lt_mask);
            ov[q] = v;
            oi[q] = (unsigned short)c;
        }
        p += __popc(bal);
    }
    if (lane == 0) hdr[u] = sp_pack(off, (uint32_t)cnt);
}

// Host side of the layout: rows given as CSR (indptr, ascending-or-not indices, values; explicit zeros are dropped)
// -> header + pool image, and back.  Used by bigclam_set_F_csr / bigclam_get_F_csr (and by the emulation tests).
// Returns the number of 8-byte words used, or -1 for an index outside [0, k) / a row longer than ld.
inline int64_t sp_host_pack(int64_t n, int32_t k, int32_t ld, const int64_t *indptr, const int32_t *indices, const double *values,
                            uint64_t *hdr, double *pool, uint64_t pool_cap8, double *colsum /* k, optional */) {
    uint64_t top = 0;
    if (colsum != nullptr)
        for (int32_t c = 0; c < k; ++c) colsum[c] = 0.0;
    for (int64_t u = 0; u < n; ++u) {
        uint32_t cnt = 0;
        for (int64_t i = indptr[u]; i < indptr[u + 1]; ++i) {
            if (indices[i] < 0 || indices[i] >= k) return -1;
            if (values[i] != 0.0) ++cnt;
        }
        if (cnt > (uint32_t)ld) return -1;
        const uint64_t words = sp_words(cnt);
        if (top + words > pool_cap8) return -2;
        double *ov = pool + top;
        unsigned short *oi = sp_idx(ov, cnt);
        for (uint64_t z = 0; z < words; ++z) ov[z] = 0.0;
        uint32_t q = 0;
        for (int64_t i = indptr[u]; i < indptr[u + 1]; ++i) {
            if (values[i] == 0.0) continue;
            // insertion keeps the indices ascending (rows arrive sorted in practice: one comparison per entry)
            uint32_t p = q;
            while (p > 0 && oi[p - 1] > (unsigned short)indices[i]) { oi[p] = oi[p - 1]; ov[p] = ov[p - 1]; --p; }
            oi[p] = (unsigned short)indices[i];
            ov[p] = values[i];
            ++q;
            if (colsum != nullptr) colsum[indices[i]] += values[i];
        }
        hdr[u] = sp_pack(cnt ? top : 0, cnt);
        top += words;
    }
    return (int64_t)top;
}

inline int64_t sp_host_nnz(int64_t n, const uint64_t *hdr) {
    int64_t t = 0;
    for (int64_t u = 0; u < n; ++u) t += sp_cnt(hdr[u]);
    return t;
}

inline void sp_host_unpack(int64_t n, const uint64_t *hdr, const double *pool, int64_t *indptr, int32_t *indices, double *values) {
    int64_t t = 0;
    for (int64_t u = 0; u < n; ++u) {
        indptr[u] = t;
        const uint32_t cnt = sp_cnt(hdr[u]);
        const double *ov = pool + sp_off8(hdr[u]);
        const unsigned short *oi = sp_idx(ov, cnt);
        for (uint32_t i = 0; i < cnt; ++i) { indices[t] = oi[i]; values[t] = ov[i]; ++t; }
    }
    indptr[n] = t;
}

// Sparse rows -> dense n x ld (rows are zeroed here, no separate memset).
__global__ void sparse_to_dense_kernel(const uint64_t *hdr, const double *pool, int64_t n, int ld, double *F) {
    const int lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= n) return;
    double *row = F + (size_t)u * ld;
    for (int c = lane; c < ld; c += 32) row[c] = 0.0;
    __syncwarp();
    const uint64_t h = hdr[u];
    const int cnt = (int)sp_cnt(h);
    const double *vals = pool + sp_off8(h);
    const unsigned short *idx = sp_idx(vals, (uint32_t)cnt);
    for (int i = lane; i < cnt; i += 32) row[idx[i]] = vals[i];
}

}  // namespace bigclam
