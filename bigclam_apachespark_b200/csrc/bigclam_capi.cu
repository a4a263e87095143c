// bigclam_capi.cu — C ABI (include/bigclam_b200.h) over the sm_100a kernels.
// No CPU fallback: every compute entry point launches CUDA kernels or fails.
#include "../../include/bigclam_b200.h"
#include "bigclam_kernels.cuh"
#include "bigclam_sparse.cuh"
#include "bigclam_tile.cuh"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdint>
#include <cstdlib>
#include <numeric>
#include <string>
#include <utility>
#include <vector>

using namespace bigclam;

struct bigclam_ctx {
    bigclam_params p{};
    int64_t n = 0, nnz = 0;
    int32_t ld = 0, c2 = 0;
    int device = 0;
    int num_sms = 0;
    int grid = 0;
    size_t smem_bytes = 0;
    int nsteps = 0;
    double steps[kMaxSteps]{};

    int64_t *d_rowptr = nullptr;
    int32_t *d_col = nullptr;
    NodeMeta *d_meta = nullptr;
    int32_t maxm = 0;
    int64_t order_n = 0;
    int32_t n_hubs = 0;
    int32_t n_hub_items = 0, n_mega = 0;
    HubItem *d_hub_items = nullptr;
    double *d_hub_scratch = nullptr;
    unsigned int *d_hub_counters = nullptr;
    int64_t lo = 0, hi = 0;
    double *d_F[2] = {nullptr, nullptr};
    double *d_sumF[2] = {nullptr, nullptr};
    int cur = 0;                // index of the current F / sumF buffer
    double *d_partials = nullptr;
    int8_t *d_accepted = nullptr;   // accepted step index per node of the last COMMITTED step
    int8_t *d_accepted_spec = nullptr;   // written by a speculative step (bigclam_step), swapped in at commit
    bool spec_valid = false;        // the next step has already been computed speculatively (see bigclam_step)
    bool spec_null_mask = true;
    std::vector<uint8_t> spec_mask;    // the uset the speculative step was computed with (exact comparison)
    uint8_t *d_mask = nullptr;
    int32_t *d_done = nullptr;
    unsigned int *d_work = nullptr;
    int8_t *d_changed = nullptr;   // multi-GPU: row changed in the most recent step
    int n_peers = 0;
    double *peer_F[2][7] = {{nullptr}};   // peers' F buffers (both halves), IPC-mapped
    RunState *d_state = nullptr;
    double *d_trace = nullptr;
    int64_t trace_cap = 0;
    double *h_pinned = nullptr; // small pinned staging (partials / state)

    cudaStream_t stream = nullptr;
    bool own_stream = false;

    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    double last_step_ms = 0.0;
    int64_t last_step_launches = 0, last_all_launches = 0;

    unsigned int h_work_init = 0;

    // sparse rows of F (BIGCLAM_F_SPARSE_ROWS, bigclam_sparse.cuh): header + pool per F buffer
    bool sparse = false;
    uint64_t *d_hdr[2] = {nullptr, nullptr};
    double *d_pool[2] = {nullptr, nullptr};
    uint64_t pool_cap8 = 0;
    unsigned long long *d_pool_top = nullptr;   // [2]
    int32_t *d_overflow = nullptr;
    int sp_grid = 0, sp_wpb = kSpWarps;
    size_t sp_smem = 0;
    bool dense_valid = true;       // d_F[cur] mirrors the sparse state (set_F; refreshed on demand by ensure_dense)
    uint64_t region_base8 = 0, region_cap8 = 0;   // this rank's part of every replica's output pool (multi-GPU)
    uint64_t *peer_hdr[2][7] = {{nullptr}};       // peers' headers / pools (both halves), IPC-mapped
    double *peer_pool[2][7] = {{nullptr}};
    // per-node results of a launch and the fixed-order reduction behind it (bigclam_tile.cuh)
    double *d_node_llh = nullptr;
    unsigned short *d_dcnt = nullptr;
    double *d_block_part = nullptr;
    unsigned int *d_ticket = nullptr;
    int red_grid = 0;
    // tiles of small nodes (bigclam_tile.cuh) and the nodes of the general path in front of them
    TileMeta *d_tiles = nullptr;
    int32_t *d_tcol = nullptr;
    int32_t ntiles = 0, n_gen = 0;
    int32_t tile_edges = kTlMaxEdges;             // edge budget of a tile (0: no tiles), see retile()
    int32_t tile_nodes = kTlMaxNodes;             // node budget of a tile
    double tile_avg16 = 1.0;                      // average row size (16-byte chunks) the tiles were cut for
    unsigned int stats_seen[2] = {0u, 0u};        // d_stats at the last look (maybe_retile)
    unsigned int stats_read[2] = {0u, 0u};        // d_stats at the last bigclam_get_tile_stats
    unsigned int *d_stats = nullptr;              // [tiles on the tile path, tiles that fell back, nodes line-searched, nodes that asked for it]
    unsigned int ls_read[2] = {0u, 0u};           // d_stats[2..3] at the last bigclam_get_ls_stats
    int ls_level = 1;                             // bounds on the tile path (1); 2 = on the general path too (BIGCLAM_LS_PRUNE=2: pays off only
                                                  // where most nodes have stopped moving AND the general path matters, e.g. com-amazon K=500: -4 %;
                                                  // Email-Enron K=50 +27 %, R-MAT K=1000 +38 %: the chunks are staged once more)
    bool ls_exhaustive = false;                   // BIGCLAM_F_LS_EXHAUSTIVE (or the environment variable BIGCLAM_LS_EXHAUSTIVE=1)
    // fused collective of the node-partitioned path (reduce_kernel publishes, xreduce_kernel adds up): this rank's
    // exchange buffer [2 halves][world][ld + 2] and flags [world], and every rank's (peer memory, incl. our own)
    int x_world = 0, x_rank = 0;
    unsigned long long x_seq = 0;                 // collectives issued so far (same count on every rank)
    double *d_xbuf = nullptr;
    unsigned long long *d_xflags = nullptr;
    double *x_peer_buf[8] = {nullptr};
    unsigned long long *x_peer_flags[8] = {nullptr};
    bool x_ipc = false;                           // peers' buffers came through CUDA IPC (closed on destroy)
    bool local_mask = false;                      // bigclam_set_uset: the node-partitioned step kernels honour d_mask
    bool work_clean = false;                      // the previous launch's reduction has reset the work counter
    bool top_clean[2] = {false, false};           // ... and zeroed this pool's bump allocator
    std::vector<int64_t> h_rowptr;                // host copy of the CSR row pointers (order / tile rebuilds)
    std::vector<int32_t> h_col;
    std::vector<int32_t> h_owned;                 // owned nodes (processing order is derived from it)
    // held-out pairs (bigclam_set_holdout): while set, the steps and the LLH use the masked objective and every node
    // goes through the general path (tile_step_kernel<.., .., true>: no tiles, no split hubs, no bounds)
    bool ho = false;
    int64_t *d_ho_rowptr = nullptr;
    int32_t *d_ho_col = nullptr;
    uint8_t *d_ho_edge = nullptr;
    double *d_ho_part = nullptr;                  // per-node partials of the held-out LLH (n) | their sum
    int64_t ho_pairs = 0;                         // unordered held-out pairs

    std::string err;
};

static thread_local std::string g_create_err;   // bigclam_create failures (no context yet), per calling thread

static int fail(bigclam_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    std::vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c != nullptr) c->err = buf; else g_create_err = buf;
    return code;
}

#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return fail(ctx, BIGCLAM_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                      \
    } while (0)

// The reduction behind a sparse step kernel resets the work counter and the next output pool's allocator on the
// device; whenever the host changes the state behind its back (or a loop may have ended on no-op kernels) the next
// launch does it with memory operations again.
static void invalidate_resets(bigclam_ctx *ctx) {
    ctx->work_clean = false;
    ctx->top_clean[0] = ctx->top_clean[1] = false;
}

// A speculative step (bigclam_step) left its partial sums in d_partials: forget both.
static int drop_speculation(bigclam_ctx *ctx) {
    if (!ctx->spec_valid) return BIGCLAM_OK;
    ctx->spec_valid = false;
    CU(cudaMemsetAsync(ctx->d_partials, 0, sizeof(double) * (2 * (size_t)ctx->ld + 2), ctx->stream));
    return BIGCLAM_OK;
}

static int ensure_dense(bigclam_ctx *ctx);
static int check_overflow(bigclam_ctx *ctx);

extern "C" const char *bigclam_version(void) { return "bigclam_b200 0.1 (sm_100a)"; }

extern "C" int bigclam_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return BIGCLAM_ECUDA; }
    return n;
}

extern "C" int bigclam_default_params(bigclam_params *p, int32_t k) {
    if (p == nullptr || k <= 0) return BIGCLAM_EINVAL;
    p->k = k;
    p->max_inter = 15;
    p->alpha = 0.05;
    p->beta = 0.1;
    p->min_p = 0.0001;
    p->max_p = 0.9999;
    p->min_f = 0.0;
    p->max_f = 1000.0;
    p->device = -1;
    p->flags = 0;
    return BIGCLAM_OK;
}

extern "C" int bigclam_step_sizes(double beta, int32_t max_inter, double *out) {
    if (out == nullptr || max_inter < 0) return BIGCLAM_EINVAL;
    double s = 1.0;                       // bigclam4-7.scala:28
    out[0] = s;
    for (int i = 1; i <= max_inter; ++i) { s *= beta; out[i] = s; }   // :31-32
    return BIGCLAM_OK;
}

extern "C" const char *bigclam_last_error(const bigclam_ctx *ctx) {
    return ctx != nullptr ? ctx->err.c_str() : g_create_err.c_str();
}

static void free_ctx(bigclam_ctx *c) {
    if (c == nullptr) return;
    cudaSetDevice(c->device);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    cudaFree(c->d_rowptr); cudaFree(c->d_col); cudaFree(c->d_meta);
    cudaFree(c->d_F[0]); cudaFree(c->d_F[1]);
    cudaFree(c->d_sumF[0]); cudaFree(c->d_sumF[1]);
    cudaFree(c->d_partials); cudaFree(c->d_accepted); cudaFree(c->d_accepted_spec); cudaFree(c->d_mask);
    cudaFree(c->d_done); cudaFree(c->d_work); cudaFree(c->d_hub_items); cudaFree(c->d_hub_scratch); cudaFree(c->d_hub_counters); cudaFree(c->d_changed);
    for (int h = 0; h < 2; ++h)
        for (int r = 0; r < c->n_peers; ++r) {
            if (c->peer_F[h][r]) cudaIpcCloseMemHandle(c->peer_F[h][r]);
            if (c->peer_hdr[h][r]) cudaIpcCloseMemHandle(c->peer_hdr[h][r]);
            if (c->peer_pool[h][r]) cudaIpcCloseMemHandle(c->peer_pool[h][r]);
        }
    cudaFree(c->d_state); cudaFree(c->d_trace);
    cudaFree(c->d_hdr[0]); cudaFree(c->d_hdr[1]); cudaFree(c->d_pool[0]); cudaFree(c->d_pool[1]);
    cudaFree(c->d_pool_top); cudaFree(c->d_overflow);
    cudaFree(c->d_node_llh); cudaFree(c->d_dcnt); cudaFree(c->d_block_part); cudaFree(c->d_ticket);
    cudaFree(c->d_tiles); cudaFree(c->d_tcol); cudaFree(c->d_stats);
    cudaFree(c->d_ho_rowptr); cudaFree(c->d_ho_col); cudaFree(c->d_ho_edge); cudaFree(c->d_ho_part);
    if (c->x_ipc)
        for (int r = 0; r < c->x_world; ++r)
            if (r != c->x_rank) {
                if (c->x_peer_buf[r]) cudaIpcCloseMemHandle(c->x_peer_buf[r]);
                if (c->x_peer_flags[r]) cudaIpcCloseMemHandle(c->x_peer_flags[r]);
            }
    cudaFree(c->d_xbuf); cudaFree(c->d_xflags);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" void bigclam_destroy(bigclam_ctx *ctx) { free_ctx(ctx); }

template <int C2, bool kHub, bool kPush>
static cudaError_t configure_one(size_t smem, int *blocks_per_sm) {
    constexpr int R = RowsInFlight<C2>::value;
    cudaError_t e = cudaFuncSetAttribute(step_kernel<C2, R, kHub, kPush>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, step_kernel<C2, R, kHub, kPush>, kBlockThreads, smem);
}

template <int C2>
static cudaError_t configure_kernel(size_t smem, int *blocks_per_sm) {
    // the persistent grid must be resident for EVERY variant that may be launched on it (mega-hub slices wait for each other
    // across blocks): the smallest occupancy of the four sizes it (the hub variants use more static shared memory and registers)
    int b = 0;
    cudaError_t e = configure_one<C2, false, false>(smem, blocks_per_sm);
    if (e == cudaSuccess) { e = configure_one<C2, true, false>(smem, &b); if (e == cudaSuccess && b > 0) *blocks_per_sm = std::min(*blocks_per_sm, b); }
    if (e == cudaSuccess) { e = configure_one<C2, false, true>(smem, &b); if (e == cudaSuccess && b > 0) *blocks_per_sm = std::min(*blocks_per_sm, b); }
    if (e == cudaSuccess) { e = configure_one<C2, true, true>(smem, &b); if (e == cudaSuccess && b > 0) *blocks_per_sm = std::min(*blocks_per_sm, b); }
    return e;
}

template <int C2>
static void launch_step_t(const StepArgs &a, int grid, size_t smem, cudaStream_t st) {
    constexpr int R = RowsInFlight<C2>::value;
    const bool hub = a.n_hubs > 0, push = a.n_peers > 0;
    if (hub && push) step_kernel<C2, R, true, true><<<grid, kBlockThreads, smem, st>>>(a);
    else if (hub) step_kernel<C2, R, true, false><<<grid, kBlockThreads, smem, st>>>(a);
    else if (push) step_kernel<C2, R, false, true><<<grid, kBlockThreads, smem, st>>>(a);
    else step_kernel<C2, R, false, false><<<grid, kBlockThreads, smem, st>>>(a);
}

static void launch_step(int c2, const StepArgs &a, int grid, size_t smem, cudaStream_t st) {
    switch (c2) {
        case 1: launch_step_t<1>(a, grid, smem, st); break;
        case 2: launch_step_t<2>(a, grid, smem, st); break;
        case 4: launch_step_t<4>(a, grid, smem, st); break;
        case 8: launch_step_t<8>(a, grid, smem, st); break;
        default: launch_step_t<16>(a, grid, smem, st); break;
    }
}

// Sparse rows: hub items, the nodes of the general path and the tiles of small nodes (bigclam_tile.cuh) for the
// processing order `meta` (degree descending).  Needs the host copy of col (ctx->h_col).
static int rebuild_sparse_lists(bigclam_ctx *ctx, const std::vector<NodeMeta> &meta) {
    const int64_t cnt = (int64_t)meta.size();
    int64_t own_nnz = 0;
    for (int64_t i = 0; i < cnt; ++i) own_nnz += meta[(size_t)i].deg;
    // a hub is split into kSpHubSeg-edge segments over warps when one warp walking it would take a sizeable
    // part of the launch: from an eighth of a warp's share of the owned entries upwards, at least 2 segments' worth
    // of edges (a 1,383-edge node of Email-Enron walked by one warp WAS the launch: 1.3 ms for 367 K entries)
    // (BIGCLAM_SPARSE_HUB_DEG overrides the threshold: tests)
    int32_t nh = 0;
    if (ctx->nsteps <= 16 && !ctx->ho) {
        const int64_t sp_per_warp = own_nnz / std::max<int64_t>(1, (int64_t)ctx->sp_grid * ctx->sp_wpb);
        int64_t sp_hub_deg = std::max<int64_t>(2 * kSpHubSeg, sp_per_warp / 8);
        if (const char *ev = std::getenv("BIGCLAM_SPARSE_HUB_DEG")) sp_hub_deg = std::max<int64_t>(1, std::atoll(ev));
        while (nh < cnt && meta[(size_t)nh].deg >= sp_hub_deg) ++nh;
    }
    ctx->n_hubs = nh;
    {
        std::vector<HubItem> i1, i2, i3;
        int32_t slots = 0;
        for (int32_t i = 0; i < nh; ++i) {
            const int32_t deg = meta[(size_t)i].deg;
            HubItem it{};
            it.hub = i;
            it.seg = std::max(kSpHubSeg, (deg + kSpHubMaxSlices - 1) / kSpHubMaxSlices);
            it.nslices = (deg + it.seg - 1) / it.seg;
            it.mslot = slots;                           // first scratch slot of the hub: nslices + 1 slots
            slots += it.nslices + 1;
            for (int32_t sl = 0; sl < it.nslices; ++sl) {
                it.slice = sl;
                it.phase = 1; i1.push_back(it);
                it.phase = 2; i2.push_back(it);
            }
            it.slice = 0;
            it.phase = 3; i3.push_back(it);
        }
        std::vector<HubItem> items;
        items.insert(items.end(), i1.begin(), i1.end());
        items.insert(items.end(), i2.begin(), i2.end());
        items.insert(items.end(), i3.begin(), i3.end());
        cudaFree(ctx->d_hub_items); ctx->d_hub_items = nullptr;
        cudaFree(ctx->d_hub_scratch); ctx->d_hub_scratch = nullptr;
        cudaFree(ctx->d_hub_counters); ctx->d_hub_counters = nullptr;
        ctx->n_hub_items = (int32_t)items.size();
        ctx->n_mega = nh;
        if (!items.empty()) {
            CU(cudaMalloc(&ctx->d_hub_items, sizeof(HubItem) * items.size()));
            CU(cudaMemcpy(ctx->d_hub_items, items.data(), sizeof(HubItem) * items.size(), cudaMemcpyHostToDevice));
        }
        CU(cudaMalloc(&ctx->d_hub_scratch, sizeof(double) * (size_t)std::max<int32_t>(1, slots) * sp_hub_stride(ctx->ld)));
        CU(cudaMalloc(&ctx->d_hub_counters, sizeof(unsigned int) * (2 * (size_t)std::max<int32_t>(1, nh) + 1)));   // + the item counter
        CU(cudaMemset(ctx->d_hub_counters, 0, sizeof(unsigned int) * (2 * (size_t)std::max<int32_t>(1, nh) + 1)));
    }
    // after the hubs: nodes above the tile budget go one per warp (general path), the rest in tiles of up to
    // kTlMaxNodes consecutive nodes with at most tile_edges edges (held-out pairs: no tiles)
    const int32_t budget = (ctx->nsteps <= 16 && !ctx->ho) ? ctx->tile_edges : 0;
    int64_t pos = nh;
    while (pos < cnt && (budget <= 0 || meta[(size_t)pos].deg > budget)) ++pos;
    ctx->n_gen = (int32_t)(pos - nh);
    std::vector<TileMeta> tiles;
    std::vector<int32_t> tcol;
    while (pos < cnt) {
        TileMeta t{};
        t.pos0 = (int32_t)pos;
        t.ecol0 = (int32_t)tcol.size();
        while (pos < cnt && t.nn < ctx->tile_nodes && t.ne + meta[(size_t)pos].deg <= budget) {
            const NodeMeta &m = meta[(size_t)pos];
            for (int32_t e = 0; e < m.deg; ++e) tcol.push_back(ctx->h_col[(size_t)(m.e0 + e)] | (int32_t)((uint32_t)t.nn << 28));
            t.ne += m.deg;
            ++t.nn;
            ++pos;
        }
        tiles.push_back(t);
    }
    ctx->ntiles = (int32_t)tiles.size();
    cudaFree(ctx->d_tiles); ctx->d_tiles = nullptr;
    cudaFree(ctx->d_tcol); ctx->d_tcol = nullptr;
    if (!tiles.empty()) {
        CU(cudaMalloc(&ctx->d_tiles, sizeof(TileMeta) * tiles.size()));
        CU(cudaMemcpy(ctx->d_tiles, tiles.data(), sizeof(TileMeta) * tiles.size(), cudaMemcpyHostToDevice));
        CU(cudaMalloc(&ctx->d_tcol, sizeof(int32_t) * std::max<size_t>(1, tcol.size())));
        if (!tcol.empty()) CU(cudaMemcpy(ctx->d_tcol, tcol.data(), sizeof(int32_t) * tcol.size(), cudaMemcpyHostToDevice));
    }
    // the reduction walks the processing order with a fixed grid
    ctx->red_grid = (int)std::max<int64_t>(1, std::min<int64_t>(2 * (int64_t)ctx->num_sms, (cnt + 32 * red_warps(ctx->ld) - 1) / (32 * red_warps(ctx->ld))));
    cudaFree(ctx->d_block_part); ctx->d_block_part = nullptr;
    CU(cudaMalloc(&ctx->d_block_part, sizeof(double) * (size_t)ctx->red_grid * ((size_t)ctx->ld + 2)));
    invalidate_resets(ctx);
    ctx->h_work_init = 0;                                  // every item of the sparse kernel is handed out dynamically
    if (ctx->d_work != nullptr) CU(cudaMemcpy(ctx->d_work + 1, &ctx->h_work_init, sizeof(unsigned int), cudaMemcpyHostToDevice));
    return BIGCLAM_OK;
}

static int rebuild_order_list(bigclam_ctx *ctx, const std::vector<int64_t> &rowptr_host, std::vector<int32_t> &order) {
    // Processing order over the owned nodes: degree descending (hubs first so the tail of the
    // launch is made of cheap nodes), ties by id; packed as NodeMeta so one 16-byte load gives a
    // warp everything it needs to start a node.
    const int64_t cnt = (int64_t)order.size();
    ctx->h_owned = order;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
        return (rowptr_host[a + 1] - rowptr_host[a]) > (rowptr_host[b + 1] - rowptr_host[b]);
    });
    std::vector<NodeMeta> meta((size_t)cnt);
    for (int64_t i = 0; i < cnt; ++i) {
        const int32_t u = order[(size_t)i];
        meta[(size_t)i].u = u;
        meta[(size_t)i].deg = (int32_t)(rowptr_host[u + 1] - rowptr_host[u]);
        meta[(size_t)i].e0 = rowptr_host[u];
    }
    if (ctx->d_meta == nullptr) CU(cudaMalloc(&ctx->d_meta, sizeof(NodeMeta) * std::max<size_t>(1, (size_t)ctx->n)));
    if (cnt > 0) CU(cudaMemcpy(ctx->d_meta, meta.data(), sizeof(NodeMeta) * (size_t)cnt, cudaMemcpyHostToDevice));
    ctx->order_n = cnt;
    if (ctx->sparse) return rebuild_sparse_lists(ctx, meta);
    // hubs (block-cooperative phase): only the C2 <= 4 kernels have the staging buffers the phase uses
    int32_t nh = 0;
    // a node is worth sharing among a block's warps when its serial chain (~ its degree) is a sizeable
    // fraction of what one warp processes in the whole launch (owned entries / #warps); below that the
    // hubs-first order already hides it
    int64_t own_nnz = 0;
    for (int64_t i = 0; i < cnt; ++i) own_nnz += meta[(size_t)i].deg;
    const int64_t per_warp = own_nnz / std::max<int64_t>(1, (int64_t)ctx->grid * kWarpsPerBlock);
    // When even the largest node's serial chain fits well inside one warp's share of the launch, the
    // hubs-first order hides it and the launch uses the leaner hub-free kernel variant; otherwise nodes
    // from a fifth of that share upwards (at most 512 edges) are shared by blocks.
    const int64_t max_deg = (cnt > 0) ? meta[0].deg : 0;
    const int64_t hub_deg = (4 * max_deg <= 3 * per_warp) ? INT64_MAX
                                                          : std::min<int64_t>(512, std::max<int64_t>(kHubDegree, per_warp / 5));
    if (ctx->c2 <= 4) while (nh < cnt && meta[(size_t)nh].deg >= hub_deg) ++nh;
    ctx->n_hubs = nh;
    // work items of the hub phase: hubs above kHubSlice edges are split into slices handled by different
    // blocks (phases 1-3), the others are done by one block (phase 0); see hub_phase
    {
        std::vector<HubItem> i1, i0, i2, i3;
        int32_t n_mega = 0;
        for (int32_t i = 0; i < nh; ++i) {
            const int32_t deg = meta[(size_t)i].deg;
            const int32_t nsl = (deg + kHubSlice - 1) / kHubSlice;
            HubItem it{};
            it.hub = i;
            if (nsl > 1 && ctx->nsteps <= 16) {
                it.mslot = n_mega++;
                it.nslices = nsl;
                for (int32_t sl = 0; sl < nsl; ++sl) {
                    it.slice = sl;
                    it.phase = 1; i1.push_back(it);
                    it.phase = 2; i2.push_back(it);
                }
                it.slice = 0;
                it.phase = 3; i3.push_back(it);
            } else {
                it.phase = 0; it.nslices = 1; it.mslot = 0;
                i0.push_back(it);
            }
        }
        std::vector<HubItem> items;
        items.insert(items.end(), i1.begin(), i1.end());
        items.insert(items.end(), i0.begin(), i0.end());
        items.insert(items.end(), i2.begin(), i2.end());
        items.insert(items.end(), i3.begin(), i3.end());
        cudaFree(ctx->d_hub_items); ctx->d_hub_items = nullptr;
        cudaFree(ctx->d_hub_scratch); ctx->d_hub_scratch = nullptr;
        cudaFree(ctx->d_hub_counters); ctx->d_hub_counters = nullptr;
        ctx->n_hub_items = (int32_t)items.size();
        ctx->n_mega = n_mega;
        if (!items.empty()) {
            CU(cudaMalloc(&ctx->d_hub_items, sizeof(HubItem) * items.size()));
            CU(cudaMemcpy(ctx->d_hub_items, items.data(), sizeof(HubItem) * items.size(), cudaMemcpyHostToDevice));
        }
        const size_t slots = (size_t)std::max<int32_t>(1, n_mega);
        CU(cudaMalloc(&ctx->d_hub_scratch, sizeof(double) * slots * ((size_t)ctx->ld + 32)));
        CU(cudaMalloc(&ctx->d_hub_counters, sizeof(unsigned int) * (2 * slots + 1)));
        CU(cudaMemset(ctx->d_hub_counters, 0, sizeof(unsigned int) * (2 * slots + 1)));
    }
    const unsigned int init = (unsigned int)nh + 3u * (unsigned int)ctx->grid * kWarpsPerBlock;
    ctx->h_work_init = init;
    if (ctx->d_work != nullptr) CU(cudaMemcpy(ctx->d_work + 1, &init, sizeof(unsigned int), cudaMemcpyHostToDevice));
    return BIGCLAM_OK;
}

static int rebuild_order(bigclam_ctx *ctx, const std::vector<int64_t> &rowptr_host) {
    std::vector<int32_t> order((size_t)(ctx->hi - ctx->lo));
    std::iota(order.begin(), order.end(), (int32_t)ctx->lo);
    return rebuild_order_list(ctx, rowptr_host, order);
}

extern "C" int bigclam_create(bigclam_ctx **out, int64_t n, const int64_t *rowptr, const int32_t *col,
                              const bigclam_params *params) {
    bigclam_ctx *ctx = nullptr;   // errors before allocation go to g_create_err
    if (out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: out is NULL");
    *out = nullptr;
    if (params == nullptr || rowptr == nullptr || n <= 0 || n >= ((int64_t)1 << 31))
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: bad n/rowptr/params");
    if (params->k <= 0) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: k must be > 0");
    if (params->max_inter < 0 || params->max_inter + 1 > kMaxSteps)
        return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_create: max_inter must be in [0,%d]", kMaxSteps - 1);
    if (!(params->min_p > 0.0 && params->min_p < params->max_p && params->max_p < 1.0))
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: need 0 < min_p < max_p < 1");
    if (!(params->min_f <= params->max_f)) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: min_f > max_f");
    const int32_t ld = (params->k + 3) & ~3;
    if (ld > 1024)
        return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_create: k = %d > 1024 not supported by this build", params->k);
    const int64_t nnz = rowptr[n];
    if (rowptr[0] != 0 || nnz < 0) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: rowptr[0] != 0 or nnz < 0");
    for (int64_t u = 0; u < n; ++u)
        if (rowptr[u + 1] < rowptr[u]) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: rowptr not monotone at %lld", (long long)u);
    if (nnz > 0 && col == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: col is NULL");
    for (int64_t e = 0; e < nnz; ++e)
        if (col[e] < 0 || col[e] >= n) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: col[%lld] out of range", (long long)e);

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        (void)cudaGetLastError();
        return fail(ctx, BIGCLAM_ECUDA, "bigclam_create: no CUDA device (this library has no CPU fallback)");
    }
    int dev = params->device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= ndev) return fail(ctx, BIGCLAM_EINVAL, "bigclam_create: device %d of %d", dev, ndev);

    ctx = new (std::nothrow) bigclam_ctx();
    if (ctx == nullptr) return fail(nullptr, BIGCLAM_ENOMEM, "bigclam_create: out of host memory");
    ctx->p = *params;
    ctx->n = n;
    ctx->nnz = nnz;
    ctx->ld = ld;
    ctx->device = dev;
    ctx->lo = 0;
    ctx->hi = n;
    ctx->nsteps = params->max_inter + 1;
    bigclam_step_sizes(params->beta, params->max_inter, ctx->steps);
    const int ld2 = ld / 2;
    const int c2raw = (ld2 + 31) / 32;
    ctx->c2 = c2raw <= 1 ? 1 : c2raw <= 2 ? 2 : c2raw <= 4 ? 4 : c2raw <= 8 ? 8 : 16;
    ctx->maxm = std::min<int32_t>(ld, kMaxActiveCap);
    ctx->smem_bytes = block_smem_bytes(ld, ctx->maxm);

#define CUC(call)                                                                                 \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            fail(nullptr, BIGCLAM_ECUDA, "%s failed: %s", #call, cudaGetErrorString(e__));        \
            free_ctx(ctx);                                                                        \
            return BIGCLAM_ECUDA;                                                                 \
        }                                                                                         \
    } while (0)

    CUC(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, dev));
    ctx->num_sms = prop.multiProcessorCount;
    if (prop.major < 10) {
        fail(nullptr, BIGCLAM_ECUDA, "bigclam_create: device sm_%d%d, this library is built for sm_100a only", prop.major, prop.minor);
        free_ctx(ctx);
        return BIGCLAM_ECUDA;
    }
    int bps = 0;
    cudaError_t ce;
    switch (ctx->c2) {
        case 1: ce = configure_kernel<1>(ctx->smem_bytes, &bps); break;
        case 2: ce = configure_kernel<2>(ctx->smem_bytes, &bps); break;
        case 4: ce = configure_kernel<4>(ctx->smem_bytes, &bps); break;
        case 8: ce = configure_kernel<8>(ctx->smem_bytes, &bps); break;
        default: ce = configure_kernel<16>(ctx->smem_bytes, &bps); break;
    }
    if (ce != cudaSuccess || bps <= 0) {
        fail(nullptr, BIGCLAM_ECUDA, "bigclam_create: kernel configuration failed: %s (smem %zu B)",
             cudaGetErrorString(ce), ctx->smem_bytes);
        free_ctx(ctx);
        return BIGCLAM_ECUDA;
    }
    ctx->grid = ctx->num_sms * bps;
    ctx->h_work_init = 3u * (unsigned int)ctx->grid * kWarpsPerBlock;
    if (params->flags & BIGCLAM_F_SPARSE_ROWS) {
        if (params->min_f != 0.0) {
            fail(nullptr, BIGCLAM_EUNSUPPORTED, "bigclam_create: BIGCLAM_F_SPARSE_ROWS needs min_f == 0");
            free_ctx(ctx);
            return BIGCLAM_EUNSUPPORTED;
        }
        if (n >= ((int64_t)1 << 28)) {
            fail(nullptr, BIGCLAM_EUNSUPPORTED, "bigclam_create: BIGCLAM_F_SPARSE_ROWS supports n < 2^28 nodes");
            free_ctx(ctx);
            return BIGCLAM_EUNSUPPORTED;
        }
        ctx->sparse = true;
        ctx->sp_wpb = tl_warps_per_block(ld);
        ctx->sp_smem = tl_block_smem_bytes(ld, ctx->sp_wpb);
        int sbps = 0;
        CUC(cudaFuncSetAttribute(tile_step_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->sp_smem));
        CUC(cudaFuncSetAttribute(tile_step_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->sp_smem));
        CUC(cudaFuncSetAttribute(tile_step_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->sp_smem));
        CUC(cudaFuncSetAttribute(tile_step_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->sp_smem));
        CUC(cudaFuncSetAttribute(reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * red_warps(ld) * (size_t)sp_ldp(ld))));
        int sb2 = 0;                         // the grid must be resident for every variant (hub items wait for each other)
        CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sbps, tile_step_kernel<true, true>, 32 * ctx->sp_wpb, ctx->sp_smem));
        CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sb2, tile_step_kernel<false, false>, 32 * ctx->sp_wpb, ctx->sp_smem));
        sbps = std::min(sbps, sb2);
        if (sbps <= 0) {
            fail(nullptr, BIGCLAM_ECUDA, "bigclam_create: sparse kernel does not fit an SM (smem %zu B)", ctx->sp_smem);
            free_ctx(ctx);
            return BIGCLAM_ECUDA;
        }
        sbps = std::min(sbps, tl_blocks_that_fit(ld, ctx->sp_wpb));
        ctx->sp_grid = ctx->num_sms * sbps;
        ctx->h_work_init = 0;
        ctx->ls_exhaustive = (params->flags & BIGCLAM_F_LS_EXHAUSTIVE) != 0;
        if (const char *ev = std::getenv("BIGCLAM_LS_EXHAUSTIVE")) ctx->ls_exhaustive = std::atoi(ev) != 0;
        if (const char *ev = std::getenv("BIGCLAM_LS_PRUNE")) ctx->ls_level = std::max(1, std::min(2, std::atoi(ev)));
        if (const char *ev = std::getenv("BIGCLAM_TILE_EDGES")) ctx->tile_edges = std::max(0, std::min(kTlMaxEdges, std::atoi(ev)));
    }

    CUC(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
    const size_t fbytes = sizeof(double) * (size_t)n * (size_t)ld;
    CUC(cudaMalloc(&ctx->d_rowptr, sizeof(int64_t) * ((size_t)n + 1)));
    CUC(cudaMalloc(&ctx->d_col, sizeof(int32_t) * std::max<size_t>(1, (size_t)nnz)));
    if (!ctx->sparse) {            // sparse rows: the dense buffers are only a mirror, allocated on first use (alloc_dense)
        CUC(cudaMalloc(&ctx->d_F[0], fbytes));
        CUC(cudaMalloc(&ctx->d_F[1], fbytes));
    }
    CUC(cudaMalloc(&ctx->d_sumF[0], sizeof(double) * ld));
    CUC(cudaMalloc(&ctx->d_sumF[1], sizeof(double) * ld));
    CUC(cudaMalloc(&ctx->d_partials, sizeof(double) * (2 * (size_t)ld + 2)));
    CUC(cudaMalloc(&ctx->d_accepted, (size_t)n));
    CUC(cudaMalloc(&ctx->d_accepted_spec, (size_t)n));
    CUC(cudaMalloc(&ctx->d_mask, (size_t)n));
    CUC(cudaMalloc(&ctx->d_done, sizeof(int32_t)));
    CUC(cudaMalloc(&ctx->d_work, 2 * sizeof(unsigned int)));      // [0] live counter, [1] its initial value
    CUC(cudaMemcpy(ctx->d_work + 1, &ctx->h_work_init, sizeof(unsigned int), cudaMemcpyHostToDevice));
    CUC(cudaMalloc(&ctx->d_state, sizeof(RunState)));
    CUC(cudaMallocHost(&ctx->h_pinned, sizeof(double) * (2 * (size_t)ld + 2) + sizeof(RunState) + 64));
    CUC(cudaMemcpy(ctx->d_rowptr, rowptr, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice));
    if (nnz > 0) CUC(cudaMemcpy(ctx->d_col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice));
    if (!ctx->sparse) {
        CUC(cudaMemset(ctx->d_F[0], 0, fbytes));
        CUC(cudaMemset(ctx->d_F[1], 0, fbytes));
    }
    CUC(cudaMemset(ctx->d_sumF[0], 0, sizeof(double) * ld));
    CUC(cudaMemset(ctx->d_sumF[1], 0, sizeof(double) * ld));
    CUC(cudaMemset(ctx->d_partials, 0, sizeof(double) * (2 * (size_t)ld + 2)));
    CUC(cudaMemset(ctx->d_accepted, 0xff, (size_t)n));
    CUC(cudaMemset(ctx->d_done, 0, sizeof(int32_t)));
    CUC(cudaMemset(ctx->d_state, 0, sizeof(RunState)));
    if (ctx->sparse) {
        // worst case: every row full (ld entries) — a step can then never overflow its pool.  When two such
        // pools do not fit in 80 % of the free memory, each pool gets 40 % of it and a step that runs out reports
        // BIGCLAM_ENOMEM (its input is untouched).  BIGCLAM_SPARSE_POOL_WORDS overrides the size (tests).
        ctx->pool_cap8 = (uint64_t)n * 2 * sp_words((uint32_t)ld);        // a full row and a full delta block per node
        {
            size_t free_b = 0, total_b = 0;
            CUC(cudaMemGetInfo(&free_b, &total_b));
            if ((double)ctx->pool_cap8 * 16.0 > 0.8 * (double)free_b) ctx->pool_cap8 = (uint64_t)(0.4 * (double)free_b / 8.0);
            if (const char *ev = std::getenv("BIGCLAM_SPARSE_POOL_WORDS")) ctx->pool_cap8 = (uint64_t)std::max<long long>(64, std::atoll(ev));
        }
        ctx->region_base8 = 0;
        ctx->region_cap8 = ctx->pool_cap8;
        for (int b = 0; b < 2; ++b) {
            CUC(cudaMalloc(&ctx->d_hdr[b], sizeof(uint64_t) * (size_t)n));
            CUC(cudaMemset(ctx->d_hdr[b], 0, sizeof(uint64_t) * (size_t)n));
            CUC(cudaMalloc(&ctx->d_pool[b], sizeof(double) * (size_t)ctx->pool_cap8));
        }
        CUC(cudaMalloc(&ctx->d_pool_top, 2 * sizeof(unsigned long long)));
        CUC(cudaMemset(ctx->d_pool_top, 0, 2 * sizeof(unsigned long long)));
        CUC(cudaMalloc(&ctx->d_overflow, sizeof(int32_t)));
        CUC(cudaMemset(ctx->d_overflow, 0, sizeof(int32_t)));
        CUC(cudaMalloc(&ctx->d_node_llh, sizeof(double) * (size_t)n));
        CUC(cudaMemset(ctx->d_node_llh, 0, sizeof(double) * (size_t)n));
        CUC(cudaMalloc(&ctx->d_dcnt, sizeof(unsigned short) * (size_t)n));
        CUC(cudaMemset(ctx->d_dcnt, 0, sizeof(unsigned short) * (size_t)n));
        CUC(cudaMalloc(&ctx->d_ticket, sizeof(unsigned int)));
        CUC(cudaMemset(ctx->d_ticket, 0, sizeof(unsigned int)));
        CUC(cudaMalloc(&ctx->d_stats, 4 * sizeof(unsigned int)));
        CUC(cudaMemset(ctx->d_stats, 0, 4 * sizeof(unsigned int)));
        ctx->h_col.assign(col, col + nnz);
    }
#undef CUC
    ctx->h_rowptr.assign(rowptr, rowptr + n + 1);
    {
        const std::vector<int64_t> &rp = ctx->h_rowptr;
        int rc = rebuild_order(ctx, rp);
        if (rc != BIGCLAM_OK) { g_create_err = ctx->err; free_ctx(ctx); return rc; }
    }
    *out = ctx;
    return BIGCLAM_OK;
}

extern "C" int bigclam_set_stream(bigclam_ctx *ctx, void *cuda_stream) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return BIGCLAM_OK;
}

extern "C" int bigclam_device_state(bigclam_ctx *ctx, void **F_dev, void **F_next_dev, void **sumF_dev, int64_t *ld) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (ctx->sparse && (F_dev != nullptr || F_next_dev != nullptr)) {
        // the dense buffers are only a mirror here: build / refresh it — only when the caller asks for dense rows
        // (n x K may not fit anywhere: R-MAT 10M x 1000)
        CU(cudaSetDevice(ctx->device));
        if (int re = ensure_dense(ctx)) return re;
    }
    if (F_dev) *F_dev = ctx->d_F[ctx->cur];
    if (F_next_dev) *F_next_dev = ctx->d_F[ctx->cur ^ 1];
    if (sumF_dev) *sumF_dev = ctx->d_sumF[ctx->cur];
    if (ld) *ld = ctx->ld;
    return BIGCLAM_OK;
}

static int colsum_current(bigclam_ctx *ctx) {
    const int nchunks = (int)((ctx->n + kColsumRows - 1) / kColsumRows);
    double *part = nullptr;
    CU(cudaMalloc(&part, sizeof(double) * (size_t)nchunks * ctx->ld));
    dim3 grid((ctx->ld + 31) / 32, nchunks);
    colsum_partial_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_F[ctx->cur], ctx->n, ctx->ld, part);
    colsum_final_kernel<<<(ctx->ld + 127) / 128, 128, 0, ctx->stream>>>(part, nchunks, ctx->ld, ctx->d_sumF[ctx->cur]);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(part);
    if (e != cudaSuccess) return fail(ctx, BIGCLAM_ECUDA, "column sums of F: %s", cudaGetErrorString(e));
    return BIGCLAM_OK;
}

// Sparse mode: the dense n x ld buffers exist only while somebody needs dense rows.
static int alloc_dense(bigclam_ctx *ctx, int b) {
    if (ctx->d_F[b] != nullptr) return BIGCLAM_OK;
    CU(cudaMalloc(&ctx->d_F[b], sizeof(double) * (size_t)ctx->n * (size_t)ctx->ld));
    return BIGCLAM_OK;
}

// Sparse mode: rebuild the sparse rows of the current buffer from its dense mirror d_F[cur].
static int sparse_from_dense(bigclam_ctx *ctx) {
    const int b = ctx->cur;
    invalidate_resets(ctx);
    CU(cudaMemsetAsync(ctx->d_pool_top + b, 0, sizeof(unsigned long long), ctx->stream));
    CU(cudaMemsetAsync(ctx->d_overflow, 0, sizeof(int32_t), ctx->stream));
    const int wpb = 8;
    dense_to_sparse_kernel<<<(unsigned)((ctx->n + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(
        ctx->d_F[b], ctx->n, ctx->ld, ctx->d_hdr[b], ctx->d_pool[b], ctx->d_pool_top + b, ctx->pool_cap8, ctx->d_overflow);
    CU(cudaGetLastError());
    ctx->dense_valid = true;
    return BIGCLAM_OK;
}

// Sparse mode: entry points that hand out dense rows refresh the mirror d_F[cur] first.
static int ensure_dense(bigclam_ctx *ctx) {
    if (!ctx->sparse || (ctx->dense_valid && ctx->d_F[ctx->cur] != nullptr)) return BIGCLAM_OK;
    const int b = ctx->cur;
    if (int ra = alloc_dense(ctx, b)) return ra;
    const int wpb = 8;
    sparse_to_dense_kernel<<<(unsigned)((ctx->n + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(
        ctx->d_hdr[b], ctx->d_pool[b], ctx->n, ctx->ld, ctx->d_F[b]);
    CU(cudaGetLastError());
    ctx->dense_valid = true;
    return BIGCLAM_OK;
}

// Sparse mode: a step that ran out of pool space left garbage rows; report it (cannot happen with the
// worst-case pool bigclam_create allocates, kept as a guard for smaller pools).
static int check_overflow(bigclam_ctx *ctx) {
    if (!ctx->sparse) return BIGCLAM_OK;
    int32_t ov = 0;
    CU(cudaMemcpyAsync(&ov, ctx->d_overflow, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ov) return fail(ctx, BIGCLAM_ENOMEM, "sparse row pool exhausted");
    return BIGCLAM_OK;
}

// Sparse rows: the edge budget of a tile follows the rows' average size (the rows of a tile are staged in
// kTlStage16 16-byte chunks of shared memory); called when F is set.  BIGCLAM_TILE_EDGES pins it instead.
static int retile(bigclam_ctx *ctx, uint64_t words_used) {
    if (!ctx->sparse || std::getenv("BIGCLAM_TILE_EDGES") != nullptr) return BIGCLAM_OK;
    std::vector<uint64_t> hdr((size_t)ctx->n);
    CU(cudaMemcpy(hdr.data(), ctx->d_hdr[ctx->cur], sizeof(uint64_t) * (size_t)ctx->n, cudaMemcpyDeviceToHost));
    const double nn = (double)std::max<int64_t>(1, ctx->n);
    const double avg_cnt = std::max(1.0, (double)sp_host_nnz(ctx->n, hdr.data()) / nn);
    const double avg16 = std::max(1.0, (double)words_used / 2.0 / nn);
    ctx->tile_avg16 = avg16;
    // the neighbour rows of a tile must fit the staging chunks, its nodes' own rows theirs, and all their entries
    // the slots (worst case: no two of them on the same component) — with 10-15 % to spare
    int nodes = std::max(0, std::min(kTlMaxNodes, (int)((double)kTlOwn16 / (1.15 * avg16))));
    const double rows = std::min((double)kTlStage16 / (1.1 * avg16), (double)kTlSlots / (1.1 * avg_cnt) - nodes);
    int budget = std::max(0, std::min(kTlMaxEdges, (int)rows));
    if (budget < 6 || nodes < 2) budget = 0;
    if (budget == ctx->tile_edges && nodes == ctx->tile_nodes) return BIGCLAM_OK;
    ctx->tile_nodes = std::max(1, nodes);
    ctx->tile_edges = budget;
    std::vector<int32_t> order = ctx->h_owned;
    return rebuild_order_list(ctx, ctx->h_rowptr, order);
}

// The rows change size while the solver runs (they fill up on small-K problems): when the tiles were cut for rows
// of a very different size, cut them again.  Call at a point where the stream is idle.
static int maybe_retile(bigclam_ctx *ctx) {
    if (!ctx->sparse || std::getenv("BIGCLAM_TILE_EDGES") != nullptr) return BIGCLAM_OK;
    // (1) tiles that keep falling back to the general path (too many active components / entries for the warp's
    //     buffers: small K, rows filling up) are cut smaller: the fallback costs three times the tile path
    unsigned int st[2] = {0u, 0u};
    CU(cudaMemcpy(st, ctx->d_stats, sizeof(st), cudaMemcpyDeviceToHost));
    const unsigned int done = st[0] - ctx->stats_seen[0], fb = st[1] - ctx->stats_seen[1];
    ctx->stats_seen[0] = st[0];
    ctx->stats_seen[1] = st[1];
    if (ctx->tile_edges > 0 && done + fb > 0 && (double)fb > 0.2 * (double)(done + fb)) {
        const int edges = std::max(6, (ctx->tile_edges * 5) / 8), nodes = std::max(2, (ctx->tile_nodes * 5 + 7) / 8);
        if (edges != ctx->tile_edges || nodes != ctx->tile_nodes) {
            ctx->tile_edges = edges;
            ctx->tile_nodes = nodes;
            std::vector<int32_t> order = ctx->h_owned;
            return rebuild_order_list(ctx, ctx->h_rowptr, order);
        }
    }
    // (2) rows of a very different size than the tiles were cut for
    unsigned long long used = 0;
    CU(cudaMemcpy(&used, ctx->d_pool_top + ctx->cur, sizeof(used), cudaMemcpyDeviceToHost));
    if (used == 0) return BIGCLAM_OK;
    const double avg16 = std::max(1.0, (double)used / 2.0 / (double)std::max<int64_t>(1, ctx->order_n));   // (this rank's rows; deltas included: conservative)
    const double ratio = avg16 / std::max(1.0, ctx->tile_avg16);
    if (ratio < 1.3 && ratio > 0.6) return BIGCLAM_OK;
    if (ctx->n_peers > 0) return BIGCLAM_OK;     // (replicated pools: pool_top only counts the owned region; the caller retiles through set_F)
    return retile(ctx, used);
}

extern "C" int bigclam_retile(bigclam_ctx *ctx) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    return maybe_retile(ctx);
}

extern "C" int bigclam_set_F(bigclam_ctx *ctx, const double *F) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (F == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_F: F is NULL");
    CU(cudaSetDevice(ctx->device));
    if (int rd = drop_speculation(ctx)) return rd;
    const int k = ctx->p.k, ld = ctx->ld;
    if (ctx->sparse) { if (int ra = alloc_dense(ctx, ctx->cur)) return ra; }
    // values must already satisfy the invariant the reference maintains: MIN_F <= F <= MAX_F
    CU(cudaMemsetAsync(ctx->d_F[ctx->cur], 0, sizeof(double) * (size_t)ctx->n * ld, ctx->stream));
    CU(cudaMemcpy2DAsync(ctx->d_F[ctx->cur], sizeof(double) * ld, F, sizeof(double) * k, sizeof(double) * k,
                         (size_t)ctx->n, cudaMemcpyHostToDevice, ctx->stream));
    int rc = colsum_current(ctx);
    if (rc != BIGCLAM_OK) return rc;
    if (ctx->sparse) {
        rc = sparse_from_dense(ctx);
        if (rc == BIGCLAM_OK) rc = check_overflow(ctx);        // a pool smaller than the rows: BIGCLAM_ENOMEM
        if (rc != BIGCLAM_OK) return rc;
        unsigned long long used = 0;
        CU(cudaMemcpy(&used, ctx->d_pool_top + ctx->cur, sizeof(used), cudaMemcpyDeviceToHost));
        if (int rt = retile(ctx, used)) return rt;
    }
    // with peer replicas every row counts as changed again: the next step publishes all owned rows
    if (ctx->d_changed != nullptr) CU(cudaMemsetAsync(ctx->d_changed, 1, (size_t)ctx->n, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return BIGCLAM_OK;
}

// F given / returned as CSR rows — the shape of the reference's RDD[(Long, BSV[Double])] (bigclam4-7.scala:97-104).
// With BIGCLAM_F_SPARSE_ROWS nothing dense is ever materialised (n x K may not fit anywhere); a dense context
// goes through a dense host image.
extern "C" int bigclam_set_F_csr(bigclam_ctx *ctx, const int64_t *indptr, const int32_t *indices, const double *values) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (indptr == nullptr || (indptr[ctx->n] > 0 && (indices == nullptr || values == nullptr)))
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_F_csr: NULL argument");
    const int64_t n = ctx->n;
    const int32_t k = ctx->p.k, ld = ctx->ld;
    if (!ctx->sparse) {
        std::vector<double> dense((size_t)n * k, 0.0);
        for (int64_t u = 0; u < n; ++u)
            for (int64_t i = indptr[u]; i < indptr[u + 1]; ++i) {
                if (indices[i] < 0 || indices[i] >= k) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_F_csr: index out of range in row %lld", (long long)u);
                dense[(size_t)u * k + indices[i]] = values[i];
            }
        return bigclam_set_F(ctx, dense.data());
    }
    CU(cudaSetDevice(ctx->device));
    if (int rd = drop_speculation(ctx)) return rd;
    invalidate_resets(ctx);
    uint64_t need = 0;
    for (int64_t u = 0; u < n; ++u) {
        uint32_t cnt = 0;
        for (int64_t i = indptr[u]; i < indptr[u + 1]; ++i) cnt += (values[i] != 0.0);
        need += sp_words(cnt);
    }
    if (need > ctx->pool_cap8) return fail(ctx, BIGCLAM_ENOMEM, "bigclam_set_F_csr: rows need %llu pool words, %llu available", (unsigned long long)need, (unsigned long long)ctx->pool_cap8);
    std::vector<uint64_t> hdr((size_t)n);
    std::vector<double> pool((size_t)need + 1), colsum((size_t)ld, 0.0);
    const int64_t used = sp_host_pack(n, k, ld, indptr, indices, values, hdr.data(), pool.data(), need, colsum.data());
    if (used < 0) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_F_csr: index outside [0, k) or more than ld entries in a row");
    const int b = ctx->cur;
    const unsigned long long top = (unsigned long long)used;
    CU(cudaMemcpyAsync(ctx->d_hdr[b], hdr.data(), sizeof(uint64_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if (used > 0) CU(cudaMemcpyAsync(ctx->d_pool[b], pool.data(), sizeof(double) * (size_t)used, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->d_pool_top + b, &top, sizeof(top), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->d_sumF[b], colsum.data(), sizeof(double) * (size_t)ld, cudaMemcpyHostToDevice, ctx->stream));   // :105-106
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->dense_valid = false;
    if (int rt = retile(ctx, (uint64_t)used)) return rt;
    return BIGCLAM_OK;
}

// Downloads the sparse state (sparse context) or the dense F (dense context) for the two getters below.
static int fetch_rows_host(bigclam_ctx *ctx, std::vector<uint64_t> &hdr, std::vector<double> &pool, std::vector<double> &dense) {
    const int64_t n = ctx->n;
    if (ctx->sparse) {
        const int b = ctx->cur;
        hdr.resize((size_t)n);
        CU(cudaMemcpyAsync(hdr.data(), ctx->d_hdr[b], sizeof(uint64_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        uint64_t extent = 0;
        for (int64_t u = 0; u < n; ++u)
            if (sp_cnt(hdr[u]) > 0) extent = std::max<uint64_t>(extent, sp_off8(hdr[u]) + sp_words(sp_cnt(hdr[u])));
        pool.resize((size_t)extent + 1);
        if (extent > 0) CU(cudaMemcpyAsync(pool.data(), ctx->d_pool[b], sizeof(double) * (size_t)extent, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        return BIGCLAM_OK;
    }
    dense.resize((size_t)n * ctx->p.k);
    return bigclam_get_F(ctx, dense.data());
}

extern "C" int bigclam_get_F_nnz(bigclam_ctx *ctx, int64_t *nnz_out) {
    if (ctx == nullptr || nnz_out == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    std::vector<uint64_t> hdr;
    std::vector<double> pool, dense;
    if (ctx->sparse) {                       // the headers are enough
        hdr.resize((size_t)ctx->n);
        CU(cudaMemcpyAsync(hdr.data(), ctx->d_hdr[ctx->cur], sizeof(uint64_t) * (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        *nnz_out = sp_host_nnz(ctx->n, hdr.data());
        return BIGCLAM_OK;
    }
    if (int rf = fetch_rows_host(ctx, hdr, pool, dense)) return rf;
    int64_t t = 0;
    for (double v : dense) t += (v != 0.0);
    *nnz_out = t;
    return BIGCLAM_OK;
}

// indptr_out: n + 1; indices_out / values_out: bigclam_get_F_nnz() entries (ascending indices inside a row).
extern "C" int bigclam_get_F_csr(bigclam_ctx *ctx, int64_t *indptr_out, int32_t *indices_out, double *values_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (indptr_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_F_csr: indptr_out is NULL");
    CU(cudaSetDevice(ctx->device));
    std::vector<uint64_t> hdr;
    std::vector<double> pool, dense;
    if (int rf = fetch_rows_host(ctx, hdr, pool, dense)) return rf;
    if (ctx->sparse) {
        if (sp_host_nnz(ctx->n, hdr.data()) > 0 && (indices_out == nullptr || values_out == nullptr))
            return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_F_csr: NULL output");
        sp_host_unpack(ctx->n, hdr.data(), pool.data(), indptr_out, indices_out, values_out);
        return BIGCLAM_OK;
    }
    int64_t t = 0;
    const int k = ctx->p.k;
    for (int64_t u = 0; u < ctx->n; ++u) {
        indptr_out[u] = t;
        for (int c = 0; c < k; ++c) {
            const double v = dense[(size_t)u * k + c];
            if (v != 0.0) { indices_out[t] = c; values_out[t] = v; ++t; }
        }
    }
    indptr_out[ctx->n] = t;
    return BIGCLAM_OK;
}

extern "C" int bigclam_set_sumF(bigclam_ctx *ctx, const double *sumF) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (sumF == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_sumF: sumF is NULL");
    CU(cudaSetDevice(ctx->device));
    if (int rd = drop_speculation(ctx)) return rd;
    CU(cudaMemsetAsync(ctx->d_sumF[ctx->cur], 0, sizeof(double) * ctx->ld, ctx->stream));
    CU(cudaMemcpyAsync(ctx->d_sumF[ctx->cur], sumF, sizeof(double) * ctx->p.k, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return BIGCLAM_OK;
}

extern "C" int bigclam_get_F(bigclam_ctx *ctx, double *F_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (F_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_F: F_out is NULL");
    CU(cudaSetDevice(ctx->device));
    if (int re = ensure_dense(ctx)) return re;
    const int k = ctx->p.k, ld = ctx->ld;
    CU(cudaMemcpy2DAsync(F_out, sizeof(double) * k, ctx->d_F[ctx->cur], sizeof(double) * ld, sizeof(double) * k,
                         (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return BIGCLAM_OK;
}

extern "C" int bigclam_get_sumF(bigclam_ctx *ctx, double *sumF_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (sumF_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_sumF: out is NULL");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyAsync(sumF_out, ctx->d_sumF[ctx->cur], sizeof(double) * ctx->p.k, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return BIGCLAM_OK;
}

extern "C" int bigclam_get_accepted(bigclam_ctx *ctx, int8_t *accepted_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (accepted_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_accepted: out is NULL");
    if (!(ctx->p.flags & BIGCLAM_F_RECORD_ACCEPTED))
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_accepted: context created without BIGCLAM_F_RECORD_ACCEPTED");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyAsync(accepted_out, ctx->d_accepted, (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return BIGCLAM_OK;
}

// ------------------------------------------------------------------------------------------------
static void fill_args(bigclam_ctx *ctx, StepArgs &a, bool linesearch, const uint8_t *d_mask, bool use_done) {
    const bigclam_params &p = ctx->p;
    a.n = ctx->n;
    a.rowptr = ctx->d_rowptr;
    a.col = ctx->d_col;
    a.F_in = ctx->d_F[ctx->cur];
    a.F_out = ctx->d_F[ctx->cur ^ 1];
    a.sumF = ctx->d_sumF[ctx->cur];
    a.k = p.k;
    a.ld = ctx->ld;
    a.nsteps = ctx->nsteps;
    for (int i = 0; i < kMaxSteps; ++i) a.steps[i] = i < ctx->nsteps ? ctx->steps[i] : 0.0;
    a.alpha = p.alpha;
    a.min_p = p.min_p; a.max_p = p.max_p; a.min_f = p.min_f; a.max_f = p.max_f;
    // exp(-x) >= max_p  <=>  x <= -log(max_p);  exp(-x) <= min_p  <=>  x >= -log(min_p)
    a.x_lo = -std::log(p.max_p) * (1.0 - 1e-12);
    a.x_hi = -std::log(p.min_p) * (1.0 + 1e-12);
    a.t_lo = std::log(1.0 - p.max_p);
    a.t_hi = std::log(1.0 - p.min_p);
    a.w_lo = 1.0 / (1.0 - p.max_p);
    a.w_hi = 1.0 / (1.0 - p.min_p);
    a.meta = ctx->d_meta;
    a.work_counter = ctx->d_work;
    a.n_peers = linesearch ? ctx->n_peers : 0;
    for (int r = 0; r < 7; ++r) a.peer_out[r] = (r < ctx->n_peers) ? ctx->peer_F[ctx->cur ^ 1][r] : nullptr;
    a.changed = ctx->d_changed;
    a.maxm = ctx->maxm;
    a.order_n = ctx->order_n;
    a.n_hubs = ctx->n_hubs;
    a.n_hub_items = ctx->n_hub_items;
    a.hub_items = ctx->d_hub_items;
    a.hub_scratch = ctx->d_hub_scratch;
    a.hub_counters = ctx->d_hub_counters;
    a.node_mask = d_mask;
    a.partials = ctx->d_partials;
    a.accepted = (linesearch && (p.flags & BIGCLAM_F_RECORD_ACCEPTED)) ? ctx->d_accepted : nullptr;
    a.done_flag = use_done ? ctx->d_done : nullptr;
    a.do_linesearch = linesearch ? 1 : 0;
}

static int timed_launch(bigclam_ctx *ctx, const StepArgs &a, bool is_step) {
    const bool timing = (ctx->p.flags & BIGCLAM_F_TIME_KERNELS) && is_step;
    if (timing) {
        while (ctx->ev_pool.size() < ctx->ev_used + 2) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            ctx->ev_pool.push_back(e);
        }
        CU(cudaEventRecord(ctx->ev_pool[ctx->ev_used], ctx->stream));
    }
    if (ctx->n_mega > 0) {     // mega-hub scratch, slice counters (and the sparse kernel's item counter) start every launch at zero
        if (!ctx->sparse)      // (the sparse kernel writes every scratch slot before it is read)
            CU(cudaMemsetAsync(ctx->d_hub_scratch, 0, sizeof(double) * (size_t)ctx->n_mega * ((size_t)ctx->ld + 32), ctx->stream));
        CU(cudaMemsetAsync(ctx->d_hub_counters, 0, sizeof(unsigned int) * (2 * (size_t)ctx->n_mega + 1), ctx->stream));
    }
    // positions 0 .. 3*#warps-1 are pre-assigned statically, the rest is handed out dynamically
    // (sparse engine: the previous launch's reduce_kernel has usually done this already)
    if (!(ctx->sparse && ctx->work_clean))
        CU(cudaMemcpyAsync(ctx->d_work, ctx->d_work + 1, sizeof(unsigned int), cudaMemcpyDeviceToDevice, ctx->stream));
    if (ctx->sparse) {
        // reads hdr/pool of the current buffer, writes the other one (its bump allocator starts at zero)
        const int in = ctx->cur, out = in ^ 1;
        SparseArgs sp{};
        sp.hdr_in = ctx->d_hdr[in];
        sp.pool_in = ctx->d_pool[in];
        sp.hdr_out = ctx->d_hdr[out];
        sp.pool_out = ctx->d_pool[out];
        sp.pool_top = ctx->d_pool_top + out;
        sp.pool_cap8 = ctx->region_cap8;
        sp.region_base8 = ctx->region_base8;
        sp.overflow = ctx->d_overflow;
        sp.n_peers = a.do_linesearch ? ctx->n_peers : 0;
        for (int r = 0; r < 7; ++r) {
            sp.peer_hdr[r] = (r < ctx->n_peers) ? ctx->peer_hdr[out][r] : nullptr;
            sp.peer_pool[r] = (r < ctx->n_peers) ? ctx->peer_pool[out][r] : nullptr;
        }
        if (a.do_linesearch) {
            if (!ctx->top_clean[out]) CU(cudaMemsetAsync(sp.pool_top, 0, sizeof(unsigned long long), ctx->stream));
            ctx->top_clean[out] = false;
            ctx->dense_valid = false;
        }
        sp.hub_work = ctx->d_hub_counters + 2 * (size_t)std::max<int32_t>(1, ctx->n_mega);
        sp.node_llh = ctx->d_node_llh;
        sp.dcnt = ctx->d_dcnt;
        sp.accepted = (a.accepted != nullptr) ? a.accepted : ctx->d_accepted;
        sp.n_gen = ctx->n_gen;
        sp.ntiles = ctx->ntiles;
        sp.tiles = ctx->d_tiles;
        sp.tcol = ctx->d_tcol;
        sp.stats = ctx->d_stats;
        // line search by bounds (bigclam_tile.cuh, H2): needs the reference's clamps in their usual order
        sp.ls_prune = (ctx->ls_exhaustive || !(ctx->p.min_f == 0.0 && ctx->p.min_p > 0.0 && ctx->p.min_p < ctx->p.max_p && ctx->p.max_p < 1.0 && ctx->p.alpha > 0.0)) ? 0 : ctx->ls_level;
        sp.pr_xlo = std::nextafterf((float)a.x_lo, 0.0f);
        sp.pr_kinv = std::nextafterf((float)(1.0 / (1.0 - ctx->p.max_p)), INFINITY) * 1.000001f;
        sp.pr_cap = std::nextafterf((float)(a.t_hi - a.t_lo), INFINITY) * 1.000001f;
        sp.ho_rowptr = ctx->d_ho_rowptr;
        sp.ho_col = ctx->d_ho_col;
        const bool hub = a.n_hub_items > 0, push = sp.n_peers > 0;
        const int threads = 32 * ctx->sp_wpb;
        if (ctx->ho) tile_step_kernel<false, false, true><<<ctx->sp_grid, threads, ctx->sp_smem, ctx->stream>>>(a, sp);   // (no hubs, no peers)
        else if (hub && push) tile_step_kernel<true, true><<<ctx->sp_grid, threads, ctx->sp_smem, ctx->stream>>>(a, sp);
        else if (hub) tile_step_kernel<false, true><<<ctx->sp_grid, threads, ctx->sp_smem, ctx->stream>>>(a, sp);
        else if (push) tile_step_kernel<true, false><<<ctx->sp_grid, threads, ctx->sp_smem, ctx->stream>>>(a, sp);
        else tile_step_kernel<false, false><<<ctx->sp_grid, threads, ctx->sp_smem, ctx->stream>>>(a, sp);
        CU(cudaGetLastError());
        if (timing) {
            CU(cudaEventRecord(ctx->ev_pool[ctx->ev_used + 1], ctx->stream));
            ctx->ev_used += 2;
        }
        // the sums over the nodes, in a fixed order (no floating-point atomics): partials = [D | - | llh | n_updated]
        ReduceArgs r{};
        r.world = 0;
        if (ctx->x_world > 1) {              // publish this rank's sums to every rank (fused collective)
            const unsigned long long seq = ++ctx->x_seq;
            const size_t half = (size_t)(seq & 1ull) * (size_t)ctx->x_world * ((size_t)ctx->ld + 2);
            r.world = ctx->x_world;
            r.seq = seq;
            for (int q = 0; q < ctx->x_world; ++q) {
                r.xslot[q] = ctx->x_peer_buf[q] + half + (size_t)ctx->x_rank * ((size_t)ctx->ld + 2);
                r.xflag[q] = ctx->x_peer_flags[q] + ctx->x_rank;
            }
        }
        r.meta = ctx->d_meta;
        r.order_n = ctx->order_n;
        r.hdr_out = sp.hdr_out;
        r.pool_out = sp.pool_out;
        r.node_llh = ctx->d_node_llh;
        r.dcnt = ctx->d_dcnt;
        r.accepted = sp.accepted;
        r.ld = ctx->ld;
        r.do_linesearch = a.do_linesearch;
        r.block_part = ctx->d_block_part;
        r.ticket = ctx->d_ticket;
        r.partials = ctx->d_partials;
        r.done_flag = a.done_flag;
        r.work_counter = ctx->d_work;
        r.work_init = ctx->h_work_init;
        // the input pool of a step is the output pool of the next one: its allocator can be zeroed now.  Not under a
        // Not for a PRE-only launch (the state stays where it is).
        // (under a done flag the kernels of a converged loop are no-ops and skip this: the loops invalidate the host's
        // bookkeeping when they end, see invalidate_resets)
        r.pool_top_in = a.do_linesearch ? ctx->d_pool_top + in : nullptr;
        ctx->work_clean = true;
        if (a.do_linesearch) ctx->top_clean[in] = true;
        reduce_kernel<<<ctx->red_grid, red_warps(ctx->ld) * 32, sizeof(double) * red_warps(ctx->ld) * (size_t)sp_ldp(ctx->ld), ctx->stream>>>(r);
        CU(cudaGetLastError());
        if (is_step) ++ctx->last_step_launches;
        ctx->last_all_launches += 2;
        return BIGCLAM_OK;
    } else {
        launch_step(ctx->c2, a, ctx->grid, ctx->smem_bytes, ctx->stream);
    }
    CU(cudaGetLastError());
    if (timing) {
        CU(cudaEventRecord(ctx->ev_pool[ctx->ev_used + 1], ctx->stream));
        ctx->ev_used += 2;
    }
    if (is_step) ++ctx->last_step_launches;
    ++ctx->last_all_launches;
    return BIGCLAM_OK;
}

static int collect_timing(bigclam_ctx *ctx) {
    ctx->last_step_ms = 0.0;
    if (ctx->p.flags & BIGCLAM_F_TIME_KERNELS) ctx->last_step_launches = (int64_t)(ctx->ev_used / 2);
    for (size_t i = 0; i + 1 < ctx->ev_used; i += 2) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, ctx->ev_pool[i], ctx->ev_pool[i + 1]));
        ctx->last_step_ms += ms;
    }
    ctx->ev_used = 0;
    return BIGCLAM_OK;
}

// Node-partitioned launches: every rank's sums of the most recent reduce_kernel -> partials (all ranks: same bits).
static int launch_xreduce(bigclam_ctx *ctx, bool use_done) {
    if (ctx->x_world <= 1) return BIGCLAM_OK;
    XReduceArgs x{};
    const unsigned long long seq = ctx->x_seq;
    x.xbuf = ctx->d_xbuf + (size_t)(seq & 1ull) * (size_t)ctx->x_world * ((size_t)ctx->ld + 2);
    x.flags = ctx->d_xflags;
    x.seq = seq;
    x.world = ctx->x_world;
    x.ld = ctx->ld;
    x.partials = ctx->d_partials;
    x.done_flag = use_done ? ctx->d_done : nullptr;
    xreduce_kernel<<<1, 256, 0, ctx->stream>>>(x);
    CU(cudaGetLastError());
    ++ctx->last_all_launches;
    return BIGCLAM_OK;
}

static int launch_finish(bigclam_ctx *ctx, long long kernel_index, int variant, double rel_tol, bool apply,
                         bool llh_is_final) {
    FinishArgs f;
    f.partials = ctx->d_partials;
    f.sumF_cur = ctx->d_sumF[ctx->cur];
    f.sumF_next = ctx->d_sumF[ctx->cur ^ 1];
    f.ld = ctx->ld;
    f.st = ctx->d_state;
    f.done_flag = ctx->d_done;
    f.trace = ctx->d_trace;
    f.trace_cap = ctx->trace_cap;
    f.kernel_index = kernel_index;
    f.variant = variant;
    f.rel_tol = rel_tol;
    f.apply = apply ? 1 : 0;
    f.llh_is_final = llh_is_final ? 1 : 0;
    finish_kernel<<<1, 256, 0, ctx->stream>>>(f);
    CU(cudaGetLastError());
    ++ctx->last_all_launches;
    return BIGCLAM_OK;
}

static int reset_run_state(bigclam_ctx *ctx) {
    ctx->spec_valid = false;
    invalidate_resets(ctx);
    CU(cudaMemsetAsync(ctx->d_done, 0, sizeof(int32_t), ctx->stream));
    CU(cudaMemsetAsync(ctx->d_state, 0, sizeof(RunState), ctx->stream));
    CU(cudaMemsetAsync(ctx->d_partials, 0, sizeof(double) * (2 * (size_t)ctx->ld + 2), ctx->stream));
    ctx->last_step_launches = 0;
    ctx->last_all_launches = 0;
    ctx->ev_used = 0;
    return BIGCLAM_OK;
}

extern "C" int bigclam_loglikelihood(bigclam_ctx *ctx, double *llh_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (llh_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_loglikelihood: llh_out is NULL");
    CU(cudaSetDevice(ctx->device));
    int rc = reset_run_state(ctx);
    if (rc) return rc;
    StepArgs a;
    fill_args(ctx, a, false, nullptr, false);
    rc = timed_launch(ctx, a, false);
    if (rc) return rc;
    CU(cudaMemcpyAsync(ctx->h_pinned, ctx->d_partials + 2 * ctx->ld, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    *llh_out = ctx->h_pinned[0];
    return BIGCLAM_OK;
}

// One call of backtrackingLineSearchs.  The LLH it has to return is the PRE sum of the NEXT call, so
// instead of a separate LLH pass the next call's whole step kernel is launched speculatively (same uset):
// its PRE delivers this call's LLH, and when the next call arrives with the same uset its result is simply
// committed (sumF update + buffer flip).  Any other entry point that touches the state drops the speculation.
extern "C" int bigclam_step(bigclam_ctx *ctx, const uint8_t *node_mask, double *llh_out, int64_t *n_updated_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    const bool speculate = (ctx->n_peers == 0);         // peers' replicas must never see uncommitted rows
    const bool null_mask = (node_mask == nullptr);
    const bool hit = speculate && ctx->spec_valid && ctx->spec_null_mask == null_mask &&
                     (null_mask || (ctx->spec_mask.size() == (size_t)ctx->n &&
                                    std::memcmp(ctx->spec_mask.data(), node_mask, (size_t)ctx->n) == 0));
    int rc;
    StepArgs a;
    const uint8_t *d_mask = null_mask ? nullptr : ctx->d_mask;
    if (!hit) {
        rc = reset_run_state(ctx);
        if (rc) return rc;
    }
    // the uset of this call always travels to the device (on a hit it equals what the speculative kernel used)
    if (!null_mask) CU(cudaMemcpyAsync(ctx->d_mask, node_mask, (size_t)ctx->n, cudaMemcpyHostToDevice, ctx->stream));
    if (!hit) {
        fill_args(ctx, a, true, d_mask, false);
        if (a.accepted != nullptr) a.accepted = ctx->d_accepted_spec;
        rc = timed_launch(ctx, a, true);                   // PRE + LS + swap
        if (rc) return rc;
    } else {
        ctx->last_step_launches = 0;
        ctx->last_all_launches = 0;
    }
    // commit: sumF update (:192), n_updated, zero the partials; the step's accepted[] becomes current
    rc = launch_finish(ctx, 0, 0, 0.0, true, false);
    if (rc) return rc;
    ctx->cur ^= 1;
    ctx->dense_valid = false;
    std::swap(ctx->d_accepted, ctx->d_accepted_spec);
    CU(cudaMemcpyAsync(ctx->h_pinned + 8, ctx->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, ctx->stream));
    if (speculate) {
        fill_args(ctx, a, true, d_mask, false);            // next call, speculatively: its PRE is this call's LLH
        if (a.accepted != nullptr) a.accepted = ctx->d_accepted_spec;
        rc = timed_launch(ctx, a, true);
        if (rc) return rc;
        ctx->spec_valid = true;
        ctx->spec_null_mask = null_mask;
        if (!null_mask && !hit) ctx->spec_mask.assign(node_mask, node_mask + ctx->n);   // on a hit it is already equal
    } else {
        fill_args(ctx, a, false, nullptr, false);          // LLH with new F, new sumF (:196-219)
        rc = timed_launch(ctx, a, false);
        if (rc) return rc;
    }
    CU(cudaMemcpyAsync(ctx->h_pinned, ctx->d_partials + 2 * ctx->ld, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (int ro = check_overflow(ctx)) return ro;
    if (llh_out) *llh_out = ctx->h_pinned[0];
    if (n_updated_out) *n_updated_out = reinterpret_cast<RunState *>(ctx->h_pinned + 8)->n_updated;
    return collect_timing(ctx);
}

extern "C" int bigclam_run(bigclam_ctx *ctx, int32_t variant, double rel_tol, int64_t max_outer,
                           double *llh_out, int64_t *calls_out, double *llh_trace, int64_t trace_cap) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (variant != 2 && variant != 3 && variant != 4) return fail(ctx, BIGCLAM_EINVAL, "bigclam_run: variant must be 2, 3 or 4");
    if (max_outer < 0 || trace_cap < 0) return fail(ctx, BIGCLAM_EINVAL, "bigclam_run: negative max_outer/trace_cap");
    CU(cudaSetDevice(ctx->device));
    int rc = reset_run_state(ctx);
    if (rc) return rc;
    if (llh_trace != nullptr && trace_cap > 0) {
        if (ctx->trace_cap < trace_cap) {
            cudaFree(ctx->d_trace);
            ctx->d_trace = nullptr;
            ctx->trace_cap = 0;
            CU(cudaMalloc(&ctx->d_trace, sizeof(double) * (size_t)trace_cap));
            ctx->trace_cap = trace_cap;
        }
    }
    const int64_t saved_cap = ctx->trace_cap;
    if (llh_trace == nullptr) ctx->trace_cap = 0; else ctx->trace_cap = trace_cap;

    RunState *hst = reinterpret_cast<RunState *>(ctx->h_pinned + 8);
    const int start_cur = ctx->cur;
    const int64_t batch = 8;       // the stream drains once per batch: the host reads the loop state and may re-cut the tiles
    int64_t c = 0;                 // step kernels enqueued so far (kernel c maps S_{c-1} -> S_c)
    bool done = false;
    StepArgs a;
    while (!done) {
        int64_t todo = batch;
        if (max_outer > 0) todo = std::min<int64_t>(batch, max_outer - c);
        for (int64_t i = 0; i < todo; ++i) {
            ++c;
            ctx->cur = (start_cur + (int)((c - 1) & 1)) & 1;       // S_{c-1} lives in buffer (c-1)%2
            fill_args(ctx, a, true, nullptr, true);
            rc = timed_launch(ctx, a, true);
            if (rc) return rc;
            rc = launch_finish(ctx, c, variant, rel_tol, true, false);   // tests call c-1, builds sumF_c
            if (rc) return rc;
        }
        CU(cudaMemcpyAsync(hst, ctx->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        if (hst->done) { done = true; break; }
        if (max_outer > 0 && c >= max_outer) break;
        {   // the stream is idle: a good moment to re-cut the tiles when the rows have changed size a lot
            const int keep = ctx->cur;
            ctx->cur = (start_cur + (int)(c & 1)) & 1;            // S_c, the current state
            const int rt = maybe_retile(ctx);
            ctx->cur = keep;
            if (rt) return rt;
        }
    }
    int64_t calls;
    if (done) {
        calls = hst->conv_call;                                   // final state S_calls, untouched
    } else {
        calls = c;                                                // cut by max_outer: need LLH(S_c)
        ctx->cur = (start_cur + (int)(c & 1)) & 1;
        fill_args(ctx, a, false, nullptr, false);
        rc = timed_launch(ctx, a, false);
        if (rc) return rc;
        rc = launch_finish(ctx, c, variant, rel_tol, false, true);
        if (rc) return rc;
        CU(cudaMemcpyAsync(hst, ctx->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    ctx->cur = (start_cur + (int)(calls & 1)) & 1;
    ctx->dense_valid = false;
    invalidate_resets(ctx);
    if (int ro = check_overflow(ctx)) return ro;
    if (llh_out) *llh_out = hst->ret_llh;
    if (calls_out) *calls_out = calls;
    if (llh_trace != nullptr && trace_cap > 0) {
        const int64_t cnt = std::min<int64_t>(calls, trace_cap);
        if (cnt > 0) CU(cudaMemcpy(llh_trace, ctx->d_trace, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost));
    }
    ctx->trace_cap = saved_cap;
    return collect_timing(ctx);
}

extern "C" int bigclam_get_kernel_time(bigclam_ctx *ctx, double *step_kernel_ms_sum, int64_t *step_kernel_launches,
                                       int64_t *all_kernel_launches) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (step_kernel_ms_sum) *step_kernel_ms_sum = ctx->last_step_ms;
    if (step_kernel_launches) *step_kernel_launches = ctx->last_step_launches;
    if (all_kernel_launches) *all_kernel_launches = ctx->last_all_launches;
    return BIGCLAM_OK;
}

extern "C" int bigclam_get_ls_stats(bigclam_ctx *ctx, int64_t *nodes_asked, int64_t *nodes_searched) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    unsigned int st[4] = {0u, 0u, 0u, 0u};
    if (ctx->sparse && ctx->d_stats != nullptr) {
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamSynchronize(ctx->stream));
        CU(cudaMemcpy(st, ctx->d_stats, sizeof(st), cudaMemcpyDeviceToHost));
    }
    if (nodes_searched) *nodes_searched = (int64_t)(st[2] - ctx->ls_read[0]);
    if (nodes_asked) *nodes_asked = (int64_t)(st[3] - ctx->ls_read[1]);
    ctx->ls_read[0] = st[2];
    ctx->ls_read[1] = st[3];
    return BIGCLAM_OK;
}

extern "C" int bigclam_get_tile_stats(bigclam_ctx *ctx, int64_t *tiles_done, int64_t *tiles_fallback, int64_t *n_tiles,
                                      int64_t *n_general_nodes, int64_t *n_split_hubs) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    unsigned int st[2] = {0u, 0u};
    if (ctx->sparse && ctx->d_stats != nullptr) {
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamSynchronize(ctx->stream));
        CU(cudaMemcpy(st, ctx->d_stats, sizeof(st), cudaMemcpyDeviceToHost));
    }
    if (tiles_done) *tiles_done = (int64_t)(st[0] - ctx->stats_read[0]);
    if (tiles_fallback) *tiles_fallback = (int64_t)(st[1] - ctx->stats_read[1]);
    ctx->stats_read[0] = st[0];
    ctx->stats_read[1] = st[1];
    if (n_tiles) *n_tiles = ctx->sparse ? ctx->ntiles : 0;
    if (n_general_nodes) *n_general_nodes = ctx->sparse ? ctx->n_gen : 0;
    if (n_split_hubs) *n_split_hubs = ctx->sparse ? ctx->n_hubs : 0;
    return BIGCLAM_OK;
}

// ------------------------------------------------------------------------------------------------
// Held-out pairs (thesis p.20; DESIGN.md (f) f-5): the masked objective drops every held-out pair (u, v) from the edge
// and the non-edge term, which leaves one linear term x_uv per pair in the per-node form (see SpGen::node).
extern "C" int bigclam_set_holdout(bigclam_ctx *ctx, const int64_t *ho_rowptr, const int32_t *ho_col, const uint8_t *ho_is_edge) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (!ctx->sparse) return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_set_holdout: needs a BIGCLAM_F_SPARSE_ROWS context");
    if (ctx->n_peers > 0 || ctx->x_world > 0)
        return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_set_holdout: the context has peers open (the masked objective runs on one GPU)");
    const int64_t n = ctx->n;
    bool all_owned = ctx->lo == 0 && ctx->hi == n && (int64_t)ctx->h_owned.size() == n;
    if (all_owned) {
        std::vector<uint8_t> seen((size_t)n, 0);
        for (int32_t u : ctx->h_owned) {
            if (seen[(size_t)u]) { all_owned = false; break; }
            seen[(size_t)u] = 1;
        }
    }
    if (!all_owned) return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_set_holdout: the context owns a node range or set (the masked objective needs all nodes)");
    CU(cudaSetDevice(ctx->device));
    if (ho_rowptr != nullptr) {
        // every check before anything on the device changes
        if (ho_rowptr[0] != 0) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: ho_rowptr[0] != 0");
        for (int64_t u = 0; u < n; ++u)
            if (ho_rowptr[u + 1] < ho_rowptr[u]) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: ho_rowptr not monotone at %lld", (long long)u);
        const int64_t m = ho_rowptr[n];
        if (m > 0 && (ho_col == nullptr || ho_is_edge == nullptr)) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: ho_col / ho_is_edge is NULL");
        for (int64_t e = 0; e < m; ++e) {
            if (ho_col[e] < 0 || ho_col[e] >= n) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: ho_col[%lld] out of range", (long long)e);
            if (ho_is_edge[e] > 1) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: ho_is_edge[%lld] is neither 0 nor 1", (long long)e);
        }
        // per row: (partner, label) sorted by partner, and the training neighbours sorted
        std::vector<std::pair<int32_t, uint8_t>> hs((size_t)m);
        for (int64_t e = 0; e < m; ++e) hs[(size_t)e] = {ho_col[e], ho_is_edge[e]};
        std::vector<int32_t> tr(ctx->h_col);
        const std::vector<int64_t> &rp = ctx->h_rowptr;
        for (int64_t u = 0; u < n; ++u) {
            std::sort(hs.begin() + ho_rowptr[u], hs.begin() + ho_rowptr[u + 1]);
            std::sort(tr.begin() + rp[u], tr.begin() + rp[u + 1]);
        }
        for (int64_t u = 0; u < n; ++u) {
            for (int64_t e = ho_rowptr[u]; e < ho_rowptr[u + 1]; ++e) {
                const int32_t v = hs[(size_t)e].first;
                const uint8_t lab = hs[(size_t)e].second;
                if (v == u) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: self pair at node %lld", (long long)u);
                if (e > ho_rowptr[u] && hs[(size_t)e - 1].first == v)
                    return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: pair (%lld, %d) listed twice", (long long)u, v);
                if (std::binary_search(tr.begin() + rp[u], tr.begin() + rp[u + 1], v))
                    return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: pair (%lld, %d) is also a training edge", (long long)u, v);
                const auto vb = hs.begin() + ho_rowptr[v], ve = hs.begin() + ho_rowptr[v + 1];
                const auto it = std::lower_bound(vb, ve, std::make_pair((int32_t)u, (uint8_t)0));
                if (it == ve || it->first != (int32_t)u)
                    return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: pair (%lld, %d) has no mirror (%d, %lld)", (long long)u, v, v, (long long)u);
                if (it->second != lab)
                    return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_holdout: pair (%lld, %d) and its mirror have different labels", (long long)u, v);
            }
        }
        if (int rd = drop_speculation(ctx)) return rd;
        CU(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_ho_rowptr); cudaFree(ctx->d_ho_col); cudaFree(ctx->d_ho_edge); cudaFree(ctx->d_ho_part);
        ctx->d_ho_rowptr = nullptr; ctx->d_ho_col = nullptr; ctx->d_ho_edge = nullptr; ctx->d_ho_part = nullptr;
        ctx->ho = false;
        CU(cudaMalloc(&ctx->d_ho_rowptr, sizeof(int64_t) * ((size_t)n + 1)));
        CU(cudaMalloc(&ctx->d_ho_col, sizeof(int32_t) * std::max<size_t>(1, (size_t)m)));
        CU(cudaMalloc(&ctx->d_ho_edge, std::max<size_t>(1, (size_t)m)));
        CU(cudaMalloc(&ctx->d_ho_part, sizeof(double) * ((size_t)n + 1)));
        CU(cudaMemcpy(ctx->d_ho_rowptr, ho_rowptr, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice));
        if (m > 0) {
            CU(cudaMemcpy(ctx->d_ho_col, ho_col, sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice));
            CU(cudaMemcpy(ctx->d_ho_edge, ho_is_edge, (size_t)m, cudaMemcpyHostToDevice));
        }
        CU(cudaFuncSetAttribute(tile_step_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->sp_smem));
        CU(cudaFuncSetAttribute(holdout_llh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * kHoWarps * (size_t)sp_ldp(ctx->ld))));
        ctx->ho_pairs = m / 2;
        ctx->ho = true;
    } else {
        if (int rd = drop_speculation(ctx)) return rd;
        CU(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_ho_rowptr); cudaFree(ctx->d_ho_col); cudaFree(ctx->d_ho_edge); cudaFree(ctx->d_ho_part);
        ctx->d_ho_rowptr = nullptr; ctx->d_ho_col = nullptr; ctx->d_ho_edge = nullptr; ctx->d_ho_part = nullptr;
        ctx->ho_pairs = 0;
        ctx->ho = false;
    }
    std::vector<int32_t> order = ctx->h_owned;            // the routing follows ctx->ho (rebuild_sparse_lists)
    return rebuild_order_list(ctx, ctx->h_rowptr, order);
}

extern "C" int bigclam_holdout_loglikelihood(bigclam_ctx *ctx, double *llh_out, int64_t *n_pairs_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (llh_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_holdout_loglikelihood: llh_out is NULL");
    if (!ctx->ho) return fail(ctx, BIGCLAM_EINVAL, "bigclam_holdout_loglikelihood: no held-out pairs (bigclam_set_holdout)");
    CU(cudaSetDevice(ctx->device));
    const bigclam_params &p = ctx->p;
    HoLlhArgs h{};
    h.hdr = ctx->d_hdr[ctx->cur];
    h.pool = ctx->d_pool[ctx->cur];
    h.ho_rowptr = ctx->d_ho_rowptr;
    h.ho_col = ctx->d_ho_col;
    h.ho_edge = ctx->d_ho_edge;
    h.n = ctx->n;
    h.ld = ctx->ld;
    h.min_p = p.min_p;
    h.max_p = p.max_p;
    h.x_lo = -std::log(p.max_p) * (1.0 - 1e-12);           // (fill_args)
    h.x_hi = -std::log(p.min_p) * (1.0 + 1e-12);
    h.part = ctx->d_ho_part;
    const unsigned blocks = (unsigned)((ctx->n + kHoWarps - 1) / kHoWarps);
    holdout_llh_kernel<<<blocks, kHoWarps * 32, sizeof(double) * kHoWarps * (size_t)sp_ldp(ctx->ld), ctx->stream>>>(h);
    CU(cudaGetLastError());
    holdout_sum_kernel<<<1, kHoSumThreads, 0, ctx->stream>>>(ctx->d_ho_part, ctx->n, ctx->d_ho_part + ctx->n);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(ctx->h_pinned, ctx->d_ho_part + ctx->n, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    *llh_out = ctx->h_pinned[0];
    if (n_pairs_out) *n_pairs_out = ctx->ho_pairs;
    return BIGCLAM_OK;
}

// ------------------------------------------------------------------------------------------------
// Node-partitioned pieces (DESIGN.md (e)).
extern "C" int bigclam_set_owned_range(bigclam_ctx *ctx, int64_t lo, int64_t hi) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (lo < 0 || hi < lo || hi > ctx->n) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_owned_range: bad range");
    if (ctx->ho) return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_set_owned_range: the context has held-out pairs (bigclam_set_holdout)");
    CU(cudaSetDevice(ctx->device));
    const std::vector<int64_t> &rp = ctx->h_rowptr;
    ctx->lo = lo;
    ctx->hi = hi;
    if (int rd = drop_speculation(ctx)) return rd;
    return rebuild_order(ctx, rp);
}

// uset of the following bigclam_step_local calls (n bytes from host memory, copied asynchronously; NULL = all vertices)
extern "C" int bigclam_set_uset(bigclam_ctx *ctx, const uint8_t *node_mask) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    ctx->local_mask = node_mask != nullptr;
    if (node_mask != nullptr) CU(cudaMemcpyAsync(ctx->d_mask, node_mask, (size_t)ctx->n, cudaMemcpyHostToDevice, ctx->stream));
    return BIGCLAM_OK;
}

extern "C" int bigclam_step_local(bigclam_ctx *ctx, void **partials_dev) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    if (int rd = drop_speculation(ctx)) return rd;
    // dense kernels accumulate their sums into d_partials: whatever an earlier call left there must not be counted
    // (the sparse engine's reduction overwrites them)
    if (!ctx->sparse) CU(cudaMemsetAsync(ctx->d_partials, 0, sizeof(double) * (2 * (size_t)ctx->ld + 2), ctx->stream));
    StepArgs a;
    fill_args(ctx, a, true, ctx->local_mask ? ctx->d_mask : nullptr, false);
    int rc = timed_launch(ctx, a, true);
    if (rc) return rc;
    if (partials_dev) *partials_dev = ctx->d_partials;
    return BIGCLAM_OK;
}

extern "C" int bigclam_finish_local(bigclam_ctx *ctx, double *llh_pre_out, int64_t *n_updated_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    const bool want = (llh_pre_out != nullptr) || (n_updated_out != nullptr);
    if (int rx = launch_xreduce(ctx, false)) return rx;      // (with the fused collective: every rank's sums first)
    if (want)
        CU(cudaMemcpyAsync(ctx->h_pinned, ctx->d_partials + 2 * ctx->ld, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    int rc = launch_finish(ctx, 0, 0, 0.0, true, false);
    if (rc) return rc;
    ctx->cur ^= 1;
    if (!want) return BIGCLAM_OK;            // fully asynchronous: nothing is read back, no host sync
    CU(cudaStreamSynchronize(ctx->stream));
    if (llh_pre_out) *llh_pre_out = ctx->h_pinned[0];
    if (n_updated_out) *n_updated_out = (int64_t)(ctx->h_pinned[1] + 0.5);
    return collect_timing(ctx);
}

extern "C" int bigclam_llh_local(bigclam_ctx *ctx, void **partials_dev) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    if (int rd = drop_speculation(ctx)) return rd;
    CU(cudaMemsetAsync(ctx->d_partials, 0, sizeof(double) * (2 * (size_t)ctx->ld + 2), ctx->stream));
    StepArgs a;
    fill_args(ctx, a, false, nullptr, false);
    int rc = timed_launch(ctx, a, false);
    if (rc) return rc;
    if (partials_dev) *partials_dev = ctx->d_partials;
    return BIGCLAM_OK;
}

extern "C" int bigclam_rollback(bigclam_ctx *ctx) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    if (int rd = drop_speculation(ctx)) return rd;
    invalidate_resets(ctx);
    ctx->cur ^= 1;
    ctx->dense_valid = false;
    return BIGCLAM_OK;
}


extern "C" int bigclam_device_accepted(bigclam_ctx *ctx, void **accepted_dev) {
    if (ctx == nullptr || accepted_dev == nullptr) return BIGCLAM_EINVAL;
    if (!(ctx->p.flags & BIGCLAM_F_RECORD_ACCEPTED))
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_device_accepted: context created without BIGCLAM_F_RECORD_ACCEPTED");
    *accepted_dev = ctx->d_accepted;
    return BIGCLAM_OK;
}

// ------------------------------------------------------------------------------------------------
// Peer replicas over NVLink (one process per GPU): every rank exports the CUDA IPC handles of its two
// F buffers, the host framework all-gathers them, every rank opens the others'.  After that the step
// kernel pushes changed rows straight into the peers' replicas (see StepArgs::peer_out).
extern "C" int bigclam_ipc_export(bigclam_ctx *ctx, void *handles_out /* 2 x 64 bytes */) {
    if (ctx == nullptr || handles_out == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    if (ctx->sparse) {                       // 4 handles: hdr[0], hdr[1], pool[0], pool[1]
        cudaIpcMemHandle_t h[4];
        CU(cudaIpcGetMemHandle(&h[0], ctx->d_hdr[0]));
        CU(cudaIpcGetMemHandle(&h[1], ctx->d_hdr[1]));
        CU(cudaIpcGetMemHandle(&h[2], ctx->d_pool[0]));
        CU(cudaIpcGetMemHandle(&h[3], ctx->d_pool[1]));
        std::memcpy(handles_out, h, sizeof(h));
        return BIGCLAM_OK;
    }
    cudaIpcMemHandle_t h[2];
    CU(cudaIpcGetMemHandle(&h[0], ctx->d_F[0]));
    CU(cudaIpcGetMemHandle(&h[1], ctx->d_F[1]));
    std::memcpy(handles_out, h, sizeof(h));
    return BIGCLAM_OK;
}

extern "C" int bigclam_ipc_open_peers(bigclam_ctx *ctx, int32_t world, int32_t rank, const void *all_handles /* world x 2 x 64 */) {
    if (ctx == nullptr || all_handles == nullptr || world < 1 || world > 8 || rank < 0 || rank >= world)
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_ipc_open_peers: bad world/rank (at most 8 GPUs)");
    if (ctx->ho) return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_ipc_open_peers: the context has held-out pairs (bigclam_set_holdout)");
    CU(cudaSetDevice(ctx->device));
    const cudaIpcMemHandle_t *h = reinterpret_cast<const cudaIpcMemHandle_t *>(all_handles);
    for (int half = 0; half < 2; ++half)            // a second call replaces the first mapping
        for (int r = 0; r < ctx->n_peers; ++r) {
            if (ctx->peer_F[half][r]) { cudaIpcCloseMemHandle(ctx->peer_F[half][r]); ctx->peer_F[half][r] = nullptr; }
            if (ctx->peer_hdr[half][r]) { cudaIpcCloseMemHandle(ctx->peer_hdr[half][r]); ctx->peer_hdr[half][r] = nullptr; }
            if (ctx->peer_pool[half][r]) { cudaIpcCloseMemHandle(ctx->peer_pool[half][r]); ctx->peer_pool[half][r] = nullptr; }
        }
    ctx->n_peers = 0;
    int np = 0;
    const int per = ctx->sparse ? 4 : 2;            // handles per rank (bigclam_ipc_handle_count)
    for (int r = 0; r < world; ++r) {
        if (r == rank) continue;
        for (int half = 0; half < 2; ++half) {
            void *p = nullptr;
            CU(cudaIpcOpenMemHandle(&p, h[per * r + half], cudaIpcMemLazyEnablePeerAccess));
            if (ctx->sparse) {
                ctx->peer_hdr[half][np] = reinterpret_cast<uint64_t *>(p);
                void *q = nullptr;
                CU(cudaIpcOpenMemHandle(&q, h[per * r + 2 + half], cudaIpcMemLazyEnablePeerAccess));
                ctx->peer_pool[half][np] = reinterpret_cast<double *>(q);
            } else {
                ctx->peer_F[half][np] = reinterpret_cast<double *>(p);
            }
        }
        ++np;
    }
    ctx->n_peers = np;
    if (ctx->d_changed == nullptr) CU(cudaMalloc(&ctx->d_changed, (size_t)ctx->n));
    // every row counts as changed before the first step, so the first step publishes all owned rows
    CU(cudaMemset(ctx->d_changed, 1, (size_t)ctx->n));
    return BIGCLAM_OK;
}

extern "C" int bigclam_mark_all_changed(bigclam_ctx *ctx) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (ctx->d_changed == nullptr) return BIGCLAM_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemsetAsync(ctx->d_changed, 1, (size_t)ctx->n, ctx->stream));
    return BIGCLAM_OK;
}

// Handles per rank that bigclam_ipc_export writes and bigclam_ipc_open_peers expects (64 bytes each).
extern "C" int bigclam_ipc_handle_count(const bigclam_ctx *ctx) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    return ctx->sparse ? 4 : 2;
}

// Sparse rows, multi-GPU: the part [base, base + cap) (8-byte words) of every replica's output pool that this
// rank allocates its owned rows in.  The parts of the ranks must not overlap; cap >= owned nodes * words of a
// full row can never overflow.
extern "C" int bigclam_set_pool_region(bigclam_ctx *ctx, int64_t base_words, int64_t cap_words) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (!ctx->sparse) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_pool_region: context without BIGCLAM_F_SPARSE_ROWS");
    if (base_words < 0 || cap_words < 0 || (uint64_t)base_words + (uint64_t)cap_words > ctx->pool_cap8)
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_pool_region: region outside the pool (%llu words)", (unsigned long long)ctx->pool_cap8);
    ctx->region_base8 = (uint64_t)base_words;
    ctx->region_cap8 = (uint64_t)cap_words;
    return BIGCLAM_OK;
}

// Sparse rows: capacity of each row pool in 8-byte words (the regions of bigclam_set_pool_region partition it).
extern "C" int bigclam_get_pool_capacity(bigclam_ctx *ctx, int64_t *words_out) {
    if (ctx == nullptr || words_out == nullptr) return BIGCLAM_EINVAL;
    if (!ctx->sparse) return fail(ctx, BIGCLAM_EINVAL, "bigclam_get_pool_capacity: context without BIGCLAM_F_SPARSE_ROWS");
    *words_out = (int64_t)ctx->pool_cap8;
    return BIGCLAM_OK;
}

// Sums the CUDA-event timings recorded since the last collection (asynchronous multi-GPU loops).
extern "C" int bigclam_collect_timing(bigclam_ctx *ctx) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    int rc = collect_timing(ctx);
    return rc;
}

// Arbitrary (non-contiguous) owned node set, e.g. the degree-sorted node list dealt round-robin over
// the ranks so that every rank gets the same mix of hubs and leaves (used with the peer-store exchange).
extern "C" int bigclam_set_owned_nodes(bigclam_ctx *ctx, const int32_t *nodes, int64_t count) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (count < 0 || count > ctx->n || (count > 0 && nodes == nullptr))
        return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_owned_nodes: bad node list");
    if (ctx->ho) return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_set_owned_nodes: the context has held-out pairs (bigclam_set_holdout)");
    for (int64_t i = 0; i < count; ++i)
        if (nodes[i] < 0 || nodes[i] >= ctx->n) return fail(ctx, BIGCLAM_EINVAL, "bigclam_set_owned_nodes: node out of range");
    CU(cudaSetDevice(ctx->device));
    const std::vector<int64_t> &rp = ctx->h_rowptr;
    std::vector<int32_t> order(nodes, nodes + count);
    ctx->lo = 0;
    ctx->hi = ctx->n;
    if (int rd = drop_speculation(ctx)) return rd;
    return rebuild_order_list(ctx, rp, order);
}

// Community extraction on the current F (Bigclamv2.scala:223-230); see extract_kernel.
extern "C" int bigclam_extract(bigclam_ctx *ctx, double delta, uint8_t *member_out /* n x k */, double *fmax_out /* n, optional */) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    if (member_out == nullptr) return fail(ctx, BIGCLAM_EINVAL, "bigclam_extract: member_out is NULL");
    CU(cudaSetDevice(ctx->device));
    if (int re = ensure_dense(ctx)) return re;
    const int k = ctx->p.k;
    uint8_t *d_member = nullptr;
    double *d_fmax = nullptr;
    cudaError_t e = cudaMalloc(&d_member, (size_t)ctx->n * k);
    if (e == cudaSuccess) e = cudaMalloc(&d_fmax, sizeof(double) * (size_t)ctx->n);
    const int wpb = 8;
    if (e == cudaSuccess) {
        extract_kernel<<<(unsigned)((ctx->n + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(ctx->d_F[ctx->cur], ctx->n, k, ctx->ld, delta, d_member, d_fmax);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(member_out, d_member, (size_t)ctx->n * k, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && fmax_out != nullptr) e = cudaMemcpyAsync(fmax_out, d_fmax, sizeof(double) * (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_member);
    cudaFree(d_fmax);
    if (e != cudaSuccess) return fail(ctx, BIGCLAM_ECUDA, "bigclam_extract: %s", cudaGetErrorString(e));
    return BIGCLAM_OK;
}

// ------------------------------------------------------------------------------------------------
// Fused collective of the node-partitioned path: exchange buffers (see bigclam_ctx::x_*).
static int xchg_alloc(bigclam_ctx *ctx, int32_t world, int32_t rank) {
    if (world < 1 || world > 8 || rank < 0 || rank >= world) return fail(ctx, BIGCLAM_EINVAL, "exchange buffers: bad world/rank (at most 8 GPUs)");
    if (!ctx->sparse) return fail(ctx, BIGCLAM_EUNSUPPORTED, "the fused collective needs BIGCLAM_F_SPARSE_ROWS");
    if (ctx->ho) return fail(ctx, BIGCLAM_EUNSUPPORTED, "exchange buffers: the context has held-out pairs (bigclam_set_holdout)");
    CU(cudaSetDevice(ctx->device));
    cudaFree(ctx->d_xbuf); ctx->d_xbuf = nullptr;
    cudaFree(ctx->d_xflags); ctx->d_xflags = nullptr;
    const size_t nb = sizeof(double) * 2 * (size_t)world * ((size_t)ctx->ld + 2);
    CU(cudaMalloc(&ctx->d_xbuf, nb));
    CU(cudaMemset(ctx->d_xbuf, 0, nb));
    CU(cudaMalloc(&ctx->d_xflags, sizeof(unsigned long long) * 8));
    CU(cudaMemset(ctx->d_xflags, 0, sizeof(unsigned long long) * 8));
    ctx->x_world = world;
    ctx->x_rank = rank;
    ctx->x_seq = 0;
    for (int r = 0; r < 8; ++r) { ctx->x_peer_buf[r] = nullptr; ctx->x_peer_flags[r] = nullptr; }
    ctx->x_peer_buf[rank] = ctx->d_xbuf;
    ctx->x_peer_flags[rank] = ctx->d_xflags;
    return BIGCLAM_OK;
}

extern "C" int bigclam_xchg_export(bigclam_ctx *ctx, int32_t world, int32_t rank, void *handles_out /* 2 x 64 bytes */) {
    if (ctx == nullptr || handles_out == nullptr) return BIGCLAM_EINVAL;
    if (int rc = xchg_alloc(ctx, world, rank)) return rc;
    cudaIpcMemHandle_t h[2];
    CU(cudaIpcGetMemHandle(&h[0], ctx->d_xbuf));
    CU(cudaIpcGetMemHandle(&h[1], ctx->d_xflags));
    std::memcpy(handles_out, h, sizeof(h));
    return BIGCLAM_OK;
}

extern "C" int bigclam_xchg_open_peers(bigclam_ctx *ctx, const void *all_handles /* world x 2 x 64 bytes, rank order */) {
    if (ctx == nullptr || all_handles == nullptr) return BIGCLAM_EINVAL;
    if (ctx->x_world < 1) return fail(ctx, BIGCLAM_EINVAL, "bigclam_xchg_open_peers: call bigclam_xchg_export first");
    if (ctx->ho) return fail(ctx, BIGCLAM_EUNSUPPORTED, "bigclam_xchg_open_peers: the context has held-out pairs (bigclam_set_holdout)");
    CU(cudaSetDevice(ctx->device));
    const cudaIpcMemHandle_t *h = reinterpret_cast<const cudaIpcMemHandle_t *>(all_handles);
    for (int r = 0; r < ctx->x_world; ++r) {
        if (r == ctx->x_rank) continue;
        void *p = nullptr, *q = nullptr;
        CU(cudaIpcOpenMemHandle(&p, h[2 * r], cudaIpcMemLazyEnablePeerAccess));
        CU(cudaIpcOpenMemHandle(&q, h[2 * r + 1], cudaIpcMemLazyEnablePeerAccess));
        ctx->x_peer_buf[r] = reinterpret_cast<double *>(p);
        ctx->x_peer_flags[r] = reinterpret_cast<unsigned long long *>(q);
    }
    ctx->x_ipc = true;
    return BIGCLAM_OK;
}

// After bigclam_llh_local: the all-rank sum of the PRE block's llh_u (fused collective), synchronous.
extern "C" int bigclam_llh_finish_local(bigclam_ctx *ctx, double *llh_out) {
    if (ctx == nullptr) return BIGCLAM_EINVAL;
    CU(cudaSetDevice(ctx->device));
    if (int rx = launch_xreduce(ctx, false)) return rx;
    CU(cudaMemcpyAsync(ctx->h_pinned, ctx->d_partials + 2 * ctx->ld, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (llh_out) *llh_out = ctx->h_pinned[0];
    return BIGCLAM_OK;
}

// ------------------------------------------------------------------------------------------------
// All the GPUs of one box behind ONE handle, for a single-threaded caller (the JVM driver of INTEGRATION.md): one
// context per device, nodes dealt over the ranks by degree, every rank's new rows stored into all replicas by the
// step kernel (peer memory over NVLink), the sums combined by the fused collective above.  No NCCL, no Python.
struct bigclam_multi {
    int world = 0;
    std::vector<bigclam_ctx *> r;
    int64_t n = 0;
    int32_t k = 0, ld = 0;
    std::string err;
};
static thread_local std::string g_multi_err;

static int mfail(bigclam_multi *m, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    std::vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (m != nullptr) m->err = buf; else g_multi_err = buf;
    return code;
}
static int mfail_from(bigclam_multi *m, int code, bigclam_ctx *c) { return mfail(m, code, "%s", bigclam_last_error(c)); }

extern "C" const char *bigclam_multi_last_error(const bigclam_multi *m) { return m != nullptr ? m->err.c_str() : g_multi_err.c_str(); }

extern "C" void bigclam_multi_destroy(bigclam_multi *m) {
    if (m == nullptr) return;
    for (bigclam_ctx *c : m->r) {
        if (c == nullptr) continue;
        for (int h = 0; h < 2; ++h)
            for (int q = 0; q < 7; ++q) { c->peer_hdr[h][q] = nullptr; c->peer_pool[h][q] = nullptr; }   // direct pointers, not IPC mappings
        c->n_peers = 0;
        free_ctx(c);
    }
    delete m;
}

extern "C" int bigclam_multi_create(bigclam_multi **out, int64_t n, const int64_t *rowptr, const int32_t *col,
                                    const bigclam_params *params, int32_t world, const int32_t *devices) {
    if (out == nullptr) return mfail(nullptr, BIGCLAM_EINVAL, "bigclam_multi_create: out is NULL");
    *out = nullptr;
    if (params == nullptr || world < 1 || world > 8) return mfail(nullptr, BIGCLAM_EINVAL, "bigclam_multi_create: world must be 1..8");
    bigclam_multi *m = new (std::nothrow) bigclam_multi();
    if (m == nullptr) return mfail(nullptr, BIGCLAM_ENOMEM, "bigclam_multi_create: out of host memory");
    m->world = world;
    m->n = n;
    m->k = params->k;
    m->ld = (params->k + 3) & ~3;
    m->r.assign((size_t)world, nullptr);
#define MFAIL(code, ...)                             \
    do {                                             \
        mfail(nullptr, code, __VA_ARGS__);           \
        bigclam_multi_destroy(m);                    \
        return code;                                 \
    } while (0)
    for (int i = 0; i < world; ++i) {
        bigclam_params p = *params;
        p.device = devices != nullptr ? devices[i] : i;
        p.flags |= BIGCLAM_F_SPARSE_ROWS;
        int rc = bigclam_create(&m->r[(size_t)i], n, rowptr, col, &p);
        if (rc != BIGCLAM_OK) MFAIL(rc, "bigclam_multi_create: device %d: %s", p.device, bigclam_last_error(nullptr));
    }
    if (world > 1) {
        // peer access both ways (already enabled is fine)
        for (int i = 0; i < world; ++i)
            for (int j = 0; j < world; ++j) {
                if (i == j || m->r[(size_t)i]->device == m->r[(size_t)j]->device) continue;
                if (cudaSetDevice(m->r[(size_t)i]->device) != cudaSuccess) MFAIL(BIGCLAM_ECUDA, "bigclam_multi_create: cudaSetDevice failed");
                int can = 0;
                cudaDeviceCanAccessPeer(&can, m->r[(size_t)i]->device, m->r[(size_t)j]->device);
                if (!can) MFAIL(BIGCLAM_EUNSUPPORTED, "bigclam_multi_create: device %d cannot access device %d", m->r[(size_t)i]->device, m->r[(size_t)j]->device);
                cudaError_t e = cudaDeviceEnablePeerAccess(m->r[(size_t)j]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) MFAIL(BIGCLAM_ECUDA, "bigclam_multi_create: cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
                (void)cudaGetLastError();
            }
        // owned nodes: the degree-sorted node list dealt to the least loaded rank (load = neighbour-list entries + 1 per
        // node, ties to the lowest rank): equal work even when a few hubs hold a sizeable part of the edges; pool
        // regions in proportion to the owned counts
        std::vector<int32_t> order((size_t)n);
        std::iota(order.begin(), order.end(), 0);
        std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return (rowptr[a + 1] - rowptr[a]) > (rowptr[b + 1] - rowptr[b]); });
        std::vector<std::vector<int32_t>> mine((size_t)world);
        {
            std::vector<int64_t> load((size_t)world, 0);
            for (int64_t q = 0; q < n; ++q) {
                int best = 0;
                for (int i = 1; i < world; ++i)
                    if (load[(size_t)i] < load[(size_t)best]) best = i;
                const int32_t u = order[(size_t)q];
                mine[(size_t)best].push_back(u);
                load[(size_t)best] += (rowptr[u + 1] - rowptr[u]) + 1;
            }
        }
        uint64_t cap = m->r[0]->pool_cap8;
        for (int i = 1; i < world; ++i) cap = std::min(cap, m->r[(size_t)i]->pool_cap8);
        uint64_t base = 0;
        for (int i = 0; i < world; ++i) {
            bigclam_ctx *c = m->r[(size_t)i];
            int rc = bigclam_set_owned_nodes(c, mine[(size_t)i].data(), (int64_t)mine[(size_t)i].size());
            if (rc != BIGCLAM_OK) MFAIL(rc, "bigclam_multi_create: %s", bigclam_last_error(c));
            uint64_t share = (uint64_t)((double)cap * (double)mine[(size_t)i].size() / (double)n) & ~(uint64_t)1;
            if (i == world - 1) share = (cap - base) & ~(uint64_t)1;
            rc = bigclam_set_pool_region(c, (int64_t)base, (int64_t)share);
            if (rc != BIGCLAM_OK) MFAIL(rc, "bigclam_multi_create: %s", bigclam_last_error(c));
            base += share;
            rc = xchg_alloc(c, world, i);
            if (rc != BIGCLAM_OK) MFAIL(rc, "bigclam_multi_create: %s", bigclam_last_error(c));
        }
        for (int i = 0; i < world; ++i) {
            bigclam_ctx *c = m->r[(size_t)i];
            int np = 0;
            for (int j = 0; j < world; ++j) {
                bigclam_ctx *o = m->r[(size_t)j];
                c->x_peer_buf[j] = o->d_xbuf;
                c->x_peer_flags[j] = o->d_xflags;
                if (j == i) continue;
                for (int h = 0; h < 2; ++h) { c->peer_hdr[h][np] = o->d_hdr[h]; c->peer_pool[h][np] = o->d_pool[h]; }
                ++np;
            }
            c->n_peers = np;
        }
    }
#undef MFAIL
    *out = m;
    return BIGCLAM_OK;
}

#define MCALL(expr, c)                                           \
    do {                                                         \
        int rc__ = (expr);                                       \
        if (rc__ != BIGCLAM_OK) return mfail_from(m, rc__, c);   \
    } while (0)

extern "C" int bigclam_multi_set_F(bigclam_multi *m, const double *F) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    for (bigclam_ctx *c : m->r) MCALL(bigclam_set_F(c, F), c);
    return BIGCLAM_OK;
}
extern "C" int bigclam_multi_set_F_csr(bigclam_multi *m, const int64_t *indptr, const int32_t *indices, const double *values) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    for (bigclam_ctx *c : m->r) MCALL(bigclam_set_F_csr(c, indptr, indices, values), c);
    return BIGCLAM_OK;
}
extern "C" int bigclam_multi_set_sumF(bigclam_multi *m, const double *sumF) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    for (bigclam_ctx *c : m->r) MCALL(bigclam_set_sumF(c, sumF), c);
    return BIGCLAM_OK;
}
extern "C" int bigclam_multi_get_F(bigclam_multi *m, int32_t rank, double *F_out) {
    if (m == nullptr || rank < 0 || rank >= m->world) return BIGCLAM_EINVAL;
    MCALL(bigclam_get_F(m->r[(size_t)rank], F_out), m->r[(size_t)rank]);
    return BIGCLAM_OK;
}
extern "C" int bigclam_multi_get_sumF(bigclam_multi *m, int32_t rank, double *sumF_out) {
    if (m == nullptr || rank < 0 || rank >= m->world) return BIGCLAM_EINVAL;
    MCALL(bigclam_get_sumF(m->r[(size_t)rank], sumF_out), m->r[(size_t)rank]);
    return BIGCLAM_OK;
}
extern "C" int bigclam_multi_get_F_nnz(bigclam_multi *m, int64_t *nnz_out) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    MCALL(bigclam_get_F_nnz(m->r[0], nnz_out), m->r[0]);
    return BIGCLAM_OK;
}
extern "C" int bigclam_multi_get_F_csr(bigclam_multi *m, int64_t *indptr_out, int32_t *indices_out, double *values_out) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    MCALL(bigclam_get_F_csr(m->r[0], indptr_out, indices_out, values_out), m->r[0]);
    return BIGCLAM_OK;
}

// One kernel round over all ranks: every rank's step (or PRE-only) kernel and reduction first, then every rank's
// combine + finish — a rank's combine waits on device flags for the other ranks' reductions, so nothing of the
// second half may be queued in front of another rank's first half.
static int multi_round(bigclam_multi *m, bool linesearch, const uint8_t *host_mask, bool use_done, long long kernel_index,
                       int variant, double rel_tol, bool apply, bool llh_is_final) {
    for (bigclam_ctx *c : m->r) {
        if (cudaSetDevice(c->device) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "cudaSetDevice(%d) failed", c->device);
        const uint8_t *d_mask = nullptr;
        if (host_mask != nullptr) {
            if (cudaMemcpyAsync(c->d_mask, host_mask, (size_t)c->n, cudaMemcpyHostToDevice, c->stream) != cudaSuccess)
                return mfail(m, BIGCLAM_ECUDA, "uset upload failed");
            d_mask = c->d_mask;
        }
        StepArgs a;
        fill_args(c, a, linesearch, d_mask, use_done);
        MCALL(timed_launch(c, a, linesearch), c);
    }
    for (bigclam_ctx *c : m->r) {
        if (cudaSetDevice(c->device) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "cudaSetDevice(%d) failed", c->device);
        MCALL(launch_xreduce(c, use_done), c);
        MCALL(launch_finish(c, kernel_index, variant, rel_tol, apply, llh_is_final), c);
    }
    return BIGCLAM_OK;
}

static int multi_sync(bigclam_multi *m) {
    for (bigclam_ctx *c : m->r) {
        if (cudaSetDevice(c->device) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
            return mfail(m, BIGCLAM_ECUDA, "device %d: %s", c->device, cudaGetErrorString(cudaGetLastError()));
        if (int ro = check_overflow(c)) return mfail_from(m, ro, c);
    }
    return BIGCLAM_OK;
}

// PRE-only round; the all-rank LLH lands in every rank's partials (finish with apply = 0 leaves the state alone)
static int multi_llh(bigclam_multi *m, double *llh_out) {
    for (bigclam_ctx *c : m->r) {
        if (cudaSetDevice(c->device) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "cudaSetDevice(%d) failed", c->device);
        StepArgs a;
        fill_args(c, a, false, nullptr, false);
        MCALL(timed_launch(c, a, false), c);
    }
    for (bigclam_ctx *c : m->r) {
        if (cudaSetDevice(c->device) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "cudaSetDevice(%d) failed", c->device);
        MCALL(launch_xreduce(c, false), c);
    }
    bigclam_ctx *c0 = m->r[0];
    if (cudaSetDevice(c0->device) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "cudaSetDevice failed");
    if (cudaMemcpyAsync(c0->h_pinned, c0->d_partials + 2 * c0->ld, sizeof(double), cudaMemcpyDeviceToHost, c0->stream) != cudaSuccess)
        return mfail(m, BIGCLAM_ECUDA, "LLH download failed");
    if (int rs = multi_sync(m)) return rs;
    if (llh_out) *llh_out = c0->h_pinned[0];
    return BIGCLAM_OK;
}

extern "C" int bigclam_multi_loglikelihood(bigclam_multi *m, double *llh_out) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    for (bigclam_ctx *c : m->r) { if (cudaSetDevice(c->device) == cudaSuccess) { int rc = reset_run_state(c); if (rc) return mfail_from(m, rc, c); } }
    return multi_llh(m, llh_out);
}

// backtrackingLineSearchs(uset) over all GPUs: one step round, then a PRE-only round for the LLH it returns.
extern "C" int bigclam_multi_step(bigclam_multi *m, const uint8_t *node_mask, double *llh_out, int64_t *n_updated_out) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    for (bigclam_ctx *c : m->r) { if (cudaSetDevice(c->device) == cudaSuccess) { int rc = reset_run_state(c); if (rc) return mfail_from(m, rc, c); } }
    if (int rr = multi_round(m, true, node_mask, false, 0, 0, 0.0, true, false)) return rr;
    for (bigclam_ctx *c : m->r) { c->cur ^= 1; c->dense_valid = false; }
    bigclam_ctx *c0 = m->r[0];
    cudaSetDevice(c0->device);
    if (cudaMemcpyAsync(c0->h_pinned + 8, c0->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, c0->stream) != cudaSuccess)
        return mfail(m, BIGCLAM_ECUDA, "state download failed");
    double llh = 0.0;
    if (int rl = multi_llh(m, &llh)) return rl;
    if (llh_out) *llh_out = llh;
    if (n_updated_out) *n_updated_out = reinterpret_cast<RunState *>(c0->h_pinned + 8)->n_updated;
    for (bigclam_ctx *c : m->r) { cudaSetDevice(c->device); collect_timing(c); }
    return BIGCLAM_OK;
}

// The outer loop (bigclam_run) over all GPUs: same device-side bookkeeping on every rank (they all see the same sums).
extern "C" int bigclam_multi_run(bigclam_multi *m, int32_t variant, double rel_tol, int64_t max_outer, double *llh_out,
                                 int64_t *calls_out, double *llh_trace, int64_t trace_cap) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    if (variant != 2 && variant != 3 && variant != 4) return mfail(m, BIGCLAM_EINVAL, "bigclam_multi_run: variant must be 2, 3 or 4");
    if (max_outer < 0 || trace_cap < 0) return mfail(m, BIGCLAM_EINVAL, "bigclam_multi_run: negative max_outer/trace_cap");
    bigclam_ctx *c0 = m->r[0];
    for (bigclam_ctx *c : m->r) {
        if (cudaSetDevice(c->device) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "cudaSetDevice failed");
        int rc = reset_run_state(c);
        if (rc) return mfail_from(m, rc, c);
        c->trace_cap = 0;
    }
    cudaSetDevice(c0->device);
    if (llh_trace != nullptr && trace_cap > 0) {
        cudaFree(c0->d_trace);
        c0->d_trace = nullptr;
        if (cudaMalloc(&c0->d_trace, sizeof(double) * (size_t)trace_cap) != cudaSuccess) return mfail(m, BIGCLAM_ENOMEM, "trace buffer");
        c0->trace_cap = trace_cap;
    }
    RunState *hst = reinterpret_cast<RunState *>(c0->h_pinned + 8);
    const int start_cur = c0->cur;
    const int64_t batch = 8;
    int64_t cdone = 0;
    bool done = false;
    while (!done) {
        int64_t todo = batch;
        if (max_outer > 0) todo = std::min<int64_t>(batch, max_outer - cdone);
        for (int64_t i = 0; i < todo; ++i) {
            ++cdone;
            for (bigclam_ctx *c : m->r) c->cur = (start_cur + (int)((cdone - 1) & 1)) & 1;
            if (int rr = multi_round(m, true, nullptr, true, cdone, variant, rel_tol, true, false)) return rr;
        }
        cudaSetDevice(c0->device);
        if (cudaMemcpyAsync(hst, c0->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, c0->stream) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "state download failed");
        if (int rs = multi_sync(m)) return rs;
        if (hst->done) { done = true; break; }
        if (max_outer > 0 && cdone >= max_outer) break;
    }
    int64_t calls;
    if (done) {
        calls = hst->conv_call;
    } else {
        calls = cdone;
        for (bigclam_ctx *c : m->r) c->cur = (start_cur + (int)(cdone & 1)) & 1;
        if (int rr = multi_round(m, false, nullptr, false, cdone, variant, rel_tol, false, true)) return rr;
        cudaSetDevice(c0->device);
        if (cudaMemcpyAsync(hst, c0->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, c0->stream) != cudaSuccess) return mfail(m, BIGCLAM_ECUDA, "state download failed");
        if (int rs = multi_sync(m)) return rs;
    }
    for (bigclam_ctx *c : m->r) { c->cur = (start_cur + (int)(calls & 1)) & 1; c->dense_valid = false; invalidate_resets(c); }
    if (llh_out) *llh_out = hst->ret_llh;
    if (calls_out) *calls_out = calls;
    if (llh_trace != nullptr && trace_cap > 0) {
        const int64_t cnt = std::min<int64_t>(calls, trace_cap);
        cudaSetDevice(c0->device);
        if (cnt > 0 && cudaMemcpy(llh_trace, c0->d_trace, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost) != cudaSuccess)
            return mfail(m, BIGCLAM_ECUDA, "trace download failed");
    }
    for (bigclam_ctx *c : m->r) { cudaSetDevice(c->device); collect_timing(c); }
    return BIGCLAM_OK;
}

// Step-kernel time of the most recent bigclam_multi_step / bigclam_multi_run: the slowest rank's sum (BIGCLAM_F_TIME_KERNELS).
extern "C" int bigclam_multi_get_kernel_time(bigclam_multi *m, double *max_rank_ms_sum, int64_t *step_kernel_launches) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    double mx = 0.0;
    for (bigclam_ctx *c : m->r) mx = std::max(mx, c->last_step_ms);
    if (max_rank_ms_sum) *max_rank_ms_sum = mx;
    if (step_kernel_launches) *step_kernel_launches = m->r[0]->last_step_launches;
    return BIGCLAM_OK;
}

extern "C" int bigclam_multi_get_ls_stats(bigclam_multi *m, int64_t *nodes_asked, int64_t *nodes_searched) {
    if (m == nullptr) return BIGCLAM_EINVAL;
    int64_t asked = 0, searched = 0;
    for (bigclam_ctx *c : m->r) {                      // every rank counts the nodes it owns
        int64_t a = 0, s = 0;
        const int rc = bigclam_get_ls_stats(c, &a, &s);
        if (rc) return mfail_from(m, rc, c);
        asked += a;
        searched += s;
    }
    if (nodes_asked) *nodes_asked = asked;
    if (nodes_searched) *nodes_searched = searched;
    return BIGCLAM_OK;
}

extern "C" int bigclam_multi_world(const bigclam_multi *m) { return m != nullptr ? m->world : BIGCLAM_EINVAL; }
#undef MCALL
