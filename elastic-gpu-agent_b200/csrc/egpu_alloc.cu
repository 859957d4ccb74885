// egpu_alloc.cu — best-fit fractional-GPU allocation on B200 (sm_100a) + its C ABI.
//
// Product path.  There is no CPU fallback in this file and nothing here
// includes or links oracle/: when no CUDA device is usable every entry point
// returns EGPU_ERR_NO_DEVICE.
//
// Reference slot this fills: baseDevicePlugin.GetPreferredAllocation, an empty
// stub in elastic-ai/elastic-gpu-agent (pkg/plugins/base.go:94-96); units from
// pkg/common/const.go:4 and pkg/plugins/gpushare.go:24-33,159-168.  The decision
// rule is the builder-defined spec of DESIGN.md §2 (the reference has none).
#include "egpu_kernels.cuh"

#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/egpu_alloc.h"

#include "egpu_scan.cuh"
#include "egpu_replay.cuh"
#include "egpu_cards.cuh"

// =============================================================================
// Host side: context + C ABI
// =============================================================================
using namespace egpu;

#include "egpu_ctx.h"

namespace {

constexpr int64_t kMaxRows = (1ll << 31) - 1;  // EGPU_MAX_ROWS

// host copy of resort_table_cta: sorted view of a freshly set table
void fill_sorted(DevState& h) {
    const int D = h.D;
    for (int j = 0; j < kMaxD; ++j) {
        h.sorted_k[j] = kPadWord;
        h.sorted_dev[j] = -1;
    }
    unsigned long long packed = ~0ull;
    for (int d = 0; d < D; ++d) {
        const uint32_t mine = (static_cast<uint32_t>(h.free_core[d]) << 24) | (static_cast<uint32_t>(h.free_mem[d]) << 6) | d;
        int pos = 0;
        for (int k = 0; k < D; ++k) {
            const uint32_t other = (static_cast<uint32_t>(h.free_core[k]) << 24) | (static_cast<uint32_t>(h.free_mem[k]) << 6) | k;
            pos += other < mine;
        }
        h.sorted_k[pos] = pack_table_word(h.free_core[d], h.free_mem[d]) | (static_cast<uint32_t>(pos) & 31u);
        h.sorted_dev[pos] = d;
        if (pos < 8) packed = (packed & ~(0xffull << (8 * pos))) | (static_cast<unsigned long long>(d) << (8 * pos));
    }
    h.dev_packed = packed;
}

// ---- output ranges of the launches in flight (pipelined launches must not share outputs) ----
// the three outputs of one batch: indices, demand sums, table'
void batch_outputs(egpu_ctx::Range* r, const void* idx, int64_t R, const void* delta, const void* table_out, int D) {
    const uintptr_t pi = reinterpret_cast<uintptr_t>(idx), pd = reinterpret_cast<uintptr_t>(delta),
                    pt = reinterpret_cast<uintptr_t>(table_out);
    r[0] = {pi, pi + static_cast<uintptr_t>(R) * sizeof(int32_t)};
    r[1] = {pd, pd + (pd ? sizeof(long long) * 2 * D : 0)};
    r[2] = {pt, pt + (pt ? sizeof(int32_t) * 3 * D : 0)};
}
// `r[0..n)`: drops empty ranges, sorts by address; returns the new count, or -1 when two of
// them overlap each other.
int prepare_ranges(egpu_ctx::Range* r, int n) {
    int m = 0;
    for (int i = 0; i < n; ++i)
        if (r[i].hi > r[i].lo) r[m++] = r[i];
    std::sort(r, r + m, [](const egpu_ctx::Range& a, const egpu_ctx::Range& b) { return a.lo < b.lo; });
    for (int i = 1; i < m; ++i)
        if (r[i].lo < r[i - 1].hi) return -1;
    return m;
}
// both sorted and internally disjoint: one sweep
bool overlaps_inflight(const std::vector<egpu_ctx::Range>& f, const egpu_ctx::Range* r, int n) {
    size_t i = 0;
    int k = 0;
    while (i < f.size() && k < n) {
        if (f[i].hi <= r[k].lo) ++i;
        else if (r[k].hi <= f[i].lo) ++k;
        else return true;
    }
    return false;
}
void add_inflight(egpu_ctx* ctx, const egpu_ctx::Range* r, int n) {
    ctx->range_tmp.resize(ctx->inflight.size() + static_cast<size_t>(n));
    std::merge(ctx->inflight.begin(), ctx->inflight.end(), r, r + n, ctx->range_tmp.begin(),
               [](const egpu_ctx::Range& a, const egpu_ctx::Range& b) { return a.lo < b.lo; });
    ctx->inflight.swap(ctx->range_tmp);
}
void new_group(egpu_ctx* ctx) {
    ctx->group_len = 0;
    ctx->group_mbatches = 0;
    ctx->inflight.clear();
}

// ---- the scan kernels ----
int d_bucket(int D) { return D <= 8 ? 0 : D <= 16 ? 1 : D <= 32 ? 2 : 3; }

// Every scan kernel of one D bucket.  The register scans run 256 threads per CTA (128 at D = 64),
// the lookup scans 256 whatever D is.
template <int DT, int THREADS = (DT == 64 ? 128 : 256)>
void fill_bucket(egpu_ctx* ctx, int b) {
    using Snap = SnapSmem<DT, THREADS>;
    using Lut = LutSmem<256>;
    ctx->single[kSorted][b] = {bestfit_sorted_kernel<DT, THREADS>, THREADS, sizeof(Snap)};
    ctx->single[kGrid][b] = {bestfit_grid_kernel<DT, THREADS>, THREADS, sizeof(Snap)};
    ctx->single[kLut][b] = {bestfit_lut_kernel<256>, 256, sizeof(Lut)};
    ctx->single[kSortedContig][b] = {bestfit_sorted_kernel<DT, THREADS, true>, THREADS, sizeof(Snap)};
    ctx->single[kLutContig][b] = {bestfit_lut_kernel<256, true>, 256, sizeof(Lut)};
    ctx->multi[0][b] = {bestfit_sorted_multi_kernel<DT, THREADS>, THREADS, sizeof(Snap)};
    ctx->multi[1][b] = {bestfit_lut_multi_kernel<256>, 256, sizeof(Lut)};
    ctx->packed[b] = {bestfit_sorted_packed_kernel<DT, THREADS>, THREADS, sizeof(Snap)};
    ctx->cards[b] = {cards_scan_kernel<DT, THREADS>, THREADS, sizeof(CardsSmem<DT, THREADS>)};
}

// first use of a kernel on this context: opt in to its shared-memory size, ask its occupancy
template <class Fn>
int configure(egpu_ctx* ctx, ScanKernel<Fn>& k) {
    if (k.ctas_per_sm != 0) return EGPU_OK;
    int per_sm = 0;
    EGPU_CUDA(ctx, cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(k.smem)));
    EGPU_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k.fn, k.threads, k.smem));
    k.ctas_per_sm = per_sm < 1 ? 1 : per_sm;
    return EGPU_OK;
}

// A scan launch with the programmatic-dependent-launch attribute (see pdl_flags).
template <class... Params, class... Args>
int launch_pdl(egpu_ctx* ctx, const ScanKernel<void (*)(Params...)>& k, int64_t ctas, cudaStream_t s, const Args&... args) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(ctas));
    cfg.blockDim = dim3(static_cast<unsigned>(k.threads));
    cfg.dynamicSmemBytes = k.smem;
    cfg.stream = s;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    EGPU_CUDA(ctx, cudaLaunchKernelEx(&cfg, k.fn, args...));
    ctx->launches += 1;
    return EGPU_OK;
}

bool uses_lut(const egpu_ctx* ctx) {
    return ctx->variant == EGPU_VARIANT_LUT || (ctx->variant == EGPU_VARIANT_AUTO && ctx->D > 16);
}

// rebuild the lookup tables on the launching stream when the table has changed since they were built
int refresh_lut(egpu_ctx* ctx, cudaStream_t s) {
    if (!ctx->lut_dirty) return EGPU_OK;
    lut_build_kernel<<<1, 256, 0, s>>>(ctx->d_state, ctx->d_lut);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    ctx->lut_dirty = false;
    ctx->prev_is_scan = false;
    return EGPU_OK;
}

// Launches per pipelined group.  With a ring of 32 output buffers, groups of 24 with boundary
// launches give 2.34 us per step against 2.45 for groups of 16 (B200, DESIGN.md 7.2).
constexpr int kPipeGroup = 24;
static_assert(kPipeGroup + 1 < kEpiSlots, "every launch in flight needs its own epilogue slot");

// Programmatic dependent launch.  Every scan carries the PDL attribute, so the
// hardware may schedule it while its predecessor is still running.  A fully
// ordered launch waits (griddepcontrol.wait) before it touches anything.  A
// pipelined launch (kFlagLateWait) runs scan and epilogue at once — its epilogue
// state is its own slot — and waits only before exiting.  That is allowed when
//  - the caller vouches its inputs were complete before the previous launch on
//    this stream (EGPU_F_INPUTS_READY),
//  - the previous launch was a scan of this context on the same stream that
//    does not rewrite the table, and this one is a plain scan (`may_pipeline`),
//  - it does not commit (a committing launch rewrites the table the launches still in
//    flight read and compute their table' from: it is always fully ordered),
//  - its outputs (indices, demand sums, table') are disjoint from the outputs
//    of every launch since the last fully ordered one, and
//  - fewer than kPipeGroup launches have been issued since then, which bounds
//    the launches in flight to kPipeGroup + 1 < kEpiSlots, and the epi_multi slots
//    they hold (`mbatches` more for this launch) to half of that ring.
// Returns the launch's PDL flags; starts a new group unless the launch pipelines.
int pdl_flags(egpu_ctx* ctx, bool may_pipeline, int user_flags, cudaStream_t s, const egpu_ctx::Range* mine, int n_mine,
              int mbatches) {
    const bool pipelined = may_pipeline && (user_flags & EGPU_F_INPUTS_READY) && !(user_flags & EGPU_F_COMMIT) &&
                           ctx->prev_is_scan && !ctx->prev_changes_table && ctx->prev_stream == s && ctx->group_len > 0 &&
                           !overlaps_inflight(ctx->inflight, mine, n_mine);
    int flags = 0;
    if (pipelined) {
        flags |= kFlagLateWait;
        if (ctx->group_len >= kPipeGroup || ctx->group_mbatches + mbatches > kMultiSlots - kMultiMax) {
            // group boundary: this launch still scans alongside its predecessors, but it waits
            // for them before its epilogue and only then lets its successors start; it becomes
            // the first member of the next group
            flags |= kFlagBoundary;
            new_group(ctx);
        }
    } else {
        new_group(ctx);
    }
    // Early trigger (griddepcontrol.launch_dependents before the work is done) only helps when
    // the next launch is another scan of a pipelined stream, so only those launches do it.
    // (Checked on B200, scripts/probes/pdl_event_probe.cu and scripts/eager_probe.py: events
    // and ordinary kernels enqueued after a PDL launch still wait for its completion.)
    if (user_flags & EGPU_F_INPUTS_READY) flags |= kFlagEarlyTrigger;
    return flags;
}

// after a scan launch that went through pdl_flags: it joins the group, and the next scan may pipeline behind it
void note_scan(egpu_ctx* ctx, cudaStream_t s, const egpu_ctx::Range* mine, int n_mine, bool commit, int mbatches) {
    add_inflight(ctx, mine, n_mine);
    ctx->group_len += 1;
    ctx->group_mbatches += mbatches;
    ctx->prev_is_scan = true;
    ctx->prev_changes_table = commit;
    ctx->prev_stream = s;
    if (commit) ctx->lut_dirty = true;
}

// Grid of a single-batch launch: one resident wave at most.  A lone launch wants every SM pulling
// at once (8 rows per thread, one trip); launches of a pipelined stream overlap each other, so a
// smaller grid with more rows per thread (48) costs fewer CTA launches, fewer atomics and leaves
// room for the neighbours — measured best on B200 at R = 1M.  A lone lookup scan has a 13 KB
// per-CTA table tile to amortise (32).  The zero-copy path passes its own hint (see egpu_bestfit_batch).
// (Measured and dropped: giving the launches of a pipelined stream that could not themselves be
// pipelined - the first of a graph - the lone-launch grid: 2.80 against 2.68 us per step.)
constexpr int kRowsPerThread = 8;
constexpr int kRowsPerThreadPipelined = 48;  // lookup scan or D <= 16
constexpr int kRowsPerThreadLoneLut = 32;
// Batches this large get two waves of CTAs: the CTA scheduler then evens out the SMs (see launch_multi).
constexpr int64_t kTwoWaveRows = 16ll << 20;

// CTAs of a single-batch launch with `rpt` rows per thread: at most one resident wave, two for
// batches of kTwoWaveRows rows and more when `two_waves`.  0 when a lane would sum 2^19 rows or
// more: its lane-private demand sums (kAccShift) would overflow.
template <class Fn>
int64_t single_ctas(const egpu_ctx* ctx, const ScanKernel<Fn>& kern, int64_t R, int rpt, bool two_waves) {
    const int64_t per_cta = static_cast<int64_t>(kern.threads) * ((rpt + 3) / 4);
    int64_t want = ((R >> 2) + per_cta - 1) / per_cta;
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * kern.ctas_per_sm * ((R >= kTwoWaveRows && two_waves) ? 2 : 1);
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    if (R / (want * kern.threads) + 8 >= (1ll << 19)) return 0;
    return want;
}

// One batch.  user_flags: EGPU_F_COMMIT | EGPU_F_INPUTS_READY.
int launch_snapshot(egpu_ctx* ctx, const int32_t* d_rc, const int32_t* d_rm, int64_t R, int32_t* d_idx,
                    long long* d_delta, int32_t* d_table_out, int user_flags, cudaStream_t s,
                    int rpt_hint = 0, unsigned long long push_step_plus1 = 0, bool contig = false, int* n_tiles_out = nullptr,
                    int lag = 0) {
    if (R > kMaxRows) return EGPU_ERR_INVALID;  // the scans index 128-bit vectors with 32 bits
    const bool grid_variant = ctx->variant == EGPU_VARIANT_GRID;
    const bool lut = uses_lut(ctx);
    if (contig && grid_variant) return EGPU_ERR_STATE;  // the literal variant has no prefix-commit mode
    ScanKernel<SingleFn>& kern =
        ctx->single[contig ? (lut ? kLutContig : kSortedContig) : grid_variant ? kGrid : (lut ? kLut : kSorted)][d_bucket(ctx->D)];
    int rc = configure(ctx, kern);
    if (rc == EGPU_OK && lut) rc = refresh_lut(ctx, s);
    if (rc != EGPU_OK) return rc;
    egpu_ctx::Range mine[3];
    batch_outputs(mine, d_idx, R, d_delta, d_table_out, ctx->D);
    const int n_mine = prepare_ranges(mine, 3);
    if (n_mine < 0) return EGPU_ERR_INVALID;  // two of this launch's own outputs overlap
    const bool commit = (user_flags & EGPU_F_COMMIT) != 0;
    const int flags = kFlagFinalize | (commit ? kFlagCommit : 0) | pdl_flags(ctx, !grid_variant && !contig, user_flags, s, mine, n_mine, 0);
    const unsigned long long slot = (ctx->seq % kEpiSlots) | (push_step_plus1 << 8) | (static_cast<unsigned long long>(lag) << 56);

    int rpt = kRowsPerThread;
    if (user_flags & EGPU_F_INPUTS_READY) rpt = (lut || ctx->D <= 16) ? kRowsPerThreadPipelined : kRowsPerThread;
    else if (lut) rpt = kRowsPerThreadLoneLut;
    if (rpt_hint > 0) rpt = rpt_hint;
    if (grid_variant) rpt = 4;
    const int64_t want = single_ctas(ctx, kern, R, rpt, !contig);
    if (want == 0) return EGPU_ERR_INVALID;

    unsigned long long* tile_sums = nullptr;
    if (contig) {  // one tile per CTA: make room for their sums
        if (want > ctx->tile_cap) {
            cudaFree(ctx->d_tile_sums);
            ctx->d_tile_sums = nullptr;
            ctx->tile_cap = 0;
            EGPU_CUDA(ctx, cudaMalloc(&ctx->d_tile_sums, sizeof(unsigned long long) * 2 * kMaxD * static_cast<size_t>(want)));
            ctx->tile_cap = want;
        }
        tile_sums = ctx->d_tile_sums;
        if (n_tiles_out) *n_tiles_out = static_cast<int>(want);
    }
    rc = launch_pdl(ctx, kern, want, s, ctx->d_state, d_rc, d_rm, static_cast<long long>(R), d_idx, d_delta, d_table_out, flags,
                    slot, static_cast<const DevLut*>(ctx->d_lut), tile_sums);
    if (rc != EGPU_OK) return rc;
    ctx->seq += 1;
    note_scan(ctx, s, mine, n_mine, commit, 0);
    return EGPU_OK;
}

// One batch of whole-card rows (spec 2.8): the register scan whatever the context's variant, pipelined,
// committed and ordered with the other scans under the same rules (pdl_flags, note_scan).  d_cards
// may be nullptr.  user_flags: EGPU_F_COMMIT | EGPU_F_INPUTS_READY.
int launch_cards(egpu_ctx* ctx, const int32_t* d_rc, const int32_t* d_rm, int64_t R, int32_t* d_idx,
                 unsigned long long* d_cards, long long* d_delta, int32_t* d_table_out, int user_flags, cudaStream_t s) {
    ScanKernel<CardsFn>& kern = ctx->cards[d_bucket(ctx->D)];
    int rc = configure(ctx, kern);
    if (rc != EGPU_OK) return rc;
    egpu_ctx::Range mine[4];
    batch_outputs(mine, d_idx, R, d_delta, d_table_out, ctx->D);
    const uintptr_t pc = reinterpret_cast<uintptr_t>(d_cards);
    mine[3] = {pc, pc + (pc ? sizeof(unsigned long long) * static_cast<uintptr_t>(R) : 0)};
    const int n_mine = prepare_ranges(mine, 4);
    if (n_mine < 0) return EGPU_ERR_INVALID;  // two of this launch's own outputs overlap
    const bool commit = (user_flags & EGPU_F_COMMIT) != 0;
    const int flags = kFlagFinalize | (commit ? kFlagCommit : 0) | pdl_flags(ctx, true, user_flags, s, mine, n_mine, 0);
    const int rpt = ((user_flags & EGPU_F_INPUTS_READY) && ctx->D <= 16) ? kRowsPerThreadPipelined : kRowsPerThread;
    const int64_t want = single_ctas(ctx, kern, R, rpt, true);
    if (want == 0) return EGPU_ERR_INVALID;
    rc = launch_pdl(ctx, kern, want, s, ctx->d_state, d_rc, d_rm, static_cast<long long>(R), d_idx, d_cards, d_delta, d_table_out,
                    flags, static_cast<unsigned long long>(ctx->seq % kEpiSlots));
    if (rc != EGPU_OK) return rc;
    ctx->seq += 1;
    note_scan(ctx, s, mine, n_mine, commit, 0);
    return EGPU_OK;
}

// Multi-batch grids: enough CTAs per batch that a thread has at least this many rows.
constexpr int kMultiRowsPerThread = 8;

// Multi-batch launch: K batches, all scored against the current table, one grid (CTA (b, t) =
// tile t of batch b), one epilogue slot per batch.  Pipelines behind its predecessor under the
// same conditions as a single-batch launch; a launch group never holds more than half of the
// epi_multi ring, so the slots of everything that can be in flight are distinct.
// push_base = first exchange step + 1 when every batch also pushes its demand vector to the peers.
int launch_multi(egpu_ctx* ctx, const egpu_batch* bs, int K, int user_flags, cudaStream_t s, unsigned long long push_base) {
    if (ctx->variant == EGPU_VARIANT_GRID) return EGPU_ERR_STATE;  // the literal variant has no multi-batch form
    const bool lut = uses_lut(ctx);
    ScanKernel<MultiFn>& kern = ctx->multi[lut ? 1 : 0][d_bucket(ctx->D)];
    int rc = configure(ctx, kern);
    if (rc == EGPU_OK && lut) rc = refresh_lut(ctx, s);
    if (rc != EGPU_OK) return rc;
    MultiArgs args;
    std::memset(&args, 0, sizeof args);
    egpu_ctx::Range* mine = ctx->multi_ranges;
    int64_t max_r = 0;
    for (int k = 0; k < K; ++k) {
        const egpu_batch& b = bs[k];
        args.b[k].rc = b.d_req_core;
        args.b[k].rm = b.d_req_mem;
        args.b[k].idx = b.d_out_idx;
        args.b[k].delta = reinterpret_cast<long long*>(b.d_delta);
        // sharded: table' comes from an apply call, or (EGPU_F_APPLY) from the batch's own last CTA
        args.b[k].table_out = (push_base && !(user_flags & EGPU_F_APPLY)) ? nullptr : b.d_table_out;
        args.b[k].R = b.R;
        if (b.R > max_r) max_r = b.R;
        batch_outputs(mine + 3 * k, b.d_out_idx, b.R, b.d_delta, args.b[k].table_out, ctx->D);
    }
    const int n_mine = prepare_ranges(mine, 3 * K);
    if (n_mine < 0) return EGPU_ERR_INVALID;  // two batches of one launch share an output: their order would be undefined
    const int flags = kFlagFinalize | ((push_base && (user_flags & EGPU_F_APPLY)) ? kFlagApplyNow : 0) | pdl_flags(ctx, true, user_flags, s, mine, n_mine, K);

    // tiles per batch: enough CTAs that a thread has >= kMultiRowsPerThread rows, at most the resident
    // capacity of the GPU shared out among the K batches
    const int64_t per_cta = static_cast<int64_t>(kern.threads) * ((kMultiRowsPerThread + 3) / 4);
    int64_t tiles = ((max_r >> 2) + per_cta - 1) / per_cta;
    if (tiles < 1) tiles = 1;
    // CTAs resident at once, x waves.  One wave is best for 1 M-row batches (every extra CTA is an extra
    // epilogue); for a few huge batches two waves of half-size CTAs let the hardware's CTA scheduler even
    // out the SMs (64 Mi rows: 129 -> 124 us per batch, same-box A/B)
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * kern.ctas_per_sm * (max_r >= kTwoWaveRows ? 2 : 1);
    int64_t extra = 0;
    if (tiles * K > cap) {  // capped: hand the resident CTAs out evenly, the first `extra` batches get one more
        tiles = cap / K;
        extra = cap % K;
        if (tiles < 1) {
            tiles = 1;
            extra = 0;
        }
    }
    if (tiles > 0xffff) tiles = 0xffff;
    if (max_r / (tiles * kern.threads) + 8 >= (1ll << 19)) return EGPU_ERR_INVALID;  // lane-private sums hold 2^19 rows per lane
    const int tiles_extra = static_cast<int>(tiles | (extra << 16));
    const unsigned int slot_base = static_cast<unsigned int>(ctx->mseq % kMultiSlots);
    rc = launch_pdl(ctx, kern, tiles * K + extra, s, ctx->d_state, args, tiles_extra, flags, slot_base, push_base,
                    static_cast<const DevLut*>(ctx->d_lut));
    if (rc != EGPU_OK) return rc;
    ctx->mseq += static_cast<uint64_t>(K);
    note_scan(ctx, s, mine, n_mine, false, K);
    return EGPU_OK;
}

// Prefix-commit pipeline on device buffers (spec 2.5): CONTIG scan -> per-device cut ->
// rewrite of the deferred indices -> delta / table' of the committed rows only.
int launch_prefix_commit(egpu_ctx* ctx, const int32_t* d_rc, const int32_t* d_rm, int64_t R, int32_t* d_idx,
                         long long* d_delta, int32_t* d_table_out, int user_flags, cudaStream_t s) {
    if (!ctx->d_prefix_out) EGPU_CUDA(ctx, cudaMalloc(&ctx->d_prefix_out, sizeof(PrefixOut) + sizeof(long long) * 2 * kMaxD));
    int n_tiles = 0;
    // the scan itself must neither publish nor commit: its sums are the uncapped ones
    int rc = launch_snapshot(ctx, d_rc, d_rm, R, d_idx, nullptr, nullptr, 0, s, 0, 0, true, &n_tiles);
    if (rc != EGPU_OK) return rc;
    PrefixOut* pf = static_cast<PrefixOut*>(ctx->d_prefix_out);
    prefix_cut_kernel<<<ctx->D, 256, 0, s>>>(ctx->d_state, d_idx, d_rc, d_rm, R, n_tiles, ctx->d_tile_sums, pf);
    int64_t blocks = (R + 1023) / 1024;
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    prefix_apply_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(pf, ctx->D, R, d_idx);
    prefix_finalize_kernel<<<1, kMaxD, 0, s>>>(ctx->d_state, pf, d_delta, d_table_out, (user_flags & EGPU_F_COMMIT) ? 1 : 0);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 3;
    ctx->prev_is_scan = false;
    if (user_flags & EGPU_F_COMMIT) ctx->lut_dirty = true;
    return EGPU_OK;
}

// Rounds of committing prefix-commit until nothing is deferred (spec 2.5, "rounds").  Round 1
// runs on the caller's device arrays; the rows it defers are gathered, in order, into dense
// scratch arrays and re-submitted against the table round 1 committed, and so on.  Every round
// needs two numbers on the host (rows still deferred, the round's committed demand), so this
// is a synchronous host loop around asynchronous launches.
struct RoundInfo {
    unsigned long long deferred;
    long long delta[2 * kMaxD];
};

int run_rounds(egpu_ctx* ctx, const int32_t* d_rc, const int32_t* d_rm, int64_t R, int32_t* d_idx, int max_rounds,
               long long* total_delta /* host [2*D] */, int32_t* rounds_out, int64_t* left_out, cudaStream_t s) {
    const int D = ctx->D;
    for (int j = 0; j < 2 * D; ++j) total_delta[j] = 0;
    *rounds_out = 0;
    *left_out = 0;
    if (R == 0 || max_rounds < 1) return EGPU_OK;
    // Scratch owned by the context, grow-only, sized by R BEFORE anything is committed (a failed
    // allocation must not leave a half-committed batch): round info, tile counts, and two sets
    // of (core, mem, caller's row, index) arrays - the deferred rows of any round are at most R.
    const int64_t tiles_cap = (R + kCompactTile - 1) / kCompactTile;
    const size_t tiles_bytes = (sizeof(unsigned int) * static_cast<size_t>(tiles_cap) + 255) & ~static_cast<size_t>(255);
    const size_t per = (sizeof(int32_t) * static_cast<size_t>(R) + 255) & ~static_cast<size_t>(255);
    constexpr size_t kHead = 2048;  // RoundInfo
    const size_t need = kHead + tiles_bytes + 8 * per;
    if (need > ctx->rounds_bytes) {
        if (ctx->d_rounds) cudaFree(ctx->d_rounds);
        ctx->d_rounds = nullptr;
        ctx->rounds_bytes = 0;
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_rounds, need));
        ctx->rounds_bytes = need;
    }
    static_assert(sizeof(RoundInfo) <= kHead, "round info header");
    char* base = static_cast<char*>(ctx->d_rounds);
    RoundInfo* d_info = reinterpret_cast<RoundInfo*>(base);
    unsigned int* d_tiles = reinterpret_cast<unsigned int*>(base + kHead);
    // current round's arrays (round 1: the caller's) and the next round's
    const int32_t* cur_rc = d_rc;
    const int32_t* cur_rm = d_rm;
    const int32_t* cur_map = nullptr;
    int32_t* cur_idx = d_idx;
    int64_t n = R;
    int32_t* set[2][4];  // rc, rm, map, idx
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 4; ++b) set[a][b] = reinterpret_cast<int32_t*>(base + kHead + tiles_bytes + per * (a * 4 + b));
    int which = 0;
    RoundInfo h{};
    for (int round = 1;; ++round) {
        int rc = launch_prefix_commit(ctx, cur_rc, cur_rm, n, cur_idx, d_info->delta, nullptr, EGPU_F_COMMIT, s);
        if (rc != EGPU_OK) return rc;
        if (cur_map) {
            int64_t blocks = (n + 255) / 256;
            if (blocks > static_cast<int64_t>(ctx->sm_count) * 8) blocks = static_cast<int64_t>(ctx->sm_count) * 8;
            round_writeback_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(cur_idx, cur_map, n, d_idx);
            ctx->launches += 1;
        }
        const int64_t tiles = (n + kCompactTile - 1) / kCompactTile;
        deferred_count_kernel<<<static_cast<unsigned>(tiles), 256, 0, s>>>(cur_idx, n, d_tiles);
        deferred_scan_kernel<<<1, 1024, 0, s>>>(d_tiles, tiles, &d_info->deferred);
        ctx->launches += 2;
        EGPU_CUDA(ctx, cudaGetLastError());
        EGPU_CUDA(ctx, cudaMemcpyAsync(&h, d_info, sizeof h, cudaMemcpyDeviceToHost, s));
        EGPU_CUDA(ctx, cudaStreamSynchronize(s));
        for (int j = 0; j < 2 * D; ++j) total_delta[j] += h.delta[j];
        *rounds_out = round;
        *left_out = static_cast<int64_t>(h.deferred);
        if (h.deferred == 0 || round >= max_rounds) return EGPU_OK;
        int32_t** nxt = set[which];
        deferred_scatter_kernel<<<static_cast<unsigned>(tiles), 256, 0, s>>>(cur_idx, cur_rc, cur_rm, cur_map, n, d_tiles, nxt[0], nxt[1],
                                                                               nxt[2]);
        ctx->launches += 1;
        EGPU_CUDA(ctx, cudaGetLastError());
        cur_rc = nxt[0];
        cur_rm = nxt[1];
        cur_map = nxt[2];
        cur_idx = nxt[3];
        n = static_cast<int64_t>(h.deferred);
        which ^= 1;
    }
}

// Prefix-commit over row shards (one rank per GPU, rank-major row order).  Two exchange
// steps: `step` carries the uncapped demand of every shard (pushed by the scan itself),
// `step + 1` the committed demand after the cut (pushed by prefix_push_kernel).
int launch_prefix_commit_shard(egpu_ctx* ctx, const int32_t* d_rc, const int32_t* d_rm, int64_t R, int32_t* d_idx,
                               long long* d_delta, int32_t* d_table_out, int user_flags, uint64_t step, cudaStream_t s) {
    if (!ctx->d_prefix_out) EGPU_CUDA(ctx, cudaMalloc(&ctx->d_prefix_out, sizeof(PrefixOut) + sizeof(long long) * 2 * kMaxD));
    PrefixOut* pf = static_cast<PrefixOut*>(ctx->d_prefix_out);
    long long* base = reinterpret_cast<long long*>(pf + 1);
    int n_tiles = 0;
    // finalising scan without commit: its epilogue publishes (and pushes) the uncapped sums
    int rc = launch_snapshot(ctx, d_rc, d_rm, R, d_idx, nullptr, nullptr, 0, s, 0, step + 1, true, &n_tiles);
    if (rc != EGPU_OK) return rc;
    prefix_base_kernel<<<1, kMaxD, 0, s>>>(ctx->d_state, step + 1, base);
    prefix_cut_kernel<<<ctx->D, 256, 0, s>>>(ctx->d_state, d_idx, d_rc, d_rm, R, n_tiles, ctx->d_tile_sums, pf, base);
    int64_t blocks = (R + 1023) / 1024;
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    prefix_apply_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(pf, ctx->D, R, d_idx);
    prefix_push_kernel<<<1, kMaxD, 0, s>>>(ctx->d_state, pf, step + 2, d_delta);
    ApplyOuts outs{};
    outs.table_out[0] = d_table_out;
    apply_peers_kernel<<<1, kMaxD, 0, s>>>(ctx->d_state, step + 2, 1, outs, (user_flags & EGPU_F_COMMIT) ? 1 : 0);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 5;
    ctx->prev_is_scan = false;
    if (user_flags & EGPU_F_COMMIT) ctx->lut_dirty = true;
    return EGPU_OK;
}

// Packed-format scan: always a fully ordered launch (it serves the synchronous host path).
int launch_packed(egpu_ctx* ctx, const uint32_t* d_req, int64_t R, signed char* d_idx8, long long* d_delta,
                  int32_t* d_table_out, int user_flags, cudaStream_t s, int rows_per_thread) {
    ScanKernel<PackedFn>& kern = ctx->packed[d_bucket(ctx->D)];
    int rc = configure(ctx, kern);
    if (rc != EGPU_OK) return rc;
    const int64_t nchunk = R >> 9;  // 512 requests per warp trip
    const int64_t per_cta = static_cast<int64_t>(kern.threads / 32) * ((rows_per_thread + 15) / 16);
    int64_t want = (nchunk + per_cta - 1) / per_cta;
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * kern.ctas_per_sm;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    if (R / (want * kern.threads) + 16 >= (1ll << 19)) return EGPU_ERR_INVALID;
    const bool commit = (user_flags & EGPU_F_COMMIT) != 0;
    rc = launch_pdl(ctx, kern, want, s, ctx->d_state, d_req, static_cast<long long>(R), d_idx8, d_delta, d_table_out,
                    kFlagFinalize | (commit ? kFlagCommit : 0), static_cast<unsigned long long>(ctx->seq % kEpiSlots));
    if (rc != EGPU_OK) return rc;
    ctx->seq += 1;
    new_group(ctx);
    ctx->prev_is_scan = false;  // the int32 scans do not pipeline behind this one
    if (commit) ctx->lut_dirty = true;
    return EGPU_OK;
}

int ensure_staging(egpu_ctx* ctx, int64_t rows) {
    if (rows <= ctx->d_cap_rows) return EGPU_OK;
    int64_t cap = ctx->d_cap_rows ? ctx->d_cap_rows : 1024;
    while (cap < rows) cap *= 2;
    if (ctx->d_req_core) cudaFree(ctx->d_req_core);
    if (ctx->d_req_mem) cudaFree(ctx->d_req_mem);
    if (ctx->d_idx) cudaFree(ctx->d_idx);
    ctx->d_req_core = ctx->d_req_mem = ctx->d_idx = nullptr;
    ctx->d_cap_rows = 0;
    EGPU_CUDA(ctx, cudaMalloc(&ctx->d_req_core, sizeof(int32_t) * cap));
    EGPU_CUDA(ctx, cudaMalloc(&ctx->d_req_mem, sizeof(int32_t) * cap));
    EGPU_CUDA(ctx, cudaMalloc(&ctx->d_idx, sizeof(int32_t) * cap));
    ctx->d_cap_rows = cap;
    return EGPU_OK;
}

// host-buffer entry points: the requests into the staging arrays ...
int stage_requests(egpu_ctx* ctx, const int32_t* req_core, const int32_t* req_mem, int64_t R, cudaStream_t s) {
    const int rc = ensure_staging(ctx, R > 0 ? R : 1);
    if (rc != EGPU_OK) return rc;
    if (R > 0) {
        EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_core, req_core, sizeof(int32_t) * R, cudaMemcpyHostToDevice, s));
        EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_mem, req_mem, sizeof(int32_t) * R, cudaMemcpyHostToDevice, s));
    }
    return EGPU_OK;
}
// ... and the indices and demand sums back; waits for the stream
int unstage_results(egpu_ctx* ctx, int32_t* out_idx, int64_t R, cudaStream_t s) {
    if (R > 0) EGPU_CUDA(ctx, cudaMemcpyAsync(out_idx, ctx->d_idx, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, s));
    EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->h_delta, ctx->d_delta, sizeof(long long) * 2 * ctx->D, cudaMemcpyDeviceToHost, s));
    EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    return EGPU_OK;
}

// Grow-only arena of the replays: the events (kind, a, b) copied in, the int32 indices out
// (ev[0..3]), then `extra` bytes (*extra).  No cudaMalloc/cudaFree on the call path once grown.
int replay_stage(egpu_ctx* ctx, const int32_t* kind, const int32_t* a, const int32_t* b, int64_t E, size_t extra, cudaStream_t s,
                 int32_t** ev, char** extra_out) {
    const size_t ebytes = (sizeof(int32_t) * static_cast<size_t>(E) + 255) & ~static_cast<size_t>(255);
    const size_t need = 4 * ebytes + extra;
    if (need > ctx->arena_cap) {
        if (ctx->arena) cudaFree(ctx->arena);
        ctx->arena = nullptr;
        ctx->arena_cap = 0;
        EGPU_CUDA(ctx, cudaMalloc(&ctx->arena, need + need / 4));
        ctx->arena_cap = need + need / 4;
    }
    char* base = static_cast<char*>(ctx->arena);
    for (int j = 0; j < 4; ++j) ev[j] = reinterpret_cast<int32_t*>(base + j * ebytes);
    *extra_out = extra ? base + 4 * ebytes : nullptr;
    EGPU_CUDA(ctx, cudaMemcpyAsync(ev[0], kind, sizeof(int32_t) * E, cudaMemcpyHostToDevice, s));
    EGPU_CUDA(ctx, cudaMemcpyAsync(ev[1], a, sizeof(int32_t) * E, cudaMemcpyHostToDevice, s));
    EGPU_CUDA(ctx, cudaMemcpyAsync(ev[2], b, sizeof(int32_t) * E, cudaMemcpyHostToDevice, s));
    return EGPU_OK;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// device-visible alias of a pinned (mapped) host allocation, nullptr for anything else
void* mapped_alias(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return (a.type == cudaMemoryTypeHost) ? a.devicePointer : nullptr;
}

}  // namespace

extern "C" {

int egpu_abi_version(void) { return 1005; }  // 1.5: + whole-card requests: egpu_bestfit_cards[_dev], egpu_replay_cards (additive)

const char* egpu_strerror(int code) {
    switch (code) {
        case EGPU_OK: return "ok";
        case EGPU_ERR_INVALID: return "invalid argument";
        case EGPU_ERR_NO_DEVICE: return "no usable CUDA device (this library has no CPU fallback)";
        case EGPU_ERR_CUDA: return "CUDA runtime error";
        case EGPU_ERR_NOMEM: return "out of memory";
        case EGPU_ERR_NO_TABLE: return "capacity table not set";
        case EGPU_ERR_STATE: return "call not valid in the current state";
        case EGPU_ERR_PARSE: return "malformed device id";
        case EGPU_ERR_UNSAT: return "preferred allocation cannot be satisfied";
        default: return "unknown error";
    }
}

int egpu_ctx_create(int cuda_device, egpu_ctx** out) {
    if (!out) return EGPU_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        return EGPU_ERR_NO_DEVICE;
    }
    if (cuda_device < 0 || cuda_device >= n) return EGPU_ERR_INVALID;
    egpu_ctx* ctx = new (std::nothrow) egpu_ctx();
    if (!ctx) return EGPU_ERR_NOMEM;
    ctx->dev = cuda_device;
    fill_bucket<8>(ctx, 0);
    fill_bucket<16>(ctx, 1);
    fill_bucket<32>(ctx, 2);
    fill_bucket<64>(ctx, 3);
    int rc = [&]() -> int {
        EGPU_CUDA(ctx, cudaSetDevice(cuda_device));
        cudaDeviceProp prop;
        EGPU_CUDA(ctx, cudaGetDeviceProperties(&prop, cuda_device));
        ctx->sm_count = prop.multiProcessorCount;
        EGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_state, sizeof(DevState)));
        EGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_state, 0, sizeof(DevState), ctx->stream));
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_lut, sizeof(DevLut)));
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_xchg, sizeof(XchgBuf)));
        EGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_xchg, 0, sizeof(XchgBuf), ctx->stream));
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_delta, sizeof(long long) * 2 * kMaxD));
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_table_out, sizeof(int32_t) * 3 * kMaxD));
        EGPU_CUDA(ctx, cudaMallocHost(&ctx->h_delta, sizeof(long long) * 2 * kMaxD));
        EGPU_CUDA(ctx, cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->h_delta_dev), ctx->h_delta, 0));
        EGPU_CUDA(ctx, cudaMallocHost(&ctx->h_table, sizeof(int32_t) * 3 * kMaxD));
        EGPU_CUDA(ctx, cudaMallocHost(&ctx->h_qtable, offsetof(DevState, peer)));
        EGPU_CUDA(ctx, cudaMallocHost(&ctx->h_gate, sizeof(unsigned long long)));
        *ctx->h_gate = 0ull;
        EGPU_CUDA(ctx, cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->h_gate_dev), ctx->h_gate, 0));
        EGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return EGPU_OK;
    }();
    if (rc != EGPU_OK) {
        egpu_ctx_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return EGPU_OK;
}

void egpu_ctx_destroy(egpu_ctx* ctx) {
    if (!ctx) return;
    if (ctx->dev >= 0) cudaSetDevice(ctx->dev);
    if (ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    for (int r = 0; r < kMaxRanks; ++r)
        if (ctx->peer_open[r]) cudaIpcCloseMemHandle(ctx->peer_open[r]);
    cudaFree(ctx->d_xchg);
    cudaFree(ctx->d_tile_sums);
    cudaFree(ctx->d_rounds);
    cudaFree(ctx->d_prefix_out);
    cudaFree(ctx->arena);
    cudaFree(ctx->d_state);
    cudaFree(ctx->d_lut);
    cudaFree(ctx->d_req_core);
    cudaFree(ctx->d_req_mem);
    cudaFree(ctx->d_idx);
    cudaFree(ctx->d_cards);
    cudaFree(ctx->d_delta);
    cudaFree(ctx->d_table_out);
    if (ctx->h_delta) cudaFreeHost(ctx->h_delta);
    if (ctx->h_table) cudaFreeHost(ctx->h_table);
    if (ctx->h_gate) cudaFreeHost(ctx->h_gate);
    if (ctx->h_qtable) cudaFreeHost(ctx->h_qtable);
    cudaFree(ctx->d_qstate);
    (void)cudaGetLastError();
    delete ctx;
}

const char* egpu_last_error(egpu_ctx* ctx) { return ctx ? ctx->last_err : ""; }
int egpu_backend(egpu_ctx* ctx) { return ctx ? 1 : EGPU_ERR_INVALID; }
int64_t egpu_launch_count(egpu_ctx* ctx) {
    if (!ctx) return 0;
    std::lock_guard<std::mutex> g(ctx->mu);
    return ctx->launches;
}

int egpu_set_variant(egpu_ctx* ctx, int variant) {
    if (!ctx || variant < EGPU_VARIANT_AUTO || variant > EGPU_VARIANT_LUT) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    ctx->variant = variant;
    return EGPU_OK;
}

int egpu_table_set(egpu_ctx* ctx, const int32_t* free_core, const int32_t* free_mem, int32_t D) {
    if (!ctx || !free_core || !free_mem || D < 1 || D > EGPU_MAX_DEVICES) return EGPU_ERR_INVALID;
    for (int d = 0; d < D; ++d) {
        if (free_core[d] < 0 || free_core[d] > EGPU_CORE_MAX) return EGPU_ERR_INVALID;
        if (free_mem[d] < 0 || free_mem[d] > EGPU_MEM_MAX) return EGPU_ERR_INVALID;
    }
    std::lock_guard<std::mutex> g(ctx->mu);
    return egpu_table_set_locked(ctx, free_core, free_mem, D);
}

}  // extern "C"

// for the host-only translation units (egpu_restore.cc), which cannot see egpu_ctx
void egpu_note_error(egpu_ctx* ctx, const char* msg) {
    if (!ctx || !msg) return;
    std::lock_guard<std::mutex> g(ctx->mu);
    std::snprintf(ctx->last_err, sizeof ctx->last_err, "%s", msg);
}

// body of egpu_table_set; the caller holds ctx->mu and has validated the arguments
// (also used by egpu_table_restore_flat, egpu_devhash.cu)
int egpu_table_set_locked(egpu_ctx* ctx, const int32_t* free_core, const int32_t* free_mem, int32_t D) {
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    DevState h;
    std::memset(&h, 0, sizeof h);
    std::memcpy(h.free_core, free_core, sizeof(int32_t) * D);
    std::memcpy(h.free_mem, free_mem, sizeof(int32_t) * D);
    h.D = D;
    h.cand_xor = kGuards;
    h.cand_mask = kCandMask;
    fill_sorted(h);
    // pageable source: the copy is staged before the call returns
    // only the table part: the peer configuration (egpu_peer_attach) and the epilogue slots
    // that follow stay as they are
    EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_state, &h, offsetof(DevState, peer), cudaMemcpyHostToDevice, ctx->stream));
    EGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->D = D;
    ctx->has_table = true;
    ctx->prev_is_scan = false;
    ctx->lut_dirty = true;
    return EGPU_OK;
}

extern "C" {

int egpu_table_size(egpu_ctx* ctx) {
    if (!ctx) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    return ctx->has_table ? ctx->D : EGPU_ERR_NO_TABLE;
}

int egpu_table_get(egpu_ctx* ctx, int32_t* free_core, int32_t* free_mem, int32_t* oversub) {
    if (!ctx || !free_core || !free_mem) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    EGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    EGPU_CUDA(ctx, cudaMemcpy(ctx->h_table, ctx->d_state, sizeof(int32_t) * 3 * kMaxD, cudaMemcpyDeviceToHost));
    std::memcpy(free_core, ctx->h_table, sizeof(int32_t) * ctx->D);
    std::memcpy(free_mem, ctx->h_table + kMaxD, sizeof(int32_t) * ctx->D);
    if (oversub) std::memcpy(oversub, ctx->h_table + 2 * kMaxD, sizeof(int32_t) * ctx->D);
    return EGPU_OK;
}

int egpu_host_alloc(egpu_ctx* ctx, void** out, int64_t bytes) {
    if (!ctx || !out || bytes <= 0) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    EGPU_CUDA(ctx, cudaMallocHost(out, static_cast<size_t>(bytes)));
    return EGPU_OK;
}

void egpu_host_free(egpu_ctx* ctx, void* p) {
    if (!ctx || !p) return;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->dev);
    cudaFreeHost(p);
    (void)cudaGetLastError();
}

int egpu_host_register(egpu_ctx* ctx, void* p, int64_t bytes) {
    if (!ctx || !p || bytes <= 0) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    EGPU_CUDA(ctx, cudaHostRegister(p, static_cast<size_t>(bytes), cudaHostRegisterMapped | cudaHostRegisterPortable));
    return EGPU_OK;
}

int egpu_host_unregister(egpu_ctx* ctx, void* p) {
    if (!ctx || !p) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    EGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // nothing of ours may still be reading it
    EGPU_CUDA(ctx, cudaHostUnregister(p));
    return EGPU_OK;
}

int egpu_bestfit_batch_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem, int64_t R,
                           int32_t* d_out_idx, int64_t* d_delta, int32_t* d_table_out, int flags,
                           void* stream) {
    if (!ctx || R < 0) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_core || !d_req_mem || !d_out_idx)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_core) || !aligned16(d_req_mem) || !aligned16(d_out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    if (flags & EGPU_F_PREFIX_COMMIT)
        return launch_prefix_commit(ctx, d_req_core, d_req_mem, R, d_out_idx, reinterpret_cast<long long*>(d_delta), d_table_out,
                                    flags, s);
    return launch_snapshot(ctx, d_req_core, d_req_mem, R, d_out_idx, reinterpret_cast<long long*>(d_delta),
                           d_table_out, flags, s);
}

static int check_batches(const egpu_batch* batches, int32_t K) {
    if (!batches || K < 1 || K > EGPU_MAX_BATCHES) return EGPU_ERR_INVALID;
    for (int k = 0; k < K; ++k) {
        const egpu_batch& b = batches[k];
        if (b.R < 0 || b.R > kMaxRows) return EGPU_ERR_INVALID;
        if (b.R > 0 && (!b.d_req_core || !b.d_req_mem || !b.d_out_idx)) return EGPU_ERR_INVALID;
        if (!aligned16(b.d_req_core) || !aligned16(b.d_req_mem) || !aligned16(b.d_out_idx)) return EGPU_ERR_INVALID;
    }
    return EGPU_OK;
}

int egpu_bestfit_batches_dev(egpu_ctx* ctx, const egpu_batch* batches, int32_t K, int flags, void* stream) {
    if (!ctx || (flags & ~EGPU_F_INPUTS_READY)) return EGPU_ERR_INVALID;
    const int rc = check_batches(batches, K);
    if (rc != EGPU_OK) return rc;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_multi(ctx, batches, K, flags, s, 0);
}

int egpu_bestfit_batches_shard_dev(egpu_ctx* ctx, const egpu_batch* batches, int32_t K, int flags, uint64_t first_step,
                                   void* stream) {
    if (!ctx || (flags & ~(EGPU_F_INPUTS_READY | EGPU_F_APPLY)) || first_step >= (1ull << 47)) return EGPU_ERR_INVALID;
    const int rc = check_batches(batches, K);
    if (rc != EGPU_OK) return rc;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (!ctx->attached) return EGPU_ERR_STATE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_multi(ctx, batches, K, flags, s, first_step + 1);
}

int egpu_peer_gate_dev(egpu_ctx* ctx, void* stream) {
    if (!ctx) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    gate_kernel<<<1, 32, 0, s>>>(ctx->d_state, ctx->h_gate_dev);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    ctx->prev_is_scan = false;
    return EGPU_OK;
}

int64_t egpu_peer_gate_timeouts(egpu_ctx* ctx) {
    if (!ctx) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (cudaSetDevice(ctx->dev) != cudaSuccess) return EGPU_ERR_CUDA;
    unsigned long long v = 0;
    if (cudaMemcpy(&v, reinterpret_cast<char*>(ctx->d_state) + offsetof(DevState, gate_timeouts), sizeof v,
                   cudaMemcpyDeviceToHost) != cudaSuccess) {
        (void)cudaGetLastError();
        return EGPU_ERR_CUDA;
    }
    return static_cast<int64_t>(v);
}

int egpu_peer_gate_open(egpu_ctx* ctx) {
    if (!ctx) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    __atomic_fetch_add(ctx->h_gate, 1ull, __ATOMIC_RELEASE);
    return EGPU_OK;
}

int egpu_bestfit_query(egpu_ctx* ctx, const int32_t* free_core, const int32_t* free_mem, int32_t D, const int32_t* req_core,
                       const int32_t* req_mem, int64_t R, int32_t* out_idx) {
    if (!ctx || !free_core || !free_mem || D < 1 || D > EGPU_MAX_DEVICES || R < 0 || R > kMaxRows) return EGPU_ERR_INVALID;
    if (R > 0 && (!req_core || !req_mem || !out_idx)) return EGPU_ERR_INVALID;
    for (int d = 0; d < D; ++d) {
        if (free_core[d] < 0 || free_core[d] > EGPU_CORE_MAX) return EGPU_ERR_INVALID;
        if (free_mem[d] < 0 || free_mem[d] > EGPU_MEM_MAX) return EGPU_ERR_INVALID;
    }
    if (R == 0) return EGPU_OK;
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = ctx->stream;
    if (!ctx->d_qstate) {
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_qstate, sizeof(DevState)));
        EGPU_CUDA(ctx, cudaMemsetAsync(ctx->d_qstate, 0, sizeof(DevState), s));
    }
    // the scratch table: same layout and sorted view as the context's own, in its own DevState
    DevState* h = reinterpret_cast<DevState*>(ctx->h_qtable);
    std::memset(h, 0, offsetof(DevState, peer));
    std::memcpy(h->free_core, free_core, sizeof(int32_t) * D);
    std::memcpy(h->free_mem, free_mem, sizeof(int32_t) * D);
    h->D = D;
    h->cand_xor = kGuards;
    h->cand_mask = kCandMask;
    fill_sorted(*h);
    EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_qstate, h, offsetof(DevState, peer), cudaMemcpyHostToDevice, s));
    int rc = ensure_staging(ctx, R);
    if (rc != EGPU_OK) return rc;
    EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_core, req_core, sizeof(int32_t) * R, cudaMemcpyHostToDevice, s));
    EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_mem, req_mem, sizeof(int32_t) * R, cudaMemcpyHostToDevice, s));
    // the register scan whatever the context's variant: one table, used once - lookup tables would not pay
    ScanKernel<SingleFn>& kern = ctx->single[kSorted][d_bucket(D)];
    rc = configure(ctx, kern);
    if (rc != EGPU_OK) return rc;
    const int64_t per_cta = static_cast<int64_t>(kern.threads) * 2;
    int64_t want = ((R >> 2) + per_cta - 1) / per_cta;
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * kern.ctas_per_sm;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    if (R / (want * kern.threads) + 8 >= (1ll << 19)) return EGPU_ERR_INVALID;
    // fully ordered launch (no PDL flags), epilogue slot 0 of the scratch state, nothing published
    kern.fn<<<static_cast<unsigned>(want), kern.threads, kern.smem, s>>>(ctx->d_qstate, ctx->d_req_core, ctx->d_req_mem,
                                                                         static_cast<long long>(R), ctx->d_idx, nullptr, nullptr,
                                                                         kFlagFinalize, 0ull, nullptr, nullptr);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    ctx->prev_is_scan = false;
    EGPU_CUDA(ctx, cudaMemcpyAsync(out_idx, ctx->d_idx, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, s));
    EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    return EGPU_OK;
}

int egpu_bestfit_batch(egpu_ctx* ctx, const int32_t* req_core, const int32_t* req_mem, int64_t R,
                       int32_t* out_idx, int64_t* out_delta_core, int64_t* out_delta_mem, int commit) {
    if (!ctx || R < 0) return EGPU_ERR_INVALID;
    if (R > 0 && (!req_core || !req_mem || !out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = ctx->stream;
    const int D = ctx->D;
    int rc;
    // Zero-copy: when all three caller arrays are pinned (egpu_host_alloc or
    // cudaHostRegister) and 16-byte aligned, the scan reads the requests and writes
    // the indices straight across PCIe — one launch, no staging in HBM, reads and
    // writes overlap on the full-duplex link.  Demand sums land in pinned memory too.
    const int32_t* zc = R > 0 ? static_cast<const int32_t*>(mapped_alias(req_core)) : nullptr;
    const int32_t* zm = R > 0 ? static_cast<const int32_t*>(mapped_alias(req_mem)) : nullptr;
    int32_t* zi = R > 0 ? static_cast<int32_t*>(mapped_alias(out_idx)) : nullptr;
    const bool prefix = (commit & EGPU_F_PREFIX_COMMIT) != 0;  // `commit` carries EGPU_F_COMMIT | EGPU_F_PREFIX_COMMIT
    if (!prefix && zc && zm && zi && aligned16(zc) && aligned16(zm) && aligned16(zi)) {
        // 64 rows per thread: few CTAs, many trips, so reads of later rows and writes of
        // earlier ones are on the link at the same time (PCIe is full duplex)
        rc = launch_snapshot(ctx, zc, zm, R, zi, ctx->h_delta_dev, nullptr, (commit & EGPU_F_COMMIT) ? EGPU_F_COMMIT : 0, s, 64);
        if (rc != EGPU_OK) return rc;
        EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    } else {
        rc = stage_requests(ctx, req_core, req_mem, R, s);
        if (rc != EGPU_OK) return rc;
        rc = prefix ? launch_prefix_commit(ctx, ctx->d_req_core, ctx->d_req_mem, R, ctx->d_idx, ctx->d_delta, nullptr,
                                           (commit & EGPU_F_COMMIT) ? EGPU_F_COMMIT : 0, s)
                    : launch_snapshot(ctx, ctx->d_req_core, ctx->d_req_mem, R, ctx->d_idx, ctx->d_delta, nullptr,
                                      (commit & EGPU_F_COMMIT) ? EGPU_F_COMMIT : 0, s);
        if (rc == EGPU_OK) rc = unstage_results(ctx, out_idx, R, s);
        if (rc != EGPU_OK) return rc;
    }
    if (out_delta_core) std::memcpy(out_delta_core, ctx->h_delta, sizeof(int64_t) * D);
    if (out_delta_mem) std::memcpy(out_delta_mem, ctx->h_delta + D, sizeof(int64_t) * D);
    return EGPU_OK;
}

int egpu_bestfit_batch_rounds(egpu_ctx* ctx, const int32_t* req_core, const int32_t* req_mem, int64_t R, int32_t* out_idx,
                              int64_t* out_delta_core, int64_t* out_delta_mem, int32_t max_rounds, int32_t* out_rounds,
                              int64_t* out_deferred) {
    if (!ctx || R < 0 || R >= (1ll << 31) || max_rounds < 1) return EGPU_ERR_INVALID;
    if (R > 0 && (!req_core || !req_mem || !out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = ctx->stream;
    int rc = ensure_staging(ctx, R > 0 ? R : 1);
    if (rc != EGPU_OK) return rc;
    if (R > 0) {
        EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_core, req_core, sizeof(int32_t) * R, cudaMemcpyHostToDevice, s));
        EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_mem, req_mem, sizeof(int32_t) * R, cudaMemcpyHostToDevice, s));
    }
    long long total[2 * kMaxD];
    int32_t rounds = 0;
    int64_t left = 0;
    rc = run_rounds(ctx, ctx->d_req_core, ctx->d_req_mem, R, ctx->d_idx, max_rounds, total, &rounds, &left, s);
    if (rc != EGPU_OK) return rc;
    if (R > 0) EGPU_CUDA(ctx, cudaMemcpyAsync(out_idx, ctx->d_idx, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, s));
    EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    const int D = ctx->D;
    if (out_delta_core) std::memcpy(out_delta_core, total, sizeof(int64_t) * D);
    if (out_delta_mem) std::memcpy(out_delta_mem, total + D, sizeof(int64_t) * D);
    if (out_rounds) *out_rounds = rounds;
    if (out_deferred) *out_deferred = left;
    return EGPU_OK;
}

int egpu_bestfit_batch_rounds_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem, int64_t R,
                                  int32_t* d_out_idx, int64_t* out_delta /* host [2*D] */, int32_t max_rounds,
                                  int32_t* out_rounds, int64_t* out_deferred, void* stream) {
    if (!ctx || R < 0 || R >= (1ll << 31) || max_rounds < 1) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_core || !d_req_mem || !d_out_idx)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_core) || !aligned16(d_req_mem) || !aligned16(d_out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    long long total[2 * kMaxD];
    int32_t rounds = 0;
    int64_t left = 0;
    const int rc = run_rounds(ctx, d_req_core, d_req_mem, R, d_out_idx, max_rounds, total, &rounds, &left, s);
    if (rc != EGPU_OK) return rc;
    EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    if (out_delta) std::memcpy(out_delta, total, sizeof(int64_t) * 2 * ctx->D);
    if (out_rounds) *out_rounds = rounds;
    if (out_deferred) *out_deferred = left;
    return EGPU_OK;
}

int egpu_peer_export(egpu_ctx* ctx, void* handle_out) {
    if (!ctx || !handle_out) return EGPU_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == EGPU_IPC_HANDLE_BYTES, "IPC handle size");
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaIpcMemHandle_t h;
    EGPU_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->d_xchg));
    std::memcpy(handle_out, &h, sizeof h);
    return EGPU_OK;
}

int egpu_peer_attach(egpu_ctx* ctx, int rank, int world, const void* handles) {
    if (!ctx || !handles || world < 1 || world > kMaxRanks || rank < 0 || rank >= world) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (ctx->attached) return EGPU_ERR_STATE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    PeerCfg cfg;
    std::memset(&cfg, 0, sizeof cfg);
    cfg.world = world;
    cfg.rank = rank;
    for (int r = 0; r < world; ++r) {
        if (r == rank) {
            cfg.buf[r] = ctx->d_xchg;
            continue;
        }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, static_cast<const char*>(handles) + static_cast<size_t>(r) * sizeof h, sizeof h);
        void* p = nullptr;
        EGPU_CUDA(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ctx->peer_open[r] = p;
        cfg.buf[r] = static_cast<XchgBuf*>(p);
    }
    EGPU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    EGPU_CUDA(ctx, cudaMemcpy(reinterpret_cast<char*>(ctx->d_state) + offsetof(DevState, peer), &cfg, sizeof cfg,
                              cudaMemcpyHostToDevice));
    ctx->world = world;
    ctx->rank = rank;
    ctx->attached = true;
    return EGPU_OK;
}

int egpu_peer_detach(egpu_ctx* ctx) {
    if (!ctx) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->attached) return EGPU_OK;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    EGPU_CUDA(ctx, cudaDeviceSynchronize());
    for (int r = 0; r < kMaxRanks; ++r) {
        if (ctx->peer_open[r]) cudaIpcCloseMemHandle(ctx->peer_open[r]);
        ctx->peer_open[r] = nullptr;
    }
    ctx->attached = false;
    ctx->world = 1;
    ctx->rank = 0;
    return EGPU_OK;
}

int egpu_bestfit_batch_shard_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem, int64_t R,
                                 int32_t* d_out_idx, int64_t* d_delta, int flags, uint64_t step, void* stream) {
    // the commit happens in apply_peers; prefix-commit over shards has its own entry point;
    // step + 1 travels in 48 bits of the launch word
    if (!ctx || R < 0 || (flags & ~EGPU_F_INPUTS_READY) || step >= (1ull << 47)) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_core || !d_req_mem || !d_out_idx)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_core) || !aligned16(d_req_mem) || !aligned16(d_out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (!ctx->attached) return EGPU_ERR_STATE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_snapshot(ctx, d_req_core, d_req_mem, R, d_out_idx, reinterpret_cast<long long*>(d_delta), nullptr,
                           flags, s, 0, step + 1);
}

int egpu_bestfit_batch_shard_prefix_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem, int64_t R,
                                        int32_t* d_out_idx, int64_t* d_delta, int32_t* d_table_out, int flags,
                                        uint64_t step, void* stream) {
    if (!ctx || R < 0 || step >= (1ull << 47) || (flags & ~(EGPU_F_COMMIT | EGPU_F_PREFIX_COMMIT))) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_core || !d_req_mem || !d_out_idx)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_core) || !aligned16(d_req_mem) || !aligned16(d_out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (!ctx->attached) return EGPU_ERR_STATE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_prefix_commit_shard(ctx, d_req_core, d_req_mem, R, d_out_idx, reinterpret_cast<long long*>(d_delta),
                                      d_table_out, flags, step, s);
}

int egpu_bestfit_batch_shard_lag_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem, int64_t R,
                                     int32_t* d_out_idx, int64_t* d_delta, int flags, uint64_t step, int lag,
                                     int32_t* d_table_out_lagged, void* stream) {
    if (!ctx || R < 0 || (flags & EGPU_F_COMMIT) || lag < 1 || lag > 16 || step >= (1ull << 47)) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_core || !d_req_mem || !d_out_idx)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_core) || !aligned16(d_req_mem) || !aligned16(d_out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (!ctx->attached) return EGPU_ERR_STATE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_snapshot(ctx, d_req_core, d_req_mem, R, d_out_idx, reinterpret_cast<long long*>(d_delta), d_table_out_lagged,
                           flags, s, 0, step + 1, false, nullptr, lag);
}

int egpu_table_apply_peers_multi_dev(egpu_ctx* ctx, uint64_t first_step, int nsteps, int32_t* const* d_table_outs,
                                     int commit, void* stream) {
    if (!ctx || nsteps < 1 || nsteps > kApplyMax) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (!ctx->attached) return EGPU_ERR_STATE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    if (commit) {
        ctx->lut_dirty = true;
        ctx->prev_is_scan = false;  // the next scan must see the new table
    }
    ApplyOuts outs;
    for (int k = 0; k < kApplyMax; ++k) outs.table_out[k] = (d_table_outs && k < nsteps) ? d_table_outs[k] : nullptr;
    apply_peers_kernel<<<commit ? 1 : nsteps, kMaxD, 0, s>>>(ctx->d_state, first_step + 1, nsteps, outs, commit);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    return EGPU_OK;
}

int egpu_table_apply_peers_dev(egpu_ctx* ctx, uint64_t step, int32_t* d_table_out, int commit, void* stream) {
    int32_t* outs[1] = {d_table_out};
    return egpu_table_apply_peers_multi_dev(ctx, step, 1, outs, commit, stream);
}

int64_t egpu_peer_last_timeout(egpu_ctx* ctx) {
    if (!ctx) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (cudaSetDevice(ctx->dev) != cudaSuccess) return EGPU_ERR_CUDA;
    unsigned long long v = 0;
    if (cudaMemcpy(&v, reinterpret_cast<char*>(ctx->d_state) + offsetof(DevState, peer_timeout), sizeof v,
                   cudaMemcpyDeviceToHost) != cudaSuccess) {
        (void)cudaGetLastError();
        return EGPU_ERR_CUDA;
    }
    return static_cast<int64_t>(v);
}

int egpu_bestfit_batch_packed_dev(egpu_ctx* ctx, const uint32_t* d_req_packed, int64_t R, int8_t* d_out_idx8,
                                  int64_t* d_delta, int32_t* d_table_out, int flags, void* stream) {
    // the epilogue's demand sums share their word with an arrival count: they hold EGPU_MAX_ROWS rows at most
    if (!ctx || R < 0 || R > kMaxRows) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_packed || !d_out_idx8)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_packed) || !aligned16(d_out_idx8)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_packed(ctx, d_req_packed, R, reinterpret_cast<signed char*>(d_out_idx8), reinterpret_cast<long long*>(d_delta),
                         d_table_out, flags, s, 16);
}

int egpu_bestfit_batch_packed(egpu_ctx* ctx, const uint32_t* req_packed, int64_t R, int8_t* out_idx8,
                              int64_t* out_delta_core, int64_t* out_delta_mem, int commit) {
    if (!ctx || R < 0 || R > kMaxRows) return EGPU_ERR_INVALID;  // as egpu_bestfit_batch_packed_dev
    if (R > 0 && (!req_packed || !out_idx8)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = ctx->stream;
    const int D = ctx->D;
    int rc;
    const uint32_t* zr = R > 0 ? static_cast<const uint32_t*>(mapped_alias(req_packed)) : nullptr;
    signed char* zi = R > 0 ? static_cast<signed char*>(mapped_alias(out_idx8)) : nullptr;
    if (zr && zi && aligned16(zr) && aligned16(zi)) {  // zero-copy across PCIe, see egpu_bestfit_batch
        rc = launch_packed(ctx, zr, R, zi, ctx->h_delta_dev, nullptr, commit ? EGPU_F_COMMIT : 0, s, 128);
        if (rc != EGPU_OK) return rc;
        EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    } else {
        rc = ensure_staging(ctx, R > 0 ? R : 1);  // d_req_core holds the packed words, d_idx the bytes
        if (rc != EGPU_OK) return rc;
        if (R > 0) EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->d_req_core, req_packed, sizeof(uint32_t) * R, cudaMemcpyHostToDevice, s));
        rc = launch_packed(ctx, reinterpret_cast<const uint32_t*>(ctx->d_req_core), R, reinterpret_cast<signed char*>(ctx->d_idx),
                           ctx->d_delta, nullptr, commit ? EGPU_F_COMMIT : 0, s, 16);
        if (rc != EGPU_OK) return rc;
        if (R > 0) EGPU_CUDA(ctx, cudaMemcpyAsync(out_idx8, ctx->d_idx, static_cast<size_t>(R), cudaMemcpyDeviceToHost, s));
        EGPU_CUDA(ctx, cudaMemcpyAsync(ctx->h_delta, ctx->d_delta, sizeof(long long) * 2 * D, cudaMemcpyDeviceToHost, s));
        EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    }
    if (out_delta_core) std::memcpy(out_delta_core, ctx->h_delta, sizeof(int64_t) * D);
    if (out_delta_mem) std::memcpy(out_delta_mem, ctx->h_delta + D, sizeof(int64_t) * D);
    return EGPU_OK;
}

int egpu_table_apply_deltas_dev(egpu_ctx* ctx, const int64_t* d_deltas, int G, int32_t* d_table_out,
                                int commit, void* stream) {
    if (!ctx || !d_deltas || G < 1) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    ctx->prev_is_scan = false;
    if (commit) ctx->lut_dirty = true;
    apply_deltas_kernel<<<1, kMaxD, 0, s>>>(ctx->d_state, reinterpret_cast<const long long*>(d_deltas), G,
                                            d_table_out, commit);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    return EGPU_OK;
}

int egpu_synth_requests_dev(egpu_ctx* ctx, int dist, uint64_t seed, int64_t first_row, int64_t R,
                            int32_t* d_req_core, int32_t* d_req_mem, void* stream) {
    if (!ctx || R < 0 || first_row < 0 || (dist != 2 && dist != 3 && dist != 4)) return EGPU_ERR_INVALID;
    if (R == 0) return EGPU_OK;
    if (!d_req_core || !d_req_mem) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    int64_t blocks = (R + 255) / 256;
    const int64_t cap = static_cast<int64_t>(ctx->sm_count) * 8;
    if (blocks > cap) blocks = cap;
    ctx->prev_is_scan = false;
    synth_requests_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(dist, seed, first_row, R, d_req_core, d_req_mem);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    return EGPU_OK;
}

int egpu_replay(egpu_ctx* ctx, const int32_t* kind, const int32_t* a, const int32_t* b, int64_t E,
                int32_t* out_idx) {
    if (!ctx || E < 0 || E > 0x7fffffffll) return EGPU_ERR_INVALID;
    if (E > 0 && (!kind || !a || !b || !out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (E == 0) return EGPU_OK;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    // staging comes from the context's grow-only arena (three inputs, one output, the `live`
    // map when it does not fit in shared memory): no cudaMalloc/cudaFree on the call path
    cudaStream_t s = ctx->stream;
    const size_t lbytes = E > kReplaySmemEvents ? ((static_cast<size_t>(E) + 255) & ~static_cast<size_t>(255)) : 0;
    int32_t* ev[4];
    char* extra = nullptr;
    const int rc = replay_stage(ctx, kind, a, b, E, lbytes, s, ev, &extra);
    if (rc != EGPU_OK) return rc;
    int32_t *d_kind = ev[0], *d_a = ev[1], *d_b = ev[2], *d_out = ev[3];
    signed char* d_live = reinterpret_cast<signed char*>(extra);
    size_t smem = 0;
    if (E <= kReplaySmemEvents) {
        smem = static_cast<size_t>((E + 15) & ~15ll);
        if (!ctx->replay_configured) {
            EGPU_CUDA(ctx, cudaFuncSetAttribute(replay_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kReplaySmemEvents));
            ctx->replay_configured = true;
        }
    }
    ctx->prev_is_scan = false;
    ctx->lut_dirty = true;
    if (ctx->D <= 32 && E <= kReplaySmemEvents) {
        // two warps: decode off the chain, lane = device on it
        if (!ctx->replay2_configured) {
            EGPU_CUDA(ctx, cudaFuncSetAttribute(replay2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kReplaySmemEvents));
            ctx->replay2_configured = true;
        }
        replay2_kernel<<<1, 64, smem, s>>>(ctx->d_state, d_kind, d_a, d_b, E, d_out);
    } else if (ctx->D <= 8)  // only past kReplaySmemEvents events: `live` in HBM
        replay8_kernel<<<1, 32, smem, s>>>(ctx->d_state, d_kind, d_a, d_b, E, d_out, d_live);
    else
        replay_kernel<<<1, 32, smem, s>>>(ctx->d_state, d_kind, d_a, d_b, E, d_out, d_live);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    EGPU_CUDA(ctx, cudaMemcpyAsync(out_idx, d_out, sizeof(int32_t) * E, cudaMemcpyDeviceToHost, s));
    EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    return EGPU_OK;
}

int egpu_bestfit_cards_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem, int64_t R, int32_t* d_out_idx,
                           uint64_t* d_out_cards, int64_t* d_delta, int32_t* d_table_out, int flags, void* stream) {
    if (!ctx || R < 0 || R > kMaxRows || (flags & ~(EGPU_F_COMMIT | EGPU_F_INPUTS_READY))) return EGPU_ERR_INVALID;
    if (R > 0 && (!d_req_core || !d_req_mem || !d_out_idx)) return EGPU_ERR_INVALID;
    if (!aligned16(d_req_core) || !aligned16(d_req_mem) || !aligned16(d_out_idx) || !aligned16(d_out_cards) ||
        !aligned16(d_delta) || !aligned16(d_table_out))
        return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return launch_cards(ctx, d_req_core, d_req_mem, R, d_out_idx, reinterpret_cast<unsigned long long*>(d_out_cards),
                        reinterpret_cast<long long*>(d_delta), d_table_out, flags, s);
}

int egpu_bestfit_cards(egpu_ctx* ctx, const int32_t* req_core, const int32_t* req_mem, int64_t R, int32_t* out_idx,
                       uint64_t* out_cards, int64_t* out_delta_core, int64_t* out_delta_mem, int commit) {
    if (!ctx || R < 0 || R > kMaxRows || (commit & ~EGPU_F_COMMIT)) return EGPU_ERR_INVALID;
    if (R > 0 && (!req_core || !req_mem || !out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = ctx->stream;
    int rc = stage_requests(ctx, req_core, req_mem, R, s);
    if (rc != EGPU_OK) return rc;
    if (out_cards && R > ctx->d_cards_cap) {
        cudaFree(ctx->d_cards);
        ctx->d_cards = nullptr;
        ctx->d_cards_cap = 0;
        EGPU_CUDA(ctx, cudaMalloc(&ctx->d_cards, sizeof(unsigned long long) * ctx->d_cap_rows));
        ctx->d_cards_cap = ctx->d_cap_rows;
    }
    unsigned long long* d_cards = out_cards ? ctx->d_cards : nullptr;
    rc = launch_cards(ctx, ctx->d_req_core, ctx->d_req_mem, R, ctx->d_idx, d_cards, ctx->d_delta, nullptr, commit, s);
    if (rc != EGPU_OK) return rc;
    if (d_cards && R > 0)
        EGPU_CUDA(ctx, cudaMemcpyAsync(out_cards, d_cards, sizeof(unsigned long long) * R, cudaMemcpyDeviceToHost, s));
    rc = unstage_results(ctx, out_idx, R, s);
    if (rc != EGPU_OK) return rc;
    if (out_delta_core) std::memcpy(out_delta_core, ctx->h_delta, sizeof(int64_t) * ctx->D);
    if (out_delta_mem) std::memcpy(out_delta_mem, ctx->h_delta + ctx->D, sizeof(int64_t) * ctx->D);
    return EGPU_OK;
}

int egpu_replay_cards(egpu_ctx* ctx, const int32_t* kind, const int32_t* a, const int32_t* b, int64_t E, int32_t* out_idx,
                      uint64_t* out_cards) {
    if (!ctx || E < 0 || E > 0x7fffffffll) return EGPU_ERR_INVALID;
    if (E > 0 && (!kind || !a || !b || !out_idx)) return EGPU_ERR_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->has_table) return EGPU_ERR_NO_TABLE;
    if (E == 0) return EGPU_OK;
    EGPU_CUDA(ctx, cudaSetDevice(ctx->dev));
    cudaStream_t s = ctx->stream;
    // after the four event arrays: the card masks out, then every ALLOC's cards and first card
    const size_t mbytes = (sizeof(unsigned long long) * static_cast<size_t>(E) + 255) & ~static_cast<size_t>(255);
    int32_t* ev[4];
    char* extra = nullptr;
    const int rc = replay_stage(ctx, kind, a, b, E, 2 * mbytes + static_cast<size_t>(E), s, ev, &extra);
    if (rc != EGPU_OK) return rc;
    unsigned long long* d_cards = reinterpret_cast<unsigned long long*>(extra);
    unsigned long long* d_live = reinterpret_cast<unsigned long long*>(extra + mbytes);
    signed char* d_live_idx = reinterpret_cast<signed char*>(extra + 2 * mbytes);
    ctx->prev_is_scan = false;
    ctx->lut_dirty = true;
    replay_cards_kernel<<<1, 32, 0, s>>>(ctx->d_state, ev[0], ev[1], ev[2], E, ev[3], out_cards ? d_cards : nullptr, d_live,
                                         d_live_idx);
    EGPU_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    EGPU_CUDA(ctx, cudaMemcpyAsync(out_idx, ev[3], sizeof(int32_t) * E, cudaMemcpyDeviceToHost, s));
    if (out_cards) EGPU_CUDA(ctx, cudaMemcpyAsync(out_cards, d_cards, sizeof(unsigned long long) * E, cudaMemcpyDeviceToHost, s));
    EGPU_CUDA(ctx, cudaStreamSynchronize(s));
    return EGPU_OK;
}

}  // extern "C"
