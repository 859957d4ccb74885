// egpu_scan.cuh — snapshot-mode kernels of the best-fit path (sm_100a): the register scan
// (bestfit_sorted_kernel and its multi-batch form), its packed-format twin, the literal grid
// scan, the lookup-table scan for large D (single- and multi-batch) with its table builder, the
// shared epilogue (demand sums with the arrival count inside them, publication by each word's finisher, fused peer push / apply),
// the exchange-word helpers, the apply kernels, the start gate, and the prefix-commit and
// rounds kernels.  Included by egpu_alloc.cu only; see DESIGN.md §4, §5.
#pragma once
#include <type_traits>
#include "egpu_kernels.cuh"

namespace egpu {

// =============================================================================
// Snapshot scan
// =============================================================================
//
// Why "sorted" is the fast formulation.  For a fixed table the best-fit device
// of request (c, m) minimises (fc-c, fm-m, d) over feasible d, which is the same
// as minimising (fc, fm, d): the request cancels out of the comparison.  So the
// answer is the FIRST feasible device in the table sorted by (fc, fm, d).  Each
// CTA sorts the <= 64 table rows once (rank sort in shared memory), every thread
// keeps the packed sorted rows in registers, and per (request, device) pair the
// work is: one subtract (both feasibility tests at once, see kGuards), one LOP3
// producing "sorted position, or a value >= 2^18 if infeasible", and half a
// 3-input unsigned min (VIMNMX3).  The chosen position maps back to the device
// index through a shared-memory tile.

constexpr int kDevTile = kMaxD + 8;  // positions 0..63, and "none" = 32 (DT <= 32) or 64
template <int DT, int THREADS>
struct SnapSmem {
    int32_t sFc[kMaxD];                           // table tile (grid variant; re-sort scratch)
    int32_t sFm[kMaxD];
    int32_t sPosDev[kMaxD];
    unsigned long long sWarpAcc[THREADS / 32][2 * DT];
    int sLast;
    int32_t sDevTile[THREADS / 32][kDevTile];         // warp-private: sorted position -> device, -1 from DT on
    unsigned long long hist[THREADS / 32][DT + 1][32];  // lane-private demand sums; row 0 = "no device"
};

// Re-derive the sorted view of the table (DevState::sorted_k / sorted_dev /
// dev_packed).  Called by every thread of ONE CTA after thread d < D has put the
// new row d into sFc[d] / sFm[d].  Rank sort: position = rows ordering before.
__device__ __forceinline__ void resort_table_cta(DevState* st, int D, int32_t* sFc, int32_t* sFm,
                                                 int32_t* sPosDev, int tid) {
    const int nt = blockDim.x;
    __syncthreads();
    for (int d = tid; d < kMaxD; d += nt) sPosDev[d] = -1;
    __syncthreads();
    for (int d = tid; d < kMaxD; d += nt) {
        if (d < D) {
            const int32_t fc = sFc[d], fm = sFm[d];
            const uint32_t mine = (static_cast<uint32_t>(fc) << 24) | (static_cast<uint32_t>(fm) << 6) | d;
            int pos = 0;
            for (int k = 0; k < D; ++k) {
                const uint32_t other = (static_cast<uint32_t>(sFc[k]) << 24) | (static_cast<uint32_t>(sFm[k]) << 6) | k;
                pos += other < mine;
            }
            st->sorted_k[pos] = pack_table_word(fc, fm) | (static_cast<uint32_t>(pos) & 31u);
            st->sorted_dev[pos] = d;
            sPosDev[pos] = d;
        } else {  // positions >= D are never produced by a rank
            st->sorted_k[d] = kPadWord;
            st->sorted_dev[d] = -1;
        }
    }
    __syncthreads();
    if (tid == 0) {
        unsigned long long packed = 0;
        for (int j = 0; j < 8; ++j)
            packed |= static_cast<unsigned long long>(static_cast<uint32_t>(sPosDev[j]) & 0xffu) << (8 * j);
        st->dev_packed = packed;
    }
}

// First feasible sorted position; kNoCand (DT <= 32) or DT (DT = 64) when there is none.
// Per (request, row) pair: one subtract (IMAD.IADD or IADD3, ptxas balances the FMA and
// ALU pipes), one 3-input LOP3 ((t ^ G) & M, both masks in registers), half a VIMNMX3.
template <int N>
__device__ __forceinline__ uint32_t first_feasible32(const uint32_t* K, uint32_t q, uint32_t gx, uint32_t gm) {
    uint32_t best = kNoCand;
#pragma unroll
    for (int j = 0; j < N; j += 2) {
        const uint32_t c0 = ((K[j] - q) ^ gx) & gm;
        const uint32_t c1 = ((K[j + 1] - q) ^ gx) & gm;
        best = __vimin3_u32(best, c0, c1);
    }
    return best;  // 0..N-1, or >= 32
}
template <int DT>
__device__ __forceinline__ uint32_t first_feasible(const uint32_t (&K)[DT], uint32_t q, uint32_t gx, uint32_t gm) {
    if constexpr (DT <= 32) {
        return first_feasible32<DT>(K, q, gx, gm);  // 0..DT-1, or kNoCand (= 32): the tile maps both ranges
    } else {  // positions are stored mod 32: two halves
        const uint32_t lo = first_feasible32<32>(K, q, gx, gm);
        const uint32_t hi = first_feasible32<DT - 32>(K + 32, q, gx, gm);
        return lo < 32u ? lo : (hi < 32u ? 32u + hi : static_cast<uint32_t>(DT));
    }
}

template <int DT, int THREADS>
__device__ __forceinline__ void hist_zero(SnapSmem<DT, THREADS>& s, int warp, int lane) {
    // lane-private: each lane clears exactly the words it will use -> no barrier
#pragma unroll
    for (int d = 0; d <= DT; ++d) s.hist[warp][d][lane] = 0ull;
}

template <int DT, int THREADS>
__device__ __forceinline__ void hist_add(SnapSmem<DT, THREADS>& s, int warp, int lane, int32_t idx,
                                         int32_t core, int32_t mem) {
    // unconditional: infeasible rows (idx = -1) land in the dummy row 0, whose
    // content is never read (it may hold garbage from out-of-domain requests)
    s.hist[warp][idx + 1][lane] +=
        (static_cast<unsigned long long>(static_cast<uint32_t>(core)) << kAccShift) |
        static_cast<unsigned long long>(static_cast<uint32_t>(mem));
}

// ---- exchange rows (XchgRow): push this rank's sums to every peer, pull and consume ----
// word w of the 2*D-word vector (w = d: core demand on device d, w = D + d: mem demand): value v of this rank
// under exchange step step_plus1 - 1, to every rank's buffer.  Every 16-byte store is two 8-byte
// single-copy-atomic words with their own tags, so the words of a vector can come from different threads/CTAs.
__device__ __forceinline__ void xchg_push_word(DevState* st, unsigned long long step_plus1, int w, long long v) {
    const int world = st->peer.world, me = st->peer.rank;
    const int xs = static_cast<int>((step_plus1 - 1) % kXchgSlots);
    const unsigned long long tag = static_cast<unsigned long long>(xchg_tag(step_plus1)) << 32;
    const unsigned long long u = static_cast<unsigned long long>(v);
    const ulonglong2 wv = make_ulonglong2(tag | (u & 0xffffffffull), tag | (u >> 32));
    for (int p = 0; p < world; ++p) {
        XchgRow& row = st->peer.buf[p]->slot[xs][me];
        asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(&row.ll[2 * w]), "l"(wv.x), "l"(wv.y) : "memory");
    }
}
// thread d < D of one CTA; (dc, dm) = this rank's demand on device d
__device__ __forceinline__ void xchg_push(DevState* st, unsigned long long step_plus1, int d, int D, long long dc, long long dm) {
    xchg_push_word(st, step_plus1, d, dc);
    xchg_push_word(st, step_plus1, D + d, dm);
}
// waits until word w of every rank g carries the step's tag; adds those of ranks [g_lo, g_hi) into v;
// zeroes the words (consumed: a replayed sequence pushes the same steps again).  false = gave up after
// ~2 s (a rank died).  The loads of four ranks at a time are issued together (they are independent): the
// wait is one or two L2 round trips after the last word has landed, not one per rank.  Four, not eight:
// this is inlined into the scans' epilogues and must stay inside their register budget (eight ranks'
// words in flight took the 8-device scan from 60 to 88 registers and a quarter of its throughput).
constexpr int kPullGroup = 4;
__device__ __forceinline__ bool xchg_pull_word(XchgRow* rows, int world, unsigned long long step_plus1, int w, int g_lo, int g_hi,
                                               long long& v) {
    const unsigned long long tag = xchg_tag(step_plus1);
    const long long t0 = clock64();
    for (int gb = 0; gb < world; gb += kPullGroup) {
        const int ng = world - gb < kPullGroup ? world - gb : kPullGroup;
        unsigned int pending = (1u << ng) - 1u;
        for (;;) {
            unsigned long long w0[kPullGroup], w1[kPullGroup];
#pragma unroll
            for (int k = 0; k < kPullGroup; ++k) {
                w0[k] = w1[k] = 0ull;
                if ((pending >> k) & 1u)
                    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0[k]), "=l"(w1[k]) : "l"(&rows[gb + k].ll[2 * w]) : "memory");
            }
#pragma unroll
            for (int k = 0; k < kPullGroup; ++k) {
                if (((pending >> k) & 1u) && (w0[k] >> 32) == tag && (w1[k] >> 32) == tag) {
                    if (gb + k >= g_lo && gb + k < g_hi) v += static_cast<long long>((w0[k] & 0xffffffffull) | (w1[k] << 32));
                    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %1};" ::"l"(&rows[gb + k].ll[2 * w]), "l"(0ull) : "memory");
                    pending &= ~(1u << k);
                }
            }
            if (!pending) break;
            if (clock64() - t0 > 4000000000ll) return false;
            __nanosleep(40);
        }
    }
    return true;
}
// thread d < D: the two values for device d (words d and D + d) of every rank; see xchg_pull_word
__device__ __forceinline__ bool xchg_pull(XchgRow* rows, int world, unsigned long long step_plus1, int d, int D, int g_lo, int g_hi,
                                          long long& dc, long long& dm) {
    return xchg_pull_word(rows, world, step_plus1, d, g_lo, g_hi, dc) && xchg_pull_word(rows, world, step_plus1, D + d, g_lo, g_hi, dm);
}

// Where a CTA's epilogue goes: the launch's (or, in a multi-batch launch, the batch's) slot of
// running sums + arrival ticket, the exchange step to push under, and which of how many CTAs
// of that batch this one is.
struct EpiCtl {
    DevState::EpiSlot* ep;
    unsigned long long push;  // step + 1 when the demand vector must also go to the peers' exchange buffers, else 0
    unsigned int lag;         // with push: also apply the exchanged vectors of step (step - lag) here
    int tile, n_tiles;        // this CTA's number among the CTAs that share `ep`
    bool apply_now;           // with push: wait for the peers' vectors of THIS step here and write its table'
};
// Single-batch launches carry it as one word: bits 0..7 = epilogue slot, bits 8..55 = step + 1
// (0 = single GPU), bits 56..63 = lag; the CTAs of the grid are the tiles.
__device__ __forceinline__ EpiCtl epi_from_word(DevState* st, unsigned long long slot_step) {
    EpiCtl ec;
    ec.ep = &st->epi[slot_step & 0xffu];
    ec.push = (slot_step >> 8) & ((1ull << 48) - 1);
    ec.lag = static_cast<unsigned int>(slot_step >> 56);
    ec.tile = static_cast<int>(blockIdx.x);
    ec.n_tiles = static_cast<int>(gridDim.x);
    ec.apply_now = false;
    return ec;
}

// Second half of every snapshot epilogue.  `wacc` holds per-warp demand sums in shared
// memory: core sum of device d of warp w at wacc[w * wstride + core_off + d], mem sum at
// [... + mem_off + d].  Called by all threads after a __syncthreads().  Publishes the CTA's
// sums; plain snapshots finish word by word (below), every other mode adds with red.global.add.u64, takes an arrival ticket, and the last CTA
// writes delta / table', optionally commits (and re-sorts) the table and resets the slot.
template <int WARPS>
__device__ __forceinline__ void epilogue_publish(const unsigned long long* wacc, int wstride, int core_off, int mem_off,
                                                 int32_t* sFc, int32_t* sFm, int32_t* sPosDev, int* sLast,
                                                 DevState* st, int D, long long* __restrict__ delta_out,
                                                 int32_t* __restrict__ table_out, int flags, const EpiCtl& ec,
                                                 unsigned long long* __restrict__ tile_sums = nullptr) {
    DevState::EpiSlot& ep = *ec.ep;
    const unsigned long long push = ec.push;
    // with push and lag: also apply the exchanged vectors of step (step - lag) here and
    // write ITS table' to table_out: no separate apply launches, no second stream
    const unsigned long long lag = ec.lag;
    const int tid = threadIdx.x;
    if ((flags & (kFlagFinalize | kFlagCommit)) == kFlagFinalize && !lag && !tile_sums && ec.n_tiles < (1 << (64 - kEpiTicketShift))) {
        // Plain snapshot (no commit, no lagged apply): the arrival ticket rides in the top bits of
        // every running sum, so ONE returning atomic per word is the whole protocol: the CTA whose
        // add returns n_tiles - 1 arrivals holds that word's total (old + own) and publishes it.
        // Nothing is re-read, so nothing needs a fence; the words of one batch may be finished by
        // different CTAs.  The exchange is word-granular too (every pushed word carries its own
        // tag): the finisher of a word pushes it and, with apply_now, collects that word from every
        // rank.  Only the oversubscription flag needs both sums of a device: the two finishers swap
        // their sign bits through ep.pair[d] (the second one to come writes the flag).  Critical
        // path of a launch's last CTA: one L2 round trip (two with table'), against red + fence +
        // ticket + re-load in the general path below.  Sums < 2^49 (EGPU_MAX_ROWS rows of < 2^18; a whole-card row of spec 2.8 adds < 2^18 to each of its cards, so that holds).
        if (tid >= 2 * D) return;
        const int d = tid < D ? tid : tid - D;
        const int j = tid < D ? core_off + tid : mem_off + (tid - D);
        unsigned long long tot = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) tot += wacc[w * wstride + j];
        unsigned long long* word = &ep.acc[tid < D ? tid : kMaxD + d];
        const unsigned long long old = atomicAdd(word, tot + (1ull << kEpiTicketShift));
        if ((old >> kEpiTicketShift) != static_cast<unsigned long long>(ec.n_tiles - 1)) return;
        *reinterpret_cast<volatile unsigned long long*>(word) = 0ull;  // the slot's next batch is at least a launch group away
        long long total = static_cast<long long>((old + tot) & ((1ull << kEpiTicketShift) - 1));
        if (delta_out) delta_out[tid] = total;
        bool ok = true;
        if (push) {
            xchg_push_word(st, push, tid, total);  // word tid of this rank's vector, straight into every rank's buffer
            if (ec.apply_now) {
                // the ranks run the same launch at the same time (start gate): a peer-store latency.
                // This thread has pushed before it waits and no push waits for anything: no cycle.
                total = 0;
                ok = xchg_pull_word(st->peer.buf[st->peer.rank]->slot[(push - 1) % kXchgSlots], st->peer.world, push, tid, 0,
                                    st->peer.world, total);
                if (!ok) st->peer_timeout = push;  // a rank died: reported by the host, table' is not written
            }
        }
        if (table_out) {
            const long long left = static_cast<long long>(tid < D ? st->free_core[d] : st->free_mem[d]) - total;
            if (ok) table_out[tid] = sat_i32(left);
            const unsigned int mine = 2u | (left < 0 ? 1u : 0u);
            const unsigned int other = atomicExch(&ep.pair[d], mine);
            if (other & 2u) {
                table_out[2 * D + d] = static_cast<int32_t>((other | mine) & 1u);
                *reinterpret_cast<volatile unsigned int*>(&ep.pair[d]) = 0u;
            }
        }
        return;
    }
    if (tid < 2 * D) {
        const int j = tid < D ? core_off + tid : mem_off + (tid - D);
        unsigned long long tot = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) tot += wacc[w * wstride + j];
        if (tot) atomicAdd(&ep.acc[tid < D ? tid : kMaxD + (tid - D)], tot);
        // prefix-commit mode: this CTA owns a contiguous run of rows; keep its sums per device
        if (tile_sums) tile_sums[static_cast<size_t>(ec.tile) * 2 * kMaxD + (tid < D ? tid : kMaxD + (tid - D))] = tot;
        // release: only the threads that published sums need to order them before the ticket
        // (acq_rel is enough for this message-passing pattern and lighter than __threadfence's fence.sc)
        fence_acq_rel_gpu();
    }
    __syncthreads();
    if (tid == 0) {
        const unsigned int ticket = atomicAdd(&ep.ticket, 1u);
        *sLast = (ticket == static_cast<unsigned int>(ec.n_tiles - 1));
    }
    __syncthreads();
    if (!*sLast) return;
    fence_acq_rel_gpu();  // acquire: the other CTAs' sums, published before their tickets
    const bool fin = (flags & kFlagFinalize) != 0;
    const bool commit = fin && (flags & kFlagCommit);
    if (fin && tid < D) {
        volatile unsigned long long* acc = ep.acc;
        const long long dc = static_cast<long long>(acc[tid]);
        const long long dm = static_cast<long long>(acc[kMaxD + tid]);
        acc[tid] = 0ull;
        acc[kMaxD + tid] = 0ull;
        const long long nc = static_cast<long long>(st->free_core[tid]) - dc;
        const long long nm = static_cast<long long>(st->free_mem[tid]) - dm;
        const int32_t over = (nc < 0 || nm < 0) ? 1 : 0;
        if (delta_out) {
            delta_out[tid] = dc;
            delta_out[D + tid] = dm;
        }
        if (push) xchg_push(st, push, tid, D, dc, dm);  // fused exchange: this rank's vector straight into every rank's buffer
        if (table_out && !lag && !ec.apply_now) {
            table_out[tid] = sat_i32(nc);
            table_out[D + tid] = sat_i32(nm);
            table_out[2 * D + tid] = over;
        }
        if (commit) {
            // the committed table stays inside the spec's domain: negative
            // leftovers clamp to 0 and the oversubscription flag is sticky
            const int32_t cc = nc < 0 ? 0 : static_cast<int32_t>(nc);
            const int32_t cm = nm < 0 ? 0 : static_cast<int32_t>(nm);
            st->free_core[tid] = cc;
            st->free_mem[tid] = cm;
            st->oversub[tid] |= over;
            sFc[tid] = cc;
            sFm[tid] = cm;
        }
    }
    if (commit) resort_table_cta(st, D, sFc, sFm, sPosDev, tid);
    if (push && (ec.apply_now || (lag && push > lag))) {
        // Lagged apply, fused: the vectors of step (step - lag) have had `lag` launches to
        // arrive, so this wait normally falls through.  It is also the back-pressure that
        // keeps every rank within `lag` steps of the slowest one (and so inside the slots).
        // apply_now (multi-batch sharded launches): the same for THIS step - the ranks run the
        // same launch at the same time (start gate), so the wait is a peer-store latency; this
        // CTA has pushed before it waits and no rank's push waits for anything, so there is no cycle.
        const unsigned long long ap = ec.apply_now ? push : push - lag;  // step + 1 of the vectors to apply
        const int world = st->peer.world, me = st->peer.rank;
        XchgRow* rows = st->peer.buf[me]->slot[(ap - 1) % kXchgSlots];
        long long dc = 0, dm = 0;
        bool ok = true;
        if (tid < D) ok = xchg_pull(rows, world, ap, tid, D, 0, world, dc, dm);
        if (!ok) {
            st->peer_timeout = ap;
        } else if (tid < D && table_out) {
            const long long nc = static_cast<long long>(st->free_core[tid]) - dc;
            const long long nm = static_cast<long long>(st->free_mem[tid]) - dm;
            table_out[tid] = sat_i32(nc);
            table_out[D + tid] = sat_i32(nm);
            table_out[2 * D + tid] = (nc < 0 || nm < 0) ? 1 : 0;
        }
    }
    if (tid == 0) ep.ticket = 0u;
}

// Demand sums -> global running sums -> (last CTA) delta / table' publication.
template <int DT, int THREADS>
__device__ __forceinline__ void snapshot_epilogue(SnapSmem<DT, THREADS>& s, DevState* st, int D,
                                                  long long* __restrict__ delta_out,
                                                  int32_t* __restrict__ table_out, int flags, const EpiCtl& ec,
                                                  unsigned long long* __restrict__ tile_sums = nullptr) {
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    __syncwarp();
    for (int d = 0; d < D; ++d) {
        const unsigned long long v = s.hist[warp][d + 1][lane];
        const uint32_t c = static_cast<uint32_t>(v >> kAccShift);
        const uint32_t ml = static_cast<uint32_t>(v) & 0x7FFFFu;
        const uint32_t mh = static_cast<uint32_t>(v >> 19) & 0x7FFFFu;
        const uint32_t sc = __reduce_add_sync(0xffffffffu, c);
        const uint32_t sl = __reduce_add_sync(0xffffffffu, ml);
        const uint32_t sh = __reduce_add_sync(0xffffffffu, mh);
        if (lane == 0) {
            s.sWarpAcc[warp][d] = sc;
            s.sWarpAcc[warp][DT + d] = static_cast<unsigned long long>(sl) + (static_cast<unsigned long long>(sh) << 19);
        }
    }
    __syncthreads();
    epilogue_publish<THREADS / 32>(&s.sWarpAcc[0][0], 2 * DT, 0, DT, s.sFc, s.sFm, s.sPosDev, &s.sLast, st, D, delta_out,
                                   table_out, flags, ec, tile_sums);
}

// The scan of one batch by one CTA: tile `tile` of `n_tiles` (in a single-batch launch the grid's
// CTAs are the tiles; in a multi-batch launch every batch has its own run of tiles).
// CONTIG = false: vectors are dealt round-robin over the batch's tiles (the product mapping).
// CONTIG = true (prefix-commit mode): tile b scans the contiguous rows of "tile" b and the
// epilogue leaves its per-device sums in tile_sums[b][*]; everything else is the same code.
// Returns D.  Leaves the demand sums in s.hist; the caller runs snapshot_epilogue.
template <int DT, int THREADS, bool CONTIG>
__device__ __forceinline__ int sorted_scan_rows(SnapSmem<DT, THREADS>& s, DevState* __restrict__ st,
                                                const int32_t* __restrict__ req_core, const int32_t* __restrict__ req_mem,
                                                long long R, int32_t* __restrict__ out_idx, int tile_i, int n_tiles) {
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    // 32-bit vector indices (the entry points keep R below 2^31): one IMAD.WIDE per address, 32-bit compares
    const int4* __restrict__ vc = reinterpret_cast<const int4*>(req_core);
    const int4* __restrict__ vm = reinterpret_cast<const int4*>(req_mem);
    int4* __restrict__ vo = reinterpret_cast<int4*>(out_idx);
    int nvec = static_cast<int>(R >> 2);  // CONTIG: end of this CTA's tile
    int stride = n_tiles * THREADS;
    int v = tile_i * THREADS + tid;
    if (CONTIG) {
        const int per = (nvec + n_tiles - 1) / n_tiles;
        const long long lo = static_cast<long long>(tile_i) * per;  // may exceed nvec on a capped grid
        nvec = (lo + per < nvec) ? static_cast<int>(lo + per) : nvec;
        stride = THREADS;
        v = lo < nvec ? static_cast<int>(lo) + tid : nvec;
    }

    // issue the first tile's loads before anything else: the request stream is
    // the only HBM traffic that matters
    int4 c0 = make_int4(0, 0, 0, 0), m0 = c0, c1 = c0, m1 = c0;
    bool has0 = v < nvec, has1 = (v + stride) < nvec;
    if (has0) {
        c0 = ld_stream_v4(vc + v);
        m0 = ld_stream_v4(vm + v);
    }
    if (has1) {
        c1 = ld_stream_v4(vc + (v + stride));
        m1 = ld_stream_v4(vm + (v + stride));
    }

    // sorted table rows: uniform loads straight into registers, no barrier
    const int D = st->D;
    uint32_t K[DT];
#pragma unroll
    for (int j = 0; j < DT; j += 4) {
        const uint4 k4 = *reinterpret_cast<const uint4*>(&st->sorted_k[j]);
        K[j] = k4.x; K[j + 1] = k4.y; K[j + 2] = k4.z; K[j + 3] = k4.w;
    }
    const uint32_t gx = st->cand_xor, gm = st->cand_mask;
    // warp-private tile of the position -> device map: only a warp-level barrier.  "No feasible
    // row" comes out of first_feasible as DT (D > 32) or as kNoCand = 32 (DT <= 32): both map to -1.
    int32_t* tile = s.sDevTile[warp];
    for (int j = lane; j < kDevTile; j += 32) tile[j] = j < DT ? st->sorted_dev[j] : -1;
    hist_zero<DT, THREADS>(s, warp, lane);
    __syncwarp();

    auto decide = [&](int32_t core, int32_t mem) -> int32_t {
        const uint32_t best = first_feasible<DT>(K, pack_request_word(core, mem), gx, gm);
        const int32_t idx = tile[best];
        hist_add<DT, THREADS>(s, warp, lane, idx, core, mem);
        return idx;
    };
    auto decide4 = [&](const int4& c, const int4& m) -> int4 {
        int4 r;
        r.x = decide(c.x, m.x);
        r.y = decide(c.y, m.y);
        r.z = decide(c.z, m.z);
        r.w = decide(c.w, m.w);
        return r;
    };

    while (has0) {
        const int vn = v + 2 * stride;
        const bool nhas0 = vn < nvec, nhas1 = (vn + stride) < nvec;
        int4 nc0 = make_int4(0, 0, 0, 0), nm0 = nc0, nc1 = nc0, nm1 = nc0;
        if (nhas0) {
            nc0 = ld_stream_v4(vc + vn);
            nm0 = ld_stream_v4(vm + vn);
        }
        if (nhas1) {
            nc1 = ld_stream_v4(vc + (vn + stride));
            nm1 = ld_stream_v4(vm + (vn + stride));
        }
        st_stream_v4(vo + v, decide4(c0, m0));
        if (has1) st_stream_v4(vo + (v + stride), decide4(c1, m1));
        v = vn;
        has0 = nhas0;
        has1 = nhas1;
        c0 = nc0; m0 = nm0; c1 = nc1; m1 = nm1;
    }
    // ragged tail: R % 4 rows, scalar (they are the LAST rows: in CONTIG mode they belong to the last tile)
    if (tile_i == (CONTIG ? n_tiles - 1 : 0) && tid < static_cast<int>(R & 3)) {
        const long long r = ((R >> 2) << 2) + tid;
        out_idx[r] = decide(req_core[r], req_mem[r]);
    }
    return D;
}

template <int DT, int THREADS, bool CONTIG = false>
__global__ void __launch_bounds__(THREADS)  // (forcing 5 CTAs/SM = 48 registers was measured slower: ptxas then puts
                                            //  more of the adds on the ALU pipe; same-box A/B, DESIGN.md 7.2)
bestfit_sorted_kernel(DevState* __restrict__ st, const int32_t* __restrict__ req_core,
                      const int32_t* __restrict__ req_mem, long long R, int32_t* __restrict__ out_idx,
                      long long* __restrict__ delta_out, int32_t* __restrict__ table_out, int flags, unsigned long long slot_step,
                      const DevLut* __restrict__ /*glut: the lookup scan's*/, unsigned long long* __restrict__ tile_sums) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& s = *reinterpret_cast<SnapSmem<DT, THREADS>*>(smem_raw);
    const bool late = (flags & kFlagLateWait) != 0;
    const bool boundary = (flags & kFlagBoundary) != 0;
    if (!late) pdl_wait();  // predecessor may have produced our inputs or changed the table
    if ((flags & kFlagEarlyTrigger) && !boundary) pdl_trigger();
    const int D = sorted_scan_rows<DT, THREADS, CONTIG>(s, st, req_core, req_mem, R, out_idx, static_cast<int>(blockIdx.x),
                                                        static_cast<int>(gridDim.x));
    if (boundary) {  // everything older must be complete before the next group may start
        pdl_wait();
        pdl_trigger();
    }
    snapshot_epilogue<DT, THREADS>(s, st, D, delta_out, table_out, flags, epi_from_word(st, slot_step), CONTIG ? tile_sums : nullptr);
    if (late && !boundary) pdl_wait();  // do not complete before the predecessor has: keeps stream order transitive
}

// Grid of a multi-batch launch: the first `extra` batches have base + 1 tiles (CTAs), the others
// base, so that K * base + extra can be exactly the number of CTAs the GPU holds at once (every SM
// equally loaded) whatever K is.  tiles_extra = base | extra << 16.
__device__ __forceinline__ void multi_cta_to_tile(int tiles_extra, int& batch, int& tile_i, int& tiles) {
    const int base = tiles_extra & 0xffff, extra = tiles_extra >> 16;
    const int bid = static_cast<int>(blockIdx.x);
    const int cut = extra * (base + 1);
    if (bid < cut) {
        tiles = base + 1;
        batch = bid / tiles;
        tile_i = bid - batch * tiles;
    } else {
        tiles = base;
        const int b2 = (bid - cut) / base;
        batch = extra + b2;
        tile_i = (bid - cut) - b2 * base;
    }
}

// Multi-batch launch (egpu_bestfit_batches_dev): K independent batches, all scored against the
// same table, in ONE grid.  CTA (b, t) = tile t of batch b; every batch has its own epilogue
// slot, so that batch's demand sums / table' are published (and its exchange step pushed) by its
// own CTAs as soon as that batch is done.  One launch latency, one ramp and one tail for K batches
// instead of K: what the per-launch fixed cost (first DRAM touch, the epilogue's atomics) was
// eating at R = 1 M, and the launch floor at R = 1 k .. 100 k.
template <int DT, int THREADS>
__global__ void __launch_bounds__(THREADS)
bestfit_sorted_multi_kernel(DevState* __restrict__ st, const __grid_constant__ MultiArgs args, int tiles_extra, int flags,
                            unsigned int slot_base, unsigned long long push_base, const DevLut* __restrict__ /*glut: the lookup scan's*/) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& s = *reinterpret_cast<SnapSmem<DT, THREADS>*>(smem_raw);
    const bool late = (flags & kFlagLateWait) != 0;
    const bool boundary = (flags & kFlagBoundary) != 0;
    if (!late) pdl_wait();
    if ((flags & kFlagEarlyTrigger) && !boundary) pdl_trigger();
    int batch, tile_i, tiles;
    multi_cta_to_tile(tiles_extra, batch, tile_i, tiles);
    const BatchDesc b = args.b[batch];  // one read of the parameter space, then registers
    const int D = sorted_scan_rows<DT, THREADS, false>(s, st, b.rc, b.rm, b.R, b.idx, tile_i, tiles);
    if (boundary) {
        pdl_wait();
        pdl_trigger();
    }
    EpiCtl ec;
    ec.ep = &st->epi_multi[(slot_base + static_cast<unsigned int>(batch)) % kMultiSlots];
    ec.push = push_base ? push_base + static_cast<unsigned long long>(batch) : 0ull;
    ec.lag = 0;
    ec.tile = tile_i;
    ec.n_tiles = tiles;
    ec.apply_now = (flags & kFlagApplyNow) != 0;
    snapshot_epilogue<DT, THREADS>(s, st, D, b.delta, b.table_out, flags, ec);
    if (late && !boundary) pdl_wait();
}

// Packed wire format (include/egpu_alloc.h: egpu_bestfit_batch_packed): one uint32 per request
// (core << 18 | mem, anything >= 2^25 = "no valid request") and one int8 per decision - 5 bytes
// per decision instead of 12.  Same scan, same epilogue.
template <int DT, int THREADS>
__global__ void __launch_bounds__(THREADS)
bestfit_sorted_packed_kernel(DevState* __restrict__ st, const uint32_t* __restrict__ req, long long R,
                             signed char* __restrict__ out_idx8, long long* __restrict__ delta_out,
                             int32_t* __restrict__ table_out, int flags, unsigned long long slot_step) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& s = *reinterpret_cast<SnapSmem<DT, THREADS>*>(smem_raw);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const bool late = (flags & kFlagLateWait) != 0;
    if (!late) pdl_wait();
    if (flags & kFlagEarlyTrigger) pdl_trigger();

    // A warp takes chunks of 512 requests (2 KiB in, 512 B out): four fully coalesced 128-bit
    // loads per lane (lane-contiguous, 512 B per instruction) and four coalesced 32-bit stores.
    const long long nchunk = R >> 9;
    const long long wstride = static_cast<long long>(gridDim.x) * (THREADS / 32);
    long long ch = static_cast<long long>(blockIdx.x) * (THREADS / 32) + warp;
    uint4 p[4];
    bool has = ch < nchunk;
    auto load_chunk = [&](long long ci, uint4 (&dst)[4]) {
        const uint4* src = reinterpret_cast<const uint4*>(req) + 128 * ci + lane;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            int4 t = ld_stream_v4(reinterpret_cast<const int32_t*>(src + 32 * u));
            dst[u] = make_uint4(t.x, t.y, t.z, t.w);
        }
    };
    if (has) load_chunk(ch, p);

    const int D = st->D;
    uint32_t K[DT];
#pragma unroll
    for (int j = 0; j < DT; j += 4) {
        const uint4 k4 = *reinterpret_cast<const uint4*>(&st->sorted_k[j]);
        K[j] = k4.x; K[j + 1] = k4.y; K[j + 2] = k4.z; K[j + 3] = k4.w;
    }
    const uint32_t gx = st->cand_xor, gm = st->cand_mask;
    int32_t* tile = s.sDevTile[warp];
    for (int j = lane; j < kDevTile; j += 32) tile[j] = j < DT ? st->sorted_dev[j] : -1;
    hist_zero<DT, THREADS>(s, warp, lane);
    __syncwarp();

    auto decide = [&](uint32_t pw) -> uint32_t {
        // core << 18 | mem  ->  core << 24 | mem << 5; out-of-format words fail every guard
        const uint32_t q = (pw >> 25) ? (127u << 24) : (((pw & ~0x3FFFFu) << 6) | ((pw & 0x3FFFFu) << 5));
        const uint32_t best = first_feasible<DT>(K, q, gx, gm);
        const int32_t idx = tile[best];
        hist_add<DT, THREADS>(s, warp, lane, idx, static_cast<int32_t>((pw >> 18) & 127u), static_cast<int32_t>(pw & 0x3FFFFu));
        return static_cast<uint32_t>(idx) & 0xffu;
    };
    auto decide4 = [&](const uint4& v) -> uint32_t {
        return decide(v.x) | (decide(v.y) << 8) | (decide(v.z) << 16) | (decide(v.w) << 24);
    };
    while (has) {
        const long long cn = ch + wstride;
        const bool nhas = cn < nchunk;
        uint4 np[4];
        if (nhas) load_chunk(cn, np);
        uint32_t* out32 = reinterpret_cast<uint32_t*>(out_idx8) + 128 * ch + lane;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t r4 = decide4(p[u]);
            asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(out32 + 32 * u), "r"(r4) : "memory");
        }
        ch = cn;
        has = nhas;
#pragma unroll
        for (int u = 0; u < 4; ++u) p[u] = np[u];
    }
    // ragged tail: R % 512 rows, scalar, spread over the first CTA
    if (blockIdx.x == 0) {
        for (long long r = (nchunk << 9) + tid; r < R; r += THREADS) out_idx8[r] = static_cast<signed char>(decide(req[r]));
    }
    snapshot_epilogue<DT, THREADS>(s, st, D, delta_out, table_out, flags, epi_from_word(st, slot_step));
    if (late) pdl_wait();
}

// The north-star's literal formulation: every (device, request) pair is scored
// with the spec's packed key (lc << 24 | lm << 6 | d) against a shared-memory
// tile of the table and the row is reduced with a running min.  Kept as an
// independent second device implementation (tests compare the two) and as the
// baseline the sorted variant is measured against.
template <int DT, int THREADS>
__global__ void __launch_bounds__(THREADS)
bestfit_grid_kernel(DevState* __restrict__ st, const int32_t* __restrict__ req_core,
                    const int32_t* __restrict__ req_mem, long long R, int32_t* __restrict__ out_idx,
                    long long* __restrict__ delta_out, int32_t* __restrict__ table_out, int flags, unsigned long long slot_step,
                    const DevLut* __restrict__ /*glut: the lookup scan's*/,
                    unsigned long long* __restrict__ /*tile_sums: not supported by the literal variant*/) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& s = *reinterpret_cast<SnapSmem<DT, THREADS>*>(smem_raw);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    pdl_wait();  // never triggers early: the literal variant keeps plain stream semantics
    const int D = st->D;
    hist_zero<DT, THREADS>(s, warp, lane);
    if (tid < D) {
        s.sFc[tid] = st->free_core[tid];
        s.sFm[tid] = st->free_mem[tid];
    }
    __syncthreads();

    auto decide = [&](int32_t core, int32_t mem) -> int32_t {
        int32_t best = 0x7fffffff;
        const bool valid = (core | mem) >= 0;
        for (int d = 0; d < D; ++d) {
            const int32_t lc = s.sFc[d] - core;
            const int32_t lm = s.sFm[d] - mem;
            const int32_t key = (lc << 24) | (lm << 6) | d;
            best = (valid && (lc | lm) >= 0) ? min(best, key) : best;
        }
        const int32_t idx = best == 0x7fffffff ? -1 : (best & 63);
        hist_add<DT, THREADS>(s, warp, lane, idx, core, mem);
        return idx;
    };

    const long long nvec = R >> 2;
    const long long stride = static_cast<long long>(gridDim.x) * THREADS;
    for (long long v = static_cast<long long>(blockIdx.x) * THREADS + tid; v < nvec; v += stride) {
        const int4 c = ld_stream_v4(req_core + 4 * v);
        const int4 m = ld_stream_v4(req_mem + 4 * v);
        int4 r;
        r.x = decide(c.x, m.x);
        r.y = decide(c.y, m.y);
        r.z = decide(c.z, m.z);
        r.w = decide(c.w, m.w);
        st_stream_v4(out_idx + 4 * v, r);
    }
    if (blockIdx.x == 0 && tid < static_cast<int>(R & 3)) {
        const long long r = (nvec << 2) + tid;
        out_idx[r] = decide(req_core[r], req_mem[r]);
    }
    snapshot_epilogue<DT, THREADS>(s, st, D, delta_out, table_out, flags, epi_from_word(st, slot_step));
}

// =============================================================================
// Lookup-table scan for large D (EGPU_VARIANT_LUT; AUTO picks it for D > 16)
// =============================================================================
//
// The register-resident scan above costs 3.5 instructions per (request, device) pair:
// fine for D = 8 (HBM-bound), ALU-bound by 4x at D = 64.  The lookup form needs two
// shared-memory reads and ~25 instructions per request whatever D is.

// Builds DevLut from the sorted view in DevState.  One CTA; runs after every table change.
__global__ void __launch_bounds__(256)
lut_build_kernel(const DevState* __restrict__ st, DevLut* __restrict__ lut) {
    __shared__ uint32_t sFm[kMaxD], sFcs[kMaxD], sV[kMaxD + 4];
    __shared__ int sFirst[kMaxD], sRidx[kMaxD], sNv, sBlocks;
    __shared__ uint8_t sA[kLutStride * kLutStride];  // a[srow][rank]: first device at or after srow with ridx >= rank
    __shared__ uint8_t sStart[kLutCRows];
    const int tid = threadIdx.x;
    const int D = st->D;
    if (tid < kMaxD) {
        const uint32_t k = tid < D ? st->sorted_k[tid] : 0u;
        sFm[tid] = (k >> 5) & 0x3FFFFu;
        sFcs[tid] = (k >> 24) & 0x7Fu;
    }
    if (tid < kMaxD + 4) sV[tid] = 0xFFFFFFFFu;
    __syncthreads();
    if (tid < D) {  // first occurrence of its fm value?
        int first = 1;
        for (int k = 0; k < tid; ++k) first &= (sFm[k] != sFm[tid]);
        sFirst[tid] = first;
    }
    __syncthreads();
    if (tid < D) {  // ridx = number of distinct values below mine
        int r = 0;
        for (int k = 0; k < D; ++k) r += (sFirst[k] && sFm[k] < sFm[tid]);
        sRidx[tid] = r;
        sV[r] = sFm[tid];
    }
    if (tid == 0) {
        int nv = 0;
        for (int k = 0; k < D; ++k) nv += sFirst[k];
        sNv = nv;
        sBlocks = 0;
        lut->nv = nv;
    }
    __syncthreads();
    const int nv = sNv;
    if (tid < kMaxD + 4) lut->v[tid] = sV[tid];
    if (tid < kLutCRows) {  // start[c] = first sorted position with fc >= c (c = 101: none, position D)
        int n = 0;
        for (int k = 0; k < D; ++k) n += (sFcs[k] < static_cast<uint32_t>(tid));
        sStart[tid] = static_cast<uint8_t>(n);
    }
    if (tid < kLutStride) {  // column r of a[][]: walk the suffixes from the back
        const int r = tid;
        uint8_t cur = 0xFF;
        for (int srow = kMaxD; srow >= 0; --srow) {
            if (srow < D && sRidx[srow] >= r) cur = static_cast<uint8_t>(st->sorted_dev[srow]);
            if (srow > D) cur = 0xFF;
            sA[srow * kLutStride + r] = cur;
        }
    }
    __syncthreads();
    for (int i = tid; i < kLutCRows * kLutStride; i += blockDim.x) {  // a2[c][r] = a[start[c]][r]
        const int c = i / kLutStride, r = i - c * kLutStride;
        lut->a2[i] = sA[sStart[c] * kLutStride + r];
    }
    for (int b = tid; b < kLutBuckets; b += blockDim.x) {
        const uint32_t lo_v = static_cast<uint32_t>(b) << 6, hi_v = lo_v + 64u;
        int lo = 0, hi = 0;
        for (int k = 0; k < nv; ++k) {
            lo += (sV[k] < lo_v);
            hi += (sV[k] < hi_v);
        }
        const int n = hi - lo;
        uint32_t e = static_cast<uint32_t>(lo);
        if (n == 0) {
            e |= 64u << 8;
        } else if (n == 1) {
            e |= ((sV[lo] & 63u) + 1u) << 8;
        } else {  // several thresholds in this bucket: exact ranks for its 64 values of m
            const int blk = atomicAdd(&sBlocks, 1);  // < 32: two values per block at least, 64 values in all
            e = kLutMulti | static_cast<uint32_t>(blk) | (64u << 8);
            for (uint32_t x = 0; x < 64u; ++x) {
                int r = lo;
                for (int k = lo; k < hi; ++k) r += (sV[k] < lo_v + x);
                lut->ovf[blk * 64 + x] = static_cast<uint8_t>(r);
            }
        }
        lut->bucket[b] = static_cast<uint16_t>(e);
    }
}

// Demand sums of the lookup scan.  64-bit shared-memory adds compile to CAS loops on sm_100a
// (ATOMS.CAST.SPIN.64) and lane-private 64-bit sums cost 16.6 KB per warp; what is used instead is
// native 32-bit ATOMS.ADD: two UNCONDITIONAL adds per request - word 0 = core | (mem >> 16) << 20,
// word 1 = mem & 0xffff - into one of 8 copies of a small table per warp (copy = lane / 4; the
// copies are 140 words apart, i.e. rotated by 12 banks, so the hot devices of a batch spread over
// the banks), infeasible rows into a per-lane dummy word: no branches, no shared hot spot.  A copy
// receives 4 lanes x 8 rows per trip, so word 0's 12-bit mem >> 16 field (<= 3 per add) lasts 42
// trips: the words are folded into 64-bit register sums every 32.
// (Measured and dropped, DESIGN.md 7.2: round 1's three conditional adds into one table per warp;
// 64-bit sums in columns owned by lane pairs with the half-warps taking turns - fewer shared-memory
// wavefronts, 7.95 M against 10.3 M per 20 M decisions, but 8.3 KB per warp halves the occupancy.)
// (4 copies of 8 lanes would fit four CTAs per SM instead of three: measured slower, 2.97 against 2.77 us per
// batch - the extra bank conflicts of the adds cost more than the occupancy brings)
constexpr int kLutCopies = 8;
constexpr int kLutLanesPerCopy = 32 / kLutCopies;
constexpr int kLutFlushTrips = 32;                                // 12-bit field, <= 3 per add, 4 lanes x 8 rows per trip
constexpr int kLutPlane = kMaxD + kLutLanesPerCopy;               // 64 devices + one dummy word per lane of the copy
constexpr int kLutCopyStride = 2 * kLutPlane + 4;                 // 140 words = 12 banks
template <int THREADS>
struct LutSmem {
    DevLut lut;
    unsigned long long sWarpAcc[THREADS / 32][2 * kMaxD];
    int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    int sLast;
    alignas(16) uint32_t hist32[THREADS / 32][kLutCopies * kLutCopyStride];
};

// The lookup scan of one batch by one CTA (tile `tile_i` of `n_tiles`, as sorted_scan_rows).
// Leaves the warp sums in sm.sWarpAcc; the caller synchronises and runs epilogue_publish.
template <int THREADS, bool CONTIG>
__device__ __forceinline__ int lut_scan_rows(LutSmem<THREADS>& sm, DevState* __restrict__ st,
                                             const int32_t* __restrict__ req_core, const int32_t* __restrict__ req_mem,
                                             long long R, int32_t* __restrict__ out_idx, const DevLut* __restrict__ glut,
                                             int tile_i, int n_tiles) {
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int4* __restrict__ vc = reinterpret_cast<const int4*>(req_core);
    const int4* __restrict__ vm = reinterpret_cast<const int4*>(req_mem);
    int4* __restrict__ vo = reinterpret_cast<int4*>(out_idx);
    int nvec = static_cast<int>(R >> 2);
    int stride = n_tiles * THREADS;
    int v = tile_i * THREADS + tid;
    if (CONTIG) {
        const int per = (nvec + n_tiles - 1) / n_tiles;
        const long long lo = static_cast<long long>(tile_i) * per;
        nvec = (lo + per < nvec) ? static_cast<int>(lo + per) : nvec;
        stride = THREADS;
        v = lo < nvec ? static_cast<int>(lo) + tid : nvec;
    }
    // vectors past the end stay (-1, -1): infeasible requests, which land in the lane's dummy word
    int4 c0 = make_int4(-1, -1, -1, -1), m0 = c0, c1 = c0, m1 = c0;
    bool has0 = v < nvec, has1 = (v + stride) < nvec;
    if (has0) {
        c0 = ld_stream_v4(vc + v);
        m0 = ld_stream_v4(vm + v);
    }
    if (has1) {
        c1 = ld_stream_v4(vc + (v + stride));
        m1 = ld_stream_v4(vm + (v + stride));
    }
    // shared-memory tile of the lookup tables (15 KB, L2-resident source)
    {
        const uint4* src = reinterpret_cast<const uint4*>(glut);
        uint4* dst = reinterpret_cast<uint4*>(&sm.lut);
        for (int i = tid; i < static_cast<int>(sizeof(DevLut) / 16); i += THREADS) dst[i] = src[i];
    }
    const int D = st->D;
    {  // zero this warp's 32-bit tables
        uint4* hz = reinterpret_cast<uint4*>(&sm.hist32[warp][0]);
        constexpr int n16 = static_cast<int>(sizeof(sm.hist32[0]) / 16);
        for (int i = lane; i < n16; i += 32) hz[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    // 64-bit running sums of this warp: lane L keeps devices L and L + 32
    unsigned long long acc_c[2] = {0ull, 0ull}, acc_m[2] = {0ull, 0ull};
    __syncthreads();
    const DevLut& L = sm.lut;
    uint32_t* const hw = &sm.hist32[warp][0];
    uint32_t* const hcopy = hw + (lane / kLutLanesPerCopy) * kLutCopyStride;
    const uint32_t dummy_col = static_cast<uint32_t>(kMaxD) + (static_cast<uint32_t>(lane) % kLutLanesPerCopy);

    // device (0..63) or 0xFF for one request: two dependent shared-memory reads, no branch
    // (the read of ovf[] is predicated: only requests whose bucket holds several thresholds)
    auto lookup = [&](int32_t core, int32_t mem) -> uint32_t {
        const uint32_t c = min(static_cast<uint32_t>(core), static_cast<uint32_t>(kCoreMax + 1));
        const uint32_t m = min(static_cast<uint32_t>(mem), 1u << 18);
        const uint32_t e = L.bucket[m >> 6];
        const uint32_t lo7 = e & 0x7Fu, x = m & 63u;
        uint32_t rank = lo7 + (((e >> 8) - 1u - x) >> 31);  // + 1 iff x >= t
        if (e & kLutMulti) rank = L.ovf[lo7 * 64u + x];
        return L.a2[c * kLutStride + rank];
    };
    // fold this warp's 32-bit words into the 64-bit sums and clear them
    auto flush32 = [&]() {
        __syncwarp();
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int d = lane + 32 * half;
            uint32_t cs = 0, mh = 0, ml = 0;
#pragma unroll
            for (int j = 0; j < kLutCopies; ++j) {  // bank = (12 j + lane) mod 32: conflict-free
                uint32_t* h = hw + j * kLutCopyStride;
                const uint32_t w0 = h[d], w1 = h[kLutPlane + d];
                h[d] = 0u;
                h[kLutPlane + d] = 0u;
                cs += w0 & 0xFFFFFu;
                mh += w0 >> 20;
                ml += w1;
            }
            acc_c[half] += cs;
            acc_m[half] += static_cast<unsigned long long>(ml) + (static_cast<unsigned long long>(mh) << 16);
        }
        __syncwarp();
    };
    auto add1 = [&](uint32_t dev, int32_t core, int32_t mem) {
        // infeasible rows (0xFF) go to this lane's dummy word, whose content is never read
        // (their core / mem may be anything: nothing carries from one word into another)
        const uint32_t col = min(dev, dummy_col);
        atomicAdd(&hcopy[col], static_cast<uint32_t>(core) | ((static_cast<uint32_t>(mem) >> 16) << 20));
        atomicAdd(&hcopy[kLutPlane + col], static_cast<uint32_t>(mem) & 0xffffu);
    };
    auto decide = [&](int32_t core, int32_t mem) -> int32_t {
        const uint32_t dev = lookup(core, mem);
        add1(dev, core, mem);
        return static_cast<int32_t>(static_cast<int8_t>(dev));
    };
    // All the lookups of a trip first, then all the adds: the shared-memory adds order every
    // later shared-memory read behind them (the compiler cannot tell the tables apart), so
    // interleaving them request by request makes one serial chain of eight dependent reads.
    auto lookup4 = [&](const int4& c, const int4& m) -> uint4 {
        return make_uint4(lookup(c.x, m.x), lookup(c.y, m.y), lookup(c.z, m.z), lookup(c.w, m.w));
    };
    auto add4 = [&](const uint4& d, const int4& c, const int4& m) {
        add1(d.x, c.x, m.x);
        add1(d.y, c.y, m.y);
        add1(d.z, c.z, m.z);
        add1(d.w, c.w, m.w);
    };
    auto as_idx4 = [](const uint4& d) -> int4 {
        return make_int4(static_cast<int8_t>(d.x), static_cast<int8_t>(d.y), static_cast<int8_t>(d.z), static_cast<int8_t>(d.w));
    };
    int trips = 0;
    while (__any_sync(0xffffffffu, has0)) {  // warp-uniform trip count: flush32() synchronises the warp
        if (++trips == kLutFlushTrips) {
            flush32();
            trips = 0;
        }
        const int vn = v + 2 * stride;
        const bool nhas0 = vn < nvec, nhas1 = (vn + stride) < nvec;
        int4 nc0 = make_int4(-1, -1, -1, -1), nm0 = nc0, nc1 = nc0, nm1 = nc0;
        if (nhas0) {
            nc0 = ld_stream_v4(vc + vn);
            nm0 = ld_stream_v4(vm + vn);
        }
        if (nhas1) {
            nc1 = ld_stream_v4(vc + (vn + stride));
            nm1 = ld_stream_v4(vm + (vn + stride));
        }
        // no branch around the lookups (lanes past the end carry infeasible requests): the eight
        // requests of a trip overlap their dependent reads
        const uint4 d0 = lookup4(c0, m0);
        const uint4 d1 = lookup4(c1, m1);
        if (has0) st_stream_v4(vo + v, as_idx4(d0));
        if (has1) st_stream_v4(vo + (v + stride), as_idx4(d1));
        add4(d0, c0, m0);
        add4(d1, c1, m1);
        v = vn;
        has0 = nhas0;
        has1 = nhas1;
        c0 = nc0; m0 = nm0; c1 = nc1; m1 = nm1;
    }
    if (tile_i == (CONTIG ? n_tiles - 1 : 0) && warp == 0) {  // ragged tail: R % 4 rows (the last ones), lanes 0..2 of warp 0
        const bool mine = lane < static_cast<int>(R & 3);
        const long long r = ((R >> 2) << 2) + lane;
        const int32_t c = mine ? req_core[r] : -1, m = mine ? req_mem[r] : -1;
        const uint32_t dev = lookup(c, m);
        if (mine) out_idx[r] = static_cast<int32_t>(static_cast<int8_t>(dev));
        add1(dev, c, m);
    }
    flush32();
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        sm.sWarpAcc[warp][lane + 32 * half] = acc_c[half];
        sm.sWarpAcc[warp][kMaxD + lane + 32 * half] = acc_m[half];
    }
    return D;
}

template <int THREADS, bool CONTIG = false>
__global__ void __launch_bounds__(THREADS)
bestfit_lut_kernel(DevState* __restrict__ st, const int32_t* __restrict__ req_core,
                   const int32_t* __restrict__ req_mem, long long R, int32_t* __restrict__ out_idx,
                   long long* __restrict__ delta_out, int32_t* __restrict__ table_out, int flags, unsigned long long slot_step,
                   const DevLut* __restrict__ glut, unsigned long long* __restrict__ tile_sums) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& sm = *reinterpret_cast<LutSmem<THREADS>*>(smem_raw);
    const bool late = (flags & kFlagLateWait) != 0;
    const bool boundary = (flags & kFlagBoundary) != 0;
    if (!late) pdl_wait();
    if ((flags & kFlagEarlyTrigger) && !boundary) pdl_trigger();
    const int D = lut_scan_rows<THREADS, CONTIG>(sm, st, req_core, req_mem, R, out_idx, glut, static_cast<int>(blockIdx.x),
                                                      static_cast<int>(gridDim.x));
    if (boundary) {
        pdl_wait();
        pdl_trigger();
    }
    __syncthreads();
    epilogue_publish<THREADS / 32>(&sm.sWarpAcc[0][0], 2 * kMaxD, 0, kMaxD, sm.sFc, sm.sFm, sm.sPosDev, &sm.sLast, st, D,
                                   delta_out, table_out, flags, epi_from_word(st, slot_step), CONTIG ? tile_sums : nullptr);
    if (late && !boundary) pdl_wait();
}

// Multi-batch form of the lookup scan (see bestfit_sorted_multi_kernel).
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
bestfit_lut_multi_kernel(DevState* __restrict__ st, const __grid_constant__ MultiArgs args, int tiles_extra, int flags,
                         unsigned int slot_base, unsigned long long push_base, const DevLut* __restrict__ glut) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& sm = *reinterpret_cast<LutSmem<THREADS>*>(smem_raw);
    const bool late = (flags & kFlagLateWait) != 0;
    const bool boundary = (flags & kFlagBoundary) != 0;
    if (!late) pdl_wait();
    if ((flags & kFlagEarlyTrigger) && !boundary) pdl_trigger();
    int batch, tile_i, tiles;
    multi_cta_to_tile(tiles_extra, batch, tile_i, tiles);
    const BatchDesc b = args.b[batch];
    const int D = lut_scan_rows<THREADS, false>(sm, st, b.rc, b.rm, b.R, b.idx, glut, tile_i, tiles);
    if (boundary) {
        pdl_wait();
        pdl_trigger();
    }
    __syncthreads();
    EpiCtl ec;
    ec.ep = &st->epi_multi[(slot_base + static_cast<unsigned int>(batch)) % kMultiSlots];
    ec.push = push_base ? push_base + static_cast<unsigned long long>(batch) : 0ull;
    ec.lag = 0;
    ec.tile = tile_i;
    ec.n_tiles = tiles;
    ec.apply_now = (flags & kFlagApplyNow) != 0;
    epilogue_publish<THREADS / 32>(&sm.sWarpAcc[0][0], 2 * kMaxD, 0, kMaxD, sm.sFc, sm.sFm, sm.sPosDev, &sm.sLast, st, D,
                                   b.delta, b.table_out, flags, ec);
    if (late && !boundary) pdl_wait();
}

// Multi-GPU step 2: table' = table - sum over ranks of their demand vectors.
__global__ void __launch_bounds__(kMaxD)
apply_deltas_kernel(DevState* __restrict__ st, const long long* __restrict__ deltas,
                    int G, int32_t* __restrict__ table_out, int commit) {
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    const int D = st->D;
    const int d = threadIdx.x;
    if (d < D) {
        long long dc = 0, dm = 0;
        for (int g = 0; g < G; ++g) {
            dc += deltas[static_cast<long long>(g) * 2 * D + d];
            dm += deltas[static_cast<long long>(g) * 2 * D + D + d];
        }
        const long long nc = static_cast<long long>(st->free_core[d]) - dc;
        const long long nm = static_cast<long long>(st->free_mem[d]) - dm;
        const int32_t over = (nc < 0 || nm < 0) ? 1 : 0;
        if (table_out) {
            table_out[d] = sat_i32(nc);
            table_out[D + d] = sat_i32(nm);
            table_out[2 * D + d] = over;
        }
        if (commit) {
            const int32_t cc = nc < 0 ? 0 : static_cast<int32_t>(nc);
            const int32_t cm = nm < 0 ? 0 : static_cast<int32_t>(nm);
            st->free_core[d] = cc;
            st->free_mem[d] = cm;
            st->oversub[d] |= over;
            sFc[d] = cc;
            sFm[d] = cm;
        }
    }
    if (commit) resort_table_cta(st, D, sFc, sFm, sPosDev, d);
}

// Multi-GPU step 2, peer-memory form: wait until every rank's demand vector of `step` has
// landed in THIS rank's exchange buffer, then apply their sum.  One CTA.  The spin gives up
// after ~2 s (a rank died): DevState::peer_timeout records it and the table is left alone.
constexpr int kApplyMax = 64;  // steps one apply launch may cover
struct ApplyOuts {
    int32_t* table_out[kApplyMax];
};

// Start gate of a sharded sequence (egpu_peer_gate_dev).  One thread block.  Waits until THIS
// rank's host has opened the gate (egpu_peer_gate_open: the host has finished enqueueing what
// follows the gate on the stream), then tells every peer and waits until every peer has said the
// same.  What follows the gate on the stream therefore starts within a peer-flag latency of the
// same instant on every rank, and nothing after it waits for a host.  Epochs count up from 1;
// a rank can be at most one gate ahead of a peer, so ">= epoch" is the arrival test.  Gives up
// after ~2 s (counted in DevState::gate_timeouts) and lets the stream proceed.
__global__ void __launch_bounds__(32)
gate_kernel(DevState* __restrict__ st, const unsigned long long* __restrict__ host_open) {
    const int world = st->peer.world, me = st->peer.rank;
    const int lane = threadIdx.x;
    const unsigned long long epoch = st->gate_epoch + 1;
    const long long t0 = clock64();
    bool ok = true;
    if (lane == 0) {
        for (;;) {
            unsigned long long h;
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(h) : "l"(host_open) : "memory");
            if (h >= epoch) break;
            if (clock64() - t0 > 4000000000ll) { ok = false; break; }
            __nanosleep(200);
        }
    }
    __syncwarp();
    if (lane < world) {
        unsigned long long* f = &st->peer.buf[lane]->ready[me];
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"(epoch) : "memory");
        const unsigned long long* mine = &st->peer.buf[me]->ready[lane];
        for (;;) {
            unsigned long long r;
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(r) : "l"(mine) : "memory");
            if (r >= epoch) break;
            if (clock64() - t0 > 4000000000ll) { ok = false; break; }
            __nanosleep(100);
        }
    }
    ok = __all_sync(0xffffffffu, ok);
    if (lane == 0) {
        st->gate_epoch = epoch;
        if (!ok) st->gate_timeouts += 1;
    }
}

// Without commit the steps are independent of each other (each is table - its own sum): the grid
// has one CTA per step, so the waits overlap instead of queueing behind one another (the vectors of
// all the steps of a multi-batch launch arrive at about the same time, when that launch drains).
// With commit the steps apply on top of each other: one CTA walks them in order.
__global__ void __launch_bounds__(kMaxD)
apply_peers_kernel(DevState* __restrict__ st, unsigned long long first_step_plus1, int nsteps, ApplyOuts outs, int commit) {
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    __shared__ int sOk;
    const int D = st->D;
    const int d = threadIdx.x;
    const int world = st->peer.world, me = st->peer.rank;
    // running table across the steps of this launch (only installed when commit is set)
    long long cur_c = d < D ? st->free_core[d] : 0, cur_m = d < D ? st->free_mem[d] : 0;
    int32_t sticky = 0;
    const int k_begin = commit ? 0 : static_cast<int>(blockIdx.x);
    const int k_end = commit ? nsteps : k_begin + 1;
    for (int k = k_begin; k < k_end; ++k) {
        const unsigned long long step_plus1 = first_step_plus1 + k;
        XchgRow* rows = st->peer.buf[me]->slot[(step_plus1 - 1) % kXchgSlots];
        if (d == 0) sOk = 1;
        __syncthreads();
        long long dc = 0, dm = 0;
        if (d < D && !xchg_pull(rows, world, step_plus1, d, D, 0, world, dc, dm)) sOk = 0;
        __syncthreads();
        if (!sOk) {
            if (d == 0) st->peer_timeout = step_plus1;
            return;
        }
        if (d < D) {
            const long long nc = cur_c - dc, nm = cur_m - dm;
            const int32_t over = (nc < 0 || nm < 0) ? 1 : 0;
            if (outs.table_out[k]) {
                outs.table_out[k][d] = sat_i32(nc);
                outs.table_out[k][D + d] = sat_i32(nm);
                outs.table_out[k][2 * D + d] = over;
            }
            if (commit) {  // the next step of this launch is applied on top of this one
                cur_c = nc < 0 ? 0 : nc;
                cur_m = nm < 0 ? 0 : nm;
                sticky |= over;
            }
        }
    }
    if (commit) {
        if (d < D) {
            st->free_core[d] = static_cast<int32_t>(cur_c);
            st->free_mem[d] = static_cast<int32_t>(cur_m);
            st->oversub[d] |= sticky;
            sFc[d] = static_cast<int32_t>(cur_c);
            sFm[d] = static_cast<int32_t>(cur_m);
        }
        resort_table_cta(st, D, sFc, sFm, sPosDev, d);
    }
}


// =============================================================================
// Prefix-commit (spec 2.5): turn the snapshot choice into an allocation that never
// oversubscribes
// =============================================================================
//
// Row r with choice d commits iff the running demand of d over rows <= r (all rows that
// chose d, committed or not) still fits free[d]; otherwise it is DEFERRED (-2).  Demands are
// non-negative, so per device the running demand is monotone and the rule is a single cut:
// rows before cut[d] commit, rows from cut[d] on are deferred.  The scan runs in CONTIG mode
// (CTA b = contiguous tile b) and leaves per-tile per-device sums; one CTA per device then
// (1) scans the tile sums to find the tile where its device crosses capacity, (2) scans
// that one tile's rows in order for the exact cut row and the committed demand;
// prefix_apply_kernel rewrites the indices, prefix_finalize_kernel publishes delta / table'.
struct PrefixOut {
    long long cut[kMaxD];          // first deferred row of device d, R when none
    long long committed_c[kMaxD];  // demand of the committed rows
    long long committed_m[kMaxD];
};

// exclusive block scan of two 64-bit values; returns the block totals through tot_*
template <int THREADS>
__device__ __forceinline__ void block_scan2(unsigned long long& a, unsigned long long& b, unsigned long long* sh /*[2][THREADS/32]*/,
                                            unsigned long long& tot_a, unsigned long long& tot_b) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long ia = a, ib = b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long ya = __shfl_up_sync(0xffffffffu, ia, o), yb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ya; ib += yb; }
    }
    if (lane == 31) { sh[warp] = ia; sh[THREADS / 32 + warp] = ib; }
    __syncthreads();
    unsigned long long wa = 0, wb = 0;
    tot_a = 0; tot_b = 0;
    for (int w = 0; w < THREADS / 32; ++w) {
        if (w < warp) { wa += sh[w]; wb += sh[THREADS / 32 + w]; }
        tot_a += sh[w]; tot_b += sh[THREADS / 32 + w];
    }
    __syncthreads();
    a = ia - a + wa;  // exclusive
    b = ib - b + wb;
}

__global__ void __launch_bounds__(256)
prefix_cut_kernel(const DevState* __restrict__ st, const int32_t* __restrict__ idx, const int32_t* __restrict__ req_core,
                  const int32_t* __restrict__ req_mem, long long R, int n_tiles,
                  const unsigned long long* __restrict__ tile_sums, PrefixOut* __restrict__ out,
                  const long long* __restrict__ base = nullptr /* [2][kMaxD]: demand of the lower ranks' rows */) {
    constexpr int T = 256;
    __shared__ unsigned long long sh[2 * (T / 32)];
    __shared__ long long sCutTile, sCutRow;
    __shared__ unsigned long long sBaseC, sBaseM, sComC, sComM;
    const int d = blockIdx.x;
    const int tid = threadIdx.x;
    const unsigned long long cap_c = static_cast<unsigned long long>(st->free_core[d]);
    const unsigned long long cap_m = static_cast<unsigned long long>(st->free_mem[d]);
    // Multi-GPU (rank-major row order): the rows of the lower ranks come first, so their whole
    // demand on this device is already on the running sums when this shard starts
    const unsigned long long pre_c = base ? static_cast<unsigned long long>(base[d]) : 0ull;
    const unsigned long long pre_m = base ? static_cast<unsigned long long>(base[kMaxD + d]) : 0ull;
    if (pre_c > cap_c || pre_m > cap_m) {  // the device filled up on a lower rank: nothing commits here
        if (tid == 0) {
            out->cut[d] = 0;
            out->committed_c[d] = 0;
            out->committed_m[d] = 0;
        }
        return;
    }
    if (tid == 0) { sCutTile = n_tiles; sCutRow = R; sBaseC = 0; sBaseM = 0; sComC = 0; sComM = 0; }
    __syncthreads();
    // (1) which tile crosses capacity?
    unsigned long long run_c = pre_c, run_m = pre_m;
    for (int t0 = 0; t0 < n_tiles; t0 += T) {
        const int t = t0 + tid;
        unsigned long long c = t < n_tiles ? tile_sums[static_cast<size_t>(t) * 2 * kMaxD + d] : 0ull;
        unsigned long long m = t < n_tiles ? tile_sums[static_cast<size_t>(t) * 2 * kMaxD + kMaxD + d] : 0ull;
        const unsigned long long own_c = c, own_m = m;
        unsigned long long tot_c, tot_m;
        block_scan2<T>(c, m, sh, tot_c, tot_m);  // c, m = demand of the tiles before t within this pass
        const unsigned long long before_c = run_c + c, before_m = run_m + m;
        // demand is monotone: exactly one tile has "fits before it, does not fit after it"
        if (t < n_tiles && (before_c + own_c > cap_c || before_m + own_m > cap_m) && before_c <= cap_c && before_m <= cap_m)
            sCutTile = t;
        __syncthreads();
        if (sCutTile < n_tiles) break;
        run_c += tot_c;
        run_m += tot_m;
    }
    __syncthreads();
    const long long cut_tile = sCutTile;
    if (cut_tile >= n_tiles) {  // the device never fills up: everything that chose it commits
        if (tid == 0) {
            out->cut[d] = R;
            out->committed_c[d] = static_cast<long long>(run_c - pre_c);
            out->committed_m[d] = static_cast<long long>(run_m - pre_m);
        }
        return;
    }
    // demand before the cut tile: rescan (cheap) up to cut_tile with a plain strided sum
    {
        unsigned long long c = 0, m = 0;
        for (long long t = tid; t < cut_tile; t += T) {
            c += tile_sums[static_cast<size_t>(t) * 2 * kMaxD + d];
            m += tile_sums[static_cast<size_t>(t) * 2 * kMaxD + kMaxD + d];
        }
        unsigned long long tc, tm;
        block_scan2<T>(c, m, sh, tc, tm);
        if (tid == 0) { sBaseC = pre_c + tc; sBaseM = pre_m + tm; }
        __syncthreads();
    }
    // (2) rows of the cut tile, in order
    const long long nvec = R >> 2;
    const long long per = (nvec + n_tiles - 1) / n_tiles;
    long long row_lo = cut_tile * per * 4;
    if (row_lo > nvec * 4) row_lo = nvec * 4;  // capped grids: ceil(nvec / n_tiles) can leave the last tile only the ragged tail
    long long row_hi = (cut_tile + 1) * per * 4;
    if (row_hi > nvec * 4) row_hi = nvec * 4;
    if (cut_tile == n_tiles - 1) row_hi = R;  // the ragged tail belongs to the last tile
    unsigned long long base_c = sBaseC, base_m = sBaseM;
    for (long long r0 = row_lo; r0 < row_hi; r0 += 4 * T) {
        const long long r = r0 + 4ll * tid;
        unsigned long long c4[4], m4[4];
        unsigned long long c = 0, m = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool mine = (r + k) < row_hi && idx[r + k] == d;
            c4[k] = mine ? static_cast<unsigned long long>(req_core[r + k]) : 0ull;
            m4[k] = mine ? static_cast<unsigned long long>(req_mem[r + k]) : 0ull;
            c += c4[k];
            m += m4[k];
        }
        unsigned long long tot_c, tot_m;
        block_scan2<T>(c, m, sh, tot_c, tot_m);
        unsigned long long pc = base_c + c, pm = base_m + m;  // demand before this thread's first row
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if ((r + k) < row_hi && idx[r + k] == d) {
                // monotone demand: exactly one row fits before it and not with it - the cut
                if ((pc + c4[k] > cap_c || pm + m4[k] > cap_m) && pc <= cap_c && pm <= cap_m) {
                    sCutRow = r + k;
                    sComC = pc;
                    sComM = pm;
                }
                pc += c4[k];
                pm += m4[k];
            }
        }
        __syncthreads();
        if (sCutRow < R) break;
        base_c += tot_c;
        base_m += tot_m;
    }
    __syncthreads();
    if (tid == 0) {
        out->cut[d] = sCutRow;
        out->committed_c[d] = static_cast<long long>((sCutRow < R ? sComC : base_c) - pre_c);
        out->committed_m[d] = static_cast<long long>((sCutRow < R ? sComM : base_m) - pre_m);
    }
}

__global__ void __launch_bounds__(256)
prefix_apply_kernel(const PrefixOut* __restrict__ pf, int D, long long R, int32_t* __restrict__ idx) {
    __shared__ long long sCut[kMaxD];
    if (threadIdx.x < kMaxD) sCut[threadIdx.x] = threadIdx.x < D ? pf->cut[threadIdx.x] : 0;
    __syncthreads();
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; r < R; r += stride) {
        const int32_t i = idx[r];
        if (i >= 0 && r >= sCut[i]) idx[r] = -2;
    }
}

__global__ void __launch_bounds__(kMaxD)
prefix_finalize_kernel(DevState* __restrict__ st, const PrefixOut* __restrict__ pf, long long* __restrict__ delta_out,
                       int32_t* __restrict__ table_out, int commit) {
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    const int D = st->D;
    const int d = threadIdx.x;
    if (d < D) {
        const long long dc = pf->committed_c[d], dm = pf->committed_m[d];
        const long long nc = static_cast<long long>(st->free_core[d]) - dc;  // >= 0 by construction
        const long long nm = static_cast<long long>(st->free_mem[d]) - dm;
        if (delta_out) {
            delta_out[d] = dc;
            delta_out[D + d] = dm;
        }
        if (table_out) {
            table_out[d] = static_cast<int32_t>(nc);
            table_out[D + d] = static_cast<int32_t>(nm);
            table_out[2 * D + d] = 0;
        }
        if (commit) {
            st->free_core[d] = static_cast<int32_t>(nc);
            st->free_mem[d] = static_cast<int32_t>(nm);
            sFc[d] = static_cast<int32_t>(nc);
            sFm[d] = static_cast<int32_t>(nm);
        }
    }
    if (commit) resort_table_cta(st, D, sFc, sFm, sPosDev, d);
}

// Prefix-commit across GPUs (spec 2.5 "rank-major across shards").  The global row order is
// rank 0's shard, then rank 1's, ...; the scan of every rank has pushed its UNCAPPED demand
// vector of exchange step `step` to every peer (epilogue_publish).  This kernel waits for
// them in this rank's own buffer and leaves base[d] = demand of the ranks below this one:
// what is already on the running sums when this shard's first row is considered.  One CTA.
__global__ void __launch_bounds__(kMaxD)
prefix_base_kernel(DevState* __restrict__ st, unsigned long long step_plus1, long long* __restrict__ base /* [2][kMaxD] */) {
    __shared__ int sOk;
    const int D = st->D;
    const int d = threadIdx.x;
    const int world = st->peer.world, me = st->peer.rank;
    XchgRow* rows = st->peer.buf[me]->slot[(step_plus1 - 1) % kXchgSlots];
    if (d == 0) sOk = 1;
    __syncthreads();
    long long bc = 0, bm = 0;
    // waits for all ranks (every vector is consumed), sums the lower ones
    if (d < D && !xchg_pull(rows, world, step_plus1, d, D, 0, me, bc, bm)) sOk = 0;
    __syncthreads();
    if (!sOk) {  // a rank died: defer everything here (base beyond any capacity) and record it
        if (d == 0) st->peer_timeout = step_plus1;
        base[d] = 1ll << 40;
        base[kMaxD + d] = 1ll << 40;
        return;
    }
    base[d] = bc;
    base[kMaxD + d] = bm;
}

// This rank's COMMITTED demand (after the cut) to every peer as exchange step `step`;
// apply_peers_kernel of that step then makes table' = table - sum over ranks.  One CTA.
__global__ void __launch_bounds__(kMaxD)
prefix_push_kernel(DevState* __restrict__ st, const PrefixOut* __restrict__ pf, unsigned long long step_plus1,
                   long long* __restrict__ delta_out) {
    const int D = st->D;
    const int d = threadIdx.x;
    if (d < D) {
        const long long dc = pf->committed_c[d], dm = pf->committed_m[d];
        if (delta_out) {
            delta_out[d] = dc;
            delta_out[D + d] = dm;
        }
        xchg_push(st, step_plus1, d, D, dc, dm);
    }
}

// =============================================================================
// Multi-round retry of the deferred rows (spec 2.5, "rounds"): order-preserving compaction
// =============================================================================
//
// After a committing prefix-commit round the rows marked -2 are re-submitted, in their
// original order, against the table that round committed.  These kernels gather them into
// dense arrays (with the index of the caller's row each one came from) and write a later
// round's results back.  Tiles of 1024 rows, 4 consecutive rows per thread, so positions
// inside a tile follow the row order.
constexpr int kCompactTile = 1024;

__global__ void __launch_bounds__(256)
deferred_count_kernel(const int32_t* __restrict__ idx, long long n, unsigned int* __restrict__ tile_count) {
    __shared__ unsigned int sWarp[8];
    const long long r0 = static_cast<long long>(blockIdx.x) * kCompactTile + 4ll * threadIdx.x;
    unsigned int c = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) c += (r0 + k < n && idx[r0 + k] == -2) ? 1u : 0u;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) sWarp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
        for (int w = 0; w < 8; ++w) t += sWarp[w];
        tile_count[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts in place; one CTA walks them 1024 at a time
__global__ void __launch_bounds__(1024)
deferred_scan_kernel(unsigned int* __restrict__ tile_count, long long n_tiles, unsigned long long* __restrict__ total) {
    __shared__ unsigned int sWarp[32];
    __shared__ unsigned int sCarry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) sCarry = 0;
    __syncthreads();
    for (long long t0 = 0; t0 < n_tiles; t0 += 1024) {
        const long long t = t0 + threadIdx.x;
        const unsigned int own = t < n_tiles ? tile_count[t] : 0u;
        unsigned int x = own;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) sWarp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            unsigned int w = sWarp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            sWarp[lane] = w;  // inclusive over warps
        }
        __syncthreads();
        const unsigned int before = sCarry + (warp ? sWarp[warp - 1] : 0u) + x - own;
        if (t < n_tiles) tile_count[t] = before;
        __syncthreads();
        if (threadIdx.x == 0) sCarry += sWarp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = sCarry;
}

__global__ void __launch_bounds__(256)
deferred_scatter_kernel(const int32_t* __restrict__ idx, const int32_t* __restrict__ rc, const int32_t* __restrict__ rm,
                        const int32_t* __restrict__ map /* nullptr: the rows are the caller's own */, long long n,
                        const unsigned int* __restrict__ tile_off, int32_t* __restrict__ out_rc, int32_t* __restrict__ out_rm,
                        int32_t* __restrict__ out_map) {
    __shared__ unsigned int sWarp[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long r0 = static_cast<long long>(blockIdx.x) * kCompactTile + 4ll * threadIdx.x;
    bool f[4];
    unsigned int c = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        f[k] = r0 + k < n && idx[r0 + k] == -2;
        c += f[k] ? 1u : 0u;
    }
    unsigned int x = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sWarp[warp] = x;
    __syncthreads();
    unsigned int pos = tile_off[blockIdx.x] + x - c;
    for (int w = 0; w < warp; ++w) pos += sWarp[w];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (f[k]) {
            out_rc[pos] = rc[r0 + k];
            out_rm[pos] = rm[r0 + k];
            out_map[pos] = map ? map[r0 + k] : static_cast<int32_t>(r0 + k);
            ++pos;
        }
    }
}

// a later round's answers (device, -1 or still -2) back to the caller's rows
__global__ void __launch_bounds__(256)
round_writeback_kernel(const int32_t* __restrict__ idx_k, const int32_t* __restrict__ map, long long n,
                       int32_t* __restrict__ out_idx) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) out_idx[map[i]] = idx_k[i];
}

}  // namespace egpu
