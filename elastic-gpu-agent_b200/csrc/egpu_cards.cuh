// egpu_cards.cuh — whole-card requests (spec 2.8): core = 100 k with 2 <= k <= 64 asks for k
// cards that are entirely free, each giving (100, mem).  The snapshot scan cards_scan_kernel and
// the sequential replay_cards_kernel.  Included by egpu_alloc.cu only; see DESIGN.md §2.8, §4.1f.
#pragma once
#include "egpu_scan.cuh"

namespace egpu {

// Cards a request asks for, and the core each of them gives.  Whole-card requests score as
// (100, mem); any other core > 100 keeps its core, which pack_request_word clamps to
// "infeasible everywhere", and k = 1.
__device__ __forceinline__ int cards_k(int32_t core, int32_t& per_core) {
    const bool whole = core > kCoreMax && core <= kCoreMax * kMaxD && core % kCoreMax == 0;
    per_core = whole ? kCoreMax : core;
    return whole ? core / kCoreMax : 1;
}

// Why a whole-card row costs the scan what a single-card row does.  With the table sorted by
// (fc, fm, d), every row feasible for (100, mem) has fc = 100, the largest value there is: the
// feasible rows are a suffix of the sorted order, and the best fit p = first_feasible is where it
// starts.  The k best whole cards are then sorted positions [p, p + k), feasible iff p + k <= D,
// which is also what k sequential best-fit picks of (100, mem) give.  A single-card row is the
// case k = 1.  So a row is one first_feasible, one compare, and its demand lands on a run of
// positions: +w at p and -w at p + k in lane-private sums BY POSITION (two unconditional adds; an
// infeasible row adds and subtracts w on the discard row DT), which the epilogue turns into
// per-device sums with a running sum over positions.  Its card mask is pm[p + k] ^ pm[p], pm
// being the prefix-OR of the card bits over sorted positions.
template <int DT, int THREADS>
struct CardsSmem {
    SnapSmem<DT, THREADS> snap;                   // hist rows are sorted positions 0..DT-1 here, DT = discard
    unsigned long long pm[THREADS / 32][DT + 1];  // warp-private: pm[j] = cards at sorted positions < j
};

__device__ __forceinline__ void st_stream_v2u64(unsigned long long* p, unsigned long long x, unsigned long long y) {
    asm volatile("st.global.L1::no_allocate.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(x), "l"(y) : "memory");
}

// The register scan of whole-card rows by one CTA (single-batch launches: the grid's CTAs are the
// tiles, vectors dealt round-robin).  The request stream is that of sorted_scan_rows.  out_cards
// may be nullptr: then no mask is looked up or stored.  Returns D.
template <int DT, int THREADS>
__device__ __forceinline__ int cards_scan_rows(CardsSmem<DT, THREADS>& cs, DevState* __restrict__ st,
                                               const int32_t* __restrict__ req_core, const int32_t* __restrict__ req_mem,
                                               long long R, int32_t* __restrict__ out_idx,
                                               unsigned long long* __restrict__ out_cards) {
    SnapSmem<DT, THREADS>& s = cs.snap;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int4* __restrict__ vc = reinterpret_cast<const int4*>(req_core);
    const int4* __restrict__ vm = reinterpret_cast<const int4*>(req_mem);
    int4* __restrict__ vo = reinterpret_cast<int4*>(out_idx);
    const int nvec = static_cast<int>(R >> 2);
    const int stride = static_cast<int>(gridDim.x) * THREADS;
    int v = static_cast<int>(blockIdx.x) * THREADS + tid;

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

    const int D = st->D;
    uint32_t K[DT];
#pragma unroll
    for (int j = 0; j < DT; j += 4) {
        const uint4 k4 = *reinterpret_cast<const uint4*>(&st->sorted_k[j]);
        K[j] = k4.x; K[j + 1] = k4.y; K[j + 2] = k4.z; K[j + 3] = k4.w;
    }
    const uint32_t gx = st->cand_xor, gm = st->cand_mask;
    // position -> device, -1 from DT on (first_feasible's "none" is DT or 32, the discard row DT)
    int32_t* tile = s.sDevTile[warp];
    for (int j = lane; j < kDevTile; j += 32) tile[j] = j < DT ? st->sorted_dev[j] : -1;
#pragma unroll
    for (int j = 0; j <= DT; ++j) s.hist[warp][j][lane] = 0ull;
    __syncwarp();
    unsigned long long* pm = cs.pm[warp];
    if (out_cards) {  // prefix-OR of the card bits over positions: two 32-position halves, five shuffle steps each
        const int32_t d0 = tile[lane], d1 = tile[lane + 32];
        unsigned long long x0 = d0 >= 0 ? 1ull << d0 : 0ull, x1 = d1 >= 0 ? 1ull << d1 : 0ull;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y0 = __shfl_up_sync(0xffffffffu, x0, o), y1 = __shfl_up_sync(0xffffffffu, x1, o);
            if (lane >= o) {
                x0 |= y0;
                x1 |= y1;
            }
        }
        const unsigned long long lo_all = __shfl_sync(0xffffffffu, x0, 31);
        if (lane == 0) pm[0] = 0ull;
        if (lane + 1 <= DT) pm[lane + 1] = x0;
        if (lane + 33 <= DT) pm[lane + 33] = lo_all | x1;
        __syncwarp();
    }

    auto decide = [&](int32_t core, int32_t mem, unsigned long long& cards) -> int32_t {
        int32_t pc;
        const int k = cards_k(core, pc);
        const int p = static_cast<int>(first_feasible<DT>(K, pack_request_word(pc, mem), gx, gm));
        const bool ok = p + k <= D;
        const int lo = ok ? p : DT, hi = ok ? p + k : DT;
        const unsigned long long w = (static_cast<unsigned long long>(static_cast<uint32_t>(pc)) << kAccShift) |
                                     static_cast<unsigned long long>(static_cast<uint32_t>(mem));
        s.hist[warp][lo][lane] += w;
        s.hist[warp][hi][lane] -= w;
        if (out_cards) cards = pm[hi] ^ pm[lo];
        return tile[lo];
    };
    auto vec = [&](int vi, const int4& c, const int4& m) {
        int4 r;
        unsigned long long k0 = 0, k1 = 0, k2 = 0, k3 = 0;
        r.x = decide(c.x, m.x, k0);
        r.y = decide(c.y, m.y, k1);
        r.z = decide(c.z, m.z, k2);
        r.w = decide(c.w, m.w, k3);
        st_stream_v4(vo + vi, r);
        if (out_cards) {
            st_stream_v2u64(out_cards + 4ll * vi, k0, k1);
            st_stream_v2u64(out_cards + 4ll * vi + 2, k2, k3);
        }
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
        vec(v, c0, m0);
        if (has1) vec(v + stride, c1, m1);
        v = vn;
        has0 = nhas0;
        has1 = nhas1;
        c0 = nc0; m0 = nm0; c1 = nc1; m1 = nm1;
    }
    if (blockIdx.x == 0 && tid < static_cast<int>(R & 3)) {
        const long long r = ((R >> 2) << 2) + tid;
        unsigned long long cards = 0;
        out_idx[r] = decide(req_core[r], req_mem[r], cards);
        if (out_cards) out_cards[r] = cards;
    }
    return D;
}

// Per-position sums -> per-device sums (a running sum over positions, per lane), then the shared
// epilogue.  What reaches the epilogue's atomics is per device and non-negative: a row adds at most
// (100, 2^18 - 1) to any one device, so the arrival count in bits 49..63 stays clear.
template <int DT, int THREADS>
__device__ __forceinline__ void cards_epilogue(CardsSmem<DT, THREADS>& cs, DevState* st, int D, long long* __restrict__ delta_out,
                                               int32_t* __restrict__ table_out, int flags, const EpiCtl& ec) {
    SnapSmem<DT, THREADS>& s = cs.snap;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int32_t* tile = s.sDevTile[warp];
    __syncwarp();
    unsigned long long run = 0;
    for (int j = 0; j < D; ++j) {
        run += s.hist[warp][j][lane];
        const uint32_t c = static_cast<uint32_t>(run >> kAccShift);
        const uint32_t ml = static_cast<uint32_t>(run) & 0x7FFFFu;
        const uint32_t mh = static_cast<uint32_t>(run >> 19) & 0x7FFFFu;
        const uint32_t sc = __reduce_add_sync(0xffffffffu, c);
        const uint32_t sl = __reduce_add_sync(0xffffffffu, ml);
        const uint32_t sh = __reduce_add_sync(0xffffffffu, mh);
        if (lane == 0) {
            const int d = tile[j];
            s.sWarpAcc[warp][d] = sc;
            s.sWarpAcc[warp][DT + d] = static_cast<unsigned long long>(sl) + (static_cast<unsigned long long>(sh) << 19);
        }
    }
    __syncthreads();
    epilogue_publish<THREADS / 32>(&s.sWarpAcc[0][0], 2 * DT, 0, DT, s.sFc, s.sFm, s.sPosDev, &s.sLast, st, D, delta_out,
                                   table_out, flags, ec);
}

// Snapshot scan with whole-card rows (egpu_bestfit_cards[_dev]).  Same launch protocol as
// bestfit_sorted_kernel (PDL flags, epilogue slot word); the register form for every D bucket.
template <int DT, int THREADS>
__global__ void __launch_bounds__(THREADS)
cards_scan_kernel(DevState* __restrict__ st, const int32_t* __restrict__ req_core, const int32_t* __restrict__ req_mem,
                  long long R, int32_t* __restrict__ out_idx, unsigned long long* __restrict__ out_cards,
                  long long* __restrict__ delta_out, int32_t* __restrict__ table_out, int flags, unsigned long long slot_step) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    auto& cs = *reinterpret_cast<CardsSmem<DT, THREADS>*>(smem_raw);
    const bool late = (flags & kFlagLateWait) != 0;
    const bool boundary = (flags & kFlagBoundary) != 0;
    if (!late) pdl_wait();
    if ((flags & kFlagEarlyTrigger) && !boundary) pdl_trigger();
    const int D = cards_scan_rows<DT, THREADS>(cs, st, req_core, req_mem, R, out_idx, out_cards);
    if (boundary) {
        pdl_wait();
        pdl_trigger();
    }
    cards_epilogue<DT, THREADS>(cs, st, D, delta_out, table_out, flags, epi_from_word(st, slot_step));
    if (late && !boundary) pdl_wait();
}

// Sequential mode with whole-card ALLOCs, every D <= 64 and every event count: one warp, lane =
// device (two per lane when D > 32), as replay_kernel.  An ALLOC of k cards takes k successive
// CREDUX minima of the spec's key (lc, lm, d) over the feasible lanes, after one ballot has
// checked that k of them are feasible (so nothing is ever undone).  Every ALLOC records its card
// mask and first card (live_cards / live_idx, HBM, lane 0's alone: program order is their
// consistency), because a later FREE cannot recompute them from a table that has moved on.
__global__ void __launch_bounds__(32)
replay_cards_kernel(DevState* __restrict__ st, const int32_t* __restrict__ kind, const int32_t* __restrict__ ev_a,
                    const int32_t* __restrict__ ev_b, long long E, int32_t* __restrict__ out_idx,
                    unsigned long long* __restrict__ out_cards, unsigned long long* __restrict__ live_cards,
                    signed char* __restrict__ live_idx) {
    const int lane = threadIdx.x;
    const int D = st->D;
    const int d0 = lane, d1 = lane + 32;
    int32_t fc0 = d0 < D ? st->free_core[d0] : -1;
    int32_t fm0 = d0 < D ? st->free_mem[d0] : -1;
    int32_t fc1 = d1 < D ? st->free_core[d1] : -1;
    int32_t fm1 = d1 < D ? st->free_mem[d1] : -1;
    constexpr int32_t kNone = 0x7fffffff;  // above every key: lc <= 100 keeps keys below 2^31 - 2^24

    for (long long base = 0; base < E; base += 32) {
        const long long i = base + lane;
        int32_t k = -1, a = 0, b = 0, ta = 0, tb = 0;
        bool tvalid = false;
        if (i < E) {
            k = kind[i];
            a = ev_a[i];
            b = ev_b[i];
            if (k == 1 && a >= 0 && a < i) {  // gather the released event's request now
                tvalid = kind[a] == 0;
                ta = ev_a[a];
                tb = ev_b[a];
            }
        }
        int32_t my_out = -1;
        unsigned long long my_cards = 0;
        const int n = (E - base) < 32 ? static_cast<int>(E - base) : 32;
        for (int j = 0; j < n; ++j) {
            const int32_t kj = __shfl_sync(0xffffffffu, k, j);
            const int32_t aj = __shfl_sync(0xffffffffu, a, j);
            const int32_t bj = __shfl_sync(0xffffffffu, b, j);
            int32_t res = -1;
            unsigned long long cards = 0;
            if (kj == 0) {
                int32_t pc;
                const int kc = cards_k(aj, pc);
                const int32_t lc0 = fc0 - pc, lm0 = fm0 - bj;
                const int32_t lc1 = fc1 - pc, lm1 = fm1 - bj;
                const bool valid = (pc | bj) >= 0 && pc <= kCoreMax;
                const bool f0 = valid && (lc0 | lm0) >= 0 && fc0 >= 0;
                const bool f1 = valid && (lc1 | lm1) >= 0 && fc1 >= 0;
                int32_t key0 = f0 ? (lc0 << 24) | (lm0 << 6) | d0 : kNone;
                int32_t key1 = f1 ? (lc1 << 24) | (lm1 << 6) | d1 : kNone;
                const int nf = __popc(__ballot_sync(0xffffffffu, f0)) + __popc(__ballot_sync(0xffffffffu, f1));
                if (nf >= kc) {
                    bool t0 = false, t1 = false;
                    for (int c = 0; c < kc; ++c) {
                        const int32_t best = __reduce_min_sync(0xffffffffu, min(key0, key1));
                        if (c == 0) res = best & 63;
                        if (key0 == best) { t0 = true; key0 = kNone; }
                        if (key1 == best) { t1 = true; key1 = kNone; }
                    }
                    cards = static_cast<unsigned long long>(__ballot_sync(0xffffffffu, t0)) |
                            (static_cast<unsigned long long>(__ballot_sync(0xffffffffu, t1)) << 32);
                    if (t0) { fc0 -= pc; fm0 -= bj; }
                    if (t1) { fc1 -= pc; fm1 -= bj; }
                }
                if (lane == 0) {
                    live_cards[base + j] = cards;
                    live_idx[base + j] = static_cast<signed char>(res);
                }
            } else {
                const bool tv = __shfl_sync(0xffffffffu, static_cast<int>(tvalid), j) != 0;
                const int32_t taj = __shfl_sync(0xffffffffu, ta, j);
                const int32_t tbj = __shfl_sync(0xffffffffu, tb, j);
                unsigned long long held = 0;
                int32_t first = -1;
                if (lane == 0 && kj == 1 && tv) {
                    held = live_cards[aj];
                    first = live_idx[aj];
                    live_cards[aj] = 0ull;
                }
                held = __shfl_sync(0xffffffffu, held, 0);
                first = __shfl_sync(0xffffffffu, first, 0);
                if (held) {
                    int32_t pc;
                    cards_k(taj, pc);
                    if ((held >> d0) & 1ull) { fc0 += pc; fm0 += tbj; }
                    if ((held >> d1) & 1ull) { fc1 += pc; fm1 += tbj; }
                    res = first;
                    cards = held;
                }
            }
            if (lane == j) {
                my_out = res;
                my_cards = cards;
            }
        }
        if (i < E) {
            out_idx[i] = my_out;
            if (out_cards) out_cards[i] = my_cards;
        }
    }
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    if (d0 < D) { st->free_core[d0] = fc0; st->free_mem[d0] = fm0; sFc[d0] = fc0; sFm[d0] = fm0; }
    if (d1 < D) { st->free_core[d1] = fc1; st->free_mem[d1] = fm1; sFc[d1] = fc1; sFm[d1] = fm1; }
    resort_table_cta(st, D, sFc, sFm, sPosDev, lane);
}

}  // namespace egpu
