// egpu_replay.cuh — the synthetic request generator and the sequential-mode (replay)
// kernels.  Included by egpu_alloc.cu only; see DESIGN.md §4.3, §6.
#pragma once
#include "egpu_scan.cuh"  // resort_table_cta

namespace egpu {

// =============================================================================
// Synthetic request generator (same counter RNG as synth.py)
// =============================================================================
__device__ __forceinline__ unsigned long long mix64(unsigned long long seed, unsigned long long stream,
                                                    unsigned long long i) {
    unsigned long long z = seed * 0x9E3779B97F4A7C15ull + stream * 0xD1B54A32D192ED03ull + i;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ int32_t uniform_i32(unsigned long long seed, unsigned long long stream,
                                               unsigned long long i, int lo, int hi) {
    const unsigned long long z = mix64(seed, stream, i);
    const unsigned long long n = static_cast<unsigned long long>(hi - lo + 1);
    return lo + static_cast<int32_t>(((z >> 32) * n) >> 32);
}

__global__ void synth_requests_kernel(int dist, unsigned long long seed, long long first_row, long long R,
                                      int32_t* __restrict__ req_core, int32_t* __restrict__ req_mem) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; k < R; k += stride) {
        const unsigned long long r = static_cast<unsigned long long>(first_row + k);
        int32_t core, mem;
        if (dist == 2) {
            const int ci = uniform_i32(seed, 2, r, 0, 5);
            const int mi = uniform_i32(seed, 3, r, 0, 6);
            core = ci == 0 ? 5 : ci == 1 ? 10 : ci == 2 ? 20 : ci == 3 ? 25 : ci == 4 ? 50 : 100;
            mem = 256 << mi;
        } else {
            core = uniform_i32(seed, 2, r, 1, 100);
            mem = uniform_i32(seed, 3, r, 1, dist == 3 ? 65536 : 24576);
            if ((r & 15ull) == 15ull) {
                if (((r >> 4) & 1ull) == 0ull) core = 101;
                else mem = 183359 + 1;
            }
        }
        req_core[k] = core;
        req_mem[k] = mem;
    }
}

// =============================================================================
// Sequential mode: one warp, for what the two-warp kernel below does not take (D > 32, or more
// than kReplaySmemEvents events).  D <= 8: table in registers (replay8_kernel, below the general
// one); otherwise lane = device (two per lane when D > 32)
// =============================================================================
//
// Request k sees the table after k-1: a serial dependence chain, so there is no
// bandwidth roofline here — the figure of merit is cycles per event.  The warp
// loads 32 events at a time (coalesced), broadcasts them one by one with
// shuffles, scores the current table with one packed key per lane and reduces
// with CREDUX.MIN (__reduce_min_sync).  `live` (device currently held by each
// ALLOC event, -1 otherwise) sits in shared memory when it fits, else in HBM;
// only lane 0 touches it, so program order gives consistency.
constexpr int kReplaySmemEvents = 200 * 1024;

__global__ void __launch_bounds__(32)
replay_kernel(DevState* __restrict__ st, const int32_t* __restrict__ kind, const int32_t* __restrict__ ev_a,
              const int32_t* __restrict__ ev_b, long long E, int32_t* __restrict__ out_idx,
              signed char* __restrict__ live_global) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    signed char* live = (E <= kReplaySmemEvents) ? reinterpret_cast<signed char*>(smem_raw) : live_global;
    const int lane = threadIdx.x;
    const int D = st->D;
    const int d0 = lane, d1 = lane + 32;
    int32_t fc0 = d0 < D ? st->free_core[d0] : -1;
    int32_t fm0 = d0 < D ? st->free_mem[d0] : -1;
    int32_t fc1 = d1 < D ? st->free_core[d1] : -1;
    int32_t fm1 = d1 < D ? st->free_mem[d1] : -1;

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
        const int n = (E - base) < 32 ? static_cast<int>(E - base) : 32;
        for (int j = 0; j < n; ++j) {
            const int32_t kj = __shfl_sync(0xffffffffu, k, j);
            const int32_t aj = __shfl_sync(0xffffffffu, a, j);
            const int32_t bj = __shfl_sync(0xffffffffu, b, j);
            int32_t res = -1;
            if (kj == 0) {
                const int32_t lc0 = fc0 - aj, lm0 = fm0 - bj;
                const int32_t lc1 = fc1 - aj, lm1 = fm1 - bj;
                const bool valid = (aj | bj) >= 0;
                int32_t key = 0x7fffffff;
                if (valid && (lc0 | lm0) >= 0 && fc0 >= 0) key = (lc0 << 24) | (lm0 << 6) | d0;
                if (valid && (lc1 | lm1) >= 0 && fc1 >= 0) key = min(key, (lc1 << 24) | (lm1 << 6) | d1);
                const int32_t best = __reduce_min_sync(0xffffffffu, key);
                if (best != 0x7fffffff) {
                    res = best & 63;
                    if (res == d0) { fc0 -= aj; fm0 -= bj; }
                    if (res == d1) { fc1 -= aj; fm1 -= bj; }
                }
                if (lane == 0) live[base + j] = static_cast<signed char>(res);
            } else {
                const bool tv = __shfl_sync(0xffffffffu, static_cast<int>(tvalid), j) != 0;
                const int32_t taj = __shfl_sync(0xffffffffu, ta, j);
                const int32_t tbj = __shfl_sync(0xffffffffu, tb, j);
                int32_t dev = -1;
                if (lane == 0) {
                    live[base + j] = -1;
                    if (kj == 1 && tv) {
                        dev = live[aj];
                        live[aj] = -1;
                    }
                }
                dev = __shfl_sync(0xffffffffu, dev, 0);
                if (dev >= 0) {
                    if (dev == d0) { fc0 += taj; fm0 += tbj; }
                    if (dev == d1) { fc1 += taj; fm1 += tbj; }
                }
                res = dev;
            }
            if (lane == j) my_out = res;
        }
        if (i < E) out_idx[i] = my_out;
    }
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    if (d0 < D) { st->free_core[d0] = fc0; st->free_mem[d0] = fm0; sFc[d0] = fc0; sFm[d0] = fm0; }
    if (d1 < D) { st->free_core[d1] = fc1; st->free_mem[d1] = fm1; sFc[d1] = fc1; sFm[d1] = fm1; }
    resort_table_cta(st, D, sFc, sFm, sPosDev, lane);
}

// Sequential mode for D <= 8: the whole table lives in the registers of every lane as packed
// compare words (guard | free_core | guard | free_mem | device).  K[d] - Q is at once the
// feasibility test (both guards survive), the ordering key of the spec ((lc, lm, d) with the
// guards as constant top bits) and the updated table word of the chosen device — so an ALLOC
// is 8 subtracts, 8 guard tests, a 3-input-min tree and 8 selects, with no cross-lane
// traffic on the dependence chain.  All lanes compute the same thing; lane 0 keeps `live`
// and the outputs.  Events are held 32 at a time in registers (lane j = event j of the chunk),
// broadcast with shuffles; the next chunk is prefetched while the current one is processed.
__global__ void __launch_bounds__(32)
replay8_kernel(DevState* __restrict__ st, const int32_t* __restrict__ kind, const int32_t* __restrict__ ev_a,
               const int32_t* __restrict__ ev_b, long long E, int32_t* __restrict__ out_idx,
               signed char* __restrict__ live_global) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    signed char* live = (E <= kReplaySmemEvents) ? reinterpret_cast<signed char*>(smem_raw) : live_global;
    const int lane = threadIdx.x;
    const int D = st->D;
    uint32_t K[8];
#pragma unroll
    for (int d = 0; d < 8; ++d)
        K[d] = d < D ? (pack_table_word(st->free_core[d], st->free_mem[d]) | static_cast<uint32_t>(d)) : kPadWord;

    auto fetch = [&](long long i, int32_t& k, uint32_t& q, uint32_t& qt, int32_t& t) {
        k = -1; q = 0; qt = 0; t = -1;
        if (i < E) {
            k = kind[i];
            const int32_t a = ev_a[i], b = ev_b[i];
            q = pack_request_word(a, b);
            if (k == 1 && a >= 0 && a < i && kind[a] == 0) {  // FREE of an earlier ALLOC: fetch its request now
                t = a;
                qt = pack_request_word(ev_a[a], ev_b[a]);
            }
        }
    };
    int32_t nk; uint32_t nq, nqt; int32_t nt;
    fetch(lane, nk, nq, nqt, nt);
    for (long long base = 0; base < E; base += 32) {
        // this chunk's events stay in registers (lane j holds event base + j) and are broadcast
        // with shuffles, which do not sit on the dependence chain; `live` is lane 0's alone
        const int32_t ck = nk, ct = nt;
        const uint32_t cq = nq, cqt = nqt;
        fetch(base + 32 + lane, nk, nq, nqt, nt);  // prefetch the next chunk
        const int n = (E - base) < 32 ? static_cast<int>(E - base) : 32;
        int32_t my_out = -1;
#pragma unroll 4
        for (int j = 0; j < n; ++j) {
            const int32_t kj = __shfl_sync(0xffffffffu, ck, j);
            const uint32_t q = __shfl_sync(0xffffffffu, cq, j);
            int32_t res = -1;
            if (kj == 0) {
                uint32_t w[8], key[8];
#pragma unroll
                for (int d = 0; d < 8; ++d) {
                    w[d] = K[d] - q;
                    key[d] = ((w[d] & kGuards) == kGuards) ? w[d] : 0xFFFFFFFFu;
                }
                const uint32_t best = __vimin3_u32(__vimin3_u32(key[0], key[1], key[2]), __vimin3_u32(key[3], key[4], key[5]),
                                                   min(key[6], key[7]));
                if (best != 0xFFFFFFFFu) {
                    res = static_cast<int32_t>(best & 31u);
#pragma unroll
                    for (int d = 0; d < 8; ++d) K[d] = (w[d] == best) ? w[d] : K[d];
                }
                if (lane == 0) live[base + j] = static_cast<signed char>(res);
            } else {
                const int32_t t = __shfl_sync(0xffffffffu, ct, j);
                const uint32_t qt = __shfl_sync(0xffffffffu, cqt, j);
                int32_t dev = -1;
                if (lane == 0) {
                    live[base + j] = -1;
                    if (t >= 0) {
                        dev = live[t];
                        live[t] = -1;
                    }
                }
                dev = __shfl_sync(0xffffffffu, dev, 0);
                if (dev >= 0) {
#pragma unroll
                    for (int d = 0; d < 8; ++d) K[d] = (d == dev) ? K[d] + qt : K[d];
                    res = dev;
                }
            }
            if (lane == j) my_out = res;
        }
        if (base + lane < E) out_idx[base + lane] = my_out;
    }
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    if (lane < D) {
        uint32_t k = 0;
#pragma unroll
        for (int d = 0; d < 8; ++d) k = (d == lane) ? K[d] : k;
        const int32_t fc = static_cast<int32_t>((k >> 24) & 0x7Fu), fm = static_cast<int32_t>((k >> 5) & 0x3FFFFu);
        st->free_core[lane] = fc;
        st->free_mem[lane] = fm;
        sFc[lane] = fc;
        sFm[lane] = fm;
    }
    resort_table_cta(st, D, sFc, sFm, sPosDev, lane);
}


// Sequential mode, two warps (D <= 32, E <= kReplaySmemEvents): the serial chain alone on one warp.
// Warp 1 decodes events 256 at a time into a shared-memory ring - loads, the packed request word, and for a
// FREE the validity of its target (an earlier ALLOC) and that ALLOC's request word - and writes the previous
// chunk's results out, coalesced.  Warp 0 walks the ring with lane = device: one broadcast 128-bit read per
// event, and per ALLOC the dependent path is subtract -> guard test -> select -> CREDUX.MIN -> compare ->
// select (the chosen lane keeps K - Q, which is its updated table word); a FREE adds the request word back on
// the lane `live` names.  `live` is lane 0's alone (program order is its consistency: racecheck-clean); the
// device a FREE releases reaches the other lanes through one shuffle.  (All lanes keeping `live` redundantly -
// same address, same value - saved that shuffle, 40 against 48 ns per event, but is a formal shared-memory race
// that racecheck reports; warp barriers around a single writer: 80 ns; `if (lane == 0)` as a branch: 87 ns.)
constexpr int kReplayChunk = 256;
struct ReplayRing {
    uint4 ev[2][kReplayChunk];   // x = request word (ALLOC: its own; FREE: its target's), y = FREE target event or -1, z = kind
    int32_t res[2][kReplayChunk];
};
__global__ void __launch_bounds__(64)
replay2_kernel(DevState* __restrict__ st, const int32_t* __restrict__ kind, const int32_t* __restrict__ ev_a,
               const int32_t* __restrict__ ev_b, long long E, int32_t* __restrict__ out_idx) {
    // the ring is a static object and `live` the dynamic one: the compiler can see that ring reads never
    // alias `live` stores and hoists the next events' reads above the current event's stores
    __shared__ ReplayRing ring;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t live_base = static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw));  // `live`: int8 per event
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int D = st->D;
    uint32_t K = lane < D ? (pack_table_word(st->free_core[lane], st->free_mem[lane]) | static_cast<uint32_t>(lane)) : kPadWord;
    const long long n_chunks = (E + kReplayChunk - 1) / kReplayChunk;

    auto decode = [&](long long c) {  // warp 1
        const long long base = c * kReplayChunk;
        for (int j = lane; j < kReplayChunk; j += 32) {
            const long long i = base + j;
            uint4 e = make_uint4(0u, 0xFFFFFFFFu, 2u, 0u);  // past the end: a no-op kind
            if (i < E) {
                const int32_t k = kind[i], a = ev_a[i], b = ev_b[i];
                e.z = static_cast<uint32_t>(k);
                if (k == 0) {
                    e.x = pack_request_word(a, b);
                } else if (k == 1 && a >= 0 && a < i && kind[a] == 0) {  // FREE of an earlier ALLOC
                    e.y = static_cast<uint32_t>(a);
                    e.x = pack_request_word(ev_a[a], ev_b[a]);
                }
            }
            ring.ev[c & 1][j] = e;
        }
    };
    auto drain = [&](long long c) {  // warp 1: results of chunk c to HBM
        const long long base = c * kReplayChunk;
        for (int j = lane; j < kReplayChunk; j += 32)
            if (base + j < E) out_idx[base + j] = ring.res[c & 1][j];
    };
    if (warp == 1) decode(0);
    __syncthreads();
    for (long long c = 0; c < n_chunks; ++c) {
        if (warp == 1) {
            if (c + 1 < n_chunks) decode(c + 1);
            if (c > 0) drain(c - 1);
        } else {
            const long long base = c * kReplayChunk;
            const int n = (E - base) < kReplayChunk ? static_cast<int>(E - base) : kReplayChunk;
            const uint4* evs = ring.ev[c & 1];
            int32_t* res_out = ring.res[c & 1];
            uint4 nxt = evs[0];
#pragma unroll 4
            for (int j = 0; j < n; ++j) {
                const uint4 e = nxt;
                nxt = evs[(j + 1) & (kReplayChunk - 1)];  // one event ahead: its read latency is off the chain
                // Branch-free: one warp alone pays a pipeline refill for every taken branch, which cost more
                // than the work it skipped.  Both kinds are computed, the event's kind selects.
                const bool is_alloc = e.z == 0u;
                const int32_t t = static_cast<int32_t>(e.y);            // FREE target (an earlier ALLOC) or -1
                // `live` belongs to lane 0 alone (reads and writes in its program order: nothing to race with);
                // the device a FREE releases reaches the other lanes through one shuffle
                // (predicated instructions, not branches: a divergent region per event costs more than the event)
                const uint32_t live_t = live_base + static_cast<uint32_t>(t < 0 ? 0 : t);
                int32_t tdev0;
                asm volatile("{ .reg .pred p; setp.eq.s32 p, %1, 0; mov.s32 %0, -1; @p ld.shared.s8 %0, [%2]; }"
                             : "=r"(tdev0) : "r"(lane), "r"(live_t) : "memory");  // read before this event's stores
                const int32_t tdev_raw = __shfl_sync(0xffffffffu, tdev0, 0);
                // ALLOC: K - Q is never 0xFFFFFFFF (Q's low five bits are zero, K's hold a device < 32), so no
                // lane matches "none"; a FREE / no-op event carries INF on every lane
                const uint32_t w = K - e.x;
                const uint32_t key = (is_alloc && (~w & kGuards) == 0u) ? w : 0xFFFFFFFFu;
                const uint32_t best = __reduce_min_sync(0xffffffffu, key);
                const int32_t a_res = best == 0xFFFFFFFFu ? -1 : static_cast<int32_t>(best & 31u);
                const int32_t tdev = t >= 0 ? tdev_raw : -1;
                const int32_t res = is_alloc ? a_res : tdev;
                const uint32_t k_alloc = (w == best) ? w : K;
                const uint32_t k_free = (lane == tdev) ? K + e.x : K;
                K = is_alloc ? k_alloc : k_free;
                {
                    const int32_t mine = is_alloc ? a_res : -1;
                    asm volatile("{ .reg .pred p, q; setp.eq.s32 p, %0, 0; setp.ge.and.s32 q, %4, 0, p;\n\t"
                                 "@p st.shared.u8 [%1], %2; @q st.shared.u8 [%3], %5; }"
                                 ::"r"(lane), "r"(live_base + static_cast<uint32_t>(base + j)), "r"(mine), "r"(live_t), "r"(t), "r"(-1)
                                 : "memory");
                }
                res_out[j] = res;
            }
        }
        __syncthreads();
    }
    if (warp == 1 && n_chunks > 0) drain(n_chunks - 1);
    __shared__ int32_t sFc[kMaxD], sFm[kMaxD], sPosDev[kMaxD];
    if (warp == 0 && lane < D) {
        const int32_t fc = static_cast<int32_t>((K >> 24) & 0x7Fu), fm = static_cast<int32_t>((K >> 5) & 0x3FFFFu);
        st->free_core[lane] = fc;
        st->free_mem[lane] = fm;
        sFc[lane] = fc;
        sFm[lane] = fm;
    }
    __syncthreads();
    resort_table_cta(st, D, sFc, sFm, sPosDev, tid);
}

}  // namespace egpu
