// egpu_kernels.cuh — sm_100a kernels of the best-fit allocation path.
//
// Everything here is integer compare / subtract / min over int32 arrays that
// stream through HBM once: 12 algorithmic bytes per decision (two int32 in,
// one int32 out).  No tensor cores: nothing in this path is a contraction.
//
// Layout in HBM (DESIGN.md §3):
//   req_core[R], req_mem[R]  int32, SoA, 16-byte aligned  (read once, 128-bit)
//   out_idx[R]               int32, 16-byte aligned       (written once, 128-bit)
//   DevState                 ~170 KB: table (free_core, free_mem, oversub), its sorted
//                            view, epilogue slots (running int64 demand sums + arrival
//                            ticket per launch / per batch), peer configuration
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace egpu {

constexpr int kMaxD = 64;
constexpr int kCoreMax = 100;
constexpr int kMemMax = (1 << 18) - 1;

// --- packed compare word (internal; the spec's key is (lc, lm, d)) -----------
//   bit 31      guard C (1)
//   bits 24..30 free_core          (7 bits, <= 100)
//   bit 23      guard M (1)
//   bits 5..22  free_mem           (18 bits)
//   bits 0..4   sorted position mod 32
// K - Q with Q = core << 24 | mem << 5 keeps both guards iff core <= free_core and
// mem <= free_mem: each field borrows from its own guard only (|difference| < field
// range), and Q's low five bits are zero, so the position rides through the subtract.
// One subtract tests both dimensions; (t ^ G) & (G | 31) is then the position when the
// row is feasible and a value >= 2^23 when it is not - ready for an unsigned min.
constexpr uint32_t kGuardC = 1u << 31;
constexpr uint32_t kGuardM = 1u << 23;
constexpr uint32_t kGuards = kGuardC | kGuardM;
constexpr uint32_t kCandMask = kGuards | 31u;
constexpr uint32_t kNoCand = 32u;  // "no feasible row" among 32 positions
// Rows past D: guard C alone.  2^31 - Q keeps bit 31 only for Q = 0, and then guard M is
// missing; any other Q clears bit 31.  Never feasible, whatever the request.
constexpr uint32_t kPadWord = kGuardC;

// flags of the snapshot kernels
constexpr int kFlagFinalize = 1;  // set on every launch: publish delta / table'.  The epilogue keeps testing it:
                                  // without the test ptxas gives the D <= 8 register scan 60 registers instead
                                  // of 48, and pipelined single launches at D = 8 run 2.56 instead of 2.36 us
                                  // per step (B200, 1000 W)
constexpr int kFlagCommit = 2;    // table' replaces the table
constexpr int kFlagLateWait = 4;  // programmatic dependent launch: this launch shares nothing
                                  // with the launches in flight before it, so it triggers its
                                  // successor at once and waits for its predecessor only
                                  // before it exits (stream order is kept, nothing else)

constexpr int kFlagBoundary = 16;     // with kFlagLateWait: group boundary of a pipelined stream - scan
                                      // alongside the predecessors, but wait for them BEFORE the epilogue
                                      // and only then trigger: everything older is complete when the next
                                      // group starts, which bounds the launches in flight
constexpr int kFlagApplyNow = 32;     // multi-batch sharded launches: the CTAs that finish a batch's sums also apply that batch's exchange step
constexpr int kFlagEarlyTrigger = 8;  // griddepcontrol.launch_dependents before the scan: only on
                                      // streams the caller declared pipelined (EGPU_F_INPUTS_READY)

// lane-private demand accumulators pack (core sum << 38 | mem sum) in 64 bits
constexpr int kAccShift = 38;

// Multi-GPU exchange of demand vectors through peer memory (DESIGN.md §5).  Every rank owns
// one XchgBuf (kXchgSlots slots); rank r's demand vector of step s lands in slot s % kXchgSlots, row r, of EVERY
// rank's buffer (plain stores over NVLink).  Flag-in-data: every 8-byte word carries 32 bits of
// payload and a 32-bit tag derived from the step (8-byte stores are single-copy atomic), so the
// receiver polls the words themselves - no separate flag, no release fence, one NVLink one-way
// latency from the sender's last store to the receiver seeing a complete vector.  (Round 1 wrote
// the vector, fenced at system scope and then raised a flag: a fence round trip more.)
constexpr int kMaxRanks = 8;
constexpr int kXchgSlots = 256;  // 4 MB per rank; a rank's scans may run kXchgSlots / 2 steps ahead of its applies
struct XchgRow {
    // value j (core sums 0..D-1, mem sums D..2D-1) = two words: ll[2j] low half, ll[2j+1] high half,
    // each  tag << 32 | half
    unsigned long long ll[2 * 2 * kMaxD];
};
__host__ __device__ __forceinline__ uint32_t xchg_tag(unsigned long long step_plus1) {
    // non-zero (a consumed word is 0), and two uses of one slot (steps 256 apart) never share a tag
    return static_cast<uint32_t>(step_plus1) | 1u;
}
struct XchgBuf {
    XchgRow slot[kXchgSlots][kMaxRanks];
    // start gate (egpu_peer_gate_dev): rank r stores its gate epoch into ready[r] of EVERY rank's buffer
    unsigned long long ready[kMaxRanks];
};
struct PeerCfg {
    XchgBuf* buf[kMaxRanks];  // device-visible address of every rank's buffer ([rank] = own)
    int32_t world, rank;
};

constexpr int kEpiSlots = 32;      // DevState::epi, the ring of single-batch launches
constexpr int kMultiSlots = 128;   // DevState::epi_multi
constexpr int kMultiMax = 64;      // batches per multi-batch launch (descriptors travel as kernel parameters)

struct DevState {
    int32_t free_core[kMaxD];
    int32_t free_mem[kMaxD];
    int32_t oversub[kMaxD];
    // derived, refreshed whenever the table changes: rows sorted by (fc, fm, d)
    uint32_t sorted_k[kMaxD];             // packed compare words, kPadWord past D
    int32_t sorted_dev[kMaxD];            // sorted position -> device, -1 past D
    unsigned long long dev_packed;        // D <= 8: byte j = device at position j (0xff = none)
    int32_t D;
    uint32_t pad_;
    // kGuards and kCandMask, read at run time: as compile-time constants ptxas emits two
    // LOP3 with one immediate each; from registers (t ^ G) & M is a single 3-input LOP3
    uint32_t cand_xor, cand_mask, pad2_[2];
    PeerCfg peer;                         // set by egpu_peer_attach
    unsigned long long peer_timeout;      // step + 1 of the last apply that gave up waiting, else 0
    // Epilogue state is per launch (slot = launch sequence mod kEpiSlots): several scans may
    // be in flight at once and each needs its own running sums and arrival ticket.
    struct EpiSlot {
        unsigned long long acc[2 * kMaxD];  // running batch sums: core[0..63], mem[64..127]
        unsigned int ticket;
        unsigned int pad_[3];
        unsigned int pair[kMaxD];           // plain-snapshot epilogue: the two finishers of a device meet here
    } epi[kEpiSlots];
    // Multi-batch launches (egpu_bestfit_batches_dev): one slot per BATCH, taken from this ring in
    // launch order; a launch group (see launch_multi) never holds more than half of it.
    EpiSlot epi_multi[kMultiSlots];
    unsigned long long gate_epoch;        // start gates passed so far (egpu_peer_gate_dev)
    unsigned long long gate_timeouts;     // ... of which gave up waiting (~2 s) for the host or a peer
};

// One batch of a multi-batch launch: the arguments of egpu_bestfit_batch_dev, per batch.
// plain-snapshot epilogue: bits 49..63 of a running sum count the CTAs that have added to it
constexpr int kEpiTicketShift = 49;

struct BatchDesc {
    const int32_t* rc;
    const int32_t* rm;
    int32_t* idx;
    long long* delta;     // int64[2*D] or nullptr
    int32_t* table_out;   // int32[3*D] or nullptr
    long long R;
};
struct MultiArgs {
    BatchDesc b[kMultiMax];
};
static_assert(sizeof(MultiArgs) <= 3072, "descriptors + the scalar arguments must fit the 4 KB kernel-parameter space");

// Lookup form of the sorted table, for large D (DESIGN.md §4.1b).  With rows sorted by
// (fc, fm, d) the best fit of (c, m) is the first position j >= start[c] whose
// fm_j >= m.  Let V be the distinct fm values in ascending order and rank(m) = #V < m;
// then fm_j >= m  <=>  ridx_j >= rank(m)  (ridx_j = #V < fm_j), so the answer is a pure
// table lookup  a2[c][rank(m)]  (device id, 0xFF = none; a2[c] = the row of position start[c]).
// rank(m) comes from a bucket table over m >> 6.  Entry = lo << 8 | t:
//   lo = #V below the bucket (0..64);  t = (threshold & 63) + 1 when exactly one value of V
//   lies in the bucket, 64 when none (so  (m & 63) >= t  is  "threshold < m").  When several
//   values of V share a bucket (at most 32 buckets can be like that) bit 15 is set and bits
//   8..14 name a 64-byte block of ovf[]: ovf[block][m & 63] is rank(m) itself.  One predicated
//   extra read for those requests, no loop and no divergent region in the scan.
constexpr int kLutStride = kMaxD + 1;
constexpr int kLutBuckets = (1 << 18 >> 6) + 1;  // last bucket: mem clamped to 2^18 = out of domain
constexpr int kLutCRows = kCoreMax + 2;          // c = 0..100, and 101 = "core out of domain" (all 0xFF)
constexpr uint32_t kLutMulti = 0x80u;
struct DevLut {
    uint16_t bucket[kLutBuckets + 7];
    uint8_t a2[kLutCRows * kLutStride + 10];
    uint8_t ovf[(kMaxD / 2) * 64];
    uint32_t v[kMaxD + 4];  // ascending distinct fm values, 0xFFFFFFFF past nv (kept for inspection; the scan does not read it)
    int32_t nv;
    int32_t pad_[3];
};
static_assert(sizeof(DevLut) % 16 == 0, "DevLut is copied with 128-bit loads");

__host__ __device__ __forceinline__ uint32_t pack_table_word(int32_t fc, int32_t fm) {
    return kGuardC | (static_cast<uint32_t>(fc) << 24) | kGuardM | (static_cast<uint32_t>(fm) << 5);
}

__device__ __forceinline__ uint32_t pack_request_word(int32_t core, int32_t mem) {
    // out-of-domain values clamp to "infeasible everywhere": a negative int is a huge
    // unsigned; core 127 exceeds every free_core (<= 100); mem 2^18 clears guard M of
    // every table word (2^18 + free_mem - 2^18 < 2^18) without touching the core field
    const uint32_t c = min(static_cast<uint32_t>(core), 127u);
    const uint32_t m = min(static_cast<uint32_t>(mem), 1u << 18);
    return (c << 24) + (m << 5);
}

// streaming 128-bit accesses: read-once / write-once data stays out of L1
__device__ __forceinline__ int4 ld_stream_v4(const int32_t* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ int4 ld_stream_v4(const int4* p) { return ld_stream_v4(reinterpret_cast<const int32_t*>(p)); }
__device__ __forceinline__ void st_stream_v4(int32_t* p, const int4& v);
__device__ __forceinline__ void st_stream_v4(int4* p, const int4& v) { st_stream_v4(reinterpret_cast<int32_t*>(p), v); }
__device__ __forceinline__ void st_stream_v4(int32_t* p, const int4& v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
                 "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}

// programmatic dependent launch (PDL): the next launch in the stream may start
// once every CTA of this one has executed the trigger; `wait` blocks until the
// previous launch has completed and its writes are visible.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

__device__ __forceinline__ int32_t sat_i32(long long v) {
    return v > 2147483647LL ? 2147483647 : (v < -2147483648LL ? static_cast<int32_t>(-2147483648LL) : static_cast<int32_t>(v));
}

}  // namespace egpu
