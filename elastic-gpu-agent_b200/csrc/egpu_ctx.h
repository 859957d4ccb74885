// egpu_ctx.h — the context behind the opaque egpu_ctx* of include/egpu_alloc.h, shared by
// the translation units of the library (egpu_alloc.cu, egpu_devhash.cu).  Internal.
#pragma once
#include <cstdint>
#include <cstdio>
#include <mutex>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/egpu_alloc.h"
#include "egpu_kernels.cuh"

using namespace egpu;  // internal header: the context is made of the kernels' types

// The scans by launch shape: one batch (the register and grid scans ignore the lookup tables),
// several batches in one grid, the packed wire format.
using SingleFn = void (*)(DevState*, const int32_t*, const int32_t*, long long, int32_t*, long long*, int32_t*, int,
                          unsigned long long, const DevLut*, unsigned long long*);
using MultiFn = void (*)(DevState*, const MultiArgs, int, int, unsigned int, unsigned long long, const DevLut*);
using PackedFn = void (*)(DevState*, const uint32_t*, long long, signed char*, long long*, int32_t*, int, unsigned long long);
// whole-card requests (cards_scan_kernel): one batch, indices and optional card masks
using CardsFn = void (*)(DevState*, const int32_t*, const int32_t*, long long, int32_t*, unsigned long long*, long long*,
                         int32_t*, int, unsigned long long);

template <class Fn>
struct ScanKernel {
    Fn fn = nullptr;
    int threads = 0;
    size_t smem = 0;
    int ctas_per_sm = 0;  // 0 = not configured yet on this context
};

enum ScanForm { kSorted, kGrid, kLut, kSortedContig, kLutContig, kSingleForms };
constexpr int kDBuckets = 4;  // D <= 8, 16, 32, 64

struct egpu_ctx {
    std::mutex mu;
    // every scan kernel by form and D bucket (egpu_ctx_create fills them, first use configures them)
    ScanKernel<SingleFn> single[kSingleForms][kDBuckets];
    ScanKernel<MultiFn> multi[2][kDBuckets];  // [0 = register scan, 1 = lookup scan]
    ScanKernel<PackedFn> packed[kDBuckets];
    ScanKernel<CardsFn> cards[kDBuckets];
    void* h_qtable = nullptr;         // pinned host image of that table (the part of DevState before `peer`)
    DevState* d_qstate = nullptr;     // scratch table of egpu_bestfit_query (the context's own table is not touched)
    unsigned long long* h_gate = nullptr;      // pinned: start gates the host has opened (egpu_peer_gate_open)
    unsigned long long* h_gate_dev = nullptr;  // its device-visible alias
    unsigned long long* d_tile_sums = nullptr;  // prefix-commit: per-tile per-device sums [tiles][2*64]
    int64_t tile_cap = 0;
    void* d_prefix_out = nullptr;     // PrefixOut
    void* d_rounds = nullptr;         // scratch of egpu_bestfit_batch_rounds (grow-only)
    size_t rounds_bytes = 0;
    DevLut* d_lut = nullptr;
    XchgBuf* d_xchg = nullptr;        // this rank's exchange buffer (exported to the peers over CUDA IPC)
    void* peer_open[kMaxRanks] = {};  // peers' buffers as opened here (nullptr for own rank)
    int world = 1, rank = 0;
    bool attached = false;
    bool lut_dirty = true;            // table changed since the lookup tables were built
    int dev = -1;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    DevState* d_state = nullptr;
    bool has_table = false;
    int D = 0;
    int variant = EGPU_VARIANT_AUTO;
    int64_t launches = 0;
    // staging for the host-buffer entry points
    int32_t* d_req_core = nullptr;
    int32_t* d_req_mem = nullptr;
    int32_t* d_idx = nullptr;
    int64_t d_cap_rows = 0;
    long long* d_delta = nullptr;     // int64[2*64]
    int32_t* d_table_out = nullptr;   // int32[3*64]
    long long* h_delta = nullptr;     // pinned
    long long* h_delta_dev = nullptr; // its device-visible alias
    int32_t* h_table = nullptr;       // pinned int32[3*64]
    unsigned long long* d_cards = nullptr;  // card masks of egpu_bestfit_cards (grow-only)
    int64_t d_cards_cap = 0;
    bool replay_configured = false;   // shared-memory opt-in of the replay kernels done
    // bookkeeping for programmatic dependent launch (see pdl_flags)
    bool prev_is_scan = false;        // the last kernel this context launched was a snapshot scan ...
    bool prev_changes_table = false;  // ... and it may rewrite the table (commit)
    cudaStream_t prev_stream = nullptr;
    uint64_t seq = 0;                 // scans launched (epilogue slot = seq mod kEpiSlots)
    int group_len = 0;                // launches since (and including) the last fully ordered one
    int group_mbatches = 0;           // ... and the epi_multi slots (batches of multi-batch launches) they hold
    uint64_t mseq = 0;                // batches launched through multi-batch launches (slot = mseq mod kMultiSlots)
    struct Range { uintptr_t lo, hi; };
    std::vector<Range> inflight;      // output ranges of those launches, sorted by address, pairwise disjoint
    std::vector<Range> range_tmp;
    Range multi_ranges[3 * kMultiMax];  // scratch of launch_multi
    bool replay2_configured = false;
    bool sort_sets_configured = false;  // sort_sets_smem_kernel may use 128 KB of dynamic shared memory
    // grow-only device arena for multi-kernel host-buffer pipelines (egpu_devhash.cu)
    void* arena = nullptr;
    size_t arena_cap = 0;
    char last_err[256] = {0};
};

inline int cuda_fail(egpu_ctx* ctx, cudaError_t e, const char* what) {
    if (ctx) std::snprintf(ctx->last_err, sizeof ctx->last_err, "%s: %s", what, cudaGetErrorString(e));
    (void)cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? EGPU_ERR_NOMEM : EGPU_ERR_CUDA;
}

// egpu_alloc.cu: body of egpu_table_set for callers that already hold ctx->mu
int egpu_table_set_locked(egpu_ctx* ctx, const int32_t* free_core, const int32_t* free_mem, int32_t D);

#define EGPU_CUDA(ctx, call)                                   \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); \
    } while (0)
