/*
 * egpu_alloc.h — C ABI of the B200-native best-fit allocation path.
 *
 * This is the drop-in boundary: a Go DaemonSet (elastic-gpu-agent) binds these
 * symbols through cgo; nothing in the signatures is a CUDA, torch or C++ type.
 * All pointers are caller-owned and only read/written for the duration of the
 * call (cgo pointer rule) unless the name ends in `_dev`, in which case they are
 * CUDA device pointers and the call is asynchronous on the given stream.
 *
 * Reference interfaces each entry point stands behind (paths relative to the
 * reference repo elastic-ai/elastic-gpu-agent @ 2609107):
 *
 *   egpu_ctx_create / egpu_ctx_destroy
 *       constructed where the plugin is built, pkg/manager/manager.go:138
 *       (plugins.PluginFactory) and pkg/plugins/base.go:208-233.
 *   egpu_table_set
 *       the capacity table the reference derives at start-up from NVML:
 *       pkg/operator/base.go:19-75 (device count, memory bytes),
 *       pkg/plugins/gpushare.go:24-33 (100 core units per GPU),
 *       pkg/plugins/gpushare.go:159-168 (one memory unit per MiB).
 *   egpu_bestfit_batch / egpu_bestfit_batch_dev
 *       the slot of baseDevicePlugin.GetPreferredAllocation, a stub in the
 *       reference (pkg/plugins/base.go:94-96); request units follow
 *       pkg/common/const.go:4 (GPUPercentEachCard = 100) and the vendored
 *       resource names elasticgpu.io/gpu-core, elasticgpu.io/gpu-memory
 *       (vendor/elasticgpu.io/elastic-gpu/api/v1alpha1/types.go:105-112).
 *   egpu_bestfit_batches_dev / egpu_bestfit_query
 *       the same slot, for a caller with several requests' worth of batches in
 *       hand (one launch for up to 64 of them), and for the stateless what-if
 *       form GetPreferredAllocation needs (pkg/plugins/base.go:94-96: kubelet
 *       passes the available IDs of ONE admission; the node's committed table
 *       must not be touched by it).
 *   egpu_replay
 *       commits serialised under baseDevicePlugin.lock in PreStartContainer
 *       (pkg/plugins/gpushare.go:114,239) and frees issued by
 *       GPUSharePlugin.GC (pkg/plugins/base.go:241-306).
 *   egpu_preferred_allocation
 *       pluginapi.PreferredAllocationRequest/Response
 *       (vendor/k8s.io/kubelet/pkg/apis/deviceplugin/v1beta1/api.pb.go:564-571,
 *       675-677) with the device-ID format "%d-%02d" of
 *       pkg/plugins/gpushare.go:28,163.
 *   egpu_device_hash / egpu_device_hash_batch
 *       types.NewDevice + hash, pkg/types/device.go:17-25,49-54
 *       (sort.Strings, join ":", SHA-256, first 8 hex digits), used by
 *       Allocate (pkg/plugins/gpushare.go:44,179) and by
 *       KubeletDeviceLocator.Locate (pkg/kube/locator.go:62-90).
 *
 * IMPORTANT: the reference contains NO best-fit scoring loop (SURVEY.md §0);
 * the decision rule implemented here is the builder-defined specification in
 * DESIGN.md §2 ("the spec"), restated on the CPU in oracle/.
 *
 * The spec in one paragraph. D devices (1..64), free_core[d] in [0,100]
 * (percent), free_mem[d] in [0, 2^18-1] (MiB).  Request (core, mem) is feasible
 * on d iff 0 <= core <= free_core[d] and 0 <= mem <= free_mem[d].  Best fit =
 * the feasible device with the lexicographically smallest
 * (free_core[d]-core, free_mem[d]-mem, d); idx = -1 when no device is feasible.
 * Snapshot mode scores every request of a batch against the same table and
 * reports per-device demand sums (int64) and table' = table - demand
 * (saturated to int32, oversub flag when negative).  Sequential mode applies
 * each event to the table before the next one is scored.
 */
#ifndef EGPU_ALLOC_H
#define EGPU_ALLOC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EGPU_MAX_DEVICES   64
#define EGPU_CORE_MAX      100              /* pkg/common/const.go:4 */
#define EGPU_MEM_MAX       ((1 << 18) - 1)  /* MiB; B200 reports 183359 */
#define EGPU_MAX_ROWS      2147483647       /* requests per batch (R): the scans index with 32 bits */
#define EGPU_IDX_INFEASIBLE (-1)
#define EGPU_IDX_DEFERRED   (-2)            /* prefix-commit mode only */

/* return codes: 0 = OK, negative = error, never aborts the process */
#define EGPU_OK               0
#define EGPU_ERR_INVALID     (-1)   /* bad argument (NULL, range, D, sizes) */
#define EGPU_ERR_NO_DEVICE   (-2)   /* no usable CUDA device / driver */
#define EGPU_ERR_CUDA        (-3)   /* CUDA runtime error (see egpu_last_error) */
#define EGPU_ERR_NOMEM       (-4)   /* host or device allocation failed */
#define EGPU_ERR_NO_TABLE    (-5)   /* egpu_table_set has not been called */
#define EGPU_ERR_STATE       (-6)   /* call not valid in the current state */
#define EGPU_ERR_PARSE       (-7)   /* malformed device-ID string or stored record */
#define EGPU_ERR_UNSAT       (-8)   /* preferred allocation cannot be satisfied */

/* event kinds for egpu_replay */
#define EGPU_EV_ALLOC 0
#define EGPU_EV_FREE  1

/* flags of egpu_bestfit_batch_dev */
#define EGPU_F_COMMIT        1   /* table' replaces the current table */
#define EGPU_F_INPUTS_READY  2   /* the request arrays were complete before the previous
                                    launch on this stream: consecutive scans may overlap
                                    (programmatic dependent launch); anything else
                                    enqueued later on the stream still sees them
                                    complete. */

#define EGPU_F_PREFIX_COMMIT 4   /* spec 2.5: a request commits only while the running demand of
                                    its device (all earlier requests that chose it) still fits;
                                    the others get EGPU_IDX_DEFERRED, the demand sums and table'
                                    count committed requests only, so table' never goes negative.
                                    Single GPU; not with EGPU_VARIANT_GRID.  In egpu_bestfit_batch
                                    pass it in `commit` (EGPU_F_COMMIT | EGPU_F_PREFIX_COMMIT). */

#define EGPU_F_APPLY         8   /* egpu_bestfit_batches_shard_dev only: the CTAs that complete a batch's sums, having pushed the
                                    batch's demand vector, also wait for the peers' vectors of that exchange step and
                                    write table' (= table - sum over ranks) to the batch's d_table_out: no apply call,
                                    no second stream.  Never commits.  Every rank must issue the same launch; start the
                                    ranks together (egpu_peer_gate_dev) or the wait is as long as their skew. */

/* kernel variants for the snapshot scan (egpu_set_variant) */
#define EGPU_VARIANT_AUTO    0   /* SORTED for D <= 16, LUT above */
#define EGPU_VARIANT_GRID    1   /* direct (device x request) score grid, min over packed keys */
#define EGPU_VARIANT_SORTED  2   /* first feasible device in (core, mem, d)-sorted order, table in registers */
#define EGPU_VARIANT_LUT     3   /* same order, answered by shared-memory lookup tables (large D) */

typedef struct egpu_ctx egpu_ctx;

/* ---- lifetime --------------------------------------------------------- */

/* One context per CUDA device (one process per GPU).  Thread-safe: every entry
 * point takes the context mutex (mirrors baseDevicePlugin.lock) and binds the
 * CUDA device explicitly, so it may be called from any OS thread (goroutines
 * migrate).  Fails with EGPU_ERR_NO_DEVICE when there is no GPU: there is NO
 * CPU fallback in this library. */
int  egpu_ctx_create(int cuda_device, egpu_ctx** out);
void egpu_ctx_destroy(egpu_ctx* ctx);
const char* egpu_strerror(int code);
/* last error detail recorded by this context ("" if none): the failing CUDA call, or the
 * record a parse error was found in.  The pointer stays valid for the life of the context;
 * the text is overwritten by the next failing call. */
const char* egpu_last_error(egpu_ctx* ctx);
/* 1 = CUDA sm_100a path.  (0 is reserved; this library never returns it.) */
int  egpu_backend(egpu_ctx* ctx);
/* number of kernels this context has launched since creation */
int64_t egpu_launch_count(egpu_ctx* ctx);
int  egpu_set_variant(egpu_ctx* ctx, int variant);
/* ABI version: major*1000 + minor.  Minor revisions only add entry points (1.1 placement
 * restore, 1.2 prefix-commit over row shards, 1.3 rounds, 1.4 multi-batch launches, stateless query,
 * start gate, host registration); a caller built against 1.0 keeps
 * working. */
int  egpu_abi_version(void);

/* ---- capacity table --------------------------------------------------- */

int egpu_table_set(egpu_ctx* ctx, const int32_t* free_core,
                   const int32_t* free_mem, int32_t D);
/* oversub may be NULL.  Synchronises the context's stream. */
int egpu_table_get(egpu_ctx* ctx, int32_t* free_core, int32_t* free_mem,
                   int32_t* oversub);
int egpu_table_size(egpu_ctx* ctx);

/* ---- snapshot mode, host buffers (what a cgo caller uses) -------------- */

/* Scores R requests against the current table.  Copies inputs H2D from the
 * caller's arrays (pinned or pageable), runs the scan, copies idx and deltas
 * back; returns when the outputs are valid.  out_delta_* have D entries and
 * may be NULL.  commit != 0 installs table' as the current table. */
int egpu_bestfit_batch(egpu_ctx* ctx, const int32_t* req_core,
                       const int32_t* req_mem, int64_t R, int32_t* out_idx,
                       int64_t* out_delta_core, int64_t* out_delta_mem,
                       int commit);

/* Batch allocation to a fixed point (SURVEY.md §8(f) n4: "multi-round deferred retry").
 * Round 1 is egpu_bestfit_batch(..., EGPU_F_COMMIT | EGPU_F_PREFIX_COMMIT); every later round
 * re-submits the rows the previous one deferred, in their original order, against the table
 * that round committed.  It stops when a round defers nothing or after max_rounds (>= 1).
 * Every round places at least one row per device that still has takers, so it terminates; the
 * table is always committed and never oversubscribed.
 *   out_idx[r]      device index, EGPU_IDX_INFEASIBLE (in the round the row was last scored),
 *                   or EGPU_IDX_DEFERRED when max_rounds ran out first
 *   out_delta_*[D]  demand committed over all rounds (may be NULL)
 *   *out_rounds     rounds run; *out_deferred = rows still deferred (both may be NULL)
 * Scratch (32 bytes per request, kept by the context) is allocated before round 1: an
 * allocation failure returns EGPU_ERR_NOMEM with nothing committed.
 * R < 2^31.  The _dev form takes device request/index arrays (16-byte aligned) and host
 * out_delta[2*D]; it synchronises `stream` (each round needs its deferred count on the host). */
int egpu_bestfit_batch_rounds(egpu_ctx* ctx, const int32_t* req_core, const int32_t* req_mem,
                              int64_t R, int32_t* out_idx, int64_t* out_delta_core,
                              int64_t* out_delta_mem, int32_t max_rounds, int32_t* out_rounds,
                              int64_t* out_deferred);
int egpu_bestfit_batch_rounds_dev(egpu_ctx* ctx, const int32_t* d_req_core,
                                  const int32_t* d_req_mem, int64_t R, int32_t* d_out_idx,
                                  int64_t* out_delta, int32_t max_rounds, int32_t* out_rounds,
                                  int64_t* out_deferred, void* stream);

/* Packed wire format, for callers bound by PCIe rather than by the scan: 5 bytes per decision
 * instead of 12.  req_packed[r] = EGPU_PACK_REQUEST(core, mem) (core in 0..127, mem in
 * 0..2^18-1; any word >= 2^25, e.g. EGPU_PACKED_INVALID, is an infeasible request);
 * out_idx8[r] = device index 0..63 or -1.  R <= EGPU_MAX_ROWS as in every other entry point
 * (EGPU_ERR_INVALID above it: the demand sums hold that many rows).  Everything else as
 * egpu_bestfit_batch. */
#define EGPU_PACK_REQUEST(core, mem) (((uint32_t)(core) << 18) | (uint32_t)(mem))
#define EGPU_PACKED_INVALID 0xFFFFFFFFu
int egpu_bestfit_batch_packed(egpu_ctx* ctx, const uint32_t* req_packed, int64_t R, int8_t* out_idx8,
                              int64_t* out_delta_core, int64_t* out_delta_mem, int commit);
int egpu_bestfit_batch_packed_dev(egpu_ctx* ctx, const uint32_t* d_req_packed, int64_t R,
                                  int8_t* d_out_idx8, int64_t* d_delta, int32_t* d_table_out,
                                  int flags, void* stream);

/* Pinned host memory for callers that want zero staging copies. */
int  egpu_host_alloc(egpu_ctx* ctx, void** out, int64_t bytes);
void egpu_host_free(egpu_ctx* ctx, void* p);

/* Pins caller-owned memory in place (cudaHostRegister, mapped) so that buffers the caller already
 * has - a Go slice it keeps for the life of the plugin, say - take the zero-staging path of
 * egpu_bestfit_batch / _packed instead of being copied through HBM: on a PCIe Gen5 B200 that is
 * ~0.2 ms instead of ~1 ms per 1 M requests.  Registration costs about a millisecond per 10 MB, so
 * it pays only for buffers that are reused.  The range must stay allocated until
 * egpu_host_unregister (a cgo caller must not hand over memory the Go runtime may release:
 * allocate it with C.malloc or keep it pinned with runtime.Pinner).  The context does not track
 * registrations. */
int  egpu_host_register(egpu_ctx* ctx, void* p, int64_t bytes);
int  egpu_host_unregister(egpu_ctx* ctx, void* p);

/* ---- snapshot mode, device buffers (bench / multi-GPU plumbing) -------- */

/* Asynchronous on `stream` (a cudaStream_t passed as void*; NULL = the
 * context's own non-blocking stream — to name the legacy default stream pass
 * cudaStreamLegacy, not 0).  d_delta is int64[2*D]: core sums then mem sums; it
 * is overwritten, not accumulated.  d_table_out (may be NULL) receives
 * int32[3*D]: free_core', free_mem', oversub.  flags: EGPU_F_*.  The three
 * request/index arrays must be 16-byte aligned (128-bit accesses). */
int egpu_bestfit_batch_dev(egpu_ctx* ctx, const int32_t* d_req_core,
                           const int32_t* d_req_mem, int64_t R,
                           int32_t* d_out_idx, int64_t* d_delta,
                           int32_t* d_table_out, int flags, void* stream);

/* Several batches in ONE launch.  Every batch is what egpu_bestfit_batch_dev takes - its own
 * request arrays, index array, d_delta (may be NULL) and d_table_out (may be NULL) - and all K
 * (1..EGPU_MAX_BATCHES) are scored against the current table, so the result of each batch is
 * exactly what K separate non-committing calls would produce; only the launch latency, ramp and
 * tail are paid once instead of K times (at R = 1 M that fixed cost is about a third of a lone
 * launch; at R <= 100 k it is nearly all of it).  Asynchronous on `stream`.  flags:
 * EGPU_F_INPUTS_READY only (a multi-batch launch never commits: install a table' with
 * egpu_table_set or a committing single-batch call).  Outputs of different batches must not
 * overlap (EGPU_ERR_INVALID).  Batches may have different R (R = 0 allowed). */
#define EGPU_MAX_BATCHES 64
typedef struct egpu_batch {
    const int32_t* d_req_core;
    const int32_t* d_req_mem;
    int64_t        R;
    int32_t*       d_out_idx;
    int64_t*       d_delta;      /* int64[2*D] or NULL */
    int32_t*       d_table_out;  /* int32[3*D] or NULL */
} egpu_batch;
int egpu_bestfit_batches_dev(egpu_ctx* ctx, const egpu_batch* batches, int32_t K, int flags,
                             void* stream);

/* Stateless query: scores R requests against the table GIVEN HERE (free_core/free_mem[D], host
 * arrays, same domain as egpu_table_set) and returns the indices.  The context's own table,
 * its oversubscription flags and lookup tables are not read or written, so a context that
 * tracks the node's committed placement can also answer GetPreferredAllocation-style
 * what-if questions (egpu_preferred_allocation uses this).  Host buffers; returns when out_idx
 * is valid. */
int egpu_bestfit_query(egpu_ctx* ctx, const int32_t* free_core, const int32_t* free_mem, int32_t D,
                       const int32_t* req_core, const int32_t* req_mem, int64_t R,
                       int32_t* out_idx);

/* Multi-GPU step 2: after the G per-rank delta vectors (int64[G][2*D], rank
 * major) have been all-gathered, subtract their sum from the current table on
 * this rank: d_table_out (may be NULL) receives int32[3*D] as above, and with
 * commit != 0 the result becomes the current table.  Every rank ends with an
 * identical table'. */
int egpu_table_apply_deltas_dev(egpu_ctx* ctx, const int64_t* d_deltas, int G,
                                int32_t* d_table_out, int commit, void* stream);

/* ---- multi-GPU without a collective library on the data path --------------- */

/* One process per GPU.  Each rank exports a CUDA-IPC handle of its exchange buffer
 * (EGPU_IPC_HANDLE_BYTES bytes), the ranks swap handles by any means (the bench uses
 * torch.distributed.all_gather_object) and attach: handles = world * 64 bytes, rank
 * major.  After that a sharded step is two asynchronous calls:
 *   egpu_bestfit_batch_shard_dev  scans this rank's rows; its last CTA stores the
 *       rank's demand vector into EVERY rank's exchange buffer over NVLink and raises
 *       a release flag - the exchange is fused into the scan kernel;
 *   egpu_table_apply_peers_dev    waits (acquire) until all `world` vectors of `step`
 *       have landed locally, applies their sum: table' (and commit) as in snapshot mode.
 * `step` must increase by one per sharded step on every rank; a rank's scans may run at
 * most 128 steps ahead of its own applies (256 exchange slots: then no peer can be more than
 * 255 steps ahead of what this rank has consumed).  The scan itself never commits. */
#define EGPU_IPC_HANDLE_BYTES 64
#define EGPU_MAX_RANKS 8
int egpu_peer_export(egpu_ctx* ctx, void* handle_out);
int egpu_peer_attach(egpu_ctx* ctx, int rank, int world, const void* handles);
int egpu_peer_detach(egpu_ctx* ctx);
int egpu_bestfit_batch_shard_dev(egpu_ctx* ctx, const int32_t* d_req_core,
                                 const int32_t* d_req_mem, int64_t R,
                                 int32_t* d_out_idx, int64_t* d_delta, int flags,
                                 uint64_t step, void* stream);
int egpu_table_apply_peers_dev(egpu_ctx* ctx, uint64_t step, int32_t* d_table_out,
                               int commit, void* stream);
/* K sharded steps in one launch: batch k is exchange step first_step + k (egpu_bestfit_batches_dev
 * + the fused push of egpu_bestfit_batch_shard_dev).  Without EGPU_F_APPLY d_table_out of the
 * batches is ignored (table' comes from the apply calls); with it the exchange steps are consumed
 * by the launch itself and no apply call must follow. */
int egpu_bestfit_batches_shard_dev(egpu_ctx* ctx, const egpu_batch* batches, int32_t K, int flags,
                                   uint64_t first_step, void* stream);
/* Start gate for a sharded sequence.  egpu_peer_gate_dev enqueues a one-warp kernel that
 * waits (i) for this rank's host to call egpu_peer_gate_open - which the caller does after it
 * has enqueued everything that follows the gate - and (ii) for every peer's gate to have
 * reached the same point, through flags in peer memory.  The work behind the gate then starts
 * at the same time on every rank without any host in the way: launch skew between the ranks'
 * host threads no longer lands inside the sequence.  Every gate_dev needs exactly one
 * gate_open, on every rank, in the same order.  Works unattached too (host part only).
 * A gate that has waited ~2 s gives up and lets the stream proceed (this happens when kernel
 * launches are blocking - CUDA_LAUNCH_BLOCKING, a profiler - because the host then never gets
 * to open it); egpu_peer_gate_timeouts counts those (synchronises the device). */
int egpu_peer_gate_dev(egpu_ctx* ctx, void* stream);
int egpu_peer_gate_open(egpu_ctx* ctx);
int64_t egpu_peer_gate_timeouts(egpu_ctx* ctx);
/* Prefix-commit (EGPU_F_PREFIX_COMMIT semantics, see egpu_bestfit_batch) over row shards.
 * The batch is the concatenation of the ranks' shards in rank order; request r of rank g
 * commits iff the running demand of its device over ALL earlier rows - the whole shards of
 * ranks < g and the rows before r here - still fits (SURVEY.md Appendix A.5: "rank-major
 * across shards").  One asynchronous call per rank; it uses TWO exchange steps, `step` (the
 * uncapped demand of every shard, pushed by the scan itself; every rank then knows the base
 * offset of its shard) and `step + 1` (the committed demand after the cut), so the caller
 * advances `step` by 2.  Outputs: d_out_idx with EGPU_IDX_DEFERRED for the rows beyond the
 * cut; d_delta[2*D] = THIS rank's committed demand (may be NULL); d_table_out[3*D] =
 * table - committed demand of all ranks, identical on every rank (may be NULL);
 * EGPU_F_COMMIT installs it.  Never oversubscribes. */
int egpu_bestfit_batch_shard_prefix_dev(egpu_ctx* ctx, const int32_t* d_req_core,
                                        const int32_t* d_req_mem, int64_t R,
                                        int32_t* d_out_idx, int64_t* d_delta,
                                        int32_t* d_table_out, int flags, uint64_t step,
                                        void* stream);
/* Scan + lagged apply in ONE launch: as egpu_bestfit_batch_shard_dev, and the same last CTA
 * also applies the exchanged vectors of step (step - lag) (1 <= lag <= 16) and writes that
 * step's table' to d_table_out_lagged (skipped while step < lag).  A whole sharded sequence
 * is then a single stream of scan launches, finished by one
 * egpu_table_apply_peers_multi_dev(first_step = last - lag + 1, lag steps) for the tail.
 * The wait for step - lag is the back-pressure: no rank gets more than `lag` steps ahead
 * of the slowest.  A sequence restarted from step 0 (a replayed CUDA graph) must be
 * separated from the previous one by a barrier across the ranks.  Never commits. */
int egpu_bestfit_batch_shard_lag_dev(egpu_ctx* ctx, const int32_t* d_req_core,
                                     const int32_t* d_req_mem, int64_t R,
                                     int32_t* d_out_idx, int64_t* d_delta, int flags,
                                     uint64_t step, int lag, int32_t* d_table_out_lagged,
                                     void* stream);
/* Same for nsteps (1..64) consecutive steps in one launch; d_table_outs is a HOST array of
 * nsteps device pointers (entries may be NULL).  With commit the steps are applied on top
 * of each other and the last table' is installed. */
int egpu_table_apply_peers_multi_dev(egpu_ctx* ctx, uint64_t first_step, int nsteps,
                                     int32_t* const* d_table_outs, int commit,
                                     void* stream);
/* step + 1 of the last apply that gave up waiting for a peer (~2 s), 0 if none */
int64_t egpu_peer_last_timeout(egpu_ctx* ctx);

/* Deterministic synthetic request generator on the device (same counter-based
 * RNG as the CPU generators; DESIGN.md §6).  dist: 2 = cfg2, 3 = cfg3. */
int egpu_synth_requests_dev(egpu_ctx* ctx, int dist, uint64_t seed,
                            int64_t first_row, int64_t R, int32_t* d_req_core,
                            int32_t* d_req_mem, void* stream);

/* ---- sequential mode --------------------------------------------------- */

/* Applies E events in order to the current table (which is updated).
 * kind[i] = EGPU_EV_ALLOC: a[i] = core, b[i] = mem  -> out_idx[i] = device or -1
 * kind[i] = EGPU_EV_FREE : a[i] = index of the ALLOC event to release
 *                          -> out_idx[i] = device released, or -1 when that
 *                          event is not a live allocation (not an ALLOC, not
 *                          earlier than i, infeasible, or already freed). */
int egpu_replay(egpu_ctx* ctx, const int32_t* kind, const int32_t* a,
                const int32_t* b, int64_t E, int32_t* out_idx);

/* ---- whole-card requests (DESIGN.md §2.8) ------------------------------- */

/* A container asking for more than 100 gpu-core units gets whole GPUs:
 * core = 100*k with 2 <= k <= 64 asks for k cards with free_core = 100 and
 * free_mem >= mem each, and every card gives (100, mem) - memory is per card.
 * The k cards are the k best fits of (100, mem), i.e. what k sequential best-fit
 * picks give.  Any other core > 100 (not a multiple of 100, k > 64, or k > D)
 * is infeasible.  core <= 100 is the single-card rule of egpu_bestfit_batch /
 * egpu_replay, unchanged: on batches without whole-card rows these entry points
 * compute exactly what those do.
 *   out_idx[r]    the first card, the tightest one (not necessarily the lowest
 *                 index), or -1
 *   out_cards[r]  mask of every card the row holds (1 << idx for a single-card
 *                 row, 0 when infeasible); may be NULL, then no mask is stored
 *                 (12 bytes of traffic per request instead of 20)
 * Demand sums, table', commit and the sticky oversubscription flag are those of
 * egpu_bestfit_batch[_dev] with every card of a row adding (100, mem) to its own
 * device.  These entry points always run the register scan: egpu_set_variant
 * does not apply to them.
 * egpu_bestfit_cards: host buffers, commit = 0 or EGPU_F_COMMIT.
 * egpu_bestfit_cards_dev: as egpu_bestfit_batch_dev; flags = EGPU_F_COMMIT |
 * EGPU_F_INPUTS_READY (EGPU_F_PREFIX_COMMIT and any other flag are
 * EGPU_ERR_INVALID); every device array, d_out_cards, d_delta and d_table_out
 * included, must be 16-byte aligned; pipelines with the other scans of the
 * context under the same rules. */
int egpu_bestfit_cards(egpu_ctx* ctx, const int32_t* req_core, const int32_t* req_mem, int64_t R,
                       int32_t* out_idx, uint64_t* out_cards, int64_t* out_delta_core,
                       int64_t* out_delta_mem, int commit);
int egpu_bestfit_cards_dev(egpu_ctx* ctx, const int32_t* d_req_core, const int32_t* d_req_mem,
                           int64_t R, int32_t* d_out_idx, uint64_t* d_out_cards, int64_t* d_delta,
                           int32_t* d_table_out, int flags, void* stream);

/* egpu_replay with whole-card ALLOCs: ALLOC(100*k, mem) takes its k cards on
 * the current table and subtracts (100, mem) from each; a FREE of a live
 * whole-card ALLOC gives (100, mem) back to every card it holds and reports that
 * ALLOC's idx and card mask.  Every other rule is egpu_replay's.  out_cards
 * (may be NULL) = the cards of each event, 0 for -1. */
int egpu_replay_cards(egpu_ctx* ctx, const int32_t* kind, const int32_t* a, const int32_t* b,
                      int64_t E, int32_t* out_idx, uint64_t* out_cards);

#ifdef __cplusplus
}
#endif
#endif /* EGPU_ALLOC_H */
