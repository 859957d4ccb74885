/*
 * oracle/cards_oracle.c — CPU restatement of whole-card requests (DESIGN.md §2.8).
 *
 * TEST INFRASTRUCTURE ONLY, like bestfit_oracle.c: nothing in the product path may include,
 * link or call this file.  Built on its own into libcards_oracle.so (oracle/cards_c.py).
 *
 * The reference gives a container asking for more than 100 gpu-core units len/100 whole GPUs
 * (pkg/plugins/gpushare.go:62-69) and picks them one after the other.  This file follows that
 * formulation literally: k sequential best-fit picks of (100, mem) on a scratch copy of the
 * table, each pick the obvious scalar loop of spec §2.3.  It does not use the fact the CUDA
 * scan relies on (the k cards are a run of the sorted table); tests/test_cards_oracle.py checks
 * that fact against this file, and an independent numpy restatement (oracle/cards_np.py)
 * against it.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORACLE_MAX_DEVICES 64
#define ORACLE_CORE_MAX 100
#define ORACLE_MEM_MAX ((1 << 18) - 1)

static int cards_table_valid(const int32_t* free_core, const int32_t* free_mem, int32_t D) {
    if (!free_core || !free_mem || D < 1 || D > ORACLE_MAX_DEVICES) return -1;
    for (int32_t d = 0; d < D; ++d) {
        if (free_core[d] < 0 || free_core[d] > ORACLE_CORE_MAX) return -1;
        if (free_mem[d] < 0 || free_mem[d] > ORACLE_MEM_MAX) return -1;
    }
    return 0;
}

/* spec §2.3: the feasible device with the smallest (free_core - core, free_mem - mem, d), or -1 */
static int32_t cards_pick(const int32_t* free_core, const int32_t* free_mem, int32_t D, int32_t core, int32_t mem) {
    int32_t best = -1, best_lc = 0, best_lm = 0;
    if (core < 0 || mem < 0) return -1;
    for (int32_t d = 0; d < D; ++d) {
        if (free_core[d] < core || free_mem[d] < mem) continue;
        const int32_t lc = free_core[d] - core, lm = free_mem[d] - mem;
        if (best < 0 || lc < best_lc || (lc == best_lc && lm < best_lm)) {
            best = d;
            best_lc = lc;
            best_lm = lm;
        }
    }
    return best;
}

static int32_t sat_i32(int64_t v) {
    if (v > INT32_MAX) return INT32_MAX;
    if (v < INT32_MIN) return INT32_MIN;
    return (int32_t)v;
}

/* spec §2.4: table' = table - delta, saturated, with oversubscription flags (int32[3*D]) */
static void cards_apply_delta(const int32_t* free_core, const int32_t* free_mem, int32_t D, const int64_t* delta_core,
                              const int64_t* delta_mem, int32_t* table_out) {
    for (int32_t d = 0; d < D; ++d) {
        const int64_t c = (int64_t)free_core[d] - delta_core[d];
        const int64_t m = (int64_t)free_mem[d] - delta_mem[d];
        table_out[d] = sat_i32(c);
        table_out[D + d] = sat_i32(m);
        table_out[2 * D + d] = (c < 0 || m < 0) ? 1 : 0;
    }
}

/* Whole-card requests (spec §2.8).  core = 100*k with 2 <= k <= 64 asks for k whole cards,
 * each giving (100, mem); any other core > 100 is infeasible; core <= 100 is one card as in
 * §2.3.  Returns k (1 for a single-card request) and sets *per_core to the core each card
 * gives, or returns 0 when the request is infeasible whatever the table. */
static int32_t oracle_cards_k(int32_t core, int32_t* per_core) {
    *per_core = core;
    if (core <= ORACLE_CORE_MAX) return 1;
    if (core % 100 != 0 || core / 100 > ORACLE_MAX_DEVICES) return 0;
    *per_core = ORACLE_CORE_MAX;
    return core / 100;
}

/* The plugin's formulation: k sequential best-fit picks of (per_core, mem) on a scratch copy
 * of the table.  Returns the first card (-1 when fewer than k cards fit) and its card mask. */
static int32_t oracle_pick_cards(const int32_t* free_core, const int32_t* free_mem, int32_t D, int32_t core,
                                 int32_t mem, uint64_t* cards) {
    int32_t per_core;
    const int32_t k = oracle_cards_k(core, &per_core);
    int32_t sc[ORACLE_MAX_DEVICES], sm[ORACLE_MAX_DEVICES];
    int32_t first = -1;
    uint64_t mask = 0;
    *cards = 0;
    if (k == 0 || k > D) return -1;
    memcpy(sc, free_core, sizeof(int32_t) * (size_t)D);
    memcpy(sm, free_mem, sizeof(int32_t) * (size_t)D);
    for (int32_t j = 0; j < k; ++j) {
        const int32_t d = cards_pick(sc, sm, D, per_core, mem);
        if (d < 0) return -1;
        sc[d] -= per_core;
        sm[d] -= mem;
        mask |= 1ull << d;
        if (j == 0) first = d;
    }
    *cards = mask;
    return first;
}

/* Snapshot mode with whole-card requests (spec §2.4 extended by §2.8): every card of a row
 * adds (per-card core, mem) to its device's demand.  out_cards may be NULL. */
int oracle_bestfit_cards_snapshot(const int32_t* free_core, const int32_t* free_mem, int32_t D,
                                  const int32_t* req_core, const int32_t* req_mem, int64_t R,
                                  int32_t* out_idx, uint64_t* out_cards, int64_t* delta_core,
                                  int64_t* delta_mem, int32_t* table_out) {
    if (cards_table_valid(free_core, free_mem, D) != 0 || R < 0) return -1;
    int64_t dc[ORACLE_MAX_DEVICES], dm[ORACLE_MAX_DEVICES];
    memset(dc, 0, sizeof dc);
    memset(dm, 0, sizeof dm);
    for (int64_t r = 0; r < R; ++r) {
        uint64_t cards;
        int32_t per_core;
        out_idx[r] = oracle_pick_cards(free_core, free_mem, D, req_core[r], req_mem[r], &cards);
        oracle_cards_k(req_core[r], &per_core);
        if (out_cards) out_cards[r] = cards;
        for (int32_t d = 0; d < D; ++d) {
            if (!((cards >> d) & 1u)) continue;
            dc[d] += per_core;
            dm[d] += req_mem[r];
        }
    }
    if (delta_core) memcpy(delta_core, dc, sizeof(int64_t) * (size_t)D);
    if (delta_mem) memcpy(delta_mem, dm, sizeof(int64_t) * (size_t)D);
    if (table_out) cards_apply_delta(free_core, free_mem, D, dc, dm, table_out);
    return 0;
}

/* Sequential mode with whole-card requests (spec §2.6 extended by §2.8).  free_core/free_mem
 * are updated in place.  A FREE of a live ALLOC gives every card it holds back and reports
 * that ALLOC's index and card mask.  out_cards may be NULL. */
int oracle_replay_cards(int32_t* free_core, int32_t* free_mem, int32_t D, const int32_t* kind,
                        const int32_t* a, const int32_t* b, int64_t E, int32_t* out_idx,
                        uint64_t* out_cards) {
    if (cards_table_valid(free_core, free_mem, D) != 0 || E < 0) return -1;
    /* live[i] = cards an ALLOC event currently holds, 0 otherwise */
    uint64_t* live = (uint64_t*)calloc((size_t)(E > 0 ? E : 1), sizeof(uint64_t));
    if (!live) return -3;
    for (int64_t i = 0; i < E; ++i) {
        uint64_t cards = 0;
        int32_t d = -1, per_core;
        if (kind[i] == 0) {
            d = oracle_pick_cards(free_core, free_mem, D, a[i], b[i], &cards);
            oracle_cards_k(a[i], &per_core);
            for (int32_t j = 0; j < D; ++j) {
                if (!((cards >> j) & 1u)) continue;
                free_core[j] -= per_core;
                free_mem[j] -= b[i];
            }
            live[i] = cards;
        } else {
            const int64_t t = a[i];
            if (kind[i] == 1 && t >= 0 && t < i && kind[t] == 0 && live[t] != 0) {
                cards = live[t];
                d = out_idx[t];
                oracle_cards_k(a[t], &per_core);
                for (int32_t j = 0; j < D; ++j) {
                    if (!((cards >> j) & 1u)) continue;
                    free_core[j] += per_core;
                    free_mem[j] += b[t];
                }
                live[t] = 0;
            }
        }
        out_idx[i] = d;
        if (out_cards) out_cards[i] = cards;
    }
    free(live);
    return 0;
}

