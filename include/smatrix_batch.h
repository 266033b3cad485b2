/*
 * include/smatrix_batch.h — batched C-ABI entry points on top of smatrix.h (new; the reference
 * has no bulk API).  These are what a binding (JNI / Ruby / cgo / ctypes) should call for
 * throughput; INTEGRATION.md shows the stubs.
 *
 * Semantics: exactly those of calling the single-op function of the reference for
 * i = 0 .. n-1 in input order (src/smatrix.c:174-256), on the safe domain described in
 * smatrix.h: uint32 wrap-around for incr/decr, duplicate keys in one set batch resolve to the
 * LAST one in input order, rowlen reproduces the reference's running counter, getrow rows are
 * complete (compare sorted by column).
 *
 * Pointers: every array argument may be a HOST pointer (pageable or pinned) or a DEVICE pointer
 * on the matrix's GPU; the library detects which (cudaPointerGetAttributes).  Host arrays are
 * streamed through the device in chunks, pinned host memory overlaps the copy with the update.
 * `vals == NULL` means "every value is 1" (the co-occurrence workload, examples/cf_recommender.c:35-47).
 * Calls return after the work has completed on the device (results are visible to the caller).
 * Errors: "libsmatrix error: ..." on stdout + abort(), like the reference (src/smatrix.c:891-894).
 */
#ifndef SMATRIX_BATCH_H
#define SMATRIX_BATCH_H

#include "smatrix.h"

#ifdef __cplusplus
extern "C" {
#endif

/* n x smatrix_incr / smatrix_decr / smatrix_set (src/smatrix.c:225-256). */
void smatrix_incr_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                        const uint32_t* vals, size_t n);
void smatrix_decr_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                        const uint32_t* vals, size_t n);
void smatrix_set_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                       const uint32_t* vals, size_t n);

/* The same three calls, additionally returning what every single call would have returned
 * (SURVEY.md 8f N1; src/smatrix.c:230,241,252): out[i] = value of cell (xs[i], ys[i]) right after
 * op i, as if the batch had been applied one op at a time in input order — so duplicate keys see
 * each other's effect in order (running sums mod 2^32 for incr / decr; set returns its own value).
 * Costs a look-up pass, a stable sort by cell and a segmented scan on top of the plain batch. */
void smatrix_incr_batch_out(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                            const uint32_t* vals, size_t n, uint32_t* out);
void smatrix_decr_batch_out(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                            const uint32_t* vals, size_t n, uint32_t* out);
void smatrix_set_batch_out(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                           const uint32_t* vals, size_t n, uint32_t* out);

/* n x smatrix_get (src/smatrix.c:174-185): out[i] = value at (xs[i], ys[i]) or 0. */
void smatrix_get_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys, size_t n,
                       uint32_t* out);

/* n x smatrix_rowlen (src/smatrix.c:212-223). */
void smatrix_rowlen_batch(smatrix_t* self, const uint32_t* xs, size_t n, uint32_t* out);

/* n x smatrix_getrow with full-size buffers (src/smatrix.c:189-210), as CSR:
 *   offsets[0..n]  (uint64) — row i's pairs are pairs[2*offsets[i] .. 2*offsets[i+1])
 *   pairs          (uint32) — [col, value] pairs, `pairs_cap` = capacity in PAIRS
 * Returns the total number of pairs.  Size query: call with pairs == NULL (offsets are still
 * filled); if the total exceeds pairs_cap nothing is written to pairs and the total is returned
 * so the caller can retry with a larger buffer. */
uint64_t smatrix_getrow_batch(smatrix_t* self, const uint32_t* xs, size_t n, uint64_t* offsets,
                              uint32_t* pairs, uint64_t pairs_cap);

/* The read side of the co-occurrence recommender for a batch of items
 * (examples/cf_recommender.c:50-86, neighbors_for_item + cf_cosine): for every item a and every
 * pair (b, cc) of a's row — including the column-0 pair, as the example does — ids = b and
 * score = cc / (sqrt(total_a) * sqrt(total_b)), where total_x = value at (x, 0) (1 if total_b is 0)
 * and the score is 0 if the denominator is 0 or smaller than cc.  CSR like smatrix_getrow_batch:
 * offsets[0..n], ids / scores with capacity `cap` entries; size query with ids == NULL. */
uint64_t smatrix_cf_neighbors_batch(smatrix_t* self, const uint32_t* items, size_t n,
                                    uint64_t* offsets, uint32_t* ids, double* scores, uint64_t cap);

/* The recommendation itself: for every item, the first min(k, len) entries of exactly the list
 * smatrix_cf_neighbors_batch returns for it (column-0 pair included), ordered by score descending, then
 * id ascending, so the answer is unique and bit-exact.  The ranking runs on the device; the neighbour
 * lists never leave it.  Fixed-width, row-major outputs: counts[n] = min(k, len); ids[n*k] and
 * scores[n*k], where the slots past counts[i] hold id 0xFFFFFFFF and score -1.0.  An absent item or an
 * empty row has count 0.  1 <= k <= 1024.  `items` may be host or device; the three outputs are all host
 * or all device (host outputs: n * (12k + 4) bytes come down).  Items are processed in pieces whose rows
 * hold at most $SMATRIX_TOPK_PAIRS pairs (see smatrix_b200.h). */
void smatrix_cf_topk_batch(smatrix_t* self, const uint32_t* items, size_t n, uint32_t k,
                           uint32_t* counts, uint32_t* ids, double* scores);

/* Item-based recommendations for baskets (a user's items): basket i is items[basket_off[i] .. basket_off[i+1]);
 * basket_off has n + 1 entries, starts at 0, never decreases and ends at most at 2^32 - 2.  For every position j,
 * L_j is exactly the list smatrix_cf_neighbors_batch returns for items[j] (empty for an absent item).  The
 * candidates of basket i are the ids of its lists, minus its own items and minus id 0 (the column-0 pair holds the
 * item's total, not a co-occurrence).  A candidate's score is (((0.0 + s_j1) + s_j2) + ...) over the positions
 * j1 < j2 < ... of the basket whose list holds it, in IEEE double with one rounding per addition, in that order:
 * the answer is bit-exact and reproducible; an item repeated in a basket counts once per position.  Output as
 * smatrix_cf_topk_batch: counts[n] = min(k, candidates), ids[n*k] / scores[n*k] by score descending, then id
 * ascending, slots past the count hold id 0xFFFFFFFF and score -1.0; an empty basket, or one of absent items only,
 * has count 0.  1 <= k <= 1024.  basket_off and items are both host or both device arrays, the three outputs all
 * host or all device (host outputs: n * (12k + 4) bytes come down; the neighbour lists never leave the device).
 * Baskets are processed in pieces whose rows hold at most $SMATRIX_TOPK_PAIRS pairs (a basket over that is a piece
 * of its own, see smatrix_b200.h). */
void smatrix_cf_recommend_batch(smatrix_t* self, const uint64_t* basket_off, const uint32_t* items,
                                size_t n_baskets, uint32_t k, uint32_t* counts, uint32_t* ids, double* scores);

#ifdef __cplusplus
}
#endif
#endif
