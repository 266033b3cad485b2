/*
 * smx_internal.h — layouts shared by the host shim (C) and the kernels (CUDA), plus the
 * launcher prototypes.  Plain C so that smx_host.c can include it.
 *
 * HBM layout (DESIGN.md "Data layout"):
 *
 *   row directory   open addressing over 64-byte entries, position = mix_row(x) & (cap-1),
 *                   linear probing.  Entry = one 32-byte header sector + one 32-byte inline
 *                   bucket sector (4 cells), so a row with <= 4 columns costs one 64-byte burst.
 *                   Replaces the reference's cmap + the malloc'ed 48-byte rmap header
 *                   (src/smatrix.h:40-65).
 *   column buckets  per row, open addressing over 32-byte sectors of 4 packed cells
 *                   {u32 column, u32 value} (same 8-byte cell as src/smatrix.h:35-38), position
 *                   = mix_col(y) & (sectors-1), linear probing over sectors.  Column 0 is NOT
 *                   stored here: it lives in the header (c0), so cell == 0 is the empty sentinel
 *                   and a zero-valued cell with column != 0 stays live (SURVEY.md Q2/H3).
 *   slab            buckets of 16 * 2^k cells carved from cudaMalloc'ed segments by a bump
 *                   cursor; growth = allocate the bigger bucket, re-place, recycle the old one.
 */
#ifndef SMX_INTERNAL_H
#define SMX_INTERNAL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- row header flags (smx_row_t.meta) ------------------------------------------------- */
#define SMX_META_CAPLOG 0x3Fu   /* log2(bucket capacity in cells); 2 = the inline bucket     */
#define SMX_META_USED   0x100u  /* entry holds a row                                         */
#define SMX_META_ZC     0x200u  /* column 0 was already non-zero when the current batch began */
#define SMX_META_D      0x400u  /* rowlen = live + 1: a virtual resize counted column 0 (Q1)  */
#define SMX_META_SLOG_SHIFT 16  /* bits 16..20: log2(reference row size) - 4, as of the last sync */
#define SMX_META_SLOG   (0x1Fu << SMX_META_SLOG_SHIFT)
#define SMX_META_T0P    0x800u  /* column 0 turns non-zero inside the current batch at t0     */
#define SMX_META_GROW   0x1000u /* row is queued for growth in the current round              */
#define SMX_INLINE_LOG  2u
#define SMX_MIN_SLAB_LOG 4u     /* first slab bucket: 16 cells = 128 B (src/smatrix.h:21)     */
#define SMX_MAX_CAPLOG  31u
#define SMX_BIG_LOG     13u     /* buckets >= 2^13 cells are re-placed / compacted grid-wide  */
#define SMX_MID_LOG     9u      /* buckets of 2^9 .. 2^12 cells are re-placed by one block each */
#define SMX_ZERO_LOG    9u      /* vacated buckets >= 2^9 cells are zeroed when they are vacated, so a
                                   recycled one can be filled in place; smaller ones are always built in
                                   shared memory and written out whole */
#define SMX_CLASSES     32u     /* bucket size classes = log2(cells)                          */
#define SMX_PLAN_RECYCLED (1ull << 63) /* smx_plan_t.off is the address of a recycled bucket, not an offset */

typedef struct {
  uint32_t key;    /* row id x                                  } claimed together by one   */
  uint32_t meta;   /* flags | caplog                            } 64-bit CAS                */
  uint64_t slots;  /* device address of the slab bucket (caplog > 2)                        */
  uint32_t live;   /* L: number of columns != 0 ever written                                */
  uint32_t c0;     /* value of column 0                                                     */
  uint32_t t0inv;  /* ~(batch index of the first op that makes column 0 non-zero); 0 = none */
  uint32_t want;   /* ops turned away because the bucket was at its load limit (growth sizing) */
  uint64_t inl[4]; /* inline bucket                                                          */
} smx_row_t;       /* 64 bytes */

/* ---- device control block (counters the host reads back after every round) -------------- */
#define SMX_DIR_SLICES 256u      /* occupancy is tracked (and limited) per directory slice     */
#define SMX_DIR_CREATE_STEPS 256u /* dir_find creates a row at most this many probe steps - 1 from its home */
typedef struct {
  /* persistent */
  unsigned long long dir_used;   /* rows in the directory (sum of slice_used, set by the host's readers) */
  /* per chunk */
  uint32_t n_late;               /* ops parked for the LATE pass                             */
  uint32_t n_t0;                 /* rows whose column 0 turned non-zero in this chunk        */
  /* per round */
  uint32_t n_defer;              /* ops turned away this round (re-run after growth)         */
  uint32_t n_dirfull;            /*   ... because the directory was at its load limit        */
  uint32_t n_grow;               /* rows queued for growth                                   */
  uint32_t n_big;                /* of those, rows whose OLD bucket is >= 2^SMX_BIG_LOG      */
  uint32_t n_mid;                /*           rows whose OLD bucket is 2^SMX_MID_LOG .. 2^(SMX_BIG_LOG-1) */
  uint32_t n_recycled;           /* planned buckets taken from the free lists                */
  uint32_t n_spill;              /* cells k_migrate_tiles could not place inside their tile (spill list length) */
  uint32_t dir_probe_max;        /* largest probe step at which k_dir_rehash placed a row (zeroed before it runs) */
  unsigned long long plan_bytes; /* bytes of FRESH slab planned by grow_plan                 */
  unsigned long long need_zero;  /* planned buckets that are filled in place (global CAS) and so
                                    need a zeroed region; shared-memory-built buckets do not  */
  uint32_t grow_from[SMX_CLASSES]; /* growing rows per OLD size class = buckets about to be vacated */
  unsigned long long scratch;    /* misc: reductions (nnz, probe checksums)                  */
  /* persistent: vacated buckets, one stack of addresses per size class (src/smatrix.c:383-416 frees the
   * old row map on every resize; here k_free_push recycles it and k_grow_plan takes from the stacks
   * before it plans fresh slab).  The host sizes the stacks (free_stack) before every push. */
  int32_t free_cnt[SMX_CLASSES];
  unsigned long long* free_stack[SMX_CLASSES];
  /* persistent: rows per directory slice (slice = position >> dir_slice_shift); new rows are
   * refused in a slice at its limit, so that no region of the directory exceeds the load limit
   * even when a chunk is applied slice by slice */
  uint32_t slice_used[SMX_DIR_SLICES];
} smx_ctl_t;

typedef struct {
  smx_row_t* dir;
  uint64_t dir_cap;    /* entries, power of two                                             */
  uint32_t slice_shift; /* directory position >> slice_shift = slice index                  */
  uint32_t slice_limit; /* new rows are refused in a slice holding this many rows            */
  smx_ctl_t* ctl;
} smx_view_t;

typedef struct {
  const uint32_t* xs;
  const uint32_t* ys;
  const uint32_t* vs;  /* NULL: every value is v_const                                       */
  const uint32_t* idx; /* NULL: identity; else idx[p] = index of array position p in the caller's
                          input order (the batch was partitioned by directory slice)          */
  uint32_t v_const;
  uint32_t n;
} smx_ops_t;

typedef struct {
  uint32_t entry;      /* directory index of the growing row                                 */
  uint32_t newlog;     /* log2 of the new bucket capacity                                    */
  uint64_t off;        /* byte offset of the new bucket inside this round's slab region, or
                          SMX_PLAN_RECYCLED | address of a recycled bucket                      */
} smx_plan_t;

typedef struct {
  uint32_t* defer_out; /* [n]  ops turned away this round                                    */
  uint32_t* late;      /* [n]  ops parked for the LATE pass                                  */
  uint32_t* grow;      /* [n]  directory indices of rows queued for growth                   */
  uint32_t* t0rows;    /* [n]  row ids (x) whose column 0 turned non-zero in this chunk      */
  smx_plan_t* plan;    /* [n]                                                                */
  uint32_t* big;       /* [n]  plan indices of big rows                                      */
  uint32_t* mid;       /* [n]  plan indices of mid-size rows                                 */
} smx_lists_t;

enum { SMX_OP_INCR = 0, SMX_OP_DECR = 1, SMX_OP_SETZERO = 2 };
enum { SMX_PASS_COL0 = 0, SMX_PASS_EARLY = 1, SMX_PASS_LATE = 2 };

/* ---- launchers (smx_kernels.cu); `stream` is a cudaStream_t ------------------------------ */
typedef void* smx_stream_t;

void smx_launch_upsert(smx_stream_t stream, smx_view_t v, smx_ops_t ops, smx_lists_t l, int op,
                       int pass, const uint32_t* list, uint32_t m, int preaggregate);
void smx_launch_grow_plan(smx_stream_t stream, smx_view_t v, smx_lists_t l, uint32_t n_grow);
void smx_launch_free_push(smx_stream_t stream, smx_view_t v, smx_lists_t l, uint32_t n_grow);
void smx_launch_migrate(smx_stream_t stream, smx_view_t v, smx_lists_t l, uint32_t n_grow,
                        uint32_t n_mid, uint32_t n_big, void* region_base, int skip_big);
/* big rows, two steps: (1) every new bucket is built tile by tile in shared memory; cells that do not fit
 * their tile go to `spill` (capacity spill_cap entries of 16 bytes, length in ctl->n_spill — if it
 * exceeds the capacity the host enlarges the list and runs step 1 again: it only reads the old buckets);
 * (2) the spilled cells are inserted, the old buckets zeroed, the headers switched */
void smx_launch_migrate_tiles(smx_stream_t stream, smx_view_t v, smx_lists_t l, uint32_t n_big, void* region_base,
                              unsigned long long* spill, uint32_t spill_cap);
void smx_launch_migrate_tiles_finish(smx_stream_t stream, smx_view_t v, smx_lists_t l, uint32_t n_big, void* region_base,
                                     const unsigned long long* spill, uint32_t n_spill);
/* distinct-row estimate (linear counting): set bit hash(x) of a zeroed bitmap of 2^bits_log bits,
 * then count the zero bits into ctl->scratch */
void smx_launch_sketch(smx_stream_t stream, const uint32_t* xs, uint32_t n, uint32_t* bitmap,
                       uint32_t bits_log, smx_ctl_t* ctl);
void smx_launch_live_bytes(smx_stream_t stream, smx_view_t v); /* sum of 8 << caplog over slab buckets -> ctl->scratch */
void smx_launch_dir_rehash(smx_stream_t stream, smx_view_t from, smx_view_t to);
void smx_launch_finalize_t0(smx_stream_t stream, smx_view_t v, const uint32_t* t0rows, uint32_t n);
void smx_launch_sync_rowlen(smx_stream_t stream, smx_view_t v, const uint32_t* rows, uint32_t n);
void smx_launch_set_max(smx_stream_t stream, smx_view_t v, smx_ops_t ops, uint64_t* addrs);
void smx_launch_set_commit(smx_stream_t stream, smx_ops_t ops, uint64_t* addrs); /* mark + commit */
size_t smx_batch_out_sort_bytes(uint32_t n);
void smx_launch_batch_out(smx_stream_t stream, smx_view_t v, smx_ops_t ops, int op, uint32_t* out,
                          uint64_t* addrs_a, uint64_t* addrs_b, uint32_t* idx_a, uint32_t* idx_b,
                          uint64_t* seg, uint64_t* tile_agg, void* sort_tmp, size_t sort_bytes);
/* slice-ordered queries: one block per 4 x 256 consecutive queries, dispatched in order; once != 0: bucket
 * sectors are loaded evict-first */
void smx_launch_get_tiled(smx_stream_t stream, smx_view_t v, const uint32_t* xs, const uint32_t* ys,
                          uint32_t n, uint32_t* out, int once);
void smx_launch_get(smx_stream_t stream, smx_view_t v, const uint32_t* xs, const uint32_t* ys,
                    uint32_t n, uint32_t* out);
void smx_launch_rowlen(smx_stream_t stream, smx_view_t v, const uint32_t* xs, uint32_t n,
                       uint32_t* out);
void smx_launch_row_counts(smx_stream_t stream, smx_view_t v, const uint32_t* xs, uint32_t n,
                           uint32_t* counts, uint64_t* info /* nullable: directory index | caplog << 32 per row */,
                           uint32_t* big_list /* nullable */, uint32_t* big_counter);
void smx_launch_scan(smx_stream_t stream, const uint32_t* counts, uint32_t n, uint64_t base,
                     uint64_t* offsets /* n+1 */, uint64_t* block_sums /* scratch */);
void smx_launch_getrow_fill(smx_stream_t stream, smx_view_t v, const uint64_t* info, uint32_t n,
                            const uint64_t* offsets, uint64_t offset_bias, uint32_t* pairs,
                            const uint32_t* big_list, uint32_t n_big, uint32_t* cursors /* [n], zeroed */);
void smx_launch_count_nnz(smx_stream_t stream, smx_view_t v);
void smx_launch_sum_values(smx_stream_t stream, smx_view_t v, uint32_t* big_list /* [rows] */, uint32_t* big_counter /* zeroed */);
void smx_launch_sum_values_big(smx_stream_t stream, smx_view_t v, const uint32_t* big_list, uint32_t n_big);
void smx_launch_cf_scores(smx_stream_t stream, smx_view_t v, const uint32_t* items, uint32_t n,
                          const uint64_t* offsets, const uint32_t* pairs, uint32_t* ids, double* scores);
void smx_launch_pair_cols(smx_stream_t stream, const uint32_t* pairs, uint64_t total, uint32_t* cols);
void smx_launch_cf_scores_totals(smx_stream_t stream, uint32_t n, const uint64_t* offsets, const uint32_t* pairs,
                                 const uint32_t* a_tot, const uint32_t* b_tot, uint32_t* ids, double* scores);
/* top-k per segment (kernel comment in smx_kernels.cu).  offsets[0..n] index ids / scores; outputs are k slots
 * per segment.  Big segments: classify -> (host reads ctl) -> init -> passes until ctl[1] (segments still
 * selecting) is 0 -> finish.  ctl: 16 zeroed words (big count, active count, big pairs as u64, region cursor as
 * u64).  big_scratch: smx_topk_big_bytes(n_big) bytes, zeroed before init; c_ids / c_scores: big pairs slots. */
#define SMX_TOPK_MAX_K 1024u
size_t smx_topk_big_bytes(uint32_t n_big);
uint32_t smx_topk_max_passes(void); /* digits of the 96-bit key */
void smx_launch_topk_small(smx_stream_t stream, uint32_t n, const uint64_t* offsets, const uint32_t* ids,
                           const double* scores, uint32_t k, uint32_t* counts, uint32_t* out_ids, double* out_scores);
void smx_launch_topk_classify(smx_stream_t stream, uint32_t n, const uint64_t* offsets, uint32_t* big_list,
                              uint32_t* ctl);
void smx_launch_topk_init(smx_stream_t stream, const uint32_t* big_list, uint32_t n_big, const uint64_t* offsets,
                          void* big_scratch, uint32_t* ctl);
void smx_launch_topk_pass(smx_stream_t stream, void* big_scratch, uint32_t n_big, uint32_t k, const uint32_t* ids,
                          const double* scores, uint32_t* c_ids, double* c_scores, uint32_t* ctl);
void smx_launch_topk_finish(smx_stream_t stream, const void* big_scratch, uint32_t n_big, const uint32_t* c_ids,
                            const double* c_scores, uint32_t k, uint32_t* counts, uint32_t* out_ids, double* out_scores);
void smx_launch_topk_cut(smx_stream_t stream, const uint64_t* offsets, uint32_t n, uint32_t lo, uint64_t budget,
                         uint32_t* out);
/* basket recommendations (kernel comment in smx_kernels.cu).  A piece of nb baskets: boff[0..nb] absolute
 * positions, base = boff[0]; items indexed by position; off[0 .. boff[nb] - base] the per-position CSR of ids /
 * scores.  Order: rec_items (sorted item keys) -> rec_small (classify into ctl as top-k's: ctl[0] big count,
 * ctl[2..3] big pairs; small baskets into the staging arrays t_*, cnt[b] survivors) -> (host reads ctl) ->
 * rec_big (cnt of the big baskets) -> smx_launch_scan(cnt) = red_off -> rec_emit (the reduced CSR r_*).
 * sort_tmp: smx_rec_sort_bytes(max(n_pos, n_pairs)); scan_tmp: smx_scan_scratch_items(max(n_big, n_pairs)). */
size_t smx_rec_sort_bytes(uint32_t n);
void smx_launch_rec_items(smx_stream_t stream, uint32_t nb, const uint64_t* boff, uint64_t base, const uint32_t* items,
                          uint32_t n_pos, uint64_t* keys, uint64_t* sitems, void* sort_tmp, size_t sort_bytes);
void smx_launch_rec_small(smx_stream_t stream, uint32_t nb, const uint64_t* boff, uint64_t base, const uint64_t* off,
                          const uint32_t* ids, const double* scores, const uint64_t* sitems, uint32_t* big_list,
                          uint32_t* ctl, uint32_t* t_ids, double* t_scores, uint32_t* cnt);
void smx_launch_rec_big(smx_stream_t stream, const uint32_t* big_list, uint32_t n_big, uint32_t n_pairs,
                        const uint64_t* boff, uint64_t base, const uint64_t* off, const uint32_t* ids,
                        const uint64_t* sitems, uint32_t* lens, uint64_t* big_off /* n_big + 1 */, uint64_t* keys_a,
                        uint64_t* keys_b, uint32_t* vals_a, uint32_t* vals_b, uint32_t* flags,
                        uint64_t* fpos /* n_pairs + 1 */, uint64_t* scan_tmp, void* sort_tmp, size_t sort_bytes,
                        uint32_t* cnt);
void smx_launch_rec_emit(smx_stream_t stream, uint32_t nb, const uint64_t* boff, uint64_t base, const uint64_t* off,
                         const double* scores, const uint32_t* cnt, const uint64_t* red_off, const uint32_t* t_ids,
                         const double* t_scores, const uint32_t* big_list, uint32_t n_big, uint32_t n_pairs,
                         const uint64_t* big_off, const uint64_t* keys /* rec_big's keys_b */,
                         const uint32_t* vals /* vals_b */, const uint64_t* fpos, uint32_t* r_ids, double* r_scores);
/* one thread: out[0] = end of the piece of baskets from lo whose rows hold <= budget pairs (pos_off: positions'
 * pair offsets of the whole call) and <= item_budget items, at least one basket; out[1..2] = its positions */
void smx_launch_rec_cut(smx_stream_t stream, const uint64_t* pos_off, const uint64_t* boff, uint32_t nb, uint32_t lo,
                        uint64_t budget, uint64_t item_budget, uint32_t* out);
/* out[0] |= 1 if boff[0..nb] is not a valid basket CSR (starts at 0, never decreases, ends <= 2^32 - 2);
 * out[2..3] = boff[nb] as u64.  out[0] zeroed. */
void smx_launch_rec_check(smx_stream_t stream, const uint64_t* boff, uint32_t nb, uint32_t* out);
void smx_launch_list_rows(smx_stream_t stream, smx_view_t v, uint32_t* keys, uint32_t* counter /* zeroed */);
void smx_launch_row_slog(smx_stream_t stream, smx_view_t v, const uint32_t* xs, uint32_t n, uint32_t* out);
void smx_launch_snap_units(smx_stream_t stream, const uint32_t* counts, const uint32_t* slogs, uint32_t n,
                           uint32_t* units /* 2 + reference row size, in 8-byte units */);
void smx_launch_snap_rows(smx_stream_t stream, smx_view_t v, const uint64_t* info, uint32_t n,
                          const uint64_t* offsets /* n+1, 8-byte units */, uint64_t* out /* zeroed */,
                          const uint32_t* big_list, uint32_t n_big);
void smx_launch_load_fixup(smx_stream_t stream, smx_view_t v, const uint32_t* xs, const uint32_t* slogs,
                           uint32_t n);
/* a snapshot's row blocks on the device: `raw` is a window of file bytes, a tile is a row or a
 * 2^SMX_LOAD_TILE_LOG-cell part of one; count -> smx_launch_scan -> emit writes every row's
 * (key, 0, 0) op and then its cells with a non-zero value, in slot order */
#define SMX_LOAD_TILE_LOG 12u
#define SMX_LOAD_FIRST 0x80000000u /* smx_load_tile_t.cells: the row's first tile */
typedef struct {
  uint64_t off;   /* byte offset of the tile's first cell in the window */
  uint32_t key;   /* row id */
  uint32_t cells; /* cells in the tile | SMX_LOAD_FIRST */
} smx_load_tile_t;
void smx_launch_load_count(smx_stream_t stream, const void* raw, const smx_load_tile_t* tiles, uint32_t n,
                           uint32_t* counts);
void smx_launch_load_emit(smx_stream_t stream, const void* raw, const smx_load_tile_t* tiles, uint32_t n,
                          const uint64_t* offsets /* n + 1, from smx_launch_scan */, uint32_t* xs, uint32_t* ys,
                          uint32_t* vs);
void smx_launch_gen_c2_ops(smx_stream_t stream, uint64_t seed, uint64_t first, uint64_t count,
                           uint32_t rows, uint32_t ycols, uint32_t* xs, uint32_t* ys);
void smx_launch_gen_c2_queries(smx_stream_t stream, uint64_t seed_get, uint64_t seed_build,
                               uint64_t first, uint64_t count, uint64_t n_build, uint32_t rows,
                               uint32_t ycols, uint32_t* xs, uint32_t* ys);
void smx_launch_gen_c3_ops(smx_stream_t stream, uint64_t seed, uint64_t first, uint64_t count,
                           const uint64_t* thr, uint32_t items, uint32_t* xs, uint32_t* ys);
void smx_launch_gen_c3_queries(smx_stream_t stream, uint64_t seed_get, uint64_t seed_build,
                               uint64_t first, uint64_t count, uint64_t n_build, const uint64_t* thr,
                               uint32_t items, uint32_t* xs, uint32_t* ys);
void smx_launch_gen_c4_lens(smx_stream_t stream, uint64_t seed, uint64_t first, uint64_t count,
                            const uint64_t* thr, uint32_t kmax, uint32_t* lens);
void smx_launch_gen_c4_ops(smx_stream_t stream, uint64_t seed, uint64_t first, uint64_t count,
                           const uint64_t* offs, uint32_t rows, uint32_t* xs, uint32_t* ys, uint32_t* vs);
void smx_launch_probe_read(smx_stream_t stream, const void* buf, uint64_t n_units, uint64_t accesses,
                           int width, smx_ctl_t* ctl);
void smx_launch_probe_atomic(smx_stream_t stream, uint32_t* buf, uint64_t n_words, uint64_t accesses);
/* part = owner rank when shift == SMX_PART_OWNER, else directory slice (mix_row(x) & dir_mask) >> shift;
 * split0 != 0 (slice mode, world = 2 * split0): ops on column 0 go to parts split0 .. 2*split0-1 */
#define SMX_PART_OWNER 0xFFFFFFFFu
#define SMX_MAX_PARTS_H 256u
void smx_launch_partition_count(smx_stream_t stream, const uint32_t* xs, const uint32_t* ys /* or NULL */,
                                uint32_t n, uint32_t world, uint32_t dir_mask, uint32_t shift,
                                uint32_t split0, unsigned long long* counts /* [world], zeroed */);
void smx_launch_partition_scatter(smx_stream_t stream, const uint32_t* xs, const uint32_t* ys,
                                  const uint32_t* vs, uint32_t n, uint32_t world,
                                  uint32_t dir_mask, uint32_t shift, uint32_t split0,
                                  unsigned long long* cursors /* [world] start offsets */,
                                  uint32_t* oxs, uint32_t* oys, uint32_t* ovs, uint32_t* osrc,
                                  const uint32_t* src_in /* NULL: osrc = position; else osrc = src_in[position] */,
                                  uint32_t* opos /* nullable: opos[input position] = routed position */,
                                  const unsigned long long* dst_tab /* nullable, device: [5][world] =
                                     per-part x / y / v / src output bases + routed-position bases */,
                                  uint32_t src_bias /* added to every osrc value */);
void smx_launch_parts_prefix(smx_stream_t stream, const unsigned long long* counts, uint32_t parts,
                             unsigned long long* cursors /* [parts] = exclusive prefix of counts */);
void smx_launch_gather(smx_stream_t stream, uint32_t* out, const uint32_t* vals, const uint32_t* pos,
                       uint32_t n);
void smx_launch_gather_stride(smx_stream_t stream, uint32_t* out, const uint32_t* vals, const uint32_t* pos,
                              uint32_t n);
void smx_launch_route_offsets(smx_stream_t stream, const uint64_t* offs, const uint32_t* pos, uint32_t n,
                             uint32_t world, const unsigned long long* tab /* device: [2][world] */);
uint32_t smx_scan_scratch_items(uint32_t n); /* number of uint64 block sums smx_launch_scan needs */
int smx_grid_blocks(void);                   /* resident grid size used by the streaming kernels */

/* hash used by the router; host-callable */
uint32_t smx_owner_hash(uint32_t x);

#ifdef __cplusplus
}
#endif
#endif
