/*
 * include/smatrix_b200.h — device-side controls and measurement hooks of the B200 build.
 * Nothing here exists in the reference; bindings do not need it.  bench.py, the tests and the
 * multi-GPU router use it (through ctypes).
 */
#ifndef SMATRIX_B200_H
#define SMATRIX_B200_H

#include "smatrix.h"

#ifdef __cplusplus
extern "C" {
#endif

/* smatrix_open on an explicit CUDA device ordinal (smatrix_open uses $SMATRIX_DEVICE, default 0).
 * Environment read at open: SMATRIX_ARENA_GIB (reserve that much slab memory up front instead of
 * cudaMalloc'ing segments on demand), SMATRIX_CHUNK (ops per internal chunk, default 2^26),
 * SMATRIX_DIR_LOG2 (initial directory size), SMATRIX_PREAGG (warp pre-aggregation on/off),
 * SMATRIX_RECYCLE (free lists of vacated buckets on/off), SMATRIX_PRESIZE (distinct-row estimate
 * that sizes the directory before a chunk of new rows, on/off), SMATRIX_GET_SLICES / SMATRIX_GET_SLICE_MIN
 * (see smatrix_b200_set_get_slices), SMATRIX_WIDE_SLICES (default 1: a write chunk without ops on column 0
 * is ordered over 256 directory slices instead of 128 + their column-0 twins), SMATRIX_TOPK_PAIRS (default
 * 2^28: smatrix_cf_topk_batch scores and ranks the items of a call in pieces whose rows hold at most that
 * many pairs, 32 bytes of device scratch per pair; a row longer than that is a piece of its own.
 * smatrix_cf_recommend_batch cuts its baskets the same way, at basket boundaries, with up to about 100 bytes of
 * device scratch per pair; a basket whose rows hold more is a piece of its own). */
smatrix_t* smatrix_b200_open(const char* fname, int device);
/* the same with the slab arena given explicitly (bytes; 0 = segments on demand) instead of through
 * $SMATRIX_ARENA_GIB — for hosts that open several handles with different needs from several threads */
smatrix_t* smatrix_b200_open_arena(const char* fname, int device, size_t arena_bytes);

/* File-backed handles: write the snapshot NOW (temporary file, fsync, atomic rename) and return 0
 * on success, -1 on failure (or when the handle has no file).  The reference streams dirty rows to
 * its file continuously from an IO thread (src/smatrix.c:418-596); this build persists only here
 * and in smatrix_close, so a process that abort()s in between loses the updates since the last
 * snapshot — call this at the checkpoints the application can afford. */
int   smatrix_b200_snapshot(smatrix_t* self);

/* Device-level pieces of the snapshot, used by the multi-GPU router (every rank writes its part of ONE
 * .smx file, and reads a share of one).  The file is always the reference's format: 512-byte header,
 * chained directory blocks of 2^22 entries, then the row blocks.
 *   snap_extent    list this table's rows and lay out their row blocks: returns (rows, row-block bytes).
 *                  Holds the list until snap_write (or the next extent, or close).
 *   snap_rows_base where the row blocks start in a file of `total_rows` rows
 *   snap_layout    header and directory block headers of such a file into `fd`, and its final size
 *   snap_write     this table's row blocks at byte `byte_base` of fd and its directory entries from entry
 *                  `first_entry` on (entry e is slot e % 2^22 of block e / 2^22); 0 or -1
 *   snap_commit    rename(tmp, fname) and fsync of the directory that holds fname; 0 or -1
 * A table on its own (smatrix_b200_snapshot) is: extent, layout, write at snap_rows_base(rows), fsync,
 * commit. */
int      smatrix_b200_snap_extent(smatrix_t* self, uint64_t* rows, uint64_t* bytes);
uint64_t smatrix_b200_snap_rows_base(uint64_t total_rows);
int      smatrix_b200_snap_layout(int fd, uint64_t total_rows, uint64_t total_bytes);
int      smatrix_b200_snap_write(smatrix_t* self, int fd, uint64_t byte_base, uint64_t first_entry);
int      smatrix_b200_snap_commit(const char* tmp, const char* fname);
/* The reader of a .smx file: share `share` of `shares` (a contiguous range of directory entries, cut evenly)
 * is read in file order, window by window ($SMATRIX_LOAD_WINDOW bytes, default 64 MiB; a bigger row grows
 * it), every row header is checked on the host, and the device expands the raw row blocks into pieces of
 * at most $SMATRIX_LOAD_CELLS cells (default 2^24; a row never straddles two pieces).
 *   load_begin   NULL if the header or the directory is unreadable
 *   load_next    1 = a piece: the op stream (x, y, v; n_ops) as smatrix_set_batch takes it — per row
 *                (key, 0, 0) first, then its cells with a non-zero value in slot order — and the rows'
 *                (key, log2 row size) for load_fixup, which goes after the piece's ops.  DEVICE arrays of
 *                self's scratch, valid until the next call.  0 = the share is done, -1 = corrupt row.
 *   load_fixup   the rowlen state of loaded rows: S = the file's row size, d = (column 0 != 0) */
typedef struct smx_loader_s smx_loader_t;
smx_loader_t* smatrix_b200_load_begin(smatrix_t* self, int fd, int share, int shares);
int  smatrix_b200_load_next(smx_loader_t* ld, const uint32_t** d_xs, const uint32_t** d_ys, const uint32_t** d_vs,
                            size_t* n_ops, const uint32_t** d_keys, const uint32_t** d_logs, size_t* n_rows);
void smatrix_b200_load_end(smx_loader_t* ld);
void smatrix_b200_load_fixup(smatrix_t* self, const uint32_t* d_keys, const uint32_t* d_logs, size_t n);

int   smatrix_b200_device(smatrix_t* self);   /* CUDA device ordinal                            */
void* smatrix_b200_stream(smatrix_t* self);   /* the cudaStream_t every kernel is launched on   */
void  smatrix_b200_sync(smatrix_t* self);     /* cudaStreamSynchronize on that stream            */

/* CUDA-event timer on the library's own stream (torch.cuda.Event only sees torch's stream). */
void  smatrix_b200_timer_start(smatrix_t* self);
float smatrix_b200_timer_stop_ms(smatrix_t* self);   /* records, synchronises, returns elapsed ms */

enum {
  SMX_STAT_ROWS = 0,        /* rows in the directory                                      */
  SMX_STAT_NNZ = 1,         /* live cells incl. non-zero column 0 (scans the directory)   */
  SMX_STAT_DIR_CAP = 2,     /* directory capacity in entries                              */
  SMX_STAT_SLAB_BYTES = 3,  /* bytes handed out by the slab allocator                     */
  SMX_STAT_DEVICE_BYTES = 4,/* bytes of device memory held (directory + slab segments + scratch) */
  SMX_STAT_LAUNCHES = 5,    /* kernels launched by this handle so far                     */
  SMX_STAT_ROUNDS = 6,      /* upsert rounds (1 per pass + 1 per growth retry) so far     */
  SMX_STAT_ROW_GROWS = 7,   /* row growth (rehash) events so far                          */
  SMX_STAT_DIR_GROWS = 8,   /* directory rehash events so far                             */
  SMX_STAT_KERNEL_NS = 9,   /* device time of the dominant (update / get) kernels, ns, when timing is on */
  /* host wall-clock per phase of the write path since set_kernel_timing(1), ns */
  SMX_STAT_NS_PARTITION = 10, SMX_STAT_NS_UPSERT = 11, SMX_STAT_NS_GROW_PLAN = 12,
  SMX_STAT_NS_SLAB = 13, SMX_STAT_NS_MIGRATE = 14, SMX_STAT_NS_DIR = 15,
  SMX_STAT_VALUE_SUM = 16,  /* sum of every stored value mod 2^64 (scans the whole table) */
  SMX_STAT_LIVE_BUCKET_BYTES = 17, /* bytes of slab buckets rows own right now (scans the directory) */
  SMX_STAT_FREE_BYTES = 18, /* bytes of vacated buckets waiting on the free lists              */
  SMX_STAT_RECYCLED = 19,   /* row growths served from the free lists so far                   */
  SMX_STAT_H2D_BYTES = 20,  /* bytes copied host -> device by this handle so far (batches, tables) */
  SMX_STAT_D2H_BYTES = 21,  /* bytes copied device -> host (answers, control-block reads)      */
  SMX_STAT_BUCKET_BYTES = 22, /* slab bytes ever handed out for column buckets; / LIVE_BUCKET_BYTES = the
                                allocator's overhead (vacated buckets wait on the free lists)   */
  SMX_STAT_SPILLED = 23,    /* cells of big rows that did not fit their shared-memory tile during a re-placement */
  SMX_STAT_SLICED_GETS = 24,/* point reads answered in directory-slice order so far (see set_get_slices)  */
  SMX_STAT_WIDE_CHUNKS = 25,/* write chunks without ops on column 0 that were ordered over 256 slices ($SMATRIX_WIDE_SLICES) */
  SMX_STAT_NS_ALLOC = 26,   /* host time inside cudaMalloc on behalf of this handle so far, ns */
  SMX_STAT_ALLOCS = 27,     /* number of those cudaMalloc calls */
  SMX_STAT_TOPK_BIG = 28,   /* top-k segments (items) longer than 4096 pairs: ranked by the multi-block radix select */
  SMX_STAT_TOPK_PASSES = 29,/* digit passes that select ran so far */
  SMX_STAT_REC_BIG = 30     /* baskets longer than 4096 pairs: aggregated by the global sort of smatrix_cf_recommend_batch */
};
uint64_t smatrix_b200_stat(smatrix_t* self, int which);

/* When on, every update/get kernel launch is bracketed by CUDA events on the launch stream and
 * the sum is reported as SMX_STAT_KERNEL_NS (used for the roofline figure). */
void smatrix_b200_set_kernel_timing(smatrix_t* self, int on);

/* Point reads on device arrays (smatrix_get_batch): 0 = look every query up in input order; 1 (default,
 * $SMATRIX_GET_SLICES) = order a call's queries by directory slice first when there are at least
 * $SMATRIX_GET_SLICE_MIN (2^22) of them and at least one per two rows of the table (the directory
 * entries of a slice then stay in L2 and are fetched from DRAM once per row instead of once per query),
 * answers are put back into input order; 2 = always.  The answers are the same in every mode.
 * Measurement switches, OR-ed to the mode (B sides of the A/Bs in profiles/): 4 = bucket sectors with the
 * ordinary L2 priority instead of evict-first, 8 = 256 slices instead of 128, 16 = look-ups by the
 * resident-grid kernel of the input-order path, 32 = resident-grid gather. */
void smatrix_b200_set_get_slices(smatrix_t* self, int mode);

/* Pinned host memory (cudaHostAlloc) so that host-pointer batches overlap copy and update. */
void* smatrix_b200_host_alloc(size_t bytes);
void  smatrix_b200_host_free(void* p);

/* Plain device memory on the matrix's GPU, for callers that build batches on the device. */
void* smatrix_b200_dev_alloc(smatrix_t* self, size_t bytes);
void  smatrix_b200_dev_free(smatrix_t* self, void* p);
void  smatrix_b200_memcpy(smatrix_t* self, void* dst, const void* src, size_t bytes); /* any direction, synchronous */
void  smatrix_b200_memset0(smatrix_t* self, void* d_dst, size_t bytes);                /* zero device memory */

/* Synthetic streams of SURVEY.md 8(d), generated on the device (r = splitmix64(seed + i)):
 * C2 build ops [first, first+count) and C2 queries (odd j -> guaranteed miss). Device arrays. */
void smatrix_b200_gen_c2_ops(smatrix_t* self, uint64_t seed, uint64_t first, size_t count,
                             uint32_t rows, uint32_t ycols, uint32_t* d_xs, uint32_t* d_ys);
void smatrix_b200_gen_c2_queries(smatrix_t* self, uint64_t seed_get, uint64_t seed_build,
                                 uint64_t first, size_t count, uint64_t n_build, uint32_t rows,
                                 uint32_t ycols, uint32_t* d_xs, uint32_t* d_ys);

/* C3 (co-occurrence build, examples/cf_recommender.c:35-47) and C4 (Zipf row lengths) streams.
 * d_thr: inverse-CDF thresholds thr[k] = floor(2^64 * CDF(k+1)) (device array of `items` / `kmax`
 * uint64, last = 2^64 - 1), built by the caller (bench.py / oracle) so host and device draw from the
 * same table.  C3 op i: basket i/64 holds 8 Zipf item ids; op i%64 = (ids[n], 0) or (ids[n], ids[i']).
 * C3 query j: build op r % n_build, odd j with y moved out of range.  C4: lens[r] = draw(seed + r);
 * op i (given d_offs = exclusive prefix of lens, rows + 1 entries) = (r * 2654435761, a column that
 * is distinct inside row r and never 0, an odd value). */
void smatrix_b200_gen_c3_ops(smatrix_t* self, uint64_t seed, uint64_t first, size_t count,
                             const uint64_t* d_thr, uint32_t items, uint32_t* d_xs, uint32_t* d_ys);
void smatrix_b200_gen_c3_queries(smatrix_t* self, uint64_t seed_get, uint64_t seed_build, uint64_t first,
                                 size_t count, uint64_t n_build, const uint64_t* d_thr, uint32_t items,
                                 uint32_t* d_xs, uint32_t* d_ys);
void smatrix_b200_gen_c4_lens(smatrix_t* self, uint64_t seed, uint64_t first, size_t count,
                              const uint64_t* d_thr, uint32_t kmax, uint32_t* d_lens);
void smatrix_b200_gen_c4_ops(smatrix_t* self, uint64_t seed, uint64_t first, size_t count,
                             const uint64_t* d_offs, uint32_t rows, uint32_t* d_xs, uint32_t* d_ys,
                             uint32_t* d_vs);

/* Roofline denominators measured in the same process: random 32 B-sector reads and random 4 B
 * atomic adds over a `footprint_bytes` device buffer (`accesses` of them, counter-based
 * addresses).  Return achieved accesses per second. `width` = bytes per access (4/8/16/32). */
double smatrix_b200_probe_random_read(smatrix_t* self, size_t footprint_bytes, size_t accesses, int width);
double smatrix_b200_probe_random_atomic(smatrix_t* self, size_t footprint_bytes, size_t accesses);

/* Multi-GPU router, device side (K8).  smatrix_b200_owner: the rank that owns row x in a world of
 * `world` ranks (include/smatrix_shard.h).  smatrix_b200_gather(out, vals, pos, n):
 * out[i] = vals[pos[i]] puts answers that came back in routed order into input order; all three
 * arrays are DEVICE pointers. */
uint32_t smatrix_b200_owner(uint32_t x, uint32_t world);
void smatrix_b200_gather(smatrix_t* self, uint32_t* d_out, const uint32_t* d_vals,
                         const uint32_t* d_pos, size_t n);

/* K8 fused with the exchange (peer memory over NVLink instead of an NCCL all-to-all).
 * smatrix_b200_partition_count: ops per owner for a device batch.
 * smatrix_b200_route_p2p: bucket by owner and write every owner's run straight to the addresses in
 *   h_dst[5][world] = { x, y, v, src (0 = not wanted) output bases, routed-position bases } — local
 *   memory or peer mappings obtained with smatrix_b200_ipc_open (cudaIpc handles of buffers that a
 *   peer allocated with smatrix_b200_dev_alloc and exported with smatrix_b200_ipc_export).  src
 *   values are (index in this batch + src_bias); d_out_pos (nullable) receives, per op, its
 *   position in routed order (pos_base[owner] + index inside the owner's run). */
void smatrix_b200_partition_count(smatrix_t* self, const uint32_t* d_xs, size_t n, uint32_t world,
                                  uint64_t* h_counts);
void smatrix_b200_route_p2p(smatrix_t* self, const uint32_t* d_xs, const uint32_t* d_ys,
                            const uint32_t* d_vals, size_t n, uint32_t world, const uint64_t* h_dst,
                            uint32_t src_bias, uint32_t* d_out_pos);
int   smatrix_b200_ipc_export(smatrix_t* self, void* dptr, unsigned char* handle64);
void* smatrix_b200_ipc_open(smatrix_t* self, const unsigned char* handle64);
void  smatrix_b200_ipc_close(smatrix_t* self, void* p);

/* Device-level pieces of smatrix_getrow_batch, used by the multi-GPU router (an owner answers rows
 * that another rank asked for and writes the pairs straight into that rank's buffer):
 *   row_counts_batch  d_counts[i] = pairs row d_xs[i] would return (0 if the row does not exist)
 *   scan_counts       d_offsets[0..n] = exclusive prefix of d_counts; returns the total
 *   getrow_fill_at    row i's pairs go to d_pairs + 2 * d_offsets[i] (local or peer memory)
 *   route_offsets     the requester's side: offset of row i goes to the owner that holds the row,
 *                     h_tab[2][world] = { first routed position of every owner's run, address of
 *                     that owner's offset array } */
void     smatrix_b200_row_counts_batch(smatrix_t* self, const uint32_t* d_xs, size_t n, uint32_t* d_counts);
uint64_t smatrix_b200_scan_counts(smatrix_t* self, const uint32_t* d_counts, size_t n, uint64_t* d_offsets);
void     smatrix_b200_getrow_fill_at(smatrix_t* self, const uint32_t* d_xs, size_t n,
                                     const uint64_t* d_offsets, uint32_t* d_pairs);
void     smatrix_b200_route_offsets(smatrix_t* self, const uint64_t* d_offsets, const uint32_t* d_pos,
                                    size_t n, uint32_t world, const uint64_t* h_tab);
/* CF read side when the totals live on other shards: columns of a pairs array, and the scores of
 * smatrix_cf_neighbors_batch from pre-fetched totals (a_tot per item, b_tot per pair) */
void smatrix_b200_pair_cols(smatrix_t* self, const uint32_t* d_pairs, uint64_t total, uint32_t* d_cols);
void smatrix_b200_cf_scores_totals(smatrix_t* self, size_t n, const uint64_t* d_offsets, const uint32_t* d_pairs,
                                   const uint32_t* d_a_tot, const uint32_t* d_b_tot, uint32_t* d_ids,
                                   double* d_scores);
/* The selection of smatrix_cf_topk_batch over any CSR of (id, double) pairs on the device: segment i is
 * d_ids / d_scores[d_offsets[i] .. d_offsets[i+1]); its first min(k, len) pairs by score descending, then id
 * ascending, go to d_counts[i] and row i of d_out_ids / d_out_scores[n*k] (slots past the count: id
 * 0xFFFFFFFF, score -1.0).  Ids must be unique inside a segment.  1 <= k <= 1024.  All arrays DEVICE. */
void smatrix_b200_topk_segments(smatrix_t* self, size_t n, const uint64_t* d_offsets, const uint32_t* d_ids,
                                const double* d_scores, uint32_t k, uint32_t* d_counts, uint32_t* d_out_ids,
                                double* d_out_scores);
/* The aggregation and ranking of smatrix_cf_recommend_batch over neighbour lists that are already on the device:
 * basket i is positions d_basket_off[i] .. d_basket_off[i+1] (n + 1 entries, d_basket_off[0] = 0) of d_items,
 * and position j's list is d_ids / d_scores[d_offsets[j] .. d_offsets[j+1]), the layout smatrix_cf_neighbors_batch
 * produces.  Candidates, summation order, exclusions and the fixed-width outputs are those of
 * smatrix_cf_recommend_batch.  1 <= k <= 1024.  All arrays DEVICE. */
void smatrix_b200_basket_topk(smatrix_t* self, size_t n_baskets, const uint64_t* d_basket_off, const uint32_t* d_items,
                              const uint64_t* d_offsets, const uint32_t* d_ids, const double* d_scores, uint32_t k,
                              uint32_t* d_counts, uint32_t* d_out_ids, double* d_out_scores);
int  smatrix_b200_is_device_ptr(smatrix_t* self, const void* p);   /* device (or managed) memory? */
/* peers in the SAME process (one thread per GPU) need no IPC: enable direct access to `peer_device` */
int  smatrix_b200_enable_peer(smatrix_t* self, int peer_device);
/* asynchronous copy (any direction) on side stream `lane` (0..2); lane_sync waits for that lane */
void smatrix_b200_memcpy_async(smatrix_t* self, void* dst, const void* src, size_t bytes, int lane);
void smatrix_b200_lane_sync(smatrix_t* self, int lane);

/* smatrix_{incr,decr,set}_batch (op = 0, 1, 2) on DEVICE arrays whose "input order" is given
 * explicitly: d_ords[i] (unique, < 2^32 - 1) is op i's place in the sequential order the result
 * must be equal to.  Used by the multi-GPU router, where ops arrive permuted: the order decides
 * which duplicate `set` wins and the history-dependent rowlen (SURVEY.md Q1).  One chunk per call. */
void smatrix_b200_apply_ordered(smatrix_t* self, int op, const uint32_t* d_xs, const uint32_t* d_ys,
                                const uint32_t* d_vals, const uint32_t* d_ords, size_t n);

/* the same, additionally returning every op's value as if the batch had been applied one op at a time in
 * the order d_ords gives (smatrix_*_batch_out for permuted batches; used by the multi-GPU router) */
void smatrix_b200_apply_ordered_out(smatrix_t* self, int op, const uint32_t* d_xs, const uint32_t* d_ys,
                                    const uint32_t* d_vals, const uint32_t* d_ords, size_t n, uint32_t* d_out);

#ifdef __cplusplus
}
#endif
#endif
