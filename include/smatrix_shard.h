/*
 * include/smatrix_shard.h — one matrix row-sharded over the GPUs of one box, behind a C handle
 * (new; the reference is single-node shared memory and has nothing to replace here — the
 * semantics every call must reproduce are those of src/smatrix.h:87-94 applied to ONE matrix).
 *
 *     owner(x) = smatrix_b200_owner(x, world)          rows are hash-partitioned by row id
 *
 * One RANK per GPU.  Ranks are threads of one process (a JNI / Ruby / C host driving several GPUs)
 * or separate processes (one per GPU, e.g. under torchrun) — the library does not care: ranks find
 * each other through a small POSIX shared-memory segment named by the caller, exchange the
 * addresses (same process) or CUDA IPC handles (other processes) of their inboxes once, and from
 * then on a batch is routed with plain stores over NVLink / NVSwitch from inside the partition
 * kernel (k_partition_scatter writes every owner's run straight into that owner's inbox); the only
 * per-batch host traffic is the world x world count matrix and two barriers in shared memory.
 * No NCCL, no MPI, no Python on the data path.
 *
 * Every batch call is COLLECTIVE: all ranks call it (in the same order), each with ITS slice of
 * the batch; a rank may pass n = 0.  "Input order" of the collective batch is the concatenation of
 * the slices in rank order.  Arrays may be host or device pointers (device pointers must be on the
 * rank's own GPU); host arrays are staged piece by piece, uploads overlapping the routing.
 * Errors follow the reference (src/smatrix.c:891-894): "libsmatrix error: ..." on stdout + abort();
 * a rank that dies flags the segment so that its peers stop waiting instead of hanging.
 */
#ifndef SMATRIX_SHARD_H
#define SMATRIX_SHARD_H

#include "smatrix.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct smatrix_shard_s smatrix_shard_t;

/* Collective.  `name`: job-unique rendezvous name ("/dev/shm/<name>"), the same on every rank;
 * device: CUDA ordinal of this rank's GPU.  Returns NULL if CUDA is unusable or the peers' memory
 * cannot be mapped (then on EVERY rank: the outcome is agreed on before anyone returns).
 * $SMATRIX_SHARD_TIMEOUT (seconds, default 300): how long a rank waits for its peers. */
smatrix_shard_t* smatrix_b200_shard_open(const char* name, int rank, int world, int device);
/* the same with this rank's slab arena given explicitly (bytes; 0 = on demand) instead of $SMATRIX_ARENA_GIB */
smatrix_shard_t* smatrix_b200_shard_open_arena(const char* name, int rank, int world, int device, size_t arena_bytes);
/* Collective.  Like smatrix_b200_shard_open_arena, plus file mode as in smatrix_open(fname): the matrix is
 * loaded from `fname` if the file exists and is non-empty, and written back by smatrix_b200_shard_close.
 * Every rank passes the same path.  Returns NULL on EVERY rank if any rank fails: the file cannot be
 * opened or is corrupt, the paths differ, or the usual set-up failures.  A file that could not be read
 * is never overwritten.
 * The file is one ordinary .smx file in the reference's format, without sharding metadata: a file written
 * at one world size loads at any other, on one GPU through smatrix_open, and in the reference; a single-GPU
 * or reference file loads sharded.  Every rank reads an even share of the file's directory, expands its row
 * blocks on its GPU and routes the rows to their owners.
 * Durability is that of a single-GPU handle (smatrix_b200_snapshot): the matrix is persisted only by
 * smatrix_b200_shard_snapshot and smatrix_b200_shard_close, so a job that dies in between loses the updates
 * since the last snapshot. */
smatrix_shard_t* smatrix_b200_shard_open_file(const char* name, int rank, int world, int device,
                                              size_t arena_bytes, const char* fname);
/* Collective: write the snapshot now.  The file goes to a temporary name (`fname.tmp`, laid out by rank 0,
 * then every rank writes its own rows' row blocks and directory entries into it in parallel and fsyncs),
 * and rank 0 renames it over the old one and syncs the directory.  Returns 0 on every rank, or -1 on every
 * rank when no rank has a file or any step failed; a failed snapshot leaves the previous file intact. */
int smatrix_b200_shard_snapshot(smatrix_shard_t* self);
/* Collective.  With a file (smatrix_b200_shard_open_file) the snapshot is written first; if that fails,
 * the same message as smatrix_close's goes to stdout and the matrix is closed anyway. */
void smatrix_b200_shard_close(smatrix_shard_t* self);
smatrix_t* smatrix_b200_shard_local(smatrix_shard_t* self);      /* this rank's own table (stats, timers) */
int smatrix_b200_shard_rank(smatrix_shard_t* self);
int smatrix_b200_shard_world(smatrix_shard_t* self);

/* Optional, collective: size the inboxes for batches of up to max_ops ops per rank and the row
 * buffers for getrow answers of up to max_pairs pairs per rank now (they grow on demand otherwise),
 * e.g. to keep allocation and IPC set-up out of a timed region. */
void smatrix_b200_shard_reserve(smatrix_shard_t* self, size_t max_ops, size_t max_pairs);

/* n x smatrix_incr / decr / set on the sharded matrix (src/smatrix.c:225-256).
 * ordered != 0: every op travels with its global input-order index and the owners apply the batch
 * bit-exactly as if it had been applied sequentially (duplicate `set`, history-dependent rowlen,
 * SURVEY.md Q1); ordered == 0 is for incr / decr streams that never write column 0, where nothing
 * depends on the order (addition mod 2^32 commutes).  vals == NULL (on every rank): all values 1. */
void smatrix_b200_shard_incr_batch(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                   const uint32_t* vals, size_t n, int ordered);
void smatrix_b200_shard_decr_batch(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                   const uint32_t* vals, size_t n, int ordered);
void smatrix_b200_shard_set_batch(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                  const uint32_t* vals, size_t n);

/* The same three, additionally returning what every single call would have returned (out[i] = value of the
 * cell right after op i when the COLLECTIVE batch is applied one op at a time in input order; same contract
 * as smatrix_*_batch_out, src/smatrix.c:230,241,252).  Always ordered; one piece per call. */
void smatrix_b200_shard_incr_batch_out(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                       const uint32_t* vals, size_t n, uint32_t* out);
void smatrix_b200_shard_decr_batch_out(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                       const uint32_t* vals, size_t n, uint32_t* out);
void smatrix_b200_shard_set_batch_out(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                      const uint32_t* vals, size_t n, uint32_t* out);

/* n x smatrix_get / smatrix_rowlen (src/smatrix.c:174-185, :212-223): queries travel to the owners,
 * the owners' kernels write the answers straight into the asking rank's buffer. */
void smatrix_b200_shard_get_batch(smatrix_shard_t* self, const uint32_t* xs, const uint32_t* ys,
                                  size_t n, uint32_t* out);
void smatrix_b200_shard_rowlen_batch(smatrix_shard_t* self, const uint32_t* xs, size_t n, uint32_t* out);

/* n x smatrix_getrow with full-size buffers (src/smatrix.c:189-210) as CSR, same contract as
 * smatrix_getrow_batch: offsets[0..n], pairs with capacity pairs_cap PAIRS, size query with
 * pairs == NULL; returns the total.  Row ids go to their owners, the owners count, the asking rank
 * scans the counts into offsets (input order), sends every row's offset back, and the owners'
 * compaction kernels write the pairs into the asking rank's row buffer over NVLink. */
uint64_t smatrix_b200_shard_getrow_batch(smatrix_shard_t* self, const uint32_t* xs, size_t n,
                                         uint64_t* offsets, uint32_t* pairs, uint64_t pairs_cap);

/* The read side of the co-occurrence recommender across ranks (examples/cf_recommender.c:50-86): same
 * contract as smatrix_cf_neighbors_batch (offsets[0..n], ids / scores with capacity `cap`, size query
 * with ids == NULL).  Rows come through the getrow route, the totals at column 0 through two sharded
 * gets, scores are bit-exact doubles. */
uint64_t smatrix_b200_shard_cf_neighbors_batch(smatrix_shard_t* self, const uint32_t* items, size_t n,
                                               uint64_t* offsets, uint32_t* ids, double* scores, uint64_t cap);

/* The top k neighbours of this rank's items across ranks: same contract as smatrix_cf_topk_batch (counts[n],
 * ids / scores[n*k], 1 <= k <= 1024).  The scores come as in smatrix_b200_shard_cf_neighbors_batch and are
 * ranked by smatrix_b200_topk_segments on this rank's GPU.  One piece per call: this rank's row buffer and
 * scratch hold all the pairs of its items at once, as cf_neighbors_batch needs for a full fill. */
void smatrix_b200_shard_cf_topk_batch(smatrix_shard_t* self, const uint32_t* items, size_t n, uint32_t k,
                                      uint32_t* counts, uint32_t* ids, double* scores);

/* Basket recommendations for this rank's baskets across ranks: same contract as smatrix_cf_recommend_batch
 * (basket_off[n_baskets + 1], items, counts[n], ids / scores[n*k], 1 <= k <= 1024; a rank may pass no baskets).
 * The lists of the flattened items come as in smatrix_b200_shard_cf_neighbors_batch and are aggregated and ranked
 * by smatrix_b200_basket_topk on this rank's GPU, so the answers equal the single-GPU ones bit for bit at every
 * world size.  One piece per call, as smatrix_b200_shard_cf_topk_batch. */
void smatrix_b200_shard_cf_recommend_batch(smatrix_shard_t* self, const uint64_t* basket_off, const uint32_t* items,
                                           size_t n_baskets, uint32_t k, uint32_t* counts, uint32_t* ids,
                                           double* scores);

/* Host wall-clock accounting of this rank since the last reset (not collective): time spent routing
 * (count, count exchange, scatter over NVLink, arrival barrier), time spent applying the inbox,
 * number of routes, bytes this rank stored into OTHER ranks' inboxes. */
enum { SMX_SHARD_STAT_ROUTE_NS = 0, SMX_SHARD_STAT_APPLY_NS = 1, SMX_SHARD_STAT_ROUTES = 2,
       SMX_SHARD_STAT_REMOTE_BYTES = 3,
       SMX_SHARD_STAT_MAX_INBOX_OPS = 4 /* largest inbox any routed batch needed so far (the same on every rank;
                                           not reset): hash-sharding a skewed stream sends the hottest rows' ops to
                                           ONE owner, so size smatrix_b200_shard_reserve from a warm-up's value */ };
uint64_t smatrix_b200_shard_stat(smatrix_shard_t* self, int which);
void smatrix_b200_shard_stat_reset(smatrix_shard_t* self);

/* collective helpers (shared-memory barrier / sum over ranks), for hosts without another transport */
void smatrix_b200_shard_barrier(smatrix_shard_t* self);
uint64_t smatrix_b200_shard_sum(smatrix_shard_t* self, uint64_t v);
uint64_t smatrix_b200_shard_max(smatrix_shard_t* self, uint64_t v);

#ifdef __cplusplus
}
#endif
#endif
