/*
 * smx_host.c — the host side of the B200 libsmatrix hot path, in C like the reference.
 *
 * Exports the reference's 8-function API (include/smatrix.h, reference src/smatrix.h:87-94),
 * the batched entry points (include/smatrix_batch.h) and the device controls
 * (include/smatrix_b200.h).  All computation happens in the CUDA kernels of smx_kernels.cu;
 * this file only owns memory, ordering and the retry/growth loop.  There is no CPU compute
 * path: if CUDA is unusable, smatrix_open fails.
 *
 * One write batch ("chunk", <= SMATRIX_CHUNK ops) is applied as
 *     COL0 pass  -> column-0 ops (they live in the row header and define t0, see DESIGN.md)
 *     EARLY pass -> all other ops, except those ordered after t0 in a row whose column 0
 *                   turns non-zero inside this chunk
 *     LATE pass  -> those parked ops
 *     (set only) max-index + commit passes: last writer in input order wins
 * and every pass is a loop of rounds: launch, read the control block, and if ops were turned
 * away (bucket or directory at its load limit) grow and re-run only those ops.
 */
#define _GNU_SOURCE
#include <cuda_runtime_api.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <sys/types.h>
#include <unistd.h>

#include "../../include/smatrix.h"
#include "../../include/smatrix_b200.h"
#include "../../include/smatrix_batch.h"
#include "smx_internal.h"

#define SMX_DIR_LOG_DEFAULT 20u
#define SMX_CHUNK_DEFAULT (1u << 26) /* measured on B200: 5.17 vs 5.50 ms per 2^26 ops with 2^25 (profiles/r2_summary.md) */
#define SMX_STAGE_MAX (1u << 23) /* host-pointer batches: piece size with the best copy/update overlap (measured) */
#define SMX_SEG_MIN ((size_t)64 << 20)
#define SMX_SEG_MAX ((size_t)16 << 30)
#define SMX_MAX_ROUNDS 128

typedef struct {
  char* base;
  size_t size;
  size_t used;
  int owned; /* cudaMalloc'ed by us (freed at close); 0 = a block given back to the slab, e.g. a replaced directory */
} smx_seg_t;

typedef struct { void* p; size_t bytes; } smx_dbuf_t; /* device scratch that grows on demand (dbuf_need) */

/* Pinned host words that small device answers are read back into, and a single op's arguments go up from: one
 * field per value, so that no two uses share a slot. */
typedef struct {
  uint32_t op[3];      /* single ops: x, y, value on their way to d_small[DS_X..DS_V] */
  uint32_t answer;     /* single ops: the value or row length (d_small[DS_OUT]) */
  uint64_t row_total;  /* pairs of the rows of a getrow plan / of smatrix_b200_scan_counts (the last offset) */
  uint32_t n_big_rows; /* rows of a getrow plan that the whole grid compacts */
  uint32_t n_spill;    /* cells the tile-wise re-placement could not place in their tile */
  uint32_t probe_max;  /* largest probe step of a directory rehash */
  uint32_t n_big_sums; /* SMX_STAT_VALUE_SUM: rows with a big bucket, summed by a launch of their own */
  uint32_t topk_cut;   /* end of the next piece of a cf_topk_batch call */
  struct { uint32_t n_big, active; uint64_t big_pairs; } topk; /* control words 0..3 of a top-k selection */
  uint32_t rec_cut[3]; /* end of the next piece of a cf_recommend_batch call, its first and end position */
  struct { uint32_t bad, pad; uint64_t n_pos; } rec_check; /* device basket offsets: malformed?, positions */
  struct { uint32_t n_big, pad; uint64_t big_pairs; } rec;  /* big baskets of a piece and their pairs */
  struct { uint32_t n_big, pad; uint64_t big_pairs; } sort; /* big segments of a sort_rows call and their pairs */
  struct { uint32_t end, pad; uint64_t pairs; } sort_cut;   /* end of the next group of big segments, its pairs */
  uint32_t listed;     /* rows smatrix_list_rows found */
  uint32_t ck_missing; /* old directory entries of a checkpoint whose row is not in the table */
  uint64_t ck_kept;    /* ... and the number of them the keep filter kept (its last offset) */
} smx_small_t;
enum { DS_X, DS_Y, DS_V, DS_OUT, DS_WORDS }; /* the words of d_small: a single op's arguments, a one-word answer */

struct smatrix_s {
  int device;
  int prev_device; /* the caller's current device, restored by leave() */
  cudaStream_t stream;
  cudaStream_t copy_stream;
  cudaStream_t read_stream[2]; /* with stream + copy_stream: four pieces of a host-pointer read in flight */
  pthread_mutex_t mu;

  smx_row_t* dir;
  int dir_in_arena; /* the directory was carved from the slab arena: never cudaFree'd on its own */
  uint64_t dir_cap;
  uint32_t dir_log_min;
  uint64_t shrink_refused; /* largest directory size a shrink was refused at (a row would sit too far from home) */
  smx_ctl_t* d_ctl;
  smx_ctl_t* h_ctl; /* pinned */

  smx_seg_t* segs;
  int nsegs, segs_cap;
  size_t slab_bytes; /* handed out */
  size_t seg_bytes;  /* held */
  size_t arena_bytes; /* slab memory reserved at open (SMATRIX_ARENA_GIB) */

  uint32_t chunk_max;
  uint32_t list_cap;
  uint32_t* defer[2];
  smx_lists_t lists;
  uint64_t* addrs;
  uint32_t addrs_cap;

  uint32_t stage_cap;
  uint32_t stage_max; /* ops per staged piece of a host-pointer batch (SMATRIX_STAGE) */
  uint32_t* stage[2][3];
  cudaEvent_t stage_ready[2];

  uint32_t* part[4]; /* chunk partitioned by directory slice: xs, ys, vs, original index */
  uint32_t part_cap;
  uint32_t part_min; /* chunks smaller than this are applied in input order */
  uint32_t slice_log; /* log2(directory entries per slice) */
  uint32_t parts_log_max; /* at most 2^this slices (<= 7: with their column-0 twins that is 256 parts) */
  int wide_slices;        /* SMATRIX_WIDE_SLICES: chunks without ops on column 0 use 256 slices */


  uint32_t* d_small; /* DS_WORDS words */
  smx_small_t* h_small; /* pinned */

  /* scratch that grows with slack (dbuf_need), so that calls of similar size make no cudaMalloc; freed at close.
   * Only smx_dbuf_t members: smatrix_close and SMX_STAT_DEVICE_BYTES walk it as an array. */
  struct {
    smx_dbuf_t tmp, tmp64; /* general temp: ids on their way up, counts, partition counters (u32 / u64 words) */
    smx_dbuf_t plan;       /* getrow plan (rowplan) */
    smx_dbuf_t rows;       /* pairs of whole rows on their way to host outputs, scores or a snapshot */
    smx_dbuf_t host_out;   /* cf_neighbors_batch / cf_topk_batch answers on their way to host outputs */
    smx_dbuf_t spill;      /* cells that did not fit their tile (16 bytes each) */
    /* *_batch_out (exact per-op return values) */
    smx_dbuf_t bo_addr[2], bo_idx[2], bo_seg, bo_tiles, bo_out, bo_sort;
    /* top-k (smatrix_cf_topk_batch, smatrix_b200_topk_segments) */
    smx_dbuf_t tk_ctl;     /* 16 control words + the list of big segments (also of smatrix_b200_sort_rows) */
    smx_dbuf_t tk_off;     /* row offsets of the whole call (piece cuts) */
    smx_dbuf_t tk_big;     /* select state + histograms of the big segments */
    smx_dbuf_t tk_cids, tk_cscores; /* compaction regions of the big segments */
    smx_dbuf_t tk_ids, tk_scores;   /* scores of a piece */
    /* basket recommendations (smatrix_cf_recommend_batch, smatrix_b200_basket_topk): the call's offsets and items
     * on their way up, its positions' row counts and pair offsets, control words + big list + survivor counts,
     * sorted item keys, the radix sorts' storage, staged survivors, reduced offsets and the reduced CSR, and the
     * big baskets' lengths / offsets, sort keys, values, marks and their scan */
    smx_dbuf_t rc_in, rc_pos, rc_ctl, rc_items, rc_sort, rc_tids, rc_tscores, rc_red, rc_rids, rc_rscores;
    smx_dbuf_t rc_big, rc_keys, rc_vals, rc_flags;
    /* rows sorted by column (smatrix_b200_sort_rows): the big segments' lengths, offsets and scan, the sort keys and
     * values of a group of them, the radix sort's storage; the listing (smatrix_list_rows): the keys as found and
     * sorted, its radix sort's storage */
    smx_dbuf_t sr_big, sr_keys, sr_vals, sr_sort, ls_keys, ls_sort;
    /* loading a snapshot (smatrix_b200_load_next): a window of file bytes, its tiles, their counts and offsets,
     * the op stream (x, y, v) and the (key, log2 size) fixups of a piece */
    smx_dbuf_t ld_raw, ld_tiles, ld_cnt, ld_off, ld_ops, ld_fix;
    /* checkpoints (smatrix_b200_ckpt_keep): old directory entries on their way up (key, row offset lo / hi), their
     * keep flags, its scan and the kept entries packed as in the file */
    smx_dbuf_t ck_in, ck_flags, ck_off, ck_out;
  } db;
  uint32_t topk_pairs;  /* SMATRIX_TOPK_PAIRS: pairs per piece of a cf_topk_batch call */
  uint64_t n_topk_big, n_topk_passes;
  uint64_t n_rec_big; /* SMX_STAT_REC_BIG */
  uint64_t n_sort_big; /* SMX_STAT_SORT_BIG */

  unsigned long long* free_ptr[SMX_CLASSES]; /* device stacks of vacated buckets, per size class */
  uint32_t free_cap[SMX_CLASSES];
  int debug;                                 /* SMATRIX_DEBUG: growth decisions on stderr */
  int migrate_tiles;                         /* SMATRIX_MIGRATE_TILES (default 1): big rows are re-placed tile by tile in shared memory */
  uint32_t spill_cap;                        /* cells the spill list (db.spill) is sized for */
  uint64_t n_spilled;
  int recycle;                               /* SMATRIX_RECYCLE (default 1) */
  int presize;                               /* SMATRIX_PRESIZE (default 1): distinct-row estimate before a chunk of new rows */
  int get_slices;                            /* SMATRIX_GET_SLICES: 0 = point reads in input order, 1 (default) = by directory slice
                                              * when the batch revisits rows often enough, 2 = always */
  int get_flags;                             /* measurement switches of the slice-ordered look-up (SMX_GET_*) */
  uint32_t get_slice_min;                    /* SMATRIX_GET_SLICE_MIN (2^22): smaller calls are looked up in input order */
  uint64_t n_sliced_gets;                    /* queries answered through the slice-ordered path */
  uint64_t n_wide_chunks;                    /* write chunks ordered over 256 slices (no ops on column 0) */
  double alloc_ns;                           /* host time spent inside cudaMalloc by this handle */
  uint64_t n_allocs;

  uint64_t n_launches, n_rounds, n_row_grows, n_dir_grows, n_recycled;
  uint64_t bucket_bytes;         /* slab bytes handed out for column buckets (fresh, not recycled) */
  uint64_t h2d_bytes, d2h_bytes; /* bytes this handle copied between host and device (SMX_STAT_*_BYTES) */
  double phase_ns[8];
  int timing;
  cudaEvent_t ev0, ev1, t_start, t_stop;
  double kernel_ns;
  int preagg;
  char* fname;
  uint32_t* snap_keys; /* the rows smatrix_b200_snap_extent listed, until smatrix_b200_snap_write */
  uint64_t snap_rows;
  uint64_t* snap_hoff; /* a table of one chunk of rows: its layout (offsets, keys, big rows) as snap_extent */
  uint32_t* snap_hkeys; /* read it back, so that snap_write neither lays it out nor reads it again */
  int ck_base;          /* the file matched the table at some point (a load, a snapshot or a checkpoint) */
  unsigned char* ck_kept; /* kept directory entries of the checkpoint in progress (12 bytes each, file order) */
  uint64_t ck_kept_n, ck_kept_cap;
};

/* ------------------------------------------------------------------------------ errors */
static void smx_die(const char* fmt, ...) { /* reference src/smatrix.c:891-894 */
  va_list ap;
  printf("libsmatrix error: ");
  va_start(ap, fmt);
  vprintf(fmt, ap);
  va_end(ap);
  printf("\n");
  fflush(stdout);
  abort();
}
#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t e_ = (call);                                                            \
    if (e_ != cudaSuccess) smx_die("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                   __FILE__, __LINE__);                                 \
  } while (0)

static uint32_t env_u32(const char* name, uint32_t dflt) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  return (uint32_t)strtoul(v, NULL, 0);
}

static inline double now_ns(void);
static void* dmalloc(smatrix_t* s, size_t bytes) {
  void* p = NULL;
  const double t0 = now_ns();
  cudaError_t e = cudaMalloc(&p, bytes ? bytes : 256);
  if (e != cudaSuccess) smx_die("out of device memory (%zu bytes): %s", bytes, cudaGetErrorString(e));
  s->alloc_ns += now_ns() - t0; /* SMX_STAT_NS_ALLOC: cudaMalloc stalls for 2 - 150 ms on some hosts */
  s->n_allocs++;
  return p;
}

/* b, grown to at least `need` bytes.  A replaced block may still be read by work in flight on s->stream: it is
 * freed after that work; its contents are not kept. */
static void* dbuf_need(smatrix_t* s, smx_dbuf_t* b, size_t need) {
  if (need <= b->bytes) return b->p;
  if (b->p) {
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaFree(b->p));
  }
  b->bytes = need + need / 4 + 4096;
  b->p = dmalloc(s, b->bytes);
  return b->p;
}

/* host <-> device copies, counted (the end-to-end accounting of bench.py reads the counters) */
static inline void copy_h2d(smatrix_t* s, void* d, const void* h, size_t bytes, cudaStream_t st) {
  CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st));
  s->h2d_bytes += bytes;
}
static inline void copy_d2h(smatrix_t* s, void* h, const void* d, size_t bytes, cudaStream_t st) {
  CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, st));
  s->d2h_bytes += bytes;
}

static uint32_t log2_u64(uint64_t v) {
  uint32_t l = 0;
  while ((1ull << l) < v) l++;
  return l;
}

static inline smx_view_t view_for(smatrix_t* s, smx_row_t* dir, uint64_t cap) {
  smx_view_t v;
  const uint32_t lg = log2_u64(cap);
  v.dir = dir;
  v.dir_cap = cap;
  uint32_t slices_log = lg > 4 ? lg - 4 : 0;              /* slices of >= 16 entries ...        */
  if (slices_log > 8) slices_log = 8;                     /* ... at most SMX_DIR_SLICES of them */
  v.slice_shift = lg - slices_log;
  v.slice_limit = (uint32_t)((1ull << v.slice_shift) / 4); /* load limit 1/4 in every slice: every
                                                              extra directory probe is one more DRAM
                                                              touch per get (13.3 vs 11.0 Gops/s
                                                              measured at load 0.19 vs 0.39)       */
  if (v.slice_limit < 1) v.slice_limit = 1;
  v.ctl = s->d_ctl;
  return v;
}
static inline smx_view_t view_of(smatrix_t* s) { return view_for(s, s->dir, s->dir_cap); }

/* ---- phase accounting (host wall clock; see SMX_STAT_NS_*) ---- */
enum { PH_PARTITION = 0, PH_UPSERT, PH_GROW_PLAN, PH_SLAB, PH_MIGRATE, PH_DIR, PH_COUNT };
static inline double now_ns(void) {
  struct timespec t;
  clock_gettime(CLOCK_MONOTONIC, &t);
  return (double)t.tv_sec * 1e9 + (double)t.tv_nsec;
}

static void read_ctl(smatrix_t* s) {
  copy_d2h(s, s->h_ctl, s->d_ctl, sizeof(smx_ctl_t), s->stream);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  unsigned long long used = 0;
  for (uint32_t k = 0; k < SMX_DIR_SLICES; k++) used += s->h_ctl->slice_used[k];
  s->h_ctl->dir_used = used;
}

/* ------------------------------------------------------------------------------ slab */
static size_t next_segment_size(smatrix_t* s) { /* geometric x4: 64 MiB, 256 MiB, 1 GiB, 4, 16, 16, ... */
  size_t want = s->nsegs ? s->segs[s->nsegs - 1].size * 4 : SMX_SEG_MIN;
  if (want < SMX_SEG_MIN) want = SMX_SEG_MIN;
  if (want > SMX_SEG_MAX) want = SMX_SEG_MAX;
  return want;
}

static void push_segment(smatrix_t* s, char* base, size_t size) {
  if (s->nsegs == s->segs_cap) {
    s->segs_cap = s->segs_cap ? s->segs_cap * 2 : 16;
    s->segs = (smx_seg_t*)realloc(s->segs, sizeof(smx_seg_t) * (size_t)s->segs_cap);
    if (!s->segs) smx_die("out of host memory");
  }
  smx_seg_t* g = &s->segs[s->nsegs++];
  g->base = base;
  g->size = size;
  g->used = 0;
  g->owned = 1;
  s->seg_bytes += size;
}

/* a block carved from the slab that is no longer needed (a replaced directory) becomes a segment of
 * its own: later reservations are served from it before fresh slab is touched */
static void slab_give_back(smatrix_t* s, char* base, size_t size) {
  size &= ~(size_t)127;
  if (size < (1u << 16)) return;
  push_segment(s, base, size);
  s->segs[s->nsegs - 1].owned = 0;
  s->seg_bytes -= size; /* it was counted when its parent segment was pushed */
  /* keep the growing tail segment LAST (next_segment_size and the bump cursor look at it) */
  if (s->nsegs >= 2) {
    smx_seg_t t = s->segs[s->nsegs - 1];
    s->segs[s->nsegs - 1] = s->segs[s->nsegs - 2];
    s->segs[s->nsegs - 2] = t;
  }
}

/* A contiguous, 128-byte aligned device region of `bytes` (not zeroed).  Carved from the arena
 * reserved at open when there is one; otherwise (or once it is exhausted) from segments that are
 * cudaMalloc'ed on demand, x4 geometric.  On-demand cudaMalloc costs 2-10 ms per call on B200
 * hosts and far more when the driver has to scrub recently freed memory, which is why a
 * long-lived table should reserve its arena up front (SMATRIX_ARENA_GIB). */
static char* slab_reserve(smatrix_t* s, size_t bytes) {
  bytes = (bytes + 127) & ~(size_t)127;
  for (int i = 0; i + 1 < s->nsegs; i++) { /* given-back blocks and the tails of earlier segments first */
    smx_seg_t* f = &s->segs[i];
    if (!f->owned && f->size - f->used >= bytes) {
      char* p = f->base + f->used;
      f->used += bytes;
      s->slab_bytes += bytes;
      return p;
    }
  }
  smx_seg_t* g = s->nsegs ? &s->segs[s->nsegs - 1] : NULL;
  if (!g || g->size - g->used < bytes) {
    size_t size = next_segment_size(s);
    if (size < bytes) size = bytes;
    push_segment(s, (char*)dmalloc(s, size), size);
    g = &s->segs[s->nsegs - 1];
  }
  char* p = g->base + g->used;
  g->used += bytes;
  s->slab_bytes += bytes;
  return p;
}

/* ------------------------------------------------------------------------------ scratch */
/* Per-chunk scratch comes from the arena when there is one (sized once for the largest chunk, never
 * freed on its own), so that a table with a reserved arena makes no cudaMalloc call at all while
 * batches are applied; otherwise it is cudaMalloc'ed and regrown on demand. */
static void* scratch_alloc(smatrix_t* s, size_t bytes) {
  return s->arena_bytes ? (void*)slab_reserve(s, bytes) : dmalloc(s, bytes);
}
static void scratch_free(smatrix_t* s, void* p) {
  if (p && !s->arena_bytes) cudaFree(p);
}

static void ensure_lists(smatrix_t* s, uint32_t n) {
  if (n <= s->list_cap) return;
  uint32_t cap = s->list_cap ? s->list_cap : 1024;
  while (cap < n) cap *= 2;
  if (cap > s->chunk_max) cap = s->chunk_max > n ? s->chunk_max : n;
  if (s->arena_bytes && cap < s->chunk_max) cap = s->chunk_max; /* once, at full size */
  if (s->list_cap) {
    CK(cudaStreamSynchronize(s->stream));
    scratch_free(s, s->defer[0]); scratch_free(s, s->defer[1]); scratch_free(s, s->lists.late);
    scratch_free(s, s->lists.grow); scratch_free(s, s->lists.t0rows); scratch_free(s, s->lists.plan);
    scratch_free(s, s->lists.big); scratch_free(s, s->lists.mid);
  }
  s->defer[0] = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->defer[1] = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->lists.late = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->lists.grow = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->lists.t0rows = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->lists.plan = (smx_plan_t*)scratch_alloc(s, (size_t)cap * sizeof(smx_plan_t));
  s->lists.big = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->lists.mid = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->list_cap = cap;
}

static void ensure_stage(smatrix_t* s, uint32_t n) {
  if (n <= s->stage_cap) return;
  uint32_t cap = n < 4096 ? 4096 : n;
  if (s->arena_bytes && cap < s->stage_max) cap = s->stage_max; /* from the arena: once, at full size */
  if (s->stage_cap) {
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaStreamSynchronize(s->copy_stream));
    for (int b = 0; b < 2; b++)
      for (int a = 0; a < 3; a++) scratch_free(s, s->stage[b][a]);
  }
  for (int b = 0; b < 2; b++)
    for (int a = 0; a < 3; a++) s->stage[b][a] = (uint32_t*)scratch_alloc(s, (size_t)cap * 4);
  s->stage_cap = cap;
}

/* ------------------------------------------------------------------------------ growth */
static void timed_begin(smatrix_t* s) {
  if (s->timing) CK(cudaEventRecord(s->ev0, s->stream));
}
static void timed_end(smatrix_t* s) {
  if (s->timing) CK(cudaEventRecord(s->ev1, s->stream));
}
static void timed_collect(smatrix_t* s) { /* call after the stream has been synchronised */
  if (s->timing) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->kernel_ns += (double)ms * 1e6;
  }
}

/* make room on the free-list stacks for the buckets this round vacates (k_grow_plan counted them
 * per class); stacks grow geometrically and are only as large as the table needs them */
static void ensure_free_stacks(smatrix_t* s) {
  for (uint32_t c = SMX_MIN_SLAB_LOG; c < SMX_CLASSES; c++) {
    const uint32_t incoming = s->h_ctl->grow_from[c];
    if (!incoming) continue;
    const int32_t have = s->h_ctl->free_cnt[c] > 0 ? s->h_ctl->free_cnt[c] : 0;
    const uint64_t need = (uint64_t)have + incoming;
    if (need <= s->free_cap[c]) continue;
    uint64_t cap = s->free_cap[c] ? s->free_cap[c] : 1024;
    while (cap < need) cap *= 4;
    if (cap > 0x7FFFFFFFull) smx_die("free list of class %u too long", c);
    /* carved from the slab like the buckets themselves (cudaMalloc costs milliseconds on these hosts);
     * a replaced stack is simply abandoned: x4 growth keeps that below a third of the final one */
    unsigned long long* nb = (unsigned long long*)slab_reserve(s, (size_t)cap * 8);
    if (have) CK(cudaMemcpyAsync(nb, s->free_ptr[c], (size_t)have * 8, cudaMemcpyDeviceToDevice, s->stream));
    s->free_ptr[c] = nb; /* a field of the handle: stays valid while the copy below is in flight */
    copy_h2d(s, &s->d_ctl->free_stack[c], &s->free_ptr[c], sizeof nb, s->stream);
    s->free_cap[c] = (uint32_t)cap;
  }
}

static void grow_rows(smatrix_t* s, uint32_t n_grow) {
  smx_view_t v = view_of(s);
  double t0 = now_ns();
  smx_launch_grow_plan(s->stream, v, s->lists, n_grow);
  s->n_launches++;
  read_ctl(s);
  double t1 = now_ns();
  const size_t bytes = (size_t)s->h_ctl->plan_bytes;
  const uint32_t n_big = s->h_ctl->n_big, n_mid = s->h_ctl->n_mid;
  char* region = bytes ? slab_reserve(s, bytes) : NULL;
  s->bucket_bytes += bytes;
  if (s->recycle) {
    ensure_free_stacks(s);
    smx_launch_free_push(s->stream, v, s->lists, n_grow);
    s->n_launches++;
  }
  double t2 = now_ns();
  /* buckets built in shared memory are written out whole; only in-place (global CAS) fills need zeros */
  if (bytes && s->h_ctl->need_zero) CK(cudaMemsetAsync(region, 0, bytes, s->stream));
  const int tiles = s->migrate_tiles && n_big;
  smx_launch_migrate(s->stream, v, s->lists, n_grow, n_mid, n_big, region, tiles);
  if (tiles) { /* big rows: new buckets built tile by tile in shared memory (k_migrate_tiles) */
    unsigned long long* spill;
    uint32_t n_spill;
    for (;;) {
      spill = dbuf_need(s, &s->db.spill, (size_t)s->spill_cap * 16);
      CK(cudaMemsetAsync(&s->d_ctl->n_spill, 0, 4, s->stream));
      smx_launch_migrate_tiles(s->stream, v, s->lists, n_big, region, spill, s->spill_cap);
      copy_d2h(s, &s->h_small->n_spill, &s->d_ctl->n_spill, 4, s->stream);
      CK(cudaStreamSynchronize(s->stream));
      n_spill = s->h_small->n_spill;
      if (n_spill <= s->spill_cap) break;
      s->spill_cap = n_spill + n_spill / 2 + 1024; /* the list was too short: step 1 only reads the old buckets, so it can run again */
    }
    smx_launch_migrate_tiles_finish(s->stream, v, s->lists, n_big, region, spill, n_spill);
    s->n_spilled += n_spill;
  }
  if (s->timing) CK(cudaStreamSynchronize(s->stream)); /* attribute the device time to this phase */
  s->n_launches += (n_grow > n_mid + n_big ? 1 : 0) + (n_mid ? 1 : 0) + (n_big ? 3 : 0);
  s->n_row_grows += n_grow;
  s->n_recycled += s->h_ctl->n_recycled;
  s->phase_ns[PH_GROW_PLAN] += t1 - t0;
  s->phase_ns[PH_SLAB] += t2 - t1;
  s->phase_ns[PH_MIGRATE] += now_ns() - t2;
}

/* A chunk of mostly NEW rows would overflow a small directory and waste a whole round finding that
 * out (every op turned away, then one resize per doubling).  Estimate the chunk's distinct rows
 * with one streaming pass (linear counting) and size the directory for them up front. */
/* ln(r) for 0 < r <= 1 without libm (bindings link the static archive without -lm):
 * r = f * 2^-k with f in [0.5, 1), ln f = 2 atanh((f-1)/(f+1)) by its series (|y| <= 1/3) */
static double ln_unit(double r) {
  int k = 0;
  while (r < 0.5) { r *= 2.0; k++; }
  const double y = (r - 1.0) / (r + 1.0), y2 = y * y;
  double term = y, sum = 0.0;
  for (int i = 1; i < 40; i += 2) { sum += term / (double)i; term *= y2; }
  return 2.0 * sum - (double)k * 0.69314718055994530942;
}
#define SMX_SKETCH_BITS_LOG 25u
static int resize_dir(smatrix_t* s, uint64_t new_cap, int shrink);
static uint64_t pow2_at_least(uint64_t v);
static void presize_dir(smatrix_t* s, const smx_ops_t* ops) {
  const uint64_t n = ops->n, used = s->h_ctl->dir_used;
  if (n < s->part_min || !s->presize) return;      /* small batches: the grow loop is cheap        */
  if (used + n <= s->dir_cap / 4) return;          /* fits even if every op creates a row           */
  /* only for an EMPTY table: there every distinct row of the chunk is a new row.  Later chunks mix new
   * and existing rows (the sketch cannot tell them apart and would over-size the directory — measured:
   * 2^27 instead of 2^26 entries for config 2, +2 % per step); the grow loop handles those */
  if (used) return;
  const uint64_t m = 1ull << SMX_SKETCH_BITS_LOG;
  uint32_t* bitmap = dbuf_need(s, &s->db.tmp, (size_t)(m / 8));
  CK(cudaMemsetAsync(bitmap, 0, (size_t)(m / 8), s->stream));
  CK(cudaMemsetAsync(&s->d_ctl->scratch, 0, 8, s->stream));
  smx_launch_sketch(s->stream, ops->xs, ops->n, bitmap, SMX_SKETCH_BITS_LOG, s->d_ctl);
  s->n_launches += 2;
  read_ctl(s);
  const double zeros = (double)s->h_ctl->scratch;
  double est = zeros >= 1.0 ? -(double)m * ln_unit(zeros / (double)m) : (double)n;
  if (est > (double)n) est = (double)n;
  const uint64_t cap = pow2_at_least((uint64_t)(4.0 * ((double)used + 1.1 * est)) + 64);
  if (s->debug) fprintf(stderr, "[smatrix] presize: %llu ops, %.0f zero bits, ~%.0f distinct rows\n", (unsigned long long)n, zeros, est);
  if (cap > s->dir_cap) resize_dir(s, cap, 0);
}

static uint64_t pow2_at_least(uint64_t v) {
  uint64_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

/* Re-place every row into a directory of new_cap entries.  A shrink is abandoned (the current directory stays,
 * returns 0) when it would put a row SMX_DIR_CREATE_STEPS or more probe steps from its home: dir_find refuses to
 * create a row that far out, so the next new row on such a chain (rows whose mix_row share their low bits) would
 * grow the directory all the way back, and the shrink after the chunk would undo that again, batch after batch. */
static int resize_dir(smatrix_t* s, uint64_t new_cap, int shrink) {
  double t0 = now_ns();
  if (s->debug)
    fprintf(stderr, "[smatrix] directory %llu -> %llu entries (rows %llu, refused ops %u of which directory-full %u)\n",
            (unsigned long long)s->dir_cap, (unsigned long long)new_cap, (unsigned long long)s->h_ctl->dir_used,
            s->h_ctl->n_defer, s->h_ctl->n_dirfull);
  smx_view_t from = view_of(s);
  /* with an arena the directory lives in it too (cudaMalloc / cudaFree of multi-GiB blocks stall for
   * tens of ms on these hosts); a replaced directory's arena space is not reused */
  const int in_arena = s->arena_bytes != 0;
  smx_row_t* nd = in_arena ? (smx_row_t*)slab_reserve(s, (size_t)new_cap * sizeof(smx_row_t))
                           : (smx_row_t*)dmalloc(s, (size_t)new_cap * sizeof(smx_row_t));
  CK(cudaMemsetAsync(nd, 0, (size_t)new_cap * sizeof(smx_row_t), s->stream));
  CK(cudaMemsetAsync(s->d_ctl->slice_used, 0, sizeof(uint32_t) * SMX_DIR_SLICES, s->stream));
  CK(cudaMemsetAsync(&s->d_ctl->dir_probe_max, 0, 4, s->stream));
  smx_view_t to = view_for(s, nd, new_cap);
  smx_launch_dir_rehash(s->stream, from, to);
  s->n_launches++;
  if (shrink) copy_d2h(s, &s->h_small->probe_max, &s->d_ctl->dir_probe_max, 4, s->stream); /* read in the same wait */
  CK(cudaStreamSynchronize(s->stream));
  if (shrink && s->h_small->probe_max >= SMX_DIR_CREATE_STEPS) {
    if (s->debug)
      fprintf(stderr, "[smatrix] shrink to %llu entries refused: a row would sit %u probe steps from its home\n",
              (unsigned long long)new_cap, s->h_small->probe_max);
    if (in_arena) slab_give_back(s, (char*)nd, (size_t)new_cap * sizeof(smx_row_t));
    else CK(cudaFree(nd));
    /* the rehash counted the rows per slice of the new directory: put back the counts of the current one
     * (as of the last read_ctl, which followed the chunk's last update launch) */
    copy_h2d(s, s->d_ctl->slice_used, s->h_ctl->slice_used, sizeof(uint32_t) * SMX_DIR_SLICES, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->shrink_refused = new_cap;
    s->phase_ns[PH_DIR] += now_ns() - t0;
    return 0;
  }
  if (!s->dir_in_arena) CK(cudaFree(s->dir));
  else slab_give_back(s, (char*)s->dir, (size_t)s->dir_cap * sizeof(smx_row_t)); /* the old directory's arena space */
  s->dir = nd;
  s->dir_in_arena = in_arena;
  s->dir_cap = new_cap;
  s->n_dir_grows++;
  s->phase_ns[PH_DIR] += now_ns() - t0;
  return 1;
}

/* ------------------------------------------------------------------------------ write path */
static void zero_round_counters(smatrix_t* s) {
  CK(cudaMemsetAsync(&s->d_ctl->n_defer, 0,
                     offsetof(smx_ctl_t, scratch) - offsetof(smx_ctl_t, n_defer), s->stream));
  /* n_defer .. need_zero are contiguous and precede `scratch` */
}

/* Run one pass to completion: rounds of (launch, grow, re-run the ops that were turned away). */
static void run_pass(smatrix_t* s, smx_ops_t ops, int op, int pass, const uint32_t* list, uint32_t m) {
  int flip = 0;
  uint32_t prev_defer = 0xFFFFFFFFu;
  for (int round = 0; m > 0; round++) {
    if (round >= SMX_MAX_ROUNDS) smx_die("update pass does not converge (%u ops left)", m);
    double t0 = now_ns();
    const uint64_t used_before = s->h_ctl->dir_used;
    zero_round_counters(s);
    s->lists.defer_out = s->defer[flip];
    timed_begin(s);
    smx_launch_upsert(s->stream, view_of(s), ops, s->lists, op, pass, list, m, s->preagg);
    timed_end(s);
    s->n_launches++;
    s->n_rounds++;
    read_ctl(s);
    timed_collect(s);
    s->phase_ns[PH_UPSERT] += now_ns() - t0;
    const smx_ctl_t c = *s->h_ctl;
    if (c.n_grow) grow_rows(s, c.n_grow);
    if (c.n_defer == 0) break;
    if (c.n_dirfull) {
      /* n_dirfull counts refused OPS; how many new ROWS they stand for is estimated from this
       * round's accepted ops (rows created per accepted op), so a uniform first chunk jumps to its
       * final directory in one step while a duplicate-heavy one grows moderately;
       * maybe_shrink_dir() trims an over-shoot after the chunk */
      const uint64_t accepted = (uint64_t)m - c.n_defer;
      const uint64_t created = c.dir_used > used_before ? c.dir_used - used_before : 0;
      double ratio = accepted ? (double)created / (double)accepted : 1.0;
      if (ratio > 1.0) ratio = 1.0;
      if (ratio < 0.05) ratio = 0.05;
      uint64_t need = 4 * (c.dir_used + (uint64_t)(ratio * (double)c.n_dirfull));
      uint64_t cap = pow2_at_least(need);
      if (cap < s->dir_cap * 2) cap = s->dir_cap * 2;
      if (cap > s->dir_cap * 64) cap = s->dir_cap * 64;
      resize_dir(s, cap, 0);
    } else if (!c.n_grow && c.n_defer >= prev_defer) {
      smx_die("update pass made no progress (%u ops deferred)", c.n_defer);
    }
    prev_defer = c.n_defer;
    list = s->defer[flip];
    m = c.n_defer;
    flip ^= 1;
  }
}

/* After a chunk: a directory that was grown for a burst of duplicates goes back to a load
 * factor in (1/8, 1/4] so that it stays as L2-friendly as the data allows. */
static void maybe_shrink_dir(smatrix_t* s) {
  const uint64_t used = s->h_ctl->dir_used;
  uint64_t fit = pow2_at_least(4 * (used ? used : 1));
  const uint64_t floor_cap = 1ull << s->dir_log_min;
  if (fit < floor_cap) fit = floor_cap;
  /* rows are never removed, so a size at which a shrink was refused stays out of reach: not tried again */
  if (fit * 4 <= s->dir_cap && fit > s->shrink_refused) resize_dir(s, fit, 1);
}

/* directory slices of a batch: 2^parts_log of them, slice(x) = (mix_row(x) & (dir_cap - 1)) >> shift */
static void slice_geometry(const smatrix_t* s, uint32_t* parts_log, uint32_t* shift) {
  uint32_t dir_log = 0;
  while ((1ull << dir_log) < s->dir_cap) dir_log++;
  uint32_t pl = dir_log > s->slice_log ? dir_log - s->slice_log : 0; /* default: slices of 2^17 entries = 8 MiB */
  if (pl > s->parts_log_max) pl = s->parts_log_max;
  *parts_log = pl;
  *shift = dir_log - pl;
}
/* the four arrays a slice-ordered batch lives in (x, y, values / answers, index / position) */
static void ensure_parts(smatrix_t* s, uint32_t n) {
  if (n <= s->part_cap) return;
  if (s->part_cap) {
    CK(cudaStreamSynchronize(s->stream));
    for (int a = 0; a < 4; a++) scratch_free(s, s->part[a]);
  }
  s->part_cap = s->list_cap > n ? s->list_cap : n;
  for (int a = 0; a < 4; a++) s->part[a] = (uint32_t*)scratch_alloc(s, (size_t)s->part_cap * 4);
}

/* Reorder a chunk so that ops on rows of the same directory slice are adjacent: the slice of the
 * directory (a few MB) then stays in L2 while its ops are applied, and a row header costs one
 * DRAM read + one write-back per chunk instead of one per op.  Ops on column 0 go to parts of their
 * own behind all the others: [other ops by slice | column-0 ops by slice], so each pass runs over
 * a dense range.  The input-order index travels along (part[3]) only when something depends on it:
 * a set batch, a chunk that writes column 0, or a caller-supplied order.
 * Returns 1 if the chunk was partitioned; *n_main = number of ops that are not on column 0. */
static int partition_chunk(smatrix_t* s, smx_ops_t* ops, int api_op, uint32_t* n_main) {
  const uint32_t n = ops->n, mask = (uint32_t)(s->dir_cap - 1);
  uint32_t parts_log, shift;
  slice_geometry(s, &parts_log, &shift);
  uint32_t slices = 1u << parts_log, parts = 2u * slices;
  /* With the column-0 parts a chunk has at most 128 slices.  A chunk WITHOUT ops on column 0 (configs 2
   * and 5) does not need them: count over twice as many slices (+ their column-0 twins, 512 bins), and
   * use all 256 parts as slices if the twins stay empty — else fold neighbouring bins back. */
  const int fine = s->wide_slices && parts_log == 7 && parts_log + shift > s->slice_log + 7;
  ensure_parts(s, n);
  unsigned long long* d_counts = dbuf_need(s, &s->db.tmp64, 3 * SMX_MAX_PARTS_H * 8); /* up to 2 * SMX_MAX_PARTS_H bins */
  unsigned long long* d_cursors = d_counts + 2 * SMX_MAX_PARTS_H;
  unsigned long long h[2 * SMX_MAX_PARTS_H], cur[SMX_MAX_PARTS_H];
  double t0 = now_ns();
  const uint32_t bins = fine ? 2u * parts : parts;
  CK(cudaMemsetAsync(d_counts, 0, bins * 8, s->stream));
  smx_launch_partition_count(s->stream, ops->xs, ops->ys, n, bins, mask, fine ? shift - 1 : shift, bins / 2, d_counts);
  copy_d2h(s, h, d_counts, bins * 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  uint32_t split0 = slices;
  if (fine) {
    unsigned long long on_col0 = 0;
    for (uint32_t p = parts; p < bins; p++) on_col0 += h[p];
    if (on_col0 == 0) { /* 256 slices, no column-0 parts: the first half of the bins is the histogram */
      slices = parts;
      split0 = 0;
      shift -= 1;
      s->n_wide_chunks++;
    } else {
      for (uint32_t p = 0; p < parts; p++) h[p] = h[2 * p] + h[2 * p + 1]; /* in place: 2p >= p */
    }
  }
  unsigned long long at = 0;
  *n_main = n;
  for (uint32_t p = 0; p < parts; p++) {
    if (split0 && p == split0) *n_main = (uint32_t)at;
    cur[p] = at;
    at += h[p];
  }
  const int want_idx = api_op == 2 || *n_main != n || ops->idx != NULL;
  copy_h2d(s, d_cursors, cur, parts * 8, s->stream);
  smx_launch_partition_scatter(s->stream, ops->xs, ops->ys, ops->vs, n, parts, mask, shift, split0, d_cursors,
                               s->part[0], s->part[1], ops->vs ? s->part[2] : NULL,
                               want_idx ? s->part[3] : NULL, ops->idx, NULL, NULL, 0);
  s->n_launches += 2;
  if (s->timing) CK(cudaStreamSynchronize(s->stream));
  s->phase_ns[PH_PARTITION] += now_ns() - t0;
  ops->xs = s->part[0];
  ops->ys = s->part[1];
  if (ops->vs) ops->vs = s->part[2];
  ops->idx = want_idx ? s->part[3] : NULL;
  return 1;
}

static smx_ops_t ops_range(smx_ops_t o, uint32_t first, uint32_t count) {
  o.xs += first;
  o.ys += first;
  if (o.vs) o.vs += first;
  if (o.idx) o.idx += first;
  o.n = count;
  return o;
}

static void process_chunk_ordered(smatrix_t* s, int api_op, const uint32_t* d_xs, const uint32_t* d_ys,
                                  const uint32_t* d_vs, const uint32_t* d_ords, uint32_t n);
static void process_chunk(smatrix_t* s, int api_op, const uint32_t* d_xs, const uint32_t* d_ys,
                          const uint32_t* d_vs, uint32_t n) {
  process_chunk_ordered(s, api_op, d_xs, d_ys, d_vs, NULL, n);
}

/* d_ords == NULL: "input order" is the array order; else ords[i] is op i's place in that order */
static void process_chunk_ordered(smatrix_t* s, int api_op, const uint32_t* d_xs, const uint32_t* d_ys,
                                  const uint32_t* d_vs, const uint32_t* d_ords, uint32_t n) {
  if (n == 0) return;
  ensure_lists(s, n);
  smx_ops_t ops;
  ops.xs = d_xs; ops.ys = d_ys; ops.vs = d_vs; ops.idx = d_ords; ops.v_const = 1u; ops.n = n;

  presize_dir(s, &ops);
  uint32_t n_main = n;
  const int parted = (n >= s->part_min) ? partition_chunk(s, &ops, api_op, &n_main) : 0;
  /* partitioned: [0, n_main) = ops on columns != 0, [n_main, n) = ops on column 0 (dense ranges);
   * otherwise both passes scan the whole chunk and pick their ops by column */
  const smx_ops_t ops0 = parted ? ops_range(ops, n_main, n - n_main) : ops;
  const smx_ops_t opsm = parted ? ops_range(ops, 0, n_main) : ops;
  const int op = (api_op == 2) ? SMX_OP_SETZERO : api_op;
  CK(cudaMemsetAsync(&s->d_ctl->n_late, 0, 2 * sizeof(uint32_t), s->stream));
  s->h_ctl->n_late = s->h_ctl->n_t0 = 0;
  if (ops0.n) run_pass(s, ops0, op, SMX_PASS_COL0, NULL, ops0.n);
  if (opsm.n) run_pass(s, opsm, op, SMX_PASS_EARLY, NULL, opsm.n);
  if (s->h_ctl->n_t0) { /* column 0 of these rows turns non-zero now: sync their rowlen state (z = 0 so far) */
    smx_launch_sync_rowlen(s->stream, view_of(s), s->lists.t0rows, s->h_ctl->n_t0);
    s->n_launches++;
  }
  const uint32_t n_late = s->h_ctl->n_late;
  if (n_late) run_pass(s, opsm, op, SMX_PASS_LATE, s->lists.late, n_late);
  if (api_op == 2) { /* set: last writer in input order wins */
    if (n > s->addrs_cap) {
      if (s->addrs) { CK(cudaStreamSynchronize(s->stream)); scratch_free(s, s->addrs); }
      s->addrs_cap = s->list_cap > n ? s->list_cap : n;
      s->addrs = (uint64_t*)scratch_alloc(s, (size_t)s->addrs_cap * 8);
    }
    smx_launch_set_max(s->stream, view_of(s), ops, s->addrs);
    smx_launch_set_commit(s->stream, ops, s->addrs);
    s->n_launches += 3;
  }
  const uint32_t n_t0 = s->h_ctl->n_t0;
  if (n_t0) {
    smx_launch_finalize_t0(s->stream, view_of(s), s->lists.t0rows, n_t0);
    s->n_launches++;
  }
  maybe_shrink_dir(s);
}

static int is_device_ptr(const void* p) {
  struct cudaPointerAttributes a;
  if (!p) return 0;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    (void)cudaGetLastError(); /* plain host memory on old drivers */
    return 0;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

/* The arrays of one batched call must be all host or all device memory: returns 1 for device arrays and dies on a
 * mix.  Each of arrays[0..n) is checked (NULL counts as host memory), `opt` only when it is not NULL. */
static int batch_on_device(const void* opt, int n, const void* const* arrays) {
  const int dev = is_device_ptr(arrays[0]);
  int mixed = opt && is_device_ptr(opt) != dev;
  for (int i = 1; i < n; i++) mixed |= is_device_ptr(arrays[i]) != dev;
  if (mixed) smx_die("batch arrays must be all host or all device pointers");
  return dev;
}

/* Every entry point runs on the handle's GPU and puts the caller's current device back afterwards,
 * so a process that holds handles on several GPUs (or mixes the library with other CUDA code) never
 * finds its current device changed by a call. */
static void enter(smatrix_t* s) {
  if (!s) smx_die("NULL matrix handle");
  pthread_mutex_lock(&s->mu);
  int cur = s->device;
  if (cudaGetDevice(&cur) != cudaSuccess) { (void)cudaGetLastError(); cur = s->device; }
  s->prev_device = cur;
  if (cur != s->device) CK(cudaSetDevice(s->device));
}
static void leave(smatrix_t* s) {
  const int back = s->prev_device, mine = s->device;
  if (back != mine) (void)cudaSetDevice(back);
  pthread_mutex_unlock(&s->mu);
}

static void write_batch(smatrix_t* s, int api_op, const uint32_t* xs, const uint32_t* ys,
                        const uint32_t* vs, size_t n) {
  if (n == 0) return;
  enter(s);
  if (batch_on_device(vs, 2, (const void*[]){xs, ys})) {
    /* equal chunks: a batch a little over k * chunk_max must not end in a sliver that pays a whole
     * chunk's launches and round trips (the multi-GPU inbox holds 2^26 +- a few thousand ops) */
    const size_t pieces = (n + s->chunk_max - 1) / s->chunk_max;
    for (size_t k = 0; k < pieces; k++) {
      const size_t off = n * k / pieces, end = n * (k + 1) / pieces;
      process_chunk(s, api_op, xs + off, ys + off, vs ? vs + off : NULL, (uint32_t)(end - off));
    }
    CK(cudaStreamSynchronize(s->stream));
  } else {
    /* host arrays: double-buffered upload on the copy stream overlaps the previous chunk's update.
     * (Shrinking the last pieces to expose less of the final update was measured and does not pay on one
     * GPU: 10.71 vs 10.62 ms per 2^26 ops — the extra pieces cost more than the shorter tail saves.) */
    uint32_t step = s->chunk_max < s->stage_max ? s->chunk_max : s->stage_max;
    if (n < step) step = (uint32_t)n;
    ensure_stage(s, step);
    size_t off = 0;
    int b = 0;
#define SMX_PIECE_LEN(remaining) ((uint32_t)((remaining) > step ? step : (remaining)))
    uint32_t len = SMX_PIECE_LEN(n - off);
    const uint32_t* src[3] = {xs, ys, vs};
    for (int a = 0; a < 3; a++)
      if (src[a]) copy_h2d(s, s->stage[b][a], src[a] + off, (size_t)len * 4, s->copy_stream);
    CK(cudaEventRecord(s->stage_ready[b], s->copy_stream));
    while (off < n) {
      const size_t next = off + len;
      uint32_t next_len = 0;
      if (next < n) { /* start uploading the next chunk into the other buffer */
        next_len = SMX_PIECE_LEN(n - next);
        for (int a = 0; a < 3; a++)
          if (src[a]) copy_h2d(s, s->stage[b ^ 1][a], src[a] + next, (size_t)next_len * 4, s->copy_stream);
        CK(cudaEventRecord(s->stage_ready[b ^ 1], s->copy_stream));
      }
      CK(cudaStreamWaitEvent(s->stream, s->stage_ready[b], 0));
      process_chunk(s, api_op, s->stage[b][0], s->stage[b][1], vs ? s->stage[b][2] : NULL, len);
      CK(cudaStreamSynchronize(s->stream));
      off = next;
      len = next_len;
      b ^= 1;
    }
#undef SMX_PIECE_LEN
  }
  leave(s);
}

void smatrix_incr_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                        const uint32_t* vals, size_t n) {
  write_batch(self, 0, xs, ys, vals, n);
}
void smatrix_decr_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                        const uint32_t* vals, size_t n) {
  write_batch(self, 1, xs, ys, vals, n);
}
void smatrix_set_batch(smatrix_t* self, const uint32_t* xs, const uint32_t* ys,
                       const uint32_t* vals, size_t n) {
  write_batch(self, 2, xs, ys, vals, n);
}

/* ---- N1: the same batches, returning every op's value as if applied one by one in input order ---- */
/* the *_batch_out launches for the ops of a chunk just applied; their scratch is sized for at least 4096 ops */
static void batch_out(smatrix_t* s, smx_ops_t ops, int api_op, uint32_t* d_out) {
  const size_t cap = ops.n < 4096 ? 4096 : ops.n;
  smx_dbuf_t* sort = &s->db.bo_sort;
  dbuf_need(s, sort, smx_batch_out_sort_bytes((uint32_t)cap));
  smx_launch_batch_out(s->stream, view_of(s), ops, api_op == 2 ? SMX_OP_SETZERO : api_op, d_out,
                       dbuf_need(s, &s->db.bo_addr[0], cap * 8), dbuf_need(s, &s->db.bo_addr[1], cap * 8),
                       dbuf_need(s, &s->db.bo_idx[0], cap * 4), dbuf_need(s, &s->db.bo_idx[1], cap * 4),
                       dbuf_need(s, &s->db.bo_seg, cap * 8),
                       dbuf_need(s, &s->db.bo_tiles, ((size_t)smx_scan_scratch_items((uint32_t)cap) + 1) * 8),
                       sort->p, sort->bytes);
}

static void chunk_out(smatrix_t* s, int api_op, const uint32_t* d_xs, const uint32_t* d_ys, const uint32_t* d_vs,
                      uint32_t n, uint32_t* d_out) {
  process_chunk(s, api_op, d_xs, d_ys, d_vs, n);
  smx_ops_t ops;
  ops.xs = d_xs; ops.ys = d_ys; ops.vs = d_vs; ops.idx = NULL; ops.v_const = 1u; ops.n = n;
  batch_out(s, ops, api_op, d_out);
  s->n_launches += 7;
}

static void write_batch_out(smatrix_t* s, int api_op, const uint32_t* xs, const uint32_t* ys, const uint32_t* vs,
                            size_t n, uint32_t* out) {
  if (n == 0) return;
  if (!out) smx_die("batch_out: out must not be NULL");
  enter(s);
  if (batch_on_device(vs, 3, (const void*[]){xs, ys, out})) {
    for (size_t off = 0; off < n; off += s->chunk_max) {
      const uint32_t len = (uint32_t)((n - off < s->chunk_max) ? n - off : s->chunk_max);
      chunk_out(s, api_op, xs + off, ys + off, vs ? vs + off : NULL, len, out + off);
    }
    CK(cudaStreamSynchronize(s->stream));
  } else {
    uint32_t step = s->chunk_max < s->stage_max ? s->chunk_max : s->stage_max;
    if (n < step) step = (uint32_t)n;
    ensure_stage(s, step);
    uint32_t* d_out = dbuf_need(s, &s->db.bo_out, (size_t)step * 4);
    const uint32_t* src[3] = {xs, ys, vs};
    for (size_t off = 0; off < n; off += step) {
      const uint32_t len = (uint32_t)((n - off < step) ? n - off : step);
      for (int a = 0; a < 3; a++)
        if (src[a]) copy_h2d(s, s->stage[0][a], src[a] + off, (size_t)len * 4, s->stream);
      chunk_out(s, api_op, s->stage[0][0], s->stage[0][1], vs ? s->stage[0][2] : NULL, len, d_out);
      copy_d2h(s, out + off, d_out, (size_t)len * 4, s->stream);
      CK(cudaStreamSynchronize(s->stream));
    }
  }
  CK(cudaGetLastError());
  leave(s);
}

void smatrix_incr_batch_out(smatrix_t* self, const uint32_t* xs, const uint32_t* ys, const uint32_t* vals,
                            size_t n, uint32_t* out) {
  write_batch_out(self, 0, xs, ys, vals, n, out);
}
void smatrix_decr_batch_out(smatrix_t* self, const uint32_t* xs, const uint32_t* ys, const uint32_t* vals,
                            size_t n, uint32_t* out) {
  write_batch_out(self, 1, xs, ys, vals, n, out);
}
void smatrix_set_batch_out(smatrix_t* self, const uint32_t* xs, const uint32_t* ys, const uint32_t* vals,
                           size_t n, uint32_t* out) {
  write_batch_out(self, 2, xs, ys, vals, n, out);
}

void smatrix_b200_apply_ordered(smatrix_t* s, int op, const uint32_t* d_xs, const uint32_t* d_ys,
                                const uint32_t* d_vals, const uint32_t* d_ords, size_t n) {
  if (n == 0) return;
  if (op < 0 || op > 2) smx_die("apply_ordered: op must be 0 (incr), 1 (decr) or 2 (set)");
  enter(s);
  if (n > (1u << 30)) smx_die("apply_ordered: at most 2^30 ops per call (one chunk)");
  if (batch_on_device(d_vals, 3, (const void*[]){d_xs, d_ys, d_ords})) {
    process_chunk_ordered(s, op, d_xs, d_ys, d_vals, d_ords, (uint32_t)n);
    CK(cudaStreamSynchronize(s->stream));
  } else { /* host arrays: one staged copy (this entry point is meant for device-resident batches) */
    const uint32_t* src[4] = {d_xs, d_ys, d_vals, d_ords};
    uint32_t* tmp[4] = {NULL, NULL, NULL, NULL};
    for (int a = 0; a < 4; a++) {
      if (!src[a]) continue;
      tmp[a] = (uint32_t*)dmalloc(s, n * 4);
      copy_h2d(s, tmp[a], src[a], n * 4, s->stream);
    }
    process_chunk_ordered(s, op, tmp[0], tmp[1], tmp[2], tmp[3], (uint32_t)n);
    CK(cudaStreamSynchronize(s->stream));
    for (int a = 0; a < 4; a++)
      if (tmp[a]) CK(cudaFree(tmp[a]));
  }
  leave(s);
}

/* apply_ordered + the per-op return values (N1) for a permuted batch: out[i] = value of op i's cell right
 * after op i in the sequential order given by d_ords.  Device arrays, one chunk. */
void smatrix_b200_apply_ordered_out(smatrix_t* s, int op, const uint32_t* d_xs, const uint32_t* d_ys,
                                    const uint32_t* d_vals, const uint32_t* d_ords, size_t n, uint32_t* d_out) {
  if (n == 0) return;
  if (op < 0 || op > 2) smx_die("apply_ordered_out: op must be 0 (incr), 1 (decr) or 2 (set)");
  if (n > (1u << 30)) smx_die("apply_ordered_out: at most 2^30 ops per call (one chunk)");
  enter(s);
  process_chunk_ordered(s, op, d_xs, d_ys, d_vals, d_ords, (uint32_t)n);
  smx_ops_t ops;
  ops.xs = d_xs; ops.ys = d_ys; ops.vs = d_vals; ops.idx = d_ords; ops.v_const = 1u; ops.n = (uint32_t)n;
  batch_out(s, ops, op, d_out);
  s->n_launches += 9;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* ------------------------------------------------------------------------------ read path */
#define READ_STEP (1u << 26)

/* Point reads by directory slice.  A query costs two dependent random DRAM touches (directory entry,
 * bucket sector) and that, not bandwidth, bounds k_get.  When a batch asks for the same rows several
 * times — q queries over R rows touch only R (1 - e^(-q/R)) distinct entries — ordering the queries
 * by directory slice (the write path's partition, without the column-0 parts) keeps a slice's few MB
 * of entries in L2 while its queries run, so the directory touch reaches DRAM once per ROW instead
 * of once per QUERY.  Answers come out in slice order and k_gather puts them back through the
 * inverse permutation the scatter leaves; a tile's queries land in one contiguous run per slice, so
 * that gather reads whole sectors.  The cursors are prefixed on the device (k_parts_prefix): nothing
 * between the five launches waits for the host.  The look-ups run in k_get_tiled (blocks dispatched
 * in query order; the resident-grid k_get drifts across slices and loses the effect: 11.5 vs 25.4
 * Gops/s).  It already pays at 0.3 - 0.65 queries per row, where few entries are asked for twice —
 * presumably because the directory accesses of a moment are confined to one slice's 32 MB instead
 * of 4 GB (the input-order kernel moves ~0.6 fetches per query that no table access accounts for).
 * Config 2, 500 M queries over 13 M rows / 1.51 B cells: 12.8 -> 25.4 Gops/s. */
enum {
  SMX_GET_KEEP = 4,    /* bucket sectors with the ordinary L2 priority (default: evict-first, they are read once) */
  SMX_GET_WIDE = 8,    /* up to 256 slices instead of the write path's count (<= 2^SMATRIX_PARTS_LOG2 = 128) */
  SMX_GET_STRIDE = 16, /* look-ups by the resident-grid kernel of the input-order path (blocks drift across slices) */
  SMX_GET_STRIDE_GATHER = 32, /* answers put back by a resident-grid gather */
  SMX_GET_FLAGS = 4 | 8 | 16 | 32
};
static void get_geometry(const smatrix_t* s, uint32_t* parts_log, uint32_t* shift) {
  slice_geometry(s, parts_log, shift);
  if (s->get_flags & SMX_GET_WIDE) { /* no column-0 parts here, so all 256 parts can be slices */
    const uint32_t dir_log = *parts_log + *shift;
    uint32_t pl = dir_log > s->slice_log ? dir_log - s->slice_log : 0;
    if (pl > 8) pl = 8;
    *parts_log = pl;
    *shift = dir_log - pl;
  }
}
static int get_slices_pay(const smatrix_t* s, uint32_t n) {
  if (s->get_slices == 0 || n < 2) return 0;
  uint32_t parts_log, shift;
  get_geometry(s, &parts_log, &shift);
  if (parts_log == 0) return 0; /* the whole directory is one slice */
  if (s->get_slices >= 2) return 1;
  /* measured on the config-2 table (13 M rows, profiles/r2_summary.md): calls of 2^22 / 2^23 / 2^24 / 2^25 queries
   * = 0.3 / 0.65 / 1.3 / 2.6 per row: +5 / +20 / +70 / +75 % over the input order; 2^20 queries: -20 % (five launches
   * instead of one) */
  return n >= s->get_slice_min && 2 * (uint64_t)n >= s->h_ctl->dir_used;
}
static void get_sliced(smatrix_t* s, const uint32_t* d_xs, const uint32_t* d_ys, uint32_t n, uint32_t* d_out) {
  uint32_t parts_log, shift;
  get_geometry(s, &parts_log, &shift);
  const uint32_t slices = 1u << parts_log, mask = (uint32_t)(s->dir_cap - 1);
  ensure_parts(s, n);
  unsigned long long* d_counts = dbuf_need(s, &s->db.tmp64, 3 * SMX_MAX_PARTS_H * 8);
  unsigned long long* d_cursors = d_counts + 2 * SMX_MAX_PARTS_H;
  CK(cudaMemsetAsync(d_counts, 0, slices * 8, s->stream));
  smx_launch_partition_count(s->stream, d_xs, NULL, n, slices, mask, shift, 0, d_counts);
  smx_launch_parts_prefix(s->stream, d_counts, slices, d_cursors);
  smx_launch_partition_scatter(s->stream, d_xs, d_ys, NULL, n, slices, mask, shift, 0, d_cursors, s->part[0],
                               s->part[1], NULL, NULL, NULL, s->part[3], NULL, 0);
  if (s->get_flags & SMX_GET_STRIDE) smx_launch_get(s->stream, view_of(s), s->part[0], s->part[1], n, s->part[2]);
  else smx_launch_get_tiled(s->stream, view_of(s), s->part[0], s->part[1], n, s->part[2], !(s->get_flags & SMX_GET_KEEP));
  if (s->get_flags & SMX_GET_STRIDE_GATHER) smx_launch_gather_stride(s->stream, d_out, s->part[2], s->part[3], n);
  else smx_launch_gather(s->stream, d_out, s->part[2], s->part[3], n);
  s->n_launches += 5;
  s->n_sliced_gets += n;
}

void smatrix_get_batch(smatrix_t* s, const uint32_t* xs, const uint32_t* ys, size_t n,
                       uint32_t* out) {
  if (n == 0) return;
  enter(s);
  if (batch_on_device(NULL, 3, (const void*[]){xs, ys, out})) {
    for (size_t off = 0; off < n; off += READ_STEP) {
      const uint32_t len = (uint32_t)((n - off < READ_STEP) ? n - off : READ_STEP);
      timed_begin(s);
      if (get_slices_pay(s, len)) {
        get_sliced(s, xs + off, ys + off, len, out + off);
      } else {
        smx_launch_get(s->stream, view_of(s), xs + off, ys + off, len, out + off);
        s->n_launches++;
      }
      timed_end(s);
      CK(cudaStreamSynchronize(s->stream));
      timed_collect(s);
    }
  } else {
    /* four pieces in flight: the two staging buffers are used as halves, piece k owns slot k & 3 and
     * runs entirely on that slot's stream (upload, look up, download in stream order).  The upload
     * of a piece then overlaps the look-ups and downloads of the three before it (PCIe is full
     * duplex), so the call is bound by the upload alone; small pieces keep the un-overlapped first
     * upload and last download short. */
    uint32_t step = s->stage_max / 2 < 1024 ? 1024 : s->stage_max / 2;
    if (step > (1u << 22)) step = 1u << 22;
    if (n < step) step = (uint32_t)n;
    ensure_stage(s, 2 * step);
    cudaStream_t sts[4] = {s->stream, s->copy_stream, s->read_stream[0], s->read_stream[1]};
    uint32_t k = 0, len = 0;
    for (size_t off = 0; off < n; off += len, k++) {
      const size_t rem = n - off;
      len = (uint32_t)(rem > step ? step : rem);
      const uint32_t q = k & 3u;
      cudaStream_t st = sts[q];
      uint32_t* const* buf = s->stage[q >> 1];
      const size_t half = (size_t)(q & 1u) * step;
      copy_h2d(s, buf[0] + half, xs + off, (size_t)len * 4, st);
      copy_h2d(s, buf[1] + half, ys + off, (size_t)len * 4, st);
      smx_launch_get(st, view_of(s), buf[0] + half, buf[1] + half, len, buf[2] + half);
      s->n_launches++;
      copy_d2h(s, out + off, buf[2] + half, (size_t)len * 4, st);
    }
    CK(cudaStreamSynchronize(s->read_stream[0]));
    CK(cudaStreamSynchronize(s->read_stream[1]));
    CK(cudaStreamSynchronize(s->stream));
    CK(cudaStreamSynchronize(s->copy_stream));
  }
  CK(cudaGetLastError());
  leave(s);
}

void smatrix_rowlen_batch(smatrix_t* s, const uint32_t* xs, size_t n, uint32_t* out) {
  if (n == 0) return;
  enter(s);
  const int dev = batch_on_device(NULL, 2, (const void*[]){xs, out});
  for (size_t off = 0; off < n; off += READ_STEP) {
    const uint32_t len = (uint32_t)((n - off < READ_STEP) ? n - off : READ_STEP);
    if (dev) {
      smx_launch_rowlen(s->stream, view_of(s), xs + off, len, out + off);
    } else {
      uint32_t* tmp = dbuf_need(s, &s->db.tmp, (size_t)len * 8);
      copy_h2d(s, tmp, xs + off, (size_t)len * 4, s->stream);
      smx_launch_rowlen(s->stream, view_of(s), tmp, len, tmp + len);
      copy_d2h(s, out + off, tmp + len, (size_t)len * 4, s->stream);
    }
    s->n_launches++;
    CK(cudaStreamSynchronize(s->stream));
  }
  CK(cudaGetLastError());
  leave(s);
}

/* scratch of the getrow plan for n rows: per-row directory index | caplog << 32 (u64, k_row_counts), row counts,
 * the list of big rows and the per-row output cursors (u32), and the big-row counter; cursors and counter zeroed */
typedef struct { uint64_t* info; uint32_t *counts, *big, *cursors, *n_big; } smx_rowplan_t;
static smx_rowplan_t rowplan(smatrix_t* s, uint32_t n) {
  smx_rowplan_t p;
  p.info = dbuf_need(s, &s->db.plan, (size_t)n * 20 + 64);
  p.counts = (uint32_t*)(p.info + n);
  p.big = p.counts + n;
  p.cursors = p.big + n;
  p.n_big = p.cursors + n;
  CK(cudaMemsetAsync(p.cursors, 0, (size_t)n * 4 + 8, s->stream));
  return p;
}

typedef struct {
  uint64_t total;      /* pairs of all the rows */
  const uint32_t* ids; /* the row ids, on the device */
  uint64_t* offsets;   /* [n + 1], in db.tmp64 */
  uint32_t* pairs;     /* where the pairs were filled; NULL if they were not */
} smx_rows_t;

/* The start of every read that returns whole rows: rows ids[0..n) (host ids go up through db.tmp first) are
 * counted and scanned, and when 0 < total <= room their pairs are filled into d_pairs, or into db.rows when d_pairs
 * is NULL (the fill is timed for smatrix_getrow_batch's kernel time). */
static smx_rows_t gather_rows(smatrix_t* s, const uint32_t* ids, int ids_on_device, uint32_t n, uint64_t room,
                              uint32_t* d_pairs) {
  smx_rows_t r;
  r.ids = ids;
  if (!ids_on_device) {
    uint32_t* d_ids = dbuf_need(s, &s->db.tmp, (size_t)n * 4);
    copy_h2d(s, d_ids, ids, (size_t)n * 4, s->stream);
    r.ids = d_ids;
  }
  r.offsets = dbuf_need(s, &s->db.tmp64, ((size_t)n + 1 + smx_scan_scratch_items(n)) * 8);
  const smx_rowplan_t p = rowplan(s, n);
  smx_launch_row_counts(s->stream, view_of(s), r.ids, n, p.counts, p.info, p.big, p.n_big);
  smx_launch_scan(s->stream, p.counts, n, 0, r.offsets, r.offsets + (size_t)n + 1);
  s->n_launches += 4;
  copy_d2h(s, &s->h_small->row_total, r.offsets + n, 8, s->stream);
  copy_d2h(s, &s->h_small->n_big_rows, p.n_big, 4, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  r.total = s->h_small->row_total;
  r.pairs = NULL;
  if (r.total && r.total <= room) {
    r.pairs = d_pairs ? d_pairs : dbuf_need(s, &s->db.rows, (size_t)r.total * 8);
    timed_begin(s);
    smx_launch_getrow_fill(s->stream, view_of(s), p.info, n, r.offsets, 0, r.pairs, p.big, s->h_small->n_big_rows,
                           p.cursors);
    timed_end(s);
    s->n_launches++;
  }
  return r;
}

/* a call for no rows still writes offsets[0] = 0 */
static uint64_t no_rows(smatrix_t* s, uint64_t* offsets) {
  if (offsets) {
    const uint64_t zero = 0;
    enter(s);
    CK(cudaMemcpy(offsets, &zero, 8, cudaMemcpyDefault));
    leave(s);
  }
  return 0;
}

static void sort_run(smatrix_t* s, uint32_t n, const uint64_t* d_off, uint32_t* d_pairs);

/* smatrix_getrow_batch, and with sorted != 0 smatrix_getrow_sorted_batch: the filled rows are sorted by column on the
 * device before they go anywhere */
static uint64_t getrow_rows(smatrix_t* s, const char* what, int sorted, const uint32_t* xs, size_t n,
                            uint64_t* offsets, uint32_t* pairs, uint64_t pairs_cap) {
  if (n == 0) return no_rows(s, offsets);
  if (n >= 0xFFFFFFFFull) smx_die("%s: too many rows in one call", what);
  enter(s);
  const uint32_t nn = (uint32_t)n;
  const int pairs_dev = is_device_ptr(pairs);
  const smx_rows_t r = gather_rows(s, xs, is_device_ptr(xs), nn, pairs ? pairs_cap : 0, pairs_dev ? pairs : NULL);
  if (sorted && r.pairs) sort_run(s, nn, r.offsets, r.pairs);
  if (offsets) {
    CK(cudaMemcpyAsync(offsets, r.offsets, ((size_t)nn + 1) * 8, cudaMemcpyDefault, s->stream));
    if (!is_device_ptr(offsets)) s->d2h_bytes += ((size_t)nn + 1) * 8;
  }
  if (r.pairs && !pairs_dev) copy_d2h(s, pairs, r.pairs, (size_t)r.total * 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  if (r.pairs) timed_collect(s);
  CK(cudaGetLastError());
  leave(s);
  return r.total;
}

uint64_t smatrix_getrow_batch(smatrix_t* s, const uint32_t* xs, size_t n, uint64_t* offsets,
                              uint32_t* pairs, uint64_t pairs_cap) {
  return getrow_rows(s, "getrow_batch", 0, xs, n, offsets, pairs, pairs_cap);
}
uint64_t smatrix_getrow_sorted_batch(smatrix_t* s, const uint32_t* xs, size_t n, uint64_t* offsets,
                                     uint32_t* pairs, uint64_t pairs_cap) {
  return getrow_rows(s, "getrow_sorted_batch", 1, xs, n, offsets, pairs, pairs_cap);
}

/* SURVEY.md 8f N4: neighbours + cosine scores for a batch of items (examples/cf_recommender.c:50-86) */
uint64_t smatrix_cf_neighbors_batch(smatrix_t* s, const uint32_t* items, size_t n, uint64_t* offsets,
                                    uint32_t* ids, double* scores, uint64_t cap) {
  if (n == 0) return no_rows(s, offsets);
  if (n >= 0xFFFFFFFFull) smx_die("cf_neighbors_batch: too many items in one call");
  enter(s);
  const uint32_t nn = (uint32_t)n;
  const smx_rows_t r = gather_rows(s, items, is_device_ptr(items), nn, (ids && scores) ? cap : 0, NULL);
  if (offsets) CK(cudaMemcpyAsync(offsets, r.offsets, ((size_t)nn + 1) * 8, cudaMemcpyDefault, s->stream));
  if (r.pairs) {
    const int out_dev = batch_on_device(NULL, 2, (const void*[]){ids, scores});
    uint32_t* d_ids = ids;
    double* d_scores = scores;
    if (!out_dev) {
      char* o = dbuf_need(s, &s->db.host_out, (size_t)r.total * 12 + 64);
      d_scores = (double*)o;
      d_ids = (uint32_t*)(o + (size_t)r.total * 8);
    }
    smx_launch_cf_scores(s->stream, view_of(s), r.ids, nn, r.offsets, r.pairs, d_ids, d_scores);
    s->n_launches++;
    if (!out_dev) {
      copy_d2h(s, ids, d_ids, (size_t)r.total * 4, s->stream);
      copy_d2h(s, scores, d_scores, (size_t)r.total * 8, s->stream);
    }
  }
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
  return r.total;
}

/* ------------------------------------------------------------------------------ top-k */
/* the selection of smatrix_b200_topk_segments on device arrays, enqueued on s->stream (synchronises to read
 * the number of big segments and, per digit pass, how many are still selecting) */
static void topk_run(smatrix_t* s, uint32_t n, const uint64_t* d_off, const uint32_t* d_ids, const double* d_scores,
                     uint32_t k, uint32_t* d_counts, uint32_t* d_oids, double* d_oscores) {
  if (!n) return;
  uint32_t* ctl = dbuf_need(s, &s->db.tk_ctl, (size_t)n * 4 + 64);
  uint32_t* big_list = ctl + 16;
  CK(cudaMemsetAsync(ctl, 0, 64, s->stream));
  smx_launch_topk_classify(s->stream, n, d_off, big_list, ctl);
  copy_d2h(s, &s->h_small->topk, ctl, 16, s->stream);
  smx_launch_topk_small(s->stream, n, d_off, d_ids, d_scores, k, d_counts, d_oids, d_oscores);
  s->n_launches += 3;
  CK(cudaStreamSynchronize(s->stream));
  const uint32_t n_big = s->h_small->topk.n_big;
  if (!n_big) return;
  const uint64_t big_pairs = s->h_small->topk.big_pairs;
  void* big = dbuf_need(s, &s->db.tk_big, smx_topk_big_bytes(n_big));
  uint32_t* cids = dbuf_need(s, &s->db.tk_cids, (size_t)big_pairs * 4);
  double* cscores = dbuf_need(s, &s->db.tk_cscores, (size_t)big_pairs * 8);
  CK(cudaMemsetAsync(big, 0, smx_topk_big_bytes(n_big), s->stream));
  smx_launch_topk_init(s->stream, big_list, n_big, d_off, big, ctl);
  s->n_launches++;
  for (uint32_t pass = 1;; pass++) { /* every pass fixes one more digit of the k-th key */
    if (pass > smx_topk_max_passes()) smx_die("topk: the select did not end after %u digit passes", pass - 1);
    CK(cudaMemsetAsync(ctl + 1, 0, 4, s->stream));
    smx_launch_topk_pass(s->stream, big, n_big, k, d_ids, d_scores, cids, cscores, ctl);
    copy_d2h(s, &s->h_small->topk.active, ctl + 1, 4, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->n_launches += 3;
    s->n_topk_passes++;
    if (!s->h_small->topk.active) break;
  }
  smx_launch_topk_finish(s->stream, big, n_big, cids, cscores, k, d_counts, d_oids, d_oscores);
  s->n_launches++;
  s->n_topk_big += n_big;
}

void smatrix_b200_topk_segments(smatrix_t* s, size_t n, const uint64_t* d_offsets, const uint32_t* d_ids,
                                const double* d_scores, uint32_t k, uint32_t* d_counts, uint32_t* d_out_ids,
                                double* d_out_scores) {
  if (k < 1 || k > SMX_TOPK_MAX_K) smx_die("topk_segments: k = %u is outside 1..%u", k, SMX_TOPK_MAX_K);
  if (n >= 0xFFFFFFFFull) smx_die("topk_segments: too many segments in one call");
  if (!n) return;
  enter(s);
  topk_run(s, (uint32_t)n, d_offsets, d_ids, d_scores, k, d_counts, d_out_ids, d_out_scores);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* the top k neighbours of every item, ranked on the device: scores as smatrix_cf_neighbors_batch computes them,
 * for pieces of items whose pairs fit SMATRIX_TOPK_PAIRS, each piece selected by topk_run */
void smatrix_cf_topk_batch(smatrix_t* s, const uint32_t* items, size_t n, uint32_t k, uint32_t* counts, uint32_t* ids,
                           double* scores) {
  if (k < 1 || k > SMX_TOPK_MAX_K) smx_die("cf_topk_batch: k = %u is outside 1..%u", k, SMX_TOPK_MAX_K);
  if (n >= 0xFFFFFFFFull) smx_die("cf_topk_batch: too many items in one call");
  if (!n) return;
  enter(s);
  const int out_dev = batch_on_device(NULL, 3, (const void*[]){counts, ids, scores});
  const uint32_t nn = (uint32_t)n;
  uint32_t* tmp = dbuf_need(s, &s->db.tmp, (size_t)nn * 8);
  uint64_t* tmp64 = dbuf_need(s, &s->db.tmp64, ((size_t)nn + 1 + smx_scan_scratch_items(nn)) * 8);
  const uint32_t* d_items = items;
  if (!is_device_ptr(items)) {
    copy_h2d(s, tmp, items, (size_t)nn * 4, s->stream);
    d_items = tmp;
  }
  uint32_t* d_cnt = tmp + nn;
  /* the row lengths of the whole call decide where the pieces end */
  uint64_t* d_all = dbuf_need(s, &s->db.tk_off, ((size_t)nn + 1) * 8);
  smx_launch_row_counts(s->stream, view_of(s), d_items, nn, d_cnt, NULL, NULL, NULL);
  smx_launch_scan(s->stream, d_cnt, nn, 0, d_all, tmp64 + (size_t)nn + 1);
  s->n_launches += 4;
  for (uint32_t lo = 0, hi; lo < nn; lo = hi) {
    smx_launch_topk_cut(s->stream, d_all, nn, lo, s->topk_pairs, s->d_small + DS_OUT);
    copy_d2h(s, &s->h_small->topk_cut, s->d_small + DS_OUT, 4, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    hi = s->h_small->topk_cut;
    const uint32_t np = hi - lo;
    const smx_rows_t r = gather_rows(s, d_items + lo, 1, np, UINT64_MAX, NULL);
    uint32_t* p_ids = dbuf_need(s, &s->db.tk_ids, (size_t)r.total * 4);
    double* p_scores = dbuf_need(s, &s->db.tk_scores, (size_t)r.total * 8);
    if (r.total) {
      smx_launch_cf_scores(s->stream, view_of(s), r.ids, np, r.offsets, r.pairs, p_ids, p_scores);
      s->n_launches++;
    }
    uint32_t* oc = counts + lo;
    uint32_t* oi = ids + (size_t)lo * k;
    double* os = scores + (size_t)lo * k;
    if (!out_dev) {
      char* o = dbuf_need(s, &s->db.host_out, (size_t)np * (12ull * k + 4));
      os = (double*)o;
      oi = (uint32_t*)(o + (size_t)np * k * 8);
      oc = oi + (size_t)np * k;
    }
    topk_run(s, np, r.offsets, p_ids, p_scores, k, oc, oi, os);
    if (!out_dev) {
      copy_d2h(s, counts + lo, oc, (size_t)np * 4, s->stream);
      copy_d2h(s, ids + (size_t)lo * k, oi, (size_t)np * k * 4, s->stream);
      copy_d2h(s, scores + (size_t)lo * k, os, (size_t)np * k * 8, s->stream);
    }
  }
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* ------------------------------------------------------------------------------ basket recommendations */
#define REC_ITEM_BUDGET (1u << 30) /* positions per piece (the radix sorts count items in an int) */

/* Aggregation and ranking of one piece of baskets, enqueued on s->stream (synchronises to read the number of big
 * baskets and their pairs, and inside topk_run).  d_boff[0..nb] are absolute positions, base = d_boff[0], n_pos
 * positions; d_items is indexed by absolute position; d_off[0..n_pos] is the per-position CSR of d_ids / d_scores
 * (`pairs` pairs).  db.rc_ctl must already hold 64 + 8 * nb bytes. */
static void rec_run(smatrix_t* s, uint32_t nb, const uint64_t* d_boff, uint64_t base, uint64_t n_pos,
                    const uint32_t* d_items, const uint64_t* d_off, uint64_t pairs, const uint32_t* d_ids,
                    const double* d_scores, uint32_t k, uint32_t* d_counts, uint32_t* d_oids, double* d_oscores) {
  if (n_pos >= (1ull << 31)) smx_die("cf_recommend_batch: a piece of %llu items is more than 2^31 - 1",
                                     (unsigned long long)n_pos);
  uint32_t* ctl = s->db.rc_ctl.p;
  uint32_t* big_list = ctl + 16;
  uint32_t* cnt = big_list + nb;
  uint64_t* keys = dbuf_need(s, &s->db.rc_items, (size_t)n_pos * 16 + 16);
  uint64_t* sitems = keys + n_pos;
  uint32_t* t_ids = dbuf_need(s, &s->db.rc_tids, (size_t)pairs * 4);
  double* t_scores = dbuf_need(s, &s->db.rc_tscores, (size_t)pairs * 8);
  uint64_t* red_off = dbuf_need(s, &s->db.rc_red, ((size_t)nb + 1 + smx_scan_scratch_items(nb)) * 8);
  uint32_t* r_ids = dbuf_need(s, &s->db.rc_rids, (size_t)pairs * 4);
  double* r_scores = dbuf_need(s, &s->db.rc_rscores, (size_t)pairs * 8);
  size_t sort_bytes = smx_rec_sort_bytes((uint32_t)n_pos);
  void* sort_tmp = dbuf_need(s, &s->db.rc_sort, sort_bytes);
  CK(cudaMemsetAsync(ctl, 0, 64, s->stream));
  smx_launch_rec_items(s->stream, nb, d_boff, base, d_items, (uint32_t)n_pos, keys, sitems, sort_tmp, sort_bytes);
  smx_launch_rec_small(s->stream, nb, d_boff, base, d_off, d_ids, d_scores, sitems, big_list, ctl, t_ids, t_scores,
                       cnt);
  copy_d2h(s, &s->h_small->rec, ctl, 16, s->stream);
  s->n_launches += 5;
  CK(cudaStreamSynchronize(s->stream));
  const uint32_t n_big = s->h_small->rec.n_big;
  const uint64_t big_pairs = s->h_small->rec.big_pairs;
  uint64_t *big_off = NULL, *bkeys = NULL, *fpos = NULL;
  uint32_t* bvals = NULL;
  if (n_big) {
    if (big_pairs >= (1ull << 31))
      smx_die("cf_recommend_batch: the big baskets of a piece hold %llu pairs, more than 2^31 - 1",
              (unsigned long long)big_pairs);
    const uint32_t P = (uint32_t)big_pairs;
    const size_t scan_items = smx_scan_scratch_items(P > n_big ? P : n_big);
    uint32_t* lens = dbuf_need(s, &s->db.rc_big, (size_t)n_big * 4 + ((size_t)n_big + 1 + scan_items) * 8 + 16);
    big_off = (uint64_t*)(((uintptr_t)(lens + n_big) + 7) & ~(uintptr_t)7);
    uint64_t* scan_tmp = big_off + n_big + 1;
    uint64_t* keys_a = dbuf_need(s, &s->db.rc_keys, (size_t)P * 16);
    bkeys = keys_a + P;
    uint32_t* vals_a = dbuf_need(s, &s->db.rc_vals, (size_t)P * 8);
    bvals = vals_a + P;
    uint32_t* flags = dbuf_need(s, &s->db.rc_flags, (size_t)P * 4 + ((size_t)P + 1) * 8 + 16);
    fpos = (uint64_t*)(((uintptr_t)(flags + P) + 7) & ~(uintptr_t)7);
    sort_bytes = smx_rec_sort_bytes(P);
    sort_tmp = dbuf_need(s, &s->db.rc_sort, sort_bytes);
    smx_launch_rec_big(s->stream, big_list, n_big, P, d_boff, base, d_off, d_ids, sitems, lens, big_off, keys_a, bkeys,
                       vals_a, bvals, flags, fpos, scan_tmp, sort_tmp, sort_bytes, cnt);
    s->n_launches += 12;
    s->n_rec_big += n_big;
  }
  smx_launch_scan(s->stream, cnt, nb, 0, red_off, red_off + (size_t)nb + 1);
  smx_launch_rec_emit(s->stream, nb, d_boff, base, d_off, d_scores, cnt, red_off, t_ids, t_scores, big_list, n_big,
                      (uint32_t)big_pairs, big_off, bkeys, bvals, fpos, r_ids, r_scores);
  s->n_launches += n_big ? 5 : 4;
  topk_run(s, nb, red_off, r_ids, r_scores, k, d_counts, d_oids, d_oscores);
}

void smatrix_b200_basket_topk(smatrix_t* s, size_t n, const uint64_t* d_basket_off, const uint32_t* d_items,
                              const uint64_t* d_offsets, const uint32_t* d_ids, const double* d_scores, uint32_t k,
                              uint32_t* d_counts, uint32_t* d_out_ids, double* d_out_scores) {
  if (k < 1 || k > SMX_TOPK_MAX_K) smx_die("basket_topk: k = %u is outside 1..%u", k, SMX_TOPK_MAX_K);
  if (n >= 0xFFFFFFFFull) smx_die("basket_topk: too many baskets in one call");
  if (!n) return;
  enter(s);
  const uint32_t nb = (uint32_t)n;
  dbuf_need(s, &s->db.rc_ctl, 64 + (size_t)nb * 8);
  copy_d2h(s, &s->h_small->rec_check.n_pos, d_basket_off + nb, 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  const uint64_t n_pos = s->h_small->rec_check.n_pos;
  copy_d2h(s, &s->h_small->row_total, d_offsets + n_pos, 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  rec_run(s, nb, d_basket_off, 0, n_pos, d_items, d_offsets, s->h_small->row_total, d_ids, d_scores, k, d_counts,
          d_out_ids, d_out_scores);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* per basket, the k best items by the summed scores of the basket's neighbour lists: the lists as
 * smatrix_cf_neighbors_batch computes them, for pieces of baskets whose rows fit SMATRIX_TOPK_PAIRS, each piece
 * aggregated and ranked by rec_run */
void smatrix_cf_recommend_batch(smatrix_t* s, const uint64_t* basket_off, const uint32_t* items, size_t n,
                                uint32_t k, uint32_t* counts, uint32_t* ids, double* scores) {
  if (k < 1 || k > SMX_TOPK_MAX_K) smx_die("cf_recommend_batch: k = %u is outside 1..%u", k, SMX_TOPK_MAX_K);
  if (n >= 0xFFFFFFFFull) smx_die("cf_recommend_batch: too many baskets in one call");
  if (!n) return;
  if (!basket_off) smx_die("cf_recommend_batch: basket_off is NULL");
  enter(s);
  const int out_dev = is_device_ptr(counts);
  if (is_device_ptr(ids) != out_dev || is_device_ptr(scores) != out_dev)
    smx_die("cf_recommend_batch: counts, ids and scores must be all host or all device arrays");
  const uint32_t nb = (uint32_t)n;
  const int in_dev = is_device_ptr(basket_off);
  uint32_t* ctl = dbuf_need(s, &s->db.rc_ctl, 64 + (size_t)nb * 8);
  uint64_t n_pos;
  if (in_dev) {
    CK(cudaMemsetAsync(ctl, 0, 16, s->stream));
    smx_launch_rec_check(s->stream, basket_off, nb, ctl);
    copy_d2h(s, &s->h_small->rec_check, ctl, 16, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->n_launches++;
    n_pos = s->h_small->rec_check.n_pos;
    if (s->h_small->rec_check.bad) n_pos = ~0ull;
  } else {
    n_pos = basket_off[0] == 0 ? basket_off[n] : ~0ull;
    for (size_t i = 0; i < n && n_pos != ~0ull; i++)
      if (basket_off[i + 1] < basket_off[i]) n_pos = ~0ull;
  }
  if (n_pos > 0xFFFFFFFEull)
    smx_die("cf_recommend_batch: malformed basket offsets (they must start at 0, never decrease and end at most at "
            "2^32 - 2)");
  if (n_pos && is_device_ptr(items) != in_dev)
    smx_die("cf_recommend_batch: basket_off and items must both be host or both be device arrays");
  const uint32_t npos = (uint32_t)n_pos;
  const uint64_t* d_boff = basket_off;
  const uint32_t* d_items = items;
  if (!in_dev) {
    char* in = dbuf_need(s, &s->db.rc_in, ((size_t)nb + 1) * 8 + (size_t)npos * 4);
    copy_h2d(s, in, basket_off, ((size_t)nb + 1) * 8, s->stream);
    d_boff = (const uint64_t*)in;
    if (npos) copy_h2d(s, in + ((size_t)nb + 1) * 8, items, (size_t)npos * 4, s->stream);
    d_items = (const uint32_t*)(in + ((size_t)nb + 1) * 8);
  }
  /* the row lengths of the whole call decide where the pieces end */
  const size_t scan_items = smx_scan_scratch_items(npos);
  uint64_t* d_pos = dbuf_need(s, &s->db.rc_pos, ((size_t)npos + 1 + scan_items) * 8 + (size_t)npos * 4);
  uint32_t* d_cnt = (uint32_t*)(d_pos + npos + 1 + scan_items);
  smx_launch_row_counts(s->stream, view_of(s), d_items, npos, d_cnt, NULL, NULL, NULL);
  smx_launch_scan(s->stream, d_cnt, npos, 0, d_pos, d_pos + (size_t)npos + 1);
  s->n_launches += 4;
  for (uint32_t lo = 0, hi; lo < nb; lo = hi) {
    smx_launch_rec_cut(s->stream, d_pos, d_boff, nb, lo, s->topk_pairs, REC_ITEM_BUDGET, ctl + 4);
    copy_d2h(s, s->h_small->rec_cut, ctl + 4, 12, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->n_launches++;
    hi = s->h_small->rec_cut[0];
    const uint32_t p_lo = s->h_small->rec_cut[1], p_n = s->h_small->rec_cut[2] - p_lo, np = hi - lo;
    const smx_rows_t r = gather_rows(s, d_items + p_lo, 1, p_n, UINT64_MAX, NULL);
    uint32_t* p_ids = dbuf_need(s, &s->db.tk_ids, (size_t)r.total * 4);
    double* p_scores = dbuf_need(s, &s->db.tk_scores, (size_t)r.total * 8);
    if (r.total) {
      smx_launch_cf_scores(s->stream, view_of(s), r.ids, p_n, r.offsets, r.pairs, p_ids, p_scores);
      s->n_launches++;
    }
    uint32_t* oc = counts + lo;
    uint32_t* oi = ids + (size_t)lo * k;
    double* os = scores + (size_t)lo * k;
    if (!out_dev) {
      char* o = dbuf_need(s, &s->db.host_out, (size_t)np * (12ull * k + 4));
      os = (double*)o;
      oi = (uint32_t*)(o + (size_t)np * k * 8);
      oc = oi + (size_t)np * k;
    }
    rec_run(s, np, d_boff + lo, p_lo, p_n, d_items, r.offsets, r.total, p_ids, p_scores, k, oc, oi, os);
    if (!out_dev) {
      copy_d2h(s, counts + lo, oc, (size_t)np * 4, s->stream);
      copy_d2h(s, ids + (size_t)lo * k, oi, (size_t)np * k * 4, s->stream);
      copy_d2h(s, scores + (size_t)lo * k, os, (size_t)np * k * 8, s->stream);
    }
  }
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* ------------------------------------------------------------------------------ enumeration */
/* Segments d_off[0..n] of d_pairs sorted by column in place, enqueued on s->stream (synchronises to read the number
 * of big segments and, per group of them, its end): the small ones by sort_small, the big ones a group of at most
 * SMATRIX_TOPK_PAIRS pairs at a time (a longer segment is a group of its own) by one radix sort each. */
static void sort_run(smatrix_t* s, uint32_t n, const uint64_t* d_off, uint32_t* d_pairs) {
  if (!n) return;
  uint32_t* ctl = dbuf_need(s, &s->db.tk_ctl, (size_t)n * 4 + 64);
  uint32_t* big_list = ctl + 16;
  CK(cudaMemsetAsync(ctl, 0, 64, s->stream));
  smx_launch_topk_classify(s->stream, n, d_off, big_list, ctl);
  copy_d2h(s, &s->h_small->sort, ctl, 16, s->stream);
  smx_launch_sort_small(s->stream, n, d_off, d_pairs);
  s->n_launches += 3;
  CK(cudaStreamSynchronize(s->stream));
  const uint32_t n_big = s->h_small->sort.n_big;
  if (!n_big) return;
  const size_t scan_items = smx_scan_scratch_items(n_big);
  uint32_t* lens = dbuf_need(s, &s->db.sr_big, (size_t)n_big * 4 + ((size_t)n_big + 1 + scan_items) * 8 + 16);
  uint64_t* big_off = (uint64_t*)(((uintptr_t)(lens + n_big) + 7) & ~(uintptr_t)7);
  smx_launch_sort_big_lens(s->stream, big_list, n_big, d_off, lens);
  smx_launch_scan(s->stream, lens, n_big, 0, big_off, big_off + n_big + 1);
  s->n_launches += 4;
  for (uint32_t lo = 0, hi; lo < n_big; lo = hi) {
    smx_launch_sort_cut(s->stream, big_off, n_big, lo, s->topk_pairs, ctl + 4);
    copy_d2h(s, &s->h_small->sort_cut, ctl + 4, 16, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->n_launches++;
    hi = s->h_small->sort_cut.end;
    const uint64_t P = s->h_small->sort_cut.pairs;
    if (P >= (1ull << 31)) smx_die("sort_rows: a row of %llu pairs is more than 2^31 - 1", (unsigned long long)P);
    uint64_t* keys = dbuf_need(s, &s->db.sr_keys, (size_t)P * 16);
    uint32_t* vals = dbuf_need(s, &s->db.sr_vals, (size_t)P * 8);
    const size_t sort_bytes = smx_rec_sort_bytes((uint32_t)P);
    void* sort_tmp = dbuf_need(s, &s->db.sr_sort, sort_bytes);
    smx_launch_sort_big(s->stream, big_list, lo, hi - lo, (uint32_t)P, big_off, d_off, d_pairs, keys, keys + P, vals,
                        vals + P, sort_tmp, sort_bytes);
    s->n_launches += 3;
  }
  s->n_sort_big += n_big;
}

void smatrix_b200_sort_rows(smatrix_t* s, size_t n, const uint64_t* d_offsets, uint32_t* d_pairs) {
  if (n >= 0xFFFFFFFFull) smx_die("sort_rows: too many segments in one call");
  if (!n) return;
  enter(s);
  sort_run(s, (uint32_t)n, d_offsets, d_pairs);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* the n keys d_in (device) in ascending order into d_tmp (device, n keys), the first min(cap, n) of them to out */
static void sort_keys_to(smatrix_t* s, const uint32_t* d_in, uint32_t* d_tmp, uint32_t n, uint32_t* out, uint64_t cap) {
  const size_t sort_bytes = smx_sort_keys_bytes(n);
  void* sort_tmp = dbuf_need(s, &s->db.ls_sort, sort_bytes);
  smx_launch_sort_keys(s->stream, d_in, d_tmp, n, sort_tmp, sort_bytes);
  s->n_launches++;
  const size_t bytes = (size_t)(cap < n ? cap : n) * 4;
  CK(cudaMemcpyAsync(out, d_tmp, bytes, cudaMemcpyDefault, s->stream));
  if (!is_device_ptr(out)) s->d2h_bytes += bytes;
}

/* one pass over the directory for the keys >= from, then a radix sort of them (not in a size query) */
uint64_t smatrix_list_rows(smatrix_t* s, uint32_t from, uint32_t* keys, uint64_t cap) {
  enter(s);
  read_ctl(s);
  const uint64_t rows = s->h_ctl->dir_used;
  if (rows >= (1ull << 31)) smx_die("list_rows: %llu rows are more than 2^31 - 1", (unsigned long long)rows);
  uint64_t m = 0;
  if (rows) {
    uint32_t* d_keys = dbuf_need(s, &s->db.ls_keys, (size_t)rows * 8 + 4); /* as found, sorted, the counter */
    uint32_t* d_cnt = d_keys + 2 * rows;
    CK(cudaMemsetAsync(d_cnt, 0, 4, s->stream));
    smx_launch_list_rows(s->stream, view_of(s), from, SMX_META_USED, d_keys, d_cnt);
    copy_d2h(s, &s->h_small->listed, d_cnt, 4, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->n_launches++;
    m = s->h_small->listed;
    if (keys && cap && m) sort_keys_to(s, d_keys, d_keys + rows, (uint32_t)m, keys, cap);
  }
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
  return m;
}

void smatrix_b200_sort_keys(smatrix_t* s, const uint32_t* d_keys, size_t n, uint32_t* out, uint64_t cap) {
  if (n >= (1ull << 31)) smx_die("sort_keys: %zu keys are more than 2^31 - 1", n);
  if (!n || !cap) return;
  enter(s);
  sort_keys_to(s, d_keys, dbuf_need(s, &s->db.ls_keys, n * 4), (uint32_t)n, out, cap);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* ------------------------------------------------------------------------------ single ops */
/* the answer of a single op, d_small[DS_OUT] */
static uint32_t single_answer(smatrix_t* s) {
  copy_d2h(s, &s->h_small->answer, s->d_small + DS_OUT, 4, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  return s->h_small->answer;
}

static uint32_t single_write(smatrix_t* s, int api_op, uint32_t x, uint32_t y, uint32_t v) {
  enter(s);
  uint32_t* d = s->d_small;
  s->h_small->op[0] = x; s->h_small->op[1] = y; s->h_small->op[2] = v;
  copy_h2d(s, d + DS_X, s->h_small->op, 12, s->stream);
  process_chunk(s, api_op, d + DS_X, d + DS_Y, d + DS_V, 1);
  smx_launch_get(s->stream, view_of(s), d + DS_X, d + DS_Y, 1, d + DS_OUT);
  s->n_launches++;
  const uint32_t r = single_answer(s);
  leave(s);
  return r;
}

uint32_t smatrix_set(smatrix_t* self, uint32_t x, uint32_t y, uint32_t value) {
  return single_write(self, 2, x, y, value);
}
uint32_t smatrix_incr(smatrix_t* self, uint32_t x, uint32_t y, uint32_t value) {
  return single_write(self, 0, x, y, value);
}
uint32_t smatrix_decr(smatrix_t* self, uint32_t x, uint32_t y, uint32_t value) {
  return single_write(self, 1, x, y, value);
}

uint32_t smatrix_get(smatrix_t* s, uint32_t x, uint32_t y) {
  enter(s);
  uint32_t* d = s->d_small;
  s->h_small->op[0] = x; s->h_small->op[1] = y;
  copy_h2d(s, d + DS_X, s->h_small->op, 8, s->stream);
  smx_launch_get(s->stream, view_of(s), d + DS_X, d + DS_Y, 1, d + DS_OUT);
  s->n_launches++;
  const uint32_t r = single_answer(s);
  leave(s);
  return r;
}

uint32_t smatrix_rowlen(smatrix_t* s, uint32_t x) {
  enter(s);
  uint32_t* d = s->d_small;
  s->h_small->op[0] = x;
  copy_h2d(s, d + DS_X, s->h_small->op, 4, s->stream);
  smx_launch_rowlen(s->stream, view_of(s), d + DS_X, 1, d + DS_OUT);
  s->n_launches++;
  const uint32_t r = single_answer(s);
  leave(s);
  return r;
}

uint32_t smatrix_getrow(smatrix_t* s, uint32_t x, uint32_t* ret, size_t ret_len) {
  enter(s);
  s->h_small->op[0] = x;
  const smx_rows_t r = gather_rows(s, s->h_small->op, 0, 1, UINT64_MAX, NULL);
  /* reference loop (src/smatrix.c:196-205): emit, then stop once num*8 >= ret_len */
  uint64_t room = (ret_len + 7) / 8;
  if (room < 1) room = 1;
  const uint64_t n = r.total < room ? r.total : room;
  if (n > 0) {
    CK(cudaMemcpyAsync(ret, r.pairs, (size_t)n * 8, cudaMemcpyDefault, s->stream));
    CK(cudaStreamSynchronize(s->stream));
  }
  leave(s);
  return (uint32_t)n;
}


/* ------------------------------------------------------------------------------ snapshot (.smx)
 * File-backed mode = snapshot on open/close (BASELINE.json north_star), in the reference's exact
 * byte format (src/smatrix.c:30-72) so that files interchange with the CPU library:
 *   512-byte header: 8 x 0x17, u64 offset of the first directory block
 *   directory blocks: u64 entries (4 194 304), u64 next-block offset, entries {u32 row, u64 row offset}
 *   row blocks: 8 x 0x23, u64 size (cells, power of two), size x {u32 column, u32 value}
 * Row blocks are written in the REFERENCE's hash layout (position = column % size, linear probing,
 * src/smatrix.c:363-380) because the reference loads them positionally (:533-540).  Like the
 * reference's loader, ours drops cells whose value is 0 (so zero-valued cells vanish across a
 * reopen, SURVEY.md 5); zero-valued cells are written last so that dropping them never breaks
 * another cell's probe chain. */
#define SMX_F_META 512ull
#define SMX_F_DIR_ENTRIES 4194304ull
#define SMX_F_DIR_HEAD 16ull
#define SMX_F_DIR_SLOT 12ull
#define SMX_F_ROW_HEAD 16ull
#define SMX_SNAPSHOT_ROWS (1u << 18)

static int write_all(int fd, const void* buf, size_t bytes, uint64_t at) {
  const char* p = (const char*)buf;
  while (bytes) {
    ssize_t w = pwrite(fd, p, bytes, (off_t)at);
    if (w <= 0) return -1;
    p += w; bytes -= (size_t)w; at += (uint64_t)w;
  }
  return 0;
}

static void sync_parent_dir(const char* fname) { /* make the rename itself durable */
  char* dir = strdup(fname);
  if (!dir) return;
  char* slash = strrchr(dir, '/');
  if (slash) *(slash == dir ? slash + 1 : slash) = 0;
  int dfd = open(slash ? dir : ".", O_RDONLY);
  if (dfd != -1) { (void)fsync(dfd); close(dfd); }
  free(dir);
}

#define SMX_F_BLOCK_BYTES (SMX_F_DIR_HEAD + SMX_F_DIR_ENTRIES * SMX_F_DIR_SLOT)
#define SMX_LOAD_WINDOW_DEFAULT (64u << 20) /* bytes of file per pread */
#define SMX_LOAD_CELLS_DEFAULT (1u << 24)   /* cells per piece: bounds the loader's device scratch */

/* ---- save, in two device-level pieces (include/smatrix_b200.h): a table's extent in the file, then its
 * row blocks and directory entries at a given place.  One table writes a whole file (snapshot_save); the
 * ranks of a sharded matrix write their parts of one file side by side (smx_router.c). */
static void snap_free_keys(smatrix_t* s) {
  if (s->snap_keys) cudaFree(s->snap_keys);
  free(s->snap_hoff); free(s->snap_hkeys);
  s->snap_keys = s->snap_hkeys = NULL;
  s->snap_hoff = NULL;
  s->snap_rows = 0;
}

/* caller holds the handle lock: the file matches the table again (after a load, a snapshot or a checkpoint).  Like
 * the snapshot's listing, the pass is not counted in SMX_STAT_LAUNCHES, so that a snapshot or a load counts the
 * launches it always did */
static void clear_dirty(smatrix_t* s) {
  smx_launch_clear_dirty(s->stream, view_of(s));
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
}

/* rows [first, first + len) of the listed keys: row sizes -> 8-byte units -> offsets (d_off[0..len]) */
typedef struct { smx_rowplan_t p; uint64_t* d_off; uint32_t* d_slog; } smx_snapchunk_t;
static smx_snapchunk_t snap_chunk_bufs(smatrix_t* s, uint32_t len) { /* the same buffers for the same len */
  smx_snapchunk_t c;
  c.d_slog = dbuf_need(s, &s->db.tmp, (size_t)len * 8);
  c.d_off = dbuf_need(s, &s->db.tmp64, ((size_t)len + 2 + smx_scan_scratch_items(len)) * 8);
  c.p = rowplan(s, len);
  return c;
}
static smx_snapchunk_t snap_chunk(smatrix_t* s, uint64_t first, uint32_t len) {
  const uint32_t* d_xs = s->snap_keys + first;
  smx_snapchunk_t c = snap_chunk_bufs(s, len);
  uint32_t* d_slog = c.d_slog;
  uint32_t* d_units = d_slog + len;
  smx_launch_row_counts(s->stream, view_of(s), d_xs, len, c.p.counts, c.p.info, c.p.big, c.p.n_big);
  smx_launch_row_slog(s->stream, view_of(s), d_xs, len, d_slog);
  smx_launch_snap_units(s->stream, c.p.counts, d_slog, len, d_units);
  smx_launch_scan(s->stream, d_units, len, 0, c.d_off, c.d_off + (size_t)len + 1);
  s->n_launches += 6;
  return c;
}

/* caller holds the handle lock, the stream is idle.  need = SMX_META_USED: every row (a snapshot);
 * | SMX_META_DIRTY: the rows written since the file last matched the table (a checkpoint) */
static void snap_extent(smatrix_t* s, uint64_t* rows, uint64_t* bytes, uint32_t need) {
  snap_free_keys(s);
  read_ctl(s);
  uint64_t n_rows = s->h_ctl->dir_used;
  if (n_rows) {
    s->snap_keys = (uint32_t*)dmalloc(s, n_rows * 4);
    CK(cudaMemsetAsync(&s->d_ctl->scratch, 0, 8, s->stream));
    smx_launch_list_rows(s->stream, view_of(s), 0, need, s->snap_keys, (uint32_t*)&s->d_ctl->scratch);
    if (need != SMX_META_USED) {
      copy_d2h(s, &s->h_small->listed, &s->d_ctl->scratch, 4, s->stream);
      CK(cudaStreamSynchronize(s->stream));
      n_rows = s->h_small->listed;
    }
  }
  s->snap_rows = n_rows;
  uint64_t total = 0;
  for (uint64_t first = 0; first < n_rows; first += SMX_SNAPSHOT_ROWS) {
    const uint32_t len = (uint32_t)((n_rows - first < SMX_SNAPSHOT_ROWS) ? n_rows - first : SMX_SNAPSHOT_ROWS);
    const smx_snapchunk_t c = snap_chunk(s, first, len);
    if (n_rows <= SMX_SNAPSHOT_ROWS) {
      s->snap_hoff = (uint64_t*)malloc(((size_t)len + 1) * 8);
      s->snap_hkeys = (uint32_t*)malloc((size_t)len * 4);
      if (!s->snap_hoff || !s->snap_hkeys) smx_die("out of host memory");
      copy_d2h(s, s->snap_hoff, c.d_off, ((size_t)len + 1) * 8, s->stream);
      copy_d2h(s, s->snap_hkeys, s->snap_keys, (size_t)len * 4, s->stream);
      copy_d2h(s, &s->h_small->n_big_rows, c.p.n_big, 4, s->stream);
      CK(cudaStreamSynchronize(s->stream));
      total = s->snap_hoff[len] * 8;
    } else {
      copy_d2h(s, &s->h_small->row_total, c.d_off + len, 8, s->stream);
      CK(cudaStreamSynchronize(s->stream));
      total += s->h_small->row_total * 8;
    }
  }
  CK(cudaGetLastError());
  *rows = n_rows;
  *bytes = total;
}

/* directory entries e0 .. e0 + n - 1 (12 bytes each in `ents`) of the chain at dir_base: entry e is slot e % 2^22
 * of block e / 2^22 */
static int snap_write_entries(int fd, const unsigned char* ents, uint64_t dir_base, uint64_t e0, uint64_t n) {
  while (n) {
    const uint64_t b = e0 / SMX_F_DIR_ENTRIES, slot = e0 % SMX_F_DIR_ENTRIES;
    const uint64_t run = (n < SMX_F_DIR_ENTRIES - slot) ? n : SMX_F_DIR_ENTRIES - slot;
    if (write_all(fd, ents, run * SMX_F_DIR_SLOT, dir_base + b * SMX_F_BLOCK_BYTES + SMX_F_DIR_HEAD + slot * SMX_F_DIR_SLOT))
      return -1;
    ents += run * SMX_F_DIR_SLOT; e0 += run; n -= run;
  }
  return 0;
}

/* caller holds the handle lock; the rows snap_extent listed, their blocks from byte fpos on, their entries from
 * first_entry on in the directory chain at dir_base */
static int snap_write(smatrix_t* s, int fd, uint64_t fpos, uint64_t dir_base, uint64_t first_entry) {
  const uint64_t n_rows = s->snap_rows;
  unsigned char* ents = (unsigned char*)malloc((size_t)SMX_SNAPSHOT_ROWS * SMX_F_DIR_SLOT);
  uint32_t* h_keys = (uint32_t*)malloc(SMX_SNAPSHOT_ROWS * 4);
  uint64_t* h_off = (uint64_t*)malloc(((size_t)SMX_SNAPSHOT_ROWS + 1) * 8);
  unsigned char* out = NULL; /* pinned: the row blocks come down at PCIe speed */
  size_t out_cap = 0;
  int rc = 0;
  if (!ents || !h_keys || !h_off) smx_die("out of host memory");
  /* K9: every chunk of rows is laid out ON THE DEVICE in the reference's row-block format (sizes ->
   * scan -> k_snap_rows / k_snap_big place every cell by column % size); the host only moves bytes */
  for (uint64_t first = 0; first < n_rows && rc == 0; first += SMX_SNAPSHOT_ROWS) {
    const uint32_t len = (uint32_t)((n_rows - first < SMX_SNAPSHOT_ROWS) ? n_rows - first : SMX_SNAPSHOT_ROWS);
    smx_snapchunk_t c;
    if (s->snap_hoff) { /* one chunk, laid out by snap_extent: its buffers still hold it */
      c = snap_chunk_bufs(s, len);
      memcpy(h_off, s->snap_hoff, ((size_t)len + 1) * 8);
      memcpy(h_keys, s->snap_hkeys, (size_t)len * 4);
    } else {
      c = snap_chunk(s, first, len);
      copy_d2h(s, h_off, c.d_off, ((size_t)len + 1) * 8, s->stream);
      copy_d2h(s, h_keys, s->snap_keys + first, (size_t)len * 4, s->stream);
      copy_d2h(s, &s->h_small->n_big_rows, c.p.n_big, 4, s->stream);
      CK(cudaStreamSynchronize(s->stream));
    }
    const size_t need = (size_t)h_off[len] * 8;
    uint64_t* rows = dbuf_need(s, &s->db.rows, need);
    if (need > out_cap) {
      if (out) cudaFreeHost(out);
      out_cap = need + need / 8 + 4096;
      CK(cudaHostAlloc((void**)&out, out_cap, cudaHostAllocDefault));
    }
    CK(cudaMemsetAsync(rows, 0, need, s->stream));
    smx_launch_snap_rows(s->stream, view_of(s), c.p.info, len, c.d_off, rows, c.p.big, s->h_small->n_big_rows);
    s->n_launches += 2;
    copy_d2h(s, out, rows, need, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    for (uint32_t i = 0; i < len; i++) {
      unsigned char* de = ents + (size_t)i * SMX_F_DIR_SLOT;
      const uint64_t row_fpos = fpos + h_off[i] * 8;
      memcpy(de, &h_keys[i], 4);
      memcpy(de + 4, &row_fpos, 8);
    }
    if (write_all(fd, out, need, fpos) || snap_write_entries(fd, ents, dir_base, first_entry + first, len)) rc = -1;
    fpos += need;
  }
  CK(cudaGetLastError());
  if (out) cudaFreeHost(out);
  free(ents); free(h_keys); free(h_off);
  snap_free_keys(s);
  return rc;
}

uint64_t smatrix_b200_snap_rows_base(uint64_t total_rows) {
  const uint64_t n_blocks = total_rows ? (total_rows + SMX_F_DIR_ENTRIES - 1) / SMX_F_DIR_ENTRIES : 1;
  return SMX_F_META + n_blocks * SMX_F_BLOCK_BYTES;
}

int smatrix_b200_snap_layout(int fd, uint64_t total_rows, uint64_t total_bytes) {
  const uint64_t n_blocks = total_rows ? (total_rows + SMX_F_DIR_ENTRIES - 1) / SMX_F_DIR_ENTRIES : 1;
  unsigned char head[SMX_F_META];
  memset(head, 0, sizeof head);
  memset(head, 0x17, 8);
  { uint64_t first = SMX_F_META; memcpy(head + 8, &first, 8); }
  if (write_all(fd, head, sizeof head, 0)) return -1;
  for (uint64_t b = 0; b < n_blocks; b++) {
    const uint64_t bpos = SMX_F_META + b * SMX_F_BLOCK_BYTES;
    unsigned char bh[SMX_F_DIR_HEAD];
    const uint64_t entries = SMX_F_DIR_ENTRIES, next = (b + 1 < n_blocks) ? bpos + SMX_F_BLOCK_BYTES : 0;
    memcpy(bh, &entries, 8);
    memcpy(bh + 8, &next, 8);
    if (write_all(fd, bh, sizeof bh, bpos)) return -1;
  }
  /* unused directory entries read back as zeros */
  return ftruncate(fd, (off_t)(smatrix_b200_snap_rows_base(total_rows) + total_bytes)) == -1 ? -1 : 0;
}

int smatrix_b200_snap_extent(smatrix_t* s, uint64_t* rows, uint64_t* bytes) {
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  snap_extent(s, rows, bytes, SMX_META_USED);
  leave(s);
  return 0;
}

int smatrix_b200_snap_write(smatrix_t* s, int fd, uint64_t byte_base, uint64_t first_entry) {
  return smatrix_b200_snap_write_at(s, fd, byte_base, SMX_F_META, first_entry);
}

int smatrix_b200_snap_write_at(smatrix_t* s, int fd, uint64_t byte_base, uint64_t dir_base, uint64_t first_entry) {
  enter(s);
  const int rc = snap_write(s, fd, byte_base, dir_base, first_entry);
  leave(s);
  return rc;
}

int smatrix_b200_snap_commit(const char* tmp, const char* fname) {
  if (rename(tmp, fname) == -1) return -1;
  sync_parent_dir(fname);
  return 0;
}

/* caller holds the handle lock */
static int snapshot_save(smatrix_t* s) {
  size_t fl = strlen(s->fname);
  char* tmp = (char*)malloc(fl + 8);
  if (!tmp) return -1;
  memcpy(tmp, s->fname, fl);
  memcpy(tmp + fl, ".tmp", 5);
  int fd = open(tmp, O_RDWR | O_CREAT | O_TRUNC, 00600);
  if (fd == -1) { perror("cannot open file"); free(tmp); return -1; }
  uint64_t rows = 0, bytes = 0;
  snap_extent(s, &rows, &bytes, SMX_META_USED);
  int rc = smatrix_b200_snap_layout(fd, rows, bytes);
  if (snap_write(s, fd, smatrix_b200_snap_rows_base(rows), SMX_F_META, 0)) rc = -1;
  if (rc == 0 && fsync(fd) == -1) rc = -1; /* the data is on disk before the old file is replaced */
  if (close(fd) == -1) rc = -1;
  if (rc == 0) rc = smatrix_b200_snap_commit(tmp, s->fname);
  if (rc) {
    perror("libsmatrix: writing the snapshot failed");
    unlink(tmp); /* the previous snapshot, if any, is still intact */
  } else {
    clear_dirty(s); /* the file matches the table */
    s->ck_base = 1;
  }
  free(tmp);
  return rc;
}

static int read_all(int fd, void* buf, size_t bytes, uint64_t at) {
  char* p = (char*)buf;
  while (bytes) {
    ssize_t r = pread(fd, p, bytes, (off_t)at);
    if (r <= 0) return -1;
    p += r; bytes -= (size_t)r; at += (uint64_t)r;
  }
  return 0;
}

/* ---- load: one reader of row blocks for a share of the directory (include/smatrix_b200.h) ----
 * The share's rows are read in file order, window by window, into pinned memory; every row header is
 * checked here; the raw bytes go up with a tile table and k_load_count / k_load_emit expand them into
 * the op stream on the device. */
typedef struct { uint64_t rpos; uint32_t key; } smx_ldrow_t;
struct smx_loader_s {
  smatrix_t* s;
  int fd;
  uint64_t fsize;
  smx_ldrow_t* rows; /* this share, by file offset */
  uint64_t n, next;
  size_t window;     /* SMATRIX_LOAD_WINDOW: bytes per pread (grown for a bigger row) */
  uint64_t cells;    /* SMATRIX_LOAD_CELLS: cells per piece (a bigger row is a piece of its own) */
  int sorted;        /* rows are in file order (load_next); until then in directory order (load_entries) */
  unsigned char* win; size_t win_cap;   /* pinned */
  smx_load_tile_t* tiles; size_t tiles_cap;
  uint32_t* fix; size_t fix_cap;        /* keys, then log2 sizes */
};

static int ldrow_cmp(const void* a, const void* b) {
  const uint64_t x = ((const smx_ldrow_t*)a)->rpos, y = ((const smx_ldrow_t*)b)->rpos;
  return x < y ? -1 : x > y;
}

void smatrix_b200_load_end(smx_loader_t* ld) {
  if (!ld) return;
  if (ld->win) cudaFreeHost(ld->win);
  free(ld->rows); free(ld->tiles); free(ld->fix);
  free(ld);
}

smx_loader_t* smatrix_b200_load_begin(smatrix_t* s, int fd, int share, int shares) {
  unsigned char head[SMX_F_META];
  struct stat st;
  if (shares < 1 || share < 0 || share >= shares || fstat(fd, &st) != 0) return NULL;
  if (read_all(fd, head, sizeof head, 0) || head[0] != 0x17 || head[1] != 0x17) {
    fprintf(stderr, "libsmatrix: invalid file header\n");
    return NULL;
  }
  smx_loader_t* ld = (smx_loader_t*)calloc(1, sizeof *ld);
  unsigned char* block = (unsigned char*)malloc(SMX_F_DIR_ENTRIES * SMX_F_DIR_SLOT);
  if (!ld || !block) smx_die("out of host memory");
  ld->s = s;
  ld->fd = fd;
  ld->fsize = (uint64_t)st.st_size;
  ld->window = env_u32("SMATRIX_LOAD_WINDOW", SMX_LOAD_WINDOW_DEFAULT);
  if (ld->window < 64) ld->window = 64;
  ld->cells = env_u32("SMATRIX_LOAD_CELLS", SMX_LOAD_CELLS_DEFAULT);
  if (ld->cells < 1) ld->cells = 1;
  /* the chain of directory blocks (a slot with rpos = 0 ends its block, src/smatrix.c:814-815): count the
   * entries, then read this share's contiguous range of them */
  uint64_t bpos, total = 0, nblk = 0, blk_cap = 0;
  uint64_t* blk = NULL; /* per block: position, entries in use */
  memcpy(&bpos, head + 8, 8);
  int rc = 0;
  while (bpos && rc == 0) {
    unsigned char bh[SMX_F_DIR_HEAD];
    uint64_t entries, next, used = 0;
    if (nblk > ld->fsize / SMX_F_DIR_HEAD || read_all(fd, bh, sizeof bh, bpos)) { rc = -1; break; } /* or a loop */
    memcpy(&entries, bh, 8);
    memcpy(&next, bh + 8, 8);
    if (entries > SMX_F_DIR_ENTRIES || read_all(fd, block, entries * SMX_F_DIR_SLOT, bpos + SMX_F_DIR_HEAD)) { rc = -1; break; }
    for (; used < entries; used++) {
      uint64_t rpos;
      memcpy(&rpos, block + used * SMX_F_DIR_SLOT + 4, 8);
      if (!rpos) break;
    }
    if (nblk == blk_cap) {
      blk_cap = blk_cap * 2 + 16;
      blk = (uint64_t*)realloc(blk, blk_cap * 16);
      if (!blk) smx_die("out of host memory");
    }
    blk[2 * nblk] = bpos; blk[2 * nblk + 1] = used; nblk++;
    total += used;
    bpos = next;
  }
  const uint64_t lo = total * (uint64_t)share / (uint64_t)shares, hi = total * ((uint64_t)share + 1) / (uint64_t)shares;
  ld->n = hi - lo;
  ld->rows = (smx_ldrow_t*)malloc((ld->n ? ld->n : 1) * sizeof(smx_ldrow_t));
  if (!ld->rows) smx_die("out of host memory");
  for (uint64_t b = 0, e = 0; b < nblk && rc == 0; e += blk[2 * b + 1], b++) {
    const uint64_t a = lo > e ? lo : e, z = hi < e + blk[2 * b + 1] ? hi : e + blk[2 * b + 1];
    if (a >= z) continue;
    if (read_all(fd, block, (z - a) * SMX_F_DIR_SLOT, blk[2 * b] + SMX_F_DIR_HEAD + (a - e) * SMX_F_DIR_SLOT)) { rc = -1; break; }
    for (uint64_t k = a; k < z; k++) {
      smx_ldrow_t* r = &ld->rows[k - lo];
      memcpy(&r->key, block + (k - a) * SMX_F_DIR_SLOT, 4);
      memcpy(&r->rpos, block + (k - a) * SMX_F_DIR_SLOT + 4, 8);
    }
  }
  free(blk);
  free(block);
  if (rc) {
    fprintf(stderr, "libsmatrix: file is corrupt\n");
    smatrix_b200_load_end(ld);
    return NULL;
  }
  return ld;
}

uint64_t smatrix_b200_load_entries(smx_loader_t* ld, uint64_t first, uint64_t n, uint32_t* d_keys, uint32_t* d_lo,
                                   uint32_t* d_hi) {
  if (ld->sorted) smx_die("load_entries: the loader has started reading rows");
  if (!d_keys || first >= ld->n) return ld->n;
  if (n > ld->n - first) n = ld->n - first;
  smatrix_t* s = ld->s;
  uint32_t* h = (uint32_t*)malloc((size_t)n * 12 + 4);
  if (!h) smx_die("out of host memory");
  for (uint64_t i = 0; i < n; i++) {
    const smx_ldrow_t* r = &ld->rows[first + i];
    h[i] = r->key;
    h[n + i] = (uint32_t)r->rpos;
    h[2 * n + i] = (uint32_t)(r->rpos >> 32);
  }
  enter(s);
  copy_h2d(s, d_keys, h, (size_t)n * 4, s->stream);
  copy_h2d(s, d_lo, h + n, (size_t)n * 4, s->stream);
  copy_h2d(s, d_hi, h + 2 * n, (size_t)n * 4, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  leave(s);
  free(h);
  return ld->n;
}

/* the window holds file bytes [at, at + len) */
static int load_window(smx_loader_t* ld, uint64_t at, size_t len) {
  if (len > ld->win_cap) {
    if (ld->win) cudaFreeHost(ld->win);
    ld->win_cap = len;
    CK(cudaHostAlloc((void**)&ld->win, ld->win_cap, cudaHostAllocDefault));
  }
  return read_all(ld->fd, ld->win, len, at);
}

int smatrix_b200_load_next(smx_loader_t* ld, const uint32_t** d_xs, const uint32_t** d_ys, const uint32_t** d_vs,
                           size_t* n_ops, const uint32_t** d_keys, const uint32_t** d_logs, size_t* n_rows) {
  smatrix_t* s = ld->s;
  *n_ops = *n_rows = 0;
  if (!ld->sorted) { /* reads go forward through the file even where a foreign file's rows are not in directory order */
    ld->sorted = 1;
    for (uint64_t i = 1; i < ld->n; i++)
      if (ld->rows[i].rpos < ld->rows[i - 1].rpos) { qsort(ld->rows, ld->n, sizeof(smx_ldrow_t), ldrow_cmp); break; }
  }
  if (ld->next == ld->n) return 0;
  const uint64_t wstart = ld->rows[ld->next].rpos & ~7ull; /* our files keep every cell 8-byte aligned */
  size_t len = ld->window;
  uint64_t i = ld->next, cells = 0, nt = 0, nf = 0, end = 0;
  if (ld->rows[i].rpos + SMX_F_ROW_HEAD > ld->fsize) return -1;
  for (;;) { /* read; grow the window if its first row does not fit */
    if (len > ld->fsize - wstart) len = (size_t)(ld->fsize - wstart);
    if (load_window(ld, wstart, len)) return -1;
    const uint64_t rpos = ld->rows[i].rpos;
    if (rpos + SMX_F_ROW_HEAD <= wstart + len) {
      uint64_t size;
      memcpy(&size, ld->win + (rpos - wstart) + 8, 8);
      if (size == 0 || (size & (size - 1)) || size > (1ull << 32) || rpos + SMX_F_ROW_HEAD + size * 8 > ld->fsize) return -1;
      if (rpos + SMX_F_ROW_HEAD + size * 8 <= wstart + len) break;
      len = (size_t)(rpos + SMX_F_ROW_HEAD + size * 8 - wstart);
    } else {
      len = (size_t)(rpos + SMX_F_ROW_HEAD - wstart);
    }
  }
  for (; i < ld->n; i++) {
    const uint64_t rpos = ld->rows[i].rpos;
    if (rpos + SMX_F_ROW_HEAD > wstart + len) break;
    const unsigned char* rh = ld->win + (rpos - wstart);
    uint64_t size;
    memcpy(&size, rh + 8, 8);
    if (rh[0] != 0x23 || rh[7] != 0x23 || size == 0 || (size & (size - 1)) || size > (1ull << 32) ||
        rpos + SMX_F_ROW_HEAD + size * 8 > ld->fsize)
      return -1;
    if (rpos + SMX_F_ROW_HEAD + size * 8 > wstart + len) break;
    if (i > ld->next && cells + size > ld->cells) break;
    const uint64_t tile = 1ull << SMX_LOAD_TILE_LOG, ntiles = (size + tile - 1) / tile;
    if (nt + ntiles > ld->tiles_cap) {
      ld->tiles_cap = (nt + ntiles) * 2 + 1024;
      ld->tiles = (smx_load_tile_t*)realloc(ld->tiles, ld->tiles_cap * sizeof(smx_load_tile_t));
      if (!ld->tiles) smx_die("out of host memory");
    }
    for (uint64_t k = 0; k < ntiles; k++) {
      smx_load_tile_t* t = &ld->tiles[nt++];
      t->off = rpos - wstart + SMX_F_ROW_HEAD + k * tile * 8;
      t->key = ld->rows[i].key;
      t->cells = (uint32_t)(size < tile ? size : tile) | (k == 0 ? SMX_LOAD_FIRST : 0u);
    }
    if (nf + 1 > ld->fix_cap) {
      ld->fix_cap = nf * 2 + 1024;
      ld->fix = (uint32_t*)realloc(ld->fix, ld->fix_cap * 2 * 4);
      if (!ld->fix) smx_die("out of host memory");
    }
    ld->fix[nf++] = ld->rows[i].key;
    cells += size;
    end = rpos + SMX_F_ROW_HEAD + size * 8 - wstart;
  }
  for (uint64_t r = 0; r < nf; r++) { /* keys, then the log2 row sizes */
    uint64_t size;
    memcpy(&size, ld->win + (ld->rows[ld->next + r].rpos - wstart) + 8, 8);
    ld->fix[nf + r] = log2_u64(size);
  }
  ld->next = i;
  if (nt >= 0xFFFFFFFFull) smx_die("load: too many rows in one window");
  enter(s);
  /* the window up to the end of its last row goes to the device */
  void* raw = dbuf_need(s, &s->db.ld_raw, end);
  smx_load_tile_t* tiles = dbuf_need(s, &s->db.ld_tiles, nt * sizeof(smx_load_tile_t));
  uint32_t* cnt = dbuf_need(s, &s->db.ld_cnt, nt * 4);
  uint64_t* off = dbuf_need(s, &s->db.ld_off, (nt + 2 + smx_scan_scratch_items((uint32_t)nt)) * 8);
  uint32_t* fix = dbuf_need(s, &s->db.ld_fix, nf * 8);
  copy_h2d(s, raw, ld->win, end, s->stream);
  copy_h2d(s, tiles, ld->tiles, nt * sizeof(smx_load_tile_t), s->stream);
  copy_h2d(s, fix, ld->fix, nf * 8, s->stream);
  smx_launch_load_count(s->stream, raw, tiles, (uint32_t)nt, cnt);
  smx_launch_scan(s->stream, cnt, (uint32_t)nt, 0, off, off + nt + 1);
  copy_d2h(s, &s->h_small->row_total, off + nt, 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  const uint64_t ops = s->h_small->row_total;
  uint32_t* xs = dbuf_need(s, &s->db.ld_ops, ops * 12);
  smx_launch_load_emit(s->stream, raw, tiles, (uint32_t)nt, off, xs, xs + ops, xs + 2 * ops);
  s->n_launches += 5;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
  *d_xs = xs; *d_ys = xs + ops; *d_vs = xs + 2 * ops;
  *n_ops = (size_t)ops;
  *d_keys = fix; *d_logs = fix + nf;
  *n_rows = (size_t)nf;
  return 1;
}

void smatrix_b200_load_fixup(smatrix_t* s, const uint32_t* d_keys, const uint32_t* d_logs, size_t n) {
  if (!n) return;
  if (n >= 0xFFFFFFFFull) smx_die("load_fixup: batch too large");
  enter(s);
  smx_launch_load_fixup(s->stream, view_of(s), d_keys, d_logs, (uint32_t)n);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* handle is complete and not yet published: public entry points may be used.  One GPU reads the whole
 * directory as its share; every piece is applied as a device-array set batch, then its rows take the
 * file's row sizes (k_load_fixup) — the rowlen automaton continues from there. */
static int snapshot_load(smatrix_t* s, int fd) {
  smx_loader_t* ld = smatrix_b200_load_begin(s, fd, 0, 1);
  if (!ld) return -1;
  int rc;
  for (;;) {
    const uint32_t *xs, *ys, *vs, *keys, *logs;
    size_t n, nr;
    rc = smatrix_b200_load_next(ld, &xs, &ys, &vs, &n, &keys, &logs, &nr);
    if (rc <= 0) break;
    smatrix_set_batch(s, xs, ys, vs, n);
    smatrix_b200_load_fixup(s, keys, logs, nr);
  }
  if (rc) fprintf(stderr, "libsmatrix: file is corrupt\n");
  smatrix_b200_load_end(ld);
  if (rc == 0) { /* the loaded rows are what the file holds */
    enter(s);
    clear_dirty(s);
    s->ck_base = 1;
    leave(s);
  }
  return rc;
}

/* ------------------------------------------------------------------------------ checkpoint (.smx)
 * An incremental save: only the row blocks of the rows written since the file last matched the table (the
 * SMX_META_DIRTY marks k_upsert leaves) are appended, behind them a new directory chain that lists the clean rows'
 * old entries (their blocks in the file are still right) and the dirty rows' new ones, and then the header is
 * switched to that chain.  The reference's own writer leaves dead blocks behind and chains directory blocks at the
 * end of its file in the same way, so every reader of the format follows the header's pointer.  Order of the
 * steps, so that the file loads to the old or the new state at every moment: blocks at E = round_up(size, 8),
 * directory at D behind them (full 2^22-entry blocks, the unused entries left to ftruncate: sparse), fsync, the 8
 * header bytes at offset 8 := D, fsync.  Nothing before E but those 8 bytes is written. */
void smatrix_b200_clear_dirty(smatrix_t* s) {
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  clear_dirty(s);
  leave(s);
}

int smatrix_b200_ckpt_extent(smatrix_t* s, uint64_t* rows, uint64_t* bytes) {
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  snap_extent(s, rows, bytes, SMX_META_USED | SMX_META_DIRTY);
  leave(s);
  return 0;
}

static uint64_t count_dirty(smatrix_t* s) { /* caller holds the handle lock */
  read_ctl(s);
  if (!s->h_ctl->dir_used) return 0;
  CK(cudaMemsetAsync(&s->d_ctl->scratch, 0, 8, s->stream));
  smx_launch_list_rows(s->stream, view_of(s), 0, SMX_META_USED | SMX_META_DIRTY, NULL, (uint32_t*)&s->d_ctl->scratch);
  s->n_launches++;
  copy_d2h(s, &s->h_small->listed, &s->d_ctl->scratch, 4, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  return s->h_small->listed;
}

uint64_t smatrix_b200_ckpt_keep(smatrix_t* s, const uint32_t* d_keys, const uint32_t* d_lo, const uint32_t* d_hi,
                                size_t n, uint64_t* kept) {
  uint64_t missing = 0;
  enter(s);
  for (size_t first = 0; first < n;) {
    const uint32_t len = (uint32_t)(n - first < SMX_SNAPSHOT_ROWS ? n - first : SMX_SNAPSHOT_ROWS);
    uint32_t* flags = dbuf_need(s, &s->db.ck_flags, (size_t)len * 4 + 8);
    uint64_t* off = dbuf_need(s, &s->db.ck_off, ((size_t)len + 2 + smx_scan_scratch_items(len)) * 8);
    uint32_t* out = dbuf_need(s, &s->db.ck_out, (size_t)len * SMX_F_DIR_SLOT);
    uint32_t* d_missing = flags + len;
    CK(cudaMemsetAsync(d_missing, 0, 4, s->stream));
    smx_launch_keep(s->stream, view_of(s), d_keys + first, d_lo + first, d_hi + first, len, flags, off,
                    off + (size_t)len + 1, d_missing, out);
    s->n_launches += 5;
    copy_d2h(s, &s->h_small->ck_missing, d_missing, 4, s->stream);
    copy_d2h(s, &s->h_small->ck_kept, off + len, 8, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    const uint64_t k = s->h_small->ck_kept;
    missing += s->h_small->ck_missing;
    if (s->ck_kept_n + k > s->ck_kept_cap) {
      s->ck_kept_cap = (s->ck_kept_n + k) * 2 + 1024;
      s->ck_kept = (unsigned char*)realloc(s->ck_kept, (size_t)s->ck_kept_cap * SMX_F_DIR_SLOT);
      if (!s->ck_kept) smx_die("out of host memory");
    }
    copy_d2h(s, s->ck_kept + s->ck_kept_n * SMX_F_DIR_SLOT, out, (size_t)k * SMX_F_DIR_SLOT, s->stream);
    CK(cudaStreamSynchronize(s->stream));
    s->ck_kept_n += k;
    first += len;
  }
  CK(cudaGetLastError());
  *kept = s->ck_kept_n;
  leave(s);
  return missing;
}

int smatrix_b200_ckpt_write_kept(smatrix_t* s, int fd, uint64_t dir_base, uint64_t first_entry) {
  enter(s);
  const int rc = snap_write_entries(fd, s->ck_kept, dir_base, first_entry, s->ck_kept_n);
  s->ck_kept_n = 0;
  leave(s);
  return rc;
}

void smatrix_b200_ckpt_reset(smatrix_t* s) {
  enter(s);
  s->ck_kept_n = 0;
  snap_free_keys(s);
  leave(s);
}

int smatrix_b200_ckpt_layout(int fd, uint64_t dir_base, uint64_t entries) {
  const uint64_t n_blocks = entries ? (entries + SMX_F_DIR_ENTRIES - 1) / SMX_F_DIR_ENTRIES : 1;
  /* the file first reaches its final size: the unused entries read back as zeros */
  if (ftruncate(fd, (off_t)(dir_base + n_blocks * SMX_F_BLOCK_BYTES)) == -1) return -1;
  for (uint64_t b = 0; b < n_blocks; b++) {
    const uint64_t bpos = dir_base + b * SMX_F_BLOCK_BYTES;
    unsigned char bh[SMX_F_DIR_HEAD];
    const uint64_t cnt = SMX_F_DIR_ENTRIES, next = (b + 1 < n_blocks) ? bpos + SMX_F_BLOCK_BYTES : 0;
    memcpy(bh, &cnt, 8);
    memcpy(bh + 8, &next, 8);
    if (write_all(fd, bh, sizeof bh, bpos)) return -1;
  }
  return 0;
}

int smatrix_b200_ckpt_switch(int fd, uint64_t dir_base) {
  if (fsync(fd) == -1) return -1; /* blocks and directory are on disk before the header points at them */
  if (write_all(fd, &dir_base, 8, 8)) return -1;
  return fsync(fd) == -1 ? -1 : 0;
}

/* caller holds the handle lock, the stream is idle */
static int checkpoint(smatrix_t* s) {
  const uint64_t dirty = count_dirty(s);
  if (!dirty) return 0;
  if (!s->ck_base) return snapshot_save(s); /* the file never matched the table */
  const int fd = open(s->fname, O_RDWR);
  if (fd == -1) {
    if (errno == ENOENT) return snapshot_save(s);
    perror("libsmatrix: cannot open the file for a checkpoint");
    return -1;
  }
  struct stat st;
  if (fstat(fd, &st) != 0) { perror("libsmatrix: checkpoint"); close(fd); return -1; }
  if (st.st_size == 0) { close(fd); return snapshot_save(s); }
  const uint64_t fsize = (uint64_t)st.st_size;
  uint64_t rows = 0, all_bytes = 0, drows = 0, dbytes = 0, kept = 0, missing = 0;
  snap_extent(s, &rows, &all_bytes, SMX_META_USED); /* the size of a full snapshot */
  snap_free_keys(s);
  leave(s); /* the pieces below take the lock themselves */
  s->ck_kept_n = 0;
  smx_loader_t* ld = smatrix_b200_load_begin(s, fd, 0, 1);
  int match = ld != NULL;
  if (ld) {
    const uint64_t n = smatrix_b200_load_entries(ld, 0, 0, NULL, NULL, NULL);
    enter(s);
    uint32_t* d_in = dbuf_need(s, &s->db.ck_in, (size_t)(n < SMX_SNAPSHOT_ROWS ? n : SMX_SNAPSHOT_ROWS) * 12 + 16);
    leave(s);
    const uint64_t piece = SMX_SNAPSHOT_ROWS;
    for (uint64_t first = 0; first < n; first += piece) {
      const uint64_t len = n - first < piece ? n - first : piece;
      smatrix_b200_load_entries(ld, first, len, d_in, d_in + len, d_in + 2 * len);
      missing += smatrix_b200_ckpt_keep(s, d_in, d_in + len, d_in + 2 * len, (size_t)len, &kept);
    }
    smatrix_b200_load_end(ld);
  }
  enter(s);
  snap_extent(s, &drows, &dbytes, SMX_META_USED | SMX_META_DIRTY); /* held until snap_write */
  /* the old directory lists exactly the table's rows: every listed row is in the table, and the clean ones and the
   * dirty ones add up to all of them (a dirty row may be new, so it need not be listed) */
  match = match && missing == 0 && kept + drows == rows;
  const uint64_t E = (fsize + 7) & ~7ull, D = E + dbytes;
  const uint64_t end = D + smatrix_b200_snap_rows_base(kept + drows) - SMX_F_META;
  if (!match || end > 2 * (smatrix_b200_snap_rows_base(rows) + all_bytes)) {
    /* a file that does not describe this table, or one that has grown to twice a full snapshot: rewrite it */
    close(fd);
    s->ck_kept_n = 0;
    snap_free_keys(s);
    return snapshot_save(s);
  }
  int rc = smatrix_b200_ckpt_layout(fd, D, kept + drows);
  if (rc == 0 && snap_write(s, fd, E, D, kept)) rc = -1;
  snap_free_keys(s);
  if (rc == 0 && snap_write_entries(fd, s->ck_kept, D, 0, kept)) rc = -1;
  s->ck_kept_n = 0;
  if (rc) {
    (void)!ftruncate(fd, (off_t)fsize); /* the header was not switched: the old file as it was */
  } else if (smatrix_b200_ckpt_switch(fd, D)) {
    rc = -1;
  }
  if (close(fd) == -1) rc = -1;
  if (rc) {
    perror("libsmatrix: writing the checkpoint failed");
    return -1;
  }
  clear_dirty(s);
  return 0;
}

int smatrix_b200_checkpoint(smatrix_t* s) {
  if (!s->fname) return -1;
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  const int rc = checkpoint(s);
  leave(s);
  return rc;
}

/* ------------------------------------------------------------------------------ open / close */
smatrix_t* smatrix_b200_open(const char* fname, int device) {
  return smatrix_b200_open_arena(fname, device, (size_t)env_u32("SMATRIX_ARENA_GIB", 0) << 30);
}

smatrix_t* smatrix_b200_open_arena(const char* fname, int device, size_t arena_bytes) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    fprintf(stderr, "libsmatrix: no usable CUDA device (this build has no CPU path)\n");
    return NULL;
  }
  if (device < 0 || device >= ndev) {
    fprintf(stderr, "libsmatrix: CUDA device %d out of range (0..%d)\n", device, ndev - 1);
    return NULL;
  }
  int fd = -1;
  if (fname) { /* like src/smatrix.c:90-96: the file must be creatable / readable */
    fd = open(fname, O_RDWR | O_CREAT, 00600);
    if (fd == -1) {
      perror("cannot open file");
      return NULL;
    }
  }
  if (cudaSetDevice(device) != cudaSuccess) { if (fd != -1) close(fd); return NULL; }
  smatrix_t* s = (smatrix_t*)calloc(1, sizeof(smatrix_t));
  if (!s) return NULL;
  s->device = device;
  pthread_mutex_init(&s->mu, NULL);
  CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&s->read_stream[0], cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&s->read_stream[1], cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&s->stage_ready[0], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&s->stage_ready[1], cudaEventDisableTiming));
  CK(cudaEventCreate(&s->ev0));
  CK(cudaEventCreate(&s->ev1));
  CK(cudaEventCreate(&s->t_start));
  CK(cudaEventCreate(&s->t_stop));
  s->dir_log_min = env_u32("SMATRIX_DIR_LOG2", SMX_DIR_LOG_DEFAULT);
  if (s->dir_log_min < 4) s->dir_log_min = 4;
  if (s->dir_log_min > 31) s->dir_log_min = 31;
  s->chunk_max = env_u32("SMATRIX_CHUNK", SMX_CHUNK_DEFAULT);
  if (s->chunk_max < 1) s->chunk_max = 1;
  if (s->chunk_max > (1u << 30)) s->chunk_max = 1u << 30;
  s->preagg = (int)env_u32("SMATRIX_PREAGG", 1);
  s->recycle = (int)env_u32("SMATRIX_RECYCLE", 1);
  s->debug = (int)env_u32("SMATRIX_DEBUG", 0);
  s->migrate_tiles = (int)env_u32("SMATRIX_MIGRATE_TILES", 1);
  s->spill_cap = env_u32("SMATRIX_SPILL_CAP", 1u << 16);
  if (s->spill_cap < 1) s->spill_cap = 1u << 16;
  s->presize = (int)env_u32("SMATRIX_PRESIZE", 1);
  s->stage_max = env_u32("SMATRIX_STAGE", SMX_STAGE_MAX);
  if (s->stage_max < 1024) s->stage_max = 1024;
  s->get_slices = (int)env_u32("SMATRIX_GET_SLICES", 1);
  s->get_slice_min = env_u32("SMATRIX_GET_SLICE_MIN", 1u << 22);
  s->topk_pairs = env_u32("SMATRIX_TOPK_PAIRS", 1u << 28);
  if (s->topk_pairs < 1) s->topk_pairs = 1;
  s->get_flags = s->get_slices & SMX_GET_FLAGS;
  s->get_slices = (s->get_slices & 3) > 2 ? 2 : (s->get_slices & 3);
  s->part_min = env_u32("SMATRIX_PARTITION_MIN", 1u << 20);
  s->slice_log = env_u32("SMATRIX_SLICE_LOG2", 17);
  s->parts_log_max = env_u32("SMATRIX_PARTS_LOG2", 7);
  if (s->parts_log_max > 7) s->parts_log_max = 7; /* 2 x 128 = SMX_MAX_PARTS_H parts */
  s->wide_slices = (int)env_u32("SMATRIX_WIDE_SLICES", 1);
  s->arena_bytes = arena_bytes;
  if (s->arena_bytes) push_segment(s, (char*)dmalloc(s, s->arena_bytes), s->arena_bytes);
  s->dir_cap = 1ull << s->dir_log_min;
  s->dir_in_arena = s->arena_bytes != 0; /* then nothing is cudaFree'd while batches are applied */
  s->dir = s->dir_in_arena ? (smx_row_t*)slab_reserve(s, (size_t)s->dir_cap * sizeof(smx_row_t))
                           : (smx_row_t*)dmalloc(s, (size_t)s->dir_cap * sizeof(smx_row_t));
  CK(cudaMemsetAsync(s->dir, 0, (size_t)s->dir_cap * sizeof(smx_row_t), s->stream));
  s->d_ctl = (smx_ctl_t*)dmalloc(s, sizeof(smx_ctl_t));
  CK(cudaMemsetAsync(s->d_ctl, 0, sizeof(smx_ctl_t), s->stream));
  CK(cudaHostAlloc((void**)&s->h_ctl, sizeof(smx_ctl_t), cudaHostAllocDefault));
  memset(s->h_ctl, 0, sizeof(smx_ctl_t));
  s->d_small = (uint32_t*)dmalloc(s, DS_WORDS * 4);
  CK(cudaHostAlloc((void**)&s->h_small, sizeof(smx_small_t), cudaHostAllocDefault));
  if (s->arena_bytes) {
    /* a table with an arena is a bulk table: take the small cudaMalloc'ed scratch of the write path now (sketch
     * bitmap, partition counters, spill list of the tile-wise re-placement) so that no batch ever waits for
     * cudaMalloc — right after another table's arena went back to the driver a single call was seen to stall
     * for 20 - 150 ms (config 3, first step: profiles/r2_summary.md) */
    dbuf_need(s, &s->db.tmp, (size_t)1 << (SMX_SKETCH_BITS_LOG - 3));
    dbuf_need(s, &s->db.tmp64, 3 * SMX_MAX_PARTS_H * 8);
    dbuf_need(s, &s->db.spill, (size_t)s->spill_cap * 16);
  }
  CK(cudaStreamSynchronize(s->stream));
  if (fname) {
    s->fname = strdup(fname);
    struct stat st;
    int bad = 0;
    if (fstat(fd, &st) == 0 && st.st_size > 0) bad = snapshot_load(s, fd); /* a file that loads is the base of checkpoints */
    close(fd);
    if (bad) {
      free(s->fname);
      s->fname = NULL; /* do not overwrite a file we could not read */
      smatrix_close(s);
      return NULL;
    }
  }
  return s;
}

smatrix_t* smatrix_open(const char* fname) {
  return smatrix_b200_open(fname, (int)env_u32("SMATRIX_DEVICE", 0));
}

void smatrix_close(smatrix_t* s) {
  if (!s) return;
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaStreamSynchronize(s->copy_stream));
  if (s->fname && snapshot_save(s) != 0) { /* close() is void (src/smatrix.h:88): be loud instead */
    printf("libsmatrix error: could not write %s; the previous snapshot (if any) was kept\n", s->fname);
    fflush(stdout);
  }
  for (int i = 0; i < s->nsegs; i++)
    if (s->segs[i].owned) cudaFree(s->segs[i].base);
  free(s->segs);
  if (!s->dir_in_arena) cudaFree(s->dir);
  snap_free_keys(s);
  free(s->ck_kept);
  cudaFree(s->d_ctl);
  cudaFreeHost(s->h_ctl);
  cudaFree(s->d_small);
  cudaFreeHost(s->h_small);
  if (s->list_cap) {
    scratch_free(s, s->defer[0]); scratch_free(s, s->defer[1]); scratch_free(s, s->lists.late);
    scratch_free(s, s->lists.grow); scratch_free(s, s->lists.t0rows); scratch_free(s, s->lists.plan);
    scratch_free(s, s->lists.big); scratch_free(s, s->lists.mid);
  }
  scratch_free(s, s->addrs);
  if (s->part_cap)
    for (int a = 0; a < 4; a++) scratch_free(s, s->part[a]);
  if (s->stage_cap)
    for (int b = 0; b < 2; b++)
      for (int a = 0; a < 3; a++) scratch_free(s, s->stage[b][a]);
  const smx_dbuf_t* db = (const smx_dbuf_t*)&s->db;
  for (size_t b = 0; b < sizeof s->db / sizeof *db; b++) cudaFree(db[b].p);
  cudaEventDestroy(s->stage_ready[0]); cudaEventDestroy(s->stage_ready[1]);
  cudaEventDestroy(s->ev0); cudaEventDestroy(s->ev1);
  cudaEventDestroy(s->t_start); cudaEventDestroy(s->t_stop);
  cudaStreamDestroy(s->stream);
  cudaStreamDestroy(s->copy_stream);
  cudaStreamDestroy(s->read_stream[0]); cudaStreamDestroy(s->read_stream[1]);
  free(s->fname);
  leave(s);
  pthread_mutex_destroy(&s->mu);
  free(s);
}

/* ------------------------------------------------------------------------------ controls */
int smatrix_b200_snapshot(smatrix_t* s) {
  if (!s->fname) return -1;
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  const int rc = snapshot_save(s);
  leave(s);
  return rc;
}
int smatrix_b200_device(smatrix_t* s) { return s->device; }
void* smatrix_b200_stream(smatrix_t* s) { return (void*)s->stream; }
void smatrix_b200_sync(smatrix_t* s) {
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  leave(s);
}
void smatrix_b200_timer_start(smatrix_t* s) {
  enter(s);
  CK(cudaEventRecord(s->t_start, s->stream));
  leave(s);
}
float smatrix_b200_timer_stop_ms(smatrix_t* s) {
  float ms = 0.f;
  enter(s);
  CK(cudaEventRecord(s->t_stop, s->stream));
  CK(cudaEventSynchronize(s->t_stop));
  CK(cudaEventElapsedTime(&ms, s->t_start, s->t_stop));
  leave(s);
  return ms;
}
void smatrix_b200_set_kernel_timing(smatrix_t* s, int on) {
  enter(s);
  s->timing = on;
  s->kernel_ns = 0.0;
  memset(s->phase_ns, 0, sizeof s->phase_ns);
  leave(s);
}

void smatrix_b200_set_get_slices(smatrix_t* s, int mode) {
  enter(s);
  if (mode < 0) mode = 0;
  s->get_slices = (mode & 3) > 2 ? 2 : (mode & 3);
  s->get_flags = mode & SMX_GET_FLAGS;
  leave(s);
}

uint64_t smatrix_b200_stat(smatrix_t* s, int which) {
  uint64_t r = 0;
  enter(s);
  switch (which) {
    case SMX_STAT_ROWS:
      read_ctl(s);
      r = s->h_ctl->dir_used;
      break;
    case SMX_STAT_NNZ:
      CK(cudaMemsetAsync(&s->d_ctl->scratch, 0, 8, s->stream));
      smx_launch_count_nnz(s->stream, view_of(s));
      s->n_launches++;
      read_ctl(s);
      r = s->h_ctl->scratch;
      break;
    case SMX_STAT_VALUE_SUM: {
      read_ctl(s);
      const size_t rows = (size_t)s->h_ctl->dir_used;
      uint32_t* big = dbuf_need(s, &s->db.tmp, (rows + 2) * 4); /* list of the rows with a big bucket + its counter */
      uint32_t* d_cnt = big + rows + 1;
      CK(cudaMemsetAsync(&s->d_ctl->scratch, 0, 8, s->stream));
      CK(cudaMemsetAsync(d_cnt, 0, 4, s->stream));
      smx_launch_sum_values(s->stream, view_of(s), big, d_cnt);
      copy_d2h(s, &s->h_small->n_big_sums, d_cnt, 4, s->stream);
      CK(cudaStreamSynchronize(s->stream));
      smx_launch_sum_values_big(s->stream, view_of(s), big, s->h_small->n_big_sums);
      s->n_launches += 2;
      read_ctl(s);
      r = s->h_ctl->scratch;
      break;
    }
    case SMX_STAT_LIVE_BUCKET_BYTES:
      CK(cudaMemsetAsync(&s->d_ctl->scratch, 0, 8, s->stream));
      smx_launch_live_bytes(s->stream, view_of(s));
      s->n_launches++;
      read_ctl(s);
      r = s->h_ctl->scratch;
      break;
    case SMX_STAT_FREE_BYTES:
      read_ctl(s);
      for (uint32_t c = SMX_MIN_SLAB_LOG; c < SMX_CLASSES; c++)
        if (s->h_ctl->free_cnt[c] > 0) r += (uint64_t)s->h_ctl->free_cnt[c] * (8ull << c);
      break;
    case SMX_STAT_RECYCLED: r = s->n_recycled; break;
    case SMX_STAT_BUCKET_BYTES: r = s->bucket_bytes; break;
    case SMX_STAT_SPILLED: r = s->n_spilled; break;
    case SMX_STAT_SLICED_GETS: r = s->n_sliced_gets; break;
    case SMX_STAT_WIDE_CHUNKS: r = s->n_wide_chunks; break;
    case SMX_STAT_NS_ALLOC: r = (uint64_t)s->alloc_ns; break;
    case SMX_STAT_ALLOCS: r = s->n_allocs; break;
    case SMX_STAT_TOPK_BIG: r = s->n_topk_big; break;
    case SMX_STAT_TOPK_PASSES: r = s->n_topk_passes; break;
    case SMX_STAT_REC_BIG: r = s->n_rec_big; break;
    case SMX_STAT_SORT_BIG: r = s->n_sort_big; break;
    case SMX_STAT_DIRTY_ROWS: r = count_dirty(s); break;
    case SMX_STAT_H2D_BYTES: r = s->h2d_bytes; break;
    case SMX_STAT_D2H_BYTES: r = s->d2h_bytes; break;
    case SMX_STAT_DIR_CAP: r = s->dir_cap; break;
    case SMX_STAT_SLAB_BYTES: r = s->slab_bytes; break;
    case SMX_STAT_DEVICE_BYTES: {
      r = s->seg_bytes + s->dir_cap * sizeof(smx_row_t) + (uint64_t)s->list_cap * (6 * 4 + sizeof(smx_plan_t)) +
          (uint64_t)s->stage_cap * 24 + (uint64_t)s->addrs_cap * 8 + (uint64_t)s->part_cap * 16;
      const smx_dbuf_t* db = (const smx_dbuf_t*)&s->db;
      for (size_t b = 0; b < sizeof s->db / sizeof *db; b++) r += db[b].bytes;
      break;
    }
    case SMX_STAT_LAUNCHES: r = s->n_launches; break;
    case SMX_STAT_ROUNDS: r = s->n_rounds; break;
    case SMX_STAT_ROW_GROWS: r = s->n_row_grows; break;
    case SMX_STAT_DIR_GROWS: r = s->n_dir_grows; break;
    case SMX_STAT_KERNEL_NS: r = (uint64_t)s->kernel_ns; break;
    case SMX_STAT_NS_PARTITION: r = (uint64_t)s->phase_ns[PH_PARTITION]; break;
    case SMX_STAT_NS_UPSERT: r = (uint64_t)s->phase_ns[PH_UPSERT]; break;
    case SMX_STAT_NS_GROW_PLAN: r = (uint64_t)s->phase_ns[PH_GROW_PLAN]; break;
    case SMX_STAT_NS_SLAB: r = (uint64_t)s->phase_ns[PH_SLAB]; break;
    case SMX_STAT_NS_MIGRATE: r = (uint64_t)s->phase_ns[PH_MIGRATE]; break;
    case SMX_STAT_NS_DIR: r = (uint64_t)s->phase_ns[PH_DIR]; break;
    default: break;
  }
  leave(s);
  return r;
}

void* smatrix_b200_host_alloc(size_t bytes) {
  void* p = NULL;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return NULL;
  return p;
}
void smatrix_b200_host_free(void* p) {
  if (p) cudaFreeHost(p);
}
void* smatrix_b200_dev_alloc(smatrix_t* s, size_t bytes) {
  enter(s);
  void* p = dmalloc(s, bytes);
  leave(s);
  return p;
}
void smatrix_b200_dev_free(smatrix_t* s, void* p) {
  enter(s);
  CK(cudaStreamSynchronize(s->stream));
  if (p) CK(cudaFree(p));
  leave(s);
}
void smatrix_b200_memcpy(smatrix_t* s, void* dst, const void* src, size_t bytes) {
  enter(s);
  if (!is_device_ptr(src)) { if (is_device_ptr(dst)) s->h2d_bytes += bytes; }
  else if (!is_device_ptr(dst)) s->d2h_bytes += bytes;
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  leave(s);
}

void smatrix_b200_memset0(smatrix_t* s, void* d_dst, size_t bytes) {
  if (!bytes) return;
  enter(s);
  CK(cudaMemsetAsync(d_dst, 0, bytes, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  leave(s);
}

void smatrix_b200_gen_c2_ops(smatrix_t* s, uint64_t seed, uint64_t first, size_t count,
                             uint32_t rows, uint32_t ycols, uint32_t* d_xs, uint32_t* d_ys) {
  enter(s);
  smx_launch_gen_c2_ops(s->stream, seed, first, count, rows, ycols, d_xs, d_ys);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}
void smatrix_b200_gen_c2_queries(smatrix_t* s, uint64_t seed_get, uint64_t seed_build,
                                 uint64_t first, size_t count, uint64_t n_build, uint32_t rows,
                                 uint32_t ycols, uint32_t* d_xs, uint32_t* d_ys) {
  enter(s);
  smx_launch_gen_c2_queries(s->stream, seed_get, seed_build, first, count, n_build, rows, ycols,
                            d_xs, d_ys);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

void smatrix_b200_gen_c3_ops(smatrix_t* s, uint64_t seed, uint64_t first, size_t count,
                             const uint64_t* d_thr, uint32_t items, uint32_t* d_xs, uint32_t* d_ys) {
  enter(s);
  smx_launch_gen_c3_ops(s->stream, seed, first, count, d_thr, items, d_xs, d_ys);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}
void smatrix_b200_gen_c3_queries(smatrix_t* s, uint64_t seed_get, uint64_t seed_build, uint64_t first,
                                 size_t count, uint64_t n_build, const uint64_t* d_thr, uint32_t items,
                                 uint32_t* d_xs, uint32_t* d_ys) {
  enter(s);
  smx_launch_gen_c3_queries(s->stream, seed_get, seed_build, first, count, n_build, d_thr, items, d_xs, d_ys);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}
void smatrix_b200_gen_c4_lens(smatrix_t* s, uint64_t seed, uint64_t first, size_t count,
                              const uint64_t* d_thr, uint32_t kmax, uint32_t* d_lens) {
  enter(s);
  smx_launch_gen_c4_lens(s->stream, seed, first, count, d_thr, kmax, d_lens);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}
void smatrix_b200_gen_c4_ops(smatrix_t* s, uint64_t seed, uint64_t first, size_t count,
                             const uint64_t* d_offs, uint32_t rows, uint32_t* d_xs, uint32_t* d_ys,
                             uint32_t* d_vs) {
  enter(s);
  smx_launch_gen_c4_ops(s->stream, seed, first, count, d_offs, rows, d_xs, d_ys, d_vs);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

double smatrix_b200_probe_random_read(smatrix_t* s, size_t footprint, size_t accesses, int width) {
  if (width != 4 && width != 8 && width != 16 && width != 32) return 0.0;
  enter(s);
  char* buf = (char*)dmalloc(s, footprint);
  CK(cudaMemsetAsync(buf, 1, footprint, s->stream));
  float ms = 0.f;
  smx_launch_probe_read(s->stream, buf, footprint / (size_t)width, accesses / 8, width, s->d_ctl); /* warm-up */
  CK(cudaEventRecord(s->ev0, s->stream));
  smx_launch_probe_read(s->stream, buf, footprint / (size_t)width, accesses, width, s->d_ctl);
  CK(cudaEventRecord(s->ev1, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  CK(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
  CK(cudaFree(buf));
  s->n_launches += 2;
  leave(s);
  return (double)accesses / ((double)ms * 1e-3);
}
double smatrix_b200_probe_random_atomic(smatrix_t* s, size_t footprint, size_t accesses) {
  enter(s);
  uint32_t* buf = (uint32_t*)dmalloc(s, footprint);
  CK(cudaMemsetAsync(buf, 0, footprint, s->stream));
  float ms = 0.f;
  smx_launch_probe_atomic(s->stream, buf, footprint / 4, accesses / 8);
  CK(cudaEventRecord(s->ev0, s->stream));
  smx_launch_probe_atomic(s->stream, buf, footprint / 4, accesses);
  CK(cudaEventRecord(s->ev1, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  CK(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
  CK(cudaFree(buf));
  s->n_launches += 2;
  leave(s);
  return (double)accesses / ((double)ms * 1e-3);
}

/* ------------------------------------------------------------------------------ peer memory */
int smatrix_b200_ipc_export(smatrix_t* s, void* dptr, unsigned char* handle64) {
  cudaIpcMemHandle_t h;
  enter(s);
  cudaError_t e = cudaIpcGetMemHandle(&h, dptr);
  leave(s);
  if (e != cudaSuccess) { (void)cudaGetLastError(); return -1; }
  memcpy(handle64, &h, sizeof h);
  return 0;
}
void* smatrix_b200_ipc_open(smatrix_t* s, const unsigned char* handle64) {
  cudaIpcMemHandle_t h;
  void* p = NULL;
  memcpy(&h, handle64, sizeof h);
  enter(s);
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  leave(s);
  if (e != cudaSuccess) { (void)cudaGetLastError(); return NULL; }
  return p;
}
void smatrix_b200_ipc_close(smatrix_t* s, void* p) {
  enter(s);
  if (p) (void)cudaIpcCloseMemHandle(p);
  leave(s);
}

/* ------------------------------------------------------------------------------ router (K8) */
void smatrix_b200_partition_count(smatrix_t* s, const uint32_t* d_xs, size_t n, uint32_t world,
                                  uint64_t* h_counts) {
  if (world == 0 || world > 64) smx_die("partition: world size must be 1..64");
  if (n > 0xFFFFFFFFull) smx_die("partition: batch too large");
  enter(s);
  unsigned long long* d_counts = dbuf_need(s, &s->db.tmp64, (2 * 64 + 5 * 64) * 8);
  unsigned long long h[64];
  CK(cudaMemsetAsync(d_counts, 0, 64 * 8, s->stream));
  smx_launch_partition_count(s->stream, d_xs, NULL, (uint32_t)n, world, 0, SMX_PART_OWNER, 0, d_counts);
  copy_d2h(s, h, d_counts, world * 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  for (uint32_t r = 0; r < world; r++) h_counts[r] = h[r];
  s->n_launches++;
  leave(s);
}

/* K8 fused with the exchange: bucket by owner and write every owner's run straight to
 * h_dst[0..4][world] = {x, y, v, src (0 = none) output base addresses, routed-position bases}
 * (peer mappings or local memory), see k_partition_scatter. */
void smatrix_b200_route_p2p(smatrix_t* s, const uint32_t* d_xs, const uint32_t* d_ys,
                            const uint32_t* d_vals, size_t n, uint32_t world, const uint64_t* h_dst,
                            uint32_t src_bias, uint32_t* d_out_pos) {
  if (world == 0 || world > 64) smx_die("route: world size must be 1..64");
  if (n == 0) return;
  if (n > 0xFFFFFFFFull) smx_die("route: batch too large");
  enter(s);
  unsigned long long* d_cursors = (unsigned long long*)dbuf_need(s, &s->db.tmp64, (2 * 64 + 5 * 64) * 8) + 64;
  unsigned long long* d_tab = d_cursors + 64;
  CK(cudaMemsetAsync(d_cursors, 0, 64 * 8, s->stream));
  copy_h2d(s, d_tab, h_dst, 5 * (size_t)world * 8, s->stream);
  smx_launch_partition_scatter(s->stream, d_xs, d_ys, d_vals, (uint32_t)n, world, 0, SMX_PART_OWNER, 0,
                               d_cursors, NULL, NULL, NULL, NULL, NULL, d_out_pos, d_tab, src_bias);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

uint32_t smatrix_b200_owner(uint32_t x, uint32_t world) { return smx_owner_hash(x) % world; }

void smatrix_b200_gather(smatrix_t* s, uint32_t* d_out, const uint32_t* d_vals, const uint32_t* d_pos,
                         size_t n) {
  if (n == 0) return;
  if (n > 0xFFFFFFFFull) smx_die("gather: batch too large");
  enter(s);
  smx_launch_gather(s->stream, d_out, d_vals, d_pos, (uint32_t)n);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* ---- device-level getrow pieces for the multi-GPU router (include/smatrix_b200.h) ---- */
void smatrix_b200_row_counts_batch(smatrix_t* s, const uint32_t* d_xs, size_t n, uint32_t* d_counts) {
  if (n == 0) return;
  if (n >= 0xFFFFFFFFull) smx_die("row_counts: batch too large");
  enter(s);
  smx_launch_row_counts(s->stream, view_of(s), d_xs, (uint32_t)n, d_counts, NULL, NULL, NULL);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

uint64_t smatrix_b200_scan_counts(smatrix_t* s, const uint32_t* d_counts, size_t n, uint64_t* d_offsets) {
  if (n >= 0xFFFFFFFFull) smx_die("scan_counts: batch too large");
  enter(s);
  smx_launch_scan(s->stream, d_counts, (uint32_t)n, 0, d_offsets,
                  dbuf_need(s, &s->db.tmp64, ((size_t)smx_scan_scratch_items((uint32_t)n) + 2) * 8));
  s->n_launches += 3;
  copy_d2h(s, &s->h_small->row_total, d_offsets + n, 8, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  const uint64_t total = s->h_small->row_total;
  leave(s);
  return total;
}

void smatrix_b200_getrow_fill_at(smatrix_t* s, const uint32_t* d_xs, size_t n, const uint64_t* d_offsets,
                                 uint32_t* d_pairs) {
  if (n == 0) return;
  if (n >= 0xFFFFFFFFull) smx_die("getrow_fill_at: batch too large");
  enter(s);
  const uint32_t nn = (uint32_t)n;
  const smx_rowplan_t p = rowplan(s, nn);
  /* resolve the rows (directory index, bucket size) and find the ones the whole grid compacts */
  smx_launch_row_counts(s->stream, view_of(s), d_xs, nn, p.counts, p.info, p.big, p.n_big);
  copy_d2h(s, &s->h_small->n_big_rows, p.n_big, 4, s->stream);
  CK(cudaStreamSynchronize(s->stream));
  timed_begin(s);
  smx_launch_getrow_fill(s->stream, view_of(s), p.info, nn, d_offsets, 0, d_pairs, p.big, s->h_small->n_big_rows, p.cursors);
  timed_end(s);
  s->n_launches += 2;
  CK(cudaStreamSynchronize(s->stream));
  timed_collect(s);
  CK(cudaGetLastError());
  leave(s);
}

void smatrix_b200_route_offsets(smatrix_t* s, const uint64_t* d_offsets, const uint32_t* d_pos, size_t n,
                                uint32_t world, const uint64_t* h_tab) {
  if (world == 0 || world > 64) smx_die("route: world size must be 1..64");
  if (n == 0) return;
  if (n >= 0xFFFFFFFFull) smx_die("route_offsets: batch too large");
  enter(s);
  unsigned long long* d_tab = (unsigned long long*)dbuf_need(s, &s->db.tmp64, (2 * 64 + 5 * 64) * 8) + 128;
  copy_h2d(s, d_tab, h_tab, 2 * (size_t)world * 8, s->stream);
  smx_launch_route_offsets(s->stream, d_offsets, d_pos, (uint32_t)n, world, d_tab);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

/* device-level pieces of the CF read side for the multi-GPU router (all arrays on the device) */
void smatrix_b200_pair_cols(smatrix_t* s, const uint32_t* d_pairs, uint64_t total, uint32_t* d_cols) {
  if (!total) return;
  enter(s);
  smx_launch_pair_cols(s->stream, d_pairs, total, d_cols);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}
void smatrix_b200_cf_scores_totals(smatrix_t* s, size_t n, const uint64_t* d_offsets, const uint32_t* d_pairs,
                                   const uint32_t* d_a_tot, const uint32_t* d_b_tot, uint32_t* d_ids, double* d_scores) {
  if (!n) return;
  enter(s);
  smx_launch_cf_scores_totals(s->stream, (uint32_t)n, d_offsets, d_pairs, d_a_tot, d_b_tot, d_ids, d_scores);
  s->n_launches++;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
  leave(s);
}

int smatrix_b200_is_device_ptr(smatrix_t* s, const void* p) {
  enter(s);
  const int r = is_device_ptr(p);
  leave(s);
  return r;
}

int smatrix_b200_enable_peer(smatrix_t* s, int peer_device) {
  if (peer_device == s->device) return 0;
  enter(s);
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  (void)cudaGetLastError(); /* "already enabled" is fine */
  leave(s);
  return (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) ? 0 : -1;
}

/* asynchronous copies on one of the side streams (lane 0..2), for callers that overlap uploads and
 * downloads with work on the main stream; smatrix_b200_lane_sync waits for a lane */
static cudaStream_t lane_stream(smatrix_t* s, int lane) {
  return lane == 0 ? s->copy_stream : s->read_stream[(lane - 1) & 1];
}
void smatrix_b200_memcpy_async(smatrix_t* s, void* dst, const void* src, size_t bytes, int lane) {
  if (!bytes) return;
  enter(s);
  if (!is_device_ptr(src)) s->h2d_bytes += bytes;
  else if (!is_device_ptr(dst)) s->d2h_bytes += bytes;
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, lane_stream(s, lane)));
  leave(s);
}
void smatrix_b200_lane_sync(smatrix_t* s, int lane) {
  enter(s);
  CK(cudaStreamSynchronize(lane_stream(s, lane)));
  CK(cudaGetLastError());
  leave(s);
}
