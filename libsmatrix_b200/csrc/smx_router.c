/*
 * smx_router.c — the multi-GPU router of the B200 libsmatrix hot path, in C (include/smatrix_shard.h).
 *
 * Rows are hash-partitioned over the GPUs of one box, one RANK per GPU; every rank owns a complete
 * private table (smatrix_t) for its rows.  This file owns only the plumbing around the C-ABI of
 * smx_host.c — it makes no CUDA call of its own:
 *
 *   rendezvous   a POSIX shared-memory segment (name chosen by the caller) holds, per rank, the
 *                address + CUDA IPC handle of its INBOX, a world x world count matrix, a few scalar
 *                slots and a sense-reversing barrier.  Ranks may be threads of one process (peer
 *                pointers are used directly) or separate processes (IPC mappings).
 *   a write      k_partition_count (ops per owner) -> counts into the segment -> barrier ->
 *                ONE k_partition_scatter launch stores every owner's run straight into that owner's
 *                inbox over NVLink / NVSwitch -> barrier -> every rank applies its inbox with the
 *                ordinary single-GPU path.  No send buffer, no all-to-all, no NCCL.
 *   a read       the same route for the queries (+ each query's routed position), then every owner
 *                runs its look-up kernel once per asking rank with the OUTPUT pointing into that
 *                rank's answer buffer (peer stores again), staggered so that at any moment the ranks
 *                answer different requesters (a shift permutation, never many-to-one) -> barrier ->
 *                the asking rank gathers its answers into input order.
 *   getrow       counts travel like read answers; the asking rank scans them into CSR offsets, sends
 *                every row's offset to its owner (k_route_offsets), and the owners' compaction
 *                kernels write the pairs into the asking rank's row buffer.
 *
 * Replaces nothing in the reference (single node, shared memory); the semantics each call must
 * reproduce are those of src/smatrix.c:174-256 applied to one matrix (SURVEY.md 8e).
 */
#define _GNU_SOURCE
#include <errno.h>
#include <fcntl.h>
#include <sched.h>
#include <stdarg.h>
#include <stdatomic.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

#include "../../include/smatrix.h"
#include "../../include/smatrix_b200.h"
#include "../../include/smatrix_batch.h"
#include "../../include/smatrix_shard.h"

#define RT_MAXW 64
#define RT_MAGIC 0x52584d53u /* "SMXR" */
#define RT_PIECE_DEFAULT (1u << 24) /* host arrays are staged in pieces of this many ops */

typedef struct {
  int32_t pid, device;
  uint64_t inbox, rowbuf;         /* device addresses in the owner's address space */
  uint64_t cap, pairs_cap;
  unsigned char h_inbox[64], h_rowbuf[64];
  int32_t ok;                     /* set-up outcome of this rank (agreed on collectively) */
} rt_blob_t;

typedef struct {
  _Atomic uint32_t magic;
  uint32_t world;
  _Atomic uint32_t arrived, generation, failed, detached;
  rt_blob_t blob[RT_MAXW];
  uint64_t cnt[2][RT_MAXW][RT_MAXW]; /* [parity][sender][owner] */
  uint64_t val[2][RT_MAXW][4];       /* [parity][rank][slot]: tiny all-gathers */
} rt_shm_t;

struct smatrix_shard_s {
  int rank, world, device;
  char name[160];
  rt_shm_t* shm;
  smatrix_t* local;
  double timeout_s;
  unsigned cnt_seq, val_seq;      /* parities of the two exchange areas */
  /* symmetric buffers (one allocation each, mapped by every peer) */
  uint64_t cap, pairs_cap;
  char* inbox;
  char* rowbuf;
  char* peer_inbox[RT_MAXW];
  char* peer_rowbuf[RT_MAXW];
  int same_proc[RT_MAXW];
  /* staging of host arrays: two generations x (x, y, v) + answers */
  uint32_t* stage[2][4];
  size_t stage_cap;
  uint32_t piece;
  uint32_t taper_min; /* 0 = off; else the last staged piece is cut into 1/2, 1/4, 1/4 if a quarter has this many ops */
  uint64_t stat[8]; /* SMX_SHARD_STAT_* */
  char* fname;        /* file mode: the .smx file every rank loaded from and writes back to */
  int ck_base;        /* the file matched the table at some point (a load, a snapshot or a checkpoint) */
};

/* inbox layout for capacity `cap` ops (cap is a multiple of 256): shared arrays first, then the
 * arrays only the owner touches */
#define OFF_X(cap) ((size_t)0)
#define OFF_Y(cap) ((size_t)(cap) * 4)
#define OFF_V(cap) ((size_t)(cap) * 8)
#define OFF_O(cap) ((size_t)(cap) * 12)
#define OFF_ANS(cap) ((size_t)(cap) * 16)
#define OFF_Q64(cap) ((size_t)(cap) * 20)
#define OFF_POS(cap) ((size_t)(cap) * 28)   /* local: routed position of my queries */
#define OFF_CNT(cap) ((size_t)(cap) * 32)   /* local: gathered counts */
#define OFF_OFS(cap) ((size_t)(cap) * 36)   /* local: CSR offsets, cap + 1 x u64 */
#define INBOX_BYTES(cap) ((size_t)(cap) * 44 + 64)

/* ------------------------------------------------------------------------------ errors, waiting */
static void rt_die(smatrix_shard_t* sh, const char* fmt, ...) { /* reference src/smatrix.c:891-894 */
  va_list ap;
  if (sh && sh->shm) atomic_store(&sh->shm->failed, 1u); /* peers stop waiting */
  printf("libsmatrix error: ");
  va_start(ap, fmt);
  vprintf(fmt, ap);
  va_end(ap);
  printf("\n");
  fflush(stdout);
  abort();
}

static uint32_t rt_env(const char* name, uint32_t dflt) {
  const char* v = getenv(name);
  return (v && *v) ? (uint32_t)strtoul(v, NULL, 0) : dflt;
}

static double rt_now(void) {
  struct timespec t;
  clock_gettime(CLOCK_MONOTONIC, &t);
  return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

/* sense-reversing barrier in the shared segment; a rank that dies (rt_die) or never arrives makes
 * the others abort instead of hanging */
static void rt_barrier(smatrix_shard_t* sh) {
  rt_shm_t* m = sh->shm;
  if (sh->world == 1) return;
  const uint32_t gen = atomic_load(&m->generation);
  if (atomic_fetch_add(&m->arrived, 1u) + 1u == (uint32_t)sh->world) {
    atomic_store(&m->arrived, 0u);
    atomic_fetch_add(&m->generation, 1u);
    return;
  }
  double t0 = 0.0;
  for (unsigned spin = 0; atomic_load(&m->generation) == gen; spin++) {
    if (atomic_load(&m->failed)) rt_die(sh, "a peer rank of the sharded matrix failed");
    if ((spin & 1023u) == 1023u) {
      sched_yield();
      const double now = rt_now();
      if (t0 == 0.0) t0 = now;
      else if (now - t0 > sh->timeout_s) rt_die(sh, "rank %d: peers did not arrive within %.0f s", sh->rank, sh->timeout_s);
    } else {
      __builtin_ia32_pause();
    }
  }
}

/* all-gather of up to 4 scalars per rank: out[r][slot] */
static void rt_allgather(smatrix_shard_t* sh, const uint64_t mine[4], uint64_t out[RT_MAXW][4]) {
  const unsigned p = sh->val_seq++ & 1u;
  memcpy(sh->shm->val[p][sh->rank], mine, 4 * sizeof(uint64_t));
  rt_barrier(sh);
  for (int r = 0; r < sh->world; r++) memcpy(out[r], sh->shm->val[p][r], 4 * sizeof(uint64_t));
}

void smatrix_b200_shard_barrier(smatrix_shard_t* sh) { rt_barrier(sh); }
uint64_t smatrix_b200_shard_sum(smatrix_shard_t* sh, uint64_t v) {
  uint64_t mine[4] = {v, 0, 0, 0}, all[RT_MAXW][4], acc = 0;
  rt_allgather(sh, mine, all);
  for (int r = 0; r < sh->world; r++) acc += all[r][0];
  return acc;
}
uint64_t smatrix_b200_shard_max(smatrix_shard_t* sh, uint64_t v) {
  uint64_t mine[4] = {v, 0, 0, 0}, all[RT_MAXW][4], acc = 0;
  rt_allgather(sh, mine, all);
  for (int r = 0; r < sh->world; r++) acc = all[r][0] > acc ? all[r][0] : acc;
  return acc;
}

/* ------------------------------------------------------------------------------ symmetric buffers */
static void rt_unmap(smatrix_shard_t* sh, char** peers) {
  for (int r = 0; r < sh->world; r++) {
    if (r != sh->rank && peers[r] && !sh->same_proc[r]) smatrix_b200_ipc_close(sh->local, peers[r]);
    peers[r] = NULL;
  }
}

/* Collective: (re)allocate the inbox (which = 0, `units` ops) or the row buffer (which = 1, `units`
 * pairs) on every rank and map the peers'.  Returns 0, or -1 on EVERY rank if any rank failed. */
static int rt_sym_alloc(smatrix_shard_t* sh, int which, uint64_t units) {
  rt_shm_t* m = sh->shm;
  rt_blob_t* me = &m->blob[sh->rank];
  char** mine = which ? &sh->rowbuf : &sh->inbox;
  char** peers = which ? sh->peer_rowbuf : sh->peer_inbox;
  rt_unmap(sh, peers);
  rt_barrier(sh); /* nobody frees memory a peer still maps */
  if (*mine) smatrix_b200_dev_free(sh->local, *mine);
  units = (units + 255u) & ~(uint64_t)255u;
  const size_t bytes = which ? (size_t)units * 8 + 64 : INBOX_BYTES(units);
  *mine = (char*)smatrix_b200_dev_alloc(sh->local, bytes);
  int ok = *mine != NULL;
  unsigned char* hb = which ? me->h_rowbuf : me->h_inbox;
  memset(hb, 0, 64);
  if (ok && sh->world > 1 && smatrix_b200_ipc_export(sh->local, *mine, hb) != 0) {
    /* no IPC (e.g. a memory pool without export): still fine if every peer is in this process */
    for (int r = 0; r < sh->world; r++)
      if (r != sh->rank && m->blob[r].pid != me->pid) ok = 0;
  }
  if (which) { me->rowbuf = (uint64_t)(uintptr_t)*mine; me->pairs_cap = units; sh->pairs_cap = units; }
  else { me->inbox = (uint64_t)(uintptr_t)*mine; me->cap = units; sh->cap = units; }
  me->ok = ok;
  rt_barrier(sh);
  for (int r = 0; r < sh->world && ok; r++) {
    const rt_blob_t* b = &m->blob[r];
    if (!b->ok) { ok = 0; break; }
    if (r == sh->rank) { peers[r] = *mine; continue; }
    if (sh->same_proc[r]) {
      peers[r] = (char*)(uintptr_t)(which ? b->rowbuf : b->inbox);
    } else {
      peers[r] = (char*)smatrix_b200_ipc_open(sh->local, which ? b->h_rowbuf : b->h_inbox);
      if (!peers[r]) ok = 0;
    }
  }
  /* agree on the outcome: one failed mapping anywhere and everybody backs out together */
  uint64_t flag[4] = {(uint64_t)ok, 0, 0, 0}, all[RT_MAXW][4];
  rt_allgather(sh, flag, all);
  for (int r = 0; r < sh->world; r++) ok = ok && all[r][0];
  if (!ok) {
    rt_unmap(sh, peers);
    rt_barrier(sh);
    return -1;
  }
  /* first stores through a freshly opened mapping are slow (it is completed lazily): touch every
   * peer array once now, so that the first routed batch runs at NVLink speed */
  for (int r = 0; r < sh->world; r++)
    if (r != sh->rank) smatrix_b200_memcpy(sh->local, peers[r], *mine, bytes);
  rt_barrier(sh);
  return 0;
}

static void rt_need_inbox(smatrix_shard_t* sh, uint64_t ops) { /* collective, same `ops` on every rank */
  if (ops <= sh->cap) return;
  uint64_t want = ops + ops / 4 + 65536;
  if (rt_sym_alloc(sh, 0, want) != 0) rt_die(sh, "cannot map the peers' inboxes (%llu ops)", (unsigned long long)want);
}
static void rt_need_rowbuf(smatrix_shard_t* sh, uint64_t pairs) {
  if (pairs <= sh->pairs_cap) return;
  uint64_t want = pairs + pairs / 8 + 4096;
  if (rt_sym_alloc(sh, 1, want) != 0) rt_die(sh, "cannot map the peers' row buffers (%llu pairs)", (unsigned long long)want);
}

/* ------------------------------------------------------------------------------ open / close */

smatrix_shard_t* smatrix_b200_shard_open(const char* name, int rank, int world, int device) {
  return smatrix_b200_shard_open_arena(name, rank, world, device, (size_t)rt_env("SMATRIX_ARENA_GIB", 0) << 30);
}

smatrix_shard_t* smatrix_b200_shard_open_arena(const char* name, int rank, int world, int device, size_t arena_bytes) {
  if (!name || world < 1 || world > RT_MAXW || rank < 0 || rank >= world) {
    fprintf(stderr, "libsmatrix: shard_open: bad arguments\n");
    return NULL;
  }
  smatrix_shard_t* sh = (smatrix_shard_t*)calloc(1, sizeof *sh);
  if (!sh) return NULL;
  sh->rank = rank; sh->world = world; sh->device = device;
  sh->timeout_s = (double)rt_env("SMATRIX_SHARD_TIMEOUT", 300);
  sh->piece = rt_env("SMATRIX_SHARD_PIECE", RT_PIECE_DEFAULT);
  if (sh->piece < 1024) sh->piece = 1024;
  sh->taper_min = rt_env("SMATRIX_SHARD_TAPER_MIN", 0); /* off: measured at N = 2, 11.8 - 12.0 vs 11.5 ms per step */
  snprintf(sh->name, sizeof sh->name, "/%s", name[0] == '/' ? name + 1 : name);
  /* rank 0 creates the segment; the others wait for it to appear and to be initialised */
  int fd = -1;
  const double t0 = rt_now();
  if (rank == 0) {
    shm_unlink(sh->name);
    fd = shm_open(sh->name, O_CREAT | O_EXCL | O_RDWR, 0600);
    if (fd == -1 || ftruncate(fd, (off_t)sizeof(rt_shm_t)) == -1) {
      perror("libsmatrix: cannot create the rendezvous segment");
      if (fd != -1) close(fd);
      free(sh);
      return NULL;
    }
  } else {
    while ((fd = shm_open(sh->name, O_RDWR, 0600)) == -1) {
      if (rt_now() - t0 > sh->timeout_s) { fprintf(stderr, "libsmatrix: rank 0 never created %s\n", sh->name); free(sh); return NULL; }
      usleep(1000);
    }
    struct stat st;
    while (fstat(fd, &st) == 0 && (size_t)st.st_size < sizeof(rt_shm_t)) {
      if (rt_now() - t0 > sh->timeout_s) { close(fd); free(sh); return NULL; }
      usleep(1000);
    }
  }
  sh->shm = (rt_shm_t*)mmap(NULL, sizeof(rt_shm_t), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (sh->shm == MAP_FAILED) { perror("libsmatrix: mmap"); free(sh); return NULL; }
  if (rank == 0) {
    sh->shm->world = (uint32_t)world;
    atomic_store(&sh->shm->magic, RT_MAGIC); /* the fresh segment is zero-filled */
  } else {
    while (atomic_load(&sh->shm->magic) != RT_MAGIC) {
      if (rt_now() - t0 > sh->timeout_s) { munmap(sh->shm, sizeof(rt_shm_t)); free(sh); return NULL; }
      usleep(200);
    }
    if (sh->shm->world != (uint32_t)world) { fprintf(stderr, "libsmatrix: world size mismatch on %s\n", sh->name); munmap(sh->shm, sizeof(rt_shm_t)); free(sh); return NULL; }
  }
  sh->local = smatrix_b200_open_arena(NULL, device, arena_bytes);
  rt_blob_t* me = &sh->shm->blob[rank];
  me->pid = (int32_t)getpid();
  me->device = device;
  me->ok = sh->local != NULL;
  rt_barrier(sh);
  int ok = 1;
  for (int r = 0; r < world; r++) {
    ok = ok && sh->shm->blob[r].ok;
    sh->same_proc[r] = sh->shm->blob[r].pid == me->pid;
  }
  if (ok)
    for (int r = 0; r < world; r++)
      if (r != rank && sh->same_proc[r] && smatrix_b200_enable_peer(sh->local, sh->shm->blob[r].device) != 0) me->ok = 0;
  if (ok && rt_sym_alloc(sh, 0, rt_env("SMATRIX_SHARD_INBOX", 1u << 16)) != 0) ok = 0;
  if (ok && rt_sym_alloc(sh, 1, 1u << 12) != 0) ok = 0;
  uint64_t flag[4] = {(uint64_t)(ok && me->ok), 0, 0, 0}, all[RT_MAXW][4];
  rt_allgather(sh, flag, all);
  for (int r = 0; r < world; r++) ok = ok && all[r][0];
  if (!ok) { /* every rank takes this branch together */
    fprintf(stderr, "libsmatrix: rank %d: the sharded matrix could not be set up (no CUDA device or no peer access)\n", rank);
    if (sh->local) smatrix_close(sh->local);
    rt_barrier(sh);
    if (rank == 0) shm_unlink(sh->name);
    munmap(sh->shm, sizeof(rt_shm_t));
    free(sh);
    return NULL;
  }
  return sh;
}

static int rt_snapshot(smatrix_shard_t* sh);
void smatrix_b200_shard_close(smatrix_shard_t* sh) {
  if (!sh) return;
  if (sh->fname && rt_snapshot(sh) != 0 && sh->rank == 0) { /* close() is void: be loud instead */
    printf("libsmatrix error: could not write %s; the previous snapshot (if any) was kept\n", sh->fname);
    fflush(stdout);
  }
  free(sh->fname);
  rt_barrier(sh);
  rt_unmap(sh, sh->peer_inbox);
  rt_unmap(sh, sh->peer_rowbuf);
  rt_barrier(sh); /* nobody frees memory a peer still maps */
  if (sh->inbox) smatrix_b200_dev_free(sh->local, sh->inbox);
  if (sh->rowbuf) smatrix_b200_dev_free(sh->local, sh->rowbuf);
  for (int g = 0; g < 2; g++)
    for (int a = 0; a < 4; a++)
      if (sh->stage[g][a]) smatrix_b200_dev_free(sh->local, sh->stage[g][a]);
  smatrix_close(sh->local);
  rt_barrier(sh);
  if (sh->rank == 0) shm_unlink(sh->name);
  munmap(sh->shm, sizeof(rt_shm_t));
  free(sh);
}

uint64_t smatrix_b200_shard_stat(smatrix_shard_t* sh, int which) {
  return (which >= 0 && which < 8) ? sh->stat[which] : 0;
}
void smatrix_b200_shard_stat_reset(smatrix_shard_t* sh) { memset(sh->stat, 0, 4 * sizeof sh->stat[0]); /* the accounting, not the high-water marks */ }
smatrix_t* smatrix_b200_shard_local(smatrix_shard_t* sh) { return sh->local; }
int smatrix_b200_shard_rank(smatrix_shard_t* sh) { return sh->rank; }
int smatrix_b200_shard_world(smatrix_shard_t* sh) { return sh->world; }

static void rt_need_stage(smatrix_shard_t* sh, size_t ops);
void smatrix_b200_shard_reserve(smatrix_shard_t* sh, size_t max_ops, size_t max_pairs) {
  const uint64_t ops = smatrix_b200_shard_max(sh, max_ops), pairs = smatrix_b200_shard_max(sh, max_pairs);
  rt_need_inbox(sh, ops);
  if (pairs) rt_need_rowbuf(sh, pairs);
  rt_need_stage(sh, (size_t)(ops < sh->piece ? ops : sh->piece) + 1); /* staging of host-array pieces */
}

/* ------------------------------------------------------------------------------ the route */
typedef struct {
  uint64_t cnt[RT_MAXW][RT_MAXW]; /* [sender][owner] */
  uint64_t n_of[RT_MAXW];         /* ops in sender s's slice */
  uint64_t recv_start[RT_MAXW];   /* where sender s's run starts in my inbox */
  uint64_t send_base[RT_MAXW];    /* where owner o's run starts in my routed order */
  uint64_t n_recv, bias;
} rt_route_t;

/* where owner `o`'s run of sender `s` starts in s's routed order / in o's inbox */
static uint64_t rt_send_base(const rt_route_t* R, int s, int o) {
  uint64_t at = 0;
  for (int k = 0; k < o; k++) at += R->cnt[s][k];
  return at;
}
static uint64_t rt_in_base(const rt_route_t* R, int s, int o) {
  uint64_t at = 0;
  for (int k = 0; k < s; k++) at += R->cnt[k][o];
  return at;
}

/* Collective.  Device arrays d_xs / d_ys / d_vs (n ops, this rank's slice) -> every owner's inbox.
 * want_ord: the global input-order index travels along (inbox array O); want_pos: the routed
 * position of each of my ops is left in my POS array (reads un-permute with it). */
static void rt_route(smatrix_shard_t* sh, const uint32_t* d_xs, const uint32_t* d_ys, const uint32_t* d_vs,
                     size_t n, int want_ord, int want_pos, rt_route_t* R) {
  const int W = sh->world, me = sh->rank;
  const double t_begin = rt_now();
  uint64_t mine[RT_MAXW];
  memset(mine, 0, sizeof mine);
  if (n) smatrix_b200_partition_count(sh->local, d_xs, n, (uint32_t)W, mine);
  const unsigned p = sh->cnt_seq++ & 1u;
  memcpy(sh->shm->cnt[p][me], mine, sizeof(uint64_t) * (size_t)W);
  rt_barrier(sh);
  uint64_t need = 0, total = 0;
  for (int s = 0; s < W; s++) {
    memcpy(R->cnt[s], sh->shm->cnt[p][s], sizeof(uint64_t) * (size_t)W);
    R->n_of[s] = 0;
    for (int o = 0; o < W; o++) R->n_of[s] += R->cnt[s][o];
    if (R->n_of[s] > need) need = R->n_of[s];
    total += R->n_of[s];
  }
  for (int o = 0; o < W; o++) {
    uint64_t in = 0;
    for (int s = 0; s < W; s++) in += R->cnt[s][o];
    if (in > need) need = in;
  }
  if (want_ord && total >= 0xFFFFFFFFull) rt_die(sh, "ordered collective batches are limited to 2^32 - 2 ops");
  if (need > sh->stat[SMX_SHARD_STAT_MAX_INBOX_OPS]) sh->stat[SMX_SHARD_STAT_MAX_INBOX_OPS] = need;
  rt_need_inbox(sh, need); /* every rank sees the same matrix: the same decision everywhere */
  R->n_recv = 0;
  R->bias = 0;
  for (int s = 0; s < W; s++) {
    R->recv_start[s] = R->n_recv;
    R->n_recv += R->cnt[s][me];
    if (s < me) R->bias += R->n_of[s];
  }
  uint64_t tab[5 * RT_MAXW];
  const uint64_t cap = sh->cap;
  for (int o = 0; o < W; o++) {
    const uint64_t at = 4 * rt_in_base(R, me, o);
    char* base = sh->peer_inbox[o];
    R->send_base[o] = rt_send_base(R, me, o);
    tab[o] = (uint64_t)(uintptr_t)(base + OFF_X(cap) + at);
    tab[W + o] = d_ys ? (uint64_t)(uintptr_t)(base + OFF_Y(cap) + at) : 0;
    tab[2 * W + o] = d_vs ? (uint64_t)(uintptr_t)(base + OFF_V(cap) + at) : 0;
    tab[3 * W + o] = want_ord ? (uint64_t)(uintptr_t)(base + OFF_O(cap) + at) : 0;
    tab[4 * W + o] = R->send_base[o];
  }
  if (n)
    smatrix_b200_route_p2p(sh->local, d_xs, d_ys, d_vs, n, (uint32_t)W, tab, (uint32_t)R->bias,
                           want_pos ? (uint32_t*)(sh->inbox + OFF_POS(cap)) : NULL);
  rt_barrier(sh); /* every rank's runs have landed (route_p2p returns after its kernel completed) */
  sh->stat[SMX_SHARD_STAT_ROUTE_NS] += (uint64_t)((rt_now() - t_begin) * 1e9);
  sh->stat[SMX_SHARD_STAT_ROUTES]++;
  sh->stat[SMX_SHARD_STAT_REMOTE_BYTES] +=
      (uint64_t)(n - R->cnt[me][me]) * 4u * (1u + (d_ys != NULL) + (d_vs != NULL) + (want_ord != 0));
}

/* Host slices go through the device in pieces: `base` equal pieces; optionally ($SMATRIX_SHARD_TAPER_MIN) the
 * last of them is cut again into 1/2, 1/4, 1/4 so that less of the final route + update is exposed — measured:
 * the extra pieces cost more than the shorter tail saves, so it is off by default.  Boundary k of rank-local
 * slice n, the same piece count on every rank: */
static uint64_t rt_pieces(uint64_t base, int taper) { return taper ? base + 2 : base; }
static size_t rt_piece_lo(uint64_t k, uint64_t base, int taper, size_t n) {
  uint64_t q; /* boundary in quarters of a base piece */
  if (!taper) q = 4 * k;
  else if (k < base) q = 4 * k;
  else if (k == base) q = 4 * base - 2;
  else if (k == base + 1) q = 4 * base - 1;
  else q = 4 * base;
  return (size_t)((unsigned __int128)q * n / (4 * base));
}

/* ------------------------------------------------------------------------------ staging of host arrays */
static void rt_need_stage(smatrix_shard_t* sh, size_t ops) {
  if (ops <= sh->stage_cap) return;
  for (int g = 0; g < 2; g++)
    for (int a = 0; a < 4; a++) {
      if (sh->stage[g][a]) smatrix_b200_dev_free(sh->local, sh->stage[g][a]);
      sh->stage[g][a] = (uint32_t*)smatrix_b200_dev_alloc(sh->local, ops * 4 + 64);
    }
  sh->stage_cap = ops;
}

/* is p a device pointer?  (host callers hand us malloc'ed / pinned arrays) */
static int rt_is_dev(smatrix_shard_t* sh, const void* p) { return p ? smatrix_b200_is_device_ptr(sh->local, p) : 0; }

/* ------------------------------------------------------------------------------ writes */
static void rt_apply(smatrix_shard_t* sh, int op, int ordered, int has_vals, const rt_route_t* R) {
  if (!R->n_recv) return;
  const uint64_t cap = sh->cap;
  const double t_begin = rt_now();
  const uint32_t* x = (const uint32_t*)(sh->inbox + OFF_X(cap));
  const uint32_t* y = (const uint32_t*)(sh->inbox + OFF_Y(cap));
  const uint32_t* v = has_vals ? (const uint32_t*)(sh->inbox + OFF_V(cap)) : NULL;
  if (ordered) {
    smatrix_b200_apply_ordered(sh->local, op, x, y, v, (const uint32_t*)(sh->inbox + OFF_O(cap)), (size_t)R->n_recv);
  } else if (op == 0) {
    smatrix_incr_batch(sh->local, x, y, v, (size_t)R->n_recv);
  } else {
    smatrix_decr_batch(sh->local, x, y, v, (size_t)R->n_recv);
  }
  sh->stat[SMX_SHARD_STAT_APPLY_NS] += (uint64_t)((rt_now() - t_begin) * 1e9);
}

static void rt_write(smatrix_shard_t* sh, int op, const uint32_t* xs, const uint32_t* ys, const uint32_t* vals,
                     size_t n, int ordered) {
  if (n >= 0xFFFFFFFFull) rt_die(sh, "sharded batch too large for one call");
  const int dev = n ? rt_is_dev(sh, xs) : 1;
  if (n && (rt_is_dev(sh, ys) != dev || (vals && rt_is_dev(sh, vals) != dev)))
    rt_die(sh, "batch arrays must be all host or all device pointers");
  /* the ranks agree on: the largest slice, whether values travel, whether anybody needs staging */
  uint64_t mine[4] = {n, n ? (vals != NULL) + 1u : 0u, (uint64_t)!dev, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t nmax = 0;
  int has_vals = -1, any_host = 0;
  for (int r = 0; r < sh->world; r++) {
    if (all[r][0] > nmax) nmax = all[r][0];
    if (all[r][1]) {
      const int hv = (int)all[r][1] - 1;
      if (has_vals >= 0 && has_vals != hv) rt_die(sh, "every rank must pass vals, or none (NULL = all ones)");
      has_vals = hv;
    }
    any_host |= (int)all[r][2];
  }
  if (nmax == 0) return;
  if (has_vals < 0) has_vals = 0;
  rt_route_t R;
  if (!any_host) { /* device slices: one route, one update */
    rt_route(sh, xs, ys, has_vals ? vals : NULL, n, ordered, 0, &R);
    rt_apply(sh, op, ordered, has_vals, &R);
    return;
  }
  /* host slices: staged piece by piece, the upload of piece k+1 under the route + update of piece k.
   * An ordered batch is staged whole: its global order is rank-major over whole slices. */
  const uint64_t piece = ordered ? nmax : sh->piece;
  const uint64_t base = (nmax + piece - 1) / piece;
  const int taper = !ordered && sh->taper_min && nmax / base >= 4ull * sh->taper_min;
  const uint64_t pieces = rt_pieces(base, taper);
  rt_need_stage(sh, (size_t)(piece < nmax ? piece : nmax) + 1);
  const uint32_t* src[3] = {xs, ys, has_vals ? vals : NULL};
#define PIECE_LO(k) rt_piece_lo((k), base, taper, n)
  for (int a = 0; a < 3 && n && !dev; a++) /* piece 0 */
    if (src[a]) smatrix_b200_memcpy_async(sh->local, sh->stage[0][a], src[a] + PIECE_LO(0), (PIECE_LO(1) - PIECE_LO(0)) * 4, 0);
  for (uint64_t k = 0; k < pieces; k++) {
    const int g = (int)(k & 1u);
    const size_t lo = PIECE_LO(k), hi = PIECE_LO(k + 1);
    smatrix_b200_lane_sync(sh->local, 0); /* piece k is on the device */
    if (k + 1 < pieces && n && !dev) {
      const size_t nlo = hi, nhi = PIECE_LO(k + 2);
      for (int a = 0; a < 3; a++)
        if (src[a]) smatrix_b200_memcpy_async(sh->local, sh->stage[g ^ 1][a], src[a] + nlo, (nhi - nlo) * 4, 0);
    }
    if (dev) /* this rank's slice is already on the device (mixed job): just cut it */
      rt_route(sh, xs + lo, ys + lo, has_vals ? vals + lo : NULL, hi - lo, ordered, 0, &R);
    else
      rt_route(sh, sh->stage[g][0], sh->stage[g][1], has_vals ? sh->stage[g][2] : NULL, hi - lo, ordered, 0, &R);
    rt_apply(sh, op, ordered, has_vals, &R);
  }
#undef PIECE_LO
}

void smatrix_b200_shard_incr_batch(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys,
                                   const uint32_t* vals, size_t n, int ordered) {
  rt_write(sh, 0, xs, ys, vals, n, ordered);
}
void smatrix_b200_shard_decr_batch(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys,
                                   const uint32_t* vals, size_t n, int ordered) {
  rt_write(sh, 1, xs, ys, vals, n, ordered);
}
void smatrix_b200_shard_set_batch(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys,
                                  const uint32_t* vals, size_t n) {
  rt_write(sh, 2, xs, ys, vals, n, 1); /* last writer in GLOBAL input order wins */
}

/* The same batches, returning what every single call would have returned (SURVEY.md 8f N1 across ranks):
 * the ops travel with their global input-order index, every owner applies its inbox in that order and
 * computes the per-op values (smatrix_b200_apply_ordered_out), and the values travel back like read answers.
 * One piece per call (host slices are staged whole): the order is global. */
static void rt_write_out(smatrix_shard_t* sh, int op, const uint32_t* xs, const uint32_t* ys, const uint32_t* vals,
                         size_t n, uint32_t* out) {
  if (n >= 0xFFFFFFFFull) rt_die(sh, "sharded batch too large for one call");
  if (n && !out) rt_die(sh, "batch_out: out must not be NULL");
  const int W = sh->world, me = sh->rank;
  const int dev = n ? rt_is_dev(sh, xs) : 1;
  if (n && (rt_is_dev(sh, ys) != dev || (vals && rt_is_dev(sh, vals) != dev) || rt_is_dev(sh, out) != dev))
    rt_die(sh, "batch arrays must be all host or all device pointers");
  uint64_t mine[4] = {n, n ? (vals != NULL) + 1u : 0u, 0, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t nmax = 0;
  int has_vals = -1;
  for (int r = 0; r < W; r++) {
    if (all[r][0] > nmax) nmax = all[r][0];
    if (all[r][1]) {
      const int hv = (int)all[r][1] - 1;
      if (has_vals >= 0 && has_vals != hv) rt_die(sh, "every rank must pass vals, or none (NULL = all ones)");
      has_vals = hv;
    }
  }
  if (nmax == 0) return;
  if (has_vals < 0) has_vals = 0;
  const uint32_t *d_xs = xs, *d_ys = ys, *d_vs = has_vals ? vals : NULL;
  if (n && !dev) {
    rt_need_stage(sh, n + 1);
    smatrix_b200_memcpy(sh->local, sh->stage[0][0], xs, n * 4);
    smatrix_b200_memcpy(sh->local, sh->stage[0][1], ys, n * 4);
    if (has_vals) smatrix_b200_memcpy(sh->local, sh->stage[0][2], vals, n * 4);
    d_xs = sh->stage[0][0]; d_ys = sh->stage[0][1]; d_vs = has_vals ? sh->stage[0][2] : NULL;
  }
  rt_route_t R;
  rt_route(sh, d_xs, d_ys, d_vs, n, 1, 1, &R);
  const uint64_t cap = sh->cap;
  uint32_t* d_ret = (uint32_t*)(sh->inbox + OFF_CNT(cap)); /* per-op values of MY inbox, inbox order */
  if (R.n_recv)
    smatrix_b200_apply_ordered_out(sh->local, op, (const uint32_t*)(sh->inbox + OFF_X(cap)),
                                   (const uint32_t*)(sh->inbox + OFF_Y(cap)),
                                   has_vals ? (const uint32_t*)(sh->inbox + OFF_V(cap)) : NULL,
                                   (const uint32_t*)(sh->inbox + OFF_O(cap)), (size_t)R.n_recv, d_ret);
  for (int i = 0; i < W; i++) { /* every sender's run goes back into that sender's answer buffer */
    const int s = (me + i) % W;
    const uint64_t c = R.cnt[s][me];
    if (c)
      smatrix_b200_memcpy(sh->local, (uint32_t*)(sh->peer_inbox[s] + OFF_ANS(cap)) + rt_send_base(&R, s, me),
                          d_ret + R.recv_start[s], (size_t)c * 4);
  }
  rt_barrier(sh);
  if (n) {
    uint32_t* d_out = dev ? out : sh->stage[0][3];
    smatrix_b200_gather(sh->local, d_out, (const uint32_t*)(sh->inbox + OFF_ANS(cap)),
                        (const uint32_t*)(sh->inbox + OFF_POS(cap)), n);
    if (!dev) smatrix_b200_memcpy(sh->local, out, d_out, n * 4);
  }
}
void smatrix_b200_shard_incr_batch_out(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys,
                                       const uint32_t* vals, size_t n, uint32_t* out) {
  rt_write_out(sh, 0, xs, ys, vals, n, out);
}
void smatrix_b200_shard_decr_batch_out(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys,
                                       const uint32_t* vals, size_t n, uint32_t* out) {
  rt_write_out(sh, 1, xs, ys, vals, n, out);
}
void smatrix_b200_shard_set_batch_out(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys,
                                      const uint32_t* vals, size_t n, uint32_t* out) {
  rt_write_out(sh, 2, xs, ys, vals, n, out);
}

/* ------------------------------------------------------------------------------ reads */
enum { RT_GET = 0, RT_ROWLEN = 1, RT_COUNTS = 2 };

/* every owner answers the run of every asking rank, output straight into that rank's answer buffer;
 * staggered (rank r starts with requester r, then r + 1, ...) so that the stores of one moment form
 * a shift permutation instead of all ranks writing into the same GPU */
static void rt_answer(smatrix_shard_t* sh, int kind, const rt_route_t* R) {
  const int W = sh->world, me = sh->rank;
  const uint64_t cap = sh->cap;
  for (int i = 0; i < W; i++) {
    const int s = (me + i) % W;
    const uint64_t c = R->cnt[s][me];
    if (!c) continue;
    const uint32_t* qx = (const uint32_t*)(sh->inbox + OFF_X(cap)) + R->recv_start[s];
    const uint32_t* qy = (const uint32_t*)(sh->inbox + OFF_Y(cap)) + R->recv_start[s];
    uint32_t* dst = (uint32_t*)(sh->peer_inbox[s] + OFF_ANS(cap)) + rt_send_base(R, s, me);
    if (kind == RT_GET) smatrix_get_batch(sh->local, qx, qy, (size_t)c, dst);
    else if (kind == RT_ROWLEN) smatrix_rowlen_batch(sh->local, qx, (size_t)c, dst);
    else smatrix_b200_row_counts_batch(sh->local, qx, (size_t)c, dst);
  }
  rt_barrier(sh); /* all answers have landed */
}

/* one device-resident piece: route, answer, gather into d_out (device, n entries) */
static void rt_read_piece(smatrix_shard_t* sh, int kind, const uint32_t* d_xs, const uint32_t* d_ys, size_t n,
                          uint32_t* d_out) {
  rt_route_t R;
  rt_route(sh, d_xs, kind == RT_GET ? d_ys : NULL, NULL, n, 0, 1, &R);
  rt_answer(sh, kind, &R);
  if (n)
    smatrix_b200_gather(sh->local, d_out, (const uint32_t*)(sh->inbox + OFF_ANS(sh->cap)),
                        (const uint32_t*)(sh->inbox + OFF_POS(sh->cap)), n);
}

static void rt_read(smatrix_shard_t* sh, int kind, const uint32_t* xs, const uint32_t* ys, size_t n, uint32_t* out) {
  if (n >= 0xFFFFFFFFull) rt_die(sh, "sharded batch too large for one call");
  const int dev = n ? rt_is_dev(sh, xs) : 1;
  if (n && ((kind == RT_GET && rt_is_dev(sh, ys) != dev) || rt_is_dev(sh, out) != dev))
    rt_die(sh, "batch arrays must be all host or all device pointers");
  uint64_t mine[4] = {n, (uint64_t)!dev, 0, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t nmax = 0;
  int any_host = 0;
  for (int r = 0; r < sh->world; r++) {
    if (all[r][0] > nmax) nmax = all[r][0];
    any_host |= (int)all[r][1];
  }
  if (nmax == 0) return;
  if (!any_host) {
    rt_read_piece(sh, kind, xs, ys, n, out);
    return;
  }
  /* host arrays: piece k+1 goes up (lane 0) and the answers of piece k-1 come down (lane 1 / 2)
   * while piece k is routed and answered */
  const uint64_t piece = sh->piece, base = (nmax + piece - 1) / piece;
  const int taper = sh->taper_min && nmax / base >= 4ull * sh->taper_min;
  const uint64_t pieces = rt_pieces(base, taper);
  rt_need_stage(sh, (size_t)(piece < nmax ? piece : nmax) + 1);
#define PIECE_LO(k) rt_piece_lo((k), base, taper, n)
  if (!dev && n) {
    smatrix_b200_memcpy_async(sh->local, sh->stage[0][0], xs, (PIECE_LO(1) - PIECE_LO(0)) * 4, 0);
    if (kind == RT_GET) smatrix_b200_memcpy_async(sh->local, sh->stage[0][1], ys, (PIECE_LO(1) - PIECE_LO(0)) * 4, 0);
  }
  for (uint64_t k = 0; k < pieces; k++) {
    const int g = (int)(k & 1u);
    const size_t lo = PIECE_LO(k), hi = PIECE_LO(k + 1);
    smatrix_b200_lane_sync(sh->local, 0);
    if (!dev && k + 1 < pieces && n) {
      const size_t nlo = hi, nhi = PIECE_LO(k + 2);
      smatrix_b200_memcpy_async(sh->local, sh->stage[g ^ 1][0], xs + nlo, (nhi - nlo) * 4, 0);
      if (kind == RT_GET) smatrix_b200_memcpy_async(sh->local, sh->stage[g ^ 1][1], ys + nlo, (nhi - nlo) * 4, 0);
    }
    if (dev) {
      rt_read_piece(sh, kind, xs + lo, kind == RT_GET ? ys + lo : NULL, hi - lo, out + lo);
    } else {
      smatrix_b200_lane_sync(sh->local, 1 + g); /* the answer buffer of piece k-2 has been downloaded */
      rt_read_piece(sh, kind, sh->stage[g][0], sh->stage[g][1], hi - lo, sh->stage[g][3]);
      if (hi > lo) smatrix_b200_memcpy_async(sh->local, out + lo, sh->stage[g][3], (hi - lo) * 4, 1 + g);
    }
  }
  if (!dev) {
    smatrix_b200_lane_sync(sh->local, 1);
    smatrix_b200_lane_sync(sh->local, 2);
  }
#undef PIECE_LO
}

void smatrix_b200_shard_get_batch(smatrix_shard_t* sh, const uint32_t* xs, const uint32_t* ys, size_t n,
                                  uint32_t* out) {
  rt_read(sh, RT_GET, xs, ys, n, out);
}
void smatrix_b200_shard_rowlen_batch(smatrix_shard_t* sh, const uint32_t* xs, size_t n, uint32_t* out) {
  rt_read(sh, RT_ROWLEN, xs, NULL, n, out);
}

/* ------------------------------------------------------------------------------ getrow */
/* Collective core of getrow: row ids d_xs (device, n of them) -> CSR offsets in my OFS array and, if
 * this rank wants them (want != 0 and total <= cap_pairs), the pairs in my row buffer.  Returns the
 * total; *filled = whether my row buffer holds my pairs; *any_fill = whether ANY rank filled (the
 * callers' follow-up collectives hinge on it). */
static uint64_t rt_getrow_core(smatrix_shard_t* sh, const uint32_t* d_xs, size_t n, int want, uint64_t cap_pairs,
                               int* filled, int* any_fill_out) {
  const int W = sh->world, me = sh->rank;
  rt_route_t R;
  rt_route(sh, d_xs, NULL, NULL, n, 0, 1, &R);
  rt_answer(sh, RT_COUNTS, &R);
  const uint64_t cap = sh->cap;
  uint32_t* d_cnt = (uint32_t*)(sh->inbox + OFF_CNT(cap));
  uint64_t* d_off = (uint64_t*)(sh->inbox + OFF_OFS(cap));
  const uint32_t* d_pos = (const uint32_t*)(sh->inbox + OFF_POS(cap));
  uint64_t total = 0;
  if (n) {
    smatrix_b200_gather(sh->local, d_cnt, (const uint32_t*)(sh->inbox + OFF_ANS(cap)), d_pos, n);
    total = smatrix_b200_scan_counts(sh->local, d_cnt, n, d_off);
  }
  const int want_fill = want && total > 0 && total <= cap_pairs;
  uint64_t mine[4] = {(uint64_t)want_fill, want_fill ? total : 0, 0, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t most = 0;
  int any_fill = 0;
  for (int r = 0; r < W; r++) {
    any_fill |= (int)all[r][0];
    if (all[r][1] > most) most = all[r][1];
  }
  *filled = want_fill;
  *any_fill_out = any_fill;
  if (!any_fill) return total;
  rt_need_rowbuf(sh, most);
  if (want_fill) { /* every row's offset travels to the row's owner */
    uint64_t tab[2 * RT_MAXW];
    for (int o = 0; o < W; o++) {
      tab[o] = R.send_base[o];
      tab[W + o] = (uint64_t)(uintptr_t)(sh->peer_inbox[o] + OFF_Q64(cap) + 8 * rt_in_base(&R, me, o));
    }
    smatrix_b200_route_offsets(sh->local, d_off, d_pos, n, (uint32_t)W, tab);
  }
  rt_barrier(sh);
  for (int i = 0; i < W; i++) { /* owners compact the rows into the asking rank's row buffer */
    const int s = (me + i) % W;
    const uint64_t c = R.cnt[s][me];
    if (!c || !all[s][0]) continue;
    smatrix_b200_getrow_fill_at(sh->local, (const uint32_t*)(sh->inbox + OFF_X(cap)) + R.recv_start[s], (size_t)c,
                                (const uint64_t*)(sh->inbox + OFF_Q64(cap)) + R.recv_start[s],
                                (uint32_t*)sh->peer_rowbuf[s]);
  }
  rt_barrier(sh);
  return total;
}

/* row ids (or items) as a device array: host arrays are few compared with the pairs, one staged copy */
static const uint32_t* rt_ids_on_device(smatrix_shard_t* sh, const uint32_t* xs, size_t n) {
  if (!n || rt_is_dev(sh, xs)) return xs;
  rt_need_stage(sh, n + 1);
  smatrix_b200_memcpy(sh->local, sh->stage[0][0], xs, n * 4);
  return sh->stage[0][0];
}

/* smatrix_b200_shard_getrow_batch, and with sorted != 0 shard_getrow_sorted_batch: the pairs are sorted by column in
 * this rank's row buffer before they are copied out */
static uint64_t rt_getrow(smatrix_shard_t* sh, const char* what, int sorted, const uint32_t* xs, size_t n,
                          uint64_t* offsets, uint32_t* pairs, uint64_t pairs_cap) {
  if (n >= 0xFFFFFFFEull) rt_die(sh, "%s: too many rows in one call", what);
  int filled = 0, any = 0;
  const uint64_t total = rt_getrow_core(sh, rt_ids_on_device(sh, xs, n), n, pairs != NULL, pairs_cap, &filled, &any);
  if (filled && sorted)
    smatrix_b200_sort_rows(sh->local, n, (const uint64_t*)(sh->inbox + OFF_OFS(sh->cap)), (uint32_t*)sh->rowbuf);
  if (offsets) {
    if (n) {
      smatrix_b200_memcpy(sh->local, offsets, sh->inbox + OFF_OFS(sh->cap), (n + 1) * 8);
    } else {
      const uint64_t zero = 0;
      smatrix_b200_memcpy(sh->local, offsets, &zero, 8);
    }
  }
  if (filled) smatrix_b200_memcpy(sh->local, pairs, sh->rowbuf, (size_t)total * 8);
  return total;
}

uint64_t smatrix_b200_shard_getrow_batch(smatrix_shard_t* sh, const uint32_t* xs, size_t n, uint64_t* offsets,
                                         uint32_t* pairs, uint64_t pairs_cap) {
  return rt_getrow(sh, "getrow_batch", 0, xs, n, offsets, pairs, pairs_cap);
}
uint64_t smatrix_b200_shard_getrow_sorted_batch(smatrix_shard_t* sh, const uint32_t* xs, size_t n, uint64_t* offsets,
                                                uint32_t* pairs, uint64_t pairs_cap) {
  return rt_getrow(sh, "getrow_sorted_batch", 1, xs, n, offsets, pairs, pairs_cap);
}

/* The first cap keys >= from of the whole matrix are among the first cap of every rank's own.  Those lists (their
 * lengths all-gathered) go into every rank's row buffer side by side, in rank order, and every rank sorts the lot. */
uint64_t smatrix_b200_shard_list_rows(smatrix_shard_t* sh, uint32_t from, uint32_t* keys, uint64_t cap) {
  const int W = sh->world, me = sh->rank;
  const uint64_t mine_m = smatrix_list_rows(sh->local, from, NULL, 0);
  const uint64_t take = mine_m < cap ? mine_m : cap;
  uint64_t mine[4] = {mine_m, take, (uint64_t)(keys != NULL && cap > 0), 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t m = 0, T = 0, at = 0;
  int want = 0;
  for (int r = 0; r < W; r++) {
    m += all[r][0];
    if (r < me) at += all[r][1];
    T += all[r][1];
    want |= (int)all[r][2];
  }
  if (!want || !T) return m;
  rt_need_rowbuf(sh, (T + 1) / 2); /* T keys of 4 bytes in a buffer of 8-byte pairs; the same T on every rank */
  uint32_t* d_keys = (uint32_t*)sh->rowbuf;
  if (take) {
    smatrix_list_rows(sh->local, from, d_keys + at, cap);
    for (int r = 0; r < W; r++)
      if (r != me) smatrix_b200_memcpy(sh->local, (uint32_t*)sh->peer_rowbuf[r] + at, d_keys + at, (size_t)take * 4);
  }
  rt_barrier(sh);
  if (keys) smatrix_b200_sort_keys(sh->local, d_keys, (size_t)T, keys, cap);
  rt_barrier(sh); /* nobody writes into a row buffer that its rank still sorts from */
  return m;
}

/* The collective core of both CF calls: rows through the getrow route, totals through two sharded gets, scores
 * on this rank's GPU.  Returns the total; when any rank fills, c->scratch holds (with `extra` more bytes at
 * c->extra) and, if this rank filled, c->off / c->ids / c->scores are its CSR of scores on the device.  The
 * caller frees c->scratch. */
typedef struct {
  char* scratch;
  void* extra;
  uint64_t* off;
  uint32_t* ids;
  double* scores;
  int filled;
} rt_cf_t;
static uint64_t rt_cf_scores(smatrix_shard_t* sh, const uint32_t* items, size_t n, int want, uint64_t cap,
                             uint64_t* offsets, size_t extra, rt_cf_t* c) {
  const uint32_t* d_items = rt_ids_on_device(sh, items, n);
  int filled = 0, any = 0;
  const uint64_t total = rt_getrow_core(sh, d_items, n, want, cap, &filled, &any);
  if (offsets) {
    if (n) {
      smatrix_b200_memcpy(sh->local, offsets, sh->inbox + OFF_OFS(sh->cap), (n + 1) * 8);
    } else {
      const uint64_t zero = 0;
      smatrix_b200_memcpy(sh->local, offsets, &zero, 8);
    }
  }
  memset(c, 0, sizeof *c);
  c->filled = filled;
  if (!any) return total;
  /* scratch on my GPU: neighbour ids, their totals, my items' totals, zeros (column 0), scores, and a
   * copy of the CSR offsets + items (the gets below reuse the inbox's local arrays) */
  const size_t np = filled ? (size_t)total : 0, nn = filled ? n : 0;
  const size_t big = np > nn ? np : nn;
  char* scratch = (char*)smatrix_b200_dev_alloc(sh->local, big * 4 * 2 + np * 4 + nn * 4 * 2 + np * 8 + (nn + 1) * 8 +
                                                extra + 256);
  uint32_t* d_zero = (uint32_t*)scratch;
  uint32_t* d_cols = d_zero + big;
  uint32_t* d_btot = d_cols + big;
  uint32_t* d_atot = d_btot + np;
  uint32_t* d_keep = d_atot + nn;                                        /* my items */
  uint64_t* d_off = (uint64_t*)(((uintptr_t)(d_keep + nn) + 7) & ~(uintptr_t)7);
  double* d_scores = (double*)(d_off + nn + 1);
  if (filled) {
    smatrix_b200_memcpy(sh->local, d_off, sh->inbox + OFF_OFS(sh->cap), (n + 1) * 8);
    smatrix_b200_memcpy(sh->local, d_keep, d_items, n * 4);
    smatrix_b200_memset0(sh->local, d_zero, big * 4);
    smatrix_b200_pair_cols(sh->local, (const uint32_t*)sh->rowbuf, total, d_cols);
  }
  rt_read_piece(sh, RT_GET, d_cols, d_zero, np, d_btot);                  /* collective: n = 0 on ranks that do not fill */
  rt_read_piece(sh, RT_GET, d_keep, d_zero, nn, d_atot);
  /* the ids go out through d_cols' slot again (same values), the scores through d_scores */
  if (filled) smatrix_b200_cf_scores_totals(sh->local, n, d_off, (const uint32_t*)sh->rowbuf, d_atot, d_btot, d_cols, d_scores);
  c->scratch = scratch;
  c->extra = d_scores + np;
  c->off = d_off;
  c->ids = d_cols;
  c->scores = d_scores;
  return total;
}

/* The read side of the co-occurrence recommender across ranks (examples/cf_recommender.c:50-86, same
 * contract as smatrix_cf_neighbors_batch): the rows come through the getrow route; the totals
 * (value at (item, 0) and at (neighbour, 0)) are two sharded gets; the scores are computed where the
 * pairs landed. */
uint64_t smatrix_b200_shard_cf_neighbors_batch(smatrix_shard_t* sh, const uint32_t* items, size_t n,
                                               uint64_t* offsets, uint32_t* ids, double* scores, uint64_t cap) {
  if (n >= 0xFFFFFFFEull) rt_die(sh, "cf_neighbors_batch: too many items in one call");
  rt_cf_t c;
  const uint64_t total = rt_cf_scores(sh, items, n, ids != NULL && scores != NULL, cap, offsets, 0, &c);
  if (c.filled) {
    smatrix_b200_memcpy(sh->local, ids, c.ids, (size_t)total * 4);
    smatrix_b200_memcpy(sh->local, scores, c.scores, (size_t)total * 8);
  }
  if (c.scratch) smatrix_b200_dev_free(sh->local, c.scratch);
  return total;
}

void smatrix_b200_shard_cf_topk_batch(smatrix_shard_t* sh, const uint32_t* items, size_t n, uint32_t k,
                                      uint32_t* counts, uint32_t* ids, double* scores) {
  if (k < 1 || k > 1024u) rt_die(sh, "cf_topk_batch: k = %u is outside 1..1024", k);
  if (n >= 0xFFFFFFFEull) rt_die(sh, "cf_topk_batch: too many items in one call");
  const int out_dev = rt_is_dev(sh, counts);
  if (n && (rt_is_dev(sh, ids) != out_dev || rt_is_dev(sh, scores) != out_dev))
    rt_die(sh, "batch arrays must be all host or all device pointers");
  /* room for the answers on the device when they go to host arrays, and for all-zero offsets when this rank's
   * rows are empty (then it fills nothing but still ranks: every count is 0) */
  const size_t out_bytes = out_dev ? 0 : n * (12ull * k + 4);
  rt_cf_t c;
  rt_cf_scores(sh, items, n, 1, ~0ull, NULL, out_bytes + (n + 1) * 8 + 64, &c);
  if (n) {
    char* extra = c.scratch ? (char*)(((uintptr_t)c.extra + 7) & ~(uintptr_t)7)
                            : (char*)smatrix_b200_dev_alloc(sh->local, out_bytes + (n + 1) * 8 + 64);
    const uint64_t* d_off = c.off;
    if (!c.filled) {
      smatrix_b200_memset0(sh->local, extra, (n + 1) * 8);
      d_off = (const uint64_t*)extra;
    }
    double* os = out_dev ? scores : (double*)(extra + (n + 1) * 8);
    uint32_t* oi = out_dev ? ids : (uint32_t*)(os + n * k);
    uint32_t* oc = out_dev ? counts : oi + n * k;
    smatrix_b200_topk_segments(sh->local, n, d_off, c.ids, c.scores, k, oc, oi, os);
    if (!out_dev) {
      smatrix_b200_memcpy(sh->local, counts, oc, n * 4);
      smatrix_b200_memcpy(sh->local, ids, oi, n * k * 4);
      smatrix_b200_memcpy(sh->local, scores, os, n * k * 8);
    }
    if (!c.scratch) smatrix_b200_dev_free(sh->local, extra);
  }
  if (c.scratch) smatrix_b200_dev_free(sh->local, c.scratch);
}

/* Basket recommendations across ranks: the flattened items' lists come as in shard_cf_neighbors_batch, and
 * smatrix_b200_basket_topk aggregates and ranks them on this rank's GPU, the same code as the single-GPU call. */
void smatrix_b200_shard_cf_recommend_batch(smatrix_shard_t* sh, const uint64_t* basket_off, const uint32_t* items,
                                           size_t n, uint32_t k, uint32_t* counts, uint32_t* ids, double* scores) {
  if (k < 1 || k > 1024u) rt_die(sh, "cf_recommend_batch: k = %u is outside 1..1024", k);
  if (n >= 0xFFFFFFFEull) rt_die(sh, "cf_recommend_batch: too many baskets in one call");
  const int out_dev = rt_is_dev(sh, counts);
  if (n && (rt_is_dev(sh, ids) != out_dev || rt_is_dev(sh, scores) != out_dev))
    rt_die(sh, "cf_recommend_batch: counts, ids and scores must be all host or all device arrays");
  /* the offsets on the host, to check them and to know the number of items */
  const int in_dev = n && rt_is_dev(sh, basket_off);
  uint64_t* hb = NULL;
  uint64_t n_pos = 0;
  if (n) {
    if (!basket_off) rt_die(sh, "cf_recommend_batch: basket_off is NULL");
    hb = (uint64_t*)malloc((n + 1) * 8);
    if (!hb) rt_die(sh, "out of host memory");
    smatrix_b200_memcpy(sh->local, hb, basket_off, (n + 1) * 8);
    int bad = hb[0] != 0 || hb[n] > 0xFFFFFFFEull;
    for (size_t i = 0; i < n && !bad; i++) bad = hb[i + 1] < hb[i];
    if (bad)
      rt_die(sh, "cf_recommend_batch: malformed basket offsets (they must start at 0, never decrease and end at "
                 "most at 2^32 - 2)");
    n_pos = hb[n];
    if (n_pos && rt_is_dev(sh, items) != in_dev)
      rt_die(sh, "cf_recommend_batch: basket_off and items must both be host or both be device arrays");
  }
  /* room for: the answers when they go to host arrays, all-zero offsets when this rank's rows are empty, the
   * offsets and items when they are host arrays */
  const size_t out_bytes = out_dev ? 0 : n * (12ull * k + 4);
  const size_t in_bytes = in_dev ? 0 : (n + 1) * 8 + n_pos * 4;
  const size_t extra = out_bytes + (n_pos + 1) * 8 + in_bytes + 64;
  rt_cf_t c;
  rt_cf_scores(sh, items, n_pos, 1, ~0ull, NULL, extra, &c);
  if (n) {
    char* ex = c.scratch ? (char*)(((uintptr_t)c.extra + 7) & ~(uintptr_t)7)
                         : (char*)smatrix_b200_dev_alloc(sh->local, extra);
    const uint64_t* d_off = c.off;
    char* at = ex;
    if (!c.filled) {
      smatrix_b200_memset0(sh->local, at, (n_pos + 1) * 8);
      d_off = (const uint64_t*)at;
    }
    at += (n_pos + 1) * 8;
    const uint64_t* d_boff = basket_off;
    const uint32_t* d_items = items;
    if (!in_dev) {
      smatrix_b200_memcpy(sh->local, at, hb, (n + 1) * 8);
      d_boff = (const uint64_t*)at;
      at += (n + 1) * 8;
      if (n_pos) smatrix_b200_memcpy(sh->local, at, items, n_pos * 4);
      d_items = (const uint32_t*)at;
      at += (n_pos * 4 + 7) & ~(size_t)7;
    }
    double* os = out_dev ? scores : (double*)at;
    uint32_t* oi = out_dev ? ids : (uint32_t*)(os + n * k);
    uint32_t* oc = out_dev ? counts : oi + n * k;
    smatrix_b200_basket_topk(sh->local, n, d_boff, d_items, d_off, c.ids, c.scores, k, oc, oi, os);
    if (!out_dev) {
      smatrix_b200_memcpy(sh->local, counts, oc, n * 4);
      smatrix_b200_memcpy(sh->local, ids, oi, n * k * 4);
      smatrix_b200_memcpy(sh->local, scores, os, n * k * 8);
    }
    if (!c.scratch) smatrix_b200_dev_free(sh->local, ex);
  }
  free(hb);
  if (c.scratch) smatrix_b200_dev_free(sh->local, c.scratch);
}

/* ------------------------------------------------------------------------------ file mode */
/* Collective: the .smx snapshot of the whole sharded matrix, one ordinary file in the reference's format.
 * Every rank lays out its own rows (snap_extent); exclusive prefixes of the (rows, bytes) pairs give each rank
 * its first directory entry and the byte where its row blocks go.  Rank 0 creates `fname.tmp` with the header
 * and directory block headers at its final size, then every rank writes its part and fsyncs, and rank 0
 * renames the file over the old one.  The outcome is agreed on: 0 or -1 on every rank. */
static int rt_all_ok(smatrix_shard_t* sh, int ok) {
  uint64_t mine[4] = {(uint64_t)(ok != 0), 0, 0, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  for (int r = 0; r < sh->world; r++) ok = ok && all[r][0];
  return ok;
}

static int rt_snapshot(smatrix_shard_t* sh) {
  const int W = sh->world, me = sh->rank;
  uint64_t rows = 0, bytes = 0;
  if (sh->fname) smatrix_b200_snap_extent(sh->local, &rows, &bytes);
  uint64_t mine[4] = {sh->fname != NULL, rows, bytes, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t total_rows = 0, total_bytes = 0, first = 0, base = 0;
  int have = 1;
  for (int r = 0; r < W; r++) {
    have = have && all[r][0];
    if (r == me) { first = total_rows; base = total_bytes; }
    total_rows += all[r][1];
    total_bytes += all[r][2];
  }
  if (!have) return -1;
  base += smatrix_b200_snap_rows_base(total_rows);
  const size_t fl = strlen(sh->fname);
  char* tmp = (char*)malloc(fl + 8);
  if (!tmp) rt_die(sh, "out of host memory");
  memcpy(tmp, sh->fname, fl);
  memcpy(tmp + fl, ".tmp", 5);
  int fd = -1, ok = 1;
  if (me == 0) {
    fd = open(tmp, O_RDWR | O_CREAT | O_TRUNC, 00600);
    ok = fd != -1 && smatrix_b200_snap_layout(fd, total_rows, total_bytes) == 0;
  }
  if (rt_all_ok(sh, ok)) { /* the file exists at its final size: the others open it without O_TRUNC */
    if (me != 0) fd = open(tmp, O_RDWR);
    ok = fd != -1 && smatrix_b200_snap_write(sh->local, fd, base, first) == 0 && fsync(fd) == 0;
  } else {
    ok = 0;
  }
  if (fd != -1 && close(fd) == -1) ok = 0;
  ok = rt_all_ok(sh, ok);
  if (me == 0) {
    if (ok && smatrix_b200_snap_commit(tmp, sh->fname) != 0) ok = 0;
    if (!ok) {
      perror("libsmatrix: writing the snapshot failed");
      unlink(tmp); /* the previous snapshot, if any, is still intact */
    }
  }
  free(tmp);
  if (!rt_all_ok(sh, ok)) return -1;
  smatrix_b200_clear_dirty(sh->local); /* the file matches the table */
  sh->ck_base = 1;
  return 0;
}

int smatrix_b200_shard_snapshot(smatrix_shard_t* sh) { return rt_snapshot(sh); }

/* Collective: the checkpoint of smatrix_b200_checkpoint for the whole sharded matrix.  Every decision is taken from
 * all-gathered values, so every rank takes the same branch: no file -> -1; nothing written -> 0; no base (the file
 * was or is missing or empty) -> the full snapshot.  Then every rank reads an even share of the old directory and
 * routes its (key, row offset lo, hi) entries to the rows' owners in pieces, and each owner runs the keep filter on
 * its inbox.  A listed row missing anywhere, Σ (kept + dirty) != Σ rows, or an appended file past twice a full
 * snapshot -> the full snapshot.  Otherwise exclusive prefixes give every rank the byte where its dirty rows' blocks
 * go behind E and its first entry in the new chain at D (its kept entries, then its dirty rows'); rank 0 extends the
 * file and writes the block headers, every rank writes its part and fsyncs, rank 0 switches the header and fsyncs,
 * and every rank clears its marks.  Each step's outcome is agreed on: 0 or -1 on every rank. */
static int rt_checkpoint(smatrix_shard_t* sh) {
  const int W = sh->world, me = sh->rank;
  uint64_t dirty = sh->fname ? smatrix_b200_stat(sh->local, SMX_STAT_DIRTY_ROWS) : 0;
  uint64_t fstate = 0; /* rank 0: 0 = the file is missing, 1 = it cannot be read, else its size + 2 */
  if (me == 0 && sh->fname) {
    struct stat st;
    if (stat(sh->fname, &st) == 0) fstate = S_ISREG(st.st_mode) ? (uint64_t)st.st_size + 2 : 1;
    else fstate = errno == ENOENT ? 0 : 1;
  }
  uint64_t mine[4] = {sh->fname != NULL, dirty, fstate, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  uint64_t total_dirty = 0;
  int have = 1;
  for (int r = 0; r < W; r++) { have = have && all[r][0]; total_dirty += all[r][1]; }
  if (!have) return -1;
  if (!total_dirty) return 0;
  fstate = all[0][2];
  if (fstate == 1) {
    if (me == 0) fprintf(stderr, "libsmatrix: cannot open %s for a checkpoint\n", sh->fname);
    return -1;
  }
  if (!sh->ck_base || fstate <= 2) return rt_snapshot(sh); /* the file never matched the table, or is gone */
  const uint64_t fsize = fstate - 2;
  uint64_t rows = 0, bytes = 0, drows = 0, dbytes = 0;
  smatrix_b200_snap_extent(sh->local, &rows, &bytes);
  const int fd = open(sh->fname, O_RDWR);
  smx_loader_t* ld = fd == -1 ? NULL : smatrix_b200_load_begin(sh->local, fd, me, W);
  const uint64_t n = ld ? smatrix_b200_load_entries(ld, 0, 0, NULL, NULL, NULL) : 0;
  const uint64_t piece = sh->piece, pieces = (n + piece - 1) / piece;
  uint64_t m1[4] = {ld != NULL, pieces, 0, 0};
  rt_allgather(sh, m1, all);
  int ok = 1;
  uint64_t max_pieces = 0;
  for (int r = 0; r < W; r++) { ok = ok && all[r][0]; if (all[r][1] > max_pieces) max_pieces = all[r][1]; }
  uint64_t missing = 0, kept = 0;
  if (ok) {
    rt_need_stage(sh, (size_t)(n < piece ? n : piece) + 1);
    for (uint64_t k = 0; k < max_pieces; k++) { /* the same number of routes on every rank */
      const uint64_t lo = k * piece < n ? k * piece : n, len = (n - lo < piece) ? n - lo : piece;
      if (len) smatrix_b200_load_entries(ld, lo, len, sh->stage[0][0], sh->stage[0][1], sh->stage[0][2]);
      rt_route_t R;
      rt_route(sh, sh->stage[0][0], sh->stage[0][1], sh->stage[0][2], (size_t)len, 0, 0, &R);
      const uint64_t cap = sh->cap;
      missing += smatrix_b200_ckpt_keep(sh->local, (const uint32_t*)(sh->inbox + OFF_X(cap)),
                                        (const uint32_t*)(sh->inbox + OFF_Y(cap)),
                                        (const uint32_t*)(sh->inbox + OFF_V(cap)), (size_t)R.n_recv, &kept);
      rt_barrier(sh); /* the inboxes are read before the next route fills them */
    }
  }
  smatrix_b200_load_end(ld);
  /* held until snap_write_at; laid out only now, because the routes above reuse the scratch that holds it */
  smatrix_b200_ckpt_extent(sh->local, &drows, &dbytes);
  uint64_t m2[4] = {(uint64_t)ok, missing, kept, 0}, m3[4] = {rows, bytes, drows, dbytes}, all3[RT_MAXW][4];
  rt_allgather(sh, m2, all);
  rt_allgather(sh, m3, all3);
  uint64_t t_rows = 0, t_bytes = 0, t_drows = 0, t_dbytes = 0, t_missing = 0, t_kept = 0, byte_off = 0, first = 0;
  for (int r = 0; r < W; r++) {
    ok = ok && all[r][0];
    if (r == me) { byte_off = t_dbytes; first = t_kept + t_drows; }
    t_missing += all[r][1]; t_kept += all[r][2];
    t_rows += all3[r][0]; t_bytes += all3[r][1]; t_drows += all3[r][2]; t_dbytes += all3[r][3];
  }
  const uint64_t E = (fsize + 7) & ~7ull, D = E + t_dbytes;
  const uint64_t end = D + smatrix_b200_snap_rows_base(t_kept + t_drows) - 512; /* the chain without the header */
  const int match = ok && t_missing == 0 && t_kept + t_drows == t_rows;
  if (!match || end > 2 * (smatrix_b200_snap_rows_base(t_rows) + t_bytes)) {
    /* a file that does not describe this table, or one that has grown to twice a full snapshot: rewrite it */
    if (fd != -1) close(fd);
    smatrix_b200_ckpt_reset(sh->local);
    return rt_snapshot(sh);
  }
  ok = me != 0 || smatrix_b200_ckpt_layout(fd, D, t_kept + t_drows) == 0;
  if (rt_all_ok(sh, ok)) { /* the file has its final size */
    ok = smatrix_b200_snap_write_at(sh->local, fd, E + byte_off, D, first + kept) == 0;
    ok = smatrix_b200_ckpt_write_kept(sh->local, fd, D, first) == 0 && ok;
    ok = ok && fsync(fd) == 0;
  } else {
    ok = 0;
  }
  smatrix_b200_ckpt_reset(sh->local);
  ok = rt_all_ok(sh, ok);
  if (me == 0) {
    if (!ok) (void)!ftruncate(fd, (off_t)fsize); /* the header was not switched: the old file as it was */
    else if (smatrix_b200_ckpt_switch(fd, D) != 0) ok = 0;
  }
  if (close(fd) == -1) ok = 0;
  if (!rt_all_ok(sh, ok)) {
    if (me == 0) perror("libsmatrix: writing the checkpoint failed");
    return -1;
  }
  smatrix_b200_clear_dirty(sh->local);
  return 0;
}

int smatrix_b200_shard_checkpoint(smatrix_shard_t* sh) { return rt_checkpoint(sh); }

static uint64_t rt_fnv(const char* p) {
  uint64_t h = 0xcbf29ce484222325ull;
  for (; *p; p++) h = (h ^ (unsigned char)*p) * 0x100000001b3ull;
  return h;
}

/* Collective: every rank reads its share of the file's directory (smatrix_b200_load_next) and routes each
 * piece to the rows' owners as an ordered set batch, then the pieces' (key, log2 size) fixups, which every
 * owner applies after the ops.  Ranks whose share has run out join with n = 0 until no rank has more. */
static int rt_load(smatrix_shard_t* sh, int fd) {
  smx_loader_t* ld = smatrix_b200_load_begin(sh->local, fd, sh->rank, sh->world);
  int bad = ld == NULL;
  for (;;) {
    const uint32_t *xs = NULL, *ys = NULL, *vs = NULL, *keys = NULL, *logs = NULL;
    size_t n = 0, nr = 0;
    const int r = bad ? 0 : smatrix_b200_load_next(ld, &xs, &ys, &vs, &n, &keys, &logs, &nr);
    if (r < 0) bad = 1;
    if (r <= 0) n = nr = 0;
    uint64_t mine[4] = {(uint64_t)bad, (uint64_t)(r > 0), 0, 0}, all[RT_MAXW][4];
    rt_allgather(sh, mine, all);
    int any_bad = 0, any_more = 0;
    for (int k = 0; k < sh->world; k++) { any_bad |= (int)all[k][0]; any_more |= (int)all[k][1]; }
    if (any_bad) { bad = 1; break; }
    if (!any_more) break;
    rt_write(sh, 2, xs, ys, vs, n, 1);
    rt_route_t R;
    rt_route(sh, keys, logs, NULL, nr, 0, 0, &R);
    if (R.n_recv)
      smatrix_b200_load_fixup(sh->local, (const uint32_t*)(sh->inbox + OFF_X(sh->cap)),
                              (const uint32_t*)(sh->inbox + OFF_Y(sh->cap)), (size_t)R.n_recv);
  }
  smatrix_b200_load_end(ld);
  if (bad && sh->rank == 0) fprintf(stderr, "libsmatrix: file is corrupt\n");
  return bad ? -1 : 0;
}

smatrix_shard_t* smatrix_b200_shard_open_file(const char* name, int rank, int world, int device, size_t arena_bytes,
                                              const char* fname) {
  smatrix_shard_t* sh = smatrix_b200_shard_open_arena(name, rank, world, device, arena_bytes);
  if (!sh || !fname) return sh;
  /* like smatrix_open(fname): the file must be creatable / readable, on every rank, under one path */
  const int fd = open(fname, O_RDWR | O_CREAT, 00600);
  if (fd == -1) perror("cannot open file");
  struct stat st;
  const int has_data = fd != -1 && fstat(fd, &st) == 0 && st.st_size > 0;
  uint64_t mine[4] = {(uint64_t)(fd != -1), rt_fnv(fname), (uint64_t)has_data, 0}, all[RT_MAXW][4];
  rt_allgather(sh, mine, all);
  int ok = 1, same = 1;
  for (int r = 0; r < world; r++) {
    ok = ok && all[r][0];
    same = same && all[r][1] == all[0][1] && all[r][2] == all[0][2];
  }
  if (ok && !same) {
    if (rank == 0) fprintf(stderr, "libsmatrix: shard_open_file: the ranks were given different files\n");
    ok = 0;
  }
  if (ok && all[0][2] && rt_load(sh, fd) != 0) ok = 0;
  if (fd != -1) close(fd);
  if (ok) { /* the loaded rows are what the file holds */
    smatrix_b200_clear_dirty(sh->local);
    sh->ck_base = all[0][2] != 0;
  }
  if (!ok) { /* every rank takes this branch together; a file we could not read is not overwritten */
    smatrix_b200_shard_close(sh);
    return NULL;
  }
  sh->fname = strdup(fname);
  if (!sh->fname) rt_die(sh, "out of host memory");
  return sh;
}
