/*
 * smx_kernels.cu — hand-written sm_100a kernels for the libsmatrix in-memory hot path and their
 * extern "C" launchers.  No tensor cores: nothing on this path is a dense contraction; every
 * kernel is bound by random 32-byte-sector HBM accesses (update / get) or by streaming HBM
 * bandwidth (row growth, getrow), so the levers are sector-exact accesses (one 256-bit
 * LDG per probe), enough resident threads to cover ~1 us dependent-miss chains, and atomics that
 * resolve in L2.
 *
 * Kernel                replaces (reference src/smatrix.c)
 *   k_upsert            smatrix_lookup(write) + cmap_lookup/insert + rmap_probe/insert + the
 *                       value update of set/incr/decr  (:225-304, :343-380, :621-713)
 *   k_grow_plan, k_free_push, k_migrate / _mid / _big
 *                       smatrix_rmap_resize + smatrix_mfree of the old map (:383-416, :151-166)
 *   k_dir_rehash, k_sketch_*   smatrix_cmap_resize (:715-741)
 *   k_get, k_get_tiled  smatrix_get (:174-185): queries in input order (resident grid) / in directory-slice
 *                       order (one block per 1024 consecutive queries, dispatched in order)
 *   k_rowlen            smatrix_rowlen (:212-223)
 *   k_row_counts, scan, k_getrow_inline / _fill / _chunks   smatrix_getrow (:189-210) for batches of rows
 *   k_set_max/mark/commit  last-writer-wins resolution for smatrix_set batches (:225-234 applied
 *                       sequentially)
 *   k_snap_units / _rows / _big   the row blocks of the .smx file (:454-482) in the loader's layout (:499-545)
 *   k_load_count / _emit          the loader's parse of raw row blocks into (x, y, v) ops (:499-545)
 *   k_partition_count / _scatter  no counterpart: chunk ordering by directory slice (writes and large read
 *                       calls), and the multi-GPU route (every owner's run stored straight into that
 *                       owner's inbox over NVLink)
 *   k_parts_prefix, k_gather      cursors of the parts on the device; answers back into input order
 *
 * Concurrency rules the code relies on (DESIGN.md "Concurrency"):
 *   - cells and directory entries are only ever claimed 0 -> key by a 64-bit CAS and keys never
 *     change afterwards, so a stale "occupied by another key" view is always still true and a
 *     stale "empty" view is corrected by the CAS; probing always tries cells in probe order.
 *   - buckets move only in the k_migrate kernels and k_dir_rehash, which never run concurrently with k_upsert.
 *   - no thread ever waits for another thread: anything that cannot complete (directory at its
 *     load limit, bucket at its load limit) is appended to a retry list and the host grows the
 *     structure between launches.
 */
#include "smx_internal.h"

#ifdef SMX_HOSTSIM
#include "hostsim.h"
#include "cuda_runtime_api.h"
#include <algorithm>
#include <vector>
#else
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh> /* only for the optional *_batch_out ordering step (N1) */
#define SMX_WARP 32
#define SMX_LAUNCH(kern, grid, block, stream, ...) \
  kern<<<(grid), (block), 0, (cudaStream_t)(stream)>>>(__VA_ARGS__)
/* opportunistic aggregation over whichever lanes happen to be converged here.  `key` is only read by the
 * 32-lane CPU simulator (tests/hostsim/warp_sched.cpp), which has no instruction addresses to tell two inlined
 * copies of a helper apart: lanes are grouped only if they agree on it */
#define SMX_ACTIVEMASK(key) __activemask()
#endif

typedef unsigned long long ull;
#define SMX_FULL 0xffffffffu
#if defined(SMX_HOSTSIM) && SMX_WARP == 1
#define SMX_BLOCK 1 /* sequential simulation: __syncthreads() is a no-op, so blocks have 1 thread */
#else
#define SMX_BLOCK (8 * SMX_WARP) /* 256 threads: 8 blocks/SM = 2048 resident threads */
#endif

#define SCAN_PER_THREAD 8
#define SCAN_TILE (SMX_BLOCK * SCAN_PER_THREAD)

enum { ST_OK = 0, ST_DEFER = 1, ST_LATE = 2, ST_DIRFULL = 3 };
enum { DIR_FOUND = 0, DIR_CREATED = 1, DIR_MISS = 2, DIR_FULL = 3 };

/* ------------------------------------------------------------------------------------------
 * small device helpers
 * ---------------------------------------------------------------------------------------- */

/* murmur3 finaliser: row ids are dense or strided in practice (SURVEY.md 8d scrambles them). */
__host__ __device__ __forceinline__ uint32_t smx_mix_row(uint32_t x) {
  x ^= x >> 16; x *= 0x85ebca6bu; x ^= x >> 13; x *= 0xc2b2ae35u; x ^= x >> 16;
  return x;
}
/* a different bijection for columns, so row and column placement are independent */
__host__ __device__ __forceinline__ uint32_t smx_mix_col(uint32_t y) {
  y ^= y >> 16; y *= 0x7feb352du; y ^= y >> 15; y *= 0x846ca68bu; y ^= y >> 16;
  return y;
}
/* and a third one for the owner rank, independent of the directory position */
__host__ __device__ __forceinline__ uint32_t smx_mix_owner(uint32_t x) {
  x *= 0x9E3779B1u; x ^= x >> 15; x *= 0x2C1B3C6Du; x ^= x >> 12; x *= 0x297A2D39u; x ^= x >> 15;
  return x;
}
__host__ __device__ __forceinline__ ull smx_splitmix64(ull z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

/* One 32-byte sector with a single 256-bit load that bypasses L1 (coherent at L2).  With the
 * L2::64B hint a miss fetches 64 bytes from DRAM instead of the whole 128-byte line (SASS
 * LDG.E.ENL2.LTC64B.256).  Measured on the full config-2 table (profiles/r2_summary.md): the speed is
 * the same with 64- and 128-byte fetches — the path is bound by the number of random DRAM touches,
 * not by their width — but the DRAM bytes per op drop (k_upsert 233 -> 173, k_get 322 -> 238 with the
 * hint on the buckets alone), so both the buckets and the 64-byte directory entries use it.  The
 * directory's probe order still visits both entries of a 128-byte line before moving on: the second
 * one is then a hit in the same DRAM page. */
#ifndef SMX_CELL_FETCH64
#define SMX_CELL_FETCH64 1
#endif
#ifndef SMX_HDR_FETCH64
#define SMX_HDR_FETCH64 1
#endif
template <bool FETCH64>
__device__ __forceinline__ void ld_sector_t(const void* p, ull c[4]) {
#ifdef SMX_HOSTSIM
  memcpy(c, p, 32);
#else
  if (FETCH64)
    asm volatile("ld.global.cg.L2::64B.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(c[0]), "=l"(c[1]), "=l"(c[2]), "=l"(c[3]) : "l"(p) : "memory");
  else
    asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(c[0]), "=l"(c[1]), "=l"(c[2]), "=l"(c[3]) : "l"(p) : "memory");
#endif
}
__device__ __forceinline__ void ld_sector(const void* p, ull c[4]) { ld_sector_t<SMX_CELL_FETCH64 != 0>(p, c); }
/* the same sector for a reader that will not come back to it: no L1 allocation, first in line for
 * eviction from L2 (SASS LDG.E.NA.EFL2.LTC64B.256).  The slice-ordered point reads use it for bucket
 * sectors, so that the single-use bucket lines do not push the slice's directory entries — which are
 * asked for again and again while the slice's queries run — out of L2. */
__device__ __forceinline__ void ld_sector_once(const void* p, ull c[4]) {
#ifdef SMX_HOSTSIM
  memcpy(c, p, 32);
#else
  asm volatile("ld.global.L1::no_allocate.L2::evict_first.L2::64B.v4.u64 {%0,%1,%2,%3}, [%4];"
               : "=l"(c[0]), "=l"(c[1]), "=l"(c[2]), "=l"(c[3]) : "l"(p) : "memory");
#endif
}
__device__ __forceinline__ void ld_hsector(const void* p, ull c[4]) { ld_sector_t<SMX_HDR_FETCH64 != 0>(p, c); }

struct Hdr {
  uint32_t key, meta;
  ull slots;
  uint32_t live, c0, t0inv, want;
};
__device__ __forceinline__ Hdr ld_hdr(const smx_row_t* e) {
  ull c[4];
  ld_hsector(e, c);
  Hdr h;
  h.key = (uint32_t)c[0];
  h.meta = (uint32_t)(c[0] >> 32);
  h.slots = c[1];
  h.live = (uint32_t)c[2];
  h.c0 = (uint32_t)(c[2] >> 32);
  h.t0inv = (uint32_t)c[3];
  h.want = (uint32_t)(c[3] >> 32);
  return h;
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x % SMX_WARP; }

/* warp-aggregated "give me a unique index": one atomic per converged group of threads */
__device__ __forceinline__ uint32_t agg_inc(uint32_t* ctr) {
  unsigned m = SMX_ACTIVEMASK(ctr);
  uint32_t lane = lane_id();
  int leader = __ffs(m) - 1;
  uint32_t base = 0;
  if ((int)lane == leader) base = atomicAdd(ctr, (uint32_t)__popc(m));
  base = __shfl_sync(m, base, leader);
  return base + (uint32_t)__popc(m & ((1u << lane) - 1u));
}
__device__ __forceinline__ void agg_inc64(ull* ctr) {
  unsigned m = SMX_ACTIVEMASK(ctr);
  if ((int)lane_id() == __ffs(m) - 1) atomicAdd(ctr, (ull)__popc(m));
}

/* rowlen: the reference returns its running `used` counter (src/smatrix.c:212-223).  With L =
 * number of columns != 0 in the row, used = L + d where the pair (S, d) follows the reference's
 * automaton: inserting a new column when L_before + d > S/2 doubles S (src/smatrix.c:346-348) and
 * recounts, which makes d = (column 0 is non-zero at that moment) (:397-402).  Because that rule is
 * monotone in L, the state can be caught up lazily from (S, d) as of any earlier moment as long
 * as z = (c0 != 0) did not change in between: the loop below gives the same (S, d) as stepping
 * through every insertion.  The table therefore only has to materialise the state right before z
 * flips (k_sync_rowlen); the hot update kernel never touches it. */
__host__ __device__ __forceinline__ uint32_t rowlen_catch_up(uint32_t meta, uint32_t live, bool z) {
  uint32_t slog = 4u + ((meta & SMX_META_SLOG) >> SMX_META_SLOG_SHIFT);
  uint32_t d = (meta & SMX_META_D) ? 1u : 0u;
  if (live) {
    const ull last = (ull)live - 1u; /* L_before of the latest insertion */
    while (slog < 36u && last + d > (1ull << (slog - 1u))) {
      ++slog;
      d = z ? 1u : d;
    }
  }
  return (meta & ~(SMX_META_SLOG | SMX_META_D)) | ((slog - 4u) << SMX_META_SLOG_SHIFT) | (d ? SMX_META_D : 0u);
}

/* ------------------------------------------------------------------------------------------
 * row directory: find or claim (replaces smatrix_cmap_lookup/probe/insert, :621-713)
 * ---------------------------------------------------------------------------------------- */
/* Probe order: both 64-byte entries of the home 128-byte line first (the line is already paid for
 * by the first probe), then the next line, and so on.  step -> position for home position p. */
__host__ __device__ __forceinline__ ull dir_probe_pos(ull p, ull step, ull mask) {
  return ((((p & ~1ull) + (step & ~1ull)) & mask) | ((p ^ step) & 1ull));
}

__device__ __forceinline__ int dir_find(const smx_view_t& V, uint32_t x, bool create,
                                        smx_row_t** out, Hdr* hdr) {
  const ull mask = V.dir_cap - 1;
  const ull home = smx_mix_row(x) & mask;
  for (ull step = 0; step < V.dir_cap; ++step) {
    const ull pos = dir_probe_pos(home, step, mask);
    smx_row_t* e = V.dir + pos;
    Hdr h = ld_hdr(e);
    if (h.meta & SMX_META_USED) {
      if (h.key == x) { *out = e; *hdr = h; return DIR_FOUND; }
      continue;
    }
    if (!create) return DIR_MISS;
    const uint32_t sl = (uint32_t)(pos >> V.slice_shift);
    uint32_t* slice = &V.ctl->slice_used[sl];
    if (step >= SMX_DIR_CREATE_STEPS || __ldcg(slice) >= V.slice_limit) return DIR_FULL;
    const ull fresh = (ull)x | ((ull)(SMX_META_USED | SMX_INLINE_LOG) << 32);
    ull old = atomicCAS((ull*)e, 0ull, fresh);
    if (old == 0ull) {
      /* occupancy counter of the slice: in a partitioned chunk nearly every row created at the same
       * time lives in the same slice, so the lanes that got here together add once for all of them */
      const unsigned grp = __match_any_sync(SMX_ACTIVEMASK(0), sl);
      if ((int)lane_id() == __ffs(grp) - 1) atomicAdd(slice, (uint32_t)__popc(grp));
      h.key = x; h.meta = SMX_META_USED | SMX_INLINE_LOG;
      h.slots = 0; h.live = 0; h.c0 = 0; h.t0inv = 0; h.want = 0;
      *out = e; *hdr = h;
      return DIR_CREATED;
    }
    if ((uint32_t)old == x && ((old >> 32) & SMX_META_USED)) {
      *out = e; *hdr = ld_hdr(e);
      return DIR_FOUND;
    }
    /* somebody claimed it for another row: keep probing */
  }
  return create ? DIR_FULL : DIR_MISS;
}

/* ------------------------------------------------------------------------------------------
 * column bucket: find-or-claim + value update (replaces rmap_probe/insert, :343-380, and the
 * arithmetic of set/incr/decr, :230,:241,:252)
 * ---------------------------------------------------------------------------------------- */
/* fire-and-forget add on a GLOBAL address: the bucket pointer comes out of a header word, so the
 * compiler would otherwise emit a generic ATOM (a round trip to L2) instead of a RED */
__device__ __forceinline__ void red_add(uint32_t* vp, uint32_t v) {
#ifdef SMX_HOSTSIM
  *vp += v;
#else
  asm volatile("red.global.add.u32 [%0], %1;" ::"l"(vp), "r"(v) : "memory");
#endif
}
template <int OP>
__device__ __forceinline__ void apply_value(uint32_t* vp, uint32_t v) {
  if (OP == SMX_OP_INCR) red_add(vp, v);
  else if (OP == SMX_OP_DECR) red_add(vp, 0u - v);
  else *(volatile uint32_t*)vp = 0u;
}

/* Two thresholds per bucket: above `soft` (1/2 load, the reference's own limit, src/smatrix.c:346)
 * the row asks for growth (SLOT_DONE_GROW) but keeps accepting new columns up to `hard` (7/8
 * load); only then is an op turned away (SLOT_FULL, re-run after the growth).  Final bucket sizes
 * are the same as with a single 1/2 limit, but ops are almost never deferred. */
enum { SLOT_FULL = 0, SLOT_DONE = 1, SLOT_DONE_GROW = 2 };
template <int OP>
__device__ __forceinline__ int slot_upsert(smx_row_t* e, const Hdr& h, uint32_t y, uint32_t v) {
  const uint32_t caplog = h.meta & SMX_META_CAPLOG;
  ull* base = (caplog == SMX_INLINE_LOG) ? (ull*)e->inl : (ull*)h.slots;
  const uint32_t nsec = 1u << (caplog - 2u);
  const uint32_t soft = (caplog == SMX_INLINE_LOG) ? 4u : (1u << (caplog - 1u));
  const uint32_t hard = (caplog == SMX_INLINE_LOG) ? 4u : (1u << caplog) - (1u << (caplog - 3u));
  const uint32_t init = (OP == SMX_OP_INCR) ? v : (OP == SMX_OP_DECR) ? (0u - v) : 0u;
  const ull fresh = (ull)y | ((ull)init << 32);
  uint32_t s = smx_mix_col(y) & (nsec - 1u);
  for (uint32_t probe = 0; probe < nsec; ++probe, s = (s + 1u) & (nsec - 1u)) {
    ull* sec = base + 4ull * s;
    ull c[4];
    ld_sector(sec, c);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if ((uint32_t)c[k] == y) { /* y != 0, so this is a live cell of ours */
        apply_value<OP>((uint32_t*)(sec + k) + 1, v);
        return SLOT_DONE;
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (c[k] != 0ull) continue;
      if (h.live >= hard) return SLOT_FULL;
      ull old = atomicCAS(sec + k, 0ull, fresh);
      if (old == 0ull) { /* new column */
        const uint32_t n = atomicAdd(&e->live, 1u) + 1u;
        return (n > soft && caplog < SMX_MAX_CAPLOG) ? SLOT_DONE_GROW : SLOT_DONE;
      }
      if ((uint32_t)old == y) {
        apply_value<OP>((uint32_t*)(sec + k) + 1, v);
        return SLOT_DONE;
      }
      /* claimed for another column meanwhile: try the next cell in probe order */
    }
  }
  return SLOT_FULL;
}

/* read-only probe: value of column y (y != 0) or 0 */
template <bool ONCE = false>
__device__ __forceinline__ uint32_t slot_find(const smx_row_t* e, const Hdr& h, uint32_t y,
                                              uint32_t** where) {
  const uint32_t caplog = h.meta & SMX_META_CAPLOG;
  const ull* base = (caplog == SMX_INLINE_LOG) ? (const ull*)e->inl : (const ull*)h.slots;
  const uint32_t nsec = 1u << (caplog - 2u);
  uint32_t s = smx_mix_col(y) & (nsec - 1u);
  for (uint32_t probe = 0; probe < nsec; ++probe, s = (s + 1u) & (nsec - 1u)) {
    const ull* sec = base + 4ull * s;
    ull c[4];
    if (ONCE) ld_sector_once(sec, c);
    else ld_sector(sec, c);
    bool hole = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if ((uint32_t)c[k] == y) {
        if (where) *where = (uint32_t*)(sec + k) + 1;
        return (uint32_t)(c[k] >> 32);
      }
      hole |= (c[k] == 0ull);
    }
    if (hole) break; /* cells fill in probe order and never empty again */
  }
  if (where) *where = nullptr;
  return 0u;
}

/* ------------------------------------------------------------------------------------------
 * K1+K2+K3: the update kernel
 * ---------------------------------------------------------------------------------------- */
/* `ord` is the op's index in the caller's input order (what "sequential application" refers to) */
template <int OP>
__device__ __forceinline__ int upsert_one(const smx_view_t& V, const smx_lists_t& S, int pass,
                                          uint32_t ord, uint32_t x, uint32_t y, uint32_t v) {
  smx_row_t* e;
  Hdr h;
  int r = dir_find(V, x, true, &e, &h);
  if (r == DIR_FULL) return ST_DIRFULL; /* counted per block by the caller */
  if (pass == SMX_PASS_COL0) {
    apply_value<OP>(&e->c0, v);
    /* column 0 of this row turns non-zero inside this batch: remember the first such op
     * (SURVEY.md Q1: rowlen depends on whether column 0 was non-zero at each virtual resize) */
    if (v != 0u && !(h.meta & SMX_META_ZC)) {
      atomicMax(&e->t0inv, ~ord);
      if (!(h.meta & SMX_META_T0P)) {
        uint32_t old = atomicOr(&e->meta, SMX_META_T0P);
        if (!(old & SMX_META_T0P)) S.t0rows[agg_inc(&V.ctl->n_t0)] = x;
      }
    }
    return ST_OK;
  }
  if (pass == SMX_PASS_EARLY && (h.meta & SMX_META_T0P)) {
    if (ord > ~h.t0inv) return ST_LATE; /* ordered after column 0 became non-zero */
  }
  const int r2 = slot_upsert<OP>(e, h, y, v);
  if (r2 == SLOT_DONE) return ST_OK;
  if (r2 == SLOT_FULL) atomicAdd(&e->want, 1u);
  if (!(h.meta & SMX_META_GROW)) { /* queue the row for growth, once per round */
    uint32_t old = atomicOr(&e->meta, SMX_META_GROW);
    if (!(old & SMX_META_GROW)) S.grow[agg_inc(&V.ctl->n_grow)] = (uint32_t)(e - V.dir);
  }
  return r2 == SLOT_FULL ? ST_DEFER : ST_OK;
}

#ifndef SMX_UPSERT_MIN_BLOCKS
#define SMX_UPSERT_MIN_BLOCKS 6 /* measured: 6 blocks (40 registers, no spills) beats 8 (32 registers, spills) on the whole build */
#endif
template <int OP>
__global__ void __launch_bounds__(SMX_BLOCK, SMX_UPSERT_MIN_BLOCKS)
k_upsert(smx_view_t V, smx_ops_t O, smx_lists_t S, int pass, const uint32_t* list, uint32_t m,
         int preagg) {
  /* ops that are turned away are staged per block and appended to the retry list with ONE global
   * atomic per block: in a round where most ops are refused (directory at its limit) per-warp
   * atomics on the same counter would serialise ~1 M times */
  __shared__ uint32_t s_defer[4 * SMX_BLOCK];
  __shared__ uint32_t s_ndefer, s_ndirfull, s_base;
  if (threadIdx.x == 0) { s_ndefer = 0u; s_ndirfull = 0u; }
  __syncthreads();
  const uint32_t lane = lane_id();
  const uint32_t stride = gridDim.x * blockDim.x;
  const uint32_t m_up = (m + (SMX_WARP - 1)) / SMX_WARP * SMX_WARP; /* whole warps stay in the loop */
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m_up; j += stride) {
    bool act = j < m;
    uint32_t pos = 0, ord = 0, x = 0, y = 0, v = 0;
    if (act) {
      pos = list ? list[j] : j;           /* position in the (possibly partitioned) batch arrays */
      ord = O.idx ? O.idx[pos] : pos;     /* index in the caller's input order */
      x = O.xs[pos];
      y = O.ys[pos];
      v = O.vs ? O.vs[pos] : O.v_const;
      if (!list) act = (pass == SMX_PASS_COL0) ? (y == 0u) : (y != 0u);
    }
    /* K1: collapse duplicate (x,y) keys inside the warp before they reach the table; the member
     * that comes first in input order leads (it decides EARLY vs LATE for the group) */
    bool lead = act;
    uint32_t vsum = v;
    unsigned peers = 1u << lane;
    int leader = (int)lane;
    if (preagg) {
      const ull k64 = ((ull)x << 32) | (ull)y;
      const unsigned valid = __ballot_sync(SMX_FULL, act);
      peers = __match_any_sync(SMX_FULL, k64) & valid;
      const bool dup = act && (peers != (1u << lane));
      if (__any_sync(SMX_FULL, dup)) {
        vsum = 0u;
        uint32_t best = 0xFFFFFFFFu, best_nz = 0xFFFFFFFFu;
        int leader_nz = -1;
        for (int src = 0; src < SMX_WARP; ++src) { /* segmented sum + arg-min of ord */
          const uint32_t tv = __shfl_sync(SMX_FULL, v, src);
          const uint32_t to = __shfl_sync(SMX_FULL, ord, src);
          if ((peers >> src) & 1u) {
            vsum += tv;
            if (to < best) { best = to; leader = src; }
            if (tv != 0u && to < best_nz) { best_nz = to; leader_nz = src; }
          }
        }
        /* column 0: t0 is the first op that makes the value non-zero, so a zero delta cannot lead */
        if (pass == SMX_PASS_COL0 && leader_nz >= 0) leader = leader_nz;
        if (OP == SMX_OP_SETZERO && pass == SMX_PASS_COL0) vsum = leader_nz >= 0 ? 1u : 0u; /* only "is any value non-zero" matters */
        lead = act && (leader == (int)lane);
      }
    }
    int status = ST_OK;
    if (lead) status = upsert_one<OP>(V, S, pass, ord, x, y, vsum);
    if (preagg) { /* members of a group share their leader's fate (retry / late pass) */
      __syncwarp();
      const int ls = __shfl_sync(SMX_FULL, status, act ? leader : (int)lane);
      if (act && !lead) status = ls;
    }
    if (act && (status == ST_DEFER || status == ST_DIRFULL)) {
      const uint32_t k = atomicAdd(&s_ndefer, 1u);
      if (k < 4u * SMX_BLOCK) s_defer[k] = pos;
      else S.defer_out[agg_inc(&V.ctl->n_defer)] = pos; /* cannot happen with the launch geometry; safe anyway */
      if (status == ST_DIRFULL) atomicAdd(&s_ndirfull, 1u);
    } else if (act && status == ST_LATE) {
      S.late[agg_inc(&V.ctl->n_late)] = pos;
    }
  }
  __syncthreads();
  const uint32_t nd = s_ndefer < 4u * SMX_BLOCK ? s_ndefer : 4u * SMX_BLOCK;
  if (threadIdx.x == 0 && nd) {
    s_base = atomicAdd(&V.ctl->n_defer, nd);
    if (s_ndirfull) atomicAdd(&V.ctl->n_dirfull, s_ndirfull);
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k < nd; k += blockDim.x) S.defer_out[s_base + k] = s_defer[k];
}

/* ------------------------------------------------------------------------------------------
 * K7: row growth (replaces smatrix_rmap_resize, :383-416)
 * ---------------------------------------------------------------------------------------- */
#define SMX_SMEM_MIGRATE_LOG 8u /* new buckets up to 2^8 cells are built in shared memory by k_migrate */
#define SMX_MID_SMEM_LOG 12u    /* ... and up to 2^12 cells by k_migrate_mid (one block per row) */

/* Plan the growth of the queued rows: new size class, and where the new bucket comes from — the
 * free list of that class (a bucket some other row vacated earlier) or fresh slab (an offset into
 * this round's region, handed out by a warp scan + one atomic per warp). */
__global__ void __launch_bounds__(SMX_BLOCK)
k_grow_plan(smx_view_t V, smx_lists_t S, uint32_t n_grow) {
  const uint32_t lane = lane_id();
  const uint32_t stride = gridDim.x * blockDim.x;
  const uint32_t n_up = (n_grow + (SMX_WARP - 1)) / SMX_WARP * SMX_WARP;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_up; j += stride) {
    const bool act = j < n_grow;
    ull bytes = 0, recycled = 0;
    uint32_t entry = 0, newlog = 0, caplog = 0;
    if (act) {
      entry = S.grow[j];
      Hdr h = ld_hdr(V.dir + entry);
      caplog = h.meta & SMX_META_CAPLOG;
      const ull need = 2ull * ((ull)h.live + (ull)h.want); /* load factor <= 1/2 after growth */
      /* small buckets grow x8 (4 -> 32 -> 256 cells: two re-placements on the way to a 256-cell
       * bucket instead of three, and less vacated memory); 256 -> 512 like the reference (:390); buckets of
       * 512 cells and more grow x4: rows that get there are a skewed workload's hot rows on their way up,
       * and every re-placement of a big row is millions of random atomics (config 3 spent a third of each
       * step on it with x2) — memory is the cheaper side of that trade on a 180 GB part */
      newlog = caplog + (caplog < 8u ? 3u : (caplog >= SMX_MID_LOG ? 2u : 1u));
      if (newlog > 8u && caplog < 8u) newlog = 8u;
      if (newlog < SMX_MIN_SLAB_LOG) newlog = SMX_MIN_SLAB_LOG;
      while ((1ull << newlog) < need && newlog < SMX_MAX_CAPLOG) ++newlog;
      /* take a vacated bucket of that class if there is one: one atomic per group of lanes that
       * want the same class (only pops run in this kernel; pushes happen in k_free_push) */
      {
        const unsigned grp = __match_any_sync(SMX_ACTIVEMASK(0), newlog);
        const int leader = __ffs(grp) - 1;
        const int cnt = __popc(grp), rank = __popc(grp & ((1u << lane) - 1u));
        int base = 0;
        if ((int)lane == leader) {
          base = atomicSub(&V.ctl->free_cnt[newlog], cnt);
          if (base < cnt) atomicAdd(&V.ctl->free_cnt[newlog], cnt - (base > 0 ? base : 0));
        }
        base = __shfl_sync(grp, base, leader);
        const int at = base - 1 - rank;
        if (at >= 0) recycled = (ull)V.ctl->free_stack[newlog][at];
      }
      bytes = recycled ? 0ull : (8ull << newlog);
      if (caplog > SMX_INLINE_LOG) { /* the bucket this row vacates, per class (sizes the stacks) */
        const unsigned grp = __match_any_sync(SMX_ACTIVEMASK(0), caplog);
        if ((int)lane == __ffs(grp) - 1) atomicAdd(&V.ctl->grow_from[caplog], (uint32_t)__popc(grp));
      }
    }
    ull incl = bytes; /* inclusive warp scan */
    for (uint32_t d = 1; d < SMX_WARP; d <<= 1) {
      ull t = __shfl_up_sync(SMX_FULL, incl, d);
      if (lane >= d) incl += t;
    }
    const ull total = __shfl_sync(SMX_FULL, incl, SMX_WARP - 1);
    ull base = 0;
    if (lane == 0 && total) base = atomicAdd(&V.ctl->plan_bytes, total);
    base = __shfl_sync(SMX_FULL, base, 0);
    if (act) {
      smx_plan_t p;
      p.entry = entry;
      p.newlog = newlog;
      p.off = recycled ? (SMX_PLAN_RECYCLED | recycled) : (base + incl - bytes);
      S.plan[j] = p;
      if (recycled) agg_inc(&V.ctl->n_recycled);
      /* which kernel re-places the row: old buckets of >= 512 cells whose NEW bucket fits 32 KB of shared
       * memory go to one block each (k_migrate_mid); anything bigger is filled in place by the whole grid
       * (k_migrate_big); the rest (old < 512 cells) by one warp (k_migrate) */
      const bool by_grid = caplog >= SMX_BIG_LOG || (caplog >= SMX_MID_LOG && newlog > SMX_MID_SMEM_LOG);
      if (by_grid) S.big[agg_inc(&V.ctl->n_big)] = j;
      else if (caplog >= SMX_MID_LOG) S.mid[agg_inc(&V.ctl->n_mid)] = j;
      /* fresh buckets that are filled in place (global CAS) need a zeroed region */
      const bool in_place = by_grid || (caplog < SMX_MID_LOG && newlog > SMX_SMEM_MIGRATE_LOG);
      if (in_place && !recycled) agg_inc64(&V.ctl->need_zero);
    }
  }
}

/* Recycle the buckets the planned rows are about to vacate: push their addresses on the stack of
 * their size class.  Runs after k_grow_plan (which only pops) and before the re-placement kernels
 * (the header still holds the old bucket); nothing pops again before the next round's plan. */
__global__ void __launch_bounds__(SMX_BLOCK)
k_free_push(smx_view_t V, smx_lists_t S, uint32_t n_grow) {
  const uint32_t lane = lane_id();
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_grow; j += gridDim.x * blockDim.x) {
    const Hdr h = ld_hdr(V.dir + S.plan[j].entry);
    const uint32_t caplog = h.meta & SMX_META_CAPLOG;
    if (caplog <= SMX_INLINE_LOG) continue;
    const unsigned grp = __match_any_sync(SMX_ACTIVEMASK(0), caplog);
    const int leader = __ffs(grp) - 1;
    int base = 0;
    if ((int)lane == leader) base = atomicAdd(&V.ctl->free_cnt[caplog], __popc(grp));
    base = __shfl_sync(grp, base, leader);
    V.ctl->free_stack[caplog][base + __popc(grp & ((1u << lane) - 1u))] = h.slots;
  }
}

/* place a whole cell into a zeroed / partially filled bucket (keys are unique) */
__device__ __forceinline__ void place_cell(ull* base, uint32_t caplog, ull cell) {
  const uint32_t nsec = 1u << (caplog - 2u);
  uint32_t s = smx_mix_col((uint32_t)cell) & (nsec - 1u);
  for (uint32_t probe = 0; probe < nsec; ++probe, s = (s + 1u) & (nsec - 1u)) {
    ull* sec = base + 4ull * s;
    ull c[4];
    ld_sector(sec, c);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (c[k] != 0ull) continue;
      if (atomicCAS(sec + k, 0ull, cell) == 0ull) return;
    }
  }
}
/* the same, into a bucket under construction in shared memory */
__device__ __forceinline__ void place_cell_smem(ull* sb, uint32_t nsec, ull c) {
  uint32_t sidx = smx_mix_col((uint32_t)c) & (nsec - 1u);
  for (bool placed = false; !placed; sidx = (sidx + 1u) & (nsec - 1u))
    for (int k = 0; k < 4 && !placed; ++k)
      placed = (atomicCAS(&sb[4u * sidx + k], 0ull, c) == 0ull); /* same probe order as slot_upsert */
}

__device__ __forceinline__ ull* plan_bucket(const smx_plan_t& p, char* region) {
  return (p.off & SMX_PLAN_RECYCLED) ? (ull*)(p.off & ~SMX_PLAN_RECYCLED) : (ull*)(region + p.off);
}

__device__ __forceinline__ void finish_growth(smx_row_t* e, const Hdr& h, ull* nb, uint32_t newlog) {
  e->slots = (ull)nb;
  e->want = 0u;
  e->meta = (h.meta & ~(SMX_META_CAPLOG | SMX_META_GROW)) | newlog;
}

/* one warp per growing row with a small old bucket (< 2^SMX_MID_LOG cells).  New buckets of up to
 * 2^SMX_SMEM_MIGRATE_LOG cells — the bulk of all growth events — are built in shared memory and
 * written out as whole lines (streaming); larger ones are filled in place with global CAS. */
__global__ void __launch_bounds__(SMX_BLOCK)
k_migrate(smx_view_t V, smx_lists_t S, uint32_t n_grow, char* region) {
  __shared__ ull sbuf[SMX_BLOCK / SMX_WARP][1u << SMX_SMEM_MIGRATE_LOG];
  const uint32_t lane = lane_id();
  const uint32_t wib = threadIdx.x / SMX_WARP;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t j = warp; j < n_grow; j += nwarps) {
    const smx_plan_t p = S.plan[j];
    smx_row_t* e = V.dir + p.entry;
    const Hdr h = ld_hdr(e);
    const uint32_t caplog = h.meta & SMX_META_CAPLOG;
    if (caplog >= SMX_MID_LOG) continue;
    ull* ob = (caplog == SMX_INLINE_LOG) ? (ull*)e->inl : (ull*)h.slots;
    ull* nb = plan_bucket(p, region);
    const uint32_t cap = 1u << caplog;
    if (p.newlog <= SMX_SMEM_MIGRATE_LOG) {
      ull* sb = sbuf[wib];
      const uint32_t ncap = 1u << p.newlog, nsec = ncap >> 2;
      for (uint32_t i = lane; i < ncap; i += SMX_WARP) sb[i] = 0ull;
      __syncwarp();
      for (uint32_t s0 = lane; s0 < cap; s0 += SMX_WARP) {
        const ull c = ob[s0];
        if (c != 0ull) place_cell_smem(sb, nsec, c);
      }
      __syncwarp();
      for (uint32_t i = lane; i < ncap; i += SMX_WARP) nb[i] = sb[i];
    } else {
      for (uint32_t s0 = lane; s0 < cap; s0 += SMX_WARP) {
        const ull c = ob[s0];
        if (c != 0ull) place_cell(nb, p.newlog, c);
      }
    }
    __syncwarp();
    if (lane == 0) finish_growth(e, h, nb, p.newlog);
  }
}

/* mid-size rows (old bucket 2^SMX_MID_LOG .. 2^(SMX_BIG_LOG-1) cells): one BLOCK per row.  New
 * buckets of up to 2^SMX_MID_SMEM_LOG cells are built in shared memory (32 KB) and streamed out;
 * larger ones are filled in place.  The vacated bucket is zeroed (it goes to the free list). */
__global__ void __launch_bounds__(SMX_BLOCK)
k_migrate_mid(smx_view_t V, smx_lists_t S, uint32_t n_mid, char* region) {
  __shared__ ull sb[1u << SMX_MID_SMEM_LOG];
  for (uint32_t j = blockIdx.x; j < n_mid; j += gridDim.x) {
    const smx_plan_t p = S.plan[S.mid[j]];
    smx_row_t* e = V.dir + p.entry;
    const Hdr h = ld_hdr(e);
    const uint32_t caplog = h.meta & SMX_META_CAPLOG;
    ull* ob = (ull*)h.slots;
    ull* nb = plan_bucket(p, region);
    const uint32_t cap = 1u << caplog;
    { /* k_grow_plan only sends rows here whose new bucket fits the shared-memory buffer */
      const uint32_t ncap = 1u << p.newlog, nsec = ncap >> 2;
      for (uint32_t i = threadIdx.x; i < ncap; i += blockDim.x) sb[i] = 0ull;
      __syncthreads();
      for (uint32_t s0 = threadIdx.x; s0 < cap; s0 += blockDim.x) {
        const ull c = ob[s0];
        ob[s0] = 0ull;
        if (c != 0ull) place_cell_smem(sb, nsec, c);
      }
      __syncthreads();
      for (uint32_t i = threadIdx.x; i < ncap; i += blockDim.x) nb[i] = sb[i];
    }
    __syncthreads(); /* every thread has read the header and finished with sb */
    if (threadIdx.x == 0) finish_growth(e, h, nb, p.newlog);
    __syncthreads();
  }
}

/* big rows: the whole grid (x) re-places one row (y) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_migrate_big(smx_view_t V, smx_lists_t S, uint32_t big_first, char* region) {
  const smx_plan_t p = S.plan[S.big[big_first + blockIdx.y]];
  smx_row_t* e = V.dir + p.entry;
  const Hdr h = ld_hdr(e);
  const uint32_t caplog = h.meta & SMX_META_CAPLOG;
  ull* ob = (ull*)h.slots;
  ull* nb = plan_bucket(p, region);
  const ull cap = 1ull << caplog;
  for (ull s = blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (ull)gridDim.x * blockDim.x) {
    const ull c = ob[s];
    ob[s] = 0ull; /* the vacated bucket goes to the free list zeroed */
    if (c != 0ull) place_cell(nb, p.newlog, c);
  }
}
__global__ void k_migrate_big_finish(smx_view_t V, smx_lists_t S, uint32_t n_big, char* region) {
  for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < n_big; b += gridDim.x * blockDim.x) {
    const smx_plan_t p = S.plan[S.big[b]];
    smx_row_t* e = V.dir + p.entry;
    const Hdr h = ld_hdr(e);
    finish_growth(e, h, plan_bucket(p, region), p.newlog);
  }
}

/* Big rows, built instead of filled: the new bucket is cut into tiles of MIG_TILE sectors; a block zeroes a
 * tile in shared memory, streams in the old sectors whose cells can have their new home in it (old home =
 * new home mod old size; plus the few sectors behind that range that linear probing pushed cells into),
 * places the cells with shared-memory CAS in the usual probe order and streams the tile out — no global
 * atomic, no zeroed target.  A cell whose probe run reaches the end of its tile goes to a small spill
 * list and is inserted with the ordinary global probe (place_cell) once all tiles are written: from its
 * home to the tile's end every sector is full, so the probe invariant holds.  k_migrate_big (one global
 * CAS per cell, 80 % of the random-atomic rate) stays as the reference path (SMATRIX_MIGRATE_TILES=0). */
#ifndef MIG_TILE_LOG
#define MIG_TILE_LOG 10u /* the CPU tests also build a variant with tiny tiles, where cells spill all the time */
#endif
#define MIG_TILE (1u << MIG_TILE_LOG) /* sectors per tile: 4096 cells = 32 KB */
__device__ __forceinline__ bool sector_is_full(const ull* sec) {
  ull c[4];
  ld_sector(sec, c);
  return c[0] != 0ull && c[1] != 0ull && c[2] != 0ull && c[3] != 0ull;
}
/* the cells of one old sector whose new home lies in the tile [t0, t0 + MIG_TILE) go into the tile */
__device__ __forceinline__ void tile_take_sector(const ull* sec, ull* sm, uint32_t t0, uint32_t n_new, uint32_t j,
                                                 smx_ctl_t* ctl, ull* spill, uint32_t spill_cap) {
  ull c[4];
  ld_sector(sec, c);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (c[k] == 0ull) continue;
    const uint32_t hn = smx_mix_col((uint32_t)c[k]) & (n_new - 1u);
    if (hn - t0 >= MIG_TILE) continue; /* its home is in another tile */
    bool placed = false;
    for (uint32_t q = hn - t0; q < MIG_TILE && !placed; ++q) /* same probe order as slot_upsert, inside the tile */
      for (int w = 0; w < 4 && !placed; ++w) placed = (atomicCAS(&sm[4u * q + w], 0ull, c[k]) == 0ull);
    if (!placed) { /* the run of full sectors reaches the end of the tile: global probe later */
      const uint32_t at = atomicAdd(&ctl->n_spill, 1u);
      if (at < spill_cap) { spill[2ull * at] = (ull)j; spill[2ull * at + 1] = c[k]; }
    }
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_migrate_tiles(smx_view_t V, smx_lists_t S, uint32_t big_first, char* region, ull* spill, uint32_t spill_cap) {
  __shared__ ull sm[4u * MIG_TILE];
  __shared__ uint32_t s_stop;
  const uint32_t j = S.big[big_first + blockIdx.y];
  const smx_plan_t p = S.plan[j];
  const smx_row_t* e = V.dir + p.entry;
  const Hdr h = ld_hdr(e);
  const ull* ob = (const ull*)h.slots;
  ull* nb = plan_bucket(p, region);
  const uint32_t n_old = 1u << ((h.meta & SMX_META_CAPLOG) - 2u), n_new = 1u << (p.newlog - 2u); /* sectors */
  const uint32_t n_tiles = n_new >> MIG_TILE_LOG, mask = n_old - 1u;
  const uint32_t len = n_old < MIG_TILE ? n_old : MIG_TILE;
  for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const uint32_t t0 = t << MIG_TILE_LOG;
    const uint32_t r0 = n_old < MIG_TILE ? 0u : (t0 & mask); /* old home = new home mod old size */
    for (uint32_t i = threadIdx.x; i < 4u * MIG_TILE; i += blockDim.x) sm[i] = 0ull;
    __syncthreads();
    for (uint32_t s = threadIdx.x; s < len; s += blockDim.x)
      tile_take_sector(ob + 4ull * ((r0 + s) & mask), sm, t0, n_new, j, V.ctl, spill, spill_cap);
    /* cells with a home in the range that linear probing pushed behind it: they can only sit in the
     * sectors that follow as long as the sector before is full.  Usually none or a handful — but a row
     * that grows because ops were turned away is 7/8 full and has runs of hundreds of full sectors, so
     * the block walks them together: 32 sectors first, then 256 at a time, up to the first hole */
    if (len < n_old) {
      for (uint32_t base = len, step = SMX_WARP; base < n_old; base += step, step = blockDim.x) {
        if (threadIdx.x == 0) s_stop = 0xFFFFFFFFu;
        __syncthreads();
        const uint32_t s = base + threadIdx.x;
        const bool in = threadIdx.x < step && s < n_old;
        if (in && !sector_is_full(ob + 4ull * ((r0 + s - 1u) & mask))) atomicMin(&s_stop, s);
        __syncthreads();
        const uint32_t stop = s_stop; /* the first sector whose predecessor has a hole: nothing of ours from there on */
        if (in && s < stop) tile_take_sector(ob + 4ull * ((r0 + s) & mask), sm, t0, n_new, j, V.ctl, spill, spill_cap);
        __syncthreads();
        if (stop != 0xFFFFFFFFu) break;
      }
    }
    __syncthreads();
    ull* out = nb + 4ull * t0;
    for (uint32_t i = threadIdx.x; i < 4u * MIG_TILE; i += blockDim.x) out[i] = sm[i];
    __syncthreads();
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_spill_insert(smx_view_t V, smx_lists_t S, char* region, const ull* spill, uint32_t n_spill) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_spill; i += gridDim.x * blockDim.x) {
    const smx_plan_t p = S.plan[(uint32_t)spill[2ull * i]];
    place_cell(plan_bucket(p, region), p.newlog, spill[2ull * i + 1]);
  }
}
/* the vacated buckets of the big rows go to the free lists zeroed (grid x strides over one row, y) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_zero_old_big(smx_view_t V, smx_lists_t S, uint32_t big_first) {
  const smx_plan_t p = S.plan[S.big[big_first + blockIdx.y]];
  const Hdr h = ld_hdr(V.dir + p.entry);
  ull* ob = (ull*)h.slots;
  const ull cap = 1ull << (h.meta & SMX_META_CAPLOG);
  for (ull s = blockIdx.x * (ull)blockDim.x + threadIdx.x; s < cap; s += (ull)gridDim.x * blockDim.x) ob[s] = 0ull;
}

/* ------------------------------------------------------------------------------------------
 * directory growth (replaces smatrix_cmap_resize, :715-741): re-place every entry into `to`
 * ---------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(SMX_BLOCK) k_dir_rehash(smx_view_t from, smx_view_t to) {
  const ull mask = to.dir_cap - 1;
  uint32_t far = 0; /* largest probe step of this thread's rows: the host refuses a shrink that puts a row beyond
                       dir_find's create limit */
  for (ull pos = blockIdx.x * blockDim.x + threadIdx.x; pos < from.dir_cap;
       pos += (ull)gridDim.x * blockDim.x) {
    const smx_row_t* o = from.dir + pos;
    ull a[4], b[4];
    ld_hsector(o, a);
    if (!((a[0] >> 32) & SMX_META_USED)) continue;
    ld_hsector((const char*)o + 32, b);
    const ull home = smx_mix_row((uint32_t)a[0]) & mask;
    for (ull step = 0;; ++step) { /* same probe order as dir_find */
      const ull q = dir_probe_pos(home, step, mask);
      ull* dst = (ull*)(to.dir + q);
      if (atomicCAS(dst, 0ull, a[0]) == 0ull) {
        dst[1] = a[1]; dst[2] = a[2]; dst[3] = a[3];
        dst[4] = b[0]; dst[5] = b[1]; dst[6] = b[2]; dst[7] = b[3];
        atomicAdd(&to.ctl->slice_used[q >> to.slice_shift], 1u);
        if (step > far) far = step < 0xFFFFFFFFull ? (uint32_t)step : 0xFFFFFFFFu;
        break;
      }
    }
  }
  if (far) atomicMax(&to.ctl->dir_probe_max, far);
}

/* between the EARLY and LATE passes: column 0 of these rows turns non-zero HERE in input order, so
 * bring their (S, d) up to date with z = 0 for the columns inserted so far */
__global__ void k_sync_rowlen(smx_view_t V, const uint32_t* rows, uint32_t n) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    if (dir_find(V, rows[j], false, &e, &h) != DIR_FOUND) continue;
    e->meta = rowlen_catch_up(h.meta, h.live, (h.meta & SMX_META_ZC) != 0u);
  }
}

/* end of a chunk: column 0 of these rows is now (and stays) non-zero */
__global__ void k_finalize_t0(smx_view_t V, const uint32_t* t0rows, uint32_t n) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    if (dir_find(V, t0rows[j], false, &e, &h) != DIR_FOUND) continue;
    e->t0inv = 0u;
    e->meta = (h.meta & ~SMX_META_T0P) | SMX_META_ZC;
  }
}

/* ------------------------------------------------------------------------------------------
 * set: last writer in input order wins.  After k_upsert<SETZERO> created every cell and stored
 * 0 in it, k_set_max leaves max(i)+1 in the cell, k_set_mark finds the op that holds it and
 * k_set_commit lets that op store its value.
 * ---------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(SMX_BLOCK) k_set_max(smx_view_t V, smx_ops_t O, ull* addrs) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < O.n; i += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    uint32_t* vp = nullptr;
    if (dir_find(V, O.xs[i], false, &e, &h) == DIR_FOUND) {
      const uint32_t y = O.ys[i];
      if (y == 0u) vp = &e->c0;
      else slot_find(e, h, y, &vp);
    }
    const uint32_t ord = O.idx ? O.idx[i] : i;
    if (vp) atomicMax(vp, ord + 1u);
    addrs[i] = (ull)vp;
  }
}
/* read-only: keep the cell address only for the op that holds the maximum (no value is stored
 * in this kernel, so a stored VALUE can never be mistaken for somebody's index + 1) */
__global__ void __launch_bounds__(SMX_BLOCK) k_set_mark(smx_ops_t O, ull* addrs) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < O.n; i += gridDim.x * blockDim.x) {
    const uint32_t* vp = (const uint32_t*)addrs[i];
    const uint32_t ord = O.idx ? O.idx[i] : i;
    if (vp && __ldcg(vp) != ord + 1u) addrs[i] = 0ull;
  }
}
__global__ void __launch_bounds__(SMX_BLOCK) k_set_commit(smx_ops_t O, const ull* addrs) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < O.n; i += gridDim.x * blockDim.x) {
    uint32_t* vp = (uint32_t*)addrs[i];
    if (vp) *vp = O.vs ? O.vs[i] : O.v_const;
  }
}


/* ------------------------------------------------------------------------------------------
 * N1: exact per-op return values of an incr / decr batch (SURVEY.md 8f): out[i] = value of the
 * cell right after op i when the batch is applied in input order (src/smatrix.c:241,:252).
 * The chunk is applied by the ordinary path first; then: (1) k_find_addr locates every op's cell,
 * (2) a STABLE sort of the op indices by cell address (input order is kept inside a cell's group),
 * (3) a segmented inclusive scan over the REVERSED sorted sequence gives, per op, the sum of its
 * own and all later deltas of the same cell, (4) out[i] = final - (that sum - own delta).
 * ---------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(SMX_BLOCK) k_find_addr(smx_view_t V, smx_ops_t O, ull* addrs, uint32_t* iota) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < O.n; i += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    uint32_t* vp = nullptr;
    if (dir_find(V, O.xs[i], false, &e, &h) == DIR_FOUND) {
      const uint32_t y = O.ys[i];
      if (y == 0u) vp = &e->c0;
      else slot_find(e, h, y, &vp);
    }
    addrs[i] = (ull)vp;
    iota[i] = i;
  }
}
/* reversed sorted order: element q <-> sorted position n-1-q; flag = first of its group in that order */
__global__ void __launch_bounds__(SMX_BLOCK)
k_out_gather(smx_ops_t O, int negate, const ull* sorted_addr, const uint32_t* sorted_idx, ull* seg) {
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < O.n; q += gridDim.x * blockDim.x) {
    const uint32_t p = O.n - 1u - q;
    const uint32_t i = sorted_idx[p];
    uint32_t v = O.vs ? O.vs[i] : O.v_const;
    if (negate) v = 0u - v;
    const bool head = (p == O.n - 1u) || (sorted_addr[p + 1] != sorted_addr[p]);
    seg[q] = (ull)v | ((ull)(head ? 1u : 0u) << 32);
  }
}
/* segmented inclusive scan of (flag, value) pairs: value = low 32 bits (mod 2^32), flag = bit 32 */
__device__ __forceinline__ ull seg_op(ull a, ull b) { /* a then b */
  return (b >> 32) ? b : (((a >> 32) << 32) | (uint32_t)((uint32_t)a + (uint32_t)b));
}
__global__ void __launch_bounds__(SMX_BLOCK) k_seg_tile(const ull* seg, uint32_t n, ull* tile_agg) {
  __shared__ ull sh[SMX_BLOCK];
  const ull first = (ull)blockIdx.x * SCAN_TILE + (ull)threadIdx.x * SCAN_PER_THREAD;
  ull acc = 0;
  for (int k = 0; k < SCAN_PER_THREAD; ++k)
    if (first + k < n) acc = seg_op(acc, seg[first + k]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    ull t = 0;
    for (uint32_t k = 0; k < blockDim.x; ++k) t = seg_op(t, sh[k]);
    tile_agg[blockIdx.x] = t;
  }
}
__global__ void k_seg_tiles(ull* tile_agg, uint32_t n_tiles) { /* one thread: exclusive carry per tile */
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ull run = 0;
    for (uint32_t t = 0; t < n_tiles; ++t) {
      const ull a = tile_agg[t];
      tile_agg[t] = run;
      run = seg_op(run, a);
    }
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_seg_apply(ull* seg, uint32_t n, const ull* tile_carry) {
  __shared__ ull sh[SMX_BLOCK];
  const ull first = (ull)blockIdx.x * SCAN_TILE + (ull)threadIdx.x * SCAN_PER_THREAD;
  ull c[SCAN_PER_THREAD];
  ull acc = 0;
  for (int k = 0; k < SCAN_PER_THREAD; ++k) {
    c[k] = (first + k < n) ? seg[first + k] : 0ull;
    acc = seg_op(acc, c[k]);
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    ull run = tile_carry[blockIdx.x] & 0xFFFFFFFFull; /* a carry never carries a flag into the tile */
    for (uint32_t k = 0; k < blockDim.x; ++k) {
      const ull v = sh[k];
      sh[k] = run;
      run = seg_op(run, v);
    }
  }
  __syncthreads();
  ull run = sh[threadIdx.x] & 0xFFFFFFFFull;
  for (int k = 0; k < SCAN_PER_THREAD; ++k) {
    if (first + k < n) {
      run = seg_op(run, c[k]);
      seg[first + k] = run;
      run &= 0xFFFFFFFFull;
    }
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_out_write(smx_ops_t O, int negate, const ull* sorted_addr, const uint32_t* sorted_idx, const ull* seg,
            uint32_t* out) {
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < O.n; q += gridDim.x * blockDim.x) {
    const uint32_t p = O.n - 1u - q;
    const uint32_t i = sorted_idx[p];
    uint32_t v = O.vs ? O.vs[i] : O.v_const;
    if (negate) v = 0u - v;
    const uint32_t* vp = (const uint32_t*)sorted_addr[p];
    const uint32_t fin = vp ? __ldcg(vp) : 0u;
    out[i] = fin - ((uint32_t)seg[q] - v); /* final minus the deltas applied after op i */
  }
}
__global__ void __launch_bounds__(SMX_BLOCK) k_fill_out(smx_ops_t O, uint32_t* out) { /* set returns its value */
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < O.n; i += gridDim.x * blockDim.x)
    out[i] = O.vs ? O.vs[i] : O.v_const;
}

/* ------------------------------------------------------------------------------------------
 * K4 / K5: point reads
 * ---------------------------------------------------------------------------------------- */
__device__ __forceinline__ uint32_t get_one(const smx_view_t& V, uint32_t x, uint32_t y, bool once) {
  smx_row_t* e;
  Hdr h;
  if (dir_find(V, x, false, &e, &h) != DIR_FOUND) return 0u;
  if (y == 0u) return h.c0;
  return once ? slot_find<true>(e, h, y, nullptr) : slot_find<false>(e, h, y, nullptr);
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_get(smx_view_t V, const uint32_t* xs, const uint32_t* ys, uint32_t n, uint32_t* out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = get_one(V, xs[i], ys[i], false);
}
/* The look-up of SLICE-ORDERED queries.  Not a resident grid with a stride loop: blocks of a resident
 * grid drift apart (an SM that is a few per cent faster is several slices ahead after the ~200
 * iterations of a 2^26-query batch), and then the directory entries of many slices compete for L2
 * at once.  One block per GET_TILE consecutive queries, dispatched in order as earlier blocks retire
 * (like k_upsert), keeps all resident blocks inside a window of ~1 M queries = one or two slices. */
#define GET_TILE_ITEMS 4
template <bool ONCE>
__global__ void __launch_bounds__(SMX_BLOCK, 8)
k_get_tiled(smx_view_t V, const uint32_t* xs, const uint32_t* ys, uint32_t n, uint32_t* out) {
  const ull base = (ull)blockIdx.x * (GET_TILE_ITEMS * SMX_BLOCK);
  uint32_t x[GET_TILE_ITEMS], y[GET_TILE_ITEMS];
#pragma unroll
  for (int k = 0; k < GET_TILE_ITEMS; ++k) {
    const ull i = base + (ull)k * SMX_BLOCK + threadIdx.x;
    x[k] = i < n ? xs[i] : 0u;
    y[k] = i < n ? ys[i] : 0u;
  }
#pragma unroll
  for (int k = 0; k < GET_TILE_ITEMS; ++k) {
    const ull i = base + (ull)k * SMX_BLOCK + threadIdx.x;
    if (i < n) out[i] = get_one(V, x[k], y[k], ONCE);
  }
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_rowlen(smx_view_t V, const uint32_t* xs, uint32_t n, uint32_t* out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    uint32_t len = 0u;
    if (dir_find(V, xs[i], false, &e, &h) == DIR_FOUND) { /* the reference's `used` (Q1) */
      const uint32_t m2 = rowlen_catch_up(h.meta, h.live, (h.meta & (SMX_META_ZC | SMX_META_T0P)) != 0u);
      len = h.live + ((m2 & SMX_META_D) ? 1u : 0u);
    }
    out[i] = len;
  }
}

/* ------------------------------------------------------------------------------------------
 * K6: getrow for a batch of rows -> CSR (replaces smatrix_getrow, src/smatrix.c:189-210, for whole
 * batches).  k_row_counts resolves every row ONCE (directory probe) and leaves, besides the pair
 * count, an `info` word per row (directory index | log2 capacity << 32, ~0 = no such row) that the
 * compaction kernels start from; the exclusive scan of the counts gives the CSR offsets; then three
 * compaction kernels, by bucket size:
 *   k_getrow_inline  rows that never left their directory entry (<= 4 cells): one THREAD per row
 *   k_getrow_fill    16 .. 1024 cells: one WARP per row, 16-byte loads, the live cells of a 64-cell
 *                    step are compacted with a warp prefix-sum, staged in shared memory and written
 *                    out as one contiguous run
 *   k_getrow_chunks  >= 2048 cells: the bucket is cut into 2048-cell chunks that all blocks of the
 *                    grid share; a chunk is compacted in shared memory (block prefix-sum), reserves
 *                    its output range with one atomic on the row's cursor and streams out
 * ---------------------------------------------------------------------------------------- */
#define SMX_GETROW_BIG_LOG 11u
#define SMX_NO_ROW 0xFFFFFFFFFFFFFFFFull
__global__ void __launch_bounds__(SMX_BLOCK)
k_row_counts(smx_view_t V, const uint32_t* xs, uint32_t n, uint32_t* counts, ull* info, uint32_t* big_list,
             uint32_t* big_counter) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    uint32_t c = 0u;
    ull inf = SMX_NO_ROW;
    if (dir_find(V, xs[i], false, &e, &h) == DIR_FOUND) {
      c = h.live + (h.c0 != 0u ? 1u : 0u);
      const uint32_t caplog = h.meta & SMX_META_CAPLOG;
      inf = (ull)(e - V.dir) | ((ull)caplog << 32);
      if (big_list && caplog >= SMX_GETROW_BIG_LOG) big_list[agg_inc(big_counter)] = i;
    }
    counts[i] = c;
    if (info) info[i] = inf;
  }
}

/* exclusive scan of one value per thread over the block (warp shuffles + one shared-memory hop);
 * returns the exclusive prefix, *total = the block's sum */
__device__ __forceinline__ ull block_exclusive_scan(ull v, ull* total) {
  __shared__ ull s_warp[SMX_BLOCK / SMX_WARP + 1];
  const uint32_t lane = lane_id(), wib = threadIdx.x / SMX_WARP;
  ull incl = v;
  for (uint32_t d = 1; d < SMX_WARP; d <<= 1) {
    const ull t = __shfl_up_sync(SMX_FULL, incl, d);
    if (lane >= d) incl += t;
  }
  __syncthreads(); /* s_warp may still be read from a previous call */
  if (lane == SMX_WARP - 1) s_warp[wib] = incl;
  __syncthreads();
  if (wib == 0) {
    const uint32_t nw = blockDim.x / SMX_WARP;
    ull w = lane < nw ? s_warp[lane] : 0ull, wi = w;
    for (uint32_t d = 1; d < SMX_WARP; d <<= 1) {
      const ull t = __shfl_up_sync(SMX_FULL, wi, d);
      if (lane >= d) wi += t;
    }
    if (lane < nw) s_warp[lane] = wi - w;
    if (lane == nw - 1) s_warp[nw] = wi;
  }
  __syncthreads();
  *total = s_warp[blockDim.x / SMX_WARP];
  return s_warp[wib] + incl - v;
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_scan_tile_sums(const uint32_t* counts, uint32_t n, ull* tile_sums) {
  const ull first = (ull)blockIdx.x * SCAN_TILE + (ull)threadIdx.x * SCAN_PER_THREAD;
  ull s = 0;
  for (int k = 0; k < SCAN_PER_THREAD; ++k)
    if (first + k < n) s += counts[first + k];
  ull total;
  block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
/* one block: exclusive scan of the tile sums, total goes to offsets[n] */
__global__ void __launch_bounds__(SMX_BLOCK)
k_scan_tiles(ull* tile_sums, uint32_t n_tiles, ull base, ull* offsets, uint32_t n) {
  ull carry = base;
  for (uint32_t t0 = 0; t0 < n_tiles; t0 += blockDim.x) {
    const uint32_t t = t0 + threadIdx.x;
    const ull v = (t < n_tiles) ? tile_sums[t] : 0ull;
    ull total;
    const ull excl = block_exclusive_scan(v, &total);
    if (t < n_tiles) tile_sums[t] = carry + excl;
    carry += total;
  }
  if (threadIdx.x == 0) offsets[n] = carry;
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_scan_apply(const uint32_t* counts, uint32_t n, const ull* tile_sums, ull* offsets) {
  const ull first = (ull)blockIdx.x * SCAN_TILE + (ull)threadIdx.x * SCAN_PER_THREAD;
  uint32_t c[SCAN_PER_THREAD];
  ull s = 0;
  for (int k = 0; k < SCAN_PER_THREAD; ++k) {
    c[k] = (first + k < n) ? counts[first + k] : 0u;
    s += c[k];
  }
  ull total;
  ull run = tile_sums[blockIdx.x] + block_exclusive_scan(s, &total);
  for (int k = 0; k < SCAN_PER_THREAD; ++k) {
    if (first + k < n) offsets[first + k] = run;
    run += c[k];
  }
}

/* 16-byte load of two adjacent cells */
__device__ __forceinline__ void ld_cells2(const ull* p, ull* a, ull* b) {
#ifdef SMX_HOSTSIM
  *a = p[0]; *b = p[1];
#else
  const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p);
  *a = v.x; *b = v.y;
#endif
}

/* rows that live in their directory entry: one thread per row */
__global__ void __launch_bounds__(SMX_BLOCK)
k_getrow_inline(smx_view_t V, const ull* info, uint32_t n, const ull* offsets, ull bias, uint32_t* pairs) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const ull inf = info[i];
    if (inf == SMX_NO_ROW || (uint32_t)(inf >> 32) != SMX_INLINE_LOG) continue;
    const smx_row_t* e = V.dir + (uint32_t)inf;
    ull hdr[4], c[4];
    ld_hsector(e, hdr);
    ld_hsector((const char*)e + 32, c);
    ull* out = (ull*)pairs + (offsets[i] - bias);
    const uint32_t c0 = (uint32_t)(hdr[2] >> 32);
    if (c0 != 0u) *out++ = (ull)c0 << 32; /* (column 0, c0) */
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (c[k] != 0ull) *out++ = c[k];
  }
}

/* one warp per row, buckets of 16 .. 2^(SMX_GETROW_BIG_LOG-1) cells */
__global__ void __launch_bounds__(SMX_BLOCK)
k_getrow_fill(smx_view_t V, const ull* info, uint32_t n, const ull* offsets, ull bias, uint32_t* pairs) {
  __shared__ ull s_out[SMX_BLOCK / SMX_WARP][2 * SMX_WARP];
  const uint32_t lane = lane_id(), wib = threadIdx.x / SMX_WARP;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  ull* stage = s_out[wib];
  for (uint32_t i = warp; i < n; i += nwarps) {
    const ull inf = info[i];
    const uint32_t caplog = (uint32_t)(inf >> 32);
    if (inf == SMX_NO_ROW || caplog == SMX_INLINE_LOG || caplog >= SMX_GETROW_BIG_LOG) continue;
    const smx_row_t* e = V.dir + (uint32_t)inf;
    const Hdr h = ld_hdr(e);
    ull* out = (ull*)pairs + (offsets[i] - bias);
    ull pos = 0;
    if (h.c0 != 0u) {
      if (lane == 0) out[0] = (ull)h.c0 << 32; /* (column 0, c0) */
      pos = 1;
    }
    const ull* base = (const ull*)h.slots;
    const ull cap = 1ull << caplog;
    for (ull s0 = 0; s0 < cap; s0 += 2ull * SMX_WARP) {
      const ull s = s0 + 2ull * lane;
      ull a = 0, b = 0;
      if (s < cap) ld_cells2(base + s, &a, &b); /* cap is a multiple of 4, s is even: both cells are in range */
      const uint32_t mine = (a != 0ull) + (b != 0ull);
      uint32_t incl = mine;
      for (uint32_t d = 1; d < SMX_WARP; d <<= 1) {
        uint32_t t = __shfl_up_sync(SMX_FULL, incl, d);
        if (lane >= d) incl += t;
      }
      const uint32_t total = __shfl_sync(SMX_FULL, incl, SMX_WARP - 1);
      uint32_t w = incl - mine; /* compact into shared memory, then one contiguous run goes out */
      if (a != 0ull) stage[w++] = a;
      if (b != 0ull) stage[w] = b;
      __syncwarp();
      for (uint32_t k = lane; k < total; k += SMX_WARP) out[pos + k] = stage[k];
      __syncwarp();
      pos += total;
    }
  }
}

/* big rows (>= 2^SMX_GETROW_BIG_LOG cells), cut into chunks of GETROW_CHUNK cells that the blocks of a
 * persistent grid share; pair order inside a row is arbitrary (the contract compares sorted) */
#define GETROW_CHUNK_LOG 11u
#define GETROW_CHUNK (1u << GETROW_CHUNK_LOG)
#define GETROW_PER_THREAD (GETROW_CHUNK / SMX_BLOCK) /* 8 cells = 4 x 16-byte loads per thread */
#define GETROW_BLOCKS_PER_ROW 32u /* grid.x: blocks that share one big row's chunks (grid.y = rows) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_getrow_chunks(smx_view_t V, const ull* info, const uint32_t* big_list, uint32_t big_first, const ull* offsets,
                ull bias, uint32_t* pairs, uint32_t* cursors) {
  __shared__ ull s_stage[GETROW_CHUNK + 1];
  __shared__ uint32_t s_base;
  const uint32_t i = big_list[big_first + blockIdx.y];
  const ull inf = info[i];
  const ull nchunks = (1ull << (uint32_t)(inf >> 32)) >> GETROW_CHUNK_LOG;
  if (blockIdx.x >= nchunks) return;
  const smx_row_t* e = V.dir + (uint32_t)inf;
  const Hdr h = ld_hdr(e);
  ull* const out_row = (ull*)pairs + (offsets[i] - bias);
  for (ull c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const ull* base = (const ull*)h.slots + (c << GETROW_CHUNK_LOG) + (ull)threadIdx.x * GETROW_PER_THREAD;
    ull cell[GETROW_PER_THREAD];
#pragma unroll
    for (int k = 0; k < (int)GETROW_PER_THREAD; k += 2) ld_cells2(base + k, &cell[k], &cell[k + 1]);
    uint32_t mine = 0;
#pragma unroll
    for (int k = 0; k < (int)GETROW_PER_THREAD; ++k) mine += cell[k] != 0ull;
    const bool with_c0 = (c == 0 && threadIdx.x == 0 && h.c0 != 0u);
    ull total;
    uint32_t w = (uint32_t)block_exclusive_scan((ull)mine + (with_c0 ? 1u : 0u), &total);
    if (with_c0) s_stage[w++] = (ull)h.c0 << 32;
#pragma unroll
    for (int k = 0; k < (int)GETROW_PER_THREAD; ++k)
      if (cell[k] != 0ull) s_stage[w++] = cell[k];
    if (threadIdx.x == 0) s_base = total ? atomicAdd(&cursors[i], (uint32_t)total) : 0u;
    __syncthreads();
    ull* out = out_row + s_base;
    for (uint32_t k = threadIdx.x; k < (uint32_t)total; k += blockDim.x) out[k] = s_stage[k];
    __syncthreads(); /* before the next chunk reuses the staging buffer */
  }
}

/* ---- the read side of the co-occurrence recommender (examples/cf_recommender.c:50-86) ------
 * one warp per item a: total_a = value at (a, 0); for every pair (b, cc) of a's row (already
 * compacted into `pairs`): total_b = value at (b, 0), 1 if zero; score = cc / (sqrt(total_a) *
 * sqrt(total_b)), 0 if the denominator is 0 or smaller than cc (cf_cosine, :67-86).  IEEE double
 * sqrt / mul / div are correctly rounded on the device too, so scores are bit-exact with the CPU. */
__global__ void __launch_bounds__(SMX_BLOCK)
k_cf_scores(smx_view_t V, const uint32_t* items, uint32_t n, const ull* offsets, const uint32_t* pairs,
            uint32_t* ids, double* scores) {
  const uint32_t lane = lane_id();
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t i = warp; i < n; i += nwarps) {
    smx_row_t* e;
    Hdr h;
    uint32_t a_total = 0u;
    if (dir_find(V, items[i], false, &e, &h) == DIR_FOUND) a_total = h.c0;
    const double sa = sqrt((double)a_total);
    for (ull k = offsets[i] + lane; k < offsets[i + 1]; k += SMX_WARP) {
      const uint32_t b = pairs[2 * k], cc = pairs[2 * k + 1];
      uint32_t b_total = 0u;
      if (dir_find(V, b, false, &e, &h) == DIR_FOUND) b_total = h.c0;
      if (b_total == 0u) b_total = 1u;
      const double num = (double)cc, den = sa * sqrt((double)b_total);
      ids[k] = b;
      scores[k] = (den == 0.0 || num > den) ? 0.0 : num / den;
    }
  }
}

/* the same scores when the totals come from OTHER shards (multi-GPU): cols[k] = column of pair k,
 * a_tot[i] / b_tot[k] = value at (item i, 0) / (cols[k], 0), fetched by sharded gets */
__global__ void __launch_bounds__(SMX_BLOCK) k_pair_cols(const uint32_t* pairs, ull total, uint32_t* cols) {
  for (ull k = blockIdx.x * (ull)blockDim.x + threadIdx.x; k < total; k += (ull)gridDim.x * blockDim.x)
    cols[k] = pairs[2 * k];
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_cf_scores_totals(uint32_t n, const ull* offsets, const uint32_t* pairs, const uint32_t* a_tot,
                   const uint32_t* b_tot, uint32_t* ids, double* scores) {
  const uint32_t lane = lane_id();
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t i = warp; i < n; i += nwarps) {
    const double sa = sqrt((double)a_tot[i]);
    for (ull k = offsets[i] + lane; k < offsets[i + 1]; k += SMX_WARP) {
      const uint32_t cc = pairs[2 * k + 1];
      const uint32_t bt = b_tot[k] ? b_tot[k] : 1u;
      const double num = (double)cc, den = sa * sqrt((double)bt);
      ids[k] = pairs[2 * k];
      scores[k] = (den == 0.0 || num > den) ? 0.0 : num / den;
    }
  }
}

/* ---- top-k per segment of (id, score) pairs (smatrix_cf_topk_batch, smatrix_b200_topk_segments) ------------
 * Order: score descending, then id ascending.  The key of a pair is 96 bits: the score mapped to an order-
 * preserving uint64 (flip every bit of a negative, set the sign bit of a positive), then ~id, so a larger key
 * is always better and keys inside a segment are unique.  Three size classes, like getrow's:
 *   k_topk_warp    segments of <= TOPK_WARP_MAX pairs: one warp per segment, bitonic sort in shared memory
 *   k_topk_block   <= TOPK_BLOCK_MAX pairs: one block per segment, the same sort over 48 KB of shared memory
 *   big segments   MSB radix select over the key, TOPK_DIGIT_BITS per pass, for all big segments of a call at
 *                  once: k_topk_hist (TOPK_BIG_BLOCKS blocks per segment build shared-memory histograms of the
 *                  candidates and merge them with one global atomic per bin), k_topk_pick (one thread per
 *                  segment: the digit of the k-th key), k_topk_compact (the pairs at or above the boundary go to
 *                  a private region once they are at most half the segment, and again once they fit).  When the
 *                  pairs above the boundary plus the candidates fit TOPK_BLOCK_MAX, k_topk_finish sorts them.
 * Launches are bounded by the number of digits, not by the number of segments.  The CPU tests lower the class
 * thresholds and the digit width with -D so that rows of a few thousand pairs take every path. */
#ifndef TOPK_WARP_MAX
#define TOPK_WARP_MAX 256u
#endif
#ifndef TOPK_BLOCK_MAX
#define TOPK_BLOCK_MAX 4096u /* 4096 x 12 B = the 48 KB of static shared memory a block may have */
#endif
#ifndef TOPK_DIGIT_BITS
#define TOPK_DIGIT_BITS 8u
#endif
#define TOPK_RADIX (1u << TOPK_DIGIT_BITS)
#define TOPK_BIG_BLOCKS (SMX_WARP > 1 ? 32u : 2u) /* grid.x per big segment (grid.y = segments) */
static_assert(32u % TOPK_DIGIT_BITS == 0u, "a digit must not straddle the score / id boundary of the key");
static_assert((TOPK_WARP_MAX & (TOPK_WARP_MAX - 1u)) == 0u && (TOPK_BLOCK_MAX & (TOPK_BLOCK_MAX - 1u)) == 0u,
              "the bitonic sorts need power-of-two buffers");
static_assert(TOPK_BLOCK_MAX >= SMX_TOPK_MAX_K && TOPK_WARP_MAX < TOPK_BLOCK_MAX, "size classes");

__device__ __forceinline__ ull topk_map(double d) {
#ifdef SMX_HOSTSIM
  ull b;
  memcpy(&b, &d, 8);
#else
  const ull b = (ull)__double_as_longlong(d);
#endif
  return (b >> 63) ? ~b : (b | (1ull << 63));
}
__device__ __forceinline__ double topk_unmap(ull m) {
  const ull b = (m >> 63) ? (m & ~(1ull << 63)) : ~m;
#ifdef SMX_HOSTSIM
  double d;
  memcpy(&d, &b, 8);
  return d;
#else
  return __longlong_as_double((long long)b);
#endif
}
/* a ranks before b */
__device__ __forceinline__ bool topk_better(ull a_hi, uint32_t a_id, ull b_hi, uint32_t b_id) {
  return a_hi > b_hi || (a_hi == b_hi && a_id < b_id);
}
/* the top `bits` bits of key (hi, lo) compared with those of the prefix: -1, 0, 1 */
__device__ __forceinline__ int topk_cmp_top(ull hi, uint32_t lo, ull p_hi, uint32_t p_lo, uint32_t bits) {
  if (bits == 0u) return 0;
  if (bits <= 64u) {
    const ull a = hi >> (64u - bits), b = p_hi >> (64u - bits);
    return a < b ? -1 : (a > b ? 1 : 0);
  }
  if (hi != p_hi) return hi < p_hi ? -1 : 1;
  const uint32_t a = (uint32_t)((ull)lo >> (96u - bits)), b = (uint32_t)((ull)p_lo >> (96u - bits));
  return a < b ? -1 : (a > b ? 1 : 0);
}
/* the digit below the top `bits` bits */
__device__ __forceinline__ uint32_t topk_digit(ull hi, uint32_t lo, uint32_t bits) {
  if (bits < 64u) return (uint32_t)(hi >> (64u - bits - TOPK_DIGIT_BITS)) & (TOPK_RADIX - 1u);
  return (lo >> (96u - bits - TOPK_DIGIT_BITS)) & (TOPK_RADIX - 1u);
}

template <bool BLOCK>
__device__ __forceinline__ void topk_sync() {
  if (BLOCK) __syncthreads(); else __syncwarp();
}
/* bitonic sort of N (power of two) keys, best first, by the T threads of a warp or a block (t = own index) */
template <bool BLOCK>
__device__ void topk_sort(ull* hi, uint32_t* id, uint32_t N, uint32_t t, uint32_t T) {
  for (uint32_t run = 2; run <= N; run <<= 1)
    for (uint32_t j = run >> 1; j > 0; j >>= 1) {
      for (uint32_t i = t; i < N; i += T) {
        const uint32_t l = i ^ j;
        if (l <= i) continue;
        const ull hi_i = hi[i], hi_l = hi[l];
        const uint32_t id_i = id[i], id_l = id[l];
        const bool swap = (i & run) == 0 ? topk_better(hi_l, id_l, hi_i, id_i) : topk_better(hi_i, id_i, hi_l, id_l);
        if (swap) {
          hi[i] = hi_l; hi[l] = hi_i;
          id[i] = id_l; id[l] = id_i;
        }
      }
      topk_sync<BLOCK>();
    }
}
/* one segment of len <= buffer size pairs: stage, sort, write k slots (count[0] = min(k, len); the slots past
 * it get id 0xFFFFFFFF and score -1.0) */
template <bool BLOCK>
__device__ void topk_segment(const uint32_t* ids, const double* scores, uint32_t len, uint32_t k, ull* hi,
                             uint32_t* id, uint32_t t, uint32_t T, uint32_t* count, uint32_t* out_ids,
                             double* out_scores) {
  uint32_t N = 1u;
  while (N < len) N <<= 1;
  for (uint32_t i = t; i < N; i += T) {
    const bool real = i < len;
    hi[i] = real ? topk_map(scores[i]) : 0ull; /* padding ranks after every real key */
    id[i] = real ? ids[i] : 0xFFFFFFFFu;
  }
  topk_sync<BLOCK>();
  topk_sort<BLOCK>(hi, id, N, t, T);
  const uint32_t c = len < k ? len : k;
  for (uint32_t r = t; r < k; r += T) {
    out_ids[r] = r < c ? id[r] : 0xFFFFFFFFu;
    out_scores[r] = r < c ? topk_unmap(hi[r]) : -1.0;
  }
  if (t == 0u) *count = c;
  topk_sync<BLOCK>(); /* before the buffers take the next segment */
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_warp(uint32_t n, const ull* offsets, const uint32_t* ids, const double* scores, uint32_t k, uint32_t* counts,
            uint32_t* out_ids, double* out_scores) {
  __shared__ ull s_hi[SMX_BLOCK / SMX_WARP][TOPK_WARP_MAX];
  __shared__ uint32_t s_id[SMX_BLOCK / SMX_WARP][TOPK_WARP_MAX];
  const uint32_t lane = lane_id(), wib = threadIdx.x / SMX_WARP;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t i = warp; i < n; i += nwarps) {
    const ull lo = offsets[i], len = offsets[i + 1] - lo;
    if (len > TOPK_WARP_MAX) continue;
    topk_segment<false>(ids + lo, scores + lo, (uint32_t)len, k, s_hi[wib], s_id[wib], lane, SMX_WARP, counts + i,
                        out_ids + (ull)i * k, out_scores + (ull)i * k);
  }
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_block(uint32_t n, const ull* offsets, const uint32_t* ids, const double* scores, uint32_t k, uint32_t* counts,
             uint32_t* out_ids, double* out_scores) {
  __shared__ ull s_hi[TOPK_BLOCK_MAX];
  __shared__ uint32_t s_id[TOPK_BLOCK_MAX];
  for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
    const ull lo = offsets[i], len = offsets[i + 1] - lo;
    if (len <= TOPK_WARP_MAX || len > TOPK_BLOCK_MAX) continue;
    topk_segment<true>(ids + lo, scores + lo, (uint32_t)len, k, s_hi, s_id, threadIdx.x, blockDim.x, counts + i,
                       out_ids + (ull)i * k, out_scores + (ull)i * k);
  }
}

/* the select state of one big segment.  Its pairs live in the input arrays (src_kind 0) or, once compacted, in
 * its region of the compaction buffers (src_kind 1; the region has `len` slots: the first compaction writes at
 * its start, a second one into its upper half, which the first one's output never reaches). */
typedef struct {
  ull pre_hi;         /* the key bits fixed so far, left-aligned; the rest zero        */
  ull len, reg;       /* segment length, start of its compaction region              */
  ull src_off, src_len, from_off, from_len;
  uint32_t pre_lo, bits; /* key bits fixed so far (a multiple of TOPK_DIGIT_BITS)     */
  uint32_t item;      /* segment index                                               */
  uint32_t above;     /* pairs above the prefix range: all of them are in the top k  */
  uint32_t cand;      /* pairs inside the prefix range                               */
  uint32_t done, compact, cursor, src_kind, from_kind;
} topk_state_t;

/* big segments -> list; ctl[0] = their number, ctl[2..3] = their pairs (u64) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_classify(uint32_t n, const ull* offsets, uint32_t* big_list, uint32_t* ctl) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const ull len = offsets[i + 1] - offsets[i];
    if (len <= TOPK_BLOCK_MAX) continue;
    big_list[agg_inc(&ctl[0])] = i;
    atomicAdd((ull*)(ctl + 2), len);
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_init(const uint32_t* big_list, uint32_t n_big, const ull* offsets, topk_state_t* st_all, ull* reg_cursor) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_big; j += gridDim.x * blockDim.x) {
    const uint32_t i = big_list[j];
    topk_state_t st;
    memset(&st, 0, sizeof st);
    st.item = i;
    st.src_off = offsets[i];
    st.len = st.src_len = offsets[i + 1] - st.src_off;
    st.cand = (uint32_t)st.len;
    st.reg = atomicAdd(reg_cursor, st.len);
    st_all[j] = st;
  }
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_hist(const topk_state_t* st_all, uint32_t first, const uint32_t* ids, const double* scores,
            const uint32_t* c_ids, const double* c_scores, uint32_t* hist) {
  __shared__ uint32_t s_h[TOPK_RADIX];
  const uint32_t j = first + blockIdx.y;
  const topk_state_t st = st_all[j];
  if (st.done) return;
  for (uint32_t b = threadIdx.x; b < TOPK_RADIX; b += blockDim.x) s_h[b] = 0u;
  __syncthreads();
  const uint32_t* sid = (st.src_kind ? c_ids : ids) + st.src_off;
  const double* ssc = (st.src_kind ? c_scores : scores) + st.src_off;
  for (ull p = (ull)blockIdx.x * blockDim.x + threadIdx.x; p < st.src_len; p += (ull)gridDim.x * blockDim.x) {
    const ull hk = topk_map(ssc[p]);
    const uint32_t lk = ~sid[p];
    if (topk_cmp_top(hk, lk, st.pre_hi, st.pre_lo, st.bits) == 0) atomicAdd(&s_h[topk_digit(hk, lk, st.bits)], 1u);
  }
  __syncthreads();
  for (uint32_t b = threadIdx.x; b < TOPK_RADIX; b += blockDim.x)
    if (s_h[b]) atomicAdd(&hist[(ull)j * TOPK_RADIX + b], s_h[b]);
}

/* one thread per big segment: the boundary digit = the bin that holds the k-th key among the candidates */
__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_pick(topk_state_t* st_all, uint32_t n_big, uint32_t k, uint32_t* hist, uint32_t* active) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_big; j += gridDim.x * blockDim.x) {
    topk_state_t st = st_all[j];
    if (st.done) {
      st_all[j].compact = 0u; /* its last compaction ran in the pass that finished it */
      continue;
    }
    uint32_t* h = hist + (ull)j * TOPK_RADIX;
    const uint32_t need = k - st.above; /* >= 1: above < k always */
    uint32_t cum = 0u, b = TOPK_RADIX - 1u;
    for (;; --b) {
      if (cum + h[b] >= need || b == 0u) break;
      cum += h[b];
    }
    st.above += cum;
    st.cand = h[b];
    if (st.bits < 64u) st.pre_hi |= (ull)b << (64u - st.bits - TOPK_DIGIT_BITS);
    else st.pre_lo |= b << (96u - st.bits - TOPK_DIGIT_BITS);
    st.bits += TOPK_DIGIT_BITS;
    for (uint32_t d = 0; d < TOPK_RADIX; ++d) h[d] = 0u;
    const ull keep = (ull)st.above + st.cand;
    st.done = keep <= TOPK_BLOCK_MAX;
    st.compact = st.src_kind == 0u ? (st.done || 2ull * keep <= st.len) : (st.done && st.src_len != keep);
    if (st.compact) {
      st.from_kind = st.src_kind; st.from_off = st.src_off; st.from_len = st.src_len;
      st.src_kind = 1u;
      st.src_off = st.reg + (st.from_kind ? st.len / 2u : 0ull);
      st.src_len = keep;
      st.cursor = 0u;
    }
    if (!st.done) atomicAdd(active, 1u);
    st_all[j] = st;
  }
}

/* the pairs whose top `bits` key bits are >= the prefix: into the segment's region (one atomic per block tile) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_compact(topk_state_t* st_all, uint32_t first, const uint32_t* ids, const double* scores, uint32_t* c_ids,
               double* c_scores) {
  __shared__ uint32_t s_base;
  const uint32_t j = first + blockIdx.y;
  const topk_state_t st = st_all[j];
  if (!st.compact) return;
  const uint32_t* sid = (st.from_kind ? c_ids : ids) + st.from_off;
  const double* ssc = (st.from_kind ? c_scores : scores) + st.from_off;
  for (ull p0 = (ull)blockIdx.x * blockDim.x; p0 < st.from_len; p0 += (ull)gridDim.x * blockDim.x) {
    const ull p = p0 + threadIdx.x;
    uint32_t id = 0u;
    double sc = 0.0;
    bool keep = false;
    if (p < st.from_len) {
      id = sid[p];
      sc = ssc[p];
      keep = topk_cmp_top(topk_map(sc), ~id, st.pre_hi, st.pre_lo, st.bits) >= 0;
    }
    ull total;
    const uint32_t w = (uint32_t)block_exclusive_scan(keep ? 1ull : 0ull, &total);
    if (threadIdx.x == 0) s_base = total ? atomicAdd(&st_all[j].cursor, (uint32_t)total) : 0u;
    __syncthreads();
    if (keep) {
      c_ids[st.src_off + s_base + w] = id;
      c_scores[st.src_off + s_base + w] = sc;
    }
    __syncthreads(); /* s_base is rewritten by the next tile */
  }
}

/* one block per big segment: sort what the select kept (<= TOPK_BLOCK_MAX pairs) and write the first k */
__global__ void __launch_bounds__(SMX_BLOCK)
k_topk_finish(const topk_state_t* st_all, uint32_t first, const uint32_t* c_ids, const double* c_scores, uint32_t k,
              uint32_t* counts, uint32_t* out_ids, double* out_scores) {
  __shared__ ull s_hi[TOPK_BLOCK_MAX];
  __shared__ uint32_t s_id[TOPK_BLOCK_MAX];
  const topk_state_t st = st_all[first + blockIdx.x];
  topk_segment<true>(c_ids + st.src_off, c_scores + st.src_off, (uint32_t)st.src_len, k, s_hi, s_id, threadIdx.x,
                     blockDim.x, counts + st.item, out_ids + (ull)st.item * k, out_scores + (ull)st.item * k);
}

/* one thread: the end of the piece that starts at item lo = the last item whose pairs still fit the budget
 * (at least one item: a row over the budget is a piece of its own) -> out[0] */
__global__ void k_topk_cut(const ull* offsets, uint32_t n, uint32_t lo, ull budget, uint32_t* out) {
  uint32_t a = lo + 1u, b = n; /* answer in [a, b] */
  while (a < b) {
    const uint32_t m = a + (b - a + 1u) / 2u;
    if (offsets[m] - offsets[lo] <= budget) a = m; else b = m - 1u;
  }
  out[0] = a;
}

/* ---- basket recommendations (smatrix_cf_recommend_batch, smatrix_b200_basket_topk) ---------------------------
 * A piece of nb baskets: boff[0..nb] are absolute positions (base = boff[0]), items[p] is the item at position p,
 * and off[p - base] .. off[p - base + 1] is that position's neighbour list in ids / scores.  Basket b's pairs are
 * [off[boff[b] - base], off[boff[b + 1] - base]), position-major, so ordering them stably by id puts every id's
 * contributions in position order, and one thread adds each run up left to right (IEEE double, one rounding per
 * addition).  A run survives unless its id is 0 or an item of the basket (binary search in the basket's items,
 * sorted once by k_rec_item_keys + a radix sort of (basket << 32 | item) keys).  The survivors, in id order, are
 * a reduced CSR that the top-k selection ranks.  Size classes as top-k's:
 *   k_rec_warp / k_rec_block  baskets of <= TOPK_WARP_MAX / TOPK_BLOCK_MAX pairs: bitonic sort of (id << 32 |
 *                             local index) keys in shared memory; survivors go to the basket's own slots of the
 *                             staging arrays, their number to cnt[b]
 *   big baskets               all of a piece's at once: (slot << 32 | id) keys of their pairs with the local index
 *                             as value, one stable radix sort, k_rec_big_flag marks the surviving run heads, a scan
 *                             of the marks ranks them and k_rec_big_emit sums each run straight into the reduced CSR
 * k_rec_compact moves the small baskets' survivors from the staging arrays to the reduced CSR. */
__device__ __forceinline__ double rec_add(double a, double b) {
#ifdef SMX_HOSTSIM
  return a + b;
#else
  return __dadd_rn(a, b); /* never contracted or reordered */
#endif
}
/* is `id` excluded from basket b, whose sorted (b << 32 | item) keys are sitems[lo..hi)? */
__device__ __forceinline__ bool rec_excluded(uint32_t id, uint32_t b, const ull* sitems, ull lo, ull hi) {
  if (id == 0u) return true;
  const ull want = ((ull)b << 32) | id;
  while (lo < hi) {
    const ull m = lo + (hi - lo) / 2u;
    const ull v = sitems[m];
    if (v == want) return true;
    if (v < want) lo = m + 1u; else hi = m;
  }
  return false;
}
/* bitonic sort of N (power of two) keys, ascending */
template <bool BLOCK>
__device__ void rec_sort(ull* key, uint32_t N, uint32_t t, uint32_t T) {
  for (uint32_t run = 2; run <= N; run <<= 1)
    for (uint32_t j = run >> 1; j > 0; j >>= 1) {
      for (uint32_t i = t; i < N; i += T) {
        const uint32_t l = i ^ j;
        if (l <= i) continue;
        const ull a = key[i], c = key[l];
        if ((i & run) == 0 ? a > c : a < c) {
          key[i] = c;
          key[l] = a;
        }
      }
      topk_sync<BLOCK>();
    }
}
/* one small basket by a warp or a block: sort, run sums, survivors in id order to t_ids / t_scores[lo..) */
template <bool BLOCK>
__device__ void rec_segment(uint32_t b, ull p0, ull p1, ull lo, uint32_t len, const uint32_t* ids,
                            const double* scores, const ull* sitems, ull* key, uint32_t t, uint32_t T,
                            uint32_t* t_ids, double* t_scores, uint32_t* cnt) {
  uint32_t N = 1u;
  while (N < len) N <<= 1;
  for (uint32_t i = t; i < N; i += T) key[i] = i < len ? ((ull)ids[lo + i] << 32) | i : ~0ull;
  topk_sync<BLOCK>();
  rec_sort<BLOCK>(key, N, t, T);
  uint32_t kept = 0u;
  for (uint32_t c0 = 0; c0 < len; c0 += T) { /* every thread takes the same number of turns */
    const uint32_t j = c0 + t;
    bool keep = false;
    uint32_t id = 0u;
    double sum = 0.0;
    if (j < len) {
      id = (uint32_t)(key[j] >> 32);
      keep = (j == 0u || (uint32_t)(key[j - 1] >> 32) != id) && !rec_excluded(id, b, sitems, p0, p1);
      if (keep)
        for (uint32_t q = j; q < len && (uint32_t)(key[q] >> 32) == id; ++q)
          sum = rec_add(sum, scores[lo + (uint32_t)key[q]]);
    }
    uint32_t w, tot;
    if (BLOCK) {
      ull all;
      w = (uint32_t)block_exclusive_scan(keep ? 1ull : 0ull, &all);
      tot = (uint32_t)all;
    } else {
      const unsigned m = __ballot_sync(SMX_FULL, keep);
      w = (uint32_t)__popc(m & ((1u << t) - 1u));
      tot = (uint32_t)__popc(m);
    }
    if (keep) {
      t_ids[lo + kept + w] = id;
      t_scores[lo + kept + w] = sum;
    }
    kept += tot;
  }
  if (t == 0u) cnt[b] = kept;
  topk_sync<BLOCK>(); /* before the buffer takes the next basket */
}

/* keys of the piece's items: (basket << 32 | item) at position p - base; one warp per basket */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_item_keys(uint32_t nb, const ull* boff, ull base, const uint32_t* items, ull* keys) {
  const uint32_t lane = lane_id();
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t b = warp; b < nb; b += nwarps)
    for (ull p = boff[b] + lane; p < boff[b + 1]; p += SMX_WARP) keys[p - base] = ((ull)b << 32) | items[p];
}

/* big baskets -> list; ctl[0] = their number, ctl[2..3] = their pairs (u64) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_classify(uint32_t nb, const ull* boff, ull base, const ull* off, uint32_t* big_list, uint32_t* ctl) {
  for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += gridDim.x * blockDim.x) {
    const ull len = off[boff[b + 1] - base] - off[boff[b] - base];
    if (len <= TOPK_BLOCK_MAX) continue;
    big_list[agg_inc(&ctl[0])] = b;
    atomicAdd((ull*)(ctl + 2), len);
  }
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_warp(uint32_t nb, const ull* boff, ull base, const ull* off, const uint32_t* ids, const double* scores,
           const ull* sitems, uint32_t* t_ids, double* t_scores, uint32_t* cnt) {
  __shared__ ull s_key[SMX_BLOCK / SMX_WARP][TOPK_WARP_MAX];
  const uint32_t lane = lane_id(), wib = threadIdx.x / SMX_WARP;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t b = warp; b < nb; b += nwarps) {
    const ull p0 = boff[b] - base, p1 = boff[b + 1] - base, lo = off[p0], len = off[p1] - lo;
    if (len > TOPK_WARP_MAX) continue;
    rec_segment<false>(b, p0, p1, lo, (uint32_t)len, ids, scores, sitems, s_key[wib], lane, SMX_WARP, t_ids, t_scores,
                       cnt);
  }
}

__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_block(uint32_t nb, const ull* boff, ull base, const ull* off, const uint32_t* ids, const double* scores,
            const ull* sitems, uint32_t* t_ids, double* t_scores, uint32_t* cnt) {
  __shared__ ull s_key[TOPK_BLOCK_MAX];
  for (uint32_t b = blockIdx.x; b < nb; b += gridDim.x) {
    const ull p0 = boff[b] - base, p1 = boff[b + 1] - base, lo = off[p0], len = off[p1] - lo;
    if (len <= TOPK_WARP_MAX || len > TOPK_BLOCK_MAX) continue;
    rec_segment<true>(b, p0, p1, lo, (uint32_t)len, ids, scores, sitems, s_key, threadIdx.x, blockDim.x, t_ids,
                      t_scores, cnt);
  }
}

/* pairs of big basket j (= big_list[j]) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_big_lens(const uint32_t* big_list, uint32_t n_big, const ull* boff, ull base, const ull* off, uint32_t* lens) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_big; j += gridDim.x * blockDim.x) {
    const uint32_t b = big_list[j];
    lens[j] = (uint32_t)(off[boff[b + 1] - base] - off[boff[b] - base]);
  }
}
/* (slot << 32 | id) keys and local indices of the big baskets' pairs, slot j at big_off[j] */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_big_keys(const uint32_t* big_list, uint32_t first, const ull* boff, ull base, const ull* off,
               const uint32_t* ids, const ull* big_off, ull* keys, uint32_t* vals) {
  const uint32_t j = first + blockIdx.y, b = big_list[j];
  const ull lo = off[boff[b] - base], len = off[boff[b + 1] - base] - lo, at = big_off[j];
  for (ull q = (ull)blockIdx.x * blockDim.x + threadIdx.x; q < len; q += (ull)gridDim.x * blockDim.x) {
    keys[at + q] = ((ull)j << 32) | ids[lo + q];
    vals[at + q] = (uint32_t)q;
  }
}
/* flags[p] = 1 where a run of equal keys starts and its id survives */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_big_flag(const ull* keys, uint32_t P, const uint32_t* big_list, const ull* boff, ull base, const ull* sitems,
               uint32_t* flags) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
    const ull key = keys[p];
    bool keep = p == 0u || keys[p - 1] != key;
    if (keep) {
      const uint32_t b = big_list[(uint32_t)(key >> 32)];
      keep = !rec_excluded((uint32_t)key, b, sitems, boff[b] - base, boff[b + 1] - base);
    }
    flags[p] = keep ? 1u : 0u;
  }
}
/* survivors per big basket from the scan of the flags */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_big_count(const uint32_t* big_list, uint32_t n_big, const ull* big_off, const ull* fpos, uint32_t* cnt) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_big; j += gridDim.x * blockDim.x)
    cnt[big_list[j]] = (uint32_t)(fpos[big_off[j + 1]] - fpos[big_off[j]]);
}
/* every surviving run of the big baskets: its sum, at its rank inside the basket's reduced segment */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_big_emit(const ull* keys, const uint32_t* vals, uint32_t P, const uint32_t* big_list, const ull* big_off,
               const ull* boff, ull base, const ull* off, const double* scores, const ull* fpos, const ull* red_off,
               uint32_t* r_ids, double* r_scores) {
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
    if (fpos[p + 1] == fpos[p]) continue;
    const ull key = keys[p];
    const uint32_t j = (uint32_t)(key >> 32), b = big_list[j];
    const ull lo = off[boff[b] - base];
    double sum = 0.0;
    for (uint32_t q = p; q < P && keys[q] == key; ++q) sum = rec_add(sum, scores[lo + vals[q]]);
    const ull at = red_off[b] + (fpos[p] - fpos[big_off[j]]);
    r_ids[at] = (uint32_t)key;
    r_scores[at] = sum;
  }
}
/* the small baskets' survivors from their staging slots into the reduced CSR; one warp per basket */
__global__ void __launch_bounds__(SMX_BLOCK)
k_rec_compact(uint32_t nb, const ull* boff, ull base, const ull* off, const uint32_t* cnt, const ull* red_off,
              const uint32_t* t_ids, const double* t_scores, uint32_t* r_ids, double* r_scores) {
  const uint32_t lane = lane_id();
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t b = warp; b < nb; b += nwarps) {
    const ull lo = off[boff[b] - base];
    if (off[boff[b + 1] - base] - lo > TOPK_BLOCK_MAX) continue;
    const ull to = red_off[b];
    for (uint32_t q = lane; q < cnt[b]; q += SMX_WARP) {
      r_ids[to + q] = t_ids[lo + q];
      r_scores[to + q] = t_scores[lo + q];
    }
  }
}
/* one thread: the end of the piece of baskets that starts at basket lo = the last basket whose rows still fit the
 * pair budget and whose items fit the item budget (at least one basket) -> out[0]; its positions -> out[1..2] */
__global__ void k_rec_cut(const ull* pos_off, const ull* boff, uint32_t nb, uint32_t lo, ull budget, ull item_budget,
                          uint32_t* out) {
  uint32_t a = lo + 1u, b = nb; /* answer in [a, b] */
  while (a < b) {
    const uint32_t m = a + (b - a + 1u) / 2u;
    if (pos_off[boff[m]] - pos_off[boff[lo]] <= budget && boff[m] - boff[lo] <= item_budget) a = m; else b = m - 1u;
  }
  out[0] = a;
  out[1] = (uint32_t)boff[lo];
  out[2] = (uint32_t)boff[a];
}
/* basket offsets that do not start at 0, decrease or end past 2^32 - 2 set out[0]; out[2..3] = boff[nb] (u64) */
__global__ void __launch_bounds__(SMX_BLOCK) k_rec_check(const ull* boff, uint32_t nb, uint32_t* out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += gridDim.x * blockDim.x)
    if (boff[i + 1] < boff[i] || (i == 0u && boff[0] != 0ull)) atomicOr(&out[0], 1u);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (boff[nb] > 0xFFFFFFFEull) atomicOr(&out[0], 1u);
    *(ull*)(out + 2) = boff[nb];
  }
}

/* ---- snapshot support (file mode, reference src/smatrix.c:30-72) --------------------------- */
/* all row ids of the directory, in no particular order */
__global__ void __launch_bounds__(SMX_BLOCK) k_list_rows(smx_view_t V, uint32_t* keys, uint32_t* counter) {
  for (ull pos = blockIdx.x * blockDim.x + threadIdx.x; pos < V.dir_cap;
       pos += (ull)gridDim.x * blockDim.x) {
    Hdr h = ld_hdr(V.dir + pos);
    if (h.meta & SMX_META_USED) keys[agg_inc(counter)] = h.key;
  }
}
/* log2 of the reference's row size as of now (the caught-up automaton state), per row */
__global__ void __launch_bounds__(SMX_BLOCK)
k_row_slog(smx_view_t V, const uint32_t* xs, uint32_t n, uint32_t* out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    uint32_t slog = 4u;
    if (dir_find(V, xs[i], false, &e, &h) == DIR_FOUND) {
      const uint32_t m2 = rowlen_catch_up(h.meta, h.live, (h.meta & (SMX_META_ZC | SMX_META_T0P)) != 0u);
      slog = 4u + ((m2 & SMX_META_SLOG) >> SMX_META_SLOG_SHIFT);
    }
    out[i] = slog;
  }
}
/* ---- K9: the row blocks of a snapshot, built on the device in the REFERENCE's layout ------------
 * A row block is 8 x 0x23, u64 size, then `size` cells placed where the reference's loader and its
 * rmap_probe expect them: position = column % size, linear probing (src/smatrix.c:363-380, :499-545).
 * Three phases keep every probe chain intact when the loader later drops zero-valued cells
 * (src/smatrix.c:533-540): (1) cells with a non-zero value, in any order (unique keys: any insertion
 * order gives a valid table), (2) column 0 into the first cell whose column is 0, (3) zero-valued
 * cells last.  units[i] = 2 + size_i (in 8-byte units) is scanned into the block offsets. */
__global__ void __launch_bounds__(SMX_BLOCK)
k_snap_units(const uint32_t* counts, const uint32_t* slogs, uint32_t n, uint32_t* units) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    ull size = 1ull << (slogs[i] < 4u ? 4u : slogs[i]);
    while ((ull)counts[i] > size / 2) size *= 2; /* never fuller than the reference lets a row get */
    units[i] = (uint32_t)(size + 2ull);
  }
}
__device__ __forceinline__ void snap_place(ull* cells, ull size, ull cell) {
  ull at = (ull)(uint32_t)cell % size;
  for (;;) {
    if (cells[at] == 0ull && atomicCAS(&cells[at], 0ull, cell) == 0ull) return;
    at = at + 1 == size ? 0 : at + 1;
  }
}
__device__ __forceinline__ void snap_place_c0(ull* cells, ull size, uint32_t c0) {
  for (ull at = 0; at < size; ++at) /* the reference probes column 0 from position 0 % size = 0 */
    if ((uint32_t)__ldcg(&cells[at]) == 0u && atomicCAS(&cells[at], 0ull, (ull)c0 << 32) == 0ull) return;
}
/* phase selector: 1 = cells with value != 0, 3 = cells with value == 0 */
__device__ __forceinline__ bool snap_takes(ull cell, int phase) {
  return cell != 0ull && (((cell >> 32) != 0ull) == (phase == 1));
}
/* rows below 2^SMX_GETROW_BIG_LOG cells: one warp per row, all three phases */
__global__ void __launch_bounds__(SMX_BLOCK)
k_snap_rows(smx_view_t V, const ull* info, uint32_t n, const ull* offsets, ull* out) {
  const uint32_t lane = lane_id();
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t i = warp; i < n; i += nwarps) {
    const ull inf = info[i];
    const uint32_t caplog = (uint32_t)(inf >> 32);
    ull* blk = out + offsets[i];
    const ull size = offsets[i + 1] - offsets[i] - 2ull;
    if (lane == 0) { blk[0] = 0x2323232323232323ull; blk[1] = size; }
    if (inf == SMX_NO_ROW || caplog >= SMX_GETROW_BIG_LOG) continue;
    const smx_row_t* e = V.dir + (uint32_t)inf;
    const Hdr h = ld_hdr(e);
    const ull* base = (caplog == SMX_INLINE_LOG) ? (const ull*)e->inl : (const ull*)h.slots;
    const uint32_t cap = 1u << caplog;
    for (int phase = 1; phase <= 3; ++phase) {
      if (phase == 2) {
        if (lane == 0 && h.c0 != 0u) snap_place_c0(blk + 2, size, h.c0);
      } else {
        for (uint32_t c = lane; c < cap; c += SMX_WARP) {
          const ull cell = base[c];
          if (snap_takes(cell, phase)) snap_place(blk + 2, size, cell);
        }
      }
      __syncwarp();
#ifndef SMX_HOSTSIM
      __threadfence_block();
#endif
    }
  }
}
/* big rows: the grid strides over the bucket of one row (y); one launch per phase (1 or 3); phase 2
 * (column 0) is done by the first thread of the phase-3 launch BEFORE any zero-valued cell is placed
 * — so phase 3 is launched twice: c0_only = 1, then c0_only = 0 */
__global__ void __launch_bounds__(SMX_BLOCK)
k_snap_big(smx_view_t V, const ull* info, const uint32_t* big_list, uint32_t first, const ull* offsets, ull* out,
           int phase, int c0_only) {
  const uint32_t i = big_list[first + blockIdx.y];
  const ull inf = info[i];
  const smx_row_t* e = V.dir + (uint32_t)inf;
  const Hdr h = ld_hdr(e);
  ull* blk = out + offsets[i];
  const ull size = offsets[i + 1] - offsets[i] - 2ull;
  if (c0_only) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && h.c0 != 0u) snap_place_c0(blk + 2, size, h.c0);
    return;
  }
  const ull* base = (const ull*)h.slots;
  const ull cap = 1ull << (uint32_t)(inf >> 32);
  for (ull c = blockIdx.x * (ull)blockDim.x + threadIdx.x; c < cap; c += (ull)gridDim.x * blockDim.x) {
    const ull cell = base[c];
    if (snap_takes(cell, phase)) snap_place(blk + 2, size, cell);
  }
}

/* after a load: the reference recounts `used` from the file (src/smatrix.c:533-540), i.e. the row
 * size is the file's and column 0 is counted iff it is non-zero */
__global__ void __launch_bounds__(SMX_BLOCK)
k_load_fixup(smx_view_t V, const uint32_t* xs, const uint32_t* slogs, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    smx_row_t* e;
    Hdr h;
    if (dir_find(V, xs[i], false, &e, &h) != DIR_FOUND) continue;
    uint32_t slog = slogs[i] < 4u ? 4u : (slogs[i] > 35u ? 35u : slogs[i]);
    uint32_t m2 = h.meta & ~(SMX_META_SLOG | SMX_META_D | SMX_META_ZC | SMX_META_T0P);
    m2 |= (slog - 4u) << SMX_META_SLOG_SHIFT;
    if (h.c0 != 0u) m2 |= SMX_META_D | SMX_META_ZC;
    e->meta = m2;
  }
}

/* ---- loading a snapshot: raw row blocks -> the op stream of the loader ------------------------
 * The host uploads a window of file bytes and a tile table (smx_load_tile_t): a row of up to
 * 2^SMX_LOAD_TILE_LOG cells is one tile, a bigger row is cut into tiles of that many cells.  One warp
 * per tile, two passes: k_load_count counts every tile's ops, smx_launch_scan turns the counts into
 * offsets, and k_load_emit writes them in order — the first tile of a row leads with (key, 0, 0) so
 * that the row exists even when it holds no live cell, then every cell with a non-zero value follows
 * in slot order (a ballot per 32 cells, each lane's place = the popcount of the lanes below it).
 * Header checks are the host's: the device only sees validated sizes. */
__device__ __forceinline__ ull ld_file_cell(const unsigned char* p) { /* {u32 column, u32 value} */
  if (((uintptr_t)p & 7u) == 0u) return *(const ull*)p;
  ull c;
  memcpy(&c, p, 8); /* a row block at an odd offset of a foreign file */
  return c;
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_load_count(const unsigned char* raw, const smx_load_tile_t* tiles, uint32_t n, uint32_t* counts) {
  const uint32_t lane = lane_id();
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t t = warp; t < n; t += nwarps) {
    const smx_load_tile_t T = tiles[t];
    const uint32_t cells = T.cells & ~SMX_LOAD_FIRST;
    const unsigned char* p = raw + T.off;
    uint32_t live = 0;
    for (uint32_t base = 0; base < cells; base += SMX_WARP) {
      const uint32_t c = base + lane;
      const bool nz = c < cells && (uint32_t)(ld_file_cell(p + 8ull * c) >> 32) != 0u;
      live += (uint32_t)__popc(__ballot_sync(SMX_FULL, nz));
    }
    if (lane == 0) counts[t] = live + ((T.cells & SMX_LOAD_FIRST) ? 1u : 0u);
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_load_emit(const unsigned char* raw, const smx_load_tile_t* tiles, uint32_t n, const ull* offsets,
            uint32_t* xs, uint32_t* ys, uint32_t* vs) {
  const uint32_t lane = lane_id();
  const uint32_t below = (1u << lane) - 1u;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / SMX_WARP;
  const uint32_t nwarps = gridDim.x * blockDim.x / SMX_WARP;
  for (uint32_t t = warp; t < n; t += nwarps) {
    const smx_load_tile_t T = tiles[t];
    const uint32_t cells = T.cells & ~SMX_LOAD_FIRST;
    const unsigned char* p = raw + T.off;
    ull at = offsets[t];
    if (T.cells & SMX_LOAD_FIRST) {
      if (lane == 0) { xs[at] = T.key; ys[at] = 0u; vs[at] = 0u; }
      at++;
    }
    for (uint32_t base = 0; base < cells; base += SMX_WARP) {
      const uint32_t c = base + lane;
      const ull cell = c < cells ? ld_file_cell(p + 8ull * c) : 0ull;
      const uint32_t v = (uint32_t)(cell >> 32);
      const uint32_t m = __ballot_sync(SMX_FULL, v != 0u);
      if (v != 0u) {
        const ull j = at + (ull)__popc(m & below);
        xs[j] = T.key; ys[j] = (uint32_t)cell; vs[j] = v;
      }
      at += (ull)__popc(m);
    }
  }
}

/* sum of every stored value (all cells + column 0) mod 2^64 -> ctl->scratch: one warp per
 * directory entry walks that row's bucket.  For an incr-only build this must equal the sum of all
 * increments — the size-independent invariant bench.py checks at full scale. */
__global__ void __launch_bounds__(SMX_BLOCK) k_sum_values(smx_view_t V, uint32_t* big_list, uint32_t* big_counter) {
  const uint32_t lane = lane_id();
  const ull warp = (blockIdx.x * (ull)blockDim.x + threadIdx.x) / SMX_WARP;
  const ull nwarps = (ull)gridDim.x * blockDim.x / SMX_WARP;
  ull acc = 0;
  for (ull pos = warp; pos < V.dir_cap; pos += nwarps) {
    const smx_row_t* e = V.dir + pos;
    const Hdr h = ld_hdr(e);
    if (!(h.meta & SMX_META_USED)) continue;
    if (lane == 0) acc += h.c0;
    const uint32_t caplog = h.meta & SMX_META_CAPLOG;
    if (caplog >= SMX_BIG_LOG) { /* a bucket of megabytes is not one warp's job: k_sum_values_big */
      if (lane == 0) big_list[atomicAdd(big_counter, 1u)] = (uint32_t)pos;
      continue;
    }
    const ull* base = (caplog == SMX_INLINE_LOG) ? (const ull*)e->inl : (const ull*)h.slots;
    const ull cap = 1ull << caplog;
    for (ull c = lane; c < cap; c += SMX_WARP) acc += base[c] >> 32;
  }
  for (uint32_t d = SMX_WARP / 2; d > 0; d >>= 1) acc += __shfl_xor_sync(SMX_FULL, acc, d);
  if (lane == 0 && acc) atomicAdd(&V.ctl->scratch, acc);
}
/* big rows: the grid (x) strides over the bucket of one row (y) */
__global__ void __launch_bounds__(SMX_BLOCK) k_sum_values_big(smx_view_t V, const uint32_t* big_list, uint32_t first) {
  const Hdr h = ld_hdr(V.dir + big_list[first + blockIdx.y]);
  const ull* base = (const ull*)h.slots;
  const ull cap = 1ull << (h.meta & SMX_META_CAPLOG);
  ull acc = 0;
  for (ull c = blockIdx.x * (ull)blockDim.x + threadIdx.x; c < cap; c += (ull)gridDim.x * blockDim.x) acc += base[c] >> 32;
  for (uint32_t d = SMX_WARP / 2; d > 0; d >>= 1) acc += __shfl_xor_sync(SMX_FULL, acc, d);
  if (lane_id() == 0 && acc) atomicAdd(&V.ctl->scratch, acc);
}

/* nnz = sum over rows of live + (c0 != 0) -> ctl->scratch */
__global__ void __launch_bounds__(SMX_BLOCK) k_count_nnz(smx_view_t V) {
  ull acc = 0;
  for (ull pos = blockIdx.x * blockDim.x + threadIdx.x; pos < V.dir_cap;
       pos += (ull)gridDim.x * blockDim.x) {
    Hdr h = ld_hdr(V.dir + pos);
    if (h.meta & SMX_META_USED) acc += (ull)h.live + (h.c0 != 0u ? 1ull : 0ull);
  }
  for (uint32_t d = SMX_WARP / 2; d > 0; d >>= 1) acc += __shfl_xor_sync(SMX_FULL, acc, d);
  if (lane_id() == 0 && acc) atomicAdd(&V.ctl->scratch, acc);
}

/* Distinct-row estimate of a chunk by linear counting (one streaming pass): bit hash(x) of a zeroed
 * bitmap of m = 2^bits_log bits is set; with Z zero bits left, distinct ~ -m ln(Z / m).  Lets the host
 * size the directory for a chunk of mostly NEW rows before the first round instead of discovering
 * the overflow through a round that turns nearly every op away (replaces the reference's repeated
 * stop-the-world doubling, src/smatrix.c:715-741). */
__global__ void __launch_bounds__(SMX_BLOCK)
k_sketch_set(const uint32_t* xs, uint32_t n, uint32_t* bitmap, uint32_t bits_log) {
  const uint32_t mask = (uint32_t)((1ull << bits_log) - 1ull);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    /* NOT mix_owner: on a shard every row has the same mix_owner(x) mod G, which would leave part of the
     * bitmap unreachable and bias the estimate low (measured at G = 2: 16 M estimated for 24 M rows) */
    const uint32_t h = smx_mix_col(xs[i] ^ 0x5bd1e995u) & mask;
    const uint32_t bit = 1u << (h & 31u);
    if (!(__ldcg(&bitmap[h >> 5]) & bit)) atomicOr(&bitmap[h >> 5], bit);
  }
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_sketch_count(const uint32_t* bitmap, uint32_t bits_log, smx_ctl_t* ctl) {
  const ull words = (1ull << bits_log) / 32ull;
  ull zeros = 0;
  for (ull w = blockIdx.x * blockDim.x + threadIdx.x; w < words; w += (ull)gridDim.x * blockDim.x)
    zeros += 32u - (uint32_t)__popc(bitmap[w]);
  for (uint32_t d = SMX_WARP / 2; d > 0; d >>= 1) zeros += __shfl_xor_sync(SMX_FULL, zeros, d);
  if (lane_id() == 0 && zeros) atomicAdd(&ctl->scratch, zeros);
}

/* bytes of slab buckets that rows currently own -> ctl->scratch (the denominator of slab / live) */
__global__ void __launch_bounds__(SMX_BLOCK) k_live_bytes(smx_view_t V) {
  ull acc = 0;
  for (ull pos = blockIdx.x * blockDim.x + threadIdx.x; pos < V.dir_cap;
       pos += (ull)gridDim.x * blockDim.x) {
    Hdr h = ld_hdr(V.dir + pos);
    const uint32_t caplog = h.meta & SMX_META_CAPLOG;
    if ((h.meta & SMX_META_USED) && caplog > SMX_INLINE_LOG) acc += 8ull << caplog;
  }
  for (uint32_t d = SMX_WARP / 2; d > 0; d >>= 1) acc += __shfl_xor_sync(SMX_FULL, acc, d);
  if (lane_id() == 0 && acc) atomicAdd(&V.ctl->scratch, acc);
}

/* ------------------------------------------------------------------------------------------
 * synthetic streams (SURVEY.md 8d) and roofline probes
 * ---------------------------------------------------------------------------------------- */
__device__ __forceinline__ void c2_op(ull seed, ull i, uint32_t rows, uint32_t ycols, uint32_t* x,
                                      uint32_t* y) {
  const ull r = smx_splitmix64(seed + i);
  *x = (uint32_t)((r >> 32) % rows) * 2654435761u;
  *y = 1u + (uint32_t)(r & 0xFFFFFFFFull) % ycols;
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_gen_c2_ops(ull seed, ull first, ull count, uint32_t rows, uint32_t ycols, uint32_t* xs,
             uint32_t* ys) {
  for (ull i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (ull)gridDim.x * blockDim.x)
    c2_op(seed, first + i, rows, ycols, &xs[i], &ys[i]);
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_gen_c2_queries(ull seed_get, ull seed_build, ull first, ull count, ull n_build, uint32_t rows,
                 uint32_t ycols, uint32_t* xs, uint32_t* ys) {
  for (ull i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (ull)gridDim.x * blockDim.x) {
    const ull j = first + i;
    const ull k = smx_splitmix64(seed_get + j) % n_build;
    uint32_t x, y;
    c2_op(seed_build, k, rows, ycols, &x, &y);
    if (j & 1ull) y += ycols;
    xs[i] = x;
    ys[i] = y;
  }
}

/* ---- C3 (co-occurrence build, examples/cf_recommender.c:35-47) and C4 (Zipf row lengths) --------
 * Both draw from a discrete distribution by inverse CDF: thr[k] = floor(2^64 * CDF(k+1)), k = 0..m-1,
 * built once on the host; draw(r) = 1 + #{k : thr[k] < r} — a binary search that the CPU baseline's
 * generator and the device do on the same table with the same counter-based r, so they see the same
 * stream. */
__host__ __device__ __forceinline__ uint32_t smx_draw(const ull* thr, uint32_t m, ull r) {
  uint32_t lo = 0, hi = m - 1u; /* thr[m-1] = 2^64 - 1: the answer is in [0, m-1] */
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (thr[mid] < r) lo = mid + 1u; else hi = mid;
  }
  return lo + 1u;
}
/* op i of the C3 stream: basket b = i / 64 holds 8 item ids; op k = i % 64 belongs to n = k / 8:
 * j = k % 8 == 0 -> (ids[n], 0), else (ids[n], ids[i']) with i' = the (j-1)-th index != n */
__host__ __device__ __forceinline__ void smx_c3_op(ull seed, ull i, const ull* thr, uint32_t items,
                                                    uint32_t* x, uint32_t* y) {
  const ull b = i >> 6;
  const uint32_t k = (uint32_t)(i & 63ull), n = k >> 3, j = k & 7u;
  *x = smx_draw(thr, items, smx_splitmix64(seed + b * 8ull + n));
  if (j == 0u) { *y = 0u; return; }
  const uint32_t other = (j - 1u < n) ? j - 1u : j;
  *y = smx_draw(thr, items, smx_splitmix64(seed + b * 8ull + other));
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_gen_c3_ops(ull seed, ull first, ull count, const ull* thr, uint32_t items, uint32_t* xs, uint32_t* ys) {
  for (ull i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (ull)gridDim.x * blockDim.x)
    smx_c3_op(seed, first + i, thr, items, &xs[i], &ys[i]);
}
/* C3 queries: query j re-generates build op k = r % n_build; odd j moves y out of the item range */
__global__ void __launch_bounds__(SMX_BLOCK)
k_gen_c3_queries(ull seed_get, ull seed_build, ull first, ull count, ull n_build, const ull* thr,
                 uint32_t items, uint32_t* xs, uint32_t* ys) {
  for (ull i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (ull)gridDim.x * blockDim.x) {
    const ull j = first + i;
    uint32_t x, y;
    smx_c3_op(seed_build, smx_splitmix64(seed_get + j) % n_build, thr, items, &x, &y);
    if (j & 1ull) y += items + 1u;
    xs[i] = x;
    ys[i] = y;
  }
}
/* C4: row r has len[r] = draw(thr, kmax, splitmix64(seed + r)) columns */
__global__ void __launch_bounds__(SMX_BLOCK)
k_gen_c4_lens(ull seed, ull first, ull count, const ull* thr, uint32_t kmax, uint32_t* lens) {
  for (ull i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (ull)gridDim.x * blockDim.x)
    lens[i] = smx_draw(thr, kmax, smx_splitmix64(seed + first + i));
}
/* murmur3 finaliser: a bijection on uint32 with f(0) = 0, so distinct non-zero inputs give distinct
 * non-zero columns */
__host__ __device__ __forceinline__ uint32_t smx_fmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
  return h;
}
/* op i of the C4 build: row r = the row whose range [offs[r], offs[r+1]) holds i, j = i - offs[r];
 * x = r * 2654435761, y = fmix32(j + salt_r) (salt_r in [1, 2^32 - 2^21]: j + salt never wraps and
 * is never 0), v = an odd 32-bit number */
__host__ __device__ __forceinline__ void smx_c4_op(ull seed, ull i, const ull* offs, uint32_t rows,
                                                    uint32_t* x, uint32_t* y, uint32_t* v) {
  uint32_t lo = 0, hi = rows - 1u; /* last r with offs[r] <= i */
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
    if (offs[mid] <= i) lo = mid; else hi = mid - 1u;
  }
  const uint32_t j = (uint32_t)(i - offs[lo]);
  const uint32_t salt = 1u + (uint32_t)(smx_splitmix64((seed ^ 0xC4C4C4C4ull) + lo) % 0xFFE00000ull);
  *x = lo * 2654435761u;
  *y = smx_fmix32(j + salt);
  *v = (uint32_t)(smx_splitmix64(seed + 0x5EED0000ull + i) >> 32) | 1u;
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_gen_c4_ops(ull seed, ull first, ull count, const ull* offs, uint32_t rows, uint32_t* xs, uint32_t* ys,
             uint32_t* vs) {
  for (ull i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (ull)gridDim.x * blockDim.x)
    smx_c4_op(seed, first + i, offs, rows, &xs[i], &ys[i], &vs[i]);
}

/* random reads of `width` bytes at width-aligned addresses; 4 independent loads in flight */
__global__ void __launch_bounds__(SMX_BLOCK)
k_probe_read(const char* buf, ull n_units, ull accesses, int width, smx_ctl_t* ctl) {
  ull acc = 0;
  const ull tid = blockIdx.x * blockDim.x + threadIdx.x;
  const ull nth = (ull)gridDim.x * blockDim.x;
  for (ull a = tid; a < accesses; a += nth) {
    const ull u = smx_splitmix64(a) % n_units;
    const char* p = buf + u * (ull)width;
    if (width == 32) {
      ull c[4];
      ld_sector_t<false>(p, c);
      acc ^= c[0] ^ c[1] ^ c[2] ^ c[3];
    } else if (width == 16) {
      const ull* q = (const ull*)p;
      acc ^= __ldcg(q) ^ __ldcg(q + 1);
    } else if (width == 8) {
      acc ^= __ldcg((const ull*)p);
    } else {
      acc ^= __ldcg((const uint32_t*)p);
    }
  }
  if (acc == 0x123456789abcdefull) atomicAdd(&ctl->scratch, acc); /* keep the loads alive */
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_probe_atomic(uint32_t* buf, ull n_words, ull accesses) {
  const ull tid = blockIdx.x * blockDim.x + threadIdx.x;
  const ull nth = (ull)gridDim.x * blockDim.x;
  for (ull a = tid; a < accesses; a += nth) atomicAdd(buf + smx_splitmix64(a) % n_words, 1u);
}

/* ------------------------------------------------------------------------------------------
 * K8: owner-rank bucketing for the multi-GPU router
 * ---------------------------------------------------------------------------------------- */
#define SMX_MAX_PARTS 256
#define PART_ITEMS 8
#define PART_TILE (SMX_BLOCK * PART_ITEMS)
#define PART_PER_LANE (SMX_MAX_PARTS / SMX_WARP)
/* part = owner rank (shift == 0xFFFFFFFF: mix_owner(x) % world) or directory slice
 * ((mix_row(x) & dir_mask) >> shift).  With split0 != 0 (slice mode, `world` = 2 * split0 parts)
 * ops on column 0 go to parts split0 .. 2*split0-1: the partitioned chunk is then
 * [other ops by slice | column-0 ops by slice], and the column-0 pass and the main pass each run
 * over a dense range instead of scanning the whole chunk with most lanes idle. */
__device__ __forceinline__ uint32_t part_of(uint32_t x, uint32_t y, uint32_t world, uint32_t dir_mask,
                                            uint32_t shift, uint32_t split0) {
  if (shift == 0xFFFFFFFFu) return smx_mix_owner(x) % world;
  const uint32_t sl = (smx_mix_row(x) & dir_mask) >> shift;
  return (split0 && y == 0u) ? sl + split0 : sl;
}
/* counts[part] += ops of that part */
__global__ void __launch_bounds__(SMX_BLOCK)
k_partition_count(const uint32_t* xs, const uint32_t* ys, uint32_t n, uint32_t world, uint32_t dir_mask,
                  uint32_t shift, uint32_t split0, ull* counts) {
  __shared__ uint32_t hist[2 * SMX_MAX_PARTS]; /* up to 256 slices + their column-0 twins */
  for (uint32_t k = threadIdx.x; k < world; k += blockDim.x) hist[k] = 0u;
  __syncthreads();
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    atomicAdd(&hist[part_of(xs[i], split0 ? ys[i] : 1u, world, dir_mask, shift, split0)], 1u);
  __syncthreads();
  for (uint32_t k = threadIdx.x; k < world; k += blockDim.x)
    if (hist[k]) atomicAdd(&counts[k], (ull)hist[k]);
}
/* cursors[p] = first output index of part p = exclusive prefix of counts (<= 256 parts: one thread;
 * the read path uses it so that no host round trip sits between the count and the scatter) */
__global__ void k_parts_prefix(const ull* counts, uint32_t parts, ull* cursors) {
#if defined(SMX_HOSTSIM) && SMX_WARP == 1
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ull at = 0ull;
    for (uint32_t p = 0; p < parts; ++p) {
      cursors[p] = at;
      at += counts[p];
    }
  }
#else
  /* one warp: lane l owns parts [8 l, 8 l + 8) — eight independent loads, a shuffle scan, eight stores */
  const uint32_t lane = threadIdx.x;
  ull c[PART_PER_LANE], sum = 0ull;
#pragma unroll
  for (int q = 0; q < PART_PER_LANE; ++q) {
    const uint32_t p = lane * PART_PER_LANE + q;
    c[q] = p < parts ? counts[p] : 0ull;
    sum += c[q];
  }
  ull incl = sum;
  for (uint32_t d = 1; d < SMX_WARP; d <<= 1) {
    const ull t = __shfl_up_sync(SMX_FULL, incl, d);
    if (lane >= d) incl += t;
  }
  ull run = incl - sum;
#pragma unroll
  for (int q = 0; q < PART_PER_LANE; ++q) {
    const uint32_t p = lane * PART_PER_LANE + q;
    if (p < parts) cursors[p] = run;
    run += c[q];
  }
#endif
}
/* Tiled partition: a block stages a tile of ops in shared memory sorted by part, reserves one
 * contiguous range per part with a single global atomic, and writes whole runs — so every
 * (tile, part) run reaches L2 as full sectors no matter how many parts there are.  Order inside a
 * part is not the input order (osrc carries the original index).
 * The kernel is latency-bound, not bandwidth-bound, so the tile loop is software-pipelined: the next
 * tile's x / y loads are issued before this tile is written out, the cursor atomics fly while the
 * tile is being staged, and every warp keeps its own copy of the (tiny) prefix table instead of
 * waiting at a barrier for one warp to build it. */
template <bool HAS_V, bool HAS_POS> /* shared memory only for what is used: 34 - 42 KB per block */
__global__ void __launch_bounds__(SMX_BLOCK)
k_partition_scatter(const uint32_t* xs, const uint32_t* ys, const uint32_t* vs, uint32_t n,
                    uint32_t world, uint32_t dir_mask, uint32_t shift, uint32_t split0, ull* cursors, uint32_t* oxs,
                    uint32_t* oys, uint32_t* ovs, uint32_t* osrc, const uint32_t* src_in,
                    uint32_t* opos, const ull* dst_tab, uint32_t src_bias) {
  __shared__ uint32_t s_x[PART_TILE], s_y[PART_TILE], s_i[PART_TILE];
  __shared__ uint32_t s_v[HAS_V ? PART_TILE : 1], s_p[HAS_POS ? PART_TILE : 1];
  __shared__ unsigned char s_part[PART_TILE];
  __shared__ uint32_t hist[2][SMX_MAX_PARTS];
  __shared__ unsigned short off[SMX_BLOCK / SMX_WARP][SMX_MAX_PARTS]; /* < PART_TILE */
  __shared__ ull gdelta[SMX_MAX_PARTS]; /* global index of a run's first op minus its place in the tile */
  if (!HAS_V) vs = nullptr;
  const bool want_pos = opos && !src_in; /* s_i = input position when src_in == NULL */
  const uint32_t lane = lane_id(), wib = threadIdx.x / SMX_WARP;
  unsigned short* myoff = off[wib];
  const uint32_t n_tiles = (n + PART_TILE - 1) / PART_TILE;
  for (uint32_t k = threadIdx.x; k < 2u * SMX_MAX_PARTS; k += blockDim.x) (&hist[0][0])[k] = 0u;
  uint32_t x[PART_ITEMS], y[PART_ITEMS];
  if (blockIdx.x < n_tiles) {
    const uint32_t base = blockIdx.x * PART_TILE;
#pragma unroll
    for (int k = 0; k < PART_ITEMS; ++k) {
      const uint32_t j = base + k * blockDim.x + threadIdx.x;
      x[k] = j < n ? xs[j] : 0u;
      y[k] = (ys && j < n) ? ys[j] : 0u;
    }
  }
  __syncthreads();
  uint32_t buf = 0;
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, buf ^= 1u) {
    const uint32_t base = tile * PART_TILE;
    const uint32_t cnt = (n - base < PART_TILE) ? n - base : PART_TILE;
    uint32_t* h = hist[buf];
    uint32_t pr[PART_ITEMS]; /* part << 16 | rank inside the tile's run */
#pragma unroll
    for (int k = 0; k < PART_ITEMS; ++k) {
      const uint32_t j = k * blockDim.x + threadIdx.x;
      if (j < cnt) {
        const uint32_t p = part_of(x[k], y[k], world, dir_mask, shift, split0);
        pr[k] = (p << 16) | atomicAdd(&h[p], 1u);
      }
    }
    __syncthreads(); /* (1) the tile's histogram is complete */
    /* reserve the runs: one global atomic per non-empty part, not waited for until the tile is staged */
#if !defined(SMX_HOSTSIM) || SMX_WARP > 1
    ull gb = 0ull;
    if (threadIdx.x < world && h[threadIdx.x]) gb = atomicAdd(&cursors[threadIdx.x], (ull)h[threadIdx.x]);
#endif
    { /* every warp: exclusive prefix of the histogram into its own table */
      uint32_t c[PART_PER_LANE], sum = 0u;
#pragma unroll
      for (int q = 0; q < PART_PER_LANE; ++q) {
        c[q] = h[lane * PART_PER_LANE + q];
        sum += c[q];
      }
      uint32_t incl = sum;
      for (uint32_t d = 1; d < SMX_WARP; d <<= 1) {
        const uint32_t t = __shfl_up_sync(SMX_FULL, incl, d);
        if (lane >= d) incl += t;
      }
      uint32_t run = incl - sum;
#pragma unroll
      for (int q = 0; q < PART_PER_LANE; ++q) {
        myoff[lane * PART_PER_LANE + q] = (unsigned short)run;
        run += c[q];
      }
      __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < PART_ITEMS; ++k) {
      const uint32_t j = k * blockDim.x + threadIdx.x;
      if (j < cnt) {
        const uint32_t p = pr[k] >> 16;
        const uint32_t at = myoff[p] + (pr[k] & 0xFFFFu);
        s_x[at] = x[k];
        s_y[at] = y[k];
        s_part[at] = (unsigned char)p;
        if (vs) s_v[at] = vs[base + j];
        s_i[at] = src_in ? src_in[base + j] : base + j; /* carry the caller's order index */
      }
    }
    { /* next tile's loads fly while this one is written out */
      const uint32_t next = tile + gridDim.x;
      if (next < n_tiles) {
        const uint32_t nb = next * PART_TILE;
#pragma unroll
        for (int k = 0; k < PART_ITEMS; ++k) {
          const uint32_t j = nb + k * blockDim.x + threadIdx.x;
          x[k] = j < n ? xs[j] : 0u;
          y[k] = (ys && j < n) ? ys[j] : 0u;
        }
      }
    }
#if defined(SMX_HOSTSIM) && SMX_WARP == 1
    for (uint32_t k = threadIdx.x; k < world; k += blockDim.x)
      gdelta[k] = (h[k] ? atomicAdd(&cursors[k], (ull)h[k]) : 0ull) - myoff[k];
#else
    if (threadIdx.x < world) gdelta[threadIdx.x] = gb - myoff[threadIdx.x];
#endif
    for (uint32_t k = threadIdx.x; k < SMX_MAX_PARTS; k += blockDim.x) hist[buf ^ 1u][k] = 0u; /* for the next tile */
    __syncthreads(); /* (2) the tile is staged and its runs are reserved */
    for (uint32_t j = threadIdx.x; j < cnt; j += blockDim.x) {
      const uint32_t xx = s_x[j];
      const uint32_t p = s_part[j];
      ull at = gdelta[p] + j;
      if (dst_tab) {
        /* fused with the exchange: part p's run goes straight into owner p's inbox — a peer
         * mapping over NVLink (or local memory for p == this rank).  dst_tab = [x | y | v | src |
         * pos_base][world]; the cursors started at 0, so `at` is the index inside my segment. */
        ((uint32_t*)dst_tab[p])[at] = xx;
        if (ys) ((uint32_t*)dst_tab[world + p])[at] = s_y[j];
        if (vs) ((uint32_t*)dst_tab[2 * world + p])[at] = s_v[j];
        if (dst_tab[3 * world + p]) ((uint32_t*)dst_tab[3 * world + p])[at] = s_i[j] + src_bias;
        at += dst_tab[4 * world + p]; /* position in the requester's routed order, for opos */
      } else {
        oxs[at] = xx;
        if (ys) oys[at] = s_y[j];
        if (vs) ovs[at] = s_v[j];
        if (osrc) osrc[at] = s_i[j] + src_bias;
      }
      /* inverse permutation, for reads: input position -> routed position (staged in shared
       * memory so that it is written coalesced).  A tile's ops land in one run per part, so a
       * later gather through opos reads long contiguous runs. */
      if (want_pos) {
        if (HAS_POS) s_p[s_i[j] - base] = (uint32_t)at;
        else opos[s_i[j]] = (uint32_t)at; /* values AND positions: no caller on a hot path, no staging */
      }
    }
    if (HAS_POS && want_pos) {
      __syncthreads();
      for (uint32_t j = threadIdx.x; j < cnt; j += blockDim.x) opos[base + j] = s_p[j];
    }
    __syncthreads(); /* (3) before the next tile overwrites the staging arrays */
  }
}

/* out[i] = vals[pos[i]]: un-permute routed answers into input order.  A block takes one scatter tile
 * (PART_TILE consecutive inputs): the tile's ops sit in one contiguous run per part of the routed
 * order, so every sector of `vals` the block touches is used up by the block itself (L1), and a
 * thread's PART_ITEMS loads are independent. */
__global__ void __launch_bounds__(SMX_BLOCK)
k_gather(uint32_t* out, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ pos, uint32_t n) {
  const ull base = (ull)blockIdx.x * PART_TILE;
  uint32_t p[PART_ITEMS];
#pragma unroll
  for (int k = 0; k < PART_ITEMS; ++k) {
    const ull i = base + (ull)k * SMX_BLOCK + threadIdx.x;
    p[k] = i < n ? pos[i] : 0u;
  }
#pragma unroll
  for (int k = 0; k < PART_ITEMS; ++k) {
    const ull i = base + (ull)k * SMX_BLOCK + threadIdx.x;
    if (i < n) out[i] = vals[p[k]];
  }
}
/* the same as a resident grid with a stride loop (kept as the B side of the A/B: SMX_GET_STRIDE_GATHER) */
__global__ void __launch_bounds__(SMX_BLOCK)
k_gather_stride(uint32_t* out, const uint32_t* vals, const uint32_t* pos, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = vals[pos[i]];
}

/* getrow across ranks: the requester hands every routed row its output offset.  pos[i] = routed
 * position of my row i (runs by owner, run o starts at tab[o]); the offset goes to owner o's array
 * (address tab[world + o], peer memory) at the row's index inside the run. */
__global__ void __launch_bounds__(SMX_BLOCK)
k_route_offsets(const ull* offs, const uint32_t* pos, uint32_t n, uint32_t world, const ull* tab) {
  __shared__ ull s_tab[2 * 64];
  for (uint32_t k = threadIdx.x; k < 2u * world; k += blockDim.x) s_tab[k] = tab[k];
  __syncthreads();
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const ull p = pos[i];
    uint32_t o = 0;
    while (o + 1u < world && s_tab[o + 1u] <= p) ++o; /* runs may be empty: take the LAST run starting at or before p */
    ((ull*)s_tab[world + o])[p - s_tab[o]] = offs[i];
  }
}

/* ==========================================================================================
 * launchers
 * ======================================================================================== */
static int g_blocks = 0;
extern "C" int smx_grid_blocks(void) {
  if (!g_blocks) {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    g_blocks = sms * 8; /* 8 x 256 threads = 2048 resident threads per SM */
  }
  return g_blocks;
}
static inline uint32_t grid_for(ull items) {
  ull want = (items + SMX_BLOCK - 1) / SMX_BLOCK;
  ull cap = (ull)smx_grid_blocks();
  if (want < 1) want = 1;
  return (uint32_t)(want < cap ? want : cap);
}

extern "C" void smx_launch_upsert(smx_stream_t st, smx_view_t v, smx_ops_t ops, smx_lists_t l,
                                  int op, int pass, const uint32_t* list, uint32_t m,
                                  int preaggregate) {
  if (m == 0) return;
  /* NOT a persistent grid: one block per 4 x 256 ops, so blocks retire continuously and kernels of
   * other streams (uploads of the next host-array piece, a second handle's kernels) interleave with an update in
   * flight instead of waiting for 1184 resident blocks to drain */
  ull want_blocks = ((ull)m + 4ull * SMX_BLOCK - 1) / (4ull * SMX_BLOCK);
  if (want_blocks < 1) want_blocks = 1;
  const uint32_t grid = (uint32_t)want_blocks;
  const int pre = (preaggregate && !list && pass != SMX_PASS_LATE && SMX_WARP > 1) ? 1 : 0;
  if (op == SMX_OP_INCR) {
    auto k = k_upsert<SMX_OP_INCR>;
    SMX_LAUNCH(k, grid, SMX_BLOCK, st, v, ops, l, pass, list, m, pre);
  } else if (op == SMX_OP_DECR) {
    auto k = k_upsert<SMX_OP_DECR>;
    SMX_LAUNCH(k, grid, SMX_BLOCK, st, v, ops, l, pass, list, m, pre);
  } else {
    auto k = k_upsert<SMX_OP_SETZERO>;
    SMX_LAUNCH(k, grid, SMX_BLOCK, st, v, ops, l, pass, list, m, pre);
  }
}

extern "C" void smx_launch_grow_plan(smx_stream_t st, smx_view_t v, smx_lists_t l, uint32_t n_grow) {
  if (!n_grow) return;
  SMX_LAUNCH(k_grow_plan, grid_for(n_grow), SMX_BLOCK, st, v, l, n_grow);
}

extern "C" void smx_launch_free_push(smx_stream_t st, smx_view_t v, smx_lists_t l, uint32_t n_grow) {
  if (!n_grow) return;
  SMX_LAUNCH(k_free_push, grid_for(n_grow), SMX_BLOCK, st, v, l, n_grow);
}

extern "C" void smx_launch_migrate(smx_stream_t st, smx_view_t v, smx_lists_t l, uint32_t n_grow,
                                   uint32_t n_mid, uint32_t n_big, void* region, int skip_big) {
  if (!n_grow) return;
  if (n_grow > n_mid + n_big)
    SMX_LAUNCH(k_migrate, grid_for((ull)n_grow * SMX_WARP), SMX_BLOCK, st, v, l, n_grow, (char*)region);
  if (n_mid) {
    const uint32_t cap = (uint32_t)smx_grid_blocks();
    SMX_LAUNCH(k_migrate_mid, n_mid < cap ? n_mid : cap, SMX_BLOCK, st, v, l, n_mid, (char*)region);
  }
  if (skip_big) return; /* the caller re-places the big rows with smx_launch_migrate_tiles */
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    dim3 grid(SMX_WARP > 1 ? 64u : 2u, cnt, 1u);
    SMX_LAUNCH(k_migrate_big, grid, SMX_BLOCK, st, v, l, first, (char*)region);
  }
  if (n_big) SMX_LAUNCH(k_migrate_big_finish, grid_for(n_big), SMX_BLOCK, st, v, l, n_big, (char*)region);
}

extern "C" void smx_launch_migrate_tiles(smx_stream_t st, smx_view_t v, smx_lists_t l, uint32_t n_big, void* region,
                                         unsigned long long* spill, uint32_t spill_cap) {
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    dim3 grid(SMX_WARP > 1 ? 32u : 2u, cnt, 1u);
    SMX_LAUNCH(k_migrate_tiles, grid, SMX_BLOCK, st, v, l, first, (char*)region, (ull*)spill, spill_cap);
  }
}
extern "C" void smx_launch_migrate_tiles_finish(smx_stream_t st, smx_view_t v, smx_lists_t l, uint32_t n_big, void* region,
                                                const unsigned long long* spill, uint32_t n_spill) {
  if (n_spill) SMX_LAUNCH(k_spill_insert, grid_for(n_spill), SMX_BLOCK, st, v, l, (char*)region, (const ull*)spill, n_spill);
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    dim3 grid(SMX_WARP > 1 ? 32u : 2u, cnt, 1u);
    SMX_LAUNCH(k_zero_old_big, grid, SMX_BLOCK, st, v, l, first);
  }
  if (n_big) SMX_LAUNCH(k_migrate_big_finish, grid_for(n_big), SMX_BLOCK, st, v, l, n_big, (char*)region);
}
extern "C" void smx_launch_sketch(smx_stream_t st, const uint32_t* xs, uint32_t n, uint32_t* bitmap,
                                  uint32_t bits_log, smx_ctl_t* ctl) {
  if (!n) return;
  SMX_LAUNCH(k_sketch_set, grid_for(n), SMX_BLOCK, st, xs, n, bitmap, bits_log);
  SMX_LAUNCH(k_sketch_count, grid_for((1ull << bits_log) / 32u), SMX_BLOCK, st, (const uint32_t*)bitmap, bits_log, ctl);
}
extern "C" void smx_launch_live_bytes(smx_stream_t st, smx_view_t v) {
  SMX_LAUNCH(k_live_bytes, grid_for(v.dir_cap), SMX_BLOCK, st, v);
}

extern "C" void smx_launch_dir_rehash(smx_stream_t st, smx_view_t from, smx_view_t to) {
  SMX_LAUNCH(k_dir_rehash, grid_for(from.dir_cap), SMX_BLOCK, st, from, to);
}

extern "C" void smx_launch_finalize_t0(smx_stream_t st, smx_view_t v, const uint32_t* t0rows,
                                       uint32_t n) {
  if (!n) return;
  SMX_LAUNCH(k_finalize_t0, grid_for(n), SMX_BLOCK, st, v, t0rows, n);
}

extern "C" void smx_launch_sync_rowlen(smx_stream_t st, smx_view_t v, const uint32_t* rows, uint32_t n) {
  if (!n) return;
  SMX_LAUNCH(k_sync_rowlen, grid_for(n), SMX_BLOCK, st, v, rows, n);
}

extern "C" void smx_launch_set_max(smx_stream_t st, smx_view_t v, smx_ops_t ops, uint64_t* addrs) {
  if (!ops.n) return;
  SMX_LAUNCH(k_set_max, grid_for(ops.n), SMX_BLOCK, st, v, ops, (ull*)addrs);
}
extern "C" void smx_launch_set_commit(smx_stream_t st, smx_ops_t ops, uint64_t* addrs) {
  if (!ops.n) return;
  SMX_LAUNCH(k_set_mark, grid_for(ops.n), SMX_BLOCK, st, ops, (ull*)addrs);
  SMX_LAUNCH(k_set_commit, grid_for(ops.n), SMX_BLOCK, st, ops, (const ull*)addrs);
}


/* scratch layout for smx_launch_batch_out (all sized n): addrs[2] (u64), idx[2] (u32), seg (u64),
 * tile_agg (u64, smx_scan_scratch_items(n)), plus the sort's temporary storage */
extern "C" size_t smx_batch_out_sort_bytes(uint32_t n) {
#ifdef SMX_HOSTSIM
  (void)n;
  return 64;
#else
  size_t bytes = 0, bytes32 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const ull*)nullptr, (ull*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)n, 0, 48);
  cub::DeviceRadixSort::SortPairs(nullptr, bytes32, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)n, 0, 32);
  return (bytes > bytes32 ? bytes : bytes32) + 256;
#endif
}
__global__ void __launch_bounds__(SMX_BLOCK)
k_permute_addrs(const ull* addrs, const uint32_t* order, uint32_t n, ull* out) {
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) out[k] = addrs[order[k]];
}
/* ops.idx == NULL: input order = array order.  Otherwise ops.idx[i] is op i's place in the input order (the
 * multi-GPU router hands over permuted batches): the ops are first ordered by that index, then stably by
 * cell, so inside a cell's group they are in input order again. */
extern "C" void smx_launch_batch_out(smx_stream_t st, smx_view_t v, smx_ops_t ops, int op, uint32_t* out,
                                     uint64_t* addrs_a, uint64_t* addrs_b, uint32_t* idx_a, uint32_t* idx_b,
                                     uint64_t* seg, uint64_t* tile_agg, void* sort_tmp, size_t sort_bytes) {
  if (!ops.n) return;
  const uint32_t n = ops.n;
  if (op == SMX_OP_SETZERO) { /* set: the value just written */
    SMX_LAUNCH(k_fill_out, grid_for(n), SMX_BLOCK, st, ops, out);
    return;
  }
  SMX_LAUNCH(k_find_addr, grid_for(n), SMX_BLOCK, st, v, ops, (ull*)addrs_a, idx_a);
  const ull* s_addr = (const ull*)addrs_b; /* sorted cell addresses / op indices end up here */
  const uint32_t* s_idx = idx_b;
#ifdef SMX_HOSTSIM
  (void)sort_tmp; (void)sort_bytes;
  {
    std::vector<uint32_t> order(n);
    for (uint32_t i = 0; i < n; i++) order[i] = i;
    const uint32_t* ords = ops.idx;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
      if (addrs_a[a] != addrs_a[b]) return addrs_a[a] < addrs_a[b];
      return ords ? ords[a] < ords[b] : false;
    });
    for (uint32_t p = 0; p < n; p++) { addrs_b[p] = addrs_a[order[p]]; idx_b[p] = order[p]; }
  }
#else
  /* LSD radix sort: stable, so ops of one cell stay in input order (device addresses fit in 48 bits) */
  if (ops.idx) {
    cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, ops.idx, out /* scratch for the sorted keys */,
                                    (const uint32_t*)idx_a, idx_b, (int)n, 0, 32, (cudaStream_t)st);
    SMX_LAUNCH(k_permute_addrs, grid_for(n), SMX_BLOCK, st, (const ull*)addrs_a, (const uint32_t*)idx_b, n, (ull*)addrs_b);
    cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, (const ull*)addrs_b, (ull*)addrs_a, (const uint32_t*)idx_b,
                                    idx_a, (int)n, 0, 48, (cudaStream_t)st);
    s_addr = (const ull*)addrs_a;
    s_idx = idx_a;
  } else {
    cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, (const ull*)addrs_a, (ull*)addrs_b, (const uint32_t*)idx_a,
                                    idx_b, (int)n, 0, 48, (cudaStream_t)st);
  }
#endif
  const int negate = (op == SMX_OP_DECR) ? 1 : 0;
  const uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  SMX_LAUNCH(k_out_gather, grid_for(n), SMX_BLOCK, st, ops, negate, s_addr, s_idx, (ull*)seg);
  SMX_LAUNCH(k_seg_tile, tiles, SMX_BLOCK, st, (const ull*)seg, n, (ull*)tile_agg);
  SMX_LAUNCH(k_seg_tiles, 1, 1, st, (ull*)tile_agg, tiles);
  SMX_LAUNCH(k_seg_apply, tiles, SMX_BLOCK, st, (ull*)seg, n, (const ull*)tile_agg);
  SMX_LAUNCH(k_out_write, grid_for(n), SMX_BLOCK, st, ops, negate, s_addr, s_idx, (const ull*)seg, out);
}

extern "C" void smx_launch_get_tiled(smx_stream_t st, smx_view_t v, const uint32_t* xs, const uint32_t* ys,
                                     uint32_t n, uint32_t* out, int once) {
  if (!n) return;
  const uint32_t grid = (uint32_t)(((ull)n + GET_TILE_ITEMS * SMX_BLOCK - 1) / (GET_TILE_ITEMS * SMX_BLOCK));
  if (once) {
    auto k = k_get_tiled<true>;
    SMX_LAUNCH(k, grid, SMX_BLOCK, st, v, xs, ys, n, out);
  } else {
    auto k = k_get_tiled<false>;
    SMX_LAUNCH(k, grid, SMX_BLOCK, st, v, xs, ys, n, out);
  }
}
extern "C" void smx_launch_get(smx_stream_t st, smx_view_t v, const uint32_t* xs, const uint32_t* ys,
                               uint32_t n, uint32_t* out) {
  if (!n) return;
  SMX_LAUNCH(k_get, grid_for(n), SMX_BLOCK, st, v, xs, ys, n, out);
}
extern "C" void smx_launch_rowlen(smx_stream_t st, smx_view_t v, const uint32_t* xs, uint32_t n,
                                  uint32_t* out) {
  if (!n) return;
  SMX_LAUNCH(k_rowlen, grid_for(n), SMX_BLOCK, st, v, xs, n, out);
}
extern "C" void smx_launch_row_counts(smx_stream_t st, smx_view_t v, const uint32_t* xs, uint32_t n,
                                      uint32_t* counts, uint64_t* info, uint32_t* big_list, uint32_t* big_counter) {
  if (!n) return;
  SMX_LAUNCH(k_row_counts, grid_for(n), SMX_BLOCK, st, v, xs, n, counts, (ull*)info, big_list, big_counter);
}

extern "C" uint32_t smx_scan_scratch_items(uint32_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE + 1; }

extern "C" void smx_launch_scan(smx_stream_t st, const uint32_t* counts, uint32_t n, uint64_t base,
                                uint64_t* offsets, uint64_t* tile_sums) {
  const uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (tiles) SMX_LAUNCH(k_scan_tile_sums, tiles, SMX_BLOCK, st, counts, n, (ull*)tile_sums);
  SMX_LAUNCH(k_scan_tiles, 1, SMX_BLOCK, st, (ull*)tile_sums, tiles, (ull)base, (ull*)offsets, n);
  if (tiles) SMX_LAUNCH(k_scan_apply, tiles, SMX_BLOCK, st, counts, n, (const ull*)tile_sums, (ull*)offsets);
}

extern "C" void smx_launch_getrow_fill(smx_stream_t st, smx_view_t v, const uint64_t* info, uint32_t n,
                                       const uint64_t* offsets, uint64_t bias, uint32_t* pairs,
                                       const uint32_t* big_list, uint32_t n_big, uint32_t* cursors) {
  if (!n) return;
  SMX_LAUNCH(k_getrow_inline, grid_for(n), SMX_BLOCK, st, v, (const ull*)info, n, (const ull*)offsets, (ull)bias, pairs);
  SMX_LAUNCH(k_getrow_fill, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, v, (const ull*)info, n,
             (const ull*)offsets, (ull)bias, pairs);
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    dim3 grid(SMX_WARP > 1 ? GETROW_BLOCKS_PER_ROW : 2u, cnt, 1u);
    SMX_LAUNCH(k_getrow_chunks, grid, SMX_BLOCK, st, v, (const ull*)info, big_list, first, (const ull*)offsets,
               (ull)bias, pairs, cursors);
  }
}

extern "C" void smx_launch_list_rows(smx_stream_t st, smx_view_t v, uint32_t* keys, uint32_t* counter) {
  SMX_LAUNCH(k_list_rows, grid_for(v.dir_cap), SMX_BLOCK, st, v, keys, counter);
}
extern "C" void smx_launch_row_slog(smx_stream_t st, smx_view_t v, const uint32_t* xs, uint32_t n,
                                    uint32_t* out) {
  if (!n) return;
  SMX_LAUNCH(k_row_slog, grid_for(n), SMX_BLOCK, st, v, xs, n, out);
}
extern "C" void smx_launch_snap_units(smx_stream_t st, const uint32_t* counts, const uint32_t* slogs, uint32_t n,
                                      uint32_t* units) {
  if (!n) return;
  SMX_LAUNCH(k_snap_units, grid_for(n), SMX_BLOCK, st, counts, slogs, n, units);
}
/* out must be zeroed; offsets in 8-byte units (n + 1 entries) */
extern "C" void smx_launch_snap_rows(smx_stream_t st, smx_view_t v, const uint64_t* info, uint32_t n,
                                     const uint64_t* offsets, uint64_t* out, const uint32_t* big_list, uint32_t n_big) {
  if (!n) return;
  SMX_LAUNCH(k_snap_rows, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, v, (const ull*)info, n, (const ull*)offsets, (ull*)out);
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    dim3 grid(SMX_WARP > 1 ? 32u : 2u, cnt, 1u);
    SMX_LAUNCH(k_snap_big, grid, SMX_BLOCK, st, v, (const ull*)info, big_list, first, (const ull*)offsets, (ull*)out, 1, 0);
    SMX_LAUNCH(k_snap_big, grid, SMX_BLOCK, st, v, (const ull*)info, big_list, first, (const ull*)offsets, (ull*)out, 3, 1);
    SMX_LAUNCH(k_snap_big, grid, SMX_BLOCK, st, v, (const ull*)info, big_list, first, (const ull*)offsets, (ull*)out, 3, 0);
  }
}
extern "C" void smx_launch_load_fixup(smx_stream_t st, smx_view_t v, const uint32_t* xs,
                                      const uint32_t* slogs, uint32_t n) {
  if (!n) return;
  SMX_LAUNCH(k_load_fixup, grid_for(n), SMX_BLOCK, st, v, xs, slogs, n);
}
extern "C" void smx_launch_load_count(smx_stream_t st, const void* raw, const smx_load_tile_t* tiles, uint32_t n,
                                      uint32_t* counts) {
  if (!n) return;
  SMX_LAUNCH(k_load_count, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, (const unsigned char*)raw, tiles, n, counts);
}
extern "C" void smx_launch_load_emit(smx_stream_t st, const void* raw, const smx_load_tile_t* tiles, uint32_t n,
                                     const uint64_t* offsets, uint32_t* xs, uint32_t* ys, uint32_t* vs) {
  if (!n) return;
  SMX_LAUNCH(k_load_emit, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, (const unsigned char*)raw, tiles, n,
             (const ull*)offsets, xs, ys, vs);
}
extern "C" void smx_launch_cf_scores(smx_stream_t st, smx_view_t v, const uint32_t* items, uint32_t n,
                                     const uint64_t* offsets, const uint32_t* pairs, uint32_t* ids,
                                     double* scores) {
  if (!n) return;
  SMX_LAUNCH(k_cf_scores, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, v, items, n, (const ull*)offsets,
             pairs, ids, scores);
}
extern "C" void smx_launch_pair_cols(smx_stream_t st, const uint32_t* pairs, uint64_t total, uint32_t* cols) {
  if (!total) return;
  SMX_LAUNCH(k_pair_cols, grid_for(total), SMX_BLOCK, st, pairs, (ull)total, cols);
}
extern "C" void smx_launch_cf_scores_totals(smx_stream_t st, uint32_t n, const uint64_t* offsets, const uint32_t* pairs,
                                            const uint32_t* a_tot, const uint32_t* b_tot, uint32_t* ids, double* scores) {
  if (!n) return;
  SMX_LAUNCH(k_cf_scores_totals, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, n, (const ull*)offsets, pairs, a_tot,
             b_tot, ids, scores);
}
extern "C" uint32_t smx_topk_max_passes(void) { return 96u / TOPK_DIGIT_BITS; }
extern "C" size_t smx_topk_big_bytes(uint32_t n_big) {
  return (size_t)n_big * (sizeof(topk_state_t) + TOPK_RADIX * 4u);
}
extern "C" void smx_launch_topk_small(smx_stream_t st, uint32_t n, const uint64_t* offsets, const uint32_t* ids,
                                      const double* scores, uint32_t k, uint32_t* counts, uint32_t* out_ids,
                                      double* out_scores) {
  if (!n) return;
  SMX_LAUNCH(k_topk_warp, grid_for((ull)n * SMX_WARP), SMX_BLOCK, st, n, (const ull*)offsets, ids, scores, k, counts,
             out_ids, out_scores);
  const uint32_t cap = (uint32_t)smx_grid_blocks();
  SMX_LAUNCH(k_topk_block, n < cap ? n : cap, SMX_BLOCK, st, n, (const ull*)offsets, ids, scores, k, counts, out_ids,
             out_scores);
}
extern "C" void smx_launch_topk_classify(smx_stream_t st, uint32_t n, const uint64_t* offsets, uint32_t* big_list,
                                         uint32_t* ctl) {
  if (!n) return;
  SMX_LAUNCH(k_topk_classify, grid_for(n), SMX_BLOCK, st, n, (const ull*)offsets, big_list, ctl);
}
extern "C" void smx_launch_topk_init(smx_stream_t st, const uint32_t* big_list, uint32_t n_big, const uint64_t* offsets,
                                     void* big_scratch, uint32_t* ctl) {
  if (!n_big) return;
  SMX_LAUNCH(k_topk_init, grid_for(n_big), SMX_BLOCK, st, big_list, n_big, (const ull*)offsets,
             (topk_state_t*)big_scratch, (ull*)(ctl + 4));
}
extern "C" void smx_launch_topk_pass(smx_stream_t st, void* big_scratch, uint32_t n_big, uint32_t k,
                                     const uint32_t* ids, const double* scores, uint32_t* c_ids, double* c_scores,
                                     uint32_t* ctl) {
  topk_state_t* state = (topk_state_t*)big_scratch;
  uint32_t* hist = (uint32_t*)(state + n_big);
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    SMX_LAUNCH(k_topk_hist, dim3(TOPK_BIG_BLOCKS, cnt, 1u), SMX_BLOCK, st, state, first, ids, scores, c_ids, c_scores,
               hist);
  }
  SMX_LAUNCH(k_topk_pick, grid_for(n_big), SMX_BLOCK, st, state, n_big, k, hist, ctl + 1);
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    SMX_LAUNCH(k_topk_compact, dim3(TOPK_BIG_BLOCKS, cnt, 1u), SMX_BLOCK, st, state, first, ids, scores, c_ids,
               c_scores);
  }
}
extern "C" void smx_launch_topk_finish(smx_stream_t st, const void* big_scratch, uint32_t n_big, const uint32_t* c_ids,
                                       const double* c_scores, uint32_t k, uint32_t* counts, uint32_t* out_ids,
                                       double* out_scores) {
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    SMX_LAUNCH(k_topk_finish, cnt, SMX_BLOCK, st, (const topk_state_t*)big_scratch, first, c_ids, c_scores, k, counts,
               out_ids, out_scores);
  }
}
extern "C" void smx_launch_topk_cut(smx_stream_t st, const uint64_t* offsets, uint32_t n, uint32_t lo, uint64_t budget,
                                    uint32_t* out) {
  SMX_LAUNCH(k_topk_cut, 1, 1, st, (const ull*)offsets, n, lo, (ull)budget, out);
}

static inline int rec_key_bits(uint32_t n) { /* 32 id bits + enough for slots 0 .. n-1 */
  int b = 32;
  while (b < 64 && (1ull << (b - 32)) < (ull)n) b++;
  return b;
}
extern "C" size_t smx_rec_sort_bytes(uint32_t n) {
#ifdef SMX_HOSTSIM
  (void)n;
  return 64;
#else
  size_t bytes = 0, bytes_keys = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const ull*)nullptr, (ull*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)n, 0, 64);
  cub::DeviceRadixSort::SortKeys(nullptr, bytes_keys, (const ull*)nullptr, (ull*)nullptr, (int)n, 0, 64);
  return (bytes > bytes_keys ? bytes : bytes_keys) + 256;
#endif
}
extern "C" void smx_launch_rec_items(smx_stream_t st, uint32_t nb, const uint64_t* boff, uint64_t base,
                                     const uint32_t* items, uint32_t n_pos, uint64_t* keys, uint64_t* sitems,
                                     void* sort_tmp, size_t sort_bytes) {
  if (!n_pos) return;
  SMX_LAUNCH(k_rec_item_keys, grid_for((ull)nb * SMX_WARP), SMX_BLOCK, st, nb, (const ull*)boff, (ull)base, items,
             (ull*)keys);
#ifdef SMX_HOSTSIM
  (void)sort_tmp; (void)sort_bytes;
  memcpy(sitems, keys, (size_t)n_pos * 8);
  std::sort(sitems, sitems + n_pos);
#else
  cub::DeviceRadixSort::SortKeys(sort_tmp, sort_bytes, (const ull*)keys, (ull*)sitems, (int)n_pos, 0, rec_key_bits(nb),
                                 (cudaStream_t)st);
#endif
}
extern "C" void smx_launch_rec_small(smx_stream_t st, uint32_t nb, const uint64_t* boff, uint64_t base,
                                     const uint64_t* off, const uint32_t* ids, const double* scores,
                                     const uint64_t* sitems, uint32_t* big_list, uint32_t* ctl, uint32_t* t_ids,
                                     double* t_scores, uint32_t* cnt) {
  if (!nb) return;
  SMX_LAUNCH(k_rec_classify, grid_for(nb), SMX_BLOCK, st, nb, (const ull*)boff, (ull)base, (const ull*)off, big_list,
             ctl);
  SMX_LAUNCH(k_rec_warp, grid_for((ull)nb * SMX_WARP), SMX_BLOCK, st, nb, (const ull*)boff, (ull)base, (const ull*)off,
             ids, scores, (const ull*)sitems, t_ids, t_scores, cnt);
  const uint32_t cap = (uint32_t)smx_grid_blocks();
  SMX_LAUNCH(k_rec_block, nb < cap ? nb : cap, SMX_BLOCK, st, nb, (const ull*)boff, (ull)base, (const ull*)off, ids,
             scores, (const ull*)sitems, t_ids, t_scores, cnt);
}
extern "C" void smx_launch_rec_big(smx_stream_t st, const uint32_t* big_list, uint32_t n_big, uint32_t n_pairs,
                                   const uint64_t* boff, uint64_t base, const uint64_t* off, const uint32_t* ids,
                                   const uint64_t* sitems, uint32_t* lens, uint64_t* big_off, uint64_t* keys_a,
                                   uint64_t* keys_b, uint32_t* vals_a, uint32_t* vals_b, uint32_t* flags,
                                   uint64_t* fpos, uint64_t* scan_tmp, void* sort_tmp, size_t sort_bytes,
                                   uint32_t* cnt) {
  if (!n_big) return;
  SMX_LAUNCH(k_rec_big_lens, grid_for(n_big), SMX_BLOCK, st, big_list, n_big, (const ull*)boff, (ull)base,
             (const ull*)off, lens);
  smx_launch_scan(st, lens, n_big, 0, big_off, scan_tmp);
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t c = (n_big - first < 32768u) ? n_big - first : 32768u;
    SMX_LAUNCH(k_rec_big_keys, dim3(TOPK_BIG_BLOCKS, c, 1u), SMX_BLOCK, st, big_list, first, (const ull*)boff,
               (ull)base, (const ull*)off, ids, (const ull*)big_off, (ull*)keys_a, vals_a);
  }
#ifdef SMX_HOSTSIM
  (void)sort_tmp; (void)sort_bytes;
  {
    std::vector<uint32_t> order(n_pairs);
    for (uint32_t p = 0; p < n_pairs; p++) order[p] = p;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return keys_a[a] < keys_a[b]; });
    for (uint32_t p = 0; p < n_pairs; p++) { keys_b[p] = keys_a[order[p]]; vals_b[p] = vals_a[order[p]]; }
  }
#else
  /* LSD radix sort: stable, so the pairs of one (basket, id) stay in position order */
  cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, (const ull*)keys_a, (ull*)keys_b, (const uint32_t*)vals_a,
                                  vals_b, (int)n_pairs, 0, rec_key_bits(n_big), (cudaStream_t)st);
#endif
  SMX_LAUNCH(k_rec_big_flag, grid_for(n_pairs), SMX_BLOCK, st, (const ull*)keys_b, n_pairs, big_list, (const ull*)boff,
             (ull)base, (const ull*)sitems, flags);
  smx_launch_scan(st, flags, n_pairs, 0, fpos, scan_tmp);
  SMX_LAUNCH(k_rec_big_count, grid_for(n_big), SMX_BLOCK, st, big_list, n_big, (const ull*)big_off, (const ull*)fpos,
             cnt);
}
extern "C" void smx_launch_rec_emit(smx_stream_t st, uint32_t nb, const uint64_t* boff, uint64_t base,
                                    const uint64_t* off, const double* scores, const uint32_t* cnt,
                                    const uint64_t* red_off, const uint32_t* t_ids, const double* t_scores,
                                    const uint32_t* big_list, uint32_t n_big, uint32_t n_pairs, const uint64_t* big_off,
                                    const uint64_t* keys, const uint32_t* vals, const uint64_t* fpos, uint32_t* r_ids,
                                    double* r_scores) {
  if (!nb) return;
  SMX_LAUNCH(k_rec_compact, grid_for((ull)nb * SMX_WARP), SMX_BLOCK, st, nb, (const ull*)boff, (ull)base,
             (const ull*)off, cnt, (const ull*)red_off, t_ids, t_scores, r_ids, r_scores);
  if (n_big)
    SMX_LAUNCH(k_rec_big_emit, grid_for(n_pairs), SMX_BLOCK, st, (const ull*)keys, vals, n_pairs, big_list,
               (const ull*)big_off, (const ull*)boff, (ull)base, (const ull*)off, scores, (const ull*)fpos,
               (const ull*)red_off, r_ids, r_scores);
}
extern "C" void smx_launch_rec_cut(smx_stream_t st, const uint64_t* pos_off, const uint64_t* boff, uint32_t nb,
                                   uint32_t lo, uint64_t budget, uint64_t item_budget, uint32_t* out) {
  SMX_LAUNCH(k_rec_cut, 1, 1, st, (const ull*)pos_off, (const ull*)boff, nb, lo, (ull)budget, (ull)item_budget, out);
}
extern "C" void smx_launch_rec_check(smx_stream_t st, const uint64_t* boff, uint32_t nb, uint32_t* out) {
  SMX_LAUNCH(k_rec_check, grid_for(nb), SMX_BLOCK, st, (const ull*)boff, nb, out);
}
extern "C" void smx_launch_sum_values(smx_stream_t st, smx_view_t v, uint32_t* big_list, uint32_t* big_counter) {
  SMX_LAUNCH(k_sum_values, grid_for(v.dir_cap * SMX_WARP), SMX_BLOCK, st, v, big_list, big_counter);
}
extern "C" void smx_launch_sum_values_big(smx_stream_t st, smx_view_t v, const uint32_t* big_list, uint32_t n_big) {
  for (uint32_t first = 0; first < n_big; first += 32768u) {
    const uint32_t cnt = (n_big - first < 32768u) ? n_big - first : 32768u;
    dim3 grid(SMX_WARP > 1 ? 32u : 2u, cnt, 1u);
    SMX_LAUNCH(k_sum_values_big, grid, SMX_BLOCK, st, v, big_list, first);
  }
}
extern "C" void smx_launch_count_nnz(smx_stream_t st, smx_view_t v) {
  SMX_LAUNCH(k_count_nnz, grid_for(v.dir_cap), SMX_BLOCK, st, v);
}

extern "C" void smx_launch_gen_c2_ops(smx_stream_t st, uint64_t seed, uint64_t first, uint64_t count,
                                      uint32_t rows, uint32_t ycols, uint32_t* xs, uint32_t* ys) {
  if (!count) return;
  SMX_LAUNCH(k_gen_c2_ops, grid_for(count), SMX_BLOCK, st, (ull)seed, (ull)first, (ull)count, rows,
             ycols, xs, ys);
}
extern "C" void smx_launch_gen_c2_queries(smx_stream_t st, uint64_t seed_get, uint64_t seed_build,
                                          uint64_t first, uint64_t count, uint64_t n_build,
                                          uint32_t rows, uint32_t ycols, uint32_t* xs, uint32_t* ys) {
  if (!count) return;
  SMX_LAUNCH(k_gen_c2_queries, grid_for(count), SMX_BLOCK, st, (ull)seed_get, (ull)seed_build,
             (ull)first, (ull)count, (ull)n_build, rows, ycols, xs, ys);
}

extern "C" void smx_launch_gen_c3_ops(smx_stream_t st, uint64_t seed, uint64_t first, uint64_t count,
                                      const uint64_t* thr, uint32_t items, uint32_t* xs, uint32_t* ys) {
  if (!count) return;
  SMX_LAUNCH(k_gen_c3_ops, grid_for(count), SMX_BLOCK, st, (ull)seed, (ull)first, (ull)count,
             (const ull*)thr, items, xs, ys);
}
extern "C" void smx_launch_gen_c3_queries(smx_stream_t st, uint64_t seed_get, uint64_t seed_build,
                                          uint64_t first, uint64_t count, uint64_t n_build,
                                          const uint64_t* thr, uint32_t items, uint32_t* xs, uint32_t* ys) {
  if (!count) return;
  SMX_LAUNCH(k_gen_c3_queries, grid_for(count), SMX_BLOCK, st, (ull)seed_get, (ull)seed_build, (ull)first,
             (ull)count, (ull)n_build, (const ull*)thr, items, xs, ys);
}
extern "C" void smx_launch_gen_c4_lens(smx_stream_t st, uint64_t seed, uint64_t first, uint64_t count,
                                       const uint64_t* thr, uint32_t kmax, uint32_t* lens) {
  if (!count) return;
  SMX_LAUNCH(k_gen_c4_lens, grid_for(count), SMX_BLOCK, st, (ull)seed, (ull)first, (ull)count,
             (const ull*)thr, kmax, lens);
}
extern "C" void smx_launch_gen_c4_ops(smx_stream_t st, uint64_t seed, uint64_t first, uint64_t count,
                                      const uint64_t* offs, uint32_t rows, uint32_t* xs, uint32_t* ys,
                                      uint32_t* vs) {
  if (!count) return;
  SMX_LAUNCH(k_gen_c4_ops, grid_for(count), SMX_BLOCK, st, (ull)seed, (ull)first, (ull)count,
             (const ull*)offs, rows, xs, ys, vs);
}

extern "C" void smx_launch_probe_read(smx_stream_t st, const void* buf, uint64_t n_units,
                                      uint64_t accesses, int width, smx_ctl_t* ctl) {
  SMX_LAUNCH(k_probe_read, grid_for(accesses), SMX_BLOCK, st, (const char*)buf, (ull)n_units,
             (ull)accesses, width, ctl);
}
extern "C" void smx_launch_probe_atomic(smx_stream_t st, uint32_t* buf, uint64_t n_words,
                                        uint64_t accesses) {
  SMX_LAUNCH(k_probe_atomic, grid_for(accesses), SMX_BLOCK, st, buf, (ull)n_words, (ull)accesses);
}

extern "C" void smx_launch_partition_count(smx_stream_t st, const uint32_t* xs, const uint32_t* ys,
                                           uint32_t n, uint32_t world, uint32_t dir_mask,
                                           uint32_t shift, uint32_t split0, unsigned long long* counts) {
  if (!n) return;
  SMX_LAUNCH(k_partition_count, grid_for(n), SMX_BLOCK, st, xs, ys, n, world, dir_mask, shift, split0, counts);
}
extern "C" void smx_launch_partition_scatter(smx_stream_t st, const uint32_t* xs, const uint32_t* ys,
                                             const uint32_t* vs, uint32_t n, uint32_t world,
                                             uint32_t dir_mask, uint32_t shift, uint32_t split0,
                                             unsigned long long* cursors, uint32_t* oxs,
                                             uint32_t* oys, uint32_t* ovs, uint32_t* osrc,
                                             const uint32_t* src_in, uint32_t* opos,
                                             const unsigned long long* dst_tab, uint32_t src_bias) {
  if (!n) return;
  const uint32_t grid = grid_for((ull)(n + PART_ITEMS - 1) / PART_ITEMS);
  const bool pos = opos && !src_in;
#define SMX_SCATTER(V, P)                                                                            \
  {                                                                                                  \
    auto k = k_partition_scatter<V, P>;                                                              \
    SMX_LAUNCH(k, grid, SMX_BLOCK, st, xs, ys, vs, n, world, dir_mask, shift, split0, cursors, oxs, oys, ovs, \
               osrc, src_in, opos, (const ull*)dst_tab, src_bias);                                   \
  }
  if (vs) SMX_SCATTER(true, false)
  else if (pos) SMX_SCATTER(false, true)
  else SMX_SCATTER(false, false)
#undef SMX_SCATTER
}
extern "C" void smx_launch_parts_prefix(smx_stream_t st, const unsigned long long* counts, uint32_t parts,
                                        unsigned long long* cursors) {
  SMX_LAUNCH(k_parts_prefix, 1, 32, st, (const ull*)counts, parts, (ull*)cursors);
}
extern "C" void smx_launch_gather(smx_stream_t st, uint32_t* out, const uint32_t* vals,
                                  const uint32_t* pos, uint32_t n) {
  if (!n) return;
  SMX_LAUNCH(k_gather, (uint32_t)(((ull)n + PART_TILE - 1) / PART_TILE), SMX_BLOCK, st, out, vals, pos, n);
}
extern "C" void smx_launch_gather_stride(smx_stream_t st, uint32_t* out, const uint32_t* vals,
                                         const uint32_t* pos, uint32_t n) {
  if (!n) return;
  SMX_LAUNCH(k_gather_stride, grid_for(n), SMX_BLOCK, st, out, vals, pos, n);
}

extern "C" void smx_launch_route_offsets(smx_stream_t st, const uint64_t* offs, const uint32_t* pos,
                                         uint32_t n, uint32_t world, const unsigned long long* tab) {
  if (!n) return;
  SMX_LAUNCH(k_route_offsets, grid_for(n), SMX_BLOCK, st, (const ull*)offs, pos, n, world, (const ull*)tab);
}

extern "C" uint32_t smx_owner_hash(uint32_t x) { return smx_mix_owner(x); }
