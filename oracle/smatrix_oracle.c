/*
 * oracle/smatrix_oracle.c — single-threaded CPU restatement of the reference's nested
 * open-addressing hash maps (row directory "cmap" -> per-row column map "rmap").
 *
 * TEST INFRASTRUCTURE ONLY (see smatrix_oracle.h).  Written from the reference's behaviour,
 * not from its text: no locks, no IO thread (the file is read at open and written whole at
 * save / close), index-based instead of pointer-based.  Every function names the reference
 * lines whose behaviour it restates (paths relative to the reference checkout).
 *
 * What has to be reproduced for bit-exact results (SURVEY.md 8a):
 *   - column map: identity hash `y % size`, linear probing, EMPTY <=> key==0 && value==0
 *     (src/smatrix.c:363-380); grow x2 when used > size/2 BEFORE placing (:343-360); growth
 *     re-places every non-empty cell in table order, recounting `used` (:383-416)
 *   - a write to column 0 never goes through the placing path, because the probe for key 0
 *     stops on any key==0 cell and the caller treats `cell.key == y` as a hit (:297-300)
 *   - rowlen returns the running `used` counter (:212-223), getrow walks the table in order
 *     and stops once `++num * 8 >= ret_len` (:189-210)
 *   - directory: `x % size`, linear probing over {used flag, key}, grow x2 when
 *     used*4 >= size*3 (:673-741), initial 65536 entries (src/smatrix.h:24), rows start with
 *     16 cells (src/smatrix.h:21)
 *   - file mode (.smx, :30-72): a row block is the row's own cell array (:454-482); loading is
 *     positional — a row keeps its file size and its cells' slots, slots with value == 0 are
 *     cleared in place and `used` is the count of the non-empty slots left (:499-545)
 */
#include "smatrix_oracle.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define ROW_CELLS0 16u    /* src/smatrix.h:21 SMATRIX_RMAP_INITIAL_SIZE */
#define DIR_ENTRIES0 65536u /* src/smatrix.h:24 SMATRIX_CMAP_INITIAL_SIZE */

typedef struct {
  uint32_t key;
  uint32_t val;
} cell_t;

typedef struct {
  uint32_t size; /* capacity in cells, power of two */
  uint32_t used; /* the reference's running counter, NOT a live count */
  cell_t* cell;
} row_t;

typedef struct {
  uint32_t taken;
  uint32_t x;
  row_t* row;
} dirent_t;

struct smx_oracle_s {
  uint64_t dsize;
  uint64_t dused;
  dirent_t* dir;
  char* fname; /* file mode: written back at close */
};

static void* zalloc(size_t bytes) {
  void* p = calloc(1, bytes);
  if (!p) {
    fprintf(stderr, "smx_oracle: out of memory\n");
    abort();
  }
  return p;
}

static inline int cell_is_empty(const cell_t* c) { return c->key == 0 && c->val == 0; }

/* src/smatrix.c:363-380 — index of the cell where the probe for `y` stops. */
static uint32_t row_probe(const row_t* r, uint32_t y) {
  uint64_t at = y % r->size;
  for (uint64_t step = 0; step < r->size; step++) {
    const cell_t* c = &r->cell[at];
    if (c->key == y || cell_is_empty(c)) break;
    at = (at + 1) % r->size;
  }
  return (uint32_t)at;
}

static uint32_t row_place(row_t* r, uint32_t y);

/* src/smatrix.c:383-416 — double the row and re-place every non-empty cell in table order. */
static void row_double(row_t* r) {
  row_t bigger;
  bigger.size = r->size * 2;
  bigger.used = 0;
  bigger.cell = zalloc(sizeof(cell_t) * bigger.size);
  for (uint32_t i = 0; i < r->size; i++) {
    if (cell_is_empty(&r->cell[i])) continue;
    uint32_t at = row_place(&bigger, r->cell[i].key);
    bigger.cell[at].val = r->cell[i].val;
  }
  free(r->cell);
  *r = bigger;
}

/* src/smatrix.c:343-360 — make sure `y` owns a cell; counts it in `used` when newly claimed. */
static uint32_t row_place(row_t* r, uint32_t y) {
  if (r->used > r->size / 2) row_double(r);
  uint32_t at = row_probe(r, y);
  cell_t* c = &r->cell[at];
  if (c->key == 0 || c->key != y) {
    r->used++;
    c->key = y;
    c->val = 0;
  }
  return at;
}

/* src/smatrix.c:673-693 — directory probe: stops on a free entry or on the key. */
static uint64_t dir_probe(const smx_oracle_t* m, uint32_t x) {
  uint32_t walk = x; /* the reference walks an `unsigned` that wraps at 2^32 */
  for (;;) {
    uint64_t at = walk % m->dsize;
    if (!m->dir[at].taken || m->dir[at].x == x) return at;
    walk++;
  }
}

static uint64_t dir_place(smx_oracle_t* m, uint32_t x);

/* src/smatrix.c:715-741 */
static void dir_double(smx_oracle_t* m) {
  smx_oracle_t bigger;
  bigger.dsize = m->dsize * 2;
  bigger.dused = 0;
  bigger.dir = zalloc(sizeof(dirent_t) * bigger.dsize);
  bigger.fname = m->fname;
  for (uint64_t i = 0; i < m->dsize; i++) {
    if (!m->dir[i].taken) continue;
    uint64_t at = dir_place(&bigger, m->dir[i].x);
    bigger.dir[at].row = m->dir[i].row;
  }
  free(m->dir);
  *m = bigger;
}

/* src/smatrix.c:695-713 */
static uint64_t dir_place(smx_oracle_t* m, uint32_t x) {
  if (m->dused * 4 >= m->dsize * 3) dir_double(m);
  uint64_t at = dir_probe(m, x);
  dirent_t* e = &m->dir[at];
  if (!e->taken || e->x != x) {
    m->dused++;
    e->taken = 1;
    e->x = x;
    e->row = NULL;
  }
  return at;
}

/* src/smatrix.c:621-670 without the locking: find the row, optionally creating it. */
static row_t* find_row(smx_oracle_t* m, uint32_t x, int create) {
  uint64_t at = dir_probe(m, x);
  if (m->dir[at].taken && m->dir[at].x == x) return m->dir[at].row;
  if (!create) return NULL;
  row_t* r = zalloc(sizeof(row_t));
  r->size = ROW_CELLS0;
  r->used = 0;
  r->cell = zalloc(sizeof(cell_t) * ROW_CELLS0);
  at = dir_place(m, x);
  m->dir[at].row = r;
  return r;
}

/* src/smatrix.c:258-304 — resolve (x,y) to a cell; writers create row and cell. */
static cell_t* resolve(smx_oracle_t* m, uint32_t x, uint32_t y, int write, row_t** row_out) {
  row_t* r = find_row(m, x, write);
  if (row_out) *row_out = r;
  if (!r) return NULL;
  uint32_t at = row_probe(r, y);
  if (r->cell[at].key == y) return &r->cell[at];
  if (!write) return NULL;
  at = row_place(r, y);
  return &r->cell[at];
}

/* ---- file mode (.smx, src/smatrix.c:30-72) -------------------------------------------------
 *   header     512 bytes: 8 x 0x17, u64 offset of the first directory block (:564-596)
 *   directory  blocks of {u64 entries, u64 next} + entries x {u32 row, u64 row offset}, chained;
 *              an entry with offset 0 ends its block (:744-830)
 *   row block  8 x 0x23, u64 size, then the row's cell array as it is in memory (:454-482) */
#define F_HEAD 512ull
#define F_DIR_ENTRIES 4194304ull
#define F_DIR_HEAD 16ull
#define F_DIR_SLOT 12ull
#define F_ROW_HEAD 16ull
#define F_SMALL_DIR_ENTRIES 5ull /* SMX_ORACLE_SAVE_SMALL_DIR */
#define F_DEAD_CELLS 16ull       /* SMX_ORACLE_SAVE_DEAD: a row's stale first block */

static void put64(unsigned char* p, uint64_t v) { memcpy(p, &v, 8); }
static uint64_t get64(const unsigned char* p) { uint64_t v; memcpy(&v, p, 8); return v; }

/* src/smatrix.c:499-545 — one row block, positionally: the row keeps the file's size and every
 * cell's slot; a slot whose value is 0 is cleared, and `used` is the count of what is left
 * (column-0 slot included).  Returns 0, or -1 when the block does not fit the file. */
static int load_row(smx_oracle_t* m, uint32_t x, const unsigned char* d, uint64_t n, uint64_t rpos) {
  if (rpos > n || n - rpos < F_ROW_HEAD) return -1;
  for (int k = 0; k < 8; k++)
    if (d[rpos + k] != 0x23) return -1;
  const uint64_t size = get64(d + rpos + 8);
  if (size == 0 || (size & (size - 1)) || size > (1ull << 32) || (n - rpos - F_ROW_HEAD) / 8 < size) return -1;
  uint64_t at = dir_probe(m, x);
  if (m->dir[at].taken && m->dir[at].x == x) return -1; /* a row listed twice */
  row_t* r = zalloc(sizeof(row_t));
  r->size = (uint32_t)size;
  r->cell = zalloc(sizeof(cell_t) * size);
  memcpy(r->cell, d + rpos + F_ROW_HEAD, sizeof(cell_t) * size);
  r->used = 0;
  for (uint64_t i = 0; i < size; i++) {
    if (r->cell[i].val == 0) r->cell[i].key = 0;
    if (!cell_is_empty(&r->cell[i])) r->used++;
  }
  at = dir_place(m, x);
  m->dir[at].row = r;
  return 0;
}

/* src/smatrix.c:744-830 — the header, then the chain of directory blocks, every entry's row */
static int load_file(smx_oracle_t* m, const unsigned char* d, uint64_t n) {
  if (n < F_HEAD) return -1;
  for (int k = 0; k < 8; k++)
    if (d[k] != 0x17) return -1;
  uint64_t bpos = get64(d + 8), blocks = 0;
  while (bpos) {
    if (++blocks > n / F_DIR_HEAD || bpos > n || n - bpos < F_DIR_HEAD) return -1; /* a loop, or past the end */
    const uint64_t entries = get64(d + bpos), next = get64(d + bpos + 8);
    if (entries > F_DIR_ENTRIES || (n - bpos - F_DIR_HEAD) / F_DIR_SLOT < entries) return -1;
    for (uint64_t e = 0; e < entries; e++) {
      const unsigned char* ent = d + bpos + F_DIR_HEAD + e * F_DIR_SLOT;
      uint32_t x;
      memcpy(&x, ent, 4);
      const uint64_t rpos = get64(ent + 4);
      if (!rpos) break;
      if (load_row(m, x, d, n, rpos)) return -1;
    }
    bpos = next;
  }
  return 0;
}

int smx_oracle_save(smx_oracle_t* m, const char* fname, int flags) {
  uint64_t n = 0;
  for (uint64_t i = 0; i < m->dsize; i++) n += m->dir[i].taken;
  row_t** rows = malloc(sizeof(row_t*) * (n ? n : 1));
  uint32_t* keys = malloc(sizeof(uint32_t) * (n ? n : 1));
  uint64_t* rpos = malloc(sizeof(uint64_t) * (n ? n : 1));
  uint64_t* dead = malloc(sizeof(uint64_t) * (n ? n : 1));
  if (!rows || !keys || !rpos || !dead) abort();
  for (uint64_t i = 0, k = 0; i < m->dsize; i++) /* directory order = table order */
    if (m->dir[i].taken) { rows[k] = m->dir[i].row; keys[k] = m->dir[i].x; k++; }
  const uint64_t per = (flags & SMX_ORACLE_SAVE_SMALL_DIR) ? F_SMALL_DIR_ENTRIES : F_DIR_ENTRIES;
  const uint64_t nblk = n ? (n + per - 1) / per : 1, blk_bytes = F_DIR_HEAD + per * F_DIR_SLOT;
  /* layout: header, first directory block, row blocks, then the later directory blocks at the end
   * of the file, where an append-only writer puts the next block once the previous one is full */
  uint64_t pos = F_HEAD + blk_bytes;
  for (uint64_t k = 0; k < n; k++) {
    const uint64_t i = (flags & SMX_ORACLE_SAVE_SHUFFLED) ? n - 1 - k : k;
    /* two row blocks off alignment: one at 4 mod 8, one at 1 mod 8, the blocks behind them aligned */
    const uint64_t odd = !(flags & SMX_ORACLE_SAVE_UNALIGNED) ? 0 : k == n / 2 ? 4 : k == n / 2 + 1 ? 1 : 0;
    dead[i] = 0;
    if ((flags & SMX_ORACLE_SAVE_DEAD) && k % 2 == 0) { /* a row's earlier, smaller block */
      dead[i] = pos;
      pos += F_ROW_HEAD + 8 * F_DEAD_CELLS;
    }
    pos += odd;
    rpos[i] = pos;
    pos += F_ROW_HEAD + 8ull * rows[i]->size + (odd ? 8 - odd : 0);
  }
  const uint64_t later_dirs = pos;
  pos += (nblk - 1) * blk_bytes;
  unsigned char* d = calloc(1, pos);
  if (!d) abort();
  memset(d, 0x17, 8);
  put64(d + 8, F_HEAD);
  for (uint64_t b = 0; b < nblk; b++) {
    const uint64_t at = b ? later_dirs + (b - 1) * blk_bytes : F_HEAD;
    put64(d + at, per);
    put64(d + at + 8, b + 1 < nblk ? later_dirs + b * blk_bytes : 0);
    for (uint64_t e = 0; e < per && b * per + e < n; e++) {
      unsigned char* ent = d + at + F_DIR_HEAD + e * F_DIR_SLOT;
      memcpy(ent, &keys[b * per + e], 4);
      put64(ent + 4, rpos[b * per + e]);
    }
  }
  for (uint64_t i = 0; i < n; i++) {
    memset(d + rpos[i], 0x23, 8);
    put64(d + rpos[i] + 8, rows[i]->size);
    memcpy(d + rpos[i] + F_ROW_HEAD, rows[i]->cell, 8ull * rows[i]->size);
    if (dead[i]) { /* stale: every value off by one, unreferenced */
      memset(d + dead[i], 0x23, 8);
      put64(d + dead[i] + 8, F_DEAD_CELLS);
      for (uint64_t c = 0; c < F_DEAD_CELLS && c < rows[i]->size; c++) {
        cell_t stale = rows[i]->cell[c];
        stale.val += 1;
        memcpy(d + dead[i] + F_ROW_HEAD + 8 * c, &stale, 8);
      }
    }
  }
  FILE* f = fopen(fname, "wb");
  int rc = f && fwrite(d, 1, pos, f) == pos ? 0 : -1;
  if (f && fclose(f) != 0) rc = -1;
  free(d); free(rows); free(keys); free(rpos); free(dead);
  return rc;
}

smx_oracle_t* smx_oracle_open(const char* fname) {
  smx_oracle_t* m = zalloc(sizeof(*m));
  m->dsize = DIR_ENTRIES0; /* src/smatrix.c:598-612 */
  m->dused = 0;
  m->dir = zalloc(sizeof(dirent_t) * m->dsize);
  if (!fname) return m;
  m->fname = strdup(fname);
  FILE* f = fopen(fname, "rb"); /* a missing or empty file is a new matrix (:90-111) */
  if (!f) return m;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  unsigned char* d = n > 0 ? malloc((size_t)n) : NULL;
  int rc = 0;
  if (n > 0) rc = (!d || fread(d, 1, (size_t)n, f) != (size_t)n) ? -1 : load_file(m, d, (uint64_t)n);
  fclose(f);
  free(d);
  if (rc) {
    fprintf(stderr, "smx_oracle: %s is not a valid .smx file\n", fname);
    free(m->fname);
    m->fname = NULL; /* never overwrite it */
    smx_oracle_close(m);
    return NULL;
  }
  return m;
}

void smx_oracle_close(smx_oracle_t* m) { /* src/smatrix.c:113-133 */
  if (!m) return;
  if (m->fname && smx_oracle_save(m, m->fname, 0)) fprintf(stderr, "smx_oracle: cannot write %s\n", m->fname);
  for (uint64_t i = 0; i < m->dsize; i++) {
    if (m->dir[i].taken && m->dir[i].row) {
      free(m->dir[i].row->cell);
      free(m->dir[i].row);
    }
  }
  free(m->fname);
  free(m->dir);
  free(m);
}

uint32_t smx_oracle_get(smx_oracle_t* m, uint32_t x, uint32_t y) { /* src/smatrix.c:174-185 */
  cell_t* c = resolve(m, x, y, 0, NULL);
  return c ? c->val : 0;
}

uint32_t smx_oracle_set(smx_oracle_t* m, uint32_t x, uint32_t y, uint32_t v) { /* :225-234 */
  cell_t* c = resolve(m, x, y, 1, NULL);
  c->val = v;
  return c->val;
}

uint32_t smx_oracle_incr(smx_oracle_t* m, uint32_t x, uint32_t y, uint32_t v) { /* :236-245 */
  cell_t* c = resolve(m, x, y, 1, NULL);
  c->val += v;
  return c->val;
}

uint32_t smx_oracle_decr(smx_oracle_t* m, uint32_t x, uint32_t y, uint32_t v) { /* :247-256 */
  cell_t* c = resolve(m, x, y, 1, NULL);
  c->val -= v;
  return c->val;
}

uint32_t smx_oracle_rowlen(smx_oracle_t* m, uint32_t x) { /* src/smatrix.c:212-223 */
  row_t* r = find_row(m, x, 0);
  return r ? r->used : 0;
}

uint32_t smx_oracle_getrow(smx_oracle_t* m, uint32_t x, uint32_t* ret, size_t ret_len) { /* :189-210 */
  row_t* r = find_row(m, x, 0);
  uint32_t n = 0;
  if (!r) return 0;
  for (uint32_t i = 0; i < r->size; i++) {
    if (cell_is_empty(&r->cell[i])) continue;
    ret[2 * n] = r->cell[i].key;
    ret[2 * n + 1] = r->cell[i].val;
    n++;
    if ((size_t)n * 8 >= ret_len) break;
  }
  return n;
}

uint64_t smx_oracle_nrows(smx_oracle_t* m) { return m->dused; }
uint64_t smx_oracle_dirsize(smx_oracle_t* m) { return m->dsize; }
uint32_t smx_oracle_rowsize(smx_oracle_t* m, uint32_t x) {
  row_t* r = find_row(m, x, 0);
  return r ? r->size : 0;
}
