/*
 * oracle/smatrix_oracle.h — CPU restatement of libsmatrix's in-memory hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under libsmatrix_b200/ may include, link or call this.
 * It is imported only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference leg, and there only as the checker.
 *
 * Parity status: PINNED.  tests/test_oracle.py checks this restatement (a) against the
 * reference's own known-answer cases (src/java/test/TestSparseMatrix.java:22-166,
 * examples/smatrix_example.c:17-48) and (b) op-for-op against the unmodified reference compiled
 * into oracle/_ref/libsmatrix_ref.so, including getrow table order and truncation.
 */
#ifndef SMATRIX_ORACLE_H
#define SMATRIX_ORACLE_H

#include <stddef.h>
#include <stdint.h>

typedef struct smx_oracle_s smx_oracle_t;

/* fname == NULL: memory mode.  Otherwise the file (if it exists and is not empty) is loaded the
 * reference's way, and the matrix is written back to it at close; NULL for a corrupt file. */
smx_oracle_t* smx_oracle_open(const char* fname);
void     smx_oracle_close(smx_oracle_t* m);
uint32_t smx_oracle_get(smx_oracle_t* m, uint32_t x, uint32_t y);
uint32_t smx_oracle_set(smx_oracle_t* m, uint32_t x, uint32_t y, uint32_t v);
uint32_t smx_oracle_incr(smx_oracle_t* m, uint32_t x, uint32_t y, uint32_t v);
uint32_t smx_oracle_decr(smx_oracle_t* m, uint32_t x, uint32_t y, uint32_t v);
uint32_t smx_oracle_rowlen(smx_oracle_t* m, uint32_t x);
uint32_t smx_oracle_getrow(smx_oracle_t* m, uint32_t x, uint32_t* ret, size_t ret_len);

/* introspection used by the tests (not part of the reference API) */
uint64_t smx_oracle_nrows(smx_oracle_t* m);       /* directory entries in use               */
uint64_t smx_oracle_dirsize(smx_oracle_t* m);     /* directory capacity                     */
uint32_t smx_oracle_rowsize(smx_oracle_t* m, uint32_t x); /* slot capacity of row x, 0 if absent */

/* Write the matrix as a .smx file now; 0 or -1.  With flags 0 the file is laid out like a fresh
 * snapshot (rows in directory order, one directory block).  The flags make it look like a file the
 * reference's append-only writer leaves behind, with the same rows and cells: */
#define SMX_ORACLE_SAVE_SHUFFLED  1 /* row blocks in reverse directory order                        */
#define SMX_ORACLE_SAVE_DEAD      2 /* an unreferenced stale block before every other row block      */
#define SMX_ORACLE_SAVE_UNALIGNED 4 /* the middle row block at 4 mod 8, the one after it at 1 mod 8  */
#define SMX_ORACLE_SAVE_SMALL_DIR 8 /* directory blocks of 5 entries, chained, the last partly used  */
int smx_oracle_save(smx_oracle_t* m, const char* fname, int flags);

#endif
