/*
 * include/smatrix.h — the libsmatrix C API, served by the B200 (sm_100a) device table.
 *
 * Drop-in for the reference's public header: the same eight entry points with the same
 * argument meaning, return values and error behaviour (reference src/smatrix.h:87-94; bodies
 * src/smatrix.c:74-133 and :174-256).  The handle is opaque here — the reference's bindings
 * only store and pass the pointer (src/smatrix_jni.c:21-49, src/smatrix_ruby.c:47), so
 * src/smatrix_jni.c and src/smatrix_ruby.c compile and link against this header unchanged.
 *
 * Differences a caller can observe (all documented in DESIGN.md):
 *   - the matrix lives in GPU memory; every call is a kernel launch plus a synchronous
 *     read-back, so single-op latency is tens of microseconds — use smatrix_batch.h for
 *     throughput;
 *   - getrow returns pairs in the device table's order, not the reference's; the contract
 *     compares rows sorted by column (the Java wrapper sorts anyway, SparseMatrix.java:102-112);
 *   - results are bit-exact on the reference's safe domain: once non-zero, column 0 of a row
 *     must not return to 0 (the reference corrupts its own probe chains there, SURVEY.md Q3).
 *
 * Error convention (reference src/smatrix.c:891-894): smatrix_open returns NULL on failure;
 * everything else prints "libsmatrix error: ..." to stdout and abort()s.  There is no CPU
 * fallback: without a usable CUDA device smatrix_open fails.
 *
 * Thread safety (reference README.md:113,120): every function may be called concurrently from
 * any number of host threads on one handle; calls are serialised by a per-handle host mutex.
 */
#ifndef SMATRIX_H
#define SMATRIX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct smatrix_s smatrix_t;

/* replaces src/smatrix.c:74-111.  fname == NULL: memory-only matrix on the device chosen by
 * $SMATRIX_DEVICE (default 0).  fname != NULL: the table is loaded from that .smx file if it
 * exists and written back to it by smatrix_close (snapshot persistence).
 * DURABILITY differs from the reference: the reference's IO thread streams dirty rows to the
 * file all the time (src/smatrix.c:418-596); here the file changes only in smatrix_close and in
 * smatrix_b200_snapshot (smatrix_b200.h) — written to a temporary file, fsync'ed, then renamed
 * over the old one — and in smatrix_b200_checkpoint, which appends the rows written since the
 * last save and then switches the header's directory pointer, so the file on disk always loads
 * to a complete persisted state.  Updates made after the last snapshot or checkpoint are lost if
 * the process dies (every "libsmatrix error" path abort()s). */
smatrix_t* smatrix_open(const char* fname);

/* replaces src/smatrix.c:113-133.  Writes the snapshot (file mode) and frees all device memory. */
void smatrix_close(smatrix_t* self);

/* replaces src/smatrix.c:174-185: value at (x,y) or 0; never creates anything. */
uint32_t smatrix_get(smatrix_t* self, uint32_t x, uint32_t y);

/* replace src/smatrix.c:225-256: create row and cell as needed, then value = v / += v / -= v
 * (mod 2^32).  Return the cell's new value. */
uint32_t smatrix_set(smatrix_t* self, uint32_t x, uint32_t y, uint32_t value);
uint32_t smatrix_incr(smatrix_t* self, uint32_t x, uint32_t y, uint32_t value);
uint32_t smatrix_decr(smatrix_t* self, uint32_t x, uint32_t y, uint32_t value);

/* replaces src/smatrix.c:212-223: the reference's running `used` counter for row x (history
 * dependent, SURVEY.md Q1), 0 if the row does not exist. */
uint32_t smatrix_rowlen(smatrix_t* self, uint32_t x);

/* replaces src/smatrix.c:189-210: writes [col, value, col, value, ...] into ret and returns the
 * number of pairs; ret_len is the buffer size in BYTES; stops once pairs*8 >= ret_len (so at
 * least one pair is written for a non-empty row, exactly like the reference). */
uint32_t smatrix_getrow(smatrix_t* self, uint32_t x, uint32_t* ret, size_t ret_len);

#ifdef __cplusplus
}
#endif
#endif
