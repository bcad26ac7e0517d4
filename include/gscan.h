/*
 * gscan.h -- C ABI of the B200-native scan engine that replaces grab's per-chunk match loop.
 *
 * The reference (stealth/grab, master) has no plugin API; its seam is the five PCRE1 calls made
 * by class FileGrep.  A per-match pcre_exec()-shaped call is the wrong granularity for a GPU, so
 * the boundary sits one level up: one call scans a BATCH of chunks ("units": the mmap windows of
 * /root/reference/src/grab.cc:154-169) and returns exactly the sequence of matches the loop at
 * grab.cc:175-213 would have produced for each of them.
 *
 * Every entry point cites the reference interface it replaces.  No torch / C++ types cross this
 * boundary: plain pointers, sizes and PODs; int 0 / -1 + message like FileGrep (grab.h:61-64).
 *
 * Threading (mirrors "each thread owns its FileGrep", main.cc:195-199): a gscan_pattern is
 * immutable and may be shared; a gscan_ctx belongs to one host thread and one GPU, shares nothing
 * with other contexts and is not re-entrant.
 */
#ifndef GSCAN_H
#define GSCAN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSCAN_ABI_VERSION 2

typedef struct gscan_ctx gscan_ctx;
typedef struct gscan_pattern gscan_pattern;
typedef struct gscan_batch gscan_batch;

/* ---- pattern compile flags ------------------------------------------------------------- */
#define GSCAN_LITERAL 1u    /* pattern bytes are a literal string (grab -S, README.md:26) */
#define GSCAN_STRICT_REF 2u /* reproduce quirk Q2: a capturing group makes pcre_exec return 0 with
                               ovecsize 3 (grab.cc:171,178-180) => the loop prints nothing */

/* ---- scan modes: which branch of grab.cc:185-212 advances `start` ---------------------- */
#define GSCAN_MODE_ALL 0u   /* -O -l            : every non-overlapping match   (grab.cc:185,209) */
#define GSCAN_MODE_FIRST 1u /* -s / -l w/o -O   : first match of the unit only  (grab.cc:204-212) */
#define GSCAN_MODE_LINE 2u  /* line output on   : resume after the line remainder, <=511 B (grab.cc:188-209) */

/* ---- unit flags ------------------------------------------------------------------------ */
#define GSCAN_UNIT_DEVICE 1u /* ptr is a device pointer on the context's GPU (16-byte aligned,
                                readable up to the next 16-byte boundary past ptr+len) */
#define GSCAN_UNIT_FD 2u     /* ptr carries an open file descriptor ((intptr_t)ptr); the window is the `len` bytes at file
                                offset `base_off` of it.  Replaces the mmap of grab.cc:126-128,161 for callers that do not
                                need the bytes themselves (no line output): the engine's staging threads pread() straight
                                into their pinned bounce buffers -- no mapping, no page faults, no munmap (grab.cc:215)
                                under mmap_lock.  The descriptor stays the caller's (not closed); a read error or a file
                                shorter than base_off + len fails the call (the reference would take a SIGBUS) */

/* One scan unit == one mmap window of grab.cc:154-169: `content`, `clen`, `off`. */
typedef struct gscan_unit {
	const uint8_t *ptr; /* window bytes (host, or device with GSCAN_UNIT_DEVICE; a descriptor with GSCAN_UNIT_FD)  grab.cc:161 */
	uint64_t len;       /* clen                                                  grab.cc:156-159 */
	uint64_t base_off;  /* off: file offset of the window                        grab.cc:154 */
	uint32_t file_id;   /* caller's id of the file the window belongs to */
	uint32_t flags;
} gscan_unit;

/* One match: what grab.cc:186 prints (start) and ovector[1]-ovector[0] (match_len). */
typedef struct gscan_match {
	uint64_t start;     /* base_off + (start - content) + ovector[0]             grab.cc:186 */
	uint32_t file_id;
	uint32_t match_len; /* ovector[1] - ovector[0]                               grab.cc:199 */
} gscan_match;

typedef struct gscan_pattern_info {
	int32_t minlen;       /* PCRE_INFO_MINLENGTH                                  grab.cc:120 */
	int32_t maxlen;       /* longest possible match, -1 if unbounded */
	int32_t captures;     /* capturing groups in the pattern (Q2) */
	int32_t engine;       /* GSCAN_ENGINE_* below */
	int32_t n_sequences;  /* alternatives after expansion (fixed engine) */
	int32_t n_filter_tests; /* byte-pair tests of the SWAR filter; negative: hashed engine, -(table slots) */
	int32_t filter_anchor; /* byte of the pattern the SWAR filter is anchored on */
	int32_t filter_delta;  /* distance to the second filter byte (0: single-byte filter) */
	int32_t scan_kernel;   /* GSCAN_KERNEL_* below: which scan-kernel family serves the pattern */
	int32_t scan_variant;  /* the values the scan-kernel launch dispatches on (bit layout below), 0 for GSCAN_KERNEL_NONE */
} gscan_pattern_info;

/* scan_variant: raw values, not template arguments (the launcher maps e.g. 5 tests to the 6-test instantiation).
 *   PAIR / TRIPLE / BALANCED  bits 0-3  n_filter_tests (0..8)      bits 4-6  filter_delta (0..4)
 *                             bit  7    every pair test exact      bit  8    balanced pair filter
 *                             bit  9    balanced: one third-byte test per pair test (aligned stage 2)
 *                             bit 10    byte-triple stage-1 filter bits 11-15 third-byte tests (0..16)
 *                             bit 16    every triple test exact
 *   RUN                       bits 0-3  byte ranges below 0x80     bits 4-5  ranges in 0x80-0xff (0..2)
 *                             bit  6    one [A-Z]/[a-z]-style range pair folded into one test
 *                             bit  7    run minimum above 17 (bytes 17.. confirmed from global memory)
 *   HASH                      bits 0-1  key bytes (2 or 3)         bit  2    sparse path possible (class prefilter)
 *                             bits 3-8  table copies in shared memory (32, 16 or 1) */
#define GSCAN_SV_TESTS(v) ((v) & 15)
#define GSCAN_SV_DELTA(v) (((v) >> 4) & 7)
#define GSCAN_SV_EXACT 0x80
#define GSCAN_SV_BALANCED 0x100
#define GSCAN_SV_ALIGNED 0x200
#define GSCAN_SV_STAGE1_TRIPLES 0x400
#define GSCAN_SV_TRIPLES(v) (((v) >> 11) & 31)
#define GSCAN_SV_EXACT3 0x10000
#define GSCAN_SV_RUN_NLO(v) ((v) & 15)
#define GSCAN_SV_RUN_NHI(v) (((v) >> 4) & 3)
#define GSCAN_SV_RUN_FOLD 0x40
#define GSCAN_SV_RUN_LONG 0x80
#define GSCAN_SV_HASH_LEN(v) ((v) & 3)
#define GSCAN_SV_HASH_SPARSE 0x4
#define GSCAN_SV_HASH_COPIES(v) (((v) >> 3) & 63)

#define GSCAN_KERNEL_NONE 0
#define GSCAN_KERNEL_PAIR 1     /* byte-pair SWAR filter (single literals: the HBM-bound kernel) */
#define GSCAN_KERNEL_TRIPLE 2   /* byte-triple SWAR filter (masked / case-insensitive multi-alternative patterns) */
#define GSCAN_KERNEL_BALANCED 3 /* exact byte pairs on both issue pipes + inline third-byte stage (small alternations) */
#define GSCAN_KERNEL_HASH 4     /* perfect-hash membership of the leading bytes (large literal sets) */
#define GSCAN_KERNEL_RUN 5      /* byte-class runs */

#define GSCAN_ENGINE_FIXED 1 /* alternation of fixed-length byte-class sequences (literals, sets) */
#define GSCAN_ENGINE_RUN 2   /* one byte class repeated {n,} (greedy) */
#define GSCAN_ENGINE_NONE 3  /* can never print anything (STRICT_REF with a capturing group) */
#define GSCAN_ENGINE_VM 4    /* general pattern: leading-byte scan + backtracking VM on the device */

typedef struct gscan_stats {
	uint64_t bytes_scanned;  /* sum of unit lengths == algorithmic HBM bytes (SURVEY.md 8(d)) */
	uint64_t n_candidates;   /* records emitted by the scan kernel before the greedy resolve */
	uint64_t n_matches;
	uint32_t n_units, n_tiles;
	uint32_t scan_launches;  /* scan-kernel launches (re-launches after a buffer grow included) */
	uint32_t total_launches; /* all kernels launched by the last call */
	float scan_kernel_ms;    /* CUDA-event time of the scan kernel(s) on the context's stream */
	float resolve_ms;        /* CUDA-event time of the resolve/compaction kernels */
	float h2d_ms;            /* host->device staging (host units only; overlapped with scanning) */
	float total_ms;          /* wall time of the call */
	uint32_t vm_limit_hit;   /* != 0: on at least one unit the device VM ran out of backtracking stack (2048 frames) or steps;
	                            that unit's loop stopped there, as the reference's does when pcre_exec returns an error
	                            (grab.cc:179, quirk Q5) -- the matches before it and all other units are complete */
	uint32_t reserved;
} gscan_stats;

/* ---- pattern: replaces FileGrep::prepare (grab.cc:101-123) ----------------------------- */

/* pcre_compile(regex, 0, ...) + pcre_study + PCRE_INFO_MINLENGTH.  Options-0 byte semantics.
 * Returns 0, or -1 (message: gscan_last_error()) for syntax errors, constructs the device
 * engines do not serve, and patterns that can match the empty string (the reference loops
 * forever on those, grab.cc:209 -- documented deviation Q4).  Thread-safe. */
int gscan_compile(const char *pattern, size_t len, uint32_t flags, gscan_pattern **out);
void gscan_free_pattern(gscan_pattern *p);
/* d_minlen (grab.h:44, grab.cc:120): drives the small-file skip (grab.cc:133-135) and Q1. */
int gscan_minlen(const gscan_pattern *p);
int gscan_pattern_get_info(const gscan_pattern *p, gscan_pattern_info *out);
/* message of the last failed context-free call on this thread (compile) */
const char *gscan_last_error(void);

/* ---- context: replaces FileGrep's ctor/dtor (grab.cc:70-80) ---------------------------- */
gscan_ctx *gscan_open(int device); /* NULL on failure: see gscan_last_error() */
void gscan_close(gscan_ctx *ctx);
/* FileGrep::why() (grab.h:61-64) */
const char *gscan_why(const gscan_ctx *ctx);

/* ---- the hot path: replaces the loop grab.cc:175-213 over many windows ------------------ */

/* Scans units[0..n_units) (host and/or device pointers) and returns, in *out, the matches sorted
 * by (position of the unit in `units`, start) -- for each unit exactly the sequence the reference
 * loop emits, including the tail off-by-one (Q1) and, since every unit is scanned statelessly,
 * the chunk-overlap duplicates/phantoms (Q3).  Host buffers are fully consumed before the call
 * returns (the reference munmap()s right after the loop, grab.cc:215).
 * *out points into a pinned result buffer owned by the context: valid until gscan_free_matches() or gscan_close(),
 * whichever comes first (a second scan before freeing gets a different buffer).  Returns 0 / -1 (gscan_why). */
int gscan_scan_batch(gscan_ctx *ctx, const gscan_pattern *pat, const gscan_unit *units, size_t n_units,
                     uint32_t mode, gscan_match **out, size_t *n_out);
void gscan_free_matches(gscan_ctx *ctx, gscan_match *m);

/* Asynchronous variant (SURVEY.md 8(b) "explicit async variant with a completion call"): starts the same scan on a worker
 * owned by the context and returns at once, so the caller can stat / open / mmap the next batch meanwhile (what the
 * FileGrep mirror's lanes do).  `units` and the host buffers they point to must stay valid and unchanged until
 * gscan_scan_wait() has returned; the context must not be used for anything else in between (one job in flight per
 * context).  gscan_scan_wait() blocks until the job is done and delivers what gscan_scan_batch() would have:
 * 0 / -1 (gscan_why), *out / *n_out as above.  Calling it without a job in flight returns -1. */
int gscan_scan_batch_async(gscan_ctx *ctx, const gscan_pattern *pat, const gscan_unit *units, size_t n_units, uint32_t mode);
int gscan_scan_wait(gscan_ctx *ctx, gscan_match **out, size_t *n_out);

/* Resident variant: plan (and for host units upload) once, scan many times / many patterns. */
int gscan_batch_create(gscan_ctx *ctx, const gscan_unit *units, size_t n_units, gscan_batch **out);
int gscan_batch_scan(gscan_ctx *ctx, const gscan_pattern *pat, gscan_batch *batch, uint32_t mode,
                     gscan_match **out, size_t *n_out);
void gscan_batch_free(gscan_ctx *ctx, gscan_batch *batch);

int gscan_last_stats(const gscan_ctx *ctx, gscan_stats *out);
/* The records of the last successful scan as they sit in device memory (same bytes, same order as *out of that call):
 * for a device-side exchange -- BASELINE config 5's gather of (file id, offset) records to one rank over NCCL reads
 * them from here instead of bouncing through the host.  Valid until the next scan on this context. */
int gscan_last_device_matches(gscan_ctx *ctx, const gscan_match **dptr, size_t *n);

/* ---- utilities (bench / tests; not part of the reference surface) ---------------------- */

/* Pinned host memory for zero-staging H2D (cudaHostAlloc). */
void *gscan_host_alloc(size_t bytes);
void gscan_host_free(void *p);
/* Device memory on the context's GPU. */
void *gscan_device_alloc(gscan_ctx *ctx, size_t bytes);
void gscan_device_free(gscan_ctx *ctx, void *dptr);
int gscan_memcpy_d2h(gscan_ctx *ctx, void *dst, const void *dsrc, size_t bytes);
int gscan_memcpy_h2d(gscan_ctx *ctx, void *ddst, const void *src, size_t bytes);
/* Counter-based synthetic corpus written straight into HBM (host twin: tests/corpus.py):
 * n_files files of file_len bytes at dptr + i*stride, ids first_file_id.. ; printable ASCII with
 * '\n' at p = 3/256; optional needle in files with id % needle_every == needle_every/2. */
int gscan_synth_corpus(gscan_ctx *ctx, void *dptr, uint64_t seed, uint64_t first_file_id, uint64_t n_files,
                       uint64_t file_len, uint64_t stride, const uint8_t *needle, uint32_t needle_len,
                       uint32_t needle_every);
/* Read-only streaming probe (16-byte loads + trivial reduce) over [dptr, dptr+bytes): the
 * measured HBM read roofline of this GPU in the same run (SURVEY.md 8(d)).  ms = kernel time. */
int gscan_read_probe(gscan_ctx *ctx, const void *dptr, uint64_t bytes, float *ms, uint64_t *checksum);
/* The scan kernel's TMA ring with a consumer that looks at nothing: what the streaming structure itself pulls
 * from HBM for this batch (geom 0: streaming geometry, 1: balanced).  ms = kernel time. */
int gscan_tma_probe(gscan_ctx *ctx, gscan_batch *batch, int geom, float *ms);
int gscan_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif
