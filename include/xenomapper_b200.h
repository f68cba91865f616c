/*
 * xenomapper_b200.h -- C ABI of libxenomapper_b200.so
 *
 * Drop-in boundary for xenomapper's read-binning hot path.  Each entry point
 * names the piece of the reference it stands in for; all citations are into
 * xenomapper/xenomapper.py of genomematt/xenomapper v1.0.2 ("xm.py").
 *
 * The library replaces, as ONE call, what the reference does with
 *     readpairs = getReadPairs(sam1, sam2, skip_repeated_reads)     xm.py:95-118
 *     counts    = main_single_end | main_paired_end |
 *                 conservative_main_paired_end(readpairs, six outputs,
 *                                min_score, tag_func)                xm.py:291-556
 * where tag_func is get_tag (xm.py:176), get_tag_with_ZS_as_XS (xm.py:193) or
 * get_cigarbased_AS_tag (xm.py:228).  Headers (process_headers, xm.py:133)
 * and the summary table (output_summary, xm.py:558) stay in the Python host
 * shim, xenomapper_b200/xenomapper.py.
 *
 * Plain C types only: bind with ctypes / cffi / cgo / JNI alike.  There is no
 * CPU fallback: every classify call runs the sm_100a CUDA kernels and fails
 * with XM_ERR_CUDA when no usable device is present.
 */
#ifndef XENOMAPPER_B200_H
#define XENOMAPPER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XM_ABI_VERSION 6

/* States and bins share one numbering: the order of the reference's output
 * arguments (xm.py:291-297).  counts[] is indexed [state] for single-end and
 * [forward_state * 6 + reverse_state] for paired walks (xm.py:330, :420). */
enum xm_bin {
    XM_PRIMARY_SPECIFIC = 0,
    XM_SECONDARY_SPECIFIC = 1,
    XM_PRIMARY_MULTI = 2,
    XM_SECONDARY_MULTI = 3,
    XM_UNASSIGNED = 4,
    XM_UNRESOLVED = 5
};

enum xm_mode {
    XM_MODE_SE = 0,              /* main_single_end, xm.py:291 */
    XM_MODE_PE_LIBERAL = 1,      /* main_paired_end, xm.py:354 */
    XM_MODE_PE_CONSERVATIVE = 2  /* conservative_main_paired_end, xm.py:456 */
};

enum xm_score_src {
    XM_SCORE_AS_XS = 0,          /* tag_func = get_tag */
    XM_SCORE_AS_ZS = 1,          /* tag_func = get_tag_with_ZS_as_XS (--use_zs) */
    XM_SCORE_CIGAR_NM = 2        /* tag_func = get_cigarbased_AS_tag (--cigar_scores) */
};

/* Return codes.  1..4 map onto the exception the reference raises on the same
 * input; the host shim re-raises that class. */
enum xm_status {
    XM_OK = 0,
    XM_ERR_ASSERT = 1,       /* AssertionError: QNAMEs differ at a yielded index (xm.py:106) */
    XM_ERR_VALUE = 2,        /* ValueError: duplicate tag (xm.py:190) or float()/int() rejects the value */
    XM_ERR_RUNTIME = 3,      /* RuntimeError (xm.py:289) */
    XM_ERR_UNICODE = 4,      /* UnicodeDecodeError from the reference's 'rt' file layer */
    XM_ERR_UNSUPPORTED = 5,  /* valid for the reference, outside the device grammar: non-integer or
                                >31-bit scores, non-ASCII bytes, a lone '\r' line break.  Detected and
                                reported, never mis-scored. */
    XM_ERR_NOMEM = 6,
    XM_ERR_CUDA = 7,
    XM_ERR_ARG = 8,
    XM_ERR_IO = 9,
    XM_ERR_INDEX = 10        /* IndexError of the header functions: an empty or header-only file, an empty header, a trailing @PG
                                line without an ID (xm.py:40-43, :124-127) */
};

#define XM_READER_SKIP_REPEATED 1
#define XM_READER_FIRST_IS_CONTEXT 2

typedef struct xm_opts {
    int32_t mode;            /* enum xm_mode */
    int32_t score_src;       /* enum xm_score_src */
    int32_t skip_repeated;   /* reader flags.  Bit 0 (XM_READER_SKIP_REPEATED): getReadPairs(skip_repeated_reads=True), xm.py:110;
                                the CLI sets it for SE (xm.py:691).  Bit 1 (XM_READER_FIRST_IS_CONTEXT): record 0 of both inputs
                                is the record before the caller's range (sharded walks): it is the predecessor the pair predicate
                                (xm.py:402) and the run-skipping reader look at, and is neither classified nor counted. */
    uint32_t enabled_bins;   /* bit b: bin b has an output.  Disabled bins still count (xm.py:330-349) */
    double min_score;        /* --min_score; -inf default (xm.py:298) */
} xm_opts;

typedef struct xm_result {
    uint64_t counts[36];     /* category histogram; zero entries are categories that never occurred */
    uint64_t n_records;      /* records the lockstep reader yielded (xm.py:107) */
    uint64_t out_len[6];     /* bytes written to each bin (0 for disabled bins) */
    uint64_t bytes_in[2];    /* raw bytes of the yielded primary / secondary records (roofline numerator) */
    int32_t status;          /* enum xm_status of the first failing record, XM_OK otherwise */
    int32_t err_stream;      /* 0 primary, 1 secondary, -1 n/a */
    uint64_t err_record;     /* index in the yielded sequence of the failing record */
    float ms_scan;           /* device time of the secondary-stream scan kernel */
    float ms_classify;       /* device time of the primary-stream classify+emit kernel */
    float ms_total;          /* device time of the whole call (CUDA events) */
    uint32_t n_launches;     /* kernels launched by the call */
    float ms_kernel[6];      /* the walk over rows (clean inputs): secondary scan, primary scan, size, prefix + emit; rest 0 */
    uint32_t reserved[2];
} xm_result;

typedef struct xm_ctx xm_ctx;

/* ---- lifetime -------------------------------------------------------- */

/* One context per process and device.  flags: 0.  NULL on failure (see
 * xm_last_error(NULL)). */
xm_ctx *xm_create(int device, uint32_t flags);
void xm_destroy(xm_ctx *ctx);
const char *xm_last_error(const xm_ctx *ctx);
int xm_abi_version(void);

/* ---- device-resident walk ------------------------------------------- */

/* Inputs and outputs live in device memory (16-byte aligned, readable up to
 * the next multiple of 16 past their length).  d_prim / d_sec are the record
 * regions of the two SAM files: everything after the '@' header lines.
 * d_out[b] receives bin b's lines, in input order; out_cap[b] is its
 * capacity.  A bin that would overflow makes the call fail with XM_ERR_ARG
 * after reporting the needed sizes in res->out_len.  Replaces xm.py:95-118
 * + 291-556 for callers that keep SAM text on the GPU. */
int xm_classify_device(xm_ctx *ctx, const void *d_prim, uint64_t prim_len,
                       const void *d_sec, uint64_t sec_len, const xm_opts *opts,
                       void *const d_out[6], const uint64_t out_cap[6], xm_result *res);

/* ---- host-buffer walk ------------------------------------------------- */

/* Same walk on host memory (pageable or pinned): the library stages the two
 * record regions through pinned double buffers with cudaMemcpyAsync, runs the
 * kernels chunk by chunk, and returns the six bins in library-owned host
 * buffers (valid until the next classify call or xm_destroy).  This is what
 * the ctypes shim calls for file-likes without a descriptor (xm.py tests). */
int xm_classify_host(xm_ctx *ctx, const void *prim, uint64_t prim_len,
                     const void *sec, uint64_t sec_len, const xm_opts *opts, xm_result *res);
int xm_get_output(xm_ctx *ctx, int bin, const void **data, uint64_t *len);

/* ---- file-descriptor walk ---------------------------------------------- */

/* Streams two seekable SAM files from the given byte offsets (the first byte
 * after each header) and appends each bin to out_fds[b] (-1 = disabled) with
 * write(2), in record order.  The caller flushes anything it already wrote to
 * those descriptors first (process_headers output).  Replaces the CLI's use
 * of getReadPairs + main_* on real files (xm.py:702-740). */
int xm_classify_fds(xm_ctx *ctx, int fd_prim, int64_t off_prim, int fd_sec, int64_t off_sec,
                    const int out_fds[6], const xm_opts *opts, xm_result *res);

/* ---- sharded walk (one process per GPU) -------------------------------- */

/* Index pass over one resident byte range that starts at a record boundary:
 * how many records it yields (after skip_repeated de-duplication if set, the
 * reader of xm.py:95-118) and whether a blank line ends the stream inside it
 * (xm.py:105).  Ranks exchange these words (all-gather, xenomapper_b200/
 * sharded.py) to turn byte shards into record-index shards. */
typedef struct xm_shard_info {
    uint64_t n_records;      /* records the range yields */
    uint64_t first_start;    /* 0: the range starts at a record boundary */
    uint64_t stop_at;        /* == n_records when a blank line ends the stream inside the range, else UINT64_MAX */
    uint64_t end_off;        /* byte offset just past the last counted record (the blank line's offset when the stream stops) */
} xm_shard_info;
int xm_count_device(xm_ctx *ctx, const void *d_buf, uint64_t len, int skip_repeated, xm_shard_info *info);
/* Byte offsets (in the buffer) at which the records with the given indices start; `len` for indices at or past
 * the buffer's record count.  With the counts above this turns record-index partition points into byte ranges. */
int xm_locate_device(xm_ctx *ctx, const void *d_buf, uint64_t len, int skip_repeated, uint32_t n_queries,
                     const uint64_t *record_index, uint64_t *byte_offset);

/* The same with options.  XM_OUT_BGZF: every bin is written as BGZF (blocked gzip, SAM/BAM specification section
 * 4.1: members of at most 64 KiB of SAM text with the BC extra field) instead of plain text -- what the reference
 * leaves to `| samtools view -bS` (README.md:138).  The walk appends members only; the caller writes its header
 * with xm_bgzf_write before the call and ends each file with xm_bgzf_write(fd, NULL, 0, 1) after it.  Additive:
 * without the flag the six files are the reference's SAM text byte for byte.  gunzip(output) == that text. */
#define XM_OUT_BGZF 1u
int xm_classify_fds_ex(xm_ctx *ctx, int fd_prim, int64_t off_prim, int fd_sec, int64_t off_sec,
                       const int out_fds[6], const xm_opts *opts, uint32_t out_flags, xm_result *res);
/* Two aligner streams in, six bins out, in one call: header processing (xm_process_headers_fds) and the walk, for
 * inputs that cannot seek -- pipes from an aligner, process substitutions, sockets (the reference needs seekable
 * files: xm.py:586-587 -- SURVEY 8f-4).  Both headers are read from the descriptors themselves, every enabled
 * output gets its header (xm.py:133-174; as BGZF members and ended by the end-of-file member with XM_OUT_BGZF),
 * then the records are walked as they arrive.  Seekable files are accepted too (they are read from their start).
 * Returns XM_ERR_INDEX / XM_ERR_UNICODE for the header errors of xm_process_headers_fds. */
int xm_classify_streams(xm_ctx *ctx, int fd_prim, int fd_sec, const int out_fds[6], const xm_opts *opts,
                        uint32_t out_flags, const char *version, xm_result *res);
/* len bytes as BGZF members appended to fd (deflated by the host thread pool); eof != 0: the 28-byte end-of-file
 * member behind them.  No context needed. */
int xm_bgzf_write(int fd, const void *data, uint64_t len, int eof);
/* The bins of an XM_OUT_BGZF walk are deflated ON THE DEVICE before they are copied back (csrc/xm_deflate.h: one warp
 * per member, one prefix code per bin fitted to a sample of its bytes; XM_BGZF_DEFLATE=host in the environment keeps
 * zlib on the host threads).  The same compressor for a host buffer: len bytes in, BGZF members out (no end-of-file
 * member); *out stays valid until the next call on the context. */
int xm_bgzf_deflate_host(xm_ctx *ctx, const void *data, uint64_t len, const void **out, uint64_t *out_len);
typedef struct xm_bgzf_stats {
    uint64_t in_bytes, out_bytes, members;   /* of the device compressor, since the last reset */
    float kernel_ms;                         /* device time of its kernels */
    uint32_t n_launches;
} xm_bgzf_stats;
int xm_bgzf_get_stats(xm_ctx *ctx, xm_bgzf_stats *out, int reset);

/* ---- headers -------------------------------------------------------------- */

/* process_headers (xm.py:133-174) with get_sam_header (xm.py:36-46) and add_pg_tag (xm.py:120-131) on the raw
 * bytes of the two SAM files: the leading '@' lines (universal newlines, valid UTF-8), Xenomapper's @PG line chained
 * with PP: to a trailing @PG line, the @CO comment.  record_offset[k] is the BYTE offset of file k's first record --
 * what xm_classify_fds takes; no tell()/seek() on a text layer is involved.  text[b] / text_len[b]: the header of
 * output b (library-owned, valid until the calling thread's next header call); status[b]: XM_OK, or the error the
 * reference raises when it renders that output's header (it renders them in bin order, enabled outputs only).
 * Returns XM_OK, XM_ERR_INDEX (xm.py:40-43 on either input), XM_ERR_UNICODE or XM_ERR_IO.  No context needed. */
typedef struct xm_headers {
    uint64_t record_offset[2];
    const char *text[6];
    uint64_t text_len[6];
    int32_t status[6];
    int32_t failed_input;      /* which input the return code is about (0 primary, 1 secondary), -1 */
} xm_headers;
int xm_process_headers_fds(int fd_prim, int fd_sec, const char *version, xm_headers *out);
int xm_process_headers_mem(const void *prim, uint64_t prim_len, const void *sec, uint64_t sec_len, const char *version, xm_headers *out);

/* ---- the walk across the GPUs of one box (one process per GPU, NCCL inside the library) ------------ */

/* Every rank holds a BYTE shard of each record region -- bytes [len*r/W, len*(r+1)/W), cut anywhere -- and walks
 * the RECORDS its primary shard holds (getReadPairs is a lockstep reader, xm.py:95-118: the two files must stay
 * aligned by record index, and pair units / QNAME runs must not be cut, xm.py:402, :110-114).  Line heads,
 * context lines and the rows + text of the few secondary records that sit in a neighbour's shard travel over
 * NCCL; nothing else does.  Shard outputs concatenated in rank order equal the single-GPU output.
 * The launcher ferries 128 bytes: rank 0 calls xm_comm_unique_id, every rank xm_comm_init_rank with it. */
#define XM_COMM_ID_BYTES 128
int xm_comm_unique_id(void *id128);
int xm_comm_init_rank(xm_ctx *ctx, int nranks, int rank, const void *id128);
int xm_comm_destroy(xm_ctx *ctx);
/* small collectives for launchers and benchmarks, so that they need no communication library of their own */
int xm_comm_barrier(xm_ctx *ctx);
int xm_comm_allreduce_f64(xm_ctx *ctx, double *values, int n, int op /* 0 sum, 1 max */);

typedef struct xm_shard_stats {
    uint64_t rec_lo, rec_hi;        /* this rank walked records [rec_lo, rec_hi) of the yielded sequence */
    uint64_t n_records_total;       /* records of the whole job */
    uint64_t out_offset[6];         /* where this rank's bytes go inside each bin (sum of the lower ranks' lengths) */
    uint64_t out_total[6];          /* length of each bin over all ranks */
    uint64_t sliver_bytes;          /* bytes this rank received from other ranks: line heads, context lines, rows and text of record slivers */
    uint64_t sent_bytes;
    float align_ms, index_ms, sliver_ms, walk_ms;      /* host wall time of the phases: line heads + context lines, the two scans, the
                                                          sliver exchange, size + prefix + emit */
    float comm_ms;                  /* of which inside collectives / send-receive groups */
    float total_ms;
    uint32_t n_collectives;
    int32_t first_bad_rank;         /* rank that reported the first failing record, -1 if none */
} xm_shard_stats;

/* Device-resident byte shards.  d_prim / d_sec point at the first byte of this rank's shard inside an allocation
 * with at least front_room writable bytes before it and back_room after it (received line heads, slivers; 1 MiB
 * each is plenty unless the two streams' record densities differ wildly between shards).  res->counts and
 * res->n_records describe the whole job, res->out_len this rank's bins.  Clean SAM only (what the barrier-free
 * kernels handle): anything else returns XM_ERR_UNSUPPORTED on every rank, nothing written -- use
 * xm_classify_sharded_host, which then gathers the shards on rank 0 for the exact walk. */
int xm_classify_sharded_device(xm_ctx *ctx, void *d_prim, uint64_t prim_len, void *d_sec, uint64_t sec_len,
                               uint64_t front_room, uint64_t back_room, const xm_opts *opts,
                               void *const d_out[6], const uint64_t out_cap[6], xm_result *res, xm_shard_stats *stats);
/* The same from host memory: this rank's byte shards are uploaded once, walked, and the rank's six bins come back
 * in library-owned host blocks (xm_get_output).  What `torchrun -m xenomapper_b200.xenomapper` calls per rank. */
int xm_classify_sharded_host(xm_ctx *ctx, const void *prim, uint64_t prim_len, const void *sec, uint64_t sec_len,
                             const xm_opts *opts, xm_result *res, xm_shard_stats *stats);

/* ---- BAM input ---------------------------------------------------------- */

/* Replaces the two `samtools view` pipes of xm.py:48-64 (get_bam_header,
 * bam_lines) and getBamReadPairs (xm.py:66-93).  The BGZF blocks are inflated
 * on the GPU (one warp per block; XM_BAM_INFLATE=host: zlib on a pool of host
 * threads), the record chain is followed and the alignment records are rendered
 * as the SAM text lines `samtools view` prints, in device memory, a window of
 * the file at a time, and the walk runs on them; the six bins come back as with
 * xm_classify_host.
 * Float aux values (types f, B:f) print with "%g", as samtools prints them. */
int xm_classify_bam_host(xm_ctx *ctx, const void *prim_bam, uint64_t prim_len,
                         const void *sec_bam, uint64_t sec_len, const xm_opts *opts, xm_result *res);
/* The same with the bins appended to six descriptors as the walk goes (-1: bin disabled), plain or as BGZF members
 * (XM_OUT_BGZF) -- BAM in, BGZF out, inflate and deflate both on the device.  The BAM files may be mapped files:
 * they are read once, front to back. */
int xm_classify_bam_fds(xm_ctx *ctx, const void *prim_bam, uint64_t prim_len, const void *sec_bam, uint64_t sec_len,
                        const int out_fds[6], const xm_opts *opts, uint32_t out_flags, xm_result *res);

/* BAM input for the walk across GPUs (xm_classify_sharded_device).  Every rank maps the whole file; rank r of `world`
 * takes the BGZF blocks that start in its 1/world of the file's bytes and the records that start inside them, inflates
 * them (and as much of what follows as its last record reaches into) and finds its records with the parallel chain:
 *   xm_bam_shard_open   *guess = the offset in the INFLATED stream at which it believes its first record starts (rank 0
 *                       knows), *exit_off = the first record start behind its part -- the next rank's true entry.
 *                       UINT64_MAX in both: the part holds no record start of its own (header only): it passes on the
 *                       entry it is given.
 *   xm_bam_shard_chain  the caller has compared the ranks' numbers (one small all-gather): a rank whose guess was not the
 *                       exit of the rank before it follows its part again from the true entry; *exit_off as above.
 *   xm_bam_shard_text   the part's records as SAM text in device memory, front_room writable bytes before and back_room
 *                       after it: *d_text goes to xm_classify_sharded_device as this rank's byte shard of that stream.
 * stream: 0 primary, 1 secondary.  The buffers stay with the context until the next xm_bam_shard_open on the stream. */
int xm_bam_shard_open(xm_ctx *ctx, int stream, const void *bam, uint64_t len, int rank, int world, uint64_t *guess, uint64_t *exit_off);
int xm_bam_shard_chain(xm_ctx *ctx, int stream, uint64_t entry, uint64_t *exit_off);
int xm_bam_shard_text(xm_ctx *ctx, int stream, uint64_t front_room, uint64_t back_room, void **d_text, uint64_t *text_len);
/* The header text stored in a BAM file (l_text bytes; what `samtools view -H`
 * of xm.py:49 printed before samtools 1.10 began to append its own @PG line).
 * *needed receives its length; it is copied to dst when cap suffices.
 * No context needed; errors are reported through xm_last_error(NULL). */
int xm_bam_header_text(const void *bam, uint64_t len, char *dst, uint64_t cap, uint64_t *needed);
/* All records of one BAM file as SAM text on the host (library-owned, valid
 * until the next BAM call): what iterating getBamReadPairs needs. */
int xm_bam_render_host(xm_ctx *ctx, const void *bam, uint64_t len, const void **text, uint64_t *text_len);
typedef struct xm_bam_stats {
    double inflate_s;        /* wall time from the BGZF bytes to record offsets on the device: upload, inflate, record chain */
    float render_ms;         /* device time of the three BAM text kernels */
    uint32_t n_launches;
    uint64_t bam_bytes, inflated_bytes, text_bytes, records;
    double upload_s;         /* of inflate_s: pageable host memory -> device (the compressed bytes; XM_BAM_INFLATE=host: the inflated ones) */
    float inflate_ms;        /* device time of k_bgzf_inflate */
    uint32_t chain_repairs;  /* segments of the record chain whose guessed entry was not the true one */
} xm_bam_stats;
int xm_bam_get_stats(xm_ctx *ctx, xm_bam_stats *out, int reset);

/* Which kernels the last resident walk (the last step of a chunked one) ran:
 * clean, error-free inputs take the barrier-free pair; anything else the exact
 * pair (DESIGN.md section 4).  For benchmarks and tests. */
#define XM_KERNEL_SCAN2 1u
#define XM_KERNEL_CLASSIFY2 2u
#define XM_KERNEL_SCAN 4u
#define XM_KERNEL_CLASSIFY 8u
#define XM_KERNEL_ROWS 16u          /* k_scan2 over both streams + k_size / k_prefix / k_emit */
int xm_get_walk_kernels(xm_ctx *ctx, uint32_t *mask);

/* ---- device memory helpers (so bindings need no CUDA of their own) ----- */
int xm_dev_alloc(xm_ctx *ctx, uint64_t bytes, void **d_ptr);
int xm_dev_free(xm_ctx *ctx, void *d_ptr);
int xm_host_alloc_pinned(xm_ctx *ctx, uint64_t bytes, void **h_ptr);
int xm_host_free_pinned(xm_ctx *ctx, void *h_ptr);
int xm_memcpy_h2d(xm_ctx *ctx, void *d_dst, const void *h_src, uint64_t bytes);
int xm_memcpy_d2h(xm_ctx *ctx, void *h_dst, const void *d_src, uint64_t bytes);
int xm_memcpy_d2d(xm_ctx *ctx, void *d_dst, const void *d_src, uint64_t bytes);
int xm_dev_mem_info(xm_ctx *ctx, uint64_t *free_bytes, uint64_t *total_bytes);

/* What the host <-> device link alone can do for a walk that uploads h2d_bytes and brings d2h_bytes back: both
 * directions at once, pinned memory, 256 MiB pieces, no kernels.  *ms receives the time of one such round (best of
 * `reps`).  Benchmarks report it next to the end-to-end walk: the distance between the two is what the library adds. */
int xm_copy_ceiling(xm_ctx *ctx, uint64_t h2d_bytes, uint64_t d2h_bytes, int reps, float *ms);

/* tuning knobs for tests: which tile geometry and parse path the kernels use */
#define XM_DEBUG_FORCE_GENERIC 1u   /* every line through the exact byte-wise tokeniser */
#define XM_DEBUG_SMALL_TILES   2u   /* 1 KiB tiles: exercises tile-boundary logic on small inputs */
#define XM_DEBUG_ROWS          4u   /* clean inputs walk over rows (k_scan2 on both streams, k_size, k_prefix, k_emit: the kernels of
                                       the sharded walk) instead of k_scan2 + the fused k_classify2 */
#define XM_DEBUG_EXACT_NAMES   8u   /* the barrier-free kernels join the streams by a 64-bit QNAME hash (xm.py:106); with this flag they
                                       also compare the bytes, as the exact kernels always do (one scattered read of the secondary
                                       line per record: 30 % on the classify kernel).  Environment: XM_EXACT_NAMES=1 */
int xm_set_debug(xm_ctx *ctx, uint32_t flags);

#ifdef __cplusplus
}
#endif
#endif /* XENOMAPPER_B200_H */
