/*
 * inqcall.h -- C ABI of libinqcall.so, the B200 (sm_100a) implementation of the
 * `inquiSTR call` hot path.
 *
 * The reference (wdecoster/inquiSTR v0.13.0) has no FFI for this path; the
 * functions below are the cut a maintainer would bind from src/call.rs to
 * replace the per-locus work of genotype_repeat_{phased,unphased}
 * (call.rs:279-374), call_from_cigar (call.rs:377-413) and median_str_length
 * (call.rs:497-522). INTEGRATION.md shows the Rust `extern "C"` stub.
 *
 * Conventions
 *  - plain C, plain-old-data only; no exceptions cross this boundary.
 *  - every function returns 0 (INQ_OK) or a negative INQ_ERR_* code;
 *    inq_last_error(ctx) gives a human-readable message for the last failure.
 *  - the caller owns all host arrays; the library copies them to the device
 *    and does not keep host pointers after the call returns. Host arrays
 *    obtained from inq_host_alloc are pinned, which makes the copies
 *    asynchronous with respect to the host.
 *  - one ctx per GPU; a ctx is not thread-safe; distinct ctxs may be used
 *    concurrently from distinct host threads.
 *  - there is no CPU fallback: without a usable CUDA device every entry point
 *    that needs one fails with INQ_ERR_CUDA.
 */
#ifndef INQCALL_H
#define INQCALL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INQ_OK 0
#define INQ_ERR_CUDA (-1)            /* CUDA runtime error / no device */
#define INQ_ERR_ARG (-2)             /* invalid argument */
#define INQ_ERR_NOMEM (-3)           /* device or host allocation failed */
#define INQ_ERR_STATE (-4)           /* call order violated (e.g. genotype before set_loci) */
#define INQ_ERR_BAD_HP (-10)         /* a read passing the phased filter has HP not in {0,1,2}: the
                                        reference panics at call.rs:358 */
#define INQ_ERR_MEDIAN_EMPTY (-11)   /* support == 0 and a bucket without spanning reads: the
                                        reference panics at call.rs:516 */
#define INQ_ERR_LOCUS_START (-12)    /* locus start < 10: `start - 10` underflows u32 at
                                        call.rs:285/335 (rejected, SURVEY 8a A4) */
#define INQ_ERR_LOCUS_ORDER (-13)    /* loci not sorted by start within a contig, or end < start
                                        (repeats.rs:102-104) */
#define INQ_ERR_TOO_LARGE (-14)      /* a count exceeds an internal 32-bit index */
#define INQ_ERR_BAD_SA (-17)         /* a read passing the filter carries INQ_FLAG_SA_PANIC: the reference panics
                                        inside is_accidental_2d (call.rs:431,439-450) */

#define INQ_HP_ABSENT 0xFFu          /* hp[] value for a read without an HP tag (call.rs:482-491) */
#define INQ_FLAG_ACCIDENTAL_2D 0x1u  /* flags[] bit0: is_accidental_2d(read) (call.rs:415-459) */
#define INQ_FLAG_SA_PANIC 0x2u       /* flags[] bit1: the read has an S op and an SA tag that is not a string or that
                                        is_accidental_2d cannot split/parse: the reference panics when (and only
                                        when) such a read passes the filter of some locus (call.rs:394,431) */

#define INQ_VALID_H1 0x1u            /* valid_mask bit0: phase1 is a number (else NaN) */
#define INQ_VALID_H2 0x2u            /* valid_mask bit1: phase2 is a number (else NaN) */

typedef struct inq_ctx inq_ctx;

/* Counters and device timings of the last inq_genotype call. Times are CUDA-event
 * milliseconds measured on the library's own streams; the per-stage ones other than ms_total, ms_cigar
 * and ms_scan are 0 unless inq_set_option("timing", 2). */
typedef struct inq_stats {
    uint64_t n_loci;
    uint64_t n_reads;
    uint64_t n_cigar_words;      /* C  : BAM CIGAR words pushed (the device keeps them as about as many 16-bit units) */
    uint64_t n_cigar_words_joined; /* C_j: words of reads joined to >= 1 locus candidate */
    uint64_t n_reads_joined;
    uint64_t n_pairs;            /* P  : (read, locus) pairs that passed the filter into a bucket */
    uint64_t n_candidates;       /* (read, locus) candidates examined by the join */
    uint64_t n_events;           /* I/D/S ops longer than minlen found by the CIGAR scan */
    uint64_t op_visits;          /* sum over pairs of n_cigar(read): what call.rs:382 executes */
    uint32_t n_kernel_launches;  /* kernels launched by the call (direct or replayed from the CUDA graph) */
    uint32_t n_tiles;            /* 32 KB tiles of the device CIGAR stream scanned: 16384 units each (before units were
                                    16 bits, a tile held 8192 words, so the count is half what it was) */
    float ms_total;              /* start of the pass -> everything done, results in host memory */
    float ms_index;              /* memsets */
    float ms_join;               /* K1 read x locus overlap join + segment offsets (second stream, under K2) */
    float ms_cigar;              /* K2 CIGAR scan (dominant kernel) */
    float ms_fixup;              /* CIGAR scan done -> K2b start: prefix scan over the warp-tile totals (and any wait for K1) */
    float ms_scan;               /* tail: CIGAR stream scanned -> end of the pass (what the overlap does not hide) */
    float ms_pairs;              /* K2b event staging, per-pair window sums, scatter into buckets */
    float ms_median;             /* K3 per-locus sort / support filter / median: first chunk start -> last chunk end */
    float ms_h2d;                /* host->device copies of the last inq_push_reads */
    float ms_d2h;                /* last median chunk done -> last result copy done */
    uint32_t n_ranges;           /* always 1: the CIGAR stream is scanned in one launch (kept for the layout) */
    uint32_t used_graph;         /* 1: the pass was replayed from a captured CUDA graph */
    uint32_t reads_sorted;       /* 1: reads were pushed in (contig, ref_start) order */
    uint32_t n_median_chunks;
    uint32_t n_passes;           /* passes run for this call: more than 1 when a speculatively sized buffer was too small,
                                    the CTA-path guess was wrong or a call needed 64-bit keys */
    uint32_t key_bytes;          /* width of the call keys of the last pass: 4, or 8 once these reads had a call outside
                                    [-2^29, 2^29) */
} inq_stats;

/* Create / destroy a context bound to CUDA device `device`. */
int inq_ctx_create(int device, inq_ctx **out);
void inq_ctx_destroy(inq_ctx *ctx);
const char *inq_last_error(const inq_ctx *ctx);   /* ctx may be NULL: message of a failed create */
const char *inq_version(void);

/*
 * Options (both optional; the defaults are what bench.py measures). Returns INQ_ERR_ARG for any other
 * name or a value out of range.
 *   "graph"           1 (default): replay the steady state from a CUDA graph; 0: always launch directly
 *   "timing"          1 (default): three CUDA event records per pass -> inq_stats.ms_total, ms_cigar, ms_scan;
 *                     2: one per stage as well -> every inq_stats.ms_* (each record is a node of the replayed graph
 *                     and costs ~5 us on the chain: ~50 us per pass); 0: none
 */
int inq_set_option(inq_ctx *ctx, const char *name, int64_t value);

/* Pinned host memory for the caller's staging buffers (optional). */
int inq_host_alloc(size_t bytes, void **out);
int inq_host_free(void *p);

/*
 * Locus catalog (replaces RepeatIntervalIterator's Vec<RepeatInterval>, repeats.rs:4-45,
 * after validation repeats.rs:96-115 which stays on the host).
 *   contig_locus_offsets: n_contigs+1 offsets into start/end; loci of contig c are
 *                         [off[c], off[c+1]) and must be sorted by start (ties any order).
 *   start/end           : BED coordinates exactly as the reference uses them (call.rs:285-286).
 * The caller keeps the permutation back to BED order.
 */
int inq_set_loci(inq_ctx *ctx, int32_t n_contigs, const int64_t *contig_locus_offsets,
                 const int32_t *start, const int32_t *end);

/*
 * Aligned reads as flat structure-of-arrays; appends to the reads already pushed.
 * Replaces what the reference pulls off each htslib record in its per-locus loop
 * (call.rs:294-303,345-357,380-382).
 *   contig    : tid of the read (index into the catalog's contigs); reads on contigs
 *               outside [0,n_contigs) are ignored
 *   ref_start : record.reference_start()  (0-based)
 *   ref_end   : record.reference_end() = bam_endpos
 *   mapq, hp (INQ_HP_ABSENT when no HP tag), flags (INQ_FLAG_*)
 *   cigar_off : n_reads+1 offsets (first is 0) into cigar_words for this batch
 *   cigar_words: BAM packed CIGAR, len<<4 | op, ops MIDNSHP=X = 0..8
 * Reads may come in any order.
 */
int inq_push_reads(inq_ctx *ctx, uint64_t n_reads, const int32_t *contig,
                   const int32_t *ref_start, const int32_t *ref_end, const uint8_t *mapq,
                   const uint8_t *hp, const uint8_t *flags, const uint64_t *cigar_off,
                   const uint32_t *cigar_words);

/*
 * Routed push: like inq_push_reads, but keeps only the reads of the batch that htslib's fetch would return for
 * some locus of THIS context's catalog (pos < end+10 && endpos > start-10, call.rs:285-288) and that survive
 * `filter`. With N contexts holding N contiguous shards of the sorted catalog (SURVEY 8e), handing every batch to
 * every context routes the reads -- a read that reaches two shards is taken by both -- without the caller
 * knowing the cuts. The selection runs on `host_threads` host threads (0 = all cores). Coordinate-sorted
 * batches are copied straight from the caller's arrays (a few contiguous runs); scattered ones are gathered
 * through a pinned staging buffer. Reads inside a short gap (<= 256 reads) between two kept reads are shipped as
 * well: they cannot pair with anything and bridging is cheaper than gathering. *n_taken (nullable) receives the
 * number of reads pushed.
 *   INQ_ROUTE_DROP_LOW_MAPQ  drop reads with mapq <= 10: they fail both filters at every locus (call.rs:297-300,350-352)
 *   INQ_ROUTE_DROP_NO_HP     drop reads without an HP tag: they fail the phased filter at every locus (call.rs:350);
 *                            must not be set for an unphased (-u) run
 * Neither flag changes any output (TSV, op_visits): such reads never reach call_from_cigar in the reference.
 */
#define INQ_ROUTE_DROP_LOW_MAPQ 0x1u
#define INQ_ROUTE_DROP_NO_HP 0x2u
int inq_push_reads_routed(inq_ctx *ctx, uint64_t n_reads, const int32_t *contig,
                          const int32_t *ref_start, const int32_t *ref_end, const uint8_t *mapq,
                          const uint8_t *hp, const uint8_t *flags, const uint64_t *cigar_off,
                          const uint32_t *cigar_words, uint32_t filter, int host_threads,
                          uint64_t *n_taken);

/* Optional: size the device buffers once before a series of pushes. The CIGAR stream gets room for n_cigar_words
 * 16-bit units (one per word of ordinary reads); ops of 4095 or more bases take a few units more and grow it in place. */
int inq_reserve_reads(inq_ctx *ctx, uint64_t n_reads, uint64_t n_cigar_words);

/* Forget all pushed reads (device buffers are kept for reuse). */
int inq_clear_reads(inq_ctx *ctx);

/*
 * Genotype every locus of the catalog against the pushed reads.
 * Replaces genotype_repeat_unphased (unphased != 0, call.rs:279-327) or
 * genotype_repeat_phased (unphased == 0, call.rs:329-374) over all loci.
 *   minlen, support: `-m`, `-s` (main.rs:43-49); ops are counted when len > minlen.
 *   twice_h1/twice_h2: n_loci values, 2 x median (exact integer; the f64 the reference
 *                      prints is twice/2.0, call.rs:515-521); undefined where not valid
 *   valid_mask       : n_loci bytes of INQ_VALID_H1 | INQ_VALID_H2 (0 bit => NaN)
 *   stats            : nullable
 * Output order is catalog order. Outputs are host pointers; when they come from inq_host_alloc the
 * results are copied straight into them, chunk by chunk, while later loci are still being reduced.
 */
int inq_genotype(inq_ctx *ctx, uint32_t minlen, uint32_t support, int unphased,
                 int64_t *twice_h1, int64_t *twice_h2, uint8_t *valid_mask, inq_stats *stats);

/* Debug/verification hook used by the parity tests: materialises the per-read event lists of the last
 * inq_genotype (CIGAR order, 1-based anchors; the genotyping pass itself never builds them) and copies
 * them back to the host. Any pointer may be NULL. */
int inq_debug_events(inq_ctx *ctx, uint64_t *n_events, uint32_t *event_pos /*cap*/,
                     int32_t *event_val /*cap*/, uint64_t cap, uint32_t *read_event_off /*n_reads+1*/);

#ifdef __cplusplus
}
#endif
#endif
