/*
 * kbbq_b200.h -- C ABI of the B200-native kbbq recalibration hot path (libkbbq_b200.so).
 *
 * The reference (adamjorr/kbbq-py) has no FFI layer: its boundary is the Python function surface of
 * kbbq/recalibrate.py, kbbq/compare_reads.py and kbbq/gatk/applybqsr.py.  Each entry point below
 * replaces the arithmetic of one of those functions on packed structure-of-arrays batches; the
 * Python package kbbq-py_b200/kbbq keeps the reference's names and signatures and binds these
 * symbols with ctypes (see INTEGRATION.md).  File:line citations are into the reference tree.
 *
 * Conventions
 *  - plain pointers and sizes only; no torch / CUDA types in signatures (`stream` is a
 *    cudaStream_t passed as void*, NULL = default stream);
 *  - every `*_dev` pointer is a DEVICE pointer; functions named *_host take HOST pointers;
 *  - device entry points are asynchronous on `stream`, allocate nothing, keep no global state
 *    and are re-entrant per stream; data errors found on the device (quality > 42, base outside
 *    ACGTN, rg >= R) are OR-ed into the caller's device word `status_dev`
 *    (KBBQ_FLAG_*), which the caller reads after synchronising;
 *  - return value: 0 = ok, negative = KBBQ_E_* (argument / CUDA errors, reported synchronously).
 *
 * Packed batch layout (SURVEY.md section 8d): seq, qual, corr are u8[N*L] row-major by read, all reads
 * of uniform length L; qual holds the phred value (ASCII - 33); rg is u16[N] (read-group int in
 * first-seen order, kbbq/recalibrate.py:59-64; NULL = all 0), second is u8[N]
 * (fastq_infer_secondinpair, kbbq/compare_reads.py:304-306; NULL = all 0).
 * Tables: pos_* int64[R][43][2L], din_* int64[R][43][16] exactly as the reference returns them
 * (kbbq/recalibrate.py:121); the cycle axis holds read-1 cycle i at i and read-2 cycle i at 2L-1-i.
 */
#ifndef KBBQ_B200_H
#define KBBQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KBBQ_NQ 43        /* maxscore + 1 (kbbq/recalibrate.py:22) */
#define KBBQ_NDINUC 16    /* kbbq/compare_reads.py:199-214 */

/* return codes */
#define KBBQ_OK 0
#define KBBQ_E_ARG (-1)       /* bad argument (NULL, negative size, misaligned pointer, L too small) */
#define KBBQ_E_CUDA (-2)      /* a CUDA runtime call failed; see kbbq_last_cuda_error() */
#define KBBQ_E_WORKSPACE (-3) /* workspace too small */
#define KBBQ_E_DATA (-4)      /* host-API only: device status word was non-zero (see flags) */
#define KBBQ_E_IO (-5)            /* FASTQ ingest: open / read / write failed */
#define KBBQ_E_FORMAT (-6)        /* FASTQ ingest: not 4-line records, or sequence / quality lengths differ */
#define KBBQ_E_RAGGED (-7)        /* FASTQ ingest: reads of unequal length (ValueError on this path) */
#define KBBQ_E_NAME_FIELD (-8)    /* --infer-rg: a name without a second '_' field (IndexError in the reference) */
#define KBBQ_E_NAME_RG (-9)       /* --infer-rg: the second '_' field does not start with RG (AssertionError) */
#define KBBQ_E_NAME_MISMATCH (-10) /* corrected read's name does not start with the read's (AssertionError) */
#define KBBQ_E_PEER (-11)          /* multi-GPU entry points: a device cannot reach a peer's memory */
#define KBBQ_E_UNSUPPORTED (-12)   /* kbbq_recalibrate_fastq: a case for the chunked driver (files of different length, or larger than the device) */

/* bits of the device status word */
#define KBBQ_FLAG_QUAL_RANGE 1 /* a quality > 42: IndexError in the reference */
#define KBBQ_FLAG_BAD_BASE 2   /* a base outside ACGTN: TypeError in Dinucleotide.vecget */
#define KBBQ_FLAG_RG_RANGE 4   /* rg[i] >= R */
#define KBBQ_FLAG_SEGMENTS 8   /* kbbq_*_segmented: malformed span table (not sorted / not 16-row aligned / past rows_bound) */
#define KBBQ_FLAG_KMER_FULL 16 /* kbbq_kmer_count / _sieve / _flag / _correct: a probe walked the whole k-mer table */

int kbbq_abi_version(void);
const char *kbbq_strerror(int code);
const char *kbbq_last_cuda_error(void);

/* Number of int64 elements of one cycle table / one dinuc table. */
int64_t kbbq_pos_table_elems(int L, int R);
int64_t kbbq_din_table_elems(int R);

/* Scratch needed by kbbq_build / kbbq_apply for a batch of N reads (bytes, device memory). */
int kbbq_workspace_bytes(int64_t N, int L, int R, size_t *bytes);

/*
 * Table build.  Replaces the per-read body of fastq_to_covariate_arrays: find_corrected_sites
 * (kbbq/recalibrate.py:13-20), cycle and dinuc covariates (kbbq/compare_reads.py:275-302), the
 * mask block (:96-101) and the pos_* / dinuc_* np.add.at calls (:116-119).  ACCUMULATES into the
 * four int64 tables (zero them first for a fresh build; batches and ranks simply add).
 * `path`: 0 = auto, 1 = shared-memory-privatised kernel, 2 = generic global-atomic kernel.
 */
int kbbq_build(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint8_t *corr_dev,
               const uint16_t *rg_dev, const uint8_t *second_dev, int64_t N, int L, int R,
               int minscore, int64_t *pos_errs_dev, int64_t *pos_total_dev, int64_t *din_errs_dev,
               int64_t *din_total_dev, void *workspace_dev, size_t workspace_bytes,
               int *status_dev, int path, void *stream);

/*
 * Marginals + meanq.  rg_* / q_* are the sums of pos_* over cycle (and q), which is what the
 * reference's separate np.add.at calls produce (kbbq/recalibrate.py:112-115); meanq is
 * p_to_q(expected_errs / rg_total) (:111,:120; kbbq/compare_reads.py:262-271).
 * Outputs: q_* int64[R][43], rg_* int64[R], meanq int64[R].  For counts below 2^53, meanq is the exact
 * floor of -10 log10(expected / total) unless expected / total lies within 2^-96 (relative) of a bucket
 * boundary 10^(-m/10) (DESIGN.md §4 K3).  KBBQ_E_ARG for R > 65535.
 */
int kbbq_marginals(const int64_t *pos_errs_dev, const int64_t *pos_total_dev, int L, int R,
                   int64_t *q_errs_dev, int64_t *q_total_dev, int64_t *rg_errs_dev,
                   int64_t *rg_total_dev, int64_t *meanq_dev, void *stream);

/* gatk_delta_q on n independent cells (kbbq/compare_reads.py:235-260).  An inconsistent cell with
 * errs >= tot + 2 gets delta = -prior, as in the reference (its log-likelihood is -inf at every
 * candidate, outside the binomial's support, and np.argmax then gives candidate 0). */
int kbbq_delta_q(const int64_t *prior_q_dev, const int64_t *numerrs_dev,
                 const int64_t *numtotal_dev, int64_t n, int64_t *delta_dev, void *stream);

/*
 * The MAP quality itself for a REAL-valued prior: argmax over q' of prior_dist[|trunc(q' - prior)|] +
 * binom.logpmf, i.e. gatk_delta_q(prior, ...) + prior as the reference's report writer uses it for
 * the EmpiricalQuality column of the read-group table, where the prior is EstimatedQReported rounded
 * to 5 decimals (kbbq/gatk/bqsr.py:293-297; truncation at kbbq/compare_reads.py:245).
 */
int kbbq_posterior_q_real(const double *prior_q_dev, const int64_t *numerrs_dev,
                          const int64_t *numtotal_dev, int64_t n, int64_t *posterior_dev, void *stream);

/*
 * BAM side (SURVEY.md section 8 row f3).  kbbq_build_bam is the tally of bqsr.bam_to_bqsr_covariates
 * (kbbq/gatk/bqsr.py:52-123) for N reads of length L already unpacked from their BAM records:
 *   seq, qual (the OQ qualities), err, skip: u8[N*L]; err / skip = what compare_reads.find_read_errors
 *   (kbbq/compare_reads.py:84-135) and bqsr.trim_bamread (kbbq/gatk/bqsr.py:158-212) return, merged;
 *   rg u16[N]; flags u8[N] (bit 0 = read 2, bit 1 = reverse strand); aln_start / aln_end u16[N] =
 *   query_alignment_start / _end (soft clips lie outside).  skip, rg, flags, aln_* may be NULL.
 * The kernel adds the q < minscore and N skips (:94-96), counts cycles inside the aligned part,
 * backwards on the reverse strand (bamread_bqsr_cycle, :23-31), and takes dinucleotides from the
 * reverse complement there (bamread_bqsr_dinuc, :33-50).  Tables as kbbq_build's, accumulating.
 * kbbq_apply_bam is applybqsr.recalibrate_bamread (kbbq/gatk/applybqsr.py:65-78): whole-read cycles
 * flipped on the reverse strand, reverse-complement dinucleotides, same delta tables as kbbq_apply.
 * With a workspace of kbbq_bam_workspace_bytes(N, L, R) device bytes the batch is first rewritten
 * into canonical reads (position = cycle, reverse strand complemented, skipped and N bases at quality
 * 0) and goes through the shared-memory kernels of kbbq_build / kbbq_apply; with workspace == NULL the
 * direct one-thread-per-base kernels run (global atomics: correct, two orders of magnitude slower).
 * Both paths compute the same tables, qualities and status: a base outside ACGTN in a usable dinucleotide of a
 * forward read raises KBBQ_FLAG_BAD_BASE (the reference's TypeError); elsewhere such a base is tallied and
 * recalibrated as N is in the dinucleotide covariate, and as the base it is in the cycle covariate.
 * aln_start / aln_end past L are cut at L, and aln_end < aln_start is an empty window.  minscore: 0..42.
 */
int kbbq_bam_workspace_bytes(int64_t N, int L, int R, size_t *bytes);
int kbbq_build_bam(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint8_t *err_dev,
                   const uint8_t *skip_dev, const uint16_t *rg_dev, const uint8_t *flags_dev,
                   const uint16_t *aln_start_dev, const uint16_t *aln_end_dev, int64_t N, int L, int R,
                   int minscore, int64_t *pos_errs_dev, int64_t *pos_total_dev, int64_t *din_errs_dev,
                   int64_t *din_total_dev, void *workspace_dev, size_t workspace_bytes, int *status_dev,
                   void *stream);
int kbbq_apply_bam(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint16_t *rg_dev,
                   const uint8_t *flags_dev, int64_t N, int L, int R, int minscore,
                   const int64_t *meanq_dev, const int64_t *rgdq_dev, const int64_t *qdq_dev,
                   const int64_t *posdq_dev, const int64_t *dindq_dev, int nq, int ndin1,
                   uint8_t *out_qual_dev, void *workspace_dev, size_t workspace_bytes, int *status_dev,
                   void *stream);

/*
 * Calibration benchmark counts (SURVEY.md section 8 row f4): the two np.bincount calls of
 * benchmark.calculate_q (kbbq/benchmark.py:76-91), total[q] += 1 and errs[q] += error, over n bases,
 * skipping bases whose skip byte is non-zero (errors[~skips], quals[~skips], kbbq/benchmark.py:102-104).
 * error = err[i] != 0 when `err` is given, else seq[i] != corr[i] (find_corrected_sites,
 * kbbq/recalibrate.py:13-20).  `skip` may be NULL.  total / errs are int64[256] and ACCUMULATE.
 */
int kbbq_calibration_counts(const uint8_t *qual_dev, const uint8_t *err_dev, const uint8_t *seq_dev,
                            const uint8_t *corr_dev, const uint8_t *skip_dev, int64_t n,
                            int64_t *total_dev, int64_t *errs_dev, void *stream);

/*
 * get_delta_qs (kbbq/gatk/applybqsr.py:80-103) for arbitrary axis lengths: q_* is [R][nq],
 * pos_* [R][nq][ncyc], din_* [R][nq][ndin].  Outputs rgdq[R], qdq[R][nq], posdq[R][nq][ncyc],
 * dindq[R][nq][ndin+1] (last dinuc column is the zero pad, :98-101).
 */
int kbbq_get_delta_qs(const int64_t *meanq_dev, const int64_t *rg_errs_dev,
                      const int64_t *rg_total_dev, const int64_t *q_errs_dev,
                      const int64_t *q_total_dev, const int64_t *pos_errs_dev,
                      const int64_t *pos_total_dev, const int64_t *din_errs_dev,
                      const int64_t *din_total_dev, int R, int nq, int ncyc, int ndin,
                      int64_t *rgdq_dev, int64_t *qdq_dev, int64_t *posdq_dev, int64_t *dindq_dev,
                      void *stream);

/*
 * Apply.  Replaces compare_reads.recalibrate_fastq (kbbq/compare_reads.py:320-328) over a batch:
 * out = q < minscore ? q : meanq[rg] + rgdq[rg] + qdq[rg,q] + dindq[rg,q,dinuc] + posdq[rg,q,cycle]
 * with dinuc -1 gathering the last dinuc column and read-2 cycles indexing from the end.  The
 * delta tables have the reference's shapes: qdq [R][nq], posdq [R][nq][2L], dindq [R][nq][ndin1]
 * (nq <= 43; a quality >= nq raises KBBQ_FLAG_QUAL_RANGE).  out_qual is u8[N*L] (no clamp: the
 * low 8 bits of the sum, as the reference keeps whatever the sum is).  A base outside ACGTN anywhere in the
 * batch raises KBBQ_FLAG_BAD_BASE, the rule of kbbq_build, on every path (the shared-memory, generic and
 * segmented kernels write the same bytes and the same status for any input with qualities below 128).
 * minscore: 0..42 (0 has no shared-memory plan: path 1 and the segmented entry points refuse it).
 * path: 0 = shared-memory kernel when a plan fits, else generic; 1 = shared-memory kernel or KBBQ_E_ARG; 2 = generic.
 * path | KBBQ_APPLY_BASES_CHECKED skips the base check: for a caller that has passed these very bytes to kbbq_build
 * and reads the same status word (the build has flagged any base outside ACGTN), or that knows they hold ACGTN only.
 * The check costs the shared-memory kernel about 6 % (DESIGN.md).
 */
#define KBBQ_APPLY_BASES_CHECKED 0x10
int kbbq_apply(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint16_t *rg_dev,
               const uint8_t *second_dev, int64_t N, int L, int R, int minscore,
               const int64_t *meanq_dev, const int64_t *rgdq_dev, const int64_t *qdq_dev,
               const int64_t *posdq_dev, const int64_t *dindq_dev, int nq, int ndin1,
               uint8_t *out_qual_dev, void *workspace_dev, size_t workspace_bytes, int *status_dev,
               int path, void *stream);

/*
 * Segmented batch layout -- the HBM layout of batches with several read groups.
 *
 * The hot kernels keep the tables of ONE read group in shared memory.  kbbq_build / kbbq_apply accept reads of
 * all read groups in any order (rg[] per read) and then gather the pairs of each read group through a work list
 * (one bulk copy per pair: 37-53 % of the HBM roofline).  A SEGMENTED batch stores the rows sorted by
 * key = 2 * rg + second:  rows [seg[k], seg[k+1]) hold the reads of key k, every seg[k] a multiple of 16 rows,
 * rows past the last read of a span are padding (quality 0, base 'A').  Every span streams like a
 * one-read-group batch, so the kernels run at their one-read-group speed for any R; rg[] / second[] are not read.
 * Semantics are those of kbbq_build / kbbq_apply on the same reads in any order (tables are sums over reads,
 * kbbq/recalibrate.py:59-64,111-119; the apply is per base, kbbq/compare_reads.py:320-328).
 *
 *   seg_dev   uint32[kbbq_segment_table_elems(R)]: [0 .. 2R] span offsets in rows, then 2R row counts, then scratch
 *   dest_dev  uint32[N]: row of read i in the segmented batch (0xFFFFFFFF for a read with rg >= R)
 *   segmented arrays hold kbbq_segment_rows_bound(N, R) rows (N rounded up to 16 + 32 R), 16-byte aligned
 *
 * kbbq_segment_plan computes seg and dest from rg / second (either may be NULL = all 0); kbbq_segment_rows
 * moves one u8[N*L] array into the layout (dst row dest[i] = src row i), kbbq_segment_pad fills the padding rows
 * of seq / qual / corr (any may be NULL), kbbq_unsegment_rows brings an array (the recalibrated qualities) back
 * into read order.  A packer that knows rg before it writes a row can produce the layout directly.
 * kbbq_segmented_supported: 1 when the shape has a shared-memory plan (else use kbbq_build / kbbq_apply).
 */
int64_t kbbq_segment_rows_bound(int64_t N, int R);
int64_t kbbq_segment_table_elems(int R);
int kbbq_segmented_supported(int L, int R, int minscore);
int kbbq_segment_plan(const uint16_t *rg_dev, const uint8_t *second_dev, int64_t N, int R, uint32_t *seg_dev,
                      uint32_t *dest_dev, int *status_dev, void *stream);
int kbbq_segment_rows(const uint8_t *src_dev, const uint32_t *dest_dev, int64_t N, int L, uint8_t *dst_segmented_dev,
                      void *stream);
int kbbq_segment_pad(const uint32_t *seg_dev, int R, int L, uint8_t *seq_dev, uint8_t *qual_dev, uint8_t *corr_dev,
                     void *stream);
int kbbq_unsegment_rows(const uint8_t *src_segmented_dev, const uint32_t *dest_dev, int64_t N, int L,
                        int64_t rows_bound, uint8_t *dst_dev, void *stream);
/* kbbq_build / kbbq_apply on a segmented batch of at most rows_bound rows (workspace: kbbq_workspace_bytes(rows_bound, L, R)) */
int kbbq_build_segmented(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint8_t *corr_dev,
                         const uint32_t *seg_dev, int64_t rows_bound, int L, int R, int minscore,
                         int64_t *pos_errs_dev, int64_t *pos_total_dev, int64_t *din_errs_dev,
                         int64_t *din_total_dev, void *workspace_dev, size_t workspace_bytes, int *status_dev,
                         void *stream);
int kbbq_apply_segmented(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint32_t *seg_dev, int64_t rows_bound,
                         int L, int R, int minscore, const int64_t *meanq_dev, const int64_t *rgdq_dev,
                         const int64_t *qdq_dev, const int64_t *posdq_dev, const int64_t *dindq_dev, int nq,
                         int ndin1, uint8_t *out_qual_dev, void *workspace_dev, size_t workspace_bytes,
                         int *status_dev, void *stream);
/* kbbq_apply_segmented with flags = 0 or KBBQ_APPLY_BASES_CHECKED (as kbbq_apply's path flag, for a batch that went
 * through kbbq_build_segmented unchanged) */
int kbbq_apply_segmented_flags(const uint8_t *seq_dev, const uint8_t *qual_dev, const uint32_t *seg_dev,
                               int64_t rows_bound, int L, int R, int minscore, const int64_t *meanq_dev,
                               const int64_t *rgdq_dev, const int64_t *qdq_dev, const int64_t *posdq_dev,
                               const int64_t *dindq_dev, int nq, int ndin1, uint8_t *out_qual_dev, void *workspace_dev,
                               size_t workspace_bytes, int *status_dev, int flags, void *stream);

/*
 * Whole path on HOST buffers: H2D, build, marginals, deltas, apply, D2H -- what
 * recalibrate.recalibrate_fastq (kbbq/recalibrate.py:123-156) does between parsing and printing.
 * Reads are streamed in chunks over three CUDA streams (upload, compute, download); the corrected reads cross
 * PCIe as a 1-bit-per-base mismatch map (kbbq_host_mismatch_bits); with several read groups every chunk is
 * rewritten into the segmented layout on the device.  tables_host (optional, may be NULL) receives
 * [pos_errs | pos_total | din_errs | din_total]; deltas_host (optional) receives
 * [meanq R | rgdq R | qdq R*43 | posdq R*43*2L | dindq R*43*17].  Synchronous; calls are serialised.
 *
 * kbbq_recalibrate_host_multi is the same call over n_dev devices of one box (SURVEY.md section 8e): reads are
 * sharded in contiguous ranges with boundaries at multiples of 16 reads (kbbq/parallel.py: shard_range), one host
 * thread and one session per device; after the build pass every device adds up all the partial tables itself --
 * one kernel reading the peers' tables over NVLink (through pinned host memory when a device cannot reach a
 * peer) -- so all devices hold the same integers, recompute the same deltas and apply them to their shard.
 * rg[] holds the global first-seen read-group numbers (kbbq/recalibrate.py:59-64), assigned before sharding.
 * Results are bit-identical for any device list; a device may be listed more than once.
 */
int kbbq_recalibrate_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                          const uint16_t *rg, const uint8_t *second, int64_t N, int L, int R,
                          int minscore, uint8_t *out_qual, int64_t *tables_host,
                          int64_t *deltas_host, int *status_out, int device);
int kbbq_recalibrate_host_multi(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                                const uint16_t *rg, const uint8_t *second, int64_t N, int L, int R,
                                int minscore, uint8_t *out_qual, int64_t *tables_host,
                                int64_t *deltas_host, int *status_out, const int *devices, int n_dev);

/*
 * FASTQ files in, recalibrated FASTQ out -- recalibrate.recalibrate_fastq (kbbq/recalibrate.py:123-156) as one call:
 * both files are indexed side by side, names checked and read groups inferred (kbbq_fastq_*), then the reads go
 * through a session in chunks: a chunk is tokenised into pinned memory while the previous one crosses PCIe and is
 * added to the tables; after the model step a chunk is applied and copied back while the previous one is formatted
 * straight into the (mapped) output file.  out_fd: where the text goes (stdout's descriptor; a pipe works, a regular
 * file is mapped).  Returns KBBQ_E_UNSUPPORTED, having written nothing, when the files hold different numbers of
 * reads (the reference's zip() semantics) or do not fit the device at once: the chunked driver of
 * kbbq-py_b200/kbbq/recalibrate.py handles those.  *n_reads / *n_rg / *status_out as the other entry points.
 */
int kbbq_recalibrate_fastq(const char *reads_path, const char *corrected_path, int infer_rg, int minscore, int out_fd,
                           int device, int threads, int64_t *n_reads, int *n_rg, int *status_out);

/* The whole-path entry points keep their sessions (device buffers, streams) between calls: allocating several
 * GB per call costs far more than the kernels.  This frees what is cached for `device`. */
int kbbq_host_release(int device);
/* What the last whole-path call on `device` moved over PCIe (bytes of the copies it issued), and the form the
 * reads take on the way up for a session with that many host threads (<= 0: all): 0 = seq + qual + corrected as
 * they are, 1 = seq + qual + 1-bit mismatch map, 2 = qual + 4 bits per base (kbbq_host_pack_nibbles). */
int kbbq_host_last_traffic(int device, int64_t *h2d_bytes, int64_t *d2h_bytes);
int kbbq_host_pack_mode(int host_threads);

/*
 * Sessions: the two passes of kbbq/recalibrate.py:123-156 on one device, fed chunk by chunk from host memory
 * (files that do not fit host or device memory at once; several processes, one per GPU).
 *   create        chunk_reads = capacity of a chunk (<= 0: ~256 MiB per array); resident_reads_cap = how many reads
 *                 may stay in HBM between the passes (0: streaming, pass 2 sends the reads again);
 *                 host_threads = host threads for the mismatch map (<= 0: all)
 *   build_chunk   pass 1 of a chunk: upload + build, accumulating into the session's tables.  Returns once the
 *                 host buffers have been read (they may be reused); the build itself runs behind.
 *   build_range   pass 1 of n reads that lie contiguously in host memory, cut into chunks by the session and
 *                 pipelined across them: the copies of chunk k + 1 are queued before the host cores pack chunk k,
 *                 which a chunk-by-chunk caller cannot do.  Chunks stay resident iff the session was created with
 *                 resident_reads_cap > 0; they are numbered on from the chunks already built.
 *   tables / set_tables / tables_dev   the partial tables [pos_errs | pos_total | din_errs | din_total] for sums
 *                 over sessions or ranks (tables_dev: device pointer, element count and the session's compute
 *                 stream; call kbbq_session_flush before touching them from another stream)
 *   model         marginals + meanq + delta tables from the current tables (deltas_host: optional copy, layout
 *                 as kbbq_recalibrate_host's)
 *   apply_resident / apply_chunk   pass 2 of a chunk kept in pass 1 (by its index) / of reads sent again;
 *                 out_qual is complete after kbbq_session_sync (chunks drain in order)
 *   sync          wait for everything; *status_out = device status word (KBBQ_E_DATA when non-zero)
 *   reset         forget tables and chunks, keep the memory
 * One host thread at a time per session.
 */
typedef struct kbbq_session kbbq_session;
int kbbq_session_create(int device, int L, int R, int minscore, int64_t chunk_reads, int64_t resident_reads_cap,
                        int host_threads, kbbq_session **out);
void kbbq_session_destroy(kbbq_session *s);
int64_t kbbq_session_chunk_reads(const kbbq_session *s);
int kbbq_session_reset(kbbq_session *s);
int kbbq_session_build_chunk(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                             const uint16_t *rg, const uint8_t *second, int64_t n, int keep_resident);
int kbbq_session_build_range(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                             const uint16_t *rg, const uint8_t *second, int64_t n);
int kbbq_session_tables(kbbq_session *s, int64_t *tables_host);
int kbbq_session_set_tables(kbbq_session *s, const int64_t *tables_host);
int kbbq_session_tables_dev(kbbq_session *s, int64_t **tables_dev, int64_t *elems, void **stream);
int kbbq_session_model(kbbq_session *s, int64_t *deltas_host);
int kbbq_session_apply_resident(kbbq_session *s, int64_t chunk, uint8_t *out_qual);
int kbbq_session_apply_chunk(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                             const uint8_t *second, int64_t n, uint8_t *out_qual);
int kbbq_session_flush(kbbq_session *s);
int kbbq_session_sync(kbbq_session *s, int *status_out);
/* bytes the session has copied over PCIe since create / reset */
int kbbq_session_traffic(const kbbq_session *s, int64_t *h2d_bytes, int64_t *d2h_bytes);

/* Host-buffer variants of the two halves (drop-in backing of fastq_to_covariate_arrays and of
 * the apply loop when the caller keeps the tables). Synchronous. */
int kbbq_build_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                    const uint16_t *rg, const uint8_t *second, int64_t N, int L, int R,
                    int minscore, int64_t *pos_errs, int64_t *pos_total, int64_t *din_errs,
                    int64_t *din_total, int *status_out, int device);
int kbbq_apply_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                    const uint8_t *second, int64_t N, int L, int R, int minscore,
                    const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                    const int64_t *posdq, const int64_t *dindq, int nq, int ndin1,
                    uint8_t *out_qual, int *status_out, int device);
int kbbq_get_delta_qs_host(const int64_t *meanq, const int64_t *rg_errs, const int64_t *rg_total,
                           const int64_t *q_errs, const int64_t *q_total, const int64_t *pos_errs,
                           const int64_t *pos_total, const int64_t *din_errs,
                           const int64_t *din_total, int R, int nq, int ncyc, int ndin,
                           int64_t *rgdq, int64_t *qdq, int64_t *posdq, int64_t *dindq, int device);
int kbbq_delta_q_host(const int64_t *prior_q, const int64_t *numerrs, const int64_t *numtotal,
                      int64_t n, int64_t *delta, int device);
int kbbq_posterior_q_real_host(const double *prior_q, const int64_t *numerrs, const int64_t *numtotal,
                               int64_t n, int64_t *posterior, int device);
int kbbq_build_bam_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *err, const uint8_t *skip,
                        const uint16_t *rg, const uint8_t *flags, const uint16_t *aln_start,
                        const uint16_t *aln_end, int64_t N, int L, int R, int minscore, int64_t *pos_errs,
                        int64_t *pos_total, int64_t *din_errs, int64_t *din_total, int *status_out,
                        int device);
int kbbq_apply_bam_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *flags,
                        int64_t N, int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq,
                        const int64_t *qdq, const int64_t *posdq, const int64_t *dindq, int nq, int ndin1,
                        uint8_t *out_qual, int *status_out, int device);
int kbbq_calibration_counts_host(const uint8_t *qual, const uint8_t *err, const uint8_t *seq,
                                 const uint8_t *corr, const uint8_t *skip, int64_t n, int64_t *total,
                                 int64_t *errs, int device);
int kbbq_marginals_host(const int64_t *pos_errs, const int64_t *pos_total, int L, int R,
                        int64_t *q_errs, int64_t *q_total, int64_t *rg_errs, int64_t *rg_total,
                        int64_t *meanq, int device);

/*
 * Synthetic Illumina-shaped reads (SURVEY.md section 8d), counter-based so that any read range can be
 * regenerated anywhere: fills seq/qual/corr u8[n*L], rg u16[n], second u8[n] for reads
 * [first_read, first_read + n) of the stream identified by `seed`.  Bench / test input only.
 */
int kbbq_synth_reads(uint64_t seed, int64_t first_read, int64_t n, int L, int R,
                     uint8_t *seq_dev, uint8_t *qual_dev, uint8_t *corr_dev, uint16_t *rg_dev,
                     uint8_t *second_dev, void *stream);

/*
 * Shared-memory plan the build (arrays = 3) or apply (arrays = 2) kernel would run with for reads of
 * length L and R read groups (max_smem: opt-in shared memory per block, 0 = 232448 of sm_100):
 * out[10] = {reads per group, lanes per group, thread-groups, consumer threads, producer warps,
 * groups per thread-group and stage, ring depth, dinuc replicas, dynamic shared memory, table bytes}.
 * KBBQ_E_ARG when the shape falls back to the generic kernels.  Diagnostics / tests.
 * arrays | KBBQ_PLAN_SEGMENTED: the plan of kbbq_build_segmented / kbbq_apply_segmented instead (the span geometry
 * of a segmented batch, which may differ from that of the same reads in read order).
 */
#define KBBQ_PLAN_SEGMENTED 0x100
int kbbq_plan_info(int L, int R, int minscore, int arrays, int max_smem, int *out);

/*
 * Host FASTQ ingest / egress (SURVEY.md section 8 row f1): multithreaded replacement of what the
 * reference does read by read in Python around the hot path -- pysam.FastxFile + get_quality_array
 * (kbbq/recalibrate.py:56-57,92,141-142), fastq_infer_rg / fastq_infer_secondinpair
 * (kbbq/compare_reads.py:304-318, first-seen numbering kbbq/recalibrate.py:59-64), the name check of
 * find_corrected_sites (kbbq/recalibrate.py:17) and the FASTQ print (kbbq/recalibrate.py:152-156).
 * Host pointers only, no CUDA.  `threads` <= 0: all hardware threads.  4-line records (blank lines at the end are
 * ignored); gzip by its magic bytes; pipes are read into memory.
 */
typedef struct kbbq_fastq kbbq_fastq;
int kbbq_fastq_open(const char *path, int threads, kbbq_fastq **out);
int kbbq_fastq_open_mem(const void *data, size_t len, int threads, kbbq_fastq **out); /* caller keeps data alive */
void kbbq_fastq_close(kbbq_fastq *f);
int64_t kbbq_fastq_num_reads(const kbbq_fastq *f);
int kbbq_fastq_read_len(const kbbq_fastq *f); /* uniform read length; -1 when reads differ; 0 when empty */
/* reads [first, first + n) -> seq u8[n*L] (bytes as they are), qual u8[n*L] (ASCII - 33) */
int kbbq_fastq_pack(const kbbq_fastq *f, int64_t first, int64_t n, uint8_t *seq, uint8_t *qual, int threads);
/* name of read i = header after '@' up to the first blank (points into the file; not NUL terminated) */
int kbbq_fastq_name(const kbbq_fastq *f, int64_t i, const char **name, int *len);
/* second[i] = first '_' field ends in "/2"; rg[i] = 0, or with infer_rg the first-seen number of the
 * text after the last ':' of the second '_' field; *n_rg = number of read groups (>= 1) */
int kbbq_fastq_infer(kbbq_fastq *f, int infer_rg, uint16_t *rg, uint8_t *second, int *n_rg, int threads);
int kbbq_fastq_rg_key(const kbbq_fastq *f, int k, const char **key, int *len); /* after kbbq_fastq_infer */
/* corr.name.startswith(uncorr.name) for the first n reads; *first_bad = first offender */
int kbbq_fastq_check_names(const kbbq_fastq *uncorr, const kbbq_fastq *corr, int64_t n, int threads,
                           int64_t *first_bad);
/* '@' name '\n' seq '\n+\n' (out_qual + 33) '\n' for reads [first, first + n); out_qual u8[n*L] */
int kbbq_fastq_write(int fd, const kbbq_fastq *f, int64_t first, int64_t n, const uint8_t *out_qual, int threads);
/* the same records formatted into memory: *bytes = their total length; dst must hold exactly that many */
int kbbq_fastq_format_size(const kbbq_fastq *f, int64_t first, int64_t n, int threads, int64_t *bytes);
int kbbq_fastq_format(const kbbq_fastq *f, int64_t first, int64_t n, const uint8_t *out_qual, char *dst,
                      int64_t dst_bytes, int threads);

/*
 * Host helper of the host-buffer entry points: bit (i mod 32) of bits[i / 32] = (seq[i] != corr[i]),
 * i.e. find_corrected_sites (kbbq/recalibrate.py:13-20) over n packed bases, multithreaded (threads
 * <= 0: all hardware threads).  bits holds ceil(n / 32) words.  kbbq_recalibrate_host sends this map
 * over PCIe instead of the corrected reads (1/8 of the bytes) unless KBBQ_HOST_NO_BITMAP=1.
 */
int kbbq_host_mismatch_bits(const uint8_t *seq, const uint8_t *corr, int64_t n, uint32_t *bits, int threads);
/* The device side of that: corr_dev[i] = seq_dev[i] ^ bit i, a byte array that differs from seq exactly
 * where the corrected read did -- all kbbq_build looks at.  seq_dev / corr_dev 16-byte aligned. */
int kbbq_expand_mismatch_bits(const uint8_t *seq_dev, const uint32_t *bits_dev, int64_t n, uint8_t *corr_dev,
                              void *stream);

/*
 * The same idea one step further, used by the host-buffer entry points when the host has the cores for it:
 * packed[i / 2] holds, for bases 2k (low nibble) and 2k + 1 (high nibble), (base >> 1) & 7 -- A 0, C 1, T 2, G 3,
 * N 7 -- with bit 3 set where seq[i] != corr[i] (find_corrected_sites, kbbq/recalibrate.py:13-20): the reads and
 * the corrected reads cross PCIe as 0.5 byte per base and only the qualities travel as they are.  *bad_base = 1
 * if a byte of seq is none of ACGTN (the reference's TypeError, kbbq/compare_reads.py:289-302; the device never
 * sees the byte, so the check happens here).  packed holds ceil(n / 2) bytes.
 */
int kbbq_host_pack_nibbles(const uint8_t *seq, const uint8_t *corr, int64_t n, uint8_t *packed, int threads,
                           int *bad_base);
/* The device side: seq_dev from the base codes, corr_dev = a byte array that differs from seq_dev exactly where
 * bit 3 of the nibble is set.  All three pointers 16-byte aligned. */
int kbbq_expand_nibbles(const uint8_t *packed_dev, int64_t n, uint8_t *seq_dev, uint8_t *corr_dev, void *stream);

/*
 * Sequencing errors from the reads' own k-mer spectrum: the mismatch map of a batch without a corrected file
 * (DESIGN.md, "Errors from k-mer counts").  For k in 1..31, window j of a read covers bases [j, j + k); it is valid
 * when all k bases are A, C, G or T (uppercase); its key is min(forward code, reverse-complement code), first base in
 * the most significant 2 bits (A 0, C 1, G 2, T 3).  count(key) = the valid windows of the batch with that key, both
 * strands on one key, exact.  A window is solid when count >= t.  A base no solid window covers is uncovered unless
 * its read has no solid window at all (such a read is left alone).  Every maximal run [a, b] of uncovered bases flags
 * a and b when it is inside the read, b when it starts the read, a when it ends the read; a flagged base that is not
 * A/C/G/T is not flagged.  The flags are the 1-bit map of kbbq_host_mismatch_bits (bit i of the flattened batch in
 * word i / 32, LSB first), which kbbq_expand_mismatch_bits turns into the corrected reads kbbq_build takes.
 *
 * The counts live in an open-addressing table of `capacity` 16-byte slots {u64 key, u64 count} (capacity a power of
 * two, table_dev 16-byte aligned).  kbbq_kmer_table_bytes: the default capacity for N reads of length L, the smallest
 * power of two >= 1.5 x the number of windows N * max(0, L - k + 1), and its bytes.  kbbq_kmer_clear empties a table.
 * kbbq_kmer_count ADDS the windows of a batch (chunks and repeated calls accumulate); a probe that finds no free slot
 * in the whole table raises KBBQ_FLAG_KMER_FULL and stops.  kbbq_kmer_histogram writes hist_dev u64[256]: hist[c] =
 * number of distinct keys with count c, counts above 255 in hist[255], hist[0] = 0.  kbbq_kmer_flag writes all
 * ceil(N * L / 32) words of bits_dev for the threshold t = min_count >= 1 (resolve an automatic threshold with
 * kbbq_kmer_min_count first).  Device pointers, asynchronous on `stream`, no allocation; L up to what one warp's
 * L words of shared memory allow.
 */
int kbbq_kmer_table_bytes(int64_t N, int L, int k, uint64_t *capacity, size_t *bytes);
int kbbq_kmer_clear(void *table_dev, uint64_t capacity, void *stream);
int kbbq_kmer_count(const uint8_t *seq_dev, int64_t N, int L, int k, void *table_dev, uint64_t capacity,
                    int *status_dev, void *stream);
int kbbq_kmer_histogram(const void *table_dev, uint64_t capacity, uint64_t *hist_dev, void *stream);
int kbbq_kmer_flag(const uint8_t *seq_dev, int64_t N, int L, int k, const void *table_dev, uint64_t capacity,
                   int min_count, uint32_t *bits_dev, int *status_dev, void *stream);
/* The automatic threshold: the smallest c in 2..254 with hist[c] <= hist[c + 1] (the first valley of the spectrum),
 * 255 when there is none.  Host only, no device.  KBBQ_E_ARG for a NULL hist. */
int kbbq_kmer_min_count(const uint64_t *hist);

/*
 * Host-buffer forms, synchronous.  kbbq_kmer_errors_host: the map of N reads of length L (bits_out ceil(N * L / 32)
 * words; hist_out u64[256] may be NULL) with t = min_count when > 0, else kbbq_kmer_min_count of the batch's histogram
 * (*min_count_used, may be NULL).  kbbq_recalibrate_kmer_host: kbbq_recalibrate_host with that map in place of a
 * corrected file -- upload, clear + count + histogram, threshold, flag, then kbbq_expand_mismatch_bits, kbbq_build,
 * kbbq_marginals, kbbq_get_delta_qs and kbbq_apply; tables_host / deltas_host (optional) as kbbq_recalibrate_host's.
 * KBBQ_E_UNSUPPORTED when the reads and the default table do not fit the device's free memory; KBBQ_E_DATA with
 * KBBQ_FLAG_KMER_FULL in the status (kbbq_kmer_errors_host has no other flag to report) when the table fills.
 */
int kbbq_kmer_errors_host(const uint8_t *seq, int64_t N, int L, int k, int min_count, uint32_t *bits_out,
                          uint64_t *hist_out, int *min_count_used, int device);
int kbbq_recalibrate_kmer_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                               int64_t N, int L, int R, int minscore, int k, int min_count, uint8_t *out_qual,
                               int64_t *tables_host, int64_t *deltas_host, int *min_count_used, int *status_out,
                               int device);

/*
 * The same counts for inputs of any size: a SIEVED table that only has to hold the keys seen at least twice, filled in
 * two passes over all the reads (DESIGN.md §10, "Streaming").  Slots, hash, probing and empty key as above.
 *   kbbq_kmer_sieve          pass A: per valid window one 64-bit atomicOr of a few bits into one word of filter_dev
 *                            (filter_words u64, a power of two, zeroed before the first chunk); when the word already
 *                            held them all, the key is put in the table with count 0.  Every key with count >= 2 ends
 *                            up in the table whatever the schedule; a key seen once only through a false positive.
 *                            A full table raises KBBQ_FLAG_KMER_FULL.
 *   kbbq_kmer_count_present  pass B: adds 1 to the count of every window whose key is in the table, and the number of
 *                            valid windows to *windows_dev (u64, zeroed before the first chunk).  A probe that walks a
 *                            table with no empty slot raises KBBQ_FLAG_KMER_FULL.
 * Both passes stop probing once KBBQ_FLAG_KMER_FULL is in status_dev: a full table costs no more than a usable one.
 *   kbbq_kmer_histogram_sieved  hist_dev u64[256] equal to kbbq_kmer_histogram's of the exact table: bins 2..255 from
 *                            the table, hist[1] = windows - the sum of the counts >= 2.
 *   kbbq_kmer_flag_sieved    the flags for any t = min_count >= 1: t >= 2 is kbbq_kmer_flag (an absent key has count
 *                            <= 1 < t); t = 1 marks every valid window solid without a lookup.
 * The histogram, threshold and flags equal those of the exact table bit for bit; which false-positive singletons the
 * table holds depends on the schedule.  Device pointers, asynchronous on `stream`, no allocation.
 * kbbq_kmer_stream_plan (host only): sizes for a file of `windows` windows within budget_bytes -- the filter the
 * largest power of two with 8 F <= min(windows, budget / 4) bytes (at least 1 word), the table the exact rule's
 * capacity (kbbq_kmer_table_bytes) or, when that does not fit, the largest power of two with 16 cap <= budget - 8 F.
 * KBBQ_E_UNSUPPORTED when not even min(exact capacity, KBBQ_KMER_MIN_SLOTS) slots fit.  The sizes never change the
 * result, only the memory and whether the table can fill.
 */
#define KBBQ_KMER_MIN_SLOTS 65536
int kbbq_kmer_stream_plan(uint64_t windows, uint64_t budget_bytes, uint64_t *filter_words, uint64_t *capacity);
int kbbq_kmer_sieve(const uint8_t *seq_dev, int64_t N, int L, int k, void *filter_dev, uint64_t filter_words,
                    void *table_dev, uint64_t capacity, int *status_dev, void *stream);
int kbbq_kmer_count_present(const uint8_t *seq_dev, int64_t N, int L, int k, void *table_dev, uint64_t capacity,
                            uint64_t *windows_dev, int *status_dev, void *stream);
int kbbq_kmer_histogram_sieved(const void *table_dev, uint64_t capacity, const uint64_t *windows_dev, uint64_t *hist_dev,
                               void *stream);
int kbbq_kmer_flag_sieved(const uint8_t *seq_dev, int64_t N, int L, int k, const void *table_dev, uint64_t capacity,
                          int min_count, uint32_t *bits_dev, int *status_dev, void *stream);

/*
 * `kbbq recalibrate -r` through a streaming session (resident_reads_cap = 0), chunk by chunk from host memory, in the
 * session's streams and staging slots (a chunk's bytes go up while the previous chunk's kernel runs):
 *   kmer_begin      allocate and clear the filter and the table for k-mers of length k (filter_words / capacity 0:
 *                   kbbq_kmer_stream_plan of `windows`, the windows of the whole input, within 90 % of the free device
 *                   memory; KBBQ_E_UNSUPPORTED when that does not fit)
 *   kmer_sieve      pass A of a chunk of n <= chunk_reads reads (seq: n * L bytes), every chunk of the input
 *   kmer_count      pass B of a chunk, every chunk again; the first call releases the filter, and returns
 *                   KBBQ_E_DATA (KBBQ_FLAG_KMER_FULL in the status word) when the table filled in pass A
 *   kmer_threshold  wait, build the histogram (hist_out u64[256], may be NULL) and take t = min_count when > 0, else
 *                   kbbq_kmer_min_count (*t_used, may be NULL).  KBBQ_E_DATA with KBBQ_FLAG_KMER_FULL in the status
 *                   word (kbbq_session_sync) when the table filled.
 *   build_chunk_kmer  pass 1 of the build with the flags of the chunk as its mismatch map: seq crosses as bytes,
 *                   then flag, kbbq_expand_mismatch_bits and the build of kbbq_session_build_chunk
 * then kbbq_session_model and kbbq_session_apply_chunk as for any streaming session.  Calls out of this order (and
 * on a session that keeps chunks resident) return KBBQ_E_ARG, as do kbbq_session_build_chunk / _build_range /
 * _apply_chunk between kmer_begin and kmer_threshold; kbbq_session_reset releases the k-mer buffers.
 */
int kbbq_session_kmer_begin(kbbq_session *s, int k, int64_t windows, uint64_t filter_words, uint64_t capacity);
int kbbq_session_kmer_sieve(kbbq_session *s, const uint8_t *seq, int64_t n);
int kbbq_session_kmer_count(kbbq_session *s, const uint8_t *seq, int64_t n);
int kbbq_session_kmer_threshold(kbbq_session *s, int min_count, uint64_t *hist_out, int *t_used);
int kbbq_session_build_chunk_kmer(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                                  const uint8_t *second, int64_t n);
/* sizes the session's k-mer buffers were given (0 before kmer_begin) */
int kbbq_session_kmer_sizes(const kbbq_session *s, uint64_t *filter_words, uint64_t *capacity);

/*
 * The correcting walk (DESIGN.md §10): an opt-in rule that finds the errors by correcting each read against its
 * trusted k-mers, as k-mer correctors such as Lighter do.  The boundary rule above flags only the two ends of each
 * uncovered run, so it misses the inner errors of a cluster within k and the outer error of a run at a read end.
 * Counts, keys, validity, t and solid as above; nw = L - k + 1, and L < k flags nothing.  Per read:
 *   1. no solid window: nothing is flagged;
 *   2. the anchor is the longest maximal run [a0, a1] of solid windows, the leftmost of equal ones;
 *   3. right walk on a copy w of the read, j = a1 + 1 .. nw - 1: a solid window j of w goes on to j + 1; otherwise
 *      e = j + k - 1, a w[e] that is not A/C/G/T stops the walk, and for each c in A, C, G, T with c != w[e],
 *      score(c) = the consecutive solid windows j, j + 1, ... of w with w[e] = c, at most min(k, nw - j).  e is
 *      flagged; when exactly one c reaches the best score and it is >= 1, w[e] = c and the walk goes on to j + 1,
 *      else it stops;
 *   4. left walk, the mirror image: j = a0 - 1 down to 0, e = j, at most min(k, j + 1) windows j, j - 1, ...
 * Every flagged base is A/C/G/T.  The bits depend only on the counts.  On a sieved table with t >= 2 they equal the
 * exact table's (an absent key has count <= 1 < t).
 *
 * kbbq_kmer_correct: the map by this rule, on an exact or a sieved table, same arguments and buffers as
 * kbbq_kmer_flag.  min_count == 1 (every valid window solid) only zeroes the map.  A probe that walks the whole table
 * raises KBBQ_FLAG_KMER_FULL.  kbbq_kmer_errors_rule_host / kbbq_recalibrate_kmer_rule_host: kbbq_kmer_errors_host /
 * kbbq_recalibrate_kmer_host with the rule given (kbbq_kmer_errors_host and kbbq_recalibrate_kmer_host are rule
 * KBBQ_KMER_BOUNDARIES).  kbbq_session_kmer_rule: the rule of a streaming session's build_chunk_kmer, allowed from
 * kmer_begin until the first build_chunk_kmer.  An unknown rule or a call out of order returns KBBQ_E_ARG.
 */
#define KBBQ_KMER_BOUNDARIES 0
#define KBBQ_KMER_CORRECT 1
int kbbq_kmer_correct(const uint8_t *seq_dev, int64_t N, int L, int k, const void *table_dev, uint64_t capacity,
                      int min_count, uint32_t *bits_dev, int *status_dev, void *stream);
int kbbq_kmer_errors_rule_host(const uint8_t *seq, int64_t N, int L, int k, int min_count, int rule, uint32_t *bits_out,
                               uint64_t *hist_out, int *min_count_used, int device);
int kbbq_recalibrate_kmer_rule_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                                    int64_t N, int L, int R, int minscore, int k, int min_count, int rule,
                                    uint8_t *out_qual, int64_t *tables_host, int64_t *deltas_host, int *min_count_used,
                                    int *status_out, int device);
int kbbq_session_kmer_rule(kbbq_session *s, int rule);

/*
 * Several GPUs (DESIGN.md §10, "Several GPUs"): the sieved table split by key into n_parts partitions of `capacity`
 * slots each, partition p on any device.  With h = splitmix64(key), the key belongs to partition
 * owner = ((h >> 32) * n_parts) >> 32 and its home slot there is h & (capacity - 1), as in a single table.  Each
 * partition runs passes A and B over EVERY chunk and takes only the windows it owns, W included; each sieved
 * histogram (kbbq_kmer_histogram_sieved of the partition) is then that of its keys, and their sum is the exact
 * histogram of the input.  So the threshold, the flags and everything built from them equal the single table's for
 * any number of partitions and any placement.
 *   kbbq_kmer_sieve_part / kbbq_kmer_count_present_part  pass A / B of partition `part`: kbbq_kmer_sieve /
 *                            _count_present restricted to the windows that partition owns
 *   kbbq_kmer_flag_parts / kbbq_kmer_correct_parts  the map of kbbq_kmer_flag_sieved / kbbq_kmer_correct with every
 *                            lookup in its owner's table (tables[p], read from the device of `stream` -- peer
 *                            memory, NVLink, for the tables of other devices).  min_count == 1 makes no lookup.
 * n_parts == 1 (part 0) is the single-table call.  KBBQ_E_ARG for n_parts outside 1..16, part outside 0..n_parts - 1,
 * a NULL table, or n_parts > 1 with capacity > 2^32.  Device pointers, asynchronous on `stream`, no allocation.
 *
 * kbbq_session_kmer_begin_parts: kbbq_session_kmer_begin with partition p of the table on devices[p] (devices[0] the
 * session's device, KBBQ_E_ARG otherwise; a device may be listed more than once); kbbq_session_kmer_begin is its
 * n_parts = 1 case.  Each chunk of kmer_sieve / kmer_count goes up into the session's device once and is copied
 * (cudaMemcpyPeerAsync) to each other partition; kmer_threshold sums the partitions' histograms; build_chunk_kmer
 * flags on the session's device, reading the other partitions' tables as peer memory.  filter_words / capacity 0:
 * every partition gets the same sizes, kbbq_kmer_stream_plan of ceil(windows / n_parts) windows within the smallest
 * partition budget -- 90 % of its device's free memory shared by the partitions on that device, less two chunks for
 * the copies of partitions p >= 1 -- and at most 2^32 slots (kbbq_session_kmer_sizes reports them).  KBBQ_E_PEER,
 * having allocated nothing, when the session's device cannot read another partition's device (or with
 * KBBQ_MULTI_NO_P2P=1 and n_parts > 1).  A table that fills in any partition is reported as for one table.
 */
int kbbq_kmer_sieve_part(const uint8_t *seq_dev, int64_t N, int L, int k, int part, int n_parts, void *filter_dev,
                         uint64_t filter_words, void *table_dev, uint64_t capacity, int *status_dev, void *stream);
int kbbq_kmer_count_present_part(const uint8_t *seq_dev, int64_t N, int L, int k, int part, int n_parts,
                                 void *table_dev, uint64_t capacity, uint64_t *windows_dev, int *status_dev,
                                 void *stream);
int kbbq_kmer_flag_parts(const uint8_t *seq_dev, int64_t N, int L, int k, const void *const *tables_dev, int n_parts,
                         uint64_t capacity, int min_count, uint32_t *bits_dev, int *status_dev, void *stream);
int kbbq_kmer_correct_parts(const uint8_t *seq_dev, int64_t N, int L, int k, const void *const *tables_dev,
                            int n_parts, uint64_t capacity, int min_count, uint32_t *bits_dev, int *status_dev,
                            void *stream);
int kbbq_session_kmer_begin_parts(kbbq_session *s, int k, int64_t windows, uint64_t filter_words, uint64_t capacity,
                                  const int *devices, int n_parts);

/* Number of kernel launches this library has issued since load (bench.py's gpu_launches). */
int64_t kbbq_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* KBBQ_B200_H */
