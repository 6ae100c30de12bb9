/* mitty_b200 -- C ABI of the B200-native read-generation engine (libmitty_b200.so).
 *
 * Drop-in boundary for Mitty's data-parallel hot path.  The reference (alenzhao/Mitty, pure
 * Python) has no FFI; each entry point below names the reference call it replaces
 * (paths relative to the reference repo) and INTEGRATION.md shows the ctypes binding a
 * maintainer would add to mitty/simulation/{readgenerate,readcorrupt,illumina,rpc}.py.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative
 * MG_E* code, with a message available from mg_last_error(); the caller owns all host buffers
 * (pinned memory makes the copies asynchronous, pageable memory works); one mg_ctx per GPU and
 * one host thread per mg_ctx; there is no global state and NO CPU fallback -- without a CUDA
 * device mg_ctx_create fails.
 */
#ifndef MITTY_B200_H
#define MITTY_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mg_ctx mg_ctx;

#define MG_OK 0
#define MG_ECUDA (-1)      /* CUDA runtime error                                   */
#define MG_EINVAL (-2)     /* bad argument / unknown handle                        */
#define MG_ECAP (-3)       /* caller buffer too small; needed size reported        */
#define MG_EVALUE (-4)     /* input the reference would reject or cannot represent */
#define MG_EINDEX (-5)     /* read longer than the model (IndexError, illumina.py:156) */

#define MG_MODE_PHILOX_C 0 /* production: counter-based Philox draws on the device (4x32-10; corruption stream 4x32-7) */
#define MG_MODE_DET_C 1    /* deterministic: the reference's numpy RandomState draws, from host  */
#define MG_MODE_EXPLICIT_C 2 /* test hook: explicit template starts and lengths                 */

/* ---- context ------------------------------------------------------------------------------ */
/* stream: a cudaStream_t to launch on (e.g. torch's current stream) or NULL for an own stream. */
int mg_device_count(void);   /* number of CUDA devices (0 if none / no driver) */
int mg_ctx_create(int device, void *stream, mg_ctx **out);
void mg_ctx_destroy(mg_ctx *ctx);
const char *mg_last_error(mg_ctx *ctx);   /* NULL: the last failed mg_bam_write_sorted of this thread */
int mg_synchronize(mg_ctx *ctx);

/* page-locked host memory for the caller's FASTQ buffers (makes the D2H copies of
 * mg_unit_generate / mg_corrupt_fastq run at full PCIe speed and asynchronously)                 */
int mg_host_alloc(mg_ctx *ctx, int64_t bytes, void **out);
int mg_host_free(mg_ctx *ctx, void *p);

/* ---- read model: illumina.read_model_params hand-off (mitty/simulation/illumina.py:12-40) ---
 * cum_tlen f64[n_tlen]; cum_bq_mat f64[n_mates][n_cycles][n_bq]; phred_p f64[100] =
 * 10**(-arange(100)/10) (illumina.py:137); rlen = model['mean_rlen'].                          */
int mg_model_load(mg_ctx *ctx, const double *cum_tlen, int n_tlen, const double *cum_bq_mat, int n_mates,
                  int n_cycles, int n_bq, const double *phred_p, int rlen);

/* production-mode corruption tables derived from the model at load time (for tests / inspection;
 * the draw layout is documented at MgCorruptCtx in mitty_b200/csrc/mg_core.cuh): per (mate, cycle) ONE
 * Vose alias row over the joint outcomes (quality, substitution) of illumina.corrupt_single_read
 * (illumina.py:151-160).  which = 0: the table of the fused emit kernel (cycles < rlen); 1: the table of
 * the standalone corrupt kernel (all n_cycles).  alias_out u32[n_mates][n_cycles][1 << *kshift];
 * *code9 = 1 when the outcome codes are 9 bits wide (some quality >= 64 carries mass), else 8 bits;
 * *n_rows = number of leading cycles that were built.                                            */
int mg_model_tables(mg_ctx *ctx, int32_t which, uint32_t *alias_out, int64_t alias_cap, int32_t *kshift, int32_t *code9,
                    int32_t *n_rows);

/* ---- region: replaces fasta.fetch(chrom, start, end) + the str the worker keeps
 * (mitty/simulation/readgenerate.py:186).  ref_bytes = the region's bases as in the FASTA
 * (ASCII); bed_start = 0-based start.  The sequence is 2-bit packed on the device; runs of
 * non-ACGT bytes (N, IUPAC, lower case) are kept as an exception list.                          */
int mg_region_load(mg_ctx *ctx, const uint8_t *ref_bytes, int64_t len, int64_t bed_start, int64_t *region_id);
int mg_region_free(mg_ctx *ctx, int64_t region_id);

/* ---- chromosome copy: replaces rpc.create_node_list (mitty/simulation/rpc.py:38-116) and the
 * p_min/p_max computation (readgenerate.py:192).  Variants of ONE copy in VCF order (output of
 * vcfio.parse, mitty/lib/vcfio.py:105-126): pos 1-based, op 'X'/'I'/'D', oplen, ALT strings
 * pooled as alt_pool[alt_off[i] .. alt_off[i+1]).  Builds the node table (the greedy walk runs on
 * the device), the packed haplotype and the block lookup table in HBM.  POS must be sorted, as the
 * records of an indexed fetch are (MG_EVALUE otherwise); a node list that would end in 'D'
 * (deletion across the region end, readgenerate.py:192) is MG_EVALUE too.                       */
int mg_copy_build(mg_ctx *ctx, int64_t region_id, int64_t n_var, const int64_t *pos, const uint8_t *op,
                  const int64_t *oplen, const uint8_t *alt_pool, const int64_t *alt_off, int64_t *copy_id,
                  int64_t *p_min, int64_t *p_max, int64_t *n_nodes);
int mg_copy_free(mg_ctx *ctx, int64_t copy_id);
/* node table as the reference's Node tuples (rpc.py:5-35): arrays of n_nodes entries            */
int mg_copy_nodes(mg_ctx *ctx, int64_t copy_id, int64_t *ps, int64_t *pr, uint8_t *op, int64_t *oplen);
/* the copy's haplotype as ASCII (p_max - p_min bytes), read back from the packed device copy    */
int mg_copy_haplotype(mg_ctx *ctx, int64_t copy_id, uint8_t *out, int64_t cap);

/* ---- one work unit ------------------------------------------------------------------------- */
typedef struct {
  int64_t copy_id;
  int64_t n_candidates;     /* int((p_max - p_min) * p * 1.2), illumina.py:69                    */
  double p;                 /* per-base template probability (PHILOX mode gaps)                  */
  int32_t mode;             /* MG_MODE_*_C                                                       */
  uint32_t unit_seed;       /* rng_seed of the unit (readgenerate.py:150); Philox key            */
  const int64_t *ts;        /* DET/EXPLICIT [n]: geometric(p).cumsum()+p_min+1, shuffled (illumina.py:70-71) */
  const double *u_tlen;     /* DET [n]: tlen_rng.rand(n) (illumina.py:72)                        */
  const int64_t *tl;        /* EXPLICIT [n]: template lengths                                    */
  const int8_t *fo;         /* DET/EXPLICIT [n]: file_order_rng.randint(2, ...) (illumina.py:93), consumed in kept order */
  const char *qname_prefix; /* "@<sample>:<worker_id>:<ps>:"  (readgenerate.py:195,210)          */
  const char *qname_mid;    /* "|<chrom>|<cpy>"               (readgenerate.py:223)              */
  int32_t corrupt;          /* 1: fuse Illumina corruption (PHILOX draws) into the emit kernel    */
  uint32_t corrupt_seed;
  int64_t p_min, p_max;     /* only read by mg_sample_templates when copy_id == 0 (plugin call
                               generate_reads(model, p_min, p_max, seed) without a haplotype)      */
} mg_unit_desc;

/* replaces read_module.generate_reads (illumina.py:43-110): per candidate j the template start
 * ts_out[j], end te_out[j] (-1 if te >= p_max) and, in PHILOX mode, the file-order bit.          */
int mg_sample_templates(mg_ctx *ctx, const mg_unit_desc *d, int64_t *ts_out, int64_t *te_out, int8_t *fo_out);

/* replaces the per-unit body of read_generating_worker + fastq_lines + writer
 * (readgenerate.py:183-253).  Writes the unit's FASTQ records of file 1 / file 2 into out1 / out2
 * (host buffers of `cap` bytes each; NULL,NULL keeps the result on the device only).
 * n_bytes = bytes per file (both files always have the same size), n_templates = templates
 * written, n_te_kept = templates that passed te < p_max.  MG_ECAP if cap < n_bytes.             */
int mg_unit_generate(mg_ctx *ctx, const mg_unit_desc *d, uint8_t *out1, uint8_t *out2, int64_t cap,
                     int64_t *n_bytes, int64_t *n_templates, int64_t *n_te_kept);

/* same, but returns as soon as the kernels have finished and the device-to-host copies are
 * ENQUEUED (on the context's copy stream): the next unit's kernels overlap with them.  out1/out2
 * (pinned memory) are valid after mg_wait_copies(); at most two units may be in flight, i.e. a
 * buffer pair may be reused for the unit after next.                                            */
int mg_unit_generate_async(mg_ctx *ctx, const mg_unit_desc *d, uint8_t *out1, uint8_t *out2, int64_t cap,
                           int64_t *n_bytes, int64_t *n_templates, int64_t *n_te_kept);
int mg_wait_copies(mg_ctx *ctx);

/* streams a unit that was generated with out1 = out2 = NULL (bytes left on the device) through a
 * small pinned ring instead of one unit-sized host buffer: copies bytes [offset, offset + bytes) of
 * file `file` (0 / 1) of the MOST RECENT unit to dst, asynchronously on the copy stream; dst is
 * valid after mg_wait_copies().  The writer loop of readgenerate.py:233-253 then appends chunk by
 * chunk.                                                                                          */
int mg_unit_read_async(mg_ctx *ctx, int32_t file, int64_t offset, int64_t bytes, uint8_t *dst);

/* ---- output sink: replaces the FASTQ writer process (mitty/simulation/readgenerate.py:233-253,
 * readcorrupt.py:100-118) and the `>(gzip > r1.fq.gz)` the reference is piped into (Readme.md:170).
 * Native writer threads: producers (one per GPU) fill page-locked slot pairs from their own pool and
 * commit them with (unit, offset); the files receive the units in SCHEDULE order whatever the order of
 * arrival -- pwrite() at the final offset for regular files, ordered sequential writes for FIFOs /
 * pipes, and with gzip_level > 0 one deflated gzip member per piece, appended in order (a valid
 * multi-member .gz).  path2 may be NULL (`generate-reads` without --fastq2: only file 1 is written).   */
typedef struct mg_sink mg_sink;
int mg_sink_create(const char *path1, const char *path2, int64_t n_units, int32_t n_producers, int32_t slots_per_producer,
                   int64_t chunk_bytes, int32_t gzip_level, int32_t n_threads, mg_sink **out);
/* the same for several PROCESSES sharing one pair of (regular) output files, e.g. one rank per GPU:
 * table_path names a small file (on /dev/shm) that carries the unit sizes and the next-unit counter;
 * the process with table_owner = 1 creates it and truncates the outputs, the others open both after a
 * barrier of the callers.  Plain output to regular files only.                                       */
int mg_sink_create_shared(const char *path1, const char *path2, int64_t n_units, int32_t n_producers, int32_t slots_per_producer,
                          int64_t chunk_bytes, int32_t gzip_level, int32_t n_threads, const char *table_path, int32_t table_owner,
                          mg_sink **out);
/* hands out the schedule's units one by one (to threads or, with a shared table, to processes): the
 * next unit index, or -1 when all are taken.  Whoever takes a unit must announce its size.            */
int64_t mg_sink_next_unit(mg_sink *s);
/* bytes per file of a unit: announced once per unit (0 for an empty one), before its pieces          */
int mg_sink_unit_size(mg_sink *s, int64_t unit, int64_t bytes_per_file);
/* a free slot pair of the producer's pool (blocks while all are in flight)                           */
int mg_sink_acquire(mg_sink *s, int32_t producer, void **buf1, void **buf2, void **slot);
/* bytes [offset, offset + bytes) of `unit` (both files) are in the slot: write them, recycle the slot  */
int mg_sink_commit(mg_sink *s, void *slot, int64_t unit, int64_t offset, int64_t bytes);
/* one slot carrying pieces of several units (a batch of small units): sub-piece i = bytes
 * [slot_off[i], slot_off[i] + bytes[i]) of the slot = bytes [unit_off[i], ...) of unit[i]            */
int mg_sink_commit_multi(mg_sink *s, void *slot, int32_t n, const int64_t *unit, const int64_t *unit_off, const int64_t *slot_off,
                         const int64_t *bytes);
/* page-locks n buffers of chunk_bytes ahead of mg_sink_create (which takes them from the library's cache): the slow
 * part of creating a sink, overlapped by the caller with its input parsing.  -> buffers locked                  */
int32_t mg_sink_prealloc(int64_t chunk_bytes, int32_t n, int32_t n_threads);
void mg_sink_abort(mg_sink *s, const char *why);   /* wakes every blocked producer with an error       */
const char *mg_sink_error(mg_sink *s);
int64_t mg_sink_chunk_bytes(mg_sink *s);          /* bytes per slot, as given at creation             */
/* waits for everything committed, closes the files, frees the sink; bytes written per file           */
int mg_sink_close(mg_sink *s, int64_t *written1, int64_t *written2);

/* streams the MOST RECENT unit of ctx (generated with out1 = out2 = NULL: its bytes are still on the
 * device) into the sink as schedule unit `unit`: announces its size and returns; a thread of the
 * context copies it out piece by piece (copy stream) while the caller generates the next unit.  The
 * unit after next waits for this one's device buffers.  mg_drain_wait: everything queued is committed. */
int mg_unit_drain_async(mg_ctx *ctx, mg_sink *sink, int32_t producer, int64_t unit);
int mg_drain_wait(mg_ctx *ctx);

/* ---- batches of small regions (an exome-style BED): what read_generating_worker does region by region
 * and unit by unit (mitty/simulation/readgenerate.py:183-214) for MANY (region, copy) pairs and MANY
 * work units in a handful of launches.  mg_batch_build packs the regions' reference bytes
 * (ref_bytes[ref_off[r] .. ref_off[r + 1]), ref_off[0] = 0) back to back and builds ONE node table /
 * haplotype / block table over all segments (a segment = one chromosome copy of one region: its variants
 * are [seg_var_off[s], seg_var_off[s + 1]) of the variant arrays, as for mg_copy_build); seg_p_min /
 * seg_p_max are what readgenerate.py:192 computes per copy.  mg_batch_generate runs the units (unit_seg =
 * segment, unit_seed = rng_seed, unit_ncand = int((p_max - p_min) * p * 1.2) <= 2048, unit_index = index
 * in the schedule, ascending; DET mode: the units' draws concatenated, cand_off[u] = first entry of unit
 * u, cand_off[n_units] = their number) and, with a sink, streams their FASTQ into it (every unit's size
 * announced, then the pieces committed by the context's drain thread); without a sink the units' bytes
 * stay on the device back to back (mg_unit_read_async).  qnames are
 * "@<sample>:0:<unit_index>:<serial>|<chrom_pool[chrom_off[s] .. chrom_off[s + 1])>|<seg_cpy[s]>|...".
 * unit_bytes / unit_templates (n_units entries each, may be NULL): bytes per file and templates of
 * every unit.  The bytes equal those of mg_unit_generate unit by unit.                               */
int mg_batch_build(mg_ctx *ctx, int64_t n_regions, const uint8_t *ref_bytes, const int64_t *ref_off, const int64_t *bed_start,
                   int64_t n_segs, const int32_t *seg_region, const int64_t *seg_var_off, const int64_t *pos, const uint8_t *op,
                   const int64_t *oplen, const uint8_t *alt_pool, const int64_t *alt_off, int64_t *batch_id, int64_t *seg_p_min,
                   int64_t *seg_p_max);
int mg_batch_free(mg_ctx *ctx, int64_t batch_id);
int mg_batch_generate(mg_ctx *ctx, int64_t batch_id, int64_t n_units, const int32_t *unit_seg, const uint32_t *unit_seed,
                      const int64_t *unit_ncand, const int64_t *unit_index, const char *sample, const uint8_t *chrom_pool,
                      const int64_t *chrom_off, const int32_t *seg_cpy, double p, int32_t mode, const int64_t *ts, const double *u_tlen,
                      const int8_t *fo, const int64_t *cand_off, int32_t corrupt, uint32_t corrupt_seed, mg_sink *sink,
                      int32_t producer, int64_t *n_templates, int64_t *n_bytes, int64_t *unit_bytes, int64_t *unit_templates);

/* ---- FASTA front end: pysam.FastaFile(fname).fetch(reference=, start=, end=) as the reference uses it
 * (mitty/simulation/readgenerate.py:181, 186), native and free of the GIL, so that the worker threads of
 * several GPUs fetch their regions at the same time.  Plain (not gzip) files; contigs with lines of one
 * width are addressed arithmetically in the mapped file, ragged ones are stripped once.  Bytes come back
 * as they are in the file.  mg_fasta_fetch -> bases written (start / end clamped to the contig, as a numpy
 * slice), MG_EINDEX for an unknown contig.                                                            */
typedef struct mg_fasta mg_fasta;
int mg_fasta_open(const char *path, mg_fasta **out);
void mg_fasta_close(mg_fasta *f);
int64_t mg_fasta_n_contigs(mg_fasta *f);
int mg_fasta_contig(mg_fasta *f, int64_t i, const char **name, int64_t *length, int32_t *uniform);
int64_t mg_fasta_fetch(mg_fasta *f, const char *name, int64_t start, int64_t end, uint8_t *out, int32_t threads);

/* ---- corrupt-reads: replaces readcorrupt.multi_process / illumina.corrupt_template
 * (mitty/simulation/readcorrupt.py:18-118, illumina.py:113-162) over whole FASTQ buffers.
 * in2/out2 may be NULL (single-end).  DET mode consumes the reference's draws: for read k (file-1
 * read then file-2 read of each template) bq_rnd/call_rnd/base_rnd[draw_off[k] + cycle].
 * Large files are streamed in chunks: only COMPLETE templates present in both buffers are
 * processed; consumed1/2 = input bytes they occupied (carry the rest into the next call) and
 * first_template = number of templates processed by earlier calls (keeps the Philox counters,
 * hence the output, independent of the chunking).                                                */
int mg_corrupt_fastq(mg_ctx *ctx, const uint8_t *in1, int64_t len1, const uint8_t *in2, int64_t len2, int32_t mode,
                     uint32_t seed, const double *bq_rnd, const double *call_rnd, const uint8_t *base_rnd,
                     const int64_t *draw_off, uint8_t *out1, uint8_t *out2, int64_t cap, int64_t *out_len1,
                     int64_t *out_len2, int64_t *n_templates, int64_t first_template, int64_t *consumed1,
                     int64_t *consumed2);

/* ---- round-trip checker: the god-aligner contract (mitty/benchmarking/god_aligner.py:141-183 over
 * readgenerate.parse_qname, mitty/simulation/readgenerate.py:259-291) verified on the device for EVERY
 * read of a FASTQ pair of PERFECT reads: (chrom, copy, strand, POS, CIGAR) from the qname + reference +
 * node list must re-derive the bases in the file ('=' equals the reference, 'X' equals the haplotype and
 * differs from the reference, 'I' carries the inserted bases, 'D' skips reference, '>p:nI' lies inside one
 * insertion; strand 1 is reverse-complemented first).
 * mg_check_add_copy registers a built copy under the (chrom, copy) the qnames name; reference and
 * haplotype are expanded to text views on the device.  mg_check_fastq checks the COMPLETE templates
 * present in both buffers (consumed1/2 as for mg_corrupt_fastq) and reports the first bad_cap failures:
 * bad_index = file * n_records + record, bad_code = 1 malformed qname, 2 unknown chrom/copy, 3 length,
 * 4 '=' mismatch, 5 'X' mismatch, 6 inserted bases, 7 no insertion at POS, 8 unknown op, 9 out of range,
 * 10 not a 4-line record with a bare '+' line.                                                        */
typedef struct mg_checker mg_checker;
int mg_check_open(mg_ctx *ctx, mg_checker **out);
void mg_check_close(mg_checker *k);
int mg_check_add_copy(mg_checker *k, int64_t copy_id, const char *chrom, int32_t cpy);
int mg_check_fastq(mg_checker *k, const uint8_t *in1, int64_t len1, const uint8_t *in2, int64_t len2, int64_t *n_records,
                   int64_t *n_bad, int64_t *bad_index, int32_t *bad_code, int32_t bad_cap, int64_t *consumed1, int64_t *consumed2);

/* ---- god-aligner: replaces mitty/benchmarking/god_aligner.py (process_multi_threaded, god_aligner.py:43-121).
 * Every read of a FASTQ (pair) becomes one BAM record at the POS / CIGAR its qname states, strand-1 reads
 * reverse-complemented back; the records are encoded and sorted by (refID, pos, reverse bit) on the device
 * in runs of at most run_bytes of device memory (<= 0: derived from free memory) and written as a BGZF BAM
 * with a BAI index by `threads` host deflate threads at `level`.
 * mg_bam_open: the FASTA's contigs in order, the SAM header text (@HD / @SQ / @RG lines), the RG value;
 * bai_path NULL writes no index.  mg_bam_add encodes the COMPLETE templates present in both buffers
 * (consumed1/2 as for mg_corrupt_fastq; fewer when the run is full: call again with the rest); a read the
 * BAM cannot hold is MG_EVALUE with bad_index = template * files + file and bad_code = 1 not a 4-line
 * record, 2 malformed qname, 3 chrom not in the FASTA, 4 name over 254 bytes, 5 length differs from rlen /
 * CIGAR, 6 malformed CIGAR, 7 alignment outside the contig.  mg_bam_close sorts / merges the last run and
 * writes BAM + BAI (n_runs: sorted runs used; times[3] ms: device work incl. ingest, device-to-host copies,
 * writing); on error nothing is left behind.  mg_bam_abort drops everything, temporary files included.
 * mg_bam_write_sorted: the BGZF writer + BAI builder alone, without a device, over records already encoded
 * and in coordinate order.  Both reject a contig of 2^31 bases or more (MG_EVALUE, before any file is
 * created): BAM keeps its length, POS, PNEXT and TLEN in int32.                                       */
typedef struct mg_bam mg_bam;
int mg_bam_open(mg_ctx *ctx, const char *bam_path, const char *bai_path, int32_t n_ref, const char *const *ref_names, const int64_t *ref_len,
                const char *header_text, const char *sample, int32_t level, int32_t threads, int64_t run_bytes, mg_bam **out);
int mg_bam_add(mg_bam *b, const uint8_t *in1, int64_t len1, const uint8_t *in2, int64_t len2, int64_t *n_templates, int64_t *consumed1,
               int64_t *consumed2, int64_t *bad_index, int32_t *bad_code);
int mg_bam_close(mg_bam *b, int64_t *n_records, int64_t *n_runs, double *times);
void mg_bam_abort(mg_bam *b);
int mg_bam_write_sorted(const char *bam_path, const char *bai_path, int32_t n_ref, const char *const *ref_names, const int64_t *ref_len,
                        const char *header_text, const uint8_t *records, int64_t len, int32_t level, int32_t threads, int64_t *n_records);

/* ---- bam2illumina: replaces mitty/empirical/bam2illumina.py -- the per-base counts of an Illumina read model
 * over every alignment record of a BGZF BAM file or FIFO (any sort order, no index).  Host threads
 * (`threads`) inflate the BGZF members into page-locked chunks of about chunk_bytes; each chunk of whole
 * records is copied to the device and counted there while the next one is inflated.  Record k (0-based,
 * file order) is considered iff k % every == 0; it is skipped for flag & 0xB04, mapq < min_mq, l_seq == 0,
 * missing QUAL (0xFF) or l_seq > max_bp, in that order; otherwise mate = (flag & 0xC1) == 0x81, base i of
 * SEQ is cycle l_seq - 1 - i on the reverse strand (else i), and
 *   bq_mat[mate][cycle][min(qual, 93)] += 1   u64[2][max_bp][94]
 *   len_hist[l_seq] += 1                      u64[max_bp + 1]
 *   tlen[|TLEN|] += 1 for (flag & 0xC1) == 0x41 and |TLEN| < max_tlen      u64[max_tlen]
 * counts[12]: records, considered, counted, skipped for flag / mapq / empty SEQ / missing QUAL / length,
 * inflated bytes, compressed bytes, EOF member present (1 / 0), chunks.  times[6] ms: reading the file,
 * inflating (wall), walking the record chain, host-to-device copies, kernels (CUDA events), the whole call.  thread_ms[threads]
 * (may be NULL): busy time of each inflate thread.  Malformed input is MG_EVALUE with bad_code (1 not gzip,
 * 2 no BC subfield, 3 corrupt or truncated member, 4 CRC32, 5 ISIZE, 6 not a BAM header, 7 file ends in the
 * header, 10 read error: bad_where = compressed offset of the member; 8 block_size < 32, 9 file ends inside
 * the record, 11 / 12 / 13 / 14 read name / CIGAR / SEQ / QUAL overrun block_size: bad_where = record
 * ordinal); the first bad record in file order is reported, and no chunk after the one holding it is read.
 * 1 <= max_bp <= 50000, 1 <= max_tlen <= 2^20 and 1 <= every <= 2^32 - 1 (MG_EINVAL otherwise).
 * mg_bam_scan: the same reader without a device: stats[4] = records, inflated bytes, compressed bytes, EOF
 * member present; record errors 11-14 are not checked.                                            */
int mg_readmodel_bam(mg_ctx *ctx, const char *path, int32_t max_bp, int32_t max_tlen, int32_t min_mq, int64_t every, int32_t threads,
                     int64_t chunk_bytes, uint64_t *bq_mat, uint64_t *len_hist, uint64_t *tlen, int64_t *counts, double *times,
                     double *thread_ms, int64_t *bad_where, int32_t *bad_code);
int mg_bam_scan(const char *path, int32_t threads, int64_t chunk_bytes, int64_t *stats, int64_t *bad_where, int32_t *bad_code);

/* ---- alignment-analysis: replaces mitty/benchmarking/mq.py and derr.py -- an aligner's BAM (file or FIFO, any
 * sort order, no index) scored against the truth in Mitty's qnames, read and inflated as mg_readmodel_bam does.
 * Every record in file order (C = 2 * max_d + 3 columns: d_err -max_d .. max_d, then wrong_chrom = C - 2,
 * unmapped = C - 1):
 *   flag & 0x900 (secondary, supplementary): skipped, nothing else.  QC-fail and duplicates are analysed.
 *   read index i = 1 iff (flag & 0xC1) == 0x81, else 0; its qname fields (the name up to its NUL, split at '|')
 *   are 3 + 5 * i .. + 4: strand, pos, rlen, CIGAR, v_list; field 1 is the chrom.
 *   column: unmapped if flag & 0x4 or refID == -1; else wrong_chrom if the header name of refID differs byte for
 *   byte from the chrom field; else d = start(POS, aligned CIGAR) - start(qname pos - 1, qname CIGAR), where
 *   start(P, C) = P - the lengths of C's leading run of S, H and I ops (P ops skipped; '>p:nI' is nI), clamped
 *   to [-max_d, max_d] at column d + max_d.
 *   mq[MAPQ][column] += 1                                                          u64[256][C]
 *   vsize[clamp(v, -max_size - 1, max_size + 1) + max_size + 1][column] += 1 per v_list entry v, or
 *   vsize[2 * max_size + 3][column] += 1 for an empty v_list                       u64[2 * max_size + 4][C]
 * counts[14]: records, analysed, skipped, unmapped, wrong_chrom, exact (d == 0), clamped (|d| > max_d),
 * strand_mismatch (right chrom, flag & 0x10 differs from the qname strand), no_variant_reads, variant_entries,
 * inflated bytes, compressed bytes, EOF member present, chunks.  times[6] and thread_ms as mg_readmodel_bam.
 * Malformed input is MG_EVALUE with bad_code / bad_where as mg_readmodel_bam (1 .. 14), plus, for an analysed
 * record (bad_where = its ordinal), in this order: 17 refID below -1 or at or above n_ref; 15 a qname that is
 * not Mitty's (fewer than 8 fields; strand not 0 / 1; pos, a v_list entry or the '>p:' offset not a decimal
 * integer; CIGAR not digits + one of MIDNSHP=X per op); 16 no read for this mate (a read-2 record whose qname
 * has fewer than 13 fields).  The first bad record in file order is reported and no chunk after the one
 * holding it is read.  0 <= max_d, max_size <= 10000 (MG_EINVAL otherwise).                          */
int mg_alnerr_bam(mg_ctx *ctx, const char *path, int32_t max_d, int32_t max_size, int32_t threads, int64_t chunk_bytes, uint64_t *mq,
                  uint64_t *vsize, int64_t *counts, double *times, double *thread_ms, int64_t *bad_where, int32_t *bad_code);

/* ---- profiling: device time (CUDA events on the launch stream) of the emit / corrupt kernel
 * (emit_ms over emit_launches launches, emit_bytes written) and of the planning kernel (plan_ms);
 * total_launches counts every kernel this context launched since the last reset.               */
int mg_prof_reset(mg_ctx *ctx);
int mg_prof_get(mg_ctx *ctx, double *emit_ms, int64_t *emit_launches, int64_t *emit_bytes, int64_t *total_launches,
                double *plan_ms);

#ifdef __cplusplus
}
#endif
#endif
