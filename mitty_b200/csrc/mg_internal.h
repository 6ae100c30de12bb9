// Internal interface between the C-ABI host code (mg_api.cu, mg_check.cu, mg_bam.cu, mg_readmodel.cu) and the
// kernels (mg_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <functional>
#include <utility>
#include "mg_core.cuh"

struct mg_ctx;

// accessors implemented in mg_api.cu (the context's internals stay there)
cudaStream_t mg_internal_stream(mg_ctx *ctx);
int mg_internal_device(mg_ctx *ctx);
int mg_internal_fail(mg_ctx *ctx, int code, const char *msg);
int mg_internal_cuda_fail(mg_ctx *ctx, cudaError_t e, const char *call, const char *file, int line);   // -> MG_ECUDA
int mg_internal_copy_view(mg_ctx *ctx, int64_t copy_id, int64_t *region_id, const MgNode **nodes, int *n_nodes, const uint32_t **hap, uint32_t *hap_len,
                          const MgExc **exc, int *n_exc, int64_t *start1);
int mg_internal_region_view(mg_ctx *ctx, int64_t region_id, const uint32_t **ref, int64_t *len, const MgExc **exc, int *n_exc);

// returns MG_ECUDA from the enclosing function when `call` fails; the context's error names the call, the CUDA
// error and file:line
#define MG_CK(ctx, call) do { const cudaError_t e_ = (call); if (e_ != cudaSuccess) return mg_internal_cuda_fail((ctx), e_, #call, __FILE__, __LINE__); } while (0)

struct DeviceGuard {   // makes `dev` current for a scope, then restores the caller's device
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard &) = delete;
  DeviceGuard &operator=(const DeviceGuard &) = delete;
};

struct DevBuf {  // grow-only device buffer; move-only, freed with its owner
  void *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevBuf &operator=(DevBuf &&o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~DevBuf() { if (p) cudaFree(p); }
  // at least `bytes`; the contents are not kept
  cudaError_t need(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // at least `bytes`, keeping the first `keep`; grows by a quarter, since a buffer that grows this way (a
  // god-aligner run) is copied on every growth.  The old block is freed once `st` has drained.
  cudaError_t need_keep(size_t bytes, size_t keep, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    void *q = nullptr;
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) return e;
    if (keep) e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (p) cudaFree(p);
    p = q; cap = want;
    return e;
  }
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct HostBuf {  // grow-only page-locked staging buffer; move-only
  void *p = nullptr;
  size_t cap = 0;
  HostBuf() = default;
  HostBuf(const HostBuf &) = delete;
  HostBuf &operator=(const HostBuf &) = delete;
  HostBuf(HostBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  HostBuf &operator=(HostBuf &&o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~HostBuf() { if (p) cudaFreeHost(p); }
  cudaError_t need(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
    size_t want = bytes + bytes / 4 + 4096;
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// The FASTQ ingest of corrupt-reads, check-reads and god-aligner: one or two FASTQ buffers on the device with
// their newline index.  The caller handles (some of) the n_tpl complete templates and carries the rest of each
// file into its next chunk.
struct MgFastqChunk {
  DevBuf in[2], nl[2], cnt, tmp;     // tmp: the newline scan's; a caller may reuse it for its own scans
  int nf = 0;
  int64_t n_tpl = 0;                 // complete templates present in every file
};
// per file: H2D, k_nl_count, scan, k_nl_write (5 launches); one sync per file to size the index
cudaError_t mg_fastq_load(MgFastqChunk &q, const uint8_t *const in[2], const int64_t len[2], int nf, cudaStream_t st);
// enqueues the D2H of the last byte offset of the first k templates of each file into last[] (the caller syncs)
cudaError_t mg_fastq_ends(const MgFastqChunk &q, int64_t k, int64_t last[2], cudaStream_t st);

// The chunk pipeline of the BAM readers (bam2illumina, alignment-analysis; mg_readmodel.cu).  Every chunk of
// whole records of `rd` goes to the device on a copy stream while the previous one is processed on a kernel
// stream: two slots (chunk buffers on both sides), five events per slot (H2D start / end, kernel start / end,
// first_bad read back).  The caller supplies only its work:
//   begin(ks)         before the first chunk: clear its accumulators;
//   launch(c, data, off, first_bad, ks)   one chunk: c.n records at data + off[i] (record c.first + i of the file);
//                     a malformed record k is reported by atomicMin(first_bad, k << 8 | code);
//   finish(ks)        after the last chunk: copy its accumulators out (ks is synchronised afterwards).
// Each returns MG_OK or an error code.  Once a slot's read-back shows a malformed record, no further chunk is read.
// Fills times[6] (read, inflate, walk, H2D, kernel, whole call since t_start, ms), thread_ms (may be null) and
// *chunks; -> MG_OK, the error of a CUDA call or a callback, or MG_EVALUE with bad_where / bad_code set for
// malformed input (the device's first bad record, else the reader's error).
class MgBamReader;
struct MgBamChunk;
struct MgBamPipe {
  std::function<int(cudaStream_t)> begin, finish;
  std::function<int(const MgBamChunk &, const uint8_t *, const uint32_t *, unsigned long long *, cudaStream_t)> launch;
};
int mg_bam_pipeline(mg_ctx *ctx, MgBamReader &rd, const MgBamPipe &p, double t_start, int64_t *chunks, double *times, double *thread_ms,
                    int64_t *bad_where, int32_t *bad_code);
double mg_now_ms();
void *mg_pinned_alloc(size_t n);       // the reader's chunk buffers: page-locked, for the copies to the device
void mg_pinned_release(void *p);

#define MG_PLAN_TILE 256     // candidates per CTA tile of k_unit_plan
#define MG_CTA 128           // threads per CTA of k_unit_emit (4 independent warps, 32 kept templates each)
#define MG_TLEN_K 1024       // entries of the template-length alias table (outcomes 0..n_tlen)
#define MG_QN_MAX 192        // max length of the qname prefix / mid strings
#define MG_HAP_PAD 8         // 32-bit words of padding on both sides of a packed sequence

enum { MG_MODE_PHILOX = 0, MG_MODE_DET = 1, MG_MODE_EXPLICIT = 2 };

// One kept template as planned by k_unit_plan, stored at its final rank (serial - 1).
struct alignas(16) MgPlan {
  uint32_t xa, xb;     // read starts relative to p_min (mate 0 forward, mate 1 reverse)
  int32_t n0a, n0b;    // first node of each read
  uint32_t dn;         // (n1 - n0) of mate 0 | mate 1 << 16
  uint32_t fo_sz;      // file-order bit << 31 | mate 0 / mate 1 touches an exception run << 30 / 29 | record bytes (with the serial's digits)
  uint64_t off;        // byte offset of the record in each file
};

// One work unit of a BATCH of small units (one CTA of k_batch_plan each, all emitted by one launch).
#define MG_BATCH_MAXC 2048   // candidates per unit: one block's worth of the gap scan
struct MgBatchUnit {
  MgTok pre[4], mid[4];      // "@sample:0:unit:" and "|chrom|copy" as tokens (at most 32 bytes each)
  int n_pre, n_mid;
  uint32_t qn_len;           // bytes of the two strings
  uint32_t seed;             // rng_seed of the unit: every Philox key derives from it as in the one-unit path
  uint32_t x0, hap_len;      // its copy's range of the concatenated haplotype
  uint32_t n_cand, plan_off; // candidates; first plan record of the unit
  int64_t draw_off;          // DET: first entry of the unit in the concatenated ts / u_tlen / fo arrays
  int64_t p_min;             // 1-based sample coordinate of the unit's first haplotype base
};

struct MgUnitParams {
  // haplotype of one chromosome copy, resident in HBM
  const uint32_t *hap;       // 2-bit packed, 16 bases / word, pointer already biased past the front pad
  uint32_t hap_len;          // p_max - p_min
  int64_t p_min;             // 1-based sample coordinate of hap base 0
  const MgNode *nodes; int n_nodes;
  const uint32_t *blk; int blk_shift; int n_blk;
  const MgExc *exc; int n_exc;
  const uint32_t *eblk;      // block table over the exception runs (MgExcView), or null
  // read model
  const double *cum_tlen; int n_tlen; int rlen;
  const uint32_t *tlen_alias; // PHILOX: MG_TLEN_K-entry alias table (prob22 << 10 | alias) or null
  // template sampling
  int mode; uint32_t n_cand;
  const int64_t *ts_in;      // DET / EXPLICIT: shuffled template starts (1-based sample coords)
  const double *u_tlen;      // DET: uniforms for the template-length inverse CDF
  const int64_t *tl_in;      // EXPLICIT: template lengths
  const int8_t *fo_in;       // DET / EXPLICIT: file-order bits, consumed in te<p_max survivor order
  const uint32_t *ts_sorted; // PHILOX: cumulative geometric gaps (+1), relative to p_min
  uint32_t key_tlen0, key_tlen1, key_perm0, key_perm1, perm_bits;
  // qname constants as tokens: "@sample:worker:ps:", "|chrom|cpy", "|<L>|<L>=|" (built on the host, read from
  // the kernel's parameter space)
  MgQnConst qn;
  int qn_len;                // bytes of the two constant strings
  int bulk;                  // copy-out through cp.async.bulk (1) or 128-bit loads / stores (0, experiments)
  // outputs
  uint8_t *out[2]; uint64_t cap;
  MgPlan *plan;              // [n_cand] written by k_unit_plan, read by k_unit_emit
  // fused corruption (PHILOX draws, alias tables)
  int corrupt; MgCorruptCtx cor;
  int L_nd;                  // decimal digits of rlen
  // grid-wide scan state
  unsigned long long *descA, *descB; uint32_t *tile_counter;
  unsigned long long *totals;  // [0] te<p_max survivors, [1] templates written, [2] bytes per file, [3] overflow
  int n_tiles; int stage_cap;
  // a batch of small units: per-unit table, exclusive prefixes of kept templates / bytes per file over the units
  const MgBatchUnit *bunits; int n_bunits;
  const long long *kept_base, *byte_base;
  long long *unit_kept, *unit_bytes, *unit_te;
  double inv_log1mp;         // 1 / log(1 - p), computed on the host as for the one-unit gap scan
};

// the keys of a unit's Philox streams, all derived from its rng_seed: the one-unit path (mg_api.cu) and the
// batch kernels must agree, so that a unit's bytes do not depend on the path it took
struct MgUnitKeys { uint32_t gap0, gap1, tlen0, tlen1, perm0, perm1, perm_bits; };
__host__ __device__ inline MgUnitKeys mg_unit_keys(uint32_t seed, uint32_t n_cand) {
  MgUnitKeys k;
  k.gap0 = seed; k.gap1 = 0x67617031u;
  k.tlen0 = seed; k.tlen1 = 0x746c6531u;
  k.perm0 = seed ^ 0x7368756bu; k.perm1 = seed * 0x9E3779B1u + 0x66656973u;
  k.perm_bits = mg_perm_bits(n_cand);
  return k;
}

struct MgSampleParams {      // template sampling only (the read-module plugin's generate_reads)
  MgUnitParams u;
  int64_t *ts_out; int64_t *te_out; int8_t *fo_out;  // per candidate (uncompacted); te = -1 when dropped
};

struct MgCorruptParams {     // standalone corrupt-reads over FASTQ resident in HBM
  const uint8_t *in[2]; uint8_t *out[2];
  const int64_t *nl[2];      // newline positions of each input file
  const int64_t *out_off[2]; // output record offsets [n_rec + 1]
  int64_t n_rec; int n_files;
  int64_t first;             // index of the first template of this buffer in the whole file (Philox counter)
  const double *cum_bq; int n_cycles, n_bq; const double *phred;
  int mode;                  // MG_MODE_PHILOX / MG_MODE_DET
  MgCorruptCtx cor;          // PHILOX: alias tables + keys
  const double *bq_rnd, *call_rnd; const uint8_t *base_rnd; const int64_t *draw_off;  // DET: per read [2*n_rec+1]
  unsigned long long *err;   // [0] != 0 -> a read is longer than the model; [1] = bytes of the largest output record
};

// launchers (all asynchronous on `st`)
void mg_launch_pack_ref(const uint8_t *raw, int64_t len, uint32_t *packed, uint32_t *exc_cnt, int64_t *exc_start,
                        uint8_t *exc_byte, int64_t *exc_end, uint32_t exc_cap, cudaStream_t st);
// device node-list walk (k_walk_*).  The variants of one or MANY chromosome copies ("segments": one per
// (BED region, copy)), concatenated, each segment sorted by POS.  One launch sequence builds the node
// tables of all segments back to back: node keys / haplotype coordinates run through the concatenation
// (segment s owns [hap_base, hap_base + hap_len)), so a batch of small regions is ONE node table, ONE
// haplotype and ONE block table.
struct MgSeg {                // input, per segment
  int32_t v0, v1;             // its variants: [v0, v1) of the concatenated arrays
  uint32_t roff;              // offset of its region's first base in the (concatenated) packed reference
  uint32_t pad;
  int64_t start1;             // ref_start_pos = bed_start + 1 (readgenerate.py:190); also p_min
  int64_t region_len;
};
struct MgSegOut {             // output, per segment
  uint32_t hap_base, hap_len; // its haplotype: [hap_base, hap_base + hap_len) of the concatenation; p_max - p_min = hap_len
  int32_t i0, last;           // first / last accepted variant (-1: none)
  int32_t ends_in_d;          // a deletion crossed the region end: the reference's list would end in 'D'
  uint32_t node0, n_nodes;    // its nodes: [node0, node0 + n_nodes)
  uint32_t pad;
};
struct MgWalkSummary {
  unsigned long long err;     // (variant index << 8 | code) of the first invalid accepted variant, ~0 if none
  long long n_nodes, hap_len; // nodes written; length of the concatenated haplotype
  int32_t ends_in_d, bad;
};

struct MgWalkParams {
  const int64_t *pos, *oplen, *alt_off; const uint8_t *op;
  int n_var;
  const MgSeg *segs; int n_seg; MgSegOut *seg_out;
  uint32_t *nxt, *jump[2]; uint8_t *mark; int32_t *pred;
  int64_t *packed, *scanned, *scan_tmp;     // n_var + n_seg (+ 1) elements: every segment has a tail element after its variants
  MgNode *nodes; uint32_t *node_alt;        // node_alt: source of the node's bases -- '=': offset in the packed reference; 'X' / 'I': offset in the alt pool
  MgWalkSummary *sum;
};

int mg_launch_walk(const MgWalkParams &W, cudaStream_t st);   // -> number of kernels launched
void mg_launch_exc_count(const MgNode *nodes, const uint32_t *node_alt, const MgWalkSummary *sum, int max_nodes,
                         const uint8_t *alt_pool, const MgExc *rexc, int n_rexc, int64_t *cnt, cudaStream_t st);
void mg_launch_exc_write(const MgNode *nodes, const uint32_t *node_alt, const MgWalkSummary *sum, int max_nodes,
                         const uint8_t *alt_pool, const MgExc *rexc, int n_rexc, int64_t *off, MgExc *out, cudaStream_t st);
void mg_launch_hap_build(const uint32_t *ref, const uint8_t *alt_pool, const MgNode *nodes, const uint32_t *node_alt,
                         int n_nodes, const uint32_t *blk, int blk_shift, int n_blk, uint32_t hap_len, uint32_t *hap, int64_t hap_words,
                         cudaStream_t st);   // after mg_launch_blk_table
void mg_launch_blk_table(const MgNode *nodes, int n_nodes, uint32_t *blk, int n_blk, int blk_shift, cudaStream_t st);
void mg_launch_eblk_table(const MgExc *exc, int n_exc, uint32_t *eblk, int n_entries, int blk_shift, cudaStream_t st);   // n_entries = n_blk + 1
void mg_launch_gap_scan(uint32_t n, double p, uint32_t k0, uint32_t k1, uint32_t *ts_sorted, unsigned long long *partial,
                        cudaStream_t st);
int mg_unit_grid(int L, int corrupt, int stage_cap, int *smem_bytes);
void mg_launch_plan(const MgUnitParams &P, cudaStream_t st);
void mg_launch_unit(const MgUnitParams &P, int grid, int smem_bytes, cudaStream_t st);
void mg_launch_batch_plan(const MgUnitParams &P, cudaStream_t st);      // one CTA per unit of P.bunits
int mg_batch_grid(int L, int corrupt, int stage_cap, int *smem_bytes);
void mg_launch_batch_emit(const MgUnitParams &P, int grid, int smem_bytes, cudaStream_t st);
void mg_launch_sample(const MgSampleParams &P, cudaStream_t st);
void mg_launch_scan_i64(const int64_t *in, int64_t *out, int64_t n, int64_t *tmp, cudaStream_t st);  // exclusive, out[n] = total
int64_t mg_scan_tmp_elems(int64_t n);
void mg_launch_nl_count(const uint8_t *buf, int64_t len, int64_t *cnt, cudaStream_t st);
void mg_launch_nl_write(const uint8_t *buf, int64_t len, const int64_t *off, int64_t *nl, cudaStream_t st);
int64_t mg_nl_chunks(int64_t len);
void mg_launch_corrupt_sizes(const MgCorruptParams &P, int64_t *sz0, int64_t *sz1, cudaStream_t st);
void mg_launch_corrupt(const MgCorruptParams &P, cudaStream_t st);
void mg_launch_corrupt_staged(const MgCorruptParams &P, bool bulk, cudaStream_t st);   // PHILOX mode, every record <= mg_corrupt_stage_cap()
int mg_corrupt_stage_cap(void);
