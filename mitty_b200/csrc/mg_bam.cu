// god-aligner: the perfect alignments of a simulated FASTQ as a coordinate-sorted BAM (Mitty's
// mitty/benchmarking/god_aligner.py), encoded and sorted on the device.
//
// Per FASTQ chunk (both files of a pair in step):
//   ingest    H2D, newline index (mg_fastq_load, shared with corrupt-reads and check-reads)
//   k_bam_size    one thread per read: qname parse (mg_qname.cuh), contig lookup, validation; record size,
//                 sort key (refID, pos, reverse bit), error code
//   scan          record offsets of the chunk
//   k_bam_encode  one thread per read: the BAM record at its offset in the run buffer -- fixed block with
//                 bin = reg2bin(pos, end), name, CIGAR, 4-bit SEQ (strand 1 reverse-complemented while
//                 packing), QUAL, RG tag
// Per run (as many whole templates as fit run_bytes):
//   k_radix_hist / scan / k_radix_scatter   stable LSD radix sort of (key, ordinal), 8 bits a pass over the
//                 key's significant bits only
//   k_gather_sizes / scan / k_gather_copy   the records in sorted order, one warp per record
// One run goes D2H in pieces straight into the BGZF writer; with several, every run is spilled (keys +
// records) to a temporary file next to the BAM and the runs are merged on the host by key, ties in run
// order, which keeps the global sort stable.
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <queue>
#include <string>
#include <vector>

#include "../../include/mitty_b200.h"
#include "mg_bgzf.h"
#include "mg_internal.h"
#include "mg_qname.cuh"

namespace {

enum { BAM_OK = 0, BAM_FRAME = 1, BAM_QNAME = 2, BAM_CHROM = 3, BAM_NAME = 4, BAM_LEN = 5, BAM_CIGAR = 6, BAM_RANGE = 7 };

struct BamParams {
  const uint8_t *fq[2]; const int64_t *nl[2]; int64_t n_reads; int nf;
  const uint8_t *names; const int32_t *name_off; const int64_t *ref_len; int n_ref;
  int pos_bits;
  const uint8_t *rg; int rg_len;                     // the RG tag's value (the sample)
  // size pass
  int64_t *size; uint64_t *key; uint8_t *code; unsigned long long *first_bad;
  // encode pass: record j goes to rec + run_rec + off[j]; its key / size / offset to the run's arrays at run_n + j
  const int64_t *off; int64_t run_rec, run_n; uint8_t *rec;
  uint64_t *run_key; int64_t *run_size, *run_off;
};

struct BamRead {
  int64_t h0, h1, s0, L, ca, cb;
  int64_t pos, mpos, span, mspan;      // 0-based; reference span of the CIGAR
  int strand, mstrand, ref, n_ops;
};

__device__ __forceinline__ int cig_code(uint8_t op) { return op == '=' ? 7 : op == 'X' ? 8 : op == 'I' ? 1 : op == 'D' ? 2 : -1; }

__device__ __forceinline__ void st32(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }

// walks a qname CIGAR ('>p:nI' is one op nI); with out != null writes the packed ops there
__device__ bool cigar_walk(const uint8_t *q, int64_t ca, int64_t cb, int &n_ops, int64_t &qlen, int64_t &span, uint8_t *out) {
  n_ops = 0; qlen = 0; span = 0;
  if (ca >= cb) return false;
  if (q[ca] == '>') {
    int64_t colon = ca + 1;
    while (colon < cb && q[colon] != ':') colon++;
    int64_t off, n;
    if (colon >= cb || q[cb - 1] != 'I' || !mg_parse_int(q, ca + 1, colon, off) || !mg_parse_int(q, colon + 1, cb - 1, n) || off < 0 || n < 0) return false;
    n_ops = 1; qlen = n;
    if (out) st32(out, (uint32_t)n << 4 | 1u);
    return true;
  }
  while (ca < cb) {
    int64_t e = ca;
    while (e < cb && q[e] >= '0' && q[e] <= '9') e++;
    int64_t c;
    if (e == ca || e >= cb || !mg_parse_int(q, ca, e, c) || c >= (1 << 28)) return false;
    const int code = cig_code(q[e]);
    if (code < 0 || n_ops == 65535) return false;
    if (out) st32(out + 4 * n_ops, (uint32_t)c << 4 | (uint32_t)code);
    n_ops++;
    if (code != 2) qlen += c;
    if (code != 1) span += c;
    ca = e + 1;
  }
  return true;
}

__device__ int bam_parse(const BamParams &P, int64_t j, BamRead &R) {
  const int f = (int)(j % P.nf);
  const int64_t t = j / P.nf;
  const uint8_t *q = P.fq[f];
  const int64_t *nl = P.nl[f];
  R.h0 = t == 0 ? 0 : nl[4 * t - 1] + 1; R.h1 = nl[4 * t]; R.s0 = R.h1 + 1;
  const int64_t s1 = nl[4 * t + 1];
  if (R.h1 <= R.h0 || q[R.h0] != '@' || nl[4 * t + 2] != s1 + 2 || q[s1 + 1] != '+' || nl[4 * t + 3] - nl[4 * t + 2] != s1 - R.s0 + 1) return BAM_FRAME;
  if (R.h1 - R.h0 - 1 > 254) return BAM_NAME;
  int64_t fs[MG_QN_FIELDS], fe[MG_QN_FIELDS];
  const int nfld = mg_qname_split(q, R.h0 + 1, R.h1, fs, fe);
  const int base = 3 + 5 * f, mbase = 3 + 5 * (1 - f);
  if (nfld < (P.nf == 2 ? 13 : base + 5)) return BAM_QNAME;
  int64_t strand, pos, rlen;
  if (!mg_parse_int(q, fs[base], fe[base], strand) || !mg_parse_int(q, fs[base + 1], fe[base + 1], pos) ||
      !mg_parse_int(q, fs[base + 2], fe[base + 2], rlen) || (strand != 0 && strand != 1)) return BAM_QNAME;
  R.strand = (int)strand; R.pos = pos - 1;
  // contig lookup: the chrom field among the FASTA's names
  const int64_t cl = fe[1] - fs[1];
  R.ref = -1;
  for (int k = 0; k < P.n_ref && R.ref < 0; k++) {
    const int a = P.name_off[k];
    if (P.name_off[k + 1] - a != cl) continue;
    bool same = true;
    for (int64_t i = 0; i < cl && same; i++) same = P.names[a + i] == q[fs[1] + i];
    if (same) R.ref = k;
  }
  if (R.ref < 0) return BAM_CHROM;
  R.ca = fs[base + 3]; R.cb = fe[base + 3];
  int64_t qlen;
  if (!cigar_walk(q, R.ca, R.cb, R.n_ops, qlen, R.span, nullptr)) return BAM_CIGAR;
  R.L = s1 - R.s0;
  if (R.L != rlen || qlen != rlen) return BAM_LEN;
  if (R.pos < 0 || R.pos + R.span > P.ref_len[R.ref]) return BAM_RANGE;
  R.mstrand = 0; R.mpos = -1; R.mspan = 0;
  if (P.nf == 2) {
    int64_t ms, mp; int mops; int64_t mq;
    if (!mg_parse_int(q, fs[mbase], fe[mbase], ms) || !mg_parse_int(q, fs[mbase + 1], fe[mbase + 1], mp) || (ms != 0 && ms != 1)) return BAM_QNAME;
    if (!cigar_walk(q, fs[mbase + 3], fe[mbase + 3], mops, mq, R.mspan, nullptr)) return BAM_CIGAR;
    R.mstrand = (int)ms; R.mpos = mp - 1;
  }
  return BAM_OK;
}

__device__ __forceinline__ int64_t bam_size(const BamParams &P, const BamRead &R) {
  return 36 + (R.h1 - R.h0) + 4 * R.n_ops + (R.L + 1) / 2 + R.L + 4 + P.rg_len;
}

__device__ __forceinline__ uint64_t bam_key(const BamParams &P, const BamRead &R) {
  return (uint64_t)R.ref << (P.pos_bits + 1) | (uint64_t)R.pos << 1 | (uint64_t)R.strand;
}

__global__ void __launch_bounds__(256) k_bam_size(BamParams P) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= P.n_reads) return;
  BamRead R;
  const int code = bam_parse(P, j, R);
  P.code[j] = (uint8_t)code;
  if (code) { atomicMin(P.first_bad, (unsigned long long)j); P.size[j] = 0; P.key[j] = 0; return; }
  P.size[j] = bam_size(P, R);
  P.key[j] = bam_key(P, R);
}

__device__ __forceinline__ uint32_t nt16(uint32_t c) {       // htslib's seq_nt16_table: "=ACMGRSVTWYHKDBN", any case
  switch (c | 0x20) {
    case 'a': return 1; case 'c': return 2; case 'm': return 3; case 'g': return 4; case 'r': return 5; case 's': return 6;
    case 'v': return 7; case 't': return 8; case 'w': return 9; case 'y': return 10; case 'h': return 11; case 'k': return 12;
    case 'd': return 13; case 'b': return 14;
    default: return c == '=' ? 0 : 15;
  }
}
__device__ __forceinline__ uint32_t nt16_comp(uint32_t x) { return (x & 1) << 3 | (x & 2) << 1 | (x & 4) >> 1 | (x & 8) >> 3; }

// SAM spec §5.3
__device__ __forceinline__ uint32_t reg2bin(int64_t beg, int64_t end) {
  --end;
  if (beg >> 14 == end >> 14) return (uint32_t)(((1 << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (uint32_t)(((1 << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (uint32_t)(((1 << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (uint32_t)(((1 << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (uint32_t)(((1 << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

__global__ void __launch_bounds__(256) k_bam_encode(BamParams P) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= P.n_reads) return;
  BamRead R;
  bam_parse(P, j, R);                                  // valid: the size pass said so
  const int f = (int)(j % P.nf);
  const uint8_t *q = P.fq[f];
  const int64_t sz = bam_size(P, R), at = P.run_rec + P.off[j];
  uint8_t *o = P.rec + at;
  const int64_t end = R.pos + (R.span > 0 ? R.span : 1);
  uint32_t flag = R.strand ? 0x10 : 0;
  int32_t tlen = 0;
  if (P.nf == 2) {
    flag |= 0x1 | 0x2 | (f ? 0x80 : 0x40) | (R.mstrand ? 0x20 : 0);
    const int64_t mend = R.mpos + (R.mspan > 0 ? R.mspan : 1);
    const int64_t lo = R.pos < R.mpos ? R.pos : R.mpos, hi = end > mend ? end : mend;
    const bool left = R.pos < R.mpos || (R.pos == R.mpos && f == 0);
    tlen = (int32_t)(left ? hi - lo : lo - hi);
  }
  const int l_name = (int)(R.h1 - R.h0);              // name + NUL
  st32(o, (uint32_t)(sz - 4));
  st32(o + 4, (uint32_t)R.ref);
  st32(o + 8, (uint32_t)R.pos);
  st32(o + 12, reg2bin(R.pos, end) << 16 | 60u << 8 | (uint32_t)l_name);
  st32(o + 16, flag << 16 | (uint32_t)R.n_ops);
  st32(o + 20, (uint32_t)R.L);
  st32(o + 24, P.nf == 2 ? (uint32_t)R.ref : 0xFFFFFFFFu);
  st32(o + 28, P.nf == 2 ? (uint32_t)R.mpos : 0xFFFFFFFFu);
  st32(o + 32, (uint32_t)tlen);
  uint8_t *p = o + 36;
  for (int i = 0; i < l_name - 1; i++) p[i] = q[R.h0 + 1 + i];
  p[l_name - 1] = 0;
  p += l_name;
  int n_ops; int64_t ql, sp;
  cigar_walk(q, R.ca, R.cb, n_ops, ql, sp, p);
  p += 4 * n_ops;
  const int64_t L = R.L, s0 = R.s0, q0 = R.s0 + L + 3;   // quality line: after "\n+\n"
  for (int64_t i = 0; i < L; i += 2) {
    uint32_t a, b = 0;
    if (R.strand) {
      a = nt16_comp(nt16(q[s0 + L - 1 - i]));
      if (i + 1 < L) b = nt16_comp(nt16(q[s0 + L - 2 - i]));
    } else {
      a = nt16(q[s0 + i]);
      if (i + 1 < L) b = nt16(q[s0 + i + 1]);
    }
    p[i >> 1] = (uint8_t)(a << 4 | b);
  }
  p += (L + 1) / 2;
  for (int64_t i = 0; i < L; i++) p[i] = (uint8_t)(q[R.strand ? q0 + L - 1 - i : q0 + i] - 33);
  p += L;
  p[0] = 'R'; p[1] = 'G'; p[2] = 'Z';
  for (int i = 0; i < P.rg_len; i++) p[3 + i] = P.rg[i];
  p[3 + P.rg_len] = 0;
  P.run_key[P.run_n + j] = bam_key(P, R);
  P.run_size[P.run_n + j] = sz;
  P.run_off[P.run_n + j] = at;
}

// ---- stable LSD radix sort of (key, ordinal) --------------------------------------------------------

#define RS_THREADS 256
#define RS_ITEMS 16
#define RS_TILE (RS_THREADS * RS_ITEMS)
#define RS_WARPS (RS_THREADS / 32)

__global__ void __launch_bounds__(RS_THREADS) k_radix_hist(const uint64_t *__restrict__ key, int64_t n, int shift, int64_t *__restrict__ hist, int nb) {
  __shared__ unsigned int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * RS_TILE;
  for (int r = 0; r < RS_ITEMS; r++) {
    const int64_t i = base + r * RS_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&h[(key[i] >> shift) & 255], 1u);
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];     // digit-major: the scan gives every (digit, tile) its first slot
}

// a tile in RS_ITEMS rounds of RS_THREADS keys, in index order: rank = tile's slot for the digit + keys of
// that digit in earlier rounds + in earlier warps of this round + in earlier lanes of this warp
__global__ void __launch_bounds__(RS_THREADS) k_radix_scatter(const uint64_t *__restrict__ kin, const uint32_t *__restrict__ oin, uint64_t *__restrict__ kout,
                                                             uint32_t *__restrict__ oout, int64_t n, int shift, const int64_t *__restrict__ hoff, int nb) {
  __shared__ unsigned int wcnt[RS_WARPS][256];
  __shared__ int64_t run[256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  run[threadIdx.x] = hoff[(int64_t)threadIdx.x * nb + blockIdx.x];
  const int64_t base = (int64_t)blockIdx.x * RS_TILE;
  for (int r = 0; r < RS_ITEMS; r++) {
    for (int w = 0; w < RS_WARPS; w++) wcnt[w][threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = base + r * RS_THREADS + threadIdx.x;
    const bool ok = i < n;
    const uint64_t k = ok ? kin[i] : 0;
    const uint32_t o = ok ? oin[i] : 0;
    const unsigned d = ok ? (unsigned)(k >> shift) & 255u : 256u;
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, d);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (ok && rank == 0) wcnt[warp][d] = __popc(peers);
    __syncthreads();
    unsigned tot = 0;
    for (int w = 0; w < RS_WARPS; w++) { const unsigned c = wcnt[w][threadIdx.x]; wcnt[w][threadIdx.x] = tot; tot += c; }
    __syncthreads();
    if (ok) {
      const int64_t at = run[d] + wcnt[warp][d] + rank;
      kout[at] = k; oout[at] = o;
    }
    __syncthreads();
    run[threadIdx.x] += tot;
  }
}

__global__ void __launch_bounds__(256) k_iota(uint32_t *o, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = (uint32_t)i;
}

// ---- gather: the records in sorted order -----------------------------------------------------------

__global__ void __launch_bounds__(256) k_gather_sizes(const uint32_t *__restrict__ ord, const int64_t *__restrict__ size, int64_t *__restrict__ ssize, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ssize[i] = size[ord[i]];
}

__global__ void __launch_bounds__(256) k_gather_copy(const uint32_t *__restrict__ ord, const int64_t *__restrict__ roff, const int64_t *__restrict__ soff,
                                                     const uint8_t *__restrict__ rec, uint8_t *__restrict__ out, int64_t n) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n) return;
  const uint8_t *src = rec + roff[ord[w]];
  uint8_t *dst = out + soff[w];
  const int64_t len = soff[w + 1] - soff[w];
  int64_t i = 0;
  if ((((uintptr_t)src ^ (uintptr_t)dst) & 15) == 0) {     // same alignment: 16-byte bulk between a byte head and tail
    const int64_t a = (int64_t)((16 - ((uintptr_t)dst & 15)) & 15), head = a < len ? a : len;
    if (lane < head) dst[lane] = src[lane];
    const int64_t n16 = (len - head) >> 4;
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src + head);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst + head);
    for (int64_t k = lane; k < n16; k += 32) d4[k] = s4[k];
    i = head + (n16 << 4);
  }
  for (int64_t k = i + lane; k < len; k += 32) dst[k] = src[k];
}

// ---- host side ---------------------------------------------------------------------------------------

bool write_all(int fd, const void *p, size_t n) {
  const uint8_t *b = static_cast<const uint8_t *>(p);
  while (n > 0) {
    const ssize_t w = write(fd, b, n);
    if (w < 0) { if (errno == EINTR) continue; return false; }
    b += w; n -= (size_t)w;
  }
  return true;
}

bool read_at(int fd, void *p, size_t n, int64_t off) {
  uint8_t *b = static_cast<uint8_t *>(p);
  while (n > 0) {
    const ssize_t r = pread(fd, b, n, (off_t)off);
    if (r <= 0) { if (r < 0 && errno == EINTR) continue; return false; }
    b += r; n -= (size_t)r; off += r;
  }
  return true;
}

const int64_t kPiece = 64ll << 20;       // D2H piece through a page-locked buffer
const int64_t kPerRead = 72;             // device bytes per read of a run besides its record: keys, ordinals, sizes, offsets (both sort buffers)

// one spilled run, read back in order: keys and records through their own buffers
struct RunReader {
  int fd = -1; int64_t n = 0, i = 0, key_at = 0, rec_at = 0, rec_end = 0;
  std::vector<uint64_t> kb; int64_t kb0 = 0, kbn = 0;
  std::vector<uint8_t> rb; int64_t rb0 = 0, rbn = 0;     // rb holds file bytes [rb0, rb0 + rbn)
  bool key(uint64_t &k) {
    if (i >= kb0 + kbn) {
      kb0 = i; kbn = std::min<int64_t>(n - i, (int64_t)kb.size());
      if (!read_at(fd, kb.data(), (size_t)kbn * 8, key_at + 8 * kb0)) return false;
    }
    k = kb[(size_t)(i - kb0)];
    return true;
  }
  // the next record; valid until the next call
  const uint8_t *record(int64_t &sz) {
    auto have = [&](int64_t a, int64_t m) {
      if (a >= rb0 && a + m <= rb0 + rbn) return true;
      if ((int64_t)rb.size() < m) rb.resize((size_t)m);
      rb0 = a; rbn = std::min<int64_t>((int64_t)rb.size(), rec_end - a);
      return rbn >= m && read_at(fd, rb.data(), (size_t)rbn, a);
    };
    if (!have(rec_at, 4)) return nullptr;
    uint32_t bs; memcpy(&bs, rb.data() + (rec_at - rb0), 4);
    sz = 4 + (int64_t)bs;
    if (!have(rec_at, sz)) return nullptr;
    const uint8_t *p = rb.data() + (rec_at - rb0);
    rec_at += sz; i++;
    return p;
  }
};

struct Bam {
  mg_ctx *ctx = nullptr;
  std::string bam, bai;
  int n_ref = 0, pos_bits = 0, key_bits = 0, level = 6, threads = 1;
  int64_t run_bytes = 0;
  std::vector<uint8_t> header;
  std::string rg;
  // contig table, RG value
  DevBuf d_names, d_name_off, d_len, d_rg;
  // chunk
  MgFastqChunk fq;
  DevBuf d_csz, d_ckey, d_coff, d_code, d_bad;
  // run
  DevBuf d_rec, d_key, d_size, d_roff;
  int64_t run_n = 0, run_rec = 0;
  // sort / gather
  DevBuf d_key2, d_ord, d_ord2, d_hist, d_hoff, d_stmp, d_ssize, d_soff, d_out;
  HostBuf pin[2];
  cudaEvent_t ev0[2] = {}, ev1[2] = {};
  std::vector<std::string> spills;
  int64_t n_runs = 0;
  double t_dev = 0, t_d2h = 0, t_out = 0;     // ms: ingest + encode + sort + gather; device-to-host copies; writing (deflate, spill, merge)
  ~Bam() {
    for (int k = 0; k < 2; k++) { if (ev0[k]) cudaEventDestroy(ev0[k]); if (ev1[k]) cudaEventDestroy(ev1[k]); }
    for (const std::string &s : spills) unlink(s.c_str());
  }
};

double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

int bam_fail(Bam &b, int code, const std::string &msg) { return mg_internal_fail(b.ctx, code, msg.c_str()); }

// sorts and gathers the current run into d_out (records in key order, d_key2 <- keys in key order)
int sort_run(Bam &b) {
  cudaStream_t st = mg_internal_stream(b.ctx);
  const int64_t n = b.run_n;
  const int nb = (int)((n + RS_TILE - 1) / RS_TILE);
  MG_CK(b.ctx, b.d_key2.need(8 * (size_t)n + 8));
  MG_CK(b.ctx, b.d_ord.need(4 * (size_t)n + 4));
  MG_CK(b.ctx, b.d_ord2.need(4 * (size_t)n + 4));
  MG_CK(b.ctx, b.d_hist.need(8 * (size_t)nb * 256 + 8));
  MG_CK(b.ctx, b.d_hoff.need(8 * ((size_t)nb * 256 + 1)));
  MG_CK(b.ctx, b.d_stmp.need(8 * (size_t)mg_scan_tmp_elems(std::max<int64_t>({(int64_t)nb * 256, n, 1}))));
  MG_CK(b.ctx, b.d_ssize.need(8 * (size_t)n + 8));
  MG_CK(b.ctx, b.d_soff.need(8 * ((size_t)n + 1)));
  MG_CK(b.ctx, b.d_out.need((size_t)b.run_rec + 16));
  const unsigned g = (unsigned)((n + 255) / 256);
  uint64_t *k[2] = {b.d_key.as<uint64_t>(), b.d_key2.as<uint64_t>()};
  uint32_t *o[2] = {b.d_ord.as<uint32_t>(), b.d_ord2.as<uint32_t>()};
  k_iota<<<g, 256, 0, st>>>(o[0], n);
  const int passes = std::max(1, (b.key_bits + 7) / 8);
  int s = 0;
  for (int p = 0; p < passes; p++, s ^= 1) {
    k_radix_hist<<<nb, RS_THREADS, 0, st>>>(k[s], n, 8 * p, b.d_hist.as<int64_t>(), nb);
    mg_launch_scan_i64(b.d_hist.as<int64_t>(), b.d_hoff.as<int64_t>(), (int64_t)nb * 256, b.d_stmp.as<int64_t>(), st);
    k_radix_scatter<<<nb, RS_THREADS, 0, st>>>(k[s], o[s], k[s ^ 1], o[s ^ 1], n, 8 * p, b.d_hoff.as<int64_t>(), nb);
  }
  if (s == 0) {   // keep the sorted keys in d_key2 and the ordinals in d_ord2
    MG_CK(b.ctx, cudaMemcpyAsync(b.d_key2.p, b.d_key.p, 8 * (size_t)n, cudaMemcpyDeviceToDevice, st));
    MG_CK(b.ctx, cudaMemcpyAsync(b.d_ord2.p, b.d_ord.p, 4 * (size_t)n, cudaMemcpyDeviceToDevice, st));
  }
  const uint32_t *ord = b.d_ord2.as<const uint32_t>();
  k_gather_sizes<<<g, 256, 0, st>>>(ord, b.d_size.as<int64_t>(), b.d_ssize.as<int64_t>(), n);
  mg_launch_scan_i64(b.d_ssize.as<int64_t>(), b.d_soff.as<int64_t>(), n, b.d_stmp.as<int64_t>(), st);
  k_gather_copy<<<(unsigned)((32 * n + 255) / 256), 256, 0, st>>>(ord, b.d_roff.as<int64_t>(), b.d_soff.as<int64_t>(), b.d_rec.as<uint8_t>(),
                                                                  b.d_out.as<uint8_t>(), n);
  MG_CK(b.ctx, cudaGetLastError());
  MG_CK(b.ctx, cudaStreamSynchronize(st));
  return MG_OK;
}

// d_out[0, bytes) to the host in pieces; sink(ptr, n) consumes piece k while piece k + 1 is copied
template <class F>
int stream_out(Bam &b, const uint8_t *src, int64_t bytes, F sink) {
  cudaStream_t st = mg_internal_stream(b.ctx);
  int64_t prev = -1; int k = 0;
  for (int64_t off = 0; off < bytes || prev >= 0; off += kPiece, k ^= 1) {
    const int64_t m = std::min(kPiece, bytes - off);
    if (m > 0) {
      MG_CK(b.ctx, cudaEventRecord(b.ev0[k], st));
      MG_CK(b.ctx, cudaMemcpyAsync(b.pin[k].p, src + off, (size_t)m, cudaMemcpyDeviceToHost, st));
      MG_CK(b.ctx, cudaEventRecord(b.ev1[k], st));
    }
    if (prev >= 0) {
      MG_CK(b.ctx, cudaEventSynchronize(b.ev1[k ^ 1]));
      float ms = 0; cudaEventElapsedTime(&ms, b.ev0[k ^ 1], b.ev1[k ^ 1]); b.t_d2h += ms;
      const double t = now_ms();
      if (!sink(b.pin[k ^ 1].as<const uint8_t>(), prev)) return MG_EVALUE;
      b.t_out += now_ms() - t;
    }
    prev = m > 0 ? m : -1;
  }
  return MG_OK;
}

// the current run, sorted, to a temporary file next to the BAM: [n, record bytes], keys, records
int spill_run(Bam &b) {
  double t = now_ms();
  int rc = sort_run(b);
  if (rc) return rc;
  b.t_dev += now_ms() - t;
  std::string path = b.bam + ".run" + std::to_string(b.spills.size()) + ".XXXXXX";
  std::vector<char> tmpl(path.begin(), path.end()); tmpl.push_back(0);
  const int fd = mkstemp(tmpl.data());
  if (fd < 0) return bam_fail(b, MG_EVALUE, "cannot create a temporary run file next to " + b.bam);
  b.spills.push_back(tmpl.data());
  const int64_t hdr[2] = {b.run_n, b.run_rec};
  bool ok = write_all(fd, hdr, sizeof hdr);
  rc = MG_OK;
  if (ok) rc = stream_out(b, b.d_key2.as<const uint8_t>(), 8 * b.run_n, [&](const uint8_t *p, int64_t n) { return write_all(fd, p, (size_t)n); });
  if (ok && !rc) rc = stream_out(b, b.d_out.as<const uint8_t>(), b.run_rec, [&](const uint8_t *p, int64_t n) { return write_all(fd, p, (size_t)n); });
  ok = close(fd) == 0 && ok;
  if (!ok || rc) return bam_fail(b, MG_EVALUE, "cannot write the temporary run file " + b.spills.back());
  b.n_runs++;
  b.run_n = 0; b.run_rec = 0;
  return MG_OK;
}

int merge_runs(Bam &b, MgBamWriter &w) {
  std::vector<RunReader> rr(b.spills.size());
  for (size_t r = 0; r < rr.size(); r++) {
    RunReader &R = rr[r];
    R.fd = open(b.spills[r].c_str(), O_RDONLY);
    int64_t hdr[2];
    if (R.fd < 0 || !read_at(R.fd, hdr, sizeof hdr, 0)) return bam_fail(b, MG_EVALUE, "cannot read the temporary run file " + b.spills[r]);
    R.n = hdr[0]; R.key_at = 16; R.rec_at = 16 + 8 * hdr[0]; R.rec_end = R.rec_at + hdr[1];
    R.kb.resize(1 << 16); R.rb.resize(4 << 20);
  }
  typedef std::pair<uint64_t, int> Head;              // (key, run): ties go to the earlier run
  std::priority_queue<Head, std::vector<Head>, std::greater<Head>> heap;
  int rc = MG_OK;
  for (size_t r = 0; r < rr.size() && !rc; r++) {
    uint64_t k;
    if (rr[r].n == 0) continue;
    if (!rr[r].key(k)) rc = MG_EVALUE; else heap.push({k, (int)r});
  }
  while (!heap.empty() && !rc) {
    const int r = heap.top().second; heap.pop();
    int64_t sz = 0;
    const uint8_t *p = rr[(size_t)r].record(sz);
    if (!p || !w.records(p, sz)) { rc = MG_EVALUE; break; }
    uint64_t k;
    if (rr[(size_t)r].i < rr[(size_t)r].n) { if (!rr[(size_t)r].key(k)) rc = MG_EVALUE; else heap.push({k, r}); }
  }
  for (RunReader &R : rr) if (R.fd >= 0) close(R.fd);
  return rc ? bam_fail(b, MG_EVALUE, "merging the sorted runs failed: " + w.err) : MG_OK;
}

int bit_length(uint64_t x) { int n = 0; while (x) { n++; x >>= 1; } return n; }

}  // namespace

extern "C" {

struct mg_bam { Bam b; };

static void bam_delete(mg_bam *h) {       // once the stream is idle; the temporary run files go with it
  DeviceGuard g(mg_internal_device(h->b.ctx));
  cudaStreamSynchronize(mg_internal_stream(h->b.ctx));
  delete h;
}

int mg_bam_open(mg_ctx *ctx, const char *bam_path, const char *bai_path, int32_t n_ref, const char *const *ref_names, const int64_t *ref_len,
                const char *header_text, const char *sample, int32_t level, int32_t threads, int64_t run_bytes, mg_bam **out) {
  if (!ctx || !bam_path || n_ref <= 0 || !ref_names || !ref_len || !header_text || !sample || level < 0 || level > 9 || !out) return MG_EINVAL;
  std::vector<std::string> names; std::vector<int64_t> lens;
  std::vector<uint8_t> pool; std::vector<int32_t> noff(1, 0);
  int64_t max_len = 1;
  for (int i = 0; i < n_ref; i++) {
    names.push_back(ref_names[i]); lens.push_back(ref_len[i]);
    pool.insert(pool.end(), names.back().begin(), names.back().end()); noff.push_back((int32_t)pool.size());
    max_len = std::max(max_len, ref_len[i]);
  }
  // with every contig below 2^31, pos + span <= ref_len bounds POS, PNEXT and TLEN to int32
  const std::string bad = mg_bam_check_contigs(names, lens);
  if (!bad.empty()) return mg_internal_fail(ctx, MG_EVALUE, ("mg_bam_open: " + bad).c_str());
  DeviceGuard g(mg_internal_device(ctx));
  mg_bam *h = new mg_bam();
  Bam &b = h->b;
  b.ctx = ctx; b.bam = bam_path; b.bai = bai_path ? bai_path : ""; b.n_ref = n_ref; b.level = level; b.threads = std::max(1, (int)threads);
  b.rg = sample;
  b.header = mg_bam_header(header_text, names, lens);
  b.pos_bits = bit_length((uint64_t)max_len);
  b.key_bits = bit_length((uint64_t)(n_ref - 1)) + b.pos_bits + 1;
  if (run_bytes <= 0) {
    size_t fr = 0, tot = 0;
    cudaMemGetInfo(&fr, &tot);
    run_bytes = (int64_t)(fr / 10 * 6);
  }
  b.run_bytes = run_bytes;
  cudaStream_t st = mg_internal_stream(ctx);
  int rc = MG_OK;
  pool.push_back(0);
  auto up = [&](DevBuf &d, const void *src, size_t n) {
    if (d.need(std::max<size_t>(n, 8)) != cudaSuccess || cudaMemcpyAsync(d.p, src, n, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = MG_ECUDA;
  };
  up(b.d_names, pool.data(), pool.size());
  up(b.d_name_off, noff.data(), 4 * noff.size());
  up(b.d_len, lens.data(), 8 * lens.size());
  up(b.d_rg, b.rg.data(), b.rg.size() + 1);
  for (int k = 0; k < 2 && !rc; k++) {
    if (b.pin[k].need((size_t)kPiece) != cudaSuccess) rc = MG_ECUDA;
    cudaEventCreate(&b.ev0[k]); cudaEventCreate(&b.ev1[k]);
  }
  if (!rc && cudaStreamSynchronize(st) != cudaSuccess) rc = MG_ECUDA;
  if (rc) { bam_delete(h); return mg_internal_fail(ctx, MG_ECUDA, "mg_bam_open: out of device or page-locked memory"); }
  *out = h;
  return MG_OK;
}

int mg_bam_add(mg_bam *h, const uint8_t *in1, int64_t len1, const uint8_t *in2, int64_t len2, int64_t *n_templates, int64_t *consumed1,
               int64_t *consumed2, int64_t *bad_index, int32_t *bad_code) {
  if (!h || !in1 || len1 < 0 || (in2 && len2 < 0)) return MG_EINVAL;
  Bam &b = h->b;
  DeviceGuard g(mg_internal_device(b.ctx));
  cudaStream_t st = mg_internal_stream(b.ctx);
  const double t0 = now_ms();
  if (n_templates) *n_templates = 0;
  if (consumed1) *consumed1 = 0;
  if (consumed2) *consumed2 = 0;
  if (bad_index) *bad_index = -1;
  if (bad_code) *bad_code = 0;
  const int nf = in2 ? 2 : 1;
  const uint8_t *in[2] = {in1, in2}; const int64_t len[2] = {len1, len2};
  MG_CK(b.ctx, mg_fastq_load(b.fq, in, len, nf, st));
  const int64_t n_tpl = b.fq.n_tpl;
  if (n_tpl == 0) return MG_OK;
  const int64_t n = n_tpl * nf;
  BamParams P; memset(&P, 0, sizeof P);
  for (int f = 0; f < nf; f++) { P.fq[f] = b.fq.in[f].as<uint8_t>(); P.nl[f] = b.fq.nl[f].as<int64_t>(); }
  P.n_reads = n; P.nf = nf;
  P.names = b.d_names.as<uint8_t>(); P.name_off = b.d_name_off.as<int32_t>(); P.ref_len = b.d_len.as<int64_t>();
  P.n_ref = b.n_ref; P.pos_bits = b.pos_bits;
  P.rg = b.d_rg.as<uint8_t>(); P.rg_len = (int)b.rg.size();
  MG_CK(b.ctx, b.d_csz.need(8 * (size_t)n));
  MG_CK(b.ctx, b.d_ckey.need(8 * (size_t)n));
  MG_CK(b.ctx, b.d_coff.need(8 * ((size_t)n + 1)));
  MG_CK(b.ctx, b.d_code.need((size_t)n));
  MG_CK(b.ctx, b.fq.tmp.need(8 * (size_t)mg_scan_tmp_elems(n)));
  MG_CK(b.ctx, b.d_bad.need(8));
  MG_CK(b.ctx, cudaMemsetAsync(b.d_bad.p, 0xFF, 8, st));
  P.size = b.d_csz.as<int64_t>(); P.key = b.d_ckey.as<uint64_t>(); P.code = b.d_code.as<uint8_t>();
  P.first_bad = b.d_bad.as<unsigned long long>();
  k_bam_size<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P);
  MG_CK(b.ctx, cudaGetLastError());
  mg_launch_scan_i64(P.size, b.d_coff.as<int64_t>(), n, b.fq.tmp.as<int64_t>(), st);
  unsigned long long first_bad = 0; int64_t total = 0;
  MG_CK(b.ctx, cudaMemcpyAsync(&first_bad, b.d_bad.p, 8, cudaMemcpyDeviceToHost, st));
  MG_CK(b.ctx, cudaMemcpyAsync(&total, b.d_coff.as<int64_t>() + n, 8, cudaMemcpyDeviceToHost, st));
  MG_CK(b.ctx, cudaStreamSynchronize(st));
  if (first_bad != ~0ull) {
    uint8_t code = 0;
    MG_CK(b.ctx, cudaMemcpy(&code, b.d_code.as<uint8_t>() + first_bad, 1, cudaMemcpyDeviceToHost));
    if (bad_index) *bad_index = (int64_t)first_bad;
    if (bad_code) *bad_code = code;
    return bam_fail(b, MG_EVALUE, "a FASTQ record cannot be written as a BAM record");
  }
  // as many whole templates as fit the run; a full run is spilled first
  auto fits = [&](int64_t reads, int64_t bytes) { return 2 * (b.run_rec + bytes) + kPerRead * (b.run_n + reads) <= b.run_bytes; };
  int64_t k = n_tpl, bytes = total;
  if (!fits(n, total)) {
    std::vector<int64_t> off((size_t)n + 1);
    MG_CK(b.ctx, cudaMemcpy(off.data(), b.d_coff.p, 8 * off.size(), cudaMemcpyDeviceToHost));
    int64_t lo = 0, hi = n_tpl;              // largest k with fits(k templates)
    while (lo < hi) { const int64_t m = (lo + hi + 1) / 2; if (fits(m * nf, off[(size_t)(m * nf)])) lo = m; else hi = m - 1; }
    if (lo == 0) {
      if (b.run_n == 0) return bam_fail(b, MG_EVALUE, "run_bytes is too small for one template");
      b.t_dev += now_ms() - t0;
      const int rc = spill_run(b);
      if (rc) return rc;
      return mg_bam_add(h, in1, len1, in2, len2, n_templates, consumed1, consumed2, bad_index, bad_code);
    }
    k = lo; bytes = off[(size_t)(k * nf)];
  }
  const int64_t nk = k * nf;
  MG_CK(b.ctx, b.d_rec.need_keep((size_t)(b.run_rec + bytes) + 16, (size_t)b.run_rec, st));
  MG_CK(b.ctx, b.d_key.need_keep(8 * (size_t)(b.run_n + nk), 8 * (size_t)b.run_n, st));
  MG_CK(b.ctx, b.d_size.need_keep(8 * (size_t)(b.run_n + nk), 8 * (size_t)b.run_n, st));
  MG_CK(b.ctx, b.d_roff.need_keep(8 * (size_t)(b.run_n + nk), 8 * (size_t)b.run_n, st));
  P.n_reads = nk;
  P.off = b.d_coff.as<int64_t>(); P.run_rec = b.run_rec; P.run_n = b.run_n; P.rec = b.d_rec.as<uint8_t>();
  P.run_key = b.d_key.as<uint64_t>(); P.run_size = b.d_size.as<int64_t>(); P.run_off = b.d_roff.as<int64_t>();
  k_bam_encode<<<(unsigned)((nk + 255) / 256), 256, 0, st>>>(P);
  MG_CK(b.ctx, cudaGetLastError());
  int64_t last[2] = {0, 0};
  MG_CK(b.ctx, mg_fastq_ends(b.fq, k, last, st));
  MG_CK(b.ctx, cudaStreamSynchronize(st));
  b.run_n += nk; b.run_rec += bytes;
  if (n_templates) *n_templates = k;
  if (consumed1) *consumed1 = last[0] + 1;
  if (consumed2 && nf > 1) *consumed2 = last[1] + 1;
  b.t_dev += now_ms() - t0;
  return MG_OK;
}

void mg_bam_abort(mg_bam *h) {
  if (h) bam_delete(h);
}

int mg_bam_close(mg_bam *h, int64_t *n_records, int64_t *n_runs, double *times) {
  if (!h) return MG_EINVAL;
  Bam &b = h->b;
  DeviceGuard g(mg_internal_device(b.ctx));
  MgBamWriter w;
  int rc = MG_OK;
  if (!w.open(b.bam.c_str(), b.bai.empty() ? nullptr : b.bai.c_str(), b.header, b.n_ref, b.level, b.threads)) rc = bam_fail(b, MG_EVALUE, w.err);
  if (!rc && b.spills.empty()) {               // one run: straight from the device into the writer
    const double t = now_ms();
    if (b.run_n) {
      rc = sort_run(b);
      b.t_dev += now_ms() - t;
      if (!rc && stream_out(b, b.d_out.as<const uint8_t>(), b.run_rec, [&](const uint8_t *p, int64_t n) { return w.records(p, n); }))
        rc = bam_fail(b, MG_EVALUE, "cannot write " + b.bam + ": " + w.err);
      b.n_runs = 1;
    }
  } else if (!rc) {
    if (b.run_n) rc = spill_run(b);
    const double t = now_ms();
    if (!rc) rc = merge_runs(b, w);
    b.t_out += now_ms() - t;
  }
  int64_t n = 0;
  const double t = now_ms();
  if (!rc && !w.close(&n)) rc = bam_fail(b, MG_EVALUE, "cannot write " + b.bam + ": " + w.err);
  b.t_out += now_ms() - t;
  if (rc) w.discard();
  if (n_records) *n_records = n;
  if (n_runs) *n_runs = b.n_runs;
  if (times) { times[0] = b.t_dev; times[1] = b.t_d2h; times[2] = b.t_out; }
  bam_delete(h);
  return rc;
}

}  // extern "C"
