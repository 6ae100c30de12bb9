// alignment-analysis: an aligner's BAM scored against the truth in Mitty's qnames (the reference's
// mitty/benchmarking/mq.py and derr.py), counted on the device.  The rules are in include/mitty_b200.h and
// DESIGN.md §11.
//
// The chunks come from the BAM chunk pipeline (mg_bam_pipeline, mg_readmodel.cu) that bam2illumina also uses.
// One launch of k_alnerr per chunk, one thread per record (grid-stride, whole warps per step):
//   the thread checks the record against its block_size, parses only the qname fields of its read (chrom,
//   strand, pos, CIGAR, v_list; mg_parse_int), compares the chrom with the header name of refID and finds its
//   column (d_err, wrong chrom or unmapped).  The warp then aggregates its cells: __match_any_sync on the cell
//   index and one u64 atomicAdd of the popcount per distinct cell -- a good aligner puts nearly every read in
//   one cell (MAPQ 60, d = 0), so the cell is added once per warp, not once per record.  The v_list entries
//   are binned the same way, one entry per lane and step, until every lane's list is done.
//   Neither matrix fits in shared memory (256 x 403 x 4 B = 412 KB at the defaults): both live in global
//   memory.  The scalar counters are per-warp ballots into the CTA's shared counters, which go to the u64
//   global counters at the end of the launch.
#include <algorithm>
#include <cstring>

#include "../../include/mitty_b200.h"
#include "mg_bamrec.cuh"
#include "mg_bgzf.h"
#include "mg_internal.h"
#include "mg_qname.cuh"

namespace {

#define AE_THREADS 256
#define AE_MAX_D 10000
#define AE_MAX_SIZE 10000

enum { AE_ANALYSED = 0, AE_SKIPPED, AE_UNMAPPED, AE_WRONG_CHROM, AE_EXACT, AE_CLAMPED, AE_STRAND, AE_NO_VARIANT, AE_VARIANTS, AE_NCNT };
enum { AE_QNAME = 15, AE_MATE = 16, AE_REFID = 17 };     // record errors after the reader's 1 .. 14

struct AeParams {
  const uint8_t *data; const uint32_t *off; int64_t n; uint64_t first;
  const uint8_t *names; const int64_t *name_off; int n_ref;
  int max_d, max_size;
  unsigned long long *mq, *vsize, *cnt, *first_bad;
};

// end of the '|'-separated field that starts at q[a] (the name ends at len)
__device__ __forceinline__ int field_end(const uint8_t *q, int a, int len) {
  while (a < len && q[a] != '|') a++;
  return a;
}

// bases before the alignment start in the leading run of S, H and I ops of a qname CIGAR q[a, b) (P ops skipped;
// '>p:nI' is its plain form nI).  false if it is not a CIGAR: ops are digits + one of MIDNSHP=X, at least one.
__device__ bool qname_lead(const uint8_t *q, int a, int b, int64_t &lead) {
  if (a < b && q[a] == '>') {
    int colon = b - 1;
    while (colon > a && q[colon] != ':') colon--;
    int64_t p;
    if (colon == a || !mg_parse_int(q, a + 1, colon, p)) return false;
    a = colon + 1;
  }
  if (a >= b) return false;
  lead = 0;
  bool run = true;
  while (a < b) {
    int e = a;
    while (e < b && q[e] >= '0' && q[e] <= '9') e++;
    int64_t c;
    if (e == a || e >= b || !mg_parse_int(q, a, e, c)) return false;
    const uint8_t op = q[e];
    if (op == 'S' || op == 'H' || op == 'I') { if (run) lead += c; }
    else if (op == 'M' || op == 'D' || op == 'N' || op == '=' || op == 'X') run = false;
    else if (op != 'P') return false;
    a = e + 1;
  }
  return true;
}

// the v_list q[a, b): its entry count, or -1 if an entry is not an integer (empty entries are skipped)
__device__ int vlist_count(const uint8_t *q, int a, int b) {
  int n = 0;
  for (int x = a; a < b; a = x + 1) {
    x = a;
    while (x < b && q[x] != ',') x++;
    int64_t v;
    if (x > a && !mg_parse_int(q, a, x, v)) return -1;
    n += x > a;
  }
  return n;
}

// adds 1 per lane to m[key] (key < 0: nothing), one atomic per distinct key of the warp; every lane calls it
__device__ __forceinline__ void warp_add(unsigned long long *m, int key) {
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  if (key >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&m[key], (unsigned long long)__popc(peers));
}

__global__ void __launch_bounds__(AE_THREADS) k_alnerr(AeParams P) {
  __shared__ unsigned long long s_cnt[AE_NCNT];
  if (threadIdx.x < AE_NCNT) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, n_col = 2 * P.max_d + 3, none_row = 2 * P.max_size + 3;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < P.n; base += step) {
    const int64_t r = base + lane;
    int col = -1, mapq = 0, n_var = 0, va = 0, vb = 0;   // col >= 0: the record is analysed
    bool skipped = false, exact = false, clamped = false, strand_bad = false;
    const uint8_t *q = nullptr;
    if (r < P.n) {
      const uint8_t *rec = P.data + P.off[r];
      const uint64_t k = P.first + (uint64_t)r;
      int64_t qual_at;
      int bad = mg_bam_overrun(rec, qual_at);
      const int flag = rec[18] | rec[19] << 8;
      if (!bad && (flag & 0x900)) skipped = true;
      else if (!bad) {
        const int32_t ref = (int32_t)mg_ld32(rec + 4), pos = (int32_t)mg_ld32(rec + 8);
        const int l_name = rec[12], n_cig = rec[16] | rec[17] << 8;
        q = rec + 36;
        int len = 0;                                   // the qname: up to its NUL
        while (len < l_name && q[len]) len++;
        // fields 1 (chrom) and 3 + 5 * index .. + 4 of this read (strand, pos, rlen, CIGAR, v_list)
        const int last = (flag & 0xC1) == 0x81 ? 12 : 7;
        int a = 0, e = 0, ca = 0, cb = 0, sa = 0, sb = 0, pa = 0, pb = 0, ga = 0, gb = 0;
        int f = 0;
        for (; f <= last; f++) {
          if (f > 0 && e >= len) break;                // field f does not exist
          e = field_end(q, a, len);
          if (f == 1) { ca = a; cb = e; }
          else if (f == last - 4) { sa = a; sb = e; }
          else if (f == last - 3) { pa = a; pb = e; }
          else if (f == last - 1) { ga = a; gb = e; }
          else if (f == last) { va = a; vb = e; }
          a = e + 1;
        }
        int64_t strand, qpos, qlead;
        if (ref < -1 || ref >= P.n_ref) bad = AE_REFID;
        else if (f <= last) bad = f < 8 ? AE_QNAME : AE_MATE;
        else if (!mg_parse_int(q, sa, sb, strand) || (strand != 0 && strand != 1) || !mg_parse_int(q, pa, pb, qpos) || !qname_lead(q, ga, gb, qlead) ||
                 (n_var = vlist_count(q, va, vb)) < 0)
          bad = AE_QNAME;
        else {
          mapq = rec[13];
          if ((flag & 0x4) || ref == -1) col = n_col - 1;
          else {
            const int64_t na = P.name_off[ref], nb = P.name_off[ref + 1];
            bool same = nb - na == cb - ca;
            for (int i = 0; same && i < cb - ca; i++) same = P.names[na + i] == q[ca + i];
            if (!same) col = n_col - 2;
            else {
              const uint8_t *cig = rec + 36 + l_name;
              int64_t lead = 0;
              for (int i = 0; i < n_cig; i++) {
                const uint32_t o = mg_ld32(cig + 4 * i), op = o & 15;
                if (op == 1 || op == 4 || op == 5) lead += o >> 4;
                else if (op != 6) break;
              }
              const int64_t d = ((int64_t)pos - lead) - (qpos - 1 - qlead);
              col = (int)(max((int64_t)-P.max_d, min((int64_t)P.max_d, d)) + P.max_d);
              exact = d == 0;
              clamped = d > P.max_d || d < -P.max_d;
              strand_bad = ((flag >> 4) & 1) != (int)strand;
            }
          }
        }
      }
      if (bad) atomicMin(P.first_bad, (unsigned long long)(k << 8 | bad));
    }
    const bool on = col >= 0;
    const unsigned b_an = __ballot_sync(0xffffffffu, on), b_sk = __ballot_sync(0xffffffffu, skipped);
    const unsigned b_un = __ballot_sync(0xffffffffu, on && col == n_col - 1), b_wc = __ballot_sync(0xffffffffu, on && col == n_col - 2);
    const unsigned b_ex = __ballot_sync(0xffffffffu, exact), b_cl = __ballot_sync(0xffffffffu, clamped);
    const unsigned b_st = __ballot_sync(0xffffffffu, strand_bad), b_nv = __ballot_sync(0xffffffffu, on && n_var == 0);
    const unsigned n_ent = __reduce_add_sync(0xffffffffu, on ? (unsigned)n_var : 0u);
    if (lane == 0 && b_an | b_sk) {
      const unsigned v[AE_NCNT] = {(unsigned)__popc(b_an), (unsigned)__popc(b_sk), (unsigned)__popc(b_un), (unsigned)__popc(b_wc), (unsigned)__popc(b_ex),
                                   (unsigned)__popc(b_cl), (unsigned)__popc(b_st), (unsigned)__popc(b_nv), n_ent};
#pragma unroll
      for (int i = 0; i < AE_NCNT; i++) if (v[i]) atomicAdd(&s_cnt[i], (unsigned long long)v[i]);
    }
    warp_add(P.mq, on ? mapq * n_col + col : -1);
    // v_list: one entry (or the 'none' row) per lane and step
    bool more = on;
    bool none = n_var == 0;
    int x = va;
    while (__any_sync(0xffffffffu, more)) {
      int key = -1;
      if (more) {
        int row = none_row;
        if (none) more = false;
        else {
          while (q[x] == ',') x++;                     // an entry follows: n_var counted it
          int e = x;
          while (e < vb && q[e] != ',') e++;
          int64_t v;
          mg_parse_int(q, x, e, v);
          row = (int)(max((int64_t)-P.max_size - 1, min((int64_t)P.max_size + 1, v)) + P.max_size + 1);
          x = e;
          while (x < vb && q[x] == ',') x++;
          more = x < vb;
        }
        key = row * n_col + col;
      }
      warp_add(P.vsize, key);
    }
  }
  __syncthreads();
  if (threadIdx.x < AE_NCNT && s_cnt[threadIdx.x]) atomicAdd(&P.cnt[threadIdx.x], s_cnt[threadIdx.x]);
}

}  // namespace

extern "C" int mg_alnerr_bam(mg_ctx *ctx, const char *path, int32_t max_d, int32_t max_size, int32_t threads, int64_t chunk_bytes, uint64_t *mq,
                             uint64_t *vsize, int64_t *counts, double *times, double *thread_ms, int64_t *bad_where, int32_t *bad_code) {
  if (!ctx || !path || max_d < 0 || max_d > AE_MAX_D || max_size < 0 || max_size > AE_MAX_SIZE || !mq || !vsize || !counts || !times || !bad_where ||
      !bad_code)
    return MG_EINVAL;
  const double t_start = mg_now_ms();
  *bad_where = -1; *bad_code = 0;
  const int dev = mg_internal_device(ctx);
  DeviceGuard g(dev);
  int n_sm = 0, per_sm = 0;
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_alnerr, AE_THREADS, 0);

  MgBamReader rd;
  if (!rd.open(path, threads, chunk_bytes, mg_pinned_alloc, mg_pinned_release)) return mg_internal_fail(ctx, MG_EVALUE, rd.err.c_str());
  const size_t n_col = 2 * (size_t)max_d + 3, n_mq = 256 * n_col, n_vs = (2 * (size_t)max_size + 4) * n_col, n_acc = n_mq + n_vs + AE_NCNT;
  DevBuf d_acc, d_names, d_off;
  int64_t chunks = 0;
  unsigned long long cnt[AE_NCNT] = {0};
  bool names_up = false;
  AeParams P;
  memset(&P, 0, sizeof P);
  P.max_d = max_d; P.max_size = max_size;
  MgBamPipe pipe;
  pipe.begin = [&](cudaStream_t ks) -> int {
    MG_CK(ctx, d_acc.need(8 * n_acc));
    P.mq = d_acc.as<unsigned long long>(); P.vsize = P.mq + n_mq; P.cnt = P.vsize + n_vs;
    MG_CK(ctx, cudaMemsetAsync(P.mq, 0, 8 * n_acc, ks));
    return MG_OK;
  };
  pipe.launch = [&](const MgBamChunk &c, const uint8_t *data, const uint32_t *off, unsigned long long *first_bad, cudaStream_t ks) -> int {
    if (!names_up) {                                   // the header's names are complete once the first chunk is out
      names_up = true;
      P.n_ref = (int)(rd.ref_off.size() - 1);
      MG_CK(ctx, d_names.need(rd.ref_names.size() + 1));
      MG_CK(ctx, d_off.need(8 * rd.ref_off.size()));
      if (!rd.ref_names.empty()) MG_CK(ctx, cudaMemcpyAsync(d_names.p, rd.ref_names.data(), rd.ref_names.size(), cudaMemcpyHostToDevice, ks));
      MG_CK(ctx, cudaMemcpyAsync(d_off.p, rd.ref_off.data(), 8 * rd.ref_off.size(), cudaMemcpyHostToDevice, ks));
      P.names = d_names.as<uint8_t>(); P.name_off = d_off.as<int64_t>();
    }
    P.data = data; P.off = off; P.n = c.n; P.first = (uint64_t)c.first; P.first_bad = first_bad;
    const unsigned grid = (unsigned)std::min<int64_t>((int64_t)n_sm * std::max(1, per_sm), (c.n + AE_THREADS - 1) / AE_THREADS);
    k_alnerr<<<grid, AE_THREADS, 0, ks>>>(P);
    MG_CK(ctx, cudaGetLastError());
    return MG_OK;
  };
  pipe.finish = [&](cudaStream_t ks) -> int {
    MG_CK(ctx, cudaMemcpyAsync(mq, P.mq, 8 * n_mq, cudaMemcpyDeviceToHost, ks));
    MG_CK(ctx, cudaMemcpyAsync(vsize, P.vsize, 8 * n_vs, cudaMemcpyDeviceToHost, ks));
    MG_CK(ctx, cudaMemcpyAsync(cnt, P.cnt, sizeof cnt, cudaMemcpyDeviceToHost, ks));
    return MG_OK;
  };
  const int rc = mg_bam_pipeline(ctx, rd, pipe, t_start, &chunks, times, thread_ms, bad_where, bad_code);
  const int64_t out[14] = {rd.records, (int64_t)cnt[AE_ANALYSED], (int64_t)cnt[AE_SKIPPED], (int64_t)cnt[AE_UNMAPPED], (int64_t)cnt[AE_WRONG_CHROM],
                           (int64_t)cnt[AE_EXACT], (int64_t)cnt[AE_CLAMPED], (int64_t)cnt[AE_STRAND], (int64_t)cnt[AE_NO_VARIANT],
                           (int64_t)cnt[AE_VARIANTS], rd.raw_bytes, rd.comp_bytes, rd.eof_marker ? 1 : 0, chunks};
  memcpy(counts, out, sizeof out);
  return rc;
}
