// Round-trip checker (the god-aligner contract) on the device.
//
// Mitty's god-aligner trusts the qname: it writes every read into a BAM at the POS / CIGAR the qname
// states, reverse-complementing the strand-1 reads (mitty/benchmarking/god_aligner.py:141-183 over
// readgenerate.parse_qname, mitty/simulation/readgenerate.py:259-291; the '>p:nI' special CIGAR of a
// read inside a long insertion becomes 'nI').  k_roundtrip_check re-derives EVERY read of a FASTQ pair
// from (chrom, copy, strand, pos, CIGAR) + reference + VCF and compares it with the bases in the file:
//   '='  the read equals the reference at the running reference position
//   'X'  the read equals the haplotype (the SNP's ALT) and differs from the reference
//   'I'  the read carries the inserted bases of the insertion recorded at that reference position (the
//        LAST n bases of it when the read starts inside it, the first n otherwise)
//   'D'  the reference position advances, the deleted bases exist in the node list
// One thread per read.  Reference and haplotypes are expanded to ASCII views once per copy
// (k_expand_ascii / k_patch_exc), so N, IUPAC codes and lower-case stretches compare as the bytes they are.
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/mitty_b200.h"
#include "mg_internal.h"
#include "mg_qname.cuh"

namespace {

struct ChkCopy {
  char chrom[40]; int chrom_len; int cpy;
  const MgNode *nodes; int n_nodes;
  const uint8_t *hap; uint32_t hap_len;
  const uint8_t *ref; int64_t ref_len; int64_t start1;     // ref[i] = the base at 1-based reference position start1 + i
};

enum { CHK_OK = 0, CHK_QNAME = 1, CHK_COPY = 2, CHK_LEN = 3, CHK_EQ = 4, CHK_X = 5, CHK_INS = 6, CHK_NOINS = 7, CHK_OP = 8, CHK_RANGE = 9, CHK_FRAME = 10 };

__global__ void __launch_bounds__(256) k_expand_ascii(const uint32_t *__restrict__ packed, int64_t len, uint8_t *__restrict__ out) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w * 16 >= len) return;
  uint32_t v = packed[w];
  for (int i = 0; i < 16 && w * 16 + i < len; i += 4, v >>= 8) {
    const uint32_t ch = mg_chars4(v & 0xFFu);
    for (int j = 0; j < 4 && w * 16 + i + j < len; j++) out[w * 16 + i + j] = (uint8_t)(ch >> (8 * j));
  }
}

// exception runs over the expanded text: one thread per 256-base block finds the runs that touch it
__global__ void __launch_bounds__(256) k_patch_exc(const MgExc *__restrict__ exc, int n_exc, int64_t len, uint8_t *__restrict__ out) {
  const int64_t b0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 256;
  if (b0 >= len || n_exc == 0) return;
  const int64_t b1 = b0 + 256 < len ? b0 + 256 : len;
  for (int k = mg_exc_first(exc, n_exc, (uint32_t)b0); k < n_exc; k++) {
    const MgExc e = exc[k];
    if ((int64_t)e.start >= b1) break;
    const int64_t a = (int64_t)e.start > b0 ? e.start : b0, b = (int64_t)e.start + e.len < b1 ? (int64_t)e.start + e.len : b1;
    for (int64_t i = a; i < b; i++) out[i] = e.byte == MG_EXC_CASE ? (uint8_t)(out[i] | 0x20) : (uint8_t)e.byte;
  }
}

__device__ __forceinline__ int last_node_pr_le(const MgNode *nodes, int n, int64_t rp) {   // last node with pr <= rp, -1 if none
  int lo = 0, hi = n;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if ((int64_t)nodes[mid].pr <= rp) lo = mid + 1; else hi = mid; }
  return lo - 1;
}

__device__ __forceinline__ uint8_t comp_base(uint8_t c) {   // DNA_complement of the reference: ATCGN only, upper case (readgenerate.py:56)
  return c == 'A' ? 'T' : c == 'T' ? 'A' : c == 'C' ? 'G' : c == 'G' ? 'C' : c;
}

struct ChkParams {
  const uint8_t *fq[2]; const int64_t *nl[2]; int64_t n_rec; int n_files;
  const ChkCopy *copies; int n_copies;
  uint8_t *code;                  // [n_files][n_rec] error code per read
  unsigned long long *n_bad;
};

__global__ void __launch_bounds__(256) k_roundtrip_check(ChkParams P) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= P.n_rec * P.n_files) return;
  const int f = (int)(t / P.n_rec);
  const int64_t r = t - (int64_t)f * P.n_rec;
  const uint8_t *q = P.fq[f];
  const int64_t *nl = P.nl[f];
  const int64_t h0 = r == 0 ? 0 : nl[4 * r - 1] + 1, h1 = nl[4 * r], s0 = h1 + 1, s1 = nl[4 * r + 1];
  int code = CHK_OK;
  do {
    if (h1 <= h0 || q[h0] != '@' || nl[4 * r + 2] != s1 + 2 || q[s1 + 1] != '+' || nl[4 * r + 3] - nl[4 * r + 2] != s1 - s0 + 1) { code = CHK_FRAME; break; }
    // fields: 0 serial, 1 chrom, 2 copy, then strand | pos | rlen | cigar | vlist per read in file order; this file's read is the f-th
    int64_t fs[MG_QN_FIELDS], fe[MG_QN_FIELDS];
    const int nf = mg_qname_split(q, h0 + 1, h1, fs, fe);
    const int base = 3 + 5 * f;
    if (nf < base + 5) { code = CHK_QNAME; break; }
    int64_t cpy, strand, pos, rlen;
    if (!mg_parse_int(q, fs[2], fe[2], cpy) || !mg_parse_int(q, fs[base], fe[base], strand) || !mg_parse_int(q, fs[base + 1], fe[base + 1], pos) ||
        !mg_parse_int(q, fs[base + 2], fe[base + 2], rlen) || (strand != 0 && strand != 1)) { code = CHK_QNAME; break; }
    const ChkCopy *C = nullptr;
    const int cl = (int)(fe[1] - fs[1]);
    for (int k = 0; k < P.n_copies && !C; k++) {
      const ChkCopy &c = P.copies[k];
      if (c.cpy != (int)cpy || c.chrom_len != cl) continue;
      if (pos < c.start1 - 1 || pos >= c.start1 + c.ref_len) continue;     // several BED regions of one chromosome: the one that holds POS
      bool same = true;
      for (int i = 0; i < cl && same; i++) same = c.chrom[i] == (char)q[fs[1] + i];
      if (same) C = &c;
    }
    if (!C) { code = CHK_COPY; break; }
    const int64_t L = s1 - s0;
    if (L != rlen) { code = CHK_LEN; break; }
    auto fwd = [&](int64_t i) -> uint8_t { return strand ? comp_base(q[s0 + L - 1 - i]) : q[s0 + i]; };   // god_aligner.py:163-166
    int64_t ca = fs[base + 3], cb = fe[base + 3];
    if (ca < cb && q[ca] == '>') {                          // '>p:nI': the read lies inside one long insertion, POS = its anchor
      int64_t colon = ca + 1;
      while (colon < cb && q[colon] != ':') colon++;
      int64_t off, n;
      if (colon >= cb || q[cb - 1] != 'I' || !mg_parse_int(q, ca + 1, colon, off) || !mg_parse_int(q, colon + 1, cb - 1, n) || n != L) { code = CHK_QNAME; break; }
      int k = last_node_pr_le(C->nodes, C->n_nodes, pos + 1);
      while (k >= 0 && C->nodes[k].pr == pos + 1 && C->nodes[k].op != 'I') k--;
      if (k < 0 || C->nodes[k].pr != pos + 1 || C->nodes[k].op != 'I') { code = CHK_NOINS; break; }
      const MgNode nd = C->nodes[k];
      if (off < 0 || off + n > nd.oplen) { code = CHK_RANGE; break; }
      for (int64_t i = 0; i < n && code == CHK_OK; i++) if (C->hap[nd.key + off + i] != fwd(i)) code = CHK_INS;
      break;
    }
    int64_t rp = pos, i = 0;
    bool first = true;
    while (ca < cb && code == CHK_OK) {
      int64_t e = ca;
      while (e < cb && q[e] >= '0' && q[e] <= '9') e++;
      int64_t c;
      if (e == ca || e >= cb || !mg_parse_int(q, ca, e, c)) { code = CHK_QNAME; break; }
      const uint8_t op = q[e];
      ca = e + 1;
      if (op == '=') {
        const int64_t o = rp - C->start1;
        if (o < 0 || o + c > C->ref_len || i + c > L) { code = CHK_RANGE; break; }
        for (int64_t j = 0; j < c; j++) if (C->ref[o + j] != fwd(i + j)) { code = CHK_EQ; break; }
        rp += c; i += c;
      } else if (op == 'X') {
        const int k = last_node_pr_le(C->nodes, C->n_nodes, rp);
        const int64_t o = rp - C->start1;
        if (k < 0 || (C->nodes[k].op != '=' && C->nodes[k].op != 'X') || o < 0 || o + c > C->ref_len || i + c > L) { code = CHK_RANGE; break; }
        const int64_t sp = (int64_t)C->nodes[k].key + (rp - C->nodes[k].pr);
        if (sp + c > C->hap_len) { code = CHK_RANGE; break; }
        for (int64_t j = 0; j < c; j++) if (C->hap[sp + j] != fwd(i + j) || C->ref[o + j] == fwd(i + j)) { code = CHK_X; break; }
        rp += c; i += c;
      } else if (op == 'I') {
        int k = last_node_pr_le(C->nodes, C->n_nodes, rp);
        while (k >= 0 && C->nodes[k].pr == rp && C->nodes[k].op != 'I') k--;
        if (k < 0 || C->nodes[k].pr != rp || C->nodes[k].op != 'I') { code = CHK_NOINS; break; }
        const MgNode nd = C->nodes[k];
        if (c > nd.oplen || i + c > L) { code = CHK_RANGE; break; }
        const int64_t from = first ? nd.oplen - c : 0;      // a read that starts inside the insertion carries its tail
        for (int64_t j = 0; j < c; j++) if (C->hap[nd.key + from + j] != fwd(i + j)) { code = CHK_INS; break; }
        i += c;
      } else if (op == 'D') {
        rp += c;
      } else { code = CHK_OP; break; }
      first = false;
    }
    if (code == CHK_OK && i != L) code = CHK_LEN;
  } while (false);
  P.code[t] = (uint8_t)code;
  if (code) atomicAdd(P.n_bad, 1ull);
}

struct Checker {
  mg_ctx *ctx;
  std::vector<ChkCopy> copies;
  std::vector<DevBuf> owned;                       // ASCII views (moving a DevBuf leaves its device block in place)
  std::map<int64_t, const uint8_t *> ref_view;     // region id -> ASCII reference, inside `owned`
  DevBuf d_copies; bool dirty = true;
  MgFastqChunk fq;
  DevBuf d_code, d_bad;
};

}  // namespace

extern "C" {

struct mg_checker { Checker c; };

int mg_check_open(mg_ctx *ctx, mg_checker **out) {
  if (!ctx || !out) return MG_EINVAL;
  mg_checker *k = new mg_checker();
  k->c.ctx = ctx;
  *out = k;
  return MG_OK;
}

void mg_check_close(mg_checker *k) {
  if (!k) return;
  DeviceGuard g(mg_internal_device(k->c.ctx));
  cudaStreamSynchronize(mg_internal_stream(k->c.ctx));
  delete k;
}

static int expand(mg_ctx *ctx, const uint32_t *packed, int64_t len, const MgExc *exc, int n_exc, uint8_t **out, std::vector<DevBuf> &owned) {
  cudaStream_t st = mg_internal_stream(ctx);
  DevBuf v;
  v.cap = (size_t)std::max<int64_t>(len, 1);      // exact: the views of a genome are large
  if (cudaMalloc(&v.p, v.cap) != cudaSuccess) return mg_internal_fail(ctx, MG_ECUDA, "out of device memory for the checker's text views");
  *out = v.as<uint8_t>();
  owned.push_back(std::move(v));
  if (len > 0) {
    const int64_t words = (len + 15) / 16;
    k_expand_ascii<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(packed, len, *out);
    if (n_exc) k_patch_exc<<<(unsigned)(((len + 255) / 256 + 255) / 256), 256, 0, st>>>(exc, n_exc, len, *out);
  }
  MG_CK(ctx, cudaGetLastError());
  return MG_OK;
}

int mg_check_add_copy(mg_checker *k, int64_t copy_id, const char *chrom, int32_t cpy) {
  if (!k || !chrom || strlen(chrom) >= sizeof(((ChkCopy *)0)->chrom)) return MG_EINVAL;
  mg_ctx *ctx = k->c.ctx;
  DeviceGuard g(mg_internal_device(ctx));
  int64_t rid, start1, rlen; const MgNode *nodes; int n_nodes, n_exc, rn_exc; const uint32_t *hap, *ref; uint32_t hap_len; const MgExc *exc, *rexc;
  int rc = mg_internal_copy_view(ctx, copy_id, &rid, &nodes, &n_nodes, &hap, &hap_len, &exc, &n_exc, &start1);
  if (rc) return rc;
  rc = mg_internal_region_view(ctx, rid, &ref, &rlen, &rexc, &rn_exc);
  if (rc) return rc;
  ChkCopy c; memset(&c, 0, sizeof c);
  strcpy(c.chrom, chrom); c.chrom_len = (int)strlen(chrom); c.cpy = cpy;
  c.nodes = nodes; c.n_nodes = n_nodes; c.hap_len = hap_len; c.start1 = start1; c.ref_len = rlen;
  uint8_t *h = nullptr;
  rc = expand(ctx, hap, hap_len, exc, n_exc, &h, k->c.owned);
  if (rc) return rc;
  c.hap = h;
  auto it = k->c.ref_view.find(rid);
  if (it == k->c.ref_view.end()) {
    uint8_t *r = nullptr;
    rc = expand(ctx, ref, rlen, rexc, rn_exc, &r, k->c.owned);
    if (rc) return rc;
    it = k->c.ref_view.insert({rid, r}).first;
  }
  c.ref = it->second;
  k->c.copies.push_back(c);
  k->c.dirty = true;
  return MG_OK;
}

int mg_check_fastq(mg_checker *k, const uint8_t *in1, int64_t len1, const uint8_t *in2, int64_t len2, int64_t *n_records,
                   int64_t *n_bad, int64_t *bad_index, int32_t *bad_code, int32_t bad_cap, int64_t *consumed1, int64_t *consumed2) {
  if (!k || !in1 || len1 < 0 || (in2 && len2 < 0)) return MG_EINVAL;
  Checker &c = k->c;
  mg_ctx *ctx = c.ctx;
  DeviceGuard g(mg_internal_device(ctx));
  cudaStream_t st = mg_internal_stream(ctx);
  if (c.dirty) {
    MG_CK(ctx, c.d_copies.need(sizeof(ChkCopy) * std::max<size_t>(1, c.copies.size())));
    MG_CK(ctx, cudaMemcpyAsync(c.d_copies.p, c.copies.data(), sizeof(ChkCopy) * c.copies.size(), cudaMemcpyHostToDevice, st));
    c.dirty = false;
  }
  const int nf = in2 ? 2 : 1;
  const uint8_t *in[2] = {in1, in2}; const int64_t len[2] = {len1, len2};
  MG_CK(ctx, mg_fastq_load(c.fq, in, len, nf, st));
  const int64_t n_rec = c.fq.n_tpl;
  if (n_records) *n_records = n_rec;
  if (n_bad) *n_bad = 0;
  if (consumed1) *consumed1 = 0;
  if (consumed2) *consumed2 = 0;
  if (n_rec == 0) return MG_OK;
  int64_t last[2] = {0, 0};
  MG_CK(ctx, mg_fastq_ends(c.fq, n_rec, last, st));
  ChkParams P; memset(&P, 0, sizeof P);
  for (int f = 0; f < nf; f++) { P.fq[f] = c.fq.in[f].as<uint8_t>(); P.nl[f] = c.fq.nl[f].as<int64_t>(); }
  P.n_rec = n_rec; P.n_files = nf;
  P.copies = c.d_copies.as<const ChkCopy>(); P.n_copies = (int)c.copies.size();
  MG_CK(ctx, c.d_code.need((size_t)(n_rec * nf)));
  MG_CK(ctx, c.d_bad.need(8));
  MG_CK(ctx, cudaMemsetAsync(c.d_bad.p, 0, 8, st));
  P.code = c.d_code.as<uint8_t>(); P.n_bad = c.d_bad.as<unsigned long long>();
  k_roundtrip_check<<<(unsigned)((n_rec * nf + 255) / 256), 256, 0, st>>>(P);
  MG_CK(ctx, cudaGetLastError());
  unsigned long long bad = 0;
  MG_CK(ctx, cudaMemcpyAsync(&bad, c.d_bad.p, 8, cudaMemcpyDeviceToHost, st));
  MG_CK(ctx, cudaStreamSynchronize(st));
  if (consumed1) *consumed1 = last[0] + 1;
  if (consumed2 && nf > 1) *consumed2 = last[1] + 1;
  if (n_bad) *n_bad = (int64_t)bad;
  if (bad && bad_index && bad_code && bad_cap > 0) {
    std::vector<uint8_t> codes((size_t)(n_rec * nf));
    MG_CK(ctx, cudaMemcpy(codes.data(), c.d_code.p, codes.size(), cudaMemcpyDeviceToHost));
    int w = 0;
    for (size_t i = 0; i < codes.size() && w < bad_cap; i++) if (codes[i]) { bad_index[w] = (int64_t)i; bad_code[w] = codes[i]; w++; }
  }
  return MG_OK;
}

}  // extern "C"
