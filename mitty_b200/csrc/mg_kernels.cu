// Hand-written sm_100a kernels of the read-generation engine.  No tensor cores: every kernel
// here is HBM / L2-bound byte and integer work (scan, gather, format, table lookup).
//
//   k_pack_ref        ASCII reference -> 2-bit packed words + non-ACGT run boundaries
//   k_hap_build       packed reference + variant segments -> packed haplotype of one copy
//   k_blk_table       node keys -> block lookup table
//   k_gap_*           Philox geometric gaps -> grid-wide inclusive scan (template starts)
//   k_walk_*          node list of a chromosome copy (pointer doubling over the variant chain)
//   k_unit_plan       phase 1 of a unit: template sampling, te < p_max / N filters, node lookup, record
//                     sizes, decoupled look-back scan -> one 32-byte plan per kept template
//   k_unit_emit       THE hot kernel, phase 2: qname/CIGAR formatting + sequence extraction/revcomp
//                     (+ fused Philox corruption) into per-warp shared-memory stages, bulk-copied
//                     (cp.async.bulk) to the two FASTQ buffers
//   k_sample          template sampling only (read-module plugin generate_reads)
//   k_scan_*          generic exclusive scan (int64)
//   k_nl_*            FASTQ newline index
//   k_corrupt_*       standalone corrupt-reads over FASTQ in HBM
#include <algorithm>
#include <cstdlib>
#include "mg_internal.h"

#define FULL 0xffffffffu

// ------------------------------------------------------------------------------------------
// small helpers

__device__ __forceinline__ uint32_t warp_incl_scan_u32(uint32_t v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t n = __shfl_up_sync(FULL, v, d);
    if (lane >= d) v += n;
  }
  return v;
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
  return v;
}

__device__ __forceinline__ unsigned long long ld_vol64(const unsigned long long *p) {
  return *(const volatile unsigned long long *)p;
}
__device__ __forceinline__ void st_vol64(unsigned long long *p, unsigned long long v) {
  *(volatile unsigned long long *)p = v;
}

// ------------------------------------------------------------------------------------------
// k_pack_ref: 16 bases per thread

__global__ void __launch_bounds__(256) k_pack_ref(const uint8_t *__restrict__ raw, int64_t len, uint32_t *__restrict__ packed,
                                                  uint32_t *exc_cnt, int64_t *exc_start, uint8_t *exc_byte,
                                                  int64_t *exc_end, uint32_t exc_cap) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t base = w * 16;
  if (base >= len) return;
  uint8_t c[18];  // c[0] = byte before, c[1..16] = mine, c[17] = byte after
  c[0] = base > 0 ? raw[base - 1] : 0;
  if (base + 16 <= len) {
    uint4 v = *reinterpret_cast<const uint4 *>(raw + base);
    uint32_t q[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 16; i++) c[1 + i] = (uint8_t)(q[i >> 2] >> (8 * (i & 3)));
  } else {
#pragma unroll
    for (int i = 0; i < 16; i++) c[1 + i] = (base + i < len) ? raw[base + i] : (uint8_t)'A';
  }
  c[17] = (base + 16 < len) ? raw[base + 16] : 0;
  uint32_t word = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) {
    int64_t pos = base + i;
    if (pos >= len) break;
    uint32_t code = mg_base_code(c[1 + i]);
    if (code > 3) {
      // runs of one identical non-ACGT byte; lower-case a/c/g/t form "case runs" of any mix of the
      // four letters and keep their codes
      const uint32_t lc = mg_base_code((uint8_t)(c[1 + i] ^ 0x20));   // code of the upper-case letter, if c is lower-case acgt
      const bool soft = c[1 + i] >= 'a' && lc <= 3;
      bool is_start, is_end;
      if (soft) {
        const bool prev_soft = pos > 0 && c[i] >= 'a' && mg_base_code((uint8_t)(c[i] ^ 0x20)) <= 3;
        const bool next_soft = pos < len - 1 && c[2 + i] >= 'a' && mg_base_code((uint8_t)(c[2 + i] ^ 0x20)) <= 3;
        is_start = !prev_soft; is_end = !next_soft;
      } else {
        is_start = (pos == 0) || (c[i] != c[1 + i]);
        is_end = (pos == len - 1) || (c[2 + i] != c[1 + i]);
      }
      if (is_start) {
        uint32_t k = atomicAdd(&exc_cnt[0], 1u);
        if (k < exc_cap) { exc_start[k] = pos; exc_byte[k] = soft ? (uint8_t)MG_EXC_CASE : c[1 + i]; }
      }
      if (is_end) {
        uint32_t k = atomicAdd(&exc_cnt[1], 1u);
        if (k < exc_cap) exc_end[k] = pos;
      }
      code = soft ? lc : 0;
    }
    word |= code << (2 * i);
  }
  packed[w] = word;
}

void mg_launch_pack_ref(const uint8_t *raw, int64_t len, uint32_t *packed, uint32_t *exc_cnt, int64_t *exc_start,
                        uint8_t *exc_byte, int64_t *exc_end, uint32_t exc_cap, cudaStream_t st) {
  int64_t words = (len + 15) / 16;
  if (words == 0) return;
  k_pack_ref<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(raw, len, packed, exc_cnt, exc_start, exc_byte, exc_end, exc_cap);
}

// ------------------------------------------------------------------------------------------
// k_walk_*: the node list of one chromosome copy (rpc.create_node_list, rpc.py:38-116) on the device.
//
// The reference walks the variants in order and skips every variant with v.pos < ref_pos (rpc.py:55),
// where ref_pos is where the previously ACCEPTED variant left the reference cursor.  That cursor
// depends only on the accepted variant itself -- end_ref(i) = pos+1 (SNP, insertion) or pos+1+oplen
// (deletion) -- so the accepted variants form a chain i0 -> nxt(i0) -> nxt(nxt(i0)) ... with
// nxt(i) = first j with pos[j] >= end_ref(i) (POS is sorted: the records come from an indexed
// fetch).  The chain is marked by pointer doubling (ceil(log2 V) rounds), every accepted variant
// then sizes its nodes (an optional '=' run up to it, then X / I / D), one exclusive scan of
// (node count, sample-space advance) places them, and a last kernel writes the node table.

#define MG_WALK_ADV_BITS 34
#define MG_WALK_ADV_MASK ((1ull << MG_WALK_ADV_BITS) - 1)

__device__ __forceinline__ int64_t walk_end_ref(const int64_t *pos, const uint8_t *op, const int64_t *oplen, int i) {
  return pos[i] + 1 + (op[i] == 'D' ? oplen[i] : 0);
}

__device__ __forceinline__ int walk_lower_bound(const int64_t *pos, int lo, int hi, int64_t x) {   // first j in [lo, hi) with pos[j] >= x, hi if none
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (pos[mid] < x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// segment of variant i: the last segment with v0 <= i (empty segments share their v0 with the next one)
__device__ __forceinline__ int seg_of_var(const MgSeg *segs, int n_seg, int i) {
  int lo = 0, hi = n_seg - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (segs[mid].v0 <= i) lo = mid; else hi = mid - 1; }
  return lo;
}
// segment of element e (the elements of segment s are its variants v0 + s .. v1 + s - 1 and its tail v1 + s)
__device__ __forceinline__ int seg_of_elem(const MgSeg *segs, int n_seg, int e) {
  int lo = 0, hi = n_seg - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (segs[mid].v0 + mid <= e) lo = mid; else hi = mid - 1; }
  return lo;
}

__device__ __forceinline__ void walk_error(MgWalkSummary *sum, int idx, int code) {   // the first error in variant order wins
  atomicMin(&sum->err, ((unsigned long long)(uint32_t)idx << 8) | (unsigned long long)code);
}

__global__ void __launch_bounds__(256) k_walk_next(const int64_t *__restrict__ pos, const uint8_t *__restrict__ op,
                                                   const int64_t *__restrict__ oplen, int V, const MgSeg *__restrict__ segs, int n_seg,
                                                   MgSegOut *__restrict__ seg_out, uint32_t *__restrict__ nxt,
                                                   uint32_t *__restrict__ jump, uint8_t *__restrict__ mark, int32_t *__restrict__ pred,
                                                   MgWalkSummary *sum) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) { sum->err = ~0ull; sum->n_nodes = 0; sum->hap_len = 0; sum->ends_in_d = 0; sum->bad = 0; }
  if (i < n_seg) {                                   // variants before the region start are skipped (rpc.py:55)
    const MgSeg sg = segs[i];
    const int j = walk_lower_bound(pos, sg.v0, sg.v1, sg.start1);
    MgSegOut o; o.hap_base = 0; o.hap_len = 0; o.i0 = j < sg.v1 ? j : -1; o.last = -1; o.ends_in_d = 0; o.node0 = 0; o.n_nodes = 0; o.pad = 0;
    seg_out[i] = o;
  }
  if (i >= V) return;
  const MgSeg sg = segs[seg_of_var(segs, n_seg, i)];
  const int j = walk_lower_bound(pos, sg.v0, sg.v1, walk_end_ref(pos, op, oplen, i));
  const uint32_t jj = j < sg.v1 ? (uint32_t)j : (uint32_t)V;          // the chain ends at its segment's end
  nxt[i] = jj; jump[i] = jj; mark[i] = 0; pred[i] = -1;
}

__global__ void __launch_bounds__(256) k_walk_seed(const MgSegOut *__restrict__ seg_out, int n_seg, uint8_t *mark) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_seg && seg_out[s].i0 >= 0) mark[seg_out[s].i0] = 1;       // every segment's chain starts at its first accepted variant
}

// one doubling round: marked variants mark the variant 2^k links ahead, links double
__global__ void __launch_bounds__(256) k_walk_round(const uint32_t *__restrict__ jin, uint32_t *__restrict__ jout, uint8_t *mark, int V) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const uint32_t j = jin[i];
  if (mark[i] && j < (uint32_t)V) mark[j] = 1;
  jout[i] = j < (uint32_t)V ? jin[j] : (uint32_t)V;
}

__global__ void __launch_bounds__(256) k_walk_pred(const uint32_t *__restrict__ nxt, const uint8_t *__restrict__ mark,
                                                   int32_t *__restrict__ pred, const MgSeg *__restrict__ segs, int n_seg,
                                                   MgSegOut *__restrict__ seg_out, int V) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V || !mark[i]) return;
  const uint32_t j = nxt[i];
  if (j < (uint32_t)V) pred[j] = i; else seg_out[seg_of_var(segs, n_seg, i)].last = i;
}

// per element (accepted variant, or the tail of a segment): node count and sample-space advance, packed for one scan
__global__ void __launch_bounds__(256) k_walk_measure(const int64_t *__restrict__ pos, const uint8_t *__restrict__ op,
                                                      const int64_t *__restrict__ oplen, const int64_t *__restrict__ alt_off,
                                                      const uint8_t *__restrict__ mark, const int32_t *__restrict__ pred, int V,
                                                      const MgSeg *__restrict__ segs, int n_seg, const MgSegOut *__restrict__ seg_out,
                                                      int64_t *__restrict__ packed, MgWalkSummary *sum) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= V + n_seg) return;
  const int s = seg_of_elem(segs, n_seg, e);
  const MgSeg sg = segs[s];
  const int i = e - s;
  if (i >= sg.v1) {                                     // the tail '=' node (rpc.py:58-61), absent when a deletion crossed the region end
    const int last = seg_out[s].last;
    const int64_t refp = last < 0 ? sg.start1 : walk_end_ref(pos, op, oplen, last);
    const int64_t offset = refp - sg.start1;
    const bool has = offset <= sg.region_len;
    packed[e] = has ? (int64_t)((1ull << MG_WALK_ADV_BITS) | (unsigned long long)(sg.region_len - offset)) : 0;
    return;
  }
  if (!mark[i]) { packed[e] = 0; return; }
  const int64_t R = pred[i] < 0 ? sg.start1 : walk_end_ref(pos, op, oplen, pred[i]);
  const int64_t vp = pos[i], alt_len = alt_off[i + 1] - alt_off[i];
  int64_t delta, adv, cnt;
  if (op[i] == 'X') {                                   // rpc.py:75-87
    delta = vp - R; cnt = (delta > 0) + 1; adv = delta + 1;
    if (alt_len != 1) walk_error(sum, i, 1);
  } else if (op[i] == 'I') {                            // rpc.py:90-102
    delta = vp + 1 - R; cnt = 2; adv = delta + oplen[i];
    if (alt_len - 1 != oplen[i] || oplen[i] < 0) walk_error(sum, i, 2);
  } else if (op[i] == 'D') {                            // rpc.py:105-116
    delta = vp + 1 - R; cnt = 2; adv = delta;
    if (oplen[i] < 0) walk_error(sum, i, 3);
  } else {
    delta = 0; cnt = 0; adv = 0;
    walk_error(sum, i, 3);
  }
  if ((R - sg.start1) + delta > sg.region_len || oplen[i] > 0x7FFFFFFFll || adv < 0 || adv > (int64_t)MG_WALK_ADV_MASK) { sum->bad = 1; adv = 0; }
  packed[e] = (int64_t)(((unsigned long long)cnt << MG_WALK_ADV_BITS) | (unsigned long long)adv);
}

// node table + per-node sources; a segment's tail element also writes the segment's summary
__global__ void __launch_bounds__(256) k_walk_nodes(const int64_t *__restrict__ pos, const uint8_t *__restrict__ op,
                                                    const int64_t *__restrict__ oplen, const int64_t *__restrict__ alt_off,
                                                    const uint8_t *__restrict__ mark, const int32_t *__restrict__ pred, int V,
                                                    const MgSeg *__restrict__ segs, int n_seg, MgSegOut *__restrict__ seg_out,
                                                    const int64_t *__restrict__ scanned,
                                                    MgNode *__restrict__ nodes, uint32_t *__restrict__ node_alt, MgWalkSummary *sum) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int E = V + n_seg;
  if (e == E) {                                          // totals
    const unsigned long long tot = (unsigned long long)scanned[E];
    sum->n_nodes = (long long)(tot >> MG_WALK_ADV_BITS); sum->hap_len = (long long)(tot & MG_WALK_ADV_MASK);
    return;
  }
  if (e > E) return;
  const int s = seg_of_elem(segs, n_seg, e);
  const MgSeg sg = segs[s];
  const int i = e - s;
  const unsigned long long pre = (unsigned long long)scanned[e];
  uint32_t k = (uint32_t)(pre >> MG_WALK_ADV_BITS);
  int64_t S = (int64_t)(pre & MG_WALK_ADV_MASK);          // sample position in the concatenated haplotype
  if (i >= sg.v1) {
    const int last = seg_out[s].last;
    const int64_t refp = last < 0 ? sg.start1 : walk_end_ref(pos, op, oplen, last);
    const int64_t offset = refp - sg.start1;
    const unsigned long long first = (unsigned long long)scanned[sg.v0 + s];   // the segment's first element
    const uint32_t node0 = (uint32_t)(first >> MG_WALK_ADV_BITS);
    const int64_t base = (int64_t)(first & MG_WALK_ADV_MASK);
    if (offset <= sg.region_len) {
      if (S + (sg.region_len - offset) >= 0xFFF00000ll || refp >= (1ll << 31)) sum->bad = 1;
      nodes[k] = MgNode{(uint32_t)S, (int32_t)refp, (int32_t)(sg.region_len - offset), '='};
      node_alt[k] = sg.roff + (uint32_t)offset;
      seg_out[s].hap_base = (uint32_t)base; seg_out[s].hap_len = (uint32_t)(S + (sg.region_len - offset) - base);
      seg_out[s].node0 = node0; seg_out[s].n_nodes = k + 1 - node0; seg_out[s].ends_in_d = 0;
    } else {                                              // a deletion crossed the region end: the list ends in 'D'
      seg_out[s].hap_base = (uint32_t)base; seg_out[s].hap_len = (uint32_t)(S - base);
      seg_out[s].node0 = node0; seg_out[s].n_nodes = k - node0; seg_out[s].ends_in_d = 1;
      sum->ends_in_d = 1;
    }
    return;
  }
  if (!mark[i]) return;
  const int64_t R = pred[i] < 0 ? sg.start1 : walk_end_ref(pos, op, oplen, pred[i]);
  const int64_t vp = pos[i];
  const uint8_t o = op[i];
  const int64_t delta = (o == 'X') ? vp - R : vp + 1 - R;
  if (S + delta + (o == 'I' ? oplen[i] : 1) >= 0xFFF00000ll || vp + 1 + (o == 'D' ? oplen[i] : 0) >= (1ll << 31)) { sum->bad = 1; return; }
  if (delta > 0) {
    nodes[k] = MgNode{(uint32_t)S, (int32_t)R, (int32_t)delta, '='};
    node_alt[k] = sg.roff + (uint32_t)(R - sg.start1);
    k++; S += delta;
  }
  if (o == 'X') { nodes[k] = MgNode{(uint32_t)S, (int32_t)vp, 1, 'X'}; node_alt[k] = (uint32_t)alt_off[i]; }
  else if (o == 'I') { nodes[k] = MgNode{(uint32_t)S, (int32_t)(vp + 1), (int32_t)oplen[i], 'I'}; node_alt[k] = (uint32_t)(alt_off[i] + 1); }
  else if (o == 'D') { nodes[k] = MgNode{(uint32_t)S /* ps + 1, rpc.py:127 */, (int32_t)(vp + 1 + oplen[i]), (int32_t)oplen[i], 'D'}; node_alt[k] = 0; }
}

int mg_launch_walk(const MgWalkParams &W, cudaStream_t st) {   // -> kernels launched
  const int V = W.n_var, E = V + W.n_seg;
  const unsigned gv = (unsigned)((std::max(V + 1, W.n_seg) + 255) / 256), ge = (unsigned)((E + 1 + 255) / 256);
  k_walk_next<<<gv, 256, 0, st>>>(W.pos, W.op, W.oplen, V, W.segs, W.n_seg, W.seg_out, W.nxt, W.jump[0], W.mark, W.pred, W.sum);
  int cur = 0, launches = 6;       // next, measure, 3 x scan, nodes
  if (V > 0) {
    k_walk_seed<<<(unsigned)((W.n_seg + 255) / 256), 256, 0, st>>>(W.seg_out, W.n_seg, W.mark);
    int rounds = 1;
    while ((1ll << rounds) < (long long)V + 1) rounds++;
    for (int r = 0; r < rounds; r++) { k_walk_round<<<gv, 256, 0, st>>>(W.jump[cur], W.jump[cur ^ 1], W.mark, V); cur ^= 1; }
    k_walk_pred<<<gv, 256, 0, st>>>(W.nxt, W.mark, W.pred, W.segs, W.n_seg, W.seg_out, V);
    launches += rounds + 2;
  }
  k_walk_measure<<<ge, 256, 0, st>>>(W.pos, W.op, W.oplen, W.alt_off, W.mark, W.pred, V, W.segs, W.n_seg, W.seg_out, W.packed, W.sum);
  mg_launch_scan_i64(W.packed, W.scanned, (int64_t)E, W.scan_tmp, st);
  k_walk_nodes<<<ge, 256, 0, st>>>(W.pos, W.op, W.oplen, W.alt_off, W.mark, W.pred, V, W.segs, W.n_seg, W.seg_out, W.scanned, W.nodes, W.node_alt, W.sum);
  return launches;
}

// exception runs of the node table in haplotype coordinates: the reference's non-ACGT runs under every
// '=' node, non-ACGT bytes of inserted / substituted alleles.  Count, scan, write.
template <bool WRITE>
__global__ void __launch_bounds__(256) k_exc_map(const MgNode *__restrict__ nodes, const uint32_t *__restrict__ node_alt,
                                                 const MgWalkSummary *__restrict__ sum, int max_nodes,
                                                 const uint8_t *__restrict__ alt_pool, const MgExc *__restrict__ rexc, int n_rexc,
                                                 int64_t *cnt_or_off, MgExc *__restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= max_nodes) return;
  if (k >= sum->n_nodes) { if (!WRITE) cnt_or_off[k] = 0; return; }
  const MgNode nd = nodes[k];
  int64_t c = WRITE ? cnt_or_off[k] : 0;
  if (nd.op == '=' && nd.oplen > 0) {
    const int64_t a = (int64_t)node_alt[k], b = a + nd.oplen;   // the node's bases in the packed reference
    int lo = 0, hi = n_rexc;                                  // first run that ends after a
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if ((int64_t)rexc[mid].start + rexc[mid].len <= a) lo = mid + 1; else hi = mid;
    }
    for (int q = lo; q < n_rexc && (int64_t)rexc[q].start < b; q++) {
      const int64_t s0 = max(a, (int64_t)rexc[q].start), e0 = min(b, (int64_t)rexc[q].start + rexc[q].len);
      if (WRITE) out[c] = MgExc{(uint32_t)(nd.key + (s0 - a)), (uint32_t)(e0 - s0), rexc[q].byte, 0};
      c++;
    }
  } else if (nd.op == 'X' || nd.op == 'I') {
    const uint8_t *alt = alt_pool + node_alt[k];
    int run = -1;                                             // start of the current run of equal non-ACGT bytes
    for (int t = 0; t <= nd.oplen; t++) {
      const bool exc = t < nd.oplen && mg_base_code(alt[t]) > 3;
      if (run >= 0 && (!exc || alt[t] != alt[run])) {
        if (WRITE) out[c] = MgExc{(uint32_t)(nd.key + run), (uint32_t)(t - run), alt[run], 0};
        c++; run = -1;
      }
      if (exc && run < 0) run = t;
    }
  }
  if (!WRITE) cnt_or_off[k] = c;
}

void mg_launch_exc_count(const MgNode *nodes, const uint32_t *node_alt, const MgWalkSummary *sum, int max_nodes,
                         const uint8_t *alt_pool, const MgExc *rexc, int n_rexc, int64_t *cnt, cudaStream_t st) {
  k_exc_map<false><<<(unsigned)((max_nodes + 255) / 256), 256, 0, st>>>(nodes, node_alt, sum, max_nodes, alt_pool, rexc, n_rexc, cnt, nullptr);
}

void mg_launch_exc_write(const MgNode *nodes, const uint32_t *node_alt, const MgWalkSummary *sum, int max_nodes,
                         const uint8_t *alt_pool, const MgExc *rexc, int n_rexc, int64_t *off, MgExc *out, cudaStream_t st) {
  k_exc_map<true><<<(unsigned)((max_nodes + 255) / 256), 256, 0, st>>>(nodes, node_alt, sum, max_nodes, alt_pool, rexc, n_rexc, off, out);
}

// ------------------------------------------------------------------------------------------
// k_hap_build: one thread per 16-base haplotype word.  The non-'D' nodes tile the haplotype:
// node k covers [key[k], key[k+1]) ('D' nodes share the key of their successor and are empty).
// '=' nodes copy from the packed reference, 'X' / 'I' nodes from the alt pool.

__device__ __forceinline__ uint64_t hap_node_src(const MgNode &nd, uint32_t alt) {   // '=': offset in the packed reference; else in the alt pool
  return nd.op == '=' ? (uint64_t)alt : ((1ull << 63) | (uint64_t)alt);
}

__global__ void __launch_bounds__(256) k_hap_build(const uint32_t *__restrict__ ref, const uint8_t *__restrict__ alt_pool,
                                                   const MgNode *__restrict__ nodes, const uint32_t *__restrict__ node_alt,
                                                   int n_seg, const uint32_t *__restrict__ blk, int blk_shift, int n_blk,
                                                   uint32_t hap_len, uint32_t *__restrict__ hap, int64_t hap_words) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= hap_words) return;
  uint64_t s0 = (uint64_t)w * 16;
  if (s0 >= hap_len) { hap[w] = 0; return; }
  // last node with key <= s0 (of equal keys the later one: never the empty 'D'): the block table (built just
  // before) leaves a search over the few nodes of one 256-base block
  int k = mg_find_node(nodes, blk, blk_shift, n_blk, n_seg, (uint32_t)s0);
  MgNode nd = nodes[k];
  uint64_t seg_end = (k + 1 < n_seg) ? nodes[k + 1].key : hap_len;
  uint64_t src = hap_node_src(nd, node_alt[k]);
  uint32_t word;
  if (!(src >> 63) && s0 + 16 <= seg_end) {
    word = mg_codes16(ref, (int64_t)(src + (s0 - nd.key)));        // whole word from the reference
  } else {
    word = 0;
    for (int i = 0; i < 16; i++) {
      uint64_t s = s0 + i;
      if (s >= hap_len) break;
      while (s >= seg_end) {
        k++; nd = nodes[k];
        seg_end = (k + 1 < n_seg) ? nodes[k + 1].key : hap_len;
        src = hap_node_src(nd, node_alt[k]);
      }
      uint64_t off = s - nd.key;
      uint32_t code;
      if (src >> 63) {
        code = mg_base_code(alt_pool[(src & ~(1ull << 63)) + off]);
        if (code > 3) code = 0;
      } else {
        uint64_t r = src + off;
        code = (ref[r >> 4] >> (2 * (r & 15))) & 3u;
      }
      word |= code << (2 * i);
    }
  }
  hap[w] = word;
}

void mg_launch_hap_build(const uint32_t *ref, const uint8_t *alt_pool, const MgNode *nodes, const uint32_t *node_alt,
                         int n_nodes, const uint32_t *blk, int blk_shift, int n_blk, uint32_t hap_len, uint32_t *hap, int64_t hap_words,
                         cudaStream_t st) {
  if (hap_words == 0) return;
  k_hap_build<<<(unsigned)((hap_words + 255) / 256), 256, 0, st>>>(ref, alt_pool, nodes, node_alt, n_nodes, blk, blk_shift, n_blk, hap_len, hap, hap_words);
}

__global__ void __launch_bounds__(256) k_blk_table(const MgNode *__restrict__ nodes, int n_nodes, uint32_t *__restrict__ blk,
                                                   int n_blk, int blk_shift) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_blk) return;
  uint64_t x = (uint64_t)b << blk_shift;
  int lo = 0, hi = n_nodes - 1;                 // nodes[0].key == 0 always
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if ((uint64_t)nodes[mid].key <= x) lo = mid; else hi = mid - 1;
  }
  blk[b] = (uint32_t)lo;
}

// block table over the exception runs (MgExcView): eblk[b] = first run that ends beyond b << shift
__global__ void __launch_bounds__(256) k_eblk_table(const MgExc *__restrict__ exc, int n_exc, uint32_t *__restrict__ eblk, int n_entries, int blk_shift) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_entries) return;
  const uint64_t x = (uint64_t)b << blk_shift;
  int lo = 0, hi = n_exc;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((uint64_t)exc[mid].start + exc[mid].len <= x) lo = mid + 1; else hi = mid;
  }
  eblk[b] = (uint32_t)lo;
}

void mg_launch_eblk_table(const MgExc *exc, int n_exc, uint32_t *eblk, int n_entries, int blk_shift, cudaStream_t st) {
  k_eblk_table<<<(n_entries + 255) / 256, 256, 0, st>>>(exc, n_exc, eblk, n_entries, blk_shift);
}

void mg_launch_blk_table(const MgNode *nodes, int n_nodes, uint32_t *blk, int n_blk, int blk_shift, cudaStream_t st) {
  k_blk_table<<<(n_blk + 255) / 256, 256, 0, st>>>(nodes, n_nodes, blk, n_blk, blk_shift);
}

// ------------------------------------------------------------------------------------------
// Philox geometric gaps + grid-wide inclusive scan (illumina.py:70 in production mode)

#define GAP_PER_THREAD 8
#define GAP_THREADS 256
#define GAP_PER_BLOCK (GAP_PER_THREAD * GAP_THREADS)

__device__ __forceinline__ void gaps8(uint32_t i0, uint32_t n, double inv_log1mp, uint32_t k0, uint32_t k1, uint32_t g[8]) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    uint32_t i = i0 + 2 * q;
    MgPhilox r = mg_philox(i >> 1, 0u, 0u, MG_STREAM_GAP, k0, k1);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      double u = mg_u53(r.v[2 * h], r.v[2 * h + 1]);
      double gd = ceil(log(1.0 - u) * inv_log1mp);
      uint32_t gv = gd < 1.0 ? 1u : (gd > 4.0e9 ? 4000000000u : (uint32_t)gd);
      g[2 * q + h] = (i + h < n) ? gv : 0u;
    }
  }
}

__global__ void __launch_bounds__(GAP_THREADS) k_gap_partial(uint32_t n, double inv_log1mp, uint32_t k0, uint32_t k1,
                                                             unsigned long long *partial) {
  __shared__ unsigned long long s_w[GAP_THREADS / 32];
  uint32_t i0 = blockIdx.x * GAP_PER_BLOCK + threadIdx.x * GAP_PER_THREAD;
  uint32_t g[8];
  unsigned long long sum = 0;
  if (i0 < n) { gaps8(i0, n, inv_log1mp, k0, k1, g); for (int q = 0; q < 8; q++) sum += g[q]; }
  sum = warp_sum_u64(sum);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < GAP_THREADS / 32; w++) t += s_w[w];
    partial[blockIdx.x] = t;
  }
}

// exclusive scan of up to a few 10^5 partials by one block
__global__ void __launch_bounds__(1024) k_scan_partials_u64(unsigned long long *partial, int n) {
  __shared__ unsigned long long s_w[32];
  __shared__ unsigned long long s_carry;
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    int i = base + threadIdx.x;
    unsigned long long v = (i < n) ? partial[i] : 0, x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { unsigned long long y = __shfl_up_sync(FULL, x, d); if (lane >= d) x += y; }
    if (lane == 31) s_w[wid] = x;
    __syncthreads();
    if (wid == 0) {
      unsigned long long t = s_w[lane], xx = t;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { unsigned long long y = __shfl_up_sync(FULL, xx, d); if (lane >= d) xx += y; }
      s_w[lane] = xx - t;  // exclusive warp offsets
    }
    __syncthreads();
    unsigned long long carry = s_carry;
    unsigned long long incl = carry + s_w[wid] + x;
    if (i < n) partial[i] = incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = incl;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(GAP_THREADS) k_gap_final(uint32_t n, double inv_log1mp, uint32_t k0, uint32_t k1,
                                                           const unsigned long long *__restrict__ partial, uint32_t *__restrict__ ts_sorted) {
  __shared__ unsigned long long s_w[GAP_THREADS / 32];
  uint32_t i0 = blockIdx.x * GAP_PER_BLOCK + threadIdx.x * GAP_PER_THREAD;
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t g[8];
  unsigned long long sum = 0;
  if (i0 < n) { gaps8(i0, n, inv_log1mp, k0, k1, g); for (int q = 0; q < 8; q++) sum += g[q]; }
  else { for (int q = 0; q < 8; q++) g[q] = 0; }
  unsigned long long x = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { unsigned long long y = __shfl_up_sync(FULL, x, d); if (lane >= d) x += y; }
  if (lane == 31) s_w[wid] = x;
  __syncthreads();
  unsigned long long off = partial[blockIdx.x];
  for (int w = 0; w < wid; w++) off += s_w[w];
  unsigned long long run = off + x - sum;  // exclusive prefix of this thread
  if (i0 < n) {
#pragma unroll
    for (int q = 0; q < 8; q++) {
      run += g[q];
      if (i0 + q < n) {
        unsigned long long v = run + 1;      // ts = cumsum + p_min + 1, stored relative to p_min
        ts_sorted[i0 + q] = v > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)v;
      }
    }
  }
}

void mg_launch_gap_scan(uint32_t n, double p, uint32_t k0, uint32_t k1, uint32_t *ts_sorted, unsigned long long *partial,
                        cudaStream_t st) {
  if (n == 0) return;
  double inv = 1.0 / log(1.0 - p);
  int nb = (int)((n + GAP_PER_BLOCK - 1) / GAP_PER_BLOCK);
  k_gap_partial<<<nb, GAP_THREADS, 0, st>>>(n, inv, k0, k1, partial);
  k_scan_partials_u64<<<1, 1024, 0, st>>>(partial, nb);
  k_gap_final<<<nb, GAP_THREADS, 0, st>>>(n, inv, k0, k1, partial, ts_sorted);
}

// ------------------------------------------------------------------------------------------
// Template sampling for one candidate (illumina.py:66-76, 93-96)

struct Cand { int64_t ts_rel; int64_t te_rel; uint32_t fo; bool k1; };

// s_alias: the template-length alias table staged in shared memory (PHILOX mode, when the model has one)
__device__ __forceinline__ Cand sample_candidate(const MgUnitParams &P, const uint32_t *s_alias, uint32_t j) {
  Cand c;
  int64_t tl;
  c.fo = 0;
  if (P.mode == MG_MODE_PHILOX) {
    uint32_t i = mg_permute(j, P.n_cand, P.perm_bits, P.key_perm0, P.key_perm1);
    c.ts_rel = (int64_t)P.ts_sorted[i];
    MgPhilox r = mg_philox(j, 0u, 0u, MG_STREAM_TLEN, P.key_tlen0, P.key_tlen1);
    if (P.tlen_alias) {                                                        // illumina.py:72 by the alias method
      const uint32_t idx = r.v[0] >> 22, e = s_alias[idx];
      tl = (r.v[0] & 0x3FFFFFu) < (e >> 10) ? idx : (e & 1023u);
    } else {
      tl = mg_lower_bound_f64(P.cum_tlen, P.n_tlen, mg_u53(r.v[0], r.v[1]));
    }
    c.fo = r.v[2] & 1u;
  } else {
    c.ts_rel = P.ts_in[j] - P.p_min;
    tl = (P.mode == MG_MODE_DET) ? (int64_t)mg_lower_bound_f64(P.cum_tlen, P.n_tlen, P.u_tlen[j]) : P.tl_in[j];
  }
  if (tl < P.rlen) tl = P.rlen;                                                // illumina.py:73
  c.te_rel = c.ts_rel + tl;
  c.k1 = (c.te_rel < (int64_t)P.hap_len) && (c.ts_rel >= 0);                   // illumina.py:75
  return c;
}

__global__ void __launch_bounds__(256) k_sample(MgSampleParams S) {
  __shared__ uint32_t s_tlen[MG_TLEN_K];
  if (S.u.mode == MG_MODE_PHILOX && S.u.tlen_alias)
    for (int i = threadIdx.x; i < MG_TLEN_K; i += blockDim.x) s_tlen[i] = S.u.tlen_alias[i];
  __syncthreads();
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < S.u.n_cand; j += gridDim.x * blockDim.x) {
    Cand c = sample_candidate(S.u, s_tlen, j);
    S.ts_out[j] = c.ts_rel + S.u.p_min;
    S.te_out[j] = c.k1 ? c.te_rel + S.u.p_min : -1;
    S.fo_out[j] = (int8_t)c.fo;
  }
}

void mg_launch_sample(const MgSampleParams &P, cudaStream_t st) {
  if (P.u.n_cand == 0) return;
  int grid = (int)((P.u.n_cand + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  k_sample<<<grid, 256, 0, st>>>(P);
}

// ------------------------------------------------------------------------------------------
// k_unit_emit

struct Agg { unsigned long long c1, c2, by; };

#define DESC_FLAG(x) ((uint32_t)((x) >> 62))
#define DESC_MASK62 ((1ull << 62) - 1ull)

// Exclusive prefix of (c1, c2, bytes) over all tiles before `tile` (decoupled look-back), computed
// by one whole warp; every lane returns the same sums.  One round reads a window of LOOKBACK_WIN
// descriptors (LOOKBACK_WIN / 32 per lane, all loads in flight at once) and stops at the nearest
// inclusive one.  The window bounds how fast inclusive prefixes can propagate: about one window of tiles
// per L2 round trip.  At 32 tiles that is close to the rate at which tiles finish on 148 SMs.
#define LOOKBACK_WIN 128
__device__ Agg tile_lookback(const MgUnitParams &P, int tile, int lane) {
  constexpr int Q = LOOKBACK_WIN / 32;
  Agg ex = {0, 0, 0};
  int idx = tile - 1;
  while (true) {
    unsigned long long a[Q], b[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) {
      const int t = idx - 32 * q - lane;
      a[q] = 2ull << 62; b[q] = 2ull << 62;   // tiles before 0 behave like an all-zero inclusive prefix
      if (t >= 0) { a[q] = ld_vol64(P.descA + t); b[q] = ld_vol64(P.descB + t); }
    }
#pragma unroll
    for (int q = 0; q < Q; q++) {
      const int t = idx - 32 * q - lane;
      while (t >= 0 && (DESC_FLAG(a[q]) == 0 || DESC_FLAG(a[q]) != DESC_FLAG(b[q]))) {
        a[q] = ld_vol64(P.descA + t); b[q] = ld_vol64(P.descB + t);
      }
    }
    __syncwarp();
    int stop = LOOKBACK_WIN;   // window position (32 q + lane) of the nearest inclusive descriptor
#pragma unroll
    for (int q = Q - 1; q >= 0; q--) {
      const uint32_t pm = __ballot_sync(FULL, DESC_FLAG(a[q]) == 2);
      if (pm) stop = 32 * q + __ffs(pm) - 1;
    }
    unsigned long long c1 = 0, c2 = 0, by = 0;
#pragma unroll
    for (int q = 0; q < Q; q++) {
      if (32 * q + lane <= stop) {   // (the all-zero stand-ins before tile 0 add nothing)
        c1 += (a[q] >> 31) & 0x7FFFFFFFull; c2 += a[q] & 0x7FFFFFFFull; by += b[q] & DESC_MASK62;
      }
    }
    ex.c1 += warp_sum_u64(c1); ex.c2 += warp_sum_u64(c2); ex.by += warp_sum_u64(by);
    if (stop < LOOKBACK_WIN) break;
    idx -= LOOKBACK_WIN;
  }
  return ex;
}

// ---- k_unit_plan ---------------------------------------------------------------------------
// Phase 1 of a unit: one candidate per thread (sampling, te < p_max / N filter, node lookup, record
// size), block scan, decoupled look-back, and one 32-byte MgPlan per KEPT template at its final
// rank.  Small per-thread state: runs at high occupancy, which hides the dependent L2 loads of the
// node / template-start gathers.
//
// One block barrier per tile, and no warp waits for a look-back right after its tile's aggregate went
// out.  Iteration k of a CTA does the candidates of its tile T_k; warp 0 then does the look-back of
// T_{k-1}, whose aggregate went out one iteration earlier.  After the barrier every thread writes its
// plan of T_{k-1} (parked in shared memory since then) and thread 0 publishes T_k's aggregate.  So
// the other warps spend the look-back on their next candidates, and a look-back starts a whole tile
// of work after the aggregates it reads were due.  The next tile is claimed one iteration ahead,
// off the barrier.
//
// Deadlock freedom: tiles are claimed from an atomic counter, so every tile below a claimed one has
// been claimed by a CTA that is running (a CTA exits only after the plans of all its tiles).  The
// look-back of a tile T waits only for aggregates of tiles below T.  The aggregate of a tile U goes
// out once its CTA has done the look-back of its previous tile, which is below U.  By induction on the
// tile index every look-back ends, whichever CTAs are resident.
#define PLAN_THREADS 256

// 40 registers, six CTAs per SM (the look-back's window spills a few words to L1 at that bound; eight CTAs at
// 32 registers spill 68 bytes and measured slower)
__global__ void __launch_bounds__(PLAN_THREADS, 6) k_unit_plan(const __grid_constant__ MgUnitParams P) {
  __shared__ uint32_t s_tlen[MG_TLEN_K];
  // each thread's candidate of T_{k-1}: {xa, xb, n0a, n0b}, {dn, fo << 31 | ta << 30 | tb << 29 | sz}, and its
  // exclusive (ec, es) inside the tile
  __shared__ uint4 s_hold[2][PLAN_THREADS];
  __shared__ uint2 s_hold2[2][PLAN_THREADS], s_ex[PLAN_THREADS];
  __shared__ uint32_t s_wc[2][PLAN_THREADS / 32], s_ws[2][PLAN_THREADS / 32];
  __shared__ unsigned long long s_base[2][3];
  __shared__ uint32_t s_tile[2];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int L = P.rlen;
  if (P.mode == MG_MODE_PHILOX && P.tlen_alias) {
#pragma unroll 1
    for (int i = t; i < MG_TLEN_K; i += PLAN_THREADS) s_tlen[i] = P.tlen_alias[i];
  }
  if (t == 0) s_tile[0] = atomicAdd(P.tile_counter, 1u);
  __syncthreads();
  int tile = (int)s_tile[0], prev = -1;
  uint32_t prev_c1 = 0, prev_c2 = 0, prev_sz = 0;       // aggregate of T_{k-1}
#pragma unroll 1
  for (int k = 0;; k++) {
    const int cur = k & 1;
    const bool live = tile < P.n_tiles;
    if (t == 0 && live) s_tile[cur ^ 1] = atomicAdd(P.tile_counter, 1u);
    const uint32_t j = (uint32_t)tile * PLAN_THREADS + t;
    bool k1 = false, k2 = false, ta = false, tb = false;
    uint32_t xa = 0, xb = 0, fo = 0, sz = 0;
    int n0a = 0, n1a = 0, n0b = 0, n1b = 0;
    if (live && j < P.n_cand) {
      Cand c = sample_candidate(P, s_tlen, j);
      k1 = c.k1; fo = c.fo;
      if (k1) {
        xa = (uint32_t)c.ts_rel; xb = (uint32_t)(c.te_rel - L);                 // illumina.py:95-96
        k2 = true;
        if (P.n_exc) {                                                           // readgenerate.py:204
          const MgExcView ev = {P.exc, P.eblk, P.blk_shift, P.n_blk};
          const int na = mg_count_N(ev, P.n_exc, xa, L, ta), nb = mg_count_N(ev, P.n_exc, xb, L, tb);
          k2 = na <= 2 && nb <= 2;
        }
        if (k2) {
          n0a = mg_find_node(P.nodes, P.blk, P.blk_shift, P.n_blk, P.n_nodes, xa);
          n1a = mg_last_node(P.nodes, n0a, P.n_nodes, xa, L);
          n0b = mg_find_node(P.nodes, P.blk, P.blk_shift, P.n_blk, P.n_nodes, xb);
          n1b = mg_last_node(P.nodes, n0b, P.n_nodes, xb, L);
          sz = (uint32_t)P.qn_len + mg_read_fields_len(P.nodes, n0a, n1a, xa, L, P.L_nd) +
               mg_read_fields_len(P.nodes, n0b, n1b, xb, L, P.L_nd) + 2u * (uint32_t)L + 5u;
        }
      }
    }
    s_hold[cur][t] = make_uint4(xa, xb, (uint32_t)n0a, (uint32_t)n0b);
    s_hold2[cur][t] = make_uint2((uint32_t)(n1a - n0a) | ((uint32_t)(n1b - n0b) << 16),
                                 (fo << 31) | ((ta ? 1u : 0u) << 30) | ((tb ? 1u : 0u) << 29) | sz);
    // warp scans of (k1 | k2 << 16, sz) over T_k
    const uint32_t cpk = (k1 ? 1u : 0u) | (k2 ? 0x10000u : 0u);
    const uint32_t ic = warp_incl_scan_u32(cpk, lane), is = warp_incl_scan_u32(sz, lane);
    if (lane == 31) { s_wc[cur][wid] = ic; s_ws[cur][wid] = is; }
    // warp 0: exclusive prefix of T_{k-1}, and its inclusive descriptor
    if (wid == 0 && prev >= 0) {
      Agg ex = {0, 0, 0};
      if (prev > 0) ex = tile_lookback(P, prev, lane);
      if (lane == 0) {
        const unsigned long long i1 = ex.c1 + prev_c1, i2 = ex.c2 + prev_c2, ib = ex.by + prev_sz;
        if (prev > 0) {                                                          // tile 0 went out inclusive
          st_vol64(P.descA + prev, (2ull << 62) | (i1 << 31) | i2);
          st_vol64(P.descB + prev, (2ull << 62) | ib);
        }
        s_base[cur ^ 1][0] = ex.c1; s_base[cur ^ 1][1] = ex.c2; s_base[cur ^ 1][2] = ex.by;
        if (prev == P.n_tiles - 1) { P.totals[0] = i1; P.totals[1] = i2; P.totals[2] = ib + mg_digit_sum(i2); }
      }
    }
    __syncthreads();
    // the plans of T_{k-1}
    if (prev >= 0) {
      const uint2 h1 = s_hold2[cur ^ 1][t];
      if (h1.y & 0x1FFFFFFFu) {                                                  // sz != 0: kept
        const uint4 h0 = s_hold[cur ^ 1][t];
        const uint2 ex = s_ex[t];
        const unsigned long long base1 = s_base[cur ^ 1][0], base2 = s_base[cur ^ 1][1];
        const unsigned long long rank = base2 + (ex.x >> 16);                    // cnt - 1, readgenerate.py:209
        // the serial's digits change the record size: offset = scanned bytes + sum of digits of 1..rank
        const unsigned long long off = s_base[cur ^ 1][2] + ex.y + mg_digit_sum(rank);
        const uint32_t my_fo = (P.mode == MG_MODE_PHILOX) ? h1.y >> 31 : (uint32_t)(P.fo_in[base1 + (ex.x & 0xFFFFu)] & 1);   // illumina.py:93
        MgPlan pl;
        pl.xa = h0.x; pl.xb = h0.y; pl.n0a = (int32_t)h0.z; pl.n0b = (int32_t)h0.w;
        pl.dn = h1.x;
        pl.fo_sz = (my_fo << 31) | ((h1.y & 0x7FFFFFFFu) + (uint32_t)mg_ndigits32((uint32_t)(rank + 1)));
        pl.off = off;
        P.plan[rank] = pl;
      }
    }
    if (!live) break;
    // T_k: offsets inside the tile, its aggregate; tile 0 has its inclusive prefix already
    uint32_t oc = 0, os = 0, tc = 0, ts_ = 0;
#pragma unroll
    for (int w = 0; w < PLAN_THREADS / 32; w++) {
      if (w < wid) { oc += s_wc[cur][w]; os += s_ws[cur][w]; }
      tc += s_wc[cur][w]; ts_ += s_ws[cur][w];
    }
    const uint32_t ec = oc + ic - cpk, es = os + is - sz;   // exclusive
    prev_c1 = tc & 0xFFFFu; prev_c2 = tc >> 16; prev_sz = ts_;
    if (t == 0) {
      const unsigned long long fl = tile == 0 ? 2ull << 62 : 1ull << 62;
      st_vol64(P.descA + tile, fl | ((unsigned long long)prev_c1 << 31) | prev_c2);
      st_vol64(P.descB + tile, fl | prev_sz);
    }
    s_ex[t] = make_uint2(ec, es);
    prev = tile;
    tile = (int)s_tile[cur ^ 1];
  }
}

void mg_launch_plan(const MgUnitParams &P, cudaStream_t st) {
  if (P.n_tiles == 0) return;
  // as many CTAs as are resident at once: a later one would find the tile counter exhausted
  static const int resident = [] {
    int dev = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_unit_plan, PLAN_THREADS, 0);
    return std::max(1, sms * per_sm);
  }();
  k_unit_plan<<<std::min(P.n_tiles, resident), PLAN_THREADS, 0, st>>>(P);
}

// ---- k_batch_plan --------------------------------------------------------------------------
// Phase 1 for a BATCH of small units (an exome-style BED: thousands of regions of a few kb): ONE CTA per
// unit does what k_gap_* + k_unit_plan do for a big unit -- geometric gaps and their scan in shared
// memory, sampling, filters, node lookup, sizes, block scans with a running carry -- so a whole batch is
// one launch.  Same draws as the one-unit path (unit_keys), hence the same bytes.
__global__ void __launch_bounds__(PLAN_THREADS) k_batch_plan(const __grid_constant__ MgUnitParams P) {
  __shared__ uint32_t s_ts[MG_BATCH_MAXC];
  __shared__ uint32_t s_tlen[MG_TLEN_K];
  __shared__ unsigned long long s_w64[PLAN_THREADS / 32];
  __shared__ uint32_t s_wc[PLAN_THREADS / 32], s_ws[PLAN_THREADS / 32];
  __shared__ unsigned long long s_carry[3];          // te survivors, kept, bytes (without the serials' digits) so far
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int L = P.rlen;
  const MgBatchUnit U = P.bunits[blockIdx.x];
  const uint32_t n = U.n_cand;
  const MgUnitKeys K = mg_unit_keys(U.seed, n);
  if (P.mode == MG_MODE_PHILOX) {
    if (P.tlen_alias) for (int i = t; i < MG_TLEN_K; i += PLAN_THREADS) s_tlen[i] = P.tlen_alias[i];
    // template starts: cumulative geometric gaps (illumina.py:70), eight per thread, block scan
    uint32_t g[8];
    unsigned long long sum = 0;
    const uint32_t i0 = (uint32_t)t * 8u;
    if (i0 < n) { gaps8(i0, n, P.inv_log1mp, K.gap0, K.gap1, g); for (int q = 0; q < 8; q++) sum += g[q]; }
    else { for (int q = 0; q < 8; q++) g[q] = 0; }
    unsigned long long x = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { unsigned long long y = __shfl_up_sync(FULL, x, d); if (lane >= d) x += y; }
    if (lane == 31) s_w64[wid] = x;
    __syncthreads();
    unsigned long long run = x - sum;
    for (int w = 0; w < wid; w++) run += s_w64[w];
    for (int q = 0; q < 8; q++) {
      run += g[q];
      if (i0 + q < n) { const unsigned long long v = run + 1; s_ts[i0 + q] = v > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)v; }
    }
  }
  if (t == 0) { s_carry[0] = 0; s_carry[1] = 0; s_carry[2] = 0; }
  __syncthreads();
  for (uint32_t c0 = 0; c0 < n; c0 += PLAN_THREADS) {
    const uint32_t j = c0 + t;
    bool k1 = false, k2 = false, ta = false, tb = false;
    uint32_t xa = 0, xb = 0, fo = 0, sz = 0;
    int n0a = 0, n1a = 0, n0b = 0, n1b = 0;
    if (j < n) {
      int64_t ts_rel, tl;
      if (P.mode == MG_MODE_PHILOX) {
        const uint32_t i = mg_permute(j, n, K.perm_bits, K.perm0, K.perm1);
        ts_rel = (int64_t)s_ts[i];
        const MgPhilox r = mg_philox(j, 0u, 0u, MG_STREAM_TLEN, K.tlen0, K.tlen1);
        if (P.tlen_alias) { const uint32_t idx = r.v[0] >> 22, e = s_tlen[idx]; tl = (r.v[0] & 0x3FFFFFu) < (e >> 10) ? idx : (e & 1023u); }
        else tl = mg_lower_bound_f64(P.cum_tlen, P.n_tlen, mg_u53(r.v[0], r.v[1]));
        fo = r.v[2] & 1u;
      } else {
        ts_rel = P.ts_in[U.draw_off + j] - U.p_min;
        tl = mg_lower_bound_f64(P.cum_tlen, P.n_tlen, P.u_tlen[U.draw_off + j]);
      }
      if (tl < L) tl = L;                                                       // illumina.py:73
      const int64_t te_rel = ts_rel + tl;
      k1 = te_rel < (int64_t)U.hap_len && ts_rel >= 0;                           // illumina.py:75
      if (k1) {
        xa = U.x0 + (uint32_t)ts_rel; xb = U.x0 + (uint32_t)(te_rel - L);       // illumina.py:95-96, in the concatenated haplotype
        k2 = true;
        if (P.n_exc) {                                                           // readgenerate.py:204
          const MgExcView ev = {P.exc, P.eblk, P.blk_shift, P.n_blk};
          const int na = mg_count_N(ev, P.n_exc, xa, L, ta), nb = mg_count_N(ev, P.n_exc, xb, L, tb);
          k2 = na <= 2 && nb <= 2;
        }
        if (k2) {
          n0a = mg_find_node(P.nodes, P.blk, P.blk_shift, P.n_blk, P.n_nodes, xa);
          n1a = mg_last_node(P.nodes, n0a, P.n_nodes, xa, L);
          n0b = mg_find_node(P.nodes, P.blk, P.blk_shift, P.n_blk, P.n_nodes, xb);
          n1b = mg_last_node(P.nodes, n0b, P.n_nodes, xb, L);
          sz = U.qn_len + mg_read_fields_len(P.nodes, n0a, n1a, xa, L, P.L_nd) + mg_read_fields_len(P.nodes, n0b, n1b, xb, L, P.L_nd) + 2u * (uint32_t)L + 5u;
        }
      }
    }
    const uint32_t cpk = (k1 ? 1u : 0u) | (k2 ? 0x10000u : 0u);
    const uint32_t ic = warp_incl_scan_u32(cpk, lane), is = warp_incl_scan_u32(sz, lane);
    if (lane == 31) { s_wc[wid] = ic; s_ws[wid] = is; }
    __syncthreads();
    uint32_t oc = 0, os = 0, tc = 0, ts_ = 0;
#pragma unroll
    for (int w = 0; w < PLAN_THREADS / 32; w++) {
      if (w < wid) { oc += s_wc[w]; os += s_ws[w]; }
      tc += s_wc[w]; ts_ += s_ws[w];
    }
    const uint32_t ec = oc + ic - cpk, es = os + is - sz;
    const unsigned long long base1 = s_carry[0], base2 = s_carry[1], baseb = s_carry[2];
    if (k2) {
      const unsigned long long rank = base2 + (ec >> 16);                        // cnt - 1, readgenerate.py:209
      const unsigned long long off = baseb + es + mg_digit_sum(rank);
      const uint32_t my_fo = (P.mode == MG_MODE_PHILOX) ? fo : (uint32_t)(P.fo_in[U.draw_off + base1 + (ec & 0xFFFFu)] & 1);   // illumina.py:93
      MgPlan pl;
      pl.xa = xa; pl.xb = xb; pl.n0a = n0a; pl.n0b = n0b;
      pl.dn = (uint32_t)(n1a - n0a) | ((uint32_t)(n1b - n0b) << 16);
      pl.fo_sz = (my_fo << 31) | ((ta ? 1u : 0u) << 30) | ((tb ? 1u : 0u) << 29) | (sz + (uint32_t)mg_ndigits32((uint32_t)(rank + 1)));
      pl.off = off | ((unsigned long long)blockIdx.x << 40);                     // bytes inside the unit (< 2^40) | the unit
      P.plan[U.plan_off + rank] = pl;
    }
    __syncthreads();
    if (t == 0) { s_carry[0] = base1 + (tc & 0xFFFFu); s_carry[1] = base2 + (tc >> 16); s_carry[2] = baseb + ts_; }
    __syncthreads();
  }
  if (t == 0) {
    P.unit_te[blockIdx.x] = (long long)s_carry[0];
    P.unit_kept[blockIdx.x] = (long long)s_carry[1];
    P.unit_bytes[blockIdx.x] = (long long)(s_carry[2] + mg_digit_sum(s_carry[1]));
  }
}

void mg_launch_batch_plan(const MgUnitParams &P, cudaStream_t st) {
  if (P.n_bunits == 0) return;
  k_batch_plan<<<P.n_bunits, PLAN_THREADS, 0, st>>>(P);
}

// ---- k_unit_emit ---------------------------------------------------------------------------
// Phase 2: one WARP owns 32 consecutive kept templates (every lane busy), formats their records
// into its own shared-memory stage and hands the 16-byte aligned body of the byte range to the bulk
// copy engine (cp.async.bulk shared -> global, L2 evict-first); only the unaligned head / tail bytes
// go through the load/store pipe.  No block barrier and no scan: placement was decided by k_unit_plan.

// a record larger than the whole stage (only possible with absurdly long CIGARs): straight to
// global memory through generic pointers, streaming sequence source; cold and out of line
template <int CORRUPT, class STR>
__device__ __noinline__ void emit_oversize(uint8_t *dst, uint32_t qlen, const MgUnitParams &P, const STR &str, const MgCorruptCtx &cor,
                                           unsigned long long cnt, MgReadRef first, MgReadRef second, MgReadRef mine, int f) {
  const int L = P.rlen;
  MgSeqSrc<0, const uint32_t *> S;
  S.load(P.hap, mine.x, L, mine.strand);
  if constexpr (CORRUPT) {
    mg_emit_frame_qname<MgGenericSpace>(dst, P.qn, str, (uint32_t)cnt, P.nodes, first, second, L);
    mg_emit_frame_seps<MgGenericSpace>(dst, qlen, L);
    mg_emit_seq_corrupt<MgGenericSpace, CORRUPT == 2>(dst + qlen + 1, dst + qlen + 1 + L + 3, S, MgExcView{P.exc, P.eblk, P.blk_shift, P.n_blk}, P.n_exc, cor, (uint32_t)(cnt - 1), (uint32_t)f, (uint32_t)f);
  } else {
    MgStream<MgGenericSpace> ws;
    mg_emit_record<MgGenericSpace>(ws, dst, P.qn, str, (uint32_t)cnt, P.nodes, first, second, S);
    ws.end();
    if (P.n_exc) mg_patch_exc<MgGenericSpace>(dst + (qlen + 1), MgExcView{P.exc, P.eblk, P.blk_shift, P.n_blk}, P.n_exc, S.hap, S.x, L, S.strand);
  }
}

__device__ __forceinline__ void bulk_store(uint8_t *gdst, uint32_t ssrc, uint32_t bytes, unsigned long long policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
               :: "l"(gdst), "r"(ssrc), "r"(bytes), "l"(policy) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

// CORRUPT: 0 = perfect reads; 1 / 2 = fused corruption with 8- / 9-bit outcome codes
// BATCH: the templates of MANY small units (k_batch_plan) in one launch: a lane finds its unit in the
// prefix of kept templates, takes the unit's strings and corruption key from the unit table and its byte
// offset from the prefix of the units' bytes
template <int MAXW, int CORRUPT, bool BATCH = false>
__global__ void __launch_bounds__(MG_CTA, 4) k_unit_emit(const __grid_constant__ MgUnitParams P) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  uint8_t *stage = smem + (uint32_t)wid * (uint32_t)(P.stage_cap + 16);      // this warp's stage
  // its shared-window address, pinned in a register (the compiler would otherwise rebuild it at every store)
  uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
  asm volatile("" : "+r"(stage_s));
  const int L = P.rlen;
  const MgExcView ev = {P.exc, P.eblk, P.blk_shift, P.n_blk};
  const unsigned long long n_kept = BATCH ? (unsigned long long)P.kept_base[P.n_bunits] : P.totals[1];
  const unsigned long long n_bytes = BATCH ? (unsigned long long)P.byte_base[P.n_bunits] : P.totals[2];
  if (n_bytes > P.cap) { if (t == 0 && blockIdx.x == 0) P.totals[3] = 1ull; return; }   // host regrows and relaunches
  if (n_kept == 0) return;
  unsigned long long policy = 0;
  if (P.bulk) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));   // the FASTQ bytes must not push the haplotype out of L2
  bool in_flight = false;          // a bulk copy may still be reading this warp's stage
  const unsigned long long n_wt = (n_kept + 31) / 32;
  for (unsigned long long wt = (unsigned long long)blockIdx.x * (MG_CTA / 32) + wid; wt < n_wt; wt += (unsigned long long)gridDim.x * (MG_CTA / 32)) {
    const unsigned long long grank = wt * 32 + lane;
    const bool active = grank < n_kept;
    unsigned long long rank = active ? grank : n_kept - 1;      // serial - 1 within the unit
    MgPlan pl;
    const MgBatchUnit *U = nullptr;
    if constexpr (BATCH) {
      int ulo = 0, uhi = P.n_bunits - 1;                        // the last unit whose first template is <= rank
      while (ulo < uhi) { const int mid = (ulo + uhi + 1) >> 1; if ((unsigned long long)P.kept_base[mid] <= rank) ulo = mid; else uhi = mid - 1; }
      U = P.bunits + ulo;
      rank -= (unsigned long long)P.kept_base[ulo];
      pl = P.plan[U->plan_off + rank];
      pl.off = (unsigned long long)P.byte_base[ulo] + (pl.off & ((1ull << 40) - 1ull));
    } else {
      pl = P.plan[rank];
    }
    const uint32_t rec = pl.fo_sz & 0x1FFFFFFFu, my_fo = pl.fo_sz >> 31;
    // exception runs (N, IUPAC, lower case) are searched only for the reads the plan flagged
    const int ne_a = (pl.fo_sz & (1u << 30)) ? P.n_exc : 0, ne_b = (pl.fo_sz & (1u << 29)) ? P.n_exc : 0;
    const int ne_first = my_fo ? ne_b : ne_a, ne_second = my_fo ? ne_a : ne_b;
    // the next tile's plan records, and the first node of each of this tile's reads, on their way into L2 / L1
    {
      const unsigned long long nr = grank + (unsigned long long)gridDim.x * MG_CTA;
      if (!BATCH && nr < n_kept) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.plan + nr));
      asm volatile("prefetch.global.L1 [%0];" :: "l"(P.nodes + pl.n0a));
      asm volatile("prefetch.global.L1 [%0];" :: "l"(P.nodes + pl.n0b));
    }
    const uint32_t qlen = rec - (2u * (uint32_t)L + 5u);
    const unsigned long long cnt = rank + 1;
    MgReadRef ra, rb;
    ra.x = pl.xa; ra.n0 = pl.n0a; ra.n1 = pl.n0a + (int)(pl.dn & 0xFFFFu); ra.strand = 0;
    rb.x = pl.xb; rb.n0 = pl.n0b; rb.n1 = pl.n0b + (int)(pl.dn >> 16); rb.strand = 1;
    // reads[fo] = mate (readgenerate.py:207): file f holds mate 0 iff fo == f
    const MgReadRef first = my_fo ? rb : ra, second = my_fo ? ra : rb;
    const unsigned long long my_end = active ? pl.off + rec : 0ull;
    // records are emitted in batches that fit the stage (normally the whole warp tile at once)
    int lo = 0;
    const int n_act = (int)((n_kept - wt * 32 < 32ull) ? (n_kept - wt * 32) : 32ull);
    while (lo < n_act) {
      const unsigned long long goff = __shfl_sync(FULL, pl.off, lo);            // byte offset of the batch in each file
      const uint32_t pad = (uint32_t)(goff & 15);
      const bool fits = active && lane >= lo && (my_end - goff + pad) <= (unsigned long long)P.stage_cap;
      int hi = lo + __popc(__ballot_sync(FULL, fits));                           // fits is monotone in the lane index
      if (hi == lo) hi = lo + 1;                                                 // a single oversize record: see below
      const unsigned long long gend = __shfl_sync(FULL, my_end, hi - 1);
      const uint32_t batch_bytes = (uint32_t)(gend - goff);
      const bool oversize = (pad + batch_bytes) > (uint32_t)P.stage_cap;         // only a record larger than the stage
      const bool mine = active && lane >= lo && lane < hi;
      const uint32_t dst = stage_s + pad + (uint32_t)(pl.off - goff);
      MgSeqSrc<MAXW, const uint32_t *> S;
      // software pipeline with ONE load site: iteration f emits file f from the window loaded in
      // iteration f-1 and then starts the loads of file f+1 (they overlap with the copy-out)
      for (int f = -1; f < 2; f++) {
        if (f >= 0 && P.out[f] == nullptr) continue;
        // the stage keeps the qname (and, for perfect reads, the quality line) of the first file
        // written in place: the other file only rewrites its L sequence (and quality) bytes
        const bool full = (f == 0) || (P.out[0] == nullptr);
        const int ne_f = f ? ne_second : ne_first;           // file f holds `second` iff f == 1
        if (f >= 0 && !oversize) {
          if (in_flight) {                                  // the previous copy must have read the stage
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            __syncwarp();
            in_flight = false;
          }
          if constexpr (CORRUPT) {
            if (full) {
              if (mine) {
                if constexpr (BATCH) mg_emit_frame_qname<MgSharedSpace>(dst, P.qn, *U, (uint32_t)cnt, P.nodes, first, second, L);
                else mg_emit_frame_qname<MgSharedSpace>(dst, P.qn, P.qn, (uint32_t)cnt, P.nodes, first, second, L);
              }
              __syncwarp();                                 // every first word is stored: now the bytes that share a word with a neighbour
              if (mine) mg_emit_frame_seps<MgSharedSpace>(dst, qlen, L);
            }
            if (mine) {
              if constexpr (BATCH) {
                MgCorruptCtx cor = P.cor;
                cor.k1 = U->seed ^ 0x636f7231u;              // the unit's corruption key, as mg_unit_generate derives it
                mg_emit_seq_corrupt<MgSharedSpace, CORRUPT == 2>(dst + qlen + 1, dst + qlen + 1 + L + 3, S, ev, ne_f, cor, (uint32_t)rank, (uint32_t)f, (uint32_t)f);
              } else {
                mg_emit_seq_corrupt<MgSharedSpace, CORRUPT == 2>(dst + qlen + 1, dst + qlen + 1 + L + 3, S, ev, ne_f, P.cor, (uint32_t)rank, (uint32_t)f, (uint32_t)f);
              }
            }
          } else {
            if (full) {
              MgStream<MgSharedSpace> ws;
              if (mine) {
                if constexpr (BATCH) mg_emit_record<MgSharedSpace>(ws, dst, P.qn, *U, (uint32_t)cnt, P.nodes, first, second, S);
                else mg_emit_record<MgSharedSpace>(ws, dst, P.qn, P.qn, (uint32_t)cnt, P.nodes, first, second, S);
              }
              __syncwarp();
              if (mine) {
                ws.end();
                if (ne_f) mg_patch_exc<MgSharedSpace>(dst + (qlen + 1), ev, ne_f, S.hap, S.x, L, S.strand);
              }
            } else if (mine) {
              mg_rewrite_seq<MgSharedSpace>(dst + qlen + 1, S, ev, ne_f);
            }
          }
        } else if (f >= 0 && mine) {
          if constexpr (BATCH) {
            MgCorruptCtx cor = P.cor;
            cor.k1 = U->seed ^ 0x636f7231u;
            emit_oversize<CORRUPT>(P.out[f] + pl.off, qlen, P, *U, cor, cnt, first, second, f ? second : first, f);
          } else {
            emit_oversize<CORRUPT>(P.out[f] + pl.off, qlen, P, P.qn, P.cor, cnt, first, second, f ? second : first, f);
          }
        }
        if (mine && f < 1) {
          const MgReadRef nxt = (f < 0 && P.out[0] != nullptr) ? first : second;
          S.load(P.hap, nxt.x, L, nxt.strand);
        }
        if (f < 0 || oversize) continue;
        // copy-out: smem and global share the same 16-byte phase (pad)
        uint8_t *gdst = P.out[f] + goff;
        const uint8_t *ssrc = stage + pad;
        uint32_t head = (16u - pad) & 15u;
        if (head > batch_bytes) head = batch_bytes;
        const uint32_t nvec = (batch_bytes - head) >> 4;
        const uint32_t done = head + (nvec << 4);
        if (P.bulk) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // this thread's stage writes -> visible to the copy engine
          __syncwarp();
          if (lane == 0 && nvec) bulk_store(gdst + head, stage_s + pad + head, nvec << 4, policy);
          in_flight = nvec != 0;
          if ((uint32_t)lane < head) gdst[lane] = ssrc[lane];
          if (done + lane < batch_bytes) gdst[done + lane] = ssrc[done + lane];
        } else {
          __syncwarp();
          if ((uint32_t)lane < head) gdst[lane] = ssrc[lane];
          const uint4 *sv = reinterpret_cast<const uint4 *>(ssrc + head);
          uint4 *gv = reinterpret_cast<uint4 *>(gdst + head);
          for (uint32_t v = lane; v < nvec; v += 32) __stcs(gv + v, sv[v]);   // streaming stores
          if (done + lane < batch_bytes) gdst[done + lane] = ssrc[done + lane];
          __syncwarp();
        }
      }
      lo = hi;
    }
  }
  // bulk copies still reading shared memory must finish before the CTA's shared memory is released
  if (P.bulk && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

typedef void (*unit_kernel_t)(const MgUnitParams);

static unit_kernel_t unit_kernel(int L, int corrupt) {   // corrupt: 0, or 1 / 2 = fused corruption with 8- / 9-bit outcome codes
  // register window: MAXW - 1 >= ceil((15 + L) / 16)
  if (L <= 161) return corrupt == 0 ? k_unit_emit<12, 0> : corrupt == 1 ? k_unit_emit<12, 1> : k_unit_emit<12, 2>;
  if (L <= 305) return corrupt == 0 ? k_unit_emit<21, 0> : corrupt == 1 ? k_unit_emit<21, 1> : k_unit_emit<21, 2>;
  return corrupt == 0 ? k_unit_emit<0, 0> : corrupt == 1 ? k_unit_emit<0, 1> : k_unit_emit<0, 2>;
}

// -> CTAs to launch (SMs x resident CTAs per SM), or 0 when the staging area does not fit this device
int mg_unit_grid(int L, int corrupt, int stage_cap, int *smem_bytes) {
  int smem = (MG_CTA / 32) * (stage_cap + 16);
  if (const char *x = getenv("MG_EXTRA_SMEM")) smem += atoi(x);   // occupancy experiments only
  *smem_bytes = smem;
  unit_kernel_t k = unit_kernel(L, corrupt);
  int per_sm = 0, dev = 0, sms = 0, optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (smem > optin) return 0;
  if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, MG_CTA, smem);
  if (per_sm < 1) per_sm = 1;
  return sms * per_sm;
}

void mg_launch_unit(const MgUnitParams &P, int grid, int smem_bytes, cudaStream_t st) {
  if (P.n_tiles == 0) return;
  unit_kernel(P.rlen, P.corrupt ? 1 + P.cor.code9 : 0)<<<grid, MG_CTA, smem_bytes, st>>>(P);
}

static unit_kernel_t batch_kernel(int L, int corrupt) {
  if (L <= 161) return corrupt == 0 ? k_unit_emit<12, 0, true> : corrupt == 1 ? k_unit_emit<12, 1, true> : k_unit_emit<12, 2, true>;
  if (L <= 305) return corrupt == 0 ? k_unit_emit<21, 0, true> : corrupt == 1 ? k_unit_emit<21, 1, true> : k_unit_emit<21, 2, true>;
  return corrupt == 0 ? k_unit_emit<0, 0, true> : corrupt == 1 ? k_unit_emit<0, 1, true> : k_unit_emit<0, 2, true>;
}

int mg_batch_grid(int L, int corrupt, int stage_cap, int *smem_bytes) {
  const int smem = (MG_CTA / 32) * (stage_cap + 16);
  *smem_bytes = smem;
  unit_kernel_t k = batch_kernel(L, corrupt);
  int per_sm = 0, dev = 0, sms = 0, optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (smem > optin) return 0;
  if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, MG_CTA, smem);
  if (per_sm < 1) per_sm = 1;
  return sms * per_sm;
}

void mg_launch_batch_emit(const MgUnitParams &P, int grid, int smem_bytes, cudaStream_t st) {
  if (P.n_bunits == 0) return;
  batch_kernel(P.rlen, P.corrupt ? 1 + P.cor.code9 : 0)<<<grid, MG_CTA, smem_bytes, st>>>(P);
}

// ------------------------------------------------------------------------------------------
// generic exclusive scan of int64 (out[n] = total)

#define SCAN_THREADS 256
#define SCAN_PER_THREAD 4
#define SCAN_PER_BLOCK (SCAN_THREADS * SCAN_PER_THREAD)

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(const int64_t *__restrict__ in, int64_t n, unsigned long long *partial) {
  __shared__ unsigned long long s_w[SCAN_THREADS / 32];
  int64_t i0 = (int64_t)blockIdx.x * SCAN_PER_BLOCK + threadIdx.x * SCAN_PER_THREAD;
  unsigned long long sum = 0;
  for (int q = 0; q < SCAN_PER_THREAD; q++) if (i0 + q < n) sum += (unsigned long long)in[i0 + q];
  sum = warp_sum_u64(sum);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long tt = 0;
    for (int w = 0; w < SCAN_THREADS / 32; w++) tt += s_w[w];
    partial[blockIdx.x] = tt;
  }
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_final(const int64_t *__restrict__ in, int64_t *__restrict__ out, int64_t n,
                                                             const unsigned long long *__restrict__ partial) {
  __shared__ unsigned long long s_w[SCAN_THREADS / 32];
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t i0 = (int64_t)blockIdx.x * SCAN_PER_BLOCK + threadIdx.x * SCAN_PER_THREAD;
  unsigned long long v[SCAN_PER_THREAD], sum = 0;
  for (int q = 0; q < SCAN_PER_THREAD; q++) { v[q] = (i0 + q < n) ? (unsigned long long)in[i0 + q] : 0; sum += v[q]; }
  unsigned long long x = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { unsigned long long y = __shfl_up_sync(FULL, x, d); if (lane >= d) x += y; }
  if (lane == 31) s_w[wid] = x;
  __syncthreads();
  unsigned long long run = partial[blockIdx.x] + x - sum;
  for (int w = 0; w < wid; w++) run += s_w[w];
  for (int q = 0; q < SCAN_PER_THREAD; q++) {
    if (i0 + q < n) out[i0 + q] = (int64_t)run;
    run += v[q];
    if (i0 + q == n - 1) out[n] = (int64_t)run;
  }
}

int64_t mg_scan_tmp_elems(int64_t n) { return (n + SCAN_PER_BLOCK - 1) / SCAN_PER_BLOCK + 1; }

void mg_launch_scan_i64(const int64_t *in, int64_t *out, int64_t n, int64_t *tmp, cudaStream_t st) {
  if (n == 0) { cudaMemsetAsync(out, 0, sizeof(int64_t), st); return; }
  int nb = (int)((n + SCAN_PER_BLOCK - 1) / SCAN_PER_BLOCK);
  k_scan_reduce<<<nb, SCAN_THREADS, 0, st>>>(in, n, reinterpret_cast<unsigned long long *>(tmp));
  k_scan_partials_u64<<<1, 1024, 0, st>>>(reinterpret_cast<unsigned long long *>(tmp), nb);
  k_scan_final<<<nb, SCAN_THREADS, 0, st>>>(in, out, n, reinterpret_cast<const unsigned long long *>(tmp));
}

// ------------------------------------------------------------------------------------------
// FASTQ newline index

#define NL_CHUNK 4096
#define NL_THREADS 256

int64_t mg_nl_chunks(int64_t len) { return (len + NL_CHUNK - 1) / NL_CHUNK; }

__global__ void __launch_bounds__(NL_THREADS) k_nl_count(const uint8_t *__restrict__ buf, int64_t len, int64_t *__restrict__ cnt) {
  __shared__ uint32_t s_w[NL_THREADS / 32];
  int64_t base = (int64_t)blockIdx.x * NL_CHUNK + threadIdx.x * 16;
  uint32_t c = 0;
  for (int i = 0; i < 16; i++) if (base + i < len && buf[base + i] == '\n') c++;
  for (int d = 16; d >= 1; d >>= 1) c += __shfl_xor_sync(FULL, c, d);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t tt = 0; for (int w = 0; w < NL_THREADS / 32; w++) tt += s_w[w]; cnt[blockIdx.x] = tt; }
}

__global__ void __launch_bounds__(NL_THREADS) k_nl_write(const uint8_t *__restrict__ buf, int64_t len, const int64_t *__restrict__ off,
                                                         int64_t *__restrict__ nl) {
  __shared__ uint32_t s_w[NL_THREADS / 32];
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t base = (int64_t)blockIdx.x * NL_CHUNK + threadIdx.x * 16;
  uint32_t m = 0;
  for (int i = 0; i < 16; i++) if (base + i < len && buf[base + i] == '\n') m |= 1u << i;
  uint32_t c = __popc(m);
  uint32_t ic = warp_incl_scan_u32(c, lane);
  if (lane == 31) s_w[wid] = ic;
  __syncthreads();
  uint32_t o = ic - c;
  for (int w = 0; w < wid; w++) o += s_w[w];
  int64_t dst = off[blockIdx.x] + o;
  while (m) { int i = __ffs(m) - 1; m &= m - 1; nl[dst++] = base + i; }
}

void mg_launch_nl_count(const uint8_t *buf, int64_t len, int64_t *cnt, cudaStream_t st) {
  if (len == 0) return;
  k_nl_count<<<(unsigned)mg_nl_chunks(len), NL_THREADS, 0, st>>>(buf, len, cnt);
}
void mg_launch_nl_write(const uint8_t *buf, int64_t len, const int64_t *off, int64_t *nl, cudaStream_t st) {
  if (len == 0) return;
  k_nl_write<<<(unsigned)mg_nl_chunks(len), NL_THREADS, 0, st>>>(buf, len, off, nl);
}

// ------------------------------------------------------------------------------------------
// standalone corrupt-reads (readcorrupt.py:18-118 over illumina.py:113-162)

__device__ __forceinline__ void fq_lines(const int64_t *nl, int64_t r, int64_t &h0, int64_t &h1, int64_t &s0, int64_t &s1) {
  h0 = (r == 0) ? 0 : nl[4 * r - 1] + 1;   // header line [h0, h1)
  h1 = nl[4 * r];
  s0 = h1 + 1;                             // sequence line [s0, s1)
  s1 = nl[4 * r + 1];
}

// sizes of the output records; sz[f][r] = 1 + name + 1 + L + 3 + L + 1 (readcorrupt.py:113)
__global__ void __launch_bounds__(256) k_corrupt_sizes(MgCorruptParams P, int64_t *sz0, int64_t *sz1) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.n_rec) return;
  int64_t h0, h1, s0, s1;
  fq_lines(P.nl[0], r, h0, h1, s0, s1);
  int64_t ne = h0 + 1;                     // FastxFile .name: up to the first whitespace
  while (ne < h1) { uint8_t c = P.in[0][ne]; if (c == ' ' || c == '\t' || c == '\r') break; ne++; }
  int64_t name_len = ne - (h0 + 1);
  if (name_len < 0) name_len = 0;
  int64_t L0 = s1 - s0;
  if (L0 > P.n_cycles) atomicExch(P.err, 1ull);
  sz0[r] = 2 * L0 + name_len + 6;
  int64_t big = 2 * L0 + name_len + 6;
  if (P.n_files > 1) {
    fq_lines(P.nl[1], r, h0, h1, s0, s1);
    int64_t L1 = s1 - s0;
    if (L1 > P.n_cycles) atomicExch(P.err, 1ull);
    sz1[r] = 2 * L1 + name_len + 6;
    if (L1 > L0) big = 2 * L1 + name_len + 6;
  }
  atomicMax(P.err + 1, (unsigned long long)big);      // the staged kernel needs every record to fit a warp's stage
}

void mg_launch_corrupt_sizes(const MgCorruptParams &P, int64_t *sz0, int64_t *sz1, cudaStream_t st) {
  if (P.n_rec == 0) return;
  k_corrupt_sizes<<<(unsigned)((P.n_rec + 255) / 256), 256, 0, st>>>(P, sz0, sz1);
}

// one warp per template; lanes stride over name bytes and base-call pairs
__global__ void __launch_bounds__(256) k_corrupt(MgCorruptParams P) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < P.n_rec; r += warps) {
    int64_t nh0, nh1, s0, s1;
    fq_lines(P.nl[0], r, nh0, nh1, s0, s1);
    for (int f = 0; f < P.n_files; f++) {
      int64_t h0, h1;
      if (f) fq_lines(P.nl[f], r, h0, h1, s0, s1);
      const int64_t o = P.out_off[f][r];
      const int L = (int)(s1 - s0);
      const int name_len = (int)(P.out_off[f][r + 1] - o - 2 * (int64_t)L - 6);
      uint8_t *out = P.out[f] + o;
      const uint8_t *name = P.in[0] + nh0 + 1;                                 // read 1's name on both files
      if (lane == 0) { out[0] = '@'; out[1 + name_len] = '\n'; }
      for (int i = lane; i < name_len; i += 32) out[1 + i] = name[i];
      uint8_t *seq = out + 2 + name_len, *qual = seq + L + 3;
      const uint8_t *src = P.in[f] + s0;
      for (int i = lane; i < L; i += 32) seq[i] = src[i];
      if (lane == 0) { seq[L] = '\n'; seq[L + 1] = '+'; seq[L + 2] = '\n'; qual[L] = '\n'; }
      __syncwarp();
      if (L > P.n_cycles) continue;
      if (P.mode == MG_MODE_DET) {
        const int64_t d0 = P.draw_off[r * P.n_files + f];
        for (int n = lane; n < L; n += 32) {
          const double *row = P.cum_bq + ((size_t)f * P.n_cycles + n) * P.n_bq;
          mg_corrupt_call(seq, qual, n, row, P.n_bq, P.phred, P.bq_rnd[d0 + n], P.call_rnd[d0 + n], (int)P.base_rnd[d0 + n]);
        }
      } else {
        for (int g = lane; 4 * g < L; g += 32) {
          const int64_t gr = P.first + r;   // template index in the whole file
          const MgPhilox rr = mg_philox_corrupt((uint32_t)gr, (uint32_t)(gr >> 32) * 2u + (uint32_t)f, (uint32_t)g, P.cor.k0, P.cor.k1);
#pragma unroll
          for (int h = 0; h < 4; h++) {
            const int n = 4 * g + h;
            if (n < L) {
              uint32_t base = seq[n], q;
              mg_corrupt_one(P.cor, (uint32_t)f, n, rr.v[h], base, q);
              seq[n] = (uint8_t)base; qual[n] = (uint8_t)q;
            }
          }
        }
      }
      __syncwarp();
    }
  }
}

// ---- k_corrupt_staged: production-mode corrupt-reads on the emit kernel's machinery ---------------
// One WARP owns 32 consecutive templates (lane = record, so every lane is at the same cycle and the
// alias row of a cycle is shared by the warp); per file the records are rebuilt -- '@' + read 1's name,
// the sequence corrupted four cycles per step (one Philox block, four joint-table lookups, branch-free
// substitution on the letters), "+", the qualities -- in the warp's shared-memory stage and leave
// through the bulk copy engine, like k_unit_emit's.  Input bytes are read with aligned 32-bit loads and
// a funnel shift per lane.

// four letters with substitutions: A/C/G/T become "ACGT"[code ^ s]; any other byte becomes 'N' when s != 0
__device__ __forceinline__ uint32_t letters4_sub(uint32_t a4, uint32_t snib) {
  const uint32_t x = (a4 >> 1) & 0x03030303u;                   // A 0, C 1, T 2, G 3 (bits 1-2 of the letter)
  const uint32_t sd = x ^ ((x >> 1) & 0x01010101u);              // -> A 0, C 1, G 2, T 3
  uint32_t u = (sd | (sd >> 4)) & 0x00330033u;
  const uint32_t z = (u | (u >> 8)) & 0x3333u;                   // as PRMT selector nibbles
  const uint32_t plain = __byte_perm(0x54474341u, 0u, z);
  uint32_t out = __byte_perm(0x54474341u, 0u, z ^ snib);
  if (plain != a4) {                                             // some byte is not an upper-case A/C/G/T (N, IUPAC, lower case)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t c = (a4 >> (8 * j)) & 0xFFu;
      if (((plain >> (8 * j)) & 0xFFu) != c) {
        const uint32_t nb = ((snib >> (4 * j)) & 3u) ? (uint32_t)'N' : c;       // base_rot.get(base, 'NNN'), illumina.py:160
        out = (out & ~(0xFFu << (8 * j))) | (nb << (8 * j));
      }
    }
  }
  return out;
}

template <bool C9>
__global__ void __launch_bounds__(MG_CTA, 4) k_corrupt_staged(const __grid_constant__ MgCorruptParams P, const int stage_cap, const int bulk) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  uint8_t *stage = smem + (uint32_t)wid * (uint32_t)(stage_cap + 16);
  uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
  asm volatile("" : "+r"(stage_s));
  unsigned long long policy = 0;
  if (bulk) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  bool in_flight = false;
  const MgCorruptCtx &C = P.cor;
  const uint32_t ks = (uint32_t)C.kshift;
  const int64_t n_wt = (P.n_rec + 31) / 32;
  for (int64_t wt = (int64_t)blockIdx.x * (MG_CTA / 32) + wid; wt < n_wt; wt += (int64_t)gridDim.x * (MG_CTA / 32)) {
    const int64_t r = wt * 32 + lane;
    const bool active = r < P.n_rec;
    const int64_t rr = active ? r : P.n_rec - 1;
    const int64_t gr = P.first + rr;                           // template index in the whole file: the Philox counter
    // everything this tile needs from the index arrays is asked for at once (one memory latency instead of one per
    // file), and so are the line bounds of the tile this warp takes NEXT: they are used at the end of this one to
    // prefetch that tile's name / sequence lines into L2 (the kernel is bound by the latency of its cold input
    // loads: 7.8 stall cycles per issue on the long scoreboard before this, `profiles/r02_corrupt_staged_full.txt`)
    int64_t nh0, nh1, s0, s1, s0b = 0, s1b = 0;
    fq_lines(P.nl[0], rr, nh0, nh1, s0, s1);
    const bool two = P.n_files > 1;
    if (two) { s0b = P.nl[1][4 * rr] + 1; s1b = P.nl[1][4 * rr + 1]; }
    const int64_t off_a = P.out_off[0][rr], end_a = P.out_off[0][rr + 1];
    const int64_t off_b = two ? P.out_off[1][rr] : 0, end_b = two ? P.out_off[1][rr + 1] : 0;
    const int64_t rn = r + (int64_t)gridDim.x * MG_CTA;       // this lane's record of the warp's next tile
    const bool has_next = rn < P.n_rec;
    int64_t pn0 = 0, pn1 = 0, pb0 = 0, pb1 = 0;
    if (has_next) {
      pn0 = P.nl[0][4 * rn - 1] + 1; pn1 = P.nl[0][4 * rn + 1];
      if (two) { pb0 = P.nl[1][4 * rn] + 1; pb1 = P.nl[1][4 * rn + 1]; }
    }
    if (two) for (int64_t a = s0b & ~31ll; a < s1b; a += 32) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.in[1] + a));   // the other file's sequence line
    const int n_act = (int)(P.n_rec - wt * 32 < 32 ? P.n_rec - wt * 32 : 32);
    for (int f = 0; f < P.n_files; f++) {
      if (f) { s0 = s0b; s1 = s1b; }
      const int64_t off = f ? off_b : off_a;
      const uint32_t rec = (uint32_t)((f ? end_b : end_a) - off);
      const int L = (int)(s1 - s0);
      const int name_len = (int)rec - 2 * L - 6;
      const unsigned long long my_end = active ? (unsigned long long)(off + rec) : 0ull;
      const uint8_t *src = P.in[f] + s0;
      const uint32_t rowf = (uint32_t)f * (uint32_t)C.n_cycles, t_lo = (uint32_t)gr, t_hi2f = (uint32_t)((unsigned long long)gr >> 32) * 2u + (uint32_t)f;
      int lo = 0;
      while (lo < n_act) {
        const unsigned long long goff = __shfl_sync(FULL, (unsigned long long)off, lo);
        const uint32_t pad = (uint32_t)(goff & 15);
        const bool fits = active && lane >= lo && (my_end - goff + pad) <= (unsigned long long)stage_cap;
        int hi = lo + __popc(__ballot_sync(FULL, fits));
        if (hi == lo) hi = lo + 1;                               // cannot happen: the host checked that every record fits
        const unsigned long long gend = __shfl_sync(FULL, my_end, hi - 1);
        const uint32_t batch_bytes = (uint32_t)(gend - goff);
        const bool mine = active && lane >= lo && lane < hi;
        const uint32_t dst = stage_s + pad + (uint32_t)((unsigned long long)off - goff);
        if (in_flight) {
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          __syncwarp();
          in_flight = false;
        }
        if (mine) {                                              // '@' + read 1's name + '\n'
          MgStream<MgSharedSpace> wn;
          wn.begin(dst);
          const uint8_t *np_ = P.in[0] + nh0 + 1;
          const uint32_t sh = 8u * (uint32_t)((uintptr_t)np_ & 3);
          const uint32_t *wp = reinterpret_cast<const uint32_t *>(np_ - ((uintptr_t)np_ & 3));
          uint32_t carry = wp[0];
          wn.append(mg_tok('@', 0, 1));
#pragma unroll 1
          for (int i0 = 0; i0 < name_len; i0 += 32) {              // eight words (four tokens) per trip: their loads are in flight together
            uint32_t v[8];
#pragma unroll
            for (int q = 0; q < 8; q++) v[q] = (i0 + 4 * q < name_len) ? wp[(i0 >> 2) + q + 1] : 0u;
#pragma unroll
            for (int q = 0; q < 8; q += 2) {
              const int i = i0 + 4 * q;
              if (i < name_len) {
                uint32_t lo4 = __funnelshift_r(carry, v[q], sh), hi4 = __funnelshift_r(v[q], v[q + 1], sh);
                const int m = name_len - i < 8 ? name_len - i : 8;
                if (m < 8) { if (m <= 4) { hi4 = 0; lo4 = m == 4 ? lo4 : lo4 & ((1u << (8 * m)) - 1u); } else hi4 &= (1u << (8 * (m - 4))) - 1u; }
                wn.append(mg_tok(lo4, hi4, (uint32_t)m));
              }
              carry = v[q + 1];
            }
          }
          wn.append(mg_tok('\n', 0, 1));
          wn.flush_own();
        }
        __syncwarp();                                            // every first word is stored: now the bytes that share a word with a neighbour
        if (mine) {
          const uint32_t seq_dst = dst + (uint32_t)name_len + 2u, qual_dst = seq_dst + (uint32_t)L + 3u;
          MgSharedSpace::st8(qual_dst + L, '\n');
          const int NG = L >> 2, rem = L & 3;
          {   // 1. the letters as they are, parked in the record's own sequence line: PARK independent loads in flight
              //    at a time (the per-group loads of the main loop would each wait for memory on their own)
            constexpr int PARK = 16;
            MgStream<MgSharedSpace> wl;
            wl.begin_rmw(seq_dst);
            const uint32_t ish = 8u * (uint32_t)((uintptr_t)src & 3);
            const uint32_t *iw = reinterpret_cast<const uint32_t *>(src - ((uintptr_t)src & 3));
            const int NW = (L + 3) >> 2;
            uint32_t carry = iw[0];
#pragma unroll 1
            for (int w0 = 0; w0 < NW; w0 += PARK) {
              uint32_t v[PARK];
#pragma unroll
              for (int i = 0; i < PARK; i++) v[i] = (w0 + i < NW) ? iw[w0 + i + 1] : 0u;
#pragma unroll
              for (int i = 0; i < PARK; i++) {
                if (w0 + i < NG) wl.put_word(__funnelshift_r(carry, v[i], ish));
                else if (w0 + i == NG && rem) { const uint32_t ch = __funnelshift_r(carry, v[i], ish); for (int j = 0; j < rem; j++) wl.put((uint8_t)(ch >> (8 * j))); }
                carry = v[i];
              }
            }
            wl.flush_own();                                     // the bytes above are this record's own '\n+\n' ...
            MgSharedSpace::st8(seq_dst + L, '\n'); MgSharedSpace::st8(seq_dst + L + 1, '+'); MgSharedSpace::st8(seq_dst + L + 2, '\n');   // ... rewritten here
          }
          // 2. four cycles per step, in place: read the parked letters, substitute, write them back with the qualities
          MgStream<MgSharedSpace> ws, wq;
          ws.begin_rmw(seq_dst); wq.begin_rmw(qual_dst);
          const uint32_t lsh = 8u * (seq_dst & 3u), lbase = seq_dst & ~3u;
          uint32_t icarry = MgSharedSpace::ld32(lbase);
          auto draw = [&](MgGrp &G, int g) {
            const uint32_t nx = MgSharedSpace::ld32(lbase + 4u * (uint32_t)(g + 1));
            G.b4 = __funnelshift_r(icarry, nx, lsh);            // the four letters of group g
            icarry = nx;
            mg_grp_draw<true>(C, ks, t_lo, t_hi2f, rowf + 4u * (uint32_t)g, 4 * g, L, G);
          };
          auto flush = [&](const MgGrp &G) {
            uint32_t q4, snib;
            mg_grp_decode<C9>(G, ks, q4, snib);
            ws.put_word(letters4_sub(G.b4, snib)); wq.put_word(q4);
          };
          if (NG > 0) {
            MgGrp A, B;
            int g = 0;
            draw(A, 0);
#pragma unroll 1
            while (g + 2 < NG) {
              draw(B, g + 1); flush(A);
              draw(A, g + 2); flush(B);
              g += 2;
            }
            if (g + 1 < NG) { draw(B, g + 1); flush(A); flush(B); }
            else flush(A);
          }
          if (rem) {
            MgGrp G;
            const uint32_t nx = MgSharedSpace::ld32(lbase + 4u * (uint32_t)(NG + 1));
            G.b4 = __funnelshift_r(icarry, nx, lsh);
            G.b4 &= (1u << (8 * rem)) - 1u; G.b4 |= 0x41414141u << (8 * rem);       // the bytes beyond the read: harmless letters
            mg_grp_draw<false>(C, ks, t_lo, t_hi2f, rowf + 4u * (uint32_t)NG, 4 * NG, L, G);
            uint32_t q4, snib;
            mg_grp_decode<C9>(G, ks, q4, snib);
            const uint32_t ch = letters4_sub(G.b4, snib);
            for (int j = 0; j < rem; j++) { ws.put((uint8_t)(ch >> (8 * j))); wq.put((uint8_t)(q4 >> (8 * j))); }
          }
          ws.end(); wq.end();
        }
        // copy-out, as in k_unit_emit
        uint8_t *gdst = P.out[f] + goff;
        const uint8_t *ssrc = stage + pad;
        uint32_t head = (16u - pad) & 15u;
        if (head > batch_bytes) head = batch_bytes;
        const uint32_t nvec = (batch_bytes - head) >> 4;
        const uint32_t done = head + (nvec << 4);
        if (bulk) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0 && nvec) bulk_store(gdst + head, stage_s + pad + head, nvec << 4, policy);
          in_flight = nvec != 0;
          if ((uint32_t)lane < head) gdst[lane] = ssrc[lane];
          if (done + lane < batch_bytes) gdst[done + lane] = ssrc[done + lane];
        } else {
          __syncwarp();
          if ((uint32_t)lane < head) gdst[lane] = ssrc[lane];
          const uint4 *sv = reinterpret_cast<const uint4 *>(ssrc + head);
          uint4 *gv = reinterpret_cast<uint4 *>(gdst + head);
          for (uint32_t v = lane; v < nvec; v += 32) __stcs(gv + v, sv[v]);
          if (done + lane < batch_bytes) gdst[done + lane] = ssrc[done + lane];
          __syncwarp();
        }
        lo = hi;
      }
    }
    if (has_next) {                                              // the next tile's name and sequence lines, on their way into L2
      for (int64_t a = pn0 & ~31ll; a < pn1; a += 32) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.in[0] + a));
      if (two) for (int64_t a = pb0 & ~31ll; a < pb1; a += 32) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.in[1] + a));
    }
  }
  if (bulk && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

#define MG_CORRUPT_STAGE (32 * (2 * 150 + 6 + 96) & ~15)     // bytes per warp: 32 records of 2 x 150 + a ~90-byte name

int mg_corrupt_stage_cap(void) { return MG_CORRUPT_STAGE; }

// staged == true: every output record fits a warp's stage (the caller checked): the fast kernel
void mg_launch_corrupt_staged(const MgCorruptParams &P, bool bulk, cudaStream_t st) {
  if (P.n_rec == 0) return;
  const int smem = (MG_CTA / 32) * (MG_CORRUPT_STAGE + 16);
  auto k = P.cor.code9 ? k_corrupt_staged<true> : k_corrupt_staged<false>;
  static bool once[2] = {false, false};
  if (!once[P.cor.code9 ? 1 : 0]) { cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); once[P.cor.code9 ? 1 : 0] = true; }
  int per_sm = 0, dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, MG_CTA, smem);
  if (per_sm < 1) per_sm = 1;
  int64_t blocks = (P.n_rec + 127) / 128;
  if (blocks > (int64_t)sms * per_sm) blocks = (int64_t)sms * per_sm;
  k<<<(unsigned)blocks, MG_CTA, smem, st>>>(P, MG_CORRUPT_STAGE, bulk ? 1 : 0);
}

void mg_launch_corrupt(const MgCorruptParams &P, cudaStream_t st) {
  if (P.n_rec == 0) return;
  int64_t blocks = (P.n_rec + 7) / 8;
  if (blocks > 148 * 16) blocks = 148 * 16;
  k_corrupt<<<(unsigned)blocks, 256, 0, st>>>(P);
}
