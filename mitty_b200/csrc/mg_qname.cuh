// Device parser of Mitty's read qname (readgenerate.parse_qname, mitty/simulation/readgenerate.py:259-291):
//   @serial|chrom|copy|strand|pos|rlen|cigar|vlist|strand|pos|rlen|cigar|vlist
// three template fields, then five fields per read in file order.  Shared by k_roundtrip_check
// (mg_check.cu) and the god-aligner's size / encode kernels (mg_bam.cu).
#pragma once
#include <stdint.h>

#define MG_QN_FIELDS 16      // fields kept per qname (13 are used by a pair)

// decimal integer in p[a, b) with an optional '-'; false if empty, not a number or beyond 2^40
__device__ __forceinline__ bool mg_parse_int(const uint8_t *p, int64_t a, int64_t b, int64_t &v) {
  if (a >= b) return false;
  bool neg = false;
  if (p[a] == '-') { neg = true; a++; if (a >= b) return false; }
  int64_t x = 0;
  for (int64_t i = a; i < b; i++) { const uint8_t c = p[i]; if (c < '0' || c > '9') return false; x = x * 10 + (c - '0'); if (x > (1ll << 40)) return false; }
  v = neg ? -x : x;
  return true;
}

// splits the qname q[a, b) (after the '@', up to the newline) at '|': field k is [fs[k], fe[k]).
// Returns the number of fields, at most MG_QN_FIELDS.
__device__ __forceinline__ int mg_qname_split(const uint8_t *q, int64_t a, int64_t b, int64_t *fs, int64_t *fe) {
  int nf = 0;
  int64_t s = a;
  for (int64_t i = a; i <= b && nf < MG_QN_FIELDS; i++)
    if (i == b || q[i] == '|') { fs[nf] = s; fe[nf] = i; nf++; s = i + 1; }
  return nf;
}
