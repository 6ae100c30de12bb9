// Device-side reading of one BAM record (SAM spec v1 §4.2) handed out by MgBamReader: rec points at its
// block_size field.  Shared by k_readmodel (mg_readmodel.cu) and k_alnerr (mg_alnerr.cu).
#pragma once
#include <stdint.h>

#include "mg_bgzf.h"

__device__ __forceinline__ uint32_t mg_ld32(const uint8_t *p) { return p[0] | p[1] << 8 | p[2] << 16 | (uint32_t)p[3] << 24; }

// The four overrun checks against block_size (>= 32: the host walk checked it): -> 0, or MG_RD_NAME / CIGAR /
// SEQ / QUAL for the first field that does not fit.  qual = offset of QUAL from the end of the block_size field.
__device__ __forceinline__ int mg_bam_overrun(const uint8_t *rec, int64_t &qual) {
  const int32_t bs = (int32_t)mg_ld32(rec);
  const int l_name = rec[12], n_cig = rec[16] | rec[17] << 8;
  const int32_t l_seq = (int32_t)mg_ld32(rec + 20);
  int64_t e = 32 + l_name;
  if (e > bs) return MG_RD_NAME;
  if ((e += 4 * n_cig) > bs) return MG_RD_CIGAR;
  if (l_seq < 0 || (e += ((int64_t)l_seq + 1) / 2) > bs) return MG_RD_SEQ;
  if (e + l_seq > bs) return MG_RD_QUAL;
  qual = e;
  return 0;
}
