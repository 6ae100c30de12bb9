// bam2illumina: the per-base counts of an Illumina read model (Mitty's mitty/empirical/bam2illumina.py)
// over a BGZF BAM, counted on the device.
//
// The host reader (MgBamReader, mg_bgzf.cpp) inflates the file chunk by chunk and walks the block_size
// chain; each chunk of whole records goes to the device with its record offsets (copy stream) while the
// next chunk is inflated.  That loop, mg_bam_pipeline, is defined here and shared with alignment-analysis
// (mg_alnerr.cu).  One launch of k_readmodel per chunk:
//   one warp per record (grid-stride): validate the record against its block_size, apply the sampling and
//   skip rules, and count QUAL with lane = cycle -- 32 consecutive cycles of one read per step, so the
//   quality loads coalesce and the 32 shared-memory addresses differ.  Rows of the privatised bq_mat are
//   95 words apart (odd), so cycles c and c + 16 with equal qualities do not share a bank.
//   The CTA's u32 counters (bq_mat rows of its cycle stripe; read lengths and skip counters in stripe 0)
//   go to the u64 global counters at the end of the launch, so a u32 counts at most one chunk's records.
//   Template lengths are counted straight into global memory: one atomic per counted read 1.
// With the default max_bp = 300 one stripe covers every cycle (228 000 B of bq_mat rows, one CTA per SM);
// a larger max_bp splits the cycles into stripes, one per blockIdx.y.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <string>

#include "../../include/mitty_b200.h"
#include "mg_bamrec.cuh"
#include "mg_bgzf.h"
#include "mg_internal.h"

namespace {

#define RM_NQ 94            // qualities 0 .. 93 (higher ones are counted as 93)
#define RM_STRIDE 95        // words per (mate, cycle) row in shared memory
#define RM_THREADS 1024

enum { RM_CONSIDERED = 0, RM_COUNTED, RM_SKIP_FLAG, RM_SKIP_MAPQ, RM_SKIP_EMPTY, RM_SKIP_NOQUAL, RM_SKIP_LONG, RM_NCNT };

struct RmParams {
  const uint8_t *data; const uint32_t *off; int64_t n; uint64_t first;
  uint32_t every; int min_mq, max_bp, max_tlen, stripe;
  unsigned long long *bq, *len_hist, *tlen, *cnt, *first_bad;
};

__global__ void __launch_bounds__(RM_THREADS, 1) k_readmodel(RmParams P) {
  extern __shared__ uint32_t sm[];
  const int W = P.stripe, c0 = blockIdx.y * W, w = min(W, P.max_bp - c0);
  const bool head = blockIdx.y == 0;
  uint32_t *s_bq = sm, *s_len = sm + 2 * W * RM_STRIDE, *s_cnt = s_len + P.max_bp + 1;
  const int words = 2 * W * RM_STRIDE + P.max_bp + 1 + RM_NCNT;
  for (int i = threadIdx.x; i < words; i += blockDim.x) sm[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < P.n; r += nw) {
    const uint8_t *rec = P.data + P.off[r];
    const int mapq = rec[13], flag = rec[18] | rec[19] << 8;
    const int32_t l_seq = (int32_t)mg_ld32(rec + 20);
    int64_t e = 0;
    const int bad = mg_bam_overrun(rec, e);
    const uint64_t k = P.first + (uint64_t)r;
    if (bad) {
      if (head && lane == 0) atomicMin(P.first_bad, (unsigned long long)(k << 8 | bad));
      continue;
    }
    if (k % P.every) continue;
    const uint8_t *q = rec + 4 + e;
    const int why = flag & 0xB04 ? RM_SKIP_FLAG : mapq < P.min_mq ? RM_SKIP_MAPQ : l_seq == 0 ? RM_SKIP_EMPTY
                  : q[0] == 0xFF ? RM_SKIP_NOQUAL : l_seq > P.max_bp ? RM_SKIP_LONG : RM_COUNTED;
    if (head && lane == 0) {
      atomicAdd(&s_cnt[RM_CONSIDERED], 1u);
      atomicAdd(&s_cnt[why], 1u);
      if (why == RM_COUNTED) {
        atomicAdd(&s_len[l_seq], 1u);
        if ((flag & 0xC1) == 0x41) {
          const int32_t tl = (int32_t)mg_ld32(rec + 32);
          const int64_t t = tl < 0 ? -(int64_t)tl : (int64_t)tl;
          if (t < P.max_tlen) atomicAdd(&P.tlen[t], 1ull);
        }
      }
    }
    if (why != RM_COUNTED) continue;
    uint32_t *row = s_bq + ((flag & 0xC1) == 0x81 ? W * RM_STRIDE : 0);
    const bool rev = flag & 0x10;
    const int c1 = min(l_seq, c0 + w);
    for (int c = c0 + lane; c < c1; c += 32) {
      const int qv = min((int)q[rev ? l_seq - 1 - c : c], RM_NQ - 1);
      atomicAdd(&row[(c - c0) * RM_STRIDE + qv], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * w * RM_NQ; i += blockDim.x) {
    const int m = i / (w * RM_NQ), c = i / RM_NQ % w, qv = i % RM_NQ;
    const uint32_t v = s_bq[(m * W + c) * RM_STRIDE + qv];
    if (v) atomicAdd(&P.bq[((int64_t)m * P.max_bp + c0 + c) * RM_NQ + qv], (unsigned long long)v);
  }
  if (!head) return;
  for (int i = threadIdx.x; i < P.max_bp + 1 + RM_NCNT; i += blockDim.x) {
    const uint32_t v = s_len[i];
    if (v) atomicAdd(i <= P.max_bp ? &P.len_hist[i] : &P.cnt[i - P.max_bp - 1], (unsigned long long)v);
  }
}

}  // namespace

double mg_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

void *mg_pinned_alloc(size_t n) { void *p = nullptr; return cudaHostAlloc(&p, n, cudaHostAllocDefault) == cudaSuccess ? p : nullptr; }
void mg_pinned_release(void *p) { cudaFreeHost(p); }

int mg_bam_pipeline(mg_ctx *ctx, MgBamReader &rd, const MgBamPipe &p, double t_start, int64_t *chunks, double *times, double *thread_ms,
                    int64_t *bad_where, int32_t *bad_code) {
  *bad_where = -1; *bad_code = 0; *chunks = 0;
  DevBuf d_data[2], d_off[2], d_bad;
  HostBuf h_bad;                                     // per slot: the chunk's first_bad, read back; [2]: the final value
  cudaStream_t cs = nullptr, ks = nullptr;
  cudaEvent_t ev[2][5] = {};                         // per slot: H2D start / end, kernel start / end, first_bad read back
  bool pending[2] = {false, false}, device_bad = false;
  double h2d_ms = 0, kernel_ms = 0;
  unsigned long long first_bad = ~0ull;
  // waits for the chunk in flight in `s`, adds its copy and kernel times and notes a malformed record found so far
  auto settle = [&](int s) -> int {
    if (!pending[s]) return MG_OK;
    pending[s] = false;
    MG_CK(ctx, cudaEventSynchronize(ev[s][4]));
    if (h_bad.as<unsigned long long>()[s] != ~0ull) device_bad = true;
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, ev[s][0], ev[s][1]); cudaEventElapsedTime(&b, ev[s][2], ev[s][3]);
    h2d_ms += a; kernel_ms += b;
    return MG_OK;
  };
  // every chunk through the caller's kernel; returns at the first failure, the streams and events are released below
  auto run = [&]() -> int {
    MG_CK(ctx, cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    MG_CK(ctx, cudaStreamCreateWithFlags(&ks, cudaStreamNonBlocking));
    MG_CK(ctx, h_bad.need(3 * sizeof(unsigned long long)));
    for (int s = 0; s < 2; s++) for (int j = 0; j < 5; j++) MG_CK(ctx, cudaEventCreate(&ev[s][j]));
    MG_CK(ctx, d_bad.need(sizeof(unsigned long long)));
    unsigned long long *bad = d_bad.as<unsigned long long>();
    MG_CK(ctx, cudaMemsetAsync(bad, 0xFF, sizeof(unsigned long long), ks));
    int rc = p.begin(ks);
    if (rc) return rc;
    MgBamChunk c;
    for (int64_t k = 0;; k++) {
      const int s = (int)(k & 1);
      if ((rc = settle(s))) return rc;                 // the slot's buffers are free again
      if (device_bad || !rd.next(s, c)) break;         // a malformed record ends the input: it is reported, nothing later is
      MG_CK(ctx, d_data[s].need((size_t)c.bytes));
      MG_CK(ctx, d_off[s].need(4 * (size_t)c.n));
      MG_CK(ctx, cudaEventRecord(ev[s][0], cs));
      MG_CK(ctx, cudaMemcpyAsync(d_data[s].p, c.data, (size_t)c.bytes, cudaMemcpyHostToDevice, cs));
      MG_CK(ctx, cudaMemcpyAsync(d_off[s].p, c.off, 4 * (size_t)c.n, cudaMemcpyHostToDevice, cs));
      MG_CK(ctx, cudaEventRecord(ev[s][1], cs));
      MG_CK(ctx, cudaStreamWaitEvent(ks, ev[s][1], 0));
      MG_CK(ctx, cudaEventRecord(ev[s][2], ks));
      if ((rc = p.launch(c, d_data[s].as<uint8_t>(), d_off[s].as<uint32_t>(), bad, ks))) return rc;
      MG_CK(ctx, cudaEventRecord(ev[s][3], ks));
      MG_CK(ctx, cudaMemcpyAsync(h_bad.as<unsigned long long>() + s, bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ks));
      MG_CK(ctx, cudaEventRecord(ev[s][4], ks));
      pending[s] = true;
      ++*chunks;
    }
    for (int s = 0; s < 2; s++) if ((rc = settle(s))) return rc;
    if ((rc = p.finish(ks))) return rc;
    MG_CK(ctx, cudaMemcpyAsync(h_bad.as<unsigned long long>() + 2, bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ks));
    MG_CK(ctx, cudaStreamSynchronize(ks));
    first_bad = h_bad.as<unsigned long long>()[2];
    return MG_OK;
  };
  const int rc = run();
  if (ks) cudaStreamSynchronize(ks);
  if (cs) cudaStreamSynchronize(cs);
  for (int s = 0; s < 2; s++) for (int j = 0; j < 5; j++) if (ev[s][j]) cudaEventDestroy(ev[s][j]);
  if (cs) cudaStreamDestroy(cs);
  if (ks) cudaStreamDestroy(ks);

  times[0] = rd.read_ms; times[1] = rd.inflate_ms; times[2] = rd.walk_ms; times[3] = h2d_ms; times[4] = kernel_ms; times[5] = mg_now_ms() - t_start;
  if (thread_ms) for (size_t t = 0; t < rd.thread_ms.size(); t++) thread_ms[t] = rd.thread_ms[t];
  if (rc != MG_OK) return rc;
  if (first_bad != ~0ull) { *bad_where = (int64_t)(first_bad >> 8); *bad_code = (int32_t)(first_bad & 0xFF); }
  else if (rd.code) { *bad_where = rd.where; *bad_code = rd.code; }
  else if (!rd.err.empty()) return mg_internal_fail(ctx, MG_EVALUE, rd.err.c_str());
  return *bad_code ? mg_internal_fail(ctx, MG_EVALUE, "malformed BAM input") : MG_OK;
}

extern "C" int mg_readmodel_bam(mg_ctx *ctx, const char *path, int32_t max_bp, int32_t max_tlen, int32_t min_mq, int64_t every, int32_t threads,
                                int64_t chunk_bytes, uint64_t *bq_mat, uint64_t *len_hist, uint64_t *tlen, int64_t *counts, double *times,
                                double *thread_ms, int64_t *bad_where, int32_t *bad_code) {
  if (!ctx || !path || max_bp < 1 || max_bp > 50000 || max_tlen < 1 || max_tlen > (1 << 20) || every < 1 || every > UINT32_MAX || !bq_mat || !len_hist || !tlen || !counts ||
      !times || !bad_where || !bad_code)
    return MG_EINVAL;
  const double t_start = mg_now_ms();
  *bad_where = -1; *bad_code = 0;
  const int dev = mg_internal_device(ctx);
  DeviceGuard g(dev);
  int smem_max = 0, n_sm = 0;
  cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  const int fixed = 4 * (max_bp + 1 + RM_NCNT);
  const int stripe = std::min(max_bp, (smem_max - fixed) / (2 * RM_STRIDE * 4));
  if (stripe < 1) return mg_internal_fail(ctx, MG_EINVAL, "mg_readmodel_bam: max_bp too large for the shared-memory counters");
  const int n_stripes = (max_bp + stripe - 1) / stripe;
  const int smem = 2 * stripe * RM_STRIDE * 4 + fixed;
  if (cudaFuncSetAttribute(k_readmodel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
    return mg_internal_fail(ctx, MG_ECUDA, "mg_readmodel_bam: cannot set the kernel's shared memory");

  MgBamReader rd;
  if (!rd.open(path, threads, chunk_bytes, mg_pinned_alloc, mg_pinned_release)) return mg_internal_fail(ctx, MG_EVALUE, rd.err.c_str());
  const size_t n_bq = (size_t)2 * max_bp * RM_NQ, n_acc = n_bq + (size_t)max_bp + 1 + (size_t)max_tlen + RM_NCNT;
  DevBuf d_acc;
  int64_t chunks = 0;
  unsigned long long cnt[RM_NCNT] = {0};
  RmParams P;
  memset(&P, 0, sizeof P);
  P.every = (uint32_t)every; P.min_mq = min_mq; P.max_bp = max_bp; P.max_tlen = max_tlen; P.stripe = stripe;
  MgBamPipe pipe;
  pipe.begin = [&](cudaStream_t ks) -> int {
    MG_CK(ctx, d_acc.need(8 * n_acc));
    P.bq = d_acc.as<unsigned long long>(); P.len_hist = P.bq + n_bq; P.tlen = P.len_hist + max_bp + 1; P.cnt = P.tlen + max_tlen;
    MG_CK(ctx, cudaMemsetAsync(P.bq, 0, 8 * n_acc, ks));
    return MG_OK;
  };
  pipe.launch = [&](const MgBamChunk &c, const uint8_t *data, const uint32_t *off, unsigned long long *first_bad, cudaStream_t ks) -> int {
    P.data = data; P.off = off; P.n = c.n; P.first = (uint64_t)c.first; P.first_bad = first_bad;
    const dim3 grid((unsigned)std::min<int64_t>(n_sm, (c.n + 31) / 32), (unsigned)n_stripes);
    k_readmodel<<<grid, RM_THREADS, smem, ks>>>(P);
    MG_CK(ctx, cudaGetLastError());
    return MG_OK;
  };
  pipe.finish = [&](cudaStream_t ks) -> int {
    MG_CK(ctx, cudaMemcpyAsync(bq_mat, P.bq, 8 * n_bq, cudaMemcpyDeviceToHost, ks));
    MG_CK(ctx, cudaMemcpyAsync(len_hist, P.len_hist, 8 * ((size_t)max_bp + 1), cudaMemcpyDeviceToHost, ks));
    MG_CK(ctx, cudaMemcpyAsync(tlen, P.tlen, 8 * (size_t)max_tlen, cudaMemcpyDeviceToHost, ks));
    MG_CK(ctx, cudaMemcpyAsync(cnt, P.cnt, sizeof cnt, cudaMemcpyDeviceToHost, ks));
    return MG_OK;
  };
  const int rc = mg_bam_pipeline(ctx, rd, pipe, t_start, &chunks, times, thread_ms, bad_where, bad_code);
  const int64_t out[12] = {rd.records, (int64_t)cnt[RM_CONSIDERED], (int64_t)cnt[RM_COUNTED], (int64_t)cnt[RM_SKIP_FLAG], (int64_t)cnt[RM_SKIP_MAPQ],
                           (int64_t)cnt[RM_SKIP_EMPTY], (int64_t)cnt[RM_SKIP_NOQUAL], (int64_t)cnt[RM_SKIP_LONG], rd.raw_bytes, rd.comp_bytes,
                           rd.eof_marker ? 1 : 0, chunks};
  memcpy(counts, out, sizeof out);
  return rc;
}
