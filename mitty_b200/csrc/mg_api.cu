// C-ABI of the engine (include/mitty_b200.h): context, device-memory management and the launch
// sequences of the kernels in mg_kernels.cu.  No CPU fallback lives here.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <cstdlib>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/mitty_b200.h"
#include "mg_bgzf.h"
#include "mg_internal.h"

namespace {

struct ExcRun { int64_t start, len; uint8_t byte; };

struct Region {
  int64_t len = 0, bed_start = 0;
  uint32_t *d_ref = nullptr;      // packed, with MG_HAP_PAD words of padding on both sides
  std::vector<ExcRun> exc;        // non-ACGT runs, region-relative
  MgExc *d_exc = nullptr;         // the same runs on the device (sorted by start)
  mg_ctx *owner = nullptr;
  ~Region();
};


struct Copy {
  int64_t region_id = 0;
  int64_t p_min = 0, p_max = 0;
  int64_t n_nodes = 0;
  int64_t n_exc = 0;
  MgNode *d_nodes = nullptr; uint32_t *d_hap = nullptr; uint32_t *d_blk = nullptr; MgExc *d_exc = nullptr;
  uint32_t *d_eblk = nullptr;        // block table over d_exc (n_blk + 1 entries), when there are exception runs
  int n_blk = 0; int64_t hap_words = 0, hap_len = 0;
  std::vector<MgSegOut> segs;      // a batch of small regions: one entry per (region, copy)
  std::vector<int64_t> seg_start1;
  mg_ctx *owner = nullptr;
  ~Copy();
};

// a batch of small regions: ONE packed reference, node table, haplotype and block table over all of its segments
struct Batch {
  std::unique_ptr<Region> R;
  std::unique_ptr<Copy> C;
};

const int BLK_SHIFT = 8;

}  // namespace

struct mg_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  // model
  DevBuf m_tlen, m_bq, m_phred, m_alias[2], m_tlen_alias;
  bool has_tlen_alias = false;   // n_tlen + 1 <= 1024 outcomes: 1024-entry alias table of the template-length model
  int n_tlen = 0, n_mates = 0, n_cycles = 0, n_bq = 0, rlen = 0;
  // production-mode corruption tables (MgCorruptCtx): [0] the emit kernel's (cycles < rlen), [1] the
  // standalone corrupt kernel's (every cycle of the model); kshift / code9 are chosen per table
  std::vector<uint32_t> h_alias[2]; int a_kshift[2] = {0, 0}, a_code9[2] = {0, 0}, a_rows[2] = {0, 0};
  std::vector<std::pair<void *, size_t>> pool;   // device blocks of freed copies, reused by the next build
  size_t pool_bytes = 0;
  std::map<void *, size_t> block_size;
  // handles
  std::map<int64_t, std::unique_ptr<Region>> regions;
  std::map<int64_t, std::unique_ptr<Copy>> copies;
  std::map<int64_t, std::unique_ptr<Batch>> batches;
  int64_t next_id = 1;
  // scratch
  DevBuf s_raw, s_exc, s_ts, s_u, s_fo, s_tsorted, s_partial, s_state, s_out[2][2], s_str, s_plan, s_sample[3];
  MgFastqChunk fq;                                 // corrupt-reads: the input chunk and its newline index
  DevBuf c_out[2], c_sz[2], c_off[2], c_draw[4];
  DevBuf b_units, b_arr;                           // a batch of small units: unit table; per-unit counts and their prefixes
  HostBuf h_stage;                                 // the variant arrays of a build on their way to the device (one DMA from page-locked memory)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
  cudaStream_t copy_stream = nullptr;              // D2H of finished units, overlapping the next unit's kernels
  cudaEvent_t ev_d2h[2] = {nullptr, nullptr};      // per output-buffer set: its last D2H has finished
  int ob = 0;                                      // output-buffer set of the next unit
  int last_ob = 0; int64_t last_bytes = 0;         // where the most recent unit's bytes are (mg_unit_read_async)
  double plan_ms = 0;
  double emit_ms = 0; int64_t emit_launches = 0, emit_bytes = 0, total_launches = 0;
  // drain thread: streams finished units from the device output buffers into an mg_sink
  struct DrainJob {
    mg_sink *sink; int producer; int64_t unit; int ob; int64_t bytes;
    // a batch of small units in one stream: their schedule indices and the prefix of their sizes (n + 1 entries)
    std::shared_ptr<std::vector<int64_t>> units, base;
  };
  std::thread drain_thread;
  std::mutex dmu; std::condition_variable dcv;
  std::deque<DrainJob> djobs;
  int dbusy[2] = {0, 0};                            // queued or running drains per output-buffer set
  bool dstop = false, dfailed = false;
  std::string derr;
  cudaEvent_t ev_drain[2] = {nullptr, nullptr};
  double d_wait_slot_ms = 0, d_wait_copy_ms = 0, d_idle_ms = 0; int64_t d_bytes = 0;   // MG_TIMING: where the drain thread's time went
};

namespace {

int fail(mg_ctx *c, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  if (c) c->err = buf;
  return code;
}

// Vose's alias method over K outcomes with probabilities q (sum 1): entry i = prob << alias_bits | alias,
// prob quantised to prob_bits.  A draw takes idx uniform in [0, K) and frac uniform in [0, 2^prob_bits):
// outcome = frac < prob ? idx : alias.
void vose_raw(std::vector<double> q, int K, std::vector<double> &prob, std::vector<int> &alias) {
  std::vector<int> small, large;
  for (int i = 0; i < K; i++) { q[i] *= K; (q[i] < 1.0 ? small : large).push_back(i); }
  prob.assign(K, 1.0); alias.resize(K);
  for (int i = 0; i < K; i++) alias[i] = i;
  while (!small.empty() && !large.empty()) {
    int s = small.back(); small.pop_back();
    int l = large.back(); large.pop_back();
    prob[s] = q[s]; alias[s] = l;
    q[l] = (q[l] + q[s]) - 1.0;
    (q[l] < 1.0 ? small : large).push_back(l);
  }
}

void vose(std::vector<double> q, int K, int prob_bits, int alias_bits, uint32_t *out) {
  std::vector<double> prob; std::vector<int> alias;
  vose_raw(q, K, prob, alias);
  const double scale = (double)(1u << prob_bits);
  for (int i = 0; i < K; i++) {
    double pr = prob[i] < 0.0 ? 0.0 : (prob[i] > 1.0 ? 1.0 : prob[i]);
    uint32_t pq = (uint32_t)std::floor(pr * scale + 0.5);
    if (pq > (1u << prob_bits)) pq = 1u << prob_bits;
    if (prob_bits + alias_bits == 32 && pq == (1u << prob_bits)) pq -= 1;   // no room for the 2^bits value
    out[i] = (pq << alias_bits) | (uint32_t)alias[i];
  }
}

// Outcome probabilities of searchsorted(cum, u, side='left') for u uniform in [0,1): outcome b =
// number of entries < u, b in [0, n]; outcomes above `clip` are folded into `clip`.
std::vector<double> ss_left_probs(const double *cum, int n, int K, int clip) {
  std::vector<double> q(K, 0.0);
  double prev = 0.0;
  for (int b = 0; b < n; b++) {
    double c = cum[b]; if (c > 1.0) c = 1.0; if (c < prev) c = prev;
    if (std::min(b, clip) < K) q[std::min(b, clip)] += c - prev;   // narrow tables are only used where this mass is zero
    prev = c;
  }
  if (std::min(n, clip) < K) q[std::min(n, clip)] += 1.0 - prev;
  return q;
}

// One (mate, cycle) of the quality model as the list of its outcomes (q, s) with non-zero mass
// (MgCorruptCtx in mg_core.cuh): quality q clipped to 93 (illumina.py:156); s = 0 "called correctly"
// with P(q) (1 - phred_p[q]), s = 1..3 "called as base ^ s" with P(q) phred_p[q] / 3 each.
// code = s << qb | q.
struct Outcome { uint32_t code; double mass; };

std::vector<Outcome> row_outcomes(const double *cum, int n_bq, const double *phred_p, int qb) {
  const std::vector<double> q = ss_left_probs(cum, n_bq, 94, 93);
  std::vector<Outcome> out;
  for (int b = 0; b < 94; b++) {
    if (!(q[b] > 0.0)) continue;
    const double p = b < 100 ? phred_p[b] : 0.0;
    const double m0 = q[b] * (1.0 - p), m = q[b] * p / 3.0;
    if (m0 > 0.0) out.push_back({(uint32_t)b, m0});
    if (m > 0.0) for (uint32_t sub = 1; sub <= 3; sub++) out.push_back({(sub << qb) | (uint32_t)b, m});
  }
  return out;
}

// Vose alias row of one (mate, cycle): entry = thr << (32 - tb) | self code << cb | alias code,
// (tb, cb) = (16, 8) or (14, 9).  Entries beyond the outcome list have threshold 0 and carry their
// alias' code twice; an entry whose threshold rounds to 0 (to the maximum) carries its alias' (its own)
// code in both fields, so quantisation never produces an outcome the model gives no mass.
void build_joint_row(const double *cum, int n_bq, const double *phred_p, int K, int code9, uint32_t *out) {
  const int tb = code9 ? 14 : 16, cb = code9 ? 9 : 8;
  const std::vector<Outcome> oc = row_outcomes(cum, n_bq, phred_p, code9 ? 7 : 6);
  double tot = 0.0;
  for (const Outcome &o : oc) tot += o.mass;
  std::vector<double> q((size_t)K, 0.0);
  for (size_t i = 0; i < oc.size(); i++) q[i] = oc[i].mass / tot;
  std::vector<double> prob; std::vector<int> alias;
  vose_raw(q, K, prob, alias);
  for (int i = 0; i < K; i++) {
    const double pr = prob[i] < 0.0 ? 0.0 : (prob[i] > 1.0 ? 1.0 : prob[i]);
    uint32_t t = (uint32_t)std::floor(pr * (double)(1u << tb) + 0.5);
    if (t > (1u << tb) - 1u) t = (1u << tb) - 1u;
    uint32_t a = (size_t)alias[i] < oc.size() ? oc[(size_t)alias[i]].code : oc[0].code;
    uint32_t sf = (size_t)i < oc.size() ? oc[(size_t)i].code : a;
    if (t == 0) sf = a;
    if (t == (1u << tb) - 1u) a = sf;
    out[i] = (t << (32 - tb)) | (sf << cb) | a;
  }
}

struct Timer {   // MG_TIMING=1: host-side section timings on stderr
  const char *name; double t0; bool on;
  static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
  explicit Timer(const char *n) : name(n), t0(now()), on(getenv("MG_TIMING") != nullptr) {}
  void lap(const char *what) { if (on) { double t = now(); fprintf(stderr, "[mg] %s/%s %.2f ms\n", name, what, t - t0); t0 = t; } }
};

}  // namespace

namespace {

// Device blocks of freed regions / chromosome copies are kept and handed to the next build: cudaMalloc and
// cudaFree wait for the device -- with device-to-host copies of finished units always in flight that is
// milliseconds per call, and a worker that builds many copies per step (units pulled dynamically by several
// processes: every rank meets most chromosomes) then starves its own drain thread.  Best fit among the blocks
// that waste at most 4x / 16 MB; the blocks of a genome's chromosomes differ by 5x in size, so after the first
// pass over the genome nearly every request is served from here.
cudaError_t pool_get(mg_ctx *ctx, void **p, size_t bytes) {
  int best = -1;
  const size_t limit = std::max(4 * bytes, bytes + ((size_t)16 << 20));
  for (size_t i = 0; i < ctx->pool.size(); i++)
    if (ctx->pool[i].second >= bytes && ctx->pool[i].second <= limit &&
        (best < 0 || ctx->pool[i].second < ctx->pool[best].second)) best = (int)i;
  if (best >= 0) { *p = ctx->pool[best].first; ctx->pool_bytes -= ctx->pool[best].second; ctx->pool.erase(ctx->pool.begin() + best); return cudaSuccess; }
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess && !ctx->pool.empty()) {          // out of memory with blocks in reserve: give them back and try again
    cudaGetLastError();
    for (auto &b : ctx->pool) { ctx->block_size.erase(b.first); cudaFree(b.first); }
    ctx->pool.clear(); ctx->pool_bytes = 0;
    e = cudaMalloc(p, bytes);
  }
  if (e == cudaSuccess) ctx->block_size[*p] = bytes;
  return e;
}

void pool_free(mg_ctx *ctx, void *p) {
  if (!p) return;
  if (ctx) {
    auto it = ctx->block_size.find(p);
    if (it != ctx->block_size.end() && ctx->pool.size() < 4096 && ctx->pool_bytes + it->second <= ((size_t)48 << 30)) {
      ctx->pool.push_back({p, it->second}); ctx->pool_bytes += it->second;
      return;
    }
    if (it != ctx->block_size.end()) ctx->block_size.erase(it);
  }
  cudaFree(p);
}

Region::~Region() { pool_free(owner, d_ref); pool_free(owner, d_exc); }
Copy::~Copy() { pool_free(owner, d_nodes); pool_free(owner, d_hap); pool_free(owner, d_blk); pool_free(owner, d_exc); pool_free(owner, d_eblk); }

}  // namespace

extern "C" {

int mg_device_count(void) {
  int n = 0;
  return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

int mg_ctx_create(int device, void *stream, mg_ctx **out) {
  if (!out) return MG_EINVAL;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0 || device < 0 || device >= n) {
    fprintf(stderr, "mitty_b200: no usable CUDA device %d (%s); this engine has no CPU fallback\n", device,
            e != cudaSuccess ? cudaGetErrorString(e) : "device count");
    return MG_ECUDA;
  }
  if (cudaSetDevice(device) != cudaSuccess) return MG_ECUDA;
  mg_ctx *ctx = new mg_ctx();
  ctx->device = device;
  if (stream) ctx->stream = reinterpret_cast<cudaStream_t>(stream);
  else { if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return MG_ECUDA; } ctx->own_stream = true; }
  cudaError_t ce = cudaEventCreate(&ctx->ev0);
  if (ce == cudaSuccess) ce = cudaEventCreate(&ctx->ev1);
  if (ce == cudaSuccess) ce = cudaEventCreate(&ctx->ev2);
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ctx->ev_d2h[0], cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ctx->ev_d2h[1], cudaEventDisableTiming);
  if (ce != cudaSuccess) {
    fprintf(stderr, "mitty_b200: cannot create the context's streams / events on device %d: %s\n", device, cudaGetErrorString(ce));
    mg_ctx_destroy(ctx);
    return MG_ECUDA;
  }
  *out = ctx;
  return MG_OK;
}

void mg_ctx_destroy(mg_ctx *ctx) {
  if (!ctx) return;
  DeviceGuard g(ctx->device);
  if (ctx->drain_thread.joinable()) {
    { std::lock_guard<std::mutex> lk(ctx->dmu); ctx->dstop = true; }
    ctx->dcv.notify_all();
    ctx->drain_thread.join();
  }
  for (int i = 0; i < 2; i++) if (ctx->ev_drain[i]) cudaEventDestroy(ctx->ev_drain[i]);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
  for (int i = 0; i < 2; i++) if (ctx->ev_d2h[i]) cudaEventDestroy(ctx->ev_d2h[i]);
  ctx->batches.clear(); ctx->regions.clear(); ctx->copies.clear();
  for (auto &b : ctx->pool) cudaFree(b.first);
  ctx->pool.clear(); ctx->block_size.clear();
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->ev2) cudaEventDestroy(ctx->ev2);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *mg_last_error(mg_ctx *ctx) { return ctx ? ctx->err.c_str() : mg_bam_host_error(); }

int mg_synchronize(mg_ctx *ctx) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

int mg_host_alloc(mg_ctx *ctx, int64_t bytes, void **out) {
  if (!ctx || !out || bytes <= 0) return fail(ctx, MG_EINVAL, "mg_host_alloc: bad arguments");
  DeviceGuard g(ctx->device);
  MG_CK(ctx, cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable));
  return MG_OK;
}

int mg_host_free(mg_ctx *ctx, void *p) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->copy_stream) MG_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));   // the pinned FASTQ buffers are written by this stream
  MG_CK(ctx, cudaFreeHost(p));
  return MG_OK;
}

int mg_model_load(mg_ctx *ctx, const double *cum_tlen, int n_tlen, const double *cum_bq_mat, int n_mates, int n_cycles,
                  int n_bq, const double *phred_p, int rlen) {
  if (!ctx || !cum_tlen || !cum_bq_mat || !phred_p || n_tlen <= 0 || n_mates < 1 || n_cycles <= 0 || n_bq <= 0 || rlen <= 0)
    return fail(ctx, MG_EINVAL, "mg_model_load: bad arguments");
  DeviceGuard g(ctx->device);
  MG_CK(ctx, ctx->m_tlen.need(sizeof(double) * n_tlen));
  MG_CK(ctx, ctx->m_bq.need(sizeof(double) * (size_t)n_mates * n_cycles * n_bq));
  MG_CK(ctx, ctx->m_phred.need(sizeof(double) * 100));
  MG_CK(ctx, cudaMemcpyAsync(ctx->m_tlen.p, cum_tlen, sizeof(double) * n_tlen, cudaMemcpyHostToDevice, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(ctx->m_bq.p, cum_bq_mat, sizeof(double) * (size_t)n_mates * n_cycles * n_bq, cudaMemcpyHostToDevice, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(ctx->m_phred.p, phred_p, sizeof(double) * 100, cudaMemcpyHostToDevice, ctx->stream));
  // production-mode tables: one joint (quality, substitution) alias row per (mate, cycle).  Built
  // twice: for the emit kernel over the cycles a read of this model has (rlen), and for the standalone
  // corrupt kernel over every cycle (reads of any length up to n_cycles; the rows beyond the model's
  // max_rlen are all-zero, i.e. quality 93, which needs the 9-bit codes).
  for (int t = 0; t < 2; t++) {
    const int rows = t == 0 ? std::min(rlen, n_cycles) : n_cycles;
    int code9 = 0; size_t longest = 1;
    for (int m = 0; m < n_mates; m++)
      for (int c = 0; c < rows; c++) {
        const double *row = cum_bq_mat + ((size_t)m * n_cycles + c) * n_bq;
        const std::vector<double> qm = ss_left_probs(row, n_bq, 94, 93);
        for (int b = 64; b < 94; b++) if (qm[b] > 0.0) code9 = 1;
        longest = std::max(longest, row_outcomes(row, n_bq, phred_p, 7).size());
      }
    int ks = 5;
    while ((size_t)1 << ks < longest) ks++;
    const int K = 1 << ks;
    ctx->a_kshift[t] = ks; ctx->a_code9[t] = code9; ctx->a_rows[t] = rows;
    ctx->h_alias[t].assign((size_t)n_mates * n_cycles * K, 0u);
    for (int m = 0; m < n_mates; m++)
      for (int c = 0; c < rows; c++) {
        const size_t r = (size_t)m * n_cycles + c;
        build_joint_row(cum_bq_mat + r * n_bq, n_bq, phred_p, K, code9, ctx->h_alias[t].data() + r * K);
      }
    MG_CK(ctx, ctx->m_alias[t].need(4 * ctx->h_alias[t].size()));
    MG_CK(ctx, cudaMemcpyAsync(ctx->m_alias[t].p, ctx->h_alias[t].data(), 4 * ctx->h_alias[t].size(), cudaMemcpyHostToDevice, ctx->stream));
  }
  ctx->has_tlen_alias = (n_tlen + 1 <= MG_TLEN_K);
  if (ctx->has_tlen_alias) {
    std::vector<uint32_t> ta(MG_TLEN_K);
    vose(ss_left_probs(cum_tlen, n_tlen, MG_TLEN_K, n_tlen), MG_TLEN_K, 22, 10, ta.data());
    MG_CK(ctx, ctx->m_tlen_alias.need(4 * MG_TLEN_K));
    MG_CK(ctx, cudaMemcpy(ctx->m_tlen_alias.p, ta.data(), 4 * MG_TLEN_K, cudaMemcpyHostToDevice));
  }
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->n_tlen = n_tlen; ctx->n_mates = n_mates; ctx->n_cycles = n_cycles; ctx->n_bq = n_bq; ctx->rlen = rlen;
  return MG_OK;
}

int mg_model_tables(mg_ctx *ctx, int32_t which, uint32_t *alias_out, int64_t alias_cap, int32_t *kshift, int32_t *code9, int32_t *n_rows) {
  if (!ctx || ctx->rlen == 0) return fail(ctx, MG_EINVAL, "no read model loaded");
  if (which != 0 && which != 1) return fail(ctx, MG_EINVAL, "which must be 0 (emit kernel) or 1 (corrupt kernel)");
  const std::vector<uint32_t> &h = ctx->h_alias[which];
  if (kshift) *kshift = ctx->a_kshift[which];
  if (code9) *code9 = ctx->a_code9[which];
  if (n_rows) *n_rows = ctx->a_rows[which];
  if (alias_out) {
    if (alias_cap < (int64_t)h.size()) return fail(ctx, MG_ECAP, "alias table needs %lld entries", (long long)h.size());
    memcpy(alias_out, h.data(), 4 * h.size());
  }
  return MG_OK;
}

// ---- region ---------------------------------------------------------------------------------

}  // extern "C"

// raw reference bytes (host) -> 2-bit packed words + sorted exception runs of a Region (k_pack_ref)
static int load_packed(mg_ctx *ctx, const uint8_t *ref_bytes, int64_t len, int64_t bed_start, std::unique_ptr<Region> &R) {
  R.reset(new Region());
  uint32_t exc_cap = 1u << 20;                        // grown on demand: a soft-masked chromosome has ~10^6 case runs
  R->len = len; R->bed_start = bed_start;
  int64_t words = (len + 15) / 16;
  R->owner = ctx;
  MG_CK(ctx, pool_get(ctx, (void **)&R->d_ref, sizeof(uint32_t) * (words + 2 * MG_HAP_PAD)));
  MG_CK(ctx, cudaMemsetAsync(R->d_ref, 0, sizeof(uint32_t) * (words + 2 * MG_HAP_PAD), ctx->stream));
  if (len > 0) {
    MG_CK(ctx, ctx->s_raw.need((size_t)len + 32));
    MG_CK(ctx, cudaMemcpyAsync(ctx->s_raw.p, ref_bytes, (size_t)len, cudaMemcpyHostToDevice, ctx->stream));
    uint32_t cnt[2] = {0, 0};
    int64_t *d_start = nullptr, *d_end = nullptr;
    uint8_t *d_byte = nullptr;
    for (int attempt = 0; attempt < 2; attempt++) {
      // exception scratch: [cnt u32 x2 (padded to 16 B)][start i64 x cap][end i64 x cap][byte u8 x cap]
      MG_CK(ctx, ctx->s_exc.need(16 + (size_t)exc_cap * 17));
      uint8_t *eb = ctx->s_exc.as<uint8_t>();
      uint32_t *d_cnt = reinterpret_cast<uint32_t *>(eb);
      d_start = reinterpret_cast<int64_t *>(eb + 16);
      d_end = d_start + exc_cap;
      d_byte = reinterpret_cast<uint8_t *>(d_end + exc_cap);
      MG_CK(ctx, cudaMemsetAsync(d_cnt, 0, 16, ctx->stream));
      mg_launch_pack_ref(ctx->s_raw.as<uint8_t>(), len, R->d_ref + MG_HAP_PAD, d_cnt, d_start, d_byte, d_end, exc_cap, ctx->stream);
      ctx->total_launches++;
      MG_CK(ctx, cudaGetLastError());
      MG_CK(ctx, cudaMemcpyAsync(cnt, d_cnt, 8, cudaMemcpyDeviceToHost, ctx->stream));
      MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
      if (cnt[0] != cnt[1]) return fail(ctx, MG_ECUDA, "internal: exception run starts (%u) != ends (%u)", cnt[0], cnt[1]);
      if (cnt[0] <= exc_cap) break;
      if (attempt == 1 || cnt[0] > (1u << 27))
        return fail(ctx, MG_EVALUE, "reference has %u runs of non-ACGT bytes / lower-case stretches (limit 2^27)", cnt[0]);
      exc_cap = cnt[0];                               // second pass with room for every run
    }
    if (cnt[0]) {
      std::vector<int64_t> st(cnt[0]), en(cnt[0]);
      std::vector<uint8_t> by(cnt[0]);
      MG_CK(ctx, cudaMemcpy(st.data(), d_start, 8 * (size_t)cnt[0], cudaMemcpyDeviceToHost));
      MG_CK(ctx, cudaMemcpy(en.data(), d_end, 8 * (size_t)cnt[0], cudaMemcpyDeviceToHost));
      MG_CK(ctx, cudaMemcpy(by.data(), d_byte, (size_t)cnt[0], cudaMemcpyDeviceToHost));
      std::vector<uint32_t> order(cnt[0]);
      for (uint32_t i = 0; i < cnt[0]; i++) order[i] = i;
      std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return st[a] < st[b]; });
      std::sort(en.begin(), en.end());
      R->exc.resize(cnt[0]);
      std::vector<MgExc> dev(cnt[0]);
      for (uint32_t i = 0; i < cnt[0]; i++) {
        R->exc[i] = ExcRun{st[order[i]], en[i] - st[order[i]] + 1, by[order[i]]};
        dev[i] = MgExc{(uint32_t)R->exc[i].start, (uint32_t)R->exc[i].len, R->exc[i].byte, 0};
      }
      MG_CK(ctx, pool_get(ctx, (void **)&R->d_exc, sizeof(MgExc) * cnt[0]));
      MG_CK(ctx, cudaMemcpy(R->d_exc, dev.data(), sizeof(MgExc) * cnt[0], cudaMemcpyHostToDevice));
    }
  }
  return MG_OK;
}

extern "C" {

int mg_region_load(mg_ctx *ctx, const uint8_t *ref_bytes, int64_t len, int64_t bed_start, int64_t *region_id) {
  if (!ctx || !region_id || len < 0 || (len > 0 && !ref_bytes)) return fail(ctx, MG_EINVAL, "mg_region_load: bad arguments");
  if (len >= (int64_t)0xFFF00000ll) return fail(ctx, MG_EVALUE, "region of %lld bases exceeds the 2^32 addressing of one region", (long long)len);
  DeviceGuard g(ctx->device);
  std::unique_ptr<Region> R;
  const int rc = load_packed(ctx, ref_bytes, len, bed_start, R);
  if (rc) return rc;
  int64_t id = ctx->next_id++;
  ctx->regions[id] = std::move(R);
  *region_id = id;
  return MG_OK;
}

int mg_region_free(mg_ctx *ctx, int64_t region_id) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  return ctx->regions.erase(region_id) ? MG_OK : fail(ctx, MG_EINVAL, "unknown region %lld", (long long)region_id);
}

// ---- chromosome copy --------------------------------------------------------------------------

}  // extern "C"

// Node tables, haplotype, block table and exception runs of ONE or MANY chromosome copies ("segments",
// MgSeg) over one packed reference: the shared body of mg_copy_build (one segment) and mg_batch_build (all
// small regions of a BED at once).  One stream synchronisation; seg_out = the per-segment results.
static int build_segments(mg_ctx *ctx, const uint32_t *d_ref, const MgExc *d_rexc, int n_rexc, const std::vector<MgSeg> &segs,
                          int64_t n_var, const int64_t *pos, const uint8_t *op, const int64_t *oplen, const uint8_t *alt_pool,
                          const int64_t *alt_off, Copy &C, std::vector<MgSegOut> &seg_out) {
  Timer tm("copy_build");
  const int V = (int)n_var, S = (int)segs.size();
  const int64_t alt_bytes = V ? alt_off[V] : 0;
  if (alt_bytes >= (1ll << 32)) return fail(ctx, MG_EVALUE, "alt allele pool of %lld bytes exceeds 2^32", (long long)alt_bytes);
  // the walk's chain argument needs POS sorted inside every segment (records of an indexed fetch always are)
  for (const MgSeg &sg : segs)
    for (int i = sg.v0 + 1; i < sg.v1; i++)
      if (pos[i] < pos[i - 1]) return fail(ctx, MG_EVALUE, "variants are not sorted by POS (record %d: %lld after %lld)", i - sg.v0, (long long)pos[i], (long long)pos[i - 1]);
  tm.lap("check");

  // -- scratch layout (all 16-byte aligned): the inputs (variant arrays, segments, alt pool) first and contiguous -- they
  // travel as ONE copy from a page-locked staging buffer: pageable copies are cut into small staged pieces by the driver,
  // and each piece queues behind the 64 MB device-to-host pieces of the units being drained (14 ms per build on average,
  // up to 180 ms, measured with two ranks sharing a genome) --, then walk state and node-sized arrays
  const size_t nv = (size_t)V, ns = (size_t)S, ne = nv + ns, max_nodes = 2 * nv + ns;
  auto al = [](size_t x) { return (x + 15) & ~(size_t)15; };
  size_t o = 0;
  const size_t o_pos = o; o += al(8 * (nv + 1));
  const size_t o_oplen = o; o += al(8 * (nv + 1));
  const size_t o_altoff = o; o += al(8 * (nv + 2));
  const size_t o_op = o; o += al(nv + 1);
  const size_t o_seg = o; o += al(sizeof(MgSeg) * ns);
  const size_t o_alt = o; o += al((size_t)alt_bytes + 16);
  const size_t in_bytes = o;
  const size_t o_nxt = o; o += al(4 * (nv + 1));
  const size_t o_j0 = o; o += al(4 * (nv + 1));
  const size_t o_j1 = o; o += al(4 * (nv + 1));
  const size_t o_pred = o; o += al(4 * (nv + 1));
  const size_t o_mark = o; o += al(nv + 1);
  const size_t o_packed = o; o += al(8 * (ne + 2));
  const size_t o_scanned = o; o += al(8 * (ne + 3));
  const size_t o_tmp = o; o += al(8 * ((std::max(max_nodes, ne) + 2) / 1024 + 4));
  const size_t o_nalt = o; o += al(4 * (max_nodes + 1));
  const size_t o_ecnt = o; o += al(8 * (max_nodes + 2));
  const size_t o_eoff = o; o += al(8 * (max_nodes + 3));
  const size_t o_sum = o; o += al(sizeof(MgWalkSummary));
  const size_t o_segout = o; o += al(sizeof(MgSegOut) * ns);
  MG_CK(ctx, ctx->s_str.need(o));
  uint8_t *sb = ctx->s_str.as<uint8_t>();
  MG_CK(ctx, pool_get(ctx, (void **)&C.d_nodes, sizeof(MgNode) * std::max<size_t>(max_nodes, 1)));
  MG_CK(ctx, ctx->h_stage.need(in_bytes));
  {
    uint8_t *hs = static_cast<uint8_t *>(ctx->h_stage.p);
    if (V) {
      memcpy(hs + o_pos, pos, 8 * nv); memcpy(hs + o_oplen, oplen, 8 * nv); memcpy(hs + o_altoff, alt_off, 8 * (nv + 1));
      memcpy(hs + o_op, op, nv);
      if (alt_bytes) memcpy(hs + o_alt, alt_pool, (size_t)alt_bytes);
    }
    memcpy(hs + o_seg, segs.data(), sizeof(MgSeg) * ns);
    MG_CK(ctx, cudaMemcpyAsync(sb, hs, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  MgWalkParams W;
  W.pos = reinterpret_cast<int64_t *>(sb + o_pos); W.oplen = reinterpret_cast<int64_t *>(sb + o_oplen);
  W.alt_off = reinterpret_cast<int64_t *>(sb + o_altoff); W.op = sb + o_op;
  W.n_var = V;
  W.segs = reinterpret_cast<const MgSeg *>(sb + o_seg); W.n_seg = S; W.seg_out = reinterpret_cast<MgSegOut *>(sb + o_segout);
  W.nxt = reinterpret_cast<uint32_t *>(sb + o_nxt);
  W.jump[0] = reinterpret_cast<uint32_t *>(sb + o_j0); W.jump[1] = reinterpret_cast<uint32_t *>(sb + o_j1);
  W.mark = sb + o_mark; W.pred = reinterpret_cast<int32_t *>(sb + o_pred);
  W.packed = reinterpret_cast<int64_t *>(sb + o_packed); W.scanned = reinterpret_cast<int64_t *>(sb + o_scanned);
  W.scan_tmp = reinterpret_cast<int64_t *>(sb + o_tmp);
  W.nodes = C.d_nodes; W.node_alt = reinterpret_cast<uint32_t *>(sb + o_nalt);
  W.sum = reinterpret_cast<MgWalkSummary *>(sb + o_sum);
  ctx->total_launches += mg_launch_walk(W, ctx->stream) + 4;   // + exception count and its scan
  // exception runs of the copy: count per node, scan
  int64_t *e_cnt = reinterpret_cast<int64_t *>(sb + o_ecnt), *e_off = reinterpret_cast<int64_t *>(sb + o_eoff);
  mg_launch_exc_count(C.d_nodes, W.node_alt, W.sum, (int)max_nodes, sb + o_alt, d_rexc, n_rexc, e_cnt, ctx->stream);
  mg_launch_scan_i64(e_cnt, e_off, (int64_t)max_nodes, W.scan_tmp, ctx->stream);
  MG_CK(ctx, cudaGetLastError());
  MgWalkSummary sum;
  int64_t n_exc = 0;
  seg_out.resize(ns);
  MG_CK(ctx, cudaMemcpyAsync(&sum, W.sum, sizeof sum, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(&n_exc, e_off + max_nodes, 8, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(seg_out.data(), W.seg_out, sizeof(MgSegOut) * ns, cudaMemcpyDeviceToHost, ctx->stream));
  tm.lap("enqueue walk");
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));             // also: the caller's arrays have been consumed
  tm.lap("walk");

  if (sum.err != ~0ull) {
    const long long i = (long long)(sum.err >> 8);
    switch ((int)(sum.err & 0xFF)) {
      case 1: return fail(ctx, MG_EVALUE, "SNP at %lld has an ALT of length %lld", (long long)pos[i], (long long)(alt_off[i + 1] - alt_off[i]));
      case 2: return fail(ctx, MG_EVALUE, "insertion at %lld: oplen %lld does not match its ALT", (long long)pos[i], (long long)oplen[i]);
      default: return fail(ctx, MG_EVALUE, "variant %lld has op %d (expected X, I or D) or a negative length", i, (int)op[i]);
    }
  }
  if (sum.n_nodes == 0 || sum.ends_in_d)
    return fail(ctx, MG_EVALUE, "a deletion crosses the end of the region: the reference's node list would end in 'D' "
                "(readgenerate.py:192 assumes it never does); trim the BED region or the VCF");
  if (sum.bad) return fail(ctx, MG_EVALUE, "a variant reaches beyond the region, or positions / node lengths exceed 2^31 (haplotypes 2^32)");
  const size_t nn = (size_t)sum.n_nodes;
  const int64_t hap_len = sum.hap_len;
  if (hap_len >= (int64_t)0xFFF00000ll) return fail(ctx, MG_EVALUE, "haplotype of %lld bases exceeds 2^32", (long long)hap_len);
  C.n_nodes = (int64_t)nn;
  C.n_exc = n_exc;
  C.hap_len = hap_len;

  // -- device builds that need the sizes: exception runs, haplotype, block table
  C.hap_words = (hap_len + 15) / 16;
  C.n_blk = (int)((hap_len >> BLK_SHIFT) + 1);
  MG_CK(ctx, pool_get(ctx, (void **)&C.d_hap, sizeof(uint32_t) * (C.hap_words + 2 * MG_HAP_PAD)));
  MG_CK(ctx, pool_get(ctx, (void **)&C.d_blk, sizeof(uint32_t) * C.n_blk));
  MG_CK(ctx, pool_get(ctx, (void **)&C.d_exc, sizeof(MgExc) * std::max<size_t>(1, (size_t)n_exc)));
  if (n_exc) {
    mg_launch_exc_write(C.d_nodes, W.node_alt, W.sum, (int)max_nodes, sb + o_alt, d_rexc, n_rexc, e_off, C.d_exc, ctx->stream);
    MG_CK(ctx, pool_get(ctx, (void **)&C.d_eblk, sizeof(uint32_t) * ((size_t)C.n_blk + 1)));
    mg_launch_eblk_table(C.d_exc, (int)n_exc, C.d_eblk, C.n_blk + 1, BLK_SHIFT, ctx->stream);
    ctx->total_launches++;
  }
  MG_CK(ctx, cudaMemsetAsync(C.d_hap, 0, sizeof(uint32_t) * MG_HAP_PAD, ctx->stream));
  MG_CK(ctx, cudaMemsetAsync(C.d_hap + MG_HAP_PAD + C.hap_words, 0, sizeof(uint32_t) * MG_HAP_PAD, ctx->stream));
  mg_launch_blk_table(C.d_nodes, (int)nn, C.d_blk, C.n_blk, BLK_SHIFT, ctx->stream);
  if (hap_len > 0)
    mg_launch_hap_build(d_ref, sb + o_alt, C.d_nodes, W.node_alt, (int)nn, C.d_blk, BLK_SHIFT, C.n_blk, (uint32_t)hap_len, C.d_hap + MG_HAP_PAD,
                        C.hap_words, ctx->stream);
  ctx->total_launches += 2 + (n_exc ? 1 : 0);
  MG_CK(ctx, cudaGetLastError());
  tm.lap("enqueue build");                            // stream-ordered: units launched next wait for these kernels
  return MG_OK;
}

extern "C" {

int mg_copy_build(mg_ctx *ctx, int64_t region_id, int64_t n_var, const int64_t *pos, const uint8_t *op, const int64_t *oplen,
                  const uint8_t *alt_pool, const int64_t *alt_off, int64_t *copy_id, int64_t *p_min, int64_t *p_max,
                  int64_t *n_nodes) {
  if (!ctx || !copy_id || n_var < 0 || (n_var > 0 && (!pos || !op || !oplen || !alt_pool || !alt_off)))
    return fail(ctx, MG_EINVAL, "mg_copy_build: bad arguments");
  if (n_var >= (1ll << 28)) return fail(ctx, MG_EVALUE, "%lld variants on one copy (limit 2^28)", (long long)n_var);
  auto it = ctx->regions.find(region_id);
  if (it == ctx->regions.end()) return fail(ctx, MG_EINVAL, "unknown region %lld", (long long)region_id);
  DeviceGuard g(ctx->device);
  Region &R = *it->second;
  std::unique_ptr<Copy> C(new Copy());
  C->region_id = region_id;
  C->owner = ctx;
  MgSeg sg; memset(&sg, 0, sizeof sg);
  sg.v0 = 0; sg.v1 = (int32_t)n_var; sg.roff = 0; sg.start1 = R.bed_start + 1; sg.region_len = R.len;   // ref_start_pos, readgenerate.py:190; also p_min
  std::vector<MgSegOut> so;
  const int rc = build_segments(ctx, R.d_ref + MG_HAP_PAD, R.d_exc, (int)R.exc.size(), std::vector<MgSeg>(1, sg), n_var, pos, op, oplen, alt_pool, alt_off, *C, so);
  if (rc) return rc;
  C->p_min = sg.start1;                               // readgenerate.py:192: nodes[0].ps
  C->p_max = sg.start1 + C->hap_len;                  // nodes[-1].ps + nodes[-1].oplen (the last node is never 'D')
  int64_t id = ctx->next_id++;
  if (p_min) *p_min = C->p_min;
  if (p_max) *p_max = C->p_max;
  if (n_nodes) *n_nodes = C->n_nodes;
  ctx->copies[id] = std::move(C);
  *copy_id = id;
  return MG_OK;
}

int mg_copy_free(mg_ctx *ctx, int64_t copy_id) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  return ctx->copies.erase(copy_id) ? MG_OK : fail(ctx, MG_EINVAL, "unknown copy %lld", (long long)copy_id);
}

int mg_copy_nodes(mg_ctx *ctx, int64_t copy_id, int64_t *ps, int64_t *pr, uint8_t *op, int64_t *oplen) {
  if (!ctx) return MG_EINVAL;
  auto it = ctx->copies.find(copy_id);
  if (it == ctx->copies.end()) return fail(ctx, MG_EINVAL, "unknown copy %lld", (long long)copy_id);
  DeviceGuard g(ctx->device);
  const Copy &C = *it->second;
  std::vector<MgNode> dn((size_t)C.n_nodes);
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  MG_CK(ctx, cudaMemcpy(dn.data(), C.d_nodes, sizeof(MgNode) * dn.size(), cudaMemcpyDeviceToHost));
  for (size_t k = 0; k < dn.size(); k++) {   // the device table back in the reference's terms (rpc.py:5-35)
    ps[k] = C.p_min + (int64_t)dn[k].key - (dn[k].op == 'D' ? 1 : 0);
    pr[k] = dn[k].pr; op[k] = (uint8_t)dn[k].op; oplen[k] = dn[k].oplen;
  }
  return MG_OK;
}

int mg_copy_haplotype(mg_ctx *ctx, int64_t copy_id, uint8_t *out, int64_t cap) {
  if (!ctx || !out) return MG_EINVAL;
  auto it = ctx->copies.find(copy_id);
  if (it == ctx->copies.end()) return fail(ctx, MG_EINVAL, "unknown copy %lld", (long long)copy_id);
  DeviceGuard g(ctx->device);
  const Copy &C = *it->second;
  const int64_t n = C.p_max - C.p_min;
  if (cap < n) return fail(ctx, MG_ECAP, "haplotype needs %lld bytes", (long long)n);
  std::vector<uint32_t> w((size_t)C.hap_words);
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  if (C.hap_words) MG_CK(ctx, cudaMemcpy(w.data(), C.d_hap + MG_HAP_PAD, 4 * (size_t)C.hap_words, cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < n; i++) out[i] = (uint8_t)("ACGT"[(w[i >> 4] >> (2 * (i & 15))) & 3]);
  std::vector<MgExc> exc((size_t)C.n_exc);
  if (C.n_exc) MG_CK(ctx, cudaMemcpy(exc.data(), C.d_exc, sizeof(MgExc) * exc.size(), cudaMemcpyDeviceToHost));
  for (const MgExc &e : exc)
    for (uint32_t q = 0; q < e.len; q++) out[e.start + q] = e.byte == MG_EXC_CASE ? (uint8_t)(out[e.start + q] | 0x20) : (uint8_t)e.byte;
  return MG_OK;
}

// ---- work units -----------------------------------------------------------------------------------

static int fill_unit_params(mg_ctx *ctx, const mg_unit_desc *d, MgUnitParams &P, const Copy **copy_out, bool sample_only) {
  if (!d) return fail(ctx, MG_EINVAL, "null unit descriptor");
  if (ctx->rlen == 0) return fail(ctx, MG_EINVAL, "no read model loaded (mg_model_load)");
  if (d->n_candidates < 0 || d->n_candidates >= (1ll << 31)) return fail(ctx, MG_EVALUE, "n_candidates %lld out of range", (long long)d->n_candidates);
  memset(&P, 0, sizeof P);
  *copy_out = nullptr;
  if (sample_only && d->copy_id == 0) {
    if (d->p_max < d->p_min || d->p_max - d->p_min >= (int64_t)0xFFF00000ll) return fail(ctx, MG_EVALUE, "p_min/p_max span out of range");
    P.hap_len = (uint32_t)(d->p_max - d->p_min); P.p_min = d->p_min;
  } else {
    auto it = ctx->copies.find(d->copy_id);
    if (it == ctx->copies.end()) return fail(ctx, MG_EINVAL, "unknown copy %lld", (long long)d->copy_id);
    const Copy &C = *it->second;
    *copy_out = &C;
    P.hap = C.d_hap + MG_HAP_PAD; P.hap_len = (uint32_t)(C.p_max - C.p_min); P.p_min = C.p_min;
    P.nodes = C.d_nodes; P.n_nodes = (int)C.n_nodes;
    P.blk = C.d_blk; P.blk_shift = BLK_SHIFT; P.n_blk = C.n_blk;
    P.exc = C.d_exc; P.n_exc = (int)C.n_exc; P.eblk = C.d_eblk;
  }
  P.cum_tlen = ctx->m_tlen.as<double>(); P.n_tlen = ctx->n_tlen; P.rlen = ctx->rlen;
  P.tlen_alias = ctx->has_tlen_alias ? ctx->m_tlen_alias.as<uint32_t>() : nullptr;
  P.mode = d->mode; P.n_cand = (uint32_t)d->n_candidates;
  const size_t n = (size_t)d->n_candidates;
  if (d->mode == MG_MODE_PHILOX) {
    if (!(d->p > 0.0 && d->p < 1.0)) return fail(ctx, MG_EINVAL, "PHILOX mode needs 0 < p < 1");
    if (n) {
      MG_CK(ctx, ctx->s_tsorted.need(4 * n + 64));
      MG_CK(ctx, ctx->s_partial.need(8 * (n / 2048 + 2)));
      const MgUnitKeys K0 = mg_unit_keys(d->unit_seed, (uint32_t)n);
      mg_launch_gap_scan((uint32_t)n, d->p, K0.gap0, K0.gap1, ctx->s_tsorted.as<uint32_t>(),
                         ctx->s_partial.as<unsigned long long>(), ctx->stream);
      ctx->total_launches += 3;
    }
    P.ts_sorted = ctx->s_tsorted.as<uint32_t>();
    const MgUnitKeys K = mg_unit_keys(d->unit_seed, (uint32_t)n);
    P.key_tlen0 = K.tlen0; P.key_tlen1 = K.tlen1;
    P.key_perm0 = K.perm0; P.key_perm1 = K.perm1;
    P.perm_bits = K.perm_bits;
  } else if (d->mode == MG_MODE_DET || d->mode == MG_MODE_EXPLICIT) {
    if (n && (!d->ts || (!d->fo && !sample_only) || (d->mode == MG_MODE_DET ? !d->u_tlen : !d->tl))) return fail(ctx, MG_EINVAL, "deterministic mode needs ts, fo and u_tlen/tl arrays");
    if (n) {
      MG_CK(ctx, ctx->s_ts.need(8 * n)); MG_CK(ctx, ctx->s_u.need(8 * n)); MG_CK(ctx, ctx->s_fo.need(n));
      MG_CK(ctx, cudaMemcpyAsync(ctx->s_ts.p, d->ts, 8 * n, cudaMemcpyHostToDevice, ctx->stream));
      MG_CK(ctx, cudaMemcpyAsync(ctx->s_u.p, d->mode == MG_MODE_DET ? (const void *)d->u_tlen : (const void *)d->tl, 8 * n, cudaMemcpyHostToDevice, ctx->stream));
      if (d->fo) MG_CK(ctx, cudaMemcpyAsync(ctx->s_fo.p, d->fo, n, cudaMemcpyHostToDevice, ctx->stream));
    }
    P.ts_in = ctx->s_ts.as<int64_t>();
    if (d->mode == MG_MODE_DET) P.u_tlen = ctx->s_u.as<double>(); else P.tl_in = ctx->s_u.as<int64_t>();
    P.fo_in = ctx->s_fo.as<int8_t>();
  } else {
    return fail(ctx, MG_EINVAL, "unknown mode %d", d->mode);
  }
  return MG_OK;
}

int mg_sample_templates(mg_ctx *ctx, const mg_unit_desc *d, int64_t *ts_out, int64_t *te_out, int8_t *fo_out) {
  if (!ctx || !ts_out || !te_out || !fo_out) return fail(ctx, MG_EINVAL, "mg_sample_templates: bad arguments");
  DeviceGuard g(ctx->device);
  MgSampleParams S; const Copy *C;
  int rc = fill_unit_params(ctx, d, S.u, &C, true);
  if (rc) return rc;
  const size_t n = (size_t)d->n_candidates;
  if (!n) return MG_OK;
  MG_CK(ctx, ctx->s_sample[0].need(8 * n)); MG_CK(ctx, ctx->s_sample[1].need(8 * n)); MG_CK(ctx, ctx->s_sample[2].need(n));
  S.ts_out = ctx->s_sample[0].as<int64_t>(); S.te_out = ctx->s_sample[1].as<int64_t>(); S.fo_out = ctx->s_sample[2].as<int8_t>();
  mg_launch_sample(S, ctx->stream);
  ctx->total_launches++;
  MG_CK(ctx, cudaGetLastError());
  MG_CK(ctx, cudaMemcpyAsync(ts_out, S.ts_out, 8 * n, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(te_out, S.te_out, 8 * n, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(fo_out, S.fo_out, n, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

static int unit_generate(mg_ctx *ctx, const mg_unit_desc *d, uint8_t *out1, uint8_t *out2, int64_t cap, int64_t *n_bytes,
                         int64_t *n_templates, int64_t *n_te_kept, bool wait_copies) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  MgUnitParams P; const Copy *C;
  int rc = fill_unit_params(ctx, d, P, &C, false);
  if (rc) return rc;
  if (!d->qname_prefix || !d->qname_mid) return fail(ctx, MG_EINVAL, "qname_prefix / qname_mid missing");
  if (d->corrupt && d->mode != MG_MODE_PHILOX) return fail(ctx, MG_EINVAL, "fused corruption draws from Philox: use mg_corrupt_fastq for deterministic mode");
  if (d->corrupt && ctx->rlen > ctx->n_cycles) return fail(ctx, MG_EINDEX, "read length %d exceeds the model's %d cycles", ctx->rlen, ctx->n_cycles);
  if (d->corrupt && ctx->n_mates < 2) return fail(ctx, MG_EINVAL, "paired corruption needs a 2-mate model");
  const size_t n = (size_t)d->n_candidates;
  const int pl = (int)strlen(d->qname_prefix), ml = (int)strlen(d->qname_mid);
  const int L = ctx->rlen;

  // qname constants, tokenised on the host (mg_qn_const): they travel in the kernel parameters
  if (pl > MG_QN_MAX || ml > MG_QN_MAX) return fail(ctx, MG_EVALUE, "sample / chromosome name too long for the qname buffers (%d)", MG_QN_MAX);
  mg_qn_const(P.qn, reinterpret_cast<const uint8_t *>(d->qname_prefix), pl, reinterpret_cast<const uint8_t *>(d->qname_mid), ml, L);
  P.qn_len = pl + ml;
  {
    static const bool lsu = getenv("MG_COPYOUT_LSU") != nullptr;     // experiments: copy-out with plain loads / stores
    P.bulk = lsu ? 0 : 1;
  }
  P.corrupt = d->corrupt;
  P.cor.kshift = ctx->a_kshift[0]; P.cor.code9 = ctx->a_code9[0];
  P.cor.alias = ctx->m_alias[0].as<uint32_t>();
  P.cor.n_cycles = ctx->n_cycles; P.cor.n_mates = ctx->n_mates;
  P.cor.k0 = d->corrupt_seed; P.cor.k1 = d->unit_seed ^ 0x636f7231u;
  P.L_nd = mg_ndigits32((uint32_t)L);

  P.n_tiles = (int)((n + MG_PLAN_TILE - 1) / MG_PLAN_TILE);
  // per-warp stage of the emit kernel: 32 records with an average qname; larger batches are split
  int stage = 32 * (2 * L + 5 + 96);
  if (stage > 48 * 1024) stage = 48 * 1024;
  P.stage_cap = stage & ~15;
  int smem = 0;
  const int grid = mg_unit_grid(L, d->corrupt ? 1 + P.cor.code9 : 0, P.stage_cap, &smem);
  if (grid <= 0) return fail(ctx, MG_EVALUE, "the emit kernel's staging area (%d bytes for reads of %d bases) exceeds the shared memory of this device", smem, L);

  // scan state: [totals 4 x u64][tile counter (16 B)][descA][descB]
  const size_t state_bytes = 48 + 16 * (size_t)std::max(P.n_tiles, 1);
  MG_CK(ctx, ctx->s_state.need(state_bytes));
  uint8_t *sb = ctx->s_state.as<uint8_t>();
  P.totals = reinterpret_cast<unsigned long long *>(sb);
  P.tile_counter = reinterpret_cast<uint32_t *>(sb + 32);
  P.descA = reinterpret_cast<unsigned long long *>(sb + 48);
  P.descB = P.descA + std::max(P.n_tiles, 1);
  MG_CK(ctx, ctx->s_plan.need(sizeof(MgPlan) * std::max<size_t>(n, 1)));
  P.plan = ctx->s_plan.as<MgPlan>();

  // device output buffers: sized from an estimate, regrown to the exact size on overflow (the plan
  // stays valid: only the emit kernel is launched again)
  size_t est = n * (size_t)(2 * L + 5 + pl + ml + 12 + 2 * 36) / 6 * 5 + 4096;   // ~5/6 of the candidates survive
  const bool want_out = (out1 != nullptr) || (out2 != nullptr);
  unsigned long long tot[4] = {0, 0, 0, 0};
  MG_CK(ctx, cudaMemsetAsync(sb, 0, state_bytes, ctx->stream));
  MG_CK(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
  mg_launch_plan(P, ctx->stream);
  MG_CK(ctx, cudaGetLastError());
  {   // a drain still reading this buffer set (the unit before last) must finish first
    std::unique_lock<std::mutex> lk(ctx->dmu);
    while (ctx->dbusy[ctx->ob] > 0 && !ctx->dfailed) ctx->dcv.wait(lk);
    if (ctx->dfailed) return fail(ctx, MG_EVALUE, "output sink: %s", ctx->derr.c_str());
  }
  for (int attempt = 0; attempt < 2; attempt++) {
    DevBuf *ob = ctx->s_out[ctx->ob];
    if (ob[0].cap < est || ob[1].cap < est) MG_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));   // regrowing frees the old block
    MG_CK(ctx, ob[0].need(est)); MG_CK(ctx, ob[1].need(est));
    P.out[0] = ob[0].as<uint8_t>(); P.out[1] = ob[1].as<uint8_t>();
    P.cap = std::min(ob[0].cap, ob[1].cap);
    MG_CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_d2h[ctx->ob], 0));   // this buffer set's previous D2H must be done
    MG_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    mg_launch_unit(P, grid, smem, ctx->stream);
    MG_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    MG_CK(ctx, cudaGetLastError());
    MG_CK(ctx, cudaMemcpyAsync(tot, P.totals, sizeof tot, cudaMemcpyDeviceToHost, ctx->stream));
    MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
    if (P.n_tiles) {
      float ms = 0, ms_plan = 0;
      cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
      if (attempt == 0) { cudaEventElapsedTime(&ms_plan, ctx->ev2, ctx->ev0); ctx->plan_ms += ms_plan; ctx->total_launches++; }
      ctx->emit_ms += ms; ctx->emit_launches++; ctx->total_launches++;
      ctx->emit_bytes += 2 * (int64_t)tot[2];
    }
    if (!tot[3]) break;
    if (attempt == 1) return fail(ctx, MG_ECUDA, "internal: output overflow after regrow");
    est = (size_t)tot[2] + 4096;
    MG_CK(ctx, cudaMemsetAsync(P.totals + 3, 0, 8, ctx->stream));
  }
  ctx->last_ob = ctx->ob; ctx->last_bytes = (int64_t)tot[2];
  if (n_bytes) *n_bytes = (int64_t)tot[2];
  if (n_templates) *n_templates = (int64_t)tot[1];
  if (n_te_kept) *n_te_kept = (int64_t)tot[0];
  if (!want_out) ctx->ob ^= 1;            // the bytes stay in this set (mg_unit_read_async / mg_unit_drain_async): the next unit takes the other one
  if (want_out) {
    if ((int64_t)tot[2] > cap) return fail(ctx, MG_ECAP, "output needs %lld bytes per file, caller gave %lld", (long long)tot[2], (long long)cap);
    // the kernels have finished (totals were read back): the copies go to their own stream, so the
    // next unit's kernels overlap with them
    if (out1 && tot[2]) MG_CK(ctx, cudaMemcpyAsync(out1, P.out[0], (size_t)tot[2], cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (out2 && tot[2]) MG_CK(ctx, cudaMemcpyAsync(out2, P.out[1], (size_t)tot[2], cudaMemcpyDeviceToHost, ctx->copy_stream));
    MG_CK(ctx, cudaEventRecord(ctx->ev_d2h[ctx->ob], ctx->copy_stream));
    ctx->ob ^= 1;
    if (wait_copies) MG_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
  }
  return MG_OK;
}

int mg_unit_generate(mg_ctx *ctx, const mg_unit_desc *d, uint8_t *out1, uint8_t *out2, int64_t cap, int64_t *n_bytes,
                     int64_t *n_templates, int64_t *n_te_kept) {
  return unit_generate(ctx, d, out1, out2, cap, n_bytes, n_templates, n_te_kept, true);
}

int mg_unit_generate_async(mg_ctx *ctx, const mg_unit_desc *d, uint8_t *out1, uint8_t *out2, int64_t cap, int64_t *n_bytes,
                           int64_t *n_templates, int64_t *n_te_kept) {
  return unit_generate(ctx, d, out1, out2, cap, n_bytes, n_templates, n_te_kept, false);
}

int mg_unit_read_async(mg_ctx *ctx, int32_t file, int64_t offset, int64_t bytes, uint8_t *dst) {
  if (!ctx || !dst || file < 0 || file > 1 || offset < 0 || bytes < 0) return fail(ctx, MG_EINVAL, "mg_unit_read_async: bad arguments");
  if (offset + bytes > ctx->last_bytes) return fail(ctx, MG_EINVAL, "mg_unit_read_async: range beyond the unit's %lld bytes", (long long)ctx->last_bytes);
  DeviceGuard g(ctx->device);
  if (bytes) MG_CK(ctx, cudaMemcpyAsync(dst, ctx->s_out[ctx->last_ob][file].as<uint8_t>() + offset, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
  MG_CK(ctx, cudaEventRecord(ctx->ev_d2h[ctx->last_ob], ctx->copy_stream));   // the next unit into this buffer set waits for it
  return MG_OK;
}

int mg_wait_copies(mg_ctx *ctx) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  MG_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
  return MG_OK;
}

// ---- corrupt-reads ---------------------------------------------------------------------------------

int mg_corrupt_fastq(mg_ctx *ctx, const uint8_t *in1, int64_t len1, const uint8_t *in2, int64_t len2, int32_t mode,
                     uint32_t seed, const double *bq_rnd, const double *call_rnd, const uint8_t *base_rnd,
                     const int64_t *draw_off, uint8_t *out1, uint8_t *out2, int64_t cap, int64_t *out_len1,
                     int64_t *out_len2, int64_t *n_templates, int64_t first_template, int64_t *consumed1,
                     int64_t *consumed2) {
  if (!ctx || !in1 || len1 < 0 || (in2 && len2 < 0)) return fail(ctx, MG_EINVAL, "mg_corrupt_fastq: bad arguments");
  if (consumed1) *consumed1 = 0;
  if (consumed2) *consumed2 = 0;
  if (ctx->rlen == 0) return fail(ctx, MG_EINVAL, "no read model loaded (mg_model_load)");
  if (mode != MG_MODE_PHILOX && mode != MG_MODE_DET) return fail(ctx, MG_EINVAL, "unknown mode %d", mode);
  DeviceGuard g(ctx->device);
  const int nf = in2 ? 2 : 1;
  if (nf > ctx->n_mates) return fail(ctx, MG_EINVAL, "paired corruption needs a 2-mate model");
  const uint8_t *in[2] = {in1, in2}; const int64_t len[2] = {len1, len2};
  MgCorruptParams P; memset(&P, 0, sizeof P);
  MgFastqChunk &q = ctx->fq;
  MG_CK(ctx, mg_fastq_load(q, in, len, nf, ctx->stream));
  ctx->total_launches += 5 * nf;
  for (int f = 0; f < nf; f++) { P.in[f] = q.in[f].as<uint8_t>(); P.nl[f] = q.nl[f].as<int64_t>(); }
  const int64_t n_rec = q.n_tpl;                                    // zip() of the two readers, readcorrupt.py:53
  P.n_rec = n_rec; P.n_files = nf;
  P.cum_bq = ctx->m_bq.as<double>(); P.n_cycles = ctx->n_cycles; P.n_bq = ctx->n_bq; P.phred = ctx->m_phred.as<double>();
  P.mode = mode;
  P.cor.kshift = ctx->a_kshift[1]; P.cor.code9 = ctx->a_code9[1];   // the table over every cycle: any read length up to n_cycles
  P.cor.alias = ctx->m_alias[1].as<uint32_t>();
  P.cor.n_cycles = ctx->n_cycles; P.cor.n_mates = ctx->n_mates;
  P.cor.k0 = seed; P.cor.k1 = 0x636f7232u;
  if (out_len1) *out_len1 = 0;
  if (out_len2) *out_len2 = 0;
  if (n_templates) *n_templates = n_rec;
  if (n_rec == 0) return MG_OK;
  P.first = first_template;
  {  // bytes of each input that belong to the n_rec complete templates (the caller streams a large
     // file in chunks and carries the rest over)
    int64_t last[2] = {0, 0};
    MG_CK(ctx, mg_fastq_ends(q, n_rec, last, ctx->stream));
    MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
    if (consumed1) *consumed1 = last[0] + 1;
    if (consumed2 && nf > 1) *consumed2 = last[1] + 1;
  }

  MG_CK(ctx, ctx->s_state.need(64));
  P.err = ctx->s_state.as<unsigned long long>();
  MG_CK(ctx, cudaMemsetAsync(P.err, 0, 16, ctx->stream));
  MG_CK(ctx, q.tmp.need(8 * (size_t)mg_scan_tmp_elems(n_rec)));
  for (int f = 0; f < nf; f++) { MG_CK(ctx, ctx->c_sz[f].need(8 * (size_t)n_rec)); MG_CK(ctx, ctx->c_off[f].need(8 * (size_t)(n_rec + 1))); }
  mg_launch_corrupt_sizes(P, ctx->c_sz[0].as<int64_t>(), nf > 1 ? ctx->c_sz[1].as<int64_t>() : nullptr, ctx->stream);
  int64_t total[2] = {0, 0};
  for (int f = 0; f < nf; f++) {
    mg_launch_scan_i64(ctx->c_sz[f].as<int64_t>(), ctx->c_off[f].as<int64_t>(), n_rec, q.tmp.as<int64_t>(), ctx->stream);
    MG_CK(ctx, cudaMemcpyAsync(&total[f], ctx->c_off[f].as<int64_t>() + n_rec, 8, cudaMemcpyDeviceToHost, ctx->stream));
    P.out_off[f] = ctx->c_off[f].as<int64_t>();
    ctx->total_launches += 3;
  }
  unsigned long long errv[2] = {0, 0};
  MG_CK(ctx, cudaMemcpyAsync(errv, P.err, 16, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  const unsigned long long err = errv[0];
  if (err) return fail(ctx, MG_EINDEX, "a read is longer than the model's %d cycles (IndexError in the reference, illumina.py:156)", ctx->n_cycles);
  if (out_len1) *out_len1 = total[0];
  if (out_len2) *out_len2 = total[1];
  if (std::max(total[0], total[1]) > cap) return fail(ctx, MG_ECAP, "output needs %lld bytes, caller gave %lld", (long long)std::max(total[0], total[1]), (long long)cap);
  for (int f = 0; f < nf; f++) { MG_CK(ctx, ctx->c_out[f].need((size_t)total[f] + 16)); P.out[f] = ctx->c_out[f].as<uint8_t>(); }

  if (mode == MG_MODE_DET) {
    if (!bq_rnd || !call_rnd || !base_rnd || !draw_off) return fail(ctx, MG_EINVAL, "deterministic mode needs the draw arrays");
    const int64_t n_reads = n_rec * nf;
    const int64_t n_draws = draw_off[n_reads];
    MG_CK(ctx, ctx->c_draw[0].need(8 * (size_t)n_draws + 8)); MG_CK(ctx, ctx->c_draw[1].need(8 * (size_t)n_draws + 8));
    MG_CK(ctx, ctx->c_draw[2].need((size_t)n_draws + 8)); MG_CK(ctx, ctx->c_draw[3].need(8 * (size_t)(n_reads + 1)));
    MG_CK(ctx, cudaMemcpyAsync(ctx->c_draw[0].p, bq_rnd, 8 * (size_t)n_draws, cudaMemcpyHostToDevice, ctx->stream));
    MG_CK(ctx, cudaMemcpyAsync(ctx->c_draw[1].p, call_rnd, 8 * (size_t)n_draws, cudaMemcpyHostToDevice, ctx->stream));
    MG_CK(ctx, cudaMemcpyAsync(ctx->c_draw[2].p, base_rnd, (size_t)n_draws, cudaMemcpyHostToDevice, ctx->stream));
    MG_CK(ctx, cudaMemcpyAsync(ctx->c_draw[3].p, draw_off, 8 * (size_t)(n_reads + 1), cudaMemcpyHostToDevice, ctx->stream));
    P.bq_rnd = ctx->c_draw[0].as<double>(); P.call_rnd = ctx->c_draw[1].as<double>();
    P.base_rnd = ctx->c_draw[2].as<uint8_t>(); P.draw_off = ctx->c_draw[3].as<int64_t>();
  }
  MG_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  {
    static const bool lsu = getenv("MG_COPYOUT_LSU") != nullptr, old = getenv("MG_CORRUPT_SIMPLE") != nullptr;
    // production mode, every record fits a warp's stage: the staged kernel; else (deterministic draws, giant names) the simple one
    if (mode == MG_MODE_PHILOX && !old && errv[1] + 16 <= (unsigned long long)mg_corrupt_stage_cap()) mg_launch_corrupt_staged(P, !lsu, ctx->stream);
    else mg_launch_corrupt(P, ctx->stream);
  }
  MG_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  MG_CK(ctx, cudaGetLastError());
  if (out1) MG_CK(ctx, cudaMemcpyAsync(out1, P.out[0], (size_t)total[0], cudaMemcpyDeviceToHost, ctx->stream));
  if (nf > 1 && out2) MG_CK(ctx, cudaMemcpyAsync(out2, P.out[1], (size_t)total[1], cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->emit_ms += ms; ctx->emit_launches++; ctx->total_launches++;
  ctx->emit_bytes += 2 * (total[0] + total[1]);
  return MG_OK;
}

}  // extern "C"

// ---- FASTQ ingest (corrupt-reads, check-reads, god-aligner) ----------------------------------------

cudaError_t mg_fastq_load(MgFastqChunk &q, const uint8_t *const in[2], const int64_t len[2], int nf, cudaStream_t st) {
#define TRY(call) do { const cudaError_t e_ = (call); if (e_ != cudaSuccess) return e_; } while (0)
  int64_t n_lines[2] = {0, 0};
  for (int f = 0; f < nf; f++) {
    TRY(q.in[f].need((size_t)len[f] + 16));
    if (len[f]) TRY(cudaMemcpyAsync(q.in[f].p, in[f], (size_t)len[f], cudaMemcpyHostToDevice, st));
    const int64_t chunks = mg_nl_chunks(len[f]);
    TRY(q.cnt.need(8 * (size_t)(2 * chunks + 4)));
    TRY(q.tmp.need(8 * (size_t)mg_scan_tmp_elems(std::max<int64_t>(chunks, 1))));
    int64_t *cnt = q.cnt.as<int64_t>(), *off = cnt + chunks + 1;
    mg_launch_nl_count(q.in[f].as<uint8_t>(), len[f], cnt, st);
    mg_launch_scan_i64(cnt, off, chunks, q.tmp.as<int64_t>(), st);
    TRY(cudaMemcpyAsync(&n_lines[f], off + chunks, 8, cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    TRY(q.nl[f].need(8 * (size_t)(n_lines[f] + 1)));
    mg_launch_nl_write(q.in[f].as<uint8_t>(), len[f], off, q.nl[f].as<int64_t>(), st);
    TRY(cudaGetLastError());
  }
#undef TRY
  q.nf = nf;
  q.n_tpl = n_lines[0] / 4;
  if (nf == 2) q.n_tpl = std::min(q.n_tpl, n_lines[1] / 4);
  return cudaSuccess;
}

cudaError_t mg_fastq_ends(const MgFastqChunk &q, int64_t k, int64_t last[2], cudaStream_t st) {
  for (int f = 0; f < q.nf; f++) {
    const cudaError_t e = cudaMemcpyAsync(&last[f], q.nl[f].as<int64_t>() + (4 * k - 1), 8, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// ---- internal views for mg_check.cu, mg_bam.cu and mg_readmodel.cu ---------------------------------
int mg_internal_copy_view(mg_ctx *ctx, int64_t copy_id, int64_t *region_id, const MgNode **nodes, int *n_nodes, const uint32_t **hap, uint32_t *hap_len,
                          const MgExc **exc, int *n_exc, int64_t *start1) {
  auto it = ctx->copies.find(copy_id);
  if (it == ctx->copies.end()) return fail(ctx, MG_EINVAL, "unknown copy %lld", (long long)copy_id);
  const Copy &C = *it->second;
  *region_id = C.region_id; *nodes = C.d_nodes; *n_nodes = (int)C.n_nodes; *hap = C.d_hap + MG_HAP_PAD; *hap_len = (uint32_t)(C.p_max - C.p_min);
  *exc = C.d_exc; *n_exc = (int)C.n_exc; *start1 = C.p_min;
  return MG_OK;
}

int mg_internal_region_view(mg_ctx *ctx, int64_t region_id, const uint32_t **ref, int64_t *len, const MgExc **exc, int *n_exc) {
  auto it = ctx->regions.find(region_id);
  if (it == ctx->regions.end()) return fail(ctx, MG_EINVAL, "unknown region %lld", (long long)region_id);
  const Region &R = *it->second;
  *ref = R.d_ref + MG_HAP_PAD; *len = R.len; *exc = R.d_exc; *n_exc = (int)R.exc.size();
  return MG_OK;
}

cudaStream_t mg_internal_stream(mg_ctx *ctx) { return ctx->stream; }
int mg_internal_device(mg_ctx *ctx) { return ctx->device; }
int mg_internal_fail(mg_ctx *ctx, int code, const char *msg) { return fail(ctx, code, "%s", msg); }
int mg_internal_cuda_fail(mg_ctx *ctx, cudaError_t e, const char *call, const char *file, int line) {
  return fail(ctx, MG_ECUDA, "%s: %s (%s:%d)", call, cudaGetErrorString(e), file, line);
}

extern "C" {

// ---- draining units into an output sink -----------------------------------------------------------

static void drain_loop(mg_ctx *ctx) {
  cudaSetDevice(ctx->device);
  std::unique_lock<std::mutex> lk(ctx->dmu);
  while (true) {
    { const double ti = Timer::now(); while (ctx->djobs.empty() && !ctx->dstop) ctx->dcv.wait(lk); ctx->d_idle_ms += Timer::now() - ti; }
    if (ctx->djobs.empty()) return;
    const mg_ctx::DrainJob job = ctx->djobs.front(); ctx->djobs.pop_front();
    lk.unlock();
    std::string err;
    // two pieces in flight: the copy of piece i + 1 is enqueued before piece i is handed to the writers
    void *slot[2] = {nullptr, nullptr}; int64_t s_off[2] = {0, 0}, s_n[2] = {0, 0};
    const int64_t chunk = mg_sink_chunk_bytes(job.sink);
    int k = 0;
    std::vector<int64_t> m_unit, m_uoff, m_soff, m_bytes;
    auto finish = [&](int i) {
      if (!slot[i]) return;
      { const double tc = Timer::now(); if (cudaEventSynchronize(ctx->ev_drain[i]) != cudaSuccess && err.empty()) err = "device-to-host copy failed"; ctx->d_wait_copy_ms += Timer::now() - tc; }
      int rc;
      if (job.units) {                                      // bytes [s_off, s_off + s_n) of the batch's stream: the units they belong to
        const std::vector<int64_t> &ui = *job.units, &b = *job.base;
        m_unit.clear(); m_uoff.clear(); m_soff.clear(); m_bytes.clear();
        const int64_t lo = s_off[i], hi = s_off[i] + (err.empty() ? s_n[i] : 0);
        size_t u = (size_t)(std::upper_bound(b.begin(), b.end(), lo) - b.begin());
        u = u ? u - 1 : 0;                                  // the last unit that starts at or before lo
        for (; u < ui.size() && b[u] < hi; u++) {
          const int64_t a0 = std::max(lo, b[u]), a1 = std::min(hi, b[u + 1]);
          if (a1 <= a0) continue;
          m_unit.push_back(ui[u]); m_uoff.push_back(a0 - b[u]); m_soff.push_back(a0 - lo); m_bytes.push_back(a1 - a0);
        }
        rc = mg_sink_commit_multi(job.sink, slot[i], (int32_t)m_unit.size(), m_unit.data(), m_uoff.data(), m_soff.data(), m_bytes.data());
      } else {
        rc = mg_sink_commit(job.sink, slot[i], job.unit, s_off[i], err.empty() ? s_n[i] : 0);
      }
      if (rc != MG_OK && err.empty()) err = mg_sink_error(job.sink);
      slot[i] = nullptr;
    };
    for (int64_t off = 0; off < job.bytes && err.empty(); off += chunk, k ^= 1) {
      finish(k);                                            // the piece that used this event two steps ago
      void *b1 = nullptr, *b2 = nullptr;
      const double ta = Timer::now();
      if (mg_sink_acquire(job.sink, job.producer, &b1, &b2, &slot[k]) != MG_OK) { err = mg_sink_error(job.sink); slot[k] = nullptr; break; }
      ctx->d_wait_slot_ms += Timer::now() - ta;
      const int64_t n = std::min(chunk, job.bytes - off);
      ctx->d_bytes += 2 * n;
      s_off[k] = off; s_n[k] = n;
      cudaError_t e = cudaMemcpyAsync(b1, ctx->s_out[job.ob][0].as<uint8_t>() + off, (size_t)n, cudaMemcpyDeviceToHost, ctx->copy_stream);
      if (e == cudaSuccess && b2) e = cudaMemcpyAsync(b2, ctx->s_out[job.ob][1].as<uint8_t>() + off, (size_t)n, cudaMemcpyDeviceToHost, ctx->copy_stream);
      if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_drain[k], ctx->copy_stream);
      if (e != cudaSuccess) err = cudaGetErrorString(e);
    }
    finish(k); finish(k ^ 1);
    lk.lock();
    ctx->dbusy[job.ob]--;
    if (!err.empty() && !ctx->dfailed) { ctx->dfailed = true; ctx->derr = err; mg_sink_abort(job.sink, err.c_str()); }
    ctx->dcv.notify_all();
  }
}

int mg_unit_drain_async(mg_ctx *ctx, mg_sink *sink, int32_t producer, int64_t unit) {
  if (!ctx || !sink) return MG_EINVAL;
  if (mg_sink_unit_size(sink, unit, ctx->last_bytes) != MG_OK) return fail(ctx, MG_EVALUE, "output sink: %s", mg_sink_error(sink));
  if (ctx->last_bytes == 0) return MG_OK;
  std::lock_guard<std::mutex> lk(ctx->dmu);
  if (ctx->dfailed) return fail(ctx, MG_EVALUE, "output sink: %s", ctx->derr.c_str());
  if (!ctx->drain_thread.joinable()) {
    DeviceGuard g(ctx->device);
    for (int i = 0; i < 2; i++)
      if (!ctx->ev_drain[i] && cudaEventCreateWithFlags(&ctx->ev_drain[i], cudaEventDisableTiming) != cudaSuccess) return fail(ctx, MG_ECUDA, "cannot create the drain events");
    ctx->drain_thread = std::thread(drain_loop, ctx);
  }
  ctx->dbusy[ctx->last_ob]++;
  ctx->djobs.push_back({sink, producer, unit, ctx->last_ob, ctx->last_bytes, nullptr, nullptr});
  ctx->dcv.notify_all();
  return MG_OK;
}

int mg_drain_wait(mg_ctx *ctx) {
  if (!ctx) return MG_EINVAL;
  std::unique_lock<std::mutex> lk(ctx->dmu);
  while ((ctx->dbusy[0] > 0 || ctx->dbusy[1] > 0) && !ctx->dfailed) ctx->dcv.wait(lk);
  if (ctx->dfailed) return fail(ctx, MG_EVALUE, "output sink: %s", ctx->derr.c_str());
  if (getenv("MG_TIMING")) {
    fprintf(stderr, "[mg] drain thread of device %d: %.1f GB copied; waiting for copies %.0f ms, for slots %.0f ms, for units %.0f ms\n", ctx->device,
            ctx->d_bytes / 1e9, ctx->d_wait_copy_ms, ctx->d_wait_slot_ms, ctx->d_idle_ms);
    ctx->d_bytes = 0; ctx->d_wait_copy_ms = ctx->d_wait_slot_ms = ctx->d_idle_ms = 0;
  }
  return MG_OK;
}

// ---- batches of small regions -------------------------------------------------------------------

int mg_batch_build(mg_ctx *ctx, int64_t n_regions, const uint8_t *ref_bytes, const int64_t *ref_off, const int64_t *bed_start,
                   int64_t n_segs, const int32_t *seg_region, const int64_t *seg_var_off, const int64_t *pos, const uint8_t *op,
                   const int64_t *oplen, const uint8_t *alt_pool, const int64_t *alt_off, int64_t *batch_id, int64_t *seg_p_min,
                   int64_t *seg_p_max) {
  if (!ctx || !batch_id || n_regions < 1 || n_segs < 1 || !ref_off || !bed_start || !seg_region || !seg_var_off)
    return fail(ctx, MG_EINVAL, "mg_batch_build: bad arguments");
  const int64_t total = ref_off[n_regions], n_var = seg_var_off[n_segs];
  if (ref_off[0] != 0 || total < 0 || (total > 0 && !ref_bytes)) return fail(ctx, MG_EINVAL, "mg_batch_build: ref_off must start at 0");
  if (n_var < 0 || (n_var > 0 && (!pos || !op || !oplen || !alt_pool || !alt_off))) return fail(ctx, MG_EINVAL, "mg_batch_build: variant arrays missing");
  if (total >= (int64_t)0x7FF00000ll) return fail(ctx, MG_EVALUE, "the regions of one batch hold %lld bases (limit 2^31)", (long long)total);
  if (n_var >= (1ll << 28) || n_segs >= (1ll << 24)) return fail(ctx, MG_EVALUE, "batch too large (%lld variants, %lld segments)", (long long)n_var, (long long)n_segs);
  for (int64_t r = 0; r < n_regions; r++)
    if (ref_off[r + 1] < ref_off[r]) return fail(ctx, MG_EINVAL, "mg_batch_build: ref_off must ascend");
  DeviceGuard g(ctx->device);
  std::unique_ptr<Batch> B(new Batch());
  int rc = load_packed(ctx, ref_bytes, total, 0, B->R);
  if (rc) return rc;
  std::vector<MgSeg> segs((size_t)n_segs);
  for (int64_t s = 0; s < n_segs; s++) {
    const int32_t r = seg_region[s];
    if (r < 0 || r >= n_regions || seg_var_off[s + 1] < seg_var_off[s]) return fail(ctx, MG_EINVAL, "mg_batch_build: segment %lld is malformed", (long long)s);
    MgSeg &sg = segs[(size_t)s];
    memset(&sg, 0, sizeof sg);
    sg.v0 = (int32_t)seg_var_off[s]; sg.v1 = (int32_t)seg_var_off[s + 1];
    sg.roff = (uint32_t)ref_off[r];
    sg.start1 = bed_start[r] + 1;                     // ref_start_pos, readgenerate.py:190; also p_min
    sg.region_len = ref_off[r + 1] - ref_off[r];
  }
  B->C.reset(new Copy());
  B->C->owner = ctx;
  rc = build_segments(ctx, B->R->d_ref + MG_HAP_PAD, B->R->d_exc, (int)B->R->exc.size(), segs, n_var, pos, op, oplen, alt_pool, alt_off, *B->C, B->C->segs);
  if (rc) return rc;
  B->C->seg_start1.resize((size_t)n_segs);
  for (int64_t s = 0; s < n_segs; s++) {
    B->C->seg_start1[(size_t)s] = segs[(size_t)s].start1;
    if (seg_p_min) seg_p_min[s] = segs[(size_t)s].start1;                                   // readgenerate.py:192
    if (seg_p_max) seg_p_max[s] = segs[(size_t)s].start1 + (int64_t)B->C->segs[(size_t)s].hap_len;
  }
  const int64_t id = ctx->next_id++;
  ctx->batches[id] = std::move(B);
  *batch_id = id;
  return MG_OK;
}

int mg_batch_free(mg_ctx *ctx, int64_t batch_id) {
  if (!ctx) return MG_EINVAL;
  DeviceGuard g(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  return ctx->batches.erase(batch_id) ? MG_OK : fail(ctx, MG_EINVAL, "unknown batch %lld", (long long)batch_id);
}

int mg_batch_generate(mg_ctx *ctx, int64_t batch_id, int64_t n_units, const int32_t *unit_seg, const uint32_t *unit_seed,
                      const int64_t *unit_ncand, const int64_t *unit_index, const char *sample, const uint8_t *chrom_pool,
                      const int64_t *chrom_off, const int32_t *seg_cpy, double p, int32_t mode, const int64_t *ts, const double *u_tlen,
                      const int8_t *fo, const int64_t *cand_off, int32_t corrupt, uint32_t corrupt_seed, mg_sink *sink,
                      int32_t producer, int64_t *n_templates, int64_t *n_bytes, int64_t *unit_bytes, int64_t *unit_templates) {
  if (!ctx || n_units < 0 || (n_units > 0 && (!unit_seg || !unit_seed || !unit_ncand || !unit_index || !sample || !chrom_pool || !chrom_off || !seg_cpy)))
    return fail(ctx, MG_EINVAL, "mg_batch_generate: bad arguments");
  if (n_templates) *n_templates = 0;
  if (n_bytes) *n_bytes = 0;
  auto it = ctx->batches.find(batch_id);
  if (it == ctx->batches.end()) return fail(ctx, MG_EINVAL, "unknown batch %lld", (long long)batch_id);
  if (ctx->rlen == 0) return fail(ctx, MG_EINVAL, "no read model loaded (mg_model_load)");
  if (mode != MG_MODE_PHILOX && mode != MG_MODE_DET) return fail(ctx, MG_EINVAL, "a batch runs in PHILOX or DET mode");
  if (mode == MG_MODE_PHILOX && !(p > 0.0 && p < 1.0)) return fail(ctx, MG_EINVAL, "PHILOX mode needs 0 < p < 1");
  if (corrupt && mode != MG_MODE_PHILOX) return fail(ctx, MG_EINVAL, "fused corruption draws from Philox: use mg_corrupt_fastq for deterministic mode");
  if (corrupt && ctx->rlen > ctx->n_cycles) return fail(ctx, MG_EINDEX, "read length %d exceeds the model's %d cycles", ctx->rlen, ctx->n_cycles);
  if (corrupt && ctx->n_mates < 2) return fail(ctx, MG_EINVAL, "paired corruption needs a 2-mate model");
  if (n_units >= (1ll << 24)) return fail(ctx, MG_EVALUE, "%lld units in one batch (limit 2^24)", (long long)n_units);
  const Copy &C = *it->second->C;
  const int64_t n_segs = (int64_t)C.segs.size();
  const int L = ctx->rlen;
  if (n_units == 0) { ctx->last_bytes = 0; return MG_OK; }
  DeviceGuard g(ctx->device);

  // -- the unit table
  std::vector<MgBatchUnit> U((size_t)n_units);
  int64_t n_plan = 0, n_draws = 0;
  char text[96];
  for (int64_t u = 0; u < n_units; u++) {
    const int32_t sg = unit_seg[u];
    if (sg < 0 || sg >= n_segs) return fail(ctx, MG_EINVAL, "unit %lld names segment %d of %lld", (long long)u, (int)sg, (long long)n_segs);
    if (unit_ncand[u] < 0 || unit_ncand[u] > MG_BATCH_MAXC) return fail(ctx, MG_EVALUE, "unit %lld has %lld candidates: the batch path takes at most %d per unit", (long long)u, (long long)unit_ncand[u], MG_BATCH_MAXC);
    if (u && unit_index[u] <= unit_index[u - 1]) return fail(ctx, MG_EINVAL, "the units of a batch must be in ascending schedule order");
    MgBatchUnit &b = U[(size_t)u];
    memset(&b, 0, sizeof b);
    const int pl = snprintf(text, sizeof text, "@%s:0:%lld:", sample, (long long)unit_index[u]);          // readgenerate.py:195, 210
    if (pl < 0 || pl > 32) return fail(ctx, MG_EVALUE, "sample name too long for the batch path (qname prefix of %d bytes, limit 32)", pl);
    b.n_pre = (pl + 7) / 8;
    for (int i = 0; i < b.n_pre; i++) b.pre[i] = mg_tok_bytes(reinterpret_cast<const uint8_t *>(text), 8 * i, pl - 8 * i);
    const int64_t cl = chrom_off[sg + 1] - chrom_off[sg];
    if (cl < 0 || cl > 20) return fail(ctx, MG_EVALUE, "chromosome name too long for the batch path (%lld bytes, limit 20)", (long long)cl);
    int ml = 0;
    text[ml++] = '|';
    memcpy(text + ml, chrom_pool + chrom_off[sg], (size_t)cl); ml += (int)cl;
    ml += snprintf(text + ml, sizeof text - (size_t)ml, "|%d", (int)seg_cpy[sg]);                         // readgenerate.py:223
    if (ml > 32) return fail(ctx, MG_EVALUE, "chromosome name too long for the batch path");
    b.n_mid = (ml + 7) / 8;
    for (int i = 0; i < b.n_mid; i++) b.mid[i] = mg_tok_bytes(reinterpret_cast<const uint8_t *>(text), 8 * i, ml - 8 * i);
    b.qn_len = (uint32_t)(pl + ml);
    b.seed = unit_seed[u];
    b.x0 = C.segs[(size_t)sg].hap_base; b.hap_len = C.segs[(size_t)sg].hap_len;
    b.n_cand = (uint32_t)unit_ncand[u]; b.plan_off = (uint32_t)n_plan;
    b.p_min = C.seg_start1[(size_t)sg];
    if (mode == MG_MODE_DET) {
      if (!cand_off || !ts || !u_tlen || !fo) return fail(ctx, MG_EINVAL, "deterministic mode needs ts, u_tlen, fo and cand_off");
      b.draw_off = cand_off[u];
      if (cand_off[u + 1] - cand_off[u] < unit_ncand[u]) return fail(ctx, MG_EINVAL, "unit %lld: fewer draws than candidates", (long long)u);
      n_draws = cand_off[u + 1];
    }
    n_plan += unit_ncand[u];
  }
  if (n_plan >= (1ll << 32)) return fail(ctx, MG_EVALUE, "%lld candidates in one batch (limit 2^32)", (long long)n_plan);

  MgUnitParams P; memset(&P, 0, sizeof P);
  P.hap = C.d_hap + MG_HAP_PAD; P.hap_len = (uint32_t)C.hap_len; P.p_min = 0;
  P.nodes = C.d_nodes; P.n_nodes = (int)C.n_nodes;
  P.blk = C.d_blk; P.blk_shift = BLK_SHIFT; P.n_blk = C.n_blk;
  P.exc = C.d_exc; P.n_exc = (int)C.n_exc; P.eblk = C.d_eblk;
  P.cum_tlen = ctx->m_tlen.as<double>(); P.n_tlen = ctx->n_tlen; P.rlen = L;
  P.tlen_alias = ctx->has_tlen_alias ? ctx->m_tlen_alias.as<uint32_t>() : nullptr;
  P.mode = mode;
  if (mode == MG_MODE_PHILOX) P.inv_log1mp = 1.0 / log(1.0 - p);
  mg_qn_const(P.qn, nullptr, 0, nullptr, 0, L);       // the per-unit strings come from the unit table
  P.bulk = 1;
  P.corrupt = corrupt;
  P.cor.kshift = ctx->a_kshift[0]; P.cor.code9 = ctx->a_code9[0];
  P.cor.alias = ctx->m_alias[0].as<uint32_t>();
  P.cor.n_cycles = ctx->n_cycles; P.cor.n_mates = ctx->n_mates;
  P.cor.k0 = corrupt_seed;                            // k1: per unit, from its seed (k_unit_emit)
  P.L_nd = mg_ndigits32((uint32_t)L);
  int stage = 32 * (2 * L + 5 + 96);
  if (stage > 48 * 1024) stage = 48 * 1024;
  P.stage_cap = stage & ~15;
  int smem = 0;
  const int grid = mg_batch_grid(L, corrupt ? 1 + P.cor.code9 : 0, P.stage_cap, &smem);
  if (grid <= 0) return fail(ctx, MG_EVALUE, "the emit kernel's staging area (%d bytes for reads of %d bases) exceeds the shared memory of this device", smem, L);

  // -- device tables: [units][unit_kept n+1][unit_bytes n+1][unit_te n+1][kept_base n+2][byte_base n+2][scan tmp]
  const size_t nu = (size_t)n_units;
  MG_CK(ctx, ctx->b_units.need(sizeof(MgBatchUnit) * nu));
  const size_t tmp_elems = (size_t)mg_scan_tmp_elems((int64_t)nu);
  MG_CK(ctx, ctx->b_arr.need(8 * (3 * (nu + 1) + 2 * (nu + 2) + tmp_elems + 8)));
  long long *arr = ctx->b_arr.as<long long>();
  P.bunits = ctx->b_units.as<MgBatchUnit>(); P.n_bunits = (int)n_units;
  P.unit_kept = arr; P.unit_bytes = arr + (nu + 1); P.unit_te = arr + 2 * (nu + 1);
  long long *kept_base = arr + 3 * (nu + 1), *byte_base = kept_base + (nu + 2), *scan_tmp = byte_base + (nu + 2);
  P.kept_base = kept_base; P.byte_base = byte_base;
  MG_CK(ctx, ctx->s_state.need(64));
  P.totals = ctx->s_state.as<unsigned long long>();
  MG_CK(ctx, cudaMemsetAsync(P.totals, 0, 64, ctx->stream));
  MG_CK(ctx, ctx->s_plan.need(sizeof(MgPlan) * std::max<size_t>((size_t)n_plan, 1)));
  P.plan = ctx->s_plan.as<MgPlan>();
  MG_CK(ctx, cudaMemcpyAsync(ctx->b_units.p, U.data(), sizeof(MgBatchUnit) * nu, cudaMemcpyHostToDevice, ctx->stream));
  if (mode == MG_MODE_DET && n_draws) {
    const size_t nd = (size_t)n_draws;
    MG_CK(ctx, ctx->s_ts.need(8 * nd)); MG_CK(ctx, ctx->s_u.need(8 * nd)); MG_CK(ctx, ctx->s_fo.need(nd));
    MG_CK(ctx, cudaMemcpyAsync(ctx->s_ts.p, ts, 8 * nd, cudaMemcpyHostToDevice, ctx->stream));
    MG_CK(ctx, cudaMemcpyAsync(ctx->s_u.p, u_tlen, 8 * nd, cudaMemcpyHostToDevice, ctx->stream));
    MG_CK(ctx, cudaMemcpyAsync(ctx->s_fo.p, fo, nd, cudaMemcpyHostToDevice, ctx->stream));
  }
  P.ts_in = ctx->s_ts.as<int64_t>(); P.u_tlen = ctx->s_u.as<double>(); P.fo_in = ctx->s_fo.as<int8_t>();

  MG_CK(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
  mg_launch_batch_plan(P, ctx->stream);
  mg_launch_scan_i64(reinterpret_cast<const int64_t *>(P.unit_kept), reinterpret_cast<int64_t *>(kept_base), (int64_t)nu, reinterpret_cast<int64_t *>(scan_tmp), ctx->stream);
  mg_launch_scan_i64(reinterpret_cast<const int64_t *>(P.unit_bytes), reinterpret_cast<int64_t *>(byte_base), (int64_t)nu, reinterpret_cast<int64_t *>(scan_tmp), ctx->stream);
  MG_CK(ctx, cudaGetLastError());
  ctx->total_launches += 7;
  std::vector<long long> h_bytes(nu), h_kept(nu);
  long long tot_kept = 0, tot_bytes = 0;
  MG_CK(ctx, cudaMemcpyAsync(h_bytes.data(), P.unit_bytes, 8 * nu, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(h_kept.data(), P.unit_kept, 8 * nu, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(&tot_kept, kept_base + nu, 8, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaMemcpyAsync(&tot_bytes, byte_base + nu, 8, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));             // the sizes: the one read-back of a batch

  {   // a drain still reading this buffer set must finish first
    std::unique_lock<std::mutex> lk(ctx->dmu);
    while (ctx->dbusy[ctx->ob] > 0 && !ctx->dfailed) ctx->dcv.wait(lk);
    if (ctx->dfailed) return fail(ctx, MG_EVALUE, "output sink: %s", ctx->derr.c_str());
  }
  DevBuf *ob = ctx->s_out[ctx->ob];
  const size_t need = (size_t)tot_bytes + 4096;
  if (ob[0].cap < need || ob[1].cap < need) MG_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
  MG_CK(ctx, ob[0].need(need)); MG_CK(ctx, ob[1].need(need));
  P.out[0] = ob[0].as<uint8_t>(); P.out[1] = ob[1].as<uint8_t>();
  P.cap = std::min(ob[0].cap, ob[1].cap);
  MG_CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_d2h[ctx->ob], 0));
  MG_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  mg_launch_batch_emit(P, grid, smem, ctx->stream);
  MG_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  MG_CK(ctx, cudaGetLastError());
  MG_CK(ctx, cudaStreamSynchronize(ctx->stream));             // the drain thread copies from another stream
  {
    float ms = 0, ms_plan = 0;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1); cudaEventElapsedTime(&ms_plan, ctx->ev2, ctx->ev0);
    ctx->plan_ms += ms_plan; ctx->emit_ms += ms; ctx->emit_launches++; ctx->total_launches++;
    ctx->emit_bytes += 2 * (int64_t)tot_bytes;
  }
  ctx->last_ob = ctx->ob; ctx->last_bytes = (int64_t)tot_bytes;
  ctx->ob ^= 1;
  if (n_templates) *n_templates = (int64_t)tot_kept;
  if (n_bytes) *n_bytes = (int64_t)tot_bytes;
  for (size_t u = 0; u < nu; u++) {
    if (unit_bytes) unit_bytes[u] = h_bytes[u];
    if (unit_templates) unit_templates[u] = h_kept[u];
  }
  if (!sink) return MG_OK;

  // -- every unit's size is announced before the first piece asks for a slot; then the stream is drained
  auto ui = std::make_shared<std::vector<int64_t>>(nu), base = std::make_shared<std::vector<int64_t>>(nu + 1);
  (*base)[0] = 0;
  for (size_t u = 0; u < nu; u++) {
    (*ui)[u] = unit_index[u]; (*base)[u + 1] = (*base)[u] + h_bytes[u];
    if (mg_sink_unit_size(sink, unit_index[u], h_bytes[u]) != MG_OK) return fail(ctx, MG_EVALUE, "output sink: %s", mg_sink_error(sink));
  }
  if (tot_bytes == 0) return MG_OK;
  std::lock_guard<std::mutex> lk(ctx->dmu);
  if (ctx->dfailed) return fail(ctx, MG_EVALUE, "output sink: %s", ctx->derr.c_str());
  if (!ctx->drain_thread.joinable()) {
    for (int i = 0; i < 2; i++)
      if (!ctx->ev_drain[i] && cudaEventCreateWithFlags(&ctx->ev_drain[i], cudaEventDisableTiming) != cudaSuccess) return fail(ctx, MG_ECUDA, "cannot create the drain events");
    ctx->drain_thread = std::thread(drain_loop, ctx);
  }
  ctx->dbusy[ctx->last_ob]++;
  ctx->djobs.push_back({sink, producer, -1, ctx->last_ob, ctx->last_bytes, ui, base});
  ctx->dcv.notify_all();
  return MG_OK;
}

int mg_prof_reset(mg_ctx *ctx) {
  if (!ctx) return MG_EINVAL;
  ctx->emit_ms = 0; ctx->plan_ms = 0; ctx->emit_launches = 0; ctx->emit_bytes = 0; ctx->total_launches = 0;
  return MG_OK;
}

int mg_prof_get(mg_ctx *ctx, double *emit_ms, int64_t *emit_launches, int64_t *emit_bytes, int64_t *total_launches, double *plan_ms) {
  if (!ctx) return MG_EINVAL;
  if (emit_ms) *emit_ms = ctx->emit_ms;
  if (plan_ms) *plan_ms = ctx->plan_ms;
  if (emit_launches) *emit_launches = ctx->emit_launches;
  if (emit_bytes) *emit_bytes = ctx->emit_bytes;
  if (total_launches) *total_launches = ctx->total_launches;
  return MG_OK;
}

}  // extern "C"
