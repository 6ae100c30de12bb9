// Output sink of generate-reads / corrupt-reads: the reference's FASTQ writer process
// (mitty/simulation/readgenerate.py:233-253, readcorrupt.py:100-118) and the `>(gzip > r1.fq.gz)`
// it is always piped into (Readme.md:170, examples/reads/run.sh:15-16) as native threads inside the
// library -- no GIL, no Python objects.
//
// Producers (one per GPU) fill page-locked slot pairs (file 1 / file 2 bytes of one piece of a work
// unit) from their OWN pool and commit them with (unit, offset in the unit).  The files are written in
// SCHEDULE order, whatever the order of arrival:
//   plain, seekable target   pwrite() at base[unit] + offset by any writer thread, as soon as the sizes of
//                            all earlier units are known (a unit's size is announced right after its kernels)
//   plain, FIFO / pipe       sequential write(), one piece at a time per file, in (unit, offset) order
//   gzip                     pieces are deflated in parallel (one gzip member per piece, zlib), the members
//                            appended in order: the file is a valid multi-member .gz (what bgzip / pigz write)
// A slot goes back to its producer's pool when both of its pieces are on disk (plain) or deflated (gzip).
// Several PROCESSES (one per GPU, e.g. torchrun ranks) can share one pair of output files: with a table
// path the unit sizes and the "next unit" counter live in a small shared mapping (a file on /dev/shm);
// every process runs its own sink on the same files and pwrite()s its own units at their final offsets.
// Deadlock freedom: every producer works through its units in increasing schedule order and announces a
// unit's size before asking for a slot, and pools are per producer; so the lowest unfinished unit always
// has its base offset known and slots to travel in.
#include <cuda_runtime.h>
#include <zlib.h>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <atomic>
#include <cerrno>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/mitty_b200.h"
#include "mg_deflate.h"

void mg_deflate(const uint8_t *in, int64_t n, int level, int window_bits, std::vector<uint8_t> &out, size_t head) {
  z_stream z; memset(&z, 0, sizeof z);
  deflateInit2(&z, level, Z_DEFLATED, window_bits, 8, Z_DEFAULT_STRATEGY);
  out.resize(head + deflateBound(&z, (uLong)n) + 64);
  z.next_in = const_cast<Bytef *>(in); z.avail_in = (uInt)n;
  z.next_out = out.data() + head; z.avail_out = (uInt)(out.size() - head);
  deflate(&z, Z_FINISH);
  out.resize(out.size() - z.avail_out);
  deflateEnd(&z);
}

int mg_inflate(const uint8_t *in, int64_t n, uint8_t *out, int64_t out_len) {
  z_stream z; memset(&z, 0, sizeof z);
  if (inflateInit2(&z, -15) != Z_OK) return 1;
  z.next_in = const_cast<Bytef *>(in); z.avail_in = (uInt)n;
  uint8_t spare;                                  // a stream longer than out_len lands here and is caught
  z.next_out = out_len ? out : &spare; z.avail_out = out_len ? (uInt)out_len : 1;
  int rc = inflate(&z, Z_FINISH);
  if (rc == Z_BUF_ERROR && z.avail_out == 0) {
    z.next_out = &spare; z.avail_out = 1;
    rc = inflate(&z, Z_FINISH);
    rc = rc == Z_STREAM_END || (rc == Z_BUF_ERROR && z.avail_out == 0) ? 2 : 1;
  } else if (rc == Z_STREAM_END) {
    rc = z.avail_in != 0 ? 1 : (int64_t)z.total_out != out_len ? 2 : 0;
  } else {
    rc = 1;
  }
  inflateEnd(&z);
  return rc;
}

namespace {

struct Slot { uint8_t *buf[2]; int producer; int refs; bool pinned; };

// Page-locking is slow (hundreds of ms per GB): the buffers of closed sinks are kept for the next one.
std::mutex g_cache_mu;
std::multimap<int64_t, uint8_t *> g_cache;      // chunk bytes -> page-locked buffer

uint8_t *cache_get(int64_t bytes) {
  std::lock_guard<std::mutex> lk(g_cache_mu);
  auto it = g_cache.find(bytes);
  if (it == g_cache.end()) return nullptr;
  uint8_t *p = it->second; g_cache.erase(it);
  return p;
}

void cache_put(int64_t bytes, uint8_t *p) {
  std::lock_guard<std::mutex> lk(g_cache_mu);
  g_cache.insert({bytes, p});
}

struct Piece {                 // one file's share of a committed slot
  int file; int64_t unit, off, bytes;
  const uint8_t *data; Slot *slot;
  std::vector<uint8_t> z;      // gzip: the deflated member
  bool deflated = false;
};

}  // namespace

struct mg_sink {
  int fd[2] = {-1, -1};
  bool seekable[2] = {false, false};
  bool mapped[2] = {false, false};         // regular file: the writers memcpy into MAP_SHARED windows (write() serialises on the inode lock)
  int64_t fsize[2] = {0, 0};               // how far this process has extended each mapped file
  int n_files = 0, gzip = 0;
  int64_t n_units = 0, chunk = 0;
  std::vector<int64_t> size_own, base;     // per unit: bytes per file (-1 unknown), offset of its first byte
  int64_t *size = nullptr;                 // -> size_own, or into the shared table
  int64_t *next = nullptr;                 // "next unit to hand out" counter (own or shared)
  int64_t next_own = 0;
  void *shm = nullptr; size_t shm_bytes = 0;
  bool shared = false;
  int64_t known = 0;                       // sizes of units [0, known) are known -> base[0..known] are valid
  std::vector<std::vector<Slot *>> pool;   // free slots per producer
  std::vector<Slot *> all_slots;
  std::deque<Piece *> ready;               // plain + seekable: writable now; gzip: to be deflated
  std::multimap<int64_t, Piece *> waiting; // plain + seekable: base of the unit not known yet
  std::map<std::pair<int64_t, int64_t>, Piece *> ordered[2];   // sequential targets: (unit, off) -> piece (deflated if gzip)
  int64_t cur_unit[2] = {0, 0}, cur_off[2] = {0, 0};
  bool writing[2] = {false, false};        // one sequential writer per file at a time
  int64_t written[2] = {0, 0};
  std::mutex mu;
  std::condition_variable cv_work, cv_slot, cv_idle, cv_poll;
  std::vector<std::thread> threads;
  std::thread grower;                      // page-locks the slots beyond the first two per producer
  std::atomic<bool> stop_grow{false}, no_pin{false};
  int64_t in_flight = 0;                   // committed pieces not yet written
  bool closing = false, failed = false;
  std::string err;
};

namespace {

void fail(mg_sink *s, const char *fmt, ...) {          // with s->mu held
  if (s->failed) return;
  char b[512];
  va_list ap; va_start(ap, fmt); vsnprintf(b, sizeof b, fmt, ap); va_end(ap);
  s->err = b; s->failed = true;
  s->cv_work.notify_all(); s->cv_slot.notify_all(); s->cv_idle.notify_all();
}

bool write_all(int fd, const uint8_t *p, int64_t n, int64_t off, bool positional) {
  while (n > 0) {
    const size_t want = (size_t)(n > (1 << 30) ? (1 << 30) : n);
    const ssize_t w = positional ? pwrite(fd, p, want, (off_t)off) : write(fd, p, want);
    if (w < 0) { if (errno == EINTR) continue; return false; }
    p += w; n -= w; off += w;
  }
  return true;
}

void release(mg_sink *s, Piece *p) {                   // with s->mu held
  if (p->slot && --p->slot->refs == 0) { s->pool[(size_t)p->slot->producer].push_back(p->slot); s->cv_slot.notify_all(); }
  p->slot = nullptr;
}

bool sequential(const mg_sink *s, int f) { return s->gzip || !s->seekable[f]; }

// skip units that are known to be empty / finished on a sequential target
void advance(mg_sink *s, int f) {                       // with s->mu held
  // (a piece committed by mg_sink_commit_multi may run on through several whole units: the offset carries over)
  while (s->cur_unit[f] < s->n_units && s->size[s->cur_unit[f]] >= 0 && s->cur_off[f] >= s->size[s->cur_unit[f]]) {
    s->cur_off[f] -= s->size[s->cur_unit[f]]; s->cur_unit[f]++;
  }
}

// extend the prefix of units whose sizes are known; pieces whose base became known are made writable
void refresh_known(mg_sink *s) {                        // with s->mu held
  bool moved = false;
  while (s->known < s->n_units) {
    const int64_t sz = __atomic_load_n(&s->size[s->known], __ATOMIC_ACQUIRE);
    if (sz < 0) break;
    s->base[(size_t)s->known + 1] = s->base[(size_t)s->known] + sz;
    s->known++;
  }
  // mapped targets: the file must reach as far as any piece that becomes writable.  fallocate of the LAST byte only
  // extends (several processes sharing the file may be at different prefixes; none may ever shrink it)
  for (int f = 0; f < s->n_files; f++)
    if (s->mapped[f] && s->base[(size_t)s->known] > s->fsize[f]) {
      if (fallocate(s->fd[f], 0, (off_t)(s->base[(size_t)s->known] - 1), 1) != 0) { s->mapped[f] = false; }     // odd file system: back to pwrite
      else s->fsize[f] = s->base[(size_t)s->known];
    }
  for (auto it = s->waiting.begin(); it != s->waiting.end() && it->first < s->known;) { s->ready.push_back(it->second); it = s->waiting.erase(it); moved = true; }
  if (moved) s->cv_work.notify_all();
}

// one piece into a regular file through a shared mapping of just its pages: page faults of different threads run
// in parallel, whereas write() / pwrite() to one file are serialised by the inode lock (1.5 GB/s per tmpfs file).
// (Measured on the 16-core B200 box, 16 writers, 2 x 16 GB: a window per piece 14.0-15.9 GB/s; ONE standing mapping of
// the whole file 12.4-13.9 GB/s; either with MADV_POPULATE_WRITE before the copy 9.4-11.1 GB/s.)
bool write_mapped(int fd, const uint8_t *p, int64_t n, int64_t at) {
  const int64_t page = 4096, a0 = at & ~(page - 1), len = at + n - a0;
  void *m = mmap(nullptr, (size_t)len, PROT_READ | PROT_WRITE, MAP_SHARED, fd, (off_t)a0);
  if (m == MAP_FAILED) return false;
  memcpy(static_cast<uint8_t *>(m) + (at - a0), p, (size_t)n);
  munmap(m, (size_t)len);
  return true;
}

// shared table only: another process may have announced the size a waiting piece depends on
void poller(mg_sink *s) {
  std::unique_lock<std::mutex> lk(s->mu);
  while (!s->closing && !s->failed) {
    if (!s->waiting.empty()) refresh_known(s);
    s->cv_poll.wait_for(lk, std::chrono::microseconds(200));
  }
}

// one slot (a buffer per file) for producer p: from the cache of closed sinks, else page-locked, else ordinary memory
// (no CUDA driver -- the host logic is being exercised on a GPU-less box -- or no more lockable memory: ordinary
// memory carries the bytes just as well, the device-to-host copies are merely slower)
Slot *alloc_slot(mg_sink *s, int p) {
  Slot *sl = new Slot();
  sl->producer = p; sl->refs = 0; sl->buf[0] = sl->buf[1] = nullptr; sl->pinned = true;
  for (int f = 0; f < s->n_files; f++) {
    if ((sl->buf[f] = cache_get(s->chunk)) != nullptr) continue;
    if (!s->no_pin.load() && cudaHostAlloc((void **)&sl->buf[f], (size_t)s->chunk, cudaHostAllocPortable) != cudaSuccess) {
      cudaGetLastError();
      s->no_pin.store(true); sl->buf[f] = nullptr;
    }
    if (!sl->buf[f]) {
      sl->pinned = false;
      if (posix_memalign((void **)&sl->buf[f], 4096, (size_t)s->chunk) != 0) {
        fprintf(stderr, "mitty_b200: cannot allocate %lld bytes for the output sink\n", (long long)s->chunk);
        for (int g = 0; g < f; g++) cache_put(s->chunk, sl->buf[g]);
        delete sl;
        return nullptr;
      }
    }
  }
  return sl;
}

void deflate_piece(Piece *p, int level) { mg_deflate(p->data, p->bytes, level, 15 + 16 /* gzip wrapper */, p->z, 0); }

void worker(mg_sink *s) {
  std::unique_lock<std::mutex> lk(s->mu);
  while (true) {
    Piece *p = nullptr; int seq_file = -1;
    // 1. a sequential target whose next piece has arrived (and, for gzip, is deflated)
    for (int f = 0; f < s->n_files && !p; f++) {
      if (!sequential(s, f) || s->writing[f]) continue;
      advance(s, f);
      auto it = s->ordered[f].find({s->cur_unit[f], s->cur_off[f]});
      if (it != s->ordered[f].end() && (!s->gzip || it->second->deflated)) { p = it->second; s->ordered[f].erase(it); s->writing[f] = true; seq_file = f; }
    }
    // 2. anything in the ready queue (positional write, or a piece to deflate)
    if (!p && !s->ready.empty()) { p = s->ready.front(); s->ready.pop_front(); }
    if (!p) {
      if (s->failed || (s->closing && s->in_flight == 0)) return;
      s->cv_work.wait(lk);
      continue;
    }
    if (s->failed) { release(s, p); delete p; s->in_flight--; if (seq_file >= 0) s->writing[seq_file] = false; s->cv_idle.notify_all(); continue; }
    if (seq_file >= 0) {                                 // ordered append
      lk.unlock();
      const bool ok = s->gzip ? write_all(s->fd[seq_file], p->z.data(), (int64_t)p->z.size(), 0, false)
                              : write_all(s->fd[seq_file], p->data, p->bytes, 0, false);
      const int e = errno;
      lk.lock();
      s->writing[seq_file] = false;
      if (!ok) fail(s, "write to FASTQ file %d failed: %s", seq_file + 1, strerror(e));
      s->written[seq_file] += s->gzip ? (int64_t)p->z.size() : p->bytes;
      s->cur_off[seq_file] += p->bytes;
      if (!s->gzip) release(s, p);
      delete p; s->in_flight--;
      s->cv_work.notify_all(); s->cv_idle.notify_all();
    } else if (s->gzip) {                                // deflate, then queue for the ordered append
      lk.unlock();
      deflate_piece(p, s->gzip);
      lk.lock();
      p->deflated = true; p->data = nullptr;
      release(s, p);                                     // the pinned slot is free as soon as its bytes are deflated
      s->ordered[p->file][{p->unit, p->off}] = p;
      s->cv_work.notify_all();
    } else {                                             // positional write
      const int64_t at = s->base[(size_t)p->unit] + p->off;
      const bool mapped = s->mapped[p->file] && at + p->bytes <= s->fsize[p->file];
      lk.unlock();
      const bool ok = (mapped && write_mapped(s->fd[p->file], p->data, p->bytes, at)) || write_all(s->fd[p->file], p->data, p->bytes, at, true);
      const int e = errno;
      lk.lock();
      if (!ok) fail(s, "write to FASTQ file %d failed: %s", p->file + 1, strerror(e));
      s->written[p->file] += p->bytes;
      release(s, p);
      delete p; s->in_flight--;
      s->cv_idle.notify_all();
    }
  }
}

}  // namespace

extern "C" {

int mg_sink_create_shared(const char *path1, const char *path2, int64_t n_units, int32_t n_producers, int32_t slots_per_producer,
                          int64_t chunk_bytes, int32_t gzip_level, int32_t n_threads, const char *table_path, int32_t table_owner,
                          mg_sink **out) {
  if (!out || !path1 || n_units < 0 || n_producers < 1 || slots_per_producer < 2 || chunk_bytes < 1 || gzip_level < 0 || gzip_level > 9 ||
      chunk_bytes > (1ll << 31) - 65536 || (table_path && gzip_level)) return MG_EINVAL;
  *out = nullptr;
  mg_sink *s = new mg_sink();
  s->n_units = n_units; s->chunk = chunk_bytes; s->gzip = gzip_level;
  s->base.assign((size_t)n_units + 1, 0);
  if (table_path) {
    // [0] next-unit counter, [1] n_units, [2 ...] sizes.  The owner creates and fills it BEFORE the others open it
    // (the callers put a barrier in between); the same goes for truncating the output files.
    s->shared = true;
    s->shm_bytes = sizeof(int64_t) * (size_t)(n_units + 2);
    const int tfd = open(table_path, table_owner ? (O_RDWR | O_CREAT | O_TRUNC | O_CLOEXEC) : (O_RDWR | O_CLOEXEC), 0600);
    if (tfd < 0 || (table_owner && ftruncate(tfd, (off_t)s->shm_bytes) != 0)) {
      fprintf(stderr, "mitty_b200: cannot open the shared unit table %s: %s\n", table_path, strerror(errno));
      if (tfd >= 0) close(tfd);
      delete s;
      return MG_EVALUE;
    }
    s->shm = mmap(nullptr, s->shm_bytes, PROT_READ | PROT_WRITE, MAP_SHARED, tfd, 0);
    close(tfd);
    if (s->shm == MAP_FAILED) { delete s; return MG_EVALUE; }
    int64_t *t = static_cast<int64_t *>(s->shm);
    if (table_owner) { t[0] = 0; t[1] = n_units; for (int64_t u = 0; u < n_units; u++) t[2 + u] = -1; __atomic_thread_fence(__ATOMIC_SEQ_CST); }
    else if (t[1] != n_units) { fprintf(stderr, "mitty_b200: shared unit table %s is for %lld units, not %lld\n", table_path, (long long)t[1], (long long)n_units); munmap(s->shm, s->shm_bytes); delete s; return MG_EVALUE; }
    s->next = t; s->size = t + 2;
  } else {
    s->size_own.assign((size_t)n_units + 1, -1);
    s->size = s->size_own.data(); s->next = &s->next_own;
  }
  const char *paths[2] = {path1, path2};
  for (int f = 0; f < 2; f++) {
    if (!paths[f]) break;
    // O_TRUNC only means something for regular files; FIFOs and /dev/fd/N open as they are ('w' of the reference's writer)
    // regular (or new) targets are opened read-write: the writers map them; FIFOs / devices write-only, as the reference's 'w'
    struct stat pst;
    const bool special = stat(paths[f], &pst) == 0 && !S_ISREG(pst.st_mode);
    const int acc = special ? O_WRONLY : O_RDWR;
    s->fd[f] = open(paths[f], (table_path && !table_owner) ? (acc | O_CLOEXEC) : (acc | O_CREAT | O_TRUNC | O_CLOEXEC), 0666);
    if (s->fd[f] < 0) {
      fprintf(stderr, "mitty_b200: cannot open %s for writing: %s\n", paths[f], strerror(errno));
      for (int g = 0; g < f; g++) close(s->fd[g]);
      delete s;
      return MG_EVALUE;
    }
    struct stat st;
    // positional writes: regular files, and /dev/null-like character devices (FIFOs, pipes and ttys are not seekable)
    s->seekable[f] = fstat(s->fd[f], &st) == 0 && (S_ISREG(st.st_mode) || (S_ISCHR(st.st_mode) && lseek(s->fd[f], 0, SEEK_CUR) != (off_t)-1));
    s->mapped[f] = !gzip_level && S_ISREG(st.st_mode) && getenv("MG_SINK_PWRITE") == nullptr;
    s->n_files = f + 1;
    if (table_path && !s->seekable[f]) {
      fprintf(stderr, "mitty_b200: %s is not a regular file: several processes can only share seekable targets\n", paths[f]);
      for (int g = 0; g <= f; g++) close(s->fd[g]);
      munmap(s->shm, s->shm_bytes);
      delete s;
      return MG_EVALUE;
    }
  }
  s->pool.resize((size_t)n_producers);
  // two slots per producer now; the others are page-locked by a side thread while the first units are already
  // travelling (locking runs at about a GB/s: the 6 GB of an 8-GPU run would otherwise hold the start back for seconds)
  const int first = slots_per_producer < 2 ? slots_per_producer : 2;
  for (int k = 0; k < first; k++)
    for (int p = 0; p < n_producers; p++) {
      Slot *sl = alloc_slot(s, p);
      if (!sl) { mg_sink_close(s, nullptr, nullptr); return MG_ECUDA; }
      s->all_slots.push_back(sl);
      s->pool[(size_t)p].push_back(sl);
    }
  if (slots_per_producer > first)
    s->grower = std::thread([s, first, slots_per_producer, n_producers]() {
      for (int k = first; k < slots_per_producer; k++)
        for (int p = 0; p < n_producers; p++) {
          if (s->stop_grow.load()) return;
          Slot *sl = alloc_slot(s, p);
          if (!sl) return;                                   // the producers go on with the slots they have
          std::lock_guard<std::mutex> lk(s->mu);
          s->all_slots.push_back(sl);
          s->pool[(size_t)p].push_back(sl);
          s->cv_slot.notify_all();
        }
    });
  if (n_threads < 1) n_threads = 1;
  for (int t = 0; t < n_threads; t++) s->threads.emplace_back(worker, s);
  if (s->shared) s->threads.emplace_back(poller, s);
  *out = s;
  return MG_OK;
}

int mg_sink_create(const char *path1, const char *path2, int64_t n_units, int32_t n_producers, int32_t slots_per_producer,
                   int64_t chunk_bytes, int32_t gzip_level, int32_t n_threads, mg_sink **out) {
  return mg_sink_create_shared(path1, path2, n_units, n_producers, slots_per_producer, chunk_bytes, gzip_level, n_threads, nullptr, 1, out);
}

// Page-locking is the slow part of creating a sink (seconds for the 6 GB of an 8-GPU run): a caller that knows the
// slot size early locks the buffers from a side thread while it still parses its inputs; mg_sink_create then finds
// them in the cache.  -> buffers locked
int32_t mg_sink_prealloc(int64_t chunk_bytes, int32_t n, int32_t n_threads) {
  if (chunk_bytes < 1 || n < 1) return 0;
  if (n_threads < 1) n_threads = 1;
  if (n_threads > n) n_threads = n;
  std::vector<std::thread> th;
  std::vector<int> got((size_t)n_threads, 0);
  for (int t = 0; t < n_threads; t++)
    th.emplace_back([&, t]() {
      for (int k = t; k < n; k += n_threads) {
        uint8_t *p = nullptr;
        if (cudaHostAlloc((void **)&p, (size_t)chunk_bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return; }
        cache_put(chunk_bytes, p);
        got[(size_t)t]++;
      }
    });
  for (auto &x : th) x.join();
  int tot = 0;
  for (int g : got) tot += g;
  return tot;
}

int64_t mg_sink_next_unit(mg_sink *s) {
  if (!s) return -1;
  const int64_t k = __atomic_fetch_add(s->next, 1, __ATOMIC_ACQ_REL);
  return k < s->n_units ? k : -1;
}

const char *mg_sink_error(mg_sink *s) { return s ? s->err.c_str() : "null sink"; }

int64_t mg_sink_chunk_bytes(mg_sink *s) { return s ? s->chunk : 0; }

int mg_sink_unit_size(mg_sink *s, int64_t unit, int64_t bytes_per_file) {
  if (!s || unit < 0 || unit >= s->n_units || bytes_per_file < 0) return MG_EINVAL;
  std::lock_guard<std::mutex> lk(s->mu);
  if (s->failed) return MG_EVALUE;
  if (s->size[unit] >= 0) { fail(s, "unit %lld announced twice", (long long)unit); return MG_EINVAL; }
  __atomic_store_n(&s->size[unit], bytes_per_file, __ATOMIC_RELEASE);
  refresh_known(s);
  s->cv_work.notify_all();
  return MG_OK;
}

int mg_sink_acquire(mg_sink *s, int32_t producer, void **buf1, void **buf2, void **slot) {
  if (!s || !slot || producer < 0 || (size_t)producer >= s->pool.size()) return MG_EINVAL;
  std::unique_lock<std::mutex> lk(s->mu);
  while (s->pool[(size_t)producer].empty() && !s->failed) s->cv_slot.wait(lk);
  if (s->failed) return MG_EVALUE;
  Slot *sl = s->pool[(size_t)producer].back(); s->pool[(size_t)producer].pop_back();
  if (buf1) *buf1 = sl->buf[0];
  if (buf2) *buf2 = sl->buf[1];
  *slot = sl;
  return MG_OK;
}

int mg_sink_commit(mg_sink *s, void *slot, int64_t unit, int64_t offset, int64_t bytes) {
  if (!s || !slot || unit < 0 || unit >= s->n_units || offset < 0 || bytes < 0 || bytes > s->chunk) return MG_EINVAL;
  Slot *sl = static_cast<Slot *>(slot);
  std::lock_guard<std::mutex> lk(s->mu);
  if (s->failed || bytes == 0) { s->pool[(size_t)sl->producer].push_back(sl); s->cv_slot.notify_all(); return s->failed ? MG_EVALUE : MG_OK; }
  if (s->size[unit] < 0 || offset + bytes > s->size[unit]) { fail(s, "piece of unit %lld outside its announced size", (long long)unit); return MG_EINVAL; }
  sl->refs = s->n_files;
  for (int f = 0; f < s->n_files; f++) {
    Piece *p = new Piece();
    p->file = f; p->unit = unit; p->off = offset; p->bytes = bytes; p->data = sl->buf[f]; p->slot = sl;
    s->in_flight++;
    if (s->gzip) s->ready.push_back(p);                                        // deflate first
    else if (!s->seekable[f]) s->ordered[f][{unit, offset}] = p;
    else if (unit < s->known) s->ready.push_back(p);
    else s->waiting.insert({unit, p});
  }
  s->cv_work.notify_all();
  return MG_OK;
}

// one slot carrying SEVERAL whole or partial units (a batch of small units leaves the device as one stream): sub-piece
// i = bytes [slot_off[i], slot_off[i] + bytes[i]) of the slot = bytes [unit_off[i], ...) of unit[i].  Sub-pieces that
// follow each other in the slot AND in the files (unit k to its end, then unit k + 1 from its start) travel as one piece.
int mg_sink_commit_multi(mg_sink *s, void *slot, int32_t n, const int64_t *unit, const int64_t *unit_off, const int64_t *slot_off,
                         const int64_t *bytes) {
  if (!s || !slot || n < 0 || (n > 0 && (!unit || !unit_off || !slot_off || !bytes))) return MG_EINVAL;
  Slot *sl = static_cast<Slot *>(slot);
  std::lock_guard<std::mutex> lk(s->mu);
  struct Run { int64_t unit, off, soff, bytes; };
  std::vector<Run> runs;
  for (int i = 0; i < n && !s->failed; i++) {
    if (bytes[i] <= 0) continue;
    if (unit[i] < 0 || unit[i] >= s->n_units || s->size[unit[i]] < 0 || unit_off[i] < 0 || unit_off[i] + bytes[i] > s->size[unit[i]] ||
        slot_off[i] < 0 || slot_off[i] + bytes[i] > s->chunk) { fail(s, "piece of unit %lld outside its announced size", (long long)unit[i]); break; }
    if (!runs.empty()) {
      Run &r = runs.back();
      // the run so far ends where its last unit ends, unit[i] is the next unit of the schedule (empty ones in between do not count)
      int64_t k = r.unit, end = r.off + r.bytes;           // walk the run to its last unit
      while (k < s->n_units && s->size[k] >= 0 && end >= s->size[k] && k < unit[i]) { end -= s->size[k]; k++; }
      // (bounded, so that the writer threads share the work of one slot)
      if (k == unit[i] && end == 0 && unit_off[i] == 0 && slot_off[i] == r.soff + r.bytes && r.bytes + bytes[i] <= (4ll << 20)) { r.bytes += bytes[i]; continue; }
    }
    runs.push_back({unit[i], unit_off[i], slot_off[i], bytes[i]});
  }
  if (s->failed || runs.empty()) { s->pool[(size_t)sl->producer].push_back(sl); s->cv_slot.notify_all(); return s->failed ? MG_EVALUE : MG_OK; }
  sl->refs = s->n_files * (int)runs.size();
  for (const Run &r : runs)
    for (int f = 0; f < s->n_files; f++) {
      Piece *p = new Piece();
      p->file = f; p->unit = r.unit; p->off = r.off; p->bytes = r.bytes; p->data = sl->buf[f] + r.soff; p->slot = sl;
      s->in_flight++;
      if (s->gzip) s->ready.push_back(p);
      else if (!s->seekable[f]) s->ordered[f][{p->unit, p->off}] = p;
      else if (p->unit < s->known) s->ready.push_back(p);
      else s->waiting.insert({p->unit, p});
    }
  s->cv_work.notify_all();
  return MG_OK;
}

void mg_sink_abort(mg_sink *s, const char *why) {
  if (!s) return;
  std::lock_guard<std::mutex> lk(s->mu);
  fail(s, "%s", why ? why : "aborted");
}

int mg_sink_close(mg_sink *s, int64_t *written1, int64_t *written2) {
  if (!s) return MG_EINVAL;
  {
    std::unique_lock<std::mutex> lk(s->mu);
    while (s->in_flight > 0 && !s->failed) s->cv_idle.wait(lk);
    if (!s->failed && !s->shared)
      for (int64_t u = 0; u < s->n_units; u++)
        if (s->size[u] < 0) { fail(s, "unit %lld was never written", (long long)u); break; }
    s->closing = true;
    s->cv_work.notify_all(); s->cv_poll.notify_all();
  }
  s->stop_grow.store(true);
  if (s->grower.joinable()) s->grower.join();
  for (auto &t : s->threads) t.join();
  const bool failed = s->failed;
  if (written1) *written1 = s->written[0];
  if (written2) *written2 = s->written[1];
  for (int f = 0; f < s->n_files; f++) if (s->fd[f] >= 0 && close(s->fd[f]) != 0 && !failed) { s->err = std::string("close: ") + strerror(errno); }
  for (auto &kv : s->waiting) delete kv.second;
  for (Piece *p : s->ready) delete p;
  for (int f = 0; f < 2; f++) for (auto &kv : s->ordered[f]) delete kv.second;
  for (Slot *sl : s->all_slots) {
    for (int f = 0; f < 2; f++) if (sl->buf[f]) cache_put(s->chunk, sl->buf[f]);      // kept for the next sink of this process
    delete sl;
  }
  if (s->shm) munmap(s->shm, s->shm_bytes);
  const int rc = failed || !s->err.empty() ? MG_EVALUE : MG_OK;
  if (rc != MG_OK) fprintf(stderr, "mitty_b200: output sink: %s\n", s->err.c_str());
  delete s;
  return rc;
}

}  // extern "C"
