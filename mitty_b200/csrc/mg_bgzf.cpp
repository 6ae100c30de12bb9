// BGZF writer, BAI builder and the device-free BAM entry point of the god-aligner.
//
// BGZF (SAM spec §4.1): gzip members of at most 64 KiB with a 'BC' extra field carrying the member size
// minus one.  The uncompressed stream -- header, then records -- is cut into fixed MG_BGZF_BLOCK-byte
// blocks as htslib does, so the member layout, and with it every virtual offset of the index, depends on
// the bytes alone (not on threads or timing).  Blocks are deflated in batches by host threads
// (mg_deflate, shared with the FASTQ sink) while the caller fills the next batch.
//
// BAI (§5.2): records arrive in coordinate order; consecutive records of one bin form one chunk of that
// bin; the 16 kb linear index holds the first record that overlaps each window (windows no record
// overlaps take the next window's value); per reference the pseudo-bin 37450 holds the offset range and
// the mapped / unmapped counts.  Offsets are kept uncompressed until close, then mapped to virtual offsets
// through the block table: u -> block_start[u / 65280] << 16 | u % 65280.
#include <fcntl.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstdlib>
#include <cstdio>
#include <cstring>

#include "../../include/mitty_b200.h"
#include "mg_bgzf.h"
#include "mg_deflate.h"

namespace {

const int kBatchBlocksPerThread = 8;
const uint8_t kEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

inline uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline void put16(uint8_t *p, uint16_t v) { memcpy(p, &v, 2); }
inline void put32(uint8_t *p, uint32_t v) { memcpy(p, &v, 4); }
void app32(std::vector<uint8_t> &o, uint32_t v) { uint8_t b[4]; put32(b, v); o.insert(o.end(), b, b + 4); }
void app64(std::vector<uint8_t> &o, uint64_t v) { uint8_t b[8]; memcpy(b, &v, 8); o.insert(o.end(), b, b + 8); }

// one BGZF member: 18-byte header with BSIZE, raw deflate, CRC32, ISIZE
void bgzf_block(const uint8_t *in, int64_t n, int level, std::vector<uint8_t> &out) {
  mg_deflate(in, n, level, -15, out, 18);
  if (out.size() + 8 > 65536) mg_deflate(in, n, 0, -15, out, 18);    // incompressible at this level: stored blocks always fit
  static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0};
  memcpy(out.data(), hdr, 16);
  const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), in, (uInt)n);
  app32(out, crc); app32(out, (uint32_t)n);
  put16(out.data() + 16, (uint16_t)(out.size() - 1));
}

bool write_all(int fd, const uint8_t *p, size_t n) {
  while (n > 0) {
    const ssize_t w = write(fd, p, n);
    if (w < 0) { if (errno == EINTR) continue; return false; }
    p += w; n -= (size_t)w;
  }
  return true;
}

// SAM spec §5.3: the smallest bin that holds [beg, end)
inline uint32_t reg2bin(int64_t beg, int64_t end) {
  --end;
  if (beg >> 14 == end >> 14) return (uint32_t)(((1 << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (uint32_t)(((1 << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (uint32_t)(((1 << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (uint32_t)(((1 << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (uint32_t)(((1 << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

}  // namespace

std::string mg_bam_check_contigs(const std::vector<std::string> &names, const std::vector<int64_t> &lens) {
  for (size_t i = 0; i < names.size(); i++)
    if (lens[i] < 0 || lens[i] > INT32_MAX)
      return "contig " + names[i] + " has " + std::to_string(lens[i]) + " bases: a BAM file addresses 0 .. 2^31 - 1";
  return "";
}

static thread_local std::string host_err;
const char *mg_bam_host_error() { return host_err.c_str(); }

std::vector<uint8_t> mg_bam_header(const std::string &text, const std::vector<std::string> &names, const std::vector<int64_t> &lens) {
  std::vector<uint8_t> h = {'B', 'A', 'M', 1};
  app32(h, (uint32_t)text.size());
  h.insert(h.end(), text.begin(), text.end());
  app32(h, (uint32_t)names.size());
  for (size_t i = 0; i < names.size(); i++) {
    app32(h, (uint32_t)(names[i].size() + 1));
    h.insert(h.end(), names[i].begin(), names[i].end());
    h.push_back(0);
    app32(h, (uint32_t)lens[i]);
  }
  return h;
}

// ---- BGZF ----------------------------------------------------------------------------------------

MgBgzf::~MgBgzf() {
  if (runner_.joinable()) runner_.join();
  if (fd_ >= 0) ::close(fd_);
}

bool MgBgzf::open(const char *path, int level, int threads) {
  fd_ = ::open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (fd_ < 0) { err = std::string("cannot create ") + path + ": " + strerror(errno); return false; }
  level_ = level; threads_ = threads < 1 ? 1 : threads;
  for (Batch &b : b_) b.raw.resize((size_t)MG_BGZF_BLOCK * kBatchBlocksPerThread * threads_);
  block_start.assign(1, 0);
  return true;
}

bool MgBgzf::write(const uint8_t *p, int64_t n) {
  while (n > 0) {
    Batch &b = b_[cur_];
    const int64_t take = std::min<int64_t>(n, (int64_t)b.raw.size() - b.fill);
    memcpy(b.raw.data() + b.fill, p, (size_t)take);
    b.fill += take; p += take; n -= take; raw_ += (uint64_t)take;
    if (b.fill == (int64_t)b.raw.size() && !submit()) return false;
  }
  return true;
}

bool MgBgzf::submit() {
  if (!drain()) return false;
  Batch *b = &b_[cur_];
  const int n_blk = (int)((b->fill + MG_BGZF_BLOCK - 1) / MG_BGZF_BLOCK);
  b->z.resize((size_t)n_blk);
  const int level = level_, threads = threads_;
  runner_ = std::thread([b, n_blk, level, threads] {
    std::atomic<int> next{0};
    auto work = [&] {
      for (int k; (k = next++) < n_blk;)
        bgzf_block(b->raw.data() + (int64_t)k * MG_BGZF_BLOCK, std::min<int64_t>(MG_BGZF_BLOCK, b->fill - (int64_t)k * MG_BGZF_BLOCK), level, b->z[(size_t)k]);
    };
    std::vector<std::thread> t;
    for (int i = 1; i < std::min(threads, n_blk); i++) t.emplace_back(work);
    work();
    for (auto &x : t) x.join();
  });
  busy_ = true;
  cur_ ^= 1;
  return true;
}

bool MgBgzf::drain() {
  if (!busy_) return true;
  runner_.join();
  busy_ = false;
  Batch &b = b_[cur_ ^ 1];
  for (auto &z : b.z) {
    if (!write_all(fd_, z.data(), z.size())) { err = std::string("BAM write failed: ") + strerror(errno); return false; }
    comp_ += z.size();
    block_start.push_back(comp_);
  }
  b.fill = 0;
  return true;
}

bool MgBgzf::close() {
  if (b_[cur_].fill && !submit()) return false;
  if (!drain()) return false;
  if (!write_all(fd_, kEof, sizeof kEof)) { err = std::string("BAM write failed: ") + strerror(errno); return false; }
  const bool ok = ::close(fd_) == 0;
  fd_ = -1;
  if (!ok) err = "BAM close failed";
  return ok;
}

// ---- BAI -----------------------------------------------------------------------------------------

void MgBai::close_chunk() {
  if (cur_ref_ >= 0) refs_[(size_t)cur_ref_].bins[cur_bin_].push_back({chunk_beg_, last_end_});
}

void MgBai::push(const uint8_t *rec, uint64_t ubeg, uint64_t uend) {
  const int ref = (int)rd32(rec + 4);
  const int64_t pos = (int32_t)rd32(rec + 8);
  const uint32_t bin = rd32(rec + 12) >> 16;
  const int l_name = rec[12], n_cig = (int)(rd32(rec + 16) & 0xFFFF);
  int64_t span = 0;
  for (int i = 0; i < n_cig; i++) {
    const uint32_t c = rd32(rec + 36 + l_name + 4 * i), op = c & 15;
    if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += c >> 4;
  }
  const int64_t end = pos + (span > 0 ? span : 1);
  if (ref != cur_ref_ || bin != cur_bin_) {
    close_chunk();
    cur_ref_ = ref; cur_bin_ = bin; chunk_beg_ = ubeg;
  }
  Ref &R = refs_[(size_t)ref];
  if (R.n_mapped == 0) R.beg = ubeg;
  R.end = uend; R.n_mapped++;
  const int64_t w1 = (end - 1) >> 14;
  if ((int64_t)R.lin.size() <= w1) R.lin.resize((size_t)w1 + 1, UINT64_MAX);
  for (int64_t w = pos >> 14; w <= w1; w++) if (R.lin[(size_t)w] == UINT64_MAX) R.lin[(size_t)w] = ubeg;
  last_end_ = uend;
}

bool MgBai::write(const char *path, const std::vector<uint64_t> &bs) {
  close_chunk(); cur_ref_ = -1;
  auto v = [&](uint64_t u) { return bs[(size_t)(u / MG_BGZF_BLOCK)] << 16 | (u % MG_BGZF_BLOCK); };
  std::vector<uint8_t> o = {'B', 'A', 'I', 1};
  app32(o, (uint32_t)refs_.size());
  for (Ref &R : refs_) {
    app32(o, (uint32_t)(R.bins.size() + (R.n_mapped ? 1 : 0)));
    for (auto &b : R.bins) {
      app32(o, b.first); app32(o, (uint32_t)b.second.size());
      for (auto &c : b.second) { app64(o, v(c.first)); app64(o, v(c.second)); }
    }
    if (R.n_mapped) {
      app32(o, 37450); app32(o, 2);
      app64(o, v(R.beg)); app64(o, v(R.end)); app64(o, R.n_mapped); app64(o, 0);
    }
    for (size_t w = R.lin.size(); w-- > 1;) if (R.lin[w - 1] == UINT64_MAX) R.lin[w - 1] = R.lin[w];
    app32(o, (uint32_t)R.lin.size());
    for (uint64_t u : R.lin) app64(o, v(u));
  }
  app64(o, 0);   // n_no_coor
  const int fd = ::open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (fd < 0) return false;
  const bool ok = write_all(fd, o.data(), o.size());
  return ::close(fd) == 0 && ok;
}

// ---- BAM writer ----------------------------------------------------------------------------------

bool MgBamWriter::open(const char *bam, const char *bai, const std::vector<uint8_t> &header, int n_ref, int level, int threads) {
  bam_ = bam; bai_path_ = bai ? bai : "";
  if (!z_.open(bam, level, threads)) { err = z_.err; return false; }
  if (bai) bai_ = new MgBai(n_ref);
  return z_.write(header.data(), (int64_t)header.size()) || (err = z_.err, false);
}

bool MgBamWriter::records(const uint8_t *p, int64_t n) {
  auto emit = [&](const uint8_t *rec, int64_t sz) {
    const uint64_t u = z_.tell();
    if (!z_.write(rec, sz)) { err = z_.err; return false; }
    if (bai_) bai_->push(rec, u, u + (uint64_t)sz);
    n_++;
    return true;
  };
  while (n > 0) {
    if (!pend_.empty()) {                                 // finish the straddling record first
      const int64_t need = pend_.size() < 4 ? 4 : 4 + (int64_t)rd32(pend_.data());
      const int64_t take = std::min<int64_t>(n, need - (int64_t)pend_.size());
      pend_.insert(pend_.end(), p, p + take); p += take; n -= take;
      if (pend_.size() >= 4 && (int64_t)pend_.size() == 4 + (int64_t)rd32(pend_.data())) {
        if (!emit(pend_.data(), (int64_t)pend_.size())) return false;
        pend_.clear();
      }
      continue;
    }
    if (n < 4 || 4 + (int64_t)rd32(p) > n) { pend_.assign(p, p + n); break; }
    const int64_t sz = 4 + (int64_t)rd32(p);
    if (!emit(p, sz)) return false;
    p += sz; n -= sz;
  }
  return true;
}

bool MgBamWriter::close(int64_t *n_records) {
  if (!pend_.empty()) { err = "the record stream ends inside a record"; discard(); return false; }
  if (!z_.close()) { err = z_.err; discard(); return false; }
  if (bai_ && !bai_->write(bai_path_.c_str(), z_.block_start)) { err = "cannot write " + bai_path_; discard(); return false; }
  delete bai_; bai_ = nullptr;
  if (n_records) *n_records = n_;
  return true;
}

void MgBamWriter::discard() {
  z_.close();
  unlink(bam_.c_str());
  if (!bai_path_.empty()) unlink(bai_path_.c_str());
  delete bai_; bai_ = nullptr;
}

extern "C" int mg_bam_write_sorted(const char *bam_path, const char *bai_path, int32_t n_ref, const char *const *ref_names, const int64_t *ref_len,
                                   const char *header_text, const uint8_t *records, int64_t len, int32_t level, int32_t threads, int64_t *n_records) {
  if (!bam_path || n_ref < 0 || (n_ref && (!ref_names || !ref_len)) || !header_text || (len && !records) || level < 0 || level > 9) return MG_EINVAL;
  std::vector<std::string> names; std::vector<int64_t> lens;
  for (int i = 0; i < n_ref; i++) { names.push_back(ref_names[i]); lens.push_back(ref_len[i]); }
  host_err = mg_bam_check_contigs(names, lens);
  if (!host_err.empty()) return MG_EVALUE;
  MgBamWriter w;
  if (!w.open(bam_path, bai_path, mg_bam_header(header_text, names, lens), n_ref, level, threads) || !w.records(records, len)) {
    host_err = w.err;
    w.discard();
    return MG_EVALUE;
  }
  if (w.close(n_records)) return MG_OK;
  host_err = w.err;
  return MG_EVALUE;
}

// ---- BGZF BAM reader -----------------------------------------------------------------------------

namespace {

double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

const int64_t kMaxMember = 65536;

// -> 0: a whole member at p[0, m.bsize); > 0: bytes needed to decide; < 0: -MG_RD_* of a malformed member
int64_t parse_member(const uint8_t *p, int64_t avail, int &hdr, int &bsize) {
  if (avail < 12) return 12;
  if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return -MG_RD_GZIP;
  const int xlen = p[10] | p[11] << 8;
  if (avail < 12 + xlen) return 12 + xlen;
  bsize = -1;
  for (int i = 12; i + 4 <= 12 + xlen;) {            // subfields: SI1 SI2 SLEN data
    const int slen = p[i + 2] | p[i + 3] << 8;
    if (p[i] == 'B' && p[i + 1] == 'C' && slen == 2 && i + 6 <= 12 + xlen) bsize = (p[i + 4] | p[i + 5] << 8) + 1;
    i += 4 + slen;
  }
  if (bsize < 0) return -MG_RD_BC;
  if (avail < bsize) return bsize;
  hdr = 12 + xlen;
  for (int f : {8, 16}) {                              // FNAME, FCOMMENT: zero-terminated
    if (!(p[3] & f)) continue;
    while (hdr < bsize && p[hdr]) hdr++;
    hdr++;
  }
  if (p[3] & 2) hdr += 2;                              // FHCRC
  return hdr + 8 > bsize ? -MG_RD_DATA : 0;
}

}  // namespace

MgBamReader::~MgBamReader() {
  if (fd_ >= 0) ::close(fd_);
  for (int s = 0; s < 2; s++) {
    if (buf_[s]) release_(buf_[s]);
    if (off_[s]) release_(off_[s]);
  }
}

bool MgBamReader::open(const char *path, int threads, int64_t chunk_bytes, Alloc alloc, Release release) {
  alloc_ = alloc; release_ = release;
  threads_ = std::max(1, threads);
  thread_ms.assign((size_t)threads_, 0.0);
  fd_ = ::open(path, O_RDONLY);
  if (fd_ < 0) { err = std::string("cannot open ") + path + ": " + strerror(errno); return false; }
  const int64_t cap = std::min<int64_t>(std::max<int64_t>(chunk_bytes, 2 * kMaxMember), 1ll << 31);
  z_.resize((size_t)(cap + 2 * kMaxMember));
  return grow(0, cap, 0) && grow(1, cap, 0);
}

// buffer `slot` of at least `need` bytes, its first `keep` bytes kept; records are at least 36 bytes
bool MgBamReader::grow(int slot, int64_t need, int64_t keep) {
  if (need <= cap_[slot]) return true;
  if (need >= (1ll << 32)) { err = "a BAM record larger than 4 GB"; return false; }
  uint8_t *b = static_cast<uint8_t *>(alloc_((size_t)need));
  uint32_t *o = static_cast<uint32_t *>(alloc_((size_t)(need / 36 + 2) * 4));
  if (!b || !o) {
    if (b) release_(b);
    if (o) release_(o);
    err = "out of host memory for a chunk of " + std::to_string(need) + " bytes";
    return false;
  }
  if (keep) memcpy(b, buf_[slot], (size_t)keep);
  if (buf_[slot]) { release_(buf_[slot]); release_(off_[slot]); }
  buf_[slot] = b; off_[slot] = o; cap_[slot] = need;
  return true;
}

// moves the unparsed compressed bytes to the front and reads until the buffer is full or the input ends
void MgBamReader::read_more() {
  const double t0 = now_ms();
  memmove(z_.data(), z_.data() + zpos_, (size_t)(zend_ - zpos_));
  zoff_ += zpos_; zend_ -= zpos_; zpos_ = 0;
  while (zend_ < (int64_t)z_.size() && !in_eof_) {
    const ssize_t r = ::read(fd_, z_.data() + zend_, z_.size() - (size_t)zend_);
    if (r < 0 && errno == EINTR) continue;
    if (r < 0) { fail(MG_RD_IO, zoff_ + zend_); in_eof_ = true; break; }
    if (r == 0) in_eof_ = true;
    zend_ += r;
  }
  read_ms += now_ms() - t0;
}

// appends whole members to b[n, cap), inflated by the thread team.  -> 1 when the next member does not fit,
// 0 when the input has ended or a member is bad (code set; n then ends where that member's bytes would start)
int MgBamReader::fill(uint8_t *b, int64_t &n, int64_t cap) {
  while (true) {
    batch_.clear();
    int64_t out = n;
    int state = 2;                                     // 2: the compressed buffer needs refilling
    while (true) {
      Member m;
      const int64_t r = parse_member(z_.data() + zpos_, zend_ - zpos_, m.hdr, m.bsize);
      if (r < 0) { fail((int)-r, zoff_ + zpos_); state = 0; break; }
      if (r > 0) {
        if (in_eof_) {
          if (zend_ > zpos_) fail(MG_RD_DATA, zoff_ + zpos_);
          state = 0;
          break;
        }
        if (!batch_.empty()) break;
        read_more();
        continue;
      }
      m.z = z_.data() + zpos_;
      m.crc = rd32(m.z + m.bsize - 8); m.isize = rd32(m.z + m.bsize - 4);
      m.comp = zoff_ + zpos_;
      if (m.isize > kMaxMember) { fail(MG_RD_ISIZE, m.comp); state = 0; break; }
      if (out + m.isize > cap) { state = 1; break; }
      m.out = out; out += m.isize;
      eof_marker = m.bsize == 28 && !memcmp(m.z, kEof, 28);
      zpos_ += m.bsize; comp_bytes += m.bsize;
      batch_.push_back(m);
    }
    const int nm = (int)batch_.size();
    if (nm) {
      const double t0 = now_ms();
      std::vector<int> st((size_t)nm, 0);
      std::atomic<int> next{0};
      auto work = [&](int t) {
        const double w0 = now_ms();
        for (int i; (i = next++) < nm;) {
          const Member &m = batch_[(size_t)i];
          const int rc = mg_inflate(m.z + m.hdr, m.bsize - m.hdr - 8, b + m.out, m.isize);
          st[(size_t)i] = rc == 1 ? MG_RD_DATA : rc == 2 ? MG_RD_ISIZE
                        : (uint32_t)crc32(crc32(0L, Z_NULL, 0), b + m.out, (uInt)m.isize) != m.crc ? MG_RD_CRC : MG_RD_OK;
        }
        thread_ms[(size_t)t] += now_ms() - w0;
      };
      std::vector<std::thread> team;
      for (int t = 1; t < std::min(threads_, nm); t++) team.emplace_back(work, t);
      work(0);
      for (auto &x : team) x.join();
      inflate_ms += now_ms() - t0;
      for (int i = 0; i < nm; i++) {
        if (st[(size_t)i] == MG_RD_OK) continue;
        code = MG_RD_OK;                               // a bad member comes before any later framing error
        fail(st[(size_t)i], batch_[(size_t)i].comp);
        out = batch_[(size_t)i].out;
        state = 0;
        break;
      }
    }
    raw_bytes += out - n;
    n = out;
    if (state != 2) return state;
  }
}

// consumes BAM header bytes of b[pos, n) (magic, l_text, text, n_ref, the references) -> the new position
int64_t MgBamReader::header(const uint8_t *b, int64_t pos, int64_t n) {
  while (hstate_ != 3 || hskip_) {
    if (hskip_) {
      const int64_t t = std::min(hskip_, n - pos);
      if (hname_) {                                    // the skip starts with the reference's name: keep it up to its NUL
        const int64_t c = std::min(t, hname_);
        if (!hnul_) {
          const uint8_t *z = static_cast<const uint8_t *>(memchr(b + pos, 0, (size_t)c));
          ref_names.insert(ref_names.end(), b + pos, z ? z : b + pos + c);
          hnul_ = z != nullptr;
        }
        if ((hname_ -= c) == 0) ref_off.push_back((int64_t)ref_names.size());
      }
      pos += t; hskip_ -= t;
      if (hskip_) return pos;
      continue;
    }
    if (n - pos < (hstate_ == 0 ? 8 : 4)) return pos;
    const int32_t v = (int32_t)rd32(b + pos + (hstate_ == 0 ? 4 : 0));
    if ((hstate_ == 0 && memcmp(b + pos, "BAM\1", 4)) || v < 0) { fail(MG_RD_MAGIC, 0); hstate_ = 3; return pos; }
    pos += hstate_ == 0 ? 8 : 4;
    if (hstate_ == 0) { hskip_ = v; hstate_ = 1; }
    else if (hstate_ == 1) { hrefs_ = v; hstate_ = v ? 2 : 3; }
    else {
      hskip_ = (int64_t)v + 4; hname_ = v; hnul_ = false;
      if (!v) ref_off.push_back((int64_t)ref_names.size());
      if (--hrefs_ == 0) hstate_ = 3;
    }
  }
  return pos;
}

bool MgBamReader::next(int slot, MgBamChunk &c) {
  if (code || !err.empty() || (done_ && !carry_n_)) return false;
  if (carry_slot_ != slot && !grow(slot, carry_n_, 0)) return false;
  if (carry_n_) memmove(buf_[slot], buf_[carry_slot_] + carry_at_, (size_t)carry_n_);
  int64_t n = carry_n_, pos = 0, k = 0;
  carry_n_ = 0;
  bool stop = false;
  while (true) {
    const int more = done_ ? 0 : fill(buf_[slot], n, cap_[slot]);
    if (hstate_ != 3 || hskip_) pos = header(buf_[slot], pos, n);
    if (code == MG_RD_MAGIC) { done_ = true; break; }
    const double t0 = now_ms();
    while (hstate_ == 3 && !hskip_ && !stop && n - pos >= 4) {
      __builtin_prefetch(buf_[slot] + std::min(pos + 4096, n - 1));      // the chain runs forward through memory the inflate threads wrote
      const int32_t bs = (int32_t)rd32(buf_[slot] + pos);
      if (bs < 32) { code = MG_RD_BLOCK; where = records + k; stop = true; break; }   // before any framing error found further on
      if (4 + (int64_t)bs > n - pos) break;
      off_[slot][k++] = (uint32_t)pos;
      pos += 4 + (int64_t)bs;
    }
    walk_ms += now_ms() - t0;
    if (stop || !more) { done_ = true; break; }
    if (k) break;
    if (pos) { memmove(buf_[slot], buf_[slot] + pos, (size_t)(n - pos)); n -= pos; pos = 0; continue; }   // header bytes only
    if (!grow(slot, 2 * cap_[slot], n)) return false;                                               // a record larger than the buffer
  }
  if (done_ && !code) {
    if (hstate_ != 3 || hskip_) fail(MG_RD_HEADER, zoff_ + zend_);
    else if (pos < n) fail(MG_RD_CUT, records + k);
  }
  carry_slot_ = slot; carry_at_ = pos; carry_n_ = done_ ? 0 : n - pos;
  if (!k) return false;
  c.data = buf_[slot]; c.bytes = pos; c.off = off_[slot]; c.n = k; c.first = records;
  records += k;
  return true;
}

namespace {
void *host_alloc(size_t n) { return malloc(n); }
void host_release(void *p) { free(p); }
}  // namespace

extern "C" int mg_bam_scan(const char *path, int32_t threads, int64_t chunk_bytes, int64_t *stats, int64_t *bad_where, int32_t *bad_code) {
  if (!path || !stats || !bad_where || !bad_code) return MG_EINVAL;
  *bad_where = -1; *bad_code = 0;
  MgBamReader rd;
  if (!rd.open(path, threads, chunk_bytes, host_alloc, host_release)) return MG_EVALUE;
  MgBamChunk c;
  for (int k = 0; rd.next(k & 1, c); k++) {}
  stats[0] = rd.records; stats[1] = rd.raw_bytes; stats[2] = rd.comp_bytes; stats[3] = rd.eof_marker;
  if (rd.code) { *bad_where = rd.where; *bad_code = rd.code; return MG_EVALUE; }
  return rd.err.empty() ? MG_OK : MG_EVALUE;
}
