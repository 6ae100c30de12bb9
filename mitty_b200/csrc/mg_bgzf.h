// BGZF writer and BAI builder of the god-aligner (SAM spec v1 §4.1, §5.2) and the BGZF BAM reader of
// bam2illumina, host code only: the device encodes and sorts the BAM records (mg_bam.cu) or counts them
// (mg_readmodel.cu), these write or read them.
#pragma once
#include <stdint.h>

#include <map>
#include <string>
#include <thread>
#include <vector>

#define MG_BGZF_BLOCK 65280   // uncompressed bytes per BGZF member (htslib's BGZF_BLOCK_SIZE)

// Binary BAM header: magic, l_text, text, then the reference list.
std::vector<uint8_t> mg_bam_header(const std::string &text, const std::vector<std::string> &names, const std::vector<int64_t> &lens);

// The uncompressed stream is cut into fixed MG_BGZF_BLOCK-byte blocks, deflated by `threads` host threads
// (one batch of blocks in flight while the next one fills), written in order; close() appends the EOF block.
class MgBgzf {
 public:
  ~MgBgzf();
  bool open(const char *path, int level, int threads);
  bool write(const uint8_t *p, int64_t n);
  bool close();                               // flushes the last block, writes the EOF member
  uint64_t tell() const { return raw_; }      // uncompressed offset
  // compressed offset of block k (k = number of blocks: the EOF member's); valid after close()
  std::vector<uint64_t> block_start;
  std::string err;
 private:
  struct Batch { std::vector<uint8_t> raw; int64_t fill = 0; std::vector<std::vector<uint8_t>> z; };
  bool submit();                              // hand the filling batch to the deflate threads
  bool drain();                               // wait for the batch in flight, write it
  int fd_ = -1, level_ = 6, threads_ = 1;
  uint64_t raw_ = 0, comp_ = 0;
  Batch b_[2];
  int cur_ = 0;
  bool busy_ = false;
  std::thread runner_;
};

// BAI over records pushed in file order with their uncompressed stream offsets; the offsets become
// virtual file offsets once the block layout is known.
class MgBai {
 public:
  explicit MgBai(int n_ref) : refs_((size_t)n_ref) {}
  // one BAM record at uncompressed [ubeg, uend); the record's own bytes give refID, pos, bin and end
  void push(const uint8_t *rec, uint64_t ubeg, uint64_t uend);
  bool write(const char *path, const std::vector<uint64_t> &block_start);
 private:
  struct Ref {
    std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
    std::vector<uint64_t> lin;
    uint64_t beg = 0, end = 0, n_mapped = 0;
  };
  void close_chunk();
  std::vector<Ref> refs_;
  int cur_ref_ = -1; uint32_t cur_bin_ = 0; uint64_t chunk_beg_ = 0, last_end_ = 0;
};

// A BAM writer over a stream of whole or partial records: BGZF + BAI.
class MgBamWriter {
 public:
  bool open(const char *bam, const char *bai, const std::vector<uint8_t> &header, int n_ref, int level, int threads);
  bool records(const uint8_t *p, int64_t n);    // any cut of the record stream
  bool close(int64_t *n_records);
  void discard();                               // on error: remove what was written
  std::string err;
 private:
  MgBgzf z_;
  MgBai *bai_ = nullptr;
  std::string bam_, bai_path_;
  std::vector<uint8_t> pend_;                   // the record that straddles two calls
  int64_t n_ = 0;
};

// Reader errors (MgBamReader::code; the device adds MG_RD_NAME .. MG_RD_QUAL).  `where` is the compressed
// file offset of the member for the framing codes, the record ordinal (0-based, over the whole file) for
// the record codes.
enum {
  MG_RD_OK = 0,
  MG_RD_GZIP = 1,      // offset: not a gzip member (magic, method, or no FEXTRA flag)
  MG_RD_BC = 2,        // offset: the gzip extra field has no 'BC' subfield
  MG_RD_DATA = 3,      // offset: corrupt or truncated member
  MG_RD_CRC = 4,       // offset: CRC32 of the inflated bytes differs
  MG_RD_ISIZE = 5,     // offset: ISIZE differs from the inflated length, or exceeds 65536
  MG_RD_MAGIC = 6,     // offset 0: the stream does not start with BAM\1
  MG_RD_HEADER = 7,    // offset: the file ends inside the BAM header
  MG_RD_BLOCK = 8,     // record: block_size < 32
  MG_RD_CUT = 9,       // record: the file ends inside the record
  MG_RD_IO = 10,       // offset: read error
  MG_RD_NAME = 11,     // record: read name overruns block_size (checked on the device)
  MG_RD_CIGAR = 12,    // record: CIGAR overruns block_size
  MG_RD_SEQ = 13,      // record: SEQ overruns block_size (or l_seq < 0)
  MG_RD_QUAL = 14,     // record: QUAL overruns block_size
};

// Whole BAM records of a chunk: data[0, bytes) holds them (a chunk may start with header bytes, which no
// offset points at); off[i] = offset of record first + i.
struct MgBamChunk { const uint8_t *data; int64_t bytes; const uint32_t *off; int64_t n; int64_t first; };

// Sequential reader of a BGZF BAM file or FIFO.  Members are parsed in order (any XLEN; the 'BC'
// subfield gives the member size); the ISIZE of each member gives its output offset before anything is
// inflated, so `threads` host threads inflate a batch of members straight into the chunk buffer and check
// CRC32 and ISIZE.  next() walks the block_size chain of the inflated stream and hands out the whole
// records; the cut record carries over to the next chunk.  Two chunk buffers alternate (slot 0 / 1), so
// the caller may still be copying one while the next one is inflated; `alloc` / `release` provide them
// (page-locked memory for copies to a device).  A record larger than the buffer grows it.
class MgBamReader {
 public:
  typedef void *(*Alloc)(size_t);
  typedef void (*Release)(void *);
  ~MgBamReader();
  bool open(const char *path, int threads, int64_t chunk_bytes, Alloc alloc, Release release);
  // the next chunk (n >= 1) in buffer `slot`; false at the end of the input or at the first error (code)
  bool next(int slot, MgBamChunk &c);
  int code = MG_RD_OK; int64_t where = -1;
  std::string err;                             // open() failure
  int64_t records = 0, raw_bytes = 0, comp_bytes = 0;
  bool eof_marker = false;                     // the last member is the 28-byte EOF member
  double read_ms = 0, inflate_ms = 0, walk_ms = 0;   // reading the file; inflating (wall time); walking the record chain
  std::vector<double> thread_ms;               // busy time of each inflate thread
 private:
  struct Member { const uint8_t *z; int hdr, bsize; uint32_t crc, isize; int64_t out, comp; };
  int fill(uint8_t *b, int64_t &n, int64_t cap);          // 1: next member does not fit, 0: input ended or failed
  void read_more();
  int64_t header(const uint8_t *b, int64_t pos, int64_t n);
  void fail(int c, int64_t w) { if (!code) { code = c; where = w; } }
  bool grow(int slot, int64_t need, int64_t keep);
  int fd_ = -1, threads_ = 1;
  Alloc alloc_ = nullptr; Release release_ = nullptr;
  uint8_t *buf_[2] = {nullptr, nullptr}; uint32_t *off_[2] = {nullptr, nullptr};
  int64_t cap_[2] = {0, 0};
  std::vector<uint8_t> z_; int64_t zpos_ = 0, zend_ = 0, zoff_ = 0;
  bool in_eof_ = false, done_ = false;
  int carry_slot_ = -1; int64_t carry_at_ = 0, carry_n_ = 0;
  int hstate_ = 0; int64_t hskip_ = 0, hrefs_ = 0;          // BAM header walk
  std::vector<Member> batch_;
};
