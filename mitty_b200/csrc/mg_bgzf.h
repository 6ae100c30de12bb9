// BGZF writer and BAI builder of the god-aligner (SAM spec v1 §4.1, §5.2), host code only: the device
// encodes and sorts the BAM records (mg_bam.cu), these write them.
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
