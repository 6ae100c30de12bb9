// One zlib deflate stream, shared by the FASTQ sink (gzip members, mg_sink.cpp) and the BGZF writer
// of the god-aligner (raw deflate inside its own member framing, mg_bgzf.cpp), and the raw inflate of
// the BGZF reader (mg_bgzf.cpp).
#pragma once
#include <stdint.h>
#include <vector>

// deflates in[0, n) at `level` into out[head, ...) and resizes out to head + the compressed bytes.
// window_bits as for deflateInit2: 15 + 16 writes a gzip member, -15 raw deflate.
void mg_deflate(const uint8_t *in, int64_t n, int level, int window_bits, std::vector<uint8_t> &out, size_t head);

// inflates the raw deflate stream in[0, n) into out[0, out_len).  -> 0 when the stream ends exactly at
// in + n and produced exactly out_len bytes, 1 corrupt or truncated deflate data, 2 a different length.
int mg_inflate(const uint8_t *in, int64_t n, uint8_t *out, int64_t out_len);
