// One zlib deflate stream, shared by the FASTQ sink (gzip members, mg_sink.cpp) and the BGZF writer
// of the god-aligner (raw deflate inside its own member framing, mg_bgzf.cpp).
#pragma once
#include <stdint.h>
#include <vector>

// deflates in[0, n) at `level` into out[head, ...) and resizes out to head + the compressed bytes.
// window_bits as for deflateInit2: 15 + 16 writes a gzip member, -15 raw deflate.
void mg_deflate(const uint8_t *in, int64_t n, int level, int window_bits, std::vector<uint8_t> &out, size_t head);
