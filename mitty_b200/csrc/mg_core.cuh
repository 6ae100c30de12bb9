// Per-thread logic of the read-generation engine, shared by every kernel.
//
// Everything here is __host__ __device__ and free of CUDA-only constructs so that
// tests/emul/ can compile the very same code with g++ and check it against the oracle on
// the build box (which has no GPU).  The product never runs these on the CPU: the only
// product callers are the kernels in mg_kernels.cu.
//
// Reference semantics restated (paths under /root/reference):
//   node lookup      rpc.get_begin_end_nodes   mitty/simulation/rpc.py:119-130
//   pos/cigar/v_list rpc.generate_read         mitty/simulation/rpc.py:133-160
//   qname / record   readgenerate.fastq_lines  mitty/simulation/readgenerate.py:222-230
//   N filter/revcomp read_generating_worker    mitty/simulation/readgenerate.py:198-210
//   corruption       illumina.corrupt_single_read  mitty/simulation/illumina.py:131-162
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MG_HD __host__ __device__ __forceinline__
#else
#define MG_HD inline
#endif
// MG_NI: deliberately NOT inlined.  The emit kernel is instruction-cache bound when every helper
// is inlined at every call site (13 k SASS instructions); the formatting helpers are shared.
#if defined(__CUDACC__)
#define MG_NI static __host__ __device__ __noinline__ __attribute__((unused))
#else
#define MG_NI static __attribute__((noinline, unused))
#endif
#if defined(__CUDA_ARCH__)
#define MG_UNROLL _Pragma("unroll")
#define MG_NOUNROLL _Pragma("unroll 1")
#else
#define MG_UNROLL
#define MG_NOUNROLL
#endif

// ------------------------------------------------------------------------------------------
// Data layout in HBM

// One node of a chromosome copy (rpc.Node, rpc.py:5-35) in 16 bytes -> one 128-bit load.
//   key   = ps - p_min (+1 for 'D' nodes: the searchsorted key of rpc.py:127)
//   pr    = 1-based reference position
//   op    = '=', 'X', 'I' or 'D' (ASCII)
struct alignas(16) MgNode {
  uint32_t key;
  int32_t pr;
  int32_t oplen;
  uint32_t op;
};

// Maximal run of one non-ACGT byte on the haplotype, in sample-relative coordinates -- or, with
// byte == MG_EXC_CASE, a maximal run of lower-case a/c/g/t (a soft-masked stretch): those bases keep
// their 2-bit codes in the packed sequence and the run only records the case.
#define MG_EXC_CASE 1u
struct alignas(16) MgExc {
  uint32_t start;
  uint32_t len;
  uint32_t byte;
  uint32_t pad;
};

// ------------------------------------------------------------------------------------------
// Bit tricks with portable fall-backs (the device versions map to single instructions)

MG_HD uint32_t mg_funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) {  // ((hi:lo) >> sh) low word, sh in [0,31]
#if defined(__CUDA_ARCH__)
  return __funnelshift_r(lo, hi, sh);
#else
  return sh ? ((lo >> sh) | (hi << (32 - sh))) : lo;
#endif
}

MG_HD uint32_t mg_funnel_l(uint32_t lo, uint32_t hi, uint32_t sh) {  // ((hi:lo) << sh) high word, sh in [0,31]
#if defined(__CUDA_ARCH__)
  return __funnelshift_l(lo, hi, sh);
#else
  return sh ? ((hi << sh) | (lo >> (32 - sh))) : hi;
#endif
}

MG_HD uint32_t mg_brev(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __brev(x);
#else
  x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
  x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
  x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
  x = ((x >> 8) & 0x00FF00FFu) | ((x & 0x00FF00FFu) << 8);
  return (x >> 16) | (x << 16);
#endif
}

MG_HD uint32_t mg_prmt(uint32_t a, uint32_t sel) {  // byte i of result = byte (nibble i of sel & 3) of a
#if defined(__CUDA_ARCH__)
  return __byte_perm(a, 0u, sel);
#else
  uint32_t r = 0;
  for (int i = 0; i < 4; i++) r |= ((a >> (8 * ((sel >> (4 * i)) & 3))) & 0xFFu) << (8 * i);
  return r;
#endif
}

MG_HD uint32_t mg_prmt2(uint32_t a, uint32_t b, uint32_t sel) {  // byte i of result = byte (nibble i of sel & 7) of b:a
#if defined(__CUDA_ARCH__)
  return __byte_perm(a, b, sel);
#else
  const uint64_t ab = ((uint64_t)b << 32) | a;
  uint32_t r = 0;
  for (int i = 0; i < 4; i++) r |= (uint32_t)((ab >> (8 * ((sel >> (4 * i)) & 7))) & 0xFFu) << (8 * i);
  return r;
#endif
}

// 16 consecutive 2-bit codes starting at base index s (s >= 0) of a packed sequence
// (16 bases per 32-bit word, base i in bits [2i, 2i+1] of word i/16).
template <class P>
MG_HD uint32_t mg_codes16(P seq, int64_t s) {
  int64_t w = s >> 4;
  uint32_t sh = (uint32_t)(s & 15) * 2u;
  uint32_t lo = seq[w];
  uint32_t hi = sh ? seq[w + 1] : 0u;
  return mg_funnel_r(lo, hi, sh);
}

// reverse the order of the 16 codes in a word and complement them (A<->T, C<->G is code ^ 3)
MG_HD uint32_t mg_revcomp16(uint32_t x) {
  uint32_t y = mg_brev(x);
  y = ((y >> 1) & 0x55555555u) | ((y & 0x55555555u) << 1);
  return ~y;
}

// four 2-bit codes (low byte of b) -> four ASCII bases
MG_HD uint32_t mg_chars4(uint32_t b) {
  uint32_t y = (b | (b << 4)) & 0x0F0Fu;
  uint32_t z = (y | (y << 2)) & 0x3333u;
  return mg_prmt(0x54474341u /* 'A','C','G','T' little-endian */, z);
}

MG_HD uint32_t mg_base_code(uint8_t c) {  // ACGT -> 0..3, anything else -> 4
  return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), the counter-based generator of the production mode

struct MgPhilox { uint32_t v[4]; };

MG_HD void mg_mulhilo(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo) {
  uint64_t p = (uint64_t)a * (uint64_t)b;
  hi = (uint32_t)(p >> 32); lo = (uint32_t)p;
}

template <int ROUNDS>
MG_HD MgPhilox mg_philox_r(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  MG_UNROLL
  for (int r = 0; r < ROUNDS; r++) {
    uint32_t h0, l0, h1, l1;
    mg_mulhilo(0xD2511F53u, c0, h0, l0);
    mg_mulhilo(0xCD9E8D57u, c2, h1, l1);
    uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  MgPhilox o; o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}

// Philox4x32-10: template sampling (gaps, template length, file order)
MG_HD MgPhilox mg_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  return mg_philox_r<10>(c0, c1, c2, c3, k0, k1);
}

// Philox4x32-7 (the fewest rounds Salmon et al. report as passing BigCrush): the per-base
// corruption stream, where the generator is ~60 % of the instruction count
#define MG_CORRUPT_ROUNDS 7
MG_HD MgPhilox mg_philox_corrupt(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t k0, uint32_t k1) {
  return mg_philox_r<MG_CORRUPT_ROUNDS>(c0, c1, c2, 0x636f7272u /* MG_STREAM_CORRUPT */, k0, k1);
}

// 53-bit uniform in [0,1) from two words, the same construction numpy's random_sample uses
MG_HD double mg_u53(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) / 9007199254740992.0;
}

// Philox stream tags (counter word 3)
#define MG_STREAM_GAP 0x67617073u
#define MG_STREAM_TLEN 0x746c656eu
#define MG_STREAM_CORRUPT 0x636f7272u

// Keyed pseudo-random permutation of [0, n): a Feistel network over exactly bits = ceil(log2 n) bits (the low
// bits / 2 and the high bits - bits / 2 bits take turns being the half that is XORed: with unequal halves it
// is still a bijection of [0, 2^bits)) with cycle walking -- n > 2^(bits - 1), so at least half of the domain is
// accepted and the lanes of a warp rarely walk more than twice.  Replaces RandomState.shuffle (illumina.py:71)
// in production mode.
MG_HD uint32_t mg_feistel_round(uint32_t r, uint32_t k) {
  uint32_t x = r * 0x9E3779B1u + k;
  x ^= x >> 15; x *= 0x85EBCA77u; x ^= x >> 13; x *= 0xC2B2AE3Du; x ^= x >> 16;
  return x;
}

MG_HD uint32_t mg_perm_bits(uint32_t n) {       // ceil(log2 n), at least 2
  uint32_t bits = 2;
  while (bits < 32 && (1ull << bits) < (unsigned long long)n) bits++;
  return bits;
}

MG_HD uint32_t mg_permute(uint32_t i, uint32_t n, uint32_t bits, uint32_t k0, uint32_t k1) {
  const uint32_t wa = bits >> 1, ma = (1u << wa) - 1u, mb = (bits - wa >= 32u) ? 0xFFFFFFFFu : (1u << (bits - wa)) - 1u;
  do {
    uint32_t a = i & ma, b = (i >> wa) & mb;
    MG_UNROLL
    for (int t = 0; t < 6; t += 2) {
      a ^= mg_feistel_round(b, k0 + (uint32_t)t) & ma;
      b ^= mg_feistel_round(a, k1 + (uint32_t)t + 1u) & mb;
    }
    i = (b << wa) | a;
  } while (i >= n);
  return i;
}

// ------------------------------------------------------------------------------------------
// Decimal helpers

// No branch and no table in the digit counts below: a switch, or a table indexed per lane, serialises the lanes
// of a warp that hold numbers of different lengths.
MG_HD uint32_t mg_pow10(uint32_t d) {   // 10^d for d in 0..9, selected by the bits of d
  return ((d & 1u) ? 10u : 1u) * ((d & 2u) ? 100u : 1u) * ((d & 4u) ? 10000u : 1u) * ((d & 8u) ? 100000000u : 1u);
}

MG_HD uint32_t mg_bit_length(uint32_t v) {   // bits of v, v != 0
#if defined(__CUDA_ARCH__)
  return 32u - (uint32_t)__clz((int)v);
#else
  return 32u - (uint32_t)__builtin_clz(v);
#endif
}

// decimal digits of v, and (ones) the number 11..1 with as many ones.  With b = bits of v, t = floor(b log10 2)
// (1233 / 4096 is log10 2 rounded down, exact enough for b <= 32) and v has t or t + 1 digits: t + 1 when
// v >= 10^t.  v | 1 has the digits of v (a power of ten above 1 is even) and makes 0 one digit.
MG_HD int mg_ndigits_ones(uint32_t v, uint32_t &ones) {
  const uint32_t w = v | 1u;
  const uint32_t t = (mg_bit_length(w) * 1233u) >> 12;
  const uint32_t p = mg_pow10(t);
  const bool up = w >= p;
  ones = (p - 1u) / 9u + (up ? p : 0u);                     // 11..1 with t ones, plus 10^t for one digit more
  return (int)(t + (up ? 1u : 0u));
}

MG_HD int mg_ndigits32(uint32_t v) { uint32_t o; return mg_ndigits_ones(v, o); }

MG_HD int mg_ndigits(uint64_t v) {
  if (v <= 0xFFFFFFFFull) return mg_ndigits32((uint32_t)v);
  int d = 1;
  while (v >= 10) { v /= 10; d++; }
  return d;
}


// sum of the decimal lengths of 1..m  (closed form; used to place records whose qname carries a
// serial number that is only known after the block/grid scan):  d*(m+1) - 11..1 (d ones)
MG_HD uint64_t mg_digit_sum(uint64_t m) {
  if (m == 0) return 0;
  if (m <= 0xFFFFFFFFull) {
    uint32_t ones;
    const int d = mg_ndigits_ones((uint32_t)m, ones);
    return (uint64_t)d * (m + 1) - (uint64_t)ones;
  }
  const int d = mg_ndigits(m);
  uint64_t ones = 0, p = 1;
  for (int k = 0; k < d; k++) { ones += p; p *= 10; }
  return (uint64_t)d * (m + 1) - ones;
}

// ------------------------------------------------------------------------------------------
// Writers.  CountWriter sizes a record; MgStream writes it at any byte alignment with aligned
// 32-bit stores: whole words (sequence, qualities) cost one funnel shift + one store, tokens of
// 0..8 bytes (the qname's numbers and separators) are appended without a branch.

struct MgCountWriter {
  static constexpr bool is_bytes = false;
  uint32_t n;
  MG_HD void put(uint8_t) { n++; }
  MG_HD void put_word(uint32_t) { n += 4; }
};

// Address-space policies.  The emit kernel formats records into its warp's shared-memory stage:
// MgSharedSpace addresses it with 32-bit offsets into the kernel's dynamic shared memory, so every
// store is a plain STS (generic 64-bit pointers cost 3-4 instructions per store).  MgGenericSpace
// is any memory: host emulation, and the rare record that is larger than the stage.
struct MgGenericSpace {
  static constexpr bool is_generic = true;
  typedef uint8_t *ptr;
  static MG_HD void st8(ptr p, uint8_t v) { *p = v; }
  static MG_HD void st32(ptr p, uint32_t v) { *reinterpret_cast<uint32_t *>(p) = v; }
  static MG_HD uint32_t ld32(ptr p) { return *reinterpret_cast<const uint32_t *>(p); }
  static MG_HD uint32_t ld8(ptr p) { return *p; }
  static MG_HD uint32_t low2(ptr p) { return (uint32_t)((uintptr_t)p & 3); }
};
#if defined(__CUDACC__)
struct MgSharedSpace {
  static constexpr bool is_generic = false;
  // a byte address in the shared window (cvta.to.shared of the kernel's stage): plain 32-bit
  // st.shared / ld.shared with no generic-address arithmetic at the use sites
  typedef uint32_t ptr;
  static __device__ __forceinline__ void st8(ptr p, uint8_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(p), "r"((uint32_t)v)); }
  static __device__ __forceinline__ void st32(ptr p, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(p), "r"(v)); }
  static __device__ __forceinline__ uint32_t ld32(ptr p) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(p));
    return v;
  }
  static __device__ __forceinline__ uint32_t ld8(ptr p) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(p));
    return v;
  }
  static __device__ __forceinline__ uint32_t low2(ptr p) { return p & 3u; }
};
#endif

template <class SP> MG_HD void mg_store_tail(typename SP::ptr b, uint32_t carry, uint32_t nb) {   // nb <= 3: three predicated stores
  if (nb > 0) SP::st8(b, (uint8_t)carry);
  if (nb > 1) SP::st8(b + 1, (uint8_t)(carry >> 8));
  if (nb > 2) SP::st8(b + 2, (uint8_t)(carry >> 16));
}

// A token: n <= 8 bytes, first byte in the lowest byte of lo; the bytes beyond n are zero.
struct MgTok { uint32_t lo, hi, n; };

template <class SP>
struct MgStream {
  static constexpr bool is_bytes = false;
  typename SP::ptr wp;   // next aligned word
  uint32_t prev;         // the pending bytes are the TOP sh / 8 bytes of prev
  uint32_t sh;           // 8 * pending byte count: 0, 8, 16 or 24
  uint32_t skip;         // generic space only: low bytes of the first word that belong to the previous record

  // Start of a record.  The bytes before dst inside its word are the tail of the PREVIOUS record
  // (another thread's).  In the shared-memory stage the first word is stored whole and the previous
  // record's tail bytes are written afterwards (every stream ends with byte stores, and the kernel
  // puts a __syncwarp between the two); anywhere else the first word is written byte by byte.
  MG_HD void begin(typename SP::ptr dst) {
    const uint32_t a = SP::low2(dst);
    wp = dst - a; sh = 8 * a; prev = 0u; skip = a;
  }
  // The bytes before dst inside its word were written earlier BY THIS THREAD (the tail of its own
  // qname / separator): they are read back and carried, so every flush is a plain word store.
  MG_HD void begin_rmw(typename SP::ptr dst) {
    const uint32_t a = SP::low2(dst);
    wp = dst - a; sh = 8 * a; skip = 0;
    prev = a ? (SP::ld32(wp) << (32 - sh)) : 0u;
  }
  MG_HD void flush_word(uint32_t w) {
    if constexpr (SP::is_generic) {
      if (skip) { for (uint32_t i = skip; i < 4; i++) SP::st8(wp + i, (uint8_t)(w >> (8 * i))); skip = 0; wp += 4; return; }
    }
    SP::st32(wp, w); wp += 4;
  }
  MG_HD void put(uint8_t c) {
    prev = (prev >> 8) | ((uint32_t)c << 24);
    sh += 8;
    if (sh == 32) { flush_word(prev); sh = 0; }
  }
  MG_HD void put_word(uint32_t w) {  // four bytes, little-endian order: one funnel shift, one store
    flush_word(mg_funnel_l(prev, w, sh));    // (w << sh) | (prev >> (32 - sh)); sh == 0 gives w
    prev = w;
  }
  // 0..8 bytes without a branch: the (at most two) completed words are stored under predicates
  MG_HD void append(MgTok t) {
    const uint32_t pend = mg_funnel_l(prev, 0u, sh);            // pending bytes in the low positions (sh == 0: none)
    const uint32_t w0 = pend | (t.lo << sh);
    const uint32_t w1 = mg_funnel_l(t.lo, t.hi, sh);
    const uint32_t w2 = mg_funnel_l(t.hi, 0u, sh);
    const uint32_t tb = sh + 8u * t.n;                          // total pending bits, < 96
    if constexpr (SP::is_generic) {
      if (tb >= 32u) flush_word(w0);
      if (tb >= 64u) flush_word(w1);
    } else {
      if (tb >= 32u) SP::st32(wp, w0);
      if (tb >= 64u) SP::st32(wp + 4, w1);
      wp += (tb >> 3) & ~3u;
    }
    const uint32_t keep = tb >= 64u ? w2 : (tb >= 32u ? w1 : w0);
    sh = tb & 31u;
    prev = keep << ((32u - sh) & 31u);                          // back to the top of prev (sh == 0: nothing is pending)
  }
  // the last partial word is shared with the NEXT record (another thread): byte stores
  MG_HD void end() {
    if (sh) {
      const uint32_t nb = sh >> 3, carry = prev >> (32 - sh);
      if constexpr (SP::is_generic) { const uint32_t k = skip; skip = 0; for (uint32_t i = k; i < nb; i++) SP::st8(wp + i, (uint8_t)(carry >> (8 * i))); }
      else mg_store_tail<SP>(wp, carry, nb);
    }
    sh = 0;
  }
  // pending bytes stored as one word whose upper bytes are zero: only where those upper bytes are the
  // writer's own, still unwritten, territory (the sequence line after the qname)
  MG_HD void flush_own() { if (sh) flush_word(prev >> (32 - sh)); sh = 0; }
};

// ---- decimal text without loops or branches -------------------------------------------------------

MG_HD uint32_t mg_dec4(uint32_t x) {   // x < 10000 -> its 4 digits as ASCII, first digit in the lowest byte
  const uint32_t c = (x * 5243u) >> 19;                     // x / 100
  const uint32_t d = x - c * 100u;
  const uint32_t p = c | (d << 16);                         // two values < 100 in the two halves
  const uint32_t t = ((p * 103u) >> 10) & 0x000F000Fu;      // their tens
  const uint32_t o = p - t * 10u;                           // their ones
  return (t | (o << 8)) + 0x30303030u;
}

// pre (npre <= 3 bytes) followed by the decimal digits of v: two tokens, A = pre + the digits above
// 10^8 (at most 2), B = the other (at most 8) digits
MG_HD void mg_tok_num(uint32_t v, uint32_t pre, uint32_t npre, MgTok &A, MgTok &B) {
  const uint32_t top = v / 100000000u, low = v - top * 100000000u;
  const uint32_t a = low / 10000u, b = low - a * 10000u;
  uint32_t lo = mg_dec4(a), hi = mg_dec4(b);
  // leading zeros of the 8-digit text (bytes equal to '0' before the first other byte)
  const uint32_t xl = lo ^ 0x30303030u, xh = hi ^ 0x30303030u;
  uint32_t lz;
#if defined(__CUDA_ARCH__)
  lz = xl ? ((uint32_t)__ffs((int)xl) - 1u) >> 3 : (xh ? 4u + (((uint32_t)__ffs((int)xh) - 1u) >> 3) : 7u);
#else
  lz = xl ? ((uint32_t)__builtin_ctz(xl)) >> 3 : (xh ? 4u + (((uint32_t)__builtin_ctz(xh)) >> 3) : 7u);
#endif
  if (top) lz = 0u;                                          // the high part is printed: keep all eight
  // drop lz bytes from the front of (lo, hi)
  const bool big = lz >= 4u;
  const uint32_t l1 = big ? hi : lo, h1 = big ? 0u : hi, s2 = 8u * (lz & 3u);
  B.lo = mg_funnel_r(l1, h1, s2); B.hi = h1 >> s2; B.n = 8u - lz;
  // the high part: 0, 1 or 2 digits after the prefix
  const uint32_t tt = (top * 103u) >> 10, to = top - tt * 10u;
  const uint32_t nt = top >= 10u ? 2u : (top ? 1u : 0u);
  const uint32_t dig = top >= 10u ? ((tt + 48u) | ((to + 48u) << 8)) : (top ? to + 48u : 0u);
  // pre occupies npre <= 3 bytes, dig up to 2: five bytes over (lo, hi)
  const uint32_t ps = 8u * npre;
  A.lo = pre | (dig << ps); A.hi = mg_funnel_l(dig, 0u, ps); A.n = npre + nt;
}

template <class SP>
MG_HD void mg_put_num(MgStream<SP> &w, uint32_t v, uint32_t pre, uint32_t npre) {
  MgTok A, B;
  mg_tok_num(v, pre, npre, A, B);
  w.append(A); w.append(B);
}

// the same for the numbers that are almost always small (CIGAR lengths, variant sizes): below 10^4
// it is one token -- pre (<= 3 bytes) + at most four digits
template <class SP>
MG_HD void mg_put_small(MgStream<SP> &w, uint32_t v, uint32_t pre, uint32_t npre) {
  if (v >= 10000u) { mg_put_num(w, v, pre, npre); return; }
  const uint32_t d = mg_dec4(v), x = d ^ 0x30303030u;
  uint32_t lz;                                               // leading '0' bytes, at most 3 (v == 0 prints "0")
#if defined(__CUDA_ARCH__)
  lz = (x & 0x00FFFFFFu) ? ((uint32_t)__ffs((int)x) - 1u) >> 3 : 3u;
#else
  lz = (x & 0x00FFFFFFu) ? ((uint32_t)__builtin_ctz(x)) >> 3 : 3u;
#endif
  const uint32_t dig = d >> (8u * lz), ps = 8u * npre;
  MgTok t;
  t.lo = pre | (dig << ps); t.hi = mg_funnel_l(dig, 0u, ps); t.n = npre + 4u - lz;
  w.append(t);
}

MG_HD MgTok mg_tok(uint32_t lo, uint32_t hi, uint32_t n) { MgTok t; t.lo = lo; t.hi = hi; t.n = n; return t; }

// decimal digits through a byte-at-a-time writer (the sizing cross-check of the emulation tests)
template <class W>
MG_HD void mg_put_u32(W &w, uint32_t v) {
  uint64_t acc = 0;
  int n = 0;
  do { uint32_t q = v / 10u; acc = (acc << 4) | (v - q * 10u); v = q; n++; } while (v);
  for (; n; n--) { w.put((uint8_t)('0' + ((uint32_t)acc & 15u))); acc >>= 4; }
}

// ------------------------------------------------------------------------------------------
// Node lookup: searchsorted(keys, x, 'right') - 1 (rpc.py:127-130), accelerated by a block table
// blk[b] = last node whose key <= (b << blk_shift).

template <class NP, class BP>
MG_NI int mg_find_node(NP nodes, BP blk, int blk_shift, int n_blk, int n_nodes, uint32_t x) {
  uint32_t b = x >> blk_shift;
  if ((int)b >= n_blk) b = (uint32_t)(n_blk - 1);
  int lo = (int)blk[b];
  int hi = ((int)b + 1 < n_blk) ? (int)blk[b + 1] : n_nodes - 1;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (nodes[mid].key <= x) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Per-read geometry shared by the sizing pass and the formatting pass.
//   pos (rpc.py:148-158), whether the read lies inside one insertion (rpc.py:149-154) and the
//   last node n1 = searchsorted(keys, x+L-1, 'right') - 1, found by walking forward from n0.
template <class NP>
MG_HD int mg_last_node(NP nodes, int n0, int n_nodes, uint32_t x, int L) {
  const uint32_t last = x + (uint32_t)L - 1u;
  int n1 = n0;
  while (n1 + 1 < n_nodes && nodes[n1 + 1].key <= last) n1++;
  return n1;
}

MG_HD int32_t mg_read_pos(const MgNode &f, bool single, uint32_t x) {
  if (f.op == 'I') return single ? f.pr - 1 : f.pr;                         // rpc.py:148-156
  const int64_t ps0 = (int64_t)f.key - (f.op == 'D' ? 1 : 0);
  return (int32_t)((int64_t)x - ps0 + (int64_t)f.pr);                        // rpc.py:158
}

MG_HD int32_t mg_cigar_len(const MgNode &n, uint32_t x, int L) {             // rpc.py:145
  if (n.op == 'D') return n.oplen;
  int64_t a = (int64_t)x - (int64_t)n.key; if (a < 0) a = 0;
  int64_t b = (int64_t)x + L - (int64_t)n.key; if ((int64_t)n.oplen < b) b = n.oplen;
  return (int32_t)(b - a);
}

template <class W>
MG_HD void mg_put_i32(W &w, int32_t v) {
  if (v < 0) { w.put('-'); mg_put_u32(w, (uint32_t)(-(int64_t)v)); } else mg_put_u32(w, (uint32_t)v);
}

MG_HD int mg_nchars_i32(int32_t v) {   // one digit count for either sign
  const bool neg = v < 0;
  return (neg ? 1 : 0) + mg_ndigits32(neg ? (uint32_t)(-(int64_t)v) : (uint32_t)v);
}

// length of '|strand|pos|rlen|cigar|vlist' for one read; L_nd = decimal digits of L
template <class NP>
MG_NI uint32_t mg_read_fields_len(NP nodes, int n0, int n1, uint32_t x, int L, int L_nd) {
  const MgNode f = nodes[n0];
  const bool single = (n0 == n1);
  uint32_t n = 2u + 1u + (uint32_t)mg_nchars_i32(mg_read_pos(f, single, x)) + 1u + (uint32_t)L_nd + 1u + 1u;
  if (single && f.op == '=') return n + (uint32_t)L_nd + 1u;                 // "<L>=" and an empty v_list
  if (single && f.op == 'I')                                                 // ">p:<L>I" and "<oplen>"
    return n + 1u + (uint32_t)mg_nchars_i32((int32_t)((int64_t)x - (int64_t)f.key)) + 1u + (uint32_t)L_nd + 1u + (uint32_t)mg_nchars_i32(f.oplen);
  uint32_t nv = 0;
  for (int k = n0; k <= n1; k++) {
    const MgNode nd = nodes[k];
    n += (uint32_t)mg_nchars_i32(mg_cigar_len(nd, x, L)) + 1u;
    if (nd.op != '=') {
      n += (nv ? 1u : 0u) + (nd.op == 'X' ? 1u : nd.op == 'I' ? (uint32_t)mg_nchars_i32(nd.oplen) : (uint32_t)mg_nchars_i32(-nd.oplen));
      nv++;
    }
  }
  return n;
}

// '|strand|pos|rlen|cigar|vlist' for one read (fastq_lines, readgenerate.py:224-225, over
// generate_read, rpc.py:144-158).  x = read start relative to p_min, L = read length.
template <class W, class NP>
MG_HD void mg_fmt_read(W &w, NP nodes, int n0, int n1, uint32_t x, int L, int strand) {
  const MgNode f = nodes[n0];
  const bool single = (n0 == n1);
  w.put('|'); w.put((uint8_t)('0' + strand));
  w.put('|'); mg_put_i32(w, mg_read_pos(f, single, x));
  w.put('|'); mg_put_u32(w, (uint32_t)L);
  w.put('|');
  if (single && f.op == '=') {                                               // the common case: "<L>=" + empty v_list
    mg_put_u32(w, (uint32_t)L); w.put('='); w.put('|');
    return;
  }
  if (single && f.op == 'I') {                                               // rpc.py:154
    w.put('>'); mg_put_i32(w, (int32_t)((int64_t)x - (int64_t)f.key)); w.put(':'); mg_put_u32(w, (uint32_t)L); w.put('I');
  } else {
    for (int k = n0; k <= n1; k++) {                                         // rpc.py:145
      const MgNode n = nodes[k];
      mg_put_i32(w, mg_cigar_len(n, x, L)); w.put((uint8_t)n.op);
    }
  }
  w.put('|');
  bool first = true;
  for (int k = n0; k <= n1; k++) {                                           // rpc.py:144
    const MgNode n = nodes[k];
    if (n.op == '=') continue;
    if (!first) w.put(',');
    first = false;
    if (n.op == 'X') w.put('0');
    else mg_put_i32(w, n.op == 'I' ? n.oplen : -n.oplen);
  }
}

// Whole qname line:
//   '@' stub ':' cnt '|' chrom '|' cpy  + per read in FILE order '|strand|pos|rlen|cigar|vlist'
// prefix = "@<sample>:<worker>:<ps>:"   mid = "|<chrom>|<cpy>"
struct MgReadRef { uint32_t x; int n0, n1, strand; };

// byte-at-a-time restatement (sizing cross-check of the emulation tests; never on a kernel's path)
template <class W, class NP>
MG_HD void mg_fmt_qname(W &w, const uint8_t *prefix, int prefix_len, uint64_t cnt, bool with_cnt,
                        const uint8_t *mid, int mid_len, NP nodes, MgReadRef first, MgReadRef second, int L) {
  for (int i = 0; i < prefix_len; i++) w.put(prefix[i]);
  if (with_cnt) mg_put_u32(w, (uint32_t)cnt);
  for (int i = 0; i < mid_len; i++) w.put(mid[i]);
  MG_NOUNROLL
  for (int r = 0; r < 2; r++) {
    const MgReadRef R = r ? second : first;
    mg_fmt_read(w, nodes, R.n0, R.n1, R.x, L, R.strand);
  }
}

// Per-CTA constants of the qname: the strings every record repeats, ready as tokens (the emit
// kernel keeps one copy in shared memory).
//   pre[]      = "@<sample>:<worker>:<ps>:"   mid[] = "|<chrom>|<cpy>"     (eight bytes per token)
//   tail[0..1] = "|<L>|<L>=|"  (what follows POS when the read lies inside one '=' node: rlen, CIGAR, empty v_list)
//   rl         = "|<L>|"       (what follows POS otherwise)
#define MG_QN_TOKS 24            // 8 * 24 = MG_QN_MAX bytes
struct MgQnConst {
  MgTok pre[MG_QN_TOKS], mid[MG_QN_TOKS];
  int n_pre, n_mid;
  MgTok tail[2], rl;
  uint32_t Lnd;   // number of digits of L, or 0: "L is absurdly long, write it digit by digit"
};

MG_HD MgTok mg_tok_bytes(const uint8_t *t, int from, int cnt) {
  MgTok k; k.lo = 0; k.hi = 0; k.n = (uint32_t)(cnt < 0 ? 0 : (cnt > 8 ? 8 : cnt));
  for (uint32_t i = 0; i < k.n; i++) { if (i < 4) k.lo |= (uint32_t)t[from + i] << (8 * i); else k.hi |= (uint32_t)t[from + i] << (8 * (i - 4)); }
  return k;
}

MG_HD void mg_qn_const(MgQnConst &Q, const uint8_t *prefix, int prefix_len, const uint8_t *mid, int mid_len, int L) {
  Q.n_pre = (prefix_len + 7) / 8; Q.n_mid = (mid_len + 7) / 8;
  for (int i = 0; i < Q.n_pre; i++) Q.pre[i] = mg_tok_bytes(prefix, 8 * i, prefix_len - 8 * i);
  for (int i = 0; i < Q.n_mid; i++) Q.mid[i] = mg_tok_bytes(mid, 8 * i, mid_len - 8 * i);
  // "|<L>|<L>=|", bytewise: once per CTA, not per record
  uint8_t d[12], t[28]; int nd = 0, n = 0;
  uint32_t v = (uint32_t)L;
  do { d[nd++] = (uint8_t)('0' + v % 10u); v /= 10u; } while (v);
  t[n++] = '|';
  for (int i = nd - 1; i >= 0; i--) t[n++] = d[i];
  t[n++] = '|';
  const int nrl = n;
  for (int i = nd - 1; i >= 0; i--) t[n++] = d[i];
  t[n++] = '='; t[n++] = '|';
  const bool ok = n <= 16;                           // up to 6 digits
  Q.Lnd = ok ? (uint32_t)nd : 0u;
  Q.rl = mg_tok_bytes(t, 0, ok ? nrl : 0);
  Q.tail[0] = mg_tok_bytes(t, 0, ok ? n : 0);
  Q.tail[1] = mg_tok_bytes(t, 8, ok ? n - 8 : 0);
}

// '|strand|pos|rlen|cigar|vlist' of one read into the stream (fastq_lines, readgenerate.py:224-225,
// over generate_read, rpc.py:144-158).  x = read start relative to p_min.
template <class SP, class NP>
MG_HD void mg_put_read(MgStream<SP> &w, const MgQnConst &Q, NP nodes, MgReadRef R, int L) {
  const MgNode f = nodes[R.n0];
  const bool single = (R.n0 == R.n1);
  mg_put_num(w, (uint32_t)mg_read_pos(f, single, R.x), (uint32_t)'|' | ((uint32_t)('0' + R.strand) << 8) | ((uint32_t)'|' << 16), 3u);
  if (single && f.op == '=' && Q.Lnd) {                                       // the common case: "<L>=" + empty v_list
    w.append(Q.tail[0]); w.append(Q.tail[1]);
    return;
  }
  if (Q.Lnd) w.append(Q.rl); else mg_put_num(w, (uint32_t)L, '|', 1u), w.append(mg_tok('|', 0, 1));
  if (single && f.op == '=') {                                               // (absurd L only)
    mg_put_num(w, (uint32_t)L, 0u, 0u); w.append(mg_tok((uint32_t)'=' | ((uint32_t)'|' << 8), 0, 2));
    return;
  }
  if (single && f.op == 'I') {                                               // rpc.py:154  ">p:<L>I" and "|<oplen>"
    mg_put_small(w, (uint32_t)((int64_t)R.x - (int64_t)f.key), '>', 1u);
    mg_put_small(w, (uint32_t)L, ':', 1u);
    mg_put_small(w, (uint32_t)f.oplen, (uint32_t)'I' | ((uint32_t)'|' << 8), 2u);
    return;
  }
  // the read spans several nodes (or sits on one that is not '='): the first three are fetched at once
  // -- one memory latency instead of one per step of the two walks below
  const int k1 = R.n0 + 1 <= R.n1 ? R.n0 + 1 : R.n1, k2 = R.n0 + 2 <= R.n1 ? R.n0 + 2 : R.n1;
  const MgNode c1 = nodes[k1], c2 = nodes[k2];
  auto node_at = [&](int k) -> MgNode { const int d = k - R.n0; if (d == 0) return f; if (d == 1) return c1; if (d == 2) return c2; return nodes[k]; };
  uint32_t pre = 0, npre = 0;
  for (int k = R.n0; k <= R.n1; k++) {                                       // rpc.py:145: <len><op> per node
    const MgNode n = node_at(k);
    mg_put_small(w, (uint32_t)mg_cigar_len(n, R.x, L), pre, npre);
    pre = n.op; npre = 1;
  }
  pre |= (uint32_t)'|' << 8; npre = 2;                                       // last op, then the field separator
  bool firstv = true;
  for (int k = R.n0; k <= R.n1; k++) {                                       // rpc.py:144: v_list
    const MgNode n = node_at(k);
    if (n.op == '=') continue;
    if (!firstv) { pre = ','; npre = 1; }
    firstv = false;
    if (n.op == 'D') { pre |= (uint32_t)'-' << (8 * npre); npre++; }
    mg_put_small(w, n.op == 'X' ? 0u : (uint32_t)n.oplen, pre, npre);
    npre = 0; pre = 0;
  }
  if (npre) w.append(mg_tok(pre, 0, npre));                                  // no variant at all (cannot happen here: the read spans > 1 node)
}

// qname line + '\n' through the stream (which then goes on with the sequence line)
// STR: where the two per-unit strings come from -- the kernel's own MgQnConst, or the unit's entry of a batch table
// (any type with pre[], n_pre, mid[], n_mid)
template <class SP, class NP, class STR>
MG_HD void mg_put_qname(MgStream<SP> &w, const MgQnConst &Q, const STR &str, uint32_t cnt, NP nodes, MgReadRef first, MgReadRef second, int L) {
  for (int i = 0; i < str.n_pre; i++) w.append(str.pre[i]);
  mg_put_num(w, cnt, 0u, 0u);
  for (int i = 0; i < str.n_mid; i++) w.append(str.mid[i]);
  MG_NOUNROLL
  for (int r = 0; r < 2; r++) mg_put_read(w, Q, nodes, r ? second : first, L);
  w.append(mg_tok('\n', 0, 1));
}

// Register window over a read: the 2-bit words covering it are fetched up front (independent
// loads, all in flight at once) and, for the reverse strand, reversed and complemented word by
// word in descending order, so that BOTH strands become a forward extraction
//   codes(c) = funnel(w[c], w[c+1], 2 * off)
// with compile-time word indices.  MAXW - 1 >= ceil((15 + L) / 16).
template <int MAXW>
struct MgWin { uint32_t w[MAXW]; uint32_t off; };

template <int MAXW, class HP>
MG_HD void mg_win_load(MgWin<MAXW> &W, HP hap, uint32_t x, int L, int strand) {
  const uint32_t last = x + (uint32_t)L - 1u;
  const int64_t w_first = (int64_t)(x >> 4), w_last = (int64_t)(last >> 4);
  W.off = strand ? 15u - (last & 15u) : (x & 15u);
  const int nw = (int)((W.off + (uint32_t)L + 15u) >> 4);
  MG_UNROLL
  for (int i = 0; i < MAXW; i++) {
    uint32_t v = 0;
    if (i < nw) v = hap[strand ? w_last - i : w_first + i];
    W.w[i] = v;                 // raw: the reverse strand is turned around by mg_win_prep, when the words are first USED
  }
}

template <int MAXW>
MG_HD void mg_win_prep(MgWin<MAXW> &W, int strand) {
  if (strand) {
    MG_UNROLL
    for (int i = 0; i < MAXW; i++) W.w[i] = mg_revcomp16(W.w[i]);
  }
}

template <int MAXW>
MG_HD uint32_t mg_win_codes(const MgWin<MAXW> &W, int c) {  // c must be a compile-time constant after unrolling
  return mg_funnel_r(W.w[c], W.w[c + 1], 2u * W.off);
}

// The emission loops run over chunk PAIRS with a rolled loop (a fully unrolled read is ~1000
// instructions per site and thrashes the instruction cache): chunks (w[0],w[1]) and (w[1],w[2]) are
// consumed, then the window slides down by two registers.
template <int MAXW>
MG_HD void mg_win_slide2(MgWin<MAXW> &W) {
  MG_UNROLL
  for (int i = 0; i < MAXW; i++) W.w[i] = (i + 2 < MAXW) ? W.w[i + 2] : 0u;
}

template <class W>
MG_HD void mg_emit_fill(W &w, uint8_t c, int n) {
  uint32_t cw = 0x01010101u * c;
  int k = 0;
  for (; k + 4 <= n; k += 4) w.put_word(cw);
  for (; k < n; k++) w.put(c);
}

// Exception runs (non-ACGT bytes) overlapping [x, x+L): first run with start+len > x.
template <class EP>
MG_HD int mg_exc_first(EP exc, int n_exc, uint32_t x) {
  int lo = 0, hi = n_exc;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if ((uint64_t)exc[mid].start + exc[mid].len <= (uint64_t)x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Exception runs with a block table over them: eblk[b] = the first run that ends beyond haplotype position
// b << shift (n_blk + 1 entries).  The first run that can touch a read starting at x then lies in
// [eblk[x >> shift], eblk[(x >> shift) + 1]] -- two adjacent table entries instead of a binary search over every
// run of the chromosome (39 N runs on chr1: six dependent loads per read, a tenth of k_unit_plan's instructions;
// ~10^6 case runs on a soft-masked one: twenty).  blk == nullptr: plain binary search.
struct MgExcView {
  const MgExc *p; const uint32_t *blk; int shift, n_blk;
  MG_HD const MgExc &operator[](int k) const { return p[k]; }
};

MG_HD int mg_exc_first(MgExcView exc, int n_exc, uint32_t x) {
  int lo = 0, hi = n_exc;
  if (exc.blk) {
    uint32_t b = x >> exc.shift;
    if ((int)b > exc.n_blk - 1) b = (uint32_t)(exc.n_blk - 1);
    lo = (int)exc.blk[b]; hi = (int)exc.blk[b + 1];
    if (hi > n_exc) hi = n_exc;
    if (lo > hi) lo = hi;
  }
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if ((uint64_t)exc.p[mid].start + exc.p[mid].len <= (uint64_t)x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// number of 'N' in the read (seq.count('N'), readgenerate.py:204); touch = the read overlaps an
// exception run of any kind (its bases need patching after the word-stream emission)
template <class EP>
MG_NI int mg_count_N(EP exc, int n_exc, uint32_t x, int L, bool &touch) {
  int cnt = 0;
  touch = false;
  for (int k = mg_exc_first(exc, n_exc, x); k < n_exc; k++) {
    MgExc e = exc[k];
    if ((uint64_t)e.start >= (uint64_t)x + L) break;
    touch = true;
    if (e.byte != 'N') continue;
    uint64_t a = e.start > x ? e.start : x;
    uint64_t b = (uint64_t)e.start + e.len < (uint64_t)x + L ? (uint64_t)e.start + e.len : (uint64_t)x + L;
    cnt += (int)(b - a);
  }
  return cnt;
}

// overwrite the bases of a written read (seq points at its first byte) that fall in exception
// runs.  The reference's translate table only maps ATCGN (readgenerate.py:56), so an exception
// byte -- lower-case bases included -- is copied unchanged on either strand; only its position is
// mirrored on strand 1.
// the forward-strand byte of haplotype position i under exception run e: the run's byte, or the
// lower-case letter of the packed code for a case run
template <class HP>
MG_HD uint8_t mg_exc_byte(const MgExc &e, HP hap, uint64_t i) {
  if (e.byte != MG_EXC_CASE) return (uint8_t)e.byte;
  return (uint8_t)("acgt"[(hap[i >> 4] >> (2 * (i & 15))) & 3u]);
}

// the 2-bit codes of consecutive haplotype positions: one load per 16 bases
template <class HP>
struct MgCodeCursor {
  HP hap; uint64_t wi; uint32_t wv;
  MG_HD explicit MgCodeCursor(HP h) : hap(h), wi(~0ull), wv(0u) {}
  MG_HD uint32_t at(uint64_t i) {
    if ((i >> 4) != wi) { wi = i >> 4; wv = hap[wi]; }
    return (wv >> (2u * ((uint32_t)i & 15u))) & 3u;
  }
};

// ---- soft-masked stretches, four bases per step ------------------------------------------------------
// The case runs a read touches as a bit mask in OUTPUT order, 192 bits in six registers: bit a + n is set
// when output base n (n = L - 1 - idx on strand 1) is lower case, a = the byte phase of the sequence line in
// its first aligned word.  The patch loops below then walk the line's aligned words, four mask bits at a
// time (the whole mask shifts down by four per word).  The words at both ends also hold the '\n' before /
// after the line -- bytes of the same record, written by the same thread -- so the read-modify-write of
// whole words touches nobody else's bytes.
#define MG_CASE_WORDS 6
struct MgCaseMask {
  uint32_t m[MG_CASE_WORDS];
  MG_HD void clear() { MG_UNROLL for (int w = 0; w < MG_CASE_WORDS; w++) m[w] = 0u; }
  MG_HD void set(uint32_t lo, uint32_t hi) {            // bits [lo, hi), hi <= 32 * MG_CASE_WORDS
    MG_UNROLL
    for (int w = 0; w < MG_CASE_WORDS; w++) {
      const uint32_t l = lo > 32u * w ? lo - 32u * w : 0u, h = hi < 32u * w + 32u ? (hi > 32u * w ? hi - 32u * w : 0u) : 32u;
      if (l < h) m[w] |= (h - l == 32u ? 0xFFFFFFFFu : ((1u << (h - l)) - 1u) << l);
    }
  }
  MG_HD uint32_t next4() {                              // the low four bits; the mask moves down by four
    const uint32_t b = m[0] & 15u;
    MG_UNROLL
    for (int w = 0; w + 1 < MG_CASE_WORDS; w++) m[w] = mg_funnel_r(m[w], m[w + 1], 4u);
    m[MG_CASE_WORDS - 1] >>= 4;
    return b;
  }
  MG_HD bool any() const { uint32_t o = 0; MG_UNROLL for (int w = 0; w < MG_CASE_WORDS; w++) o |= m[w]; return o != 0u; }
};

MG_HD uint32_t mg_bits4_to_bytes(uint32_t b) { return ((b * 0x00204081u) & 0x01010101u) * 0xFFu; }   // bit j -> byte j = 0xFF
// four upper-case letters A/C/G/T -> their complements (A ^ T = 0x15, C ^ G = 0x04; bit 1 tells the pairs apart)
MG_HD uint32_t mg_complement4(uint32_t w) { return w ^ (0x15151515u ^ (((w >> 1) & 0x01010101u) * 0x11u)); }

// perfect reads: the line holds upper-case letters, complemented on strand 1.  A lower-case base is copied
// as it is on either strand (the reference's translate table only maps ATCGN, readgenerate.py:56).
template <class SP>
MG_HD void mg_patch_case_words(typename SP::ptr seq, MgCaseMask &M, int L, int strand) {
  const uint32_t a = SP::low2(seq);
  typename SP::ptr wp = seq - a;
  const int nw = (int)((a + (uint32_t)L + 3u) >> 2);
  MG_NOUNROLL
  for (int k = 0; k < nw; k++, wp += 4) {
    const uint32_t bits = M.next4();
    if (!bits) continue;
    const uint32_t bm = mg_bits4_to_bytes(bits);
    uint32_t w = SP::ld32(wp);
    const uint32_t u = strand ? mg_complement4(w) : w;
    w = (w & ~bm) | ((u | 0x20202020u) & bm);
    SP::st32(wp, w);
  }
}

template <class SP, class EP, class HP>
MG_NI void mg_patch_exc(typename SP::ptr seq, EP exc, int n_exc, HP hap, uint32_t x, int L, int strand) {
  MgCodeCursor<HP> cur(hap);
  const uint32_t ph = SP::low2(seq);
  const bool words = ph + (uint32_t)L <= 32u * MG_CASE_WORDS;      // the mask registers cover the line
  MgCaseMask M; M.clear();
  for (int k = mg_exc_first(exc, n_exc, x); k < n_exc; k++) {
    MgExc e = exc[k];
    if ((uint64_t)e.start >= (uint64_t)x + L) break;
    uint64_t a = e.start > x ? e.start : x;
    uint64_t b = (uint64_t)e.start + e.len < (uint64_t)x + L ? (uint64_t)e.start + e.len : (uint64_t)x + L;
    const bool soft = e.byte == MG_EXC_CASE;
    if (soft && words) {
      const uint32_t i0 = (uint32_t)(a - x), i1 = (uint32_t)(b - x);
      if (strand) M.set(ph + (uint32_t)L - i1, ph + (uint32_t)L - i0); else M.set(ph + i0, ph + i1);
      continue;
    }
    for (uint64_t i = a; i < b; i++) {
      int idx = (int)(i - x);
      const uint32_t out = soft ? (0x74676361u /* "acgt" */ >> (8u * cur.at(i))) & 0xFFu : (uint32_t)e.byte;
      SP::st8(seq + (uint32_t)(strand ? (L - 1 - idx) : idx), (uint8_t)out);
    }
  }
  if (M.any()) mg_patch_case_words<SP>(seq, M, L, strand);
}

// ------------------------------------------------------------------------------------------
// Corruption of one base call (illumina.py:155-160)

MG_HD uint8_t mg_base_rot(uint8_t c, int r) {  // illumina.py:131-136: A->CTG C->ATG T->ACG G->ACT else N
  uint32_t t;
  switch (c) {
    case 'A': t = 'C' | ('T' << 8) | ('G' << 16); break;
    case 'C': t = 'A' | ('T' << 8) | ('G' << 16); break;
    case 'T': t = 'A' | ('C' << 8) | ('G' << 16); break;
    case 'G': t = 'A' | ('C' << 8) | ('T' << 16); break;
    default: t = 'N' | ('N' << 8) | ('N' << 16); break;
  }
  return (uint8_t)(t >> (8 * r));
}

// searchsorted(row, u) side='left' over n doubles
template <class DP>
MG_HD int mg_lower_bound_f64(DP row, int n, double u) {
  int lo = 0, hi = n;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (row[mid] < u) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// ------------------------------------------------------------------------------------------
// Source of a read's 2-bit codes, 16 bases per chunk.  MAXW > 0: register window (MgWin, loads
// issued up front, both strands a forward extraction); MAXW == 0: streamed from memory (any L).
template <int MAXW, class HP>
struct MgSeqSrc {
  MgWin<(MAXW > 0 ? MAXW : 2)> W;
  HP hap; uint32_t x; int L, strand;
  MG_HD void load(HP hap_, uint32_t x_, int L_, int strand_) {
    hap = hap_; x = x_; L = L_; strand = strand_;
    if constexpr (MAXW > 0) mg_win_load(W, hap, x, L, strand);
  }
  // Between load() and prep() nothing waits for the loads: the kernel issues load() for the next file
  // before the copy-out of the current one, and prep() runs when the emission starts.
  MG_HD void prep() { if constexpr (MAXW > 0) mg_win_prep(W, strand); }
  // streaming source only (MAXW == 0)
  MG_HD uint32_t codes(int c) const {
    if (strand == 0) return mg_codes16(hap, (int64_t)x + 16 * c);
    // output bases [16c, 16c+16) are the complement of forward bases [L-16c-16, L-16c) reversed
    return mg_revcomp16(mg_codes16(hap, (int64_t)x + L - 16 * (int64_t)c - 16));   // may dip 15 below x: front pad
  }
};

// for_each_chunk(S, fn): fn(codes, c) for every 16-base chunk of the read, in order.  Consumes the
// register window of S.
template <int MAXW, class HP, class FN>
MG_HD void mg_for_each_chunk(MgSeqSrc<MAXW, HP> &S, FN fn) {
  const int L = S.L;
  if constexpr (MAXW > 0) {
    MG_NOUNROLL
    for (int c = 0; 16 * c < L; c += 2) {
      fn(mg_win_codes(S.W, 0), c);
      if (16 * (c + 1) < L) fn(mg_win_codes(S.W, 1), c + 1);
      mg_win_slide2(S.W);
    }
  } else {
    for (int c = 0; 16 * c < L; c++) fn(S.codes(c), c);
  }
}

// four output bases of chunk word q (n0 = first base index) through a writer
template <class WR>
MG_HD void mg_put_bases4(WR &w, uint32_t b4, int n0, int L) {
  const uint32_t ch = mg_chars4(b4);
  if (n0 + 4 <= L) w.put_word(ch);
  else for (int j = 0; n0 + j < L; j++) w.put((uint8_t)(ch >> (8 * j)));
}

template <class WR, int MAXW, class HP>
MG_HD void mg_emit_seq_src(WR &w, MgSeqSrc<MAXW, HP> &S) {
  const int L = S.L;
  mg_for_each_chunk(S, [&](uint32_t codes, int c) {
    if (16 * c + 16 <= L) {              // a whole chunk: four words, no bounds logic
      MG_UNROLL
      for (int q = 0; q < 4; q++) w.put_word(mg_chars4((codes >> (8 * q)) & 0xFFu));
      return;
    }
    MG_NOUNROLL
    for (int q = 0; q < 4; q++) if (16 * c + 4 * q < L) mg_put_bases4(w, (codes >> (8 * q)) & 0xFFu, 16 * c + 4 * q, L);
  });
}

// One FASTQ record (fastq_lines, readgenerate.py:227-230):  qname \n SEQ \n+\n ~~~~ \n
// S = the read that goes into this file (already loaded); first/second give the qname's file order.
// The stream is left OPEN: the caller ends it (tail bytes) after every thread of the warp has stored
// its first word -- see MgStream::begin -- and then patches the exception bases (mg_patch_exc).
template <class SP, int MAXW, class NP, class HP, class STR>
MG_HD void mg_emit_record(MgStream<SP> &ws, typename SP::ptr dst, const MgQnConst &Q, const STR &str, uint32_t cnt, NP nodes, MgReadRef first,
                          MgReadRef second, MgSeqSrc<MAXW, HP> &S) {
  const int L = S.L;
  ws.begin(dst);
  mg_put_qname(ws, Q, str, cnt, nodes, first, second, L);
  S.prep();
  mg_emit_seq_src(ws, S);
  ws.append(mg_tok((uint32_t)'\n' | ((uint32_t)'+' << 8) | ((uint32_t)'\n' << 16), 0, 3));
  mg_emit_fill(ws, '~', L);
  ws.append(mg_tok('\n', 0, 1));
}

// The other file's record has the same qname, the same offsets and (for perfect reads) the same
// quality line: only the L sequence bytes are rewritten in place.
template <class SP, int MAXW, class HP, class EP>
MG_HD void mg_rewrite_seq(typename SP::ptr seq_dst, MgSeqSrc<MAXW, HP> &S, EP exc, int n_exc) {
  MgStream<SP> ws;
  ws.begin_rmw(seq_dst);
  S.prep();
  mg_emit_seq_src(ws, S);
  ws.end();
  if (n_exc) mg_patch_exc<SP>(seq_dst, exc, n_exc, S.hap, S.x, S.L, S.strand);
}

// Fused corruption: the qname line first (its last partial word is stored whole: the bytes above it
// are this record's own sequence line, still to be written) ...
template <class SP, class NP, class STR>
MG_HD void mg_emit_frame_qname(typename SP::ptr dst, const MgQnConst &Q, const STR &str, uint32_t cnt, NP nodes, MgReadRef first, MgReadRef second, int L) {
  MgStream<SP> ws;
  ws.begin(dst);
  mg_put_qname(ws, Q, str, cnt, nodes, first, second, L);
  ws.flush_own();
}
// ... then (after the warp has synchronised: the record's last byte shares its word with the next
// record's first bytes) the three separator newlines around the SEQ / QUAL lines that
// mg_emit_seq_corrupt writes
template <class SP>
MG_HD void mg_emit_frame_seps(typename SP::ptr dst, uint32_t qlen, int L) {
  const typename SP::ptr p = dst + (qlen + 1 + (uint32_t)L);
  SP::st8(p, '\n'); SP::st8(p + 1, '+'); SP::st8(p + 2, '\n'); SP::st8(p + (3 + (uint32_t)L), '\n');
}

// ------------------------------------------------------------------------------------------
// Production-mode corruption (Philox draws, ONE alias-table lookup per base).
//
// The reference draws a quality per cycle, then a miscall with probability phred_p[quality], then
// one of the three other bases (illumina.py:151-160).  Per (file, cycle) that is one joint
// distribution over the outcomes (q, s): q the quality, s = 0 "called correctly" or s = 1..3 "called
// as base code ^ s" (A=0 C=1 G=2 T=3: code ^ 1, ^ 2, ^ 3 are the three other bases, each with
// probability 1/3, as base_rot + randint(0,3) give them):
//     P(q, 0) = P(q) (1 - phred_p[q]),        P(q, s) = P(q) phred_p[q] / 3,  s = 1, 2, 3
// It is sampled with ONE 32-bit Philox word and ONE lookup in a Vose alias row of K = 2^kshift
// entries that lists the row's outcomes with non-zero mass (built at model load, mg_api.cu):
//
// Draw layout (the specification tests/philox_ref.py restates in numpy): for template serial t
// (0-based count within the unit; 64-bit template index of the whole file for corrupt-reads), file f
// and cycle group g = n / 4,
//     r = Philox4x32-7(counter = (t_lo, 2 t_hi + f, g, MG_STREAM_CORRUPT), key = (k0, k1)),  w = r[n % 4]
//     e = alias[((f * n_cycles + n) << kshift) | (w & (2^kshift - 1))]        (the entry: w's LOW bits)
//     take = w < e                                (e's top bits are the acceptance threshold: w's HIGH bits decide,
//                                                  independently of the low ones up to 2^(kshift - 32))
//     code = take ? e's SELF field : e's ALIAS field,   fields of 8 bits (s << 6 | q, all q < 64):
//            e = thr16 << 16 | self8 << 8 | alias8,  or of 9 bits (s << 7 | q): e = thr14 << 18 | self9 << 9 | alias9
//     quality = code's q;  an A/C/G/T base becomes "ACGT"[code_of_base ^ s]; any other byte (N, IUPAC,
//     lower case) becomes 'N' when s != 0 (base_rot.get(base, 'NNN'), illumina.py:160) and stays otherwise.
struct MgCorruptCtx {
  const uint32_t *alias;   // [n_mates][n_cycles][1 << kshift]
  int kshift, code9, n_cycles, n_mates;
  uint32_t k0, k1;
};

// outcome code of one base: bits 0..(6|7) the quality, the two bits above the substitution
template <bool C9>
MG_HD uint32_t mg_corrupt_code(const uint32_t *alias, uint32_t ks, uint32_t row, uint32_t w) {
  const uint32_t e = alias[(row << ks) | (w & ((1u << ks) - 1u))];
  const bool take = w < e;
  return C9 ? ((take ? e >> 9 : e) & 0x1FFu) : ((take ? e >> 8 : e) & 0xFFu);
}

// one base given as ASCII (the standalone corrupt-reads kernel's tail path, exception bases)
MG_HD void mg_corrupt_one(const MgCorruptCtx &C, uint32_t f, int n, uint32_t w, uint32_t &base, uint32_t &qual) {
  const uint32_t row = f * (uint32_t)C.n_cycles + (uint32_t)n;
  const uint32_t code = C.code9 ? mg_corrupt_code<true>(C.alias, (uint32_t)C.kshift, row, w) : mg_corrupt_code<false>(C.alias, (uint32_t)C.kshift, row, w);
  const uint32_t qb = C.code9 ? 7u : 6u, s = code >> qb;
  qual = (code & ((1u << qb) - 1u)) + 33u;
  if (s) {
    const uint32_t c = mg_base_code((uint8_t)base);
    base = c > 3 ? (uint32_t)'N' : (0x54474341u >> (8u * (c ^ s))) & 0xFFu;
  }
}

// Four cycles at once.  draw: the Philox block and the four table loads; decode: the four entries
// become four ASCII quality bytes and the four substitutions as nibbles (s_j in bits 4j, 4j+1), which
// is the layout of the PRMT selector that turns 2-bit codes into letters (mg_chars4).
struct MgGrp { uint32_t w[4], e[4], b4; };

template <bool FULL>   // FULL: all four cycles are inside the read
MG_HD void mg_grp_draw(const MgCorruptCtx &C, uint32_t ks, uint32_t t_lo, uint32_t t_hi2f, uint32_t row0, int n0, int L, MgGrp &G) {
  const MgPhilox r = mg_philox_corrupt(t_lo, t_hi2f, (uint32_t)(n0 >> 2), C.k0, C.k1);
  const uint32_t mask = (1u << ks) - 1u;
  MG_UNROLL
  for (int j = 0; j < 4; j++) {
    G.w[j] = r.v[j];
    const uint32_t rj = row0 + ((FULL || n0 + j < L) ? (uint32_t)j : 0u);    // stay inside the table at the read's end
    G.e[j] = C.alias[(rj << ks) | (G.w[j] & mask)];
  }
}

template <bool C9>
MG_HD void mg_grp_decode(const MgGrp &G, uint32_t ks, uint32_t &q4, uint32_t &snib) {
  if constexpr (!C9) {
    uint32_t c[4];
    MG_UNROLL
    for (int j = 0; j < 4; j++) c[j] = (G.w[j] < G.e[j]) ? G.e[j] >> 8 : G.e[j];
    const uint32_t t4 = mg_prmt2(mg_prmt2(c[0], c[1], 0x0040u), mg_prmt2(c[2], c[3], 0x0040u), 0x5410u);   // the four code bytes
    q4 = (t4 & 0x3F3F3F3Fu) + 0x21212121u;
    uint32_t u = (t4 >> 6) & 0x03030303u;                 // s_j in bits 8j, 8j+1 -> bits 4j, 4j+1
    u = (u | (u >> 4)) & 0x00330033u;
    snib = (u | (u >> 8)) & 0x3333u;
  } else {
    q4 = 0x21212121u; snib = 0;
    MG_UNROLL
    for (int j = 0; j < 4; j++) {
      const uint32_t c = ((G.w[j] < G.e[j]) ? G.e[j] >> 9 : G.e[j]) & 0x1FFu;
      q4 += (c & 127u) << (8 * j);
      snib |= (c >> 7) << (4 * j);
    }
  }
}

// four 2-bit codes (low byte of b) with substitutions -> four ASCII bases
MG_HD uint32_t mg_chars4_sub(uint32_t b, uint32_t snib) {
  uint32_t y = (b | (b << 4)) & 0x0F0Fu;
  uint32_t z = ((y | (y << 2)) & 0x3333u) ^ snib;
  return mg_prmt(0x54474341u /* 'A','C','G','T' little-endian */, z);
}

// SEQ and QUAL lines of one read, corrupted on the fly: every thread of a warp is at the same
// cycle of its own record, so the alias row is shared by the warp.
//
// The read's 2-bit codes are first parked, strand-normalised and byte-aligned (one byte per group of
// four cycles), in the tail of the record's OWN quality line: byte coff + g, coff = L - 4 ceil(L / 16).
// The quality bytes written later never reach a parked byte that is still to be read (checked below),
// the register window dies before the main loop, and that loop can be rolled over the groups.
//
// Main loop: two groups per trip in two register sets (A, B); a set's table loads are issued one
// group of work before its decode (draw B, flush A, draw A', flush B, ...) and never copied.
template <class SP, bool C9, int MAXW, class HP, class EP>
MG_HD void mg_emit_seq_corrupt(typename SP::ptr seq_dst, typename SP::ptr qual_dst, MgSeqSrc<MAXW, HP> &S, EP exc, int n_exc,
                               const MgCorruptCtx &C, uint32_t t_lo, uint32_t t_hi2f, uint32_t f) {
  const int L = S.L;
  const struct { uint32_t x; int strand; HP hap; } mine = {S.x, S.strand, S.hap};
  const uint32_t ks = (uint32_t)C.kshift;
  const uint32_t rowf = f * (uint32_t)C.n_cycles;
  const int NCH = (L + 15) >> 4, NG = L >> 2, rem = L & 3;
  const int coff = L - 4 * NCH;                       // >= 0 iff L >= 4
  S.prep();
  uint32_t b_last = 0;                                // the codes of the last, partial group
  if (L >= 4) {
    MgStream<SP> cs;
    cs.begin_rmw(qual_dst + (uint32_t)coff);
    if constexpr (MAXW > 0) {
      MG_UNROLL
      for (int c = 0; c < MAXW - 1; c++) if (16 * c < L) cs.put_word(mg_win_codes(S.W, c));
    } else {
      for (int c = 0; 16 * c < L; c++) cs.put_word(S.codes(c));
    }
    cs.end();
    if (rem) b_last = SP::ld8(qual_dst + (uint32_t)(coff + NG));
  } else {
    if constexpr (MAXW > 0) b_last = mg_win_codes(S.W, 0) & 0xFFu; else b_last = S.codes(0) & 0xFFu;
  }
  // a quality byte never lands on a parked byte before that byte has been read: the draw of group
  // g + 2 (reading byte coff + g + 2) follows the flush of group g (quality bytes up to 4g + 3), and
  // coff + g + 2 > 4g + 3 for every g + 2 < NG whenever L >= 4 (coff >= 12 k + r - 4 for L = 16 k + r).
  MgStream<SP> ws, wq;
  ws.begin_rmw(seq_dst); wq.begin_rmw(qual_dst);
  const typename SP::ptr cbase = qual_dst + (uint32_t)(coff < 0 ? 0 : coff);
  auto draw = [&](MgGrp &G, int g) {
    G.b4 = SP::ld8(cbase + (uint32_t)g);
    mg_grp_draw<true>(C, ks, t_lo, t_hi2f, rowf + 4u * (uint32_t)g, 4 * g, L, G);
  };
  auto flush = [&](const MgGrp &G) {
    uint32_t q4, snib;
    mg_grp_decode<C9>(G, ks, q4, snib);
    ws.put_word(mg_chars4_sub(G.b4, snib)); wq.put_word(q4);
  };
  if (NG > 0) {
    MgGrp A, B;
    int g = 0;
    draw(A, 0);
    MG_NOUNROLL
    while (g + 2 < NG) {
      draw(B, g + 1); flush(A);
      draw(A, g + 2); flush(B);
      g += 2;
    }
    if (g + 1 < NG) { draw(B, g + 1); flush(A); flush(B); }
    else flush(A);
  }
  if (rem) {
    MgGrp G;
    G.b4 = b_last;
    mg_grp_draw<false>(C, ks, t_lo, t_hi2f, rowf + 4u * (uint32_t)NG, 4 * NG, L, G);
    uint32_t q4, snib;
    mg_grp_decode<C9>(G, ks, q4, snib);
    const uint32_t ch = mg_chars4_sub(G.b4, snib);
    for (int j = 0; j < rem; j++) { ws.put((uint8_t)(ch >> (8 * j))); wq.put((uint8_t)(q4 >> (8 * j))); }
  }
  ws.end(); wq.end();
  if (n_exc) {
    // bases in exception runs: a non-ACGT byte (lower case included) becomes 'N' on a miscall
    // (base_rot.get(base, 'NNN'), illumina.py:160) and is copied otherwise; the quality line is already
    // right.  Whether the call was a miscall is read off the letter the main loop wrote: it differs from
    // the letter of the packed code exactly when the substitution s was not 0 (code ^ s != code).
    MgCodeCursor<HP> cur(mine.hap);
    const uint32_t ph = SP::low2(seq_dst);
    const bool words = ph + (uint32_t)L <= 32u * MG_CASE_WORDS;
    MgCaseMask M; M.clear();
    for (int k = mg_exc_first(exc, n_exc, mine.x); k < n_exc; k++) {
      const MgExc e = exc[k];
      if ((uint64_t)e.start >= (uint64_t)mine.x + L) break;
      uint64_t a = e.start > mine.x ? e.start : mine.x;
      uint64_t b = (uint64_t)e.start + e.len < (uint64_t)mine.x + L ? (uint64_t)e.start + e.len : (uint64_t)mine.x + L;
      const bool soft = e.byte == MG_EXC_CASE;
      if (soft && words) {
        const uint32_t i0 = (uint32_t)(a - mine.x), i1 = (uint32_t)(b - mine.x);
        if (mine.strand) M.set(ph + (uint32_t)L - i1, ph + (uint32_t)L - i0); else M.set(ph + i0, ph + i1);
        continue;
      }
      for (uint64_t i = a; i < b; i++) {
        const int idx = (int)(i - mine.x), n = mine.strand ? (L - 1 - idx) : idx;
        const uint32_t code = cur.at(i);
        const uint32_t clean = (0x54474341u /* "ACGT" */ >> (8u * (mine.strand ? code ^ 3u : code))) & 0xFFu;   // what the loop writes when s == 0
        const uint32_t keep = soft ? (0x74676361u /* "acgt" */ >> (8u * code)) & 0xFFu : (uint32_t)e.byte;
        const uint32_t got = SP::ld8(seq_dst + (uint32_t)n);
        SP::st8(seq_dst + (uint32_t)n, (uint8_t)(got != clean ? (uint32_t)'N' : keep));
      }
    }
    if (M.any()) {
      // soft-masked stretches, one aligned word of the line (four cycles) per step: the clean letters are
      // rebuilt from the haplotype, a case base that was miscalled becomes 'N', the others their lower-case
      // (on strand 1: uncomplemented) letter
      typename SP::ptr wp = seq_dst - ph;
      const int nw = (int)((ph + (uint32_t)L + 3u) >> 2);
      MG_NOUNROLL
      for (int k = 0; k < nw; k++, wp += 4) {
        const uint32_t bits = M.next4();
        if (!bits) continue;
        const uint32_t bm = mg_bits4_to_bytes(bits);
        const int n0 = 4 * k - (int)ph;                                  // output position of the word's byte 0
        // haplotype position of the lowest base the word covers, relative to the read
        const int rel = mine.strand ? L - 4 - n0 : n0;
        const int64_t p = (int64_t)mine.x + rel;
        uint32_t c8;                                                     // the four codes at p .. p + 3 (zeros where p < 0)
        if (p >= 0) c8 = mg_codes16(mine.hap, p) & 0xFFu; else c8 = (mg_codes16(mine.hap, 0) << (2u * (uint32_t)(-p))) & 0xFFu;
        if (mine.strand) c8 = (((c8 & 3u) << 6) | ((c8 & 0xCu) << 2) | ((c8 >> 2) & 0xCu) | (c8 >> 6)) ^ 0xFFu;
        const uint32_t clean = mg_chars4(c8);
        const uint32_t got = SP::ld32(wp);
        const uint32_t mis = ((((got ^ clean) & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) >> 7 & 0x01010101u) * 0xFFu;   // bytes that differ
        const uint32_t low = (mine.strand ? mg_complement4(got) : got) | 0x20202020u;
        const uint32_t out = (mis & 0x4E4E4E4Eu /* 'N' */) | (~mis & low);
        SP::st32(wp, (got & ~bm) | (out & bm));
      }
    }
  }
}

// One base call with explicit draws (deterministic mode: the reference's own numpy draws)
template <class DP>
MG_HD void mg_corrupt_call(uint8_t *seq, uint8_t *qual, int n, DP cum_row, int n_bq, DP phred,
                           double u_bq, double u_call, int rot) {
  int bq = mg_lower_bound_f64(cum_row, n_bq, u_bq);                // illumina.py:156
  if (bq > 93) bq = 93;
  if (u_call < phred[bq]) seq[n] = mg_base_rot(seq[n], rot);       // illumina.py:159-160
  qual[n] = (uint8_t)(bq + 33);
}

