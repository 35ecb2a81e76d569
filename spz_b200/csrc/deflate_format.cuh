// The format logic of the device deflater (deflate_kernels.cu), written once for the device and the
// host: tokens, length-limited canonical Huffman codes, the dynamic block header, the segment layout
// and CRC-32 combination.  tests/host_emul/deflate_host.cc compiles this header with g++ so the
// format is checked against Python's zlib without a GPU; deflate_kernels.cu runs the same functions,
// the per-item ones (rankOf, pmPlace) spread over the threads of a CTA.
//
// Format (RFC 1951), DESIGN.md section 10:
//   * the input is cut into kSegBytes segments; each is coded on its own -- no back-reference crosses
//     a segment boundary -- so segments are independent pieces of one raw deflate stream;
//   * symbols: literals, and for every maximal run of one byte value of at least kRunMin bytes a
//     literal followed by distance-1 matches of at most 258 bytes;
//   * one dynamic block per segment (literal/length codes <= 15 bits, code-length codes <= 7 bits,
//     every tree with at least two non-zero lengths, end-of-block always present), ended byte-aligned
//     by an empty stored block (zlib's Z_SYNC_FLUSH) -- or, for the last segment of the input, by
//     BFINAL and padding;
//   * when the dynamic block would not be smaller, the segment is stored (blocks of <= 65535 bytes).
// Every byte depends on the segment's bytes and on whether it is the last one: nothing else.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define DFL_HD __host__ __device__ __forceinline__
#else
#define DFL_HD inline
#endif

namespace spzb200 {
namespace dfl {

constexpr int kSegBytes = 1 << 16;
constexpr int kRunMin = 12;  // shortest run coded as a match (DESIGN.md section 10: file sizes measured for 8..32)
constexpr int kSlotBytes = kSegBytes + 64;  // worst case of one coded segment (stored: 65536 + 2 * 5), 16-byte multiple
constexpr int kLitLenSyms = 286;
constexpr int kEob = 256;
constexpr int kMaxBits = 15;
constexpr int kClSyms = 19;
constexpr int kClMaxBits = 7;
constexpr int kMaxClSeq = kLitLenSyms + 2;  // one entry per code length at most (HLIT + HDIST of 2)
constexpr int kStoredMax = 65535;

// ---- symbols -------------------------------------------------------------------------------------

// Length 3..258 -> literal/length symbol 257..285 and its extra bits (RFC 1951 section 3.2.5).
DFL_HD void lengthSymbol(int len, int *sym, int *extraBits, int *extraVal) {
  if (len <= 10) {
    *sym = 254 + len; *extraBits = 0; *extraVal = 0;
  } else if (len == 258) {
    *sym = 285; *extraBits = 0; *extraVal = 0;
  } else {
    const int l = len - 3;  // 8..254
    int e = 0;
    while ((l >> (e + 3)) != 0) e++;  // l in [2^(e+2), 2^(e+3))
    *sym = 265 + (e - 1) * 4 + ((l >> e) - 4);
    *extraBits = e;
    *extraVal = l & ((1 << e) - 1);
  }
}

// The tokens of one maximal run of `len` equal bytes: f(0) for a literal, f(m) for a distance-1
// match of m bytes.  Runs shorter than kRunMin are literals; longer ones are one literal and then
// matches of at most 258 bytes, none shorter than 3 (a remainder of 1 or 2 bytes is literals).
template <class F>
DFL_HD void runTokens(int len, F &&f) {
  if (len < kRunMin) {
    for (int i = 0; i < len; i++) f(0);
    return;
  }
  f(0);
  int m = len - 1;
  while (m >= 3) {
    int take = m < 258 ? m : 258;
    if (m - take > 0 && m - take < 3) take = m - 3;
    f(take);
    m -= take;
  }
  for (; m > 0; m--) f(0);
}

// ---- length-limited Huffman code lengths (package-merge) -------------------------------------------
//
// The active symbols (non-zero frequency) sorted by (frequency, symbol) are the leaves.  Level
// maxBits-1 is the leaves alone; level d < maxBits-1 is the leaves merged with the pairwise sums
// ("packages") of level d+1's list, a leaf before a package of equal weight.  The optimal lengths
// follow from how many leaves the first 2n-2 items of level 0 take, level by level (pmLengths).
// Only the position of every leaf in every level is kept.

// Rank of active symbol s among the active symbols in (frequency, symbol) order.
DFL_HD int rankOf(const uint32_t *freq, int nsym, int s) {
  int r = 0;
  const uint32_t f = freq[s];
  for (int j = 0; j < nsym; j++) {
    const uint32_t g = freq[j];
    r += g != 0 && (g < f || (g == f && j < s));
  }
  return r;
}

// Places item `item` of the level whose leaves are w[0, n) and whose packages come from the
// previous (deeper) level's list prev[0, 2 * np): writes its weight into cur and, for a leaf, its
// position into leafPos.
DFL_HD void pmPlace(const uint32_t *w, int n, const uint32_t *prev, int np, uint32_t *cur, uint16_t *leafPos, int item) {
  if (item < n) {
    const uint32_t x = w[item];
    int lo = 0, hi = np;  // packages lighter than the leaf
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (prev[2 * mid] + prev[2 * mid + 1] < x) lo = mid + 1; else hi = mid;
    }
    cur[item + lo] = x;
    leafPos[item] = (uint16_t)(item + lo);
  } else {
    const int k = item - n;
    const uint32_t p = prev[2 * k] + prev[2 * k + 1];
    int lo = 0, hi = n;  // leaves no heavier than the package
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (w[mid] <= p) lo = mid + 1; else hi = mid;
    }
    cur[k + lo] = p;
  }
}

// Code lengths by rank from the leaf positions of every level (leafPos + d * stride).  n >= 2.
DFL_HD void pmLengths(const uint16_t *leafPos, int stride, int n, int maxBits, uint8_t *lenByRank) {
  for (int i = 0; i < n; i++) lenByRank[i] = 0;
  int m = 2 * n - 2;
  for (int d = 0; d < maxBits && m > 0; d++) {
    const uint16_t *pos = leafPos + d * stride;
    int lo = 0, hi = n;  // leaves among the first m items
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (pos[mid] < m) lo = mid + 1; else hi = mid;
    }
    for (int i = 0; i < lo; i++) lenByRank[i]++;
    m = 2 * (m - lo);
  }
}

// At least two non-zero frequencies (zlib's inflater refuses an incomplete code-length code, and
// gzip-compatible encoders never emit one-code trees): symbols 0 and 1 are the fillers.
DFL_HD void ensureTwo(uint32_t *freq, int nsym) {
  int used = 0, which = -1;
  for (int s = 0; s < nsym; s++)
    if (freq[s]) { used++; which = s; }
  if (used >= 2) return;
  if (used == 0) { freq[0] = 1; freq[1] = 1; return; }
  freq[which == 0 ? 1 : 0] = 1;
}

// The whole construction on one thread (the device uses it for the 19-symbol code-length code; the
// host for everything).  freq must already satisfy ensureTwo.  MAXN >= active symbols.
template <int MAXN, int MAXBITS>
DFL_HD void buildLengthsSerial(const uint32_t *freq, int nsym, uint8_t *lens) {
  uint32_t w[MAXN];
  uint16_t sym[MAXN];
  uint32_t list[2][2 * MAXN];
  uint16_t leafPos[MAXBITS * MAXN];
  uint8_t byRank[MAXN];
  int n = 0;
  for (int s = 0; s < nsym; s++) {
    lens[s] = 0;
    if (freq[s]) n++;
  }
  for (int s = 0; s < nsym; s++)
    if (freq[s]) {
      const int r = rankOf(freq, nsym, s);
      w[r] = freq[s];
      sym[r] = (uint16_t)s;
    }
  int prevItems = 0;
  for (int d = MAXBITS - 1; d >= 0; d--) {
    const int np = d == MAXBITS - 1 ? 0 : prevItems / 2;
    uint32_t *cur = list[d & 1], *prev = list[(d + 1) & 1];
    for (int item = 0; item < n + np; item++) pmPlace(w, n, prev, np, cur, leafPos + d * MAXN, item);
    prevItems = n + np;
  }
  pmLengths(leafPos, MAXN, n, MAXBITS, byRank);
  for (int r = 0; r < n; r++) lens[sym[r]] = byRank[r];
}

// Canonical codes (RFC 1951 section 3.2.2), bit-reversed for LSB-first output.
DFL_HD void canonicalCodes(const uint8_t *lens, int nsym, uint16_t *codes) {
  uint16_t count[16] = {0}, next[16];
  for (int s = 0; s < nsym; s++) count[lens[s]]++;
  count[0] = 0;
  uint16_t code = 0;
  for (int b = 1; b < 16; b++) {
    code = (uint16_t)((code + count[b - 1]) << 1);
    next[b] = code;
  }
  for (int s = 0; s < nsym; s++) {
    const int l = lens[s];
    uint16_t c = 0;
    if (l) {
      const uint16_t v = next[l]++;
      for (int i = 0; i < l; i++) c |= (uint16_t)(((v >> i) & 1) << (l - 1 - i));
    }
    codes[s] = c;
  }
}

// ---- the dynamic block header ------------------------------------------------------------------------

// OR-writes bits LSB first into zeroed 32-bit words.
struct BitWriter {
  uint32_t *words;
  uint32_t pos;
  DFL_HD void put(uint32_t v, int n) {
    const uint32_t w = pos >> 5, sh = pos & 31;
    words[w] |= v << sh;
    if (sh + n > 32) words[w + 1] |= v >> (32 - sh);
    pos += n;
  }
};

// Order of the code-length code lengths in the header: 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
// (a function rather than a table, so device code reads it without a __constant__ copy).
DFL_HD int clOrder(int i) {
  const uint32_t packed[5] = {0x00121110u, 0x06090708u, 0x040b050au, 0x020d030cu, 0x000f010eu};
  return (int)((packed[i >> 2] >> (8 * (i & 3))) & 0xff);
}

struct DynHeader {
  int hlit;      // literal/length lengths sent, 257..286
  int hclen;     // code-length lengths sent, 4..19
  int nseq;      // code-length symbols
  uint32_t bits;  // BFINAL + BTYPE + the whole header
  uint8_t seqSym[kMaxClSeq];
  uint8_t seqExtra[kMaxClSeq];
  uint8_t clLens[kClSyms];
  uint16_t clCodes[kClSyms];
};

// The distance code: two codes of one bit (zlib's rule of two non-zero lengths), only distance 1 used.
constexpr int kHdist = 2;
constexpr int kDistBits = 1;

// Run-length codes the HLIT literal/length lengths and the two distance lengths as one sequence
// (RFC 1951 section 3.2.7: 16 repeats the previous length 3-6 times, 17 / 18 give 3-10 / 11-138 zeros),
// then builds the code-length code and sums the header's bits.
DFL_HD void planHeader(const uint8_t *litLens, DynHeader *h) {
  int hlit = kLitLenSyms;
  while (hlit > 257 && litLens[hlit - 1] == 0) hlit--;
  h->hlit = hlit;
  const int total = hlit + kHdist;
  auto lenAt = [&](int i) -> int { return i < hlit ? litLens[i] : kDistBits; };
  int n = 0;
  for (int i = 0; i < total;) {
    const int cur = lenAt(i);
    int run = 1;
    while (i + run < total && lenAt(i + run) == cur) run++;
    if (cur == 0) {
      int left = run;
      while (left >= 11) { const int t = left < 138 ? left : 138; h->seqSym[n] = 18; h->seqExtra[n++] = (uint8_t)(t - 11); left -= t; }
      if (left >= 3) { h->seqSym[n] = 17; h->seqExtra[n++] = (uint8_t)(left - 3); left = 0; }
      while (left-- > 0) { h->seqSym[n] = 0; h->seqExtra[n++] = 0; }
    } else {
      h->seqSym[n] = (uint8_t)cur; h->seqExtra[n++] = 0;
      int left = run - 1;
      while (left >= 3) { const int t = left < 6 ? left : 6; h->seqSym[n] = 16; h->seqExtra[n++] = (uint8_t)(t - 3); left -= t; }
      while (left-- > 0) { h->seqSym[n] = (uint8_t)cur; h->seqExtra[n++] = 0; }
    }
    i += run;
  }
  h->nseq = n;
  uint32_t freq[kClSyms];
  for (int s = 0; s < kClSyms; s++) freq[s] = 0;
  for (int i = 0; i < n; i++) freq[h->seqSym[i]]++;
  ensureTwo(freq, kClSyms);
  buildLengthsSerial<kClSyms, kClMaxBits>(freq, kClSyms, h->clLens);
  canonicalCodes(h->clLens, kClSyms, h->clCodes);
  int hclen = kClSyms;
  while (hclen > 4 && h->clLens[clOrder(hclen - 1)] == 0) hclen--;
  h->hclen = hclen;
  uint32_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
  for (int i = 0; i < n; i++) {
    const int s = h->seqSym[i];
    bits += h->clLens[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
  }
  h->bits = bits;
}

DFL_HD void writeHeader(const DynHeader &h, bool final, BitWriter &bw) {
  bw.put(final ? 1 : 0, 1);
  bw.put(2, 2);  // BTYPE 10: dynamic Huffman
  bw.put((uint32_t)(h.hlit - 257), 5);
  bw.put((uint32_t)(kHdist - 1), 5);
  bw.put((uint32_t)(h.hclen - 4), 4);
  for (int i = 0; i < h.hclen; i++) bw.put(h.clLens[clOrder(i)], 3);
  for (int i = 0; i < h.nseq; i++) {
    const int s = h.seqSym[i];
    bw.put(h.clCodes[s], h.clLens[s]);
    if (s == 16) bw.put(h.seqExtra[i], 2);
    else if (s == 17) bw.put(h.seqExtra[i], 3);
    else if (s == 18) bw.put(h.seqExtra[i], 7);
  }
}

// ---- segments and gzip blocks -------------------------------------------------------------------------

// Segments of an input of `size` bytes (an empty input is one empty segment).
DFL_HD uint64_t segmentCount(uint64_t size) { return size == 0 ? 1 : (size + kSegBytes - 1) / kSegBytes; }

// Segments per block of the gzip member's "SZ" block table (spz_gzip.cc): the table holds at most
// kMaxTableBlocks entries, so a block is the fewest whole segments that keep it within that.
constexpr uint64_t kMaxTableBlocks = 16000;
DFL_HD uint64_t segmentsPerBlock(uint64_t segments) { return (segments + kMaxTableBlocks - 1) / kMaxTableBlocks; }

// ---- block sizes -------------------------------------------------------------------------------------

// Bytes of a segment coded as stored blocks (it starts byte-aligned): 5 per block of <= 65535 bytes.
DFL_HD uint32_t storedBytes(uint32_t len) {
  const uint32_t blocks = len == 0 ? 1 : (len + kStoredMax - 1) / kStoredMax;
  return len + 5 * blocks;
}

// Bytes of a segment coded as one dynamic block of `bits` bits (header, symbols, end-of-block):
// padded to a byte after BFINAL, or followed by the empty stored block of a sync flush.
DFL_HD uint32_t dynamicBytes(uint32_t bits, bool final) {
  if (final) return (bits + 7) / 8;
  return (bits + 3 + 7) / 8 + 4;
}

// Writes the stored form of in[0, len) to out (storedBytes(len) bytes).
DFL_HD void storedHeaderAt(uint32_t len, bool final, uint32_t block, uint8_t *out) {
  const uint32_t blocks = len == 0 ? 1 : (len + kStoredMax - 1) / kStoredMax;
  const uint32_t start = block * kStoredMax, n = len - start < (uint32_t)kStoredMax ? len - start : kStoredMax;
  uint8_t *p = out + start + 5 * block;
  p[0] = (final && block + 1 == blocks) ? 1 : 0;
  p[1] = (uint8_t)(n & 0xff); p[2] = (uint8_t)(n >> 8);
  p[3] = (uint8_t)(~n & 0xff); p[4] = (uint8_t)((~n >> 8) & 0xff);
}

// ---- CRC-32 (the gzip polynomial, reflected) ----------------------------------------------------------

DFL_HD uint32_t crcMulModP(uint32_t a, uint32_t b) {  // a * b modulo the CRC polynomial (zlib's multmodp)
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
  }
  return p;
}

// x^(8 * bytes) modulo the polynomial.
DFL_HD uint32_t crcShiftOp(uint64_t bytes) {
  uint32_t p = 1u << 31;   // x^0
  uint32_t sq = 1u << 23;  // x^8
  while (bytes) {
    if (bytes & 1) p = crcMulModP(sq, p);
    sq = crcMulModP(sq, sq);
    bytes >>= 1;
  }
  return p;
}

// CRC-32 of A || B from crc(A), crc(B) and |B| (zlib's crc32_combine).
DFL_HD uint32_t crcCombine(uint32_t crcA, uint32_t crcB, uint64_t lenB) { return crcMulModP(crcShiftOp(lenB), crcA) ^ crcB; }

DFL_HD uint32_t crcTableEntry(uint32_t i) {
  uint32_t c = i;
  for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
  return c;
}

}  // namespace dfl
}  // namespace spzb200
