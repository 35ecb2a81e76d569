// The format logic of the device inflater (inflate_kernels.cu), written once for the device and the
// host: one table block of a block-table gzip member (spz_gzip.cc) -- raw deflate data (RFC 1951) --
// into that block's output slice.  tests/host_emul/inflate_host.cc compiles this header with g++ and
// checks it against zlib on valid and hostile streams without a GPU; inflate_kernels.cu runs the same
// function with the lanes of one warp.
//
// The lanes run the decoder in lockstep on identical state: every lane reads the same bits and looks
// up the same shared table entries, so nothing is broadcast.  Work that is not serial is split over the
// lanes (`lane` of `lanes`): filling the code tables, copying matches and stored bytes.  Workspace
// fields are written by lane 0 only and read after sync(); the host passes lane 0 of 1 and a no-op.
//
// The input is untrusted (DESIGN.md section 10):
//   * reads stay in in[0, inLen): a read past the end is an error, never a load;
//   * writes stay in out[0, outLen); a distance may not reach before out[0] (table blocks are
//     independent streams);
//   * the decoder is never more lenient than zlib's inflate() given the same bytes and avail_out =
//     outLen: once the slice is full it goes on parsing exactly as far as zlib does (up to the first
//     byte it would have to write, the end of the input or the end of the final block), so an invalid
//     code, header or stored length that zlib reports there is reported here too.  It is stricter in
//     places (an empty code-length code, a truncated symbol after the slice is full); a block it
//     refuses goes to the host inflater, so strictness costs time, never correctness;
//   * every loop ends: each step consumes at least one bit or writes at least one byte.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define IFL_HD __host__ __device__ __forceinline__
#else
#define IFL_HD inline
#endif

namespace spzb200 {
namespace ifl {

constexpr int kMaxBits = 15;
constexpr int kLitSyms = 288;   // fixed code: 286 and 287 have codes but are invalid
constexpr int kDistSyms = 32;   // fixed code: 30 and 31 have codes but are invalid
constexpr int kClSyms = 19;
constexpr int kLitRoot = 10;    // primary lookup bits; longer codes take the canonical walk
constexpr int kDistRoot = 8;

enum Status : int {
  kOk = 0,
  kTruncated = 1,   // the input ended before the slice was full
  kShort = 2,       // the final block ended before the slice was full
  kBadBlockType = 3,
  kBadStored = 4,   // LEN != ~NLEN
  kBadHeader = 5,   // HLIT / HDIST out of range, a bad repeat, no end-of-block code
  kBadCodeSet = 6,  // over-subscribed or incomplete code lengths
  kBadSymbol = 7,   // an invalid literal/length or distance code
  kBadDistance = 8, // reaches before the slice
};

// A canonical code: counts per length, symbols sorted by (length, symbol), and a primary table of
// 2^root entries indexed by the next `root` input bits, each (symbol << 4) | length, or 0 when the code
// there is longer than root bits (or absent).
struct Code {
  uint16_t count[kMaxBits + 1];
  uint16_t sorted[kLitSyms];
  int16_t maxLen;
};

struct Workspace {
  uint8_t lens[kLitSyms + kDistSyms];
  Code lit, dist;
  uint16_t litTable[1 << kLitRoot];
  uint16_t distTable[1 << kDistRoot];
};

IFL_HD uint32_t reverseBits(uint32_t v, int n) {
  uint32_t r = 0;
  for (int i = 0; i < n; i++) r |= ((v >> i) & 1u) << (n - 1 - i);
  return r;
}

// Builds `c` and its primary table from lens[0, n).  kind 0: code-length code (must be complete);
// 1: literal/length or distance code (zlib's inflate_table also takes an empty set, and an incomplete
// one whose only code has one bit; the missing codes then decode as invalid).  false: the set is
// over-subscribed or incomplete beyond that.  All lanes return the same verdict.
template <class Sync>
IFL_HD bool buildCode(const uint8_t *lens, int n, int kind, Code *c, uint16_t *table, int root, int lane, int lanes, Sync &&sync) {
  uint16_t count[kMaxBits + 1];
  for (int b = 0; b <= kMaxBits; b++) count[b] = 0;
  for (int s = 0; s < n; s++) count[lens[s]]++;
  count[0] = 0;
  int maxLen = 0;
  int left = 1;
  for (int b = 1; b <= kMaxBits; b++) {
    left = (left << 1) - count[b];
    if (left < 0) return false;  // over-subscribed
    if (count[b]) maxLen = b;
  }
  if (left > 0 && (kind == 0 || maxLen > 1)) return false;  // incomplete
  if (lane == 0) {
    uint16_t offs[kMaxBits + 2];
    offs[1] = 0;
    for (int b = 1; b <= kMaxBits; b++) {
      c->count[b] = count[b];
      offs[b + 1] = (uint16_t)(offs[b] + count[b]);
    }
    c->count[0] = 0;
    c->maxLen = (int16_t)maxLen;
    for (int s = 0; s < n; s++)
      if (lens[s]) c->sorted[offs[lens[s]]++] = (uint16_t)s;
  }
  for (int e = lane; e < (1 << root); e += lanes) table[e] = 0;
  sync();
  // codes of at most root bits: code k of length b (canonical order) fills every entry whose low b bits
  // are its bit-reversed code
  int first = 0, index = 0;
  for (int b = 1; b <= root && b <= maxLen; b++) {
    const int cnt = count[b];
    for (int k = lane; k < cnt; k += lanes) {
      const uint32_t rev = reverseBits((uint32_t)(first + k), b);
      const uint16_t entry = (uint16_t)((c->sorted[index + k] << 4) | b);
      for (uint32_t e = rev; e < (1u << root); e += 1u << b) table[e] = entry;
    }
    index += cnt;
    first = (first + cnt) << 1;
  }
  sync();
  return true;
}

// LSB-first bits from in[0, len).  avail() bits are buffered; a read of more than are left fails.
struct BitReader {
  const uint8_t *in;
  uint64_t len, pos;  // pos: next byte to buffer
  uint64_t buf;
  int cnt;
  IFL_HD void refill() {
    while (cnt <= 56 && pos < len) {
      buf |= (uint64_t)in[pos++] << cnt;
      cnt += 8;
    }
  }
  IFL_HD bool need(int n) {
    if (cnt < n) refill();
    return cnt >= n;
  }
  IFL_HD uint32_t peek(int n) const { return (uint32_t)(buf & ((1ull << n) - 1)); }
  IFL_HD void drop(int n) {
    buf >>= n;
    cnt -= n;
  }
  // to the next byte boundary, unbuffering the whole bytes still held
  IFL_HD void alignToByte() {
    drop(cnt & 7);
    pos -= (uint64_t)(cnt >> 3);
    buf = 0;
    cnt = 0;
  }
};

// One symbol.  >= 0: the symbol; -1: the input ended inside the code; -2: no code matches (an
// incomplete or empty set).  Codes of at most `root` bits come from the table; longer ones, and the
// gaps of an incomplete set, walk the canonical code one bit at a time (RFC 1951 section 3.2.2).
IFL_HD int decodeSymbol(BitReader &br, const Code &c, const uint16_t *table, int root) {
  br.refill();
  const int have = br.cnt;
  const uint16_t e = table[br.peek(root)];
  if (e) {
    const int b = e & 15;
    if (b > have) return -1;
    br.drop(b);
    return e >> 4;
  }
  int code = 0, first = 0, index = 0;
  for (int b = 1; b <= kMaxBits; b++) {
    if (b > have) return -1;
    code |= (int)((br.buf >> (b - 1)) & 1);
    const int cnt = c.count[b];
    if (code - first < cnt) {
      br.drop(b);
      return c.sorted[index + code - first];
    }
    if (b >= c.maxLen) return -2;  // zlib's table marks the code invalid at this length
    index += cnt;
    first = (first + cnt) << 1;
    code <<= 1;
  }
  return -2;
}

IFL_HD int lengthBase(int i) {  // i = symbol - 257, 0..28
  if (i < 8) return 3 + i;
  if (i == 28) return 258;
  const int e = (i - 4) >> 2;
  return 3 + (4 << e) + ((i & 3) << e);
}
IFL_HD int lengthExtra(int i) { return (i < 8 || i == 28) ? 0 : ((i - 4) >> 2); }
IFL_HD int distBase(int d) {  // 0..29
  if (d < 4) return 1 + d;
  const int e = (d - 2) >> 1;
  return 1 + (2 << e) + ((d & 1) << e);
}
IFL_HD int distExtra(int d) { return d < 4 ? 0 : ((d - 2) >> 1); }

// Reads the code lengths of a dynamic block into ws->lens (literal/length at [0, hlit), distance at
// [kLitSyms, kLitSyms + hdist)) and builds both codes.  Returns kOk, kTruncated (the input ended) or the
// error zlib reports.
template <class Sync>
IFL_HD int readDynamic(BitReader &br, Workspace *ws, int lane, int lanes, Sync &&sync) {
  if (!br.need(14)) return kTruncated;
  const int hlit = (int)br.peek(5) + 257;
  const int hdist = (int)(br.buf >> 5 & 31) + 1;
  const int hclen = (int)(br.buf >> 10 & 15) + 4;
  br.drop(14);
  if (hlit > 286 || hdist > 30) return kBadHeader;
  uint8_t cl[kClSyms];
  for (int i = 0; i < kClSyms; i++) cl[i] = 0;
  for (int i = 0; i < hclen; i++) {
    if (!br.need(3)) return kTruncated;
    // order 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
    const uint32_t packed[5] = {0x00121110u, 0x06090708u, 0x040b050au, 0x020d030cu, 0x000f010eu};
    cl[(packed[i >> 2] >> (8 * (i & 3))) & 0xff] = (uint8_t)br.peek(3);
    br.drop(3);
  }
  // the code-length code shares the literal table's storage until the literal code is built
  if (!buildCode(cl, kClSyms, 0, &ws->lit, ws->litTable, 7, lane, lanes, sync)) return kBadCodeSet;
  const int total = hlit + hdist;
  int prev = -1;
  uint8_t *lens = ws->lens;
  for (int i = 0; i < total;) {
    const int s = decodeSymbol(br, ws->lit, ws->litTable, 7);
    if (s == -1) return kTruncated;
    if (s < 0) return kBadCodeSet;
    int val = 0, rep = 1;
    if (s < 16) {
      val = s;
    } else {
      const int eb = s == 16 ? 2 : s == 17 ? 3 : 7;
      if (s == 16 && prev < 0) return kBadHeader;  // repeat with no previous length
      if (!br.need(eb)) return kTruncated;
      rep = (s == 16 ? 3 : s == 17 ? 3 : 11) + (int)br.peek(eb);
      br.drop(eb);
      val = s == 16 ? prev : 0;
    }
    if (i + rep > total) return kBadHeader;
    for (int k = 0; k < rep; k++, i++) {
      const int at = i < hlit ? i : kLitSyms + (i - hlit);
      if (lane == 0) lens[at] = (uint8_t)val;
    }
    prev = val;
  }
  if (lane == 0) {
    for (int i = hlit; i < kLitSyms; i++) lens[i] = 0;
    for (int i = hdist; i < kDistSyms; i++) lens[kLitSyms + i] = 0;
  }
  sync();
  if (lens[256] == 0) return kBadHeader;  // no end-of-block code
  if (!buildCode(lens, kLitSyms, 1, &ws->lit, ws->litTable, kLitRoot, lane, lanes, sync)) return kBadCodeSet;
  if (!buildCode(lens + kLitSyms, kDistSyms, 1, &ws->dist, ws->distTable, kDistRoot, lane, lanes, sync)) return kBadCodeSet;
  return kOk;
}

template <class Sync>
IFL_HD void buildFixed(Workspace *ws, int lane, int lanes, Sync &&sync) {
  if (lane == 0) {
    for (int i = 0; i < kLitSyms; i++) ws->lens[i] = (uint8_t)(i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8);
    for (int i = 0; i < kDistSyms; i++) ws->lens[kLitSyms + i] = 5;
  }
  sync();
  buildCode(ws->lens, kLitSyms, 1, &ws->lit, ws->litTable, kLitRoot, lane, lanes, sync);
  buildCode(ws->lens + kLitSyms, kDistSyms, 1, &ws->dist, ws->distTable, kDistRoot, lane, lanes, sync);
}

// Inflates in[0, inLen) into out[0, outLen): kOk when the slice was filled exactly (and zlib's inflate
// would not report an error in what it parses after that), else the first error.  All lanes return the
// same status; lane 0 writes literals, all lanes share copies (sync() before each, so every lane sees
// the bytes written before it).
template <class Sync>
IFL_HD int inflateBlock(const uint8_t *in, uint64_t inLen, uint8_t *out, uint32_t outLen, Workspace *ws, int lane, int lanes,
                        Sync &&sync) {
  BitReader br{in, inLen, 0, 0, 0};
  uint32_t pos = 0;
  bool full = outLen == 0;
  for (;;) {
    if (!br.need(3)) return full ? kOk : kTruncated;
    const bool final = br.peek(1) != 0;
    const int type = (int)(br.buf >> 1 & 3);
    br.drop(3);
    if (type == 3) return kBadBlockType;
    if (type == 0) {  // stored
      br.alignToByte();
      if (br.len - br.pos < 4) return full ? kOk : kTruncated;
      const uint8_t *h = in + br.pos;
      const uint32_t n = (uint32_t)h[0] | ((uint32_t)h[1] << 8), nn = (uint32_t)h[2] | ((uint32_t)h[3] << 8);
      if (n != (nn ^ 0xffffu)) return kBadStored;
      br.pos += 4;
      if (n) {
        if (full) return kOk;  // zlib stops here: a byte to write and no room
        const uint64_t have = br.len - br.pos;
        uint32_t take = n < outLen - pos ? n : outLen - pos;
        if (take > have) take = (uint32_t)have;
        sync();
        for (uint32_t j = lane; j < take; j += lanes) out[pos + j] = in[br.pos + j];
        pos += take;
        br.pos += take;
        if (take < n) {  // the input or the slice ended inside the block
          if (pos == outLen) return kOk;
          return kTruncated;
        }
        full = pos == outLen;
      }
    } else {
      if (type == 1) {
        buildFixed(ws, lane, lanes, sync);
      } else {
        const int st = readDynamic(br, ws, lane, lanes, sync);
        if (st == kTruncated) return full ? kOk : kTruncated;
        if (st != kOk) return st;
      }
      for (;;) {
        const int s = decodeSymbol(br, ws->lit, ws->litTable, kLitRoot);
        if (s == -1) return full ? kOk : kTruncated;
        if (s < 0 || s > 285) return kBadSymbol;
        if (s < 256) {
          if (full) return kOk;
          if (lane == 0) out[pos] = (uint8_t)s;
          pos++;
          full = pos == outLen;
          continue;
        }
        if (s == 256) break;
        const int li = s - 257;
        const int leb = lengthExtra(li);
        if (!br.need(leb)) return full ? kOk : kTruncated;
        const uint32_t length = (uint32_t)lengthBase(li) + (leb ? br.peek(leb) : 0);
        br.drop(leb);
        const int d = decodeSymbol(br, ws->dist, ws->distTable, kDistRoot);
        if (d == -1) return full ? kOk : kTruncated;
        if (d < 0 || d > 29) return kBadSymbol;
        const int deb = distExtra(d);
        if (!br.need(deb)) return full ? kOk : kTruncated;
        const uint32_t dist = (uint32_t)distBase(d) + (deb ? br.peek(deb) : 0);
        br.drop(deb);
        if (full) return kOk;  // zlib leaves at MATCH with no room before checking the distance
        if (dist > pos) return kBadDistance;
        const uint32_t room = outLen - pos, take = length < room ? length : room;
        sync();
        // out[pos + j] = out[pos - dist + j % dist]: every source byte lies before pos, so the lanes
        // copy an overlapping match in one pass
        for (uint32_t j = lane; j < take; j += lanes) out[pos + j] = out[pos - dist + (j % dist)];
        pos += take;
        if (take < length) return kOk;  // the slice ended inside the match: zlib stops here too
        full = pos == outLen;
      }
    }
    if (final) return full ? kOk : kShort;
  }
}

}  // namespace ifl
}  // namespace spzb200
