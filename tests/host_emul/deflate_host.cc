// TEST-ONLY host build of spz_b200/csrc/deflate_format.cuh: the device deflater's format, run serially
// on the CPU so tests can check it against zlib without a GPU and compare the kernels' output with it
// byte for byte.  Never part of the product library.
//   g++ -O2 -std=c++17 -shared -fPIC deflate_host.cc -L../../spz_b200/_lib -lspz_b200
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../spz_b200/csrc/deflate_format.cuh"
#include "../../spz_b200/csrc/spz_internal.hpp"

using namespace spzb200::dfl;

namespace {

// Serial form of the kernel's symbol pass: the maximal runs of the segment, in order.
template <class F>
void forEachToken(const uint8_t *in, int len, F &&f) {
  for (int p = 0; p < len;) {
    int q = p + 1;
    while (q < len && in[q] == in[p]) q++;
    const uint8_t c = in[p];
    runTokens(q - p, [&](int m) { f(c, m); });
    p = q;
  }
}

}  // namespace

extern "C" {

int dfl_build_lengths(const uint32_t *freqIn, int nsym, int maxBits, uint8_t *lens) {
  uint32_t freq[kLitLenSyms];
  if (nsym < 1 || nsym > kLitLenSyms) return -1;
  std::memcpy(freq, freqIn, sizeof(uint32_t) * nsym);
  ensureTwo(freq, nsym);
  if (maxBits == kMaxBits) buildLengthsSerial<kLitLenSyms, kMaxBits>(freq, nsym, lens);
  else if (maxBits == kClMaxBits && nsym <= kClSyms) buildLengthsSerial<kClSyms, kClMaxBits>(freq, nsym, lens);
  else return -1;
  return 0;
}

// One segment (len <= kSegBytes) -> out (kSlotBytes).  Returns the byte count; *dynamic says which form.
int dfl_encode_segment(const uint8_t *in, int len, int last, uint8_t *out, int *dynamic) {
  uint32_t freq[kLitLenSyms] = {0};
  forEachToken(in, len, [&](uint8_t c, int m) {
    if (m == 0) { freq[c]++; return; }
    int s, eb, ev;
    lengthSymbol(m, &s, &eb, &ev);
    freq[s]++;
  });
  freq[kEob] = 1;
  ensureTwo(freq, kLitLenSyms);
  uint8_t lens[kLitLenSyms];
  uint16_t codes[kLitLenSyms];
  buildLengthsSerial<kLitLenSyms, kMaxBits>(freq, kLitLenSyms, lens);
  canonicalCodes(lens, kLitLenSyms, codes);
  DynHeader h;
  planHeader(lens, &h);
  uint32_t bits = h.bits + lens[kEob];
  forEachToken(in, len, [&](uint8_t c, int m) {
    if (m == 0) { bits += lens[c]; return; }
    int s, eb, ev;
    lengthSymbol(m, &s, &eb, &ev);
    bits += lens[s] + eb + kDistBits;
  });
  const uint32_t dyn = dynamicBytes(bits, last != 0), stored = storedBytes((uint32_t)len);
  std::memset(out, 0, kSlotBytes);
  if (dyn >= stored) {
    *dynamic = 0;
    const uint32_t blocks = len == 0 ? 1 : (len + kStoredMax - 1) / kStoredMax;
    for (uint32_t b = 0; b < blocks; b++) storedHeaderAt((uint32_t)len, last != 0, b, out);
    for (int i = 0; i < len; i++) out[i + 5 * (i / kStoredMax + 1)] = in[i];
    return (int)stored;
  }
  *dynamic = 1;
  std::vector<uint32_t> words(kSlotBytes / 4 + 1, 0);
  BitWriter bw{words.data(), 0};
  writeHeader(h, last != 0, bw);
  forEachToken(in, len, [&](uint8_t c, int m) {
    if (m == 0) { bw.put(codes[c], lens[c]); return; }
    int s, eb, ev;
    lengthSymbol(m, &s, &eb, &ev);
    bw.put(codes[s], lens[s]);
    if (eb) bw.put((uint32_t)ev, eb);
    bw.put(0, kDistBits);  // distance code 0: distance 1
  });
  bw.put(codes[kEob], lens[kEob]);
  if (!last) {
    bw.put(0, 3);                  // empty stored block ...
    bw.pos = (bw.pos + 7) & ~7u;   // ... byte-aligned ...
    bw.put(0xffff0000u, 32);       // ... LEN 0000, NLEN ffff
  }
  std::memcpy(out, words.data(), dyn);
  return (int)dyn;
}

// The device deflater's whole output for `size` host bytes, framed as a gzip member by the library's
// own framing (spz::detail::frameBlockMember).  *out is malloc'd.
int dfl_gzip(const uint8_t *data, size_t size, uint8_t **out, size_t *outSize) {
  const size_t segs = segmentCount(size);
  std::vector<std::vector<uint8_t>> parts(segs);
  std::vector<uint32_t> segBytes(segs);
  uint32_t crc = 0;
  for (size_t s = 0; s < segs; s++) {
    const size_t off = s * kSegBytes;
    const int len = (int)(size - off < (size_t)kSegBytes ? size - off : kSegBytes);
    parts[s].resize(kSlotBytes);
    int dynamic = 0;
    const int n = dfl_encode_segment(data + off, len, s + 1 == segs, parts[s].data(), &dynamic);
    parts[s].resize(n);
    segBytes[s] = (uint32_t)n;
    uint32_t c = 0xffffffffu;
    for (int i = 0; i < len; i++) c = crcTableEntry((c ^ data[off + i]) & 0xff) ^ (c >> 8);
    crc = crcCombine(crc, ~c, (uint64_t)len);
  }
  const size_t perBlock = segmentsPerBlock(segs);
  std::vector<uint32_t> blockBytes((segs + perBlock - 1) / perBlock, 0);
  for (size_t s = 0; s < segs; s++) blockBytes[s / perBlock] += segBytes[s];
  std::vector<uint8_t> bytes;
  const bool ok = spz::detail::frameBlockMember(size, perBlock * kSegBytes, blockBytes, crc,
                                                [&](uint8_t *dst) {
                                                  for (auto &p : parts) {
                                                    std::memcpy(dst, p.data(), p.size());
                                                    dst += p.size();
                                                  }
                                                  return true;
                                                },
                                                &bytes);
  if (!ok) return -1;
  *out = static_cast<uint8_t *>(std::malloc(bytes.size() ? bytes.size() : 1));
  std::memcpy(*out, bytes.data(), bytes.size());
  *outSize = bytes.size();
  return 0;
}

void dfl_free(void *p) { std::free(p); }

}  // extern "C"
