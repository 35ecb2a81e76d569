// Multi-threaded gzip for the .spz container (host side; SURVEY.md section 8f-2).
//
// The reference deflates the whole container on one thread (load-spz.cc:186-214); on the synthetic
// SH3 stream that runs at ~10 MB/s, about four orders of magnitude slower than the GPU codec that
// fills it.  zlib stays the compressor (north star), but nothing obliges it to run on one core:
//
//   * compressGzippedParallel cuts the input into independent blocks, deflates each on its own
//     thread as a raw deflate stream ended by a sync flush (the last by a finish), and frames the
//     concatenation as ONE ordinary gzip member: any inflater -- the reference's loadSpz, gunzip,
//     Python's gzip -- reads it.  This is pigz's "independent blocks" layout.
//   * the member's FEXTRA field carries an "SZ" subfield with the block size and the compressed
//     length of every block, so decompressGzippedParallel can inflate the blocks concurrently and
//     check the combined CRC-32.  Streams without that subfield (e.g. written by the reference)
//     are inflated serially.
//
// The compressed bytes differ from the reference's single-thread output (block boundaries reset
// the window); the inflated container is identical, which is what parity is defined on
// (SURVEY.md section 8c).  saveSpz / loadSpz use this path only when SPZ_B200_GZIP_THREADS > 1.
#include <zlib.h>

#include <atomic>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <functional>
#include <thread>
#include <vector>

#include "../../include/spz_b200/spz.hpp"
#include "spz_internal.hpp"

namespace spz {
namespace {

constexpr uint8_t kSubfieldId1 = 'S', kSubfieldId2 = 'Z';
constexpr size_t kMinBlock = (size_t)1 << 20;
constexpr size_t kMaxBlocks = 16000;  // 4 bytes each inside the 64 KiB FEXTRA limit (plus 20 of header)

void put32(std::vector<uint8_t> *v, uint32_t x) {
  for (int i = 0; i < 4; i++) v->push_back((uint8_t)(x >> (8 * i)));
}
uint32_t get32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

template <class Fn>
void parallelFor(size_t count, int threads, Fn &&fn) {
  std::atomic<size_t> next{0};
  auto work = [&] {
    for (size_t i = next.fetch_add(1); i < count; i = next.fetch_add(1)) fn(i);
  };
  std::vector<std::thread> pool;
  const int extra = (int)std::min<size_t>(count, (size_t)std::max(1, threads)) - 1;
  try {
    for (int t = 0; t < extra; t++) pool.emplace_back(work);
  } catch (const std::exception &) {
    // fewer threads than asked for: the ones that started (and this one) share the blocks
  }
  work();
  for (auto &t : pool) t.join();
}

// zlib level of the parallel path: the reference's default unless SPZ_B200_GZIP_LEVEL (0..9) says
// otherwise (level 1 is ~3x faster for a few percent of ratio; the inflated bytes never change).
int parallelLevel() {
  const char *env = std::getenv("SPZ_B200_GZIP_LEVEL");
  if (!env || !*env) return Z_DEFAULT_COMPRESSION;
  const int v = std::atoi(env);
  return v < 0 ? Z_DEFAULT_COMPRESSION : (v > 9 ? 9 : v);
}

// One block -> raw deflate bytes, reference parameters (default level, memLevel 9).
bool deflateBlock(const uint8_t *src, size_t len, bool last, int level, std::vector<uint8_t> *out) {
  z_stream zs;
  std::memset(&zs, 0, sizeof zs);
  if (deflateInit2(&zs, level, Z_DEFLATED, -MAX_WBITS, 9, Z_DEFAULT_STRATEGY) != Z_OK) return false;
  out->resize(deflateBound(&zs, (uLong)len) + 16);
  zs.next_in = const_cast<Bytef *>(src);
  zs.avail_in = (uInt)len;
  zs.next_out = out->data();
  zs.avail_out = (uInt)out->size();
  const int rc = deflate(&zs, last ? Z_FINISH : Z_SYNC_FLUSH);
  const bool ok = last ? rc == Z_STREAM_END : (rc == Z_OK && zs.avail_in == 0 && zs.avail_out > 0);
  out->resize(out->size() - zs.avail_out);
  deflateEnd(&zs);
  return ok;
}

}  // namespace

bool compressGzippedParallel(const uint8_t *data, size_t size, int threads, std::vector<uint8_t> *out) {
  if (threads <= 1 || size < 2 * kMinBlock) return compressGzipped(data, size, out);
  size_t blockSize = std::max(kMinBlock, (size + kMaxBlocks - 1) / kMaxBlocks);
  blockSize = (blockSize + 65535) / 65536 * 65536;
  if (blockSize >= ((size_t)1 << 31)) return compressGzipped(data, size, out);
  const size_t blocks = (size + blockSize - 1) / blockSize;
  std::vector<std::vector<uint8_t>> parts(blocks);
  std::vector<uint32_t> crcs(blocks);
  std::atomic<bool> ok{true};
  const int level = parallelLevel();
  parallelFor(blocks, threads, [&](size_t i) {
    const size_t off = i * blockSize, len = std::min(blockSize, size - off);
    if (!deflateBlock(data + off, len, i + 1 == blocks, level, &parts[i])) ok = false;
    crcs[i] = (uint32_t)crc32(crc32(0L, Z_NULL, 0), data + off, (uInt)len);
  });
  if (!ok) {
    out->clear();
    return false;
  }
  uLong crc = crc32(0L, Z_NULL, 0);
  std::vector<uint32_t> compressed(blocks);
  for (size_t i = 0; i < blocks; i++) {
    crc = crc32_combine(crc, crcs[i], (z_off_t)std::min(blockSize, size - i * blockSize));
    compressed[i] = (uint32_t)parts[i].size();
  }
  return detail::frameBlockMember(size, blockSize, compressed, (uint32_t)crc,
                                  [&](uint8_t *dst) {
                                    for (const auto &p : parts) {
                                      if (!p.empty()) std::memcpy(dst, p.data(), p.size());
                                      dst += p.size();
                                    }
                                    return true;
                                  },
                                  out);
}

namespace detail {
bool frameBlockMember(size_t size, size_t blockSize, const std::vector<uint32_t> &compressed, uint32_t crc,
                      const std::function<bool(uint8_t *)> &writeBody, std::vector<uint8_t> *out) {
  const size_t blocks = compressed.size();
  out->clear();
  if (blocks == 0 || blocks > kMaxBlocks || blockSize == 0 || blockSize >= ((size_t)1 << 31)) return false;
  size_t body = 0;
  for (uint32_t c : compressed) body += c;
  const size_t subLen = 16 + 4 * blocks, xlen = 4 + subLen;
  std::vector<uint8_t> head = {0x1f, 0x8b, 8, 4 /* FEXTRA */, 0, 0, 0, 0 /* mtime */, 0 /* xfl */, 3 /* unix */};
  head.push_back((uint8_t)(xlen & 0xff));
  head.push_back((uint8_t)(xlen >> 8));
  head.push_back(kSubfieldId1);
  head.push_back(kSubfieldId2);
  head.push_back((uint8_t)(subLen & 0xff));
  head.push_back((uint8_t)(subLen >> 8));
  put32(&head, (uint32_t)blockSize);
  put32(&head, (uint32_t)blocks);
  put32(&head, (uint32_t)(size & 0xffffffffu));
  put32(&head, (uint32_t)((uint64_t)size >> 32));
  for (size_t i = 0; i < blocks; i++) put32(&head, compressed[i]);
  std::vector<uint8_t> tail;
  put32(&tail, crc);
  put32(&tail, (uint32_t)(size & 0xffffffffu));
  resizeUninitialized(*out, head.size() + body + tail.size());  // the body is written in place, no zero-fill first
  std::memcpy(out->data(), head.data(), head.size());
  std::memcpy(out->data() + head.size() + body, tail.data(), tail.size());
  if (body && !writeBody(out->data() + head.size())) {
    out->clear();
    return false;
  }
  return true;
}

// Parses the gzip header; true when it carries the block table and the table is one the block-parallel
// inflaters may trust.  The table is untrusted input and sizes the output before a byte has been
// inflated, so besides fitting the member (blocks, then CRC-32 and ISIZE) it must agree with ISIZE, keep
// every block under 2 GiB (zlib counts a block in 32 bits) and claim no block larger than deflate can
// expand its compressed length to: 1032 : 1 (a 258-byte match costs at least 2 bits).  Otherwise the
// serial inflater, whose buffer only grows with what zlib really produces, gives the verdict.
bool parseBlockTable(const uint8_t *d, size_t n, BlockTable *t) {
  if (n < 18 || d[0] != 0x1f || d[1] != 0x8b || d[2] != 8) return false;
  const uint8_t flg = d[3];
  size_t pos = 10;
  bool found = false;
  if (flg & 4) {  // FEXTRA
    if (pos + 2 > n) return false;
    const size_t xlen = d[pos] | (d[pos + 1] << 8);
    pos += 2;
    if (pos + xlen > n) return false;
    size_t p = pos;
    while (p + 4 <= pos + xlen) {
      const size_t len = d[p + 2] | (d[p + 3] << 8);
      if (p + 4 + len > pos + xlen) break;
      if (d[p] == kSubfieldId1 && d[p + 1] == kSubfieldId2 && len >= 16 && (len - 16) % 4 == 0) {
        const uint8_t *q = d + p + 4;
        t->blockSize = get32(q);
        const size_t blocks = get32(q + 4);
        t->totalSize = (uint64_t)get32(q + 8) | ((uint64_t)get32(q + 12) << 32);
        if (blocks * 4 + 16 == len && t->blockSize > 0 && blocks > 0 &&
            t->totalSize > (uint64_t)(blocks - 1) * t->blockSize && t->totalSize <= (uint64_t)blocks * t->blockSize) {
          t->compressed.resize(blocks);
          for (size_t i = 0; i < blocks; i++) t->compressed[i] = get32(q + 16 + 4 * i);
          found = true;
        }
      }
      p += 4 + len;
    }
    pos += xlen;
  }
  if (flg & 8) { while (pos < n && d[pos]) pos++; pos++; }   // FNAME
  if (flg & 16) { while (pos < n && d[pos]) pos++; pos++; }  // FCOMMENT
  if (flg & 2) pos += 2;                                     // FHCRC
  if (pos > n || !found || t->compressed.empty()) return false;
  t->bodyOffset = pos;
  const size_t blocks = t->compressed.size();
  size_t end = pos;
  for (size_t i = 0; i < blocks; i++) end += t->compressed[i];
  if (end + 8 > n) return false;  // the table does not fit: not ours after all
  t->crc = get32(d + end);
  if ((uint32_t)(t->totalSize & 0xffffffffu) != get32(d + end + 4)) return false;
  constexpr uint64_t kMaxExpansion = 1032;
  if (t->blockSize >= ((size_t)1 << 31)) return false;
  for (size_t i = 0; i < blocks; i++)
    if (t->blockBytes(i) > kMaxExpansion * ((uint64_t)t->compressed[i] + 1)) return false;
  return true;
}
}  // namespace detail

bool decompressGzippedParallel(const uint8_t *data, size_t size, int threads, std::vector<uint8_t> *out) {
  detail::BlockTable t;
  if (threads <= 1 || !detail::parseBlockTable(data, size, &t)) return decompressGzipped(data, size, out);
  const size_t blocks = t.compressed.size();
  std::vector<size_t> offset(blocks + 1, t.bodyOffset);
  for (size_t i = 0; i < blocks; i++) offset[i + 1] = offset[i] + t.compressed[i];
  const uint32_t wantCrc = t.crc;
  const size_t total = (size_t)t.totalSize;
  out->clear();
  try {
    detail::resizeUninitialized(*out, total);  // every block inflates into its own slice; no zero-fill pass on one thread first
  } catch (const std::exception &) {  // the API never throws (load-spz.cc:94-100): an allocation failure is a failed load
    out->clear();
    return false;
  }
  std::vector<uint32_t> crcs(blocks);
  std::atomic<bool> ok{true};
  parallelFor(blocks, threads, [&](size_t i) {
    const size_t len = t.blockBytes(i);
    z_stream zs;
    std::memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -MAX_WBITS) != Z_OK) { ok = false; return; }
    zs.next_in = const_cast<Bytef *>(data + offset[i]);
    zs.avail_in = (uInt)t.compressed[i];
    zs.next_out = out->data() + i * t.blockSize;
    zs.avail_out = (uInt)len;
    const int rc = inflate(&zs, Z_SYNC_FLUSH);
    const bool filled = (rc == Z_OK || rc == Z_STREAM_END) && zs.avail_out == 0;  // content is vouched for by the CRC below
    inflateEnd(&zs);
    if (!filled) { ok = false; return; }  // the slice is only partly written: nothing to checksum
    crcs[i] = (uint32_t)crc32(crc32(0L, Z_NULL, 0), out->data() + i * t.blockSize, (uInt)len);
  });
  uLong crc = crc32(0L, Z_NULL, 0);
  if (ok)
    for (size_t i = 0; i < blocks; i++) crc = crc32_combine(crc, crcs[i], (z_off_t)t.blockBytes(i));
  if (!ok || (uint32_t)crc != wantCrc) {
    // a damaged table or block: let the serial inflater give the verdict the reference would
    return decompressGzipped(data, size, out);
  }
  return true;
}

}  // namespace spz

