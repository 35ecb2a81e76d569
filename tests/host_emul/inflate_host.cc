// TEST-ONLY host build of spz_b200/csrc/inflate_format.cuh: the device inflater's decoder, run on the
// CPU (one lane) so tests can check it against zlib on valid and hostile streams without a GPU.  Never
// part of the product library.
//   g++ -O2 -std=c++17 -shared -fPIC inflate_host.cc -L../../spz_b200/_lib -lspz_b200 -lz
#include <sys/mman.h>
#include <unistd.h>
#include <zlib.h>

#include <cstdint>
#include <cstring>
#include <vector>

#include "../../spz_b200/csrc/deflate_format.cuh"
#include "../../spz_b200/csrc/inflate_format.cuh"
#include "../../spz_b200/csrc/spz_internal.hpp"

using namespace spzb200;

namespace {

struct NoSync {
  void operator()() const {}
};

int inflateOne(const uint8_t *in, size_t inLen, uint8_t *out, uint32_t outLen) {
  ifl::Workspace ws;
  std::memset(&ws, 0, sizeof ws);
  return ifl::inflateBlock(in, inLen, out, outLen, &ws, 0, 1, NoSync{});
}

// A mapping of `bytes` usable bytes whose end touches an inaccessible page: a read or write one byte
// past the end faults instead of passing unnoticed.
struct Guarded {
  uint8_t *map = nullptr;
  size_t mapBytes = 0;
  uint8_t *data = nullptr;
  explicit Guarded(size_t bytes) {
    const size_t page = (size_t)sysconf(_SC_PAGESIZE);
    const size_t body = (bytes + page - 1) / page * page + page;  // one extra page of canaries in front
    mapBytes = body + page;
    void *m = mmap(nullptr, mapBytes, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (m == MAP_FAILED) return;
    map = static_cast<uint8_t *>(m);
    mprotect(map + body, page, PROT_NONE);
    data = map + body - bytes;
    std::memset(map, 0xA5, body - bytes);  // canaries before the data
  }
  ~Guarded() {
    if (map) munmap(map, mapBytes);
  }
  bool canariesIntact() const {
    for (uint8_t *p = map; p < data; p++)
      if (*p != 0xA5) return false;
    return true;
  }
};

}  // namespace

extern "C" {

// The decoder on in[0, inLen) with outLen bytes of output space.  Returns its status (ifl::Status), and
// writes the slice to out when that is kOk.
int ifl_inflate(const uint8_t *in, size_t inLen, uint8_t *out, uint32_t outLen) { return inflateOne(in, inLen, out, outLen); }

// The same, with the input and the slice each placed against an inaccessible page and canary bytes in
// front of the slice: -100 when a canary changed, -101 when the mapping failed.  The slice is copied to
// out (outLen bytes) whatever the status, so tests can see what an error left behind.
int ifl_inflate_guarded(const uint8_t *in, size_t inLen, uint8_t *out, uint32_t outLen) {
  Guarded gin(inLen), gout(outLen);
  if (!gin.map || !gout.map) return -101;
  if (inLen) std::memcpy(gin.data, in, inLen);
  std::memset(gout.data, 0x5A, outLen);
  const int st = inflateOne(gin.data, inLen, gout.data, outLen);
  if (!gout.canariesIntact() || !gin.canariesIntact()) return -100;
  if (outLen) std::memcpy(out, gout.data, outLen);
  return st;
}

// zlib's verdict the way the block-parallel host inflater asks for it (spz_gzip.cc): one inflate() call
// with Z_SYNC_FLUSH into outLen bytes; 1 when it fills them without an error.
int ifl_zlib(const uint8_t *in, size_t inLen, uint8_t *out, uint32_t outLen) {
  z_stream zs;
  std::memset(&zs, 0, sizeof zs);
  if (inflateInit2(&zs, -MAX_WBITS) != Z_OK) return -1;
  zs.next_in = const_cast<Bytef *>(in);
  zs.avail_in = (uInt)inLen;
  zs.next_out = out;
  zs.avail_out = outLen;
  const int rc = inflate(&zs, Z_SYNC_FLUSH);
  inflateEnd(&zs);
  return (rc == Z_OK || rc == Z_STREAM_END) && zs.avail_out == 0 ? 1 : 0;
}

// The device route for a whole member, serially: the shared table parser, every block through the
// decoder, the CRC-32s combined and compared with the trailer.  1: vouched for (out holds *outSize
// bytes); 0: the device would hand the member to the host inflater; -1: no trusted table.
int ifl_member(const uint8_t *bytes, size_t size, uint8_t *out, size_t capacity, size_t *outSize) {
  spz::detail::BlockTable t;
  *outSize = 0;
  if (!spz::detail::parseBlockTable(bytes, size, &t)) return -1;
  if (capacity < t.totalSize) return -1;
  size_t in = t.bodyOffset;
  uint32_t crc = 0;
  for (size_t i = 0; i < t.compressed.size(); i++) {
    const uint64_t len = t.blockBytes(i);
    uint8_t *slice = out + i * t.blockSize;
    if (inflateOne(bytes + in, t.compressed[i], slice, (uint32_t)len) != ifl::kOk) return 0;
    uint32_t c = 0xffffffffu;
    for (uint64_t k = 0; k < len; k++) c = dfl::crcTableEntry((c ^ slice[k]) & 0xff) ^ (c >> 8);
    crc = dfl::crcCombine(crc, ~c, len);
    in += t.compressed[i];
  }
  if (crc != t.crc) return 0;
  *outSize = (size_t)t.totalSize;
  return 1;
}

// The table as the shared parser reads it: 0 and the sizes, or -1.
int ifl_table(const uint8_t *bytes, size_t size, uint64_t *blockSize, uint64_t *total, uint64_t *bodyOffset, uint32_t *compressed,
              size_t capacity, size_t *blocks) {
  spz::detail::BlockTable t;
  if (!spz::detail::parseBlockTable(bytes, size, &t)) return -1;
  *blockSize = t.blockSize;
  *total = t.totalSize;
  *bodyOffset = t.bodyOffset;
  *blocks = t.compressed.size();
  for (size_t i = 0; i < t.compressed.size() && i < capacity; i++) compressed[i] = t.compressed[i];
  return 0;
}

}  // extern "C"
