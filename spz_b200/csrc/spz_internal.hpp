// Internals shared by the host-side sources of the drop-in API (spz_api.cc, spz_ply.cc).
#pragma once
#include <cstdint>
#include <cstring>
#include <functional>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/spz_b200.h"
#include "../../include/spz_b200/spz.hpp"

namespace spz {
namespace detail {

// Column layout of a gaussian-splat .ply body: every property is one float.
struct PlyLayout {
  int64_t numPoints = 0;
  int width = 0;   // floats per vertex record
  int shDim = 0;   // SH coefficients per channel present in the file (f_rest count / 3)
  int pos[3], scale[3], rot[4] /* x, y, z, w */, alpha, color[3];
  std::vector<int> rest;  // columns of f_rest_0 .. in file order ([channel][coefficient])
};

// Parses the header and reads the vertex records (load-spz.cc:691-806).  Logs and returns false the
// way loadSplatFromPly does on any malformed input.
bool readPlyRows(const std::string &filename, PlyLayout *layout, std::vector<float> *rows);

// v.resize(n) without the value-initialisation pass, for vectors the codec is about to overwrite
// completely.  The reference's value-returning signatures force std::vector outputs, and at 10M
// SH-degree-3 points resize() spends 1.7 s zero-filling 2.36 GB on one thread -- twenty times the
// whole H2D | kernel | D2H pipeline (SURVEY.md section 8f-1).  reserve() only maps address space;
// the pages are then first touched by the pipeline's copy threads, in parallel.
//
// Setting the end pointer behind the vector's back (the folly resizeWithoutInitialization idea) is
// outside the standard, so it is fenced three ways:
//   * compile time: only libstdc++ / libc++ release configurations whose std::vector is three
//     pointers wide; never under AddressSanitizer (container annotations would flag the planes),
//     _GLIBCXX_DEBUG / _GLIBCXX_ASSERTIONS / libc++ debug or hardening modes; -DSPZ_B200_NO_VECTOR_HACK
//     removes it outright (INTEGRATION.md);
//   * start-up: the {begin, end, end-of-storage} layout is probed on a scratch vector;
//   * run time: SPZ_B200_ZEROFILL=1 switches it off.
// Everything else takes the defined path: reserve(), MADV_HUGEPAGE on the reserved range, then a
// plain resize() -- the zero fill then faults 2 MiB pages instead of 4 KiB ones (about 3x faster than
// a bare resize() on a fresh 2.4 GB plane, still one thread).  `v` must be empty on entry.
#if defined(SPZ_B200_NO_VECTOR_HACK) || defined(__SANITIZE_ADDRESS__) || defined(_GLIBCXX_DEBUG) ||      \
    defined(_GLIBCXX_ASSERTIONS) || defined(_GLIBCXX_SANITIZE_VECTOR) || defined(_LIBCPP_DEBUG) ||      \
    defined(_LIBCPP_ENABLE_ASSERTIONS) || (defined(_LIBCPP_HARDENING_MODE) && _LIBCPP_HARDENING_MODE != 0) || \
    !(defined(__GLIBCXX__) || defined(_LIBCPP_VERSION))
#define SPZ_B200_VECTOR_HACK 0
#elif defined(__has_feature)
#if __has_feature(address_sanitizer)
#define SPZ_B200_VECTOR_HACK 0
#else
#define SPZ_B200_VECTOR_HACK 1
#endif
#else
#define SPZ_B200_VECTOR_HACK 1
#endif
bool vectorLayoutIsThreePointers();
void adviseHugePages(void *p, size_t bytes);  // MADV_HUGEPAGE on the 2 MiB-aligned interior (Linux; no-op elsewhere)
template <class T>
void resizeUninitialized(std::vector<T> &v, size_t n) {
  static_assert(std::is_trivial<T>::value, "only for trivially constructible and destructible elements");
  constexpr size_t kHugeWorthIt = (size_t)32 << 20;
  if (!v.empty() || n == 0) {
    v.resize(n);
    return;
  }
  v.reserve(n);
  // first touch then faults 2 MiB at a time instead of 4 KiB (3x faster fill of a fresh 2.4 GB plane)
  if (n * sizeof(T) >= kHugeWorthIt) adviseHugePages(v.data(), n * sizeof(T));
#if SPZ_B200_VECTOR_HACK
  if constexpr (sizeof(std::vector<T>) == 3 * sizeof(T *)) {
    static const bool hack = vectorLayoutIsThreePointers();
    if (hack) {
      T *raw[3];
      std::memcpy(raw, static_cast<const void *>(&v), sizeof raw);
      raw[1] = raw[0] + n;
      std::memcpy(static_cast<void *>(&v), raw, sizeof raw);
      return;
    }
  }
#endif
  v.resize(n);
}

// A context of the process-wide pool (spzb200_acquire), held for one call.  get() is null -- after one
// logged line -- when no sm_100 device is usable; there is no CPU path to fall back to.
class ContextLease {
 public:
  explicit ContextLease(int32_t device);
  ~ContextLease() {
    if (ctx_) spzb200_release(ctx_);
  }
  ContextLease(const ContextLease &) = delete;
  ContextLease &operator=(const ContextLease &) = delete;
  SpzB200Context *get() const { return ctx_; }

 private:
  SpzB200Context *ctx_ = nullptr;
};
std::vector<int32_t> configuredDevices();             // SPZ_B200_DEVICE(S)
bool finishSpz(const PackedGaussians &packed, std::vector<uint8_t> *out);  // container + gzip (serial or SPZ_B200_GZIP_THREADS)
void logLine(const char *fmt, ...);

// Frames one gzip member in the block-table layout that compressGzippedParallel writes and
// decompressGzippedParallel reads (spz_gzip.cc): header, FEXTRA "SZ" subfield {blockSize, block count,
// 64-bit input size, compressed bytes of every block}, the concatenated raw deflate body -- written by
// writeBody into the sum of `compressed` bytes at the pointer it is given -- then CRC-32 and ISIZE.  Every
// block but the last inflates to blockSize bytes and ends byte-aligned.  Both writers (host zlib
// threads, device deflater) call this.  false: at most 16000 blocks of less than 2 GiB, or writeBody failed.
bool frameBlockMember(size_t size, size_t blockSize, const std::vector<uint32_t> &compressed, uint32_t crc,
                      const std::function<bool(uint8_t *)> &writeBody, std::vector<uint8_t> *out);

// The block table of a member as frameBlockMember writes it, and the trailer's CRC-32.
struct BlockTable {
  size_t blockSize = 0;
  uint64_t totalSize = 0;            // inflated bytes of the whole member
  std::vector<uint32_t> compressed;  // bytes of each block's deflate data
  size_t bodyOffset = 0;             // where the deflate data starts
  uint32_t crc = 0;                  // the trailer's CRC-32 of the inflated bytes
  uint64_t blockBytes(size_t i) const { return i + 1 == compressed.size() ? totalSize - (uint64_t)i * blockSize : blockSize; }
};
// The one parser of the table (spz_gzip.cc), for the host and the device block-parallel inflaters:
// true when `data` is a gzip member carrying a table those may trust -- it fits the member, agrees with
// ISIZE, has blocks under 2 GiB and claims no block larger than 1032 times its compressed length plus
// one.  Reads only the header, the table and the trailer; allocates nothing but t->compressed.
bool parseBlockTable(const uint8_t *data, size_t size, BlockTable *t);

// What the 16 header bytes and the stream length of an inflated container say (load-spz.cc:548-574),
// validated before anything is allocated: parseContainer logs and returns false the way the reference
// fails.  offset / bytes are in stream order: positions, alphas, colors, scales, rotations, sh.
struct Container {
  int32_t numPoints = 0, shDegree = 0, fractionalBits = 0;
  bool antialiased = false, half = false, smallestThree = true;
  size_t offset[6] = {0, 0, 0, 0, 0, 0};
  size_t bytes[6] = {0, 0, 0, 0, 0, 0};
};
bool parseContainer(const uint8_t *data, size_t size, Container *c);
// Threads of the block-parallel inflater: SPZ_B200_GZIP_THREADS, else up to 16.
int inflateThreads();
// The first `want` bytes of the member's inflated stream (fewer if it is shorter); false if the gzip
// data is not readable up to there.
bool inflatePrefix(const uint8_t *data, size_t size, size_t want, std::vector<uint8_t> *out);
constexpr size_t kContainerHeaderBytes = 16;
constexpr uint32_t kContainerMagic = 0x5053474e;  // "NGSP"
// The 16 header bytes the writer puts in front of the planes (load-spz.cc:131-139).
void writeContainerHeader(uint32_t version, int64_t numPoints, int32_t shDegree, bool antialiased, uint8_t out[kContainerHeaderBytes]);

}  // namespace detail
}  // namespace spz
