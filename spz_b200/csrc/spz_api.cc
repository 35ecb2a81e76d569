// Host side of the drop-in C++ API (include/spz_b200/spz.hpp): namespace spz as the reference
// exports it.  packGaussians / unpackGaussians marshal the std::vector planes into the C-ABI
// (include/spz_b200.h) where the sm_100a kernels do all codec arithmetic; the rest of this file is
// the host glue the reference also keeps on the host -- container header and plane order
// (load-spz.cc:131-139, 533-596), zlib gzip framing (:141-214), file I/O (:598-668), one-element
// accessors (:383-465) and the small math of splat-types.cc.
//
// Error behaviour follows the reference: nothing throws; a failed check prints one line to stdout
// and the function returns false / an empty struct (load-spz.cc:94-100).
#include <zlib.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <fstream>
#include <limits>
#include <mutex>
#include <ostream>
#include <string>
#include <thread>
#include <vector>

#if defined(__linux__)
#include <sys/mman.h>
#endif

#include "spz_internal.hpp"

namespace spz {
namespace detail {
void logLine(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vprintf(fmt, ap);
  va_end(ap);
  printf("\n");
  fflush(stdout);
}

void adviseHugePages(void *p, size_t bytes) {
#if defined(__linux__)
  constexpr uintptr_t kHuge = (uintptr_t)2 << 20;
  const uintptr_t a = ((uintptr_t)p + kHuge - 1) & ~(kHuge - 1), e = ((uintptr_t)p + bytes) & ~(kHuge - 1);
  if (e > a) (void)madvise(reinterpret_cast<void *>(a), e - a, MADV_HUGEPAGE);  // advisory: failure changes nothing
#else
  (void)p;
  (void)bytes;
#endif
}

// true when std::vector<T> is {begin, end, end-of-storage} in that order (libstdc++, libc++)
bool vectorLayoutIsThreePointers() {
  if (const char *env = std::getenv("SPZ_B200_ZEROFILL")) {
    if (env[0] == '1') return false;  // plain resize() everywhere (A/B timing, or a safety valve)
  }
  std::vector<uint32_t> v;
  v.reserve(8);
  v.push_back(1);
  v.push_back(2);
  uint32_t *raw[3];
  if (sizeof v != sizeof raw) return false;
  std::memcpy(raw, &v, sizeof raw);
  return raw[0] == v.data() && raw[1] == v.data() + v.size() && raw[2] == v.data() + v.capacity();
}
}  // namespace detail
namespace {
using detail::logLine;
using detail::resizeUninitialized;

// The reference prints "[SPZ: ERROR] Check failed: file:line: expr" (load-spz.cc:94-100).
#define SPZ_REQUIRE(cond)                                                                \
  do {                                                                                   \
    if (!(cond)) {                                                                       \
      logLine("[SPZ: ERROR] Check failed: %s:%d: %s", __FILE__, __LINE__, #cond);        \
      return false;                                                                      \
    }                                                                                    \
  } while (0)

int shDimOf(int degree) { return degree == 0 ? 0 : degree == 1 ? 3 : degree == 2 ? 8 : degree == 3 ? 15 : 0; }

constexpr uint32_t kMagic = detail::kContainerMagic;
constexpr uint8_t kFlagAntialiased = 0x1;
constexpr size_t kHeaderBytes = detail::kContainerHeaderBytes;

// ---- devices and contexts -----------------------------------------------------------------------
// SPZ_B200_DEVICES="0,1,2,3" shards every call by point range over those GPUs (no collective);
// default is device 0 (or SPZ_B200_DEVICE).  Every call leases a context from the process-wide pool
// (spzb200_acquire) and hands it back on return, so short-lived host threads do not rebuild streams,
// tables, staging and pinned bounce buffers per thread.

}  // namespace

namespace detail {
std::vector<int32_t> configuredDevices() {
  std::vector<int32_t> devs;
  if (const char *list = std::getenv("SPZ_B200_DEVICES")) {
    const char *p = list;
    while (*p) {
      char *end = nullptr;
      const long v = std::strtol(p, &end, 10);
      if (end == p) break;
      devs.push_back((int32_t)v);
      p = (*end == ',') ? end + 1 : end;
    }
  }
  if (devs.empty()) {
    const char *one = std::getenv("SPZ_B200_DEVICE");
    devs.push_back(one ? (int32_t)std::atoi(one) : 0);
  }
  return devs;
}

ContextLease::ContextLease(int32_t device) {
  if (spzb200_acquire(device, &ctx_) != SPZB200_OK) {
    logLine("[SPZ ERROR] spz_b200: %s", spzb200_last_error());
    ctx_ = nullptr;
  }
}

}  // namespace detail

namespace {
using detail::configuredDevices;
using detail::ContextLease;

bool checkCloudSizes(const GaussianCloud &g) {
  // the reference's checks (load-spz.cc:106-117) with the products taken in 64 bits
  const int64_t n = g.numPoints;
  SPZ_REQUIRE(g.numPoints >= 0);
  SPZ_REQUIRE(g.shDegree >= 0);
  SPZ_REQUIRE(g.shDegree <= 3);
  SPZ_REQUIRE((int64_t)g.positions.size() == n * 3);
  SPZ_REQUIRE((int64_t)g.scales.size() == n * 3);
  SPZ_REQUIRE((int64_t)g.rotations.size() == n * 4);
  SPZ_REQUIRE((int64_t)g.alphas.size() == n);
  SPZ_REQUIRE((int64_t)g.colors.size() == n * 3);
  SPZ_REQUIRE((int64_t)g.sh.size() == n * shDimOf(g.shDegree) * 3);
  return true;
}

bool checkPackedSizes(const PackedGaussians &p, int64_t n, int shDim, bool usesFloat16) {
  // load-spz.cc:119-127
  SPZ_REQUIRE((int64_t)p.positions.size() == n * 3 * (usesFloat16 ? 2 : 3));
  SPZ_REQUIRE((int64_t)p.scales.size() == n * 3);
  SPZ_REQUIRE((int64_t)p.rotations.size() == n * (p.usesQuaternionSmallestThree ? 4 : 3));
  SPZ_REQUIRE((int64_t)p.alphas.size() == n);
  SPZ_REQUIRE((int64_t)p.colors.size() == n * 3);
  SPZ_REQUIRE((int64_t)p.sh.size() == n * shDim * 3);
  return true;
}

int32_t streamFlavour(bool usesFloat16, bool smallestThree) {
  if (usesFloat16) return smallestThree ? SPZB200_STREAM_HALF_POSITIONS_SMALLEST_THREE : SPZB200_STREAM_V1;
  return smallestThree ? SPZB200_STREAM_V3 : SPZB200_STREAM_V2;
}

SpzB200Packed viewOf(const PackedGaussians &p, int32_t flavour) {
  SpzB200Packed v;
  std::memset(&v, 0, sizeof v);
  v.num_points = p.numPoints;
  v.sh_degree = p.shDegree;
  v.fractional_bits = p.fractionalBits;
  v.version = flavour;
  v.positions = const_cast<uint8_t *>(p.positions.data());
  v.scales = const_cast<uint8_t *>(p.scales.data());
  v.rotations = const_cast<uint8_t *>(p.rotations.data());
  v.alphas = const_cast<uint8_t *>(p.alphas.data());
  v.colors = const_cast<uint8_t *>(p.colors.data());
  v.sh = const_cast<uint8_t *>(p.sh.data());
  return v;
}

SpzB200Cloud viewOf(const GaussianCloud &g) {
  SpzB200Cloud v;
  std::memset(&v, 0, sizeof v);
  v.num_points = g.numPoints;
  v.sh_degree = g.shDegree;
  v.positions = const_cast<float *>(g.positions.data());
  v.scales = const_cast<float *>(g.scales.data());
  v.rotations = const_cast<float *>(g.rotations.data());
  v.alphas = const_cast<float *>(g.alphas.data());
  v.colors = const_cast<float *>(g.colors.data());
  v.sh = const_cast<float *>(g.sh.data());
  return v;
}

// ---- container ------------------------------------------------------------------------------------

// The 16 header bytes, little endian (load-spz.cc:131-139).  The writer always says version 3
// (load-spz.cc:133,533-539), also for a struct that came from a version-1/2 file.
void writeHeader(const PackedGaussians &p, uint8_t out[kHeaderBytes]) {
  const uint32_t words[3] = {kMagic, 3u, (uint32_t)p.numPoints};
  std::memcpy(out, words, 12);
  out[12] = (uint8_t)p.shDegree;
  out[13] = (uint8_t)p.fractionalBits;
  out[14] = p.antialiased ? kFlagAntialiased : 0;
  out[15] = 0;
}

// plane order in the stream: positions, alphas, colors, scales, rotations, sh
const std::vector<uint8_t> *streamOrder(const PackedGaussians &p, int i) {
  const std::vector<uint8_t> *order[6] = {&p.positions, &p.alphas, &p.colors, &p.scales, &p.rotations, &p.sh};
  return order[i];
}

size_t serializedBytes(const PackedGaussians &p) {
  size_t total = kHeaderBytes;
  for (int i = 0; i < 6; i++) total += streamOrder(p, i)->size();
  return total;
}

void serializeInto(const PackedGaussians &p, uint8_t *dst) {
  writeHeader(p, dst);
  dst += kHeaderBytes;
  for (int i = 0; i < 6; i++) {
    const std::vector<uint8_t> *v = streamOrder(p, i);
    if (!v->empty()) std::memcpy(dst, v->data(), v->size());
    dst += v->size();
  }
}

// gzip policy of saveSpz / loadSpz* (spz_gzip.cc has the block-parallel framing):
//   SPZ_B200_GZIP_THREADS=1   the reference's single-thread deflate, compressed bytes identical to the reference's, always
//   SPZ_B200_GZIP_THREADS=N   N > 1: block-parallel for every container of two blocks (2 MiB) or more
//   unset                     containers below 8 MiB (~130K SH3 gaussians) as the reference writes them, byte for byte;
//                             larger ones block-parallel on up to 16 threads -- one thread deflates ~10 MB/s, i.e.
//                             7 s for a 1M-gaussian scene and a minute for a 10M-gaussian one that the GPU encodes in
//                             milliseconds (same box, 4M SH3: reference saveSpz 28.0 s, this 1.8 s; loadSpz 2.6 s vs
//                             0.11 s -- profiles/r2_file_api_timing.jsonl).  The file is one standard gzip member
//                             either way and inflates to the identical container.
// Loading inflates the blocks of a member that carries the block table concurrently (N threads, default up to 16);
// members without it -- anything the reference wrote -- take the serial inflater.
constexpr size_t kAutoParallelGzipBytes = (size_t)8 << 20;
int hostThreads() { return (int)std::min<unsigned>(16, std::max(1u, std::thread::hardware_concurrency())); }
int gzipThreadsEnv() {
  const char *env = std::getenv("SPZ_B200_GZIP_THREADS");
  return env && *env ? std::max(1, std::atoi(env)) : 0;
}
int deflateThreads(size_t containerBytes) {
  const int env = gzipThreadsEnv();
  if (env) return env;
  return containerBytes >= kAutoParallelGzipBytes ? hostThreads() : 1;
}
}  // namespace
namespace detail {
int inflateThreads() {
  const int env = gzipThreadsEnv();
  return env ? env : hostThreads();
}
}  // namespace detail
namespace {
using detail::inflateThreads;

int64_t maxPointsToRead() {
  // The reference refuses more than 10,000,000 points (load-spz.cc:549).  Lifted here so the large
  // configurations round-trip; SPZ_B200_MAX_POINTS restores any cap.
  if (const char *env = std::getenv("SPZ_B200_MAX_POINTS")) return std::atoll(env);
  return std::numeric_limits<int32_t>::max();
}

}  // namespace

namespace detail {
bool parseContainer(const uint8_t *data, size_t size, Container *c) {
  if (size < kHeaderBytes) {
    logLine("[SPZ ERROR] deserializePackedGaussians: header not found");
    return false;
  }
  uint32_t words[3];
  std::memcpy(words, data, 12);
  if (words[0] != kMagic) {
    logLine("[SPZ ERROR] deserializePackedGaussians: header not found");
    return false;
  }
  const uint32_t version = words[1], numPointsU = words[2];
  const uint8_t shDegree = data[12], fractionalBits = data[13], flags = data[14];
  if (version < 1 || version > 3) {
    logLine("[SPZ ERROR] deserializePackedGaussians: version not supported: %d", (int)version);
    return false;
  }
  if ((int64_t)numPointsU > maxPointsToRead()) {
    logLine("[SPZ ERROR] deserializePackedGaussians: Too many points: %d", (int)numPointsU);
    return false;
  }
  if (shDegree > 3) {
    logLine("[SPZ ERROR] deserializePackedGaussians: Unsupported SH degree: %d", (int)shDegree);
    return false;
  }
  const size_t n = numPointsU;
  const size_t shDim = (size_t)shDimOf(shDegree);
  c->half = version == 1;
  c->smallestThree = version >= 3;
  const size_t sizes[6] = {n * (c->half ? 6 : 9), n, n * 3, n * 3, n * (c->smallestThree ? 4 : 3), n * shDim * 3};
  size_t need = kHeaderBytes;
  for (int i = 0; i < 6; i++) {
    c->offset[i] = need;
    c->bytes[i] = sizes[i];
    need += sizes[i];
  }
  if (size < need) {  // checked before anything is allocated: a corrupt count cannot exhaust memory
    logLine("[SPZ ERROR] deserializePackedGaussians: read error");
    return false;
  }
  c->numPoints = (int32_t)numPointsU;
  c->shDegree = shDegree;
  c->fractionalBits = fractionalBits;
  c->antialiased = (flags & kFlagAntialiased) != 0;
  return true;
}

void writeContainerHeader(uint32_t version, int64_t numPoints, int32_t shDegree, bool antialiased, uint8_t out[kContainerHeaderBytes]) {
  const uint32_t words[3] = {kContainerMagic, version, (uint32_t)numPoints};
  std::memcpy(out, words, 12);
  out[12] = (uint8_t)shDegree;
  out[13] = 12;  // fractionalBits, load-spz.cc:270
  out[14] = antialiased ? kFlagAntialiased : 0;
  out[15] = 0;
}
}  // namespace detail

namespace {
using detail::Container;
using detail::parseContainer;

PackedGaussians deserialize(const uint8_t *data, size_t size) {
  Container c;
  if (!parseContainer(data, size, &c)) return {};
  PackedGaussians r;
  r.numPoints = c.numPoints;
  r.shDegree = c.shDegree;
  r.fractionalBits = c.fractionalBits;
  r.antialiased = c.antialiased;
  r.usesQuaternionSmallestThree = c.smallestThree;
  std::vector<uint8_t> *dst[6] = {&r.positions, &r.alphas, &r.colors, &r.scales, &r.rotations, &r.sh};
  for (int i = 0; i < 6; i++) dst[i]->assign(data + c.offset[i], data + c.offset[i] + c.bytes[i]);
  return r;
}

bool readFile(const std::string &filename, std::vector<uint8_t> *out) {
  std::ifstream in(filename, std::ios::binary | std::ios::ate);
  if (!in.good()) return false;
  const std::streamoff len = in.tellg();
  if (len < 0) return false;
  out->clear();
  resizeUninitialized(*out, (size_t)len);
  in.seekg(0, std::ios::beg);
  if (len > 0) in.read(reinterpret_cast<char *>(out->data()), len);
  return in.good();
}

}  // namespace

// =================================================================================================
// the codec: GPU only
// =================================================================================================

namespace {
enum class PackStatus { Ok, Rejected, DeviceError };
PackStatus packImpl(const GaussianCloud &g, const PackOptions &o, PackedGaussians *result, int32_t streamVersion = SPZB200_STREAM_V3);
PackStatus encodeInto(const GaussianCloud &g, const PackOptions &o, SpzB200Packed out, int32_t streamVersion);
bool encodeContainer(const GaussianCloud &g, const PackOptions &o, int32_t streamVersion, std::vector<uint8_t> *stream, PackStatus *status);
GaussianCloud decodeFrom(const SpzB200Packed &in, int32_t numPoints, int32_t shDegree, bool antialiased, const UnpackOptions &o);
}  // namespace

// (The reference cannot run out of memory gracefully either, but it promises "nothing throws": an allocation that
// fails here is a logged, failed call -- an empty struct -- like every other failure.)
PackedGaussians packGaussians(const GaussianCloud &g, const PackOptions &o) {
  try {
    PackedGaussians packed;
    if (packImpl(g, o, &packed) != PackStatus::Ok) return {};
    return packed;
  } catch (const std::exception &e) {
    logLine("[SPZ ERROR] packGaussians: %s", e.what());
    return {};
  }
}

// Extension (SURVEY.md 8f-4), PARITY UNPINNED: the version-2 form of the stream -- rotations as the first three
// components of the normalised, w >= 0 quaternion in 3 bytes, what unpackQuaternionFirstThree (load-spz.cc:333-345)
// reads.  The reference tree holds no encoder for it; every other plane is what packGaussians writes.
PackedGaussians packGaussiansV2(const GaussianCloud &g, const PackOptions &o) {
  try {
    PackedGaussians packed;
    if (packImpl(g, o, &packed, SPZB200_STREAM_V2) != PackStatus::Ok) return {};
    return packed;
  } catch (const std::exception &e) {
    logLine("[SPZ ERROR] packGaussiansV2: %s", e.what());
    return {};
  }
}

// ... and the container for it: header version 2 (the reference's writer always says 3, load-spz.cc:133), so that
// the reference's loadSpz takes its first-three path.
bool saveSpzV2(const GaussianCloud &g, const PackOptions &o, std::vector<uint8_t> *out) {
  try {
    std::vector<uint8_t> stream;
    PackStatus st;
    if (!encodeContainer(g, o, SPZB200_STREAM_V2, &stream, &st) || st != PackStatus::Ok) return false;
    return compressGzippedParallel(stream.data(), stream.size(), deflateThreads(stream.size()), out);
  } catch (const std::exception &e) {
    logLine("[SPZ ERROR] saveSpzV2: %s", e.what());
    return false;
  }
}

namespace {
PackStatus packImpl(const GaussianCloud &g, const PackOptions &o, PackedGaussians *result, int32_t streamVersion) {
  PackedGaussians &packed = *result;
  if (!checkCloudSizes(g)) return PackStatus::Rejected;
  const size_t n = (size_t)g.numPoints;
  const size_t shDim = (size_t)shDimOf(g.shDegree);
  packed.numPoints = g.numPoints;
  packed.shDegree = g.shDegree;
  packed.fractionalBits = 12;  // load-spz.cc:270
  packed.antialiased = g.antialiased;
  packed.usesQuaternionSmallestThree = streamVersion != SPZB200_STREAM_V2;
  // every byte is written by the encoder (or the struct is discarded on failure)
  resizeUninitialized(packed.positions, n * 9);
  resizeUninitialized(packed.scales, n * 3);
  resizeUninitialized(packed.rotations, n * (packed.usesQuaternionSmallestThree ? 4 : 3));
  resizeUninitialized(packed.alphas, n);
  resizeUninitialized(packed.colors, n * 3);
  resizeUninitialized(packed.sh, n * shDim * 3);
  if (n == 0) return PackStatus::Ok;  // nothing to encode; no device needed (load_spz_test.py:753)
  return encodeInto(g, o, viewOf(packed, streamVersion), streamVersion);
}

// The device part of packGaussians: the cloud's planes -> wherever `out` points (six vectors, or straight into a container).
PackStatus encodeInto(const GaussianCloud &g, const PackOptions &o, SpzB200Packed out, int32_t streamVersion) {
  const SpzB200Cloud in = viewOf(g);
  const std::vector<int32_t> devs = configuredDevices();
  int rc;
  if (devs.size() > 1 && streamVersion == SPZB200_STREAM_V3) {
    rc = spzb200_encode_host_multi(devs.data(), (int32_t)devs.size(), &in, (int32_t)o.from, &out, nullptr);
  } else {
    ContextLease lease(devs[0]);
    if (!lease.get()) return PackStatus::DeviceError;
    rc = spzb200_encode_host_as(lease.get(), &in, (int32_t)o.from, streamVersion, &out, nullptr);
  }
  if (rc != SPZB200_OK) {
    logLine("[SPZ ERROR] spz_b200: %s", spzb200_last_error());
    return PackStatus::DeviceError;
  }
  return PackStatus::Ok;
}

// saveSpz's packGaussians + serializePackedGaussians (load-spz.cc:598-607) without the six vectors in between: the
// container is laid out first -- 16 header bytes, then the planes in stream order at their offsets -- and the
// encoder's copy-out writes every plane straight to its place in it (SURVEY.md 8f-1; the north star's "each GPU
// writes its slice of the plane-major output at a precomputed offset", here for the file image).  Returns false only
// when the cloud is rejected by the size checks (the caller then serialises the empty struct, as the reference does).
bool encodeContainer(const GaussianCloud &g, const PackOptions &o, int32_t streamVersion, std::vector<uint8_t> *stream, PackStatus *status) {
  *status = PackStatus::Rejected;
  if (!checkCloudSizes(g)) return false;
  const size_t n = (size_t)g.numPoints, shDim = (size_t)shDimOf(g.shDegree);
  const bool s3 = streamVersion != SPZB200_STREAM_V2;
  const size_t sizes[6] = {n * 9, n, n * 3, n * 3, n * (s3 ? 4 : 3), n * shDim * 3};  // stream order
  size_t offset[6], total = kHeaderBytes;
  for (int i = 0; i < 6; i++) {
    offset[i] = total;
    total += sizes[i];
  }
  stream->clear();
  resizeUninitialized(*stream, total);  // header written below, every plane byte by the encoder
  uint8_t *base = stream->data();
  detail::writeContainerHeader(s3 ? 3u : 2u, g.numPoints, g.shDegree, g.antialiased, base);
  *status = PackStatus::Ok;
  if (n == 0) return true;
  SpzB200Packed out;
  std::memset(&out, 0, sizeof out);
  out.num_points = g.numPoints;
  out.sh_degree = g.shDegree;
  out.fractional_bits = 12;
  out.version = streamVersion;
  out.positions = base + offset[0]; out.alphas = base + offset[1]; out.colors = base + offset[2];
  out.scales = base + offset[3]; out.rotations = base + offset[4]; out.sh = base + offset[5];
  *status = encodeInto(g, o, out, streamVersion);
  return true;
}

// The device part of unpackGaussians: packed planes wherever they lie (six vectors, or inside an inflated container) ->
// a GaussianCloud.  The size checks are the caller's.
GaussianCloud decodeFrom(const SpzB200Packed &in, int32_t numPoints, int32_t shDegree, bool antialiased, const UnpackOptions &o) {
  const size_t n = (size_t)numPoints, shDim = (size_t)shDimOf(shDegree);
  GaussianCloud result;
  result.numPoints = numPoints;
  result.shDegree = shDegree;
  result.antialiased = antialiased;
  // every float is written by the decoder (or the struct is discarded on failure)
  resizeUninitialized(result.positions, n * 3);
  resizeUninitialized(result.scales, n * 3);
  resizeUninitialized(result.rotations, n * 4);
  resizeUninitialized(result.alphas, n);
  resizeUninitialized(result.colors, n * 3);
  resizeUninitialized(result.sh, n * shDim * 3);
  if (n == 0) return result;
  SpzB200Cloud out = viewOf(result);
  const std::vector<int32_t> devs = configuredDevices();
  int rc;
  if (devs.size() > 1) {
    rc = spzb200_decode_host_multi(devs.data(), (int32_t)devs.size(), &in, (int32_t)o.to, &out, nullptr);
  } else {
    ContextLease lease(devs[0]);
    if (!lease.get()) return {};
    rc = spzb200_decode_host(lease.get(), &in, (int32_t)o.to, &out, nullptr);
  }
  if (rc != SPZB200_OK) {
    logLine("[SPZ ERROR] spz_b200: %s", spzb200_last_error());
    return {};
  }
  return result;
}
}  // namespace

GaussianCloud unpackGaussians(const PackedGaussians &packed, const UnpackOptions &o) {
  const int64_t n = packed.numPoints;
  const int shDim = shDimOf(packed.shDegree);
  const bool usesFloat16 = packed.usesFloat16();
  if (n < 0 || packed.shDegree < 0 || packed.shDegree > 3) {
    // the reference indexes with these unchecked; refusing is the defined version of that
    logLine("[SPZ ERROR] unpackGaussians: invalid numPoints / shDegree");
    return {};
  }
  if (!checkPackedSizes(packed, n, shDim, usesFloat16)) return {};
  try {
    return decodeFrom(viewOf(packed, streamFlavour(usesFloat16, packed.usesQuaternionSmallestThree)), packed.numPoints, packed.shDegree,
                      packed.antialiased, o);
  } catch (const std::exception &e) {
    logLine("[SPZ ERROR] unpackGaussians: %s", e.what());
    return {};
  }
}

// =================================================================================================
// one-element accessors (load-spz.cc:383-465)
// =================================================================================================

bool PackedGaussians::usesFloat16() const { return (int64_t)positions.size() == (int64_t)numPoints * 3 * 2; }

// Pure byte gather: the i-th gaussian's bytes, SH de-interleaved per channel and padded with 128
// (the code of 0.0) up to 15 coefficients.
PackedGaussian PackedGaussians::at(int32_t i) const {
  PackedGaussian r;
  const size_t idx = (size_t)i;
  const size_t posBytes = usesFloat16() ? 6 : 9, rotBytes = usesQuaternionSmallestThree ? 4 : 3;
  std::memcpy(r.position.data(), positions.data() + idx * posBytes, posBytes);
  std::memcpy(r.scale.data(), scales.data() + idx * 3, 3);
  std::memcpy(r.rotation.data(), rotations.data() + idx * rotBytes, rotBytes);
  std::memcpy(r.color.data(), colors.data() + idx * 3, 3);
  r.alpha = alphas[idx];
  const size_t shDim = (size_t)shDimOf(shDegree);
  const uint8_t *s = sh.data() + idx * shDim * 3;
  for (size_t j = 0; j < 15; j++) {
    const bool have = j < shDim;
    r.shR[j] = have ? s[3 * j] : 128;
    r.shG[j] = have ? s[3 * j + 1] : 128;
    r.shB[j] = have ? s[3 * j + 2] : 128;
  }
  return r;
}

// One gaussian through the batched gather kernel (gather_kernels.cu): the struct IS the kernel's
// 65-byte record and the result IS its 59-float output, so there is no marshalling; for a handful of
// records the kernel reads and writes pinned host memory itself (one launch, one synchronize, ~10 us).
// A caller that wants many should use unpackGaussiansAt below: one launch for the whole list.
// Without a usable device there is no CPU path: the failure is logged and every field is NaN, which no
// valid stream decodes to -- never a plausible-looking all-zero gaussian.
static_assert(sizeof(PackedGaussian) == SPZB200_RECORD_BYTES, "PackedGaussian must be the 65-byte record");
static_assert(sizeof(UnpackedGaussian) == SPZB200_UNPACKED_FLOATS * sizeof(float), "UnpackedGaussian must be 59 floats");
static_assert(sizeof(CoordinateConverter) == 21 * sizeof(float), "CoordinateConverter must be 21 floats");

namespace {
void poison(UnpackedGaussian *u, size_t count) {
  float *f = reinterpret_cast<float *>(u);
  for (size_t i = 0; i < count * SPZB200_UNPACKED_FLOATS; i++) f[i] = std::numeric_limits<float>::quiet_NaN();
}
}  // namespace

UnpackedGaussian PackedGaussian::unpack(bool usesFloat16, bool usesQuaternionSmallestThree,
                                        int32_t fractionalBits, const CoordinateConverter &c) const {
  UnpackedGaussian u;
  ContextLease lease(configuredDevices()[0]);
  if (!lease.get() ||
      spzb200_unpack_records_host(lease.get(), reinterpret_cast<const uint8_t *>(this), 1, streamFlavour(usesFloat16, usesQuaternionSmallestThree),
                                  fractionalBits, c.flipP.data(), reinterpret_cast<float *>(&u)) != SPZB200_OK) {
    if (lease.get()) logLine("[SPZ ERROR] spz_b200: %s", spzb200_last_error());
    poison(&u, 1);
  }
  return u;
}

namespace {
std::vector<UnpackedGaussian> unpackAtImpl(const PackedGaussians &packed, const std::vector<int32_t> &indices, const CoordinateConverter &c);
}

// Extension: PackedGaussians::unpack(i, c) for a list of indices in one launch (SURVEY.md 8f-4).
// Returns an empty vector (after a logged line) when an index is out of range or no device is usable.
std::vector<UnpackedGaussian> unpackGaussiansAt(const PackedGaussians &packed, const std::vector<int32_t> &indices,
                                                const CoordinateConverter &c) {
  std::vector<UnpackedGaussian> out;
  if (indices.empty()) return out;
  try {
    return unpackAtImpl(packed, indices, c);
  } catch (const std::exception &e) {
    logLine("[SPZ ERROR] unpackGaussiansAt: %s", e.what());
    return {};
  }
}

namespace {
std::vector<UnpackedGaussian> unpackAtImpl(const PackedGaussians &packed, const std::vector<int32_t> &indices, const CoordinateConverter &c) {
  std::vector<UnpackedGaussian> out;
  const bool usesFloat16 = packed.usesFloat16();
  if (packed.numPoints < 0 || packed.shDegree < 0 || packed.shDegree > 3 ||
      !checkPackedSizes(packed, packed.numPoints, shDimOf(packed.shDegree), usesFloat16))
    return out;
  std::vector<int64_t> idx(indices.begin(), indices.end());
  const SpzB200Packed in = viewOf(packed, streamFlavour(usesFloat16, packed.usesQuaternionSmallestThree));
  resizeUninitialized(out, indices.size());  // every float is written by the kernel (or the vector is cleared on failure)
  ContextLease lease(configuredDevices()[0]);
  if (!lease.get() || spzb200_unpack_gather_host(lease.get(), &in, idx.data(), (int64_t)idx.size(), c.flipP.data(),
                                                 reinterpret_cast<float *>(out.data())) != SPZB200_OK) {
    if (lease.get()) logLine("[SPZ ERROR] spz_b200: %s", spzb200_last_error());
    out.clear();
  }
  return out;
}
}  // namespace

// A consumer that walks a cloud with `for (i...) packed.unpack(i, c)` -- what this accessor is for -- would pay one
// launch + one synchronize (~16 us) per gaussian.  So the accessor reads ahead: once two calls in a row ask for
// consecutive indices, a miss decodes a window of the following records in ONE launch (16, 64, ... up to 4096) and the
// next calls are served from it.  The window is a memo, not a cache of the cloud: it keeps the 65 record bytes it was
// decoded from, and a call is answered from it only if at(i) still yields exactly those bytes under the same stream
// flavour, fractionalBits and converter -- the decoder is a pure function of those, so the answer cannot go stale
// whatever the caller does to the planes between calls.  Random access stays on the one-record path.
// SPZ_B200_UNPACK_READAHEAD=<records> caps the window (0 or 1: off).
namespace {
struct UnpackWindow {
  std::vector<PackedGaussian> records;
  std::vector<UnpackedGaussian> values;
  int64_t first = 0, count = 0;
  int32_t flavour = 0, fractionalBits = 0;
  CoordinateConverter conv;
  int64_t lastIndex = -2;
};

int64_t readAheadLimit() {
  static const int64_t limit = [] {
    const char *env = std::getenv("SPZ_B200_UNPACK_READAHEAD");
    const long long v = env ? std::atoll(env) : 4096;
    return (int64_t)std::min<long long>(std::max<long long>(v, 0), 1 << 16);
  }();
  return limit;
}
}  // namespace

UnpackedGaussian PackedGaussians::unpack(int32_t i, const CoordinateConverter &c) const {
  const bool half = usesFloat16();
  const PackedGaussian rec = at(i);
  const int64_t limit = readAheadLimit();
  if (limit <= 1) return rec.unpack(half, usesQuaternionSmallestThree, fractionalBits, c);
  thread_local UnpackWindow w;
  const int32_t flavour = streamFlavour(half, usesQuaternionSmallestThree);
  const bool sequential = (int64_t)i == w.lastIndex + 1;
  w.lastIndex = i;
  const bool sameDecoder = w.count > 0 && flavour == w.flavour && fractionalBits == w.fractionalBits &&
                           std::memcmp(&c, &w.conv, sizeof c) == 0;
  if (sameDecoder && i >= w.first && i < w.first + w.count &&
      std::memcmp(&rec, &w.records[(size_t)(i - w.first)], sizeof rec) == 0)
    return w.values[(size_t)(i - w.first)];
  // Reading ahead gathers records i+1.. with at(): only inside a struct whose planes really hold numPoints records
  // (at(i) of an inconsistent struct is the caller's business, as in the reference; at(i + k) would be this function's).
  const int64_t n = numPoints;
  const size_t shDim = (size_t)shDimOf(shDegree);
  const bool consistent = n > 0 && i >= 0 && i < n && shDegree >= 0 && shDegree <= 3 &&
                          positions.size() == (size_t)n * (half ? 6 : 9) && scales.size() == (size_t)n * 3 &&
                          rotations.size() == (size_t)n * (usesQuaternionSmallestThree ? 4 : 3) && alphas.size() == (size_t)n &&
                          colors.size() == (size_t)n * 3 && sh.size() == (size_t)n * shDim * 3;
  int64_t want = 1;
  if (sequential && consistent) want = std::min<int64_t>({limit, std::max<int64_t>(16, 4 * w.count), n - i});
  if (want <= 1) {
    w.count = 0;  // the run is broken (or has not started): one record, nothing kept
    return rec.unpack(half, usesQuaternionSmallestThree, fractionalBits, c);
  }
  try {
    w.records.resize((size_t)want);
    w.values.resize((size_t)want);
  } catch (const std::exception &) {
    w.count = 0;
    return rec.unpack(half, usesQuaternionSmallestThree, fractionalBits, c);
  }
  w.records[0] = rec;
  for (int64_t k = 1; k < want; k++) w.records[(size_t)k] = at((int32_t)(i + k));
  w.count = 0;
  ContextLease lease(configuredDevices()[0]);
  if (!lease.get() ||
      spzb200_unpack_records_host(lease.get(), reinterpret_cast<const uint8_t *>(w.records.data()), want, flavour, fractionalBits,
                                  c.flipP.data(), reinterpret_cast<float *>(w.values.data())) != SPZB200_OK) {
    if (lease.get()) logLine("[SPZ ERROR] spz_b200: %s", spzb200_last_error());
    UnpackedGaussian u;
    poison(&u, 1);
    return u;
  }
  w.first = i;
  w.count = want;
  w.flavour = flavour;
  w.fractionalBits = fractionalBits;
  w.conv = c;
  return w.values[0];
}

// =================================================================================================
// container + gzip + files
// =================================================================================================

void serializePackedGaussians(const PackedGaussians &packed, std::ostream *out) {
  uint8_t header[kHeaderBytes];
  writeHeader(packed, header);
  out->write(reinterpret_cast<const char *>(header), kHeaderBytes);
  for (int i = 0; i < 6; i++) {
    const std::vector<uint8_t> *v = streamOrder(packed, i);
    out->write(reinterpret_cast<const char *>(v->data()), (std::streamsize)v->size());
  }
}

// gzip member -> bytes (windowBits 16 + MAX_WBITS: gzip framing only, load-spz.cc:169-173).  The
// ISIZE trailer sizes the first allocation; the loop still grows if it lied.  Stops at the end of
// the first member, like the reference.
bool decompressGzipped(const uint8_t *data, size_t size, std::vector<uint8_t> *out) {
  out->clear();
  z_stream zs;
  std::memset(&zs, 0, sizeof zs);
  if (inflateInit2(&zs, 16 | MAX_WBITS) != Z_OK) return false;
  // The member's ISIZE trailer sizes the buffer in one go -- but only as a hint: in a truncated or damaged blob
  // those four bytes are arbitrary, so the hint is capped at 8x the compressed size (the loop below grows the buffer
  // if a stream really expands more) instead of zero-filling up to 4 GiB for a file that then fails to inflate.
  size_t capacity = 1 << 16;
  if (size >= 18) {
    uint32_t isize;
    std::memcpy(&isize, data + size - 4, 4);
    capacity = std::max<size_t>(capacity, std::min<size_t>(isize, size * 8));
  }
  resizeUninitialized(*out, capacity);  // inflate fills it; trimmed to what was produced below
  constexpr size_t kChunk = (size_t)1 << 30;  // zlib counts in 32 bits
  size_t fed = 0, produced = 0;
  bool ok = false;
  while (true) {
    if (zs.avail_in == 0 && fed < size) {
      const size_t take = std::min(size - fed, kChunk);
      zs.next_in = const_cast<Bytef *>(data + fed);
      zs.avail_in = (uInt)take;
      fed += take;
    }
    if (produced == out->size()) out->resize(out->size() + out->size() / 2);
    const size_t room = std::min(out->size() - produced, kChunk);
    zs.next_out = out->data() + produced;
    zs.avail_out = (uInt)room;
    const int rc = inflate(&zs, Z_NO_FLUSH);
    produced += room - zs.avail_out;
    if (rc == Z_STREAM_END) {
      ok = true;
      break;
    }
    if (rc == Z_OK) continue;
    if (rc == Z_BUF_ERROR && (zs.avail_out == 0 || fed < size)) continue;  // wants room or input
    break;  // corrupt, or the input ended inside the member
  }
  inflateEnd(&zs);
  if (!ok) {
    out->clear();
    return false;
  }
  out->resize(produced);
  return true;
}

namespace detail {
bool inflatePrefix(const uint8_t *data, size_t size, size_t want, std::vector<uint8_t> *out) {
  out->assign(want, 0);
  z_stream zs;
  std::memset(&zs, 0, sizeof zs);
  if (inflateInit2(&zs, 16 | MAX_WBITS) != Z_OK) return false;
  zs.next_in = const_cast<Bytef *>(data);
  zs.avail_in = (uInt)std::min<size_t>(size, (size_t)1 << 30);
  zs.next_out = out->data();
  zs.avail_out = (uInt)want;
  int rc = Z_OK;
  while (zs.avail_out > 0 && rc == Z_OK) rc = inflate(&zs, Z_NO_FLUSH);
  const bool ok = zs.avail_out == 0 || rc == Z_STREAM_END;
  out->resize(want - zs.avail_out);
  inflateEnd(&zs);
  return ok;
}
}  // namespace detail

// zlib deflate with the reference's parameters (default level, gzip wrapper, memLevel 9,
// load-spz.cc:186-214), so the compressed bytes are the same for the same input.
bool compressGzipped(const uint8_t *data, size_t size, std::vector<uint8_t> *out) {
  z_stream zs;
  std::memset(&zs, 0, sizeof zs);
  if (deflateInit2(&zs, Z_DEFAULT_COMPRESSION, Z_DEFLATED, 16 + MAX_WBITS, 9, Z_DEFAULT_STRATEGY) != Z_OK) return false;
  out->clear();
  out->resize(std::max<size_t>(size / 4, 4096));
  size_t produced = 0, consumed = 0;
  bool ok = false;
  while (true) {
    const size_t inChunk = std::min<size_t>(size - consumed, (size_t)1 << 30);
    const bool last = consumed + inChunk == size;
    zs.next_in = const_cast<Bytef *>(reinterpret_cast<const Bytef *>(data) + consumed);
    zs.avail_in = (uInt)inChunk;
    if (produced == out->size()) out->resize(out->size() * 2);
    const size_t outChunk = std::min<size_t>(out->size() - produced, (size_t)1 << 30);
    zs.next_out = out->data() + produced;
    zs.avail_out = (uInt)outChunk;
    const int rc = deflate(&zs, last ? Z_FINISH : Z_NO_FLUSH);
    consumed += inChunk - zs.avail_in;
    produced += outChunk - zs.avail_out;
    if (rc == Z_STREAM_END) {
      ok = true;
      break;
    }
    if (rc != Z_OK && rc != Z_BUF_ERROR) break;
  }
  deflateEnd(&zs);
  if (!ok) {
    out->clear();
    return false;
  }
  out->resize(produced);
  return true;
}

namespace detail {
bool finishSpz(const PackedGaussians &packed, std::vector<uint8_t> *out) {
  std::vector<uint8_t> stream;
  resizeUninitialized(stream, serializedBytes(packed));  // serializeInto writes every byte
  serializeInto(packed, stream.data());
  return compressGzippedParallel(stream.data(), stream.size(), deflateThreads(stream.size()), out);
}
}  // namespace detail

bool saveSpz(const GaussianCloud &g, const PackOptions &o, std::vector<uint8_t> *out) {
  try {
    std::vector<uint8_t> stream;
    PackStatus st;
    if (!encodeContainer(g, o, SPZB200_STREAM_V3, &stream, &st)) {
      // A cloud the size checks reject yields the empty struct, which the reference goes on to
      // serialize as a 0-point file (load-spz.cc:598-607); same here.
      const PackedGaussians empty;
      resizeUninitialized(stream, serializedBytes(empty));
      serializeInto(empty, stream.data());
    } else if (st == PackStatus::DeviceError) {
      return false;  // no GPU: fail loudly, never write a file
    }
    return compressGzippedParallel(stream.data(), stream.size(), deflateThreads(stream.size()), out);
  } catch (const std::exception &e) {  // out of memory: a failed save, not a throw
    logLine("[SPZ ERROR] saveSpz: %s", e.what());
    return false;
  }
}

bool saveSpz(const GaussianCloud &g, const PackOptions &o, const std::string &filename) {
  std::vector<uint8_t> bytes;
  if (!saveSpz(g, o, &bytes)) return false;
  std::ofstream out(filename, std::ios::binary | std::ios::out);
  out.write(reinterpret_cast<const char *>(bytes.data()), (std::streamsize)bytes.size());
  out.close();
  return out.good();
}

PackedGaussians loadSpzPacked(const uint8_t *data, int32_t size) {
  try {
    std::vector<uint8_t> stream;
    if (size < 0 || !decompressGzippedParallel(data, (size_t)size, inflateThreads(), &stream)) return {};
    return deserialize(stream.data(), stream.size());
  } catch (const std::exception &e) {  // out of memory on a hostile or huge file: a failed load, not a throw
    logLine("[SPZ ERROR] loadSpzPacked: %s", e.what());
    return {};
  }
}

PackedGaussians loadSpzPacked(const std::vector<uint8_t> &data) {
  return loadSpzPacked(data.data(), static_cast<int>(data.size()));
}

PackedGaussians loadSpzPacked(const std::string &filename) {
  std::vector<uint8_t> data;
  if (!readFile(filename, &data)) return {};
  return loadSpzPacked(data);
}

GaussianCloud loadSpz(const std::vector<uint8_t> &data, const UnpackOptions &o) {
  return loadSpz(data.data(), static_cast<int>(data.size()), o);
}

// unpackGaussians(loadSpzPacked(data)) (load-spz.cc:635-641) without materialising the PackedGaussians: the planes are
// decoded from where they lie in the inflated container (SURVEY.md 8f-1).
GaussianCloud loadSpz(const uint8_t *data, int32_t size, const UnpackOptions &o) {
  try {
    std::vector<uint8_t> stream;
    if (size < 0 || !decompressGzippedParallel(data, (size_t)size, inflateThreads(), &stream)) return unpackGaussians(PackedGaussians{}, o);
    Container c;
    if (!parseContainer(stream.data(), stream.size(), &c)) return unpackGaussians(PackedGaussians{}, o);
    SpzB200Packed in;
    std::memset(&in, 0, sizeof in);
    in.num_points = c.numPoints;
    in.sh_degree = c.shDegree;
    in.fractional_bits = c.fractionalBits;
    in.version = streamFlavour(c.half, c.smallestThree);
    uint8_t *base = stream.data();
    in.positions = base + c.offset[0]; in.alphas = base + c.offset[1]; in.colors = base + c.offset[2];
    in.scales = base + c.offset[3]; in.rotations = base + c.offset[4]; in.sh = base + c.offset[5];
    return decodeFrom(in, c.numPoints, c.shDegree, c.antialiased, o);
  } catch (const std::exception &e) {  // out of memory on a hostile or huge file: a failed load, not a throw
    logLine("[SPZ ERROR] loadSpz: %s", e.what());
    return {};
  }
}

GaussianCloud loadSpz(const std::string &filename, const UnpackOptions &o) {
  std::vector<uint8_t> data;
  std::ifstream probe(filename, std::ios::binary);
  if (!probe.good()) {
    logLine("[SPZ ERROR] Unable to open: %s", filename.c_str());
    return {};
  }
  probe.close();
  if (!readFile(filename, &data)) {
    logLine("[SPZ ERROR] Unable to load data from: %s", filename.c_str());
    return {};
  }
  return loadSpz(data, o);
}

// =================================================================================================
// small math (splat-types.cc)
// =================================================================================================

// IEEE binary16 -> binary32 by bit manipulation; every half value is exactly representable.
float halfToFloat(Half h) {
  const uint32_t sign = (uint32_t)(h >> 15) << 31, e = (h >> 10) & 0x1fu, mant = h & 0x3ffu;
  uint32_t bits;
  if (e == 0) {
    const float v = std::ldexp((float)mant, -24);  // subnormal half
    std::memcpy(&bits, &v, 4);
    bits |= sign;
  } else if (e == 31) {
    if (mant) return std::numeric_limits<float>::quiet_NaN();
    bits = sign | 0x7f800000u;
  } else {
    bits = sign | ((e + 112u) << 23) | (mant << 13);
  }
  float f;
  std::memcpy(&f, &bits, 4);
  return f;
}

// binary32 -> binary16 with truncation of the mantissa, the reference's conversion
// (splat-types.cc:30-60): NaN -> 0x7c01 | sign, overflow -> Inf, tiny values flush through the
// subnormal range by shifting.
Half floatToHalf(float f) {
  uint32_t b;
  std::memcpy(&b, &f, 4);
  const uint32_t sign = (b >> 16) & 0x8000u;
  const int32_t e = (int32_t)((b >> 23) & 0xffu);
  const uint32_t mant = b & 0x7fffffu;
  if (e == 0xff) return (Half)(sign | (mant ? 0x7c01u : 0x7c00u));
  const int32_t unbiased = e - 127;
  if (unbiased > 15) return (Half)(sign | 0x7c00u);
  if (unbiased > -15) return (Half)(sign | (uint32_t)((unbiased + 15) << 10) | (mant >> 13));
  const int32_t shift = -(unbiased + 14);
  const uint32_t full = 0x800000u | mant;
  // For |f| < 2^-32 the reference shifts a 32-bit value by 32..113 places, which C leaves
  // undefined; its x86-64 build takes the count modulo 32 (SHR/SAR), and so does this.
  const uint32_t shifted = full >> (shift & 31);
  return (Half)(sign | (shifted >> 13));
}

float norm(const Vec3f &a) { return std::sqrt(squaredNorm(a)); }

Vec3f normalized(const Vec3f &v) {
  const float n = norm(v);
  return {v[0] / n, v[1] / n, v[2] / n};
}

float norm(const Quat4f &q) { return std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]); }

Quat4f normalized(const Quat4f &v) {
  const float n = norm(v);
  return {v[0] / n, v[1] / n, v[2] / n, v[3] / n};
}

Quat4f axisAngleQuat(const Vec3f &scaledAxis) {
  const float t2 = squaredNorm(scaledAxis);
  float c = 1.0f, k = 0.5f;  // first-order series at the origin, where sin(t/2)/t -> 1/2
  if (t2 > 0.0f) {
    const float t = std::sqrt(t2);
    c = std::cos(0.5f * t);
    k = std::sin(0.5f * t) / t;
  }
  return normalized(Quat4f{c, scaledAxis[0] * k, scaledAxis[1] * k, scaledAxis[2] * k});
}

}  // namespace spz
