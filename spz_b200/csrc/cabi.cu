// C-ABI of the codec (include/spz_b200.h): contexts, the two host-built tables, the
// device-pointer entry points, the chunked host-pointer pipeline and its multi-GPU form.
//
// There is no CPU implementation of the codec in this library.  The only per-value arithmetic
// done on the host is the one-time construction of two small tables per context, both of which
// depend on the host's libm exactly as the reference does (load-spz.cc:85,87):
//   * the 255 thresholds of the alpha quantizer  a -> toUint8(sigmoid(a) * 255)   (uses expf)
//   * the 256 values of the alpha dequantizer    b -> invSigmoid(b / 255.0f)      (uses logf)
#include <cuda_runtime.h>
#include <zlib.h>
#if defined(__x86_64__) && (defined(__GNUC__) || defined(__clang__))
#include <immintrin.h>
#endif

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <condition_variable>
#include <atomic>
#include <cstring>
#include <deque>
#include <exception>
#include <functional>
#include <memory>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/spz_b200.h"
#include "../../include/spz_b200/spz.hpp"
#include "batch_plan.hpp"
#include "codec_kernels.cuh"
#include "codec_math.cuh"
#include "deflate_format.cuh"
#include "inflate_format.cuh"
#include "spz_internal.hpp"

namespace {

thread_local std::string tlsError;
thread_local int tlsShardCount = 1;  // > 1 on the per-device threads of a *_host_multi call

int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  tlsError = buf;
  return code;
}

int cudaFail(cudaError_t e, const char *what) {
  return fail(e == cudaErrorMemoryAllocation ? SPZB200_ERR_NOMEM : SPZB200_ERR_CUDA, "%s: %s",
              what, cudaGetErrorString(e));
}

#define CU(call)                                   \
  do {                                             \
    cudaError_t e_ = (call);                       \
    if (e_ != cudaSuccess) return cudaFail(e_, #call); \
  } while (0)

int shDimOf(int degree) { return degree == 0 ? 0 : degree == 1 ? 3 : degree == 2 ? 8 : 15; }

// ---- the two libm-dependent tables ------------------------------------------------------------

// The reference expression, load-spz.cc:301 with :85 and :74, for a non-NaN argument.  This file
// is compiled with -ffp-contract=off so the product s * 255 is rounded on its own.
uint32_t alphaByteOnHost(float a) {
  const float s = 1 / (1 + std::exp(-a));
  float r = std::round(s * 255.0f);
  r = r < 0.0f ? 0.0f : (255.0f < r ? 255.0f : r);
  return (uint32_t)r;
}

// order-preserving map float <-> uint32 (negative floats reversed below positives)
uint32_t keyOf(float f) {
  uint32_t b;
  std::memcpy(&b, &f, 4);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
float floatOf(uint32_t k) {
  const uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  float f;
  std::memcpy(&f, &b, 4);
  return f;
}

// thr[L-1] = the smallest float whose alpha byte is >= L, L = 1..255; thr[255] = +Inf.
// Exact because the byte is monotone in a (checked below on a 2^16-point grid plus both
// neighbours of every threshold; over every float of [-8, 8] against the oracle's expression in
// tests/test_oracle.py::test_alpha_quantizer_is_a_monotone_step_function and against the reference's
// golden thresholds in tests/test_cabi.py::test_host_built_tables_match_reference).
bool buildAlphaThresholds(float thr[256], std::string *why) {
  const uint32_t kLo = keyOf(-std::numeric_limits<float>::infinity());
  const uint32_t kHi = keyOf(std::numeric_limits<float>::infinity());
  for (uint32_t level = 1; level <= 255; level++) {
    uint32_t lo = kLo, hi = kHi;  // f(hi) = 255 >= level always; find the first key with f >= level
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (alphaByteOnHost(floatOf(mid)) >= level) hi = mid; else lo = mid + 1;
    }
    thr[level - 1] = floatOf(lo);
  }
  thr[255] = std::numeric_limits<float>::infinity();
  auto viaTable = [&](float a) {
    uint32_t c = 0;
    for (int i = 0; i < 255; i++) c += a >= thr[i];
    return c;
  };
  for (uint32_t level = 1; level <= 255; level++) {
    const uint32_t k = keyOf(thr[level - 1]);
    const float here = thr[level - 1], below = floatOf(k - 1);
    if (viaTable(here) != alphaByteOnHost(here) || (k > kLo && viaTable(below) != alphaByteOnHost(below))) {
      *why = "alpha quantizer is not a monotone step function with this libm";
      return false;
    }
  }
  for (uint32_t i = 0; i < 65536; i++) {
    const float a = floatOf(kLo + (uint32_t)(((uint64_t)(kHi - kLo) * i) >> 16));
    if (viaTable(a) != alphaByteOnHost(a)) {
      *why = "alpha threshold table disagrees with the direct expression";
      return false;
    }
  }
  return true;
}

void buildAlphaLut(float lut[256]) {
  for (int i = 0; i < 256; i++) {
    const float x = (float)i / 255.0f;        // load-spz.cc:518
    lut[i] = std::log(x / (1.0f - x));        // load-spz.cc:87
  }
}

// Both tables depend only on the host's libm, so they are built once per process (the threshold
// search + its self-check is ~10 ms of host time that every later context skips).
struct HostTables {
  float thr[256];
  float lut[256];
  bool ok = false;
  std::string why;
};
const HostTables &hostTables() {
  static const HostTables *t = [] {
    HostTables *h = new HostTables;
    h->ok = buildAlphaThresholds(h->thr, &h->why);
    buildAlphaLut(h->lut);
    return h;
  }();
  return *t;
}

#ifndef SPZ_STAGES
#define SPZ_STAGES 3
#endif
constexpr int kStages = SPZ_STAGES;

struct Stage {
  cudaStream_t stream = nullptr;
  uint8_t *dIn = nullptr;   // input planes of one range (device)
  uint8_t *dOut = nullptr;  // output planes of one range (device)
  size_t dInCap = 0, dOutCap = 0;
  uint8_t *hIn = nullptr;      // pinned bounce buffers, used only when the caller's planes are pageable
  uint8_t *hOut = nullptr;
  size_t hInCap = 0, hOutCap = 0;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> pieceEv;  // bounced output: one per D2H piece of the range in flight
};

// The bounce copies move each byte once and never read it back on the CPU, so large ones use non-temporal stores
// (no read-for-ownership of the destination lines, no cache pollution): on x86-64 with AVX2, chosen at run time;
// plain memcpy otherwise, for small pieces, and with SPZB200_NT_COPY=0 (profiles/r2_tuning_notes.txt section 15).
#if defined(__x86_64__) && (defined(__GNUC__) || defined(__clang__))
__attribute__((target("avx2"))) static void copyNonTemporalAvx2(uint8_t *dst, const uint8_t *src, size_t bytes) {
  const size_t head = (32 - (reinterpret_cast<uintptr_t>(dst) & 31)) & 31;
  if (head) {
    std::memcpy(dst, src, head);
    dst += head; src += head; bytes -= head;
  }
  size_t i = 0;
  for (; i + 128 <= bytes; i += 128) {
    const __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i));
    const __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i + 32));
    const __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i + 64));
    const __m256i d = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i + 96));
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i), a);
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 32), b);
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 64), c);
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 96), d);
  }
  _mm_sfence();
  if (i < bytes) std::memcpy(dst + i, src + i, bytes - i);
}
static bool nonTemporalCopyUsable() {
  static const bool ok = [] {
    const char *env = std::getenv("SPZB200_NT_COPY");
    return !(env && env[0] == '0') && __builtin_cpu_supports("avx2");
  }();
  return ok;
}
static void bounceCopy(void *dst, const void *src, size_t bytes) {
  if (bytes >= ((size_t)256 << 10) && nonTemporalCopyUsable()) copyNonTemporalAvx2(static_cast<uint8_t *>(dst), static_cast<const uint8_t *>(src), bytes);
  else std::memcpy(dst, src, bytes);
}
#else
static void bounceCopy(void *dst, const void *src, size_t bytes) { std::memcpy(dst, src, bytes); }
#endif

// A few host threads that move pieces between the caller's pageable planes and the pinned bounce buffers
// (one thread copies ~11 GB/s, eight ~65 -- scripts/host_copy_probe.cu; the PCIe link wants ~55).  A task is a
// closure: copy a piece and queue its DMA, or wait for a piece's DMA and copy it out (runBouncedStages below).
// Created on the first pageable call of a context.
class CopyPool {
 public:
  using Task = std::function<void()>;
  explicit CopyPool(int threads) {
    try {
      for (int i = 0; i < threads; i++) workers_.emplace_back([this] { loop(); });
    } catch (const std::exception &) {
      // fewer threads than asked for (none, in the limit): helpUntil() makes the calling thread a worker too
    }
  }
  ~CopyPool() {
    {
      std::lock_guard<std::mutex> g(m_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto &t : workers_) t.join();
  }
  void submit(std::vector<Task> &&tasks) {  // all or nothing: an allocation failure leaves the queue as it was and rethrows
    {
      std::lock_guard<std::mutex> g(m_);
      size_t pushed = 0;
      try {
        for (Task &t : tasks) {
          queue_.push_back(std::move(t));
          pushed++;
        }
      } catch (...) {
        while (pushed--) queue_.pop_back();
        throw;
      }
    }
    cv_.notify_all();
  }
  void resubmit(Task &&t) {  // a task that found its input not ready yet goes to the back of the queue
    {
      std::lock_guard<std::mutex> g(m_);
      queue_.push_back(std::move(t));
    }
    cv_.notify_one();
  }
  bool othersQueued() {
    std::lock_guard<std::mutex> g(m_);
    return !queue_.empty();
  }
  // The calling thread works through the queue too until done() holds; tasks announce progress with progressed().
  template <class Pred>
  void helpUntil(Pred done) {
    std::unique_lock<std::mutex> g(m_);
    while (!done()) {
      if (!queue_.empty()) {
        Task t = std::move(queue_.front());
        queue_.pop_front();
        g.unlock();
        t();
        g.lock();
      } else {
        progress_.wait(g);
      }
    }
  }
  void progressed() {
    std::lock_guard<std::mutex> g(m_);
    progress_.notify_all();
  }

 private:
  void loop() {
    std::unique_lock<std::mutex> g(m_);
    while (true) {
      cv_.wait(g, [this] { return stop_ || !queue_.empty(); });
      if (queue_.empty()) return;  // stop_
      Task t = std::move(queue_.front());
      queue_.pop_front();
      g.unlock();
      t();
      g.lock();
    }
  }
  std::vector<std::thread> workers_;
  std::deque<Task> queue_;
  std::mutex m_;
  std::condition_variable cv_, progress_;
  bool stop_ = false;
};

size_t alignUp(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

struct SpzB200Context {
  int device = 0;
  int smCount = 0;
  int packMode = spzb200::kPackAlu;
  bool cvtPackOk = false;  // the init-time probe of cvt.pack.sat.u8.s32 agreed with the ALU packer
  bool forceGeneric = false;
  bool pooled = false;  // owned by the process-wide pool (spzb200_acquire): released, never destroyed by callers
  int ctasPerSm = 0;
  int bounceMode = 1;     // pageable planes: 0 never bounce, 1 bounce large calls (see bounceMinBytes), 2 always
  size_t bounceMinBytes = (size_t)4 << 20;  // pack / unpack ms, bounced vs direct: 20K SH3 gaussians (6 MB) 0.45 / 0.55 vs 0.5 / 0.6, 60K 0.9 / 0.85 vs 1.2 / 1.4, 100K 0.9 / 1.0 vs 2.0 / 2.1 (profiles/r2_small_api_staging.txt); the one-time pinned allocation (~1 ms per MB) is small next to CUDA initialisation
  int encodeBulk = 1;  // planar encoder through the bulk-copy per-gaussian kernel: 1 = where faster (default); SPZB200_ENCODE=bulk: 2, =tiles: 0
  int decodePerGaussian = 1;  // SPZB200_DECODE=pergaussian: 2 (also SH-less clouds); =bulk / =direct: 0 (tile kernels only)
  bool plyMapped = false;  // SPZB200_PLY=mapped: canonical-layout PLY kernels off (column-map kernels for everything)
  bool decodeBulk = true;  // SH plane of the decoder staged with bulk async copies (SPZB200_DECODE=direct: registers)
  int smallTilesEncode = 2, smallTilesDecode = 0;  // 128-thread tile geometry (SH degree 0 - 2): encoder always, decoder never; SPZB200_TILE=128 / 320 set both, =auto the size rule
  bool pdl = true;       // SPZB200_PDL=0: plain stream-ordered launches (A/B timing)
  bool foldRest = true;  // SPZB200_REST=separate: the sub-tile remainder as a launch of its own (A/B timing)
  bool flatGrid = true;  // one CTA per tile: the block scheduler keeps the tile frontier compact
  bool adaptiveChunks = true;             // SPZB200_CHUNK_POINTS / spzb200_set_chunk_points pin the range size instead
  long long chunkPoints = 1 << 21;        // pinned / registered host planes: copied straight from the caller
  long long pageableChunkPoints = 1 << 18;  // pageable planes: bounced through pinned buffers of this many points
  int copyThreads = 0;                      // 0 = auto (3/4 of the hardware threads, at most 16)
  CopyPool *pool = nullptr;
  long long kernelLaunches = 0;
  float hThr[256];
  float hLut[256];
  float *dThr = nullptr;
  float *dLut = nullptr;
  Stage stage[kStages];
  // batched per-gaussian access (spzb200_unpack_*_host): two slots of pinned + device staging
  struct GatherSlot {
    uint8_t *hIn = nullptr;   // pinned, cap * 65 bytes
    float *hOut = nullptr;    // pinned, cap * 59 floats
    uint8_t *dIn = nullptr;
    float *dOut = nullptr;
    size_t cap = 0;           // records
    cudaEvent_t done = nullptr;
  } gather[2];
};

namespace {

int validDegree(int d) { return d >= 0 && d <= 3; }

int checkCloud(const SpzB200Cloud *c, const char *who) {
  if (!c) return fail(SPZB200_ERR_INVALID, "%s: null cloud view", who);
  if (c->num_points < 0) return fail(SPZB200_ERR_INVALID, "%s: num_points < 0", who);
  if (!validDegree(c->sh_degree)) return fail(SPZB200_ERR_INVALID, "%s: sh_degree %d not in 0..3", who, c->sh_degree);
  if (c->num_points > 0) {
    if (!c->positions || !c->scales || !c->rotations || !c->alphas || !c->colors)
      return fail(SPZB200_ERR_INVALID, "%s: null plane pointer", who);
    if (c->sh_degree > 0 && !c->sh) return fail(SPZB200_ERR_INVALID, "%s: null sh plane", who);
  }
  return SPZB200_OK;
}

int checkPacked(const SpzB200Packed *p, const char *who, bool needVersion) {
  if (!p) return fail(SPZB200_ERR_INVALID, "%s: null packed view", who);
  if (p->num_points < 0) return fail(SPZB200_ERR_INVALID, "%s: num_points < 0", who);
  if (!validDegree(p->sh_degree)) return fail(SPZB200_ERR_INVALID, "%s: sh_degree %d not in 0..3", who, p->sh_degree);
  if (needVersion && (p->version < 1 || p->version > SPZB200_STREAM_HALF_POSITIONS_SMALLEST_THREE))
    return fail(SPZB200_ERR_INVALID, "%s: version %d not in 1..4", who, p->version);
  if (p->num_points > 0) {
    if (!p->positions || !p->scales || !p->rotations || !p->alphas || !p->colors)
      return fail(SPZB200_ERR_INVALID, "%s: null plane pointer", who);
    if (p->sh_degree > 0 && !p->sh) return fail(SPZB200_ERR_INVALID, "%s: null sh plane", who);
  }
  return SPZB200_OK;
}

// (float)(1.0 / (1 << fractionalBits)), load-spz.cc:495.  The shift count is taken modulo 32, which
// is what the reference's x86 build does for header bytes >= 32.
float positionScaleFor(int fractionalBits) {
  const int32_t one = (int32_t)(1u << (fractionalBits & 31));
  return (float)(1.0 / one);
}

spzb200::EncodeArgs makeEncodeArgs(const SpzB200Context *ctx, const SpzB200Cloud &in,
                                   const SpzB200Packed &out, int32_t from) {
  spzb200::EncodeArgs a;
  a.positions = in.positions; a.scales = in.scales; a.rotations = in.rotations;
  a.alphas = in.alphas; a.colors = in.colors; a.sh = in.sh;
  a.oPositions = out.positions; a.oScales = out.scales; a.oRotations = out.rotations;
  a.oAlphas = out.alphas; a.oColors = out.colors; a.oSh = out.sh;
  a.n = in.num_points;
  a.shDim = shDimOf(in.sh_degree);
  a.version = out.version == 2 ? 2 : 3;
  const spzb200::m::FlipBits f = spzb200::m::make_flip_bits(from, SPZB200_COORD_RUB);
  a.flipP = f.p; a.flipQ = f.q; a.flipSh = f.sh;
  a.alphaThresholds = ctx->dThr;
  return a;
}

spzb200::DecodeArgs makeDecodeArgs(const SpzB200Context *ctx, const SpzB200Packed &in,
                                   const SpzB200Cloud &out, int32_t to) {
  spzb200::DecodeArgs a;
  a.positions = in.positions; a.scales = in.scales; a.rotations = in.rotations;
  a.alphas = in.alphas; a.colors = in.colors; a.sh = in.sh;
  a.oPositions = out.positions; a.oScales = out.scales; a.oRotations = out.rotations;
  a.oAlphas = out.alphas; a.oColors = out.colors; a.oSh = out.sh;
  a.n = in.num_points;
  a.shDim = shDimOf(in.sh_degree);
  a.version = in.version;
  a.positionScale = positionScaleFor(in.fractional_bits);
  const spzb200::m::FlipBits f = spzb200::m::make_flip_bits(SPZB200_COORD_RUB, to);
  a.flipP = f.p; a.flipQ = f.q; a.flipSh = f.sh;
  a.tables = ctx->dLut;
  return a;
}

spzb200::LaunchPlan planOf(const SpzB200Context *ctx) {
  spzb200::LaunchPlan p;
  p.smCount = ctx->smCount;
  p.packMode = ctx->packMode;
  p.forceGeneric = ctx->forceGeneric;
  p.ctasPerSm = ctx->ctasPerSm;
  p.flatGrid = ctx->flatGrid;
  p.decodeBulk = ctx->decodeBulk;
  p.plyMapped = ctx->plyMapped;
  p.foldRest = ctx->foldRest;
  p.pdl = ctx->pdl;
  p.smallTilesEncode = ctx->smallTilesEncode;
  p.smallTilesDecode = ctx->smallTilesDecode;
  p.decodePerGaussian = ctx->decodePerGaussian;
  p.encodeBulk = ctx->encodeBulk;
  return p;
}

// bytes per gaussian of each plane, in the struct order positions, scales, rotations, alphas,
// colors, sh
void floatPlaneBytes(int shDim, size_t b[6]) {
  b[0] = 12; b[1] = 12; b[2] = 16; b[3] = 4; b[4] = 12; b[5] = (size_t)12 * shDim;
}
void bytePlaneBytes(int shDim, int version, size_t b[6]) {
  b[0] = (version == 1 || version == 4) ? 6 : 9; b[1] = 3; b[2] = version >= 3 ? 4 : 3; b[3] = 1; b[4] = 3;
  b[5] = (size_t)3 * shDim;
}

int ensureStage(Stage &s, size_t inBytes_, size_t outBytes_) {
  if (s.dInCap < inBytes_) {
    if (s.dIn) cudaFree(s.dIn);
    s.dIn = nullptr; s.dInCap = 0;
    CU(cudaMalloc(&s.dIn, inBytes_));
    s.dInCap = inBytes_;
  }
  if (s.dOutCap < outBytes_) {
    if (s.dOut) cudaFree(s.dOut);
    s.dOut = nullptr; s.dOutCap = 0;
    CU(cudaMalloc(&s.dOut, outBytes_));
    s.dOutCap = outBytes_;
  }
  return SPZB200_OK;
}

// Pinned bounce buffers (cudaHostAlloc: ~1 GB/s on these VMs, i.e. 0.1-0.4 s for the 3 x 79 MB of a first bounced call; an mmap +
// MADV_HUGEPAGE + cudaHostRegister variant measured no faster -- commit 116c183, profiles/r2_tuning_notes.txt section 9).
int ensureBounce(uint8_t *&buf, size_t &cap, size_t bytes) {
  if (cap >= bytes) return SPZB200_OK;
  if (buf) cudaFreeHost(buf);
  buf = nullptr; cap = 0;
  CU(cudaHostAlloc(&buf, bytes, cudaHostAllocDefault));
  cap = bytes;
  return SPZB200_OK;
}

double nowMs() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// true when cudaMemcpyAsync from/to p would be staged by the driver (plain malloc'd memory)
bool isPageable(const void *p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

// A set of per-gaussian planes on the host or the device: pointer + bytes per gaussian each.
struct PlaneSet {
  int count = 0;
  uint8_t *ptr[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  size_t per[6] = {0, 0, 0, 0, 0, 0};
  size_t bytesPerGaussian() const {
    size_t t = 0;
    for (int i = 0; i < count; i++) t += per[i];
    return t;
  }
};

// `count` 256-byte-aligned sub-buffers for `points` gaussians inside one allocation
size_t carveSet(uint8_t *base, const PlaneSet &set, long long points, uint8_t *out[6]) {
  size_t off = 0;
  for (int i = 0; i < set.count; i++) {
    out[i] = base ? base + off : nullptr;
    off += alignUp(set.per[i] * (size_t)points, 256);
  }
  return off;
}

// The chunked H2D || kernel || D2H pipeline behind every *_host entry point.
//
// The n gaussians are cut into contiguous point ranges (multiples of `granule`, the kernel tile).
// Range c uses stage c % kStages: its own stream, device staging buffers and events, so the copy-in
// of one range overlaps the kernel and the copy-out of its predecessors.  Pinned (or registered)
// caller memory is copied directly (runPinnedStages).  Pageable caller memory -- what std::vector hands
// the C++ API -- would make every cudaMemcpyAsync a synchronous, driver-staged ~11 GB/s copy; instead the
// ranges are bounced through pinned buffers owned by the stage (runBouncedStages).
// launch(dIn, dOut, points, stream, &launches) queues the kernel(s) for one range.
struct PipelinePlan {
  long long n = 0, chunk = 0, numChunks = 0;
  bool bounceIn = false, bounceOut = false;
};

template <class Launch>
int runPinnedStages(SpzB200Context *ctx, const PlaneSet &in, const PlaneSet &out, const PipelinePlan &pp, Launch &&launch, SpzB200Timings &tm) {
  const long long n = pp.n, chunk = pp.chunk, numChunks = pp.numChunks;
  // Completes the range that last used `st`: waits for its copy-out and books its timings.
  auto finish = [&](Stage &st) -> int {
    CU(cudaEventSynchronize(st.ev[3]));
    float ms;
    CU(cudaEventElapsedTime(&ms, st.ev[0], st.ev[1])); tm.h2d_ms += ms;
    CU(cudaEventElapsedTime(&ms, st.ev[1], st.ev[2])); tm.kernel_ms += ms;
    CU(cudaEventElapsedTime(&ms, st.ev[2], st.ev[3])); tm.d2h_ms += ms;
    return SPZB200_OK;
  };
  for (long long c = 0; c < numChunks; c++) {
    Stage &st = ctx->stage[c % kStages];
    const long long a = c * chunk, b = std::min(n, a + chunk), pts = b - a;
    if (c >= kStages) {
      int rc = finish(st);
      if (rc != SPZB200_OK) return rc;
    }
    uint8_t *dIn[6], *dOut[6];
    carveSet(st.dIn, in, chunk, dIn);
    carveSet(st.dOut, out, chunk, dOut);
    CU(cudaEventRecord(st.ev[0], st.stream));
    for (int i = 0; i < in.count; i++) {
      const size_t bytes = in.per[i] * (size_t)pts;
      if (bytes) CU(cudaMemcpyAsync(dIn[i], in.ptr[i] + in.per[i] * (size_t)a, bytes, cudaMemcpyHostToDevice, st.stream));
      tm.h2d_bytes += (int64_t)bytes;
    }
    CU(cudaEventRecord(st.ev[1], st.stream));
    int launches = 0;
    CU(launch(dIn, dOut, pts, st.stream, &launches));
    ctx->kernelLaunches += launches;
    tm.kernel_launches += launches;
    CU(cudaEventRecord(st.ev[2], st.stream));
    for (int i = 0; i < out.count; i++) {
      const size_t bytes = out.per[i] * (size_t)pts;
      if (bytes) CU(cudaMemcpyAsync(out.ptr[i] + out.per[i] * (size_t)a, dOut[i], bytes, cudaMemcpyDeviceToHost, st.stream));
      tm.d2h_bytes += (int64_t)bytes;
    }
    CU(cudaEventRecord(st.ev[3], st.stream));
  }
  // drain the ranges still in flight, oldest first
  for (long long c = std::max<long long>(0, numChunks - kStages); c < numChunks; c++) {
    int rc = finish(ctx->stage[c % kStages]);
    if (rc != SPZB200_OK) return rc;
  }
  return SPZB200_OK;
}

// Pageable planes.  The calling thread only coordinates; the copy pool moves the bytes, in pieces of <= 2 MiB:
//   up    a worker copies a piece of the caller's plane into the stage's pinned buffer (non-temporal stores) and queues
//         that piece's H2D itself, on the stage's stream -- the DMA of a range starts when its first piece has landed,
//         not when its last has, and pieces of the next range are copied while this one's are on the link;
//   down  every D2H piece is followed by an event; a worker waits for a piece's event and copies it out to the caller's
//         plane while later pieces are still on the link.  The down tasks of range c are queued one range late (their
//         DMA has had a range's time to land, so workers rarely sleep on an event), and a task whose piece has not landed
//         yet steps aside for queued up tasks.
// Input and output directions therefore copy concurrently (round 1/2a: one after the other on the calling thread --
// 10M SH3 pack 100 ms, unpack 124 ms; scripts/bounce_probe.cu has the two shapes bare).  Reuse of a stage waits until
// its previous range has been copied out completely, which also covers its pinned input buffer (that range's kernel
// ran after its H2D pieces, and its D2H pieces after the kernel).
template <class Launch>
int runBouncedStages(SpzB200Context *ctx, const PlaneSet &in, const PlaneSet &out, const PipelinePlan &pp, Launch &&launch, SpzB200Timings &tm) {
  constexpr size_t kPiece = (size_t)2 << 20;
  const long long n = pp.n, chunk = pp.chunk, numChunks = pp.numChunks;
  const bool bounceIn = pp.bounceIn, bounceOut = pp.bounceOut;
  CopyPool &pool = *ctx->pool;
  struct DownPiece { uint8_t *dst; const uint8_t *src; size_t bytes; cudaEvent_t landed; };
  struct Range {
    std::atomic<int> upLeft{0}, downLeft{0};
    std::vector<DownPiece> down;
    bool downQueued = false, launched = false;
  };
  std::unique_ptr<Range[]> ranges(new Range[(size_t)numChunks]);
  std::atomic<int> firstError{(int)cudaSuccess};
  const int device = ctx->device;

  auto queueDown = [&](long long c) {
    Range &r = ranges[(size_t)c];
    if (r.downQueued || !r.launched) return;
    std::vector<CopyPool::Task> tasks;
    tasks.reserve(r.down.size());
    for (const DownPiece &d : r.down) {
      // std::function needs a copyable closure; the task re-queues a copy of itself when it steps aside
      struct DownTask {
        DownPiece d; Range *r; CopyPool *pool; std::atomic<int> *err; int device; int asides;
        void operator()() const {
          cudaSetDevice(device);
          cudaError_t e = cudaEventQuery(d.landed);
          if (e == cudaErrorNotReady) {
            if (asides < 3 && pool->othersQueued()) {  // bounded: not-ready pieces must not chase each other round the queue
              DownTask later = *this;
              later.asides++;
              pool->resubmit(CopyPool::Task(later));
              return;
            }
            e = cudaEventSynchronize(d.landed);
          }
          if (e == cudaSuccess) bounceCopy(d.dst, d.src, d.bytes);
          else {
            int expected = (int)cudaSuccess;
            err->compare_exchange_strong(expected, (int)e);
          }
          r->downLeft.fetch_sub(1);
          pool->progressed();
        }
      };
      tasks.emplace_back(DownTask{d, &r, &pool, &firstError, device, 0});
    }
    pool.submit(std::move(tasks));  // may throw (out of memory): nothing queued then, and downQueued stays false
    r.downQueued = true;
  };
  // host time of the coordinator inside the pool (helping with / waiting for copies)
  auto helpUntil = [&](std::atomic<int> &counter) {
    const double t0 = nowMs();
    pool.helpUntil([&] { return counter.load() == 0; });
    tm.host_copy_ms += nowMs() - t0;
  };
  // everything queued so far must have run before the caller's planes and `ranges` go away
  auto settle = [&](long long upTo) {
    for (long long c = 0; c < upTo; c++) {
      Range &r = ranges[(size_t)c];
      helpUntil(r.upLeft);
      if (r.downQueued) helpUntil(r.downLeft);
    }
  };
  auto finish = [&](Stage &st, long long c) -> int {
    if (bounceOut) {
      queueDown(c);
      helpUntil(ranges[(size_t)c].downLeft);
    }
    CU(cudaEventSynchronize(st.ev[3]));
    float ms;
    CU(cudaEventElapsedTime(&ms, st.ev[0], st.ev[1])); tm.h2d_ms += ms;
    CU(cudaEventElapsedTime(&ms, st.ev[1], st.ev[2])); tm.kernel_ms += ms;
    CU(cudaEventElapsedTime(&ms, st.ev[2], st.ev[3])); tm.d2h_ms += ms;
    if (firstError.load() != (int)cudaSuccess) return cudaFail((cudaError_t)firstError.load(), "bounced copy");
    return SPZB200_OK;
  };

  long long issued = 0;  // ranges whose tasks may be in the pool
  // A range goes through the coordinator twice.  begin(c): its stage is free (the range that used it is copied out),
  // its up tasks go to the pool.  launch(c), one iteration later: all its pieces are on the stream -> kernel, D2H
  // pieces with their events.  So while the coordinator does the serial part of range c - 1 (a few dozen API calls),
  // the pool already holds the pieces of range c: the workers never run dry between ranges.
  auto begin = [&](long long c) -> int {
    Stage &st = ctx->stage[c % kStages];
    Range &r = ranges[(size_t)c];
    const long long a = c * chunk, pts = std::min(n, a + chunk) - a;
    if (c >= kStages) {
      int rc = finish(st, c - kStages);
      if (rc != SPZB200_OK) return rc;
    }
    // an older range's D2H has had an iteration on the link: its pieces go out now, ahead of this range's up tasks
    if (bounceOut && c >= kStages - 1 && kStages > 1) queueDown(c - (kStages - 1));
    uint8_t *dIn[6], *hi[6];
    carveSet(st.dIn, in, chunk, dIn);
    issued = c + 1;
    CU(cudaEventRecord(st.ev[0], st.stream));
    if (bounceIn) {
      carveSet(st.hIn, in, chunk, hi);
      std::vector<CopyPool::Task> tasks;
      for (int i = 0; i < in.count; i++) {
        const size_t bytes = in.per[i] * (size_t)pts;
        const uint8_t *src = in.ptr[i] + in.per[i] * (size_t)a;
        tm.h2d_bytes += (int64_t)bytes;
        for (size_t off = 0; off < bytes; off += kPiece) {
          const size_t len = std::min(kPiece, bytes - off);
          uint8_t *pinned = hi[i] + off, *dev = dIn[i] + off;
          const uint8_t *from = src + off;
          cudaStream_t stream = st.stream;
          Range *rp = &r;
          CopyPool *pl = &pool;
          std::atomic<int> *err = &firstError;
          tasks.emplace_back([=] {
            bounceCopy(pinned, from, len);
            cudaSetDevice(device);
            const cudaError_t e = cudaMemcpyAsync(dev, pinned, len, cudaMemcpyHostToDevice, stream);
            if (e != cudaSuccess) {
              int expected = (int)cudaSuccess;
              err->compare_exchange_strong(expected, (int)e);
            }
            rp->upLeft.fetch_sub(1);
            pl->progressed();
          });
        }
      }
      r.upLeft.store((int)tasks.size());
      try {
        pool.submit(std::move(tasks));
      } catch (...) {
        r.upLeft.store(0);  // nothing was queued
        throw;
      }
    } else {
      for (int i = 0; i < in.count; i++) {
        const size_t bytes = in.per[i] * (size_t)pts;
        if (bytes) CU(cudaMemcpyAsync(dIn[i], in.ptr[i] + in.per[i] * (size_t)a, bytes, cudaMemcpyHostToDevice, st.stream));
        tm.h2d_bytes += (int64_t)bytes;
      }
    }
    return SPZB200_OK;
  };
  auto launchRange = [&](long long c) -> int {
    Stage &st = ctx->stage[c % kStages];
    Range &r = ranges[(size_t)c];
    const long long a = c * chunk, pts = std::min(n, a + chunk) - a;
    uint8_t *dIn[6], *dOut[6], *ho[6];
    carveSet(st.dIn, in, chunk, dIn);
    carveSet(st.dOut, out, chunk, dOut);
    helpUntil(r.upLeft);
    if (firstError.load() != (int)cudaSuccess) return cudaFail((cudaError_t)firstError.load(), "bounced copy");
    CU(cudaEventRecord(st.ev[1], st.stream));
    int launches = 0;
    CU(launch(dIn, dOut, pts, st.stream, &launches));
    ctx->kernelLaunches += launches;
    tm.kernel_launches += launches;
    CU(cudaEventRecord(st.ev[2], st.stream));
    if (bounceOut) {
      carveSet(st.hOut, out, chunk, ho);
      size_t pieces = 0;
      for (int i = 0; i < out.count; i++) pieces += (out.per[i] * (size_t)pts + kPiece - 1) / kPiece;
      while (st.pieceEv.size() < pieces) {
        cudaEvent_t e;
        CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        st.pieceEv.push_back(e);
      }
      size_t k = 0;
      r.down.reserve(pieces);
      for (int i = 0; i < out.count; i++) {
        const size_t bytes = out.per[i] * (size_t)pts;
        tm.d2h_bytes += (int64_t)bytes;
        for (size_t off = 0; off < bytes; off += kPiece, k++) {
          const size_t len = std::min(kPiece, bytes - off);
          CU(cudaMemcpyAsync(ho[i] + off, dOut[i] + off, len, cudaMemcpyDeviceToHost, st.stream));
          CU(cudaEventRecord(st.pieceEv[k], st.stream));
          r.down.push_back({out.ptr[i] + out.per[i] * (size_t)a + off, ho[i] + off, len, st.pieceEv[k]});
        }
      }
      r.downLeft.store((int)r.down.size());
    } else {
      for (int i = 0; i < out.count; i++) {
        const size_t bytes = out.per[i] * (size_t)pts;
        if (bytes) CU(cudaMemcpyAsync(out.ptr[i] + out.per[i] * (size_t)a, dOut[i], bytes, cudaMemcpyDeviceToHost, st.stream));
        tm.d2h_bytes += (int64_t)bytes;
      }
    }
    CU(cudaEventRecord(st.ev[3], st.stream));
    r.launched = true;
    return SPZB200_OK;
  };
  auto body = [&]() -> int {
    for (long long c = 0; c <= numChunks; c++) {
      if (c < numChunks) {
        int rc = begin(c);
        if (rc != SPZB200_OK) return rc;
      }
      if (c >= 1) {
        int rc = launchRange(c - 1);
        if (rc != SPZB200_OK) return rc;
      }
    }
    for (long long c = std::max<long long>(0, numChunks - kStages); c < numChunks; c++) {
      int rc = finish(ctx->stage[c % kStages], c);
      if (rc != SPZB200_OK) return rc;
    }
    return SPZB200_OK;
  };
  int rc;
  try {
    rc = body();
  } catch (const std::exception &e) {  // allocation failure while building a range's task list: a failed call, after the tasks already queued have run out
    rc = fail(SPZB200_ERR_NOMEM, "host pipeline: %s", e.what());
  }
  if (rc != SPZB200_OK) {
    // tasks still queued hold pointers into the caller's planes, the stage buffers and `ranges`: let them run out
    // (a down task of a range whose D2H never got queued is never submitted; its counter is not waited on)
    const std::string first = tlsError;
    settle(issued);
    tlsError = first;
  }
  return rc;
}

template <class Launch>
int runPipelineStages(SpzB200Context *ctx, const PlaneSet &in, const PlaneSet &out, long long n, long long granule,
                      Launch &&launch, SpzB200Timings *timings) {
  const double w0 = nowMs();
  CU(cudaSetDevice(ctx->device));
  // Bouncing costs a one-time pinned allocation per context (~1 GB/s on a VM), so small one-shot
  // calls are cheaper through the driver's own staging; once the buffers exist they are always used.
  const size_t callBytes = (size_t)n * (in.bytesPerGaussian() + out.bytesPerGaussian());
  const bool wantBounce = ctx->bounceMode == 2 ||
                          (ctx->bounceMode == 1 && (callBytes >= ctx->bounceMinBytes || ctx->stage[0].hIn || ctx->stage[0].hOut));
  PipelinePlan pp;
  pp.n = n;
  pp.bounceIn = n > 0 && wantBounce && isPageable(in.ptr[0]);
  pp.bounceOut = n > 0 && wantBounce && isPageable(out.ptr[0]);
  const bool bounced = pp.bounceIn || pp.bounceOut;
  long long want = bounced ? ctx->pageableChunkPoints : ctx->chunkPoints;
  // Pinned planes: 2M-point ranges keep the copy engines in long transfers, but a cloud of only a few such ranges
  // spends a visible part of the call filling and draining the three-stage pipeline (10M points = 5 ranges: 0.84 of
  // the link; in ~12 ranges: profiles/r2_tuning_notes.txt).  So mid-sized clouds are cut into about a dozen ranges,
  // never below 256K points.
  if (!bounced && ctx->adaptiveChunks) want = std::min(want, std::max<long long>(1 << 18, (n + 11) / 12));
  long long chunk = std::max<long long>(granule, (want + granule - 1) / granule * granule);
  if (chunk > n) chunk = std::max<long long>(n, 1);
  pp.chunk = chunk;
  pp.numChunks = n == 0 ? 0 : (n + chunk - 1) / chunk;
  const int stages = (int)std::min<long long>(kStages, pp.numChunks);

  SpzB200Timings tm;
  std::memset(&tm, 0, sizeof tm);
  tm.staged = (pp.bounceIn ? 1 : 0) | (pp.bounceOut ? 2 : 0);
  if (pp.numChunks > 0) {
    uint8_t *unused[6];
    const size_t inBytes = carveSet(nullptr, in, chunk, unused);
    const size_t outBytes = carveSet(nullptr, out, chunk, unused);
    for (int s = 0; s < stages; s++) {
      Stage &st = ctx->stage[s];
      int rc = ensureStage(st, inBytes, outBytes);
      if (rc == SPZB200_OK && pp.bounceIn) rc = ensureBounce(st.hIn, st.hInCap, inBytes);
      if (rc == SPZB200_OK && pp.bounceOut) rc = ensureBounce(st.hOut, st.hOutCap, outBytes);
      if (rc != SPZB200_OK) return rc;
    }
    if (bounced && !ctx->pool) {
      // 10M SH3 through the C++ API on a 16-thread host, pack / unpack ms: 4 threads 117 / 187, 8: 70 / 110, 12: 62 / 92, 16: 62 / 86
      const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
      int t = ctx->copyThreads > 0 ? ctx->copyThreads : (int)std::min<unsigned>(16, std::max(1u, hw * 3 / 4));
      // a *_host_multi call runs one pipeline per device at once: they share the host's threads (and its memory bandwidth)
      if (ctx->copyThreads <= 0 && tlsShardCount > 1) t = std::max(2, t / tlsShardCount);
      ctx->pool = new CopyPool(std::max(0, t - 1));  // the calling thread copies too while it waits
    }
    const int rc = bounced ? runBouncedStages(ctx, in, out, pp, launch, tm) : runPinnedStages(ctx, in, out, pp, launch, tm);
    if (rc != SPZB200_OK) return rc;
  }
  tm.chunks = (int32_t)pp.numChunks;
  tm.wall_ms = nowMs() - w0;
  if (timings) *timings = tm;
  return SPZB200_OK;
}

// On failure copies of earlier ranges may still be in flight on the stage streams, reading or writing
// the caller's planes and the bounce buffers; the caller is about to free or reuse both, so the
// streams are drained first (secondary errors of that drain are dropped, the first message is kept).
template <class Launch>
int runPipeline(SpzB200Context *ctx, const PlaneSet &in, const PlaneSet &out, long long n, long long granule,
                Launch &&launch, SpzB200Timings *timings) {
  int rc;
  try {
    rc = runPipelineStages(ctx, in, out, n, granule, launch, timings);
  } catch (const std::exception &e) {  // nothing may cross the C boundary
    rc = fail(SPZB200_ERR_NOMEM, "host pipeline: %s", e.what());
  }
  if (rc != SPZB200_OK) {
    const std::string first = tlsError;
    for (int s = 0; s < kStages; s++)
      if (ctx->stage[s].stream) (void)cudaStreamSynchronize(ctx->stage[s].stream);
    (void)cudaGetLastError();
    tlsError = first;
  }
  return rc;
}

PlaneSet cloudPlaneSet(const SpzB200Cloud &c) {
  PlaneSet s;
  s.count = 6;
  float *const p[6] = {c.positions, c.scales, c.rotations, c.alphas, c.colors, c.sh};
  floatPlaneBytes(shDimOf(c.sh_degree), s.per);
  for (int i = 0; i < 6; i++) s.ptr[i] = reinterpret_cast<uint8_t *>(p[i]);
  return s;
}

PlaneSet packedPlaneSet(const SpzB200Packed &p, int version) {
  PlaneSet s;
  s.count = 6;
  uint8_t *const q[6] = {p.positions, p.scales, p.rotations, p.alphas, p.colors, p.sh};
  bytePlaneBytes(shDimOf(p.sh_degree), version, s.per);
  for (int i = 0; i < 6; i++) s.ptr[i] = q[i];
  return s;
}

SpzB200Cloud cloudOn(const SpzB200Cloud &like, uint8_t *const d[6], long long pts) {
  SpzB200Cloud c = like;
  c.num_points = pts;
  c.positions = (float *)d[0]; c.scales = (float *)d[1]; c.rotations = (float *)d[2];
  c.alphas = (float *)d[3]; c.colors = (float *)d[4]; c.sh = (float *)d[5];
  return c;
}

SpzB200Packed packedOn(const SpzB200Packed &like, uint8_t *const d[6], long long pts, int version) {
  SpzB200Packed p = like;
  p.num_points = pts;
  p.version = version;
  p.positions = d[0]; p.scales = d[1]; p.rotations = d[2]; p.alphas = d[3]; p.colors = d[4]; p.sh = d[5];
  return p;
}

// encode_host / decode_host: float planes in and byte planes out, or the reverse.
int runHostPipeline(SpzB200Context *ctx, bool isEncode, const SpzB200Cloud &cloud,
                    const SpzB200Packed &packed, int32_t coord, SpzB200Timings *timings) {
  const int version = isEncode ? (packed.version == 2 ? 2 : 3) : packed.version;
  const PlaneSet fl = cloudPlaneSet(cloud), by = packedPlaneSet(packed, version);
  const long long granule = spzb200::tileGaussians(shDimOf(cloud.sh_degree));
  const spzb200::LaunchPlan plan = planOf(ctx);
  if (isEncode) {
    return runPipeline(ctx, fl, by, cloud.num_points, granule,
                       [&](uint8_t *const dIn[6], uint8_t *const dOut[6], long long pts, cudaStream_t s, int *launches) {
                         return spzb200::launchEncode(makeEncodeArgs(ctx, cloudOn(cloud, dIn, pts), packedOn(packed, dOut, pts, version), coord),
                                                      plan, s, launches);
                       }, timings);
  }
  return runPipeline(ctx, by, fl, cloud.num_points, granule,
                     [&](uint8_t *const dIn[6], uint8_t *const dOut[6], long long pts, cudaStream_t s, int *launches) {
                       return spzb200::launchDecode(makeDecodeArgs(ctx, packedOn(packed, dIn, pts, version), cloudOn(cloud, dOut, pts), coord),
                                                    plan, s, launches);
                     }, timings);
}

// Process-wide pool of contexts, one free list per device (spzb200_acquire / spzb200_release).
// A context owns device staging buffers, pinned bounce buffers, streams and a copy pool -- building
// them costs more than a small cloud's whole encode -- so the C++ API and the multi-GPU entry points
// lease one per call instead of keeping one per host thread: a server that packs from short-lived
// threads pays the set-up once per process, not once per request.  A lease is exclusive.  At most
// `maxLive` contexts exist per device (SPZ_B200_MAX_CONTEXTS, default 2: one H2D-heavy encode and one
// D2H-heavy decode keep both directions of the PCIe link busy; more callers only queue on the link, and on
// the driver's staging of pageable copies); further callers wait for a release.  Never destroyed: no CUDA
// calls at exit.
struct ContextPool {
  struct PerDevice {
    std::vector<SpzB200Context *> idle;
    int live = 0;
  };
  std::mutex m;
  std::condition_variable cv;
  std::vector<std::pair<int32_t, PerDevice>> devs;
  int maxLive = 2;
  ContextPool() {
    if (const char *env = std::getenv("SPZ_B200_MAX_CONTEXTS")) maxLive = std::max(1, std::atoi(env));
  }
  PerDevice &of(int32_t device) {
    for (auto &d : devs)
      if (d.first == device) return d.second;
    devs.emplace_back(device, PerDevice());
    return devs.back().second;
  }
  int acquire(int32_t device, SpzB200Context **out) {
    *out = nullptr;
    {
      std::unique_lock<std::mutex> g(m);
      while (true) {
        PerDevice &d = of(device);
        if (!d.idle.empty()) {
          *out = d.idle.back();
          d.idle.pop_back();
          return SPZB200_OK;
        }
        if (d.live < maxLive) {
          d.live++;
          break;
        }
        cv.wait(g);
      }
    }
    const int rc = spzb200_create(device, out);  // outside the lock: other devices' callers do not wait for it
    if (rc != SPZB200_OK) {
      std::lock_guard<std::mutex> g(m);
      of(device).live--;
      cv.notify_all();
    } else {
      (*out)->pooled = true;
    }
    return rc;
  }
  void release(SpzB200Context *ctx) {
    // A context whose stream reports an error (a failed launch, a lost device) must not be handed to the next caller:
    // it is destroyed and its slot freed, so the next lease builds a fresh one (or fails with the real reason).
    const int32_t device = ctx->device;
    bool healthy = cudaSetDevice(device) == cudaSuccess;
    if (healthy) {
      const cudaError_t e = cudaStreamQuery(ctx->stage[0].stream);
      healthy = e == cudaSuccess || e == cudaErrorNotReady;
    }
    if (!healthy) {
      (void)cudaGetLastError();
      ctx->pooled = false;
      spzb200_destroy(ctx);
    }
    {
      std::lock_guard<std::mutex> g(m);
      if (healthy) of(device).idle.push_back(ctx);
      else of(device).live--;
    }
    cv.notify_all();
  }
};
ContextPool &contextPool() {
  static ContextPool *pool = new ContextPool;
  return *pool;
}

template <class Fn>
int runSharded(const int32_t *devices, int32_t numDevices, int64_t n, int32_t shDegree, Fn &&perShard,
               SpzB200Timings *timings) {
  if (!devices || numDevices <= 0) return fail(SPZB200_ERR_INVALID, "multi: no devices given");
  std::vector<int> rc(numDevices, SPZB200_OK);
  std::vector<std::string> msg(numDevices);
  std::vector<SpzB200Timings> tms(numDevices);
  std::vector<std::thread> threads;
  const double w0 = nowMs();
  auto shard = [&](int32_t i) {
      std::memset(&tms[i], 0, sizeof(SpzB200Timings));
      int64_t a = 0, b = 0;
      rc[i] = spzb200_shard_range(n, shDegree, numDevices, i, &a, &b);
      if (rc[i] == SPZB200_OK && b > a) {
        SpzB200Context *ctx = nullptr;
        rc[i] = contextPool().acquire(devices[i], &ctx);
        if (rc[i] == SPZB200_OK) {
          tlsShardCount = numDevices;
          rc[i] = perShard(ctx, a, b, &tms[i]);
          tlsShardCount = 1;
          if (rc[i] != SPZB200_OK) msg[i] = spzb200_last_error();
          contextPool().release(ctx);
        }
      }
      if (rc[i] != SPZB200_OK && msg[i].empty()) msg[i] = spzb200_last_error();
  };
  for (int32_t i = 0; i < numDevices; i++) {
    try {
      threads.emplace_back(shard, i);
    } catch (const std::exception &) {
      shard(i);  // no thread to be had: this device's range runs on the calling thread
    }
  }
  for (auto &t : threads) t.join();
  for (int32_t i = 0; i < numDevices; i++)
    if (rc[i] != SPZB200_OK) return fail(rc[i], "device %d: %s", devices[i], msg[i].c_str());
  if (timings) {
    SpzB200Timings out;
    std::memset(&out, 0, sizeof out);
    for (auto &t : tms) {
      out.h2d_ms = std::max(out.h2d_ms, t.h2d_ms);
      out.kernel_ms = std::max(out.kernel_ms, t.kernel_ms);
      out.d2h_ms = std::max(out.d2h_ms, t.d2h_ms);
      out.h2d_bytes += t.h2d_bytes;
      out.d2h_bytes += t.d2h_bytes;
      out.kernel_launches += t.kernel_launches;
      out.chunks += t.chunks;
      out.host_copy_ms = std::max(out.host_copy_ms, t.host_copy_ms);
      out.staged |= t.staged;
    }
    out.wall_ms = nowMs() - w0;
    *timings = out;
  }
  return SPZB200_OK;
}

SpzB200Cloud sliceCloud(const SpzB200Cloud &c, int64_t a, int64_t b) {
  const int d = shDimOf(c.sh_degree);
  SpzB200Cloud s = c;
  s.num_points = b - a;
  s.positions = c.positions + 3 * a; s.scales = c.scales + 3 * a; s.rotations = c.rotations + 4 * a;
  s.alphas = c.alphas + a; s.colors = c.colors + 3 * a; s.sh = c.sh ? c.sh + (int64_t)3 * d * a : nullptr;
  return s;
}

SpzB200Packed slicePacked(const SpzB200Packed &p, int64_t a, int64_t b) {
  const int d = shDimOf(p.sh_degree);
  SpzB200Packed s = p;
  s.num_points = b - a;
  s.positions = p.positions + ((p.version == 1 || p.version == 4) ? 6 : 9) * a; s.scales = p.scales + 3 * a;
  s.rotations = p.rotations + (p.version >= 3 ? 4 : 3) * a; s.alphas = p.alphas + a;
  s.colors = p.colors + 3 * a; s.sh = p.sh ? p.sh + (int64_t)3 * d * a : nullptr;
  return s;
}

}  // namespace

extern "C" {

const char *spzb200_last_error(void) { return tlsError.c_str(); }
int32_t spzb200_version(void) { return SPZB200_VERSION; }

int spzb200_create(int32_t device, SpzB200Context **out) {
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_create: null out");
  *out = nullptr;
  // SPZB200_TRACE_INIT=1: one stderr line with where a context's creation time went (profiles/r2_cold_start.txt)
  const bool trace = std::getenv("SPZB200_TRACE_INIT") != nullptr;
  double tMark = nowMs();
  double tQuery = 0, tTables = 0, tAlloc = 0, tStreams = 0, tKernels = 0;
  auto lap = [&](double &slot) {
    const double now = nowMs();
    slot = now - tMark;
    tMark = now;
  };
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0)
    return fail(SPZB200_ERR_NO_DEVICE, "spzb200_create: no CUDA device (%s); this library has no CPU path",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (device < 0 || device >= count)
    return fail(SPZB200_ERR_NO_DEVICE, "spzb200_create: device %d out of range (0..%d)", device, count - 1);
  // (cudaGetDeviceProperties costs ~1 ms per call: it queries every property; the two attributes do not)
  int major = 0, sms = 0;
  CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (major != 10) {
    int minor = 0;
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device);
    return fail(SPZB200_ERR_NO_DEVICE, "spzb200_create: device %d is sm_%d%d; kernels are built for sm_100a only",
                device, major, minor);
  }
  CU(cudaSetDevice(device));
  CU(cudaFree(nullptr));  // forces the primary context, so the trace separates CUDA initialisation from ours
  lap(tQuery);
  const HostTables &tables = hostTables();
  if (!tables.ok) return fail(SPZB200_ERR_INVALID, "spzb200_create: %s", tables.why.c_str());
  SpzB200Context *ctx = new SpzB200Context;
  ctx->device = device;
  ctx->smCount = sms;
  std::memcpy(ctx->hThr, tables.thr, sizeof ctx->hThr);
  std::memcpy(ctx->hLut, tables.lut, sizeof ctx->hLut);
  lap(tTables);
  auto bail = [&](cudaError_t err, const char *what) {
    spzb200_destroy(ctx);
    return cudaFail(err, what);
  };
  // one allocation: [0, 256) thresholds, the decode tables, one scratch word for the probe
  if ((e = cudaMalloc(&ctx->dThr, (256 + spzb200::kDecodeTableFloats + 4) * sizeof(float))) != cudaSuccess) return bail(e, "cudaMalloc tables");
  ctx->dLut = ctx->dThr + 256;
  int *dScratch = reinterpret_cast<int *>(ctx->dLut + spzb200::kDecodeTableFloats);
  lap(tAlloc);
  for (int s = 0; s < kStages; s++) {
    if ((e = cudaStreamCreateWithFlags(&ctx->stage[s].stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    for (int k = 0; k < 4; k++)
      if ((e = cudaEventCreate(&ctx->stage[s].ev[k])) != cudaSuccess) return bail(e, "cudaEventCreate");
  }
  lap(tStreams);
  // The uploads ride on the stream the table kernels and the probe run on, and the probe ends with a
  // synchronize of that stream: everything is resident before spzb200_create returns.  (A blocking
  // cudaMemcpy on the legacy stream would not order against these non-blocking streams.)
  cudaStream_t s0 = ctx->stage[0].stream;
  if ((e = cudaMemcpyAsync(ctx->dThr, ctx->hThr, sizeof ctx->hThr, cudaMemcpyHostToDevice, s0)) != cudaSuccess) return bail(e, "table upload");
  if ((e = cudaMemcpyAsync(ctx->dLut, ctx->hLut, sizeof ctx->hLut, cudaMemcpyHostToDevice, s0)) != cudaSuccess) return bail(e, "table upload");
  if ((e = spzb200::buildDecodeTables(ctx->dLut, s0)) != cudaSuccess) return bail(e, "decode tables");
  int ok = 0;
  if ((e = spzb200::probePackCvt(s0, dScratch, &ok)) != cudaSuccess) return bail(e, "pack probe");
  if ((e = cudaStreamSynchronize(s0)) != cudaSuccess) return bail(e, "table upload");
  lap(tKernels);
  ctx->cvtPackOk = ok != 0;
  ctx->packMode = ok ? spzb200::kPackCvt : spzb200::kPackAlu;
  // development knobs (profiles/ records which settings the shipped defaults came from)
  if (const char *env = std::getenv("SPZB200_PACK")) {
    if (!std::strcmp(env, "alu")) ctx->packMode = spzb200::kPackAlu;
  }
  if (const char *env = std::getenv("SPZB200_CTAS_PER_SM")) ctx->ctasPerSm = std::atoi(env);
  if (const char *env = std::getenv("SPZB200_BOUNCE_MIN_MB")) ctx->bounceMinBytes = (size_t)std::atoll(env) << 20;
  if (const char *env = std::getenv("SPZB200_COPY_THREADS")) ctx->copyThreads = std::max(0, std::atoi(env));
  if (const char *env = std::getenv("SPZB200_PAGEABLE_CHUNK_POINTS")) {
    const long long v = std::atoll(env);
    if (v > 0) ctx->pageableChunkPoints = v;
  }
  if (const char *env = std::getenv("SPZB200_DECODE")) {
    ctx->decodeBulk = std::strcmp(env, "direct") != 0;
    ctx->decodePerGaussian = std::strcmp(env, "pergaussian") == 0 ? 2 : (std::strcmp(env, "bulk") == 0 || std::strcmp(env, "direct") == 0) ? 0 : 1;
  }
  if (const char *env = std::getenv("SPZB200_ENCODE")) ctx->encodeBulk = std::strcmp(env, "bulk") == 0 ? 2 : std::strcmp(env, "tiles") == 0 ? 0 : 1;
  if (const char *env = std::getenv("SPZB200_PLY")) ctx->plyMapped = std::strcmp(env, "mapped") == 0;
  if (const char *env = std::getenv("SPZB200_TILE"))
    ctx->smallTilesEncode = ctx->smallTilesDecode = std::strcmp(env, "320") == 0 ? 0 : std::strcmp(env, "128") == 0 ? 2 : 1;
  if (const char *env = std::getenv("SPZB200_PDL")) ctx->pdl = std::strcmp(env, "0") != 0;
  if (const char *env = std::getenv("SPZB200_REST")) ctx->foldRest = std::strcmp(env, "separate") != 0;
  if (const char *env = std::getenv("SPZB200_GRID")) ctx->flatGrid = std::strcmp(env, "persistent") != 0;
  if (const char *env = std::getenv("SPZB200_CHUNK_POINTS")) {
    const long long v = std::atoll(env);
    if (v > 0) {
      ctx->chunkPoints = v;
      ctx->adaptiveChunks = false;
    }
  }
  if (trace)
    fprintf(stderr, "[spz_b200 init] device %d: cuda init + device query %.2f ms, host tables %.2f ms, cudaMalloc %.2f ms, "
            "streams + events %.2f ms, table kernels + probe (first launch loads the module) %.2f ms\n",
            device, tQuery, tTables, tAlloc, tStreams, tKernels);
  *out = ctx;
  return SPZB200_OK;
}

int spzb200_acquire(int32_t device, SpzB200Context **out) {
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_acquire: null out");
  try {
    return contextPool().acquire(device, out);
  } catch (const std::exception &e) {
    *out = nullptr;
    return fail(SPZB200_ERR_NOMEM, "spzb200_acquire: %s", e.what());
  }
}

void spzb200_release(SpzB200Context *ctx) {
  if (!ctx) return;
  if (!ctx->pooled) {  // a context of spzb200_create: the caller owns it
    spzb200_destroy(ctx);
    return;
  }
  contextPool().release(ctx);
}

void spzb200_destroy(SpzB200Context *ctx) {
  if (!ctx) return;
  if (ctx->pooled) {  // leased contexts go back to the pool, whoever lets go of them
    contextPool().release(ctx);
    return;
  }
  cudaSetDevice(ctx->device);
  delete ctx->pool;
  for (int s = 0; s < kStages; s++) {
    Stage &st = ctx->stage[s];
    if (st.stream) cudaStreamSynchronize(st.stream);
    if (st.hIn) cudaFreeHost(st.hIn);
    if (st.hOut) cudaFreeHost(st.hOut);
    for (int k = 0; k < 4; k++) if (st.ev[k]) cudaEventDestroy(st.ev[k]);
    for (cudaEvent_t e : st.pieceEv) cudaEventDestroy(e);
    if (st.dIn) cudaFree(st.dIn);
    if (st.dOut) cudaFree(st.dOut);
    if (st.stream) cudaStreamDestroy(st.stream);
  }
  for (auto &g : ctx->gather) {
    if (g.hIn) cudaFreeHost(g.hIn);
    if (g.hOut) cudaFreeHost(g.hOut);
    if (g.dIn) cudaFree(g.dIn);
    if (g.dOut) cudaFree(g.dOut);
    if (g.done) cudaEventDestroy(g.done);
  }
  if (ctx->dThr) cudaFree(ctx->dThr);  // dLut lives in the same allocation
  delete ctx;
}

int spzb200_encode_device(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from,
                          SpzB200Packed *out, void *stream) {
  return spzb200_encode_device_as(ctx, in, from, SPZB200_STREAM_V3, out, stream);
}

int spzb200_encode_device_as(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from, int32_t stream_version,
                             SpzB200Packed *out, void *stream) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_encode_device: null context");
  if (stream_version != SPZB200_STREAM_V2 && stream_version != SPZB200_STREAM_V3)
    return fail(SPZB200_ERR_INVALID, "spzb200_encode_device: the encoder writes stream version 2 or 3, not %d", stream_version);
  int rc = checkCloud(in, "spzb200_encode_device");
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_encode_device: null out");
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  out->fractional_bits = 12;  // load-spz.cc:270
  out->version = stream_version;  // 3: load-spz.cc:133,272
  rc = checkPacked(out, "spzb200_encode_device", true);
  if (rc) return rc;
  if (from < 0 || from > 8) return fail(SPZB200_ERR_INVALID, "spzb200_encode_device: coordinate system %d", from);
  CU(cudaSetDevice(ctx->device));
  int launches = 0;
  CU(spzb200::launchEncode(makeEncodeArgs(ctx, *in, *out, from), planOf(ctx), (cudaStream_t)stream, &launches));
  ctx->kernelLaunches += launches;
  return SPZB200_OK;
}

int spzb200_decode_device(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to,
                          SpzB200Cloud *out, void *stream) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_decode_device: null context");
  int rc = checkPacked(in, "spzb200_decode_device", true);
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_decode_device: null out");
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  rc = checkCloud(out, "spzb200_decode_device");
  if (rc) return rc;
  if (to < 0 || to > 8) return fail(SPZB200_ERR_INVALID, "spzb200_decode_device: coordinate system %d", to);
  CU(cudaSetDevice(ctx->device));
  int launches = 0;
  CU(spzb200::launchDecode(makeDecodeArgs(ctx, *in, *out, to), planOf(ctx), (cudaStream_t)stream, &launches));
  ctx->kernelLaunches += launches;
  return SPZB200_OK;
}

namespace {
// An output plane may be its own input plane (in place).  Any other overlap of an output plane with an
// input or another output plane would make the result depend on the order the CTAs run in.
int checkQuantizeOverlap(const SpzB200Cloud &in, const SpzB200Cloud &out, const char *who) {
  size_t per[6];
  floatPlaneBytes(shDimOf(in.sh_degree), per);
  const float *ip[6] = {in.positions, in.scales, in.rotations, in.alphas, in.colors, in.sh};
  const float *op[6] = {out.positions, out.scales, out.rotations, out.alphas, out.colors, out.sh};
  auto overlap = [&](const float *a, size_t aBytes, const float *b, size_t bBytes) {
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + bBytes && y < x + aBytes;
  };
  for (int i = 0; i < 6; i++) {
    const size_t bi = per[i] * (size_t)out.num_points;
    if (bi == 0) continue;
    for (int j = 0; j < 6; j++) {
      const size_t bj = per[j] * (size_t)out.num_points;
      if (bj == 0) continue;
      if (overlap(op[i], bi, ip[j], bj) && !(i == j && op[i] == ip[j]))
        return fail(SPZB200_ERR_INVALID, "%s: output plane %d overlaps input plane %d other than exactly (in place)", who, i, j);
      if (j != i && overlap(op[i], bi, op[j], bj))
        return fail(SPZB200_ERR_INVALID, "%s: output planes %d and %d overlap", who, i, j);
    }
  }
  return SPZB200_OK;
}
}  // namespace

int spzb200_quantize_device(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from, int32_t to, int32_t version,
                            SpzB200Cloud *out, void *stream) {
  const char *who = "spzb200_quantize_device";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (version != SPZB200_STREAM_V2 && version != SPZB200_STREAM_V3)
    return fail(SPZB200_ERR_INVALID, "%s: the encoder writes stream version 2 or 3, not %d", who, version);
  int rc = checkCloud(in, who);
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "%s: null out", who);
  rc = checkCloud(out, who);
  if (rc) return rc;
  if (out->num_points != in->num_points || out->sh_degree != in->sh_degree)
    return fail(SPZB200_ERR_INVALID, "%s: out holds %lld points of SH degree %d, in %lld of degree %d", who, (long long)out->num_points,
                out->sh_degree, (long long)in->num_points, in->sh_degree);
  if (from < 0 || from > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, from);
  if (to < 0 || to > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, to);
  rc = checkQuantizeOverlap(*in, *out, who);
  if (rc) return rc;
  spzb200::QuantizeArgs a;
  a.positions = in->positions; a.scales = in->scales; a.rotations = in->rotations;
  a.alphas = in->alphas; a.colors = in->colors; a.sh = in->sh;
  a.oPositions = out->positions; a.oScales = out->scales; a.oRotations = out->rotations;
  a.oAlphas = out->alphas; a.oColors = out->colors; a.oSh = out->sh;
  a.n = in->num_points;
  a.shDim = shDimOf(in->sh_degree);
  a.version = version;
  const spzb200::m::FlipBits f = spzb200::m::make_flip_bits(from, SPZB200_COORD_RUB);
  a.flipP = f.p; a.flipQ = f.q; a.flipSh = f.sh;
  const spzb200::m::FlipBits g = spzb200::m::make_flip_bits(SPZB200_COORD_RUB, to);
  a.oFlipP = g.p; a.oFlipQ = g.q; a.oFlipSh = g.sh;
  a.alphaThresholds = ctx->dThr;
  a.tables = ctx->dLut;
  CU(cudaSetDevice(ctx->device));
  int launches = 0;
  CU(spzb200::launchQuantize(a, planOf(ctx), (cudaStream_t)stream, &launches));
  ctx->kernelLaunches += launches;
  return SPZB200_OK;
}

int spzb200_encode_host(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from,
                        SpzB200Packed *out, SpzB200Timings *timings) {
  return spzb200_encode_host_as(ctx, in, from, SPZB200_STREAM_V3, out, timings);
}

int spzb200_encode_host_as(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from, int32_t stream_version,
                           SpzB200Packed *out, SpzB200Timings *timings) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_encode_host: null context");
  if (stream_version != SPZB200_STREAM_V2 && stream_version != SPZB200_STREAM_V3)
    return fail(SPZB200_ERR_INVALID, "spzb200_encode_host: the encoder writes stream version 2 or 3, not %d", stream_version);
  int rc = checkCloud(in, "spzb200_encode_host");
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_encode_host: null out");
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  out->fractional_bits = 12;
  out->version = stream_version;
  rc = checkPacked(out, "spzb200_encode_host", true);
  if (rc) return rc;
  if (from < 0 || from > 8) return fail(SPZB200_ERR_INVALID, "spzb200_encode_host: coordinate system %d", from);
  return runHostPipeline(ctx, true, *in, *out, from, timings);
}

int spzb200_decode_host(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to,
                        SpzB200Cloud *out, SpzB200Timings *timings) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_decode_host: null context");
  int rc = checkPacked(in, "spzb200_decode_host", true);
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_decode_host: null out");
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  rc = checkCloud(out, "spzb200_decode_host");
  if (rc) return rc;
  if (to < 0 || to > 8) return fail(SPZB200_ERR_INVALID, "spzb200_decode_host: coordinate system %d", to);
  return runHostPipeline(ctx, false, *out, *in, to, timings);
}

int spzb200_encode_host_multi(const int32_t *devices, int32_t num_devices, const SpzB200Cloud *in,
                              int32_t from, SpzB200Packed *out, SpzB200Timings *timings) {
  int rc = checkCloud(in, "spzb200_encode_host_multi");
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_encode_host_multi: null out");
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  out->fractional_bits = 12;
  out->version = 3;
  rc = checkPacked(out, "spzb200_encode_host_multi", true);
  if (rc) return rc;
  const SpzB200Cloud cin = *in;
  const SpzB200Packed cout = *out;
  return runSharded(devices, num_devices, in->num_points, in->sh_degree,
                    [&](SpzB200Context *ctx, int64_t a, int64_t b, SpzB200Timings *tm) {
                      SpzB200Cloud ci = sliceCloud(cin, a, b);
                      SpzB200Packed po = slicePacked(cout, a, b);
                      return spzb200_encode_host(ctx, &ci, from, &po, tm);
                    }, timings);
}

int spzb200_decode_host_multi(const int32_t *devices, int32_t num_devices,
                              const SpzB200Packed *in, int32_t to, SpzB200Cloud *out,
                              SpzB200Timings *timings) {
  int rc = checkPacked(in, "spzb200_decode_host_multi", true);
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_decode_host_multi: null out");
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  rc = checkCloud(out, "spzb200_decode_host_multi");
  if (rc) return rc;
  const SpzB200Packed cin = *in;
  const SpzB200Cloud cout = *out;
  return runSharded(devices, num_devices, in->num_points, in->sh_degree,
                    [&](SpzB200Context *ctx, int64_t a, int64_t b, SpzB200Timings *tm) {
                      SpzB200Packed pi = slicePacked(cin, a, b);
                      SpzB200Cloud co = sliceCloud(cout, a, b);
                      return spzb200_decode_host(ctx, &pi, to, &co, tm);
                    }, timings);
}

static int checkPlyRows(const SpzB200PlyRows *in, const char *who) {
  if (!in) return fail(SPZB200_ERR_INVALID, "%s: null rows view", who);
  if (in->num_points < 0) return fail(SPZB200_ERR_INVALID, "%s: num_points < 0", who);
  if (!validDegree(in->sh_degree)) return fail(SPZB200_ERR_INVALID, "%s: sh_degree %d not in 0..3", who, in->sh_degree);
  if (in->width < 14 || in->width > 4096) return fail(SPZB200_ERR_INVALID, "%s: width %d out of range", who, in->width);
  if (in->num_points > 0 && !in->rows) return fail(SPZB200_ERR_INVALID, "%s: null rows pointer", who);
  auto ok = [&](int32_t c) { return c >= 0 && c < in->width; };
  bool cols = ok(in->col_alpha);
  for (int i = 0; i < 3; i++) cols = cols && ok(in->col_pos[i]) && ok(in->col_scale[i]) && ok(in->col_color[i]);
  for (int i = 0; i < 4; i++) cols = cols && ok(in->col_rot[i]);
  for (int i = 0; i < 3 * shDimOf(in->sh_degree); i++) cols = cols && ok(in->col_rest[i]);
  if (!cols) return fail(SPZB200_ERR_INVALID, "%s: column index outside the record", who);
  return SPZB200_OK;
}

static spzb200::PlyEncodeArgs makePlyArgs(const SpzB200Context *ctx, const SpzB200PlyRows &in, const float *rows, long long n,
                                          const SpzB200Packed &out, int32_t from) {
  spzb200::PlyEncodeArgs a;
  std::memset(&a, 0, sizeof a);
  a.rows = rows;
  a.n = n;
  a.width = in.width;
  a.shDim = shDimOf(in.sh_degree);
  for (int i = 0; i < 3; i++) { a.colPos[i] = in.col_pos[i]; a.colScale[i] = in.col_scale[i]; a.colColor[i] = in.col_color[i]; }
  for (int i = 0; i < 4; i++) a.colRot[i] = in.col_rot[i];
  a.colAlpha = in.col_alpha;
  for (int i = 0; i < 3 * a.shDim; i++) a.colRest[i] = in.col_rest[i];
  a.oPositions = out.positions; a.oScales = out.scales; a.oRotations = out.rotations;
  a.oAlphas = out.alphas; a.oColors = out.colors; a.oSh = out.sh;
  const spzb200::m::FlipBits f = spzb200::m::make_flip_bits(from, SPZB200_COORD_RUB);
  a.flipP = f.p; a.flipQ = f.q; a.flipSh = f.sh;
  a.alphaThresholds = ctx->dThr;
  return a;
}

static int preparePlyOut(const SpzB200PlyRows *in, SpzB200Packed *out, int32_t from, const char *who) {
  if (!out) return fail(SPZB200_ERR_INVALID, "%s: null out", who);
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  out->fractional_bits = 12;
  out->version = 3;
  int rc = checkPacked(out, who, true);
  if (rc) return rc;
  if (from < 0 || from > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, from);
  return SPZB200_OK;
}

int spzb200_encode_ply_device(SpzB200Context *ctx, const SpzB200PlyRows *in, int32_t from, SpzB200Packed *out, void *stream) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_encode_ply_device: null context");
  int rc = checkPlyRows(in, "spzb200_encode_ply_device");
  if (rc) return rc;
  rc = preparePlyOut(in, out, from, "spzb200_encode_ply_device");
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  int launches = 0;
  CU(spzb200::launchEncodePly(makePlyArgs(ctx, *in, in->rows, in->num_points, *out, from), planOf(ctx), (cudaStream_t)stream, &launches));
  ctx->kernelLaunches += launches;
  return SPZB200_OK;
}

int spzb200_encode_ply_host(SpzB200Context *ctx, const SpzB200PlyRows *in, int32_t from, SpzB200Packed *out,
                            SpzB200Timings *timings) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_encode_ply_host: null context");
  int rc = checkPlyRows(in, "spzb200_encode_ply_host");
  if (rc) return rc;
  rc = preparePlyOut(in, out, from, "spzb200_encode_ply_host");
  if (rc) return rc;
  PlaneSet rows;
  rows.count = 1;
  rows.ptr[0] = reinterpret_cast<uint8_t *>(in->rows);
  rows.per[0] = (size_t)in->width * 4;
  const PlaneSet by = packedPlaneSet(*out, 3);
  const spzb200::LaunchPlan plan = planOf(ctx);
  return runPipeline(ctx, rows, by, in->num_points, spzb200::plyTileGaussians(),
                     [&](uint8_t *const dIn[6], uint8_t *const dOut[6], long long pts, cudaStream_t s, int *launches) {
                       const SpzB200Packed dp = packedOn(*out, dOut, pts, 3);
                       return spzb200::launchEncodePly(makePlyArgs(ctx, *in, reinterpret_cast<const float *>(dIn[0]), pts, dp, from),
                                                       plan, s, launches);
                     }, timings);
}

static spzb200::PlyDecodeArgs makePlyDecodeArgs(const SpzB200Context *ctx, const SpzB200Packed &in, const SpzB200PlyRows &out, float *rows,
                                                long long n, int32_t to) {
  spzb200::PlyDecodeArgs a;
  std::memset(&a, 0, sizeof a);
  a.positions = in.positions; a.scales = in.scales; a.rotations = in.rotations;
  a.alphas = in.alphas; a.colors = in.colors; a.sh = in.sh;
  a.rows = rows;
  a.n = n;
  a.width = out.width;
  a.shDim = shDimOf(in.sh_degree);
  a.version = in.version;
  a.positionScale = positionScaleFor(in.fractional_bits);
  for (int i = 0; i < 3; i++) { a.colPos[i] = out.col_pos[i]; a.colScale[i] = out.col_scale[i]; a.colColor[i] = out.col_color[i]; }
  for (int i = 0; i < 4; i++) a.colRot[i] = out.col_rot[i];
  a.colAlpha = out.col_alpha;
  for (int i = 0; i < 3 * a.shDim; i++) a.colRest[i] = out.col_rest[i];
  // the columns nothing is decoded into (normals, extras): the kernel writes zeros there
  std::vector<bool> used((size_t)out.width, false);
  used[(size_t)a.colAlpha] = true;
  for (int i = 0; i < 3; i++) used[(size_t)a.colPos[i]] = used[(size_t)a.colScale[i]] = used[(size_t)a.colColor[i]] = true;
  for (int i = 0; i < 4; i++) used[(size_t)a.colRot[i]] = true;
  for (int i = 0; i < 3 * a.shDim; i++) used[(size_t)a.colRest[i]] = true;
  a.numUnmapped = 0;
  for (int c = 0; c < out.width && a.numUnmapped >= 0; c++) {
    if (used[(size_t)c]) continue;
    if (a.numUnmapped == spzb200::kMaxUnmappedColumns) a.numUnmapped = -1;
    else a.unmapped[a.numUnmapped++] = (uint16_t)c;
  }
  const spzb200::m::FlipBits f = spzb200::m::make_flip_bits(SPZB200_COORD_RUB, to);
  a.flipP = f.p; a.flipQ = f.q; a.flipSh = f.sh;
  a.tables = ctx->dLut;
  return a;
}

static int preparePlyDecode(const SpzB200Packed *in, int32_t to, SpzB200PlyRows *out, const char *who) {
  int rc = checkPacked(in, who, true);
  if (rc) return rc;
  if (!out) return fail(SPZB200_ERR_INVALID, "%s: null out", who);
  out->num_points = in->num_points;
  out->sh_degree = in->sh_degree;
  rc = checkPlyRows(out, who);
  if (rc) return rc;
  if (to < 0 || to > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, to);
  return SPZB200_OK;
}

int spzb200_decode_ply_device(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to, SpzB200PlyRows *out, void *stream) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_decode_ply_device: null context");
  int rc = preparePlyDecode(in, to, out, "spzb200_decode_ply_device");
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  int launches = 0;
  CU(spzb200::launchDecodePly(makePlyDecodeArgs(ctx, *in, *out, out->rows, in->num_points, to), planOf(ctx), (cudaStream_t)stream, &launches));
  ctx->kernelLaunches += launches;
  return SPZB200_OK;
}

int spzb200_decode_ply_host(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to, SpzB200PlyRows *out,
                            SpzB200Timings *timings) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_decode_ply_host: null context");
  int rc = preparePlyDecode(in, to, out, "spzb200_decode_ply_host");
  if (rc) return rc;
  PlaneSet rows;
  rows.count = 1;
  rows.ptr[0] = reinterpret_cast<uint8_t *>(out->rows);
  rows.per[0] = (size_t)out->width * 4;
  const PlaneSet by = packedPlaneSet(*in, in->version);
  const spzb200::LaunchPlan plan = planOf(ctx);
  return runPipeline(ctx, by, rows, in->num_points, spzb200::plyTileGaussians(),
                     [&](uint8_t *const dIn[6], uint8_t *const dOut[6], long long pts, cudaStream_t s, int *launches) {
                       const SpzB200Packed dp = packedOn(*in, dIn, pts, in->version);
                       return spzb200::launchDecodePly(makePlyDecodeArgs(ctx, dp, *out, reinterpret_cast<float *>(dOut[0]), pts, to),
                                                       plan, s, launches);
                     }, timings);
}

int spzb200_alloc_pinned(size_t bytes, void **out) {
  if (!out) return fail(SPZB200_ERR_INVALID, "spzb200_alloc_pinned: null out");
  *out = nullptr;
  if (bytes == 0) return SPZB200_OK;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0)
    return fail(SPZB200_ERR_NO_DEVICE, "spzb200_alloc_pinned: no CUDA device");
  e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
  if (e != cudaSuccess) {
    *out = nullptr;
    cudaGetLastError();
    return fail(SPZB200_ERR_NOMEM, "spzb200_alloc_pinned: %zu bytes: %s", bytes, cudaGetErrorString(e));
  }
  return SPZB200_OK;
}

void spzb200_free_pinned(void *ptr) {
  if (ptr) cudaFreeHost(ptr);
}

static int handOverBytes(bool ok, const char *who, std::vector<uint8_t> &bytes, uint8_t **out, size_t *outSize) {
  if (!out || !outSize) return fail(SPZB200_ERR_INVALID, "%s: null output arguments", who);
  *out = nullptr;
  *outSize = 0;
  if (!ok) return fail(SPZB200_ERR_INVALID, "%s: zlib rejected the input", who);
  *out = static_cast<uint8_t *>(std::malloc(bytes.size() ? bytes.size() : 1));
  if (!*out) return fail(SPZB200_ERR_NOMEM, "%s: out of memory (%zu bytes)", who, bytes.size());
  if (!bytes.empty()) std::memcpy(*out, bytes.data(), bytes.size());
  *outSize = bytes.size();
  return SPZB200_OK;
}

// No exception may cross the extern "C" boundary: an allocation failure becomes SPZB200_ERR_NOMEM.
int spzb200_gzip(const uint8_t *data, size_t size, int32_t threads, uint8_t **out, size_t *out_size) {
  try {
    std::vector<uint8_t> bytes;
    const bool ok = (data || size == 0) && spz::compressGzippedParallel(data, size, threads, &bytes);
    return handOverBytes(ok, "spzb200_gzip", bytes, out, out_size);
  } catch (const std::exception &e) {
    if (out) *out = nullptr;
    if (out_size) *out_size = 0;
    return fail(SPZB200_ERR_NOMEM, "spzb200_gzip: %s", e.what());
  }
}

int spzb200_gunzip(const uint8_t *data, size_t size, int32_t threads, uint8_t **out, size_t *out_size) {
  try {
    std::vector<uint8_t> bytes;
    const bool ok = data && spz::decompressGzippedParallel(data, size, threads, &bytes);
    return handOverBytes(ok, "spzb200_gunzip", bytes, out, out_size);
  } catch (const std::exception &e) {
    if (out) *out = nullptr;
    if (out_size) *out_size = 0;
    return fail(SPZB200_ERR_NOMEM, "spzb200_gunzip: %s", e.what());
  }
}

void spzb200_free(void *ptr) { std::free(ptr); }

int32_t spzb200_tile_gaussians(int32_t sh_degree) {
  return validDegree(sh_degree) ? spzb200::tileGaussians(shDimOf(sh_degree)) : 0;
}

int spzb200_shard_range(int64_t n, int32_t sh_degree, int32_t num_shards, int32_t index,
                        int64_t *begin, int64_t *end) {
  if (n < 0 || !validDegree(sh_degree) || num_shards <= 0 || index < 0 || index >= num_shards || !begin || !end)
    return fail(SPZB200_ERR_INVALID, "spzb200_shard_range: bad arguments");
  const int64_t g = spzb200::tileGaussians(shDimOf(sh_degree));
  const int64_t tiles = n / g;
  // whole tiles are dealt out as evenly as possible; the sub-tile remainder rides on the last shard
  const int64_t a = tiles * index / num_shards * g;
  const int64_t b = index == num_shards - 1 ? n : tiles * (index + 1) / num_shards * g;
  *begin = a;
  *end = b;
  return SPZB200_OK;
}

void spzb200_flip_bits(int32_t from, int32_t to, uint32_t *flip_p, uint32_t *flip_q, uint32_t *flip_sh) {
  const spzb200::m::FlipBits f = spzb200::m::make_flip_bits(from, to);
  if (flip_p) *flip_p = f.p;
  if (flip_q) *flip_q = f.q;
  if (flip_sh) *flip_sh = f.sh;
}

int spzb200_build_tables(float alpha_thresholds[256], float alpha_lut[256]) {
  std::string why;
  if (alpha_thresholds && !buildAlphaThresholds(alpha_thresholds, &why))
    return fail(SPZB200_ERR_INVALID, "spzb200_build_tables: %s", why.c_str());
  if (alpha_lut) buildAlphaLut(alpha_lut);
  return SPZB200_OK;
}

int spzb200_get_tables(const SpzB200Context *ctx, float alpha_thresholds[256], float alpha_lut[256]) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_get_tables: null context");
  if (alpha_thresholds) std::memcpy(alpha_thresholds, ctx->hThr, sizeof ctx->hThr);
  if (alpha_lut) std::memcpy(alpha_lut, ctx->hLut, sizeof ctx->hLut);
  return SPZB200_OK;
}

int spzb200_info(const SpzB200Context *ctx, int32_t *sm_count, int32_t *pack_mode, int64_t *kernel_launches) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_info: null context");
  if (sm_count) *sm_count = ctx->smCount;
  if (pack_mode) *pack_mode = ctx->packMode;
  if (kernel_launches) *kernel_launches = ctx->kernelLaunches;
  return SPZB200_OK;
}

int spzb200_selfcheck_division(SpzB200Context *ctx, int32_t part, uint64_t pairs_per_thread, uint64_t seed, uint64_t *wrong,
                               uint64_t *checked) {
  if (!ctx || !wrong) return fail(SPZB200_ERR_INVALID, "spzb200_selfcheck_division: null argument");
  if (part != 0 && part != 1) return fail(SPZB200_ERR_INVALID, "spzb200_selfcheck_division: part %d", (int)part);
  CU(cudaSetDevice(ctx->device));
  unsigned long long w = 0, c = 0;
  CU(spzb200::divisionSelfCheck(part, pairs_per_thread, seed, ctx->smCount, ctx->stage[0].stream, &w, &c));
  ctx->kernelLaunches += 1;
  *wrong = w;
  if (checked) *checked = c;
  return SPZB200_OK;
}

void spzb200_set_force_generic(SpzB200Context *ctx, int32_t on) { if (ctx) ctx->forceGeneric = on != 0; }
void spzb200_set_pack_mode(SpzB200Context *ctx, int32_t mode) {
  if (ctx) ctx->packMode = (mode && ctx->cvtPackOk) ? spzb200::kPackCvt : spzb200::kPackAlu;
}
void spzb200_set_chunk_points(SpzB200Context *ctx, int64_t points) {
  if (!ctx) return;
  if (points > 0) {
    ctx->chunkPoints = ctx->pageableChunkPoints = points;
    ctx->adaptiveChunks = false;
  } else {  // back to the defaults
    ctx->chunkPoints = 1 << 21;
    ctx->pageableChunkPoints = 1 << 18;
    ctx->adaptiveChunks = true;
  }
}
void spzb200_set_host_staging(SpzB200Context *ctx, int32_t bounce, int32_t copy_threads) {
  if (!ctx) return;
  ctx->bounceMode = bounce < 0 ? 0 : (bounce > 2 ? 2 : bounce);
  if (copy_threads >= 0 && copy_threads != ctx->copyThreads) {
    ctx->copyThreads = copy_threads;
    delete ctx->pool;
    ctx->pool = nullptr;
  }
}

}  // extern "C"

// ---- batched per-gaussian access -----------------------------------------------------------------
namespace {

constexpr long long kGatherChunk = 1 << 16;  // records per staged chunk (4.2 MB in, 15.5 MB out)
constexpr long long kGatherZeroCopy = 2048;  // up to here the kernel reads and writes the pinned host buffers itself

int ensureGatherSlot(SpzB200Context::GatherSlot &g, size_t records, bool device) {
  if (!g.done) CU(cudaEventCreateWithFlags(&g.done, cudaEventDisableTiming));
  if (g.cap < records || (device && !g.dIn)) {
    size_t cap = 256;
    while (cap < records) cap <<= 1;
    cap = std::max(cap, g.cap);
    if (g.cap < cap) {
      if (g.hIn) cudaFreeHost(g.hIn);
      if (g.hOut) cudaFreeHost(g.hOut);
      g.hIn = nullptr; g.hOut = nullptr;
      if (g.dIn) cudaFree(g.dIn);
      if (g.dOut) cudaFree(g.dOut);
      g.dIn = nullptr; g.dOut = nullptr;
      g.cap = 0;
      CU(cudaHostAlloc(&g.hIn, cap * SPZB200_RECORD_BYTES, cudaHostAllocMapped));
      CU(cudaHostAlloc(&g.hOut, cap * SPZB200_UNPACKED_FLOATS * sizeof(float), cudaHostAllocMapped));
      g.cap = cap;
    }
    if (device && !g.dIn) {
      CU(cudaMalloc(&g.dIn, g.cap * SPZB200_RECORD_BYTES));
      CU(cudaMalloc(&g.dOut, g.cap * SPZB200_UNPACKED_FLOATS * sizeof(float)));
    }
  }
  return SPZB200_OK;
}

void fillConverter(spzb200::GatherArgs &a, const float *converter) {
  for (int i = 0; i < 3; i++) { a.flipP[i] = converter ? converter[i] : 1.0f; a.flipQ[i] = converter ? converter[3 + i] : 1.0f; }
  for (int i = 0; i < 15; i++) a.flipSh[i] = converter ? converter[6 + i] : 1.0f;
}

// at(i), load-spz.cc:431-459: pure byte gather of one gaussian into the 65-byte record layout
void gatherRecord(const SpzB200Packed &p, int shDim, int64_t i, uint8_t *r) {
  const bool half = p.version == 1 || p.version == 4;
  const size_t posBytes = half ? 6 : 9, rotBytes = p.version >= 3 ? 4 : 3;
  std::memset(r, 0, 13);
  std::memcpy(r, p.positions + (size_t)i * posBytes, posBytes);
  std::memcpy(r + 9, p.rotations + (size_t)i * rotBytes, rotBytes);
  std::memcpy(r + 13, p.scales + (size_t)i * 3, 3);
  std::memcpy(r + 16, p.colors + (size_t)i * 3, 3);
  r[19] = p.alphas[i];
  const uint8_t *s = shDim ? p.sh + (size_t)i * shDim * 3 : nullptr;
  for (int j = 0; j < 15; j++) {
    const bool have = j < shDim;
    r[20 + j] = have ? s[3 * j] : 128;
    r[35 + j] = have ? s[3 * j + 1] : 128;
    r[50 + j] = have ? s[3 * j + 2] : 128;
  }
}

// fill(dst, first, count) writes records [first, first + count) into dst
template <class Fill>
int runGatherHost(SpzB200Context *ctx, long long n, int32_t version, int32_t fractionalBits, const float *converter, float *out,
                  Fill &&fill) {
  if (n == 0) return SPZB200_OK;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t stream = ctx->stage[0].stream;
  spzb200::GatherArgs a;
  std::memset(&a, 0, sizeof a);
  a.version = version;
  a.positionScale = positionScaleFor(fractionalBits);
  a.tables = ctx->dLut;
  fillConverter(a, converter);
  const bool zeroCopy = n <= kGatherZeroCopy;
  const long long chunk = std::min<long long>(n, kGatherChunk);
  const long long chunks = (n + chunk - 1) / chunk;
  const int slots = (int)std::min<long long>(2, chunks);
  for (int s = 0; s < slots; s++) {
    const int rc = ensureGatherSlot(ctx->gather[s], (size_t)chunk, !zeroCopy);
    if (rc != SPZB200_OK) return rc;
  }
  auto drain = [&](long long c) -> int {
    SpzB200Context::GatherSlot &g = ctx->gather[c & 1];
    const long long first = c * chunk, count = std::min(n, first + chunk) - first;
    CU(cudaEventSynchronize(g.done));
    std::memcpy(out + first * SPZB200_UNPACKED_FLOATS, g.hOut, (size_t)count * SPZB200_UNPACKED_FLOATS * sizeof(float));
    return SPZB200_OK;
  };
  for (long long c = 0; c < chunks; c++) {
    SpzB200Context::GatherSlot &g = ctx->gather[c & 1];
    if (c >= 2) {
      const int rc = drain(c - 2);
      if (rc != SPZB200_OK) return rc;
    }
    const long long first = c * chunk, count = std::min(n, first + chunk) - first;
    fill(g.hIn, first, count);
    int launches = 0;
    a.n = count;
    if (zeroCopy) {
      // a handful of gaussians: the kernel reads the pinned records and writes the pinned result over
      // PCIe itself -- one launch and one synchronize instead of copy, launch, copy
      a.records = g.hIn;
      a.out = g.hOut;
    } else {
      CU(cudaMemcpyAsync(g.dIn, g.hIn, (size_t)count * SPZB200_RECORD_BYTES, cudaMemcpyHostToDevice, stream));
      a.records = g.dIn;
      a.out = g.dOut;
    }
    CU(spzb200::launchUnpackRecords(a, stream, &launches));
    ctx->kernelLaunches += launches;
    if (!zeroCopy)
      CU(cudaMemcpyAsync(g.hOut, g.dOut, (size_t)count * SPZB200_UNPACKED_FLOATS * sizeof(float), cudaMemcpyDeviceToHost, stream));
    CU(cudaEventRecord(g.done, stream));
  }
  for (long long c = std::max<long long>(0, chunks - 2); c < chunks; c++) {
    const int rc = drain(c);
    if (rc != SPZB200_OK) return rc;
  }
  return SPZB200_OK;
}

int gatherFailed(SpzB200Context *ctx, int rc) {
  if (rc != SPZB200_OK) {  // nothing of this call may still be reading or writing the staging buffers
    const std::string first = tlsError;
    (void)cudaStreamSynchronize(ctx->stage[0].stream);
    (void)cudaGetLastError();
    tlsError = first;
  }
  return rc;
}

}  // namespace

extern "C" {

int spzb200_unpack_records_host(SpzB200Context *ctx, const uint8_t *records, int64_t n, int32_t version,
                                int32_t fractional_bits, const float *converter, float *out) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_records_host: null context");
  if (n < 0) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_records_host: n < 0");
  if (version < 1 || version > SPZB200_STREAM_HALF_POSITIONS_SMALLEST_THREE)
    return fail(SPZB200_ERR_INVALID, "spzb200_unpack_records_host: version %d not in 1..4", version);
  if (n > 0 && (!records || !out)) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_records_host: null pointer");
  return gatherFailed(ctx, runGatherHost(ctx, n, version, fractional_bits, converter, out, [&](uint8_t *dst, long long first, long long count) {
    std::memcpy(dst, records + (size_t)first * SPZB200_RECORD_BYTES, (size_t)count * SPZB200_RECORD_BYTES);
  }));
}

int spzb200_unpack_gather_host(SpzB200Context *ctx, const SpzB200Packed *packed, const int64_t *indices, int64_t n,
                               const float *converter, float *out) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_host: null context");
  int rc = checkPacked(packed, "spzb200_unpack_gather_host", true);
  if (rc) return rc;
  if (n < 0) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_host: n < 0");
  if (n > 0 && !out) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_host: null out");
  if (!indices && n > packed->num_points)
    return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_host: n exceeds num_points and no indices were given");
  if (indices)
    for (int64_t k = 0; k < n; k++)
      if (indices[k] < 0 || indices[k] >= packed->num_points)
        return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_host: index %lld at position %lld is outside [0, %lld)",
                    (long long)indices[k], (long long)k, (long long)packed->num_points);
  const int shDim = shDimOf(packed->sh_degree);
  const SpzB200Packed p = *packed;
  return gatherFailed(ctx, runGatherHost(ctx, n, p.version, p.fractional_bits, converter, out, [&](uint8_t *dst, long long first, long long count) {
    // at() for every record of the chunk; random reads of six planes (~0.1 us per record on one thread), so large
    // chunks are split over a few threads
    auto part = [&](long long a, long long b) {
      for (long long k = a; k < b; k++)
        gatherRecord(p, shDim, indices ? indices[first + k] : first + k, dst + (size_t)k * SPZB200_RECORD_BYTES);
    };
    const int workers = count >= 16384 ? (int)std::min<unsigned>(4, std::max(1u, std::thread::hardware_concurrency())) : 1;
    if (workers == 1) {
      part(0, count);
      return;
    }
    std::vector<std::thread> th;
    int started = 1;
    try {
      for (; started < workers; started++) th.emplace_back(part, count * started / workers, count * (started + 1) / workers);
    } catch (const std::exception &) {
      // no more threads to be had: the rest of the chunk is gathered on this one
    }
    part(0, count / workers);
    for (int w = started; w < workers; w++) part(count * w / workers, count * (w + 1) / workers);
    for (auto &t : th) t.join();
  }));
}

int spzb200_unpack_gather_device(SpzB200Context *ctx, const SpzB200Packed *packed, const int64_t *indices, int64_t n,
                                 const float *converter, float *out, void *stream) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_device: null context");
  int rc = checkPacked(packed, "spzb200_unpack_gather_device", true);
  if (rc) return rc;
  if (n < 0) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_device: n < 0");
  if (n > 0 && !out) return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_device: null out");
  if (!indices && n > packed->num_points)
    return fail(SPZB200_ERR_INVALID, "spzb200_unpack_gather_device: n exceeds num_points and no indices were given");
  if (n == 0) return SPZB200_OK;
  CU(cudaSetDevice(ctx->device));
  spzb200::GatherArgs a;
  std::memset(&a, 0, sizeof a);
  a.positions = packed->positions; a.scales = packed->scales; a.rotations = packed->rotations;
  a.alphas = packed->alphas; a.colors = packed->colors; a.sh = packed->sh;
  a.indices = reinterpret_cast<const long long *>(indices);
  a.out = out;
  a.n = n;
  a.shDim = shDimOf(packed->sh_degree);
  a.version = packed->version;
  a.positionScale = positionScaleFor(packed->fractional_bits);
  a.tables = ctx->dLut;
  fillConverter(a, converter);
  int launches = 0;
  CU(spzb200::launchUnpackRecords(a, (cudaStream_t)stream, &launches));
  ctx->kernelLaunches += launches;
  return SPZB200_OK;
}

}  // extern "C"

// =================================================================================================
// .spz files from and to device-resident planes, with the deflate stage on the device (DESIGN.md section 10)
// =================================================================================================

namespace {

// Device scratch of one call: stream-ordered allocations, handed back on the same stream on every exit.
struct DeviceScratch {
  cudaStream_t stream;
  std::vector<void *> ptrs;
  explicit DeviceScratch(cudaStream_t s) : stream(s) {}
  ~DeviceScratch() {
    for (void *p : ptrs) cudaFreeAsync(p, stream);
  }
  template <class T>
  cudaError_t alloc(T **p, size_t bytes) {
    void *v = nullptr;
    const cudaError_t e = cudaMallocAsync(&v, std::max<size_t>(bytes, 16), stream);
    if (e != cudaSuccess) return e;
    ptrs.push_back(v);
    *p = static_cast<T *>(v);
    return cudaSuccess;
  }
};

size_t deflateBodyBytes(size_t size) { return size + 16 * spzb200::dfl::segmentCount(size) + 16; }

struct HostSpan {
  const uint8_t *p;
  size_t n;
};

// The spans, end to end, from pageable host memory to dst on the device, stream-ordered after earlier
// work on `stream`, in pieces through two of the context's pinned bounce buffers: the DMA of one piece
// overlaps the host copy of the next (a pageable copy of a whole compressed body ran at ~2 GB/s on a B200
// host).  Synchronous.
int bouncedUpload(SpzB200Context *ctx, uint8_t *dst, const std::vector<HostSpan> &src, cudaStream_t stream) {
  constexpr size_t kPiece = (size_t)8 << 20;
  for (int k = 0; k < 2; k++) {
    Stage &s = ctx->stage[k];
    const int rc = ensureBounce(s.hIn, s.hInCap, kPiece);
    if (rc) return rc;
  }
  size_t bytes = 0;
  for (const HostSpan &h : src) bytes += h.n;
  const size_t pieces = (bytes + kPiece - 1) / kPiece;
  size_t span = 0, at = 0;  // read position: src[span].p + at
  for (size_t i = 0; i < pieces; i++) {  // wait until the buffer's previous DMA is done, fill it, queue its DMA
    Stage &s = ctx->stage[i & 1];
    if (i >= 2) CU(cudaEventSynchronize(s.ev[0]));
    const size_t len = std::min(kPiece, bytes - i * kPiece);
    for (size_t filled = 0; filled < len;) {
      if (at == src[span].n) {
        span++;
        at = 0;
        continue;
      }
      const size_t n = std::min(len - filled, src[span].n - at);
      bounceCopy(s.hIn + filled, src[span].p + at, n);
      filled += n;
      at += n;
    }
    CU(cudaMemcpyAsync(dst + i * kPiece, s.hIn, len, cudaMemcpyHostToDevice, stream));
    CU(cudaEventRecord(s.ev[0], stream));
  }
  CU(cudaStreamSynchronize(stream));
  return SPZB200_OK;
}

// `bytes` between pageable host memory and the device through the bounce buffers (bouncedUpload); the
// D2H direction queues piece i, then copies piece i - 1 out of its buffer.  Synchronous.
int bouncedCopy(SpzB200Context *ctx, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, cudaStream_t stream) {
  if (kind != cudaMemcpyDeviceToHost)
    return bouncedUpload(ctx, static_cast<uint8_t *>(dst), {HostSpan{static_cast<const uint8_t *>(src), bytes}}, stream);
  constexpr size_t kPiece = (size_t)8 << 20;
  for (int k = 0; k < 2; k++) {
    Stage &s = ctx->stage[k];
    const int rc = ensureBounce(s.hOut, s.hOutCap, kPiece);
    if (rc) return rc;
  }
  uint8_t *to = static_cast<uint8_t *>(dst);
  const uint8_t *from = static_cast<const uint8_t *>(src);
  const size_t pieces = (bytes + kPiece - 1) / kPiece;
  auto len = [&](size_t i) { return std::min(kPiece, bytes - i * kPiece); };
  for (size_t i = 0; i <= pieces; i++) {
    if (i < pieces) {
      Stage &s = ctx->stage[i & 1];
      CU(cudaMemcpyAsync(s.hOut, from + i * kPiece, len(i), cudaMemcpyDeviceToHost, stream));
      CU(cudaEventRecord(s.ev[0], stream));
    }
    if (i > 0) {
      Stage &s = ctx->stage[(i - 1) & 1];
      CU(cudaEventSynchronize(s.ev[0]));
      bounceCopy(to + (i - 1) * kPiece, s.hOut, len(i - 1));
    }
  }
  return SPZB200_OK;
}

// A host table to a fresh device allocation of `scratch`, stream-ordered (the host vector must live until
// the stream is synchronised).
template <class T>
int uploadTable(const std::vector<T> &host, T **dev, DeviceScratch &scratch) {
  CU(scratch.alloc(dev, host.size() * sizeof(T)));
  if (!host.empty()) CU(cudaMemcpyAsync(*dev, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice, scratch.stream));
  return SPZB200_OK;
}

// The segments of all inputs (every DeflateSegment of the batch, batch_plan.hpp) deflated in one set of
// launches, then each input's body framed as one gzip member and handed over to a malloc'd out[i] at once,
// while its bytes are still in the host's caches.  All or nothing: after a failure every out[i] is NULL.
// slots: the batch's segment count times deflateSlotBytes(); body: the sum of deflateBodyBytes over the
// inputs (may hold the inputs themselves: the body is written after the last read of them).  Synchronous.
int gzipDeviceBatch(SpzB200Context *ctx, const char *who, const uint8_t *const *src, const size_t *sizes, int count, uint8_t *slots,
                    uint8_t *body, DeviceScratch &scratch, uint8_t **out, size_t *outSize) {
  namespace dfl = spzb200::dfl;
  std::vector<unsigned long long> addr(count);
  std::vector<uint64_t> size64(count);
  for (int i = 0; i < count; i++) {
    addr[i] = (unsigned long long)(uintptr_t)src[i];
    size64[i] = sizes[i];
  }
  std::vector<spzb200::DeflateSegment> segs;
  std::vector<uint64_t> first;
  spzb200::planDeflate(addr.data(), size64.data(), count, &segs, &first);
  const size_t total = segs.size();
  spzb200::DeflateSegment *dSegs = nullptr;
  uint32_t *segBytes = nullptr;
  unsigned long long *offsets = nullptr;
  int rc = uploadTable(segs, &dSegs, scratch);
  if (rc) return rc;
  CU(scratch.alloc(&segBytes, 2 * total * sizeof(uint32_t)));
  CU(scratch.alloc(&offsets, (total + 1) * sizeof(unsigned long long)));
  uint32_t *segCrc = segBytes + total;
  int launches = 0;
  CU(spzb200::launchDeflate(dSegs, total, slots, segBytes, segCrc, offsets, body, scratch.stream, &launches));
  ctx->kernelLaunches += launches;
  std::vector<uint32_t> hostSeg(2 * total);
  CU(cudaMemcpyAsync(hostSeg.data(), segBytes, 2 * total * sizeof(uint32_t), cudaMemcpyDeviceToHost, scratch.stream));
  CU(cudaStreamSynchronize(scratch.stream));
  std::vector<uint64_t> bodyStart;
  std::vector<std::vector<uint32_t>> blockBytes;
  spzb200::planMemberBodies(hostSeg.data(), first, &bodyStart, &blockBytes);
  auto undo = [&](int upTo, int rc) {
    for (int j = 0; j < upTo; j++) {
      std::free(out[j]);
      out[j] = nullptr;
      outSize[j] = 0;
    }
    return rc;
  };
  int i = 0;
  try {
    for (; i < count; i++) {
      uLong crc = crc32(0L, Z_NULL, 0);
      for (uint64_t s = first[i]; s < first[i + 1]; s++) crc = crc32_combine(crc, hostSeg[total + s], (z_off_t)segs[s].len);
      const size_t segCount = first[i + 1] - first[i];
      std::vector<uint8_t> bytes;
      int copyRc = SPZB200_OK;
      const bool ok = spz::detail::frameBlockMember(sizes[i], dfl::segmentsPerBlock(segCount) * dfl::kSegBytes, blockBytes[i], (uint32_t)crc,
                                                    [&](uint8_t *dst) {
                                                      copyRc = bouncedCopy(ctx, dst, body + bodyStart[i], bodyStart[i + 1] - bodyStart[i],
                                                                           cudaMemcpyDeviceToHost, scratch.stream);
                                                      return copyRc == SPZB200_OK;
                                                    },
                                                    &bytes);
      if (copyRc) return undo(i, copyRc);
      if (!ok) return undo(i, fail(SPZB200_ERR_INVALID, "%zu bytes do not fit the gzip block table", sizes[i]));
      const int rc = handOverBytes(true, who, bytes, &out[i], &outSize[i]);
      if (rc) return undo(i, rc);
    }
  } catch (const std::exception &e) {  // a member handed over before the failure must not outlive it
    return undo(i, fail(SPZB200_ERR_NOMEM, "%s: %s", who, e.what()));
  }
  return SPZB200_OK;
}

// One member of a batched device inflate: its bytes in host memory, its parsed table, where it inflates to.
struct InflateMember {
  const uint8_t *bytes;
  const spz::detail::BlockTable *t;
  uint8_t *out;
};

// The inflate stage on the device for members m (every table block of every member in one launch): the
// compressed bodies cross PCIe through the bounce buffers, one kernel inflates every block and checksums
// its slice, and the host combines each member's CRCs.  (*vouched)[i]: every block of member i filled its
// slice exactly and the combined CRC-32 matches the trailer (ISIZE was checked by the parser); when false,
// its output holds nothing to use and the host inflater has to give the verdict.  Synchronous.
int inflateDeviceBatch(SpzB200Context *ctx, const std::vector<InflateMember> &m, DeviceScratch &scratch, std::vector<char> *vouched) {
  const int count = (int)m.size();
  vouched->assign(count, 0);
  std::vector<uint64_t> blockSize(count), total(count), nBlocks(count);
  std::vector<uint32_t> compressed;
  std::vector<unsigned long long> outAddr(count);
  for (int i = 0; i < count; i++) {
    blockSize[i] = m[i].t->blockSize;
    total[i] = m[i].t->totalSize;
    nBlocks[i] = m[i].t->compressed.size();
    compressed.insert(compressed.end(), m[i].t->compressed.begin(), m[i].t->compressed.end());
    outAddr[i] = (unsigned long long)(uintptr_t)m[i].out;
  }
  std::vector<spzb200::InflateBlock> blocks;
  std::vector<uint64_t> first, bodyStart;
  spzb200::planInflate(count, blockSize.data(), total.data(), nBlocks.data(), compressed.data(), outAddr.data(), &blocks, &first, &bodyStart);
  const size_t nb = blocks.size();
  if (nb == 0) return SPZB200_OK;
  uint8_t *body = nullptr;
  spzb200::InflateBlock *dBlocks = nullptr;
  uint32_t *dCrc = nullptr;
  CU(scratch.alloc(&body, bodyStart[count]));
  int rc = uploadTable(blocks, &dBlocks, scratch);
  if (rc) return rc;
  CU(scratch.alloc(&dCrc, 2 * nb * sizeof(uint32_t)));
  int32_t *dStatus = reinterpret_cast<int32_t *>(dCrc + nb);
  std::vector<HostSpan> spans(count);
  for (int i = 0; i < count; i++) spans[i] = HostSpan{m[i].bytes + m[i].t->bodyOffset, (size_t)(bodyStart[i + 1] - bodyStart[i])};
  rc = bouncedUpload(ctx, body, spans, scratch.stream);
  if (rc) return rc;
  int warps = 0;
  CU(spzb200::launchInflate(body, dBlocks, (long long)nb, dCrc, dStatus, ctx->smCount, scratch.stream, &warps));
  ctx->kernelLaunches += 1;
  std::vector<uint32_t> result(2 * nb);
  CU(cudaMemcpyAsync(result.data(), dCrc, 2 * nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, scratch.stream));
  CU(cudaStreamSynchronize(scratch.stream));
  for (int i = 0; i < count; i++) {
    uLong crc = crc32(0L, Z_NULL, 0);
    bool ok = true;
    for (uint64_t b = first[i]; b < first[i + 1] && ok; b++) {
      ok = result[nb + b] == spzb200::ifl::kOk;
      crc = crc32_combine(crc, result[b], (z_off_t)blocks[b].outBytes);
    }
    (*vouched)[i] = ok && (uint32_t)crc == m[i].t->crc;
  }
  return SPZB200_OK;
}

// No exception may cross the extern "C" boundary: allocation failures become SPZB200_ERR_NOMEM.
template <class Fn>
int guarded(const char *who, uint8_t **out, size_t *outSize, Fn &&fn) {
  try {
    return fn();
  } catch (const std::exception &e) {
    if (out) *out = nullptr;
    if (outSize) *outSize = 0;
    return fail(SPZB200_ERR_NOMEM, "%s: %s", who, e.what());
  }
}

// spzb200_gzip_device_batch after its argument checks.
int gzipBatch(SpzB200Context *ctx, const char *who, const uint8_t *const *data, const size_t *sizes, int32_t count, uint8_t **out,
              size_t *outSize, cudaStream_t stream) {
  return guarded(who, nullptr, nullptr, [&]() -> int {
    if (count == 0) return SPZB200_OK;
    CU(cudaSetDevice(ctx->device));
    size_t segs = 0, body = 0;
    for (int i = 0; i < count; i++) {
      segs += spzb200::dfl::segmentCount(sizes[i]);
      body += deflateBodyBytes(sizes[i]);
    }
    DeviceScratch scratch(stream);
    uint8_t *slots = nullptr, *dBody = nullptr;
    CU(scratch.alloc(&slots, segs * spzb200::deflateSlotBytes()));
    CU(scratch.alloc(&dBody, body));
    return gzipDeviceBatch(ctx, who, data, sizes, count, slots, dBody, scratch, out, outSize);
  });
}

// spzb200_save_spz_device_batch after every cloud has been checked: each cloud's encoder planes go to
// 16-byte-aligned places of the slots buffer, one move launch writes every header and plane into the
// containers, and the deflater codes every container's segments in one set of launches.
int saveBatch(SpzB200Context *ctx, const char *who, const SpzB200Cloud *clouds, int32_t count, int32_t from, const int32_t *antialiased,
              uint8_t **out, size_t *outSize, cudaStream_t stream) {
  return guarded(who, nullptr, nullptr, [&]() -> int {
    if (count == 0) return SPZB200_OK;
    CU(cudaSetDevice(ctx->device));
    constexpr size_t kHeader = spz::detail::kContainerHeaderBytes;
    const int streamOrder[6] = {0, 3, 4, 1, 2, 5};  // container order (positions, alphas, colors, scales, rotations, sh) -> struct order
    std::vector<std::array<size_t, 6>> plane(count), offset(count);  // struct order; offset within the container
    std::vector<uint64_t> total(count), aligned(count), bodyBound(count);
    size_t segs = 0;
    for (int i = 0; i < count; i++) {
      bytePlaneBytes(shDimOf(clouds[i].sh_degree), SPZB200_STREAM_V3, plane[i].data());
      for (size_t &b : plane[i]) b *= (size_t)clouds[i].num_points;
      total[i] = kHeader;
      for (int k = 0; k < 6; k++) {
        offset[i][streamOrder[k]] = total[i];
        total[i] += plane[i][streamOrder[k]];
        aligned[i] += alignUp(plane[i][k], 16);
      }
      bodyBound[i] = deflateBodyBytes(total[i]);
      segs += spzb200::dfl::segmentCount(total[i]);
    }
    std::vector<uint64_t> planesAt, containerAt;
    spzb200::planAligned(aligned.data(), count, &planesAt);
    spzb200::planAligned(bodyBound.data(), count, &containerAt);
    // Peak scratch: the slots (which first hold the encoder's aligned planes) + the containers (which then hold the bodies).
    DeviceScratch scratch(stream);
    uint8_t *slots = nullptr, *containers = nullptr, *headers = nullptr;
    CU(scratch.alloc(&slots, std::max<size_t>(segs * spzb200::deflateSlotBytes(), planesAt[count])));
    CU(scratch.alloc(&containers, containerAt[count]));
    CU(scratch.alloc(&headers, kHeader * count));
    std::vector<uint8_t> hostHeaders(kHeader * count);
    std::vector<spzb200::MoveSpan> spans;
    unsigned long long maxSpan = kHeader;
    std::vector<const uint8_t *> src(count);
    std::vector<size_t> sizes(count);
    for (int i = 0; i < count; i++) {
      const SpzB200Cloud &c = clouds[i];
      uint8_t *container = containers + containerAt[i];
      src[i] = container;
      sizes[i] = total[i];
      spz::detail::writeContainerHeader(3, c.num_points, c.sh_degree, antialiased && antialiased[i] != 0, &hostHeaders[kHeader * i]);
      spans.push_back({(unsigned long long)(uintptr_t)(headers + kHeader * i), (unsigned long long)(uintptr_t)container, kHeader});
      uint8_t *planes[6], *p = slots + planesAt[i];
      for (int k = 0; k < 6; k++) {
        planes[k] = p;
        p += alignUp(plane[i][k], 16);
        if (plane[i][k]) {
          spans.push_back({(unsigned long long)(uintptr_t)planes[k], (unsigned long long)(uintptr_t)(container + offset[i][k]), plane[i][k]});
          maxSpan = std::max<unsigned long long>(maxSpan, plane[i][k]);
        }
      }
      if (c.num_points == 0) continue;
      SpzB200Packed packed;
      std::memset(&packed, 0, sizeof packed);
      packed.num_points = c.num_points;
      packed.sh_degree = c.sh_degree;
      packed.positions = planes[0]; packed.scales = planes[1]; packed.rotations = planes[2];
      packed.alphas = planes[3]; packed.colors = planes[4]; packed.sh = c.sh_degree ? planes[5] : nullptr;
      const int erc = spzb200_encode_device_as(ctx, &c, from, SPZB200_STREAM_V3, &packed, stream);
      if (erc) return erc;
    }
    CU(cudaMemcpyAsync(headers, hostHeaders.data(), hostHeaders.size(), cudaMemcpyHostToDevice, stream));
    spzb200::MoveSpan *dSpans = nullptr;
    int rc = uploadTable(spans, &dSpans, scratch);
    if (rc) return rc;
    int launches = 0;
    CU(spzb200::launchMoveSpans(dSpans, (long long)spans.size(), maxSpan, stream, &launches));
    ctx->kernelLaunches += launches;
    return gzipDeviceBatch(ctx, who, src.data(), sizes.data(), count, slots, containers, scratch, out, outSize);
  });
}

// Both save entry points: every cloud is checked before anything is queued.
int saveSpzDevice(SpzB200Context *ctx, const char *who, const SpzB200Cloud *clouds, int32_t count, int32_t from, const int32_t *antialiased,
                  uint8_t **out, size_t *outSize, cudaStream_t stream) {
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (count < 0) return fail(SPZB200_ERR_INVALID, "%s: count %d", who, count);
  if (count && (!out || !outSize)) return fail(SPZB200_ERR_INVALID, "%s: null output arguments", who);
  for (int i = 0; i < count; i++) {
    out[i] = nullptr;
    outSize[i] = 0;
  }
  if (count && !clouds) return fail(SPZB200_ERR_INVALID, "%s: null cloud view", who);
  for (int i = 0; i < count; i++) {
    const int rc = checkCloud(&clouds[i], who);
    if (rc) return rc;
    if (clouds[i].num_points > std::numeric_limits<int32_t>::max())
      return fail(SPZB200_ERR_INVALID, "%s: %lld points do not fit the container's 32-bit count", who, (long long)clouds[i].num_points);
  }
  if (from < 0 || from > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, from);
  return saveBatch(ctx, who, clouds, count, from, antialiased, out, outSize, stream);
}

// spzb200_gunzip_device_batch after its argument checks: every member with a table is inflated in one
// device launch; a member the device cannot vouch for is inflated by the host inflater, alone.
int gunzipBatch(SpzB200Context *ctx, const char *who, const uint8_t *const *bytes, const size_t *sizes, int32_t count, uint8_t *const *out,
                const size_t *capacity, size_t *outSize, int32_t *onDevice, int32_t *status, cudaStream_t stream) {
  return guarded(who, nullptr, nullptr, [&]() -> int {
    std::vector<spz::detail::BlockTable> tables(count);
    std::vector<InflateMember> members;
    std::vector<int> index;
    for (int i = 0; i < count; i++) {
      outSize[i] = 0;
      if (onDevice) onDevice[i] = 0;
      status[i] = SPZB200_OK;
      const spz::detail::BlockTable &t = tables[i];
      if (!spz::detail::parseBlockTable(bytes[i], sizes[i], &tables[i]))
        status[i] = fail(SPZB200_ERR_INVALID, "%s: member %d: not a gzip member with a block table the parallel inflater trusts", who, i);
      else if (capacity[i] < t.totalSize)
        status[i] = fail(SPZB200_ERR_INVALID, "%s: member %d: out holds %zu bytes, the member inflates to %llu", who, i, capacity[i],
                         (unsigned long long)t.totalSize);
      else {
        members.push_back({bytes[i], &tables[i], out[i]});
        index.push_back(i);
      }
    }
    if (!members.empty()) {
      CU(cudaSetDevice(ctx->device));
      std::vector<char> vouched;
      {
        DeviceScratch scratch(stream);
        const int rc = inflateDeviceBatch(ctx, members, scratch, &vouched);
        if (rc) return rc;
      }
      for (size_t k = 0; k < members.size(); k++) {
        const int i = index[k];
        const spz::detail::BlockTable &t = tables[i];
        if (!vouched[k]) {  // the host inflater's verdict and bytes; they must fill exactly what the table announced
          std::vector<uint8_t> host;
          if (!spz::decompressGzippedParallel(bytes[i], sizes[i], spz::detail::inflateThreads(), &host)) {
            status[i] = fail(SPZB200_ERR_INVALID, "%s: member %d: not a readable gzip member", who, i);
            continue;
          }
          if (host.size() != t.totalSize) {
            status[i] = fail(SPZB200_ERR_INVALID, "%s: member %d: inflates to %zu bytes, its block table says %llu", who, i, host.size(),
                             (unsigned long long)t.totalSize);
            continue;
          }
          const int rc = bouncedCopy(ctx, out[i], host.data(), host.size(), cudaMemcpyHostToDevice, stream);
          if (rc) return rc;
        }
        outSize[i] = (size_t)t.totalSize;
        if (onDevice) onDevice[i] = vouched[k] ? 1 : 0;
      }
    }
    for (int i = 0; i < count; i++)
      if (status[i]) return SPZB200_ERR_INVALID;
    return SPZB200_OK;
  });
}

}  // namespace

extern "C" {

int spzb200_gzip_device(SpzB200Context *ctx, const uint8_t *data, size_t size, uint8_t **out, size_t *out_size, void *stream) {
  const char *who = "spzb200_gzip_device";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (!out || !out_size) return fail(SPZB200_ERR_INVALID, "%s: null output arguments", who);
  *out = nullptr;
  *out_size = 0;
  if (!data && size) return fail(SPZB200_ERR_INVALID, "%s: null data", who);
  return gzipBatch(ctx, who, &data, &size, 1, out, out_size, (cudaStream_t)stream);
}

int spzb200_gzip_device_batch(SpzB200Context *ctx, const uint8_t *const *data, const size_t *sizes, int32_t count, uint8_t **out,
                              size_t *out_size, void *stream) {
  const char *who = "spzb200_gzip_device_batch";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (count < 0) return fail(SPZB200_ERR_INVALID, "%s: count %d", who, count);
  if (count && (!out || !out_size)) return fail(SPZB200_ERR_INVALID, "%s: null output arguments", who);
  for (int i = 0; i < count; i++) {
    out[i] = nullptr;
    out_size[i] = 0;
  }
  if (count && (!data || !sizes)) return fail(SPZB200_ERR_INVALID, "%s: null data", who);
  for (int i = 0; i < count; i++)
    if (!data[i] && sizes[i]) return fail(SPZB200_ERR_INVALID, "%s: null data[%d]", who, i);
  return gzipBatch(ctx, who, data, sizes, count, out, out_size, (cudaStream_t)stream);
}

int spzb200_save_spz_device(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from, int32_t antialiased, uint8_t **out,
                            size_t *out_size, void *stream) {
  return saveSpzDevice(ctx, "spzb200_save_spz_device", in, 1, from, &antialiased, out, out_size, (cudaStream_t)stream);
}

int spzb200_save_spz_device_batch(SpzB200Context *ctx, const SpzB200Cloud *clouds, int32_t count, int32_t from, const int32_t *antialiased,
                                  uint8_t **out, size_t *out_size, void *stream) {
  return saveSpzDevice(ctx, "spzb200_save_spz_device_batch", clouds, count, from, antialiased, out, out_size, (cudaStream_t)stream);
}

int spzb200_spz_info(const uint8_t *bytes, size_t size, int64_t *num_points, int32_t *sh_degree) {
  const char *who = "spzb200_spz_info";
  if (!bytes || !num_points || !sh_degree) return fail(SPZB200_ERR_INVALID, "%s: null argument", who);
  try {
    std::vector<uint8_t> head;
    if (!spz::detail::inflatePrefix(bytes, size, spz::detail::kContainerHeaderBytes, &head) ||
        head.size() < spz::detail::kContainerHeaderBytes)
      return fail(SPZB200_ERR_INVALID, "%s: not a gzip member holding an .spz header", who);
    uint32_t words[3];
    std::memcpy(words, head.data(), 12);
    if (words[0] != spz::detail::kContainerMagic) return fail(SPZB200_ERR_INVALID, "%s: bad magic 0x%08x", who, words[0]);
    if (words[1] < 1 || words[1] > 3) return fail(SPZB200_ERR_INVALID, "%s: container version %u not in 1..3", who, words[1]);
    if (head[12] > 3) return fail(SPZB200_ERR_INVALID, "%s: SH degree %d not in 0..3", who, (int)head[12]);
    *num_points = words[2];
    *sh_degree = head[12];
    return SPZB200_OK;
  } catch (const std::exception &e) {
    return fail(SPZB200_ERR_NOMEM, "%s: %s", who, e.what());
  }
}

int spzb200_gzip_table_info(const uint8_t *bytes, size_t size, uint64_t *inflated_size, int64_t *blocks) {
  const char *who = "spzb200_gzip_table_info";
  if (!bytes || !inflated_size || !blocks) return fail(SPZB200_ERR_INVALID, "%s: null argument", who);
  try {
    spz::detail::BlockTable t;
    if (!spz::detail::parseBlockTable(bytes, size, &t))
      return fail(SPZB200_ERR_INVALID, "%s: not a gzip member with a block table the parallel inflater trusts", who);
    *inflated_size = t.totalSize;
    *blocks = (int64_t)t.compressed.size();
    return SPZB200_OK;
  } catch (const std::exception &e) {
    return fail(SPZB200_ERR_NOMEM, "%s: %s", who, e.what());
  }
}

int spzb200_gunzip_device(SpzB200Context *ctx, const uint8_t *bytes, size_t size, uint8_t *out, size_t out_capacity, size_t *out_size,
                          int32_t *on_device, void *stream) {
  const char *who = "spzb200_gunzip_device";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (!bytes || !out || !out_size) return fail(SPZB200_ERR_INVALID, "%s: null argument", who);
  int32_t status = SPZB200_OK;
  return gunzipBatch(ctx, who, &bytes, &size, 1, &out, &out_capacity, out_size, on_device, &status, (cudaStream_t)stream);
}

int spzb200_gunzip_device_batch(SpzB200Context *ctx, const uint8_t *const *bytes, const size_t *sizes, int32_t count, uint8_t *const *out,
                                const size_t *out_capacity, size_t *out_size, int32_t *on_device, int32_t *status, void *stream) {
  const char *who = "spzb200_gunzip_device_batch";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (count < 0) return fail(SPZB200_ERR_INVALID, "%s: count %d", who, count);
  if (count == 0) return SPZB200_OK;
  if (!bytes || !sizes || !out || !out_capacity || !out_size || !status) return fail(SPZB200_ERR_INVALID, "%s: null argument", who);
  for (int i = 0; i < count; i++)
    if (!bytes[i] || (!out[i] && out_capacity[i])) return fail(SPZB200_ERR_INVALID, "%s: null bytes[%d] or out[%d]", who, i, i);
  return gunzipBatch(ctx, who, bytes, sizes, count, out, out_capacity, out_size, on_device, status, (cudaStream_t)stream);
}

}  // extern "C"

namespace {

// Table blocks from this size up are loaded through the host route.  Each block is one serial decode on
// the device, so few large blocks leave most of the GPU idle: a 10M SH3 file of 620 zlib blocks of 1 MiB
// (saveSpz) loads in 339 ms on the device route against 293 ms on the host route, while the 9919 blocks
// of 64 KiB of a save_spz_device file load in 129 ms against 262 ms (B200 at 1000 W,
// profiles/r4_device_inflate_timing_unrouted.jsonl; DESIGN.md section 10b).
constexpr size_t kDeviceLoadMaxBlock = (size_t)1 << 20;

// The packed planes of a parsed container whose planes sit at `planes` (struct order).
SpzB200Packed packedOfContainer(const spz::detail::Container &c, uint8_t *const planes[6]) {
  SpzB200Packed in;
  std::memset(&in, 0, sizeof in);
  in.num_points = c.numPoints;
  in.sh_degree = c.shDegree;
  in.fractional_bits = c.fractionalBits;
  in.version = c.half ? SPZB200_STREAM_V1 : c.smallestThree ? SPZB200_STREAM_V3 : SPZB200_STREAM_V2;
  in.positions = planes[0]; in.scales = planes[1]; in.rotations = planes[2];
  in.alphas = planes[3]; in.colors = planes[4]; in.sh = c.shDegree ? planes[5] : nullptr;
  return in;
}

// stream order -> struct order (positions, scales, rotations, alphas, colors, sh)
constexpr int kStructOf[6] = {0, 3, 4, 1, 2, 5};

// load_spz_device's host route: inflate on the host (block-parallel where a table allows), validate, copy
// each plane up and decode on the device.  Its verdict is the file's.  Synchronous.
int loadSpzHostRoute(SpzB200Context *ctx, const char *who, const uint8_t *bytes, size_t size, int32_t to, SpzB200Cloud *out,
                     int32_t *antialiased, cudaStream_t st) {
  std::vector<uint8_t> container;
  if (!spz::decompressGzippedParallel(bytes, size, spz::detail::inflateThreads(), &container))
    return fail(SPZB200_ERR_INVALID, "%s: not a readable gzip member", who);
  spz::detail::Container c;
  if (!spz::detail::parseContainer(container.data(), container.size(), &c))
    return fail(SPZB200_ERR_INVALID, "%s: not an .spz container (bad magic, version, degree or size)", who);
  if (out->num_points != c.numPoints || out->sh_degree != c.shDegree)
    return fail(SPZB200_ERR_INVALID, "%s: out holds %lld points of SH degree %d, the file %d of degree %d (spzb200_spz_info)", who,
                (long long)out->num_points, out->sh_degree, c.numPoints, c.shDegree);
  int rc = checkCloud(out, who);
  if (rc) return rc;
  if (antialiased) *antialiased = c.antialiased ? 1 : 0;
  if (c.numPoints == 0) return SPZB200_OK;
  CU(cudaSetDevice(ctx->device));
  size_t aligned = 0;
  for (int i = 0; i < 6; i++) aligned += alignUp(c.bytes[i], 16);
  DeviceScratch scratch(st);
  uint8_t *base = nullptr;
  CU(scratch.alloc(&base, aligned));
  uint8_t *planes[6];
  for (int i = 0; i < 6; i++) {
    planes[kStructOf[i]] = base;
    if (c.bytes[i]) CU(cudaMemcpyAsync(base, container.data() + c.offset[i], c.bytes[i], cudaMemcpyHostToDevice, st));
    base += alignUp(c.bytes[i], 16);
  }
  const SpzB200Packed in = packedOfContainer(c, planes);
  rc = spzb200_decode_device(ctx, &in, to, out, st);
  if (rc) return rc;
  CU(cudaStreamSynchronize(st));
  return SPZB200_OK;
}

// A file of a load batch that may take the device route: a member with a block table of blocks under
// kDeviceLoadMaxBlock whose header (inflated on the host, 16 bytes) agrees with its `out`.
struct DeviceLoad {
  int index;
  spz::detail::BlockTable t;
  spz::detail::Container c;
};

bool deviceLoadCandidate(const uint8_t *bytes, size_t size, const SpzB200Cloud *out, const char *who, DeviceLoad *d) {
  if (!spz::detail::parseBlockTable(bytes, size, &d->t) || d->t.blockSize >= kDeviceLoadMaxBlock) return false;
  std::vector<uint8_t> head;
  if (!spz::detail::inflatePrefix(bytes, size, spz::detail::kContainerHeaderBytes, &head) || head.size() < spz::detail::kContainerHeaderBytes)
    return false;
  if (!spz::detail::parseContainer(head.data(), (size_t)d->t.totalSize, &d->c)) return false;  // reads the 16 bytes and the size
  if (out->num_points != d->c.numPoints || out->sh_degree != d->c.shDegree || d->c.numPoints == 0) return false;
  return checkCloud(out, who) == SPZB200_OK;
}

// load_spz_device of `count` files (DESIGN.md section 10c).  The device-route candidates are inflated in one
// launch into containers at 16-byte-aligned places of one buffer; one move launch puts every vouched
// container's planes at aligned places; each cloud is decoded by its own launches, queued with no host
// wait in between.  Every other file, and every candidate the device cannot vouch for or whose device
// scratch cannot be allocated, takes the host route alone.  status[i] is the file's verdict; a CUDA or
// allocation failure outside the device route's own scratch ends the call.
int loadBatch(SpzB200Context *ctx, const char *who, const uint8_t *const *bytes, const size_t *sizes, int32_t count, int32_t to,
              SpzB200Cloud *out, int32_t *antialiased, int32_t *status, cudaStream_t st) {
  return guarded(who, nullptr, nullptr, [&]() -> int {
    std::vector<char> hostRoute(count, 1);
    std::vector<DeviceLoad> dev;
    for (int i = 0; i < count; i++) {
      status[i] = SPZB200_OK;
      DeviceLoad d;
      d.index = i;
      if (deviceLoadCandidate(bytes[i], sizes[i], &out[i], who, &d)) dev.push_back(std::move(d));
    }
    if (!dev.empty() && cudaSetDevice(ctx->device) == cudaSuccess) {
      const int n = (int)dev.size();
      std::vector<uint64_t> containerBytes(n), planeBytes(n), containerAt, planesAt;
      for (int k = 0; k < n; k++) {
        containerBytes[k] = dev[k].t.totalSize;
        for (int p = 0; p < 6; p++) planeBytes[k] += alignUp(dev[k].c.bytes[p], 16);
      }
      spzb200::planAligned(containerBytes.data(), n, &containerAt);
      spzb200::planAligned(planeBytes.data(), n, &planesAt);
      DeviceScratch scratch(st);
      uint8_t *containers = nullptr, *base = nullptr;
      std::vector<char> vouched;
      bool inflated = false;
      if (scratch.alloc(&containers, containerAt[n]) == cudaSuccess && scratch.alloc(&base, planesAt[n]) == cudaSuccess) {
        std::vector<InflateMember> members(n);
        for (int k = 0; k < n; k++) members[k] = {bytes[dev[k].index], &dev[k].t, containers + containerAt[k]};
        inflated = inflateDeviceBatch(ctx, members, scratch, &vouched) == SPZB200_OK;
      }
      if (!inflated) cudaGetLastError();
      // From here on a vouched file's result is this route's: its container is what the host route would inflate.
      std::vector<spzb200::MoveSpan> spans;
      std::vector<SpzB200Packed> packed;
      std::vector<int> decoded;
      unsigned long long maxSpan = 0;
      for (int k = 0; inflated && k < n; k++) {
        if (!vouched[k]) continue;
        const int i = dev[k].index;
        const spz::detail::Container &c = dev[k].c;
        hostRoute[i] = 0;
        if (antialiased) antialiased[i] = c.antialiased ? 1 : 0;
        uint8_t *planes[6], *p = base + planesAt[k];
        for (int s = 0; s < 6; s++) {  // plane offsets such as 16 + 9n are not aligned: move the planes
          planes[kStructOf[s]] = p;
          if (c.bytes[s]) {
            spans.push_back({(unsigned long long)(uintptr_t)(containers + containerAt[k] + c.offset[s]), (unsigned long long)(uintptr_t)p,
                             c.bytes[s]});
            maxSpan = std::max<unsigned long long>(maxSpan, c.bytes[s]);
          }
          p += alignUp(c.bytes[s], 16);
        }
        packed.push_back(packedOfContainer(c, planes));
        decoded.push_back(i);
      }
      if (!spans.empty()) {
        spzb200::MoveSpan *dSpans = nullptr;
        int rc = uploadTable(spans, &dSpans, scratch);
        if (rc) return rc;
        int launches = 0;
        CU(spzb200::launchMoveSpans(dSpans, (long long)spans.size(), maxSpan, st, &launches));
        ctx->kernelLaunches += launches;
        for (size_t k = 0; k < decoded.size(); k++) {
          rc = spzb200_decode_device(ctx, &packed[k], to, &out[decoded[k]], st);
          if (rc) return rc;
        }
        CU(cudaStreamSynchronize(st));
      }
    }
    bool failed = false;
    for (int i = 0; i < count; i++) {
      if (!hostRoute[i]) continue;
      const int rc = loadSpzHostRoute(ctx, who, bytes[i], sizes[i], to, &out[i], antialiased ? &antialiased[i] : nullptr, st);
      if (rc == SPZB200_ERR_INVALID) {
        status[i] = rc;
        failed = true;
      } else if (rc) {
        return rc;
      }
    }
    return failed ? SPZB200_ERR_INVALID : SPZB200_OK;
  });
}

}  // namespace

extern "C" {

int spzb200_load_spz_device(SpzB200Context *ctx, const uint8_t *bytes, size_t size, int32_t to, SpzB200Cloud *out,
                            int32_t *antialiased, void *stream) {
  const char *who = "spzb200_load_spz_device";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (!bytes || !out) return fail(SPZB200_ERR_INVALID, "%s: null argument", who);
  if (to < 0 || to > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, to);
  int32_t status = SPZB200_OK;
  return loadBatch(ctx, who, &bytes, &size, 1, to, out, antialiased, &status, (cudaStream_t)stream);
}

int spzb200_load_spz_device_batch(SpzB200Context *ctx, const uint8_t *const *bytes, const size_t *sizes, int32_t count, int32_t to,
                                  SpzB200Cloud *out, int32_t *antialiased, int32_t *status, void *stream) {
  const char *who = "spzb200_load_spz_device_batch";
  if (!ctx) return fail(SPZB200_ERR_INVALID, "%s: null context", who);
  if (count < 0) return fail(SPZB200_ERR_INVALID, "%s: count %d", who, count);
  if (to < 0 || to > 8) return fail(SPZB200_ERR_INVALID, "%s: coordinate system %d", who, to);
  if (count == 0) return SPZB200_OK;
  if (!bytes || !sizes || !out || !status) return fail(SPZB200_ERR_INVALID, "%s: null argument", who);
  for (int i = 0; i < count; i++)
    if (!bytes[i]) return fail(SPZB200_ERR_INVALID, "%s: null bytes[%d]", who, i);
  return loadBatch(ctx, who, bytes, sizes, count, to, out, antialiased, status, (cudaStream_t)stream);
}

}  // extern "C"
