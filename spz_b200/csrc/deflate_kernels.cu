// Device deflater: device inputs -> raw deflate segments -> one contiguous body (DESIGN.md sections 10
// and 10c).
//
// One CTA per 64 KiB segment; a DeflateSegment descriptor names its bytes and whether it ends its input,
// so the segments of many inputs are coded in one launch.  The segment is staged in shared memory with one bulk async copy; the
// symbols (literals, distance-1 matches for runs) are found by every thread for its 128-byte slice --
// a run crossing slices belongs to the slice it starts in, whose thread learns its full length from a
// CTA-wide pointer-jumping pass over the slices' head runs.  A histogram, the length-limited code
// (package-merge, per-item steps spread over the threads), the header (one thread), a scan of the
// threads' bit counts and an OR-assembly of the codes into shared words follow; the coded segment (or
// its stored form, when that is not larger) goes to the segment's worst-case slot.  A second kernel
// scans the segment sizes of the whole batch and a third packs the slots into one body, each input's
// segments at a contiguous range of it.  All format decisions live in
// deflate_format.cuh, which tests compile for the host.
#include <cuda_runtime.h>
#include <stdint.h>

#include "batch_plan.hpp"
#include "codec_kernels.cuh"
#include "deflate_format.cuh"
#include "kernel_utils.cuh"

namespace spzb200 {
namespace {

using namespace dfl;

constexpr int kThreads = 512;
constexpr int kSlice = kSegBytes / kThreads;
constexpr int kWarps = kThreads / 32;

struct DeflateSmem {
  alignas(16) uint8_t in[kSegBytes];
  alignas(16) uint32_t out[kSlotBytes / 4];
  uint32_t freq[kLitLenSyms];
  uint32_t crcTab[256];
  uint32_t sortW[kLitLenSyms];
  uint32_t list[2][2 * kLitLenSyms];
  uint16_t sortSym[kLitLenSyms];
  uint16_t leafPos[kMaxBits * kLitLenSyms];
  uint16_t codes[kLitLenSyms];
  uint8_t lens[kLitLenSyms];
  uint8_t byRank[kLitLenSyms];
  uint32_t runVal[2][kThreads];
  uint8_t runLink[2][kThreads];
  uint32_t crc[kThreads];
  uint32_t warpSum[kWarps];
  DynHeader hdr;
  alignas(8) unsigned long long bar;
};

__global__ void __launch_bounds__(kThreads, 1)
    deflateSegmentsKernel(const DeflateSegment *__restrict__ desc, uint8_t *__restrict__ slots, uint32_t *__restrict__ segBytes,
                          uint32_t *__restrict__ segCrc) {
  extern __shared__ __align__(16) uint8_t smemRaw[];
  DeflateSmem &S = *reinterpret_cast<DeflateSmem *>(smemRaw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned long long seg = blockIdx.x;
  const DeflateSegment d = desc[seg];
  const int len = (int)d.len;
  const bool last = d.last != 0;
  const uint8_t *g = reinterpret_cast<const uint8_t *>(d.src);

  // ---- stage the segment; clear the output words and the histogram --------------------------------
  const int bulkBytes = (d.src & 15) == 0 ? (len & ~15) : 0;
  if (tid == 0 && bulkBytes) {
    mbarInit(&S.bar);
    bulkLoad(S.in, g, (uint32_t)bulkBytes, &S.bar);
  }
  for (int i = bulkBytes + tid; i < len; i += kThreads) S.in[i] = g[i];
  for (int i = tid; i < kSlotBytes / 4; i += kThreads) S.out[i] = 0;
  for (int i = tid; i < kLitLenSyms; i += kThreads) S.freq[i] = 0;
  if (tid < 256) S.crcTab[tid] = crcTableEntry(tid);
  __syncthreads();
  if (bulkBytes) mbarWait(&S.bar, 0);
  __syncthreads();

  // ---- this thread's slice: CRC-32 and the run it starts with -------------------------------------
  const int a = min(tid * kSlice, len), b = min(tid * kSlice + kSlice, len);
  int head = 0;
  {
    uint32_t c = 0xffffffffu;
    for (int p = a; p < b; p++) c = S.crcTab[(c ^ S.in[p]) & 0xff] ^ (c >> 8);
    S.crc[tid] = ~c;
    if (a < b) {
      head = 1;
      while (a + head < b && S.in[a + head] == S.in[a]) head++;
    }
  }
  const bool continues = b < len && S.in[b] == S.in[b - 1];  // the slice's last run goes on into the next slice
  S.runVal[0][tid] = (uint32_t)head;
  S.runLink[0][tid] = (a < b && head == b - a && continues) ? 1 : 0;
  __syncthreads();
  // runVal -> length of the run starting at slice t's first byte, across slices (pointer jumping)
  int cur = 0;
  for (int d = 1; d < kThreads; d <<= 1) {
    uint32_t v = S.runVal[cur][tid];
    uint8_t l = S.runLink[cur][tid];
    if (l && tid + d < kThreads) {
      v += S.runVal[cur][tid + d];
      l = S.runLink[cur][tid + d];
    }
    S.runVal[cur ^ 1][tid] = v;
    S.runLink[cur ^ 1][tid] = l;
    __syncthreads();
    cur ^= 1;
  }
  const int ext = continues ? (int)S.runVal[cur][tid + 1] : 0;
  // the symbols this thread owns: the runs that start in its slice, at their full length
  auto tokens = [&](auto &&f) {
    int p = (a > 0 && a < b && S.in[a] == S.in[a - 1]) ? a + head : a;  // a run from an earlier slice goes on here
    while (p < b) {
      const uint8_t c = S.in[p];
      int q = p + 1;
      while (q < b && S.in[q] == c) q++;
      const int run = q - p + (q == b ? ext : 0);
      runTokens(run, [&](int m) { f(c, m); });
      p = q;
    }
  };

  // ---- histogram, segment CRC ----------------------------------------------------------------------
  tokens([&](uint8_t c, int m) {
    int s = c;
    if (m) {
      int eb, ev;
      lengthSymbol(m, &s, &eb, &ev);
    }
    atomicAdd(&S.freq[s], 1u);
  });
  for (int d = 1; d < kThreads; d <<= 1) {
    __syncthreads();
    if ((tid & (2 * d - 1)) == 0 && tid + d < kThreads) {
      const int ra = min((tid + d) * kSlice, len), rb = min((tid + 2 * d) * kSlice, len);
      S.crc[tid] = crcCombine(S.crc[tid], S.crc[tid + d], (uint64_t)(rb - ra));
    }
  }
  if (tid == 0) {
    S.freq[kEob] = 1;
    ensureTwo(S.freq, kLitLenSyms);
  }
  __syncthreads();

  // ---- length-limited code: rank the symbols, package-merge level by level ------------------------
  const int n = __syncthreads_count(tid < kLitLenSyms && S.freq[tid] != 0);
  if (tid < kLitLenSyms && S.freq[tid]) {
    const int r = rankOf(S.freq, kLitLenSyms, tid);
    S.sortW[r] = S.freq[tid];
    S.sortSym[r] = (uint16_t)tid;
  }
  __syncthreads();
  int prevItems = 0;
  for (int d = kMaxBits - 1; d >= 0; d--) {
    const int np = d == kMaxBits - 1 ? 0 : prevItems / 2;
    for (int item = tid; item < n + np; item += kThreads)
      pmPlace(S.sortW, n, S.list[(d + 1) & 1], np, S.list[d & 1], S.leafPos + d * kLitLenSyms, item);
    prevItems = n + np;
    __syncthreads();
  }
  if (tid == 0) {
    pmLengths(S.leafPos, kLitLenSyms, n, kMaxBits, S.byRank);
    for (int s = 0; s < kLitLenSyms; s++) S.lens[s] = 0;
    for (int r = 0; r < n; r++) S.lens[S.sortSym[r]] = S.byRank[r];
    canonicalCodes(S.lens, kLitLenSyms, S.codes);
    planHeader(S.lens, &S.hdr);
  }
  __syncthreads();

  // ---- bit offsets: each thread's symbol bits, exclusive scan over the CTA -------------------------
  uint32_t myBits = 0;
  tokens([&](uint8_t c, int m) {
    if (!m) {
      myBits += S.lens[c];
      return;
    }
    int s, eb, ev;
    lengthSymbol(m, &s, &eb, &ev);
    myBits += S.lens[s] + eb + kDistBits;
  });
  uint32_t x = myBits;
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) S.warpSum[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < kWarps ? S.warpSum[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    __syncwarp();
    if (lane < kWarps) S.warpSum[lane] = w;
  }
  __syncthreads();
  const uint32_t before = (warp ? S.warpSum[warp - 1] : 0) + x - myBits;
  const uint32_t symbolBits = S.warpSum[kWarps - 1];

  const uint32_t dynBytes = dynamicBytes(S.hdr.bits + symbolBits + S.lens[kEob], last);
  const uint32_t stBytes = storedBytes((uint32_t)len);
  uint8_t *slot = slots + seg * kSlotBytes;
  if (dynBytes < stBytes) {
    if (tid == 0) {
      BitWriter bw{S.out, 0};
      writeHeader(S.hdr, last, bw);
    }
    __syncthreads();
    // codes, LSB first, OR-ed into the shared words (neighbouring threads share the boundary words)
    uint64_t acc = 0;
    int nb = (int)((S.hdr.bits + before) & 31);
    uint32_t w = (S.hdr.bits + before) >> 5;
    auto put = [&](uint32_t v, int bits) {
      acc |= (uint64_t)v << nb;
      nb += bits;
      if (nb >= 32) {
        atomicOr(&S.out[w++], (uint32_t)acc);
        acc >>= 32;
        nb -= 32;
      }
    };
    tokens([&](uint8_t c, int m) {
      if (!m) {
        put(S.codes[c], S.lens[c]);
        return;
      }
      int s, eb, ev;
      lengthSymbol(m, &s, &eb, &ev);
      put(S.codes[s], S.lens[s]);
      if (eb) put((uint32_t)ev, eb);
      put(0, kDistBits);  // distance code 0: distance 1
    });
    if (nb > 0) atomicOr(&S.out[w], (uint32_t)acc);
    __syncthreads();
    if (tid == 0) {
      BitWriter bw{S.out, S.hdr.bits + symbolBits};
      bw.put(S.codes[kEob], S.lens[kEob]);
      if (!last) {
        bw.put(0, 3);                 // empty stored block (sync flush) ...
        bw.pos = (bw.pos + 7) & ~7u;  // ... byte-aligned ...
        bw.put(0xffff0000u, 32);      // ... LEN 0000, NLEN ffff
      }
    }
    __syncthreads();
    const int vecs = (int)((dynBytes + 15) / 16);
    for (int i = tid; i < vecs; i += kThreads) reinterpret_cast<uint4 *>(slot)[i] = reinterpret_cast<const uint4 *>(S.out)[i];
  } else {
    for (int i = tid; i < len; i += kThreads) slot[i + 5 * (i / kStoredMax + 1)] = S.in[i];
    const int blocks = len == 0 ? 1 : (len + kStoredMax - 1) / kStoredMax;
    if (tid < blocks) storedHeaderAt((uint32_t)len, last, (uint32_t)tid, slot);
  }
  if (tid == 0) {
    segBytes[seg] = dynBytes < stBytes ? dynBytes : stBytes;
    segCrc[seg] = S.crc[0];
  }
}

// offsets[s] = bytes of segments [0, s); offsets[segments] = the body's size.  One CTA.
constexpr int kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads)
    segmentOffsetsKernel(const uint32_t *__restrict__ segBytes, unsigned long long segments, unsigned long long *__restrict__ offsets) {
  __shared__ unsigned long long part[kScanThreads];
  const int tid = threadIdx.x;
  const unsigned long long per = (segments + kScanThreads - 1) / kScanThreads;
  const unsigned long long lo = min(segments, tid * per), hi = min(segments, lo + per);
  unsigned long long sum = 0;
  for (unsigned long long s = lo; s < hi; s++) sum += segBytes[s];
  part[tid] = sum;
  __syncthreads();
  for (int d = 1; d < kScanThreads; d <<= 1) {  // inclusive scan
    const unsigned long long v = tid >= d ? part[tid - d] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  unsigned long long run = part[tid] - sum;
  for (unsigned long long s = lo; s < hi; s++) {
    offsets[s] = run;
    run += segBytes[s];
  }
  if (tid == kScanThreads - 1) offsets[segments] = part[tid];
}

// Every slot's coded bytes to its place in the body.
__global__ void __launch_bounds__(256)
    packSlotsKernel(const uint8_t *__restrict__ slots, const uint32_t *__restrict__ segBytes,
                    const unsigned long long *__restrict__ offsets, uint8_t *__restrict__ body) {
  const unsigned long long seg = blockIdx.x;
  const uint8_t *from = slots + seg * kSlotBytes;
  uint8_t *to = body + offsets[seg];
  const uint32_t bytes = segBytes[seg];
  for (uint32_t i = threadIdx.x * 4; i < bytes; i += blockDim.x * 4) {
    const uint32_t w = *reinterpret_cast<const uint32_t *>(from + i);  // slots are 16-byte aligned
    const uint32_t k = bytes - i < 4 ? bytes - i : 4;
    for (uint32_t j = 0; j < k; j++) to[i + j] = (uint8_t)(w >> (8 * j));
  }
}

}  // namespace

size_t deflateSlotBytes() { return kSlotBytes; }

cudaError_t launchDeflate(const DeflateSegment *segs, unsigned long long segments, uint8_t *slots, uint32_t *segBytes, uint32_t *segCrc,
                          unsigned long long *offsets, uint8_t *body, cudaStream_t stream, int *launches) {
  cudaError_t e = cudaFuncSetAttribute(deflateSegmentsKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DeflateSmem));
  if (e != cudaSuccess) return e;
  deflateSegmentsKernel<<<(unsigned)segments, kThreads, sizeof(DeflateSmem), stream>>>(segs, slots, segBytes, segCrc);
  segmentOffsetsKernel<<<1, kScanThreads, 0, stream>>>(segBytes, segments, offsets);
  packSlotsKernel<<<(unsigned)segments, 256, 0, stream>>>(slots, segBytes, offsets, body);
  *launches = 3;
  return cudaGetLastError();
}

}  // namespace spzb200
