// Plane moves of the batched file routes (DESIGN.md section 10c): a table of MoveSpan copies, device to
// device, in one launch -- the encoder's aligned planes and the headers into the containers of a save,
// the planes of inflated containers (at offsets such as 16 + 9n) to 16-byte-aligned places for the
// decoder on a load.
//
// CTA (x, y) copies part y of span x; the parts of a span stride over it in 16-byte vectors of its
// destination.  Bytes before the destination's first 16-byte boundary and after its last one are copied
// one by one.  When the source is misaligned against the destination, each vector is assembled from the
// two aligned source vectors it straddles: both hold bytes of the span, so neither read leaves the source.
#include <cuda_runtime.h>
#include <stdint.h>

#include "batch_plan.hpp"
#include "codec_kernels.cuh"

namespace spzb200 {
namespace {

constexpr int kMoveThreads = 256;
constexpr unsigned long long kMoveStep = kMoveThreads * 16;  // bytes one CTA moves per pass
constexpr long long kMoveCtas = 1 << 18;                     // bound on spans * parts

// Bytes k .. 15 of lo followed by bytes 0 .. k - 1 of hi (k in 1 .. 15).
__device__ __forceinline__ uint4 straddle(const uint4 lo, const uint4 hi, int k) {
  uint32_t a0, a1, a2, a3, a4;
  switch (k >> 2) {
    case 0: a0 = lo.x; a1 = lo.y; a2 = lo.z; a3 = lo.w; a4 = hi.x; break;
    case 1: a0 = lo.y; a1 = lo.z; a2 = lo.w; a3 = hi.x; a4 = hi.y; break;
    case 2: a0 = lo.z; a1 = lo.w; a2 = hi.x; a3 = hi.y; a4 = hi.z; break;
    default: a0 = lo.w; a1 = hi.x; a2 = hi.y; a3 = hi.z; a4 = hi.w; break;
  }
  const int r = (k & 3) * 8;
  return make_uint4(__funnelshift_r(a0, a1, r), __funnelshift_r(a1, a2, r), __funnelshift_r(a2, a3, r), __funnelshift_r(a3, a4, r));
}

__global__ void __launch_bounds__(kMoveThreads) moveSpansKernel(const MoveSpan *__restrict__ spans) {
  const MoveSpan m = spans[blockIdx.x];
  const uint8_t *src = reinterpret_cast<const uint8_t *>(m.src);
  uint8_t *dst = reinterpret_cast<uint8_t *>(m.dst);
  const unsigned long long n = m.bytes;
  const unsigned long long head = min(n, (16 - (m.dst & 15)) & 15);
  const unsigned long long vecs = (n - head) / 16, tail = head + vecs * 16;
  const int tid = threadIdx.x;
  if (blockIdx.y == 0) {
    if (tid < head) dst[tid] = src[tid];
    if (tail + tid < n) dst[tail + tid] = src[tail + tid];
  }
  uint4 *d4 = reinterpret_cast<uint4 *>(dst + head);
  const unsigned long long first = (unsigned long long)blockIdx.y * kMoveThreads + tid, stride = (unsigned long long)gridDim.y * kMoveThreads;
  const int k = (int)((m.src + head) & 15);
  if (k == 0) {
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src + head);
    for (unsigned long long v = first; v < vecs; v += stride) d4[v] = s4[v];
  } else {
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src + head - k);
    for (unsigned long long v = first; v < vecs; v += stride) d4[v] = straddle(s4[v], s4[v + 1], k);
  }
}

}  // namespace

cudaError_t launchMoveSpans(const MoveSpan *spans, long long count, unsigned long long maxBytes, cudaStream_t stream, int *launches) {
  *launches = 0;
  if (count == 0) return cudaSuccess;
  long long parts = (long long)((maxBytes + kMoveStep - 1) / kMoveStep);
  parts = max(1ll, min(parts, max(1ll, kMoveCtas / count)));
  moveSpansKernel<<<dim3((unsigned)count, (unsigned)min(parts, 65535ll)), kMoveThreads, 0, stream>>>(spans);
  *launches = 1;
  return cudaGetLastError();
}

}  // namespace spzb200
