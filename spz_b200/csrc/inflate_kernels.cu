// Device inflater: the table blocks of block-table gzip members -> their slices of the outputs
// (DESIGN.md sections 10 and 10c).
//
// One warp per table block; an InflateBlock descriptor names the block's compressed bytes and its output
// slice, so the blocks of many members, each with its own block size, go to their own outputs in one launch.  The warp's lanes run inflate_format.cuh's decoder in lockstep on identical
// state (no shuffles: they read the same bits and the same shared table entries); the code tables are
// filled lane-parallel in the warp's shared workspace, lane 0 writes literals, and match and stored
// copies are spread over the lanes.  Output goes straight to the block's slice in global memory,
// which also serves as the window.  The block's CRC-32 follows: each lane checksums 1/32 of the slice
// and the lanes' CRCs are combined in a shuffle tree.  All format decisions live in inflate_format.cuh,
// which tests compile for the host.
#include <cuda_runtime.h>
#include <stdint.h>

#include "batch_plan.hpp"
#include "codec_kernels.cuh"
#include "deflate_format.cuh"
#include "inflate_format.cuh"

namespace spzb200 {
namespace {

constexpr int kMaxWarps = 8;

struct WarpSync {
  __device__ __forceinline__ void operator()() const { __syncwarp(); }
};

__device__ __forceinline__ uint32_t crcBytes(const uint32_t *tab, uint32_t c, const uint8_t *p, uint64_t n) {
  uint64_t i = 0;
  for (; i < n && ((uintptr_t)(p + i) & 15); i++) c = tab[(c ^ p[i]) & 0xff] ^ (c >> 8);
  for (; i + 16 <= n; i += 16) {
    const uint4 v = *reinterpret_cast<const uint4 *>(p + i);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
      for (int b = 0; b < 4; b++) c = tab[(c ^ (w[k] >> (8 * b))) & 0xff] ^ (c >> 8);
  }
  for (; i < n; i++) c = tab[(c ^ p[i]) & 0xff] ^ (c >> 8);
  return c;
}

__global__ void __launch_bounds__(kMaxWarps * 32)
    inflateBlocksKernel(const uint8_t *__restrict__ body, const InflateBlock *__restrict__ desc, long long blocks,
                        uint32_t *__restrict__ crcOut, int32_t *__restrict__ status) {
  extern __shared__ __align__(16) uint8_t smemRaw[];
  uint32_t *crcTab = reinterpret_cast<uint32_t *>(smemRaw);
  ifl::Workspace *ws = reinterpret_cast<ifl::Workspace *>(smemRaw + 256 * sizeof(uint32_t)) + (threadIdx.x >> 5);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) crcTab[i] = dfl::crcTableEntry(i);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= blocks) return;
  const InflateBlock d = desc[b];
  const uint32_t len = d.outBytes;
  uint8_t *slice = reinterpret_cast<uint8_t *>(d.out);
  const int st = ifl::inflateBlock(body + d.in, d.inBytes, slice, len, ws, lane, 32, WarpSync{});
  if (st != ifl::kOk) {
    if (lane == 0) status[b] = st;
    return;
  }
  __syncwarp();
  // CRC-32: 16-byte-aligned chunks, one per lane, combined pairwise (lane 0 ends with the slice's CRC)
  const uint64_t chunk = ((len + 31) / 32 + 15) & ~15ull;
  const uint64_t a = min((uint64_t)lane * chunk, (uint64_t)len), e = min(a + chunk, (uint64_t)len);
  uint32_t c = ~crcBytes(crcTab, 0xffffffffu, slice + a, e - a);
  unsigned long long n = e - a;
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t oc = __shfl_down_sync(0xffffffffu, c, o);
    const unsigned long long on = __shfl_down_sync(0xffffffffu, n, o);
    if ((lane & (2 * o - 1)) == 0) {
      c = dfl::crcCombine(c, oc, on);
      n += on;
    }
  }
  if (lane == 0) {
    crcOut[b] = c;
    status[b] = ifl::kOk;
  }
}

}  // namespace

cudaError_t launchInflate(const uint8_t *body, const InflateBlock *blocksDesc, long long blocks, uint32_t *crc, int32_t *status, int smCount,
                          cudaStream_t stream, int *warpsPerCta) {
  // Each block is one serial decode, so the block count of the whole batch bounds the parallelism: with fewer than
  // kMaxWarps blocks per SM (1 MiB zlib blocks: 620 for a 10M SH3 file) every warp gets a CTA of its
  // own so the blocks spread over all SMs; otherwise kMaxWarps warps share a CTA and its CRC table.
  const int warps = blocks >= (long long)kMaxWarps * (smCount > 0 ? smCount : 1) ? kMaxWarps : 1;
  *warpsPerCta = warps;
  const size_t smem = 256 * sizeof(uint32_t) + warps * sizeof(ifl::Workspace);
  cudaError_t e = cudaFuncSetAttribute(inflateBlocksKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long long ctas = (blocks + warps - 1) / warps;
  inflateBlocksKernel<<<(unsigned)ctas, warps * 32, smem, stream>>>(body, blocksDesc, blocks, crc, status);
  return cudaGetLastError();
}

}  // namespace spzb200
