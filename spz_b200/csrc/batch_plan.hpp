// Descriptor tables of the batched device file routes (DESIGN.md section 10c): which bytes each CTA or
// warp of the deflate, inflate and plane-move kernels reads and writes when one launch serves many
// files.  Plain host code over integers (device addresses are carried as unsigned long long), shared by
// cabi.cu and tests/host_emul/batch_host.cc, which checks it against a Python restatement without a GPU.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "deflate_format.cuh"

namespace spzb200 {

// One 64 KiB segment of one deflater input: `len` bytes at address `src`; `last` = 1 for the input's
// final segment (BFINAL), 0 for the others (ended by the sync-flush marker).
struct DeflateSegment {
  unsigned long long src;
  uint32_t len;
  uint32_t last;
};

// One table block of one gzip member: inBytes raw deflate bytes at `in` (an offset into the batch's
// compressed body buffer) inflate to exactly outBytes bytes at address `out`.
struct InflateBlock {
  unsigned long long in, out;
  uint32_t inBytes, outBytes;
};

// `bytes` bytes from address src to address dst (the plane-move kernel).
struct MoveSpan {
  unsigned long long src, dst, bytes;
};

// Inputs i of sizes[i] bytes at src[i] -> their segments, input by input: segment s of input i covers
// bytes [s * kSegBytes, ...) of it, and an empty input is one empty final segment (dfl::segmentCount).
// first[i] = index of input i's first segment, first[count] = the batch's segment count.
inline void planDeflate(const unsigned long long *src, const uint64_t *sizes, int count, std::vector<DeflateSegment> *segs,
                        std::vector<uint64_t> *first) {
  first->assign((size_t)count + 1, 0);
  for (int i = 0; i < count; i++) (*first)[i + 1] = (*first)[i] + dfl::segmentCount(sizes[i]);
  segs->resize((*first)[count]);
  for (int i = 0; i < count; i++) {
    const uint64_t n = (*first)[i + 1] - (*first)[i];
    for (uint64_t s = 0; s < n; s++) {
      const uint64_t off = s * dfl::kSegBytes;
      DeflateSegment &d = (*segs)[(*first)[i] + s];
      d.src = src[i] + off;
      d.len = (uint32_t)(sizes[i] - off < (uint64_t)dfl::kSegBytes ? sizes[i] - off : dfl::kSegBytes);
      d.last = s + 1 == n ? 1u : 0u;
    }
  }
}

// After the deflate kernels: segBytes[s] = coded bytes of segment s.  bodyStart[i] = where input i's body
// begins in the batch's body buffer (the exclusive scan of segBytes at first[i]); bodyStart[count] = the
// whole body.  blockBytes[i] = the compressed sizes of input i's gzip table blocks, each the fewest whole
// segments that keep the table within dfl::kMaxTableBlocks entries (dfl::segmentsPerBlock).
inline void planMemberBodies(const uint32_t *segBytes, const std::vector<uint64_t> &first, std::vector<uint64_t> *bodyStart,
                             std::vector<std::vector<uint32_t>> *blockBytes) {
  const size_t count = first.size() - 1;
  bodyStart->assign(count + 1, 0);
  blockBytes->assign(count, {});
  for (size_t i = 0; i < count; i++) {
    const uint64_t segs = first[i + 1] - first[i], per = dfl::segmentsPerBlock(segs);
    std::vector<uint32_t> &b = (*blockBytes)[i];
    b.assign((segs + per - 1) / per, 0);
    uint64_t body = 0;
    for (uint64_t s = 0; s < segs; s++) {
      b[s / per] += segBytes[first[i] + s];
      body += segBytes[first[i] + s];
    }
    (*bodyStart)[i + 1] = (*bodyStart)[i] + body;
  }
}

// Members i with table blocks of blockSize[i] inflated bytes (the last one holds the rest of total[i]),
// whose nBlocks[i] compressed sizes follow one another in `compressed`, inflated to address out[i].
// Their bodies are laid end to end in one buffer: bodyStart[i] (count + 1 entries) is member i's.
// first[i] = index of member i's first block in `blocks`.
inline void planInflate(int count, const uint64_t *blockSize, const uint64_t *total, const uint64_t *nBlocks, const uint32_t *compressed,
                        const unsigned long long *out, std::vector<InflateBlock> *blocks, std::vector<uint64_t> *first,
                        std::vector<uint64_t> *bodyStart) {
  first->assign((size_t)count + 1, 0);
  bodyStart->assign((size_t)count + 1, 0);
  for (int i = 0; i < count; i++) (*first)[i + 1] = (*first)[i] + nBlocks[i];
  blocks->resize((*first)[count]);
  uint64_t in = 0;
  for (int i = 0; i < count; i++) {
    (*bodyStart)[i] = in;
    for (uint64_t k = 0; k < nBlocks[i]; k++) {
      const uint64_t at = (*first)[i] + k, start = k * blockSize[i];
      InflateBlock &d = (*blocks)[at];
      d.in = in;
      d.out = out[i] + start;
      d.inBytes = compressed[at];
      d.outBytes = (uint32_t)(k + 1 == nBlocks[i] ? total[i] - start : blockSize[i]);
      in += compressed[at];
    }
  }
  (*bodyStart)[count] = in;
}

// Places of `count` buffers of sizes[i] bytes end to end in one allocation, each at a multiple of 16:
// at[i], and at[count] = the allocation's size.
inline void planAligned(const uint64_t *sizes, int count, std::vector<uint64_t> *at) {
  at->assign((size_t)count + 1, 0);
  for (int i = 0; i < count; i++) (*at)[i + 1] = (*at)[i] + (sizes[i] + 15) / 16 * 16;
}

}  // namespace spzb200
