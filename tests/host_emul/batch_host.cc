// TEST-ONLY host build of spz_b200/csrc/batch_plan.hpp: the descriptor tables of the batched device file
// routes, exposed flat so tests check them against a Python restatement without a GPU.  Never part of
// the product library.
//   g++ -O2 -std=c++17 -shared -fPIC batch_host.cc
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../spz_b200/csrc/batch_plan.hpp"

using namespace spzb200;

extern "C" {

// Segments of the batch (at most `cap`); returns their number, or -1 when cap is too small.  first[count + 1].
long long bp_plan_deflate(const unsigned long long *src, const uint64_t *sizes, int count, uint64_t *first, DeflateSegment *segs,
                          long long cap) {
  std::vector<DeflateSegment> s;
  std::vector<uint64_t> f;
  planDeflate(src, sizes, count, &s, &f);
  std::memcpy(first, f.data(), f.size() * sizeof(uint64_t));
  if ((long long)s.size() > cap) return -1;
  std::memcpy(segs, s.data(), s.size() * sizeof(DeflateSegment));
  return (long long)s.size();
}

// bodyStart[count + 1]; blockBytes: every member's table blocks, member after member (at most `cap`);
// nBlocks[count].  Returns the number of table blocks, or -1 when cap is too small.
long long bp_member_bodies(const uint32_t *segBytes, const uint64_t *first, int count, uint64_t *bodyStart, uint32_t *blockBytes,
                           uint64_t *nBlocks, long long cap) {
  std::vector<uint64_t> f(first, first + count + 1), b;
  std::vector<std::vector<uint32_t>> blocks;
  planMemberBodies(segBytes, f, &b, &blocks);
  std::memcpy(bodyStart, b.data(), b.size() * sizeof(uint64_t));
  long long n = 0;
  for (int i = 0; i < count; i++) {
    nBlocks[i] = blocks[i].size();
    for (uint32_t v : blocks[i]) {
      if (n >= cap) return -1;
      blockBytes[n++] = v;
    }
  }
  return n;
}

// blocks[sum nBlocks], first[count + 1], bodyStart[count + 1].
void bp_plan_inflate(int count, const uint64_t *blockSize, const uint64_t *total, const uint64_t *nBlocks, const uint32_t *compressed,
                     const unsigned long long *out, InflateBlock *blocks, uint64_t *first, uint64_t *bodyStart) {
  std::vector<InflateBlock> b;
  std::vector<uint64_t> f, s;
  planInflate(count, blockSize, total, nBlocks, compressed, out, &b, &f, &s);
  std::memcpy(blocks, b.data(), b.size() * sizeof(InflateBlock));
  std::memcpy(first, f.data(), f.size() * sizeof(uint64_t));
  std::memcpy(bodyStart, s.data(), s.size() * sizeof(uint64_t));
}

// at[count + 1]
void bp_plan_aligned(const uint64_t *sizes, int count, uint64_t *at) {
  std::vector<uint64_t> a;
  planAligned(sizes, count, &a);
  std::memcpy(at, a.data(), a.size() * sizeof(uint64_t));
}

int bp_sizes(int *seg, int *block, int *span) {
  *seg = (int)sizeof(DeflateSegment);
  *block = (int)sizeof(InflateBlock);
  *span = (int)sizeof(MoveSpan);
  return dfl::kSegBytes;
}

}  // extern "C"
