// Launch interface of the codec kernels (internal to the library; the public boundary is the
// C-ABI in include/spz_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spzb200 {

// GaussianCloud planes (splat-types.h:90-115) -> PackedGaussians planes (load-spz.h:42-59),
// both device-resident.  n gaussians, shDim in {0,3,8,15}.
struct EncodeArgs {
  const float *positions, *scales, *rotations, *alphas, *colors, *sh;
  uint8_t *oPositions, *oScales, *oRotations, *oAlphas, *oColors, *oSh;
  long long n;
  int shDim;
  int version;                    // 3: smallest-three rotations, 4 bytes each (what the reference writes); 2: first-three, 3 bytes
                                  // each (upstream's earlier form: parity unpinned, codec_math.cuh: quant_rotation_first3)
  uint32_t flipP, flipQ, flipSh;  // sign-bit sets of coordinateConverter(from, RUB)
  const float *alphaThresholds;   // device, 256 floats (255 thresholds + +Inf pad)
};

struct DecodeArgs {
  const uint8_t *positions, *scales, *rotations, *alphas, *colors, *sh;
  float *oPositions, *oScales, *oRotations, *oAlphas, *oColors, *oSh;
  long long n;
  int shDim;
  int version;                    // 1: half positions + first-three; 2: 24-bit + first-three; 3
  float positionScale;            // (float)(1.0 / (1 << fractionalBits)), load-spz.cc:495
  uint32_t flipP, flipQ, flipSh;  // sign-bit sets of coordinateConverter(RUB, to)
  const float *tables;            // device, kDecodeTableFloats floats: [0,256) alpha LUT
                                  // invSigmoid(a / 255.0f) (host-built, libm logf), [256,512)
                                  // colour LUT, [512,1024) smallest-three magnitudes (device-built)
};

constexpr int kDecodeTableFloats = 1024;

// GaussianCloud planes -> the planes launchDecode(launchEncode(x)) gives back, both device-resident,
// without packed planes in between (quantize_kernels.cu).  An output plane may be its input plane (in
// place); no other overlap is allowed.  Positions use 12 fractional bits, as the encoder writes them.
struct QuantizeArgs {
  const float *positions, *scales, *rotations, *alphas, *colors, *sh;
  float *oPositions, *oScales, *oRotations, *oAlphas, *oColors, *oSh;
  long long n;
  int shDim;
  int version;                       // 3: smallest-three rotations; 2: first-three (as EncodeArgs)
  uint32_t flipP, flipQ, flipSh;     // sign-bit sets of coordinateConverter(from, RUB)
  uint32_t oFlipP, oFlipQ, oFlipSh;  // sign-bit sets of coordinateConverter(RUB, to)
  const float *alphaThresholds;      // as EncodeArgs
  const float *tables;               // as DecodeArgs
};

// PLY vertex records (row-major, `width` floats per vertex) -> PackedGaussians planes, both
// device-resident: loadSplatFromPly's column shuffle (load-spz.cc:808-838) fused with packGaussians.
struct PlyEncodeArgs {
  const float *rows;
  long long n;
  int width;   // floats per record
  int shDim;   // 0, 3, 8, 15
  int colPos[3], colScale[3], colRot[4] /* x, y, z, w */, colAlpha, colColor[3];
  int colRest[45];  // f_rest_0 .. : channel-major [C][S], as the file stores them
  uint8_t *oPositions, *oScales, *oRotations, *oAlphas, *oColors, *oSh;
  uint32_t flipP, flipQ, flipSh;  // sign-bit sets of coordinateConverter(from, RUB)
  const float *alphaThresholds;
};

constexpr int kMaxUnmappedColumns = 64;

// PackedGaussians planes -> PLY vertex records: unpackGaussians fused with saveSplatToPly's row
// layout (load-spz.cc:846-934).  Columns no plane maps to (nx, ny, nz, extras) are written as 0.
struct PlyDecodeArgs {
  const uint8_t *positions, *scales, *rotations, *alphas, *colors, *sh;
  float *rows;
  long long n;
  int width, shDim, version;
  float positionScale;
  int colPos[3], colScale[3], colRot[4] /* x, y, z, w */, colAlpha, colColor[3];
  int colRest[45];
  int numUnmapped;                          // columns no plane maps to, or -1 if more than the list holds
  uint16_t unmapped[kMaxUnmappedColumns];
  uint32_t flipP, flipQ, flipSh;  // sign-bit sets of coordinateConverter(RUB, to)
  const float *tables;
};

// Batched PackedGaussians::at(i) + PackedGaussian::unpack (load-spz.cc:383-463), gather_kernels.cu.
// Either `records` (n x 65-byte PackedGaussian) or the six packed planes (+ optional index list) is
// the source; `out` receives n x 59 floats (UnpackedGaussian).  All pointers are device-accessible.
struct GatherArgs {
  const uint8_t *records;  // non-null: array of PackedGaussian; null: gather from the planes below
  const uint8_t *positions, *scales, *rotations, *alphas, *colors, *sh;
  const long long *indices;  // null = gaussians 0..n-1 of the planes
  float *out;
  long long n;
  int shDim;
  int version;             // stream flavour 1..4 (include/spz_b200.h)
  float positionScale;     // (float)(1.0 / (1 << fractionalBits))
  float flipP[3], flipQ[3], flipSh[15];  // the caller's CoordinateConverter, applied by multiplication
  const float *tables;
};
cudaError_t launchUnpackRecords(const GatherArgs &a, cudaStream_t stream, int *launches);

enum PackMode { kPackAlu = 0, kPackCvt = 1 };

struct LaunchPlan {
  int smCount;
  int packMode;        // encode only: how four bytes are saturated and packed into a word
  bool forceGeneric;   // test hook: route everything through the scalar kernels
  int ctasPerSm;       // persistent grid only: smCount * ctasPerSm CTAs (1..4); 0 = default (4)
  bool flatGrid;       // one CTA per tile (default) instead of persistent grid-stride CTAs
  bool decodeBulk;     // decode the SH plane through bulk async copies (TMA) instead of registers
  int encodeBulk;      // planar encoder through the one-thread-per-gaussian bulk-copy kernel: 0 never, 1 where it measured
                       // faster (SH degree 3 up to 24M gaussians per launch, degree 2 from 1M to 24M, degree 1 up to 6M; default), 2 wherever it exists
  int decodePerGaussian;   // planar decoder through the one-thread-per-gaussian bulk-copy kernel: 0 never, 1 where it
                           // measured faster (SH degree 1 - 3; default), 2 also for SH-less clouds
  int smallTilesEncode, smallTilesDecode;  // 128-thread tile geometry for SH degree 0 - 2: 0 never, 1 up to 16M gaussians per launch, 2 always.
                                            // Defaults: encoder always, decoder never (measured); SPZB200_TILE=128 / 320 set both
  bool pdl;            // launch with programmatic stream serialization (kernel_utils.cuh); default on, SPZB200_PDL=0 turns it off
  bool foldRest;       // the sub-tile remainder rides in the vector kernel's first CTA(s) instead of a launch of its own (default)
  bool plyMapped;      // test hook: PLY rows always through the column-map kernels, never the canonical-layout ones
};

// Number of kernels launched is returned through *launches (0, 1 or 2).
cudaError_t launchEncode(const EncodeArgs &a, const LaunchPlan &plan, cudaStream_t stream,
                         int *launches);
cudaError_t launchDecode(const DecodeArgs &a, const LaunchPlan &plan, cudaStream_t stream,
                         int *launches);
// One launch (none for n = 0); uses plan.pdl only.
cudaError_t launchQuantize(const QuantizeArgs &a, const LaunchPlan &plan, cudaStream_t stream, int *launches);

cudaError_t launchEncodePly(const PlyEncodeArgs &a, const LaunchPlan &plan, cudaStream_t stream, int *launches);
cudaError_t launchDecodePly(const PlyDecodeArgs &a, const LaunchPlan &plan, cudaStream_t stream, int *launches);
int plyTileGaussians();
// canonical property order only (pergaussian_kernels.cu); *done = leading gaussians handled
cudaError_t launchEncodePlyCanonical(const PlyEncodeArgs &a, const LaunchPlan &plan, cudaStream_t stream, long long *done);
cudaError_t launchEncodePerGaussianPlanar(const EncodeArgs &a, const LaunchPlan &plan, cudaStream_t stream, long long *done);
cudaError_t launchDecodePerGaussianPlanar(const DecodeArgs &a, const LaunchPlan &plan, cudaStream_t stream, long long *done);
cudaError_t launchDecodePlyCanonical(const PlyDecodeArgs &a, const LaunchPlan &plan, cudaStream_t stream, long long *done);

// Gaussians per tile of the vector kernels for a given shDim (the sharding granule).
int tileGaussians(int shDim);

// Fills tables[256, 1024) on the device (colour LUT load-spz.cc:522, smallest-three magnitude LUT
// load-spz.cc:367); tables[0, 256) is uploaded by the caller.
cudaError_t buildDecodeTables(float *tables, cudaStream_t stream);

// Device self-check of the division identities of the rotation quantizer (see divisionSelfCheckKernel).
cudaError_t divisionSelfCheck(int part, unsigned long long pairsPerThread, unsigned long long seed, int smCount, cudaStream_t stream,
                              unsigned long long *wrong, unsigned long long *checked);

// Runs both byte packers on probe values; *ok = 1 when cvt.pack.sat.u8.s32.b32 orders and
// saturates bytes the way the kernels assume (decided once per context).  `scratch` = one device int.
cudaError_t probePackCvt(cudaStream_t stream, int *scratch, int *ok);

struct DeflateSegment;
struct InflateBlock;
struct MoveSpan;

// Device deflater (deflate_kernels.cu, DESIGN.md sections 10 and 10c): the `segments` segments of one or
// more inputs (DeflateSegment descriptors on the device, batch_plan.hpp: planDeflate) -> coded segments in
// slots (deflateSlotBytes() each), their byte counts and CRC-32s, offsets[0..segments] (the exclusive scan
// of the byte counts; offsets[segments] = body bytes) and the packed raw deflate body, each input's
// segments at a contiguous range (at most its size + 16 bytes per segment).  Three launches,
// asynchronous on `stream`.
size_t deflateSlotBytes();
cudaError_t launchDeflate(const DeflateSegment *segs, unsigned long long segments, uint8_t *slots, uint32_t *segBytes, uint32_t *segCrc,
                          unsigned long long *offsets, uint8_t *body, cudaStream_t stream, int *launches);

// Device inflater (inflate_kernels.cu, DESIGN.md sections 10 and 10c): `blocks` table blocks of one or
// more block-table gzip members (InflateBlock descriptors on the device, batch_plan.hpp: planInflate),
// block i's raw deflate bytes at body + desc[i].in into its slice desc[i].out.  status[i] = ifl::kOk when
// the block filled its slice exactly, crc[i] its CRC-32 then.  One launch (blocks > 0), asynchronous on
// `stream`; *warpsPerCta is the geometry chosen for the batch's block count and the SM count.
cudaError_t launchInflate(const uint8_t *body, const InflateBlock *desc, long long blocks, uint32_t *crc, int32_t *status, int smCount,
                          cudaStream_t stream, int *warpsPerCta);

// Device-to-device copies of `count` MoveSpan descriptors (on the device) in one launch (move_kernels.cu);
// maxBytes = the largest span.  None for count = 0.
cudaError_t launchMoveSpans(const MoveSpan *spans, long long count, unsigned long long maxBytes, cudaStream_t stream, int *launches);

}  // namespace spzb200
