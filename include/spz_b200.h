/*
 * spz_b200 -- C-ABI of the B200-native .spz per-gaussian codec.
 *
 * This is the drop-in boundary for the reference's hot path (citations: lanxinger/spz, src/cc/):
 *
 *     spz::packGaussians(const GaussianCloud&, const PackOptions&)        load-spz.cc:257-331
 *     spz::unpackGaussians(const PackedGaussians&, const UnpackOptions&)  load-spz.cc:467-531
 *
 * Plain C: pointers, sizes, integer status codes; no C++ or torch types.  Everything the codec
 * does runs in hand-written sm_100a kernels; there is NO CPU implementation behind these entry
 * points -- without a usable CUDA device every call fails with SPZB200_ERR_NO_DEVICE.
 *
 * The C++ drop-in API of the reference (namespace spz, include/spz/load-spz.h) and the Python
 * mirror (spz_b200/) are thin layers over exactly these functions.  INTEGRATION.md shows the
 * binding a maintainer of the reference would add.
 *
 * Plane layouts are the reference's own:
 *   float side  (GaussianCloud, splat-types.h:90-115): positions[3n] scales[3n] rotations[4n]
 *               (x,y,z,w) alphas[n] colors[3n] sh[3*shDim*n] (coefficient-major, colour channel
 *               innermost), shDim = 0/3/8/15 for shDegree 0..3 (load-spz.cc:58-72).
 *   packed side (PackedGaussians, load-spz.h:42-59): positions[9n] (24-bit LE fixed point; 6n
 *               float16 for version 1) scales[3n] rotations[4n] (version 3 smallest-three) or
 *               [3n] (versions 1,2) alphas[n] colors[3n] sh[3*shDim*n].
 */
#ifndef SPZ_B200_H_
#define SPZ_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPZB200_VERSION 200 /* 0.2.0: context pool, batched per-gaussian access, stream-version-2 encoder */

/* Status codes.  0 = success; negative = failure, message via spzb200_last_error(). */
enum {
  SPZB200_OK = 0,
  SPZB200_ERR_INVALID = -1,    /* bad sizes / degree / version / null pointer: the cases the
                                  reference's checkSizes (load-spz.cc:106-127) rejects */
  SPZB200_ERR_NO_DEVICE = -2,  /* no CUDA device, or not an sm_100 part */
  SPZB200_ERR_CUDA = -3,       /* a CUDA call failed */
  SPZB200_ERR_NOMEM = -4       /* device or pinned-host allocation failed */
};

/* CoordinateSystem (splat-types.h:24-34); passed as int32. */
enum {
  SPZB200_COORD_UNSPECIFIED = 0,
  SPZB200_COORD_LDB = 1, SPZB200_COORD_RDB = 2, SPZB200_COORD_LUB = 3, SPZB200_COORD_RUB = 4,
  SPZB200_COORD_LDF = 5, SPZB200_COORD_RDF = 6, SPZB200_COORD_LUF = 7, SPZB200_COORD_RUF = 8
};

/* Stream flavours a decoder accepts in SpzB200Packed.version.  1..3 are the container versions
 * (load-spz.cc:571-572): 1 = float16 positions + first-three rotations, 2 = 24-bit positions +
 * first-three, 3 = 24-bit + smallest-three.  4 has no file form: it is the in-memory combination
 * "float16 positions with usesQuaternionSmallestThree = true" that unpackGaussians accepts for a
 * hand-built PackedGaussians (load-spz.cc:465,509) -- notably the default-constructed empty one. */
enum {
  SPZB200_STREAM_V1 = 1,
  SPZB200_STREAM_V2 = 2,
  SPZB200_STREAM_V3 = 3,
  SPZB200_STREAM_HALF_POSITIONS_SMALLEST_THREE = 4
};

/* Float planes of n gaussians: a borrowed view of GaussianCloud (splat-types.h:90-115).  The
 * pointers are device pointers for the *_device entry points and host pointers for *_host. */
typedef struct {
  int64_t num_points;
  int32_t sh_degree; /* 0..3 */
  int32_t reserved;
  float *positions;
  float *scales;
  float *rotations;
  float *alphas;
  float *colors;
  float *sh; /* may be NULL when sh_degree == 0 */
} SpzB200Cloud;

/* Byte planes of n gaussians: a borrowed view of PackedGaussians (load-spz.h:42-59). */
typedef struct {
  int64_t num_points;
  int32_t sh_degree;       /* 0..3 */
  int32_t fractional_bits; /* header byte; the encoder always writes 12 (load-spz.cc:270) */
  int32_t version;         /* container version 1..3 (load-spz.cc:571-572), or
                              SPZB200_STREAM_HALF_POSITIONS_SMALLEST_THREE; the encoder writes 3 */
  int32_t reserved;
  uint8_t *positions;
  uint8_t *scales;
  uint8_t *rotations;
  uint8_t *alphas;
  uint8_t *colors;
  uint8_t *sh; /* may be NULL when sh_degree == 0 */
} SpzB200Packed;

/* Per-phase timings of a *_host call, milliseconds, measured with CUDA events on the call's own
 * streams (kernel_ms = sum over chunks) plus the host wall clock of the whole call. */
typedef struct {
  double h2d_ms;
  double kernel_ms;
  double d2h_ms;
  double wall_ms;
  int64_t h2d_bytes;
  int64_t d2h_bytes;
  int32_t kernel_launches;
  int32_t chunks;
  double host_copy_ms;     /* calling-thread time inside the copy pool (helping with / waiting for the bounce copies of pageable planes) */
  int32_t staged;          /* bit 0: input planes were pageable and bounced, bit 1: output planes */
  int32_t reserved;
} SpzB200Timings;

/* A context: immutable codec tables resident on one device, three worker streams and the staging
 * buffers of the host-pointer pipeline.  A context is not thread-safe: one caller at a time (own one
 * per host thread with spzb200_create, or lease one per call with spzb200_acquire).  Creation fails
 * (no CPU fallback) without an sm_100 device. */
typedef struct SpzB200Context SpzB200Context;

int spzb200_create(int32_t device, SpzB200Context **out);
void spzb200_destroy(SpzB200Context *ctx);

/* Process-wide pool: lease a context of `device` for one call (or a batch of calls) and hand it back.
 * Contexts are created on demand, at most SPZ_B200_MAX_CONTEXTS (default 2) per device -- further
 * callers block until one is released -- and live until the process exits, so threads that come and go
 * do not pay for streams, tables, staging and pinned bounce buffers again.  A lease is exclusive.  This
 * is what the C++ API (spz::packGaussians, ...) and the *_multi entry points use.  spzb200_release
 * of a context that came from spzb200_create destroys it. */
int spzb200_acquire(int32_t device, SpzB200Context **out);
void spzb200_release(SpzB200Context *ctx);

/* ---- device-resident codec: what the benchmark's `value` times ------------------------------
 *
 * Replaces packGaussians (load-spz.cc:257-331).  `from` is PackOptions::from (load-spz.h:61-63);
 * the flips of coordinateConverter(from, RUB) (splat-types.h:55-81) are folded into the kernel.
 * in/out hold DEVICE pointers; out->fractional_bits and out->version are set to 12 and 3.
 * Asynchronous on `stream` (a cudaStream_t, NULL = the legacy default stream); nothing is
 * retained after the call returns except work queued on the stream.  num_points is 64-bit: the
 * reference's int32 size arithmetic (load-spz.cc:110-115) does not limit this implementation. */
int spzb200_encode_device(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from,
                          SpzB200Packed *out, void *stream);

/* The same encoder writing another stream flavour.  stream_version = SPZB200_STREAM_V3 is
 * spzb200_encode_device; SPZB200_STREAM_V2 stores rotations as the first three components in 3 bytes
 * (out->rotations = 3n bytes), the form unpackQuaternionFirstThree (load-spz.cc:333-345) reads.
 * PARITY UNPINNED for version 2: the reference tree has only that decoder, no encoder to compare with;
 * this follows upstream nianticlabs/spz before smallest-three (normalise, make w >= 0, toUint8(xyz * 127.5
 * + 127.5)).  Every other plane is byte-identical to version 3. */
int spzb200_encode_device_as(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from, int32_t stream_version,
                             SpzB200Packed *out, void *stream);

/* Replaces unpackGaussians (load-spz.cc:467-531) including its trailing
 * convertCoordinates(RUB, to) (load-spz.cc:529, splat-types.h:134-164), fused into the kernel.
 * `to` is UnpackOptions::to.  in->version selects the stream flavour: 3 = smallest-three
 * rotations, 2 = first-three rotations, 1 = float16 positions + first-three, 4 = float16 +
 * smallest-three. */
int spzb200_decode_device(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to,
                          SpzB200Cloud *out, void *stream);

/* The cloud an .spz file of `in` gives back: spzb200_encode_device_as(in, from, version) followed by
 * spzb200_decode_device(to), bit for bit, in one kernel that writes no packed planes (no device scratch).
 * For training with the quantizer in the loop.  version is SPZB200_STREAM_V3 (smallest-three rotations)
 * or SPZB200_STREAM_V2 (first-three).  in and out hold DEVICE pointers; out->num_points and out->sh_degree
 * must equal in's.  Planes need only float alignment (16-byte aligned ones are faster).
 * Aliasing: each output plane is either exactly its input plane (same pointer: in place) or overlaps no
 * input plane; output planes do not overlap each other.  Anything else fails with SPZB200_ERR_INVALID.
 * Every failure is reported before any work is queued, so `out` is untouched then.  Asynchronous on
 * `stream`, as spzb200_encode_device. */
int spzb200_quantize_device(SpzB200Context *ctx, const SpzB200Cloud *in /* device */, int32_t from, int32_t to,
                            int32_t version, SpzB200Cloud *out /* device */, void *stream);

/* ---- host-pointer codec: what the C++ / Python drop-in API calls ----------------------------
 *
 * Same contracts with HOST pointers.  The cloud is cut into contiguous point ranges; each range is
 * copied in, transformed and copied out on one of three streams so H2D, kernel and D2H of
 * neighbouring ranges overlap.  Pinned planes (spzb200_alloc_pinned, cudaHostRegister) are copied
 * directly; pageable planes are bounced through pinned buffers by a few host threads.
 * Synchronous: returns when `out` is complete.  timings may be NULL. */
int spzb200_encode_host(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from,
                        SpzB200Packed *out, SpzB200Timings *timings);
int spzb200_encode_host_as(SpzB200Context *ctx, const SpzB200Cloud *in, int32_t from, int32_t stream_version,
                           SpzB200Packed *out, SpzB200Timings *timings);
int spzb200_decode_host(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to,
                        SpzB200Cloud *out, SpzB200Timings *timings);

/* Multi-GPU form: shards [0, n) by contiguous point range (spzb200_shard_range) over the given
 * devices, one host thread and one context per device; every device writes its slice of each
 * output plane at its precomputed offset.  No collective, no peer traffic.  timings (may be
 * NULL) receives the slowest device's figures. */
int spzb200_encode_host_multi(const int32_t *devices, int32_t num_devices, const SpzB200Cloud *in,
                              int32_t from, SpzB200Packed *out, SpzB200Timings *timings);
int spzb200_decode_host_multi(const int32_t *devices, int32_t num_devices,
                              const SpzB200Packed *in, int32_t to, SpzB200Cloud *out,
                              SpzB200Timings *timings);

/* ---- fused PLY-rows encoder (SURVEY.md 8f-3) ------------------------------------------------------
 *
 * The vertex records of a gaussian-splat .ply -- row-major, `width` floats each, the layout
 * loadSplatFromPly parses (load-spz.cc:691-844) -- straight to PackedGaussians planes.  Equals
 * packGaussians(loadSplatFromPly(rows, to = X), from = X): the loader's [N,C,S] -> [N,S,C] SH shuffle and
 * wxyz -> xyzw reorder, then the encoder.  `from` is the frame the records are in (RDF for PLY files;
 * UNSPECIFIED = no flips, which is what the reference's ply_to_spz tool does).  Column indices are
 * positions inside a record; col_rest lists f_rest_0 .. f_rest_{3*shDim-1} in file order. */
typedef struct {
  int64_t num_points;
  int32_t width;      /* floats per record */
  int32_t sh_degree;  /* 0..3 */
  float *rows;        /* device pointer for *_device, host pointer for *_host; read by the encoder, written by the decoder */
  int32_t col_pos[3], col_scale[3], col_rot[4] /* x, y, z, w = rot_1, rot_2, rot_3, rot_0 */, col_alpha, col_color[3];
  int32_t col_rest[45];
} SpzB200PlyRows;

int spzb200_encode_ply_device(SpzB200Context *ctx, const SpzB200PlyRows *in, int32_t from, SpzB200Packed *out, void *stream);
int spzb200_encode_ply_host(SpzB200Context *ctx, const SpzB200PlyRows *in, int32_t from, SpzB200Packed *out,
                            SpzB200Timings *timings);

/* The mirror image: PackedGaussians planes -> vertex records, i.e. saveSplatToPly(unpackGaussians(in, to = X),
 * from = X)'s body (load-spz.cc:846-934) in one kernel.  `to` is the frame of the records (RDF for a
 * PLY file, UNSPECIFIED = no flips).  out->rows receives num_points * width floats; columns no
 * plane maps to (nx, ny, nz, anything extra) are written as 0.  in->version as for spzb200_decode_*. */
int spzb200_decode_ply_device(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to, SpzB200PlyRows *out, void *stream);
int spzb200_decode_ply_host(SpzB200Context *ctx, const SpzB200Packed *in, int32_t to, SpzB200PlyRows *out,
                            SpzB200Timings *timings);

/* ---- batched per-gaussian access (SURVEY.md 8f-4) ----------------------------------------------
 *
 * PackedGaussians::at(i) followed by PackedGaussian::unpack (load-spz.cc:383-463) for many gaussians
 * in one call.  The unit structs are the reference's own, so arrays of them pass through unchanged:
 *   record  = PackedGaussian   (load-spz.h:28-37), 65 bytes: position[9] rotation[4] scale[3] color[3]
 *             alpha shR[15] shG[15] shB[15]
 *   output  = UnpackedGaussian (load-spz.h:13-24), 59 floats: position[3] rotation[4] (x,y,z,w) scale[3]
 *             color[3] alpha shR[15] shG[15] shB[15]
 *   converter = CoordinateConverter (splat-types.h:36-41), 21 floats: flipP[3] flipQ[3] flipSh[15];
 *             NULL = identity.  Applied by multiplication in the reference's order, so any values work.
 * `version` is the stream flavour (SPZB200_STREAM_*): which position / rotation encoding the records hold. */
#define SPZB200_RECORD_BYTES 65
#define SPZB200_UNPACKED_FLOATS 59

/* records (HOST, n x 65 bytes) -> out (HOST, n x 59 floats).  Synchronous. */
int spzb200_unpack_records_host(SpzB200Context *ctx, const uint8_t *records, int64_t n, int32_t version,
                                int32_t fractional_bits, const float *converter, float *out);
/* at(indices[k]) for k < n on HOST planes, then as above.  indices == NULL means 0..n-1 (then n must
 * not exceed packed->num_points).  An index outside [0, num_points) fails with SPZB200_ERR_INVALID
 * (the reference reads out of bounds). */
int spzb200_unpack_gather_host(SpzB200Context *ctx, const SpzB200Packed *packed, const int64_t *indices, int64_t n,
                               const float *converter, float *out);
/* The same with DEVICE planes, DEVICE indices (or NULL) and a DEVICE output, asynchronous on `stream`:
 * the kernel does the gather itself.  Indices are not range-checked. */
int spzb200_unpack_gather_device(SpzB200Context *ctx, const SpzB200Packed *packed, const int64_t *indices, int64_t n,
                                 const float *converter, float *out, void *stream);

/* Page-locked host buffers for the *_host entry points (cudaHostAlloc, portable across devices).
 * Pageable memory works too but its copies neither overlap nor reach PCIe bandwidth. */
int spzb200_alloc_pinned(size_t bytes, void **out);
void spzb200_free_pinned(void *ptr);

/* ---- host-side helpers (no GPU needed) ------------------------------------------------------ */

/* The container's gzip stage (load-spz.cc:141-214) for FFI callers: zlib with the reference's
 * parameters.  threads <= 1 gives the reference's byte-identical single-thread stream; threads > 1
 * deflates independent blocks concurrently into one standard gzip member (same inflated bytes,
 * different compressed bytes) and inflates such members block-parallel.  *out is malloc'd; release
 * it with spzb200_free. */
int spzb200_gzip(const uint8_t *data, size_t size, int32_t threads, uint8_t **out, size_t *out_size);
int spzb200_gunzip(const uint8_t *data, size_t size, int32_t threads, uint8_t **out, size_t *out_size);
void spzb200_free(void *ptr);

/* ---- .spz files of device-resident clouds ---------------------------------------------------
 *
 * The gzip stage on the device: the input is cut into 64 KiB segments, each coded by one CTA as an
 * independent piece of a raw deflate stream (Huffman-coded literals plus distance-1 matches for runs of
 * one byte value; stored when that is not larger), and the pieces are framed as ONE standard gzip member
 * with the block table spzb200_gzip(threads > 1) writes, so any inflater reads it and spzb200_gunzip
 * inflates it block-parallel.  The bytes depend only on the input bytes (not on the device, context,
 * stream or timing).  Only compressed bytes cross PCIe.  *out is malloc'd: release it with spzb200_free.
 * Synchronous: each returns when *out is complete, after work queued earlier on `stream` (a
 * cudaStream_t, NULL = legacy default stream).  Device scratch, allocated and freed on `stream`:
 * about 2 bytes per input byte (the 64 KiB + 64 byte worst-case slot of every segment plus the
 * compacted body). */
int spzb200_gzip_device(SpzB200Context *ctx, const uint8_t *data /* device */, size_t size, uint8_t **out, size_t *out_size,
                        void *stream);

/* saveSpz for a device cloud: the encoder's planes, the 16-byte header and the planes in container order
 * (positions, alphas, colors, scales, rotations, sh) on the device, then spzb200_gzip_device's deflater.
 * The file inflates to the container saveSpz writes for the same cloud, `from` and antialiased flag.
 * Device scratch peaks at about twice the container (65 bytes per point at SH degree 3).  A cloud the
 * reference's checkSizes rejects, or one of more than 2^31 - 1 points, fails with SPZB200_ERR_INVALID;
 * nothing is written to any file. */
int spzb200_save_spz_device(SpzB200Context *ctx, const SpzB200Cloud *in /* device */, int32_t from, int32_t antialiased,
                            uint8_t **out, size_t *out_size, void *stream);

/* Point count and SH degree from the header of an .spz file in host memory (inflates only the first 16
 * bytes), to size the output of spzb200_load_spz_device. */
int spzb200_spz_info(const uint8_t *bytes, size_t size, int64_t *num_points, int32_t *sh_degree);

/* Inflated size and block count of a gzip member carrying the "SZ" block table (what spzb200_gzip with
 * threads > 1, saveSpz from 8 MiB, spzb200_gzip_device and spzb200_save_spz_device write).  No GPU.
 * SPZB200_ERR_INVALID for a member without the table or with one the parallel inflater would not trust. */
int spzb200_gzip_table_info(const uint8_t *bytes, size_t size, uint64_t *inflated_size, int64_t *blocks);

/* The inflate stage on the device: a block-table gzip member in HOST memory -> its inflated bytes at
 * `out` (DEVICE, out_capacity >= the table's size).  The compressed bytes cross PCIe; each table block
 * is inflated by the device and the CRC-32 and ISIZE are checked.  The result is exactly what
 * spzb200_gunzip(threads > 1) returns for the same bytes, and the call fails where that fails: when the device cannot
 * vouch for a block, the host inflater produces the bytes.  *on_device (may be NULL) = 1 when the device
 * produced them.  Synchronous, after earlier work on `stream`.  A member without the table fails with
 * SPZB200_ERR_INVALID before anything is allocated; after a failure the contents of `out` are undefined.
 * Device scratch: the compressed body and 24 bytes per table block. */
int spzb200_gunzip_device(SpzB200Context *ctx, const uint8_t *bytes, size_t size, uint8_t *out,
                          size_t out_capacity, size_t *out_size, int32_t *on_device, void *stream);

/* loadSpz into caller-allocated DEVICE planes (container versions 1-3).  out->num_points and
 * out->sh_degree must be what spzb200_spz_info reports.  `to` is UnpackOptions::to; *antialiased (may be
 * NULL) receives the header flag.  A member whose block table has blocks of less than 1 MiB (every
 * spzb200_save_spz_device file) is inflated on the device: its header is validated the way loadSpz does
 * before anything is allocated, only the compressed bytes cross PCIe, and the planes are moved into
 * aligned places on the device and decoded there.  Other members (the reference's files, saveSpz files,
 * whose zlib blocks of 1 MiB or more the host inflates faster), and any member the device cannot vouch
 * for, take the host route: inflate on the host (block-parallel where a table allows), validate, copy
 * each plane up and decode on the device.
 * Both routes give the same verdict and the same planes.  A file that does not inflate or parse fails
 * with SPZB200_ERR_INVALID and leaves `out` untouched.  Device scratch: the container and its packed
 * planes (twice the container's size) plus the compressed body on the device route, the packed planes
 * on the host route.  Returns when `out` is complete. */
int spzb200_load_spz_device(SpzB200Context *ctx, const uint8_t *bytes /* host */, size_t size, int32_t to,
                            SpzB200Cloud *out /* device */, int32_t *antialiased, void *stream);

/* ---- batches of .spz files of device-resident clouds (DESIGN.md section 10c) ------------------
 *
 * One call for many files: the table blocks of all members go to one inflate launch, the segments of all
 * inputs to one set of deflate launches, and the planes of all files to one plane-move launch, so small
 * files share the GPU instead of each paying a launch and its latency.  Entry i of every result is
 * exactly what the single-file call gives for input i alone.  Synchronous, after earlier work on
 * `stream`; device scratch is allocated and freed on `stream` and peaks at the sum over the files of
 * what the single call uses.  count may be 0 (nothing is done). */

/* spzb200_gzip_device of each of data[0..count) (device; sizes[i] bytes): out[i], out_size[i] are what
 * spzb200_gzip_device writes for input i.  Release each out[i] with spzb200_free.  All or nothing: on
 * failure every out[i] is NULL. */
int spzb200_gzip_device_batch(SpzB200Context *ctx, const uint8_t *const *data /* device */, const size_t *sizes, int32_t count,
                              uint8_t **out, size_t *out_size, void *stream);

/* spzb200_save_spz_device of each of clouds[0..count) (device planes), all from coordinate system
 * `from`; antialiased[i] is cloud i's header flag (antialiased may be NULL: none is).  Every cloud is
 * checked before anything is queued.  All or nothing: on failure every out[i] is NULL. */
int spzb200_save_spz_device_batch(SpzB200Context *ctx, const SpzB200Cloud *clouds /* device */, int32_t count, int32_t from,
                                  const int32_t *antialiased, uint8_t **out, size_t *out_size, void *stream);

/* spzb200_gunzip_device of each member bytes[i] (host; sizes[i] bytes) into out[i] (device,
 * out_capacity[i] bytes): status[i], out_size[i], on_device[i] (on_device may be NULL) and the bytes are
 * what spzb200_gunzip_device gives for member i alone.  A member the device cannot vouch for is inflated
 * by the host inflater on its own; its neighbours are not affected.  Returns SPZB200_ERR_INVALID when any
 * member failed, OK otherwise; a CUDA or allocation failure ends the call with its code. */
int spzb200_gunzip_device_batch(SpzB200Context *ctx, const uint8_t *const *bytes /* host */, const size_t *sizes, int32_t count,
                                uint8_t *const *out /* device */, const size_t *out_capacity, size_t *out_size, int32_t *on_device,
                                int32_t *status, void *stream);

/* spzb200_load_spz_device of each file bytes[i] (host; sizes[i] bytes) into out[i] (device planes sized
 * by spzb200_spz_info), all to coordinate system `to`; antialiased[i] (antialiased may be NULL) receives
 * file i's header flag.  Per file, the route and the verdict are those of spzb200_load_spz_device: the
 * members with table blocks under 1 MiB whose headers agree with their out[i] are inflated together on
 * the device, every other file and every member the device cannot vouch for takes the host route.  A file
 * that fails has status[i] = SPZB200_ERR_INVALID and out[i] untouched; the others are complete.  Returns
 * SPZB200_ERR_INVALID when any file failed, OK otherwise; a CUDA or allocation failure ends the call with
 * its code. */
int spzb200_load_spz_device_batch(SpzB200Context *ctx, const uint8_t *const *bytes /* host */, const size_t *sizes, int32_t count,
                                  int32_t to, SpzB200Cloud *out /* device */, int32_t *antialiased, int32_t *status, void *stream);

/* Point range [*begin, *end) of shard `index` out of `num_shards` over n gaussians of the given
 * SH degree.  Boundaries are multiples of the kernel tile, so every shard but the last runs
 * entirely on the vector path and every plane slice stays 16-byte aligned. */
int spzb200_shard_range(int64_t n, int32_t sh_degree, int32_t num_shards, int32_t index,
                        int64_t *begin, int64_t *end);

/* Gaussians per kernel tile for an SH degree (the sharding granule). */
int32_t spzb200_tile_gaussians(int32_t sh_degree);

/* Sign sets of coordinateConverter(from, to) (splat-types.h:55-81): bit i of *flip_p negates
 * position axis i, of *flip_q quaternion component i (x,y,z), of *flip_sh SH coefficient i. */
void spzb200_flip_bits(int32_t from, int32_t to, uint32_t *flip_p, uint32_t *flip_q,
                       uint32_t *flip_sh);

/* The two host-built tables of a context (for inspection and tests): the 255 ascending alpha
 * thresholds (out[255] = +Inf) and the 256-entry inverse-sigmoid table. */
int spzb200_get_tables(const SpzB200Context *ctx, float alpha_thresholds[256],
                       float alpha_lut[256]);
/* The same construction without a context or a GPU (what spzb200_create runs on the host). */
int spzb200_build_tables(float alpha_thresholds[256], float alpha_lut[256]);

/* Context facts: 148 on a B200, which byte packer the encoder uses (1 = cvt.pack/I2IP, 0 = ALU),
 * kernels launched through this context so far. */
int spzb200_info(const SpzB200Context *ctx, int32_t *sm_count, int32_t *pack_mode,
                 int64_t *kernel_launches);

/* Self-check on the device of the two division identities the smallest-three packer uses in place of
 * IEEE divisions (spz_b200/csrc/codec_math.cuh: div_by_sqrt1_2, div_by_rcp).  part 0: a / sqrt1_2 for
 * every float in {0} U [2^-81, 1.01]; part 1: x / b on pseudo-random operand pairs of the domain the
 * packer's guard admits, pairs_per_thread of them on each of sm_count * 2048 threads.  *wrong receives
 * the number of quotients that differ from the device's IEEE division in any bit (0 is the only
 * acceptable answer), *checked the number compared. */
int spzb200_selfcheck_division(SpzB200Context *ctx, int32_t part, uint64_t pairs_per_thread, uint64_t seed,
                               uint64_t *wrong, uint64_t *checked);

/* Test hooks: force the scalar kernels (1) / restore (0); choose the byte packer. */
void spzb200_set_force_generic(SpzB200Context *ctx, int32_t on);
void spzb200_set_pack_mode(SpzB200Context *ctx, int32_t mode);
/* Point ranges of at most this many gaussians per pipeline stage of the *_host calls; 0 restores
 * the defaults (2M points for pinned planes, 256K for pageable ones). */
void spzb200_set_chunk_points(SpzB200Context *ctx, int64_t points);
/* Pageable host planes (plain malloc / std::vector memory) are bounced through pinned buffers by
 * `copy_threads` host threads (0 = auto: three quarters of the hardware threads, at most 16; SPZB200_COPY_THREADS)
 * in 2 MiB pieces whose DMAs overlap the copies: 4-5x the speed of handing them to cudaMemcpyAsync as they are
 * (driver-staged, synchronous).  bounce: 0 = never,
 * 1 = calls of >= 4 MiB (SPZB200_BOUNCE_MIN_MB) or once the buffers exist (default: the pinned
 * allocation is a one-time cost small one-shot calls would not earn back), 2 = always. */
void spzb200_set_host_staging(SpzB200Context *ctx, int32_t bounce, int32_t copy_threads);

/* Thread-local message of the last failing call on this thread ("" if none). */
const char *spzb200_last_error(void);
int32_t spzb200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SPZ_B200_H_ */
