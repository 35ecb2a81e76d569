// The codec's round trip on float planes: launchDecode(launchEncode(x)) in one kernel that never puts
// a packed byte in global memory (DESIGN.md section 11).  What a trainer calls to see, at every step,
// the cloud its .spz file will give back.
//
// Every float is quantised with the encoder's functions (codec_math.cuh) and expanded again with the
// decoder's functions and tables, so the result is the encoder-then-decoder result bit for bit, NaN,
// Inf and denormal inputs included.  Apart from the rotations, each float of every plane is a value
// of its own: its parameters (flip sign, SH bucket) depend only on its index modulo the plane's floats
// per gaussian.  So every plane is an elementwise stream, and a CTA takes a slice of ONE plane:
//
//   * about kSliceFloats floats of it -- a whole number of gaussians, a multiple of four, so a slice
//     of a 16-byte aligned plane is 16-byte aligned too -- read and written as float4s, four per
//     thread, all four loads issued before the first store;
//   * the CTAs of the six planes follow each other in the grid (positions, scales, rotations, alphas,
//     colours, SH), so every CTA does about the same work and the block scheduler keeps the set of
//     pages in use compact;
//   * a plane whose input or output is not 16-byte aligned (a slice of a larger tensor, say) takes the
//     same path with scalar loads and stores: the scalar-path idea of scalar_path.cuh, per plane;
//   * a CTA stages the one table its plane needs (alpha thresholds and inverse sigmoid, colour LUT or
//     smallest-three magnitudes) in shared memory before it waits on the previous kernel.
//
// In place is allowed: a thread reads every float it writes before writing it and touches no other
// thread's floats, so an output plane may be its input plane.  Partial overlaps are refused by the
// caller (cabi.cu).
#include "codec_kernels.cuh"

#define SPZ_COLD_NOINLINE  // the general rotation forms are taken only for degenerate quaternions
// the host pass of nvcc sees the header's device-only `#pragma unroll`s; nothing here runs on the host
#pragma GCC diagnostic push
#pragma GCC diagnostic ignored "-Wunknown-pragmas"
#include "codec_math.cuh"
#include "kernel_utils.cuh"
#pragma GCC diagnostic pop

namespace spzb200 {
namespace {

constexpr int kQThreads = 256;
constexpr int kQuadsPerThread = 4;
constexpr int kSliceFloats = 4 * kQThreads * kQuadsPerThread;  // 4096 floats in and out per CTA at most

enum QPlane { kQPos = 0, kQScale, kQRot, kQAlpha, kQColor, kQSh };

// Host-computed launch geometry: plane p owns CTAs [firstCta[p], firstCta[p + 1]), each covering
// `gaussians[p]` gaussians (the last one fewer).  Bit p of `vec`: plane p's input and output are both
// 16-byte aligned.
struct QuantizeGrid {
  long long firstCta[7];
  int gaussians[6];
  uint32_t vec;
};

// gaussians per slice for a plane of w floats per gaussian: a multiple of 4 with at most kSliceFloats floats
constexpr int sliceGaussians(int w) { return (kSliceFloats / w) & ~3; }

// One float of a plane that is not rotations; k = its index modulo W.
template <int P, int W>
__device__ __forceinline__ float roundTrip(const QuantizeArgs &a, const float *sTab, float x, int k) {
  if constexpr (P == kQPos) {
    const uint32_t lo24 = m::quant_position24(x, signedConst(4096.0f, (a.flipP >> k) & 1u));
    return m::dequant_position24(lo24, signedConst(1.0f / 4096.0f, (a.oFlipP >> k) & 1u));  // fractional bits 12
  } else if constexpr (P == kQScale) {
    return m::dequant_scale(m::quant_scale(x));
  } else if constexpr (P == kQAlpha) {
    return sTab[256 + m::quant_alpha(x, sTab)];
  } else if constexpr (P == kQColor) {
    return sTab[m::quant_color(x)];
  } else {
    const uint32_t j = (uint32_t)k / 3u;  // SH coefficient
    const uint32_t bucket = k < 9 ? 8u : 16u;
    const uint32_t b = m::quant_sh(x, signedConst(128.0f, (a.flipSh >> j) & 1u), 128u + bucket / 2u, ~(bucket - 1u));
    return m::dequant_sh(b, signedConst(0.0078125f, (a.oFlipSh >> j) & 1u));
  }
}

template <int P, int W>
__device__ __forceinline__ float4 roundTrip4(const QuantizeArgs &a, const float *sTab, float4 v, int e) {
  if constexpr (P == kQRot) {
    float r[4];
    if (a.version == 2) {
      const uint32_t b = m::quant_rotation_first3(v.x, v.y, v.z, v.w, a.flipQ);
      m::dequant_rotation_first3(b & 0xffu, (b >> 8) & 0xffu, (b >> 16) & 0xffu, a.oFlipQ, r);
    } else {
      m::dequant_rotation_smallest3(m::quant_rotation_smallest3(v.x, v.y, v.z, v.w, a.flipQ), sTab, a.oFlipQ, r);
    }
    return make_float4(r[0], r[1], r[2], r[3]);
  } else {
    const int k = e % W;
    return make_float4(roundTrip<P, W>(a, sTab, v.x, k), roundTrip<P, W>(a, sTab, v.y, (k + 1) % W),
                       roundTrip<P, W>(a, sTab, v.z, (k + 2) % W), roundTrip<P, W>(a, sTab, v.w, (k + 3) % W));
  }
}

template <bool VEC>
__device__ __forceinline__ float4 load4(const float *p) {
  if constexpr (VEC) return *reinterpret_cast<const float4 *>(p);
  return make_float4(p[0], p[1], p[2], p[3]);
}
template <bool VEC>
__device__ __forceinline__ void store4(float *p, float4 v) {
  if constexpr (VEC) {
    *reinterpret_cast<float4 *>(p) = v;
  } else {
    p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
  }
}

// The slice's `floats` floats from `src` to `dst`, both already advanced to the slice.  Loads are plain
// (not .nc): in place, dst is src.
template <int P, int W, bool VEC>
__device__ __forceinline__ void slicePass(const QuantizeArgs &a, const float *sTab, const float *src, float *dst, int floats) {
  const int t = threadIdx.x;
  const int quads = floats >> 2;
#pragma unroll 1
  for (int base = 0; base < quads; base += kQThreads * kQuadsPerThread) {
    float4 v[kQuadsPerThread];
#pragma unroll
    for (int u = 0; u < kQuadsPerThread; u++) {
      const int q = base + u * kQThreads + t;
      if (q < quads) v[u] = load4<VEC>(src + 4 * q);
    }
#pragma unroll
    for (int u = 0; u < kQuadsPerThread; u++) {
      const int q = base + u * kQThreads + t;
      if (q < quads) store4<VEC>(dst + 4 * q, roundTrip4<P, W>(a, sTab, v[u], 4 * q));
    }
  }
  if constexpr (P != kQRot) {  // the last slice of a plane may end 1 - 3 floats past a whole float4
    const int e = 4 * quads + t;
    if (e < floats) dst[e] = roundTrip<P, W>(a, sTab, src[e], e % W);
  }
}

template <int P, int W>
__device__ __forceinline__ void planeSlice(const QuantizeArgs &a, const QuantizeGrid &gr, float *sTab, const float *in, float *out,
                                           long long slice) {
  // the plane's table: [0, 256) thresholds and [256, 512) inverse sigmoid for alphas, the colour LUT, or
  // the 512 smallest-three magnitudes
  if constexpr (P == kQAlpha) {
    for (int i = threadIdx.x; i < 256; i += kQThreads) {
      sTab[i] = a.alphaThresholds[i];
      sTab[256 + i] = a.tables[i];
    }
  } else if constexpr (P == kQColor) {
    for (int i = threadIdx.x; i < 256; i += kQThreads) sTab[i] = a.tables[256 + i];
  } else if constexpr (P == kQRot) {
    if (a.version != 2)
      for (int i = threadIdx.x; i < 512; i += kQThreads) sTab[i] = a.tables[512 + i];
  }
  if constexpr (P == kQAlpha || P == kQColor || P == kQRot) __syncthreads();
  const long long g0 = slice * gr.gaussians[P];
  const long long left = a.n - g0;
  const int floats = (int)(left < gr.gaussians[P] ? left : gr.gaussians[P]) * W;
  pdlWait();  // the planes may only be touched from here on (kernel_utils.cuh)
  if ((gr.vec >> P) & 1u) slicePass<P, W, true>(a, sTab, in + g0 * W, out + g0 * W, floats);
  else slicePass<P, W, false>(a, sTab, in + g0 * W, out + g0 * W, floats);
}

__global__ void __launch_bounds__(kQThreads) quantizeKernel(const __grid_constant__ QuantizeArgs a, const __grid_constant__ QuantizeGrid gr) {
  __shared__ float sTab[512];
  pdlTrigger();
  const long long cta = blockIdx.x;
  int p = 0;
  while (p < 5 && cta >= gr.firstCta[p + 1]) p++;
  const long long slice = cta - gr.firstCta[p];
  switch (p) {
    case kQPos: planeSlice<kQPos, 3>(a, gr, sTab, a.positions, a.oPositions, slice); break;
    case kQScale: planeSlice<kQScale, 3>(a, gr, sTab, a.scales, a.oScales, slice); break;
    case kQRot: planeSlice<kQRot, 4>(a, gr, sTab, a.rotations, a.oRotations, slice); break;
    case kQAlpha: planeSlice<kQAlpha, 1>(a, gr, sTab, a.alphas, a.oAlphas, slice); break;
    case kQColor: planeSlice<kQColor, 3>(a, gr, sTab, a.colors, a.oColors, slice); break;
    default:
      switch (a.shDim) {
        case 3: planeSlice<kQSh, 9>(a, gr, sTab, a.sh, a.oSh, slice); break;
        case 8: planeSlice<kQSh, 24>(a, gr, sTab, a.sh, a.oSh, slice); break;
        default: planeSlice<kQSh, 45>(a, gr, sTab, a.sh, a.oSh, slice); break;
      }
  }
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

cudaError_t launchQuantize(const QuantizeArgs &a, const LaunchPlan &plan, cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (a.n <= 0) return cudaSuccess;
  if (a.shDim != 0 && a.shDim != 3 && a.shDim != 8 && a.shDim != 15) return cudaErrorInvalidValue;
  const int widths[6] = {3, 3, 4, 1, 3, 3 * a.shDim};
  const float *in[6] = {a.positions, a.scales, a.rotations, a.alphas, a.colors, a.sh};
  const float *out[6] = {a.oPositions, a.oScales, a.oRotations, a.oAlphas, a.oColors, a.oSh};
  QuantizeGrid gr = {};
  gr.firstCta[0] = 0;
  for (int p = 0; p < 6; p++) {
    const long long ctas = widths[p] ? (a.n + sliceGaussians(widths[p]) - 1) / sliceGaussians(widths[p]) : 0;
    gr.gaussians[p] = widths[p] ? sliceGaussians(widths[p]) : 0;
    gr.firstCta[p + 1] = gr.firstCta[p] + ctas;
    if (aligned16(in[p]) && aligned16(out[p])) gr.vec |= 1u << p;
  }
  if (gr.firstCta[6] > 0x7fffffffLL) return cudaErrorInvalidValue;
  cudaError_t e = launchKernel(quantizeKernel, (unsigned)gr.firstCta[6], kQThreads, 0, stream, plan.pdl, a, gr);
  if (e == cudaSuccess && launches) *launches = 1;
  return e;
}

}  // namespace spzb200
