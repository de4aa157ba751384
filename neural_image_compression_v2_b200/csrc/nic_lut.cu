// nic_lut.cu — applying a baked 3-D colour LUT (nic.h nic_lut_pack / nic_lut_apply).
//   lut_pack_kernel   the bake's last step: a dense fp32 decode [N, cout] -> [N][4] texels of fp32 or fp16, padding channels 0;
//   lut_apply_kernel  the per-pixel gather: RGB -> coordinates -> 8 (trilinear, sample_tap) or 4 (tetrahedral, tetra_corners)
//                     table texels, one 8-byte (fp16) or 16-byte (fp32) read-only load each, blended in fp32 on CUDA cores.
// The apply is a streaming kernel: a persistent grid-stride loop over chunks of 16 pixels, whose input (48 elements) and
// output (16 * cout elements) are whole 16-byte vectors; a scalar loop takes the pixels before the first aligned chunk and
// after the last one, so any element alignment of the two buffers works.
#include <type_traits>

#include "nic_internal.cuh"

namespace nic {

constexpr int kLutPix = 16;        // pixels per thread and chunk: 48 u8 inputs = three 16-byte loads

template <typename TableT>
__global__ void __launch_bounds__(256) lut_pack_kernel(const float* __restrict__ dense, long long n, int cout,
                                                       TableT* __restrict__ table) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n * 4; e += (long long)gridDim.x * blockDim.x) {
    const long long t = e >> 2;
    const int c = (int)(e & 3);
    store_as(table + e, c < cout ? __ldg(dense + t * cout + c) : 0.0f);
  }
}

__device__ __forceinline__ float4 lut_texel(const float* __restrict__ t, int i) {
  return __ldg(reinterpret_cast<const float4*>(t) + i);
}
__device__ __forceinline__ float4 lut_texel(const __half* __restrict__ t, int i) {
  const uint2 r = __ldg(reinterpret_cast<const uint2*>(t) + i);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

__device__ __forceinline__ void lut_accumulate(float* acc, float w, float4 v) {
  acc[0] = __fadd_rn(acc[0], __fmul_rn(w, v.x));
  acc[1] = __fadd_rn(acc[1], __fmul_rn(w, v.y));
  acc[2] = __fadd_rn(acc[2], __fmul_rn(w, v.z));
  acc[3] = __fadd_rn(acc[3], __fmul_rn(w, v.w));
}

// One pixel at normalised coordinates u (R, G, B -> x, y, z): the blend of nic.h, all four table channels.
template <typename TableT, int INTERP>
__device__ __forceinline__ void lut_pixel(const DevSampler& s, const TableT* __restrict__ table, const float* u, float* acc) {
  acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
  if (INTERP == NIC_INTERP_TRILINEAR) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      int p[3];
      const float w = sample_tap(s, 3, u, k, p);
      lut_accumulate(acc, w, lut_texel(table, (p[0] * s.S[1] + p[1]) * s.S[2] + p[2]));
    }
  } else {
    int p[4][3];
    float w[4];
    tetra_corners(s.S, u, p, w);
#pragma unroll
    for (int k = 0; k < 4; ++k) lut_accumulate(acc, w[k], lut_texel(table, (p[k][0] * s.S[1] + p[k][1]) * s.S[2] + p[k][2]));
  }
}

// The normalised coordinate of one input channel: an 8-bit value through the block's table of v / 255, a float as given.
__device__ __forceinline__ float lut_unit(const float* s_unit, uint8_t v) { return s_unit[v]; }
__device__ __forceinline__ float lut_unit(const float*, float v) { return v; }

struct LutArgs {
  const void* table;
  int S[3];
  const void* src;
  void* dst;
  long long pixels;
  long long head;      // pixels before the first 16-byte-aligned chunk (scalar)
  long long chunks;    // whole chunks of kLutPix pixels after the head; the rest is the scalar tail
};

template <int BYTES>
struct alignas(16) LutVec {
  uint4 v[BYTES / 16];
};

template <typename SrcT, typename DstT, typename TableT, int INTERP, int COUT>
__global__ void __launch_bounds__(256) lut_apply_kernel(LutArgs a) {
  constexpr bool kU8In = std::is_same<SrcT, uint8_t>::value;
  __shared__ float s_unit[256];                     // v / 255 of every 8-bit input value (__fdiv_rn, as nic.h states)
  if (kU8In) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_unit[i] = __fdiv_rn((float)i, 255.0f);
    __syncthreads();
  }
  DevSampler s;                                     // align_corners, clamp: constants the tap rule folds
  s.coords = nullptr;
  s.prev = nullptr;
  s.blend_weight = 0.f;
  s.address = NIC_ADDRESS_CLAMP;
  s.align_corners = 1;
  s.S[0] = a.S[0];
  s.S[1] = a.S[1];
  s.S[2] = a.S[2];
  const TableT* __restrict__ table = static_cast<const TableT*>(a.table);
  const SrcT* __restrict__ src = static_cast<const SrcT*>(a.src);
  DstT* __restrict__ dst = static_cast<DstT*>(a.dst);
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;

  for (long long c = tid; c < a.chunks; c += stride) {
    const long long p0 = a.head + c * kLutPix;
    LutVec<kLutPix * 3 * sizeof(SrcT)> in;
    const uint4* ps = reinterpret_cast<const uint4*>(src + p0 * 3);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(in) / 16); ++i) in.v[i] = __ldcs(ps + i);
    const SrcT* e = reinterpret_cast<const SrcT*>(&in);
    LutVec<kLutPix * COUT * sizeof(DstT)> out;
    DstT* o = reinterpret_cast<DstT*>(&out);
#pragma unroll
    for (int px = 0; px < kLutPix; ++px) {
      float u[3], acc[4];
#pragma unroll
      for (int k = 0; k < 3; ++k) u[k] = lut_unit(s_unit, e[px * 3 + k]);
      lut_pixel<TableT, INTERP>(s, table, u, acc);
#pragma unroll
      for (int k = 0; k < COUT; ++k) store_out(o + px * COUT + k, acc[k]);
    }
    uint4* pd = reinterpret_cast<uint4*>(dst + p0 * COUT);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(out) / 16); ++i) __stcs(pd + i, out.v[i]);
  }

  const long long tail0 = a.head + a.chunks * kLutPix, scalar = a.head + (a.pixels - tail0);
  for (long long i = tid; i < scalar; i += stride) {
    const long long p = i < a.head ? i : tail0 + (i - a.head);
    float u[3], acc[4];
#pragma unroll
    for (int k = 0; k < 3; ++k) u[k] = lut_unit(s_unit, src[p * 3 + k]);
    lut_pixel<TableT, INTERP>(s, table, u, acc);
#pragma unroll
    for (int k = 0; k < COUT; ++k) store_out(dst + p * COUT + k, acc[k]);
  }
}

int launch_lut_pack(Handle* h, const float* dense, long long texels, int cout, void* table, int table_dtype, cudaStream_t st) {
  const long long cap = (long long)h->sms * 8, blocks = (texels * 4 + 255) / 256;
  const int grid = (int)(blocks < cap ? blocks : cap);
  if (table_dtype == NIC_DT_F32)
    lut_pack_kernel<float><<<grid, 256, 0, st>>>(dense, texels, cout, (float*)table);
  else
    lut_pack_kernel<__half><<<grid, 256, 0, st>>>(dense, texels, cout, (__half*)table);
  h->launches++;
  return (int)cudaGetLastError();
}

template <typename SrcT, typename DstT, typename TableT, int INTERP>
static void launch_apply(int cout, const LutArgs& a, int grid, cudaStream_t st) {
  switch (cout) {
    case 1: lut_apply_kernel<SrcT, DstT, TableT, INTERP, 1><<<grid, 256, 0, st>>>(a); break;
    case 2: lut_apply_kernel<SrcT, DstT, TableT, INTERP, 2><<<grid, 256, 0, st>>>(a); break;
    case 3: lut_apply_kernel<SrcT, DstT, TableT, INTERP, 3><<<grid, 256, 0, st>>>(a); break;
    default: lut_apply_kernel<SrcT, DstT, TableT, INTERP, 4><<<grid, 256, 0, st>>>(a); break;
  }
}

template <typename SrcT, typename DstT, typename TableT>
static void launch_apply(int interp, int cout, const LutArgs& a, int grid, cudaStream_t st) {
  if (interp == NIC_INTERP_TRILINEAR)
    launch_apply<SrcT, DstT, TableT, NIC_INTERP_TRILINEAR>(cout, a, grid, st);
  else
    launch_apply<SrcT, DstT, TableT, NIC_INTERP_TETRAHEDRAL>(cout, a, grid, st);
}

template <typename SrcT, typename DstT>
static void launch_apply(int table_dtype, int interp, int cout, const LutArgs& a, int grid, cudaStream_t st) {
  if (table_dtype == NIC_DT_F32)
    launch_apply<SrcT, DstT, float>(interp, cout, a, grid, st);
  else
    launch_apply<SrcT, DstT, __half>(interp, cout, a, grid, st);
}

int launch_lut_apply(Handle* h, const NicLut& lut, const void* src, int src_dtype, long long pixels, void* dst, int dst_dtype,
                     int interp, cudaStream_t st) {
  LutArgs a;
  a.table = lut.table;
  for (int k = 0; k < 3; ++k) a.S[k] = lut.extent[k];
  a.src = src;
  a.dst = dst;
  a.pixels = pixels;
  // the first pixel at which both buffers are 16-byte aligned (the chunk sizes are multiples of 16 bytes on both sides, so
  // every later chunk is aligned too); when no such pixel exists every pixel takes the scalar loop
  const int in_bytes = src_dtype == NIC_DT_U8 ? 3 : 12, out_bytes = lut.cout * (dst_dtype == NIC_DT_U8 ? 1 : 4);
  a.head = pixels;
  for (long long p = 0; p < kLutPix && p < pixels; ++p)
    if (((uintptr_t)src + p * in_bytes) % 16 == 0 && ((uintptr_t)dst + p * out_bytes) % 16 == 0) {
      a.head = p;
      break;
    }
  a.chunks = (pixels - a.head) / kLutPix;
  const long long scalar = pixels - a.chunks * kLutPix, work = a.chunks > scalar ? a.chunks : scalar;
  const long long cap = (long long)h->sms * 8, blocks = (work + 255) / 256;
  const int grid = (int)(blocks < cap ? blocks : cap);
  if (src_dtype == NIC_DT_U8) {
    if (dst_dtype == NIC_DT_U8)
      launch_apply<uint8_t, uint8_t>(lut.table_dtype, interp, lut.cout, a, grid, st);
    else
      launch_apply<uint8_t, float>(lut.table_dtype, interp, lut.cout, a, grid, st);
  } else {
    if (dst_dtype == NIC_DT_U8)
      launch_apply<float, uint8_t>(lut.table_dtype, interp, lut.cout, a, grid, st);
    else
      launch_apply<float, float>(lut.table_dtype, interp, lut.cout, a, grid, st);
  }
  h->launches++;
  return (int)cudaGetLastError();
}

}  // namespace nic
