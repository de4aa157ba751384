// nic_sample.cu — the reference-exact (fp32) arm of nic_sample: the parity reference of the tensor-core sampling kernel
// (decode_tc_gws_kernel with TAPS > 0, nic_tc.cu).  Three steps on handle scratch:
//   sample_taps_kernel   the 2^D tap texels (int64 origins of one-texel blocks) and weights of every query (sample_tap);
//   mlp_forward_kernel   the fused fp32 decode of those Q * 2^D texels (launch_mlp_forward_f32, as nic_decode f32);
//   sample_blend_kernel  sum_k w_k * value_k in tap order, the optional mip blend, the output dtype.
// and of nic_sample_lod: 2 * 2^D rows per query (the taps at mip m, then at mip min(m + 1, L)), decoded by one pass of the
// same fp32 decode per mip of the chain (each pass keeps the rows of its mip), then the tap sums and the blend of nic.h.
#include "nic_tc_common.cuh"

namespace nic {

__global__ void __launch_bounds__(256) sample_taps_kernel(DevSampler s, int dim, long long rows, long long* __restrict__ taps,
                                                          float* __restrict__ weights) {
  const int T = 1 << dim;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
    const long long q = r >> dim;
    float u[3] = {0.f, 0.f, 0.f};
    for (int a = 0; a < dim; ++a) u[a] = __ldg(s.coords + q * dim + a);
    int p[3];
    weights[r] = sample_tap(s, dim, u, (int)(r & (T - 1)), p);
    for (int a = 0; a < dim; ++a) taps[r * dim + a] = p[a];
  }
}

template <typename OutT>
__global__ void __launch_bounds__(256) sample_blend_kernel(DevSampler s, int dim, int cout, long long total,
                                                           const float* __restrict__ weights, const float* __restrict__ values,
                                                           OutT* __restrict__ out) {
  const int T = 1 << dim;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long q = e / cout, c = e - q * cout;
    float acc = 0.f;
    for (int k = 0; k < T; ++k) {
      const long long r = q * T + k;
      acc = __fadd_rn(acc, __fmul_rn(weights[r], values[r * cout + c]));
    }
    store_out(out + e, sample_blend_prev(s, e, acc));
  }
}

int launch_sample_f32(Handle* h, const DevGeom& g, const DevSampler& smp, const MlpDev& m, const float* g0, const float* g1,
                      void* out, int out_dtype, cudaStream_t st) {
  const long long Q = g.nblocks, rows = Q << g.dim;
  if (Q == 0) return NIC_OK;
  const size_t b_taps = ((size_t)rows * g.dim * 8 + 255) & ~(size_t)255, b_w = ((size_t)rows * 4 + 255) & ~(size_t)255;
  const size_t b_val = (size_t)rows * m.cout * 4;
  int rc = ensure_scratch(&h->sample_scratch, &h->sample_scratch_bytes, b_taps + b_w + b_val);
  if (rc) return rc;
  long long* taps = (long long*)h->sample_scratch;
  float* weights = (float*)((uint8_t*)h->sample_scratch + b_taps);
  float* values = (float*)((uint8_t*)h->sample_scratch + b_taps + b_w);
  const long long cap = (long long)h->sms * 8;
  long long blocks = (rows + 255) / 256;
  sample_taps_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, st>>>(smp, g.dim, rows, taps, weights);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  DevGeom gt = g;                                   // every tap a one-texel block whose origin is the tap texel
  gt.nblocks = (int)rows;
  gt.N = rows;
  rc = launch_mlp_forward_f32(h, &gt, m, g0, g1, taps, nullptr, 0, rows, values, NIC_DT_F32, nullptr, nullptr, st);
  if (rc) return rc;
  const long long total = Q * m.cout;
  blocks = (total + 255) / 256;
  const int grid = (int)(blocks < cap ? blocks : cap);
  if (out_dtype == NIC_DT_U8)
    sample_blend_kernel<uint8_t><<<grid, 256, 0, st>>>(smp, g.dim, m.cout, total, weights, values, (uint8_t*)out);
  else
    sample_blend_kernel<float><<<grid, 256, 0, st>>>(smp, g.dim, m.cout, total, weights, values, (float*)out);
  h->launches++;
  return (int)cudaGetLastError();
}

// Rows of mip `mip` in the chain: row r = tap (r % 2T) of query r / 2T; the rows of other mips point at texel 0 (always
// inside the grids) and are dropped by sample_lod_keep_kernel.  Also records every row's mip and weight.
__global__ void __launch_bounds__(256) sample_lod_taps_kernel(DevChain c, DevSampler s, long long rows, int mip,
                                                              long long* __restrict__ taps, float* __restrict__ weights,
                                                              int* __restrict__ row_mip) {
  const int dim = c.dim, T = 1 << dim;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
    const long long q = r >> (dim + 1);
    const int k = (int)(r & (2 * T - 1));
    const int m = (int)floorf(lod_clamped(c, q));
    const int mi = min(m + (k >= T), c.num_mips - 1);
    float u[3] = {0.f, 0.f, 0.f};
    for (int a = 0; a < dim; ++a) u[a] = __ldg(s.coords + q * dim + a);
    for (int a = 0; a < 3; ++a) s.S[a] = c.mip[mi].S[a];
    int p[3];
    weights[r] = sample_tap(s, dim, u, k & (T - 1), p);
    row_mip[r] = mi;
    for (int a = 0; a < dim; ++a) taps[r * dim + a] = mi == mip ? p[a] : 0;
  }
}

__global__ void __launch_bounds__(256) sample_lod_keep_kernel(long long total, int cout, int mip, const int* __restrict__ row_mip,
                                                              const float* __restrict__ pass, float* __restrict__ values) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x)
    if (row_mip[e / cout] == mip) values[e] = pass[e];
}

template <typename OutT>
__global__ void __launch_bounds__(256) sample_lod_blend_kernel(DevChain c, int cout, long long total,
                                                               const float* __restrict__ weights,
                                                               const float* __restrict__ values, OutT* __restrict__ out) {
  const int T = 1 << c.dim;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long q = e / cout, ch = e - q * cout;
    const float lc = lod_clamped(c, q), t = __fsub_rn(lc, floorf(lc));
    float acc[2] = {0.f, 0.f};
    for (int h = 0; h < 2; ++h)
      for (int k = 0; k < T; ++k) {
        const long long r = q * 2 * T + h * T + k;
        acc[h] = __fadd_rn(acc[h], __fmul_rn(weights[r], values[r * cout + ch]));
      }
    store_out(out + e, lod_blend(t, acc[0], acc[1]));
  }
}

int launch_sample_lod_f32(Handle* h, const DevGeom* g, const DevChain& c, const DevSampler& smp, const MlpDev& m,
                          const float* const* g0, const float* const* g1, void* out, int out_dtype, cudaStream_t st) {
  const long long Q = g[0].nblocks, rows = Q << (c.dim + 1);
  if (Q == 0) return NIC_OK;
  const size_t b_taps = ((size_t)rows * c.dim * 8 + 255) & ~(size_t)255, b_w = ((size_t)rows * 4 + 255) & ~(size_t)255;
  const size_t b_val = ((size_t)rows * m.cout * 4 + 255) & ~(size_t)255;
  int rc = ensure_scratch(&h->sample_scratch, &h->sample_scratch_bytes, b_taps + 2 * b_w + 2 * b_val);
  if (rc) return rc;
  uint8_t* base = (uint8_t*)h->sample_scratch;
  long long* taps = (long long*)base;
  float* weights = (float*)(base + b_taps);
  int* row_mip = (int*)(base + b_taps + b_w);
  float* values = (float*)(base + b_taps + 2 * b_w);
  float* pass = (float*)(base + b_taps + 2 * b_w + b_val);
  const long long cap = (long long)h->sms * 8, total_rows = rows * m.cout;
  long long blocks = (rows + 255) / 256;
  const int grid_rows = (int)(blocks < cap ? blocks : cap);
  blocks = (total_rows + 255) / 256;
  const int grid_vals = (int)(blocks < cap ? blocks : cap);
  for (int i = 0; i < c.num_mips; ++i) {
    sample_lod_taps_kernel<<<grid_rows, 256, 0, st>>>(c, smp, rows, i, taps, weights, row_mip);
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    DevGeom gt = g[i];                              // every row a one-texel block whose origin is its tap texel
    gt.nblocks = (int)rows;
    gt.N = rows;
    rc = launch_mlp_forward_f32(h, &gt, m, g0[i], g1[i], taps, nullptr, 0, rows, pass, NIC_DT_F32, nullptr, nullptr, st);
    if (rc) return rc;
    sample_lod_keep_kernel<<<grid_vals, 256, 0, st>>>(total_rows, m.cout, i, row_mip, pass, values);
    h->launches++;
  }
  const long long total = Q * m.cout;
  blocks = (total + 255) / 256;
  const int grid = (int)(blocks < cap ? blocks : cap);
  if (out_dtype == NIC_DT_U8)
    sample_lod_blend_kernel<uint8_t><<<grid, 256, 0, st>>>(c, m.cout, total, weights, values, (uint8_t*)out);
  else
    sample_lod_blend_kernel<float><<<grid, 256, 0, st>>>(c, m.cout, total, weights, values, (float*)out);
  h->launches++;
  return (int)cudaGetLastError();
}

}  // namespace nic
