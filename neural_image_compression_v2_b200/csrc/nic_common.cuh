// nic_common.cuh — geometry, coordinate math, positional encodings and grid-tile staging shared by every
// kernel of libnic.so.  Arithmetic follows SURVEY.md Appendix A (reference: Projects/fp_def.py:115-223,
// Projects/utils.py:198-227); every quantity the reference computes with dyadic floats is computed with
// the same float32 operations here, so fp32 results are bit-identical.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "../../include/nic.h"

#define NIC_MAX_C 16        // channels per grid node supported by the staged kernels
#define NIC_MAX_PE 8        // PE channels per axis

// ------------------------------------------------------------------------------------------------ device geometry
// Flattened, kernel-friendly copy of NicGeom (built on the host by nic_api.cu).
struct DevGeom {
  int method, dim, C, PE, pe_kind, mip, interp;   // interp: 0 only when step == 2 (fp_def.py:136)
  int ncorner0;                                   // 4 (2-D, v2) or 8 (3-D)
  int cin;                                        // C*(ncorner0+1) + PE*dim + 1
  int n0[3], n1[3];                               // nodes along x,y,z
  int B[3];                                       // block extent along x,y,z (B[2] = 1 in 2-D)
  int nblocks;
  int origin0[3];
  float step;                                     // 2^step_log2, exact
  float lod;                                      // float(mip)
  float pe_div[NIC_MAX_PE];
  long long per_block;                            // B[0]*B[1]*B[2]
  long long N;                                    // nblocks*per_block
  // exact division of n < 2^31 by per_block, B[1]*B[2] and B[2]: q = (n * mul) >> (31 + shift)
  unsigned fd_mul[3], fd_shift[3];
  int metrics;                                    // training: also accumulate the squared error of the 8-bit outputs (loss_sum[1])
};

// corner tables, (dz,dy,dx) as the reference orders them
__device__ __constant__ int8_t kCorner2D[4][3] = {{0, 0, 0}, {0, 1, 0}, {0, 0, 1}, {0, 1, 1}};            // fp_def.py:81-86
__device__ __constant__ int8_t kCorner3D[8][3] = {{0, 0, 0}, {1, 0, 0}, {0, 1, 0}, {1, 1, 0},
                                                  {0, 0, 1}, {1, 0, 1}, {0, 1, 1}, {1, 1, 1}};            // fp_def.py:96-103
__device__ __constant__ int8_t kCorner3Dv2[4][3] = {{0, 0, 0}, {1, 1, 0}, {1, 0, 1}, {0, 1, 1}};          // fp_def.py:108-111
// AS-CODED 3-D G1 weights (fp_def.py:176-183): which factor (k = 1, 1-k = 0) axes x,y,z contribute per corner.
__device__ __constant__ int8_t kW3D[8][3] = {{0, 0, 0}, {0, 0, 1}, {0, 1, 0}, {1, 0, 0},
                                             {1, 1, 0}, {1, 0, 1}, {0, 1, 1}, {1, 1, 1}};

struct AxisCoord {
  int i0, i1;   // floor(u0), floor(u1)
  float u1, k;  // u1 = u0/2, k = u1 - i1
};

// fp_def.py:116-123,137-138 for one axis.  p = origin + offset (integer texel coordinate).
__device__ __forceinline__ AxisCoord axis_coord(int p, float step) {
  AxisCoord a;
  float u0 = __fmul_rn((float)p, step);
  a.i0 = (int)floorf(u0);
  a.u1 = __fmul_rn(u0, 0.5f);
  a.i1 = (int)floorf(a.u1);
  a.k = __fsub_rn(a.u1, (float)a.i1);
  return a;
}

// utils.py:226-227: tri(x, o) = 2*|((x - o) mod 2) - 1| - 1 with floor-mod.
__device__ __forceinline__ float tri_wave(float x, float offset) {
  float v = __fsub_rn(x, offset);
  float m = __fsub_rn(v, __fmul_rn(2.0f, floorf(__fmul_rn(v, 0.5f))));   // exact for dyadic v
  return __fsub_rn(__fmul_rn(2.0f, fabsf(__fsub_rn(m, 1.0f))), 1.0f);
}

// Row r (0..PE-1) of the triangular encoding of coordinate u (utils.py:211-223):
// r = PE - (2*octave + i + 1), (i, offset) in ((0, .5), (1, 0)), (octave 0, i 0) skipped -> stays 0.
__device__ __forceinline__ float pe_triangular(float u, int r, int PE) {
  int q = PE - 1 - r;          // = 2*octave + i
  if (q <= 0 || q >= 2 * (PE / 2)) return 0.0f;
  int octave = q >> 1, i = q & 1;
  float x = __fmul_rn(u, __int_as_float((127 - octave) << 23));   // u / 2^octave, exact (power-of-two divisor)
  return tri_wave(x, i ? 0.0f : 0.5f);
}

// Row r of the sinusoidal encoding (utils.py:198-208): even rows sin(u*div[r/2]), odd rows cos(u*div[r/2]).
__device__ __forceinline__ float pe_sinusoidal(float u, int r, const float* div) {
  float arg = __fmul_rn(u, div[r >> 1]);
  return (r & 1) ? cosf(arg) : sinf(arg);
}

__device__ __forceinline__ float pe_value(const DevGeom& g, float u, int r) {
  return g.pe_kind == NIC_PE_TRIANGULAR ? pe_triangular(u, r, g.PE) : pe_sinusoidal(u, r, g.pe_div);
}

// Texel of sample n: block, offsets, integer coordinates.
struct Texel {
  int b;
  int p[3];
};

__device__ __forceinline__ Texel texel_of(const DevGeom& g, long long n, const long long* origins) {
  Texel t;
  t.b = (int)(n / g.per_block);
  long long r = n - (long long)t.b * g.per_block;
  int iz = (int)(r % g.B[2]);
  r /= g.B[2];
  int iy = (int)(r % g.B[1]);
  int ix = (int)(r / g.B[1]);
  int o[3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
    o[a] = origins ? (a < g.dim ? (int)origins[(long long)t.b * g.dim + a] : 0) : (t.b == 0 ? g.origin0[a] : 0);
  t.p[0] = o[0] + ix;
  t.p[1] = o[1] + iy;
  t.p[2] = o[2] + iz;
  return t;
}

// n / d for n < 2^31 with mul = ceil(2^(31+shift) / d), shift = ceil(log2 d): one wide multiply and a shift.
__device__ __forceinline__ unsigned fastdiv31(unsigned n, unsigned mul, unsigned shift) {
  return (unsigned)(((unsigned long long)n * mul) >> (31 + shift));
}

// texel_of for N < 2^31 without 64-bit division (the tensor-core kernels' per-tile index math).
__device__ __forceinline__ Texel texel_of_fast(const DevGeom& g, unsigned n, const long long* origins) {
  Texel t;
  unsigned b = fastdiv31(n, g.fd_mul[0], g.fd_shift[0]);
  unsigned r = n - b * (unsigned)g.per_block;
  unsigned ix = fastdiv31(r, g.fd_mul[1], g.fd_shift[1]);
  unsigned r2 = r - ix * (unsigned)(g.B[1] * g.B[2]);
  unsigned iy = fastdiv31(r2, g.fd_mul[2], g.fd_shift[2]);
  unsigned iz = r2 - iy * (unsigned)g.B[2];
  t.b = (int)b;
  int o[3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
    o[a] = origins ? (a < g.dim ? (int)origins[(long long)b * g.dim + a] : 0) : (b == 0 ? g.origin0[a] : 0);
  t.p[0] = o[0] + (int)ix;
  t.p[1] = o[1] + (int)iy;
  t.p[2] = o[2] + (int)iz;
  return t;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ------------------------------------------------------------------------------------------------ filtered sampling
// What nic_sample / nic_sample_codes filter: the texel extent of the mip and how coordinates map onto it (nic.h NicSampler).
struct DevSampler {
  const float* coords;    // [Q, dim] normalised (x, y[, z])
  int S[3];               // texels per axis (1 on unused axes)
  int address;            // NIC_ADDRESS_*
  int align_corners;
  float blend_weight;     // out = (1 - t) * prev + t * sample when prev != NULL
  const float* prev;      // [Q, cout] fp32 or NULL
};

// Tap `tap` (0 .. 2^dim - 1, x slowest) of the linear filter at normalised coordinates u[0..dim): writes the integer texel
// of the mip to p[0..3) and returns the tap's weight.  Every step is one explicit fp32 operation (nic.h documents the rule),
// so the oracle reproduces it bit for bit; after the clamp to +-2^24 the index arithmetic is exact (NaN -> -2^24).
__device__ __forceinline__ float sample_tap(const DevSampler& s, int dim, const float* u, int tap, int* p) {
  float w = 1.0f;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    p[a] = 0;
    if (a >= dim) continue;
    const int S = s.S[a];
    float x = s.align_corners ? __fmul_rn(u[a], (float)(S - 1)) : __fsub_rn(__fmul_rn(u[a], (float)S), 0.5f);
    x = fminf(fmaxf(x, -16777216.0f), 16777216.0f);
    const float i0 = floorf(x), f = __fsub_rn(x, i0);
    const int hi = (tap >> (dim - 1 - a)) & 1;
    int i = (int)i0 + hi;
    if (s.address == NIC_ADDRESS_WRAP) {
      i %= S;                 // = fmodf(i, S): exact, sign of the dividend
      if (i < 0) i += S;
    } else {
      i = clampi(i, 0, S - 1);
    }
    p[a] = i;
    w = __fmul_rn(w, hi ? f : __fsub_rn(1.0f, f));
  }
  return w;
}

// Tetrahedral interpolation of an S[0] x S[1] x S[2] table at normalised coordinates u[0..3) (nic.h nic_lut_apply), on
// sample_tap's axis rule with align_corners and clamp addressing: writes the texels of the 4 corners to p[k][0..3) and their
// weights to w[k], k = 0..3 in summation order.  The axes are ordered by descending fraction with a fixed compare-exchange
// network (swaps only on a strictly larger fraction, so ties keep x before y before z), which compiles to selects.
__device__ __forceinline__ void tetra_corners(const int* S, const float* u, int (*p)[3], float* w) {
  float f[3];
  int lo[3], hi[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float x = __fmul_rn(u[a], (float)(S[a] - 1));
    x = fminf(fmaxf(x, -16777216.0f), 16777216.0f);
    const float i0 = floorf(x);
    f[a] = __fsub_rn(x, i0);
    lo[a] = clampi((int)i0, 0, S[a] - 1);
    hi[a] = clampi((int)i0 + 1, 0, S[a] - 1);
  }
  float f1 = f[0], f2 = f[1], f3 = f[2];
  int m1 = 1, m2 = 2, m3 = 4;                       // the axis of each rank as a bit: x = 1, y = 2, z = 4
  auto cx = [](float& fa, int& ma, float& fb, int& mb) {
    const bool sw = fb > fa;
    const float tf = sw ? fb : fa;
    const int tm = sw ? mb : ma;
    fb = sw ? fa : fb;
    mb = sw ? ma : mb;
    fa = tf;
    ma = tm;
  };
  cx(f1, m1, f2, m2);
  cx(f2, m2, f3, m3);
  cx(f1, m1, f2, m2);
  const int mask[4] = {0, m1, m1 | m2, 7};
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int a = 0; a < 3; ++a) p[k][a] = (mask[k] >> a) & 1 ? hi[a] : lo[a];
  w[0] = __fsub_rn(1.0f, f1);
  w[1] = __fsub_rn(f1, f2);
  w[2] = __fsub_rn(f2, f3);
  w[3] = f3;
}

// The last step of a sample: the optional blend with the previous mip's result, element `idx` of [Q, cout].
__device__ __forceinline__ float sample_blend_prev(const DevSampler& s, long long idx, float v) {
  if (!s.prev) return v;
  return __fadd_rn(__fmul_rn(__fsub_rn(1.0f, s.blend_weight), __ldg(s.prev + idx)), __fmul_rn(s.blend_weight, v));
}

// Per-query level of detail (nic.h NicMipChain): what varies from one mip of the chain to the next, and the LOD inputs.
struct DevMip {
  int n0[3], n1[3];       // nodes of the mip's two grids along x, y, z
  int S[3];               // texels per axis (1 on unused axes)
  float step;             // 2^step_log2
  int interp;             // 0 at step 2 (fp_def.py:136)
  int lut_shift;          // tensor-core PE: index (p << lut_shift) & 63 of the 64-entry LUT built at step 1/4
  unsigned s0, s1;        // tensor-core path: offsets (in uint2) of the mip's shadow grids
};
struct DevChain {
  int num_mips, dim, address, align_corners;
  const float* lod;       // [Q], or NULL with ddx / ddy [Q, dim]
  const float* ddx;
  const float* ddy;
  float E0[3];            // extent of mip 0 (derivatives are in normalised units)
  DevMip mip[NIC_MAX_MIPS];
};
// nic_decode_mips (tensor core): the chain table of the dense pass over mips 1 .. L and the pass's first row of each mip
// (row0[0] = row0[1] = 0: mip 0 has no rows in the pass; 0xffffffff past the last mip).  Row n belongs to the mip with the
// largest row0 <= n.
struct DevMipRows {
  DevChain c;
  unsigned row0[NIC_MAX_MIPS];
};

// lambda of query q clamped to [0, L] (nic.h nic_sample_lod; every step one fp32 operation).  fmaxf maps NaN and the -inf
// of zero derivatives to 0.
__device__ __forceinline__ float lod_clamped(const DevChain& c, long long q) {
  float lam;
  if (c.lod) {
    lam = __ldg(c.lod + q);
  } else {
    float sx = 0.f, sy = 0.f;
    for (int a = 0; a < c.dim; ++a) {
      const float px = __fmul_rn(__ldg(c.ddx + q * c.dim + a), c.E0[a]), py = __fmul_rn(__ldg(c.ddy + q * c.dim + a), c.E0[a]);
      sx = a == 0 ? __fmul_rn(px, px) : __fadd_rn(sx, __fmul_rn(px, px));
      sy = a == 0 ? __fmul_rn(py, py) : __fadd_rn(sy, __fmul_rn(py, py));
    }
    lam = __fmul_rn(0.5f, log2f(fmaxf(sx, sy)));
  }
  return fminf(fmaxf(lam, 0.0f), (float)(c.num_mips - 1));
}

// out = (1 - t) * s_m + t * s_m1: the fp32 sequence of sample_blend_prev.
__device__ __forceinline__ float lod_blend(float t, float s_m, float s_m1) {
  return __fadd_rn(__fmul_rn(__fsub_rn(1.0f, t), s_m), __fmul_rn(t, s_m1));
}

// Linear node index in a channel-major grid [C, (z,) y, x]; indices clamped for memory safety (the reference
// raises IndexError instead; host-known origins are validated in nic_api.cu).
__device__ __forceinline__ long long node_index(const int* nodes, int dim, int x, int y, int z) {
  x = clampi(x, 0, nodes[0] - 1);
  y = clampi(y, 0, nodes[1] - 1);
  if (dim == 2) return (long long)y * nodes[0] + x;
  z = clampi(z, 0, nodes[2] - 1);
  return ((long long)z * nodes[1] + y) * nodes[0] + x;
}

__device__ __forceinline__ long long plane_size(const int* nodes, int dim) {
  return dim == 2 ? (long long)nodes[0] * nodes[1] : (long long)nodes[0] * nodes[1] * nodes[2];
}

// G1 interpolation weight of corner j (SURVEY Appendix A): 2-D true bilinear evaluated as (wx)*(wy) factors
// applied left to right on the value; 3-D uses the AS-CODED (permuted) table.  Returns the three factors.
__device__ __forceinline__ void g1_factors(const DevGeom& g, int j, const AxisCoord* ax, float* f) {
  if (!g.interp) {
    f[0] = f[1] = f[2] = 1.0f;
    return;
  }
  if (g.dim == 2) {
    int dy = kCorner2D[j][1], dx = kCorner2D[j][2];
    f[0] = dx ? ax[0].k : __fsub_rn(1.0f, ax[0].k);
    f[1] = dy ? ax[1].k : __fsub_rn(1.0f, ax[1].k);
    f[2] = 1.0f;
  } else {
#pragma unroll
    for (int a = 0; a < 3; ++a) f[a] = kW3D[j][a] ? ax[a].k : __fsub_rn(1.0f, ax[a].k);
  }
}

// Value of decoder-input column `col` for a texel, straight from global memory (used by the generic gather
// kernel and as the reference device implementation the staged kernels are tested against).
__device__ __forceinline__ float gather_column(const DevGeom& g, const float* __restrict__ g0,
                                               const float* __restrict__ g1, const AxisCoord* ax, int col) {
  const int C = g.C;
  const int n0c = g.ncorner0 * C;
  if (col < n0c) {
    int j = col / C, c = col - j * C;
    const int8_t* d = g.dim == 2 ? kCorner2D[j] : (g.method == NIC_METHOD_3D ? kCorner3D[j] : kCorner3Dv2[j]);
    long long idx = node_index(g.n0, g.dim, ax[0].i0 + d[2], ax[1].i0 + d[1], ax[2].i0 + d[0]);
    return __ldg(g0 + (long long)c * plane_size(g.n0, g.dim) + idx);
  }
  if (col < n0c + C) {
    int c = col - n0c;
    const float* plane = g1 + (long long)c * plane_size(g.n1, g.dim);
    const int nc1 = g.dim == 2 ? 4 : 8;
    float acc = 0.0f;
    for (int j = 0; j < nc1; ++j) {
      const int8_t* d = g.dim == 2 ? kCorner2D[j] : kCorner3D[j];
      float v = __ldg(plane + node_index(g.n1, g.dim, ax[0].i1 + d[2], ax[1].i1 + d[1], ax[2].i1 + d[0]));
      if (g.interp) {
        float f[3];
        g1_factors(g, j, ax, f);
        v = __fmul_rn(__fmul_rn(v, f[0]), f[1]);
        if (g.dim == 3) v = __fmul_rn(v, f[2]);
      }
      acc = j == 0 ? v : __fadd_rn(acc, v);
    }
    return acc;
  }
  int q = col - (n0c + C);
  if (q < g.PE * g.dim) {
    int a = q / g.PE, r = q - a * g.PE;
    return pe_value(g, ax[a].u1, r);
  }
  return g.lod;
}

// ------------------------------------------------------------------------------------------------ misc helpers
__device__ __forceinline__ float gelu_erf(float z) { return 0.5f * z * (1.0f + erff(z * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_erf_grad(float z) {
  float cdf = 0.5f * (1.0f + erff(z * 0.70710678118654752440f));
  float pdf = 0.39894228040143267794f * __expf(-0.5f * z * z);
  return cdf + z * pdf;
}
__device__ __forceinline__ float sigmoidf_exact(float z) { return 1.0f / (1.0f + expf(-z)); }

// floor(v*scale + .5) with SEPARATE multiply and add (no FMA contraction), models.py:55-64.
__device__ __forceinline__ float quant_round(float v, float scale) { return floorf(__fadd_rn(__fmul_rn(v, scale), 0.5f)); }
