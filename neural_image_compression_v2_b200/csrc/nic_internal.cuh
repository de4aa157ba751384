// nic_internal.cuh — host-side handle, device-side parameter blocks and the launch prototypes that tie
// nic_api.cu (the C ABI) to the kernel translation units.
#pragma once
#include "nic_common.cuh"

#define NIC_MAX_CIN 160     // widest decoder input the fp32 kernels accept (method 3: 9C + 3PE + 1 = 127 at C=12)
#define NIC_MAX_COUT 16     // widest decoder output

namespace nic {

struct MlpDev {
  int cin, hidden, cout;
  const float *w1, *b1, *w2, *b2, *w3, *b3;
};
struct MlpGradDev {
  float *w1, *b1, *w2, *b2, *w3, *b3;
};

struct Handle {
  int device;
  int sms;
  int cc_major, cc_minor;
  long long launches;
  char err[256];
  // scratch owned by the handle (device memory)
  void* tc_weights;          // packed f16/bf16 UMMA operand images of the decoder weights
  size_t tc_weights_bytes;
  void* tc_shadow;           // 16-bit channel-last shadows of the two active grids
  size_t tc_shadow_bytes;
  void* tc_gscratch;         // channel-last fp32 grid-gradient scratch of the tensor-core training step (kept zero)
  size_t tc_gscratch_bytes;
  unsigned* xch_err;         // device words: [0] an exchange timed out waiting for a peer (nic_exchange_status), [1] release word
  unsigned xch_seq;          // launches of the exchange kernel so far
  unsigned* xch_host_err;    // mapped pinned host copy of xch_err[0] (read by the next API call without a sync) + its device alias
  unsigned* xch_host_err_dev;
  int xch_resident_blocks;   // occupancy-bounded co-resident blocks of adam_exchange_kernel on this device
  int xch_timeout_ms;        // NIC_OPT_EXCHANGE_TIMEOUT_MS (0 = default 10 s)
  void* tc_partials;         // per-CTA MLP-gradient partial sums of the tensor-core training step
  size_t tc_partials_bytes;
  int disable_fast2d;        // testing knob: force the general tensor-core kernel
  int reuse_prepared;        // NIC_OPT_REUSE_PREPARED
  int debug_flags;           // knock-out experiments (option 100), never set in production
  unsigned long long* dbg_counters;   // 16 device counters (nic_debug_counters), allocated on first use
  int static_tiles;          // NIC_OPT_STATIC_TILES: static tile order in the tensor-core training kernel
  int step_metrics;          // NIC_OPT_STEP_METRICS: training steps also accumulate the 8-bit squared error in loss_sum[1]
  void* data_scratch;        // nic_data.cu: resample coefficient tables + 8-bit intermediate
  size_t data_scratch_bytes;
  void* sample_scratch;      // nic_sample.cu: tap texels, tap weights and tap outputs of the fp32 sampling arm
  size_t sample_scratch_bytes;
  void* lod_chain;           // nic_sample_lod / nic_decode_mips (tensor core): device copy of the call's chain table
                             // (sizeof(DevMipRows) bytes)
  int gelu_poly;             // NIC_OPT_GELU_POLY: -1 = tuned default, 0..8 = activation pairs (of 8) on the polynomial GELU
  struct PreparedKey {       // what the tables in tc_weights / tc_shadow were last built from (compared with memcmp)
    int kind;                // PreparedKind: the kernel they were built for (PREP_NONE: nothing valid)
    int fmt, code_bits, npoly, method, pe_kind, mip, num_mips;
    const void *w1, *b1, *w2, *b2, *w3, *b3;
    struct Mip {             // each mip the call reads: one for a single-mip call, the whole chain for nic_sample_lod
      const void *g0, *g1;
      int n0[3], n1[3];
      float step;
    } mips[NIC_MAX_MIPS];
  } prepared;
  void* adam_desc;           // device copy of NicAdamTensor descriptors
  size_t adam_desc_bytes;
  // NIC_OPT_TIME_KERNELS: event pairs around the dominant kernel of each call (ring of NIC_MAX_TIMED pairs)
  int time_kernels;
  int timed_count;
  cudaEvent_t timed_ev[2 * 256];
};
#define NIC_MAX_TIMED 256

// The kernels whose tables a PreparedKey describes: each builds its own weight image (and shadows or G1 rows), so tables
// are shared only between calls of the same kind.
enum PreparedKind { PREP_NONE = 0, PREP_GENERAL, PREP_FAST2D, PREP_CODES, PREP_CHAIN };
// Marks the prepared tables stale: their scratch was reallocated, or overwritten by the training step.
static inline void invalidate_prepared(Handle* h) { h->prepared.kind = PREP_NONE; }

// Brackets the dominant kernel of a call with events when NIC_OPT_TIME_KERNELS is on (no-op otherwise).
// Programmatic dependent launch (sm_90+): a kernel launched with launch_pdl() may start while its predecessor in the
// stream is still running (after every CTA of the predecessor has called pdl_launch_dependents() or exited); it must call
// pdl_wait() before touching anything the predecessor writes.  Hides the launch latency between the small dependent
// kernels of a training step.  Both calls are no-ops in a normally launched kernel.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

struct KernelTimer {
  Handle* h;
  cudaStream_t st;
  int slot;
  KernelTimer(Handle* h_, cudaStream_t st_) : h(h_), st(st_), slot(-1) {
    if (!h->time_kernels || h->timed_count >= NIC_MAX_TIMED) return;
    slot = h->timed_count;
    for (int i = 0; i < 2; ++i)
      if (!h->timed_ev[2 * slot + i] && cudaEventCreate(&h->timed_ev[2 * slot + i]) != cudaSuccess) { slot = -1; return; }
    cudaEventRecord(h->timed_ev[2 * slot], st);
  }
  ~KernelTimer() {
    if (slot < 0) return;
    cudaEventRecord(h->timed_ev[2 * slot + 1], st);
    h->timed_count = slot + 1;
  }
};

// ---------------------------------------------------------------------------------------------- typed stores
__device__ __forceinline__ void store_as(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_as(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void store_as(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
// decoder outputs: float as is, uint8 = floor(v*255 + .5) (models.quantize_to_bit, models.py:29-40)
__device__ __forceinline__ void store_out(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_out(uint8_t* p, float v) {
  float q = quant_round(v, 255.0f);
  *p = (uint8_t)(q < 0.f ? 0.f : (q > 255.f ? 255.f : q));
}

// ---------------------------------------------------------------------------------------------- row iterator
// Calls f(col, value) for every decoder-input column of one texel in reference column order
// (image_compression.py:94-96): G0 corners | sum of weighted G1 corners | PE per axis | LOD.
template <class F>
__device__ __forceinline__ void for_each_input(const DevGeom& g, const float* __restrict__ g0,
                                               const float* __restrict__ g1, const AxisCoord* ax, F&& f) {
  const int C = g.C;
  const long long ps0 = plane_size(g.n0, g.dim), ps1 = plane_size(g.n1, g.dim);
  int col = 0;
  for (int j = 0; j < g.ncorner0; ++j) {
    const int8_t* d = g.dim == 2 ? kCorner2D[j] : (g.method == NIC_METHOD_3D ? kCorner3D[j] : kCorner3Dv2[j]);
    const float* p = g0 + node_index(g.n0, g.dim, ax[0].i0 + d[2], ax[1].i0 + d[1], ax[2].i0 + d[0]);
    for (int c = 0; c < C; ++c) f(col++, __ldg(p + (long long)c * ps0));
  }
  const int nc1 = g.dim == 2 ? 4 : 8;
  long long idx1[8];
  float fac[8][3];
  for (int j = 0; j < nc1; ++j) {
    const int8_t* d = g.dim == 2 ? kCorner2D[j] : kCorner3D[j];
    idx1[j] = node_index(g.n1, g.dim, ax[0].i1 + d[2], ax[1].i1 + d[1], ax[2].i1 + d[0]);
    g1_factors(g, j, ax, fac[j]);
  }
  for (int c = 0; c < C; ++c) {
    const float* plane = g1 + (long long)c * ps1;
    float acc = 0.f;
    for (int j = 0; j < nc1; ++j) {
      float v = __ldg(plane + idx1[j]);
      if (g.interp) {
        v = __fmul_rn(__fmul_rn(v, fac[j][0]), fac[j][1]);
        if (g.dim == 3) v = __fmul_rn(v, fac[j][2]);
      }
      acc = j == 0 ? v : __fadd_rn(acc, v);
    }
    f(col++, acc);
  }
  for (int a = 0; a < g.dim; ++a)
    for (int r = 0; r < g.PE; ++r) f(col++, pe_value(g, ax[a].u1, r));
  f(col, g.lod);
}

// Transpose of one grid column of the gather: adds v (d loss / d X[col]) into the grid gradients.
__device__ __forceinline__ void scatter_column(const DevGeom& g, float* __restrict__ dg0, float* __restrict__ dg1,
                                               const AxisCoord* ax, int col, float v) {
  const int C = g.C;
  const int n0c = g.ncorner0 * C;
  if (col < n0c) {
    int j = col / C, c = col - j * C;
    const int8_t* d = g.dim == 2 ? kCorner2D[j] : (g.method == NIC_METHOD_3D ? kCorner3D[j] : kCorner3Dv2[j]);
    long long idx = node_index(g.n0, g.dim, ax[0].i0 + d[2], ax[1].i0 + d[1], ax[2].i0 + d[0]);
    atomicAdd(dg0 + (long long)c * plane_size(g.n0, g.dim) + idx, v);
    return;
  }
  int c = col - n0c;
  if (c >= C) return;
  float* plane = dg1 + (long long)c * plane_size(g.n1, g.dim);
  const int nc1 = g.dim == 2 ? 4 : 8;
  for (int j = 0; j < nc1; ++j) {
    const int8_t* d = g.dim == 2 ? kCorner2D[j] : kCorner3D[j];
    float f[3];
    g1_factors(g, j, ax, f);
    float w = f[0] * f[1] * f[2];
    if (w != 0.f) atomicAdd(plane + node_index(g.n1, g.dim, ax[0].i1 + d[2], ax[1].i1 + d[1], ax[2].i1 + d[0]), w * v);
  }
}

// ---------------------------------------------------------------------------------------------- Philox4x32-10
template <int ROUNDS>
__device__ __forceinline__ uint4 philox4x32_r(unsigned long long seed, unsigned long long offset, unsigned long long counter) {
  unsigned int k0 = (unsigned int)seed, k1 = (unsigned int)(seed >> 32);
  unsigned int c0 = (unsigned int)counter, c1 = (unsigned int)(counter >> 32);
  unsigned int c2 = (unsigned int)offset, c3 = (unsigned int)(offset >> 32);
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    unsigned int n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ uint4 philox4x32(unsigned long long seed, unsigned long long offset, unsigned long long counter) {
  return philox4x32_r<10>(seed, offset, counter);
}

// Quantisation noise of image_compression.py:250: (U[0,1) - 0.5) / 2^bits for element `idx` of step `step`.
// Element idx uses word idx%4 of Philox block idx/4 (key = seed, high counter words = step).
__device__ __forceinline__ float philox_noise(unsigned long long seed, unsigned long long step,
                                              unsigned long long idx, int bits) {
  uint4 r = philox4x32(seed, step, idx >> 2);
  unsigned int w = (idx & 3) == 0 ? r.x : ((idx & 3) == 1 ? r.y : ((idx & 3) == 2 ? r.z : r.w));
  float u = (float)(w >> 8) * (1.0f / 16777216.0f);
  return (u - 0.5f) * exp2f(-(float)bits);
}

// ---------------------------------------------------------------------------------------------- launchers
int launch_gather(Handle* h, const DevGeom& g, const float* g0, const float* g1, const long long* origins, void* x,
                  int x_dtype, cudaStream_t st);
bool gather_tile_eligible(const DevGeom& g, const void* x);
int launch_gather_tile(Handle* h, const DevGeom& g, const float* g0, const float* g1, const long long* origins, void* x,
                       int x_dtype, cudaStream_t st);
int launch_scatter(Handle* h, const DevGeom& g, const float* dx, const long long* origins, float* dg0, float* dg1,
                   cudaStream_t st);
int launch_sample_crops(Handle* h, const float* img, int dim, int ci, const int* size, const long long* origins, int ncrops,
                        const int* crop, float* out, cudaStream_t st);
int launch_sample_crops_random(Handle* h, const float* img, int dim, int ci, const int* size, int ncrops, const int* crop,
                               unsigned long long seed, unsigned long long step, long long* origins_out, float* out,
                               cudaStream_t st);
int launch_resize_bilinear_u8(Handle* h, const uint8_t* src, int H, int W, int C, int out_h, int out_w, uint8_t* dst_u8,
                              float* dst_f32, cudaStream_t st);
int launch_atlas(Handle* h, uint8_t* frames, uint8_t* atlas, int T, int S, int C, int A, int unpack, cudaStream_t st);
int launch_pe(Handle* h, const float* coord, int dim, long long n, int PE, int kind, const float* div_host, float* out,
              cudaStream_t st);
int launch_mlp_forward_f32(Handle* h, const DevGeom* g, const MlpDev& m, const float* g0, const float* g1,
                           const long long* origins, const float* x, long long ldx, long long N, void* out,
                           int out_dtype, float* z1, float* z2, cudaStream_t st);
int launch_mlp_backward_f32(Handle* h, const MlpDev& m, const MlpGradDev& gm, const float* x, long long ldx,
                            long long N, const float* z1, const float* z2, const float* out, const float* dout,
                            float* dx, cudaStream_t st);
int launch_train_f32(Handle* h, const DevGeom& g, const MlpDev& m, const MlpGradDev& gm, const float* g0,
                     const float* g1, const long long* origins, const float* targets, const float* noise,
                     int noise_bits, unsigned long long seed, unsigned long long step, float grad_scale, float* dg0,
                     float* dg1, float* loss_sum, float* out_save, cudaStream_t st);
// The tensor-core launchers read the grids as float32 (code_bits = 0) or as uint8 codes of width code_bits (1..8).
int launch_decode_tc(Handle* h, const DevGeom& g, const MlpDev& m, const void* g0, const void* g1, int code_bits,
                     const long long* origins, void* out, int out_dtype, int precision, cudaStream_t st);
// nic_sample / nic_sample_codes: g describes the mip with nblocks = queries (one texel each); smp the filter.
int launch_sample_tc(Handle* h, const DevGeom& g, const DevSampler& smp, const MlpDev& m, const void* g0, const void* g1,
                     int code_bits, void* out, int out_dtype, int precision, cudaStream_t st);
int launch_sample_f32(Handle* h, const DevGeom& g, const DevSampler& smp, const MlpDev& m, const float* g0, const float* g1,
                      void* out, int out_dtype, cudaStream_t st);
// nic_sample_lod / nic_sample_lod_codes: g[i] describes mip i of the chain as launch_sample_* take it; c the chain.
int launch_sample_lod_tc(Handle* h, const DevGeom* g, const DevChain& c, const DevSampler& smp, const MlpDev& m,
                         const void* const* g0, const void* const* g1, int code_bits, void* out, int out_dtype,
                         int precision, cudaStream_t st);
int launch_sample_lod_f32(Handle* h, const DevGeom* g, const DevChain& c, const DevSampler& smp, const MlpDev& m,
                          const float* const* g0, const float* const* g1, void* out, int out_dtype, cudaStream_t st);
// nic_decode_mips / nic_decode_mips_codes (tensor core): g[i] describes mip i as one whole-mip block; c the chain.
int launch_decode_mips_tc(Handle* h, const DevGeom* g, const DevChain& c, const MlpDev& m, const void* const* g0,
                          const void* const* g1, int code_bits, void* out, int out_dtype, int precision, cudaStream_t st);
// nic_lut_pack / nic_lut_apply (nic_lut.cu): arguments validated by nic_api.cu.
int launch_lut_pack(Handle* h, const float* dense, long long texels, int cout, void* table, int table_dtype, cudaStream_t st);
int launch_lut_apply(Handle* h, const NicLut& lut, const void* src, int src_dtype, long long pixels, void* dst, int dst_dtype,
                     int interp, cudaStream_t st);
int launch_train_tc(Handle* h, const DevGeom& g, const MlpDev& m, const MlpGradDev& gm, const float* g0, const float* g1,
                    const long long* origins, const float* targets, const float* noise, int noise_bits,
                    unsigned long long seed, unsigned long long step, float grad_scale, float* dg0, float* dg1,
                    float* loss_sum, float* out_save, int precision, cudaStream_t st);
int launch_adam(Handle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                float grad_scale, int zero_grad, float* loss_sum, float* loss_out, float loss_scale, cudaStream_t st);
int launch_adam_exchange(Handle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                         float grad_scale, const NicExchange& x, const float* loss_sum, float* loss_out, float loss_scale,
                         cudaStream_t st);
int launch_quantize4fp(Handle* h, const float* src, float* dst, long long n, int bits, cudaStream_t st);
int launch_quantize_pack(Handle* h, const float* src, uint8_t* codes, long long n, int bits, cudaStream_t st);
int launch_unpack(Handle* h, const uint8_t* codes, float* dst, long long n, int bits, cudaStream_t st);
int launch_pack_bits(Handle* h, const uint8_t* src, uint8_t* dst, long long n, int bits, int unpack, cudaStream_t st);
int launch_clamp(Handle* h, float* p, long long n, float lo, float hi, cudaStream_t st);
int launch_output_to_u8(Handle* h, const float* src, uint8_t* dst, long long n, int bits, cudaStream_t st);
int launch_sse_u8(Handle* h, const uint8_t* a, const uint8_t* b, long long n, double* sse, cudaStream_t st);

}  // namespace nic
