// nic_train_tc.cu — K3 + K4 on tensor cores: one fused training step (gather, quantisation noise, decoder forward, MSE,
// full backward, weight-gradient sums, grid-gradient scatter) with EVERY GEMM on tcgen05.mma (sm_100a).
// Reference behaviour: the body of train_models up to loss.backward() (Projects/image_compression.py:239-265) on the
// 2-D path (create_decoder_input_2d :71-100, fp_def.create_g0_g1 fp_def.py:115-145) and the 3-D "v2" path (method 4:
// create_decoder_input_3d_v2 :137-167, fp_def.create_g0_g1_3d_v2 fp_def.py:187-223), ColorDecoder :54-68.
//
// Per CTA (persistent, 256 threads = 2 warpgroups, TWO CTAs per SM: 106 KB smem, 256 TMEM columns, <= 128 registers), per tile of 128 samples (= MMA M = TMEM lanes):
//   activations live in shared memory as [sample-group of 8][feature-group of 8][8 samples][8 features] 16-bit core
//   matrices.  ONE copy serves three operand views (no transposes are ever materialised):
//     * K-major A  (M = samples,  K = features)  for the forward GEMMs and the delta-propagation GEMMs,
//     * MN-major A (M = features, K = samples)   for the weight-gradient GEMMs (the reduction runs over the samples),
//     * MN-major B (N = features, K = samples)   likewise;
//   and the forward weight images W' (K-major B) double as MN-major B for the delta-propagation GEMMs (W'^T).
//   forward : Z1 = X~ W1'^T           (5 MMAs K=16)  -> h1' = 2 gelu(z1), g1' = d h1'/d z1 (registers)   -> H1
//             Z2 = [H1|1] W2'^T       (5)            -> h2', g2'                                        -> H2
//             Z3 = [H2|1] W3'^T       (5, N=16)      -> out = sigmoid, loss, dz3 = S (out - t) out (1 - out) -> DZ[0:16)
//   backward: dH2 = dZ3 W3'           (1)   and  D3^T += [H2|1]^T dZ3 (8 MMAs, M=128 N=16 K=128: dW3'^T, db3 in row 64)
//             dZ2 = dH2 * g2' -> DZ[16:80)
//             dH1 = dZ2 W2'           (4)   and  D2 += DZ^T [H1|1]   (8: dW2', db2 in rows 16..79)
//             dZ1 = dH1 * g1' -> the H2 buffer, features [0:64) (H2 is dead by then; DZ is still read by the D2 batch)
//             dX  = dZ1 W1'           (4)   and  D1 += dZ1^T X~      (8: dW1', db1 in rows 0..63)
//             dX -> warp-aggregated red.global.add.v4.f32 into channel-last fp32 scratch grids (K4)
//   The three weight-gradient batches are DEFERRED: issued behind the delta-propagation MMAs of their stage but not waited
//   for — they run under the next epilogue / the scatter; the last one is awaited before the next tile overwrites X~.
//   D1, D2, D3 (fp32, TMEM) accumulate over ALL tiles of the CTA and are flushed once per launch with atomics.
//   Biases ride in K (a constant-1 feature); the 1/2 of GELU is folded into the next layer's weights; dz3 carries a
//   power-of-two loss scale S so that f16 deltas stay normal; S and the 2/(N*Cout) of the MSE mean are applied at the flush.
//   GELU is the tanh form in forward AND backward (the gradient of the function actually evaluated).
//   Noise: X~ = x + (U - 1/2) / 2^bits on all Cin columns (image_compression.py:248-251), Philox4x32-10 keyed by
//   (seed), counter (sample, block of 16 features, step); 8-bit uniforms, sixteen per Philox call.
// Algorithmic work: 3 * 2 * (Cin*64 + 64*64 + 64*Cout) = 53,760 FLOP/sample; tensor-bound roofline.
#include "nic_tc_common.cuh"

namespace nic {

constexpr int TT_ROWS = 128, TT_THREADS = 256;
constexpr int TT_H = 64, TT_K2 = 80;
constexpr int TT_SG80 = 10 * 128;          // sample-group stride of an 80-feature activation / delta buffer (bytes)
constexpr int TT_W2 = 64 * 80 * 2, TT_W3 = 16 * 80 * 2;
constexpr int TT_ACT = 16 * TT_SG80;       // 20480
constexpr int TT_SG16 = 2 * 128, TT_DZ3 = 16 * TT_SG16;       // dZ3: 16 output features per sample, sample-group stride 256 B
// Everything that depends on the decoder-input width.  2-D: Cin = 5C + 2 PE + 1 = 73 and 3-D "v2" (method 4): 79 both
// fit K1 = 80 (with the bias carrier) -> 106 KB smem, 240 TMEM columns, two CTAs per SM;  3-D method 3: Cin = 9C + 3 PE
// + 1 = 127 -> K1 = 128, dX is 108 columns wide (N = 128), 122 KB smem, 352 TMEM columns, one CTA per SM.
template <int METHOD> struct TrainShape {
  static constexpr int DIM = METHOD == NIC_METHOD_2D ? 2 : 3;
  static constexpr int NC0 = METHOD == NIC_METHOD_3D ? 8 : 4;      // G0 corners
  static constexpr int NC1 = DIM == 2 ? 4 : 8;                     // G1 corners
  static constexpr int CIN = 12 * (NC0 + 1) + 6 * DIM + 1;
  static constexpr int K1 = (CIN + 1 + 15) / 16 * 16;              // 80 / 128
  static constexpr int KG1 = K1 / 8, SGX = KG1 * 128, XBYTES = 16 * SGX, W1BYTES = 64 * K1 * 2;
  static constexpr int NDX = 12 * (NC0 + 1) <= 64 ? 64 : 128;      // N of the dX GEMM = width of the D accumulator
  static constexpr int C0 = METHOD == NIC_METHOD_3D ? 9 : 6;       // feature groups (of 8) gathered by warp-group 0
  static constexpr int XV = 8 * C0 > K1 - 8 * C0 ? 8 * C0 : K1 - 8 * C0;
  // One persistent CTA per SM runs NSLOT tiles at a time, each on its own 256 threads ("slot": own activation buffers, own D
  // accumulator, own mbarriers and named barrier); the weight images and the three weight-gradient accumulators D1, D2, D3
  // are shared by the slots.  K1 = 80: three slots (768 threads, <= 80 registers); K1 = 128: one.
  static constexpr int NSLOT = K1 == 80 ? 3 : 1;
  static constexpr int THREADS = NSLOT * TT_THREADS;
  static constexpr int COL_D = 0, COL_D1 = NSLOT * NDX, COL_D2 = COL_D1 + K1, COL_D3 = COL_D2 + 80;       // D3 (transposed): 16 columns
  static constexpr int COL_GD = COL_D3 + 16;           // NSLOT > 1: d h1'/d z1 of a tile parks here between forward and backward (32 columns per slot)
  static constexpr int TMEM = COL_GD + (NSLOT > 1 ? 32 * NSLOT : 0) <= 256 ? 256 : 512;
  static constexpr int WIMG = W1BYTES + TT_W2 + TT_W3;
  static constexpr int OFF_W1 = 0, OFF_W2 = W1BYTES, OFF_W3 = OFF_W2 + TT_W2, OFF_SLOT0 = OFF_W3 + TT_W3;
  // A slot: X~ | B1 | B2 | dZ3.   B1: H1, then the selector matrix S, then T (FS).  B2: H2, then dZ2, then dZ1 — each
  // overwrite waits for the deferred weight-gradient batch that still reads the previous content (D3, D2).
  // MN-major A operands with M = 128 read 16 feature groups per sample group from buffers that hold 10: groups 10..15
  // alias the start of the next sample group (accumulator rows 80..127, never read); for the last sample group that is 768
  // bytes past the buffer: B1's overrun lands in B2, B2's in dZ3 (4 KB).
  static constexpr int SOFF_X = 0, SOFF_B1 = XBYTES, SOFF_B2 = SOFF_B1 + TT_ACT, SOFF_DZ3 = SOFF_B2 + TT_ACT;
  static constexpr int SLOT_BYTES = SOFF_DZ3 + TT_DZ3;
  static constexpr int OFF_MISC = OFF_SLOT0 + NSLOT * SLOT_BYTES, OFF_PELUT = OFF_MISC + 128 * NSLOT + 64, SMEM = OFF_PELUT + 1024;
};
constexpr float TT_LOSS_SCALE = 64.0f;
// The quantisation dither takes 8 bits per feature from Philox4x32 with SEVEN rounds — the fewest that pass BigCrush (Salmon et
// al., SC'11; ten is the library default with its safety margin).  73 bytes per sample are five calls; at ten rounds the
// generator was 9 % of the kernel's instructions.  (The crop sampler keeps the ten-round generator of the known-answer test.)
constexpr int TT_NOISE_ROUNDS = 7;

// Instruction descriptor with explicit operand majors (bit 15: A is MN-major, bit 16: B is MN-major).
__host__ __device__ constexpr uint32_t tt_idesc(int fmt, int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// Training weight images (K-major B, no swizzle): element (n, k) at (k/8)*(NR/8)*128 + (n/8)*128 + (n%8)*16 + (k%8)*2.
//   W1' [64 x K1]: k < Cin: W1[n][k]; k = Cin: b1[n]; rest 0     (the LOD column is a real, noisy input in training)
//   W2' [64 x 80]: k < 64: W2[n][k]/2; k = 64: b2[n]
//   W3' [16 x 80]: n < cout: k < 64: W3[n][k]/2; k = 64: b3[n]
template <int FMT>
__device__ __forceinline__ void pack_train_weights_item(int i, const MlpDev& m, int K1, uint16_t* __restrict__ img) {
  const int n1 = 64 * K1, n2 = 64 * 80;
  {
    int which = i < n1 ? 0 : (i < n1 + n2 ? 1 : 2);
    int local = which == 0 ? i : (which == 1 ? i - n1 : i - n1 - n2);
    int nrows = which == 2 ? 16 : 64;
    int kc = local / (nrows * 8), rem = local - kc * nrows * 8;
    int n = rem / 8, k = kc * 8 + (rem - n * 8);
    float v = 0.f;
    if (which == 0) v = k < m.cin ? m.w1[n * m.cin + k] : (k == m.cin ? m.b1[n] : 0.f);
    else if (which == 1) v = k < 64 ? 0.5f * m.w2[n * 64 + k] : (k == 64 ? m.b2[n] : 0.f);
    else if (n < m.cout) v = k < 64 ? 0.5f * m.w3[n * 64 + k] : (k == 64 ? m.b3[n] : 0.f);
    img[i] = to16<FMT>(v);
  }
}

// dg[c][y][x] += scale * s[(x*ny + y)*C + c];  s <- 0   (channel-last fp32 scratch -> the caller's channel-major grid)
// Tile = 32 nodes along x  x  GR_TF along y, all channels: the scratch is read in runs of GR_TF * C contiguous floats, the
// gradient is written in 128-byte runs along x, every loop runs over the whole tile in parallel.
constexpr int GR_TF = 8;
__global__ void __launch_bounds__(256) grad_relayout_add_kernel(float* __restrict__ s, float* __restrict__ dg, int C, int nx,
                                                                int ny, float scale) {
  extern __shared__ float tile_f[];            // [GR_TF * C][33]
  const int x0 = blockIdx.x * 32, y0 = blockIdx.y * GR_TF;
  const int yw = ny - y0 < GR_TF ? ny - y0 : GR_TF, xw = nx - x0 < 32 ? nx - x0 : 32;
  const int run = yw * C;
  for (int i = threadIdx.x; i < xw * run; i += blockDim.x) {
    const int xi = i / run, e = i - xi * run;        // e = yi * C + c
    float* p = s + ((size_t)(x0 + xi) * ny + y0) * C + e;
    const float v = *p;
    tile_f[e * 33 + xi] = v;
    if (v != 0.f) *p = 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C * GR_TF * 32; i += blockDim.x) {
    const int c = i / (GR_TF * 32), r = i - c * (GR_TF * 32), yi = r >> 5, xi = r & 31;
    if (xi < xw && yi < yw) {
      const float v = tile_f[(yi * C + c) * 33 + xi];
      if (v != 0.f) dg[((size_t)c * ny + y0 + yi) * nx + x0 + xi] += scale * v;
    }
  }
}

// Small-grid variants (one thread per element): the tiled kernels above are bandwidth-shaped and take tens of
// microseconds of pure latency on a [12, 129, 129] grid, which is a third of a 0.36 ms training step.
__device__ __forceinline__ void grad_add_small_item(long long i, float* __restrict__ s, float* __restrict__ dg, int C, int nx, int ny,
                                                    int nz, float scale) {
  const float v = s[i];                              // s is [x][y][z][C]: i walks it linearly (coalesced read + zero)
  if (v == 0.f) return;
  const unsigned u = (unsigned)i, node = u / 12u, c = u - node * 12u;      // C == 12 on this path; < 2^32 elements (launcher)
  const unsigned nyz = node / (unsigned)nz, z = node - nyz * (unsigned)nz;
  const unsigned x = nyz / (unsigned)ny, y = nyz - x * (unsigned)ny;
  if (v != 0.f) {
    dg[(((size_t)c * nz + z) * ny + y) * nx + x] += scale * v;      // dg is [C][z][y][x]
    s[i] = 0.f;
  }
}
template <int FMT>
__device__ __forceinline__ void relayout_small_item(long long i, const float* __restrict__ g, uint16_t* __restrict__ sh, int C, int nx,
                                                    int ny, int nz) {
  const unsigned u = (unsigned)i, node = u / 12u, c = u - node * 12u;      // C == 12 on this path; < 2^32 elements (launcher)
  const unsigned nyz = node / (unsigned)nz, z = node - nyz * (unsigned)nz;
  const unsigned x = nyz / (unsigned)ny, y = nyz - x * (unsigned)ny;
  sh[i] = to16<FMT>(__ldg(g + (((size_t)c * nz + z) * ny + y) * nx + x));
}

// (h', g') for a pair: h' = 2 gelu_tanh(x) = x + x t,  g' = d h'/dx = (1 + t) + x (1 - t^2)(c1 + 3 c2 x^2),
// t = tanh(x (c1 + c2 x^2)).  Packed 16-bit math; the activation feeds the next MMA, the derivative stays in registers.
template <int FMT>
__device__ __forceinline__ void gelu2x_pair_grad(float a, float b, uint32_t& h_out, uint32_t& g_out) {
  using P = Pair<FMT>;
  typename P::T2 x = P::pack(a, b);
  typename P::T2 x2 = __hmul2(x, x);
  typename P::T2 p = __hfma2(x2, P::cst(0.0356774081f), P::cst(0.7978845608f));
  typename P::T2 t = P::tanh2(__hmul2(p, x));
  typename P::T2 h = __hfma2(x, t, x);
  typename P::T2 q = __hfma2(x2, P::cst(3.0f * 0.0356774081f), P::cst(0.7978845608f));
  typename P::T2 s = __hfma2(__hneg2(t), t, P::cst(1.0f));
  typename P::T2 gd = __hfma2(__hmul2(x, s), q, __hadd2(t, P::cst(1.0f)));
  h_out = *reinterpret_cast<uint32_t*>(&h);
  g_out = *reinterpret_cast<uint32_t*>(&gd);
}

template <int FMT>
__device__ __forceinline__ float2 unpack2(uint32_t v) {
  if (FMT == 0) return __half22float2(*reinterpret_cast<__half2*>(&v));
  return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v));
}

// hw = two f16 values 1024 + b (b = a uniform byte)  ->  ((b + 1/2) / 256 - 1/2) * amp for both, exactly, in packed f16:
// sc = amp / 256, hs = sc / 2.
__device__ __forceinline__ uint32_t noise_h2(uint32_t hw, __half2 sc, __half2 hs) {
  __half2 v = __hadd2(*reinterpret_cast<const __half2*>(&hw), __float2half2_rn(-1152.0f));
  v = __hfma2(v, sc, hs);
  return *reinterpret_cast<uint32_t*>(&v);
}


// Segmented warp reduction for the scatter: lanes whose `key` (grid node) is equal and contiguous are summed into the
// first lane of the run; runs are also cut every 2^steps lanes so that `steps` shuffle rounds always suffice.
// The run structure depends only on the grid (corner keys differ by lane-independent offsets), so it is computed once
// per grid (SegInfo) and reused by every corner and 4-channel part; the values travel as two f16x2 words (they carry
// the loss scale, so they are well inside f16 range, and dX itself comes from 16-bit MMA operands).
struct SegInfo {
  unsigned same;     // bit s: lane + 2^s belongs to the same run
  bool head;         // this lane issues the atomic
};
__device__ __forceinline__ SegInfo seg_info(int key, int steps, int lane) {
  const int prev = __shfl_up_sync(0xffffffffu, key, 1);
  const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || prev != key);
  const int start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
  const int L = 1 << steps, sub = (lane - start) & (L - 1);
  SegInfo si;
  si.same = 0u;
  si.head = sub == 0;
  for (int s = 0, d = 1; s < steps; ++s, d <<= 1) {
    const int kd = __shfl_down_sync(0xffffffffu, key, d);
    if (lane + d < 32 && kd == key && sub + d < L) si.same |= 1u << s;
  }
  return si;
}
struct TrainArgs {
  const uint2* s0;            // 16-bit channel-last shadow of G0: [x][y][12]
  const uint2* s1;            // ... of G1
  const long long* origins;   // [nblocks, 2]
  const uint4* wimg;          // packed W1' W2' W3'
  const float* targets;       // [N, cout]
  const float* noise;         // optional injected noise [N, cin]
  float* dgs0;                // channel-last fp32 gradient scratch of G0 (NULL: grids frozen)
  float* dgs1;
  float* loss_sum;
  float* out_save;
  MlpGradDev gm;
  float noise_amp;            // 2^-bits, 0 = no in-kernel noise
  unsigned long long seed, step;
  float flush_scale;          // 2 / (N_global * cout) / S
  int cout;
  int steps0, steps1;         // segmented-reduction depths of the scatter (lanes sharing a G0 / G1 node)
  float* partials;            // [gridDim.x][pstride]: this CTA's MLP-gradient sums (w1 | b1 | w2 | b2 | w3 | b3), plain stores
  int pstride;
  int dbg;                    // knock-out experiments (NIC_OPT_DEBUG_KNOCKOUT): bit 4 skips the grid-gradient REDs
  unsigned* tile_ctr;         // dynamic tile scheduler: next tile to hand out minus gridDim.x (zeroed by train_prep_kernel);
                              // NULL: static round-robin (NIC_OPT_STATIC_TILES: run-to-run identical decoder gradients)
  unsigned long long* prof;   // NULL, or 16 device counters: cycles per phase seen by thread 0 (nic_debug_counters)
};

// FS ("fast scatter", 2-D, step 1/4, interpolation on, crop rows of whole tiles): the grid-gradient reduction over the samples
// that share a node runs ON THE TENSOR CORE.  A tile is 128 consecutive texels of one image row, so its samples touch <= 33
// consecutive G0 node rows and <= 17 G1 node rows; with the selector matrix S [128 samples x 80 slots] (slot < 40: one-hot
// G0 node row of the sample; 40 + q / 58 + q: its G1 node row q weighted by (1 - ky) / ky)
//     T = S^T dZ1           (8 MMAs, reduction over the samples: S is an MN-major A operand exactly like the weight gradients)
//     U = T W1'             (4 MMAs: the dX GEMM applied to 80 slot rows instead of 128 sample rows)
// and U's rows leave as fp32 red.global.add.v4 — no dX epilogue, no shuffles, no 16-bit packing of the gradients.  S is
// written into the H1 buffer (dead once D2 has been accumulated), T (16 bit) into the DZ buffer.
template <int FMT, int METHOD, int FS = 0>
__global__ void __launch_bounds__(TrainShape<METHOD>::THREADS, 1) train_tc_kernel(DevGeom g, TrainArgs a) {
  static_assert(!FS || METHOD == NIC_METHOD_2D, "the tensor-core scatter covers the 2-D method");
  using P = Pair<FMT>;
  using TS = TrainShape<METHOD>;
  constexpr int DIM = TS::DIM, CIN = TS::CIN, NC0 = TS::NC0, NC1 = TS::NC1, K1 = TS::K1, SGX = TS::SGX, NDX = TS::NDX, C0 = TS::C0;
  constexpr int NSLOT = TS::NSLOT;
  constexpr bool GD_TMEM = NSLOT > 1;             // d h1'/d z1 parks in tensor memory instead of 16 registers
  constexpr int TT_COL_D1 = TS::COL_D1, TT_COL_D2 = TS::COL_D2, TT_COL_D3 = TS::COL_D3;
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp_cta = uniform_warp_index();      // provably uniform (MMA issue)
  const int slot = warp_cta >> 3, warp = warp_cta & 7;
  const int tid = threadIdx.x & (TT_THREADS - 1), lane = tid & 31;
  uint8_t* sSlot = smem + TS::OFF_SLOT0 + slot * TS::SLOT_BYTES;
  uint8_t* sX = sSlot + TS::SOFF_X;
  uint8_t* sH1 = sSlot + TS::SOFF_B1;             // B1: H1 | S | T
  uint8_t* sH2 = sSlot + TS::SOFF_B2;             // B2: H2 | dZ2 | dZ1
  uint8_t* sDZ3 = sSlot + TS::SOFF_DZ3;
  uint8_t* sMisc = smem + TS::OFF_MISC + 128 * slot;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sMisc);          // completion of the awaited batch of a stage
  uint64_t* mbar2 = mbar + 1;                     // completion of the LAST deferred batch of a tile (D1 += dZ1^T X~): X~, B2 free
  uint64_t* mbar3 = mbar + 2;                     // completion of D2 (B1 = H1 and B2 = dZ2 may be overwritten)
  uint64_t* mbar4 = mbar + 3;                     // completion of D3 (B2 = H2 may be overwritten)
  float* sRed = reinterpret_cast<float*>(sMisc + 32);           // [8] loss partials
  // [2] x {tile, px, py0, -}: the next tile (dynamic scheduler) and, FS, the image coordinates of its first texel — worked out
  // by thread 0 of the slot one tile ahead (the tile's 128 texels are consecutive in y), not by every thread
  volatile int* sInfo = reinterpret_cast<volatile int*>(sMisc + 64);
  const uint4* sPE = reinterpret_cast<const uint4*>(smem + TS::OFF_PELUT);      // FS: triangular encoding of p mod 64 (3 packed words)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + TS::OFF_MISC + 128 * NSLOT);
  // timeline (debug, bit 9 with bit 3): nanosecond stamps of CTA entry / first tile / flush / exit, min and max over the CTAs
  const bool tl = a.prof && (a.dbg & 512);
  auto gtime = [] {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
  };
  const unsigned long long tl_entry = tl ? gtime() : 0ull;
  const int wg = warp >> 2;                       // column half of the epilogues / row half of the gather
  const int row = tid & (TT_ROWS - 1);            // sample of the tile = TMEM lane
  const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
  // byte offset of this sample's 16-byte chunk inside a feature group, for the three buffer widths
  const int roff80 = (row >> 3) * TT_SG80 + (row & 7) * 16, roffx = (row >> 3) * SGX + (row & 7) * 16;
  const int roff16 = (row >> 3) * TT_SG16 + (row & 7) * 16;
  auto slot_sync = [&] {                          // barrier of the 256 threads of this slot
    if (NSLOT == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "n"(TT_THREADS) : "memory");
  };

  if (warp_cta == 0) tmem_alloc(tmem_slot, TS::TMEM);
  if (tid == 0) {
    mbar_init(mbar, 1);
    mbar_init(mbar2, 1);
    mbar_init(mbar3, 1);
    mbar_init(mbar4, 1);
  }
  {
    // zero the activation / delta buffers once (padding features must be finite), then the constant-1 bias features
    uint4* act = reinterpret_cast<uint4*>(smem + TS::OFF_SLOT0);
    for (int i = threadIdx.x; i < NSLOT * TS::SLOT_BYTES / 16; i += TS::THREADS) act[i] = make_uint4(0, 0, 0, 0);
    pdl_wait();                  // everything above overlaps the tail of train_prep_kernel; its outputs are read from here on
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = threadIdx.x; i < TS::WIMG / 16; i += TS::THREADS) dst[i] = __ldg(a.wimg + i);
  }
  __syncthreads();
  if (wg == 0) {
    auto one = P::pack(1.0f, 0.0f);
    const uint32_t o = *reinterpret_cast<uint32_t*>(&one);
    *reinterpret_cast<uint4*>(sH1 + roff80 + 8 * 128) = make_uint4(o, 0, 0, 0);     // feature 64 = 1
    *reinterpret_cast<uint4*>(sH2 + roff80 + 8 * 128) = make_uint4(o, 0, 0, 0);
  }
  // FS: first texel of a tile (b = crop, then x, then the tile's 128 y)
  auto tile_first_texel = [&](unsigned tl_, int& px, int& py0) {
    px = py0 = 0;
    if (tl_ < (unsigned)((g.N + TT_ROWS - 1) / TT_ROWS)) {
      const unsigned tpb = (unsigned)g.per_block >> 7, tpr = (unsigned)g.B[1] >> 7;
      const unsigned b = tl_ / tpb, r = tl_ - b * tpb, ix = r / tpr;
      px = (int)a.origins[2 * (size_t)b] + (int)ix;
      py0 = (int)a.origins[2 * (size_t)b + 1] + (int)((r - ix * tpr) << 7);
    }
  };
  // The scheduler runs on ONE otherwise idle thread per slot (thread 128: warp-group 1 has nothing to do while warp-group 0
  // evaluates the loss), two tiles ahead: during tile k it holds the index of tile k + 1, asks the counter for tile k + 2 and —
  // the two memory round trips overlap — looks up the first texel of tile k + 1.  (Fetching in thread 0 at the top of a tile
  // cost 1,500 cycles per tile: at 80 registers the compiler spills the returned index at once, i.e. waits for the atomic.)
  const unsigned tile_stride = gridDim.x * NSLOT;
  const unsigned ntiles = (unsigned)((g.N + TT_ROWS - 1) / TT_ROWS);
  volatile unsigned* sSched = reinterpret_cast<volatile unsigned*>(sMisc + 96);      // tile k + 1 (thread 128 only)
  if (tid == 128) sSched[0] = a.tile_ctr ? atomicAdd(a.tile_ctr, 1u) + tile_stride : blockIdx.x * NSLOT + slot + tile_stride;
  if (FS) {
    if (tid == 0) {
      int px, py0;
      const unsigned t0 = blockIdx.x * NSLOT + slot;
      tile_first_texel(t0, px, py0);
      sInfo[4] = (int)t0, sInfo[5] = px, sInfo[6] = py0;
    }
    if (threadIdx.x < 64 && g.pe_kind == NIC_PE_TRIANGULAR) {
      const float u1 = __fmul_rn(__fmul_rn((float)threadIdx.x, g.step), 0.5f);
      uint32_t w[3];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        auto v = P::pack(pe_triangular(u1, 2 * r, 6), pe_triangular(u1, 2 * r + 1, 6));
        w[r] = *reinterpret_cast<uint32_t*>(&v);
      }
      reinterpret_cast<uint4*>(smem + TS::OFF_PELUT)[threadIdx.x] = make_uint4(w[0], w[1], w[2], 0u);
    }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t TT_COL_D = (uint32_t)(slot * NDX);       // this slot's D accumulator
  if (slot == 0 && wg == 0) {
    // D1, D2, D3 are shared by the slots and accumulate from the first MMA on: clear them here
    uint32_t z[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) z[i] = 0u;
#pragma unroll
    for (int c = TT_COL_D1; c < TT_COL_D3 + 16; c += 16) tmem_st16(tmem + lane_base + c, z);
    tc_wait_st();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t aW1 = smem_u32(smem + TS::OFF_W1), aW2 = smem_u32(smem + TS::OFF_W2), aW3 = smem_u32(smem + TS::OFF_W3);
  const uint32_t aX = smem_u32(sX), aH1 = smem_u32(sH1), aH2 = smem_u32(sH2), aDZ3 = smem_u32(sDZ3);
  constexpr uint32_t ID_F64 = tt_idesc(FMT, 128, 64, 0, 0), ID_F16 = tt_idesc(FMT, 128, 16, 0, 0);
  constexpr uint32_t ID_B64 = tt_idesc(FMT, 128, 64, 0, 1);        // delta propagation: A K-major, B = W'^T (MN-major view)
  constexpr uint32_t ID_G16 = tt_idesc(FMT, 128, 16, 1, 1);        // D3^T = [H2|1]^T dZ3
  constexpr uint32_t ID_G80 = tt_idesc(FMT, 128, 80, 1, 1);        // weight gradients: both operands MN-major
  constexpr uint32_t ID_GX = tt_idesc(FMT, 128, K1, 1, 1);         // ... against the K1-wide input buffer
  constexpr uint32_t ID_BDX = tt_idesc(FMT, 128, NDX, 0, 1);       // dX = dZ1 W1' (N = NDX input columns)
  constexpr uint32_t WG64 = 8 * 128, WG16 = 2 * 128;               // k-group strides of the 64-row / 16-row weight images
  uint32_t phase = 0;
  float loss_local = 0.f, sse8_local = 0.f;
  unsigned tiles_done = 0;

  // phase profile (debug): thread 0 adds the cycles since its previous mark to counter `i`
  const bool prof0 = a.prof && threadIdx.x == 0;      // thread 0 of slot 0
  long long prof_t = a.prof ? clock64() : 0;
  const long long prof_start = prof_t;
  auto mark = [&](int i) {
    if (prof0 && !tl) {
      const long long t = clock64();
      atomicAdd(a.prof + i, (unsigned long long)(t - prof_t));
      prof_t = t;
    }
  };
  // hand the tensor core a batch of MMAs and wait for them
  // `issue` is waited for; `deferred` (the weight-gradient MMAs, which nothing in the next stage reads) is issued behind
  // it and runs under the next epilogue.  tcgen05.commit tracks ALL earlier MMAs of the issuing thread, so the next
  // stage's wait also covers this stage's deferred batch; the last one of a tile commits to mbar2 (`last`).
  auto run_mmas2 = [&](auto&& issue, auto&& deferred, bool last) {
    fence_async_smem();
    tc_fence_before();
    slot_sync();
    if (warp == 0) {               // uniform branch + elected lane: operands stay in uniform registers (nic_tc_common.cuh)
      if (elect_one()) {
        tc_fence_after();
        issue();
        tc_commit(mbar);
        deferred();
        if (last) tc_commit(mbar2);
      }
      __syncwarp();
    }
    mbar_wait(mbar, phase);
    phase ^= 1;
    tc_fence_after();
  };
  auto run_mmas = [&](auto&& issue) { run_mmas2(issue, [] {}, false); };
  // weight-gradient GEMM: Dacc[128 x 80] (+)= Abuf^T (features x samples) . Bbuf (samples x 80 features)
  auto issue_wgrad = [&](uint32_t dcol, uint32_t abuf, uint32_t bbuf, uint32_t sgb, uint32_t idesc) {
#pragma unroll
    for (int kc = 0; kc < 8; ++kc)
      mma_ss(tmem + dcol, make_smem_desc(abuf + kc * 2 * TT_SG80, TT_SG80, 128),
             make_smem_desc(bbuf + kc * 2 * sgb, sgb, 128), idesc, 1u);
  };
  uint32_t phase2 = 0, phase3 = 0, phase4 = 0;

  // FS: the last GEMM of a tile (U = T W1') is NOT awaited at the end of the tile — its rows are scattered after the NEXT
  // tile's gather, which hides that round trip; the geometry the scatter needs travels in these registers.
  bool u_pending = false;
  int u_x0 = 0, u_x1 = 0, u_base0 = 0, u_base1 = 0, u_nslot0 = 0, u_nslot1 = 0;
  float u_kx = 0.f;
  // rows of U -> the channel-last fp32 gradient scratch.  Row r < 40: G0 node row base0 + r, columns [12 j, +12) = corner
  // j = (dy, dx) -> node (x0 + dx, base0 + r + dy); rows 40 + q / 58 + q: G1 node row base1 + q (+ 1), columns [48, 60), times
  // wx(dx) for the two x nodes.  Warp-group 0 holds columns [0, 32), 1 holds [32, 64).
  auto fs_scatter_rows = [&] {
    mbar_wait(mbar, phase);
    phase ^= 1;
    tc_fence_after();
    uint32_t acc[32];
    tmem_ld32(tmem + TT_COL_D + lane_base + wg * 32, acc);
    tc_wait_ld();
    auto red4f = [](float* dst, float x0, float x1, float x2, float x3) {
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(x0), "f"(x1), "f"(x2), "f"(x3) : "memory");
    };
    if (!(a.dbg & 16)) {
      if (row < u_nslot0 && row < 40) {
#pragma unroll
        for (int gi = 0; gi < 8; ++gi) {
          const int col = 32 * wg + 4 * gi;
          if (col < 48) {
            const int j = col / 12, q = (col - 12 * j) >> 2, dy = j & 1, dx = j >> 1;
            float* dst = a.dgs0 + ((size_t)(u_x0 + dx) * g.n0[1] + (u_base0 + row + dy)) * 12 + 4 * q;
            red4f(dst, __uint_as_float(acc[4 * gi]), __uint_as_float(acc[4 * gi + 1]), __uint_as_float(acc[4 * gi + 2]),
                  __uint_as_float(acc[4 * gi + 3]));
          }
        }
      } else if (wg == 1 && row >= 40 && row < 76) {
        const int dy = row >= 58, q = row - 40 - 18 * dy;
        if (q < u_nslot1) {
#pragma unroll
          for (int dx = 0; dx < 2; ++dx) {
            const float wx = dx ? u_kx : __fsub_rn(1.0f, u_kx);
#pragma unroll
            for (int part = 0; part < 3; ++part) {
              float* dst = a.dgs1 + ((size_t)(u_x1 + dx) * g.n1[1] + (u_base1 + q + dy)) * 12 + 4 * part;
              red4f(dst, wx * __uint_as_float(acc[16 + 4 * part]), wx * __uint_as_float(acc[17 + 4 * part]),
                    wx * __uint_as_float(acc[18 + 4 * part]), wx * __uint_as_float(acc[19 + 4 * part]));
            }
          }
        }
      }
    }
    u_pending = false;
    tc_fence_before();          // the next MMAs into D are ordered after these tcgen05.ld by the barrier of run_mmas
  };

  if (tl && prof0) {
    const unsigned long long t = gtime();
    atomicMax(a.prof + 0, ~tl_entry);
    atomicMax(a.prof + 1, tl_entry);
    atomicMax(a.prof + 2, ~t);
    atomicMax(a.prof + 3, t);
  }
  // Tiles are handed out by an atomic counter: the CTAs of one launch finish their static share up to 20 % apart (13 or 14
  // tiles each at config 1, and the per-tile time varies from SM to SM), and the kernel ends with the slowest.  Thread 0
  // fetches the next index at the top of a tile; it reaches the others through shared memory, several barriers later.
  unsigned tile = blockIdx.x * NSLOT + slot;
  for (; tile < ntiles; ++tiles_done) {
    const unsigned n = tile * TT_ROWS + row;
    const bool live = FS ? true : n < (unsigned)g.N;           // FS: crop rows are whole tiles
    const unsigned nc = live ? n : (unsigned)g.N - 1;
    float tgt[4] = {0.f, 0.f, 0.f, 0.f};           // targets of the first 4 outputs: loaded now, used after the forward pass
    if (wg == 0 && live) {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < a.cout)       // volatile: keep the load HERE (the compiler would sink it to its use, 2,000 cycles later)
          asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(tgt[c]) : "l"(a.targets + (size_t)n * a.cout + c));
    }
    if (prof0 && tiles_done == 0) prof_t = clock64();      // later tiles: the gather phase starts at the end of the previous tile
    // ------------------------------------------------------------------------------------------ gather + noise -> X~
    Texel t;
    if constexpr (FS) {
      t.b = 0;
      t.p[0] = sInfo[4 * ((tiles_done & 1) ^ 1) + 1];
      t.p[1] = sInfo[4 * ((tiles_done & 1) ^ 1) + 2] + row;
      t.p[2] = 0;
    } else {
      t = texel_of_fast(g, nc, a.origins);
    }
    AxisCoord ax[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      ax[d] = axis_coord(d < DIM ? t.p[d] : 0, g.step);
      ax[d].i0 = clampi(ax[d].i0, 0, g.n0[d] - 2 < 0 ? 0 : g.n0[d] - 2);
      ax[d].i1 = clampi(ax[d].i1, 0, g.n1[d] - 2 < 0 ? 0 : g.n1[d] - 2);
    }
    // shadow node order: x slowest, then y, then z (2-D: x, y).  Linear index of corner (0,0,0) and the axis strides.
    const int sy0 = DIM == 2 ? 1 : g.n0[2], sx0 = g.n0[1] * sy0, sy1 = DIM == 2 ? 1 : g.n1[2], sx1 = g.n1[1] * sy1;
    const int node0 = ax[0].i0 * sx0 + ax[1].i0 * sy0 + (DIM == 3 ? ax[2].i0 : 0);
    const int node1 = ax[0].i1 * sx1 + ax[1].i1 * sy1 + (DIM == 3 ? ax[2].i1 : 0);
    // corner tables are (dz, dy, dx): offset of G0 corner j / G1 corner j from corner 0
    auto off0 = [&](int j) {
      const int8_t* d = DIM == 2 ? kCorner2D[j] : (METHOD == NIC_METHOD_3D ? kCorner3D[j] : kCorner3Dv2[j]);
      return d[2] * sx0 + d[1] * sy0 + (DIM == 3 ? d[0] : 0);
    };
    auto off1 = [&](int j) {
      const int8_t* d = DIM == 2 ? kCorner2D[j] : kCorner3D[j];
      return d[2] * sx1 + d[1] * sy1 + (DIM == 3 ? d[0] : 0);
    };
    auto w1 = [&](int j) {          // interpolation weight of G1 corner j (2-D bilinear; 3-D: the AS-CODED table)
      if (!g.interp) return 1.0f;
      float f[3];
      g1_factors(g, j, ax, f);
      return DIM == 2 ? f[0] * f[1] : f[0] * f[1] * f[2];
    };
    constexpr bool PACKED_ROW = FMT == 0 && METHOD == NIC_METHOD_2D;
    if constexpr (PACKED_ROW) {
      // f16, 2-D: the row is assembled as PACKED 16-bit words, never as fp32 values.  The G0 corners go from the shadow grid to
      // the operand buffer as loaded (one packed add for the noise, no conversions), G1 is interpolated with packed FMAs (the
      // result is rounded to f16 anyway), only the 12 encoding values are converted.  Same Philox counters and the same
      // feature <-> noise-byte mapping as the generic path below.
      auto ldg2 = [](const uint2* p) {
        uint2 v;
        asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
        return v;
      };
      auto as_h2 = [](uint32_t v) { return *reinterpret_cast<const __half2*>(&v); };
      auto bits2 = [](__half2 v) { return *reinterpret_cast<uint32_t*>(&v); };
      const bool gen = !a.noise && a.noise_amp > 0.f;
      const __half2 nsc = __float2half2_rn(a.noise_amp * (1.0f / 256.0f)), nhs = __float2half2_rn(a.noise_amp * (0.5f / 256.0f));
      auto noise16 = [&](int b16, uint32_t* nzw) {
        const uint4 r = philox4x32_r<TT_NOISE_ROUNDS>(a.seed, a.step, ((unsigned long long)nc << 4) | (unsigned)(8 * wg + b16));
        const uint32_t wds[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          nzw[2 * k] = noise_h2(__byte_perm(wds[k], 0x64646464u, 0x5140), nsc, nhs);
          nzw[2 * k + 1] = noise_h2(__byte_perm(wds[k], 0x64646464u, 0x5342), nsc, nhs);
        }
      };
      auto add_inj = [&](uint32_t w, float n0, float n1) {     // injected fp32 noise (parity tests)
        const float2 x = __half22float2(as_h2(w));
        return bits2(__floats2half2_rn(x.x + n0, x.y + n1));
      };
      auto wait_prev = [&] {          // the previous tile's deferred D1 += dZ1^T X~ still reads X~ (and the H2 buffer)
        if (tiles_done > 0) {
          mbar_wait_sleep(mbar2, phase2);
          phase2 ^= 1;
        }
      };
      if (wg == 0) {                  // features [0, 48): the four raw G0 corners
        uint32_t w[24];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            const uint2 v = ldg2(a.s0 + 3 * (size_t)(node0 + off0(j)) + q);
            w[6 * j + 2 * q] = v.x;
            w[6 * j + 2 * q + 1] = v.y;
          }
        if (a.noise) {
          const float* nz = a.noise + (size_t)nc * CIN;
#pragma unroll
          for (int i = 0; i < 24; ++i) w[i] = add_inj(w[i], nz[2 * i], nz[2 * i + 1]);
        } else if (gen) {
#pragma unroll
          for (int b16 = 0; b16 < 3; ++b16) {
            uint32_t nzw[8];
            noise16(b16, nzw);
#pragma unroll
            for (int i = 0; i < 8; ++i) w[8 * b16 + i] = bits2(__hadd2(as_h2(w[8 * b16 + i]), as_h2(nzw[i])));
          }
        }
        wait_prev();
#pragma unroll
        for (int c = 0; c < 6; ++c)
          *reinterpret_cast<uint4*>(sX + roffx + c * 128) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
      } else {                        // features [48, 80): G1 (12), PE (12), LOD, bias carrier, zero padding
        uint2 raw1[12];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int q = 0; q < 3; ++q) raw1[3 * j + q] = ldg2(a.s1 + 3 * (size_t)(node1 + off1(j)) + q);
        uint32_t w[16];
        {
          __half2 acc[6];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const __half2 wj = __float2half2_rn(w1(j));
#pragma unroll
            for (int q = 0; q < 3; ++q) {
              acc[2 * q] = j == 0 ? __hmul2(wj, as_h2(raw1[3 * j + q].x)) : __hfma2(wj, as_h2(raw1[3 * j + q].x), acc[2 * q]);
              acc[2 * q + 1] = j == 0 ? __hmul2(wj, as_h2(raw1[3 * j + q].y)) : __hfma2(wj, as_h2(raw1[3 * j + q].y), acc[2 * q + 1]);
            }
          }
#pragma unroll
          for (int i = 0; i < 6; ++i) w[i] = bits2(acc[i]);
        }
        if (FS && g.pe_kind == NIC_PE_TRIANGULAR) {        // step 1/4: the encoding has period 64 in the texel coordinate
          const uint4 lx = sPE[t.p[0] & 63], ly = sPE[t.p[1] & 63];
          w[6] = lx.x, w[7] = lx.y, w[8] = lx.z, w[9] = ly.x, w[10] = ly.y, w[11] = ly.z;
        } else if (g.pe_kind == NIC_PE_TRIANGULAR) {
#pragma unroll
          for (int d = 0; d < 2; ++d)
#pragma unroll
            for (int r = 0; r < 3; ++r)
              w[6 + 3 * d + r] = bits2(__floats2half2_rn(pe_triangular(ax[d].u1, 2 * r, 6), pe_triangular(ax[d].u1, 2 * r + 1, 6)));
        } else {
#pragma unroll 1
          for (int d = 0; d < 2; ++d) {
#pragma unroll 1
            for (int h = 0; h < 3; ++h) {
              float sv, cv;
              sincosf(__fmul_rn(ax[d].u1, g.pe_div[h]), &sv, &cv);
              const uint32_t pv = bits2(__floats2half2_rn(sv, cv));
#pragma unroll
              for (int i = 0; i < 6; ++i)
                if (i == 3 * d + h) w[6 + i] = pv;
            }
          }
        }
        float lodv = g.lod;
        if (a.noise) {
          const float* nz = a.noise + (size_t)nc * CIN + 48;
#pragma unroll
          for (int i = 0; i < 12; ++i) w[i] = add_inj(w[i], nz[2 * i], nz[2 * i + 1]);
          lodv += nz[24];
          w[12] = bits2(__floats2half2_rn(lodv, 1.0f));          // (LOD, bias carrier: not an input, no noise)
        } else {
          w[12] = bits2(__floats2half2_rn(lodv, 1.0f));
          if (gen) {
            uint32_t nzw[8];
            noise16(0, nzw);
#pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = bits2(__hadd2(as_h2(w[i]), as_h2(nzw[i])));
            noise16(1, nzw);
#pragma unroll
            for (int i = 0; i < 4; ++i) w[8 + i] = bits2(__hadd2(as_h2(w[8 + i]), as_h2(nzw[i])));
            w[12] = bits2(__hadd2(as_h2(w[12]), as_h2(nzw[4] & 0x0000FFFFu)));      // no noise beyond the real input columns
          }
        }
        w[13] = w[14] = w[15] = 0u;
        wait_prev();
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<uint4*>(sX + roffx + (6 + c) * 128) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
      }
    } else {
    constexpr int NCW0 = 8 * C0 / 12;          // G0 corners gathered by warp-group 0 (4 / 6); the rest go to warp-group 1
    constexpr int R0 = 12 * (NC0 - NCW0);      // ... which therefore starts with R0 raw G0 features (0 / 24)
    {
      float xv[TS::XV];        // this thread's part of the row: wg 0 -> features [0, 8 C0), wg 1 -> features [8 C0, K1)
      // All grid loads of this thread are issued FIRST (volatile: the compiler keeps them here instead of sinking each
      // next to its use, which serialised four ~800-cycle L2 round trips per tile); the arithmetic follows.
      auto ldg2 = [](const uint2* p) {
        uint2 v;
        asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
        return v;
      };
      auto unpack_corner = [&](const uint2* raw, float* dst) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          float2 lo = unpack2<FMT>(raw[q].x), hi = unpack2<FMT>(raw[q].y);
          dst[4 * q] = lo.x;
          dst[4 * q + 1] = lo.y;
          dst[4 * q + 2] = hi.x;
          dst[4 * q + 3] = hi.y;
        }
      };
      if (wg == 0) {
        uint2 raw[3 * NCW0];
#pragma unroll
        for (int j = 0; j < NCW0; ++j)
#pragma unroll
          for (int q = 0; q < 3; ++q) raw[3 * j + q] = ldg2(a.s0 + 3 * (size_t)(node0 + off0(j)) + q);
#pragma unroll
        for (int j = 0; j < NCW0; ++j) unpack_corner(raw + 3 * j, xv + 12 * j);
      } else {
        uint2 raw0[3 * (NC0 - NCW0) + 1], raw1[3 * NC1];
#pragma unroll
        for (int j = NCW0; j < NC0; ++j)
#pragma unroll
          for (int q = 0; q < 3; ++q) raw0[3 * (j - NCW0) + q] = ldg2(a.s0 + 3 * (size_t)(node0 + off0(j)) + q);
#pragma unroll
        for (int j = 0; j < NC1; ++j)
#pragma unroll
          for (int q = 0; q < 3; ++q) raw1[3 * j + q] = ldg2(a.s1 + 3 * (size_t)(node1 + off1(j)) + q);
#pragma unroll
        for (int j = NCW0; j < NC0; ++j) unpack_corner(raw0 + 3 * (j - NCW0), xv + 12 * (j - NCW0));
#pragma unroll
        for (int j = 0; j < NC1; ++j) {
          const float w = w1(j);
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            float2 lo = unpack2<FMT>(raw1[3 * j + q].x), hi = unpack2<FMT>(raw1[3 * j + q].y);
            xv[R0 + 4 * q] = j == 0 ? w * lo.x : fmaf(w, lo.x, xv[R0 + 4 * q]);
            xv[R0 + 4 * q + 1] = j == 0 ? w * lo.y : fmaf(w, lo.y, xv[R0 + 4 * q + 1]);
            xv[R0 + 4 * q + 2] = j == 0 ? w * hi.x : fmaf(w, hi.x, xv[R0 + 4 * q + 2]);
            xv[R0 + 4 * q + 3] = j == 0 ? w * hi.y : fmaf(w, hi.y, xv[R0 + 4 * q + 3]);
          }
        }
        // ONE branch on the encoding kind (pe_value per element interleaves twelve copies of the sin/cos slow path with
        // the code that actually runs: 112 KB of SASS and instruction-cache misses every tile)
        if (g.pe_kind == NIC_PE_TRIANGULAR) {
#pragma unroll
          for (int d = 0; d < DIM; ++d)
#pragma unroll
            for (int r = 0; r < 6; ++r) xv[R0 + 12 + 6 * d + r] = pe_triangular(ax[d].u1, r, 6);
        } else {
#pragma unroll 1
          for (int d = 0; d < DIM; ++d) {
#pragma unroll 1
            for (int h = 0; h < 3; ++h) {
              float sv, cv;
              sincosf(__fmul_rn(ax[d].u1, g.pe_div[h]), &sv, &cv);
#pragma unroll
              for (int dd = 0; dd < DIM; ++dd)
#pragma unroll
                for (int hh = 0; hh < 3; ++hh)
                  if (dd == d && hh == h) {
                    xv[R0 + 12 + 6 * dd + 2 * hh] = sv;
                    xv[R0 + 12 + 6 * dd + 2 * hh + 1] = cv;
                  }
            }
          }
        }
        xv[R0 + 12 + 6 * DIM] = g.lod;
#pragma unroll
        for (int i = R0 + 13 + 6 * DIM; i < K1 - 8 * C0; ++i) xv[i] = 0.f;
      }
      const int col0 = wg == 0 ? 0 : 8 * C0, ncols = wg == 0 ? 8 * C0 : CIN - 8 * C0;     // real (noisy) columns of this part
      if (a.noise) {
        const float* nz = a.noise + (size_t)nc * CIN + col0;
#pragma unroll
        for (int i = 0; i < TS::XV; ++i)
          if (i < ncols) xv[i] += nz[i];
      }
      if (wg == 1) xv[CIN - 8 * C0] = 1.0f;          // feature CIN: the bias carrier (not an input: no noise)
      // Pack to 16-byte chunks of 8 features -> X~ buffer, adding the in-kernel noise on the way: one Philox call
      // yields 16 bytes = the 8-bit uniforms of 16 features (two chunks).  (b - 127.5) * amp / 256 is built in packed
      // f16 (0x6400 | b = 1024 + b exactly) — 8 bits are far below what a 16-bit X~ resolves.
      if (tiles_done > 0) {          // the previous tile's deferred D1 += dZ1^T X~ still reads X~ (and the H2 buffer)
        mbar_wait_sleep(mbar2, phase2);
        phase2 ^= 1;
      }
      const bool gen = !a.noise && a.noise_amp > 0.f;
      const __half2 nsc = __float2half2_rn(a.noise_amp * (1.0f / 256.0f)), nhs = __float2half2_rn(a.noise_amp * (0.5f / 256.0f));
      const int fg0 = wg == 0 ? 0 : C0, nfg = wg == 0 ? C0 : TS::KG1 - C0;
#pragma unroll
      for (int b16 = 0; b16 < (TS::XV + 15) / 16; ++b16) {
        uint32_t nzw[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) nzw[i] = 0u;
        if (gen && 16 * b16 < ncols) {
          const uint4 r = philox4x32_r<TT_NOISE_ROUNDS>(a.seed, a.step, ((unsigned long long)nc << 4) | (unsigned)(8 * wg + b16));
          const uint32_t wds[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            nzw[2 * k] = noise_h2(__byte_perm(wds[k], 0x64646464u, 0x5140), nsc, nhs);
            nzw[2 * k + 1] = noise_h2(__byte_perm(wds[k], 0x64646464u, 0x5342), nsc, nhs);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {          // no noise beyond the real input columns
            if (16 * b16 + 2 * i >= ncols) nzw[i] = 0u;
            else if (16 * b16 + 2 * i + 1 >= ncols) nzw[i] &= 0x0000FFFFu;
          }
        }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int f = 2 * b16 + hh;
          if (f < TS::XV / 8 && f < nfg) {
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (FMT == 0) {
                __half2 v = __hadd2(__floats2half2_rn(xv[8 * f + 2 * i], xv[8 * f + 2 * i + 1]),
                                    *reinterpret_cast<const __half2*>(&nzw[4 * hh + i]));
                w[i] = *reinterpret_cast<uint32_t*>(&v);
              } else {
                const float2 z = __half22float2(*reinterpret_cast<const __half2*>(&nzw[4 * hh + i]));
                auto v = P::pack(xv[8 * f + 2 * i] + z.x, xv[8 * f + 2 * i + 1] + z.y);
                w[i] = *reinterpret_cast<uint32_t*>(&v);
              }
            }
            *reinterpret_cast<uint4*>(sX + roffx + (fg0 + f) * 128) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
    }
    }
    if (FS && u_pending) fs_scatter_rows();     // the previous tile's gradient rows (its last GEMM ran under this gather)
    mark(0);
    // ------------------------------------------------------------------------------------------ forward
    // d h'/d z of this thread's 32 hidden columns, layers 1 and 2.  The two layer loops below are FULLY unrolled: with a
    // rolled loop (layer a run-time value) nvcc 12.9 mis-compiled the conditional writes into these register arrays.
    uint32_t gd1[16], gd2[16];
    run_mmas([&] {
#pragma unroll
      for (int kc = 0; kc < K1 / 16; ++kc)
        mma_ss(tmem + TT_COL_D, make_smem_desc(aX + kc * 256, 128, SGX), make_smem_desc(aW1 + kc * 2 * WG64, WG64, 128),
               ID_F64, kc > 0);
    });
    mark(1);
#pragma unroll
    for (int layer = 0; layer < 2; ++layer) {
      uint32_t acc[32];
      tmem_ld32(tmem + TT_COL_D + lane_base + wg * 32, acc);
      tc_wait_ld();
      uint8_t* dstb = (layer == 0 ? sH1 : sH2) + roff80 + wg * 4 * 128;
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        uint32_t hp[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t gg;
          gelu2x_pair_grad<FMT>(__uint_as_float(acc[8 * f + 2 * i]), __uint_as_float(acc[8 * f + 2 * i + 1]), hp[i], gg);
          if (layer == 0) gd1[4 * f + i] = gg;
          else gd2[4 * f + i] = gg;
        }
        *reinterpret_cast<uint4*>(dstb + f * 128) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
      }
      if (FS && layer == 0 && a.dgs0) {      // the previous tile's selector matrix overwrote H1's bias carrier / padding
        auto one = P::pack(1.0f, 0.0f);
        *reinterpret_cast<uint4*>(sH1 + roff80 + (8 + wg) * 128) = make_uint4(wg == 0 ? *reinterpret_cast<uint32_t*>(&one) : 0u, 0, 0, 0);
      }
      if (GD_TMEM && layer == 0) {           // park d h1'/d z1 in tensor memory until the backward pass
        tmem_st16(tmem + TS::COL_GD + slot * 32 + wg * 16 + lane_base, gd1);
        tc_wait_st();
      }
      mark(layer == 0 ? 2 : 4);
      if (layer == 0) {
        run_mmas([&] {
#pragma unroll
          for (int kc = 0; kc < TT_K2 / 16; ++kc)
            mma_ss(tmem + TT_COL_D, make_smem_desc(aH1 + kc * 256, 128, TT_SG80),
                   make_smem_desc(aW2 + kc * 2 * WG64, WG64, 128), ID_F64, kc > 0);
        });
      } else {
        run_mmas([&] {
#pragma unroll
          for (int kc = 0; kc < TT_K2 / 16; ++kc)
            mma_ss(tmem + TT_COL_D, make_smem_desc(aH2 + kc * 256, 128, TT_SG80),
                   make_smem_desc(aW3 + kc * 2 * WG16, WG16, 128), ID_F16, kc > 0);
        });
      }
      mark(layer == 0 ? 3 : 5);
    }
    // ------------------------------------------------------------------------------------------ output, loss, dz3
    if (wg == 0) {
      uint32_t acc[16];
      tmem_ld16(tmem + TT_COL_D + lane_base, acc);
      tc_wait_ld();
      float dz[16];
      const bool save = a.out_save != nullptr;
#pragma unroll
      for (int c = 0; c < 4; ++c) {                  // branch-free for the usual 3 outputs (targets were prefetched)
        const bool on = live && c < a.cout;
        const float o = __fdividef(1.0f, 1.0f + __expf(-__uint_as_float(acc[c])));
        const float d = o - tgt[c];
        loss_local += on ? d * d : 0.f;
        if (g.metrics) {            // squared error of the 8-bit outputs (per-step PSNR, image_compression.py:260-261)
          const float d8 = quant_round(o, 255.0f) - quant_round(tgt[c], 255.0f);
          sse8_local += on ? d8 * d8 : 0.f;
        }
        if (on && save) a.out_save[(size_t)n * a.cout + c] = o;
        dz[c] = on ? TT_LOSS_SCALE * d * o * (1.0f - o) : 0.f;
      }
#pragma unroll
      for (int c = 4; c < 16; ++c) dz[c] = 0.f;
      if (a.cout > 4 && live) {
#pragma unroll
        for (int c = 4; c < 16; ++c) {
          if (c < a.cout) {
            const float o = __fdividef(1.0f, 1.0f + __expf(-__uint_as_float(acc[c])));
            const float tv = a.targets[(size_t)n * a.cout + c];
            const float d = o - tv;
            loss_local += d * d;
            if (g.metrics) {
              const float d8 = quant_round(o, 255.0f) - quant_round(tv, 255.0f);
              sse8_local += d8 * d8;
            }
            if (save) a.out_save[(size_t)n * a.cout + c] = o;
            dz[c] = TT_LOSS_SCALE * d * o * (1.0f - o);
          }
        }
      }
#pragma unroll
      for (int f = 0; f < 2; ++f) {
        auto p0 = P::pack(dz[8 * f], dz[8 * f + 1]), p1 = P::pack(dz[8 * f + 2], dz[8 * f + 3]);
        auto p2 = P::pack(dz[8 * f + 4], dz[8 * f + 5]), p3 = P::pack(dz[8 * f + 6], dz[8 * f + 7]);
        *reinterpret_cast<uint4*>(sDZ3 + roff16 + f * 128) =
            make_uint4(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1), *reinterpret_cast<uint32_t*>(&p2),
                       *reinterpret_cast<uint32_t*>(&p3));
      }
    } else if (tid == 128) {         // the tile scheduler (see the prologue)
      // tile k + 1 and its crop origin, and the request for tile k + 2: the origin load is issued BEFORE the atomic and nothing
      // uses either result until both are in flight, so the two round trips overlap inside the loss phase; the atomic's result
      // goes straight to shared memory.  (Requesting earlier — before the layer-3 wait — and posting here was slower: a result
      // that has to survive a long wait in a register is spilled at once, i.e. awaited at the point of issue.)
      const unsigned t1 = sSched[0];
      long long ox = 0, oy = 0;
      unsigned ix = 0, iy0 = 0;
      if (FS && t1 < ntiles) {
        const unsigned tpb = (unsigned)g.per_block >> 7, tpr = (unsigned)g.B[1] >> 7;
        const unsigned b = t1 / tpb, r = t1 - b * tpb;
        ix = r / tpr;
        iy0 = (r - ix * tpr) << 7;
        asm volatile("ld.global.nc.v2.s64 {%0, %1}, [%2];" : "=l"(ox), "=l"(oy) : "l"(a.origins + 2 * (size_t)b));
      }
      const unsigned t2 = a.tile_ctr ? atomicAdd(a.tile_ctr, 1u) + tile_stride : t1 + tile_stride;
      volatile int* d = sInfo + 4 * (tiles_done & 1);
      d[0] = (int)t1, d[1] = (int)ox + (int)ix, d[2] = (int)oy + (int)iy0;
      sSched[0] = t2;
    }
    mark(6);
    // ------------------------------------------------------------------------------------------ backward
    // dH2 = dZ3 W3' (K = 16 output features) and D3^T += [H2 | 1]^T dZ3.
    run_mmas2([&] { mma_ss(tmem + TT_COL_D, make_smem_desc(aDZ3, 128, TT_SG16), make_smem_desc(aW3, 128, WG16), ID_B64, 0); },
              [&] {
                // D3^T [H2 feature x output c] += [H2|1]^T (MN-major A, M = 128 aliased) . dZ3 (MN-major B, N = 16)
#pragma unroll
                for (int kc = 0; kc < 8; ++kc)
                  mma_ss(tmem + TT_COL_D3, make_smem_desc(aH2 + kc * 2 * TT_SG80, TT_SG80, 128),
                         make_smem_desc(aDZ3 + kc * 2 * TT_SG16, TT_SG16, 128), ID_G16, 1u);
                tc_commit(mbar4);      // D3 has read H2: dZ2 may overwrite it
              },
              false);
    mark(7);
#pragma unroll
    for (int layer = 1; layer >= 0; --layer) {
      uint32_t acc[32];
      tmem_ld32(tmem + TT_COL_D + lane_base + wg * 32, acc);
      tc_wait_ld();
      // dZ2, then dZ1 -> B2, features [0, 64) (H2 / dZ2 are dead once D3 / D2 have been accumulated: awaited HERE, after the
      // arithmetic).  B2's constant-1 feature 64 is left alone.
      uint8_t* dstb = sH2 + roff80 + (wg * 4) * 128;
      uint32_t gdl[16];
      if (layer == 0 && GD_TMEM) {
        tmem_ld16(tmem + TS::COL_GD + slot * 32 + wg * 16 + lane_base, gdl);
        tc_wait_ld();
      }
      uint32_t dp[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        // dZ = dH * g' in packed 16-bit math (the product is rounded to 16 bits for the next MMA anyway; dH carries the loss scale)
        const uint32_t ggw = layer == 1 ? gd2[i] : (GD_TMEM ? gdl[i] : gd1[i]);
        auto v = __hmul2(P::pack(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1])), *reinterpret_cast<const typename P::T2*>(&ggw));
        dp[i] = *reinterpret_cast<uint32_t*>(&v);
      }
      if (layer == 1) {
        mbar_wait(mbar4, phase4);
        phase4 ^= 1;
      } else {
        mbar_wait(mbar3, phase3);
        phase3 ^= 1;
      }
      tc_fence_after();
#pragma unroll
      for (int f = 0; f < 4; ++f) *reinterpret_cast<uint4*>(dstb + f * 128) = make_uint4(dp[4 * f], dp[4 * f + 1], dp[4 * f + 2], dp[4 * f + 3]);
      mark(layer == 1 ? 8 : 10);
      const bool fs = FS && a.dgs0;
      if (layer == 1) {
        auto issue_dh1 = [&] {
#pragma unroll
          for (int kc = 0; kc < 4; ++kc)
            mma_ss(tmem + TT_COL_D, make_smem_desc(aH2 + 2 * kc * 128, 128, TT_SG80),
                   make_smem_desc(aW2 + kc * 256, 128, WG64), ID_B64, kc > 0);
        };
        // dH1 = dZ2 W2'  and (deferred)  D2 += dZ2^T [H1 | 1]   (rows 0..63 = hidden units).  dZ1 will overwrite dZ2 (and the
        // selector matrix H1), so D2 signals its own mbarrier, awaited in the dZ1 epilogue
        run_mmas2(issue_dh1,
                  [&] {
                    issue_wgrad(TT_COL_D2, aH2, aH1, TT_SG80, ID_G80);
                    tc_commit(mbar3);
                  },
                  false);
      } else if (!fs) {
        run_mmas2(      // dX = dZ1 W1' (grid columns only)  and (deferred)  D1 += dZ1^T X~   (rows 0..63 = hidden units)
            [&] {
              if (a.dgs0) {
#pragma unroll
                for (int kc = 0; kc < 4; ++kc)
                  mma_ss(tmem + TT_COL_D, make_smem_desc(aH2 + 2 * kc * 128, 128, TT_SG80),
                         make_smem_desc(aW1 + kc * 256, 128, WG64), ID_BDX, kc > 0);
              }
            },
            [&] { issue_wgrad(TT_COL_D1, aH2, aX, SGX, ID_GX); }, true);
      }
      mark(layer == 1 ? 9 : 11);
    }
    // ------------------------------------------------------------------------------------------ grid-gradient scatter
    if (FS && a.dgs0) {
      // ---- selector matrix S -> H1 buffer.  This thread: sample `row`; warp-group 0 writes slots [0, 40), 1 writes [40, 80).
      const AxisCoord ayf = axis_coord(t.p[1] - row, g.step);       // first sample of the tile (same image row)
      const int base0 = clampi(ayf.i0, 0, g.n0[1] - 2 < 0 ? 0 : g.n0[1] - 2);
      const int base1 = clampi(ayf.i1, 0, g.n1[1] - 2 < 0 ? 0 : g.n1[1] - 2);
      {
        auto h16 = [](float v) -> uint32_t {
          auto p2 = P::pack(v, 0.0f);
          return *reinterpret_cast<uint32_t*>(&p2) & 0xFFFFu;
        };
        // (slot, value) pairs of this thread's half of the row; a slot outside [0, 40) never matches (invalid origins)
        int sa, sb;
        uint32_t va, vb;
        if (wg == 0) {
          sa = clampi(ax[1].i0 - base0, 0, 39);
          va = h16(1.0f);
          sb = -1;
          vb = 0u;
        } else {
          const int q = clampi(ax[1].i1 - base1, 0, 17);
          sa = q;                                                  // slots 40 + q: weight 1 - ky (corner dy = 0)
          va = h16(__fsub_rn(1.0f, ax[1].k));
          sb = 18 + q;                                             // slots 58 + q: weight ky (corner dy = 1)
          vb = h16(ax[1].k);
        }
        if (!live) va = vb = 0u;
        // (D2 += dZ2^T [H1 | 1] has read H1: awaited in the dZ1 epilogue)
        // one or two non-zero 16-bit entries in this thread's 80 bytes: five zero chunks, then the entries as 4-byte words on top
        // (same thread, same addresses: program order)
        uint8_t* srow = sH1 + roff80 + 5 * wg * 128;
#pragma unroll
        for (int c = 0; c < 5; ++c) *reinterpret_cast<uint4*>(srow + c * 128) = make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint32_t*>(srow + (sa >> 3) * 128 + ((sa >> 1) & 3) * 4) = va << ((sa & 1) * 16);
        if (sb >= 0) *reinterpret_cast<uint32_t*>(srow + (sb >> 3) * 128 + ((sb >> 1) & 3) * 4) = vb << ((sb & 1) * 16);
      }
      // ---- T = S^T dZ1 (awaited)  and (deferred)  D1 += dZ1^T X~
      run_mmas2(
          [&] {
#pragma unroll
            for (int kc = 0; kc < 8; ++kc)
              mma_ss(tmem + TT_COL_D, make_smem_desc(aH1 + kc * 2 * TT_SG80, TT_SG80, 128),
                     make_smem_desc(aH2 + kc * 2 * TT_SG80, TT_SG80, 128), tt_idesc(FMT, 128, 64, 1, 1), kc > 0);
          },
          [&] { issue_wgrad(TT_COL_D1, aH2, aX, SGX, ID_GX); }, true);
      mark(11);
      // ---- T (rows = slots) -> 16 bit, K-major A operand in B1 (the selector matrix is dead: T = S^T dZ1 is complete)
      {
        uint32_t acc[32];
        tmem_ld32(tmem + TT_COL_D + lane_base + wg * 32, acc);
        tc_wait_ld();
        if (row < 80) {
#pragma unroll
          for (int f = 0; f < 4; ++f) {
            uint32_t tp[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              auto v = P::pack(__uint_as_float(acc[8 * f + 2 * i]), __uint_as_float(acc[8 * f + 2 * i + 1]));
              tp[i] = *reinterpret_cast<uint32_t*>(&v);
            }
            *reinterpret_cast<uint4*>(sH1 + roff80 + (wg * 4 + f) * 128) = make_uint4(tp[0], tp[1], tp[2], tp[3]);
          }
        }
      }
      // ---- U = T W1'  (the dX GEMM on slot rows): issued, NOT awaited (fs_scatter_rows after the next tile's gather)
      fence_async_smem();
      tc_fence_before();
      slot_sync();
      if (warp == 0) {
        if (elect_one()) {
          tc_fence_after();
#pragma unroll
          for (int kc = 0; kc < 4; ++kc)
            mma_ss(tmem + TT_COL_D, make_smem_desc(aH1 + 2 * kc * 128, 128, TT_SG80), make_smem_desc(aW1 + kc * 256, 128, WG64),
                   ID_BDX, kc > 0);
          tc_commit(mbar);
        }
        __syncwarp();
      }
      u_pending = true;
      u_x0 = ax[0].i0;
      u_x1 = ax[0].i1;
      u_base0 = base0;
      u_base1 = base1;
      u_kx = ax[0].k;
      u_nslot0 = clampi(axis_coord(t.p[1] - row + TT_ROWS - 1, g.step).i0, 0, g.n0[1] - 2 < 0 ? 0 : g.n0[1] - 2) - base0 + 1;
      u_nslot1 = clampi(axis_coord(t.p[1] - row + TT_ROWS - 1, g.step).i1, 0, g.n1[1] - 2 < 0 ? 0 : g.n1[1] - 2) - base1 + 1;
    } else if (a.dgs0) {
      constexpr int HW = NDX / 2;                     // dX columns read by each warp-group: [HW wg, HW wg + HW)
      uint32_t acc[HW];
#pragma unroll
      for (int c = 0; c < HW; c += 32) tmem_ld32(tmem + TT_COL_D + lane_base + wg * HW + c, acc + c);
      uint32_t accg1[16];                             // dX columns [12 NC0, +12): the G1 block, read by BOTH warp-groups
      tmem_ld16(tmem + TT_COL_D + lane_base + 12 * NC0, accg1);
      tc_wait_ld();
      // The run structure (which lanes share a node) is the same for every corner of a grid: corner keys differ from
      // node0 / node1 by a lane-independent offset.  All groups of a grid are reduced TOGETHER, one shuffle round at a
      // time, so that the 2 x groups independent shuffles of a round are in flight at once (reducing group after group
      // serialises ~30-cycle shuffle latencies: 9,200 of the 25,000 cycles of a tile in the first version).
      const SegInfo si0 = seg_info(node0, a.steps0, lane), si1 = seg_info(node1, a.steps1, lane);
      auto pack_h2 = [](uint32_t x, uint32_t y) {
        __half2 h = __floats2half2_rn(__uint_as_float(x), __uint_as_float(y));
        return *reinterpret_cast<uint32_t*>(&h);
      };
      auto red4 = [](float* dst, uint32_t lo, uint32_t hi) {
        const float2 fa = __half22float2(*reinterpret_cast<const __half2*>(&lo)), fb = __half22float2(*reinterpret_cast<const __half2*>(&hi));
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(fa.x), "f"(fa.y), "f"(fb.x), "f"(fb.y) : "memory");
      };
      // ---- G0: v4 group gi of this thread covers dX columns [HW wg + 4 gi, +4); group gq = (corner gq / 3, part gq % 3)
      constexpr int NG0 = HW / 4;
      const int ng0 = 3 * NC0 - NG0 * wg < NG0 ? 3 * NC0 - NG0 * wg : NG0;      // groups of this warp-group that exist
      uint32_t pk[2 * NG0];
#pragma unroll
      for (int gi = 0; gi < NG0; ++gi) {
        pk[2 * gi] = pack_h2(acc[4 * gi], acc[4 * gi + 1]);
        pk[2 * gi + 1] = pack_h2(acc[4 * gi + 2], acc[4 * gi + 3]);
      }
#pragma unroll
      for (int s = 0; s < 5; ++s) {
        if (s < a.steps0) {
          uint32_t o[2 * NG0];
#pragma unroll
          for (int i = 0; i < 2 * NG0; ++i)
            if (i < 2 * ng0) o[i] = __shfl_down_sync(0xffffffffu, pk[i], 1 << s);
          const uint32_t m = (si0.same >> s) & 1u ? 0xffffffffu : 0u;      // + 0 where the partner is another node
#pragma unroll
          for (int i = 0; i < 2 * NG0; ++i)
            if (i < 2 * ng0) {
              const uint32_t om = o[i] & m;
              __half2 r = __hadd2(*reinterpret_cast<const __half2*>(&pk[i]), *reinterpret_cast<const __half2*>(&om));
              pk[i] = *reinterpret_cast<uint32_t*>(&r);
            }
        }
      }
      if (live && si0.head && !(a.dbg & 16)) {
#pragma unroll
        for (int gi = 0; gi < NG0; ++gi) {
          const int gq = NG0 * wg + gi;
          if (gi < ng0) {
            const int j = gq / 3, q = gq - 3 * j;
            red4(a.dgs0 + (size_t)(node0 + off0(j)) * 12 + 4 * q, pk[2 * gi], pk[2 * gi + 1]);
          }
        }
      }
      // ---- G1: the NC1 corners are split between the warp-groups (balance: G0 gives wg 0 eight groups and wg 1 four)
      constexpr int NG1 = 3 * (NC1 / 2);
      uint32_t pk1[2 * NG1];
#pragma unroll
      for (int jj = 0; jj < NC1 / 2; ++jj) {
        const float w = w1(wg * (NC1 / 2) + jj);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          __half2 lo = __floats2half2_rn(w * __uint_as_float(accg1[4 * q]), w * __uint_as_float(accg1[4 * q + 1]));
          __half2 hi = __floats2half2_rn(w * __uint_as_float(accg1[4 * q + 2]), w * __uint_as_float(accg1[4 * q + 3]));
          pk1[2 * (3 * jj + q)] = *reinterpret_cast<uint32_t*>(&lo);
          pk1[2 * (3 * jj + q) + 1] = *reinterpret_cast<uint32_t*>(&hi);
        }
      }
#pragma unroll
      for (int s = 0; s < 5; ++s) {
        if (s < a.steps1) {
          uint32_t o[2 * NG1];
#pragma unroll
          for (int i = 0; i < 2 * NG1; ++i) o[i] = __shfl_down_sync(0xffffffffu, pk1[i], 1 << s);
          const uint32_t m = (si1.same >> s) & 1u ? 0xffffffffu : 0u;
#pragma unroll
          for (int i = 0; i < 2 * NG1; ++i) {
            const uint32_t om = o[i] & m;
            __half2 r = __hadd2(*reinterpret_cast<const __half2*>(&pk1[i]), *reinterpret_cast<const __half2*>(&om));
            pk1[i] = *reinterpret_cast<uint32_t*>(&r);
          }
        }
      }
      if (live && si1.head && !(a.dbg & 16)) {
#pragma unroll
        for (int jj = 0; jj < NC1 / 2; ++jj) {
          const int key = node1 + off1(wg * (NC1 / 2) + jj);
#pragma unroll
          for (int q = 0; q < 3; ++q) red4(a.dgs1 + (size_t)key * 12 + 4 * q, pk1[2 * (3 * jj + q)], pk1[2 * (3 * jj + q) + 1]);
        }
      }
    }
    mark(12);
    if (a.prof && !tl && tid == 0) atomicAdd(a.prof + 15, 1ull);      // (every slot counts its tiles)
    // (the next tile's first MMA batch is preceded by tcgen05.fence::before_thread_sync + the slot barrier in run_mmas, which
    // orders it after this tile's tcgen05.ld)
    tile = (unsigned)sInfo[4 * (tiles_done & 1)];
  }
  if (FS && u_pending) fs_scatter_rows();       // the last tile's gradient rows
  // -------------------------------------------------------------------------------------------- flush: MLP gradients
  pdl_launch_dependents();       // train_finish_kernel may be scheduled now; it waits for this grid to complete
  if (prof0) prof_t = clock64();
  if (tl && prof0) {
    const unsigned long long t = gtime();
    atomicMax(a.prof + 4, ~t);
    atomicMax(a.prof + 5, t);
  }
  if (tiles_done > 0) mbar_wait_sleep(mbar2, phase2);       // the last tile's deferred D1 batch (and everything before it)
  tc_fence_before();
  __syncthreads();               // all slots: every MMA of the CTA is complete
  tc_fence_after();
  {
    // Every CTA writes its sums to its OWN slice with plain stores (each element exactly once); mlp_grad_reduce_kernel
    // adds the slices up in a fixed order.  (296 CTAs x 9,091 atomicAdds onto the same 9,091 addresses took a fifth of
    // the kernel, and made the MLP gradients depend on the order of arrival.)
    // Slice layout (TRANSPOSED, so that the 32 lanes = 32 consecutive accumulator rows of a store write one 128-byte run):
    //   [K1' = CIN + 1 columns][64 hidden units]  dW1 (column CIN: db1)  |  [65][64]  dW2 (column 64: db2)  |  [cout][64] dW3 | db3
    const float fs = a.flush_scale;
    float* part = a.partials + (size_t)blockIdx.x * a.pstride;
    float* p_w1t = part;
    float* p_w2t = p_w1t + 64 * (CIN + 1);
    float* p_w3 = p_w2t + 64 * 65;
    float* p_b3 = p_w3 + 64 * a.cout;
    // D3^T: rows 0..63 = hidden unit h, row 64 = the bias feature; columns c < cout: dW3'[c][h] (W3' = W3/2) / db3[c]
    // D2: rows 0..63 = hidden unit j; columns 0..63 = dW2'[j][k] (W2' = W2/2), 64 = db2[j];
    // D1: rows 0..63 = hidden unit j (dZ2 and dZ1 live in B2's features 0..63); columns 0..72 = dW1[j][cin], 73 = db1[j].
    // Warp-group 0 reads columns [0,48), 1 reads [48,80).  Slot 0 flushes D3 and D2, slot 1 (if any) D1.
    if (wg == 0 && slot == 0) {
      uint32_t acc[16];
      tmem_ld16(tmem + TT_COL_D3 + lane_base, acc);
      tc_wait_ld();
#pragma unroll
      for (int c = 0; c < 16; ++c)
        if (c < a.cout) {
          const float v = __uint_as_float(acc[c]) * fs;
          if (row < 64) p_w3[c * 64 + row] = 0.5f * v;
          else if (row == 64) p_b3[c] = v;
        }
    }
    for (int which = 1; which < 3; ++which) {
      if (slot != (NSLOT > 1 ? which - 1 : 0)) continue;
      const uint32_t dcol = which == 1 ? TT_COL_D2 : TT_COL_D1;
      const int width = which == 1 ? 80 : K1;                            // 80-wide: wg 0 reads [0,48), wg 1 [48,80); 128: halves
      const int c0 = width == 80 ? wg * 48 : wg * 64, cw = width == 80 ? (wg == 0 ? 48 : 32) : 64;
      uint32_t acc[64];
#pragma unroll
      for (int c = 0; c < 64; c += 16)
        if (c < cw) tmem_ld16(tmem + dcol + lane_base + c0 + c, acc + c);
      tc_wait_ld();
#pragma unroll
      for (int i = 0; i < 64; ++i) {
        if (i >= cw) continue;
        const int col = c0 + i;
        const float v = __uint_as_float(acc[i]) * fs;
        if (which == 1) {
          if (row < 64 && col <= 64) p_w2t[col * 64 + row] = col < 64 ? 0.5f * v : v;
        } else if (row < 64 && col <= CIN) {
          p_w1t[col * 64 + row] = v;
        }
      }
    }
  }
  if (a.loss_sum) {
    float v = loss_local;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) sRed[warp] = v;
    slot_sync();
    if (tid == 0) atomicAdd(a.loss_sum, ((sRed[0] + sRed[1]) + (sRed[2] + sRed[3])));
    if (g.metrics) {
      slot_sync();
      v = sse8_local;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0) sRed[warp] = v;
      slot_sync();
      if (tid == 0) atomicAdd(a.loss_sum + 1, ((sRed[0] + sRed[1]) + (sRed[2] + sRed[3])));
    }
  }
  tc_fence_before();
  __syncthreads();
  mark(13);                    // the flush, once per CTA
  if (prof0 && !tl) atomicAdd(a.prof + 14, (unsigned long long)(clock64() - prof_start));      // CTA lifetime
  if (tl && prof0) {
    const unsigned long long t = gtime();
    atomicMax(a.prof + 6, ~t);
    atomicMax(a.prof + 7, t);
  }
  if (warp_cta == 0) tmem_dealloc(tmem, TS::TMEM);
}

// gm.* += sum over the CTAs' slices, in a fixed order (deterministic).  One block of 256 threads = 32 elements x 8 slice
// lanes, eight independent loads in flight per thread (the slices are L2-resident: just written).
constexpr int TF_THREADS = 256, TF_LANES = TF_THREADS / 32;
__device__ __forceinline__ void mlp_grad_reduce_block(int block, const float* __restrict__ part, int nparts, int pstride,
                                                      const MlpGradDev& gm, int cin, int cout) {
  __shared__ float red[TF_LANES][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i = block * 32 + tx;
  float s = 0.f;
  if (i < pstride) {
    for (int c0 = ty; c0 < nparts; c0 += 8 * TF_LANES) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = c0 + k * TF_LANES < nparts ? part[(size_t)(c0 + k * TF_LANES) * pstride + i] : 0.f;
      s += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    }
  }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && i < pstride) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < TF_LANES; ++k) t += red[k][tx];
    const int o_w2t = 64 * (cin + 1), o_w3 = o_w2t + 64 * 65, o_b3 = o_w3 + 64 * cout;      // the slice layout of train_tc_kernel
    float* dst;
    if (i < o_w2t) {
      const int col = i >> 6, r = i & 63;
      dst = col < cin ? gm.w1 + r * cin + col : gm.b1 + r;
    } else if (i < o_w3) {
      const int col = (i - o_w2t) >> 6, r = (i - o_w2t) & 63;
      dst = col < 64 ? gm.w2 + r * 64 + col : gm.b2 + r;
    } else {
      dst = i < o_b3 ? gm.w3 + (i - o_w3) : gm.b3 + (i - o_b3);
    }
    *dst += t;
  }
}

// The small kernels around train_tc_kernel, fused: a training step at config 1 is 0.16 ms of train_tc_kernel, and every
// extra launch costs 5-8 us of latency on a [12, 129, 129] grid.
//   prep   : 16-bit channel-last shadows of both grids + the packed weight images         (before train_tc_kernel)
//   finish : grid-gradient scratch -> the caller's channel-major gradients (+ re-zero), MLP partial sums -> gm  (after)
struct TrainSideArgs {
  const float* g0;            // prep: source grids [C][z][y][x]
  const float* g1;
  uint16_t* s0;               // prep: shadows [x][y][z][C]
  uint16_t* s1;
  uint16_t* img;              // prep: weight images
  MlpDev m;
  int K1;
  float* gs0;                 // finish: channel-last fp32 scratch (NULL: grids frozen)
  float* gs1;
  float* dg0;
  float* dg1;
  float scale;
  const float* part;          // finish: per-CTA MLP partial sums
  int nparts, pstride;
  MlpGradDev gm;
  int C, n0[3], n1[3];        // nodes per axis (x, y, z), z = 1 in 2-D
  long long t0, t1;           // elements of G0 / G1 handled here (0: the tiled kernels do the grids)
  int nb_items;               // finish: blocks [0, nb_items) walk the grid elements, the rest reduce the partial sums
  unsigned* tile_ctr;         // prep: the training kernel's tile counter, reset every step
};

template <int FMT>
__global__ void __launch_bounds__(256) train_prep_kernel(TrainSideArgs p) {
  pdl_launch_dependents();       // train_tc_kernel's prologue (TMEM allocation, shared-memory clear) may start
  if (blockIdx.x == 0 && threadIdx.x == 0) *p.tile_ctr = 0u;
  const long long nw = 64 * p.K1 + 64 * 80 + 16 * 80, total = p.t0 + p.t1 + nw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (i < p.t0) relayout_small_item<FMT>(i, p.g0, p.s0, p.C, p.n0[0], p.n0[1], p.n0[2]);
    else if (i < p.t0 + p.t1) relayout_small_item<FMT>(i - p.t0, p.g1, p.s1, p.C, p.n1[0], p.n1[1], p.n1[2]);
    else pack_train_weights_item<FMT>((int)(i - p.t0 - p.t1), p.m, p.K1, p.img);
  }
}

__global__ void __launch_bounds__(TF_THREADS) train_finish_kernel(TrainSideArgs p) {
  pdl_wait();                    // launched programmatically behind train_tc_kernel
  pdl_launch_dependents();       // ... and the Adam kernel behind this one
  if ((int)blockIdx.x < p.nb_items) {
    const long long total = p.t0 + p.t1;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)p.nb_items * blockDim.x) {
      if (i < p.t0) grad_add_small_item(i, p.gs0, p.dg0, p.C, p.n0[0], p.n0[1], p.n0[2], p.scale);
      else grad_add_small_item(i - p.t0, p.gs1, p.dg1, p.C, p.n1[0], p.n1[1], p.n1[2], p.scale);
    }
  } else {
    mlp_grad_reduce_block((int)blockIdx.x - p.nb_items, p.part, p.nparts, p.pstride, p.gm, p.m.cin, p.m.cout);
  }
}

// ------------------------------------------------------------------------------------------------ launcher
template <int FMT, int METHOD>
static int launch_train_tc_t(Handle* h, const DevGeom& g, const MlpDev& m, const MlpGradDev& gm, const float* g0,
                             const float* g1, const long long* origins, const float* targets, const float* noise,
                             int noise_bits, unsigned long long seed, unsigned long long step, float grad_scale, float* dg0,
                             float* dg1, float* loss_sum, float* out_save, cudaStream_t st) {
  const long long nodes0 = plane_size_host(g.n0, g.dim), nodes1 = plane_size_host(g.n1, g.dim);
  const void* grids[2] = {g0, g1};
  const ShadowLayout sl = shadow_layout(&g, &grids[0], &grids[1], 1);
  int rc = tc_scratch(h, sl.total);
  if (rc) return rc;
  invalidate_prepared(h);                      // the decode tables share this scratch
  uint16_t* s0 = (uint16_t*)h->tc_shadow;
  uint16_t* s1 = (uint16_t*)((uint8_t*)h->tc_shadow + sl.off[0][1]);
  // channel-last fp32 gradient scratch (zero between steps: grad_relayout_add_kernel re-zeroes what it consumes)
  const size_t gb0 = (size_t)nodes0 * g.C * 4, gb1 = (size_t)nodes1 * g.C * 4;
  float *gs0 = nullptr, *gs1 = nullptr;
  if (dg0) {
    size_t have = h->tc_gscratch_bytes;
    rc = ensure_scratch(&h->tc_gscratch, &h->tc_gscratch_bytes, gb0 + gb1 + 256);
    if (rc) return rc;
    if (h->tc_gscratch_bytes != have) {
      cudaError_t e = cudaMemsetAsync(h->tc_gscratch, 0, h->tc_gscratch_bytes, st);
      if (e != cudaSuccess) return (int)e;
    }
    gs0 = (float*)h->tc_gscratch;
    gs1 = (float*)((uint8_t*)h->tc_gscratch + ((gb0 + 255) & ~(size_t)255));
  }
  cudaError_t e = cudaSuccess;
  // The one-thread-per-element side kernels read / write the channel-major grids with a stride of a whole plane between
  // neighbouring threads: fine (and one launch each) while the grids are L2-resident and tiny — [12, 129, 129] at config 1 —
  // but 19 + 40 us per step on [12, 513, 513] (2048^2 image).  From 160^2 nodes on, the tiled (shared-memory transposing)
  // relayout / relayout-add kernels take over (2-D only).
  const bool small = nodes0 <= 160 * 160 || g.dim == 3;
  TrainSideArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.g0 = g0;
  sa.g1 = g1;
  sa.s0 = s0;
  sa.s1 = s1;
  sa.img = (uint16_t*)h->tc_weights;
  sa.tile_ctr = (unsigned*)((uint8_t*)h->tc_weights + 60 * 1024);       // behind the weight images (<= 29 KB)
  sa.m = m;
  sa.K1 = TrainShape<METHOD>::K1;
  sa.C = g.C;
  for (int d = 0; d < 3; ++d) {
    sa.n0[d] = d < g.dim ? g.n0[d] : 1;
    sa.n1[d] = d < g.dim ? g.n1[d] : 1;
  }
  sa.t0 = small ? nodes0 * g.C : 0;
  sa.t1 = small ? nodes1 * g.C : 0;
  if (sa.t0 >= (1ll << 32) || sa.t1 >= (1ll << 32)) return NIC_ERR_UNSUPPORTED;        // 32-bit index math in the side kernels
  if (!small) {
    rc = build_shadows<FMT>(h, sl, &g, &grids[0], &grids[1], 0, st);
    if (rc) return rc;
  }
  {
    const long long items = sa.t0 + sa.t1 + 64 * sa.K1 + 64 * 80 + 16 * 80;
    const long long nb = (items + 255) / 256, cap = 8ll * h->sms;
    train_prep_kernel<FMT><<<(int)(nb < cap ? nb : cap), 256, 0, st>>>(sa);
  }
  h->launches++;
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;

  TrainArgs a;
  memset(&a, 0, sizeof(a));
  a.s0 = (const uint2*)s0;
  a.s1 = (const uint2*)s1;
  a.origins = origins;
  a.wimg = (const uint4*)h->tc_weights;
  a.targets = targets;
  a.noise = noise;
  a.dgs0 = gs0;
  a.dgs1 = gs1;
  a.loss_sum = loss_sum;
  a.out_save = out_save;
  a.gm = gm;
  a.noise_amp = (!noise && noise_bits > 0) ? ldexpf(1.0f, -noise_bits) : 0.f;
  a.seed = seed;
  a.step = step;
  a.flush_scale = 2.0f * grad_scale / TT_LOSS_SCALE;
  a.cout = m.cout;
  int s0n = 0;
  while (s0n < 5 && ldexpf(1.0f, -s0n) > g.step) ++s0n;       // lanes sharing a G0 node along the fast axis: 1/step
  a.steps0 = s0n;
  a.steps1 = s0n + 1 > 5 ? 5 : s0n + 1;
  a.dbg = h->debug_flags;
  a.tile_ctr = h->static_tiles ? nullptr : sa.tile_ctr;
  if (h->debug_flags & 8) {
    if (!h->dbg_counters) {
      e = cudaMalloc(&h->dbg_counters, 16 * 8);
      if (e == cudaSuccess) e = cudaMemsetAsync(h->dbg_counters, 0, 16 * 8, st);
      if (e != cudaSuccess) return (int)e;
    }
    a.prof = h->dbg_counters;
  }
  void (*kern)(DevGeom, TrainArgs) = train_tc_kernel<FMT, METHOD, 0>;
  if constexpr (METHOD == NIC_METHOD_2D) {
    // full-resolution crops whose rows are whole tiles: the node reduction of the scatter runs on the tensor core
    // (NIC_OPT_DEBUG_KNOCKOUT bit 8 keeps the shuffle path for A/B runs)
    if (dg0 && g.step == 0.25f && g.interp && g.B[1] % TT_ROWS == 0 && !(h->debug_flags & 256)) kern = train_tc_kernel<FMT, METHOD, 1>;
  }
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, TrainShape<METHOD>::SMEM);
  if (e != cudaSuccess) return (int)e;
  if (g.N >= (1ll << 27)) return NIC_ERR_UNSUPPORTED;          // Philox counter packs (sample << 4 | block)
  constexpr int NSLOT = TrainShape<METHOD>::NSLOT;
  long long ntiles = (g.N + TT_ROWS - 1) / TT_ROWS;
  const long long want = (ntiles + NSLOT - 1) / NSLOT, cap = h->sms;          // one persistent CTA per SM, NSLOT tiles in flight each
  int grid = (int)(want < cap ? want : cap);
  a.pstride = 64 * m.cin + 64 + 64 * 64 + 64 + 64 * m.cout + m.cout;
  rc = ensure_scratch(&h->tc_partials, &h->tc_partials_bytes, (size_t)grid * a.pstride * sizeof(float));
  if (rc) return rc;
  a.partials = (float*)h->tc_partials;
  if (h->time_kernels) {          // the event records between the kernels rule out a programmatic launch
    KernelTimer timer(h, st);
    kern<<<grid, TrainShape<METHOD>::THREADS, TrainShape<METHOD>::SMEM, st>>>(g, a);
  } else {
    e = launch_pdl(kern, dim3(grid), dim3(TrainShape<METHOD>::THREADS), TrainShape<METHOD>::SMEM, st, g, a);
    if (e != cudaSuccess) return (int)e;
  }
  h->launches++;
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  sa.gs0 = gs0;
  sa.gs1 = gs1;
  sa.dg0 = dg0;
  sa.dg1 = dg1;
  sa.scale = 2.0f * grad_scale / TT_LOSS_SCALE;
  sa.part = a.partials;
  sa.nparts = grid;
  sa.pstride = a.pstride;
  sa.gm = gm;
  if (!(dg0 && small)) sa.t0 = sa.t1 = 0;                       // frozen grids, or the tiled kernels below do them
  {
    const long long nb = (sa.t0 + sa.t1 + TF_THREADS - 1) / TF_THREADS, cap = 16ll * h->sms;
    sa.nb_items = (int)(nb < cap ? nb : cap);
    e = launch_pdl(train_finish_kernel, dim3(sa.nb_items + (a.pstride + 31) / 32), dim3(TF_THREADS), 0, st, sa);
    if (e != cudaSuccess) return (int)e;
  }
  h->launches++;
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if (dg0 && !small) {
    size_t smem = (size_t)g.C * GR_TF * 33 * sizeof(float);
    if (smem > 48 * 1024) return NIC_ERR_UNSUPPORTED;
    grad_relayout_add_kernel<<<dim3((g.n0[0] + 31) / 32, (g.n0[1] + GR_TF - 1) / GR_TF), 256, smem, st>>>(gs0, dg0, g.C, g.n0[0], g.n0[1], sa.scale);
    grad_relayout_add_kernel<<<dim3((g.n1[0] + 31) / 32, (g.n1[1] + GR_TF - 1) / GR_TF), 256, smem, st>>>(gs1, dg1, g.C, g.n1[0], g.n1[1], sa.scale);
    h->launches += 2;
    e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  return NIC_OK;
}

int launch_train_tc(Handle* h, const DevGeom& g, const MlpDev& m, const MlpGradDev& gm, const float* g0, const float* g1,
                    const long long* origins, const float* targets, const float* noise, int noise_bits,
                    unsigned long long seed, unsigned long long step, float grad_scale, float* dg0, float* dg1,
                    float* loss_sum, float* out_save, int precision, cudaStream_t st) {
  if (g.N == 0) return NIC_OK;
  if (!tc_shape_ok(g, m) || !origins) return NIC_ERR_UNSUPPORTED;
  return dispatch_method_fmt(g.method, precision, [&](auto M, auto FMT) -> int {
    if (m.cin != TrainShape<M.value>::CIN) return NIC_ERR_UNSUPPORTED;
    return launch_train_tc_t<FMT.value, M.value>(h, g, m, gm, g0, g1, origins, targets, noise, noise_bits, seed, step,
                                                 grad_scale, dg0, dg1, loss_sum, out_save, st);
  });
}

}  // namespace nic
