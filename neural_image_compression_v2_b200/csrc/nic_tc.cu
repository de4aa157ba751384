// nic_tc.cu — K2, the fused tensor-core decode: gather -> Linear/GELU/Linear/GELU/Linear/Sigmoid -> output,
// with all three layer GEMMs on tcgen05.mma (sm_100a) and every activation resident in TMEM / registers.
// Reference behaviour: finally_decode_input_* + ColorDecoder.forward inside decode_image
// (Projects/image_compression.py:54-68, 170-211, 313-327).
//
// Two kernel bodies, both ONE persistent CTA per SM made of independent groups of 4 warps (a group = one tile of 128
// texels = the MMA M = the TMEM lanes; a group owns 64 accumulator columns of TMEM and its operand buffers in shared memory):
//   decode_tc2d_ws_kernel   aligned full-resolution 2-D frames; layer 1 re-associated so no input row is ever built;
//   decode_tc_gws_body      everything else (any mip / origin / block shape, both 3-D methods, random-access queries),
//                           behind two entry points that differ in where the grids come from:
//     decode_tc_gws_kernel      16-bit shadows of the grids in global memory (ShadowGeom);
//     decode_codes_smem_kernel  random-access queries on a small model whose uint8 codes stay resident in shared memory
//                               (ResidentCodes).
// Per tile: layer 1 (KX/16 or 5 tcgen05.mma, M=128 N=64 K=16, SS form) -> epilogue: tcgen05.ld, packed GELU, st.shared in
// the UMMA K-major layout -> layer 2 (4 MMAs + 1 bias MMA against a constant ones block) -> epilogue -> layer 3 (N=16)
// -> sigmoid, quantise, store.  The 1/2 of GELU is folded into the next layer's weights.
//
// Algorithmic work: 2*(Cin*64 + 64*64 + 64*Cout) FLOP/texel (17,920 for the 2-D default); tensor-bound roofline.
#include "nic_tc_common.cuh"

namespace nic {

// ------------------------------------------------------------------------------------------------ weight images
// Operand-B images in global memory, already in the shared-memory UMMA layout (K-major, no swizzle):
//   byte offset of element (n, k) = (k/8)*LBO + (n/8)*128 + (n%8)*16 + (k%8)*2,  LBO = (Nrows/8)*128.
// W1': [64 x KX]  col k < cin-1: W1[n][k];  col cin-1: b1[n] + lod*W1[n][cin-1];  rest 0.
// W2': [64 x 80]  col k < 64: W2[n][k]/2 (W2[n][k] for hidden columns on the polynomial GELU);   col 64: b2[n];  rest 0.
// W3': [16 x 80]  row n < cout: col k < 64: W3[n][k]/2 (same rule); col 64: b3[n];  rest 0.
// (code-resident path, the general body reading ResidentCodes: the A operand holds the integer grid codes minus their
//  offset, so the grid columns k < grid_cols of W1 carry the 1 / (2^bits - 1) of models.load4fp: gscale.)
template <int FMT>
__global__ void pack_weights_kernel(MlpDev m, float lod, int KX, uint16_t* __restrict__ img, int npoly, int grid_cols = 0,
                                    float gscale = 1.0f) {
  const int H = 64;
  const int n1 = H * KX, n2 = H * 80, n3 = 16 * 80;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n1 + n2 + n3; i += gridDim.x * blockDim.x) {
    int which = i < n1 ? 0 : (i < n1 + n2 ? 1 : 2);
    int local = which == 0 ? i : (which == 1 ? i - n1 : i - n1 - n2);
    int nrows = which == 2 ? 16 : H;
    // decode the position inside the image: [k/8][n/8][n%8][k%8]
    int kc = local / (nrows * 8);
    int rem = local - kc * nrows * 8;
    int n = rem / 8, ke = rem - n * 8;
    int k = kc * 8 + ke;
    float v = 0.f;
    // hidden column k arrives as 2*gelu (MUFU tanh form) or as gelu (polynomial form, gelu_poly_pair)
    const float half = gelu_poly_column(k, npoly) ? 1.0f : 0.5f;
    if (which == 0) {
      if (k < m.cin - 1) v = k < grid_cols ? __fmul_rn(m.w1[n * m.cin + k], gscale) : m.w1[n * m.cin + k];
      else if (k == m.cin - 1) v = m.b1[n] + lod * m.w1[n * m.cin + k];
    } else if (which == 1) {
      if (k < H) v = half * m.w2[n * H + k];
      else if (k == H) v = m.b2[n];
    } else if (n < m.cout) {
      if (k < H) v = half * m.w3[n * H + k];
      else if (k == H) v = m.b3[n];
    }
    img[i] = to16<FMT>(v);
  }
}

// nic_sample_lod (decode_tc_gws_kernel with TAPS = 2 * 2^D): the row carries the mip in column cin - 1 against
// W1[:, cin - 1] and the constant 1 in column cin against b1 (the reference's own [... | pe | lod] layout), so W1' gets
// those two columns instead of the folded bias.
template <int FMT>
__global__ void pack_lod_columns_kernel(MlpDev m, uint16_t* __restrict__ img) {
  const int n = threadIdx.x;
  if (n >= 64) return;
  auto at = [&](int k) { return img + (k / 8) * 64 * 8 + n * 8 + (k % 8); };
  *at(m.cin - 1) = to16<FMT>(m.w1[n * m.cin + m.cin - 1]);
  *at(m.cin) = to16<FMT>(m.b1[n]);
}

// ------------------------------------------------------------------------------------------------ decoder-input row
// Decoder-input row of one texel for C = 12, PE = 6 as packed 16-bit pairs (the layer-1 A operand):
//   pairs [6j, 6j+6)         corner j of G0 (raw copy of the shadow node)
//   pairs [6*NC0, 6*NC0+6)   sum_j w_j * G1 corner j   (packed fma; w_j exact in f16)
//   then 3 pairs per axis    positional encoding (shared-memory LUT for the triangular kind)
//   half CIN-1               constant 1 carrying the layer-1 bias (+ LOD), remaining halves 0.
template <int METHOD>
struct RowShape {
  static constexpr int DIM = METHOD == NIC_METHOD_2D ? 2 : 3;
  static constexpr int NC0 = METHOD == NIC_METHOD_3D ? 8 : 4;
  static constexpr int NC1 = METHOD == NIC_METHOD_2D ? 4 : 8;
  static constexpr int C = 12, PE = 6;
  static constexpr int CIN = C * (NC0 + 1) + PE * DIM + 1;    // 73 / 127 / 79
  static constexpr int KX = (CIN + 15) / 16 * 16;            // 80 / 128 / 80
};

__device__ __forceinline__ int node_lin(const int* n, int dim, int x, int y, int z) {
  // shadow order: x slowest, then y, then z (2-D: x, y)
  return dim == 2 ? x * n[1] + y : (x * n[1] + y) * n[2] + z;
}

constexpr int TC_ROWS = 128;    // texels per tile = MMA M = TMEM lanes
constexpr int TC_K2 = 80;       // K of layers 2/3: 64 hidden + the bias block
constexpr int TC_LUT_MAX = 256; // positional-encoding LUT entries (period 16/step texels)

// ================================================================================================ 2-D fast path
// Full-resolution 2-D decode (step 1/4, interpolation on, triangular PE, block aligned to 8 x 16 texels): layer 1 is
// re-associated so that NO per-texel input is ever built.  For a tile of 8 x 16 texels:
//   z1 = W1[:, 0:48] * (G0 corners of the texel's cell)          -> the 128 rows alias 8 cell rows (descriptor SBO = 0)
//      + sum_nodes tent(node, texel) * R[node]                   R[node] = W1[:, 48:60] * G1[node]   (per-node table)
//      + LUTx[px mod 64] + LUTy[py mod 64]                       LUT = W1[:, 60:72] * PE(p) (+ bias and LOD in LUTx)
// The last two lines are ONE constant 128 x 32 selector/weight matrix (tent weights, one-hot x, one-hot y) that stays
// in shared memory for the life of the CTA, times per-tile table rows that are addressed in shared memory as an MN-major
// B operand.  Row m of a tile is texel (cell = m % 8, within-cell index = m / 8).
constexpr int F_TX = 8, F_TY = 16;                 // tile extent in texels (x = first image axis)
constexpr int F_W1G0 = b_image_bytes(64, 48);      // 6144
constexpr int F_LUT = 64 * 64 * 2;                 // 8192 per axis
constexpr int F_IMG = F_W1G0 + b_image_bytes(64, TC_K2) + b_image_bytes(16, TC_K2) + 2 * F_LUT;

// R[node][n] = sum_c W1[n][4C + c] * G1[c][node], stored [x][y][64] 16-bit (128 B per node).  Persistent blocks walk tiles of
// 8 (x) x 16 (y) nodes.  A thread owns FOUR of the 64 outputs and keeps their 4 x 12 weights in registers for the life of the
// block; the 16 threads of an output row share a node, whose 12 channels come from a channel-last shared-memory patch as three
// 16-byte loads (48 FMAs per 3 loads), and together write the node's 128 bytes as one run.  A thread does 8 nodes per tile,
// two at a time.  The next tile's patch is in flight in registers while the block works on the current one.
// (History: one thread per node with 64 accumulators, stores 64 KB apart: 52 us for a 513 x 513 grid; four threads per node
// pair with the weights re-read from shared memory for every channel — 6 loads per 32 FMAs, half of them two-wavefront bank
// conflicts — 40 us, 30 us without the conflicts: the kernel waited on shared-memory latency.)
constexpr int G1R_TX = 8, G1R_TY = 16;
template <int FMT>
__global__ void __launch_bounds__(256, 2) g1_rows_kernel(MlpDev m, const float* __restrict__ g1, int nx, int ny,
                                                         uint16_t* __restrict__ R, int code_bits) {
  constexpr int C = 12, PER = C * G1R_TY * G1R_TX / 256;    // patch elements per thread (6)
  constexpr int ROW = G1R_TX * C + 4;                       // floats per y-row of the patch (+4: rows shifted by 4 banks)
  __shared__ __align__(16) float patch[G1R_TY * ROW];       // [y][x][c], channel-last
  const int oq = threadIdx.x & 15, ns = threadIdx.x >> 4;   // outputs 4 oq .. 4 oq + 3; node row y = ns of the tile
  float wr[4][C];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int c = 0; c < C; ++c) wr[j][c] = m.w1[(4 * oq + j) * m.cin + 4 * C + c];
  const int tiles_x = (nx + G1R_TX - 1) / G1R_TX, tiles_y = (ny + G1R_TY - 1) / G1R_TY, ntiles = tiles_x * tiles_y;
  const size_t nodes = (size_t)nx * ny;
  float pf[PER];
  auto fetch = [&](int tile) {
    const int x0 = (tile / tiles_y) * G1R_TX, y0 = (tile % tiles_y) * G1R_TY;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
      const int i = threadIdx.x + 256 * k;
      const int c = i / (G1R_TY * G1R_TX), r = i - c * (G1R_TY * G1R_TX), yl = r / G1R_TX, xl = r - yl * G1R_TX;
      const int x = x0 + xl, y = y0 + yl;
      pf[k] = (x < nx && y < ny) ? grid_value(g1, (long long)(c * nodes + (size_t)y * nx + x), code_bits) : 0.f;
    }
  };
  int tile = blockIdx.x;
  if (tile < ntiles) fetch(tile);
  for (; tile < ntiles; tile += gridDim.x) {
#pragma unroll
    for (int k = 0; k < PER; ++k) {
      const int i = threadIdx.x + 256 * k;
      const int c = i / (G1R_TY * G1R_TX), r = i - c * (G1R_TY * G1R_TX), yl = r / G1R_TX, xl = r - yl * G1R_TX;
      patch[yl * ROW + xl * C + c] = pf[k];
    }
    __syncthreads();
    if (tile + (int)gridDim.x < ntiles) fetch(tile + gridDim.x);
    const int x0 = (tile / tiles_y) * G1R_TX, y = (tile % tiles_y) * G1R_TY + ns;
    if (y < ny) {
#pragma unroll
      for (int xl = 0; xl < G1R_TX; xl += 2) {
        float g[2][C];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float4* p = reinterpret_cast<const float4*>(patch + ns * ROW + (xl + u) * C);
          const float4 a = p[0], bq = p[1], cq = p[2];
          g[u][0] = a.x; g[u][1] = a.y; g[u][2] = a.z; g[u][3] = a.w;
          g[u][4] = bq.x; g[u][5] = bq.y; g[u][6] = bq.z; g[u][7] = bq.w;
          g[u][8] = cq.x; g[u][9] = cq.y; g[u][10] = cq.z; g[u][11] = cq.w;
        }
        float acc[2][4];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[u][j] = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c)
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[u][j] = fmaf(g[u][c], wr[j][c], acc[u][j]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int x = x0 + xl + u;
          if (x < nx) {
            uint2 v;
            v.x = to16<FMT>(acc[u][0]) | ((uint32_t)to16<FMT>(acc[u][1]) << 16);
            v.y = to16<FMT>(acc[u][2]) | ((uint32_t)to16<FMT>(acc[u][3]) << 16);
            *reinterpret_cast<uint2*>(R + ((size_t)x * ny + y) * 64 + 4 * oq) = v;
          }
        }
      }
    }
    __syncthreads();
  }
}

// Weight images of the fast path: [W1g0 K-major 64x48][W2' 64x80][W3' 16x80][LUTx][LUTy]; LUT element (n, k = p mod 64)
// at (k/8)*1024 + (n/8)*128 + (k%8)*16 + (n%8)*2  (MN-major B operand, 8 k-rows x 8 n per 128-byte block).
template <int FMT>
__global__ void pack_fast_kernel(MlpDev m, float lod, float step, uint16_t* __restrict__ img, int npoly) {
  const int H = 64, C = 12, PE = 6;
  const int n1 = H * 48, n2 = H * 80, n3 = 16 * 80, nl = 64 * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n1 + n2 + n3 + 2 * nl; i += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i < n1 + n2 + n3) {
      int which = i < n1 ? 0 : (i < n1 + n2 ? 1 : 2);
      int local = which == 0 ? i : (which == 1 ? i - n1 : i - n1 - n2);
      int nrows = which == 2 ? 16 : H;
      int kc = local / (nrows * 8), rem = local - kc * nrows * 8;
      int n = rem / 8, k = kc * 8 + (rem - n * 8);
      // hidden column k arrives as 2*gelu (MUFU tanh form) or as gelu (polynomial form, gelu_poly_pair)
      const float half = gelu_poly_column(k, npoly) ? 1.0f : 0.5f;
      if (which == 0) v = m.w1[n * m.cin + k];
      else if (which == 1) v = k < H ? half * m.w2[n * H + k] : (k == H ? m.b2[n] : 0.f);
      else if (n < m.cout) v = k < H ? half * m.w3[n * H + k] : (k == H ? m.b3[n] : 0.f);
    } else {
      int local = i - (n1 + n2 + n3);
      int axis = local / nl;
      local -= axis * nl;
      int kg = local / 512, rem = local - kg * 512;       // 512 elements per k-group: [n/8][k%8][n%8]
      int ng = rem / 64, r2 = rem - ng * 64;
      int k = kg * 8 + r2 / 8, n = ng * 8 + (r2 & 7);
      float u1 = __fmul_rn(__fmul_rn((float)k, step), 0.5f);
      float acc = axis == 0 ? m.b1[n] + lod * m.w1[n * m.cin + (m.cin - 1)] : 0.f;
      for (int r = 0; r < PE; ++r) acc = fmaf(m.w1[n * m.cin + 5 * C + axis * PE + r], pe_triangular(u1, r, PE), acc);
      v = acc;
    }
    img[i] = to16<FMT>(v);
  }
}

// ================================================================================================ 2-D fast path, v2
// Warp-specialised persistent form of the kernel above.  Knock-out experiments (NIC option 100, tools/run_decode.py)
// showed the first versions were bound by the LATENCY of the per-tile chain (epilogue -> barrier -> MMA issue ->
// MMAs (then ~95 cycles each: they were still issued from divergent control flow, see elect_one() in nic_tc_common.cuh)
// -> commit -> wake-up -> tcgen05.ld), i.e. by how many tiles are in flight, not by any pipe.
// TMEM caps that number: with the next layer's A operand in TMEM a tile needs 104 columns (4 tiles).  Here the
// activations go to SHARED memory instead (st.shared in the UMMA K-major core-matrix layout, SS-form MMAs), a tile
// needs only its 64 accumulator columns, and EIGHT tiles are in flight per SM:
//   * ONE CTA of 1024 threads per SM = eight independent warp-groups of 4 warps; group s owns TMEM columns [64 s, +64),
//     a 16 KB activation buffer and a double-buffered 2 KB operand staging area;
//   * a group runs its tiles as a private pipeline: tcgen05.ld 16 columns -> packed 2*gelu -> one 16-byte st.shared per
//     8 columns; after a 128-thread named barrier its elected lane issues the next tcgen05.mma batch (layer 1: 3
//     aliased-cell MMAs + selector x [G1 rows | LUTx] + selector x LUTy; layers 2, 3: 4 MMAs + 1 bias MMA against a
//     shared constant ones block) and the group waits on its own mbarrier (tcgen05.commit).  Groups never meet at a
//     CTA-wide barrier, so one group's MMAs and hand-offs run under the other groups' epilogues;
//   * the group stages its own operands: its threads fetch the pieces (8 B of a G0 cell row / 16 B of a G1 node row)
//     of the tile after next into registers while the current tile is processed.
constexpr int WS_SLOTS = 8, WS_GROUP = 128, WS_THREADS = WS_SLOTS * WS_GROUP;
constexpr int WS_NPOLY_F16 = 3, WS_NPOLY_BF16 = 3;   // default share (of 8) of activation pairs on the polynomial GELU
constexpr int WS_TMEM_COLS = 512;
constexpr int WS_STAGE = WS_SLOTS * 2 * 2048;       // [slot][buffer][Ag0 1 KB | G1 rows 1 KB]
constexpr int WS_KG = 16 * 128;                     // bytes of one k-group (8 columns) of a 128-row K-major A operand
constexpr int WS_OFF_SEL = WS_STAGE + F_IMG;        // selector matrix, 128 x 32 (4 k-groups)
constexpr int WS_OFF_ONE = WS_OFF_SEL + 4 * WS_KG;  // ones block, 128 x 16: column 0 = 1
constexpr int WS_OFF_ACT = WS_OFF_ONE + 2 * WS_KG;  // [slot] 128 x 64 activations (8 k-groups)
constexpr int WS_OFF_BAR = WS_OFF_ACT + WS_SLOTS * 8 * WS_KG;
constexpr int WS_SMEM = WS_OFF_BAR + 256;

// Output activation of the warp-specialised kernels: sigmoid(z) = 1/2 + 1/2 tanh(z/2) — one MUFU instead of ex2 + rcp; the
// 8-bit code is floor(v * 255 + .5) of exactly the float this kernel would store (separate multiply and add like
// models.quantize_to_bit), and needs no clamp because v is in [0, 1].
__device__ __forceinline__ float sigmoid_tanh(float z) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(z * 0.5f));
  return fmaf(t, 0.5f, 0.5f);
}
__device__ __forceinline__ void store_sigmoid(float* p, float z) { *p = sigmoid_tanh(z); }
__device__ __forceinline__ void store_sigmoid(uint8_t* p, float z) {
  *p = (uint8_t)__float2uint_rd(__fadd_rn(__fmul_rn(sigmoid_tanh(z), 255.0f), 0.5f));
}

__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}

// CO = 3: the production instance for RGB outputs (no knock-out flags, channel count folded: the per-tile integer work of
// the generic instance — three uniform branches per channel, the output pointer re-read per store — was 100 of the 755
// instructions per texel, profiles/r02f); CO = 0: any channel count <= 16, honours NIC_OPT_DEBUG_KNOCKOUT.
template <int FMT, typename OutT, int NPOLY, int CO>
__global__ void __launch_bounds__(WS_THREADS, 1) decode_tc2d_ws_kernel(DevGeom g, const uint2* __restrict__ shadow0,
                                                                       const uint4* __restrict__ R,
                                                                       const uint4* __restrict__ wimg, int cout_arg,
                                                                       unsigned tiles_y, unsigned fd_mul, unsigned fd_shift,
                                                                       OutT* __restrict__ out, int dbg_arg) {
  using P = Pair<FMT>;
  const int cout = CO ? CO : cout_arg, dbg = CO ? 0 : dbg_arg;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint8_t* sW = smem_raw + WS_STAGE;                // weight images + LUTs sit ABOVE the staging buffers (LBO = distance)
  uint8_t* sW1 = sW;
  uint8_t* sW2 = sW1 + F_W1G0;
  uint8_t* sW3 = sW2 + b_image_bytes(64, TC_K2);
  uint8_t* sLx = sW3 + b_image_bytes(16, TC_K2);
  uint8_t* sLy = sLx + F_LUT;
  uint8_t* sSel = smem_raw + WS_OFF_SEL;
  uint8_t* sOne = smem_raw + WS_OFF_ONE;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem_raw + WS_OFF_BAR);     // [8]: tensor core -> group
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_full + WS_SLOTS);

  const int tid = threadIdx.x, warp = uniform_warp_index(), lane = tid & 31;     // warp: provably uniform (MMA operands)
  const int slot = warp >> 2;                        // warp-group = tile slot
  const int row = 32 * (warp & 3) + lane;            // texel row of the tile = TMEM lane
  const int cell = row & 7, within = row >> 3;
  const int lx = 4 * (cell >> 2) + (within >> 2), ly = 4 * (cell & 3) + (within & 3);
  const int roff = (row >> 3) * 128 + (row & 7) * 16;      // this row's 16-byte chunk inside a k-group block
  if (warp == 0) tmem_alloc(tmem_slot, WS_TMEM_COLS);
  if (tid == 0)
    for (int s = 0; s < WS_SLOTS; ++s) mbar_init(bar_full + s, 1);
  {
    uint4* dst = reinterpret_cast<uint4*>(sW);
    for (int i = tid; i < F_IMG / 16; i += WS_THREADS) dst[i] = __ldg(wimg + i);
    for (int i = tid; i < WS_STAGE / 16; i += WS_THREADS) reinterpret_cast<uint4*>(smem_raw)[i] = make_uint4(0, 0, 0, 0);
  }
  if (slot == 0) {
    // selector row of this texel: [6 tent weights of the 2 x 3 G1 nodes, 0, 0 | one-hot x (8) | one-hot y (16)]
    float kx = (float)lx * 0.125f, ky = (float)(ly & 7) * 0.125f;
    int cy1 = ly >> 3;
    float sel[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) sel[i] = 0.f;
#pragma unroll
    for (int ix = 0; ix < 2; ++ix)
#pragma unroll
      for (int iy = 0; iy < 3; ++iy) {
        float wx = ix ? kx : 1.0f - kx;
        float wy = iy == cy1 ? 1.0f - ky : (iy == cy1 + 1 ? ky : 0.f);
        sel[ix * 3 + iy] = wx * wy;
      }
#pragma unroll
    for (int j = 0; j < 8; ++j) sel[8 + j] = j == lx ? 1.f : 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) sel[16 + j] = j == ly ? 1.f : 0.f;
#pragma unroll
    for (int kg = 0; kg < 4; ++kg) {
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        auto v = P::pack(sel[8 * kg + 2 * i], sel[8 * kg + 2 * i + 1]);
        w[i] = *reinterpret_cast<uint32_t*>(&v);
      }
      *reinterpret_cast<uint4*>(sSel + kg * WS_KG + roff) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    auto one = P::pack(1.0f, 0.0f);
    *reinterpret_cast<uint4*>(sOne + roff) = make_uint4(*reinterpret_cast<uint32_t*>(&one), 0, 0, 0);
    *reinterpret_cast<uint4*>(sOne + WS_KG + roff) = make_uint4(0, 0, 0, 0);
  }
  fence_async_smem();
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const unsigned ntiles = (unsigned)(g.B[0] / F_TX) * tiles_y;
  const unsigned my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  auto tile_origin = [&](unsigned tile, int& px0, int& py0, int& bx0, int& by0) {
    unsigned tx = fastdiv31(tile, fd_mul, fd_shift), ty = tile - tx * tiles_y;
    bx0 = (int)tx * F_TX;
    by0 = (int)ty * F_TY;
    px0 = g.origin0[0] + bx0;
    py0 = g.origin0[1] + by0;
  };

  const int gt = tid & (WS_GROUP - 1);               // thread index inside the group
  const uint32_t tDs = tmem + slot * 64;             // this slot's accumulator columns
  const uint32_t tD = tDs + ((uint32_t)((warp & 3) * 32) << 16);
  uint8_t* sAct = smem_raw + WS_OFF_ACT + slot * 8 * WS_KG;
  // the group's issuing (and polling) warp: a different lane quarter for consecutive groups, so the eight issuers are
  // spread over the four SM sub-partitions (warp % 4) instead of all sitting on sub-partition 0
  const bool issuer_warp = (warp & 3) == (slot & 3);
  // f16 operands: the two hidden layers accumulate in f16 (tcgen05 D format F16), so the epilogue reads packed pairs
  // (tcgen05.ld.pack::16b) and skips 32 f32 -> f16x2 conversions per row and layer; measured on the goldens this changes
  // the share of bit-identical 8-bit texels by 0.1 % (the activations are rounded to f16 right after anyway).  bf16
  // operands have no 16-bit accumulator format; the output layer always accumulates in fp32.
  constexpr bool ACC16 = FMT == 0;
  constexpr uint32_t IDESC_64 = make_idesc(FMT, 128, 64, 0, ACC16), IDESC_16 = make_idesc(FMT, 128, 16);
  constexpr uint32_t IDESC_64_BMN = make_idesc(FMT, 128, 64, 1, ACC16);
  constexpr uint32_t LBO_64 = (64 / 8) * 128, LBO_16 = (16 / 8) * 128, SBO = 128;
  const uint32_t aStage = smem_u32(smem_raw), aW1 = smem_u32(sW1), aW2 = smem_u32(sW2), aW3 = smem_u32(sW3);
  const uint32_t aLx = smem_u32(sLx), aLy = smem_u32(sLy), aSel = smem_u32(sSel), aOne = smem_u32(sOne), aAct = smem_u32(sAct);
  const int ny0 = g.n0[1], ny1 = g.n1[1];
  auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + slot), "n"(WS_GROUP) : "memory"); };
  // wait for the group's MMA batch: ONE warp polls the mbarrier, the other three park at the group's named barrier
  // (a hardware wait: no issue slots) — polling by all four warps was 10 % of the kernel's issued instructions
  auto group_wait = [&](uint32_t phase) {
    if (issuer_warp) mbar_wait(bar_full + slot, phase);
    group_sync();
  };
  // ---- operand staging: 144 pieces per tile over 128 threads (threads 0..15 take a second piece).  Piece p of a tile:
  //   p < 96 : 8 bytes of a G0 cell row  (cell c8 = p / 12; the two 24-byte halves of a row are the nodes (x, y) and
  //            (x, y + 1), contiguous in the channel-last shadow, for x and x + 1);
  //   p >= 96: 16 bytes of one of the 2 x 3 G1 node rows R[node] the tile touches.
  // Which piece a thread moves never changes, so everything but the tile's base node is formed once, here: a thread
  // keeps a pointer (pre-offset by its piece) and its shared-memory offset per piece.
  const bool g0_piece = gt < 96;                     // warp-uniform (warps 0..2 of a group: G0, warp 3: G1 rows)
  const uint8_t* src0;                               // this thread's primary piece at tile base 0
  uint32_t dst0;                                     // and where it goes inside a staging buffer
  if (g0_piece) {
    const int c8 = gt / 12, piece = gt - c8 * 12, seg = piece >= 6, off = piece - seg * 6, k = seg * 24 + off * 4;
    src0 = reinterpret_cast<const uint8_t*>(shadow0 + ((size_t)((c8 >> 2) + seg) * ny0 + (c8 & 3)) * 3 + off);
    dst0 = (k >> 3) * 128 + c8 * 16 + (k & 7) * 2;
  } else {
    const int t2 = gt - 96, r6 = t2 >> 3, piece = t2 & 7;
    src0 = reinterpret_cast<const uint8_t*>(R + ((size_t)(r6 / 3) * ny1 + r6 % 3) * 8 + piece);
    dst0 = 1024 + piece * 128 + r6 * 16;
  }
  const int r6b = 4 + (gt >> 3);                     // second piece of threads 0..15: G1 rows 4, 5
  const uint8_t* src1 = reinterpret_cast<const uint8_t*>(R + ((size_t)(r6b / 3) * ny1 + r6b % 3) * 8 + (gt & 7));
  const uint32_t dst1 = 1024 + (gt & 7) * 128 + r6b * 16;
  const uint32_t out_thread = (uint32_t)lx * (uint32_t)g.B[1] + (uint32_t)ly;      // this thread's texel inside a tile
  uint4 pre0 = make_uint4(0, 0, 0, 0), pre1 = make_uint4(0, 0, 0, 0);
  auto fetch = [&](unsigned i) {          // pieces of tile i -> registers
    if (i >= my_tiles) return;
    int px0, py0, bx0, by0;
    tile_origin(blockIdx.x + i * gridDim.x, px0, py0, bx0, by0);
    // byte offsets of the tile's base nodes: the launcher guarantees both tables are smaller than 4 GB
    const uint32_t b0 = ((uint32_t)(px0 >> 2) * (uint32_t)ny0 + (uint32_t)(py0 >> 2)) * 24u;
    const uint32_t b1 = ((uint32_t)(px0 >> 3) * (uint32_t)ny1 + (uint32_t)(py0 >> 3)) * 128u;
    if (g0_piece) {
      const uint2 v = __ldg(reinterpret_cast<const uint2*>(src0 + b0));
      pre0 = make_uint4(v.x, v.y, 0, 0);
    } else {
      pre0 = __ldg(reinterpret_cast<const uint4*>(src0 + b1));
    }
    if (gt < 16) pre1 = __ldg(reinterpret_cast<const uint4*>(src1 + b1));
  };
  auto stage = [&](unsigned i) {          // store the fetched pieces of tile i into its staging buffer
    if (i >= my_tiles) return;
    uint8_t* base = smem_raw + (slot * 2 + ((i / WS_SLOTS) & 1)) * 2048;
    if (g0_piece) *reinterpret_cast<uint2*>(base + dst0) = make_uint2(pre0.x, pre0.y);
    else *reinterpret_cast<uint4*>(base + dst0) = pre0;
    if (gt < 16) *reinterpret_cast<uint4*>(base + dst1) = pre1;
    fence_async_smem();
  };
  // Descriptors as 32-bit halves (mma_ss_lohi): everything that does not depend on the tile is formed once, here; per
  // tile the issuing thread adds the staging-buffer parity and the two LUT groups.
  constexpr uint32_t HI_SBO = smem_desc_hi(SBO), HI_SBO0 = smem_desc_hi(0);
  const uint32_t loAg0 = smem_desc_lo(aStage + slot * 2 * 2048, 128);        // + parity * 128 + kc * 16
  const uint32_t loW1 = smem_desc_lo(aW1, LBO_64);                           // + kc * (2 * LBO_64 >> 4)
  const uint32_t loSel = smem_desc_lo(aSel, WS_KG);
  const uint32_t loLy = smem_desc_lo(aLy, 1024);                             // + group * 64
  const uint32_t loAct = smem_desc_lo(aAct, WS_KG), loOne = smem_desc_lo(aOne, WS_KG);
  const uint32_t loW2 = smem_desc_lo(aW2, LBO_64), loW3 = smem_desc_lo(aW3, LBO_16);
  auto issue_layer1 = [&](unsigned i) {          // elected lane only; tile i's operands are staged
    int px0, py0, bx0, by0;
    tile_origin(blockIdx.x + i * gridDim.x, px0, py0, bx0, by0);
    const uint32_t par = (i / WS_SLOTS) & 1;
    const uint32_t aG1 = aStage + (slot * 2 + par) * 2048 + 1024;
#pragma unroll
    for (int kc = 0; kc < 3; ++kc)
      if (!((dbg & 4) && kc > 0))
        mma_ss_lohi(tDs, loAg0 + par * 128 + kc * 16, HI_SBO0, loW1 + kc * (2 * LBO_64 >> 4), HI_SBO, IDESC_64, kc > 0);
    if (!(dbg & 4)) {
      // selector x [G1 rows of this tile | LUTx group]: the B operand's LBO is the distance between the two pieces
      const uint32_t lx_grp = aLx + ((px0 & 63) >> 3) * 1024;
      mma_ss_lohi(tDs, loSel, HI_SBO, (aG1 >> 4) | (((lx_grp - aG1) >> 4) << 16), HI_SBO, IDESC_64_BMN, 1);
      mma_ss_lohi(tDs, loSel + (2 * WS_KG >> 4), HI_SBO, loLy + ((py0 & 63) >> 3) * 64, HI_SBO, IDESC_64_BMN, 1);
    }
    tc_commit(bar_full + slot);
  };
  auto issue_layer23 = [&](int layer) {          // elected lane only: A = this slot's activations (+ the ones block: bias)
    const uint32_t loW = layer == 0 ? loW2 : loW3, stepW = layer == 0 ? (2 * LBO_64 >> 4) : (2 * LBO_16 >> 4);
    const uint32_t idesc = layer == 0 ? IDESC_64 : IDESC_16;
#pragma unroll
    for (int kc = 0; kc < 4; ++kc)
      if (!((dbg & 4) && kc > 0)) mma_ss_lohi(tDs, loAct + kc * (2 * WS_KG >> 4), HI_SBO, loW + kc * stepW, HI_SBO, idesc, kc > 0);
    if (!(dbg & 4)) mma_ss_lohi(tDs, loOne, HI_SBO, loW + 4 * stepW, HI_SBO, idesc, 1);
    tc_commit(bar_full + slot);
  };

  // ---- prologue: first tile of this slot
  fetch(slot);
  stage(slot);
  tc_fence_before();
  group_sync();
  if (issuer_warp && (unsigned)slot < my_tiles) {
    if (elect_one()) {
      tc_fence_after();
      issue_layer1(slot);
    }
    __syncwarp();
  }
  fetch(slot + WS_SLOTS);
  uint32_t ph = 0;
  for (unsigned i = slot; i < my_tiles; i += WS_SLOTS) {
    const unsigned tile = blockIdx.x + i * gridDim.x;
#pragma unroll 1
    for (int layer = 0; layer < 2; ++layer) {
      group_wait(ph);
      ph ^= 1;
      tc_fence_after();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t acc[16];
        uint32_t hp[8];
        if constexpr (ACC16) {
          tmem_ld8_pack16(tD + 16 * q, acc);
          tc_wait_ld();
#pragma unroll
          for (int k = 0; k < 8; ++k) hp[k] = gelu_poly_pair_sel(k, NPOLY) ? gelu_poly_packed<FMT>(acc[k]) : gelu2x_packed<FMT>(acc[k]);
          *reinterpret_cast<uint4*>(sAct + (2 * q) * WS_KG + roff) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
          *reinterpret_cast<uint4*>(sAct + (2 * q + 1) * WS_KG + roff) = make_uint4(hp[4], hp[5], hp[6], hp[7]);
          continue;
        }
        tmem_ld16(tD + 16 * q, acc);
        tc_wait_ld();
        if (dbg & 2) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            auto v = P::pack(__uint_as_float(acc[2 * k]), __uint_as_float(acc[2 * k + 1]));
            hp[k] = *reinterpret_cast<uint32_t*>(&v);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            hp[k] = gelu_poly_pair_sel(k, NPOLY) ? gelu_poly_pair<FMT>(__uint_as_float(acc[2 * k]), __uint_as_float(acc[2 * k + 1]))
                                                 : gelu2x_pair<FMT>(__uint_as_float(acc[2 * k]), __uint_as_float(acc[2 * k + 1]));
        }
        *reinterpret_cast<uint4*>(sAct + (2 * q) * WS_KG + roff) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
        *reinterpret_cast<uint4*>(sAct + (2 * q + 1) * WS_KG + roff) = make_uint4(hp[4], hp[5], hp[6], hp[7]);
      }
      fence_async_smem();                           // the activations (generic-proxy stores) -> visible to the tensor core
      tc_fence_before();
      group_sync();
      if (issuer_warp) {
        if (elect_one()) {
          tc_fence_after();
          issue_layer23(layer);
        }
        __syncwarp();
      }
    }
    group_wait(ph);
    ph ^= 1;
    tc_fence_after();
    uint32_t acc[16];
    if (cout > 4) tmem_ld16(tD, acc);               // multi-channel outputs (material stacks): up to 16 channels
    else tmem_ld4(tD, acc);
    tc_wait_ld();
    stage(i + WS_SLOTS);                          // operands of this slot's next tile (fetched one tile ago)
    tc_fence_before();
    group_sync();                                 // D has been read and the next operands are staged
    if (issuer_warp && i + WS_SLOTS < my_tiles) {
      if (elect_one()) {
        tc_fence_after();
        issue_layer1(i + WS_SLOTS);
      }
      __syncwarp();
    }
    fetch(i + 2 * WS_SLOTS);
    {
      int px0, py0, bx0, by0;
      tile_origin(tile, px0, py0, bx0, by0);
      const size_t n = (size_t)((uint32_t)bx0 * (uint32_t)g.B[1] + (uint32_t)by0 + out_thread);      // < 2^31 (launcher)
      if constexpr (CO == 3) {
        OutT* o = out + n * 3;
        store_sigmoid(o, __uint_as_float(acc[0]));
        store_sigmoid(o + 1, __uint_as_float(acc[1]));
        store_sigmoid(o + 2, __uint_as_float(acc[2]));
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < cout && !(dbg & 1)) store_sigmoid(out + n * cout + c, __uint_as_float(acc[c]));
        if (cout > 4) {
#pragma unroll
          for (int c = 4; c < 16; ++c)
            if (c < cout) store_sigmoid(out + n * cout + c, __uint_as_float(acc[c]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, WS_TMEM_COLS);
}

// ================================================================================================ grid sources
// Where the general body reads a corner's 12 features.  stage() runs in the CTA prologue and may fill the shared memory
// behind the barriers (the place of the CHAIN modes' chain table: a source that stages never runs in a CHAIN mode),
// start() once after the CTA barrier.  Then node(grid, i) locates node i of G0 (grid 0) or G1 (grid 1), piece(node, q)
// loads what holds the node's features [4q, 4q + 4), and pair(piece, h) is features 4q + 2h, 4q + 2h + 1 as a packed
// 16-bit pair.

// The 16-bit channel-last shadows of both grids in global memory, read with __ldg: every decode_tc_gws_kernel launch.
struct ShadowGeom {
  const uint2* s0;   // shadow of G0, 3 x uint2 per node
  const uint2* s1;   // shadow of G1
  __device__ __forceinline__ void stage(uint8_t*, const DevGeom&, int, int, int) {}
  __device__ __forceinline__ void start() {}
  // CHAIN modes: the shadows of the row's mip, at its offsets in the chain table
  __device__ __forceinline__ ShadowGeom at_mip(const DevMip& m) const { return {s0 + m.s0, s1 + m.s1}; }
  __device__ __forceinline__ const uint2* node(int grid, int i) const { return (grid ? s1 : s0) + 3 * i; }
  __device__ __forceinline__ uint2 piece(const uint2* node, int q) const { return __ldg(node + q); }
  __device__ __forceinline__ uint32_t pair(uint2 v, int h) const { return h ? v.y : v.x; }
};

// Random-access decode of a SMALL model straight from its saved uint8 codes (BASELINE config 4: a 65^3 colour LUT, 1e9
// query points): both grids live in SHARED MEMORY as channel-last codes for the life of the CTA (18^3 + 10^3 nodes x 12
// bytes = 82 KB), so a query's 16 corner reads are shared-memory loads instead of 48 uncoalesced 8-byte global loads —
// with the grids in global memory a tile of 128 queries costs ~6,000 L1 wavefronts (one 32-byte sector per thread and
// load), which is what bounds ShadowGeom at 6 Gquery/s.  The A operand holds the INTEGER codes minus their
// offset (bytes -> exact f16 integers through 0x6400 | b = 1024 + b), and 1 / (2^bits - 1) rides in W1 (pack_weights_kernel
// gscale).  f16 only: the byte trick needs 11 mantissa bits.
struct ResidentCodes {
  const uint8_t* codes0;   // the caller's codes, channel-major [C][z][y][x] (x fastest)
  const uint8_t* codes1;
  int code_off;            // the offset of the codes: the A operand holds code - code_off
  int bytes0;              // shared-memory bytes of G0 (a multiple of 16); G1 follows
  const uint8_t* base;     // set by stage(): both grids in shared memory, channel-last [x][y][z][12]
  __half2 neg;             // set by start(): -(1024 + code_off)

  __device__ __forceinline__ void stage(uint8_t* smem, const DevGeom& g, int dim, int tid, int threads) {
    // read the codes linearly (coalesced), store them channel-last
    for (int which = 0; which < 2; ++which) {
      const uint8_t* src = which == 0 ? codes0 : codes1;
      uint8_t* dstg = which == 0 ? smem : smem + bytes0;
      const int* nn = which == 0 ? g.n0 : g.n1;
      const int nx = nn[0], ny = nn[1], nz = dim == 3 ? nn[2] : 1;
      const int plane = nx * ny * nz;
      for (int i = tid; i < 12 * plane; i += threads) {
        const int c = i / plane, r = i - c * plane;               // r = (z * ny + y) * nx + x
        const int x = r % nx, yz = r / nx, y = yz % ny, z = yz / ny;
        dstg[((x * ny + y) * nz + z) * 12 + c] = __ldg(src + i);
      }
    }
    base = smem;
  }
  __device__ __forceinline__ void start() { neg = __float2half2_rn(-(1024.0f + (float)code_off)); }
  __device__ __forceinline__ const uint32_t* node(int grid, int i) const {
    return reinterpret_cast<const uint32_t*>((grid ? base + bytes0 : base) + 12 * i);
  }
  // code word q of the node; its pair h: code bytes 2h, 2h + 1 -> a packed pair of exact f16 integers (code - offset)
  __device__ __forceinline__ uint32_t piece(const uint32_t* node, int q) const { return node[q]; }
  __device__ __forceinline__ uint32_t pair(uint32_t w, int h) const {
    const uint32_t v = __byte_perm(w, 0x64646464u, h ? 0x5342 : 0x5140);
    const __half2 p = __hadd2(*reinterpret_cast<const __half2*>(&v), neg);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};

// ================================================================================================ general kernel, v2
// The general decode (any mip / origin / block shape, 2-D and both 3-D methods, random-access queries) in the same
// warp-specialised form as decode_tc2d_ws_kernel: ONE persistent CTA per SM made of NG independent groups of 4 warps
// (NG = 8 for a decoder input of <= 80 columns, 5 for method 3's 128), group s owning TMEM columns [64 s, +64) and one
// [128 x KX] operand buffer in shared memory.  A group's thread = one texel of its tile:
//   gather : the texel's decoder-input row goes STRAIGHT from the grid source to the operand buffer — a G0 corner is
//            three 8-byte pieces and three 8-byte shared stores, G1 is interpolated in packed 16-bit math (6 registers),
//            the triangular PE comes from a shared LUT — so no thread ever holds the row;
//   layers : SS-form tcgen05.mma issued by the group's elected lane after a 128-thread named barrier (layer 1: KX/16
//            MMAs; layers 2, 3: 4 MMAs + 1 bias MMA against a shared constant ones block), the epilogue overwrites the
//            operand buffer with the next layer's activations;  the groups never meet at a CTA-wide barrier.
// TAPS > 0 (nic_sample: 4 in 2-D, 8 in 3-D): row n is tap n % TAPS of query n / TAPS, its texel comes from the query's
// coordinates (sample_tap); the TAPS rows of a query are adjacent lanes of one warp, which blend their weighted sigmoid
// outputs with a shuffle butterfly before tap 0 stores the query.  TAPS = 0 is the plain decode.
// TAPS = 2 * 2^D (nic_sample_lod, 8 in 2-D, 16 in 3-D): every query carries its own LOD; its first 2^D rows are the taps at
// mip m, the next 2^D the taps at mip min(m + 1, L).  Each lane computes its query's lambda and from it its row's mip; what
// varies by mip (nodes, shadow-grid offsets, step, interpolation, extent) comes from the chain table, which `origins`
// points at and the CTA copies to shared memory (lanes of a warp read different mips).  The mip is a decoder input
// (column CIN - 1; the bias moves to column CIN), one PE LUT built at step 1/4 serves every mip, and the two halves of a
// query blend after their butterflies.
// TAPS = TAPS_MIPS (nic_decode_mips): the dense chain.  Row n is a texel of the mip whose first row (DevMipRows::row0, in
// shared memory behind the chain table) is the largest one <= n, at index n - row0 inside that mip, x slowest.  Everything
// that varies by mip comes from the chain table as in the per-query-LOD mode, and so do the mip column and the step-1/4 PE
// LUT; the epilogue is TAPS = 0's: each row stores its own output row.  Tiles may straddle mips, so small mips share tiles.
constexpr int GW_GROUP = 128;
constexpr int TAPS_MIPS = -1;

// NGT / LUTCAP: groups per CTA and capacity of the positional-encoding LUT.  The defaults (8 groups, or 5 for method 3's
// 32 KB operand buffers, 256 LUT entries) always fit; with a 64-entry LUT (step >= 1/4: every full-resolution decode) a
// SIXTH 32 KB group fits the 227 KB of shared memory for method 3 (225.8 KB), 20 % more tiles in flight.
constexpr int gws_groups(int kx, int ngt) { return ngt ? ngt : (kx > 80 ? 5 : 8); }
template <int METHOD, int FMT, int NPOLY, int NGT, int LUTCAP, int TAPS, typename OutT, class Grids>
__device__ __forceinline__ void decode_tc_gws_body(const DevGeom& g, Grids grids, const long long* origins, const uint4* wimg,
                                                   int cout, int lut_n, OutT* out, const DevSampler& smp) {
  using S = RowShape<METHOD>;
  using P = Pair<FMT>;
  constexpr int KX = S::KX, NG = gws_groups(KX, NGT), THREADS = NG * GW_GROUP;
  constexpr int W1_BYTES = b_image_bytes(64, KX), W2_BYTES = b_image_bytes(64, TC_K2), W3_BYTES = b_image_bytes(16, TC_K2);
  constexpr int KG = 16 * 128;                       // bytes of one k-group (8 columns) of a 128-row K-major operand
  constexpr int OFF_LUT = W1_BYTES + W2_BYTES + W3_BYTES, OFF_ONE = OFF_LUT + LUTCAP * 16, OFF_ACT = OFF_ONE + 2 * KG;
  constexpr int ACT_BYTES = (KX / 8) * KG, OFF_BAR = OFF_ACT + NG * ACT_BYTES;
  constexpr bool LODQ = TAPS == (2 << S::DIM);
  constexpr bool DENSE = TAPS == TAPS_MIPS;
  constexpr bool CHAIN = LODQ || DENSE;              // per-row mip from the chain table
  constexpr int TQ = LODQ ? TAPS / 2 : TAPS;         // taps of one mip
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const DevChain* sChain = reinterpret_cast<const DevChain*>(smem_raw + OFF_BAR + 256);     // CHAIN only
  const unsigned* sRow0 = reinterpret_cast<const DevMipRows*>(sChain)->row0;                // DENSE only
  uint8_t* sW1 = smem_raw;
  uint8_t* sW2 = sW1 + W1_BYTES;
  uint8_t* sW3 = sW2 + W2_BYTES;
  uint4* sLut = reinterpret_cast<uint4*>(smem_raw + OFF_LUT);
  uint8_t* sOne = smem_raw + OFF_ONE;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem_raw + OFF_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_full + NG);

  const int tid = threadIdx.x, warp = uniform_warp_index(), lane = tid & 31;     // warp: provably uniform (MMA operands)
  const int slot = warp >> 2;
  const int row = 32 * (warp & 3) + lane;
  const int roff = (row >> 3) * 128 + (row & 7) * 16;
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 0)
    for (int s = 0; s < NG; ++s) mbar_init(bar_full + s, 1);
  {
    uint4* dst = reinterpret_cast<uint4*>(smem_raw);
    for (int i = tid; i < OFF_LUT / 16; i += THREADS) dst[i] = __ldg(wimg + i);
    for (int i = tid; i < lut_n; i += THREADS) {
      float u1 = __fmul_rn(__fmul_rn((float)i, CHAIN ? 0.25f : g.step), 0.5f);
      uint4 e;
      auto v0 = P::pack(pe_triangular(u1, 0, 6), pe_triangular(u1, 1, 6));
      auto v1 = P::pack(pe_triangular(u1, 2, 6), pe_triangular(u1, 3, 6));
      auto v2 = P::pack(pe_triangular(u1, 4, 6), pe_triangular(u1, 5, 6));
      e.x = *reinterpret_cast<uint32_t*>(&v0);
      e.y = *reinterpret_cast<uint32_t*>(&v1);
      e.z = *reinterpret_cast<uint32_t*>(&v2);
      e.w = 0u;
      sLut[i] = e;
    }
    if constexpr (CHAIN) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(origins);
      uint32_t* cdst = reinterpret_cast<uint32_t*>(smem_raw + OFF_BAR + 256);
      for (int i = tid; i < (int)((LODQ ? sizeof(DevChain) : sizeof(DevMipRows)) / 4); i += THREADS) cdst[i] = __ldg(src + i);
    }
    if (slot == 0) {
      auto one = P::pack(1.0f, 0.0f);
      *reinterpret_cast<uint4*>(sOne + roff) = make_uint4(*reinterpret_cast<uint32_t*>(&one), 0, 0, 0);
      *reinterpret_cast<uint4*>(sOne + KG + roff) = make_uint4(0, 0, 0, 0);
    }
    grids.stage(smem_raw + OFF_BAR + 256, g, S::DIM, tid, THREADS);
  }
  fence_async_smem();
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tDs = tmem + slot * 64;
  const uint32_t tD = tDs + ((uint32_t)((warp & 3) * 32) << 16);
  uint8_t* sAct = smem_raw + OFF_ACT + slot * ACT_BYTES;
  // the group's issuing (and polling) warp: a different lane quarter for consecutive groups, so the eight issuers are
  // spread over the four SM sub-partitions (warp % 4) instead of all sitting on sub-partition 0
  const bool issuer_warp = (warp & 3) == (slot & 3);
  constexpr bool ACC16 = FMT == 0;                    // f16 operands: 16-bit accumulators for the hidden layers (see above)
  constexpr uint32_t IDESC_64 = make_idesc(FMT, 128, 64, 0, ACC16), IDESC_16 = make_idesc(FMT, 128, 16);
  constexpr uint32_t LBO_64 = (64 / 8) * 128, LBO_16 = (16 / 8) * 128, SBO = 128;
  const uint32_t aW1 = smem_u32(sW1), aW2 = smem_u32(sW2), aW3 = smem_u32(sW3), aOne = smem_u32(sOne), aAct = smem_u32(sAct);
  auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + slot), "n"(GW_GROUP) : "memory"); };
  auto group_wait = [&](uint32_t phase) {          // one polling warp per group, the others park at the named barrier
    if (issuer_warp) mbar_wait(bar_full + slot, phase);
    group_sync();
  };
  constexpr uint32_t HI_SBO = smem_desc_hi(SBO);      // descriptors as 32-bit halves (mma_ss_lohi)
  const uint32_t loAct = smem_desc_lo(aAct, KG), loOne = smem_desc_lo(aOne, KG);
  const uint32_t loW1 = smem_desc_lo(aW1, LBO_64), loW2 = smem_desc_lo(aW2, LBO_64), loW3 = smem_desc_lo(aW3, LBO_16);
  // this thread's 8-byte piece holding features [f, f + 4) of its row (f a multiple of 4)
  auto piece = [&](int f) -> uint2* { return reinterpret_cast<uint2*>(sAct + (f >> 3) * KG + roff + (f & 7) * 2); };
  grids.start();

  const unsigned ntiles = (unsigned)((g.N + TC_ROWS - 1) / TC_ROWS);
  const int lut_mask = lut_n - 1;
  uint32_t ph = 0;
  for (unsigned tile = blockIdx.x + gridDim.x * slot; tile < ntiles; tile += gridDim.x * NG) {
    const unsigned n = tile * TC_ROWS + row;
    const bool live = n < (unsigned)g.N;
    float tap_w = 0.f;                               // TAPS > 0: this row's filter weight (0 on dead rows)
    float lod_t = 0.f;                               // LODQ: the query's weight of mip m + 1
    int row_mip = 0;                                 // CHAIN: this row's mip and its entry of the chain table
    const DevMip* mp = nullptr;
    // ------------------------------------------------------------------------------------ gather -> operand buffer
    {
      Texel t;
      if constexpr (TAPS > 0) {
        const unsigned q = (live ? n : (unsigned)g.N - 1) / TAPS;
        float u[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int a = 0; a < S::DIM; ++a) u[a] = __ldg(smp.coords + (size_t)q * S::DIM + a);
        if constexpr (LODQ) {
          const float lc = lod_clamped(*sChain, q);
          const int m = (int)floorf(lc);
          lod_t = __fsub_rn(lc, (float)m);
          row_mip = min(m + (row % TAPS >= TQ), sChain->num_mips - 1);
          mp = &sChain->mip[row_mip];
          DevSampler sm = smp;
#pragma unroll
          for (int a = 0; a < 3; ++a) sm.S[a] = mp->S[a];
          const float w = sample_tap(sm, S::DIM, u, row % TQ, t.p);
          tap_w = live ? w : 0.f;
        } else {
          const float w = sample_tap(smp, S::DIM, u, row % TAPS, t.p);
          tap_w = live ? w : 0.f;
        }
      } else if constexpr (DENSE) {
        const unsigned r = live ? n : (unsigned)g.N - 1;
#pragma unroll
        for (int i = 1; i < NIC_MAX_MIPS; ++i) row_mip += r >= sRow0[i];
        mp = &sChain->mip[row_mip];
        const unsigned idx = r - sRow0[row_mip];     // x slowest: ((ix * Sy) + iy) * Sz + iz
        const unsigned yz = (unsigned)mp->S[1] * (unsigned)mp->S[2];
        const unsigned ix = idx / yz, r2 = idx - ix * yz;
        const unsigned iy = S::DIM == 3 ? r2 / (unsigned)mp->S[2] : r2;
        t.b = 0;
        t.p[0] = (int)ix;
        t.p[1] = (int)iy;
        t.p[2] = S::DIM == 3 ? (int)(r2 - iy * (unsigned)mp->S[2]) : 0;
      } else {
        t = texel_of_fast(g, live ? n : (unsigned)g.N - 1, origins);
      }
      const int* n0 = CHAIN ? mp->n0 : g.n0;
      const int* n1 = CHAIN ? mp->n1 : g.n1;
      Grids src = grids;
      if constexpr (CHAIN) src = grids.at_mip(*mp);
      AxisCoord ax[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        ax[a] = axis_coord(t.p[a], CHAIN ? mp->step : g.step);
        ax[a].i0 = clampi(ax[a].i0, 0, n0[a] - 2 < 0 ? 0 : n0[a] - 2);
        ax[a].i1 = clampi(ax[a].i1, 0, n1[a] - 2 < 0 ? 0 : n1[a] - 2);
      }
#pragma unroll
      for (int j = 0; j < S::NC0; ++j) {             // G0 corners: the source's pairs, unweighted
        const int8_t* d = S::DIM == 2 ? kCorner2D[j] : (METHOD == NIC_METHOD_3D ? kCorner3D[j] : kCorner3Dv2[j]);
        const int dz = S::DIM == 3 ? d[0] : 0;
        const auto node = src.node(0, node_lin(n0, S::DIM, ax[0].i0 + d[2], ax[1].i0 + d[1], ax[2].i0 + dz));
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const auto v = src.piece(node, q);
          *piece(12 * j + 4 * q) = make_uint2(src.pair(v, 0), src.pair(v, 1));
        }
      }
      typename P::T2 acc[6];                          // G1: weighted sum of corners
#pragma unroll
      for (int j = 0; j < S::NC1; ++j) {
        const int8_t* d = S::DIM == 2 ? kCorner2D[j] : kCorner3D[j];
        const int dz = S::DIM == 3 ? d[0] : 0;
        const auto node = src.node(1, node_lin(n1, S::DIM, ax[0].i1 + d[2], ax[1].i1 + d[1], ax[2].i1 + dz));
        float f[3];
        g1_factors(g, j, ax, f);
        if constexpr (CHAIN) {
          if (!mp->interp) f[0] = f[1] = f[2] = 1.0f;
        }
        float w = f[0] * f[1];
        if (S::DIM == 3) w *= f[2];
        typename P::T2 w2 = P::cst(w);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const auto v = src.piece(node, q);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t pr = src.pair(v, h);
            typename P::T2 vh = *reinterpret_cast<typename P::T2*>(&pr);
            acc[2 * q + h] = j == 0 ? __hmul2(vh, w2) : __hfma2(vh, w2, acc[2 * q + h]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 3; ++q)
        *piece(12 * S::NC0 + 4 * q) = make_uint2(*reinterpret_cast<uint32_t*>(&acc[2 * q]), *reinterpret_cast<uint32_t*>(&acc[2 * q + 1]));
      // positional encoding (3 pairs per axis), the bias carrier (feature CIN - 1 = 1) and zero padding up to KX: the
      // tail of the row, [12 (NC0 + 1), KX), is assembled as packed pairs and stored in 8-byte pieces
      constexpr int T0 = 12 * (S::NC0 + 1), NTAIL = (KX - T0) / 2;      // pairs in the tail
      uint32_t tail[NTAIL];
#pragma unroll
      for (int i = 0; i < NTAIL; ++i) tail[i] = 0u;
#pragma unroll
      for (int a = 0; a < S::DIM; ++a) {
        if (g.pe_kind == NIC_PE_TRIANGULAR) {
          uint4 e = sLut[CHAIN ? ((t.p[a] << mp->lut_shift) & 63) : (t.p[a] & lut_mask)];
          tail[3 * a] = e.x;
          tail[3 * a + 1] = e.y;
          tail[3 * a + 2] = e.z;
        } else {
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            float arg = __fmul_rn(ax[a].u1, g.pe_div[q]);
            auto v = P::pack(sinf(arg), cosf(arg));
            tail[3 * a + q] = *reinterpret_cast<uint32_t*>(&v);
          }
        }
      }
      {
        auto one = P::pack(CHAIN ? (float)row_mip : 1.0f, CHAIN ? 1.0f : 0.0f);   // CHAIN: [... | pe | mip | 1]
        tail[(S::CIN - 1 - T0) / 2] = *reinterpret_cast<uint32_t*>(&one);
      }
#pragma unroll
      for (int i = 0; i < NTAIL / 2; ++i) *piece(T0 + 4 * i) = make_uint2(tail[2 * i], tail[2 * i + 1]);
    }
    fence_async_smem();
    tc_fence_before();
    group_sync();
    if (issuer_warp) {
      if (elect_one()) {
        tc_fence_after();
#pragma unroll
        for (int kc = 0; kc < KX / 16; ++kc)
          mma_ss_lohi(tDs, loAct + kc * (2 * KG >> 4), HI_SBO, loW1 + kc * (2 * LBO_64 >> 4), HI_SBO, IDESC_64, kc > 0);
        tc_commit(bar_full + slot);
      }
      __syncwarp();
    }
    // ------------------------------------------------------------------------------------ layers 1, 2: epilogues
#pragma unroll 1
    for (int layer = 0; layer < 2; ++layer) {
      group_wait(ph);
      ph ^= 1;
      tc_fence_after();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t acc[16];
        uint32_t hp[8];
        if constexpr (ACC16) {
          tmem_ld8_pack16(tD + 16 * q, acc);
          tc_wait_ld();
#pragma unroll
          for (int k = 0; k < 8; ++k) hp[k] = gelu_poly_pair_sel(k, NPOLY) ? gelu_poly_packed<FMT>(acc[k]) : gelu2x_packed<FMT>(acc[k]);
          *reinterpret_cast<uint4*>(sAct + (2 * q) * KG + roff) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
          *reinterpret_cast<uint4*>(sAct + (2 * q + 1) * KG + roff) = make_uint4(hp[4], hp[5], hp[6], hp[7]);
          continue;
        }
        tmem_ld16(tD + 16 * q, acc);
        tc_wait_ld();
#pragma unroll
        for (int k = 0; k < 8; ++k)
          hp[k] = gelu_poly_pair_sel(k, NPOLY) ? gelu_poly_pair<FMT>(__uint_as_float(acc[2 * k]), __uint_as_float(acc[2 * k + 1]))
                                               : gelu2x_pair<FMT>(__uint_as_float(acc[2 * k]), __uint_as_float(acc[2 * k + 1]));
        *reinterpret_cast<uint4*>(sAct + (2 * q) * KG + roff) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
        *reinterpret_cast<uint4*>(sAct + (2 * q + 1) * KG + roff) = make_uint4(hp[4], hp[5], hp[6], hp[7]);
      }
      fence_async_smem();
      tc_fence_before();
      group_sync();
      if (issuer_warp) {
        if (elect_one()) {
          tc_fence_after();
          const uint32_t loW = layer == 0 ? loW2 : loW3, stepW = layer == 0 ? (2 * LBO_64 >> 4) : (2 * LBO_16 >> 4);
          const uint32_t idesc = layer == 0 ? IDESC_64 : IDESC_16;
#pragma unroll
          for (int kc = 0; kc < 4; ++kc)
            mma_ss_lohi(tDs, loAct + kc * (2 * KG >> 4), HI_SBO, loW + kc * stepW, HI_SBO, idesc, kc > 0);
          mma_ss_lohi(tDs, loOne, HI_SBO, loW + 4 * stepW, HI_SBO, idesc, 1);
          tc_commit(bar_full + slot);
        }
        __syncwarp();
      }
    }
    // ------------------------------------------------------------------------------------ output
    group_wait(ph);
    ph ^= 1;
    tc_fence_after();
    uint32_t acc[16];
    if (cout > 4) tmem_ld16(tD, acc);
    else tmem_ld4(tD, acc);
    tc_wait_ld();
    tc_fence_before();
    if constexpr (TAPS > 0) {
      // weighted taps, reduced over the TAPS lanes of the query in a fixed butterfly order (every lane takes part: the
      // shuffles run before the live test); tap 0 applies the optional mip blend and stores, quantising once
      float v[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) v[c] = (c < cout) ? __fmul_rn(tap_w, sigmoid_tanh(__uint_as_float(acc[c]))) : 0.f;
#pragma unroll
      for (int msk = 1; msk < TQ; msk <<= 1) {
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = __fadd_rn(v[c], __shfl_xor_sync(0xffffffffu, v[c], msk));
        if (cout > 4) {
#pragma unroll
          for (int c = 4; c < 16; ++c) v[c] = __fadd_rn(v[c], __shfl_xor_sync(0xffffffffu, v[c], msk));
        }
      }
      if constexpr (LODQ) {                           // tap 0 holds S_m, tap TQ S_m1: tap 0 blends (1 - t) * S_m + t * S_m1
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = lod_blend(lod_t, v[c], __shfl_xor_sync(0xffffffffu, v[c], TQ));
        if (cout > 4) {
#pragma unroll
          for (int c = 4; c < 16; ++c) v[c] = lod_blend(lod_t, v[c], __shfl_xor_sync(0xffffffffu, v[c], TQ));
        }
      }
      if (live && row % TAPS == 0) {
        const size_t o = (size_t)(n / TAPS) * cout;
#pragma unroll
        for (int c = 0; c < 16; ++c)
          if (c < cout) store_out(out + o + c, LODQ ? v[c] : sample_blend_prev(smp, (long long)(o + c), v[c]));
      }
    } else if (live) {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < cout) store_sigmoid(out + (size_t)n * cout + c, __uint_as_float(acc[c]));
      if (cout > 4) {
#pragma unroll
        for (int c = 4; c < 16; ++c)
          if (c < cout) store_sigmoid(out + (size_t)n * cout + c, __uint_as_float(acc[c]));
      }
    }
    // (every thread passes its own tcgen05.wait::ld above before it reaches the next tile's pre-MMA barrier, so the next
    //  layer-1 MMAs cannot overwrite D early)
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// The general kernel: the grids come from their 16-bit shadows in global memory.
template <int METHOD, int FMT, typename OutT, int NPOLY, int NGT = 0, int LUTCAP = TC_LUT_MAX, int TAPS = 0>
__global__ void __launch_bounds__(gws_groups(RowShape<METHOD>::KX, NGT) * GW_GROUP, 1)
    decode_tc_gws_kernel(DevGeom g, ShadowGeom sg, const long long* __restrict__ origins, const uint4* __restrict__ wimg,
                         int cout, int lut_n, OutT* __restrict__ out, DevSampler smp) {
  decode_tc_gws_body<METHOD, FMT, NPOLY, NGT, LUTCAP, TAPS>(g, sg, origins, wimg, cout, lut_n, out, smp);
}

// Code-resident queries: the general body on random-access queries with both grids resident in shared memory as codes
// (ResidentCodes), f16, three groups (the grids take the shared memory of the others).
constexpr int CQ_NG = 3;
template <int METHOD, typename OutT, int NPOLY>
__global__ void __launch_bounds__(CQ_NG * GW_GROUP, 1)
    decode_codes_smem_kernel(DevGeom g, const uint8_t* __restrict__ codes0, const uint8_t* __restrict__ codes1, int code_off,
                             int bytes0, const long long* __restrict__ origins, const uint4* __restrict__ wimg, int cout,
                             int lut_n, OutT* __restrict__ out) {
  decode_tc_gws_body<METHOD, 0, NPOLY, CQ_NG, TC_LUT_MAX, 0>(g, ResidentCodes{codes0, codes1, code_off, bytes0}, origins,
                                                            wimg, cout, lut_n, out, DevSampler{});
}

// ------------------------------------------------------------------------------------------------ launcher
// NIC_OPT_REUSE_PREPARED: what the tables of a call are built from.  gm, g0 and g1 hold num_mips entries.
static Handle::PreparedKey make_key(int kind, int fmt, int code_bits, int npoly, const MlpDev& m, const DevGeom* gm,
                                    const void* const* g0, const void* const* g1, int num_mips) {
  Handle::PreparedKey k;
  memset(&k, 0, sizeof(k));                            // (padding included: keys are compared with memcmp)
  k.kind = kind; k.fmt = fmt; k.code_bits = code_bits; k.npoly = npoly;
  k.method = gm[0].method; k.pe_kind = gm[0].pe_kind; k.mip = gm[0].mip; k.num_mips = num_mips;
  k.w1 = m.w1; k.b1 = m.b1; k.w2 = m.w2; k.b2 = m.b2; k.w3 = m.w3; k.b3 = m.b3;
  for (int i = 0; i < num_mips; ++i) {
    Handle::PreparedKey::Mip& p = k.mips[i];
    p.g0 = g0[i];
    p.g1 = g1[i];
    memcpy(p.n0, gm[i].n0, sizeof(p.n0));
    memcpy(p.n1, gm[i].n1, sizeof(p.n1));
    p.step = gm[i].step;
  }
  return k;
}
// Runs build() (NIC_OK or an error) unless reuse is on and the tables already describe `key`; the key is kept only when
// the build succeeds.
template <class Build>
static int prepare_tables(Handle* h, const Handle::PreparedKey& key, Build&& build) {
  if (h->reuse_prepared && memcmp(&h->prepared, &key, sizeof(key)) == 0) return NIC_OK;
  invalidate_prepared(h);
  const int rc = build();
  if (rc == NIC_OK) memcpy(&h->prepared, &key, sizeof(key));
  return rc;
}

// How many of every 8 activation pairs take the polynomial (FMA-pipe) GELU instead of MUFU.TANH: tuned per format so that
// the XU and FMA pipes finish together (profiles/r02*); NIC_OPT_GELU_POLY overrides it for A/B runs.
static int resolve_npoly(const Handle* h, int fmt) {
  return h->gelu_poly >= 0 ? h->gelu_poly : (fmt == 0 ? WS_NPOLY_F16 : WS_NPOLY_BF16);
}

// Positional-encoding LUT length, or NIC_ERR_UNSUPPORTED: the triangular encoding has period 16/step texels.
static int pe_lut_len(const DevGeom& g) {
  const float period = 16.0f / g.step;
  int n = 1;
  while (n < period && n < TC_LUT_MAX) n <<= 1;
  return g.pe_kind == NIC_PE_TRIANGULAR && (float)n < period ? NIC_ERR_UNSUPPORTED : n;
}

// Dynamic shared memory of decode_tc_gws_body with NG groups and a LUTCAP-entry LUT: weight images, LUT, ones block,
// operand buffers, barriers, and behind them the `table` bytes of the chain table of a per-query-LOD (DevChain) or dense-chain
// (DevMipRows) launch.  With ResidentCodes (CQ_NG groups) the two grids take that place instead.
template <int METHOD>
constexpr int gws_smem(int ng, int lutcap, size_t table = 0) {
  using S = RowShape<METHOD>;
  return b_image_bytes(64, S::KX) + b_image_bytes(64, TC_K2) + b_image_bytes(16, TC_K2) + lutcap * 16 + 2 * 2048 +
         ng * (S::KX / 8) * 2048 + 256 + (int)((table + 15) & ~(size_t)15);
}

// One launch of a persistent tensor-core kernel: at most one CTA per SM for `units` work units (tiles or tile groups).
template <typename... KArgs, typename... Args>
static int launch_persistent(Handle* h, void (*kern)(KArgs...), long long units, int threads, int smem, cudaStream_t st,
                             const Args&... args) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return (int)e;
  {
    KernelTimer timer(h, st);
    kern<<<(int)(units < h->sms ? units : h->sms), threads, smem, st>>>(args...);
  }
  h->launches++;
  return (int)cudaGetLastError();
}

static bool fast2d_eligible(const DevGeom& g, const long long* origins) {
  return g.method == NIC_METHOD_2D && g.step == 0.25f && g.interp && g.pe_kind == NIC_PE_TRIANGULAR && !origins &&
         g.nblocks == 1 && g.B[0] % F_TX == 0 && g.B[1] % F_TY == 0 && g.origin0[0] % F_TX == 0 &&
         g.origin0[1] % F_TY == 0 && g.B[0] > 0 && g.B[1] > 0;
}

// Random-access queries (1-texel blocks) on a model given as uint8 codes whose two grids fit shared memory next to three
// operand buffers: the code-resident kernel.
static long long codes_bytes(const int* nodes, int dim) { return (plane_size_host(nodes, dim) * 12 + 15) & ~15ll; }
template <int METHOD>
static long long codes_smem(const DevGeom& g) {
  return gws_smem<METHOD>(CQ_NG, TC_LUT_MAX) + codes_bytes(g.n0, g.dim) + codes_bytes(g.n1, g.dim);
}
template <int METHOD>
static bool codes_smem_eligible(const DevGeom& g, int bits, const long long* origins) {
  return bits >= 1 && bits <= 8 && origins && g.per_block == 1 && codes_smem<METHOD>(g) <= 227 * 1024;
}

template <int METHOD, typename OutT>
static int launch_codes_smem(Handle* h, const DevGeom& g, const MlpDev& m, const void* c0, const void* c1, int bits,
                             const long long* origins, OutT* out, cudaStream_t st) {
  using S = RowShape<METHOD>;
  int rc = tc_scratch(h, 0);
  if (rc) return rc;
  const int npoly = resolve_npoly(h, 0);
  rc = prepare_tables(h, make_key(PREP_CODES, 0, bits, npoly, m, &g, &c0, &c1, 1), [&] {
    pack_weights_kernel<0><<<16, 256, 0, st>>>(m, g.lod, S::KX, (uint16_t*)h->tc_weights, npoly, 12 * (S::NC0 + 1),
                                               1.0f / (float)((1 << bits) - 1));
    h->launches++;
    return (int)cudaGetLastError();
  });
  if (rc) return rc;
  const int lut_n = pe_lut_len(g);
  if (lut_n < 0) return lut_n;
  if (g.N >= (1ll << 31) - TC_ROWS) return NIC_ERR_UNSUPPORTED;
  void (*kern)(DevGeom, const uint8_t*, const uint8_t*, int, int, const long long*, const uint4*, int, int, OutT*) = nullptr;
  switch (npoly) {
    case 0: kern = decode_codes_smem_kernel<METHOD, OutT, 0>; break;
    case 3: kern = decode_codes_smem_kernel<METHOD, OutT, 3>; break;
    default: return NIC_ERR_UNSUPPORTED;
  }
  const long long ntiles = (g.N + TC_ROWS - 1) / TC_ROWS;
  return launch_persistent(h, kern, (ntiles + CQ_NG - 1) / CQ_NG, CQ_NG * GW_GROUP, (int)codes_smem<METHOD>(g), st, g,
                           (const uint8_t*)c0, (const uint8_t*)c1, (1 << (bits - 1)) - 1, (int)codes_bytes(g.n0, g.dim),
                           origins, (const uint4*)h->tc_weights, m.cout, lut_n, out);
}

// Bytes of tc_shadow the fast path's tables take: the G0 shadow (b0, rounded to 256 bytes), then R (b1).
static void fast2d_table_bytes(const DevGeom& g, size_t* b0, size_t* b1) {
  *b0 = ((size_t)plane_size_host(g.n0, 2) * g.C * 2 + 255) & ~(size_t)255;
  *b1 = (size_t)plane_size_host(g.n1, 2) * 128;
}

template <int FMT, typename OutT>
static int launch_fast2d(Handle* h, const DevGeom& g, const MlpDev& m, const void* g0, const void* g1, int code_bits,
                         OutT* out, cudaStream_t st) {
  size_t b0, b1;
  fast2d_table_bytes(g, &b0, &b1);
  int rc = tc_scratch(h, b0 + b1);
  if (rc) return rc;
  uint16_t* s0 = (uint16_t*)h->tc_shadow;
  uint16_t* R = (uint16_t*)((uint8_t*)h->tc_shadow + b0);
  const int npoly = resolve_npoly(h, FMT);
  rc = prepare_tables(h, make_key(PREP_FAST2D, FMT, code_bits, npoly, m, &g, &g0, &g1, 1), [&] {
    const int e = launch_relayout<FMT>(h, g, g0, code_bits, g.n0, s0, st);
    if (e) return e;
    const long long tiles_r = (long long)((g.n1[0] + G1R_TX - 1) / G1R_TX) * ((g.n1[1] + G1R_TY - 1) / G1R_TY);
    const long long cap_r = 2ll * h->sms;
    g1_rows_kernel<FMT><<<(int)(tiles_r < cap_r ? tiles_r : cap_r), 256, 0, st>>>(m, (const float*)g1, g.n1[0], g.n1[1], R,
                                                                                 code_bits);
    pack_fast_kernel<FMT><<<32, 256, 0, st>>>(m, g.lod, g.step, (uint16_t*)h->tc_weights, npoly);
    h->launches += 2;
    return (int)cudaGetLastError();
  });
  if (rc) return rc;
  unsigned tiles_y = (unsigned)(g.B[1] / F_TY);
  long long ntiles = (long long)(g.B[0] / F_TX) * tiles_y;
  if (ntiles >= (1ll << 31) || g.N >= (1ll << 31)) return NIC_ERR_UNSUPPORTED;     // 32-bit texel index in the kernel
  unsigned sh = 0;
  while ((1ull << sh) < tiles_y) ++sh;
  unsigned mul = (unsigned)(((1ull << (31 + sh)) + tiles_y - 1) / tiles_y);
  // warp-specialised persistent kernel: one CTA per SM (all 512 TMEM columns)
  static_assert(WS_SMEM <= 227 * 1024, "shared memory budget");
  if (b0 >= (1ull << 32) || b1 >= (1ull << 32)) return NIC_ERR_UNSUPPORTED;          // 32-bit table offsets in the kernel
  void (*kern)(DevGeom, const uint2*, const uint4*, const uint4*, int, unsigned, unsigned, unsigned, OutT*, int) = nullptr;
  const bool rgb = m.cout == 3 && h->debug_flags == 0;       // the specialised instance; anything else takes the generic one
  switch (npoly) {
    case 0: kern = decode_tc2d_ws_kernel<FMT, OutT, 0, 0>; break;
    case 3: kern = rgb ? decode_tc2d_ws_kernel<FMT, OutT, 3, 3> : decode_tc2d_ws_kernel<FMT, OutT, 3, 0>; break;
#ifdef NIC_GELU_SWEEP
    case 2: kern = decode_tc2d_ws_kernel<FMT, OutT, 2, 0>; break;
    case 4: kern = decode_tc2d_ws_kernel<FMT, OutT, 4, 0>; break;
    case 5: kern = decode_tc2d_ws_kernel<FMT, OutT, 5, 0>; break;
    case 6: kern = decode_tc2d_ws_kernel<FMT, OutT, 6, 0>; break;
    case 8: kern = decode_tc2d_ws_kernel<FMT, OutT, 8, 0>; break;
#endif
    default: return NIC_ERR_UNSUPPORTED;
  }
  return launch_persistent(h, kern, ntiles, WS_THREADS, WS_SMEM, st, g, (const uint2*)s0, (const uint4*)R,
                           (const uint4*)h->tc_weights, m.cout, tiles_y, mul, sh, out, h->debug_flags);
}

// TAPS > 0: filtered sampling (smp set, g.N = queries * TAPS rows) always runs on the general kernel: the fast 2-D kernel
// has no per-row texel and no tap epilogue, and the code-resident kernel is built for TAPS = 0 only.
template <int METHOD, int FMT, int TAPS, typename OutT>
static int launch_tc_t(Handle* h, const DevGeom& g, const MlpDev& m, const void* g0, const void* g1, int code_bits,
                       const long long* origins, OutT* out, cudaStream_t st, const DevSampler& smp = DevSampler{}) {
  using S = RowShape<METHOD>;
  if constexpr (METHOD == NIC_METHOD_2D && TAPS == 0) {
    if (fast2d_eligible(g, origins) && !h->disable_fast2d) return launch_fast2d<FMT, OutT>(h, g, m, g0, g1, code_bits, out, st);
  }
  if constexpr (METHOD == NIC_METHOD_3D && FMT == 0 && TAPS == 0) {       // small models given as codes, random-access queries
    if (codes_smem_eligible<METHOD>(g, code_bits, origins) && !h->disable_fast2d)
      return launch_codes_smem<METHOD, OutT>(h, g, m, g0, g1, code_bits, origins, out, st);
  }
  const int npoly = resolve_npoly(h, FMT);
  if (npoly != 0 && npoly != 3) return NIC_ERR_UNSUPPORTED;      // (the NIC_GELU_SWEEP values exist for the fast 2-D kernel only)
  const ShadowLayout sl = shadow_layout(&g, &g0, &g1, 1);
  int rc = tc_scratch(h, sl.total);
  if (rc) return rc;
  rc = prepare_tables(h, make_key(PREP_GENERAL, FMT, code_bits, npoly, m, &g, &g0, &g1, 1), [&] {
    const int e = build_shadows<FMT>(h, sl, &g, &g0, &g1, code_bits, st);
    if (e) return e;
    pack_weights_kernel<FMT><<<16, 256, 0, st>>>(m, g.lod, S::KX, (uint16_t*)h->tc_weights, npoly);
    h->launches++;
    return (int)cudaGetLastError();
  });
  if (rc) return rc;
  const int lut_n = pe_lut_len(g);
  if (lut_n < 0) return lut_n;
  if (g.N >= (1ll << 31) - TC_ROWS) return NIC_ERR_UNSUPPORTED;     // 32-bit sample index in the kernel
  const ShadowGeom sg = {(const uint2*)h->tc_shadow, (const uint2*)((uint8_t*)h->tc_shadow + sl.off[0][1])};
  // warp-specialised persistent kernel: one CTA per SM, NG groups of 4 warps
  constexpr int NG0 = gws_groups(S::KX, 0), GSMEM0 = gws_smem<METHOD>(NG0, TC_LUT_MAX);
  constexpr int GSMEM6 = gws_smem<METHOD>(6, 64);                  // method 3: six groups, 64-entry LUT
  static_assert(GSMEM0 <= 227 * 1024 && (S::KX <= 80 || GSMEM6 <= 227 * 1024), "shared memory budget");
  // (not for random-access queries: they live on L1 hits, and the sixth group's 32 KB come out of the L1 — measured
  //  4.8 -> 4.2 Gquery/s on a 256^3 volume)
  const bool six = TAPS == 0 && S::KX > 80 && lut_n <= 64 && g.per_block > 1 && !(h->debug_flags & 128);
  const int NG = six ? 6 : NG0;
  void (*kern)(DevGeom, ShadowGeom, const long long*, const uint4*, int, int, OutT*, DevSampler) =
      npoly == 0 ? decode_tc_gws_kernel<METHOD, FMT, OutT, 0, 0, TC_LUT_MAX, TAPS>
                 : decode_tc_gws_kernel<METHOD, FMT, OutT, 3, 0, TC_LUT_MAX, TAPS>;
  if constexpr (S::KX > 80 && TAPS == 0) {
    if (six) kern = npoly == 0 ? decode_tc_gws_kernel<METHOD, FMT, OutT, 0, 6, 64> : decode_tc_gws_kernel<METHOD, FMT, OutT, 3, 6, 64>;
  }
  const long long ntiles = (g.N + TC_ROWS - 1) / TC_ROWS;
  return launch_persistent(h, kern, (ntiles + NG - 1) / NG, NG * GW_GROUP, six ? GSMEM6 : GSMEM0, st, g, sg, origins,
                           (const uint4*)h->tc_weights, m.cout, lut_n, out, smp);
}

// The chain table of a per-query-LOD or dense-chain launch (`bytes` of it) in the handle's device copy, on the call's stream.
static int upload_chain_table(Handle* h, const void* table, size_t bytes, cudaStream_t st) {
  if (!h->lod_chain && cudaMalloc(&h->lod_chain, sizeof(DevMipRows)) != cudaSuccess) {
    h->lod_chain = nullptr;
    return NIC_ERR_SCRATCH;
  }
  return (int)cudaMemcpyAsync(h->lod_chain, table, bytes, cudaMemcpyHostToDevice, st);
}

// The tables of a chain pass over mips gm[0, n) (per-query LOD or dense chain), keyed by the whole chain: the shadow grids of
// every pyramid level those mips reach (layout `sl`, which tc_scratch already holds) and the W1 image with the mip column.
template <int METHOD, int FMT>
static int prepare_chain(Handle* h, const ShadowLayout& sl, const DevGeom* gm, const void* const* g0, const void* const* g1,
                         int n, int code_bits, int npoly, const MlpDev& m, cudaStream_t st) {
  return prepare_tables(h, make_key(PREP_CHAIN, FMT, code_bits, npoly, m, gm, g0, g1, n), [&] {
    const int e = build_shadows<FMT>(h, sl, gm, g0, g1, code_bits, st);
    if (e) return e;
    pack_weights_kernel<FMT><<<16, 256, 0, st>>>(m, 0.0f, RowShape<METHOD>::KX, (uint16_t*)h->tc_weights, npoly);
    pack_lod_columns_kernel<FMT><<<1, 64, 0, st>>>(m, (uint16_t*)h->tc_weights);
    h->launches += 2;
    return (int)cudaGetLastError();
  });
}

// Per-query LOD: the shadow grids of every pyramid level the chain reaches (built once, keyed by the whole chain), the
// W1 image with the mip column, the chain table in device memory, one pass of the general kernel with 2 * 2^D rows a query.
template <int METHOD, int FMT, typename OutT>
static int launch_lod_t(Handle* h, const DevGeom* gm, DevChain c, const DevSampler& smp, const MlpDev& m,
                        const void* const* g0, const void* const* g1, int code_bits, OutT* out, cudaStream_t st) {
  using S = RowShape<METHOD>;
  constexpr int TAPS = 2 << S::DIM;
  const ShadowLayout sl = shadow_layout(gm, g0, g1, c.num_mips);
  if (sl.total / 8 >= (1ull << 32)) return NIC_ERR_UNSUPPORTED;            // 32-bit shadow offsets in the chain table
  int rc = tc_scratch(h, sl.total);
  if (rc) return rc;
  for (int i = 0; i < c.num_mips; ++i) {
    c.mip[i].s0 = (unsigned)(sl.off[i][0] / 8);
    c.mip[i].s1 = (unsigned)(sl.off[i][1] / 8);
  }
  const int npoly = resolve_npoly(h, FMT);
  if (npoly != 0 && npoly != 3) return NIC_ERR_UNSUPPORTED;
  rc = prepare_chain<METHOD, FMT>(h, sl, gm, g0, g1, c.num_mips, code_bits, npoly, m, st);
  if (rc) return rc;
  rc = upload_chain_table(h, &c, sizeof(DevChain), st);
  if (rc) return rc;
  DevGeom g = gm[0];                                  // method, PE, coordinates; the rest is per row from the chain
  g.N = (long long)g.nblocks * TAPS;
  g.interp = 1;                                       // (g1_factors computes the weights; rows of step-2 mips drop them)
  const ShadowGeom sg = {(const uint2*)h->tc_shadow, (const uint2*)h->tc_shadow};
  constexpr int NG = gws_groups(S::KX, 0), GSMEM = gws_smem<METHOD>(NG, TC_LUT_MAX, sizeof(DevChain));
  static_assert(GSMEM <= 227 * 1024, "shared memory budget");
  void (*kern)(DevGeom, ShadowGeom, const long long*, const uint4*, int, int, OutT*, DevSampler) =
      npoly == 0 ? decode_tc_gws_kernel<METHOD, FMT, OutT, 0, 0, TC_LUT_MAX, TAPS>
                 : decode_tc_gws_kernel<METHOD, FMT, OutT, 3, 0, TC_LUT_MAX, TAPS>;
  const long long ntiles = (g.N + TC_ROWS - 1) / TC_ROWS;
  return launch_persistent(h, kern, (ntiles + NG - 1) / NG, NG * GW_GROUP, GSMEM, st, g, sg, (const long long*)h->lod_chain,
                           (const uint4*)h->tc_weights, m.cout, 64, out, smp);
}

// Whole mip chain: mip 0 through the single-mip path (launch_tc_t: it equals nic_decode), then mips 1 .. L in ONE pass of
// the general kernel in its dense-chain mode, on the tables of launch_lod_t built for those mips.  tc_scratch is sized for
// the larger of the two passes before either builds: growing it between them would cudaFree, which synchronises the device.
template <int METHOD, int FMT, typename OutT>
static int launch_mips_t(Handle* h, const DevGeom* gm, const DevChain& c, const MlpDev& m, const void* const* g0,
                         const void* const* g1, int code_bits, OutT* out, cudaStream_t st) {
  using S = RowShape<METHOD>;
  const int L = c.num_mips - 1;
  const ShadowLayout sl = shadow_layout(gm + 1, g0 + 1, g1 + 1, L);
  if (sl.total / 8 >= (1ull << 32)) return NIC_ERR_UNSUPPORTED;            // 32-bit shadow offsets in the chain table
  const int npoly = resolve_npoly(h, FMT);
  if (L > 0 && npoly != 0 && npoly != 3) return NIC_ERR_UNSUPPORTED;
  size_t need0;                                       // what launch_tc_t takes for mip 0 (it never takes the code-resident path)
  if (METHOD == NIC_METHOD_2D && fast2d_eligible(gm[0], nullptr) && !h->disable_fast2d) {
    size_t b0, b1;
    fast2d_table_bytes(gm[0], &b0, &b1);
    need0 = b0 + b1;
  } else {
    need0 = shadow_layout(gm, g0, g1, 1).total;
  }
  int rc = tc_scratch(h, need0 > sl.total ? need0 : sl.total);
  if (rc) return rc;
  rc = launch_tc_t<METHOD, FMT, 0>(h, gm[0], m, g0[0], g1[0], code_bits, nullptr, out, st);
  if (rc || L == 0) return rc;
  rc = prepare_chain<METHOD, FMT>(h, sl, gm + 1, g0 + 1, g1 + 1, L, code_bits, npoly, m, st);
  if (rc) return rc;
  DevMipRows t;
  t.c = c;
  long long rows = 0;                                 // < 2^31 - TC_ROWS (launch_decode_mips_tc)
  for (int i = 0; i < NIC_MAX_MIPS; ++i) {
    t.row0[i] = i <= L ? (unsigned)rows : 0xffffffffu;
    if (i < 1 || i > L) continue;
    rows += gm[i].N;
    t.c.mip[i].s0 = (unsigned)(sl.off[i - 1][0] / 8);
    t.c.mip[i].s1 = (unsigned)(sl.off[i - 1][1] / 8);
  }
  rc = upload_chain_table(h, &t, sizeof(t), st);
  if (rc) return rc;
  DevGeom g = gm[1];                                  // method and PE; the rest is per row from the chain
  g.N = rows;
  g.interp = 1;                                       // (g1_factors computes the weights; rows of step-2 mips drop them)
  const ShadowGeom sg = {(const uint2*)h->tc_shadow, (const uint2*)h->tc_shadow};
  constexpr int NG = gws_groups(S::KX, 0), GSMEM = gws_smem<METHOD>(NG, TC_LUT_MAX, sizeof(DevMipRows));
  static_assert(GSMEM <= 227 * 1024, "shared memory budget");
  void (*kern)(DevGeom, ShadowGeom, const long long*, const uint4*, int, int, OutT*, DevSampler) =
      npoly == 0 ? decode_tc_gws_kernel<METHOD, FMT, OutT, 0, 0, TC_LUT_MAX, TAPS_MIPS>
                 : decode_tc_gws_kernel<METHOD, FMT, OutT, 3, 0, TC_LUT_MAX, TAPS_MIPS>;
  const long long ntiles = (g.N + TC_ROWS - 1) / TC_ROWS;
  return launch_persistent(h, kern, (ntiles + NG - 1) / NG, NG * GW_GROUP, GSMEM, st, g, sg, (const long long*)h->lod_chain,
                           (const uint4*)h->tc_weights, m.cout, 64, out + (size_t)gm[0].N * m.cout, DevSampler{});
}

// f(IntC<METHOD>, IntC<FMT>, out as OutT*) for the call's method, precision and output dtype (uint8 or float).
template <class F>
static int dispatch_tc(int method, int precision, int out_dtype, void* out, F&& f) {
  return dispatch_method_fmt(method, precision, [&](auto M, auto FMT) {
    return out_dtype == NIC_DT_U8 ? f(M, FMT, (uint8_t*)out) : f(M, FMT, (float*)out);
  });
}

int launch_decode_tc(Handle* h, const DevGeom& g, const MlpDev& m, const void* g0, const void* g1, int code_bits,
                     const long long* origins, void* out, int out_dtype, int precision, cudaStream_t st) {
  if (g.N == 0) return NIC_OK;
  if (!tc_shape_ok(g, m)) return NIC_ERR_UNSUPPORTED;
  return dispatch_tc(g.method, precision, out_dtype, out, [&](auto M, auto FMT, auto* o) {
    return launch_tc_t<M.value, FMT.value, 0>(h, g, m, g0, g1, code_bits, origins, o, st);
  });
}

int launch_sample_tc(Handle* h, const DevGeom& gq, const DevSampler& smp, const MlpDev& m, const void* g0, const void* g1,
                     int code_bits, void* out, int out_dtype, int precision, cudaStream_t st) {
  if (gq.nblocks == 0) return NIC_OK;
  if (!tc_shape_ok(gq, m)) return NIC_ERR_UNSUPPORTED;
  DevGeom g = gq;                                   // one row per tap: queries x 2^dim rows
  g.N = (long long)gq.nblocks << gq.dim;
  if (g.N >= (1ll << 31) - TC_ROWS) return NIC_ERR_UNSUPPORTED;     // 32-bit row index in the kernel
  return dispatch_tc(g.method, precision, out_dtype, out, [&](auto M, auto FMT, auto* o) {
    return launch_tc_t<M.value, FMT.value, 1 << RowShape<M.value>::DIM>(h, g, m, g0, g1, code_bits, nullptr, o, st, smp);
  });
}

int launch_sample_lod_tc(Handle* h, const DevGeom* gm, const DevChain& c, const DevSampler& smp, const MlpDev& m,
                         const void* const* g0, const void* const* g1, int code_bits, void* out, int out_dtype,
                         int precision, cudaStream_t st) {
  if (gm[0].nblocks == 0) return NIC_OK;
  if (!tc_shape_ok(gm[0], m)) return NIC_ERR_UNSUPPORTED;
  for (int i = 0; i < c.num_mips; ++i)               // one 64-entry LUT at step 1/4 serves the triangular PE of every mip
    if (gm[0].pe_kind == NIC_PE_TRIANGULAR && gm[i].step < 0.25f) return NIC_ERR_UNSUPPORTED;
  return dispatch_tc(gm[0].method, precision, out_dtype, out, [&](auto M, auto FMT, auto* o) {
    return launch_lod_t<M.value, FMT.value>(h, gm, c, smp, m, g0, g1, code_bits, o, st);
  });
}

int launch_decode_mips_tc(Handle* h, const DevGeom* gm, const DevChain& c, const MlpDev& m, const void* const* g0,
                          const void* const* g1, int code_bits, void* out, int out_dtype, int precision, cudaStream_t st) {
  if (!tc_shape_ok(gm[0], m)) return NIC_ERR_UNSUPPORTED;
  long long rows = 0;                                 // of the chain pass: mips 1 .. L
  for (int i = 1; i < c.num_mips; ++i) {              // one 64-entry LUT at step 1/4 serves the triangular PE of every mip
    if (gm[0].pe_kind == NIC_PE_TRIANGULAR && gm[i].step < 0.25f) return NIC_ERR_UNSUPPORTED;
    rows += gm[i].N;
  }
  if (rows >= (1ll << 31) - TC_ROWS) return NIC_ERR_UNSUPPORTED;     // 32-bit row index in the kernel
  return dispatch_tc(gm[0].method, precision, out_dtype, out, [&](auto M, auto FMT, auto* o) {
    return launch_mips_t<M.value, FMT.value>(h, gm, c, m, g0, g1, code_bits, o, st);
  });
}

}  // namespace nic
