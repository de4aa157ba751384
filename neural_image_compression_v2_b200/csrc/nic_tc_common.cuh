// nic_tc_common.cuh — tcgen05 / TMEM / mbarrier PTX wrappers, UMMA descriptors, packed 16-bit math and the shadow-grid
// relayout shared by the tensor-core kernels (nic_tc.cu: decode, nic_train_tc.cu: training step).
#pragma once
#include <cstring>
#include <type_traits>

#include "nic_internal.cuh"

namespace nic {

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// try_wait with a suspend-time hint: the warp sleeps in hardware until the phase completes (or the hint expires)
// instead of burning issue slots in a spin loop.
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAITS_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONES_%=;\n\t"
      "bra WAITS_%=;\n\t"
      "DONES_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"(1000000u) : "memory");
}
// tcgen05.commit: the mbarrier receives one arrival when every tcgen05.mma issued so far by this thread is done.
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem desc]   (kind::f16: f16 or bf16 operands, fp32 accumulate)
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// The same with the two shared-memory descriptors given as 32-bit halves.  The high half of a K-major no-swizzle
// descriptor (SBO, version bit) is a constant and the low half is (address >> 4) | (LBO >> 4) << 16, so stepping an operand
// through shared memory is ONE 32-bit add on the low half — the issuing thread of the decode kernels spends ~10 uniform
// instructions per MMA batch on descriptors this way instead of ~90 when every descriptor is rebuilt from its fields.
__host__ __device__ constexpr uint32_t smem_desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__device__ __forceinline__ void mma_ss_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi),
      "r"(idesc), "r"(accumulate)
      : "memory");
}

// One elected lane of a CONVERGED warp.  tcgen05.mma must be issued from warp-uniform control flow with warp-uniform
// operands: `if (warp_u == X) if (elect_one()) mma(...)` with warp_u = uniform_warp_index() keeps descriptors in uniform
// registers and the UTCHMMAs back to back (48 cycles each for M128 N64 SS, 32 for TS; tools/ubench/mma_rate2.cu).
// `if (lane == 0)` instead makes the compiler wrap EVERY mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall loop
// (operands are then per-thread values): 95..120 cycles per mma from one issuing thread.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ int uniform_warp_index() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

// Shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor): in 16-byte units the
// canonical layout is ((8,n),2):((1,SBO),LBO) — 8 rows x 16 B form a 128-byte core matrix, SBO steps to the next
// 8-row group, LBO to the next 8-element K chunk.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version for sm_100
  return d;                 // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}

// Instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A/B format fmt (0 f16, 1 bf16), both K-major.
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int M, int N, int b_mn_major = 0, int d_f16 = 0) {
  return ((d_f16 ? 0u : 1u) << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// tcgen05.ld / st, shape 32x32b: thread i of warp w touches TMEM lane 32*(w%4)+i, one 32-bit column per register.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 16 columns of 16-bit accumulators (idesc d_f16) as 8 registers of packed pairs (columns 2i, 2i+1 -> register i)
__device__ __forceinline__ void tmem_ld8_pack16(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.pack::16b.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// ------------------------------------------------------------------------------------------------ 16-bit math
template <int FMT> struct Pair;   // FMT 0 = f16, 1 = bf16
template <> struct Pair<0> {
  using T2 = __half2;
  static __device__ __forceinline__ T2 pack(float a, float b) { return __floats2half2_rn(a, b); }
  static __device__ __forceinline__ T2 cst(float a) { return __float2half2_rn(a); }
  static __device__ __forceinline__ T2 tanh2(T2 x) {
    uint32_t r, v = *reinterpret_cast<uint32_t*>(&x);
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(r) : "r"(v));
    return *reinterpret_cast<T2*>(&r);
  }
};
template <> struct Pair<1> {
  using T2 = __nv_bfloat162;
  static __device__ __forceinline__ T2 pack(float a, float b) { return __floats2bfloat162_rn(a, b); }
  static __device__ __forceinline__ T2 cst(float a) { return __float2bfloat162_rn(a); }
  static __device__ __forceinline__ T2 tanh2(T2 x) {
    uint32_t r, v = *reinterpret_cast<uint32_t*>(&x);
    asm("tanh.approx.bf16x2 %0, %1;" : "=r"(r) : "r"(v));
    return *reinterpret_cast<T2*>(&r);
  }
};

// 2*GELU_tanh on a packed pair: x + x*tanh(x*(c1 + c2*x^2)); the factor 1/2 lives in the next layer's weights.
template <int FMT>
__device__ __forceinline__ uint32_t gelu2x_packed(uint32_t xin) {
  using P = Pair<FMT>;
  typename P::T2 x = *reinterpret_cast<typename P::T2*>(&xin);
  typename P::T2 x2 = __hmul2(x, x);
  typename P::T2 p = __hfma2(x2, P::cst(0.0356774081f), P::cst(0.7978845608f));
  typename P::T2 t = P::tanh2(__hmul2(p, x));
  typename P::T2 h = __hfma2(x, t, x);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <int FMT>
__device__ __forceinline__ uint32_t gelu2x_pair(float a, float b) {
  using P = Pair<FMT>;
  typename P::T2 x = P::pack(a, b);
  typename P::T2 x2 = __hmul2(x, x);
  typename P::T2 p = __hfma2(x2, P::cst(0.0356774081f), P::cst(0.7978845608f));
  typename P::T2 t = P::tanh2(__hmul2(p, x));
  typename P::T2 h = __hfma2(x, t, x);
  return *reinterpret_cast<uint32_t*>(&h);
}

// GELU without MUFU (the decode kernels are bound by the XU pipe when every activation costs one MUFU.TANH):
//   gelu(x) = x * Phi(x),  Phi(x) ~ clamp(1/2 + x * Q(x^2), 0, 1),  Q a minimax polynomial of degree 4 in x^2
// evaluated on the FMA pipe in packed 16-bit math.  Exhaustively checked over all 63,488 finite f16 inputs against the
// exact erf GELU (tools/gelu_poly_fit.py): f16 max |err| 4.4e-3 (at |x| ~ 2.8), rms 4.1e-4 for |x| < 4 — the MUFU tanh
// form has 1.7e-3 / 1.5e-4, bf16 tanh 9.2e-3 / 8.7e-4.  The result is gelu(x), NOT 2*gelu(x) like gelu2x_pair: columns
// evaluated this way take the next layer's weights unscaled (pack_fast_kernel / gelu_poly_column).
//   f16 : the degree-4 Q has a positive leading coefficient and x*Q(x^2) stays above 1/2 beyond the fitted range, so no
//         argument clamp is needed; fma.rn.sat clamps Phi to [0, 1]  (7 FMA-pipe instructions + the pack).
//   bf16: no .sat form exists and the 8-bit mantissa needs the argument clamped: min(x^2, L^2), fma.relu, min(., 1).
template <int FMT>
__device__ __forceinline__ uint32_t gelu_poly_packed(uint32_t xin);
template <int FMT>
__device__ __forceinline__ uint32_t gelu_poly_pair(float a, float b) {
  auto x = Pair<FMT>::pack(a, b);
  return gelu_poly_packed<FMT>(*reinterpret_cast<uint32_t*>(&x));
}
template <int FMT>
__device__ __forceinline__ uint32_t gelu_poly_packed(uint32_t xin) {
  using P = Pair<FMT>;
  typename P::T2 x = *reinterpret_cast<typename P::T2*>(&xin);
  typename P::T2 s = __hmul2(x, x);
  typename P::T2 h;
  if constexpr (FMT == 0) {
    typename P::T2 q = __hfma2(s, P::cst(1.1074006e-05f), P::cst(-4.2891181e-04f));
    q = __hfma2(q, s, P::cst(6.8348698e-03f));
    q = __hfma2(q, s, P::cst(-6.0208798e-02f));
    q = __hfma2(q, s, P::cst(3.9457067e-01f));
    h = __hmul2(x, __hfma2_sat(x, q, P::cst(0.5f)));
  } else {
    s = __hmin2(s, P::cst(11.56f));
    typename P::T2 q = __hfma2(s, P::cst(1.1117739e-05f), P::cst(-4.2903416e-04f));
    q = __hfma2(q, s, P::cst(6.8217828e-03f));
    q = __hfma2(q, s, P::cst(-6.0079083e-02f));
    q = __hfma2(q, s, P::cst(3.9425993e-01f));
    h = __hmul2(x, __hmin2(__hfma2_relu(x, q, P::cst(0.5f)), P::cst(1.0f)));
  }
  return *reinterpret_cast<uint32_t*>(&h);
}
// Which of the 8 activation pairs of a 16-column chunk use gelu_poly_pair when NPOLY of them do (evenly interleaved with
// the MUFU pairs, so both pipes stay busy), and the same question for a hidden column (weight packing).
__host__ __device__ constexpr bool gelu_poly_pair_sel(int pair, int npoly) {
  return ((pair + 1) * npoly) / 8 > (pair * npoly) / 8;
}
__host__ __device__ constexpr bool gelu_poly_column(int col, int npoly) { return gelu_poly_pair_sel((col & 15) >> 1, npoly); }

template <int FMT>
__device__ __forceinline__ uint16_t to16(float v) {
  if (FMT == 0) {
    __half h = __float2half_rn(v);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __nv_bfloat16 h = __float2bfloat16_rn(v);
  return *reinterpret_cast<uint16_t*>(&h);
}

__host__ __device__ constexpr int b_image_bytes(int nrows, int k) { return nrows * k * 2; }

// ------------------------------------------------------------------------------------------------ shadow grids
// The tensor-core path reads 16-bit, channel-LAST copies of the two active grids, transposed so that the fast texel
// axis is contiguous: shadow[((x*Ny + y)*Nz + z)*C + c] = grid[c][z][y][x]  (2-D: Nz = 1, shadow[(x*Ny + y)*C + c]).
// One node = C*2 bytes (24 B at C = 12) -> a corner is three 8-byte loads that land in the operand registers as is.
// Written once per decode call by relayout_kernel (coalesced both ways through shared memory).
// A grid element from the caller's tensor: float32 as is, or (code_bits > 0) a uint8 code of models.save4fp de-quantised
// exactly as models.load4fp does, (code - 2^(b-1) + 1) / (2^b - 1) — the quantiser fused into the grid read.
__device__ __forceinline__ float grid_value(const float* __restrict__ src, long long idx, int code_bits) {
  if (code_bits == 0) return __ldg(src + idx);
  const float c = (float)__ldg(reinterpret_cast<const uint8_t*>(src) + idx);
  const float z = __fadd_rn(__fsub_rn(c, (float)(1 << (code_bits - 1))), 1.0f);
  return __fdiv_rn(z, (float)((1 << code_bits) - 1));
}

// tile: 32 nodes along x  x  RL_TF nodes along the output-fast axis f, all channels.  RL_TF = 32 writes 768-byte runs and is
// the faster one once the grid yields enough blocks (1025^2 nodes: 1,089 blocks, 20 us against 36 us with RL_TF = 8); on
// smaller grids (513^2: 289 blocks of 48 serial loads per thread, 28 us) RL_TF = 8 gives 4x the blocks.
template <int FMT, int RL_TF>
__global__ void __launch_bounds__(256) relayout_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, int C,
                                                       int nx, int nf, int no, long long sf, long long so,
                                                       long long plane, int code_bits) {
  // blockIdx.z = the third axis.  tile[e * 33 + xi] with e = fi * C + c = the element's position in output row xi:
  // conflict-free both ways.
  extern __shared__ uint16_t tile[];           // [RL_TF * C][33]
  const int x0 = blockIdx.x * 32, f0 = blockIdx.y * RL_TF, o = blockIdx.z;
  for (int i = threadIdx.x; i < C * RL_TF * 32; i += blockDim.x) {
    int c = i / (RL_TF * 32), r = i - c * (RL_TF * 32), fi = r >> 5, xi = r & 31;
    int x = x0 + xi, f = f0 + fi;
    float v = (x < nx && f < nf) ? grid_value(src, (long long)c * plane + (long long)f * sf + (long long)o * so + x, code_bits) : 0.f;
    tile[(fi * C + c) * 33 + xi] = to16<FMT>(v);
  }
  __syncthreads();
  const int fw = nf - f0 < RL_TF ? nf - f0 : RL_TF;   // valid nodes along f in this tile
  const int xw = nx - x0 < 32 ? nx - x0 : 32;         // valid output rows
  const int row_elems = fw * C;
  if ((C & 3) == 0) {
    // 8-byte stores (rows start 8-byte aligned when C % 4 == 0), all rows of the tile in parallel
    const int per_row = row_elems >> 2;
    for (int j = threadIdx.x; j < xw * per_row; j += blockDim.x) {
      const int xi = j / per_row, q = j - xi * per_row;
      const uint16_t* t = tile + (4 * q) * 33 + xi;
      uint2 v;
      v.x = (uint32_t)t[0] | ((uint32_t)t[33] << 16);
      v.y = (uint32_t)t[66] | ((uint32_t)t[99] << 16);
      uint16_t* row = dst + (((long long)(x0 + xi) * no + o) * nf + f0) * C;
      *reinterpret_cast<uint2*>(row + 4 * q) = v;
    }
  } else {
    for (int j = threadIdx.x; j < xw * row_elems; j += blockDim.x) {
      const int xi = j / row_elems, e = j - xi * row_elems;
      dst[(((long long)(x0 + xi) * no + o) * nf + f0) * C + e] = tile[e * 33 + xi];
    }
  }
}

__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
               : "memory");
}

// stores registers [lo, lo+n) of a row to operand-A columns [lo, lo+n) with the widest tcgen05.st shapes
template <int N>
__device__ __forceinline__ void store_row_part(uint32_t taddr, const uint32_t* r) {
  if constexpr (N >= 16) {
    tmem_st16(taddr, r);
    store_row_part<N - 16>(taddr + 16, r + 16);
  } else if constexpr (N >= 8) {
    tmem_st8(taddr, r);
    store_row_part<N - 8>(taddr + 8, r + 8);
  } else if constexpr (N >= 4) {
    tmem_st4(taddr, r);
    store_row_part<N - 4>(taddr + 4, r + 4);
  } else {
    static_assert(N == 0, "row parts are multiples of 4 registers");
  }
}

static inline long long plane_size_host(const int* n, int dim) {
  return dim == 2 ? (long long)n[0] * n[1] : (long long)n[0] * n[1] * n[2];
}

static inline int ensure_scratch(void** ptr, size_t* have, size_t need) {
  if (*have >= need) return NIC_OK;
  if (*ptr) cudaFree(*ptr);
  *ptr = nullptr;
  *have = 0;
  size_t sz = (need + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
  if (cudaMalloc(ptr, sz) != cudaSuccess) return NIC_ERR_SCRATCH;
  *have = sz;
  return NIC_OK;
}

template <int FMT>
static inline int launch_relayout(Handle* h, const DevGeom& g, const void* src, int code_bits, const int* nodes, uint16_t* dst,
                                  cudaStream_t st) {
  const int dim = g.dim;
  const int nx = nodes[0], nf = dim == 2 ? nodes[1] : nodes[2], no = dim == 2 ? 1 : nodes[1];
  const long long sf = dim == 2 ? nx : (long long)nodes[1] * nx, so = dim == 2 ? 0 : nx;
  const long long plane = (long long)nx * nodes[1] * (dim == 2 ? 1 : nodes[2]);
  const bool tall = (long long)((nx + 31) / 32) * ((nf + 31) / 32) * no >= 4ll * h->sms;
  const int tf = tall ? 32 : 8;
  dim3 grid((nx + 31) / 32, (nf + tf - 1) / tf, no);
  size_t smem = (size_t)g.C * tf * 33 * sizeof(uint16_t);
  if (tall) {
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(relayout_kernel<FMT, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
    }
    relayout_kernel<FMT, 32><<<grid, 256, smem, st>>>((const float*)src, dst, g.C, nx, nf, no, sf, so, plane, code_bits);
  } else {
    relayout_kernel<FMT, 8><<<grid, 256, smem, st>>>((const float*)src, dst, g.C, nx, nf, no, sf, so, plane, code_bits);
  }
  h->launches++;
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ launcher helpers
// The shapes the tensor-core kernels are built for.
static inline bool tc_shape_ok(const DevGeom& g, const MlpDev& m) {
  return g.C == 12 && g.PE == 6 && m.hidden == 64 && m.cout <= 16;
}

// The scratch of the tensor-core tables: the weight images (64 KB of tc_weights) and shadow_bytes of tc_shadow.  A
// reallocated buffer holds no tables.
static inline int tc_scratch(Handle* h, size_t shadow_bytes) {
  const size_t wb = h->tc_weights_bytes, sb = h->tc_shadow_bytes;
  int rc = ensure_scratch(&h->tc_weights, &h->tc_weights_bytes, 64 * 1024);
  if (rc == NIC_OK) rc = ensure_scratch(&h->tc_shadow, &h->tc_shadow_bytes, shadow_bytes);
  if (h->tc_weights_bytes != wb || h->tc_shadow_bytes != sb) invalidate_prepared(h);
  return rc;
}

// The 16-bit shadows of the grids of mips [0, n) in tc_shadow: G0 then G1 of each mip, each rounded up to 256 bytes.  A mip
// whose grids (pointers and node counts) equal an earlier mip's shares that mip's shadows.
struct ShadowLayout {
  int n;
  size_t off[NIC_MAX_MIPS][2];       // byte offsets of mip i's G0 and G1 shadows
  bool own[NIC_MAX_MIPS];            // mip i's shadows are built from its own grids
  size_t total;
};
static inline ShadowLayout shadow_layout(const DevGeom* gm, const void* const* g0, const void* const* g1, int n) {
  ShadowLayout s;
  s.n = n;
  s.total = 0;
  for (int i = 0; i < n; ++i) {
    int first = i;
    for (int j = 0; j < i && first == i; ++j)
      if (g0[j] == g0[i] && g1[j] == g1[i] && !memcmp(gm[j].n0, gm[i].n0, sizeof(gm[i].n0)) &&
          !memcmp(gm[j].n1, gm[i].n1, sizeof(gm[i].n1)))
        first = j;
    s.own[i] = first == i;
    for (int k = 0; k < 2; ++k) {
      s.off[i][k] = s.own[i] ? s.total : s.off[first][k];
      if (s.own[i]) s.total += ((size_t)plane_size_host(k ? gm[i].n1 : gm[i].n0, gm[i].dim) * gm[i].C * 2 + 255) & ~(size_t)255;
    }
  }
  return s;
}
template <int FMT>
static inline int build_shadows(Handle* h, const ShadowLayout& s, const DevGeom* gm, const void* const* g0,
                                const void* const* g1, int code_bits, cudaStream_t st) {
  uint8_t* base = (uint8_t*)h->tc_shadow;
  for (int i = 0; i < s.n; ++i) {
    if (!s.own[i]) continue;
    int rc = launch_relayout<FMT>(h, gm[i], g0[i], code_bits, gm[i].n0, (uint16_t*)(base + s.off[i][0]), st);
    if (rc == NIC_OK) rc = launch_relayout<FMT>(h, gm[i], g1[i], code_bits, gm[i].n1, (uint16_t*)(base + s.off[i][1]), st);
    if (rc != NIC_OK) return rc;
  }
  return NIC_OK;
}

// The one place where a call's method and precision become template parameters: f(IntC<METHOD>, IntC<FMT>) with FMT 0
// for NIC_PREC_F16 and 1 (bf16) otherwise.
template <int V>
using IntC = std::integral_constant<int, V>;
template <class F>
static inline int dispatch_method_fmt(int method, int precision, F&& f) {
  auto by_fmt = [&](auto M) { return precision == NIC_PREC_F16 ? f(M, IntC<0>{}) : f(M, IntC<1>{}); };
  switch (method) {
    case NIC_METHOD_2D: return by_fmt(IntC<NIC_METHOD_2D>{});
    case NIC_METHOD_3D: return by_fmt(IntC<NIC_METHOD_3D>{});
    case NIC_METHOD_3D_V2: return by_fmt(IntC<NIC_METHOD_3D_V2>{});
  }
  return NIC_ERR_UNSUPPORTED;
}

}  // namespace nic
