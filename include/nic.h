/*
 * nic.h — C ABI of libnic.so: the B200 (sm_100a) implementation of the per-texel decode / training-step
 * hot path of 21K1113/Neural_Image_Compression_V2.
 *
 * The reference has no FFI of its own (pure Python/PyTorch); the seam this ABI replaces is the set of
 * module-level functions that `train_models`, `decode_image` and `process_images` call
 * (Projects/image_compression.py:233-269, 313-345, 380-396).  Each entry point below cites the reference
 * interface it stands in for.  `INTEGRATION.md` shows the ctypes binding a maintainer of the reference adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch), borrowed for the duration of the stream
 *     work the call enqueues; the library never frees caller memory.  Scratch lives in the NicHandle.
 *   - calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - return value: 0 = success, < 0 = NicStatus library error, > 0 = cudaError_t.  Nothing throws.
 *   - there is NO CPU fallback: a device that is not compute capability 10.x yields NIC_ERR_DEVICE.
 *   - a handle is bound to one device and is not thread-safe; use one handle per rank.
 *   - grids keep the reference layout: float32, contiguous, channel-major `[C, y, x]` (2-D) or
 *     `[C, z, y, x]` (3-D), where x is the FIRST image axis (Projects/fp_def.py:81-86, 96-103).
 *   - a step's samples are ordered n = block*Bx*By*Bz + ix*By*Bz + iy*Bz + iz (meshgrid 'ij',
 *     Projects/fp_def.py:124,161), blocks = crops (training) or decode blocks.
 */
#ifndef NIC_H_
#define NIC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NIC_ABI_VERSION 1

typedef enum NicStatus {
  NIC_OK = 0,
  NIC_ERR_ARG = -1,          /* null pointer / negative size / inconsistent descriptor            */
  NIC_ERR_UNSUPPORTED = -2,  /* configuration outside what the kernels are built for              */
  NIC_ERR_DEVICE = -3,       /* not an sm_100 device, or handle bound to another device           */
  NIC_ERR_BOUNDS = -4,       /* a host-known origin would index outside the grids                 */
  NIC_ERR_ALIGN = -5,        /* pointer not aligned as documented                                 */
  NIC_ERR_SCRATCH = -6,      /* scratch allocation failed                                         */
  NIC_ERR_EXCHANGE = -7      /* a data-parallel exchange timed out waiting for a peer (sticky, see
                                nic_adam_step_exchange): parameters are no longer updated on this handle */
} NicStatus;

/* COMPRESSION_METHOD of Projects/var2.py:51-55 (2 = 2-D atlas, handled by the caller as method 1). */
enum { NIC_METHOD_2D = 1, NIC_METHOD_3D = 3, NIC_METHOD_3D_V2 = 4 };
/* positional encodings: Projects/utils.py:211-227 (triangular) and :198-208 (sinusoidal). */
enum { NIC_PE_TRIANGULAR = 0, NIC_PE_SINUSOIDAL = 1 };
/* arithmetic of the decoder MLP. F32 = reference-exact erf GELU on CUDA cores (1e-5 parity path);
 * F16 / BF16 = tcgen05 tensor-core path, fp32 accumulate, tanh-form GELU (+-1 LSB on 8-bit output). */
enum { NIC_PREC_F32 = 0, NIC_PREC_F16 = 1, NIC_PREC_BF16 = 2 };
/* element types of outputs */
enum { NIC_DT_F32 = 0, NIC_DT_F16 = 1, NIC_DT_BF16 = 2, NIC_DT_U8 = 3 };

/* Geometry of one gather problem: which grids, which texels.  Mirrors the arguments of
 * fp_def.create_g0_g1 / create_g0_g1_3d / create_g0_g1_3d_v2 (Projects/fp_def.py:115,148,187) plus the
 * crop loop of create_decoder_input_* (Projects/image_compression.py:71-167). */
typedef struct NicGeom {
  int32_t method;        /* NIC_METHOD_*                                                            */
  int32_t channels;      /* C, FEATURE_PYRAMID_CHANNELS                                             */
  int32_t pe_channels;   /* PE_CHANNELS per axis                                                    */
  int32_t pe_kind;       /* NIC_PE_*                                                                */
  int32_t step_log2;     /* log2(step_number) = mip - 2(fl+1)  (image_compression.py:79)            */
  int32_t mip_level;     /* value written to the LOD column                                         */
  int32_t g0_nodes[3];   /* nodes of G0 along image axes x,y,z (z ignored in 2-D)                   */
  int32_t g1_nodes[3];   /* nodes of G1 along x,y,z                                                 */
  int32_t block[3];      /* texels per block along x,y,z (reference: a cube of sample_number)       */
  int32_t num_blocks;    /* crops per step, or decode blocks                                        */
  int32_t origin0[3];    /* origin of block 0 when `origins` is NULL (single-block decode)          */
  int32_t reserved;
  float pe_div[8];       /* sinusoidal div_term (utils.py:202), float32 as torch evaluates it        */
} NicGeom;

/* The decoder MLP of ColorDecoder (Projects/image_compression.py:54-68), nn.Linear layout [out,in]. */
typedef struct NicMlp {
  int32_t cin, hidden, cout, reserved;
  const float* w1; const float* b1;   /* [hidden, cin], [hidden]    */
  const float* w2; const float* b2;   /* [hidden, hidden], [hidden] */
  const float* w3; const float* b3;   /* [cout, hidden], [cout]     */
} NicMlp;

/* Gradients / mutable views of the same six tensors. */
typedef struct NicMlpGrad {
  float* w1; float* b1; float* w2; float* b2; float* w3; float* b3;
} NicMlpGrad;

typedef struct NicHandle NicHandle;

/* ---- lifecycle ---------------------------------------------------------------------------------------- */
int nic_abi_version(void);
/* Binds a handle to CUDA device `device`; fails with NIC_ERR_DEVICE unless it is compute capability 10.x. */
int nic_create(int device, NicHandle** out);
int nic_destroy(NicHandle* h);
/* Message for the last non-zero status returned on this handle (or a generic one when h is NULL). */
const char* nic_last_error_string(const NicHandle* h);
const char* nic_status_string(int status);
/* Number of kernel launches this handle has enqueued so far (bench.py reports it as `gpu_launches`). */
int64_t nic_launch_count(const NicHandle* h);

/* Tuning / testing knobs.  NIC_OPT_DISABLE_FAST2D = 1 forces the general tensor-core decode kernel even when the
 * geometry qualifies for the aligned full-resolution 2-D fast path (both must give the same image). */
/* NIC_OPT_REUSE_PREPARED = 1: the caller asserts that grids and decoder weights have not changed since the previous
 * tensor-core call on this handle (nic_decode, nic_decode_codes, nic_sample, nic_sample_codes, nic_sample_lod,
 * nic_sample_lod_codes, nic_decode_mips, nic_decode_mips_codes); if that call prepared its private tables (shadow grids, per-node G1 rows, packed weights) for the
 * same kernel, pointers, node counts, steps, mip level, code width and precision, they are reused instead of being
 * rebuilt (decoding one frame as several row bands).  A training step on the handle discards them.  Off by default: every
 * call rebuilds from the caller's tensors. */
/* NIC_OPT_DEBUG_KNOCKOUT: profiling only (tools/run_decode.py, tools/run_train.py) — decode: bit 0 skips the output
 * stores, bit 1 replaces GELU by a plain pack, bit 2 issues one MMA per layer; training: bit 4 skips the grid-gradient
 * atomics, bits 5 / 6 make nic_adam_step_exchange skip the flag wait / read only its own buffer (timing experiments in
 * tools/dp_timing.py), bit 8 keeps the shuffle-based grid scatter where the tensor-core scatter would run (results stay correct:
 * A/B timing); results are otherwise WRONG on purpose.  Bit 3 only enables the training phase counters (nic_debug_counters) and
 * leaves the results unchanged.  nic_gather (16-bit rows, tools/run_gather.py): bit 0 skips the row build, bit 1 the bulk
 * stores, bit 4 keeps 4-row super-tiles, bit 6 the run-time-geometry kernel.  nic_adam_step_exchange (sliced): bit 7 reduces
 * one item per thread and round.  Any non-zero value makes nic_decode's fast path run its generic instance instead of the
 * RGB-specialised one (same results: A/B timing).  Never set in production. */
/* NIC_OPT_GELU_POLY: how many of every 8 hidden activations of the fast 2-D tensor-core decode kernel evaluate GELU as a
 * clamped minimax polynomial on the FMA pipe instead of MUFU.TANH (the kernel is bound by the XU pipe when all of them
 * use the transcendental).  -1 = the tuned default; 0 = all MUFU (round-1 behaviour); values the library was not built
 * with return NIC_ERR_UNSUPPORTED from nic_decode.  Both forms stay inside the tensor-core tolerance (+-1 LSB). */
/* NIC_OPT_EXCHANGE_TIMEOUT_MS: how long nic_adam_step_exchange waits on the device for a peer before it gives up
 * (default 10,000 ms, counted in SM clock cycles at 2 GHz; raise it when a rank may legitimately stall, e.g. a rank-0 evaluation between steps). */
/* NIC_OPT_STEP_METRICS = 1: the per-step PSNR bookkeeping of train_models (calculate_psnr(quantize_to_bit(out),
 * quantize_to_bit(target)), image_compression.py:260-261) without a host sync: nic_train_step additionally accumulates
 * loss_sum[1] += sum((floor(out*255+.5) - floor(target*255+.5))^2), and nic_adam_step_loss / nic_adam_step_exchange
 * additionally write loss_out[1] = loss_sum[1] * loss_scale (and clear it).  loss_sum and loss_out must then hold TWO floats.
 * FusedTrainer points loss_out into a device ring buffer and reads it back every k steps. */
/* NIC_OPT_STATIC_TILES = 1: the tensor-core training kernel walks its tiles in a static round-robin order instead of handing
 * them out through an atomic counter (A/B timing of the scheduler: the dynamic order balances the CTAs, -7 % kernel time at
 * config 1).  Either way the decoder gradients are reproducible to fp32 rounding, like the grid gradients (float atomics): the
 * tile slots of a CTA share their weight-gradient accumulators. */
enum { NIC_OPT_DISABLE_FAST2D = 1, NIC_OPT_TIME_KERNELS = 2, NIC_OPT_REUSE_PREPARED = 3,
       NIC_OPT_GELU_POLY = 5, NIC_OPT_EXCHANGE_TIMEOUT_MS = 6, NIC_OPT_STEP_METRICS = 7, NIC_OPT_STATIC_TILES = 8,
       NIC_OPT_DEBUG_KNOCKOUT = 100 };
int nic_set_option(NicHandle* h, int option, int value);
/* With NIC_OPT_TIME_KERNELS = 1 every nic_decode / nic_train_step / nic_gather call brackets its DOMINANT kernel
 * (not the small preparation kernels) with CUDA events on the call's stream.  This call synchronises on the recorded
 * events, adds up their durations, returns the sum (milliseconds) and the number of bracketed launches, and clears
 * the list.  bench.py uses it for the roofline fraction of the dominant kernel. */
int nic_kernel_time_ms(NicHandle* h, double* total_ms, int64_t* launches);
/* Profiling aid (tools/run_train.py phases): with bit 3 of NIC_OPT_DEBUG_KNOCKOUT set, thread 0 of every CTA of the
 * tensor-core training kernel adds the SM cycles it spends in each of its 13 per-tile phases (gather, 3 forward MMA
 * waits, 2 GELU epilogues, loss, 3 backward MMA waits, 2 delta epilogues, scatter) to device counters; counter 15 counts
 * tiles.  This call synchronises the device, copies counters[0, n) (n <= 16) to `out` and clears them. */
int nic_debug_counters(NicHandle* h, int64_t* out, int n);

/* ---- decoder input (K1) ------------------------------------------------------------------------------- */
/* Width of the decoder input for a geometry: C*(corners+1) + PE*D + 1 (Projects/var2.py:114-118). */
int nic_cin(const NicGeom* g);
/* Replaces create_decoder_input_2d/3d/3d_v2 and finally_decode_input_* (image_compression.py:71-211):
 * writes X [N, Cin] row-major, N = num_blocks*Bx*By*Bz.  `origins` = int64 [num_blocks, D] device pointer
 * (the reference's `coord` tensor) or NULL to use g->origin0.  x_dtype: NIC_DT_F32 (bit-exact with the
 * reference for triangular PE), NIC_DT_F16 or NIC_DT_BF16 (rounded once from the fp32 value). */
int nic_gather(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const int64_t* origins,
               void* x, int x_dtype, void* stream);
/* Transpose of nic_gather for autograd (the reference's 64 index_put(accumulate) calls,
 * image_compression.py:265): dX [N, Cin] fp32 -> accumulates into dG0 / dG1 (grid-shaped, fp32). */
int nic_scatter(NicHandle* h, const NicGeom* g, const float* dx, const int64_t* origins, float* dg0, float* dg1,
                void* stream);

/* Target gather of random_crop_dataset (image_compression.py:44-47): image [channels, S0, S1(, S2)] fp32 -> targets
 * [num_crops, crop0*crop1(*crop2), channels] fp32 for crops whose origins are the DEVICE tensor `origins` [num_crops, dim]
 * (the reference's `coord`).  size / crop: HOST pointers to dim ints.  Origins are clamped into the image. */
int nic_sample_crops(NicHandle* h, const float* image, int dim, int channels, const int32_t* size, const int64_t* origins,
                     int num_crops, const int32_t* crop, float* targets, void* stream);

/* random_crop_dataset without the host (image_compression.py:36-49): crop origins are drawn ON THE DEVICE, uniform over the
 * integers [0, size - crop] per axis like torch.randint (Philox4x32-10, key = seed, counter = (crop index, step); word a of
 * the block -> axis a), written to origins_out [num_crops, dim] (int64, the reference's `coord`) and used for the target
 * gather of nic_sample_crops in the same launch.  Data-parallel ranks pass different seeds.  The LOD of the step (which
 * fixes `image`, `crop` and every launch shape) stays a host integer: FusedTrainer.draw_lod evaluates the reference's
 * distribution (:29-34) with a counter-based generator, identically on every rank, without touching the device. */
int nic_sample_crops_random(NicHandle* h, const float* image, int dim, int channels, const int32_t* size, int num_crops,
                            const int32_t* crop, uint64_t seed, uint64_t step, int64_t* origins_out, float* targets, void* stream);

/* The mip-pyramid builder of the script: transforms.Resize((h, w)) on the 8-bit PIL image followed by ToTensor
 * (image_compression.py:433-442, 462-469).  src: uint8 [height, width, channels] (PIL / numpy HWC layout).  Reproduces
 * Pillow's antialiased BILINEAR resample bit for bit: separable triangle filter of support max(scale, 1), fixed-point
 * coefficients (22 fractional bits), horizontal pass rounded to 8 bits before the vertical pass.  dst_u8 (optional):
 * [out_height, out_width, channels]; dst_f32 (optional): ToTensor's [channels, out_height, out_width] = u8 / 255.
 * An init-time call: it synchronises `stream` (host-built coefficient tables live in handle scratch). */
int nic_resize_bilinear_u8(NicHandle* h, const uint8_t* src, int height, int width, int channels, int out_height, int out_width,
                           uint8_t* dst_u8, float* dst_f32, void* stream);

/* COMPRESSION_METHOD 2 (a volume flattened into one 2-D image): frame i of frames [num_frames, S, S, channels] (uint8) sits
 * at atlas rows [r S, (r+1) S), columns [q S, (q+1) S), r = i / (atlas_size / S), q = i % (atlas_size / S)
 * (image_compression.py:453-460); unused atlas cells are zero.  nic_atlas_unpack is the inverse applied to the decoded
 * frame (:413-419). */
int nic_atlas_pack(NicHandle* h, const uint8_t* frames, int num_frames, int frame_size, int channels, int atlas_size,
                   uint8_t* atlas, void* stream);
int nic_atlas_unpack(NicHandle* h, const uint8_t* atlas, int atlas_size, int channels, int num_frames, int frame_size,
                     uint8_t* frames, void* stream);

/* Stand-alone positional encodings, utils.triangular_positional_encoding (utils.py:211-223) and
 * utils.positional_encoding (utils.py:198-208): coord [dim, n] fp32 -> out [pe_channels*dim, n] fp32.
 * pe_div: HOST pointer to pe_channels/2 floats (sinusoidal div_term), ignored for the triangular kind. */
int nic_positional_encoding(NicHandle* h, const float* coord, int dim, int64_t n, int pe_channels, int pe_kind,
                            const float* pe_div, float* out, void* stream);

/* ---- decoder MLP on a materialised input (ColorDecoder.forward, image_compression.py:66-68) ------------ */
/* out [N, cout] fp32 = sigmoid(W3 gelu(W2 gelu(W1 x + b1) + b2) + b3); x [N, cin] fp32 row-major with row
 * stride `ldx` elements.  If z1/z2 are non-NULL the pre-activations [N, hidden] are saved for backward. */
int nic_mlp_forward(NicHandle* h, const NicMlp* m, const float* x, int64_t ldx, int64_t n, float* out, float* z1,
                    float* z2, void* stream);
/* Backward of the above given dOut [N, cout]: accumulates weight/bias gradients into `gm` and, when dx is
 * non-NULL, writes dX [N, cin]. */
int nic_mlp_backward(NicHandle* h, const NicMlp* m, const float* x, int64_t ldx, int64_t n, const float* z1,
                     const float* z2, const float* out, const float* dout, const NicMlpGrad* gm, float* dx,
                     void* stream);

/* ---- fused decode (K2): gather -> MLP -> output, X never materialised ---------------------------------- */
/* Replaces finally_decode_input_* + arc_decoder(...) inside decode_image (image_compression.py:313-345).
 * out: [N, cout] row-major in out_dtype (NIC_DT_F32, or NIC_DT_U8 = floor(v*255+.5), models.py:29-40).
 * precision: NIC_PREC_F32 (reference-exact) or NIC_PREC_F16/BF16 (tcgen05). */
int nic_decode(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const int64_t* origins,
               const NicMlp* m, void* out, int out_dtype, int precision, void* stream);

/* The same from the SAVED model: codes0 / codes1 are the uint8 grid codes of models.save4fp (one code per byte, `bits`
 * wide, same [C, (z,) y, x] layout); they are de-quantised exactly as models.load4fp does inside the grid read, so the
 * float32 grids of fp_load are never materialised (image_compression.py:393-400).  Tensor-core precisions only. */
int nic_decode_codes(NicHandle* h, const NicGeom* g, const uint8_t* codes0, const uint8_t* codes1, int bits,
                     const int64_t* origins, const NicMlp* m, void* out, int out_dtype, int precision, void* stream);

/* ---- filtered sampling at continuous coordinates ------------------------------------------------------- */
/* Bilinear (2-D) / trilinear (3-D) sampling of the decoded mip: what a renderer's texture read or a colour-LUT
 * application does, without materialising the taps.  coords: [Q, D] fp32 normalised coordinates in axis order (x, y[, z]),
 * x the first image axis (the slow axis of nic_decode's output).  The geometry describes the mip exactly as for a
 * random-access nic_decode, with num_blocks = Q and block = 1; `origins` / origin0 are not used.  On each axis, with S the
 * extent of the mip (every step one fp32 operation, so the result is reproducible bit for bit):
 *   p  = align_corners ? u * (S - 1) : u * S - 0.5;      p = min(max(p, -2^24), 2^24)   (NaN -> -2^24)
 *   i0 = floor(p), f = p - i0;  taps i0 and i0 + 1 with weights 1 - f and f;
 *   NIC_ADDRESS_CLAMP: each tap clamped to [0, S - 1];  NIC_ADDRESS_WRAP: each tap reduced modulo S (fmod, + S if negative).
 * The T = 2^D taps are ordered with x slowest; a tap's weight is the product of its per-axis weights (x first) and its value
 * is nic_decode's output for that integer texel (fp32 sigmoid output, before any quantisation).  out [Q, cout] in out_dtype
 * (NIC_DT_F32, or NIC_DT_U8 = floor(v*255+.5) of the blended value, quantised once) holds sum_k w_k * value_k, or with
 * blend_prev set (1 - blend_weight) * prev + blend_weight * that sum (blending two mips: fractional LOD).
 * precision NIC_PREC_F32: the taps are decoded by the reference-exact kernel and summed in tap order; F16 / BF16: one
 * tensor-core pass, the T taps of a query are T adjacent rows of a tile and are summed in registers.  Q * T must stay below
 * 2^31 - 128 (NIC_ERR_UNSUPPORTED).  An extent whose last texel would index outside the grids
 * gives NIC_ERR_BOUNDS (the rule of a host-known origin, with origin 0 and block = extent). */
enum { NIC_ADDRESS_CLAMP = 0, NIC_ADDRESS_WRAP = 1 };
typedef struct NicSampler {
  int32_t address;          /* NIC_ADDRESS_*                                                     */
  int32_t align_corners;    /* 0: texel i centred at (i + .5)/S; 1: texel i at i/(S - 1)         */
  int32_t extent[3];        /* texels of this mip along x, y, z (z ignored in 2-D)               */
  float blend_weight;       /* used when blend_prev != NULL                                      */
  const float* blend_prev;  /* optional [Q, cout] fp32: out = (1 - w) * prev + w * sample        */
} NicSampler;
int nic_sample(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const float* coords,
               const NicSampler* s, const NicMlp* m, void* out, int out_dtype, int precision, void* stream);
/* The same from the saved model's uint8 codes (as nic_decode_codes).  Tensor-core precisions only. */
int nic_sample_codes(NicHandle* h, const NicGeom* g, const uint8_t* codes0, const uint8_t* codes1, int bits,
                     const float* coords, const NicSampler* s, const NicMlp* m, void* out, int out_dtype,
                     int precision, void* stream);

/* ---- per-query level of detail: trilinear mip filtering --------------------------------------------------- */
/* Each query carries its own LOD, given directly or computed from screen-space derivatives, and is filtered across the
 * two mips around it (2 x 4 taps in 2-D, 2 x 8 in 3-D).  For query q, with L = num_mips - 1 (every step one fp32 operation):
 *   lambda = lod[q]                                                    (LOD given), or
 *   lambda = 0.5 * log2f(max(|ddx[q] * E0|^2, |ddy[q] * E0|^2))        (derivatives of the normalised coordinates along the
 *            screen's x and y; E0 = extent[0]; |v|^2 summed x first; the isotropic rule of the GL / Vulkan specifications)
 *   lc = min(max(lambda, 0), L)                                        (fmaxf: NaN -> 0, -inf from zero derivatives -> 0)
 *   m  = floor(lc),  t = lc - m                                        (lc = L gives t = 0)
 *   out = (1 - t) * S_m + t * S_min(m+1, L)
 * S_i is nic_sample's tap sum at mip i (its extent, the chain's address mode and align_corners) in fp32, before any
 * quantisation, and the blend is the fp32 sequence of NicSampler's blend_prev; NIC_DT_U8 quantises the blended value once.
 * So NIC_PREC_F32 equals, bit for bit, scalar nic_sample calls composed the same way (at t = 0 the result is S_m).
 * F16 / BF16: one tensor-core pass, the 2 x 2^D taps of a query are adjacent rows of a tile; the row's mip is a decoder
 * input (the reference's LOD column) instead of being folded into the bias, so a result may differ from a scalar-LOD
 * tensor-core call at the same lambda by 16-bit rounding.
 * Exactly one of `lod` ([Q] fp32) or the pair `ddx`, `ddy` ([Q, D] fp32 each) is given (NIC_ERR_ARG).  Every mip is
 * validated as nic_sample validates one (NIC_ERR_BOUNDS, NIC_ERR_ARG); all mips share method, channels, PE channels and PE
 * kind, geom[i].mip_level = i and geom[i].num_blocks = Q, and num_mips is in [1, NIC_MAX_MIPS] (NIC_ERR_ARG).
 * Q * 2 * 2^D must stay below 2^31 - 128 (NIC_ERR_UNSUPPORTED).  With the triangular PE the tensor-core path needs every
 * mip's step >= 1/4, as every mip of a model has (NIC_ERR_UNSUPPORTED otherwise). */
#define NIC_MAX_MIPS 16
typedef struct NicMipChain {
  int32_t num_mips;                 /* mips 0 .. num_mips - 1 that a query may reach                                      */
  int32_t address, align_corners;   /* as NicSampler                                                                      */
  int32_t reserved;                 /* 0                                                                                  */
  NicGeom geom[NIC_MAX_MIPS];       /* mip i exactly as nic_sample takes it: num_blocks = Q, block = 1, mip_level = i      */
  const void* g0[NIC_MAX_MIPS];     /* mip i's two grids (fp32) or codes (uint8); mips of one pyramid level share them    */
  const void* g1[NIC_MAX_MIPS];
  int32_t extent[NIC_MAX_MIPS][3];  /* texels of mip i along x, y, z (z ignored in 2-D)                                   */
} NicMipChain;
int nic_sample_lod(NicHandle* h, const NicMipChain* c, const float* coords, const float* lod, const float* ddx,
                   const float* ddy, const NicMlp* m, void* out, int out_dtype, int precision, void* stream);
/* The same from the saved model's uint8 codes (as nic_sample_codes).  Tensor-core precisions only. */
int nic_sample_lod_codes(NicHandle* h, const NicMipChain* c, int bits, const float* coords, const float* lod,
                         const float* ddx, const float* ddy, const NicMlp* m, void* out, int out_dtype, int precision,
                         void* stream);

/* ---- the whole mip chain in one call --------------------------------------------------------------------- */
/* Decodes every mip 0 .. L = num_mips - 1 of a model (what a renderer uploads as a mipmapped texture; the reference's
 * process_images decodes each mip in turn, image_compression.py:400).  c->geom[i] describes mip i exactly as nic_decode takes
 * a whole-mip block: num_blocks = 1, block = c->extent[i], origin0 = 0, mip_level = i; c->g0[i] / c->g1[i] are its grids
 * (fp32) or codes (uint8); address and align_corners are not used.  Every mip is validated as nic_decode validates a
 * host-known block (NIC_ERR_BOUNDS); num_mips outside [1, NIC_MAX_MIPS], an extent < 1, geom[i].block != extent[i],
 * num_blocks != 1, a non-zero origin, mip_level != i, NULL grids or mips that differ in method, channels, PE channels or PE
 * kind give NIC_ERR_ARG.
 * out is the concatenated chain in mip order: mip i starts at row sum_{j<i} texels_j and is laid out exactly as nic_decode
 * writes that block, [Sx, Sy(, Sz), cout] with x slowest, in out_dtype (NIC_DT_F32, or NIC_DT_U8 = floor(v*255+.5)).
 *   NIC_PREC_F32: every mip equals nic_decode of that mip at NIC_PREC_F32 bit for bit (the reference-exact kernel once per mip).
 *   F16 / BF16: mip 0 is decoded exactly as nic_decode decodes it (bit for bit).  Mips 1 .. L are ONE tensor-core pass in
 *   which the mip is a decoder input, as in nic_sample_lod: texel idx of mip i equals nic_sample_lod at its centre
 *   ((idx + .5) / S per axis, align_corners 0) with lambda = i bit for bit, and may differ from a scalar nic_decode of that
 *   mip by 16-bit rounding.  The pass's rows, sum_{i>=1} texels_i, must stay below 2^31 - 128, and with the triangular PE
 *   every mip >= 1 needs step >= 1/4 (NIC_ERR_UNSUPPORTED otherwise). */
int nic_decode_mips(NicHandle* h, const NicMipChain* c, const NicMlp* m, void* out, int out_dtype, int precision,
                    void* stream);
/* The same from the saved model's uint8 codes (as nic_decode_codes).  Tensor-core precisions only. */
int nic_decode_mips_codes(NicHandle* h, const NicMipChain* c, int bits, const NicMlp* m, void* out, int out_dtype,
                          int precision, void* stream);

/* ---- applying a baked 3-D colour LUT to images ------------------------------------------------------------ */
/* A colour LUT is decoded once (nic_decode / nic_decode_codes of the whole 3-D mip, fp32 out), packed into a table of 4-channel
 * texels by nic_lut_pack (the bake), and then applied to every pixel of an image by nic_lut_apply, a pure gather: no decoder
 * runs per pixel.  Channel k of a pixel indexes LUT axis k: R -> x (the first, slowest axis of the decoded [Sx, Sy, Sz, C]),
 * G -> y, B -> z, which is nic_sample's coordinate order.  For each pixel (every step one fp32 operation):
 *   u  = NIC_DT_U8 input: __fdiv_rn((float)v, 255.f); NIC_DT_F32 input: the value as given;
 *   on each axis nic_sample's rule with align_corners = 1 and NIC_ADDRESS_CLAMP: p = u * (S - 1), clamped to +-2^24 (NaN ->
 *   -2^24), i0 = floor(p), f = p - i0; the low tap i0 and the high tap i0 + 1, each clamped to [0, S - 1];
 *   NIC_INTERP_TRILINEAR: the 8 taps, weights and order of nic_sample (x slowest; weight = product of the per-axis weights,
 *     x first), summed as acc = 0, acc = acc + w_k * v_k for k = 0..7 (each product and sum rounded): fp32 apply of a table
 *     baked at NIC_PREC_F32 equals nic_sample at NIC_PREC_F32 bit for bit;
 *   NIC_INTERP_TETRAHEDRAL: the axes ordered by descending f, ties broken x before y before z (a stable sort): a1, a2, a3.
 *     Corners v0 = c(lo), v1 = c(lo + e_a1), v2 = c(lo + e_a1 + e_a2), v3 = c(hi) (each step moves one axis from its low tap to
 *     its high tap); weights w0 = 1 - f_a1, w1 = f_a1 - f_a2, w2 = f_a2 - f_a3, w3 = f_a3; acc = 0, acc = acc + w_k * v_k for
 *     k = 0..3.  It reads 4 texels instead of 8 and reproduces the table exactly on the neutral axis of a cubic table;
 *   out: NIC_DT_F32 the fp32 result; NIC_DT_U8 floor(v * 255 + .5) of it, clamped to [0, 255] (quantised once).
 * Errors: NIC_ERR_ARG for a NULL pointer with pixels > 0, a bad dtype, cout, interp or reserved field, an extent < 1, pixels < 0
 * or src / dst overlapping (no in-place apply); NIC_ERR_UNSUPPORTED for Sx * Sy * Sz >= 2^31.  pixels == 0 launches nothing. */
enum { NIC_INTERP_TRILINEAR = 0, NIC_INTERP_TETRAHEDRAL = 1 };
typedef struct NicLut {
  const void* table;     /* [Sx][Sy][Sz][4] of table_dtype, x slowest (nic_decode's texel order); channels >= cout are 0 */
  int32_t table_dtype;   /* NIC_DT_F32 (the exact arm) or NIC_DT_F16                                               */
  int32_t cout;          /* 1..4                                                                                   */
  int32_t extent[3];     /* Sx, Sy, Sz >= 1, Sx*Sy*Sz < 2^31                                                       */
  int32_t reserved;      /* 0                                                                                      */
} NicLut;
/* dense [Sx, Sy, Sz, cout] fp32 (what nic_decode / nic_decode_codes write for a 3-D block) -> the table layout above
 * (NIC_DT_F16: __float2half_rn of each value; channels cout..3 written as 0). */
int nic_lut_pack(NicHandle* h, const float* dense, const int32_t extent[3], int cout, void* table, int table_dtype,
                 void* stream);
/* src [pixels, 3] (NIC_DT_U8 or NIC_DT_F32) -> dst [pixels, cout] (NIC_DT_U8 or NIC_DT_F32); dst must not overlap src.
 * Any element alignment of src and dst is accepted (a view that starts 3 bytes into a buffer works). */
int nic_lut_apply(NicHandle* h, const NicLut* lut, const void* src, int src_dtype, int64_t pixels, void* dst,
                  int dst_dtype, int interp, void* stream);

/* ---- fused training forward+backward (K3+K4) ----------------------------------------------------------- */
/* One step of train_models up to loss.backward() (image_compression.py:239-265).
 *   targets [N, cout] fp32; noise: NULL (no noise), or [N, Cin] fp32 injected tensor (parity tests), or use
 *   in-kernel Philox when noise == NULL and noise_bits > 0: X += (U[0,1) - .5) / 2^noise_bits with
 *   (seed, step) as the Philox key/offset (U has 24 bits on the fp32 path and 8 bits on the tensor-core paths, whose
 *   16-bit X~ cannot resolve more; the two paths draw different streams).
 *   On the tensor-core precisions the decoder gradients are summed in a fixed order (bit-reproducible); the grid
 *   gradients are scattered with float atomics (reproducible to rounding).
 *   Writes: loss_sum[0] += sum((out-target)^2) (caller divides by N*cout), gradients ACCUMULATED into
 *   gm / dg0 / dg1 (caller zeroes them), already scaled by 2/(N*cout*loss_scale_den) where loss_scale_den
 *   lets data-parallel callers pass the GLOBAL sample count (0 = use local N).
 *   dg0/dg1 may both be NULL (grids frozen, image_compression.py:227-231): the grid scatter is skipped.
 *   out (optional, may be NULL): decoder output [N, cout] fp32. */
int nic_train_step(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const int64_t* origins,
                   const NicMlp* m, const float* targets, const float* noise, int noise_bits, uint64_t seed,
                   uint64_t step, int64_t global_n, const NicMlpGrad* gm, float* dg0, float* dg1,
                   float* loss_sum, float* out, int precision, void* stream);

/* ---- optimiser (K5): torch.optim.Adam + CosineAnnealingLR + fp_quantize_clamp -------------------------- */
/* One fused Adam update of `count` tensors (image_compression.py:266-269, 361-365).  For tensor i:
 *   m,v,p updated with step count t[i] (>=1), lr[i] already cosine-scheduled by the caller, betas/eps
 *   torch defaults unless overridden; if clamp[i] != 0 the result is clamped to [clamp_lo, clamp_hi]
 *   (fp_quantize_clamp, fp_def.py:227-232).  grad_scale multiplies the gradient first (1/world for DP);
 *   if zero_grad != 0 the gradient buffer is zeroed after use. */
typedef struct NicAdamTensor {
  float* p; float* g; float* m; float* v;
  int64_t numel;
  float lr; int32_t t;
  int32_t clamp; float clamp_lo, clamp_hi;
} NicAdamTensor;
int nic_adam_step(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                  float grad_scale, int zero_grad, void* stream);
/* The same, and in the same launch: loss_out[0] = loss_sum[0] * loss_scale, loss_sum[0] = 0 — the `loss.item()`
 * bookkeeping of image_compression.py:275 without a host sync or extra kernels (the caller reads loss_out when it
 * wants to). */
int nic_adam_step_loss(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                       float grad_scale, int zero_grad, float* loss_sum, float* loss_out, float loss_scale, void* stream);

/* ---- the exchange step of data-parallel training, fused into the optimiser (NVLink peer memory) ------------------- */
/* Replaces `all_reduce(flat gradient buffer); Adam` (the one collective of the path; reference: single-GPU, so this is
 * the drop-in for what a DistributedDataParallel wrapper would add around image_compression.py:265-269) by ONE kernel:
 * every rank keeps its flat gradient buffer in IPC-shared ("symmetric") device memory, and the Adam kernel itself waits
 * until all ranks have published this step's token, reads the `world` peer buffers over NVLink in rank order (every
 * rank forms bit-identical sums, so the replicas never drift) and updates its parameters.
 *   nic_sym_alloc: cudaMalloc'ed, zero-filled memory + its 64-byte IPC handle (send it to the other ranks out of band).
 *   nic_sym_open / nic_sym_close: map / unmap another rank's allocation.  nic_sym_free: release one's own.
 * Protocol (FusedTrainer implements it): gradient buffers are double-buffered by use parity; tensors[i].g points into
 * THIS rank's current buffer `peer_flat[rank]`; peer_flat[r] / peer_flag[r] are the same buffer / the flag array (`world`
 * 32-bit words: slot s is written by rank s) of rank r; `token` increases by one per use; `zero_buf` (the OTHER parity buffer of this rank, `zero_numel` floats) is
 * cleared in the same launch — no peer can still be reading it once every flag shows `token`.
 * A timeout is FATAL and sticky: a rank that waits longer than NIC_OPT_EXCHANGE_TIMEOUT_MS for a peer applies NO update in
 * that launch nor in any later one (nobody ever consumes a partial sum, a lost peer cannot hang the GPU), and the next
 * nic_adam_step_exchange on the handle returns NIC_ERR_EXCHANGE without launching.  nic_exchange_status reports and clears the
 * flag; the caller must re-synchronise the replicas (broadcast parameters + Adam state) before it resumes.  All blocks of the
 * kernel are co-resident by construction (grid capped by occupancy), so the intra-kernel release cannot deadlock. */
#define NIC_MAX_PEERS 16
#define NIC_EXCHANGE_ONE_SHOT 0   /* every rank reads all `world` buffers (small buffers: one handshake) */
#define NIC_EXCHANGE_SLICED 1     /* rank r sums slice r of all buffers and writes it back to all; second handshake; Adam from
                                     the own buffer: 2 (world-1)/world of the buffer crosses NVLink per rank instead of world-1
                                     times.  The flag array then needs 2 NIC_MAX_PEERS words, and peer_flat must be writable. */
typedef struct NicExchange {
  int32_t world, rank;
  uint32_t token;
  int32_t reserved;           /* mode: NIC_EXCHANGE_ONE_SHOT or NIC_EXCHANGE_SLICED */
  const float* peer_flat[NIC_MAX_PEERS];
  uint32_t* peer_flag[NIC_MAX_PEERS];
  float* zero_buf;
  int64_t zero_numel;
} NicExchange;
int nic_sym_alloc(NicHandle* h, int64_t bytes, void** ptr, uint8_t ipc_handle[64]);
int nic_sym_open(NicHandle* h, const uint8_t ipc_handle[64], void** ptr);
int nic_sym_close(NicHandle* h, void* ptr);
int nic_sym_free(NicHandle* h, void* ptr);
/* nic_adam_step_loss with the gradient (and the loss sum) of every element taken as the sum over the peers' buffers. */
int nic_adam_step_exchange(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                           float grad_scale, const NicExchange* x, const float* loss_sum, float* loss_out, float loss_scale,
                           void* stream);
/* Synchronises the device and reports whether any exchange so far timed out waiting for a peer (then clears the sticky flag). */
int nic_exchange_status(NicHandle* h, int* timed_out);

/* ---- quantisers (K6) ------------------------------------------------------------------------------------ */
/* models.quantize4fp (models.py:55-57): dst = floor(src*(2^b-1)+.5)/(2^b-1), separate fp32 mul and add. */
int nic_quantize4fp(NicHandle* h, const float* src, float* dst, int64_t n, int bits, void* stream);
/* models.save4fp (models.py:61-64): code = floor(src*(2^b-1)+.5) + 2^(b-1) - 1 -> uint8, one code per byte. */
int nic_quantize_pack(NicHandle* h, const float* src, uint8_t* codes, int64_t n, int bits, void* stream);
/* models.load4fp (models.py:68-71) with the intended float result (the reference call site passes uint8 and
 * wraps, image_compression.py:396): dst = (code - 2^(b-1) + 1)/(2^b-1). */
int nic_unpack(NicHandle* h, const uint8_t* codes, float* dst, int64_t n, int bits, void* stream);
/* Sub-byte storage of the codes above (an extension: the reference's fp_savable keeps one code per byte even for
 * FP_BITS 4 / 2, fp_def.py:250-255): 8/bits codes per byte, code i in bits [(i mod 8/bits)*bits, +bits) of byte
 * i / (8/bits); bits in {1, 2, 4, 8}; `packed` holds ceil(n*bits/8) bytes. */
int nic_pack_codes(NicHandle* h, const uint8_t* codes, uint8_t* packed, int64_t n, int bits, void* stream);
int nic_unpack_codes(NicHandle* h, const uint8_t* packed, uint8_t* codes, int64_t n, int bits, void* stream);
/* fp_quantize_clamp / models.quantize_clamp (fp_def.py:227-232, models.py:48-51): in-place clamp. */
int nic_clamp(NicHandle* h, float* p, int64_t n, float lo, float hi, void* stream);
/* models.quantize_to_bit + astype(uint8) (models.py:29-40, image_compression.py:406-407):
 * dst = (uint8) floor(src*(2^b-1)+.5) for src in [0,1]. */
int nic_output_to_u8(NicHandle* h, const float* src, uint8_t* dst, int64_t n, int bits, void* stream);
/* Sum of squared differences of two 8-bit images, for utils.calculate_psnr (utils.py:117-130):
 * sse[0] += sum((a-b)^2) as float64. */
int nic_sse_u8(NicHandle* h, const uint8_t* a, const uint8_t* b, int64_t n, double* sse, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NIC_H_ */
