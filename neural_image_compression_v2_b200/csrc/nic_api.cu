// nic_api.cu — the C ABI of libnic.so (include/nic.h): argument validation, geometry flattening, dispatch.
// No torch types, no exceptions across the boundary, no CPU fallback.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

#include "nic_internal.cuh"

using namespace nic;

struct NicHandle : public Handle {};

static thread_local char g_err[256] = "no error";

static int fail(NicHandle* h, int code, const char* fmt, ...) {
  char buf[256];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) {
    strncpy(h->err, buf, sizeof(h->err) - 1);
    h->err[sizeof(h->err) - 1] = 0;
  }
  strncpy(g_err, buf, sizeof(g_err) - 1);
  return code;
}

static int cuda_fail(NicHandle* h, int e, const char* what) {
  if (e == 0) return 0;
  if (e < 0) return fail(h, e, "%s: %s", what, nic_status_string(e));
  return fail(h, e, "%s: CUDA error %d (%s)", what, e, cudaGetErrorString((cudaError_t)e));
}

extern "C" {

int nic_abi_version(void) { return NIC_ABI_VERSION; }

const char* nic_status_string(int status) {
  switch (status) {
    case NIC_OK: return "ok";
    case NIC_ERR_ARG: return "invalid argument";
    case NIC_ERR_UNSUPPORTED: return "unsupported configuration";
    case NIC_ERR_DEVICE: return "not an sm_100 device (no CPU or other-GPU fallback exists)";
    case NIC_ERR_BOUNDS: return "origin would index outside the grids";
    case NIC_ERR_ALIGN: return "misaligned pointer";
    case NIC_ERR_SCRATCH: return "scratch allocation failed";
    case NIC_ERR_EXCHANGE: return "data-parallel exchange timed out waiting for a peer";
    default: return status > 0 ? cudaGetErrorString((cudaError_t)status) : "unknown status";
  }
}

const char* nic_last_error_string(const NicHandle* h) { return h ? h->err : g_err; }

int nic_create(int device, NicHandle** out) {
  if (!out) return fail(nullptr, NIC_ERR_ARG, "nic_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(nullptr, NIC_ERR_DEVICE, "nic_create: no CUDA device visible (%s)", cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(nullptr, NIC_ERR_ARG, "nic_create: device %d out of range", device);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, (int)e, "nic_create: cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return fail(nullptr, NIC_ERR_DEVICE, "nic_create: device %d is sm_%d%d; libnic.so is built for sm_100a only", device,
                prop.major, prop.minor);
  NicHandle* h = new (std::nothrow) NicHandle();
  if (!h) return fail(nullptr, NIC_ERR_SCRATCH, "nic_create: out of host memory");
  memset(static_cast<Handle*>(h), 0, sizeof(Handle));
  h->device = device;
  h->sms = prop.multiProcessorCount;
  h->cc_major = prop.major;
  h->cc_minor = prop.minor;
  h->gelu_poly = -1;
  strcpy(h->err, "no error");
  *out = h;
  return NIC_OK;
}

int nic_destroy(NicHandle* h) {
  if (!h) return NIC_OK;
  int cur = 0;
  cudaGetDevice(&cur);
  cudaSetDevice(h->device);
  if (h->tc_weights) cudaFree(h->tc_weights);
  if (h->tc_shadow) cudaFree(h->tc_shadow);
  if (h->tc_gscratch) cudaFree(h->tc_gscratch);
  if (h->tc_partials) cudaFree(h->tc_partials);
  if (h->xch_err) cudaFree(h->xch_err);
  if (h->xch_host_err) cudaFreeHost(h->xch_host_err);
  if (h->dbg_counters) cudaFree(h->dbg_counters);
  if (h->data_scratch) cudaFree(h->data_scratch);
  if (h->sample_scratch) cudaFree(h->sample_scratch);
  if (h->lod_chain) cudaFree(h->lod_chain);
  if (h->adam_desc) cudaFree(h->adam_desc);
  for (int i = 0; i < 2 * NIC_MAX_TIMED; ++i)
    if (h->timed_ev[i]) cudaEventDestroy(h->timed_ev[i]);
  cudaSetDevice(cur);
  delete h;
  return NIC_OK;
}

int64_t nic_launch_count(const NicHandle* h) { return h ? h->launches : 0; }

int nic_set_option(NicHandle* h, int option, int value) {
  if (!h) return fail(nullptr, NIC_ERR_ARG, "handle is NULL");
  if (option == NIC_OPT_DISABLE_FAST2D) { h->disable_fast2d = value != 0; return NIC_OK; }
  if (option == NIC_OPT_DEBUG_KNOCKOUT) { h->debug_flags = value; return NIC_OK; }
  if (option == NIC_OPT_REUSE_PREPARED) { h->reuse_prepared = value != 0; return NIC_OK; }
  if (option == NIC_OPT_TIME_KERNELS) { h->time_kernels = value != 0; h->timed_count = 0; return NIC_OK; }
  if (option == NIC_OPT_STEP_METRICS) { h->step_metrics = value != 0; return NIC_OK; }
  if (option == NIC_OPT_STATIC_TILES) { h->static_tiles = value != 0; return NIC_OK; }
  if (option == NIC_OPT_EXCHANGE_TIMEOUT_MS) {
    if (value < 0) return fail(h, NIC_ERR_ARG, "nic_set_option: NIC_OPT_EXCHANGE_TIMEOUT_MS must be >= 0 (0 = default)");
    h->xch_timeout_ms = value;
    return NIC_OK;
  }
  if (option == NIC_OPT_GELU_POLY) {
    if (value < -1 || value > 8) return fail(h, NIC_ERR_ARG, "nic_set_option: NIC_OPT_GELU_POLY takes -1 (default) or 0..8");
    h->gelu_poly = value;
    return NIC_OK;
  }
  return fail(h, NIC_ERR_ARG, "nic_set_option: unknown option %d", option);
}

int nic_kernel_time_ms(NicHandle* h, double* total_ms, int64_t* launches) {
  if (!h || !total_ms || !launches) return fail(h, NIC_ERR_ARG, "nic_kernel_time_ms: NULL argument");
  double sum = 0.0;
  for (int i = 0; i < h->timed_count; ++i) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(h->timed_ev[2 * i + 1]);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, h->timed_ev[2 * i], h->timed_ev[2 * i + 1]);
    if (e != cudaSuccess) return fail(h, (int)e, "nic_kernel_time_ms: %s", cudaGetErrorString(e));
    sum += ms;
  }
  *total_ms = sum;
  *launches = h->timed_count;
  h->timed_count = 0;
  return NIC_OK;
}

int nic_debug_counters(NicHandle* h, int64_t* out, int n) {
  if (!h || !out || n < 0 || n > 16) return fail(h, NIC_ERR_ARG, "nic_debug_counters: bad argument");
  for (int i = 0; i < n; ++i) out[i] = 0;
  if (!h->dbg_counters) return NIC_OK;
  int cur = 0;
  cudaGetDevice(&cur);
  cudaSetDevice(h->device);
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out, h->dbg_counters, (size_t)n * 8, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemset(h->dbg_counters, 0, 16 * 8);
  cudaSetDevice(cur);
  if (e != cudaSuccess) return fail(h, (int)e, "nic_debug_counters: %s", cudaGetErrorString(e));
  return NIC_OK;
}

int nic_cin(const NicGeom* g) {
  if (!g) return NIC_ERR_ARG;
  int dim = g->method == NIC_METHOD_2D ? 2 : 3;
  int corners = g->method == NIC_METHOD_3D ? 8 : 4;
  return g->channels * (corners + 1) + g->pe_channels * dim + 1;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ helpers
static int flatten_geom(NicHandle* h, const NicGeom* g, bool have_origins, DevGeom* d) {
  if (!g) return fail(h, NIC_ERR_ARG, "geometry is NULL");
  if (g->method != NIC_METHOD_2D && g->method != NIC_METHOD_3D && g->method != NIC_METHOD_3D_V2)
    return fail(h, NIC_ERR_UNSUPPORTED, "method %d (expected 1, 3 or 4)", g->method);
  memset(d, 0, sizeof(*d));
  d->method = g->method;
  d->dim = g->method == NIC_METHOD_2D ? 2 : 3;
  d->ncorner0 = g->method == NIC_METHOD_3D ? 8 : 4;
  d->C = g->channels;
  d->PE = g->pe_channels;
  d->pe_kind = g->pe_kind;
  if (d->C < 1 || d->PE < 0 || d->PE > NIC_MAX_PE) return fail(h, NIC_ERR_UNSUPPORTED, "channels %d / pe_channels %d", d->C, d->PE);
  if (g->pe_kind != NIC_PE_TRIANGULAR && g->pe_kind != NIC_PE_SINUSOIDAL) return fail(h, NIC_ERR_ARG, "pe_kind %d", g->pe_kind);
  d->cin = d->C * (d->ncorner0 + 1) + d->PE * d->dim + 1;
  if (d->cin > NIC_MAX_CIN) return fail(h, NIC_ERR_UNSUPPORTED, "decoder input width %d > %d", d->cin, NIC_MAX_CIN);
  d->mip = g->mip_level;
  d->lod = (float)g->mip_level;
  if (g->step_log2 < -24 || g->step_log2 > 24) return fail(h, NIC_ERR_ARG, "step_log2 %d", g->step_log2);
  d->step = ldexpf(1.0f, g->step_log2);
  d->interp = g->step_log2 != 1;                 // fp_def.py:136: int(1 // (step/2)) != 1
  d->nblocks = g->num_blocks;
  if (g->num_blocks < 0) return fail(h, NIC_ERR_ARG, "num_blocks %d", g->num_blocks);
  d->per_block = 1;
  for (int a = 0; a < 3; ++a) {
    bool used = a < d->dim;
    d->n0[a] = used ? g->g0_nodes[a] : 1;
    d->n1[a] = used ? g->g1_nodes[a] : 1;
    d->B[a] = used ? g->block[a] : 1;
    d->origin0[a] = used ? g->origin0[a] : 0;
    if (used && (d->n0[a] < 2 || d->n1[a] < 2)) return fail(h, NIC_ERR_ARG, "grid axis %d has < 2 nodes", a);
    if (d->B[a] < 0) return fail(h, NIC_ERR_ARG, "block extent %d on axis %d", d->B[a], a);
    d->per_block *= d->B[a];
  }
  d->N = d->per_block * d->nblocks;
  {
    long long divs[3] = {d->per_block, (long long)d->B[1] * d->B[2], d->B[2]};
    for (int i = 0; i < 3; ++i) {
      unsigned long long dv = divs[i] > 0 ? (unsigned long long)divs[i] : 1ull;
      unsigned sh = 0;
      while ((1ull << sh) < dv) ++sh;
      if (dv >= (1ull << 31)) { d->fd_mul[i] = 0; d->fd_shift[i] = 0; continue; }   // quotient is 0 for n < 2^31
      unsigned long long num = 1ull << (31 + sh);
      d->fd_mul[i] = (unsigned)((num + dv - 1) / dv);
      d->fd_shift[i] = sh;
    }
  }
  for (int i = 0; i < NIC_MAX_PE; ++i) d->pe_div[i] = g->pe_div[i];
  if (!have_origins) {
    if (d->nblocks > 1) return fail(h, NIC_ERR_ARG, "origins is NULL but num_blocks = %d", d->nblocks);
    // host-known origin: reproduce the reference's IndexError instead of clamping silently
    for (int a = 0; a < d->dim && d->N > 0; ++a) {
      double last = (double)(d->origin0[a] + d->B[a] - 1) * (double)d->step;
      long long i0 = (long long)floor(last), i1 = (long long)floor(last / 2);
      if (d->origin0[a] < 0 || i0 + 1 >= d->n0[a] || i1 + 1 >= d->n1[a])
        return fail(h, NIC_ERR_BOUNDS, "axis %d: origin %d + block %d at step %g reaches node %lld/%lld of %d/%d", a,
                    d->origin0[a], d->B[a], (double)d->step, i0 + 1, i1 + 1, d->n0[a], d->n1[a]);
    }
  }
  return NIC_OK;
}

static int flatten_mlp(NicHandle* h, const NicMlp* m, MlpDev* d, int expect_cin) {
  if (!m || !m->w1 || !m->b1 || !m->w2 || !m->b2 || !m->w3 || !m->b3) return fail(h, NIC_ERR_ARG, "MLP descriptor has NULL tensors");
  if (expect_cin > 0 && m->cin != expect_cin) return fail(h, NIC_ERR_ARG, "MLP cin %d != geometry cin %d", m->cin, expect_cin);
  if (m->cin < 1 || m->cin > NIC_MAX_CIN) return fail(h, NIC_ERR_UNSUPPORTED, "MLP cin %d", m->cin);
  if (m->cout < 1 || m->cout > NIC_MAX_COUT) return fail(h, NIC_ERR_UNSUPPORTED, "MLP cout %d", m->cout);
  if (m->hidden != 64 && m->hidden != 32) return fail(h, NIC_ERR_UNSUPPORTED, "MLP hidden %d (32 or 64)", m->hidden);
  d->cin = m->cin; d->hidden = m->hidden; d->cout = m->cout;
  d->w1 = m->w1; d->b1 = m->b1; d->w2 = m->w2; d->b2 = m->b2; d->w3 = m->w3; d->b3 = m->b3;
  return NIC_OK;
}

struct DeviceGuard {
  int prev;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define NIC_ENTER(h)                                         \
  if (!(h)) return fail(nullptr, NIC_ERR_ARG, "handle is NULL"); \
  DeviceGuard guard_((h)->device);                           \
  cudaStream_t st = (cudaStream_t)stream

extern "C" {

int nic_gather(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const int64_t* origins, void* x,
               int x_dtype, void* stream) {
  NIC_ENTER(h);
  DevGeom d;
  int rc = flatten_geom(h, g, origins != nullptr, &d);
  if (rc) return rc;
  if (!g0 || !g1 || (!x && d.N > 0)) return fail(h, NIC_ERR_ARG, "nic_gather: NULL pointer");
  return cuda_fail(h, launch_gather(h, d, g0, g1, (const long long*)origins, x, x_dtype, st), "nic_gather");
}

int nic_scatter(NicHandle* h, const NicGeom* g, const float* dx, const int64_t* origins, float* dg0, float* dg1,
                void* stream) {
  NIC_ENTER(h);
  DevGeom d;
  int rc = flatten_geom(h, g, origins != nullptr, &d);
  if (rc) return rc;
  if ((!dx && d.N > 0) || !dg0 || !dg1) return fail(h, NIC_ERR_ARG, "nic_scatter: NULL pointer");
  return cuda_fail(h, launch_scatter(h, d, dx, (const long long*)origins, dg0, dg1, st), "nic_scatter");
}

int nic_sample_crops(NicHandle* h, const float* image, int dim, int channels, const int32_t* size, const int64_t* origins,
                     int num_crops, const int32_t* crop, float* targets, void* stream) {
  NIC_ENTER(h);
  if ((dim != 2 && dim != 3) || channels < 1 || num_crops < 0 || !size || !crop)
    return fail(h, NIC_ERR_ARG, "nic_sample_crops: dim %d channels %d num_crops %d", dim, channels, num_crops);
  for (int a = 0; a < dim; ++a)
    if (size[a] < 1 || crop[a] < 0 || crop[a] > size[a]) return fail(h, NIC_ERR_ARG, "nic_sample_crops: axis %d size %d crop %d", a, size[a], crop[a]);
  if (num_crops > 0 && (!image || !origins || !targets)) return fail(h, NIC_ERR_ARG, "nic_sample_crops: NULL pointer");
  int rc = launch_sample_crops(h, image, dim, channels, size, (const long long*)origins, num_crops, crop, targets, st);
  if (rc == NIC_ERR_UNSUPPORTED) return fail(h, rc, "nic_sample_crops: num_crops * 12 + 1 KB * (channels | 1) must fit 48 KB of shared memory");
  return cuda_fail(h, rc, "nic_sample_crops");
}

int nic_sample_crops_random(NicHandle* h, const float* image, int dim, int channels, const int32_t* size, int num_crops,
                            const int32_t* crop, uint64_t seed, uint64_t step, int64_t* origins_out, float* targets, void* stream) {
  NIC_ENTER(h);
  if ((dim != 2 && dim != 3) || channels < 1 || num_crops < 0 || !size || !crop)
    return fail(h, NIC_ERR_ARG, "nic_sample_crops_random: dim %d channels %d num_crops %d", dim, channels, num_crops);
  for (int a = 0; a < dim; ++a)
    if (size[a] < 1 || crop[a] < 1 || crop[a] > size[a])
      return fail(h, NIC_ERR_ARG, "nic_sample_crops_random: axis %d size %d crop %d", a, size[a], crop[a]);
  if (num_crops > 0 && (!image || !origins_out || !targets)) return fail(h, NIC_ERR_ARG, "nic_sample_crops_random: NULL pointer");
  int rc = launch_sample_crops_random(h, image, dim, channels, size, num_crops, crop, seed, step, (long long*)origins_out, targets, st);
  if (rc == NIC_ERR_UNSUPPORTED) return fail(h, rc, "nic_sample_crops_random: num_crops * 12 + 1 KB * (channels | 1) must fit 48 KB of shared memory");
  return cuda_fail(h, rc, "nic_sample_crops_random");
}

int nic_resize_bilinear_u8(NicHandle* h, const uint8_t* src, int height, int width, int channels, int out_height, int out_width,
                           uint8_t* dst_u8, float* dst_f32, void* stream) {
  NIC_ENTER(h);
  if (height < 1 || width < 1 || channels < 1 || out_height < 1 || out_width < 1)
    return fail(h, NIC_ERR_ARG, "nic_resize_bilinear_u8: %dx%dx%d -> %dx%d", height, width, channels, out_height, out_width);
  if (!src || (!dst_u8 && !dst_f32)) return fail(h, NIC_ERR_ARG, "nic_resize_bilinear_u8: NULL pointer");
  int rc = launch_resize_bilinear_u8(h, src, height, width, channels, out_height, out_width, dst_u8, dst_f32, st);
  if (rc == NIC_ERR_SCRATCH) return fail(h, rc, "nic_resize_bilinear_u8: scratch allocation failed");
  return cuda_fail(h, rc, "nic_resize_bilinear_u8");
}

static int check_atlas(NicHandle* h, int num_frames, int frame_size, int channels, int atlas_size, const char* who) {
  if (num_frames < 0 || frame_size < 1 || channels < 1 || atlas_size < frame_size)
    return fail(h, NIC_ERR_ARG, "%s: %d frames of %d^2 x %d into %d^2", who, num_frames, frame_size, channels, atlas_size);
  const long long per_row = atlas_size / frame_size;
  if (per_row * per_row < num_frames) return fail(h, NIC_ERR_ARG, "%s: %d frames do not fit a %d^2 atlas", who, num_frames, atlas_size);
  return NIC_OK;
}

int nic_atlas_pack(NicHandle* h, const uint8_t* frames, int num_frames, int frame_size, int channels, int atlas_size,
                   uint8_t* atlas, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_atlas(h, num_frames, frame_size, channels, atlas_size, "nic_atlas_pack")) return rc;
  if (!atlas || (num_frames > 0 && !frames)) return fail(h, NIC_ERR_ARG, "nic_atlas_pack: NULL pointer");
  return cuda_fail(h, launch_atlas(h, const_cast<uint8_t*>(frames), atlas, num_frames, frame_size, channels, atlas_size, 0, st),
                   "nic_atlas_pack");
}

int nic_atlas_unpack(NicHandle* h, const uint8_t* atlas, int atlas_size, int channels, int num_frames, int frame_size,
                     uint8_t* frames, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_atlas(h, num_frames, frame_size, channels, atlas_size, "nic_atlas_unpack")) return rc;
  if (!atlas || (num_frames > 0 && !frames)) return fail(h, NIC_ERR_ARG, "nic_atlas_unpack: NULL pointer");
  return cuda_fail(h, launch_atlas(h, frames, const_cast<uint8_t*>(atlas), num_frames, frame_size, channels, atlas_size, 1, st),
                   "nic_atlas_unpack");
}

int nic_positional_encoding(NicHandle* h, const float* coord, int dim, int64_t n, int pe_channels, int pe_kind,
                            const float* pe_div, float* out, void* stream) {
  NIC_ENTER(h);
  if (dim < 1 || dim > 3 || n < 0 || pe_channels < 0 || pe_channels > NIC_MAX_PE) return fail(h, NIC_ERR_ARG, "nic_positional_encoding: dim %d pe %d", dim, pe_channels);
  if (pe_kind != NIC_PE_TRIANGULAR && pe_kind != NIC_PE_SINUSOIDAL) return fail(h, NIC_ERR_ARG, "nic_positional_encoding: kind %d", pe_kind);
  if (pe_kind == NIC_PE_SINUSOIDAL && !pe_div) return fail(h, NIC_ERR_ARG, "nic_positional_encoding: pe_div is NULL");
  if (n > 0 && (!coord || !out)) return fail(h, NIC_ERR_ARG, "nic_positional_encoding: NULL pointer");
  return cuda_fail(h, launch_pe(h, coord, dim, n, pe_channels, pe_kind, pe_div, out, st), "nic_positional_encoding");
}

int nic_mlp_forward(NicHandle* h, const NicMlp* m, const float* x, int64_t ldx, int64_t n, float* out, float* z1,
                    float* z2, void* stream) {
  NIC_ENTER(h);
  MlpDev md;
  int rc = flatten_mlp(h, m, &md, 0);
  if (rc) return rc;
  if (n < 0 || ldx < md.cin) return fail(h, NIC_ERR_ARG, "nic_mlp_forward: n %lld ldx %lld", (long long)n, (long long)ldx);
  if (n > 0 && (!x || !out)) return fail(h, NIC_ERR_ARG, "nic_mlp_forward: NULL pointer");
  if ((((uintptr_t)z1 | (uintptr_t)z2) & 15) != 0) return fail(h, NIC_ERR_ALIGN, "nic_mlp_forward: z1/z2 must be 16-byte aligned");
  return cuda_fail(h, launch_mlp_forward_f32(h, nullptr, md, nullptr, nullptr, nullptr, x, ldx, n, out, NIC_DT_F32, z1, z2, st),
                   "nic_mlp_forward");
}

int nic_mlp_backward(NicHandle* h, const NicMlp* m, const float* x, int64_t ldx, int64_t n, const float* z1,
                     const float* z2, const float* out, const float* dout, const NicMlpGrad* gm, float* dx,
                     void* stream) {
  NIC_ENTER(h);
  MlpDev md;
  int rc = flatten_mlp(h, m, &md, 0);
  if (rc) return rc;
  if (!gm || !gm->w1 || !gm->b1 || !gm->w2 || !gm->b2 || !gm->w3 || !gm->b3) return fail(h, NIC_ERR_ARG, "nic_mlp_backward: NULL gradient tensor");
  if (n < 0 || ldx < md.cin) return fail(h, NIC_ERR_ARG, "nic_mlp_backward: n %lld ldx %lld", (long long)n, (long long)ldx);
  if (n > 0 && (!x || !z1 || !z2 || !out || !dout)) return fail(h, NIC_ERR_ARG, "nic_mlp_backward: NULL pointer");
  MlpGradDev gd = {gm->w1, gm->b1, gm->w2, gm->b2, gm->w3, gm->b3};
  return cuda_fail(h, launch_mlp_backward_f32(h, md, gd, x, ldx, n, z1, z2, out, dout, dx, st), "nic_mlp_backward");
}

// Each decode / sampling entry point and its *_codes twin share one body.  `codes` says which of the two was called: the
// grids are float32 (bits is 0) or uint8 codes of width bits.  It is a flag of its own because a codes call with bits 0
// must be refused, not read as floats.
// check_call: the checks a call makes once its geometry and MLP are flattened, in this order: the code width of a codes
// call (1..8), the NULL pointers, out_dtype, the precision.  Codes are read by the tensor-core kernels only.
static int check_call(NicHandle* h, bool codes, int bits, bool null_ptr, const char* null_msg, int out_dtype, int precision,
                      const char* who) {
  if (codes && (bits < 1 || bits > 8)) return fail(h, NIC_ERR_ARG, "%s: bits %d (1..8)", who, bits);
  if (null_ptr) return fail(h, NIC_ERR_ARG, "%s: %s", who, null_msg);
  if (out_dtype != NIC_DT_F32 && out_dtype != NIC_DT_U8) return fail(h, NIC_ERR_ARG, "%s: out_dtype %d", who, out_dtype);
  if (codes && precision != NIC_PREC_F16 && precision != NIC_PREC_BF16)
    return fail(h, NIC_ERR_UNSUPPORTED, "%s: tensor-core precisions only (f16 / bf16); unpack the codes for NIC_PREC_F32", who);
  if (precision != NIC_PREC_F32 && precision != NIC_PREC_F16 && precision != NIC_PREC_BF16)
    return fail(h, NIC_ERR_ARG, "%s: precision %d", who, precision);
  return NIC_OK;
}

static int decode_impl(NicHandle* h, const NicGeom* g, const void* g0, const void* g1, bool codes, int bits,
                       const int64_t* origins, const NicMlp* m, void* out, int out_dtype, int precision, void* stream) {
  NIC_ENTER(h);
  const char* who = codes ? "nic_decode_codes" : "nic_decode";
  DevGeom d;
  int rc = flatten_geom(h, g, origins != nullptr, &d);
  if (rc) return rc;
  MlpDev md;
  rc = flatten_mlp(h, m, &md, d.cin);
  if (rc) return rc;
  rc = check_call(h, codes, bits, !g0 || !g1 || (!out && d.N > 0), "NULL pointer", out_dtype, precision, who);
  if (rc) return rc;
  if (precision == NIC_PREC_F32)
    return cuda_fail(h, launch_mlp_forward_f32(h, &d, md, (const float*)g0, (const float*)g1, (const long long*)origins, nullptr,
                                               0, d.N, out, out_dtype, nullptr, nullptr, st), "nic_decode(f32)");
  return cuda_fail(h, launch_decode_tc(h, d, md, g0, g1, bits, (const long long*)origins, out, out_dtype, precision, st),
                   codes ? who : "nic_decode(tensor core)");
}

int nic_decode(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const int64_t* origins,
               const NicMlp* m, void* out, int out_dtype, int precision, void* stream) {
  return decode_impl(h, g, g0, g1, false, 0, origins, m, out, out_dtype, precision, stream);
}

int nic_decode_codes(NicHandle* h, const NicGeom* g, const uint8_t* codes0, const uint8_t* codes1, int bits,
                     const int64_t* origins, const NicMlp* m, void* out, int out_dtype, int precision, void* stream) {
  return decode_impl(h, g, codes0, codes1, true, bits, origins, m, out, out_dtype, precision, stream);
}

// Geometry of a sampling call: the mip is validated like a host-known block (origin 0, block = extent), then described as
// num_blocks one-texel queries.
static int flatten_sampler(NicHandle* h, const NicGeom* g, const NicSampler* s, const float* coords, DevGeom* d,
                           DevSampler* ds, const char* who) {
  if (!g || !s) return fail(h, NIC_ERR_ARG, "%s: geometry or sampler is NULL", who);
  if (s->address != NIC_ADDRESS_CLAMP && s->address != NIC_ADDRESS_WRAP) return fail(h, NIC_ERR_ARG, "%s: address mode %d", who, s->address);
  if (g->num_blocks < 0) return fail(h, NIC_ERR_ARG, "%s: num_blocks %d", who, g->num_blocks);
  if (g->num_blocks > 0 && !coords) return fail(h, NIC_ERR_ARG, "%s: coords is NULL", who);
  const int dim = g->method == NIC_METHOD_2D ? 2 : 3;
  NicGeom whole = *g;
  whole.num_blocks = 1;
  for (int a = 0; a < 3; ++a) {
    if (a < dim && s->extent[a] < 1) return fail(h, NIC_ERR_ARG, "%s: extent %d on axis %d", who, s->extent[a], a);
    if (a < dim && g->block[a] != 1) return fail(h, NIC_ERR_ARG, "%s: block must be 1 (one query per block)", who);
    whole.block[a] = a < dim ? s->extent[a] : 1;
    whole.origin0[a] = 0;
  }
  int rc = flatten_geom(h, &whole, false, d);
  if (rc) return rc;
  if (((long long)g->num_blocks << dim) >= (1ll << 31) - 128)
    return fail(h, NIC_ERR_UNSUPPORTED, "%s: %d queries x %d taps reach 2^31 - 128 rows; split the batch", who, g->num_blocks, 1 << dim);
  d->nblocks = g->num_blocks;
  for (int a = 0; a < 3; ++a) d->B[a] = 1;
  d->per_block = 1;
  d->N = g->num_blocks;
  memset(ds, 0, sizeof(*ds));
  ds->coords = coords;
  for (int a = 0; a < 3; ++a) ds->S[a] = a < dim ? s->extent[a] : 1;
  ds->address = s->address;
  ds->align_corners = s->align_corners != 0;
  ds->blend_weight = s->blend_weight;
  ds->prev = s->blend_prev;
  return NIC_OK;
}

static int sample_impl(NicHandle* h, const NicGeom* g, const void* g0, const void* g1, bool codes, int bits,
                       const float* coords, const NicSampler* s, const NicMlp* m, void* out, int out_dtype, int precision,
                       void* stream) {
  NIC_ENTER(h);
  const char* who = codes ? "nic_sample_codes" : "nic_sample";
  DevGeom d;
  DevSampler ds;
  int rc = flatten_sampler(h, g, s, coords, &d, &ds, who);
  if (rc) return rc;
  MlpDev md;
  rc = flatten_mlp(h, m, &md, d.cin);
  if (rc) return rc;
  rc = check_call(h, codes, bits, !g0 || !g1 || (!out && d.N > 0), "NULL pointer", out_dtype, precision, who);
  if (rc) return rc;
  if (precision == NIC_PREC_F32)
    return cuda_fail(h, launch_sample_f32(h, d, ds, md, (const float*)g0, (const float*)g1, out, out_dtype, st),
                     "nic_sample(f32)");
  return cuda_fail(h, launch_sample_tc(h, d, ds, md, g0, g1, bits, out, out_dtype, precision, st),
                   codes ? who : "nic_sample(tensor core)");
}

int nic_sample(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const float* coords,
               const NicSampler* s, const NicMlp* m, void* out, int out_dtype, int precision, void* stream) {
  return sample_impl(h, g, g0, g1, false, 0, coords, s, m, out, out_dtype, precision, stream);
}

int nic_sample_codes(NicHandle* h, const NicGeom* g, const uint8_t* codes0, const uint8_t* codes1, int bits,
                     const float* coords, const NicSampler* s, const NicMlp* m, void* out, int out_dtype,
                     int precision, void* stream) {
  return sample_impl(h, g, codes0, codes1, true, bits, coords, s, m, out, out_dtype, precision, stream);
}

// Mip i of a nic_decode_mips chain: one block that covers the whole mip (num_blocks 1, block = extent, origin 0), validated as
// nic_decode validates a host-known block.
static int flatten_whole_mip(NicHandle* h, const NicGeom* g, const int32_t* extent, int i, DevGeom* d, const char* who) {
  const int dim = g->method == NIC_METHOD_2D ? 2 : 3;
  if (g->num_blocks != 1) return fail(h, NIC_ERR_ARG, "%s: geom[%d].num_blocks is %d (one whole-mip block)", who, i, g->num_blocks);
  for (int a = 0; a < dim; ++a) {
    if (extent[a] < 1) return fail(h, NIC_ERR_ARG, "%s: extent %d of mip %d on axis %d", who, extent[a], i, a);
    if (g->block[a] != extent[a] || g->origin0[a] != 0)
      return fail(h, NIC_ERR_ARG, "%s: geom[%d] must be the whole mip (block = extent, origin 0) on axis %d", who, i, a);
  }
  return flatten_geom(h, g, false, d);
}

// Every mip of a chain, validated as flatten_sampler validates one (whole false: a sampling call's Q queries) or as
// flatten_whole_mip does (whole true: nic_decode_mips), and the chain's shared description: method, channels and PE.
static int flatten_mips(NicHandle* h, const NicMipChain* c, const float* coords, bool whole, DevGeom* d, DevChain* dc,
                        DevSampler* ds, const char* who) {
  if (!c) return fail(h, NIC_ERR_ARG, "%s: chain is NULL", who);
  if (c->num_mips < 1 || c->num_mips > NIC_MAX_MIPS) return fail(h, NIC_ERR_ARG, "%s: num_mips %d (1..%d)", who, c->num_mips, NIC_MAX_MIPS);
  memset(dc, 0, sizeof(*dc));
  for (int i = 0; i < c->num_mips; ++i) {
    int rc;
    if (whole) {
      rc = flatten_whole_mip(h, &c->geom[i], c->extent[i], i, &d[i], who);
    } else {
      NicSampler s;
      memset(&s, 0, sizeof(s));
      s.address = c->address;
      s.align_corners = c->align_corners;
      for (int a = 0; a < 3; ++a) s.extent[a] = c->extent[i][a];
      rc = flatten_sampler(h, &c->geom[i], &s, coords, &d[i], ds, who);
    }
    if (rc) return rc;
    if (c->geom[i].mip_level != i) return fail(h, NIC_ERR_ARG, "%s: geom[%d].mip_level is %d", who, i, c->geom[i].mip_level);
    if (!c->g0[i] || !c->g1[i]) return fail(h, NIC_ERR_ARG, "%s: grids of mip %d are NULL", who, i);
    if (d[i].method != d[0].method || d[i].C != d[0].C || d[i].PE != d[0].PE || d[i].pe_kind != d[0].pe_kind ||
        d[i].nblocks != d[0].nblocks || memcmp(d[i].pe_div, d[0].pe_div, sizeof(d[0].pe_div)) != 0)
      return fail(h, NIC_ERR_ARG, "%s: mip %d differs from mip 0 in method, channels, PE or query count", who, i);
    DevMip& mp = dc->mip[i];
    for (int a = 0; a < 3; ++a) { mp.n0[a] = d[i].n0[a]; mp.n1[a] = d[i].n1[a]; mp.S[a] = a < d[i].dim ? c->extent[i][a] : 1; }
    mp.step = d[i].step;
    mp.interp = d[i].interp;
    const int k = c->geom[i].step_log2 + 2;
    mp.lut_shift = k < 0 ? 0 : (k > 6 ? 6 : k);
  }
  dc->num_mips = c->num_mips;
  dc->dim = d[0].dim;
  return NIC_OK;
}

// Geometry of a per-query-LOD call: every mip validated as flatten_sampler validates one, the chain's shared description,
// and exactly one LOD source.
static int flatten_chain(NicHandle* h, const NicMipChain* c, const float* coords, const float* lod, const float* ddx,
                         const float* ddy, DevGeom* d, DevChain* dc, DevSampler* ds, const char* who) {
  if (!((lod && !ddx && !ddy) || (!lod && ddx && ddy)))
    return fail(h, NIC_ERR_ARG, "%s: give exactly one of lod or the pair ddx / ddy", who);
  int rc = flatten_mips(h, c, coords, false, d, dc, ds, who);
  if (rc) return rc;
  if (((long long)d[0].nblocks << (d[0].dim + 1)) >= (1ll << 31) - 128)
    return fail(h, NIC_ERR_UNSUPPORTED, "%s: %d queries x %d taps reach 2^31 - 128 rows; split the batch", who, d[0].nblocks,
                2 << d[0].dim);
  ds->S[0] = ds->S[1] = ds->S[2] = 1;                // per mip: DevMip::S
  dc->address = ds->address;
  dc->align_corners = ds->align_corners;
  dc->lod = lod;
  dc->ddx = ddx;
  dc->ddy = ddy;
  for (int a = 0; a < 3; ++a) dc->E0[a] = a < d[0].dim ? (float)c->extent[0][a] : 1.0f;
  return NIC_OK;
}

static int sample_lod_impl(NicHandle* h, const NicMipChain* c, bool codes, int bits, const float* coords, const float* lod,
                           const float* ddx, const float* ddy, const NicMlp* m, void* out, int out_dtype, int precision,
                           void* stream) {
  NIC_ENTER(h);
  const char* who = codes ? "nic_sample_lod_codes" : "nic_sample_lod";
  DevGeom d[NIC_MAX_MIPS];
  DevChain dc;
  DevSampler ds;
  int rc = flatten_chain(h, c, coords, lod, ddx, ddy, d, &dc, &ds, who);
  if (rc) return rc;
  MlpDev md;
  rc = flatten_mlp(h, m, &md, d[0].cin);
  if (rc) return rc;
  rc = check_call(h, codes, bits, !out && d[0].N > 0, "out is NULL", out_dtype, precision, who);
  if (rc) return rc;
  if (precision == NIC_PREC_F32)
    return cuda_fail(h, launch_sample_lod_f32(h, d, dc, ds, md, reinterpret_cast<const float* const*>(c->g0),
                                              reinterpret_cast<const float* const*>(c->g1), out, out_dtype, st),
                     "nic_sample_lod(f32)");
  return cuda_fail(h, launch_sample_lod_tc(h, d, dc, ds, md, c->g0, c->g1, bits, out, out_dtype, precision, st),
                   codes ? who : "nic_sample_lod(tensor core)");
}

int nic_sample_lod(NicHandle* h, const NicMipChain* c, const float* coords, const float* lod, const float* ddx,
                   const float* ddy, const NicMlp* m, void* out, int out_dtype, int precision, void* stream) {
  return sample_lod_impl(h, c, false, 0, coords, lod, ddx, ddy, m, out, out_dtype, precision, stream);
}

int nic_sample_lod_codes(NicHandle* h, const NicMipChain* c, int bits, const float* coords, const float* lod,
                         const float* ddx, const float* ddy, const NicMlp* m, void* out, int out_dtype, int precision,
                         void* stream) {
  return sample_lod_impl(h, c, true, bits, coords, lod, ddx, ddy, m, out, out_dtype, precision, stream);
}

static int decode_mips_impl(NicHandle* h, const NicMipChain* c, bool codes, int bits, const NicMlp* m, void* out, int out_dtype,
                            int precision, void* stream) {
  NIC_ENTER(h);
  const char* who = codes ? "nic_decode_mips_codes" : "nic_decode_mips";
  DevGeom d[NIC_MAX_MIPS];
  DevChain dc;
  int rc = flatten_mips(h, c, nullptr, true, d, &dc, nullptr, who);
  if (rc) return rc;
  MlpDev md;
  rc = flatten_mlp(h, m, &md, d[0].cin);
  if (rc) return rc;
  rc = check_call(h, codes, bits, !out, "out is NULL", out_dtype, precision, who);
  if (rc) return rc;
  if (precision == NIC_PREC_F32) {                   // the reference-exact kernel once per mip, into its slice of out
    uint8_t* o = (uint8_t*)out;
    for (int i = 0; i < c->num_mips; ++i) {
      rc = launch_mlp_forward_f32(h, &d[i], md, (const float*)c->g0[i], (const float*)c->g1[i], nullptr, nullptr, 0, d[i].N, o,
                                  out_dtype, nullptr, nullptr, st);
      if (rc) return cuda_fail(h, rc, "nic_decode_mips(f32)");
      o += (size_t)d[i].N * md.cout * (out_dtype == NIC_DT_U8 ? 1 : sizeof(float));
    }
    return NIC_OK;
  }
  return cuda_fail(h, launch_decode_mips_tc(h, d, dc, md, c->g0, c->g1, bits, out, out_dtype, precision, st),
                   codes ? who : "nic_decode_mips(tensor core)");
}

int nic_decode_mips(NicHandle* h, const NicMipChain* c, const NicMlp* m, void* out, int out_dtype, int precision, void* stream) {
  return decode_mips_impl(h, c, false, 0, m, out, out_dtype, precision, stream);
}

int nic_decode_mips_codes(NicHandle* h, const NicMipChain* c, int bits, const NicMlp* m, void* out, int out_dtype,
                          int precision, void* stream) {
  return decode_mips_impl(h, c, true, bits, m, out, out_dtype, precision, stream);
}

// Texels of a LUT extent: NIC_ERR_ARG for an extent < 1, NIC_ERR_UNSUPPORTED from 2^31 texels on (int texel indices).
static int lut_texels(NicHandle* h, const int32_t* extent, long long* texels, const char* who) {
  if (!extent) return fail(h, NIC_ERR_ARG, "%s: extent is NULL", who);
  for (int a = 0; a < 3; ++a)
    if (extent[a] < 1) return fail(h, NIC_ERR_ARG, "%s: extent %d on axis %d", who, extent[a], a);
  *texels = (long long)extent[0] * extent[1] * extent[2];
  if (*texels >= (1ll << 31)) return fail(h, NIC_ERR_UNSUPPORTED, "%s: %lld texels reach 2^31", who, *texels);
  return NIC_OK;
}

int nic_lut_pack(NicHandle* h, const float* dense, const int32_t extent[3], int cout, void* table, int table_dtype,
                 void* stream) {
  NIC_ENTER(h);
  if (!dense || !table) return fail(h, NIC_ERR_ARG, "nic_lut_pack: NULL pointer");
  if (cout < 1 || cout > 4) return fail(h, NIC_ERR_ARG, "nic_lut_pack: cout %d (1..4)", cout);
  if (table_dtype != NIC_DT_F32 && table_dtype != NIC_DT_F16) return fail(h, NIC_ERR_ARG, "nic_lut_pack: table_dtype %d", table_dtype);
  long long texels = 0;
  int rc = lut_texels(h, extent, &texels, "nic_lut_pack");
  if (rc) return rc;
  return cuda_fail(h, launch_lut_pack(h, dense, texels, cout, table, table_dtype, st), "nic_lut_pack");
}

int nic_lut_apply(NicHandle* h, const NicLut* lut, const void* src, int src_dtype, int64_t pixels, void* dst,
                  int dst_dtype, int interp, void* stream) {
  NIC_ENTER(h);
  if (!lut) return fail(h, NIC_ERR_ARG, "nic_lut_apply: lut is NULL");
  if (pixels < 0) return fail(h, NIC_ERR_ARG, "nic_lut_apply: pixels %lld", (long long)pixels);
  if (pixels > 0 && (!lut->table || !src || !dst)) return fail(h, NIC_ERR_ARG, "nic_lut_apply: NULL pointer");
  if (lut->table_dtype != NIC_DT_F32 && lut->table_dtype != NIC_DT_F16)
    return fail(h, NIC_ERR_ARG, "nic_lut_apply: table_dtype %d", lut->table_dtype);
  if (lut->cout < 1 || lut->cout > 4) return fail(h, NIC_ERR_ARG, "nic_lut_apply: cout %d (1..4)", lut->cout);
  if (lut->reserved != 0) return fail(h, NIC_ERR_ARG, "nic_lut_apply: reserved is %d (must be 0)", lut->reserved);
  if (src_dtype != NIC_DT_U8 && src_dtype != NIC_DT_F32) return fail(h, NIC_ERR_ARG, "nic_lut_apply: src_dtype %d", src_dtype);
  if (dst_dtype != NIC_DT_U8 && dst_dtype != NIC_DT_F32) return fail(h, NIC_ERR_ARG, "nic_lut_apply: dst_dtype %d", dst_dtype);
  if (interp != NIC_INTERP_TRILINEAR && interp != NIC_INTERP_TETRAHEDRAL) return fail(h, NIC_ERR_ARG, "nic_lut_apply: interp %d", interp);
  long long texels = 0;
  int rc = lut_texels(h, lut->extent, &texels, "nic_lut_apply");
  if (rc) return rc;
  if (pixels == 0) return NIC_OK;
  const uintptr_t s0 = (uintptr_t)src, s1 = s0 + (uintptr_t)pixels * 3 * (src_dtype == NIC_DT_U8 ? 1 : 4);
  const uintptr_t d0 = (uintptr_t)dst, d1 = d0 + (uintptr_t)pixels * lut->cout * (dst_dtype == NIC_DT_U8 ? 1 : 4);
  if (s0 < d1 && d0 < s1) return fail(h, NIC_ERR_ARG, "nic_lut_apply: src and dst overlap (no in-place apply)");
  return cuda_fail(h, launch_lut_apply(h, *lut, src, src_dtype, pixels, dst, dst_dtype, interp, st), "nic_lut_apply");
}

int nic_train_step(NicHandle* h, const NicGeom* g, const float* g0, const float* g1, const int64_t* origins,
                   const NicMlp* m, const float* targets, const float* noise, int noise_bits, uint64_t seed,
                   uint64_t step, int64_t global_n, const NicMlpGrad* gm, float* dg0, float* dg1, float* loss_sum,
                   float* out, int precision, void* stream) {
  NIC_ENTER(h);
  DevGeom d;
  int rc = flatten_geom(h, g, origins != nullptr, &d);
  if (rc) return rc;
  MlpDev md;
  rc = flatten_mlp(h, m, &md, d.cin);
  if (rc) return rc;
  if (!g0 || !g1 || !gm || !gm->w1 || !gm->b1 || !gm->w2 || !gm->b2 || !gm->w3 || !gm->b3 || (!targets && d.N > 0))
    return fail(h, NIC_ERR_ARG, "nic_train_step: NULL pointer");
  if ((dg0 == nullptr) != (dg1 == nullptr)) return fail(h, NIC_ERR_ARG, "nic_train_step: dg0 and dg1 must both be set or both NULL");
  if (noise_bits < 0 || noise_bits > 24) return fail(h, NIC_ERR_ARG, "nic_train_step: noise_bits %d", noise_bits);
  if (precision != NIC_PREC_F32 && precision != NIC_PREC_F16 && precision != NIC_PREC_BF16)
    return fail(h, NIC_ERR_ARG, "nic_train_step: precision %d", precision);
  d.metrics = h->step_metrics;
  long long denom = (global_n > 0 ? global_n : d.N) * (long long)md.cout;
  float grad_scale = denom > 0 ? (float)(1.0 / (double)denom) : 0.f;
  MlpGradDev gd = {gm->w1, gm->b1, gm->w2, gm->b2, gm->w3, gm->b3};
  if (precision != NIC_PREC_F32) {
    int trc = launch_train_tc(h, d, md, gd, g0, g1, (const long long*)origins, targets, noise, noise_bits, seed, step, grad_scale,
                              dg0, dg1, loss_sum, out, precision, st);
    if (trc == NIC_ERR_UNSUPPORTED)
      return fail(h, trc, "nic_train_step: the tensor-core step covers the 2-D method with C=12, PE=6, hidden 64 and crop origins; "
                          "use NIC_PREC_F32 for this configuration");
    return cuda_fail(h, trc, "nic_train_step(tensor core)");
  }
  return cuda_fail(h, launch_train_f32(h, d, md, gd, g0, g1, (const long long*)origins, targets, noise, noise_bits, seed, step,
                                       grad_scale, dg0, dg1, loss_sum, out, st), "nic_train_step");
}

static int adam_common(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                       float grad_scale, int zero_grad, float* loss_sum, float* loss_out, float loss_scale, cudaStream_t st) {
  if (count < 0 || (count > 0 && !tensors)) return fail(h, NIC_ERR_ARG, "nic_adam_step: count %d", count);
  for (int i = 0; i < count; ++i) {
    const NicAdamTensor& t = tensors[i];
    if (t.numel < 0 || t.t < 1 || (t.numel > 0 && (!t.p || !t.g || !t.m || !t.v)))
      return fail(h, NIC_ERR_ARG, "nic_adam_step: tensor %d invalid (numel %lld, t %d)", i, (long long)t.numel, t.t);
  }
  return cuda_fail(h, launch_adam(h, tensors, count, beta1, beta2, eps, grad_scale, zero_grad, loss_sum, loss_out, loss_scale, st),
                   "nic_adam_step");
}

int nic_adam_step(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                  float grad_scale, int zero_grad, void* stream) {
  NIC_ENTER(h);
  return adam_common(h, tensors, count, beta1, beta2, eps, grad_scale, zero_grad, nullptr, nullptr, 0.f, st);
}

int nic_adam_step_loss(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                       float grad_scale, int zero_grad, float* loss_sum, float* loss_out, float loss_scale, void* stream) {
  NIC_ENTER(h);
  if (count < 1 || !loss_sum || !loss_out) return fail(h, NIC_ERR_ARG, "nic_adam_step_loss: needs tensors and loss buffers");
  return adam_common(h, tensors, count, beta1, beta2, eps, grad_scale, zero_grad, loss_sum, loss_out, loss_scale, st);
}

int nic_sym_alloc(NicHandle* h, int64_t bytes, void** ptr, uint8_t ipc_handle[64]) {
  if (!h || !ptr || !ipc_handle || bytes <= 0) return fail(h, NIC_ERR_ARG, "nic_sym_alloc: bad argument");
  DeviceGuard guard_(h->device);
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);
  if (e == cudaSuccess) e = cudaMemset(p, 0, (size_t)bytes);
  cudaIpcMemHandle_t hd;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&hd, p);
  if (e != cudaSuccess) {
    if (p) cudaFree(p);
    return fail(h, (int)e, "nic_sym_alloc: %s", cudaGetErrorString(e));
  }
  memcpy(ipc_handle, &hd, 64);
  *ptr = p;
  return NIC_OK;
}

int nic_sym_open(NicHandle* h, const uint8_t ipc_handle[64], void** ptr) {
  if (!h || !ptr || !ipc_handle) return fail(h, NIC_ERR_ARG, "nic_sym_open: bad argument");
  DeviceGuard guard_(h->device);
  cudaIpcMemHandle_t hd;
  memcpy(&hd, ipc_handle, 64);
  cudaError_t e = cudaIpcOpenMemHandle(ptr, hd, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return fail(h, (int)e, "nic_sym_open: %s", cudaGetErrorString(e));
  return NIC_OK;
}

int nic_sym_close(NicHandle* h, void* ptr) {
  if (!h) return fail(nullptr, NIC_ERR_ARG, "handle is NULL");
  DeviceGuard guard_(h->device);
  cudaError_t e = ptr ? cudaIpcCloseMemHandle(ptr) : cudaSuccess;
  if (e != cudaSuccess) return fail(h, (int)e, "nic_sym_close: %s", cudaGetErrorString(e));
  return NIC_OK;
}

int nic_sym_free(NicHandle* h, void* ptr) {
  if (!h) return fail(nullptr, NIC_ERR_ARG, "handle is NULL");
  DeviceGuard guard_(h->device);
  cudaError_t e = ptr ? cudaFree(ptr) : cudaSuccess;
  if (e != cudaSuccess) return fail(h, (int)e, "nic_sym_free: %s", cudaGetErrorString(e));
  return NIC_OK;
}

int nic_adam_step_exchange(NicHandle* h, const NicAdamTensor* tensors, int count, float beta1, float beta2, float eps,
                           float grad_scale, const NicExchange* x, const float* loss_sum, float* loss_out, float loss_scale,
                           void* stream) {
  NIC_ENTER(h);
  if (!x || count < 1 || !tensors) return fail(h, NIC_ERR_ARG, "nic_adam_step_exchange: NULL argument");
  if (x->world < 1 || x->world > NIC_MAX_PEERS || x->rank < 0 || x->rank >= x->world)
    return fail(h, NIC_ERR_ARG, "nic_adam_step_exchange: rank %d of world %d (max %d)", x->rank, x->world, NIC_MAX_PEERS);
  for (int r = 0; r < x->world; ++r)
    if (!x->peer_flat[r] || !x->peer_flag[r]) return fail(h, NIC_ERR_ARG, "nic_adam_step_exchange: peer %d not mapped", r);
  if ((loss_out != nullptr) != (loss_sum != nullptr)) return fail(h, NIC_ERR_ARG, "nic_adam_step_exchange: loss buffers");
  if (x->zero_buf && ((((uintptr_t)x->zero_buf) & 15) || (x->zero_numel & 3) || x->zero_numel < 0))
    return fail(h, NIC_ERR_ARG, "nic_adam_step_exchange: zero_buf must be 16-byte aligned, a multiple of 4 floats");
  for (int i = 0; i < count; ++i) {
    const NicAdamTensor& t = tensors[i];
    if (t.numel < 0 || t.t < 1 || (t.numel > 0 && (!t.p || !t.g || !t.m || !t.v)))
      return fail(h, NIC_ERR_ARG, "nic_adam_step_exchange: tensor %d invalid", i);
  }
  int rc = launch_adam_exchange(h, tensors, count, beta1, beta2, eps, grad_scale, *x, loss_sum, loss_out, loss_scale, st);
  if (rc == NIC_ERR_EXCHANGE)
    return fail(h, rc, "nic_adam_step_exchange: an earlier exchange timed out waiting for a peer; no update has been applied "
                       "since.  Re-synchronise the replicas and clear the flag with nic_exchange_status");
  return cuda_fail(h, rc, "nic_adam_step_exchange");
}

int nic_exchange_status(NicHandle* h, int* timed_out) {
  if (!h || !timed_out) return fail(h, NIC_ERR_ARG, "nic_exchange_status: NULL argument");
  *timed_out = 0;
  if (!h->xch_err) return NIC_OK;
  DeviceGuard guard_(h->device);
  unsigned v = 0;
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(&v, h->xch_err, sizeof(v), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemset(h->xch_err, 0, sizeof(v));
  if (h->xch_host_err) {
    if (*reinterpret_cast<volatile unsigned*>(h->xch_host_err)) v = 1u;
    *h->xch_host_err = 0u;
  }
  if (e != cudaSuccess) return fail(h, (int)e, "nic_exchange_status: %s", cudaGetErrorString(e));
  *timed_out = (int)v;
  return NIC_OK;
}

static int check_bits(NicHandle* h, int bits, const char* who) {
  if (bits < 1 || bits > 8) return fail(h, NIC_ERR_ARG, "%s: bits %d (1..8)", who, bits);
  return NIC_OK;
}

int nic_quantize4fp(NicHandle* h, const float* src, float* dst, int64_t n, int bits, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_bits(h, bits, "nic_quantize4fp")) return rc;
  if (n < 0 || (n > 0 && (!src || !dst))) return fail(h, NIC_ERR_ARG, "nic_quantize4fp: bad buffer");
  return cuda_fail(h, launch_quantize4fp(h, src, dst, n, bits, st), "nic_quantize4fp");
}

int nic_quantize_pack(NicHandle* h, const float* src, uint8_t* codes, int64_t n, int bits, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_bits(h, bits, "nic_quantize_pack")) return rc;
  if (n < 0 || (n > 0 && (!src || !codes))) return fail(h, NIC_ERR_ARG, "nic_quantize_pack: bad buffer");
  return cuda_fail(h, launch_quantize_pack(h, src, codes, n, bits, st), "nic_quantize_pack");
}

int nic_unpack(NicHandle* h, const uint8_t* codes, float* dst, int64_t n, int bits, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_bits(h, bits, "nic_unpack")) return rc;
  if (n < 0 || (n > 0 && (!codes || !dst))) return fail(h, NIC_ERR_ARG, "nic_unpack: bad buffer");
  return cuda_fail(h, launch_unpack(h, codes, dst, n, bits, st), "nic_unpack");
}

static int check_pack_bits(NicHandle* h, int bits, const char* who) {
  if (bits != 1 && bits != 2 && bits != 4 && bits != 8) return fail(h, NIC_ERR_ARG, "%s: bits %d (1, 2, 4 or 8)", who, bits);
  return NIC_OK;
}

int nic_pack_codes(NicHandle* h, const uint8_t* codes, uint8_t* packed, int64_t n, int bits, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_pack_bits(h, bits, "nic_pack_codes")) return rc;
  if (n < 0 || (n > 0 && (!codes || !packed))) return fail(h, NIC_ERR_ARG, "nic_pack_codes: bad buffer");
  return cuda_fail(h, launch_pack_bits(h, codes, packed, n, bits, 0, st), "nic_pack_codes");
}

int nic_unpack_codes(NicHandle* h, const uint8_t* packed, uint8_t* codes, int64_t n, int bits, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_pack_bits(h, bits, "nic_unpack_codes")) return rc;
  if (n < 0 || (n > 0 && (!codes || !packed))) return fail(h, NIC_ERR_ARG, "nic_unpack_codes: bad buffer");
  return cuda_fail(h, launch_pack_bits(h, packed, codes, n, bits, 1, st), "nic_unpack_codes");
}

int nic_clamp(NicHandle* h, float* p, int64_t n, float lo, float hi, void* stream) {
  NIC_ENTER(h);
  if (n < 0 || (n > 0 && !p) || !(lo <= hi)) return fail(h, NIC_ERR_ARG, "nic_clamp: bad arguments");
  return cuda_fail(h, launch_clamp(h, p, n, lo, hi, st), "nic_clamp");
}

int nic_output_to_u8(NicHandle* h, const float* src, uint8_t* dst, int64_t n, int bits, void* stream) {
  NIC_ENTER(h);
  if (int rc = check_bits(h, bits, "nic_output_to_u8")) return rc;
  if (n < 0 || (n > 0 && (!src || !dst))) return fail(h, NIC_ERR_ARG, "nic_output_to_u8: bad buffer");
  return cuda_fail(h, launch_output_to_u8(h, src, dst, n, bits, st), "nic_output_to_u8");
}

int nic_sse_u8(NicHandle* h, const uint8_t* a, const uint8_t* b, int64_t n, double* sse, void* stream) {
  NIC_ENTER(h);
  if (n < 0 || !sse || (n > 0 && (!a || !b))) return fail(h, NIC_ERR_ARG, "nic_sse_u8: bad buffer");
  return cuda_fail(h, launch_sse_u8(h, a, b, n, sse, st), "nic_sse_u8");
}

}  // extern "C"
