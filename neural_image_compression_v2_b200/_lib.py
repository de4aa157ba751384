"""ctypes binding of libnic.so (include/nic.h).  Plumbing only: device memory and streams come from torch,
every computation happens in the CUDA library.  There is no CPU fallback — a missing library or a
non-sm_100 device raises."""
import ctypes as C
import math
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NIC_LIB_PATH") or os.path.join(_HERE, "libnic.so")     # override: A/B runs of kernel builds

METHOD_2D, METHOD_3D, METHOD_3D_V2 = 1, 3, 4
PE_TRIANGULAR, PE_SINUSOIDAL = 0, 1
PREC_F32, PREC_F16, PREC_BF16 = 0, 1, 2
DT_F32, DT_F16, DT_BF16, DT_U8 = 0, 1, 2, 3
PRECISIONS = {"f32": PREC_F32, "fp32": PREC_F32, "f16": PREC_F16, "fp16": PREC_F16, "bf16": PREC_BF16}


class NicError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"libnic status {status}: {message}")
        self.status = status


class NicGeom(C.Structure):
    _fields_ = [("method", C.c_int32), ("channels", C.c_int32), ("pe_channels", C.c_int32), ("pe_kind", C.c_int32),
                ("step_log2", C.c_int32), ("mip_level", C.c_int32), ("g0_nodes", C.c_int32 * 3),
                ("g1_nodes", C.c_int32 * 3), ("block", C.c_int32 * 3), ("num_blocks", C.c_int32),
                ("origin0", C.c_int32 * 3), ("reserved", C.c_int32), ("pe_div", C.c_float * 8)]


class NicMlp(C.Structure):
    _fields_ = [("cin", C.c_int32), ("hidden", C.c_int32), ("cout", C.c_int32), ("reserved", C.c_int32),
                ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w3", C.c_void_p), ("b3", C.c_void_p)]


ADDRESS_CLAMP, ADDRESS_WRAP = 0, 1


class NicSampler(C.Structure):
    _fields_ = [("address", C.c_int32), ("align_corners", C.c_int32), ("extent", C.c_int32 * 3),
                ("blend_weight", C.c_float), ("blend_prev", C.c_void_p)]


MAX_MIPS = 16


class NicMipChain(C.Structure):
    _fields_ = [("num_mips", C.c_int32), ("address", C.c_int32), ("align_corners", C.c_int32), ("reserved", C.c_int32),
                ("geom", NicGeom * MAX_MIPS), ("g0", C.c_void_p * MAX_MIPS), ("g1", C.c_void_p * MAX_MIPS),
                ("extent", (C.c_int32 * 3) * MAX_MIPS)]


INTERP_TRILINEAR, INTERP_TETRAHEDRAL = 0, 1


class NicLut(C.Structure):
    _fields_ = [("table", C.c_void_p), ("table_dtype", C.c_int32), ("cout", C.c_int32), ("extent", C.c_int32 * 3),
                ("reserved", C.c_int32)]


class NicMlpGrad(C.Structure):
    _fields_ = [("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w3", C.c_void_p), ("b3", C.c_void_p)]


class NicAdamTensor(C.Structure):
    _fields_ = [("p", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("numel", C.c_int64),
                ("lr", C.c_float), ("t", C.c_int32), ("clamp", C.c_int32), ("clamp_lo", C.c_float),
                ("clamp_hi", C.c_float)]


MAX_PEERS = 16


EXCHANGE_ONE_SHOT, EXCHANGE_SLICED = 0, 1      # NicExchange.reserved (nic.h: NIC_EXCHANGE_*)


class NicExchange(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("token", C.c_uint32), ("reserved", C.c_int32),
                ("peer_flat", C.c_void_p * MAX_PEERS), ("peer_flag", C.c_void_p * MAX_PEERS),
                ("zero_buf", C.c_void_p), ("zero_numel", C.c_int64)]


# every symbol include/nic.h declares: name -> (restype, argtypes)
_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float
SYMBOLS = {
    "nic_abi_version": (_I, []),
    "nic_create": (_I, [_I, C.POINTER(_P)]),
    "nic_destroy": (_I, [_P]),
    "nic_last_error_string": (C.c_char_p, [_P]),
    "nic_status_string": (C.c_char_p, [_I]),
    "nic_launch_count": (_L, [_P]),
    "nic_set_option": (_I, [_P, _I, _I]),
    "nic_kernel_time_ms": (_I, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "nic_debug_counters": (_I, [_P, C.POINTER(C.c_int64), _I]),
    "nic_cin": (_I, [C.POINTER(NicGeom)]),
    "nic_gather": (_I, [_P, C.POINTER(NicGeom), _P, _P, _P, _P, _I, _P]),
    "nic_scatter": (_I, [_P, C.POINTER(NicGeom), _P, _P, _P, _P, _P]),
    "nic_mlp_forward": (_I, [_P, C.POINTER(NicMlp), _P, _L, _L, _P, _P, _P, _P]),
    "nic_mlp_backward": (_I, [_P, C.POINTER(NicMlp), _P, _L, _L, _P, _P, _P, _P, C.POINTER(NicMlpGrad), _P, _P]),
    "nic_decode": (_I, [_P, C.POINTER(NicGeom), _P, _P, _P, C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_decode_codes": (_I, [_P, C.POINTER(NicGeom), _P, _P, _I, _P, C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_sample": (_I, [_P, C.POINTER(NicGeom), _P, _P, _P, C.POINTER(NicSampler), C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_sample_codes": (_I, [_P, C.POINTER(NicGeom), _P, _P, _I, _P, C.POINTER(NicSampler), C.POINTER(NicMlp), _P, _I,
                              _I, _P]),
    "nic_sample_lod": (_I, [_P, C.POINTER(NicMipChain), _P, _P, _P, _P, C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_sample_lod_codes": (_I, [_P, C.POINTER(NicMipChain), _I, _P, _P, _P, _P, C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_decode_mips": (_I, [_P, C.POINTER(NicMipChain), C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_decode_mips_codes": (_I, [_P, C.POINTER(NicMipChain), _I, C.POINTER(NicMlp), _P, _I, _I, _P]),
    "nic_lut_pack": (_I, [_P, _P, C.POINTER(C.c_int32), _I, _P, _I, _P]),
    "nic_lut_apply": (_I, [_P, C.POINTER(NicLut), _P, _I, _L, _P, _I, _I, _P]),
    "nic_train_step": (_I, [_P, C.POINTER(NicGeom), _P, _P, _P, C.POINTER(NicMlp), _P, _P, _I, C.c_uint64, C.c_uint64,
                            _L, C.POINTER(NicMlpGrad), _P, _P, _P, _P, _I, _P]),
    "nic_adam_step": (_I, [_P, C.POINTER(NicAdamTensor), _I, _F, _F, _F, _F, _I, _P]),
    "nic_adam_step_loss": (_I, [_P, C.POINTER(NicAdamTensor), _I, _F, _F, _F, _F, _I, _P, _P, _F, _P]),
    "nic_sym_alloc": (_I, [_P, _L, C.POINTER(_P), C.c_char_p]),
    "nic_sym_open": (_I, [_P, C.c_char_p, C.POINTER(_P)]),
    "nic_sym_close": (_I, [_P, _P]),
    "nic_sym_free": (_I, [_P, _P]),
    "nic_adam_step_exchange": (_I, [_P, C.POINTER(NicAdamTensor), _I, _F, _F, _F, _F, C.POINTER(NicExchange), _P, _P, _F, _P]),
    "nic_exchange_status": (_I, [_P, C.POINTER(_I)]),
    "nic_quantize4fp": (_I, [_P, _P, _P, _L, _I, _P]),
    "nic_quantize_pack": (_I, [_P, _P, _P, _L, _I, _P]),
    "nic_unpack": (_I, [_P, _P, _P, _L, _I, _P]),
    "nic_pack_codes": (_I, [_P, _P, _P, _L, _I, _P]),
    "nic_unpack_codes": (_I, [_P, _P, _P, _L, _I, _P]),
    "nic_clamp": (_I, [_P, _P, _L, _F, _F, _P]),
    "nic_output_to_u8": (_I, [_P, _P, _P, _L, _I, _P]),
    "nic_sse_u8": (_I, [_P, _P, _P, _L, _P, _P]),
    "nic_sample_crops": (_I, [_P, _P, _I, _I, _P, _P, _I, _P, _P, _P]),
    "nic_sample_crops_random": (_I, [_P, _P, _I, _I, _P, _I, _P, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "nic_resize_bilinear_u8": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "nic_atlas_pack": (_I, [_P, _P, _I, _I, _I, _I, _P, _P]),
    "nic_atlas_unpack": (_I, [_P, _P, _I, _I, _I, _I, _P, _P]),
    "nic_positional_encoding": (_I, [_P, _P, _I, _L, _I, _I, _P, _P, _P]),
}

_lib = None


def load_library():
    """Loads libnic.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -m neural_image_compression_v2_b200.build` "
                          "(there is no CPU or PyTorch fallback for this path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype, fn.argtypes = res, args
    if lib.nic_abi_version() != 1:
        raise ImportError("libnic.so ABI version mismatch")
    _lib = lib
    return lib


_handles = {}


def handle(device):
    """One NicHandle per CUDA device (created lazily)."""
    device = torch.device(device)
    if device.type != "cuda":
        raise NicError(-3, f"tensor on {device}: this path only runs on a CUDA sm_100 device (no CPU fallback)")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _handles:
        lib = load_library()
        h = _P()
        rc = lib.nic_create(idx, C.byref(h))
        if rc != 0:
            raise NicError(rc, lib.nic_last_error_string(None).decode())
        _handles[idx] = h
    return _handles[idx]


OPT_DISABLE_FAST2D = 1
OPT_TIME_KERNELS = 2
OPT_REUSE_PREPARED = 3
OPT_GELU_POLY = 5            # share (of 8) of hidden activations on the polynomial GELU; -1 = tuned default
OPT_EXCHANGE_TIMEOUT_MS = 6  # device-side wait for a peer in nic_adam_step_exchange (default 10 s)
OPT_STEP_METRICS = 7         # loss_sum / loss_out carry [squared error, squared error of the 8-bit outputs]
ERR_EXCHANGE = -7
ERR_UNSUPPORTED = -2
OPT_STATIC_TILES = 8         # static tile order in the tensor-core training kernel (A/B timing of the dynamic scheduler)
OPT_DEBUG_KNOCKOUT = 100     # profiling only (nic.h); bit 3 = training phase counters


def kernel_time_ms(device):
    """(sum of the dominant kernels' durations in ms, launches bracketed) since the last call; see nic.h."""
    h = handle(device)
    ms, n = C.c_double(0.0), C.c_int64(0)
    check(h, load_library().nic_kernel_time_ms(h, C.byref(ms), C.byref(n)))
    return float(ms.value), int(n.value)


def debug_counters(device, n=16):
    """The 16 device debug counters (nic_debug_counters): read and cleared; see nic.h."""
    h = handle(device)
    out = (C.c_int64 * 16)()
    check(h, load_library().nic_debug_counters(h, out, int(n)))
    return [int(v) for v in out[:n]]


class SymmetricBuffer:
    """A float32 device buffer in IPC-shared memory (nic_sym_alloc) that the other ranks of a process group can map.
    `tensor` aliases the memory (CUDA array interface); `handle` is the 64-byte IPC handle to send to the peers."""

    def __init__(self, device, numel):
        self.device = torch.device(device)
        self.numel = int(numel)
        h = handle(self.device)
        p = _P()
        buf = C.create_string_buffer(64)
        check(h, load_library().nic_sym_alloc(h, self.numel * 4, C.byref(p), buf))
        self.ptr = int(p.value)
        self.handle = bytes(buf.raw)
        self.__cuda_array_interface__ = {"shape": (self.numel,), "typestr": "<f4", "data": (self.ptr, False), "version": 3,
                                         "strides": None}
        self.tensor = torch.as_tensor(self, device=self.device)
        self._peers = []

    def open_peer(self, ipc_handle):
        """Maps another rank's buffer; returns its device pointer in THIS process."""
        h = handle(self.device)
        p = _P()
        check(h, load_library().nic_sym_open(h, C.c_char_p(ipc_handle), C.byref(p)))
        self._peers.append(int(p.value))
        return int(p.value)

    def close(self):
        h = handle(self.device)
        lib = load_library()
        for p in self._peers:
            lib.nic_sym_close(h, _P(p))
        self._peers = []
        if self.ptr:
            self.tensor = None
            lib.nic_sym_free(h, _P(self.ptr))
            self.ptr = 0


def exchange_status(device):
    """True if an exchange kernel on this device timed out waiting for a peer since the last call (synchronises)."""
    h = handle(device)
    v = C.c_int(0)
    check(h, load_library().nic_exchange_status(h, C.byref(v)))
    return bool(v.value)


def set_option(device, option, value):
    h = handle(device)
    check(h, load_library().nic_set_option(h, option, int(value)))


def check(h, rc):
    if rc != 0:
        raise NicError(rc, load_library().nic_last_error_string(h).decode())


def stream_ptr(device):
    return _P(torch.cuda.current_stream(device).cuda_stream)


def launch_count(device):
    return int(load_library().nic_launch_count(handle(device)))


def ptr(t):
    return _P(t.data_ptr()) if t is not None else _P(None)


def _f32c(t, name):
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise TypeError(f"{name} must be a contiguous float32 tensor (got {t.dtype}, contiguous={t.is_contiguous()})")
    return t


def sin_div_term(pe_channels):
    """utils.py:202 as torch evaluates it in float32."""
    return np.exp(np.arange(0, pe_channels, 2, dtype=np.float32) * np.float32(-(math.log(10000.0) / pe_channels)))


def make_geom(method, g0, g1, block, num_blocks, step_log2, mip_level, pe_channels, pe_kind, origin0=None):
    """NicGeom for grids g0/g1 (`[C, (z,) y, x]`) and blocks of `block` texels along image axes x,y(,z)."""
    dim = 2 if method == METHOD_2D else 3
    if g0.dim() != dim + 1 or g1.dim() != dim + 1 or g0.shape[0] != g1.shape[0]:
        raise ValueError(f"grids must be [C, {'z, ' if dim == 3 else ''}y, x]; got {tuple(g0.shape)} and {tuple(g1.shape)}")
    if pe_channels > 8:
        raise ValueError("PE_CHANNELS > 8 is not supported")
    g = NicGeom()
    g.method, g.channels, g.pe_channels, g.pe_kind = method, g0.shape[0], pe_channels, pe_kind
    g.step_log2, g.mip_level, g.num_blocks = step_log2, mip_level, num_blocks
    if isinstance(block, int):
        block = (block,) * dim
    for a in range(3):
        # grid tensors are indexed [c, (z,) y, x]: image axis a (x=0, y=1, z=2) is tensor dim (dim - a)
        g.g0_nodes[a] = g0.shape[dim - a] if a < dim else 1
        g.g1_nodes[a] = g1.shape[dim - a] if a < dim else 1
        g.block[a] = block[a] if a < dim else 1
        g.origin0[a] = int(origin0[a]) if (origin0 is not None and a < dim) else 0
    if pe_kind == PE_SINUSOIDAL:
        for i, v in enumerate(sin_div_term(pe_channels)):
            g.pe_div[i] = float(v)
    return g


def cin_of(geom):
    return int(load_library().nic_cin(C.byref(geom)))


def make_mlp(params):
    """NicMlp from (W1, b1, W2, b2, W3, b3) float32 CUDA tensors in nn.Linear layout."""
    w1, b1, w2, b2, w3, b3 = [_f32c(p, "decoder parameter") for p in params]
    m = NicMlp()
    m.cin, m.hidden, m.cout = w1.shape[1], w1.shape[0], w3.shape[0]
    if tuple(w2.shape) != (m.hidden, m.hidden) or w3.shape[1] != m.hidden:
        raise ValueError("decoder must be Linear(cin,H) / Linear(H,H) / Linear(H,cout)")
    m.w1, m.b1, m.w2, m.b2, m.w3, m.b3 = [t.data_ptr() for t in (w1, b1, w2, b2, w3, b3)]
    return m


def make_mlp_grad(grads):
    g = NicMlpGrad()
    g.w1, g.b1, g.w2, g.b2, g.w3, g.b3 = [_f32c(t, "decoder gradient").data_ptr() for t in grads]
    return g


def origins_tensor(coord, device, dim):
    """The reference's `coord` ([num_crops, D] int64 on DEVICE) as a contiguous device tensor."""
    if not torch.is_tensor(coord):
        coord = torch.as_tensor(np.asarray(coord), dtype=torch.int64)
    coord = coord.to(device=device, dtype=torch.int64).contiguous()
    if coord.dim() != 2 or coord.shape[1] != dim:
        raise ValueError(f"coord must be [num_crops, {dim}], got {tuple(coord.shape)}")
    return coord
