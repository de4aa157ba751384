"""Host-side mirror of the hot-path functions of the reference's `Projects/image_compression.py`.

Same function names, argument order, return shapes and `state_dict` keys as the reference, so a maintainer
can swap the imports (INTEGRATION.md).  Each function cites the reference lines it replaces.  All arithmetic
runs in libnic.so on a B200; tensors must live on a CUDA device (there is no CPU fallback).

Two ways to drive the path:
  * the reference's own two-call sequence — `create_decoder_input_*` / `finally_decode_input_*` followed by
    `decoder(x)`, `loss.backward()` and a torch optimiser — works unchanged through autograd Functions;
  * the fused entry points `decode(...)` and `FusedTrainer.step(...)`, which never materialise X.
"""
import ctypes as C
import math
import random

import torch
import torch.nn as nn

from . import _lib as L
from . import var2
from .fp_def import create_pyramid_mip_levels, fp_all_quantize, fp_freeze, fp_quantize_clamp
from .models import quantize4fp


# ------------------------------------------------------------------------------------------------ helpers
def _method():
    return {1: L.METHOD_2D, 2: L.METHOD_2D, 3: L.METHOD_3D, 4: L.METHOD_3D_V2}[var2.COMPRESSION_METHOD]


def _pe_kind(method):
    """2-D: TF_USE_TRI_PE chooses (fp_def.py:132-135); method 3 always triangular (:169); method 4 always
    sinusoidal (:208)."""
    if method == L.METHOD_2D:
        return L.PE_TRIANGULAR if var2.TF_USE_TRI_PE else L.PE_SINUSOIDAL
    return L.PE_TRIANGULAR if method == L.METHOD_3D else L.PE_SINUSOIDAL


def feature_pyramid_mip_levels():
    """The reference's global `feature_pyramid_mip_levels_dict` (image_compression.py:360)."""
    return create_pyramid_mip_levels(var2.IMAGE_SIZE, var2.FEATURE_PYRAMID_SIZE)


def _step_log2(mip_level, fl):
    """image_compression.py:79 — step_number = 2^(mip - 2(fl+1))."""
    return mip_level - (fl + 1) * 2


def _check_grid(g):
    if not g.is_cuda:
        raise L.NicError(-3, "grids must be CUDA tensors (no CPU fallback)")
    if g.dtype != torch.float32 or not g.is_contiguous():
        raise TypeError("grids must be contiguous float32")
    return g


class _GatherFn(torch.autograd.Function):
    """X = gather(G0, G1): fp_def.create_g0_g1* + the torch.cat of image_compression.py:90-100.  Backward is the
    scatter-add the reference gets from autograd's index_put(accumulate) (image_compression.py:265)."""

    @staticmethod
    def forward(ctx, g0, g1, coord, geom):
        g0d, g1d = _check_grid(g0.detach()), _check_grid(g1.detach())
        n = geom.num_blocks * geom.block[0] * geom.block[1] * geom.block[2]
        x = torch.empty((n, L.cin_of(geom)), dtype=torch.float32, device=g0.device)
        h = L.handle(g0.device)
        L.check(h, L.load_library().nic_gather(h, C.byref(geom), L.ptr(g0d), L.ptr(g1d), L.ptr(coord), L.ptr(x),
                                               L.DT_F32, L.stream_ptr(g0.device)))
        ctx.geom, ctx.coord, ctx.shapes = geom, coord, (g0.shape, g1.shape)
        return x

    @staticmethod
    def backward(ctx, dx):
        dx = dx.contiguous()
        dg0 = torch.zeros(ctx.shapes[0], dtype=torch.float32, device=dx.device)
        dg1 = torch.zeros(ctx.shapes[1], dtype=torch.float32, device=dx.device)
        h = L.handle(dx.device)
        L.check(h, L.load_library().nic_scatter(h, C.byref(ctx.geom), L.ptr(dx), L.ptr(ctx.coord), L.ptr(dg0),
                                                L.ptr(dg1), L.stream_ptr(dx.device)))
        return dg0, dg1, None, None


class _MlpFn(torch.autograd.Function):
    """ColorDecoder.forward on a materialised input (image_compression.py:57-68), exact-erf GELU in fp32."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, w3, b3):
        if not x.is_cuda:
            raise L.NicError(-3, "decoder input must be a CUDA tensor (no CPU fallback)")
        params = [p.detach().contiguous() for p in (w1, b1, w2, b2, w3, b3)]
        xd = x.detach()
        if xd.dtype != torch.float32:
            raise TypeError("decoder input must be float32")
        if xd.dim() != 2:
            raise ValueError("decoder input must be [N, Cin]")
        if xd.stride(1) != 1:
            xd = xd.contiguous()
        m = L.make_mlp(params)
        if xd.shape[1] != m.cin:
            raise ValueError(f"decoder input has {xd.shape[1]} columns, decoder expects {m.cin}")
        n = xd.shape[0]
        need_grad = any(ctx.needs_input_grad)
        out = torch.empty((n, m.cout), dtype=torch.float32, device=x.device)
        z1 = torch.empty((n, m.hidden), dtype=torch.float32, device=x.device) if need_grad else None
        z2 = torch.empty((n, m.hidden), dtype=torch.float32, device=x.device) if need_grad else None
        h = L.handle(x.device)
        L.check(h, L.load_library().nic_mlp_forward(h, C.byref(m), L.ptr(xd), xd.stride(0), n, L.ptr(out), L.ptr(z1),
                                                    L.ptr(z2), L.stream_ptr(x.device)))
        if need_grad:
            ctx.save_for_backward(xd, z1, z2, out, *params)
        return out

    @staticmethod
    def backward(ctx, dout):
        xd, z1, z2, out, *params = ctx.saved_tensors
        m = L.make_mlp(params)
        grads = [torch.zeros_like(p) for p in params]
        gm = L.make_mlp_grad(grads)
        dx = torch.empty((xd.shape[0], m.cin), dtype=torch.float32, device=xd.device) if ctx.needs_input_grad[0] else None
        h = L.handle(xd.device)
        L.check(h, L.load_library().nic_mlp_backward(h, C.byref(m), L.ptr(xd), xd.stride(0), xd.shape[0], L.ptr(z1),
                                                     L.ptr(z2), L.ptr(out), L.ptr(dout.contiguous()), C.byref(gm),
                                                     L.ptr(dx), L.stream_ptr(xd.device)))
        return (dx, *grads)


# ------------------------------------------------------------------------------------------------ decoder
class _FusedSequential(nn.Sequential):
    """nn.Sequential(Linear, GELU, Linear, GELU, Linear, Sigmoid) whose forward is one fused CUDA kernel."""

    def forward(self, x):
        lin = [self[0], self[2], self[4]]
        return _MlpFn.apply(x, lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias, lin[2].weight, lin[2].bias)


class ColorDecoder(nn.Module):
    """image_compression.py:54-68 — same construction and `state_dict` keys (`decoder.{0,2,4}.{weight,bias}`)."""

    def __init__(self, in_channels=None, hidden=None, out_channels=None):
        super().__init__()
        cin = var2.DECODER_INPUT_CHANNELS if in_channels is None else in_channels
        hid = var2.HIDDEN_LAYER_CHANNELS if hidden is None else hidden
        cout = var2.OUTPUT_CHANNELS if out_channels is None else out_channels
        self.decoder = _FusedSequential(nn.Linear(cin, hid), nn.GELU(), nn.Linear(hid, hid), nn.GELU(),
                                        nn.Linear(hid, cout), nn.Sigmoid())

    def forward(self, x):
        return self.decoder(x)

    def parameters_list(self):
        d = self.decoder
        return [d[0].weight, d[0].bias, d[2].weight, d[2].bias, d[4].weight, d[4].bias]


# ------------------------------------------------------------------------------------------------ decoder inputs
def _create_decoder_input(fp, coord, num_crops, fl, mip_level, method):
    g0, g1 = fp[fl * 2], fp[fl * 2 + 1]
    dim = 2 if method == L.METHOD_2D else 3
    # image_compression.py:78 hard-codes 8 in 2-D; :110/:144 use CROP_MIP_LEVEL in 3-D
    sample_number = pow(2, max(0, (8 if dim == 2 else var2.CROP_MIP_LEVEL) - mip_level))
    coord = L.origins_tensor(coord, g0.device, dim)[:num_crops].contiguous()
    geom = L.make_geom(method, g0, g1, sample_number, num_crops, _step_log2(mip_level, fl), mip_level,
                       var2.PE_CHANNELS, _pe_kind(method))
    return _GatherFn.apply(g0, g1, coord, geom)


def create_decoder_input_2d(fp, coord, num_crops, fl, mip_level):
    """image_compression.py:71-100 -> X [num_crops * S^2, Cin]."""
    return _create_decoder_input(fp, coord, num_crops, fl, mip_level, L.METHOD_2D)


def create_decoder_input_3d(fp, coord, num_crops, fl, mip_level):
    """image_compression.py:103-134."""
    return _create_decoder_input(fp, coord, num_crops, fl, mip_level, L.METHOD_3D)


def create_decoder_input_3d_v2(fp, coord, num_crops, fl, mip_level):
    """image_compression.py:137-167."""
    return _create_decoder_input(fp, coord, num_crops, fl, mip_level, L.METHOD_3D_V2)


def _finally_decode_input(fp, image_size, mip_level, origin, method):
    fl = feature_pyramid_mip_levels()[mip_level]
    g0, g1 = fp[fl * 2], fp[fl * 2 + 1]
    geom = L.make_geom(method, g0, g1, image_size, 1, _step_log2(mip_level, fl), mip_level, var2.PE_CHANNELS,
                       _pe_kind(method), origin0=origin)
    return _GatherFn.apply(g0, g1, None, geom)


def finally_decode_input_2d(fp, image_size, mip_level, x=0, y=0):
    """image_compression.py:170-181."""
    return _finally_decode_input(fp, image_size, mip_level, (x, y), L.METHOD_2D)


def finally_decode_input_3d(fp, image_size, mip_level, x=0, y=0, z=0):
    """image_compression.py:184-196."""
    return _finally_decode_input(fp, image_size, mip_level, (x, y, z), L.METHOD_3D)


def finally_decode_input_3d_v2(fp, image_size, mip_level, x=0, y=0, z=0):
    """image_compression.py:199-211."""
    return _finally_decode_input(fp, image_size, mip_level, (x, y, z), L.METHOD_3D_V2)


# ------------------------------------------------------------------------------------------------ fused decode
def _check_codes(codes):
    for c in codes:
        if not c.is_cuda or c.dtype != torch.uint8 or not c.is_contiguous():
            raise TypeError("codes must be contiguous uint8 CUDA tensors")
    return codes


def _check_grids(grids, bits):
    """The grids a call reads: float32 grids (bits None) or uint8 codes (the list fp_savable returns)."""
    return [_check_grid(g.detach()) for g in grids] if bits is None else _check_codes(grids)


def _launch(h, fn, fn_codes, bits, pname, head, tail, stream):
    """fn(h, *head, *tail, precision, stream) on float32 grids (bits None), fn_codes(h, *head, bits, *tail, precision,
    stream) on codes (the library checks bits); raises on failure.  "auto" (float32 grids only): the tensor-core kernels
    where they exist (C = 12, PE = 6, hidden 64), else the reference-exact CUDA-core kernel."""
    if bits is not None:
        rc = fn_codes(h, *head, bits, *tail, L.PRECISIONS[pname], stream)
    else:
        for prec in (("f16", "f32") if pname == "auto" else (pname,)):
            rc = fn(h, *head, *tail, L.PRECISIONS[prec], stream)
            if not (rc == L.ERR_UNSUPPORTED and pname == "auto" and prec != "f32"):
                break
    L.check(h, rc)


def _decode(fp_like, bits, decoder, mip_level, size, origin, coords, precision, out_dtype, out, method, level_table):
    """Common body of decode / decode_points (bits None: float32 grids) and decode_codes / decode_points_codes (uint8 codes of
    width bits).  coords None: one block of `size` texels at `origin`; else Q one-texel blocks at coords [Q, D]."""
    method = _method() if method is None else method
    dim = 2 if method == L.METHOD_2D else 3
    table = feature_pyramid_mip_levels() if level_table is None else level_table
    fl = table[mip_level]
    g0, g1 = _check_grids((fp_like[fl * 2], fp_like[fl * 2 + 1]), bits)
    if coords is None:
        if size is None:
            size = var2.IMAGE_SIZE // pow(2, mip_level)
        block = (size,) * dim if isinstance(size, int) else tuple(size)
        blocks, shape = 1, block
    else:
        coords = L.origins_tensor(coords, g0.device, dim)
        blocks = coords.shape[0]
        if blocks >= 2 ** 31 - 128:
            raise ValueError("at most 2^31 - 129 queries per call; split the batch")
        block, shape = 1, (blocks,)
    params = [p.detach().contiguous() for p in decoder.parameters_list()]
    m = L.make_mlp(params)
    geom = L.make_geom(method, g0, g1, block, blocks, _step_log2(mip_level, fl), mip_level, var2.PE_CHANNELS, _pe_kind(method),
                       origin0=origin)
    if out_dtype not in (torch.float32, torch.uint8):
        raise TypeError("out_dtype must be torch.float32 or torch.uint8")
    shape += (m.cout,)
    if out is None:
        out = torch.empty(shape, dtype=out_dtype, device=g0.device)
    elif tuple(out.shape) != shape or out.dtype != out_dtype or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous {out_dtype} tensor of shape {shape}")
    lib = L.load_library()
    _launch(L.handle(g0.device), lib.nic_decode, lib.nic_decode_codes, bits, (precision or var2.DECODE_PRECISION).lower(),
            (C.byref(geom), L.ptr(g0), L.ptr(g1)),
            (L.ptr(coords), C.byref(m), L.ptr(out), L.DT_U8 if out_dtype == torch.uint8 else L.DT_F32), L.stream_ptr(g0.device))
    return out


def decode(fp, decoder, mip_level=0, size=None, origin=None, precision=None, out_dtype=torch.float32, out=None,
           method=None, level_table=None):
    """Fused gather + MLP for one block: the body of decode_image's single-shot branch
    (image_compression.py:313-327) without materialising X.

    size: texels per axis (int) or per-axis tuple (x, y[, z]); default IMAGE_SIZE >> mip_level.
    origin: block origin in texels of this mip level.  precision: "f32" | "f16" | "bf16" | "auto" (default
    var2.DECODE_PRECISION).  out_dtype: torch.float32 or torch.uint8 (floor(v*255+.5)).
    Returns [Sx, Sy(, Sz), Cout]."""
    return _decode(fp, None, decoder, mip_level, size, origin, None, precision, out_dtype, out, method, level_table)


def decode_codes(codes, decoder, num_bits, mip_level=0, size=None, origin=None, precision="f16", out_dtype=torch.uint8,
                 out=None, method=None, level_table=None):
    """`decode` straight from the saved model: `codes` is the list fp_savable / torch.load returns (uint8, one code per
    byte).  The de-quantisation of models.load4fp is fused into the grid read (no float32 grids are materialised)."""
    return _decode(codes, num_bits, decoder, mip_level, size, origin, None, precision, out_dtype, out, method, level_table)


def decode_points(fp, decoder, coords, mip_level=0, precision=None, out_dtype=torch.float32, method=None,
                  level_table=None):
    """Random-access decode: coords `[Q, D]` integer texel coordinates of mip `mip_level` -> `[Q, Cout]`.
    Each query is a 1-texel block whose origin is the query (the `coord` mechanism of create_decoder_input_*,
    image_compression.py:71-167, with sample_number = 1); used for LUT look-ups (BASELINE config 4).
    precision: "f32" | "f16" | "bf16" | "auto" (default var2.DECODE_PRECISION), as for `decode`."""
    return _decode(fp, None, decoder, mip_level, None, None, coords, precision, out_dtype, None, method, level_table)


def decode_points_codes(codes, decoder, coords, num_bits, mip_level=0, precision="f16", out_dtype=torch.uint8, method=None,
                        level_table=None):
    """`decode_points` straight from the saved model (`codes`: the uint8 list of fp_savable, one code per byte): the
    deployment form of a colour LUT (BASELINE config 4).  When both active grids fit into shared memory next to the
    operand buffers (a 65^3 LUT: 18^3 + 10^3 nodes = 82 KB of codes) and the precision is f16, the queries run on the
    code-resident kernel (decode_codes_smem_kernel: corner reads are shared-memory loads, models.load4fp is folded into the
    first layer); otherwise on the general tensor-core kernel with the de-quantisation fused into the grid read."""
    return _decode(codes, num_bits, decoder, mip_level, None, None, coords, precision, out_dtype, None, method, level_table)


# ------------------------------------------------------------------------------------------------ filtered sampling
_ADDRESS = {"clamp": L.ADDRESS_CLAMP, "wrap": L.ADDRESS_WRAP}


def _sample_coords(coords, dim):
    if not torch.is_tensor(coords) or coords.dtype != torch.float32 or not coords.is_contiguous():
        raise TypeError("coords must be a contiguous float32 tensor [Q, D] of normalised coordinates")
    if coords.dim() != 2 or coords.shape[1] != dim:
        raise ValueError(f"coords must be [Q, {dim}], got {tuple(coords.shape)}")
    if not coords.is_cuda:
        raise L.NicError(-3, "coords must be a CUDA tensor (no CPU fallback)")
    if coords.shape[0] << dim >= 2 ** 31 - 128:
        raise ValueError(f"at most (2^31 - 129) / {1 << dim} queries per call; split the batch")
    return coords


def _sample_passes(lod, size, table):
    """[(mip, weight)] of a sample at `lod`: one pass, or two for a fractional lod between two mips of the table."""
    if size is not None and float(lod) != math.floor(float(lod)):
        raise ValueError("size may only be given with an integer lod")
    lod = min(max(float(lod), 0.0), float(var2.MAX_MIP_LEVEL))
    m = int(math.floor(lod))
    t = lod - m
    if t == 0.0 or m >= max(table):
        return [(m, 1.0)]
    return [(m, 1.0), (m + 1, t)]


def _lod_args(lod, grad, size):
    """Is this a per-query LOD call (lod a tensor, or grad given)?  Checks what needs no tensor."""
    if grad is None and not torch.is_tensor(lod):
        return False
    if grad is not None and lod is not None:
        raise ValueError("give lod or grad, not both")
    if size is not None:
        raise ValueError("size may not be given with a per-query lod or grad (each mip has its own extent)")
    return True


def _lod_inputs(lod, grad, coords, dim):
    """(lod, ddx, ddy) of a per-query LOD call (lod a tensor [Q], or grad = (ddx, ddy) tensors [Q, D])."""
    q = coords.shape[0] if torch.is_tensor(coords) and coords.dim() == 2 else None      # (coords are checked next)
    named = [("lod", lod, (q,))] if grad is None else []
    if grad is not None:
        if not isinstance(grad, (tuple, list)) or len(grad) != 2:
            raise TypeError("grad must be a pair (ddx, ddy) of float32 tensors [Q, D]")
        named = [("ddx", grad[0], (q, dim)), ("ddy", grad[1], (q, dim))]
    for name, t, shape in named:
        if not torch.is_tensor(t) or t.dtype != torch.float32 or not t.is_contiguous():
            raise TypeError(f"{name} must be a contiguous float32 tensor {list(shape)}")
        if q is not None and tuple(t.shape) != shape:
            raise ValueError(f"{name} must be {list(shape)}, got {tuple(t.shape)}")
    for name, t, _ in named:
        if not t.is_cuda:
            raise L.NicError(-3, f"{name} must be a CUDA tensor (no CPU fallback)")
        if q is not None and coords.is_cuda and t.device != coords.device:
            raise ValueError(f"{name} is on {t.device}, coords on {coords.device}")
    return (lod, None, None) if grad is None else (None, grad[0], grad[1])


def _mip_chain(fp_like, q, address, align_corners, method, table):
    """NicMipChain of mips 0 .. min(MAX_MIP_LEVEL, max(table)), each at its default extent IMAGE_SIZE >> mip: q one-texel
    queries per mip (nic_sample_lod), or with q None one block that covers the whole mip (nic_decode_mips)."""
    dim = 2 if method == L.METHOD_2D else 3
    last = min(var2.MAX_MIP_LEVEL, max(table))
    if last + 1 > L.MAX_MIPS:
        what = "a per-query lod reaches" if q is not None else "a mip chain holds"
        raise ValueError(f"{what} at most {L.MAX_MIPS} mips; the table has {last + 1}")
    c = L.NicMipChain()
    c.num_mips, c.address, c.align_corners = last + 1, _ADDRESS[address], int(bool(align_corners))
    grids = []
    for mip in range(last + 1):
        fl = table[mip]
        g0, g1 = fp_like[fl * 2], fp_like[fl * 2 + 1]
        grids += [g0, g1]
        extent = [var2.IMAGE_SIZE // pow(2, mip) if a < dim else 1 for a in range(3)]
        block, blocks = (1, q) if q is not None else (extent[:dim], 1)
        c.geom[mip] = L.make_geom(method, g0, g1, block, blocks, _step_log2(mip, fl), mip, var2.PE_CHANNELS, _pe_kind(method))
        c.g0[mip], c.g1[mip] = L.ptr(g0), L.ptr(g1)
        for a in range(3):
            c.extent[mip][a] = extent[a]
    return c, grids


def _sample(fp_like, bits, decoder, coords, lod, size, address, align_corners, precision, out_dtype, method, level_table, grad):
    """Common body of sample (bits None: float32 grids) and sample_codes (uint8 codes of width bits)."""
    method = _method() if method is None else method
    dim = 2 if method == L.METHOD_2D else 3
    table = feature_pyramid_mip_levels() if level_table is None else level_table
    if address not in _ADDRESS:
        raise ValueError(f"address must be 'clamp' or 'wrap', got {address!r}")
    if out_dtype not in (torch.float32, torch.uint8):
        raise TypeError("out_dtype must be torch.float32 or torch.uint8")
    per_query = _lod_args(lod, grad, size)
    passes = None if per_query else _sample_passes(0 if lod is None else lod, size, table)
    lod_inputs = _lod_inputs(lod, grad, coords, dim) if per_query else None
    coords = _sample_coords(coords, dim)
    params = [p.detach().contiguous() for p in decoder.parameters_list()]
    m = L.make_mlp(params)
    q = coords.shape[0]
    out = torch.empty((q, m.cout), dtype=out_dtype, device=coords.device)
    pname = (precision or var2.DECODE_PRECISION).lower()
    lib = L.load_library()
    if per_query:
        if q > 0:
            chain, grids = _mip_chain(fp_like, q, address, align_corners, method, table)
            _check_grids(grids, bits)
            _launch(L.handle(coords.device), lib.nic_sample_lod, lib.nic_sample_lod_codes, bits, pname, (C.byref(chain),),
                    (L.ptr(coords), *[L.ptr(t) for t in lod_inputs], C.byref(m), L.ptr(out),
                     L.DT_U8 if out_dtype == torch.uint8 else L.DT_F32), L.stream_ptr(coords.device))
        return out
    prev = None
    for i, (mip, t) in enumerate(passes):
        fl = table[mip]
        g0, g1 = fp_like[fl * 2], fp_like[fl * 2 + 1]
        s = (var2.IMAGE_SIZE // pow(2, mip)) if size is None else size
        extent = (s,) * dim if isinstance(s, int) else tuple(s)
        geom = L.make_geom(method, g0, g1, 1, q, _step_log2(mip, fl), mip, var2.PE_CHANNELS, _pe_kind(method))
        smp = L.NicSampler()
        smp.address, smp.align_corners = _ADDRESS[address], int(bool(align_corners))
        for a in range(3):
            smp.extent[a] = int(extent[a]) if a < dim else 1
        smp.blend_weight, smp.blend_prev = t, (prev.data_ptr() if prev is not None else None)
        last = i == len(passes) - 1
        dst = out if last else torch.empty((q, m.cout), dtype=torch.float32, device=coords.device)
        g0, g1 = _check_grids((g0, g1), bits)
        _launch(L.handle(g0.device), lib.nic_sample, lib.nic_sample_codes, bits, pname, (C.byref(geom), L.ptr(g0), L.ptr(g1)),
                (L.ptr(coords), C.byref(smp), C.byref(m), L.ptr(dst), L.DT_U8 if last and out_dtype == torch.uint8 else L.DT_F32),
                L.stream_ptr(g0.device))
        prev = dst
    return out


def sample(fp, decoder, coords, lod=None, size=None, address="clamp", align_corners=False, precision=None,
           out_dtype=torch.float32, method=None, level_table=None, grad=None):
    """Filtered sampling at continuous coordinates: bilinear (2-D) / trilinear (3-D) reads of the decoded mip, as a renderer
    samples a texture or a colour LUT is applied, without materialising the taps (nic.h nic_sample has the exact rule).

    coords: float32 `[Q, D]` CUDA tensor of normalised coordinates in axis order (x, y[, z]).  lod: mip level; a fractional
    lod blends the two mips around it ((1 - t) * mip m + t * mip m + 1), clamped to [0, MAX_MIP_LEVEL].  size: texel extent
    of the mip (int or per-axis tuple), default IMAGE_SIZE >> lod; integer lod only.  address: "clamp" or "wrap".
    align_corners: texel i at i / (S - 1) instead of (i + .5) / S.  precision: "f32" | "f16" | "bf16" | "auto" (default
    var2.DECODE_PRECISION).  Returns `[Q, Cout]` in out_dtype (torch.float32, or torch.uint8 = floor(v*255+.5)).

    Per-query level of detail (nic.h nic_sample_lod has the exact rule): lod a float32 CUDA tensor `[Q]`, or
    grad=(ddx, ddy), float32 CUDA tensors `[Q, D]` holding the derivatives of the normalised coordinates along the screen's
    x and y (lambda = log2 of the longer one in texels of mip 0).  Each query blends the two mips around its clamped lambda,
    over mips 0 .. min(MAX_MIP_LEVEL, max(level_table)) at their default extents (no `size`), in one pass."""
    return _sample(fp, None, decoder, coords, lod, size, address, align_corners, precision, out_dtype, method, level_table, grad)


def sample_codes(codes, decoder, coords, num_bits, lod=None, size=None, address="clamp", align_corners=False,
                 precision="f16", out_dtype=torch.float32, method=None, level_table=None, grad=None):
    """`sample` straight from the saved model (`codes`: the uint8 list of fp_savable, one code per byte); the de-quantisation
    of models.load4fp is fused into the grid read.  Tensor-core precisions only."""
    return _sample(codes, num_bits, decoder, coords, lod, size, address, align_corners, precision, out_dtype, method,
                   level_table, grad)


# ------------------------------------------------------------------------------------------------ whole mip chain
def _decode_mips(fp_like, bits, decoder, precision, out_dtype, out, method, level_table):
    """Common body of decode_mips (bits None: float32 grids) and decode_mips_codes (uint8 codes of width bits)."""
    method = _method() if method is None else method
    dim = 2 if method == L.METHOD_2D else 3
    table = feature_pyramid_mip_levels() if level_table is None else level_table
    if out_dtype not in (torch.float32, torch.uint8):
        raise TypeError("out_dtype must be torch.float32 or torch.uint8")
    chain, grids = _mip_chain(fp_like, None, "clamp", False, method, table)
    params = [p.detach().contiguous() for p in decoder.parameters_list()]
    m = L.make_mlp(params)
    shapes = [tuple(chain.extent[i][:dim]) for i in range(chain.num_mips)]
    total = sum(math.prod(s) for s in shapes)
    device = grids[0].device
    if out is None:
        out = torch.empty((total, m.cout), dtype=out_dtype, device=device)
    elif (not torch.is_tensor(out) or tuple(out.shape) != (total, m.cout) or out.dtype != out_dtype or not out.is_contiguous()
          or out.device != device):
        raise ValueError(f"out must be a contiguous {out_dtype} tensor of shape {(total, m.cout)} on {device}")
    _check_grids(grids, bits)
    lib = L.load_library()
    _launch(L.handle(device), lib.nic_decode_mips, lib.nic_decode_mips_codes, bits, (precision or var2.DECODE_PRECISION).lower(),
            (C.byref(chain),), (C.byref(m), L.ptr(out), L.DT_U8 if out_dtype == torch.uint8 else L.DT_F32),
            L.stream_ptr(device))
    views, row = [], 0
    for s in shapes:
        views.append(out[row:row + math.prod(s)].view(s + (m.cout,)))
        row += math.prod(s)
    return views


def decode_mips(fp, decoder, precision=None, out_dtype=torch.float32, out=None, method=None, level_table=None):
    """Every mip of the model in one call (nic.h nic_decode_mips has the exact rule): mips 0 .. min(MAX_MIP_LEVEL,
    max(level_table)) at extents IMAGE_SIZE >> mip, the mips and extents `sample(lod=tensor)` filters across — what
    process_images decodes mip by mip (image_compression.py:400) and a renderer uploads as a mipmapped texture.

    Returns a list of per-mip tensors `[S, S(, S), Cout]` that are consecutive views of one contiguous `[total_texels, Cout]`
    buffer; `out`, if given, is that buffer.  precision: "f32" | "f16" | "bf16" | "auto" (default var2.DECODE_PRECISION), as
    for `decode`.  At f32 every mip equals `decode` of that mip bit for bit; on the tensor-core precisions mip 0 equals
    `decode` bit for bit and mips 1 .. L run as one pass with the mip as a decoder input, so a texel equals
    `sample(lod=tensor)` at its centre and may differ from `decode` of its mip by 16-bit rounding (+-1 LSB of 8 bits)."""
    return _decode_mips(fp, None, decoder, precision, out_dtype, out, method, level_table)


def decode_mips_codes(codes, decoder, num_bits, precision="f16", out_dtype=torch.uint8, out=None, method=None,
                      level_table=None):
    """`decode_mips` straight from the saved model (`codes`: the uint8 list of fp_savable, one code per byte); the
    de-quantisation of models.load4fp is fused into the grid read.  Tensor-core precisions only."""
    return _decode_mips(codes, num_bits, decoder, precision, out_dtype, out, method, level_table)


# ------------------------------------------------------------------------------------------------ baked colour LUTs
_INTERP = {"trilinear": L.INTERP_TRILINEAR, "tetrahedral": L.INTERP_TETRAHEDRAL}
_TABLE_DT = {torch.float32: L.DT_F32, torch.float16: L.DT_F16}


class BakedLut:
    """A 3-D colour LUT decoded once and packed for application to images (nic.h nic_lut_apply has the exact rule): `apply`
    is a pure gather per pixel, no decoder runs.  `table` is the `[Sx, Sy, Sz, 4]` float32 or float16 CUDA tensor (x slowest,
    channels from `cout` on are 0), `extent` is (Sx, Sy, Sz) and `cout` the number of output channels (1..4).  Build one with
    `bake_lut`, `bake_lut_codes` or `BakedLut.from_table`."""

    def __init__(self, table, extent, cout):
        self.table, self.extent, self.cout = table, tuple(int(e) for e in extent), int(cout)

    @classmethod
    def from_table(cls, dense, table_dtype=torch.float32):
        """A plain LUT: `dense` is a contiguous float32 CUDA tensor `[Sx, Sy, Sz, C]`, C in 1..4 (what `decode` writes for a
        3-D block), packed as float32 (exact) or float16 (`__float2half_rn` of each value)."""
        if not torch.is_tensor(dense) or dense.dtype != torch.float32 or not dense.is_contiguous():
            raise TypeError("dense must be a contiguous float32 tensor [Sx, Sy, Sz, C]")
        if dense.dim() != 4 or not 1 <= dense.shape[3] <= 4 or dense.numel() == 0:
            raise ValueError(f"dense must be [Sx, Sy, Sz, C] with every extent >= 1 and C in 1..4, got {tuple(dense.shape)}")
        if table_dtype not in _TABLE_DT:
            raise TypeError("table_dtype must be torch.float32 or torch.float16")
        if not dense.is_cuda:
            raise L.NicError(-3, "dense must be a CUDA tensor (no CPU fallback)")
        extent, cout = tuple(dense.shape[:3]), int(dense.shape[3])
        table = torch.empty(extent + (4,), dtype=table_dtype, device=dense.device)
        h = L.handle(dense.device)
        L.check(h, L.load_library().nic_lut_pack(h, L.ptr(dense), (C.c_int32 * 3)(*extent), cout, L.ptr(table),
                                                 _TABLE_DT[table_dtype], L.stream_ptr(dense.device)))
        return cls(table, extent, cout)

    def apply(self, image, interpolation="trilinear", out_dtype=torch.uint8, out=None):
        """Applies the LUT to every pixel of `image`, a contiguous uint8 or float32 CUDA tensor `[..., 3]` (`[H, W, 3]`,
        `[F, H, W, 3]`, `[N, 3]`): R, G, B index the x, y, z axes; uint8 values are read as v / 255, floats as given
        (align_corners, clamped at the edges).  interpolation: "trilinear" (8 texels) or "tetrahedral" (4 texels, exact on
        the neutral axis).  Returns `[..., cout]` in out_dtype (torch.uint8 = floor(v*255+.5), or torch.float32), written
        into `out` when given (a contiguous tensor of that shape and dtype that does not overlap `image`)."""
        if interpolation not in _INTERP:
            raise ValueError(f"interpolation must be 'trilinear' or 'tetrahedral', got {interpolation!r}")
        if out_dtype not in (torch.float32, torch.uint8):
            raise TypeError("out_dtype must be torch.float32 or torch.uint8")
        if not torch.is_tensor(image) or image.dtype not in (torch.uint8, torch.float32) or not image.is_contiguous():
            raise TypeError("image must be a contiguous uint8 or float32 tensor [..., 3]")
        if image.dim() < 1 or image.shape[-1] != 3:
            raise ValueError(f"image must be [..., 3] (R, G, B last), got {tuple(image.shape)}")
        if not image.is_cuda:
            raise L.NicError(-3, "image must be a CUDA tensor (no CPU fallback)")
        if image.device != self.table.device:
            raise ValueError(f"image is on {image.device}, the LUT on {self.table.device}")
        shape = tuple(image.shape[:-1]) + (self.cout,)
        if out is None:
            out = torch.empty(shape, dtype=out_dtype, device=image.device)
        elif (not torch.is_tensor(out) or tuple(out.shape) != shape or out.dtype != out_dtype or not out.is_contiguous()
              or out.device != image.device):
            raise ValueError(f"out must be a contiguous {out_dtype} tensor of shape {shape} on {image.device}")
        pixels = image.numel() // 3
        s0, d0 = image.data_ptr(), out.data_ptr()
        if pixels > 0 and s0 < d0 + out.numel() * out.element_size() and d0 < s0 + image.numel() * image.element_size():
            raise ValueError("out overlaps image (the LUT is not applied in place)")
        lut = L.NicLut()
        lut.table, lut.table_dtype, lut.cout = self.table.data_ptr(), _TABLE_DT[self.table.dtype], self.cout
        for a in range(3):
            lut.extent[a] = self.extent[a]
        h = L.handle(image.device)
        L.check(h, L.load_library().nic_lut_apply(h, C.byref(lut), L.ptr(image), L.DT_U8 if image.dtype == torch.uint8 else L.DT_F32,
                                                  pixels, L.ptr(out), L.DT_U8 if out_dtype == torch.uint8 else L.DT_F32,
                                                  _INTERP[interpolation], L.stream_ptr(image.device)))
        return out


def _lut_method(method):
    method = _method() if method is None else method
    if method == L.METHOD_2D:
        raise ValueError("a 2-D model is a texture (read it with sample); a colour LUT needs a 3-D model (method 3 or 4)")
    return method


def bake_lut(fp, decoder, mip_level=0, size=None, precision=None, method=None, level_table=None):
    """Bakes a 3-D model into a `BakedLut`: one dense `decode` of the whole mip with float32 output (size and defaults as
    `decode`; a 65^3 LUT passes size=65), packed as a float32 table when precision is "f32" (default
    var2.DECODE_PRECISION) and as float16 for the tensor-core precisions."""
    method = _lut_method(method)
    pname = (precision or var2.DECODE_PRECISION).lower()
    dense = decode(fp, decoder, mip_level, size, None, pname, torch.float32, None, method, level_table)
    return BakedLut.from_table(dense, torch.float32 if L.PRECISIONS.get(pname) == L.PREC_F32 else torch.float16)


def bake_lut_codes(codes, decoder, num_bits, mip_level=0, size=None, precision="f16", method=None, level_table=None):
    """`bake_lut` straight from the saved model (`codes`: the uint8 list of fp_savable): one dense `decode_codes`."""
    method = _lut_method(method)
    dense = decode_codes(codes, decoder, num_bits, mip_level, size, None, precision, torch.float32, None, method, level_table)
    return BakedLut.from_table(dense, torch.float32 if L.PRECISIONS.get(precision.lower()) == L.PREC_F32 else torch.float16)


class DecodeSession:
    """A model that is decoded many times (regions, mips, repeated frames): the private tensor-core tables (16-bit
    channel-last shadow grids, per-node G1 rows, packed weight images) are built by the first `decode` and REUSED by the
    following ones (NIC_OPT_REUSE_PREPARED) — the grids and the decoder are the model's weights, and this is their
    load-time re-packing.  The caller promises not to modify `fp` / `decoder` between calls; call `refresh()` after a
    change (or simply use `decode(...)`, which always rebuilds)."""

    def __init__(self, fp, decoder, precision="f16"):
        self.fp, self.decoder, self.precision = fp, decoder, precision
        self._fresh = False

    def refresh(self):
        self._fresh = False

    def decode(self, mip_level=0, size=None, origin=None, out_dtype=torch.uint8, out=None, **kw):
        dev = self.fp[0].device
        L.set_option(dev, L.OPT_REUSE_PREPARED, int(self._fresh))
        try:
            res = decode(self.fp, self.decoder, mip_level, size, origin, self.precision, out_dtype, out, **kw)
        finally:
            L.set_option(dev, L.OPT_REUSE_PREPARED, 0)
        self._fresh = True          # (a different mip level / path re-keys the tables inside the library and rebuilds)
        return res

    def sample(self, coords, lod=None, size=None, out_dtype=torch.uint8, **kw):
        """`sample(...)` of this model, reusing the tensor-core tables like `decode` (the library rebuilds them when the mip or
        the kernel they were built for differs).  A per-query lod or grad= reuses the tables of the whole mip chain."""
        dev = self.fp[0].device
        L.set_option(dev, L.OPT_REUSE_PREPARED, int(self._fresh))
        try:
            res = sample(self.fp, self.decoder, coords, lod, size, precision=self.precision, out_dtype=out_dtype, **kw)
        finally:
            L.set_option(dev, L.OPT_REUSE_PREPARED, 0)
        self._fresh = True
        return res


class HostDecodePipeline:
    """End-to-end decode of 2-D frames from HOST buffers to a HOST buffer (what `process_images` does with a saved
    model, image_compression.py:393-407), as a three-stream pipeline:
      upload stream : pinned H2D of the uint8 grid codes and the decoder parameters (double-buffered on the device);
      caller stream : decode-from-codes in row bands (the tables are built by the first band and reused by the others);
      copy stream   : D2H of each 8-bit band while the next band decodes (the device frame is double-buffered too).
    With `wait=False` the H2D of frame i + 1 and the D2H of frame i overlap the decode of frame i (PCIe is full
    duplex).  `decode_frame` never blocks the host on the device, with either `wait`, so the host buffers of a frame stay
    in use after it returns:
      * `codes` and `host_params` are read by the frame's upload, which may still be pending (it waits for the decode
        of frame i - 2 to release its device buffer).  Overwrite them, e.g. with the next frame's model, only after
        `self.uploaded.synchronize()` (the upload event of the latest frame) or a later host synchronisation of the
        caller's stream.
      * `host_out` is written by the frame's downloads.  Read it only after synchronising the caller's stream: with
        `wait=True` that stream already waits for the downloads, with `wait=False` call `finish()` first.  A later frame
        may write the same `host_out` at once (the downloads are ordered on one stream)."""

    def __init__(self, size, device, precision="f16", bands=4, bits=8):
        self.size, self.device, self.precision, self.bits = size, torch.device(device), precision, bits
        self.bands = [(r0, n) for r0, n in (_band(size, b, bands) for b in range(bands)) if n > 0]
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.up_stream = torch.cuda.Stream(device=self.device)
        self.decoders = None
        self.dcodes = None
        self.out = None
        self.d2h_done = [None, None]
        self.dec_done = [None, None]
        self.uploaded = None
        self.frame = 0
        self._last = None

    def decode_frame(self, codes, host_params, host_out, mip_level=0, wait=True):
        dev = self.device
        if self.dcodes is None:
            self.dcodes = [[torch.empty(c.shape, dtype=torch.uint8, device=dev) for c in codes] for _ in range(2)]
            self.decoders = [ColorDecoder(host_params[0].shape[1], host_params[0].shape[0], host_params[4].shape[0]).to(dev)
                             for _ in range(2)]
            shape = (self.size, self.size, host_params[4].shape[0])
            self.out = [torch.empty(shape, dtype=torch.uint8, device=dev) for _ in range(2)]
        main = torch.cuda.current_stream(dev)
        k = self.frame & 1
        self.frame += 1
        # ---- upload (buffer k was last read by the decode of frame - 2)
        if self.dec_done[k] is not None:
            self.up_stream.wait_event(self.dec_done[k])
        else:
            # first use of buffer k: it was allocated on the caller's stream, and the caching allocator may have handed
            # out a block whose previous use on that stream is still pending
            self.up_stream.wait_stream(main)
            self.copy_stream.wait_stream(main)
            for t in self.dcodes[k] + list(self.decoders[k].parameters_list()):
                t.record_stream(self.up_stream)
            self.out[k].record_stream(self.copy_stream)
        with torch.cuda.stream(self.up_stream):
            for d, c in zip(self.dcodes[k], codes):
                d.copy_(c, non_blocking=True)
            with torch.no_grad():
                for p, hp in zip(self.decoders[k].parameters_list(), host_params):
                    p.copy_(hp, non_blocking=True)
            uploaded = torch.cuda.Event()
            uploaded.record(self.up_stream)
        self.uploaded = uploaded
        main.wait_event(uploaded)
        if self.d2h_done[k] is not None:
            main.wait_event(self.d2h_done[k])        # the frame that used this device buffer two frames ago has left
        out = self.out[k]
        try:
            for i, (r0, n) in enumerate(self.bands):
                L.set_option(dev, L.OPT_REUSE_PREPARED, int(i > 0))
                band = out[r0:r0 + n]
                decode_codes(self.dcodes[k], self.decoders[k], self.bits, mip_level, size=(n, self.size), origin=(r0, 0),
                             precision=self.precision, out_dtype=torch.uint8, out=band)
                ready = torch.cuda.Event()
                ready.record(main)
                self.copy_stream.wait_event(ready)
                with torch.cuda.stream(self.copy_stream):
                    host_out[r0:r0 + n].copy_(band, non_blocking=True)
        finally:
            L.set_option(dev, L.OPT_REUSE_PREPARED, 0)
        self.dec_done[k] = torch.cuda.Event()
        self.dec_done[k].record(main)
        done = torch.cuda.Event()
        done.record(self.copy_stream)
        self.d2h_done[k] = done
        self._last = done
        if wait:
            main.wait_event(done)            # the frame is complete (in host memory) when the caller's stream gets here
        return host_out

    def finish(self):
        """Makes the caller's stream wait for every outstanding device-to-host copy."""
        if self._last is not None:
            torch.cuda.current_stream(self.device).wait_event(self._last)


def _band(size, b, bands):
    from .parallel import shard_rows
    return shard_rows(size, b, bands)


def decode_image(fp, arc_decoder, mip_level, pr=True, div_size=10, precision=None):
    """image_compression.py:307-346 — full-frame decode; <= 2^div_size-texel tiles when the frame is larger.
    Differences from the reference, both deliberate: the tiled result is assembled on the device (the
    reference assembles it in a CPU tensor, :329), and 3-D tiling passes all three origins (the reference's
    3-D tiled branch passes only x,y, :338-340)."""
    with torch.no_grad():
        power = var2.MAX_MIP_LEVEL - mip_level
        div_slice = pow(2, max(power - div_size, 0))
        div_count = pow(div_slice, 2)
        decode_size = var2.IMAGE_SIZE // pow(2, mip_level)
        dim = var2.FP_DIMENSION
        fused = isinstance(arc_decoder, ColorDecoder)

        def one(size, origin):
            if fused:
                return decode(fp, arc_decoder, mip_level, size, origin, precision)
            method = _method()
            x = _finally_decode_input(fp, size, mip_level, origin, method)
            return arc_decoder(x).reshape((size,) * dim + (-1,))

        if div_count == 1:
            out = one(decode_size, (0,) * dim)
            if pr:
                print(torch.Size([out.numel() // out.shape[-1], out.shape[-1]]))
            return out
        if dim != 2:
            raise NotImplementedError("tiled decode is 2-D only, as in the reference (image_compression.py:329-345)")
        result = torch.zeros(decode_size, decode_size, var2.OUTPUT_CHANNELS, dtype=torch.float32, device=fp[0].device)
        sample_number = var2.IMAGE_SIZE // pow(2, mip_level + max(power - div_size, 0))
        for i in range(div_count):
            x, y = i % div_slice, i // div_slice
            tile = one(sample_number, (sample_number * x, sample_number * y))
            if pr:
                print(torch.Size([tile.numel() // tile.shape[-1], tile.shape[-1]]))
            result[sample_number * x:sample_number * (x + 1), sample_number * y:sample_number * (y + 1), :] = tile
        return result


# ------------------------------------------------------------------------------------------------ crop sampler
def sample_crops(dataset, coord, crop_size):
    """Target gather of random_crop_dataset (image_compression.py:44-47) as ONE kernel: `dataset` [Ci, S, S(, S)]
    float32 on the device, `coord` [NC, D] crop origins -> `[NC, crop^D, Ci]`."""
    dim = dataset.dim() - 1
    if not dataset.is_cuda:
        raise L.NicError(-3, "dataset must be a CUDA tensor (no CPU fallback)")
    if dataset.dtype != torch.float32 or not dataset.is_contiguous():
        raise TypeError("dataset must be contiguous float32")
    coord = L.origins_tensor(coord, dataset.device, dim)
    nc, ci = coord.shape[0], dataset.shape[0]
    out = torch.empty((nc, crop_size ** dim, ci), dtype=torch.float32, device=dataset.device)
    size = (C.c_int32 * 3)(*(list(dataset.shape[1:]) + [1] * (3 - dim)))
    crop = (C.c_int32 * 3)(*([crop_size] * dim + [1] * (3 - dim)))
    h = L.handle(dataset.device)
    L.check(h, L.load_library().nic_sample_crops(h, L.ptr(dataset), dim, ci, C.cast(size, C.c_void_p), L.ptr(coord), nc,
                                                 C.cast(crop, C.c_void_p), L.ptr(out), L.stream_ptr(dataset.device)))
    return out


def random_crop_dataset(datasets, crop_size, num_crops, uniform_distribution, dim=2):
    """image_compression.py:26-50 — host RNG LOD draw + integer crop origins (as in the reference); the target
    slices `[NC, S^D, C]` are gathered by one kernel instead of NC slice/reshape/transpose chains."""
    if uniform_distribution:
        lod = random.randint(0, var2.MAX_MIP_LEVEL)
    else:
        lod = int(math.floor(-math.log2(random.random()) / 2))
        if lod > var2.MAX_MIP_LEVEL:
            lod = var2.MAX_MIP_LEVEL
    dataset = datasets[lod]
    data_size = dataset.shape[1]
    re_crop_size = max(1, crop_size // pow(2, lod))
    coord = torch.randint(0, data_size - re_crop_size + 1, (num_crops, dim)).to(dataset.device)
    return sample_crops(dataset, coord, re_crop_size), coord, lod


def random_crop_dataset_device(datasets, crop_size, num_crops, lod, seed, step, dim=2):
    """random_crop_dataset (image_compression.py:36-49) with NO host work after the LOD draw: the crop origins are drawn on
    the device (Philox keyed by (seed, step), uniform over [0, size - crop] like torch.randint) and the targets are
    gathered in the same launch (nic_sample_crops_random).  `lod` is the step's mip level (FusedTrainer.draw_lod or
    DataParallelPlan.next_lod).  Returns (inputs [NC, crop^D, C], coord [NC, D] int64 on the device)."""
    dataset = datasets[lod]
    if not dataset.is_cuda:
        raise L.NicError(-3, "dataset must be a CUDA tensor (no CPU fallback)")
    if dataset.dtype != torch.float32 or not dataset.is_contiguous():
        raise TypeError("dataset must be contiguous float32")
    if dataset.dim() != dim + 1:
        raise ValueError(f"dataset must be [C, {'S, ' * dim}] for dim {dim}")
    re_crop_size = max(1, crop_size // pow(2, lod))
    ci = dataset.shape[0]
    out = torch.empty((num_crops, re_crop_size ** dim, ci), dtype=torch.float32, device=dataset.device)
    coord = torch.empty((num_crops, dim), dtype=torch.int64, device=dataset.device)
    size = (C.c_int32 * 3)(*(list(dataset.shape[1:]) + [1] * (3 - dim)))
    crop = (C.c_int32 * 3)(*([min(re_crop_size, dataset.shape[1 + a]) for a in range(dim)] + [1] * (3 - dim)))
    h = L.handle(dataset.device)
    L.check(h, L.load_library().nic_sample_crops_random(h, L.ptr(dataset), dim, ci, C.cast(size, C.c_void_p), num_crops,
                                                        C.cast(crop, C.c_void_p), int(seed) & (2 ** 64 - 1), int(step),
                                                        L.ptr(coord), L.ptr(out), L.stream_ptr(dataset.device)))
    return out, coord


# ------------------------------------------------------------------------------------------------ data front end
def resize_image(image_u8, out_height, out_width, want_u8=False):
    """transforms.Resize((h, w)) + transforms.ToTensor() on an 8-bit image (image_compression.py:436-441), on the device:
    `image_u8` uint8 [H, W, C] (PIL / numpy layout) -> float32 [C, h, w] in [0, 1].  Bit-exact with Pillow's antialiased
    BILINEAR resample (nic_resize_bilinear_u8).  want_u8: also return the 8-bit [h, w, C] image."""
    if not image_u8.is_cuda:
        raise L.NicError(-3, "image must be a CUDA tensor (no CPU fallback)")
    if image_u8.dtype != torch.uint8 or image_u8.dim() != 3 or not image_u8.is_contiguous():
        raise TypeError("image must be a contiguous uint8 [H, W, C] tensor")
    hh, ww, cc = image_u8.shape
    out = torch.empty((cc, out_height, out_width), dtype=torch.float32, device=image_u8.device)
    out8 = torch.empty((out_height, out_width, cc), dtype=torch.uint8, device=image_u8.device) if want_u8 else None
    h = L.handle(image_u8.device)
    L.check(h, L.load_library().nic_resize_bilinear_u8(h, L.ptr(image_u8), hh, ww, cc, out_height, out_width, L.ptr(out8),
                                                       L.ptr(out), L.stream_ptr(image_u8.device)))
    return (out, out8) if want_u8 else out


def build_mip_pyramid(image_u8, image_size=None, max_mip_level=None):
    """The `images` list of the script (image_compression.py:433-442): mip i = Resize((S >> i, S >> i)) of the ORIGINAL
    8-bit image, ToTensor -> float32 [C, S >> i, S >> i] on the device, for i = 0..MAX_MIP_LEVEL."""
    size = var2.IMAGE_SIZE if image_size is None else image_size
    top = var2.MAX_MIP_LEVEL if max_mip_level is None else max_mip_level
    return [resize_image(image_u8, size // pow(2, i), size // pow(2, i)) for i in range(top + 1)]


def flatten_movie_to_atlas(movie_u8, image_size=None):
    """COMPRESSION_METHOD 2 (image_compression.py:453-460): frames [T, S, S, C] uint8 -> one [IMAGE_SIZE, IMAGE_SIZE, C] image,
    frame i at tile (i // (IMAGE_SIZE // S), i % (IMAGE_SIZE // S)); unused tiles are zero."""
    if not movie_u8.is_cuda:
        raise L.NicError(-3, "movie must be a CUDA tensor (no CPU fallback)")
    if movie_u8.dtype != torch.uint8 or movie_u8.dim() != 4 or movie_u8.shape[1] != movie_u8.shape[2] or not movie_u8.is_contiguous():
        raise TypeError("movie must be a contiguous uint8 [T, S, S, C] tensor")
    t, sz, _, cc = movie_u8.shape
    a = var2.IMAGE_SIZE if image_size is None else image_size
    atlas = torch.empty((a, a, cc), dtype=torch.uint8, device=movie_u8.device)
    h = L.handle(movie_u8.device)
    L.check(h, L.load_library().nic_atlas_pack(h, L.ptr(movie_u8), t, sz, cc, a, L.ptr(atlas), L.stream_ptr(movie_u8.device)))
    return atlas


def unflatten_atlas(image_u8, size_3d=None, num_frames=None):
    """The inverse on the decoded frame (image_compression.py:410-419): [A, A, C] uint8 -> [T, S, S, C], S = IMAGE_3D_SIZE,
    T = S frames unless `num_frames` says otherwise."""
    if not image_u8.is_cuda:
        raise L.NicError(-3, "image must be a CUDA tensor (no CPU fallback)")
    if image_u8.dtype != torch.uint8 or image_u8.dim() != 3 or image_u8.shape[0] != image_u8.shape[1] or not image_u8.is_contiguous():
        raise TypeError("image must be a contiguous uint8 [A, A, C] tensor")
    sz = var2.IMAGE_3D_SIZE if size_3d is None else size_3d
    t = sz if num_frames is None else num_frames
    a, _, cc = image_u8.shape
    frames = torch.empty((t, sz, sz, cc), dtype=torch.uint8, device=image_u8.device)
    h = L.handle(image_u8.device)
    L.check(h, L.load_library().nic_atlas_unpack(h, L.ptr(image_u8), a, cc, t, sz, L.ptr(frames), L.stream_ptr(image_u8.device)))
    return frames


# ------------------------------------------------------------------------------------------------ fused training
class FusedTrainer:
    """The body of train_models (image_compression.py:215-269) as fused CUDA launches per step:
    one forward+backward kernel (gather, noise, MLP, MSE, backward, grid-gradient scatter), an optional
    single NCCL all-reduce of the flat gradient buffer (data parallel), and one fused Adam (+ cosine LR,
    + clamp of the active grids, + gradient zeroing).

    Semantics kept from the reference: Adam defaults with lr 0.01 (grids) / 0.005 (decoder) and
    CosineAnnealingLR(T_max=NUM_EPOCHS) (:361-365); per-tensor Adam step counts — grids of inactive levels
    are skipped entirely (SURVEY A.2); noise on every input column while epoch < 0.95 N (:248-254); freeze +
    quantise the grids once epoch > 0.95 N (:227-231); clamp of the two active grids after each step (:269).
    """

    PEER_EXCHANGE_MAX_BYTES = 4 << 20      # above this (and more than two ranks) the fused exchange runs sliced: see _peer_level
    PEER_SYMMETRIC_MAX_BYTES = 1 << 30     # "auto" keeps nccl for flat buffers beyond this (symmetric memory is allocated twice)

    def __init__(self, fp, decoder, num_epochs=None, fp_bits=None, lr_fp=0.01, lr_mlp=0.005, betas=(0.9, 0.999),
                 eps=1e-8, method=None, level_table=None, process_group=None, seed=0, precision="f32", exchange="auto",
                 metrics_ring=4096, data_parallel=True, exchange_timeout_ms=None):
        self.fp = [_check_grid(g.detach()) for g in fp]
        self.decoder = decoder
        self.params = [p.detach() for p in decoder.parameters_list()]
        self.num_epochs = var2.NUM_EPOCHS if num_epochs is None else num_epochs
        self.bits = var2.FP_BITS if fp_bits is None else fp_bits
        self.lr_fp, self.lr_mlp, self.betas, self.eps = lr_fp, lr_mlp, betas, eps
        self.method = _method() if method is None else method
        self.dim = 2 if self.method == L.METHOD_2D else 3
        self.table = feature_pyramid_mip_levels() if level_table is None else level_table
        self.pg = process_group
        self.world = 1
        if data_parallel and torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world = torch.distributed.get_world_size(process_group)
        self.seed = seed
        self.rank = torch.distributed.get_rank(process_group) if self.world > 1 else 0
        self._cache = {}
        # "f32" reference-exact; "f16" / "bf16" tcgen05 path; "auto": f16 where the tensor-core kernels exist (C = 12, PE = 6,
        # hidden 64, <= 16 outputs), else f32 — decided once, from the shapes
        if precision.lower() == "auto":
            c_ok = self.fp[0].shape[0] == 12 and var2.PE_CHANNELS == 6
            m_ok = self.params[0].shape[0] == 64 and self.params[4].shape[0] <= 16
            precision = "f16" if (c_ok and m_ok) else "f32"
        self.precision_name = precision.lower()
        self.precision = L.PRECISIONS[precision.lower()]
        self.epoch = 0
        self.frozen = False
        dev = self.fp[0].device
        self.device = dev
        if exchange_timeout_ms is not None:      # how long the fused exchange waits on the device for a peer (default 10 s)
            L.set_option(dev, L.OPT_EXCHANGE_TIMEOUT_MS, int(exchange_timeout_ms))
        # one flat gradient buffer per pyramid level: [dG0 | dG1 | dW1 db1 dW2 db2 dW3 db3 | loss] -> one all-reduce
        self._flat = {}
        # The exchange step under data parallelism: "nccl" = all_reduce(flat) then Adam; "peer" = ONE kernel that reads the
        # peers' flat buffers over NVLink and applies Adam (nic_adam_step_exchange); "auto" = peer for flat buffers up to
        # PEER_EXCHANGE_MAX_BYTES when every rank could map every peer, else nccl.
        # A one-shot exchange reads all `world` buffers on every rank; beyond PEER_EXCHANGE_MAX_BYTES (and two ranks) the
        # kernel runs SLICED: rank r sums slice r of every buffer, writes it back to all of them, second handshake, Adam
        # from the own buffer — 2 (world-1)/world of the buffer per rank over NVLink ("sliced" forces that mode).
        if exchange not in ("auto", "nccl", "peer", "sliced"):
            raise ValueError("exchange must be 'auto', 'nccl', 'peer' or 'sliced'")
        self.exchange = exchange
        self._peer = {}          # level -> symmetric buffers, peer pointers, use count (None: this level uses nccl)
        self.state = {}          # id -> (m, v, t)
        self.q_min = -(pow(2, self.bits) - 1) / pow(2, self.bits + 1)
        # per-step metrics stay on the device (the reference syncs with loss.item() every step, :275): every step writes
        # (loss, mse of the 8-bit outputs) into a ring slot; flush_metrics() reads the steps since the last flush at once
        self.metrics_ring = max(16, int(metrics_ring))
        self._ring = torch.zeros((self.metrics_ring, 2), dtype=torch.float32, device=dev)
        self._ring_base = 0      # first step held by the current ring tensor
        self._flushed = 0        # steps already returned by flush_metrics
        self._old_rings = []     # (base, tensor) of rings that still hold unflushed steps
        from .parallel import DataParallelPlan
        self._plan = DataParallelPlan(var2.MAX_MIP_LEVEL, var2.UNIFORM_DISTRIBUTION_RATE, seed=seed, rank=self.rank,
                                      world=self.world, group=process_group)
        self._checked_uniform = False
        self._sample_stream, self._sample_key, self._sample_slots, self._sample_geo = None, None, None, {}
        self._prefetched = None  # the sampler launch of the NEXT step (step_sampled)

    # -- buffers
    def _level_buffers(self, fl):
        if fl not in self._flat:
            sizes, offs, total = self._level_layout(fl)          # every view 16-byte aligned
            flat = torch.zeros(total, dtype=torch.float32, device=self.device)
            views = [flat[o:o + s] for o, s in zip(offs, sizes)]
            self._flat[fl] = (flat, views)
        return self._flat[fl]

    def _level_layout(self, fl):
        sizes = [self.fp[2 * fl].numel(), self.fp[2 * fl + 1].numel()] + [p.numel() for p in self.params] + [4]
        offs, total = [], 0
        for s in sizes:
            offs.append(total)
            total += (s + 3) // 4 * 4
        return sizes, offs, total

    def _peer_level(self, fl):
        """Symmetric double-buffered flat gradient buffers of level `fl`, mapped on every rank (collective on first
        use: all ranks reach it in the same step because they draw the same LOD sequence).  None -> use nccl."""
        if fl in self._peer:
            return self._peer[fl]
        dist = torch.distributed
        sizes, offs, total = self._level_layout(fl)
        want = self.world > 1 and self.world <= L.MAX_PEERS and self.exchange != "nccl" and \
            (self.exchange != "auto" or total * 4 <= self.PEER_SYMMETRIC_MAX_BYTES)
        sliced = self.exchange == "sliced" or (self.exchange != "nccl" and self.world > 2 and
                                               total * 4 > self.PEER_EXCHANGE_MAX_BYTES)
        ent = None
        if want:
            ok, buf, bases = 1, None, []
            try:
                buf = L.SymmetricBuffer(self.device, 2 * total + 64)          # [parity 0 | parity 1 | flag words]
                handles = [None] * self.world
                dist.all_gather_object(handles, buf.handle, group=self.pg)
                bases = [buf.ptr if r == self.rank else buf.open_peer(handles[r]) for r in range(self.world)]
            except Exception:                                                  # no IPC / no peer access on this box
                ok = 0
                if buf is None:       # keep the collective below matched even when the allocation itself failed
                    dist.all_gather_object([None] * self.world, b"", group=self.pg)
            flag = torch.tensor([ok], dtype=torch.int32, device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.pg)
            if int(flag.item()) == 1:
                flats = []
                for par in range(2):
                    flat = buf.tensor[par * total:(par + 1) * total]
                    flats.append((flat, [flat[o:o + s] for o, s in zip(offs, sizes)]))
                ent = {"buf": buf, "bases": bases, "flats": flats, "total": total, "uses": 0, "xch": {},
                       "mode": L.EXCHANGE_SLICED if sliced else L.EXCHANGE_ONE_SHOT}
            else:
                if self.exchange in ("peer", "sliced"):
                    raise RuntimeError(f"exchange='{self.exchange}': the ranks could not map each other's buffers (CUDA IPC)")
                if buf is not None:
                    buf.close()
        self._peer[fl] = ent
        return ent

    def close(self):
        """Unmaps the peers' buffers and frees this rank's symmetric buffers (call on every rank, after a barrier).
        Raises if an exchange timed out since the last check (the replicas then stopped updating, see nic.h)."""
        used_peer = any(v is not None for v in self._peer.values())
        failed = used_peer and L.exchange_status(self.device)
        self._close_buffers()
        if failed:
            raise L.NicError(L.ERR_EXCHANGE, "a data-parallel exchange timed out waiting for a peer; parameters were not "
                                             "updated from that step on")

    def _close_buffers(self):
        for ent in self._peer.values():
            if ent is not None:
                ent["flats"], ent["xch"] = [], {}
                ent["buf"].close()
        self._peer = {}
        self._cache.clear()

    def exchange_in_use(self):
        """'none' (single process), 'peer' / 'sliced' (every level used so far exchanges over peer memory, one-shot / sliced),
        'nccl' or 'mixed'."""
        if self.world == 1:
            return "none"
        kinds = {"nccl" if v is None else ("sliced" if v["mode"] == L.EXCHANGE_SLICED else "peer") for v in self._peer.values()}
        return kinds.pop() if len(kinds) == 1 else ("mixed" if kinds else "nccl")

    def _exchange_desc(self, ent, parity):
        x = ent["xch"].get(parity)
        if x is None:
            x = L.NicExchange()
            x.world, x.rank, x.reserved = self.world, self.rank, ent["mode"]
            for r, base in enumerate(ent["bases"]):
                x.peer_flat[r] = base + 4 * parity * ent["total"]
                x.peer_flag[r] = base + 8 * ent["total"]
            x.zero_buf = ent["bases"][self.rank] + 4 * (1 - parity) * ent["total"]
            x.zero_numel = ent["total"]
            ent["xch"][parity] = x
        return x

    def _adam_state(self, key, like):
        if key not in self.state:
            self.state[key] = [torch.zeros_like(like), torch.zeros_like(like), 0]
        return self.state[key]

    def lr_scale(self, epoch):
        """CosineAnnealingLR closed form, eta_min = 0 (image_compression.py:365)."""
        return (1.0 + math.cos(math.pi * epoch / self.num_epochs)) / 2.0 if self.num_epochs > 0 else 1.0

    def step(self, coord, targets, lod, noise=None, out=None):
        """One training step.  coord [NC, D] crop origins (int64), targets [NC, S^D, Cout] or [N, Cout] float32,
        lod = mip level of this step.  noise: None -> in-kernel Philox noise while epoch < .95 N;
        a tensor [N, Cin] -> injected noise (parity tests); False -> no noise.  Returns the loss (0-dim
        device tensor, mean over N*Cout, averaged over ranks when data parallel)."""
        lib = L.load_library()
        epoch = self.epoch
        if epoch > self.num_epochs * 0.95 and not self.frozen:       # image_compression.py:227-231
            for i, g in enumerate(self.fp):
                g.copy_(quantize4fp(g, self.bits))
            self.frozen = True
            self._cache.clear()
        fl = self.table[lod]
        g0, g1 = self.fp[2 * fl], self.fp[2 * fl + 1]
        sample_number = pow(2, max(0, (8 if self.dim == 2 else var2.CROP_MIP_LEVEL) - lod))
        coord = L.origins_tensor(coord, self.device, self.dim)
        nc = coord.shape[0]
        if self.world > 1 and not self._checked_uniform:
            # every rank must pass the same (lod, crop count): the gradient denominator is n * world, and the peer
            # buffers and flag tokens are keyed per level.  Checked on the first step (all ranks are here together);
            # draw_lod() / step_sampled() make it true by construction afterwards.
            chk = torch.tensor([lod, -lod, nc, -nc], dtype=torch.int64, device=self.device)
            torch.distributed.all_reduce(chk, op=torch.distributed.ReduceOp.MAX, group=self.pg)
            mx = chk.tolist()
            if mx[0] != -mx[1] or mx[2] != -mx[3]:
                raise ValueError(f"data-parallel step: ranks disagree on (lod, crops): lod {-mx[1]}..{mx[0]}, crops {-mx[3]}..{mx[2]}")
            self._checked_uniform = True
        peer = self._peer_level(fl) if self.world > 1 else None
        parity = (peer["uses"] & 1) if peer else 0
        # descriptors that only depend on (lod, crops) are built once (host overhead matters at ~0.2 ms per step)
        key = (lod, nc, parity)
        ent = self._cache.get(key)
        if ent is None:
            geom = L.make_geom(self.method, g0, g1, sample_number, nc, _step_log2(lod, fl), lod, var2.PE_CHANNELS,
                               _pe_kind(self.method))
            m = L.make_mlp(self.params)
            flat, views = peer["flats"][parity] if peer else self._level_buffers(fl)
            gm = L.make_mlp_grad(views[2:8])
            entries = []
            if not self.frozen:
                for j, (g, dg) in enumerate(((g0, views[0]), (g1, views[1]))):
                    entries.append((("g", 2 * fl + j), g.view(-1), dg, self.lr_fp, True))
            for i, p in enumerate(self.params):
                entries.append((("p", i), p.view(-1), views[2 + i], self.lr_mlp, False))
            arr = (L.NicAdamTensor * len(entries))()
            states = []
            for k, (skey, p, g, lr, clamp) in enumerate(entries):
                stt = self._adam_state(skey, p)
                states.append((stt, lr))
                a = arr[k]
                a.p, a.g, a.m, a.v = p.data_ptr(), g.data_ptr(), stt[0].data_ptr(), stt[1].data_ptr()
                a.numel = p.numel()
                a.clamp, a.clamp_lo, a.clamp_hi = int(clamp), self.q_min, 0.5
            loss_out = torch.zeros(1, dtype=torch.float32, device=self.device)
            ent = (geom, m, flat, views, gm, arr, states, loss_out)
            self._cache[key] = ent
        geom, m, flat, views, gm, arr, states, _ = ent
        n = nc * sample_number ** self.dim
        if targets.dtype != torch.float32 or not targets.is_contiguous():
            targets = targets.detach().to(torch.float32).contiguous()
        if targets.numel() != n * m.cout:
            raise ValueError(f"targets must hold {n} x {m.cout} values")
        noise_bits, noise_t = 0, None
        if epoch < self.num_epochs * 0.95 and noise is not False:   # image_compression.py:248-254
            if torch.is_tensor(noise):
                noise_t = noise.detach().to(torch.float32).contiguous()
                if tuple(noise_t.shape) != (n, m.cin):
                    raise ValueError(f"noise must be [{n}, {m.cin}]")
            else:
                noise_bits = self.bits
        h = L.handle(self.device)
        st = L.stream_ptr(self.device)
        lib.nic_set_option(h, L.OPT_STEP_METRICS, 1)
        try:
            return self._launch_step(lib, h, st, geom, m, g0, g1, coord, targets, noise_t, noise_bits, epoch, n, gm, views,
                                     out, peer, parity, flat, states, arr)
        finally:
            lib.nic_set_option(h, L.OPT_STEP_METRICS, 0)

    def _ring_slot(self, epoch):
        if epoch - self._ring_base >= self.metrics_ring:       # ring full: a FRESH tensor, so handles returned earlier stay valid
            self._old_rings.append((self._ring_base, self._ring))
            self._ring = torch.zeros((self.metrics_ring, 2), dtype=torch.float32, device=self.device)
            self._ring_base = epoch
        return self._ring[epoch - self._ring_base]

    def flush_metrics(self):
        """The per-step scalars the reference logs (image_compression.py:275-279) for every step since the last flush, with
        ONE device-to-host copy: a list of (step, loss, psnr) where psnr = calculate_psnr of the 8-bit-rounded outputs and
        targets (:260-261; 10 log10(256^2 / mse8))."""
        res = []
        rings = self._old_rings + [(self._ring_base, self._ring)]
        for base, ring in rings:
            lo, hi = max(self._flushed, base), min(self.epoch, base + self.metrics_ring)
            if hi <= lo:
                continue
            vals = ring[lo - base:hi - base].cpu().tolist()
            for i, (loss, mse8) in enumerate(vals):
                res.append((lo + i, loss, float("inf") if mse8 == 0 else 10.0 * math.log10(65536.0 / mse8)))
        self._old_rings = []
        self._flushed = self.epoch
        return res

    def draw_lod(self):
        """The step's LOD with the reference's distribution (image_compression.py:221-226 + :29-34), identical on every
        rank of the process group (a shared counter-free host stream: no device work, no collective)."""
        return self._plan.next_lod()

    def step_sampled(self, datasets, crop_size=None, num_crops=None, noise=None):
        """One whole iteration of train_models' loop body: LOD draw, device-side crop sampling + target gather
        (random_crop_dataset), fused step.  `datasets`: the mip list (build_mip_pyramid).  Returns (loss, lod).
        The sampler of step i + 1 is launched on a side stream BEFORE step i is enqueued (its inputs — the image and a
        Philox counter — do not depend on the step), so it runs in the shadow of step i's small kernels instead of
        between two steps."""
        crop = (var2.CROP_SIZE if crop_size is None else crop_size)
        nc = var2.NUM_CROPS if num_crops is None else num_crops
        key = (id(datasets), crop, nc)
        if self._sample_stream is None or self._sample_key != key:
            # three preallocated (targets, coord) slots sized for LOD 0 — no allocator traffic and no stream-context
            # switches per step (the host enqueue time of a step is of the order of its 0.18 ms device time)
            self._sample_stream = self._sample_stream or torch.cuda.Stream(device=self.device)
            ci = datasets[0].shape[0]
            n0 = nc * max(1, crop) ** self.dim
            torch.cuda.current_stream(self.device).synchronize()
            self._sample_slots = [(torch.empty(n0 * ci, dtype=torch.float32, device=self.device),
                                   torch.empty((nc, self.dim), dtype=torch.int64, device=self.device),
                                   torch.cuda.Event(), torch.cuda.Event()) for _ in range(3)]
            self._sample_key, self._prefetched = key, None
            self._sample_geo = {}
        main = torch.cuda.current_stream(self.device)
        lib = L.load_library()
        h = L.handle(self.device)
        sp = C.c_void_p(self._sample_stream.cuda_stream)

        def launch(index):
            lod = self.draw_lod()
            geo = self._sample_geo.get(lod)
            if geo is None:
                ds = datasets[lod]
                if not ds.is_cuda or ds.dtype != torch.float32 or not ds.is_contiguous() or ds.dim() != self.dim + 1:
                    raise TypeError("datasets must be contiguous float32 CUDA tensors [C, S, S(, S)]")
                rc = max(1, crop // pow(2, lod))
                size = (C.c_int32 * 3)(*(list(ds.shape[1:]) + [1] * (3 - self.dim)))
                cr = (C.c_int32 * 3)(*([min(rc, ds.shape[1 + a]) for a in range(self.dim)] + [1] * (3 - self.dim)))
                geo = (ds, size, cr, nc * rc ** self.dim, ds.shape[0])
                self._sample_geo[lod] = geo
            ds, size, cr, n, ci = geo
            buf, coord, filled, consumed = self._sample_slots[index % 3]
            if index >= 3:
                self._sample_stream.wait_event(consumed)     # the step that last read this slot (index - 3) has run
            L.check(h, lib.nic_sample_crops_random(h, L.ptr(ds), self.dim, ci, C.cast(size, C.c_void_p), nc, C.cast(cr, C.c_void_p),
                                                   (self.seed + 7919 * self.rank + 1) & (2 ** 64 - 1), index, L.ptr(coord),
                                                   L.ptr(buf), sp))
            filled.record(self._sample_stream)
            return index, lod, buf[:n * ci].view(nc, -1, ci), coord, filled, consumed

        cur = self._prefetched
        if cur is None or cur[0] != self.epoch:
            cur = launch(self.epoch)
        self._prefetched = launch(self.epoch + 1)
        _, lod, targets, coord, filled, consumed = cur
        main.wait_event(filled)
        loss = self.step(coord, targets, lod, noise=noise)
        consumed.record(main)
        return loss, lod

    def _launch_step(self, lib, h, st, geom, m, g0, g1, coord, targets, noise_t, noise_bits, epoch, n, gm, views, out, peer,
                     parity, flat, states, arr):
        L.check(h, lib.nic_train_step(h, C.byref(geom), L.ptr(g0), L.ptr(g1), L.ptr(coord), C.byref(m), L.ptr(targets),
                                      L.ptr(noise_t), noise_bits, self.seed + 7919 * self.rank, epoch, n * self.world,
                                      C.byref(gm), L.ptr(None if self.frozen else views[0]),
                                      L.ptr(None if self.frozen else views[1]), L.ptr(views[8]), L.ptr(out),
                                      self.precision, st))
        if self.world > 1 and not peer:                              # the one exchange step of the path, as a collective
            torch.distributed.all_reduce(flat, group=self.pg)
        # Adam on the tensors that received a gradient this step (per-tensor step counts); the same launch turns the
        # loss sum into the mean (a fresh 1-element tensor per step, so callers may keep the handles) and re-zeroes it
        scale = self.lr_scale(epoch)
        for k, (stt, lr0) in enumerate(states):
            stt[2] += 1
            arr[k].lr = lr0 * scale
            arr[k].t = stt[2]
        loss = self._ring_slot(epoch)                                # [loss, mse of the 8-bit outputs]
        if peer:                                                     # ... or fused into the optimiser over NVLink peer memory
            x = self._exchange_desc(peer, parity)
            peer["uses"] += 1
            x.token = peer["uses"]
            L.check(h, lib.nic_adam_step_exchange(h, arr, len(states), self.betas[0], self.betas[1], self.eps, 1.0,
                                                  C.byref(x), L.ptr(views[8]), L.ptr(loss),
                                                  1.0 / float(n * self.world * m.cout), st))
        else:
            L.check(h, lib.nic_adam_step_loss(h, arr, len(states), self.betas[0], self.betas[1], self.eps, 1.0, 1,
                                              L.ptr(views[8]), L.ptr(loss), 1.0 / float(n * self.world * m.cout), st))
        loss = loss[0]
        self.epoch += 1
        return loss
