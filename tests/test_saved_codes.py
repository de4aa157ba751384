"""Decoding from the saved model: the uint8 grid codes of fp_savable (optionally bit-packed) and the decoder weights.
Without a GPU: the quantiser oracle (tests/codes_oracle.py) against float64 evaluations of the same formulas, and the
sub-byte layout in numpy.  On the GPU, at every code width: the quantiser kernels bit for bit against the oracle, packing
through the raw C ABI, decode_codes against decode of the loaded grids bit for bit on each path, the code-resident query
kernel, sample / bake from codes, the refusals, and HostDecodePipeline frame by frame against per-band decodes.

Grids are built as codes (uniform in [0, 2^b - 1] with both extreme codes in every channel), not by quantising float grids,
which would make the extreme codes rare."""
import numpy as np
import pytest
import torch

import codes_oracle as CO
import inputs as I
from helpers import T, configure, dev, lsb_stats, make_decoder

F32 = np.float32
BITS = list(range(1, 9))
PACK_BITS = [1, 2, 4, 8]
ERR_ARG, ERR_UNSUPPORTED = -1, -2


def nic():
    import neural_image_compression_v2_b200 as n
    return n


def assert_same_f32(got, want, what):
    """Bit-for-bit equality of float32 arrays; any NaN matches any NaN (payloads are not part of the contract)."""
    got, want = np.asarray(got, F32), np.asarray(want, F32)
    assert got.shape == want.shape, what
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), what
    bad = np.flatnonzero(got[~nan].view(np.uint32) != want[~nan].view(np.uint32))
    assert bad.size == 0, (what, got[~nan][bad[:8]], want[~nan][bad[:8]])


def wide_inputs(rng, bits, n=20000):
    """The special inputs plus uniform values over three times the clamp range."""
    lo = float(CO.q_min(bits))
    x = rng.uniform(3 * lo - 1, 2.0, n).astype(F32)
    return np.concatenate([CO.special_inputs(bits), x]).astype(F32)


# ------------------------------------------------------------------------------------------------ no GPU
@pytest.mark.parametrize("bits", BITS)
def test_oracle_quantisers_against_float64(bits):
    """The float32 oracle against float64: x * s and x * s + 1/2 are exact in float64 (24 + 8 significant bits), so float64
    gives the exact code; the float32 op sequence may differ only where fl(x * s) rounds onto or across a half-integer, i.e.
    where x * s + 1/2 lies within one float32 ulp of x * s of an integer.  The tie neighbours must produce such cases at the
    widths where s has more than one significant bit, or the inputs would not test the rounding."""
    rng = np.random.default_rng(700 + bits)
    x = wide_inputs(rng, bits)
    fin = np.isfinite(x) & (np.abs(x) < 1e4)
    s = 2 ** bits - 1
    xs = x[fin].astype(np.float64) * s
    exact = np.floor(xs + 0.5)
    q32 = CO._round(x[fin], bits).astype(np.float64)
    ulp = np.spacing(np.maximum(np.abs(xs), np.abs(xs + 0.5)).astype(F32)).astype(np.float64)
    near = np.abs(xs + 0.5 - np.round(xs + 0.5)) <= ulp
    differ = q32 != exact
    assert not (differ & ~near).any(), x[fin][differ & ~near][:8]
    assert (np.abs(q32 - exact) <= 1).all()
    if s & (s - 1) and bits > 1:              # s = 3, 7, ..., 255: some tie neighbour rounds onto the half-integer
        assert differ.any()
    # quantize4fp / save4fp / output_to_u8 / clamp from the float32 code, each remaining step checked in float64
    q = CO._round(x, bits).astype(np.float64)
    with np.errstate(invalid="ignore"):
        assert_same_f32(CO.quantize4fp(x, bits), (q / s).astype(F32), "quantize4fp")
        code = np.where(np.isnan(q), 0, np.clip(q + 2 ** (bits - 1) - 1, 0, 255)).astype(np.uint8)
        u8 = np.where(np.isnan(q), 0, np.clip(q, 0, s)).astype(np.uint8)
    assert np.array_equal(CO.save4fp(x, bits), code)
    assert np.array_equal(CO.output_to_u8(x, bits), u8)
    assert_same_f32(CO.quantize_to_bit(x, bits), u8.astype(F32), "quantize_to_bit")
    lo = float(CO.q_min(bits))
    assert lo == -(2 ** bits - 1) / 2 ** (bits + 1)
    assert_same_f32(CO.quantize_clamp(x, bits), np.where(np.isnan(x), lo, np.clip(x.astype(np.float64), lo, 0.5)).astype(F32),
                    "quantize_clamp")
    # load4fp of all 256 codes: (c - 2^(b-1) + 1) is an exact small integer, one correctly rounded division
    c = np.arange(256, dtype=np.uint8)
    assert_same_f32(CO.load4fp(c, bits), ((c.astype(np.float64) - 2 ** (bits - 1) + 1) / s).astype(F32), "load4fp")
    # the documented values for non-finite inputs
    nf = np.array([np.nan, np.inf, -np.inf], F32)
    assert np.isnan(CO.quantize4fp(nf, bits)[0]) and list(CO.quantize4fp(nf, bits)[1:]) == [np.inf, -np.inf]
    assert list(CO.save4fp(nf, bits)) == [0, 255, 0]
    assert list(CO.output_to_u8(nf, bits)) == [0, s, 0]
    assert list(CO.quantize_clamp(nf, bits)) == [lo, 0.5, lo]
    # in range, the saved code reloads as the quantised value
    xi = CO.in_range_inputs(rng, bits, 5000)
    assert (CO.save4fp(xi, bits) <= s).all()
    assert_same_f32(CO.load4fp(CO.save4fp(xi, bits), bits), CO.quantize4fp(xi, bits), "load4fp(save4fp(x))")


@pytest.mark.parametrize("bits", PACK_BITS)
def test_oracle_pack_layout(bits):
    """The numpy layout against a per-code loop and a hand-packed byte; unpack(pack(c)) == c & mask."""
    per, mask = 8 // bits, (1 << bits) - 1
    rng = np.random.default_rng(720 + bits)
    for n in (1, per - 1, per, per + 1, 3 * per + 2, 1000):
        c = rng.integers(0, 256, n, dtype=np.uint8)
        want = np.zeros((n * bits + 7) // 8, np.uint8)
        for i in range(n):
            want[i // per] |= (int(c[i]) & mask) << ((i % per) * bits)
        assert np.array_equal(CO.pack(c, bits), want), n
        assert np.array_equal(CO.unpack(CO.pack(c, bits), n, bits), c & mask), n
    hand = {1: ([1, 0, 1, 1, 0, 0, 0, 1, 1], [0b10001101, 0b1]), 2: ([1, 2, 3, 0, 1], [0b00111001, 0b01]),
            4: ([0x3, 0xC, 0x5], [0xC3, 0x05]), 8: ([7, 200], [7, 200])}[bits]
    assert list(CO.pack(np.array(hand[0], np.uint8), bits)) == hand[1]


@pytest.mark.parametrize("bits", BITS)
def test_random_codes_hold_both_extremes_in_every_channel(bits):
    c = CO.random_codes(np.random.default_rng(730 + bits), (12, 9, 9), bits)
    flat = c.reshape(12, -1)
    assert c.dtype == np.uint8 and int(c.max()) == 2 ** bits - 1
    assert (flat.min(1) == 0).all() and (flat.max(1) == 2 ** bits - 1).all()


# ------------------------------------------------------------------------------------------------ GPU: quantisers, packing
@pytest.mark.gpu
@pytest.mark.parametrize("bits", BITS)
def test_quantiser_kernels_bit_exact(bits):
    """quantize4fp, save4fp, load4fp (all 256 codes), output_to_u8, quantize_to_bit and quantize_clamp against the oracle, bit
    for bit, on ties and their neighbours, both clamp ends, out-of-range values, +-0, large magnitudes, +-inf and NaN."""
    m = nic().models
    rng = np.random.default_rng(740 + bits)
    x = wide_inputs(rng, bits)
    xt = T(x)
    assert_same_f32(m.quantize4fp(xt, bits).cpu().numpy(), CO.quantize4fp(x, bits), "quantize4fp")
    assert np.array_equal(m.save4fp(xt, bits).cpu().numpy(), CO.save4fp(x, bits))
    codes = np.arange(256, dtype=np.uint8)
    assert_same_f32(m.load4fp(T(codes), bits).cpu().numpy(), CO.load4fp(codes, bits), "load4fp")
    assert np.array_equal(m.output_to_u8(xt, bits).cpu().numpy(), CO.output_to_u8(x, bits))
    assert_same_f32(m.quantize_to_bit(xt, bits).cpu().numpy(), CO.quantize_to_bit(x, bits), "quantize_to_bit")
    assert_same_f32(m.quantize_clamp(xt, bits).cpu().numpy(), CO.quantize_clamp(x, bits), "quantize_clamp")
    # in range, load4fp(save4fp(x)) == quantize4fp(x) on the device as well
    xi = T(CO.in_range_inputs(rng, bits, 100000))
    assert torch.equal(m.load4fp(m.save4fp(xi, bits), bits), m.quantize4fp(xi, bits))


def _raw(name, src, dst, n, bits):
    L = nic()._lib
    h = L.handle(dev())
    return getattr(L.load_library(), name)(h, L.ptr(src), L.ptr(dst), n, bits, L.stream_ptr(dev()))


@pytest.mark.gpu
@pytest.mark.parametrize("bits", PACK_BITS)
def test_pack_codes_raw_abi_layout(bits):
    """nic_pack_codes / nic_unpack_codes: the byte layout against numpy at n in {1, per - 1, per, per + 1, 2^20 + 3}, codes
    over all 256 byte values (only the low `bits` bits are kept), no byte written past the end, unpack(pack(c)) == c & mask;
    unpack of arbitrary bytes against numpy; widths other than 1, 2, 4, 8 refused."""
    per, mask = 8 // bits, (1 << bits) - 1
    rng = np.random.default_rng(750 + bits)
    guard = 16
    for n in (1, per - 1, per, per + 1, 2 ** 20 + 3):
        c = rng.integers(0, 256, n, dtype=np.uint8)
        nbytes = (n * bits + 7) // 8
        packed = torch.full((nbytes + guard,), 0xA5, dtype=torch.uint8, device=dev())
        assert _raw("nic_pack_codes", T(c), packed, n, bits) == 0
        p = packed.cpu().numpy()
        assert np.array_equal(p[:nbytes], CO.pack(c, bits)), n
        assert (p[nbytes:] == 0xA5).all(), n
        out = torch.full((n + guard,), 0x5A, dtype=torch.uint8, device=dev())
        assert _raw("nic_unpack_codes", packed, out, n, bits) == 0
        o = out.cpu().numpy()
        assert np.array_equal(o[:n], c & mask) and (o[n:] == 0x5A).all(), n
        anyb = rng.integers(0, 256, nbytes, dtype=np.uint8)
        out = torch.empty((n,), dtype=torch.uint8, device=dev())
        assert _raw("nic_unpack_codes", T(anyb), out, n, bits) == 0
        assert np.array_equal(out.cpu().numpy(), CO.unpack(anyb, n, bits)), n
    torch.cuda.synchronize()
    one = torch.zeros(8, dtype=torch.uint8, device=dev())
    for bad in (0, 3, 5, 9):
        assert _raw("nic_pack_codes", one, one, 1, bad) == ERR_ARG
        assert _raw("nic_unpack_codes", one, one, 1, bad) == ERR_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("bits", PACK_BITS)
def test_packed_grids_reload_as_quantize4fp(bits):
    """fp_load_packed(fp_savable_packed(g)) == quantize4fp(g) for in-range grids with the ties and both clamp ends among
    their values, ragged sizes included."""
    fpd, models = nic().fp_def, nic().models
    rng = np.random.default_rng(760 + bits)
    grids = []
    for shape in ((12, 33, 33), (12, 17, 17), (3, 5, 7), (1, 1, 3), (1, 1, 1)):
        g = CO.in_range_inputs(rng, bits, int(np.prod(shape)))[-int(np.prod(shape)):]
        grids.append(T(rng.permutation(g).reshape(shape)))
    packed = fpd.fp_savable_packed(grids, bits)
    for g, r, (p, shape) in zip(grids, fpd.fp_load_packed(packed, bits), packed):
        assert shape == tuple(g.shape) and p.numel() == (g.numel() * bits + 7) // 8
        assert torch.equal(r, models.quantize4fp(g, bits))
        assert_same_f32(r.cpu().numpy(), CO.quantize4fp(g.cpu().numpy(), bits), "fp_load_packed")


# ------------------------------------------------------------------------------------------------ GPU: decode from codes
def _codes(rng, shapes, bits):
    return [T(CO.random_codes(rng, s, bits)) for s in shapes]


@pytest.mark.gpu
@pytest.mark.parametrize("bits", BITS)
def test_decode_codes_equals_decode_of_loaded_grids(bits):
    """decode_codes(codes, bits) == decode(fp_load(codes, bits)) bit for bit, f16 and bf16, uint8 and float32 out: the
    aligned 2-D fast path (whole frame), the general 2-D kernel (an unaligned block), mips at step 1 and step 2 (no
    interpolation), and dense 3-D for methods 3 and 4."""
    n = nic()
    ic, fpd = n.image_compression, n.fp_def
    rng = np.random.default_rng(800 + bits)
    size = 256
    configure(IMAGE_SIZE=size)
    codes = _codes(rng, [(12, s, s) for s in I.pyramid_sizes(size, True)], bits)
    loaded = fpd.fp_load(codes, bits)
    dec = make_decoder(I.make_mlp(73, seed=801, gain=2.0))
    table = {0: 0, 2: 0, 3: 0}                   # mip 2: step 1; mip 3: step 2, G1 interpolation off
    cases = [dict(mip=0, size=size), dict(mip=0, size=(37, 50), origin=(5, 9)), dict(mip=2, size=size >> 2),
             dict(mip=3, size=(29, 31), origin=(3, 1))]
    for prec in ("f16", "bf16"):
        for dt in (torch.uint8, torch.float32):
            for kw in cases:
                kw = dict(kw)
                mip = kw.pop("mip")
                a = ic.decode_codes(codes, dec, bits, mip, precision=prec, out_dtype=dt, level_table=table, **kw)
                b = ic.decode(loaded, dec, mip, precision=prec, out_dtype=dt, level_table=table, **kw)
                assert torch.equal(a, b), (prec, dt, mip, kw)
    for method, cin in ((3, 127), (4, 79)):
        configure(IMAGE_SIZE=32, IMAGE_DIMENSION=3, COMPRESSION_METHOD=method, CROP_MIP_LEVEL=3)
        c3 = _codes(rng, [(12, s, s, s) for s in I.pyramid_sizes(32, True)], bits)
        l3 = fpd.fp_load(c3, bits)
        d3 = make_decoder(I.make_mlp(cin, seed=802 + method, gain=2.0))
        for prec in ("f16", "bf16"):
            for dt in (torch.uint8, torch.float32):
                a = ic.decode_codes(c3, d3, bits, 0, precision=prec, out_dtype=dt, method=method, level_table={0: 0})
                b = ic.decode(l3, d3, 0, precision=prec, out_dtype=dt, method=method, level_table={0: 0})
                assert torch.equal(a, b), (method, prec, dt)
    configure()


def _lut_codes(rng, bits):
    """A 65^3 LUT as codes: 18^3 and 10^3 nodes, 12 channels."""
    return _codes(rng, [(12, 18, 18, 18), (12, 10, 10, 10)], bits)


@pytest.mark.gpu
@pytest.mark.parametrize("bits", BITS)
def test_code_resident_queries_at_every_width(bits):
    """decode_points_codes on a 65^3 LUT (f16: the code-resident kernel, load4fp folded into layer 1 with the code offset
    2^(b-1) - 1) against the fp32 decode of the loaded grids and against the same queries on the general kernel: +-1 LSB
    for >= 99.9 % of the queries, none further than 2; the corner queries included."""
    n = nic()
    ic, fpd, L = n.image_compression, n.fp_def, n._lib
    configure(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3, CROP_MIP_LEVEL=3)
    rng = np.random.default_rng(820 + bits)
    codes = _lut_codes(rng, bits)
    dec = make_decoder(I.make_mlp(127, seed=821, gain=2.0))
    table = {0: 0}
    dense = ic.decode(fpd.fp_load(codes, bits), dec, 0, size=65, precision="f32", out_dtype=torch.uint8, level_table=table)
    q = rng.integers(0, 65, (20011, 3))
    q[:3] = [[64, 64, 64], [0, 0, 64], [64, 0, 0]]
    qt = torch.tensor(q)
    pts = ic.decode_points_codes(codes, dec, qt, bits, 0, precision="f16", level_table=table).cpu().numpy()
    want = dense[q[:, 0], q[:, 1], q[:, 2]].cpu().numpy()
    within1, same, worst = lsb_stats(pts, want)
    assert within1 >= 0.999 and worst <= 2, (bits, within1, same, worst)
    L.set_option(dev(), L.OPT_DISABLE_FAST2D, 1)             # the same call on the general kernel
    try:
        gen = ic.decode_points_codes(codes, dec, qt, bits, 0, precision="f16", level_table=table).cpu().numpy()
    finally:
        L.set_option(dev(), L.OPT_DISABLE_FAST2D, 0)
    within1, same, worst = lsb_stats(pts, gen)
    assert within1 >= 0.999 and worst <= 2, (bits, within1, same, worst)
    configure()


def _query_coords(rng, q, dim):
    c = (rng.random((q, dim), dtype=F32) * F32(1.5) - F32(0.25)).astype(F32)
    c[:6] = [[0.0] * dim, [1.0] * dim, [-0.3] * dim, [1.7] * dim, [np.nan] * dim, [0.5] * dim]
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [3, 5])
def test_sample_and_bake_from_codes_at_odd_widths(bits):
    """sample_codes (a scalar LOD, a fractional scalar LOD and a per-query LOD tensor) and bake_lut_codes equal the same
    calls on the loaded grids bit for bit, f16 and bf16."""
    n = nic()
    ic, fpd = n.image_compression, n.fp_def
    rng = np.random.default_rng(840 + bits)
    for method, size, dim in ((1, 64, 2), (3, 32, 3)):
        if method == 1:
            configure(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=6)
        else:
            configure(IMAGE_SIZE=size, IMAGE_DIMENSION=3, COMPRESSION_METHOD=method, TF_NO_MIP=False, MAX_MIP_LEVEL=5)
        codes = _codes(rng, [(12,) + (s,) * dim for s in I.pyramid_sizes(size, False)], bits)
        loaded = fpd.fp_load(codes, bits)
        dec = make_decoder(I.make_mlp(73 if dim == 2 else 127, seed=841, gain=2.0))
        table = fpd.create_pyramid_mip_levels(size, size // 4)
        last = int(np.log2(size))
        c = T(_query_coords(rng, 3001, dim))
        lam = (rng.random(3001, dtype=F32) * F32(last + 2.5) - F32(1)).astype(F32)
        lam[:6] = [np.nan, -np.inf, np.inf, 0.0, 1.0, float(last)]
        for prec in ("f16", "bf16"):
            for dt in (torch.uint8, torch.float32):
                for lod, sz in ((0, size), (1.25, None), (T(lam), None)):
                    kw = dict(align_corners=True, precision=prec, out_dtype=dt, method=method, level_table=table)
                    a = ic.sample_codes(codes, dec, c, bits, lod, sz, **kw)
                    b = ic.sample(loaded, dec, c, lod, sz, **kw)
                    assert torch.equal(a, b), (method, prec, dt, lod if not torch.is_tensor(lod) else "tensor")
    for method, cin in ((3, 127), (4, 79)):
        configure(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=method, CROP_MIP_LEVEL=3)
        codes = _lut_codes(rng, bits)
        dec = make_decoder(I.make_mlp(cin, seed=842, gain=2.0))
        for prec in ("f16", "bf16"):
            a = ic.bake_lut_codes(codes, dec, bits, 0, size=65, precision=prec, level_table={0: 0})
            b = ic.bake_lut(fpd.fp_load(codes, bits), dec, 0, size=65, precision=prec, level_table={0: 0})
            assert a.extent == b.extent == (65, 65, 65) and torch.equal(a.table, b.table), (method, prec)
    configure()


@pytest.mark.gpu
def test_decode_codes_refusals():
    """A float32-precision decode or sample from codes is NIC_ERR_UNSUPPORTED; code widths 0 and 9 are NIC_ERR_ARG.
    sample_codes at an integer lod, at a fractional lod (two passes) and with a per-query lod tensor."""
    n = nic()
    ic, fpd = n.image_compression, n.fp_def
    configure(IMAGE_SIZE=64, TF_NO_MIP=False, MAX_MIP_LEVEL=6)
    codes = _codes(np.random.default_rng(860), [(12, s, s) for s in I.pyramid_sizes(64, False)], 8)
    dec = make_decoder(I.make_mlp(73, seed=861))
    table = fpd.create_pyramid_mip_levels(64, 16)
    c = T(_query_coords(np.random.default_rng(862), 64, 2))
    lam = T(np.linspace(-1, 7, 64, dtype=F32))
    calls = [lambda **kw: ic.decode_codes(codes, dec, level_table=table, **kw),
             lambda **kw: ic.decode_points_codes(codes, dec, torch.tensor([[3, 5]]), level_table=table, **kw)]
    calls += [lambda lod=lod, **kw: ic.sample_codes(codes, dec, c, lod=lod, level_table=table, **kw) for lod in (0, 1.25, lam)]
    for call in calls:
        with pytest.raises(n.NicError) as e:
            call(num_bits=8, precision="f32")
        assert e.value.status == ERR_UNSUPPORTED
        for bad in (0, 9):
            with pytest.raises(n.NicError) as e:
                call(num_bits=bad, precision="f16")
            assert e.value.status == ERR_ARG, bad
    configure()


# ------------------------------------------------------------------------------------------------ GPU: HostDecodePipeline
GRID_SIZE = 512          # every pipeline model is a 2-D no-mip model of a 512^2 image (129^2 and 65^2 nodes)


def _pipeline_models(rng, bits, cout, count=3):
    """`count` models, each with its own codes and its own decoder weights (numpy)."""
    shapes = [(12, s, s) for s in I.pyramid_sizes(GRID_SIZE, True)]
    return [([CO.random_codes(rng, s, bits) for s in shapes], I.make_mlp(73, cout=cout, seed=870 + i, gain=2.0))
            for i in range(count)]


def _host(a, pinned):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.pin_memory() if pinned else t


def _references(ic, par, fpd, model, size, bands, bits, mip, prec):
    """(per-band reference frame, fp32 frame) of one model: each band decoded on its own from codes with the band
    boundaries of parallel.shard_rows, and the fp32 decode of the loaded grids."""
    codes, params = model
    dcodes, dec = [T(c) for c in codes], make_decoder(params)
    ref = torch.empty((size, size, len(params[5])), dtype=torch.uint8, device=dev())
    rows = 0
    for b in range(bands):
        r0, n = par.shard_rows(size, b, bands)
        assert r0 == rows or n == 0
        rows += n
        if n:
            ic.decode_codes(dcodes, dec, bits, mip, size=(n, size), origin=(r0, 0), precision=prec, out=ref[r0:r0 + n])
    assert rows == size
    f32 = ic.decode(fpd.fp_load(dcodes, bits), dec, mip, size=size, precision="f32", out_dtype=torch.uint8)
    return ref.cpu().numpy(), f32.cpu().numpy()


PIPELINE_CASES = {
    # id: (frame size, bands, bits, cout, mip, precision, wait, pinned, side stream, frames)
    "models_cycle_wait": (512, 4, 8, 3, 0, "f16", True, True, False, 6),
    "models_cycle_nowait": (512, 4, 8, 3, 0, "f16", False, True, False, 6),
    "bands1": (512, 1, 8, 3, 0, "f16", False, True, False, 3),
    "bands3": (512, 3, 8, 3, 0, "f16", True, True, False, 3),
    "bands7": (512, 7, 8, 3, 0, "f16", False, True, False, 3),
    "general_kernel_500": (500, 3, 8, 3, 0, "f16", False, True, False, 3),
    "empty_bands_40": (40, 7, 8, 3, 0, "f16", True, True, False, 3),
    "bits4_cout5_bf16": (512, 4, 4, 5, 0, "bf16", False, True, False, 3),
    "bits2": (512, 4, 2, 3, 0, "f16", True, True, False, 3),
    "mip1": (256, 4, 8, 3, 1, "f16", False, True, False, 3),
    "pageable_nowait": (512, 4, 8, 3, 0, "f16", False, False, False, 4),
    "pageable_wait": (512, 3, 8, 3, 0, "f16", True, False, False, 3),
    "side_stream_wait": (512, 4, 8, 3, 0, "f16", True, True, True, 4),
    "side_stream_nowait": (512, 4, 8, 3, 0, "f16", False, True, True, 4),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PIPELINE_CASES))
def test_host_decode_pipeline(case):
    """HostDecodePipeline frame by frame, cycling through 3 models (own codes, own decoder weights), so both device buffer
    sets are refilled with other models: every band of each host frame equals that model's own per-band decode_codes bit
    for bit, and the frame is within +-1 LSB (>= 99.9 %) of the fp32 decode of the loaded grids.  The host buffers follow
    the documented rule: with wait=True the frame is read after synchronising the caller's stream; with wait=False each
    frame has its own host_out, read after finish(), and the inputs come from one staging set that is overwritten for the
    next frame only after `uploaded.synchronize()`.  Afterwards a plain decode_codes rebuilds its tables (the pipeline
    leaves NIC_OPT_REUSE_PREPARED off): decoding one model, overwriting its tensors in place with another and decoding
    again gives the other model."""
    size, bands, bits, cout, mip, prec, wait, pinned, side, frames = PIPELINE_CASES[case]
    n = nic()
    ic, par, fpd = n.image_compression, n.parallel, n.fp_def
    configure(IMAGE_SIZE=GRID_SIZE)
    rng = np.random.default_rng(880 + list(PIPELINE_CASES).index(case))
    models = _pipeline_models(rng, bits, cout)
    refs = [_references(ic, par, fpd, m, size, bands, bits, mip, prec) for m in models]
    if case == "empty_bands_40":
        assert any(par.shard_rows(size, b, bands)[1] == 0 for b in range(bands))
    host = [([_host(c, pinned) for c in codes], [_host(p, pinned) for p in params]) for codes, params in models]
    order = [i % len(models) for i in range(frames)]
    torch.cuda.synchronize()

    pipe = ic.HostDecodePipeline(size, dev(), precision=prec, bands=bands, bits=bits)
    stream = torch.cuda.Stream(device=dev()) if side else torch.cuda.current_stream(dev())
    got = []
    with torch.cuda.stream(stream):
        if wait:
            host_out = _host(np.zeros((size, size, cout), np.uint8), pinned)
            for m in order:
                pipe.decode_frame(host[m][0], host[m][1], host_out, mip_level=mip, wait=True)
                stream.synchronize()
                got.append(host_out.numpy().copy())
        else:
            stage_codes = [_host(np.zeros_like(c), pinned) for c in models[0][0]]
            stage_params = [_host(np.zeros_like(p), pinned) for p in models[0][1]]
            outs = [_host(np.zeros((size, size, cout), np.uint8), pinned) for _ in order]
            for i, m in enumerate(order):
                if pipe.uploaded is not None:
                    pipe.uploaded.synchronize()          # the previous frame's upload has read the staging set
                for d, s in zip(stage_codes + stage_params, host[m][0] + host[m][1]):
                    d.copy_(s)
                pipe.decode_frame(stage_codes, stage_params, outs[i], mip_level=mip, wait=False)
            pipe.finish()
            stream.synchronize()
            got = [o.numpy() for o in outs]
    torch.cuda.synchronize()
    for i, m in enumerate(order):
        ref, f32 = refs[m]
        for b in range(bands):
            r0, rows = par.shard_rows(size, b, bands)
            assert np.array_equal(got[i][r0:r0 + rows], ref[r0:r0 + rows]), (case, i, m, b)
        within1, same, worst = lsb_stats(got[i], f32)
        assert within1 >= 0.999, (case, i, within1, same, worst)

    # after the pipeline: a plain decode from codes does not reuse tables across a change of the model's contents
    (ca, pa), (cb, pb) = models[0], models[1]
    dcodes, dec = [T(c) for c in ca], make_decoder(pa)
    ic.decode_codes(dcodes, dec, bits, mip, size=size, precision=prec)
    for d, c in zip(dcodes, cb):
        d.copy_(T(c))
    with torch.no_grad():
        for p, v in zip(dec.parameters_list(), pb):
            p.copy_(T(v))
    again = ic.decode_codes(dcodes, dec, bits, mip, size=size, precision=prec).cpu().numpy()
    assert np.array_equal(again, ic.decode_codes([T(c) for c in cb], make_decoder(pb), bits, mip, size=size,
                                                 precision=prec).cpu().numpy())
    configure()


@pytest.mark.gpu
def test_host_decode_pipeline_rebuilds_tables_for_every_frame():
    """Band 0 of each frame rebuilds the prepared tables even when the handle's tables were last built from the very device
    buffers the frame refills, with the model they held before (what a caller's decode of those buffers leaves behind, or
    a new pipeline whose buffers land on the addresses of a freed one): the frame is the new model's."""
    n = nic()
    ic, par, fpd = n.image_compression, n.parallel, n.fp_def
    size, bands, bits = 512, 4, 8
    configure(IMAGE_SIZE=GRID_SIZE)
    models = _pipeline_models(np.random.default_rng(890), bits, 3)
    refs = [_references(ic, par, fpd, m, size, bands, bits, 0, "f16")[0] for m in models]
    host = [([_host(c, True) for c in codes], [_host(p, True) for p in params]) for codes, params in models]
    host_out = _host(np.zeros((size, size, 3), np.uint8), True)
    pipe = ic.HostDecodePipeline(size, dev(), precision="f16", bands=bands, bits=bits)
    for i in range(2):                                           # frames 0 and 1: device buffer sets 0 and 1
        pipe.decode_frame(host[i][0], host[i][1], host_out, wait=True)
        torch.cuda.synchronize()
        assert np.array_equal(host_out.numpy(), refs[i]), i
    r0, rows = par.shard_rows(size, 0, bands)
    ic.decode_codes(pipe.dcodes[0], pipe.decoders[0], bits, 0, size=(rows, size), origin=(r0, 0), precision="f16")
    torch.cuda.synchronize()                                     # the handle's tables now describe buffer set 0 (model 0)
    pipe.decode_frame(host[2][0], host[2][1], host_out, wait=True)   # frame 2 refills buffer set 0 with model 2
    torch.cuda.synchronize()
    assert np.array_equal(host_out.numpy(), refs[2])
    configure()
