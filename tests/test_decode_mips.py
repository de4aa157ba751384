"""The whole mip chain in one call (nic_decode_mips / nic_decode_mips_codes, image_compression.decode_mips /
decode_mips_codes): host checks and the chain the binding builds; on the GPU the fp32 arm against per-mip decode, the
tensor-core arm against decode (mip 0) and per-query-LOD sampling at texel centres (mips >= 1), decode from codes, the
config-2 chain and its launch count, table reuse, `out=` and the C ABI's error codes."""
import ctypes
import math

import numpy as np
import pytest
import torch

import inputs as I
from helpers import T, configure, dev, lsb_stats, make_decoder, psnr256

F32 = np.float32


def nic():
    import neural_image_compression_v2_b200 as n
    return n


def cpu_model():
    """A 64^2 2-D model on the host (mips 0 .. 6) with its decoder: enough for the checks that run before any launch."""
    ic = nic().image_compression
    configure(IMAGE_SIZE=64, TF_NO_MIP=False, MAX_MIP_LEVEL=6)
    fp = [torch.zeros((12, s, s)) for s in I.pyramid_sizes(64, False)]
    return ic, fp, ic.ColorDecoder(in_channels=73, hidden=64, out_channels=3), ic.feature_pyramid_mip_levels()


# ------------------------------------------------------------------------------------------------ no GPU
def test_host_checks_raise_before_any_launch():
    n = nic()
    ic, fp, dec, table = cpu_model()
    total = sum((64 >> i) ** 2 for i in range(7))
    for bad in (torch.empty((total + 1, 3)), torch.empty((total, 3), dtype=torch.float64), torch.empty((3, total)).T,
                torch.empty((total, 4))):
        with pytest.raises(ValueError):
            ic.decode_mips(fp, dec, precision="f16", out=bad, level_table=table)
    with pytest.raises(ValueError):                       # uint8 output asked for, float32 buffer given
        ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8, out=torch.empty((total, 3)), level_table=table)
    with pytest.raises(TypeError):
        ic.decode_mips(fp, dec, out_dtype=torch.float16, level_table=table)
    with pytest.raises(TypeError):                        # codes must be uint8
        ic.decode_mips_codes(fp, dec, 8, level_table=table)
    configure(IMAGE_SIZE=1 << 17, TF_NO_MIP=False, MAX_MIP_LEVEL=16)
    long_table = {i: 0 for i in range(17)}
    with pytest.raises(ValueError, match="at most 16 mips"):
        ic.decode_mips(fp, dec, level_table=long_table)
    configure(IMAGE_SIZE=64, TF_NO_MIP=False, MAX_MIP_LEVEL=6)
    with pytest.raises(n.NicError):                       # everything checked: host tensors have no fallback
        ic.decode_mips(fp, dec, precision="f16", out=torch.empty((total, 3)), level_table=table)
    configure()


def test_chain_of_whole_mip_blocks():
    L = nic()._lib
    ic, fp, dec, table = cpu_model()
    chain, grids = ic._mip_chain(fp, None, "clamp", False, L.METHOD_2D, table)
    assert chain.num_mips == 7 and len(grids) == 14
    for i in range(7):
        g = chain.geom[i]
        assert g.num_blocks == 1 and g.mip_level == i
        assert list(g.block) == list(chain.extent[i]) == [64 >> i, 64 >> i, 1]
        assert list(g.origin0) == [0, 0, 0]
        assert g.step_log2 == i - 2 * (table[i] + 1)
    configure()


# ------------------------------------------------------------------------------------------------ GPU
_MODELS = {}


def model(kind):
    """(grids, params, table, method, size, last) of a test model with mips.  2-D 64^2: mips 0 .. 6 (mip 3 at step 2 without
    G1 interpolation, mip 6 one texel); 2-D 96^2: extents 96, 48, .., 3, 1 (not powers of two); 3-D 32^3: mips 0 .. 5."""
    if kind not in _MODELS:
        from neural_image_compression_v2_b200.fp_def import create_pyramid_mip_levels
        method, size, seed = {"2d": (1, 64, 720), "2d_96": (1, 96, 730), "3d_m3": (3, 32, 740), "3d_m4": (4, 32, 750)}[kind]
        dim = 2 if method == 1 else 3
        grids = I.make_grids(size, dim, seed=seed, quantized=True)
        params = I.make_mlp({1: 73, 3: 127, 4: 79}[method], seed=seed + 1, gain=2.0)
        last = int(math.log2(size)) if size & (size - 1) == 0 else 6
        _MODELS[kind] = (grids, params, create_pyramid_mip_levels(size, size // 4), method, size, last)
    return _MODELS[kind]


def setup(kind):
    grids, params, table, method, size, last = model(kind)
    dim = 2 if method == 1 else 3
    configure(IMAGE_SIZE=size, IMAGE_DIMENSION=dim, COMPRESSION_METHOD=method, TF_NO_MIP=False, MAX_MIP_LEVEL=last)
    return [T(g) for g in grids], make_decoder(params), table, method, size, last


def centres(s, dim):
    """Texel centres (idx + .5) / S of an S^dim mip in decode's texel order (x slowest)."""
    axis = (np.arange(s, dtype=F32) + F32(0.5)) / F32(s)
    mesh = np.meshgrid(*[axis] * dim, indexing="ij")
    return np.stack([m.reshape(-1) for m in mesh], 1).astype(F32)


def smooth_target(s, dim):
    """A smooth 8-bit signal over an S^dim mip (only its distance to the two arms matters)."""
    c = centres(s, dim).astype(np.float64)
    v = 0.5 + 0.4 * np.sin(5 * c[:, :1]) * np.cos(3 * c[:, 1:2])
    return np.floor(np.repeat(v, 3, 1) * 255 + 0.5)


KINDS = ["2d", "2d_96", "3d_m3", "3d_m4"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_f32_chain_equals_per_mip_decode(kind):
    ic = nic().image_compression
    fp, dec, table, method, size, last = setup(kind)
    for dt in (torch.float32, torch.uint8):
        mips = ic.decode_mips(fp, dec, precision="f32", out_dtype=dt, method=method, level_table=table)
        assert len(mips) == last + 1
        for i, got in enumerate(mips):
            want = ic.decode(fp, dec, i, precision="f32", out_dtype=dt, method=method, level_table=table)
            assert tuple(got.shape) == tuple(want.shape) and torch.equal(got, want), (kind, dt, i)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16"])
@pytest.mark.parametrize("kind", KINDS)
def test_tensor_core_chain(precision, kind):
    """Mip 0 is decode's own result; every mip >= 1 of a power-of-two chain is sample(lod = i) at its texel centres bit for
    bit; every mip is within +-1 LSB of the fp32 arm on >= 99.9 % of its texels, and the PSNR of the chain and of every mip
    of >= 256 texels is within 0.05 dB of the fp32 arm's (the PSNR of a few texels is no image statistic: one 1-LSB step of
    one channel of the 1-texel mip moves its PSNR by 0.09 dB)."""
    ic = nic().image_compression
    fp, dec, table, method, size, last = setup(kind)
    dim = 2 if method == 1 else 3
    kw = dict(method=method, level_table=table)
    ref = ic.decode_mips(fp, dec, precision="f32", out_dtype=torch.uint8, **kw)
    for dt in (torch.float32, torch.uint8):
        mips = ic.decode_mips(fp, dec, precision=precision, out_dtype=dt, **kw)
        assert torch.equal(mips[0], ic.decode(fp, dec, 0, precision=precision, out_dtype=dt, **kw)), dt
        if size & (size - 1) == 0:
            for i in range(1, last + 1):
                s = size >> i
                c = T(centres(s, dim))
                want = ic.sample(fp, dec, c, T(np.full(s ** dim, i, F32)), precision=precision, out_dtype=dt, **kw)
                assert torch.equal(mips[i].reshape(-1, 3), want), (dt, i)
        if dt == torch.uint8:
            chain_got, chain_ref, chain_target = [], [], []
            for i, (got, r) in enumerate(zip(mips, ref)):
                got, r = got.cpu().numpy().reshape(-1, 3), r.cpu().numpy().reshape(-1, 3)
                within1, same, worst = lsb_stats(got, r)
                assert within1 >= 0.999, (i, within1, same, worst)
                target = smooth_target(size >> i, dim)
                if len(target) >= 256:
                    assert abs(psnr256(got, target) - psnr256(r, target)) <= 0.05, i
                chain_got.append(got)
                chain_ref.append(r)
                chain_target.append(target)
            got, r, target = (np.concatenate(x) for x in (chain_got, chain_ref, chain_target))
            assert abs(psnr256(got, target) - psnr256(r, target)) <= 0.05
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 4, 2])
def test_chain_from_codes_equals_chain_of_loaded_grids(bits):
    n = nic()
    ic, fp_def = n.image_compression, n.fp_def
    for kind, precision in (("2d", "f16"), ("3d_m3", "bf16"), ("3d_m4", "f16")):
        fp, dec, table, method, size, last = setup(kind)
        codes = fp_def.fp_savable(fp, bits)
        loaded = fp_def.fp_load(codes, bits)
        for dt in (torch.uint8, torch.float32):
            a = ic.decode_mips_codes(codes, dec, bits, precision=precision, out_dtype=dt, method=method, level_table=table)
            b = ic.decode_mips(loaded, dec, precision=precision, out_dtype=dt, method=method, level_table=table)
            assert all(torch.equal(x, y) for x, y in zip(a, b)), (kind, dt)
    configure()


def config2_model():
    """BASELINE config 2's shape with a mip pyramid: a 4096^2 RGB model, C = 12, every pyramid level."""
    size = 4096
    gen = torch.Generator(device=dev()).manual_seed(760)
    lo, hi = I.q_range(8)
    fp = [(torch.floor((torch.rand((12, s, s), generator=gen, device=dev()) * (hi - lo) + lo) * 255 + 0.5) / 255).contiguous()
          for s in I.pyramid_sizes(size, False)]
    return fp, make_decoder(I.make_mlp(73, seed=761, gain=2.0))


@pytest.mark.gpu
def test_config2_chain_and_its_launches():
    """4096^2, mips 0 .. 12, f16, uint8: mip 0 is decode's, mips >= 1 within +-1 LSB of per-mip decode, and a call launches
    the tables' builders plus exactly two decode kernels, whatever the number of mips."""
    n = nic()
    ic = n.image_compression
    fp, dec = config2_model()
    for last in (6, 12):
        configure(IMAGE_SIZE=4096, TF_NO_MIP=False, MAX_MIP_LEVEL=last)
        table = ic.feature_pyramid_mip_levels()
        before = n.launch_count(dev())
        mips = ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8)
        launches = n.launch_count(dev()) - before
        # mip 0 on the fast 2-D path: its G0 shadow (launch_relayout), g1_rows_kernel and pack_fast_kernel; the chain pass:
        # two shadows (build_shadows) per distinct pyramid level of mips 1 .. L, pack_weights_kernel, pack_lod_columns_kernel;
        # and the two decode kernels
        levels = len({table[i] for i in range(1, last + 1)})
        assert launches == 3 + 2 * levels + 2 + 2, (last, launches)
        assert len(mips) == last + 1
        for i, got in enumerate(mips):
            want = ic.decode(fp, dec, i, precision="f16", out_dtype=torch.uint8)
            if i == 0:
                assert torch.equal(got, want)
            else:
                assert int((got.to(torch.int16) - want.to(torch.int16)).abs().max()) <= 1, i
    configure()


@pytest.mark.gpu
def test_reuse_and_an_interleaved_lod_sample():
    n = nic()
    ic, L = n.image_compression, n._lib
    fp, dec, table, method, size, last = setup("2d")
    kw = dict(method=method, level_table=table)
    rng = np.random.default_rng(770)
    c = T(rng.random((4096, 2), dtype=F32))
    lam = T((rng.random(4096, dtype=F32) * F32(last + 1)).astype(F32))
    want = torch.cat([m.reshape(-1, 3) for m in ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8, **kw)])
    want_s = ic.sample(fp, dec, c, lam, precision="f16", out_dtype=torch.uint8, **kw)
    L.set_option(dev(), L.OPT_REUSE_PREPARED, 1)
    try:
        runs = []
        for _ in range(2):
            runs.append(ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8, **kw))
            got_s = ic.sample(fp, dec, c, lam, precision="f16", out_dtype=torch.uint8, **kw)
            assert torch.equal(got_s, want_s)
        runs.append(ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8, **kw))
    finally:
        L.set_option(dev(), L.OPT_REUSE_PREPARED, 0)
    for r in runs:
        assert torch.equal(torch.cat([m.reshape(-1, 3) for m in r]), want)
    configure()


@pytest.mark.gpu
def test_out_buffer_is_the_documented_layout():
    ic = nic().image_compression
    fp, dec, table, method, size, last = setup("3d_m3")
    kw = dict(method=method, level_table=table)
    total = sum((size >> i) ** 3 for i in range(last + 1))
    out = torch.full((total, 3), 7, dtype=torch.uint8, device=dev())
    mips = ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8, out=out, **kw)
    row = 0
    for i, m in enumerate(mips):
        s = size >> i
        assert tuple(m.shape) == (s, s, s, 3)
        assert m.data_ptr() == out.data_ptr() + row * 3 and m.is_contiguous()
        assert torch.equal(m, out[row:row + s ** 3].view(s, s, s, 3))
        row += s ** 3
    assert row == total
    fresh = ic.decode_mips(fp, dec, precision="f16", out_dtype=torch.uint8, **kw)
    assert all(torch.equal(a, b) for a, b in zip(mips, fresh))
    configure()


@pytest.mark.gpu
def test_c_abi_error_codes():
    n = nic()
    ic, fp_def, L = n.image_compression, n.fp_def, n._lib
    fp, dec, table, method, size, last = setup("2d")
    lib, h, st = L.load_library(), L.handle(dev()), L.stream_ptr(dev())
    m = L.make_mlp([p.detach().contiguous() for p in dec.parameters_list()])
    total = sum((size >> i) ** 2 for i in range(last + 1))
    out = torch.empty((total, 3), device=dev())
    codes = fp_def.fp_savable(fp, 8)

    def chain(grids=fp):
        return ic._mip_chain(grids, None, "clamp", False, method, table)[0]

    def call(c, prec=L.PREC_F16, dst=out):
        return lib.nic_decode_mips(h, ctypes.byref(c), ctypes.byref(m), L.ptr(dst), L.DT_F32, prec, st)

    def call_codes(c, bits, prec=L.PREC_F16):
        return lib.nic_decode_mips_codes(h, ctypes.byref(c), bits, ctypes.byref(m), L.ptr(out), L.DT_F32, prec, st)

    assert call(chain()) == 0 and call(chain(), L.PREC_F32) == 0 and call_codes(chain(codes), 8) == 0
    for bits in (0, 9):
        assert call_codes(chain(codes), bits) == -1, bits
    assert call_codes(chain(codes), 8, L.PREC_F32) == L.ERR_UNSUPPORTED
    for num in (0, 17):
        c = chain()
        c.num_mips = num
        assert call(c) == -1, num
    c = chain()
    c.geom[2].mip_level = 3
    assert call(c) == -1
    c = chain()
    c.geom[1].block[0] = 31                                # extent 32
    assert call(c) == -1
    c = chain()
    c.geom[2].channels = 11
    assert call(c) == -1
    c = chain()
    c.geom[3].method = L.METHOD_3D
    assert call(c) == -1
    assert call(chain(), dst=None) == -1
    c = chain()
    c.extent[0][0] = c.geom[0].block[0] = 65               # texel 64 at step 1/4 reaches node 17 of 17
    assert call(c) == -4
    c = chain()
    c.extent[1][0] = c.geom[1].block[0] = 0
    assert call(c) == -1
    torch.cuda.synchronize()
    configure()
