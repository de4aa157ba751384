"""Which calls share the prepared tensor-core tables (NIC_OPT_REUSE_PREPARED): the 16-bit shadow grids, the G1 rows and the
packed weight images built by one call are reused by the next only when they describe the same inputs for the same kernel.
Each case runs two calls with reuse on and checks the second call's launch count (exactly one kernel when it reuses the
tables, more when it rebuilds them) and that it returns the same bytes as the same call with reuse off."""
import numpy as np
import pytest
import torch

import inputs as I
from helpers import T, configure, dev, make_decoder


def nic():
    import neural_image_compression_v2_b200 as n
    return n


def coords(q, dim, seed):
    rng = np.random.default_rng(seed)
    return T((rng.random((q, dim), dtype=np.float32) * np.float32(1.5) - np.float32(0.25)).astype(np.float32))


def model_2d(size=256, seed=700):
    configure(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=8)
    fp = [T(a) for a in I.make_grids(size, 2, seed=seed, quantized=True)]
    return fp, make_decoder(I.make_mlp(73, seed=seed + 1, gain=2.0))


def model_3d(seed=710):
    """A method-3 model of a 64^3 volume whose grids hold one node more than mip 0 needs, so a 65^3 block fits."""
    configure(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3)
    fp = [T(a) for a in I.make_grids(64, 3, seed=seed, no_mip=True, quantized=True)]
    fp = [T(np.pad(g.cpu().numpy(), ((0, 0), (0, 1), (0, 1), (0, 1)), mode="edge")) for g in fp]
    return fp, make_decoder(I.make_mlp(127, seed=seed + 1, gain=2.0)), {0: 0}


def second_call(first, second):
    """Runs first() then second() on one handle with reuse on; returns (second's output, second's launches) and checks that
    the output equals second() with reuse off."""
    n = nic()
    L = n._lib
    L.set_option(dev(), L.OPT_REUSE_PREPARED, 1)
    try:
        first()
        torch.cuda.synchronize()
        before = n.launch_count(dev())
        got = second()
        launches = n.launch_count(dev()) - before
    finally:
        L.set_option(dev(), L.OPT_REUSE_PREPARED, 0)
    want = second()
    assert torch.equal(got, want)
    return got, launches


@pytest.mark.gpu
def test_chain_sample_then_scalar_sample_rebuilds():
    """The chain's W1 image carries the mip column; a scalar sample of the same grids must not use it."""
    ic = nic().image_compression
    fp, dec = model_2d()
    c = coords(4096, 2, 720)
    lam = T(np.random.default_rng(721).random(4096, dtype=np.float32) * np.float32(3))
    _, launches = second_call(lambda: ic.sample(fp, dec, c, lam, precision="f16"),
                              lambda: ic.sample(fp, dec, c, 0, precision="f16", out_dtype=torch.uint8))
    assert launches > 1
    configure()


@pytest.mark.gpu
def test_scalar_sample_then_chain_sample_rebuilds():
    ic = nic().image_compression
    fp, dec = model_2d()
    c = coords(4096, 2, 730)
    lam = T(np.random.default_rng(731).random(4096, dtype=np.float32) * np.float32(3))
    _, launches = second_call(lambda: ic.sample(fp, dec, c, 0, precision="f16"),
                              lambda: ic.sample(fp, dec, c, lam, precision="f16", out_dtype=torch.uint8))
    assert launches > 1
    configure()


@pytest.mark.gpu
def test_code_resident_queries_then_general_decode_codes_rebuilds():
    """decode_points_codes on a 65^3 LUT runs on the code-resident kernel (its own weight image, no shadows); decode_codes of
    the whole mip from the same codes runs on the general kernel and must build its own tables."""
    n = nic()
    ic, fpd = n.image_compression, n.fp_def
    fp, dec, table = model_3d()
    codes = fpd.fp_savable(fp, 8)
    q = torch.tensor(np.random.default_rng(740).integers(0, 65, (5000, 3)))
    _, launches = second_call(lambda: ic.decode_points_codes(codes, dec, q, 8, 0, precision="f16", level_table=table),
                              lambda: ic.decode_codes(codes, dec, 8, 0, size=65, precision="f16", level_table=table))
    assert launches > 1
    configure()


@pytest.mark.gpu
def test_3d_decode_then_sample_reuses():
    """A 3-D decode of mip 0 and a sample at lod 0 of the same model build the same general-kernel tables."""
    ic = nic().image_compression
    fp, dec, table = model_3d()
    c = coords(4096, 3, 750)
    _, launches = second_call(lambda: ic.decode(fp, dec, 0, precision="f16", level_table=table),
                              lambda: ic.sample(fp, dec, c, 0, precision="f16", out_dtype=torch.uint8, level_table=table))
    assert launches == 1
    configure()


@pytest.mark.gpu
def test_fast_2d_decode_then_sample_rebuilds():
    """A full-resolution 2-D decode runs on the fast 2-D kernel (G1 rows, its own weight image); a sample needs the general
    kernel's tables."""
    ic = nic().image_compression
    fp, dec = model_2d()
    c = coords(4096, 2, 760)
    _, launches = second_call(lambda: ic.decode(fp, dec, 0, precision="f16"),
                              lambda: ic.sample(fp, dec, c, 0, precision="f16", out_dtype=torch.uint8))
    assert launches > 1
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("raw", [False, True])
def test_training_step_invalidates_the_tables(raw):
    """A training step on the handle's device overwrites the scratch the tables live in and changes the grids in place: the
    session's next decode rebuilds and equals a fresh decode of the trained model."""
    n = nic()
    ic, L = n.image_compression, n._lib
    size = 256
    fp, dec = model_2d(size, seed=770)
    ses = ic.DecodeSession(fp, dec, precision="f16")
    ses.decode(0)
    before = n.launch_count(dev())
    ses.decode(0)
    assert n.launch_count(dev()) - before == 1
    coord = torch.zeros((1, 2), dtype=torch.int64, device=dev())
    targets = T(np.random.default_rng(771).random((size * size, 3), dtype=np.float32))
    if raw:
        import ctypes as C
        h = L.handle(dev())
        geom = L.make_geom(L.METHOD_2D, fp[0], fp[1], size, 1, -2, 0, 6, L.PE_TRIANGULAR)
        m = L.make_mlp([p.detach().contiguous() for p in dec.parameters_list()])
        gm = L.make_mlp_grad([torch.zeros_like(p) for p in dec.parameters_list()])
        dg = [torch.zeros_like(fp[0]), torch.zeros_like(fp[1])]
        loss = torch.zeros(4, dtype=torch.float32, device=dev())
        L.check(h, L.load_library().nic_train_step(h, C.byref(geom), L.ptr(fp[0]), L.ptr(fp[1]), L.ptr(coord), C.byref(m),
                                                   L.ptr(targets), None, 0, 0, 0, 0, C.byref(gm), L.ptr(dg[0]),
                                                   L.ptr(dg[1]), L.ptr(loss), None, L.PREC_F16, L.stream_ptr(dev())))
        with torch.no_grad():
            fp[0].sub_(dg[0].sign() * (1.0 / 255))          # changes the grids where the tables were built from
    else:
        tr = ic.FusedTrainer(fp, dec, num_epochs=100, fp_bits=8, precision="f16")
        tr.step(coord, targets, 0, noise=False)
    torch.cuda.synchronize()
    before = n.launch_count(dev())
    got = ses.decode(0)
    assert n.launch_count(dev()) - before > 1
    assert torch.equal(got, ic.decode(fp, dec, 0, precision="f16", out_dtype=torch.uint8))
    configure()
