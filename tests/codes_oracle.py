"""numpy oracle of the quantisers and of the sub-byte code layout (nic_quantize4fp, nic_quantize_pack, nic_unpack,
nic_output_to_u8, nic_clamp, nic_pack_codes / nic_unpack_codes; include/nic.h), float32 step by step in the kernels'
order, so that it reproduces them bit for bit at every code width b = 1..8.  With s = 2^b - 1 and off = 2^(b-1):

  round(x)        = floor(fl(fl(x * s) + 0.5))          (separate fp32 multiply and add, as models.py)
  quantize4fp(x)  = fl(round(x) / s)
  save4fp(x)      = uint8(fminf(fmaxf(fl(fl(round(x) + off) - 1), 0), 255))
  load4fp(c)      = fl(fl(fl(c - off) + 1) / s)
  output_to_u8(x) = uint8(fminf(fmaxf(round(x), 0), s))
  quantize_clamp  = fminf(fmaxf(x, q_min), 0.5),         q_min = -(2^b - 1) / 2^(b+1)

What the op sequences give for non-finite inputs (fmaxf / fminf return the other operand when one is NaN):
  * quantize4fp: NaN -> NaN, +-inf -> +-inf.
  * save4fp: NaN -> code 0, +inf -> 255, -inf -> 0.  torch's reference (`(floor(..) + off - 1).to(uint8)`) converts a
    NaN, an infinity or any value outside [0, 255] with an undefined float-to-uint8 cast; the kernel saturates instead.
    Inside [0, 255] the two agree, including codes above 2^b - 1 from grid values above 1/2 (they are not clamped to b bits).
  * output_to_u8 / quantize_to_bit: NaN -> 0, +inf -> s, -inf -> 0.  The reference's quantize_to_bit returns the
    unclamped float fl(fl(round(x) / s) * s); the product clamps to [0, s] first, as the `astype(uint8)` at its call site
    needs, so the two differ outside [0, 1].
  * quantize_clamp: NaN -> q_min (fmaxf(NaN, q_min) = q_min); torch.clamp keeps the NaN.
"""
import numpy as np

F32 = np.float32


def scale(bits):
    return F32(2 ** bits - 1)


def q_min(bits):
    return F32(-(2 ** bits - 1) / 2 ** (bits + 1))          # a dyadic rational with <= 9 significant bits: exact in fp32


def _round(x, bits):
    x = np.asarray(x, F32)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.floor(((x * scale(bits)).astype(F32) + F32(0.5)).astype(F32)).astype(F32)


def quantize4fp(x, bits):
    with np.errstate(invalid="ignore"):
        return (_round(x, bits) / scale(bits)).astype(F32)


def save4fp(x, bits):
    with np.errstate(invalid="ignore"):
        c = ((_round(x, bits) + F32(2 ** (bits - 1))).astype(F32) - F32(1)).astype(F32)
    return np.fmin(np.fmax(c, F32(0)), F32(255)).astype(np.uint8)


def load4fp(codes, bits):
    z = ((np.asarray(codes).astype(F32) - F32(2 ** (bits - 1))).astype(F32) + F32(1)).astype(F32)
    return (z / scale(bits)).astype(F32)


def output_to_u8(x, bits):
    return np.fmin(np.fmax(_round(x, bits), F32(0)), scale(bits)).astype(np.uint8)


def quantize_to_bit(x, bits):
    return output_to_u8(x, bits).astype(F32)


def quantize_clamp(x, bits):
    return np.fmin(np.fmax(np.asarray(x, F32), q_min(bits)), F32(0.5)).astype(F32)


def special_inputs(bits):
    """float32 inputs where a quantiser can go wrong: every exact tie (k + 0.5) / s (the float32 nearest it) for k from
    -s - 2 to s + 1 together with one float32 ulp either side, both clamp ends q_min and 0.5 with their neighbours, values
    outside [q_min, 1/2], +-0, large magnitudes, +-inf and NaN."""
    s = 2 ** bits - 1
    ties = np.array([(k + 0.5) / s for k in range(-s - 2, s + 2)], F32)
    ends = np.array([q_min(bits), 0.5, 1.0, -1.0], F32)
    near = np.concatenate([ties, ends])
    up, down = np.nextafter(near, F32(np.inf)), np.nextafter(near, F32(-np.inf))
    other = np.array([0.0, -0.0, 0.75, -0.75, 2.0, -2.0, 3.0e3, -3.0e3, 1.0e30, -1.0e30, np.finfo(F32).max,
                      -np.finfo(F32).max, np.finfo(F32).tiny, -np.finfo(F32).tiny, 1e-45, np.inf, -np.inf, np.nan], F32)
    return np.concatenate([near, up, down, other]).astype(F32)


def in_range_inputs(rng, bits, n):
    """float32 values in [q_min, 1/2]: uniform draws, the ties inside the range with their neighbours, and both ends."""
    lo = q_min(bits)
    x = (rng.random(n, dtype=F32) * (F32(0.5) - lo) + lo).astype(F32)
    sp = special_inputs(bits)
    sp = sp[np.isfinite(sp) & (sp >= lo) & (sp <= F32(0.5))]
    return np.concatenate([x, sp]).astype(F32)


def pack(codes, bits):
    """nic_pack_codes' layout: 8 / bits codes per byte, code i in bits [(i mod per) * bits, +bits) of byte i / per, only the
    low `bits` bits of each code kept, the unused high part of the last byte zero."""
    per = 8 // bits
    c = np.asarray(codes, np.uint8).reshape(-1)
    nbytes = (c.size * bits + 7) // 8
    padded = np.zeros(nbytes * per, np.uint32)
    padded[:c.size] = c & np.uint8((1 << bits) - 1)
    shifts = (np.arange(per, dtype=np.uint32) * bits)
    return (padded.reshape(nbytes, per) << shifts).sum(1).astype(np.uint8)


def unpack(packed, n, bits):
    per = 8 // bits
    i = np.arange(n)
    p = np.asarray(packed, np.uint8)[i // per].astype(np.uint32)
    return ((p >> ((i % per) * bits).astype(np.uint32)) & ((1 << bits) - 1)).astype(np.uint8)


def random_codes(rng, shape, bits):
    """uint8 codes uniform in [0, 2^b - 1] of shape [C, ...], with code 0 and code 2^b - 1 in every channel (at random
    positions), so the extreme codes are as common as any other rather than rare."""
    top = 2 ** bits - 1
    c = rng.integers(0, top + 1, shape, dtype=np.uint8)
    flat = c.reshape(shape[0], -1)
    for ch in range(shape[0]):
        i, j = rng.choice(flat.shape[1], 2, replace=False)
        flat[ch, i], flat[ch, j] = 0, top
    return c
