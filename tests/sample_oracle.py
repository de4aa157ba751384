"""numpy oracle of filtered sampling (nic_sample, include/nic.h): the fp32 tap rule step for step (np.fmax / np.fmin /
np.floor on float32, the wrap as np.fmod), the blend of the taps in float64, and the blend of two mips (fractional LOD)."""
import numpy as np

F32 = np.float32


def tap_rule(coords, extent, align_corners, address):
    """coords [Q, D] float32 -> (taps int64 [Q, 2^D, D], weights float32 [Q, 2^D]); taps ordered with x slowest."""
    c = np.asarray(coords, F32)
    q, dim = c.shape
    idx, wts = [], []
    for a in range(dim):
        s = int(extent[a])
        u = c[:, a]
        p = u * F32(s - 1) if align_corners else u * F32(s) - F32(0.5)
        p = np.fmin(np.fmax(p, F32(-2.0 ** 24)), F32(2.0 ** 24))         # NaN -> -2^24 (fmax ignores a NaN operand)
        i0 = np.floor(p)
        f = (p - i0).astype(F32)
        t = np.stack([i0.astype(np.int64), i0.astype(np.int64) + 1], 1)
        if address == "wrap":
            t = np.fmod(t, s)
            t = np.where(t < 0, t + s, t)
        else:
            t = np.clip(t, 0, s - 1)
        idx.append(t)
        wts.append(np.stack([(F32(1) - f).astype(F32), f], 1))
    T = 1 << dim
    taps = np.zeros((q, T, dim), np.int64)
    w = np.ones((q, T), F32)
    for k in range(T):
        for a in range(dim):
            hi = (k >> (dim - 1 - a)) & 1
            taps[:, k, a] = idx[a][:, hi]
            w[:, k] = (w[:, k] * wts[a][:, hi]).astype(F32)
    return taps, w


def sample_filtered(dense, coords, align_corners, address="clamp"):
    """Bilinear / trilinear sample of a decoded frame `dense` [Sx, Sy(, Sz), C] at normalised coords [Q, D] -> [Q, C]
    float64: sum over the taps of weight * texel, in tap order."""
    dense = np.asarray(dense)
    dim = dense.ndim - 1
    taps, w = tap_rule(coords, dense.shape[:dim], align_corners, address)
    out = np.zeros((taps.shape[0], dense.shape[-1]), np.float64)
    for k in range(taps.shape[1]):
        v = dense[tuple(taps[:, k, a] for a in range(dim))].astype(np.float64)
        out += w[:, k, None].astype(np.float64) * v
    return out


def blend_lod(a, b, t):
    """A fractional LOD m + t: (1 - t) * sample at mip m + t * sample at mip m + 1."""
    return (1.0 - t) * np.asarray(a, np.float64) + t * np.asarray(b, np.float64)
