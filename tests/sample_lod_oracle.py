"""numpy oracle of per-query level-of-detail sampling (nic_sample_lod, include/nic.h): lambda from a LOD or from screen-space
derivatives, the clamp to [0, L], the mip pair m, min(m + 1, L) and the weight t, all in float32 as the library computes
them, and the blend of sample_oracle.sample_filtered over the decoded mip frames."""
import numpy as np

from sample_oracle import sample_filtered

F32 = np.float32


def lod_from_derivatives(ddx, ddy, extent0):
    """lambda = 0.5 * log2(max(|ddx * E0|^2, |ddy * E0|^2)), every product and sum one float32 operation, x first."""
    ddx, ddy = np.asarray(ddx, F32), np.asarray(ddy, F32)
    e = np.asarray(extent0, F32)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        sx = sy = None
        for a in range(ddx.shape[1]):
            px = (ddx[:, a] * e[a]).astype(F32)
            py = (ddy[:, a] * e[a]).astype(F32)
            sx = (px * px).astype(F32) if sx is None else (sx + (px * px).astype(F32)).astype(F32)
            sy = (py * py).astype(F32) if sy is None else (sy + (py * py).astype(F32)).astype(F32)
        return (F32(0.5) * np.log2(np.fmax(sx, sy))).astype(F32)


def mip_pair(lam, last):
    """(m, m1, t) of each query: lambda clamped to [0, last] (NaN -> 0, -inf -> 0), m = floor, t = lambda - m."""
    lam = np.asarray(lam, F32)
    lc = np.fmin(np.fmax(lam, F32(0)), F32(last)).astype(F32)
    m = np.floor(lc).astype(np.int64)
    t = (lc - m.astype(F32)).astype(F32)
    return m, np.minimum(m + 1, last), t


def blend_mips(s_m, s_m1, t):
    """(1 - t) * S_m + t * S_m1 in float32, one rounding per operation (the library's blend sequence)."""
    t = np.asarray(t, F32)[:, None]
    a = ((F32(1) - t).astype(F32) * np.asarray(s_m, F32)).astype(F32)
    return (a + (t * np.asarray(s_m1, F32)).astype(F32)).astype(F32)


def sample_lod(frames, coords, lam, align_corners, address="clamp"):
    """Trilinear mip filtering of the decoded frames [mip 0 .. L] (each [Sx, Sy(, Sz), C]) at coords [Q, D] with per-query
    lambda -> [Q, C] float64: each mip's tap sum (sample_filtered), blended with float64 weights (1 - t, t)."""
    last = len(frames) - 1
    m, m1, t = mip_pair(lam, last)
    per_mip = [sample_filtered(f, coords, align_corners, address) for f in frames]
    stack = np.stack(per_mip)                                                  # [L + 1, Q, C]
    q = np.arange(len(t))
    t64 = t.astype(np.float64)[:, None]
    return (1.0 - t64) * stack[m, q] + t64 * stack[m1, q]
