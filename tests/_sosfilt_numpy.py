"""numpy emulation of kernel 10 (csrc/iqw_sosfilt.cu): the fp32 cascade per chunk through scipy's complex64
sosfilt, the chunk and group folds and the carry in float64, in the kernels' geometry and order.  scipy's loop
rounds each product where the device fuses multiply-adds, so the emulation matches the device within the error
bound, not bit for bit; emulation against emulation is bitwise."""
import numpy as np
import scipy.signal as ss
import torch

from iqwaveform_b200 import _plan, fourier

FILTERS = {
    'dc_blocker': np.array([[1, -1, 0, 1, -0.999, 0]]),
    'butter4': ss.butter(4, 0.002, output='sos'),
    'ellip8': ss.ellip(8, 0.1, 80, 0.05, output='sos'),
    'ellip16': ss.ellip(16, 0.1, 100, 0.2, output='sos'),
    'butter32': ss.butter(32, 0.3, output='sos'),
    'integrator': np.array([[1, 0, 0, 1, -1, 0]]),
}


def _fold(P, t, b, every=False):
    """t <- P t + b[:, k] for k in order, vectorised over the leading axis; optionally the state before each k"""
    out = np.empty_like(b) if every else None
    for k in range(b.shape[1]):
        if every:
            out[:, k] = t
        t = t @ P.T + b[:, k]
    return t, out


def states(x, sos32):
    """-> (chunk states (chunks, 2S) complex64, group states (groups, 2S) complex128) of one row"""
    S = len(sos32)
    L, G, _ = fourier._sosfilt_geometry(S)
    P = _plan.sosfilt_powers(sos32, L, G, 1)[0]
    ng = -(-x.size // (L * G))
    xp = np.zeros(ng * G * L, np.complex64)
    xp[:x.size] = x
    _, zf = ss.sosfilt(sos32, xp.reshape(-1, L), axis=-1, zi=np.zeros((S, ng * G, 2), np.complex64))
    bc = zf.transpose(1, 0, 2).reshape(ng * G, 2 * S)
    bg, _ = _fold(P, np.zeros((ng, 2 * S), np.complex128), bc.reshape(ng, G, 2 * S).astype(np.complex128))
    return bc, bg


def carry(bg, sos32, zi=None):
    """group states of the whole row -> start state of each group, from zi (2S,) complex64 or zero"""
    S = len(sos32)
    L, G, H = fourier._sosfilt_geometry(S)
    _, PG, PH = _plan.sosfilt_powers(sos32, L, G, H)
    ng = bg.shape[0]
    nb = -(-ng // H)
    b = np.zeros((nb * H, 2 * S), np.complex128)
    b[:ng] = bg
    b = b.reshape(nb, H, 2 * S)
    blocks, _ = _fold(PG, np.zeros((nb, 2 * S), np.complex128), b)
    t0 = np.zeros((1, 2 * S), np.complex128) if zi is None else np.asarray(zi, np.complex64)[None].astype(np.complex128)
    _, starts = _fold(PH, t0, blocks[None], every=True)
    _, sg = _fold(PG, starts[0], b, every=True)
    return sg.reshape(nb * H, 2 * S)[:ng]


def apply(x, sos32, bc, sg, want_zf=False):
    """-> (y, zf (2S,) complex64 or None) of one row from its chunk states and its groups' start states"""
    S = len(sos32)
    L, G, _ = fourier._sosfilt_geometry(S)
    P = _plan.sosfilt_powers(sos32, L, G, 1)[0]
    ng = sg.shape[0]
    _, sc = _fold(P, sg.astype(np.complex128), bc.reshape(ng, G, 2 * S).astype(np.complex128), every=True)
    sc = sc.reshape(ng * G, 2 * S).astype(np.complex64)
    xp = np.zeros(ng * G * L, np.complex64)
    xp[:x.size] = x
    zi = sc.reshape(-1, S, 2).transpose(1, 0, 2)
    y, _ = ss.sosfilt(sos32, xp.reshape(-1, L), axis=-1, zi=zi)
    zf = None
    if want_zf:
        c = (x.size - 1) // L
        _, zf = ss.sosfilt(sos32, x[c * L:], zi=sc[c].reshape(S, 2))
        zf = zf.reshape(2 * S).astype(np.complex64)
    return y.reshape(-1)[:x.size].astype(np.complex64), zf


def emulate(x, sos32, zi=None):
    """one row through the three passes -> (y, zf (S, 2) or None); zi (S, 2)"""
    S = len(sos32)
    if x.size == 0:
        return x.astype(np.complex64), (None if zi is None else np.asarray(zi, np.complex64))
    bc, bg = states(x, sos32)
    sg = carry(bg, sos32, None if zi is None else np.asarray(zi).reshape(2 * S))
    y, zf = apply(x, sos32, bc, sg, want_zf=zi is not None)
    return y, (None if zi is None else zf.reshape(S, 2))


class NumpyOps:
    """the three steps of distributed.SosfiltShardOps in numpy, on torch CPU tensors"""

    def states(self, x, sos32):
        self._bc, bg = states(np.asarray(x), sos32)
        return torch.from_numpy(bg)

    def carry(self, g, sos32, zi):
        return torch.from_numpy(carry(g.numpy(), sos32, None if zi is None else zi.numpy()))

    def apply(self, x, sos32, s, want_zf):
        x = np.asarray(x)
        if x.size == 0:
            return torch.zeros(0, dtype=torch.complex64), None
        y, zf = apply(x, sos32, self._bc, s.numpy(), want_zf)
        return torch.from_numpy(y), (None if zf is None else torch.from_numpy(zf))


def reference(x, sos32, zi=None):
    """(y64, E32): scipy's float64 sosfilt of the float32 sos, and the max error of scipy's complex64 sosfilt
    against it (per row along the last axis); with zi also (zf64, zf32)"""
    s64 = sos32.astype(np.float64)
    if zi is None:
        y64 = ss.sosfilt(s64, x.astype(np.complex128))
        y32 = ss.sosfilt(sos32, x)
        return y64, np.abs(y32 - y64).max(axis=-1)
    y64, zf64 = ss.sosfilt(s64, x.astype(np.complex128), zi=np.asarray(zi, np.complex128))
    y32, zf32 = ss.sosfilt(sos32, x, zi=np.asarray(zi, np.complex64))
    return y64, np.abs(y32 - y64).max(axis=-1), zf64, zf32


def ratio(y, y64, e32, floor_ulps=4):
    """max |y - y64| per row in units of the bound: E32, floored at a few ulp of max |y64|"""
    unit = np.maximum(e32, floor_ulps * 2.0 ** -24 * np.abs(y64).max(axis=-1))
    unit = np.where(unit > 0, unit, 1e-30)
    return (np.abs(y - y64).max(axis=-1) / unit).max()


def zf_unit(zf32, zf64, e32):
    """the unit of the zf bound: scipy's complex64 error on the final state itself, or on the row's outputs when
    that is larger (the state at one instant can be accurate by chance; its error is of the outputs' order)"""
    return max(float(np.abs(zf32 - zf64).max()), float(np.max(e32)))


def signal(rng, n, burst=True):
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    if burst and n:
        x[n // 3] += 1000
    return x
