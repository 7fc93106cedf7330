"""A CPU double of Engine.register_spectrum (K14) and Engine.mle_f64 for the `-m "not gpu"` tests, and the float-count
transcription of the oracle's Ertl MLE that both the double and the GPU tests check against.

TEST INFRASTRUCTURE: the product never imports this module."""
import math

import numpy as np
import torch

from tests.fake_engine import FakeEngine

BINS = 64


def spectrum_numpy(regs, begin=0, end=None) -> np.ndarray:
    """int64 [nk, 64, n]: entry (k, v, c - 1) = registers of [begin, end) where exactly c genomes hold a value >= v
    (values clamped at 63), from regs [n, nk, 2^p]."""
    x = np.minimum(np.asarray(regs)[:, :, begin:end], BINS - 1).astype(np.int16)
    n, nk, _ = x.shape
    out = np.zeros((nk, BINS, n), dtype=np.int64)
    for k in range(nk):
        for v in range(1, BINS):
            c = (x[:, k, :] >= v).sum(axis=0)
            out[k, v] = np.bincount(c, minlength=n + 1)[1:]
    return out


def ertl_mle_float(c, p: int) -> float:
    """oracle/ref_numpy.ertl_mle_py with float counts: the same steps, every count a Python float."""
    q = 64 - p
    m = float(1 << p)
    c = [float(v) for v in c] + [0.0] * (q + 2 - len(c))
    if c[q + 1] == m:
        return math.inf
    kmin = next(j for j in range(q + 2) if c[j])
    kmax = next(j for j in range(q + 1, -1, -1) if c[j])
    kminp, kmaxp = max(1, kmin), min(q, kmax)
    z = 0.0
    for j in range(kmaxp, kminp - 1, -1):
        z = 0.5 * z + c[j]
    z = math.ldexp(z, -kminp)
    cp = c[q + 1] + (c[kmaxp] if q >= 1 else 0.0)
    a = z + c[0]
    mp_ = m - c[0]
    b = z + math.ldexp(c[q + 1], -q)
    x = mp_ / (0.5 * b + a) if b <= 1.5 * a else mp_ / b * math.log1p(b / a)
    gprev, dx, relerr = 0.0, x, 1e-2 / math.sqrt(m)
    while dx > x * relerr:
        kap = math.frexp(x)[1]
        xp = math.ldexp(x, -max(kmaxp + 1, kap + 2))
        xp2 = xp * xp
        h = xp - xp2 / 3.0 + (xp2 * xp2) * (1.0 / 45.0 - xp2 / 472.5)
        for _ in range(kap, kmaxp - 1, -1):
            hp = 1.0 - h
            h = (xp + h * hp) / (xp + hp)
            xp += xp
        g = cp * h
        for j in range(kmaxp - 1, kminp - 1, -1):
            hp = 1.0 - h
            h = (xp + h * hp) / (xp + hp)
            xp += xp
            g += c[j] * h
        g += x * a
        dx = dx * (g - mp_) / (gprev - g) if (gprev < g <= mp_) else 0.0
        x += dx
        gprev = g
    return x * m


class RegisterSpectrumFakeEngine(FakeEngine):
    """FakeEngine plus Engine.register_spectrum (numpy counts over the registers) and Engine.mle_f64 (ertl_mle_float)."""

    def register_spectrum(self, regs, p, reg_range=None, out=None):
        self.calls["register_spectrum"] = self.calls.get("register_spectrum", 0) + 1
        begin, end = reg_range if reg_range is not None else (0, 1 << p)
        assert begin % 16 == 0 and end % 16 == 0 and regs.shape[2] == 1 << p
        got = torch.from_numpy(spectrum_numpy(regs.numpy(), begin, end).astype(np.int32))
        return got if out is None else out.add_(got)

    def mle_f64(self, hist, p):
        flat = hist.reshape(-1, BINS).numpy()
        return torch.tensor([ertl_mle_float(row.tolist(), p) for row in flat], dtype=torch.float64).view(hist.shape[:-1])
