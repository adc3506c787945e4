"""Reference quantiles for the quantile-field tests: NumPy's 'linear' np.quantile of a float32 array restated in torch float32
arithmetic, so that a reference can be formed on the device for fields too large for the host."""
import numpy as np


def numpy_rank(n, q):
    """(i, j, t) of np.quantile(x, q) for n float32 values and a Python float q (NumPy 2.x converts q to float32):
    pos = float32(n-1) * float32(q), i = floor(pos), j = min(i+1, n-1), t = pos - i."""
    pos = np.float32(n - 1) * np.float32(q)
    i = int(np.floor(pos))
    return i, min(i + 1, n - 1), np.float32(pos - np.float32(i))


def quantile_sorted(zs, q):
    """np.quantile(z, q, axis=0) of float32 samples already sorted along dim 0 (torch.sort: NaN last): the lerp of
    numpy.lib._function_base_impl._lerp in float32 ops, NaN wherever a column holds a NaN."""
    import torch
    i, j, t = numpy_rank(zs.shape[0], q)
    a, b = zs[i], zs[j]
    d = b - a

    def f32(v):
        return torch.tensor(float(v), dtype=torch.float32, device=zs.device)
    r = b - d * f32(np.float32(1) - t) if t >= 0.5 else a + d * f32(t)
    return torch.where(torch.isnan(zs[-1]), torch.full_like(r, float('nan')), r)
