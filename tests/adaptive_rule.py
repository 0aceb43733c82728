"""numpy restatement of rh_render_adaptive's selection rule (include/rayhs_b200.h), in the header's operation order so
that it gives the library's decision bit for bit."""
import numpy as np


def active_pixels(counts, sums, sumsq, spp: int, stream_spp: int, min_spp: int, threshold: float, valid=None):
    """counts uint [...], sums / sumsq float64 [..., 3] -> bool [...]: the pixels the next call traces.  `valid`: False
    for padding rows of a shard (never active)."""
    n = np.asarray(counts).astype(np.int64)
    S = np.asarray(sums, dtype=np.float64)
    Q = np.asarray(sumsq, dtype=np.float64)
    tt = np.float64(threshold) * np.float64(threshold)
    nf = n.astype(np.float64)
    nn = nf * (n - 1).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        d = Q - S * (S / nf[..., None])
        over = (d > (tt * nn)[..., None]).any(axis=-1)
    act = (n + spp <= stream_spp) & ((n < min_spp) | over)
    if valid is not None:
        act &= valid
    return act


def fold(samples):
    """samples float64 [n, ..., 3] in sample order -> (S, Q) as the library folds them: S = foldl (+) 0 x, Q = foldl (+)
    0 (x * x), each square rounded before it is added."""
    S = np.zeros(samples.shape[1:], dtype=np.float64)
    Q = np.zeros(samples.shape[1:], dtype=np.float64)
    for x in samples:
        S = S + x
        Q = Q + x * x
    return S, Q
