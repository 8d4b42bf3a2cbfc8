"""Seeded DEMs for the upslope-area tests and tools/upslope_bench.py."""
from __future__ import annotations

import numpy as np


def fractal_dem(n_rows: int, n_cols: int, seed: int, relief: float = 1500.0, tilt: float = 800.0, sea: float = 0.2):
    """Spectral-synthesis fractal surface (amplitude ~ 1/k^1.6) plus a large-scale tilt down to the south-west, rounded
    to centimetres; the lowest `sea` fraction of the cells is NaN (sea), so the grid has coasts and islands."""
    rng = np.random.default_rng(seed)
    ky = np.fft.fftfreq(n_rows)[:, None]
    kx = np.fft.rfftfreq(n_cols)[None, :]
    k = np.hypot(ky, kx)
    k[0, 0] = 1.0
    spec = np.fft.rfft2(rng.standard_normal((n_rows, n_cols))) / k ** 1.6
    spec[0, 0] = 0.0
    z = np.fft.irfft2(spec, s=(n_rows, n_cols))
    z = (z - z.min()) / max(np.ptp(z), 1e-300) * relief
    y, x = np.mgrid[0:n_rows, 0:n_cols]
    z = z + tilt * (1.0 - y / max(n_rows - 1, 1)) * 0.5 + tilt * (x / max(n_cols - 1, 1)) * 0.5
    z = np.round(z * 100.0) / 100.0
    if sea > 0:
        z[z < np.quantile(z, sea)] = np.nan
    return z
