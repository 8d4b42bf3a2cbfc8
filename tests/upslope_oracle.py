"""tests/upslope_oracle.py -- TEST INFRASTRUCTURE: numpy restatement of the upslope contributing area
(include/splash_cuda.h, splash_upslope_area_run; PARITY UNPINNED).

topmodel::sinkfill / topidx are CRAN code that is not in the reference tree; this restates the published definition
the header gives, with DIFFERENT algorithms from the kernels (which run Jacobi sweeps and level-synchronous rounds):
the fill is a priority flood (Barnes et al. 2014) and the accumulation visits the cells in descending filled
elevation.  Both reach the same least surface and the same sums in the same order, so equal bits are a real check.
Cell sizes follow the terrain slice's restatement (oracle/terrain_oracle.py: R_EARTH, PIR), but are computed per row
with the math module, the same libm the library's host code calls.
"""
import heapq
import math

import numpy as np

from oracle.terrain_oracle import PIR, R_EARTH

# D8 code order E, SE, S, SW, W, NW, N, NE (north row first: S is row + 1)
D8 = ((0, 1), (1, 1), (1, 0), (1, -1), (0, -1), (-1, -1), (-1, 0), (-1, 1))


def upslope_rows(n_rows, ymax, xres, yres, lonlat=True, min_slope_deg=0.1):
    """Per-row metrics with the math module (the C library's cos / tan / sqrt, as the library's host code uses), in
    the same operation order: dx, dy, dd, cell area, cardinal / diagonal contour length, fill step E-W / N-S / diagonal."""
    t = math.tan(min_slope_deg * PIR)
    out = np.empty((n_rows, 9))
    for r in range(n_rows):
        lat_c = ymax - (r + 0.5) * yres
        dy = R_EARTH * (yres * PIR) if lonlat else float(yres)
        dx = R_EARTH * math.cos(lat_c * PIR) * (xres * PIR) if lonlat else float(xres)
        dd = math.sqrt(dx * dx + dy * dy)
        rl = math.sqrt(dx * dy)
        out[r] = (dx, dy, dd, dx * dy, 0.5 * rl, 0.354 * rl, dx * t, dy * t, dd * t)
    return out


def d8_dist_col(k):
    """Column of upslope_rows() with the distance of direction k (E, W: dx; S, N: dy; diagonals: dd); +6 is its eps."""
    return 2 if k & 1 else (1 if k & 2 else 0)


def boundary_mask(z):
    """Valid cells on the grid edge or next to an NA cell."""
    valid = ~np.isnan(z)
    pad = np.zeros((z.shape[0] + 2, z.shape[1] + 2), dtype=bool)
    pad[1:-1, 1:-1] = valid
    all_nb = np.ones(z.shape, dtype=bool)
    for dr, dc in D8:
        all_nb &= pad[1 + dr:1 + dr + z.shape[0], 1 + dc:1 + dc + z.shape[1]]
    return valid & ~all_nb


def fill_priority_flood(z, rows):
    """Priority flood from the boundary cells with Dijkstra's relaxation (a cell keeps the cheapest offer
    max(Z(n), W(c) + eps(n->c)) of any neighbour, since the steps differ by direction and row)."""
    z = np.asarray(z, dtype=np.float64)
    nr, nc = z.shape
    valid = ~np.isnan(z)
    w = np.where(valid, np.inf, np.nan)
    bnd = boundary_mask(z)
    w[bnd] = z[bnd]
    heap = [(z[r, c], r, c) for r, c in zip(*np.nonzero(bnd))]
    heapq.heapify(heap)
    done = np.zeros(z.shape, dtype=bool)
    while heap:
        wc, r, c = heapq.heappop(heap)
        if done[r, c]:
            continue
        done[r, c] = True
        for k, (dr, dc) in enumerate(D8):
            rr, cc = r + dr, c + dc
            if rr < 0 or rr >= nr or cc < 0 or cc >= nc or done[rr, cc] or not valid[rr, cc] or bnd[rr, cc]:
                continue
            # the step from n = (rr, cc) back to c: the opposite direction, same kind, n's row
            v = wc + rows[rr, 6 + d8_dist_col(k)]
            cand = v if v > z[rr, cc] else z[rr, cc]
            if cand < w[rr, cc]:
                w[rr, cc] = cand
                heapq.heappush(heap, (cand, rr, cc))
    return w


def accumulate(w, rows):
    """Quinn et al. (1991) MFD area on the filled surface, cells in descending W: each pulls from its donors (higher
    valid neighbours) in D8 order, area(c) = dx*dy + sum area(u) * (w_uc / S_u), w = ((W(u) - W(c)) / dist) * L."""
    w = np.asarray(w, dtype=np.float64)
    nr, nc = w.shape
    valid = ~np.isnan(w)
    pad = np.full((nr + 2, nc + 2), np.nan)
    pad[1:-1, 1:-1] = w
    nb = [pad[1 + dr:1 + dr + nr, 1 + dc:1 + dc + nc] for dr, dc in D8]
    rr = np.arange(nr)[:, None]
    s = np.zeros(w.shape)
    for k in range(8):        # S in D8 order; + 0.0 where n is not lower leaves the sum's bits alone
        lower = nb[k] < w
        wt = ((w - nb[k]) / rows[rr, d8_dist_col(k)]) * rows[rr, 5 if k & 1 else 4]
        s = s + np.where(lower, wt, 0.0)
    area = np.full(w.shape, np.nan)
    order = np.argsort(-np.where(valid, w, -np.inf), axis=None, kind="stable")[:int(valid.sum())]
    for i in order:
        r, c = divmod(int(i), nc)
        w0 = w[r, c]
        a = rows[r, 3]
        for k, (dr, dc) in enumerate(D8):
            r2, c2 = r + dr, c + dc
            if 0 <= r2 < nr and 0 <= c2 < nc and w[r2, c2] > w0:
                wt = ((w[r2, c2] - w0) / rows[r2, d8_dist_col(k)]) * rows[r2, 5 if k & 1 else 4]
                a = a + area[r2, c2] * (wt / s[r2, c2])
        area[r, c] = a
    return area


def upslope_area(elev, ymax, xres, yres, lonlat=True, min_slope_deg=0.1):
    z = np.asarray(elev, dtype=np.float64)
    rows = upslope_rows(z.shape[0], ymax, xres, yres, lonlat, min_slope_deg)
    w = fill_priority_flood(z, rows)
    return dict(filled=w, area=accumulate(w, rows))
