"""tests/dinf_oracle.py -- TEST INFRASTRUCTURE: numpy restatement of the D-infinity contributing area
(include/splash_cuda.h, splash_upslope_dinf_run; PARITY UNPINNED).

TauDEM is not in this tree; this restates the definition the header gives, with DIFFERENT algorithms from the kernels
wherever the definition allows (the kernels run Jacobi sweeps and level-synchronous frontier rounds):
  * fill: the priority flood of tests/upslope_oracle.py with zero fill steps;
  * flats: Barnes et al. (2014)'s queue-based labelling and breadth-first searches, one flat after another;
  * facets: vectorised numpy with the header's comparison forms;
  * accumulation: cells taken from a CPU Kahn queue, each pulling from its donors in D8 order.
Per-row metrics are upslope_oracle.upslope_rows (the math module, the library's host libm) plus the two facet angles.
"""
import math
from collections import deque

import numpy as np

from tests import upslope_oracle as uo

D8 = uo.D8
# facets in Tarboton's order: (cardinal e1, diagonal e2) as D8 codes (E 0, SE 1, S 2, SW 3, W 4, NW 5, N 6, NE 7), ac, af
FACETS = ((0, 7, 0, 1), (6, 7, 1, -1), (6, 5, 1, 1), (4, 5, 2, -1), (4, 3, 2, 1), (2, 3, 3, -1), (2, 1, 3, 1), (0, 1, 4, -1))
HALF_PI = math.pi / 2
TWO_PI = 4.0 * HALF_PI
TX, TY = 9, 10  # columns of dinf_rows(): atan2(dy, dx), atan2(dx, dy)


def dinf_rows(n_rows, ymax, xres, yres, lonlat=True):
    """upslope_rows with zero fill steps, plus the facet angles theta = atan2(d2, d1) of the two facet orientations."""
    base = uo.upslope_rows(n_rows, ymax, xres, yres, lonlat, 0.0)
    th = np.array([(math.atan2(dy, dx), math.atan2(dx, dy)) for dx, dy in base[:, :2]]).reshape(n_rows, 2)
    return np.concatenate([base, th], axis=1)


def _shift(a, k, fill):
    """a at the neighbour in D8 direction k of every cell (fill outside the grid)."""
    dr, dc = D8[k]
    nr, nc = a.shape
    pad = np.full((nr + 2, nc + 2), fill, dtype=a.dtype)
    pad[1:-1, 1:-1] = a
    return pad[1 + dr:1 + dr + nr, 1 + dc:1 + dc + nc]


def _neighbours(i, nr, nc):
    r, c = divmod(i, nc)
    for dr, dc in D8:
        rr, cc = r + dr, c + dc
        if 0 <= rr < nr and 0 <= cc < nc:
            yield rr * nc + cc


def _bfs(seeds, is_flat, nr, nc):
    """Breadth-first distance over flat cells from the seeds (distance 1); 0 where not reached."""
    dist = np.zeros(nr * nc, dtype=np.int64)
    q = deque()
    for i in seeds:
        dist[i] = 1
        q.append(i)
    while q:
        i = q.popleft()
        for n in _neighbours(i, nr, nc):
            if is_flat[n] and dist[n] == 0:
                dist[n] = dist[i] + 1
                q.append(n)
    return dist


def flats(w):
    """Flat cells, their labels (least index of the 8-connected flat), the two distances, H and the mask M (0 off the
    flats: outlets count as 0)."""
    nr, nc = w.shape
    valid = ~np.isnan(w)
    inner = valid & ~uo.boundary_mask(w)
    lower = np.zeros(w.shape, dtype=bool)
    higher = np.zeros(w.shape, dtype=bool)
    for k in range(8):
        nb = _shift(w, k, np.nan)
        lower |= nb < w
        higher |= nb > w
    flat = inner & ~lower
    fl = flat.ravel()
    wf = w.ravel()
    label = np.full(nr * nc, -1, dtype=np.int64)
    for s in np.flatnonzero(fl):       # raster order: the first cell met is the least index of its flat
        if label[s] >= 0:
            continue
        label[s] = s
        q = deque([s])
        while q:
            i = q.popleft()
            for n in _neighbours(i, nr, nc):
                if fl[n] and label[n] < 0:
                    label[n] = s
                    q.append(n)
    outlet_next = [i for i in np.flatnonzero(fl) if any(not fl[n] and wf[n] == wf[i] for n in _neighbours(i, nr, nc))]
    tow = _bfs(outlet_next, fl, nr, nc)
    away = _bfs(np.flatnonzero(fl & (flat & higher).ravel()), fl, nr, nc)
    hmax = np.zeros(nr * nc, dtype=np.int64)
    np.maximum.at(hmax, label[fl], away[fl])
    mask = np.where(fl, 2 * tow + hmax[np.maximum(label, 0)] - away, 0)
    assert (tow[fl] >= 1).all(), "a flat without an outlet"
    return dict(flat=flat, label=label.reshape(w.shape), towards=tow.reshape(w.shape), away=away.reshape(w.shape),
                mask=mask.reshape(w.shape))


def directions(w, rows, flat, mask):
    """Receivers (cardinal and diagonal D8 code, -1 = none), the diagonal receiver's proportion pd and the angle."""
    nr, nc = w.shape
    inner = ~np.isnan(w) & ~uo.boundary_mask(w)
    rr = np.arange(nr)[:, None]
    dx = np.broadcast_to(rows[rr, 0], w.shape)
    dy = np.broadcast_to(rows[rr, 1], w.shape)
    dd = np.broadcast_to(rows[rr, 2], w.shape)
    m = mask.astype(np.float64)
    e0 = np.where(flat, m, w)
    wn = [_shift(w, k, np.nan) for k in range(8)]
    mn = [_shift(m, k, 0.0) for k in range(8)]
    best = np.zeros(w.shape)
    bf = np.full(w.shape, -1)
    bk = np.zeros(w.shape, dtype=np.int64)
    bs1 = np.zeros(w.shape)
    bs2 = np.zeros(w.shape)
    with np.errstate(invalid="ignore", divide="ignore"):
        for f, (k1, k2, _, _) in enumerate(FACETS):
            ok = inner & (~flat | ((wn[k1] == w) & (wn[k2] == w)))
            e1 = np.where(flat, mn[k1], wn[k1])
            e2 = np.where(flat, mn[k2], wn[k2])
            ew = (k1 & 2) == 0
            d1, d2 = (dx, dy) if ew else (dy, dx)
            s1 = (e0 - e1) / d1
            s2 = (e1 - e2) / d2
            inside = (s2 > 0.0) & (s1 > 0.0) & (s2 * d1 < s1 * d2)
            diag = ~inside & (s2 > 0.0)
            s = np.where(inside, np.sqrt(s1 * s1 + s2 * s2), np.where(diag, (e0 - e2) / dd, s1))
            win = ok & (s > best)
            best = np.where(win, s, best)
            bf = np.where(win, f, bf)
            bk = np.where(win, np.where(inside, 2, np.where(diag, 1, 0)), bk)
            bs1 = np.where(win, s1, bs1)
            bs2 = np.where(win, s2, bs2)
        card = np.full(w.shape, -1)
        dgn = np.full(w.shape, -1)
        pd = np.zeros(w.shape)
        angle = np.full(w.shape, np.nan)
        for f, (k1, k2, ac, af) in enumerate(FACETS):
            th = np.broadcast_to(rows[rr, TX if (k1 & 2) == 0 else TY], w.shape)
            sel = bf == f
            c0, c1, c2 = sel & (bk == 0), sel & (bk == 1), sel & (bk == 2)
            card[c0 | c2] = k1
            dgn[c1 | c2] = k2
            r = np.where(c2, np.arctan(bs2 / bs1), np.where(c1, th, 0.0))
            pd = np.where(c1, 1.0, np.where(c2, np.minimum(r / th, 1.0), pd))
            a = ac * HALF_PI + af * r
            angle = np.where(sel, np.where(a >= TWO_PI, a - TWO_PI, a), angle)
    # flat cells without a facet of positive slope: steepest descent in M over the neighbours at their W
    for i in np.flatnonzero((flat & (bf < 0)).ravel()):
        r, c = divmod(int(i), nc)
        g, kb = 0.0, -1
        for k, (dr, dc) in enumerate(D8):
            if w[r + dr, c + dc] != w[r, c]:
                continue
            v = (float(mask[r, c]) - float(mask[r + dr, c + dc])) / rows[r, uo.d8_dist_col(k)]
            if v > g:
                g, kb = v, k
        assert kb >= 0, "a flat cell without a lower neighbour in M"
        f = 0 if kb == 0 else 7 - kb
        k1, _, ac, af = FACETS[f]
        if kb & 1:
            dgn[r, c], pd[r, c] = kb, 1.0
            a = ac * HALF_PI + af * rows[r, TX if (k1 & 2) == 0 else TY]
        else:
            card[r, c] = kb
            a = ac * HALF_PI + af * 0.0
        angle[r, c] = a - TWO_PI if a >= TWO_PI else a
    return dict(card=card, diag=dgn, pd=pd, angle=angle)


def accumulate(w, rows, card, diag, pd):
    """Kahn's algorithm with a FIFO queue: a cell is taken once all its donors are done, and pulls
    area(u) * p(u -> c) from them in D8 order (p = pd for a diagonal step, 1 - pd for a cardinal one)."""
    nr, nc = w.shape
    valid = ~np.isnan(w).ravel()
    cf, df, pf = card.ravel(), diag.ravel(), pd.ravel()

    def receivers(i):
        r, c = divmod(i, nc)
        return [(r + D8[k][0]) * nc + c + D8[k][1] for k in (cf[i], df[i]) if k >= 0]

    ndon = np.zeros(nr * nc, dtype=np.int64)
    for i in np.flatnonzero(valid):
        for n in receivers(int(i)):
            ndon[n] += 1
    area = np.full(nr * nc, np.nan)
    q = deque(int(i) for i in np.flatnonzero(valid & (ndon == 0)))
    done = 0
    while q:
        i = q.popleft()
        r, c = divmod(i, nc)
        a = rows[r, 3]
        for k, (dr, dc) in enumerate(D8):
            r2, c2 = r + dr, c + dc
            if not (0 <= r2 < nr and 0 <= c2 < nc):
                continue
            u = r2 * nc + c2
            back = (k + 4) & 7
            if back & 1 and df[u] == back:
                a = a + area[u] * pf[u]
            elif not back & 1 and cf[u] == back:
                a = a + area[u] * (1.0 - pf[u])
        area[i] = a
        done += 1
        for n in receivers(i):
            ndon[n] -= 1
            if ndon[n] == 0:
                q.append(n)
    assert done == int(valid.sum()), "the receiver graph has a cycle"
    return area.reshape(w.shape)


def upslope_areav2(elev, ymax, xres, yres, lonlat=True):
    z = np.asarray(elev, dtype=np.float64)
    rows = dinf_rows(z.shape[0], ymax, xres, yres, lonlat)
    w = uo.fill_priority_flood(z, rows)
    fl = flats(w)
    dr = directions(w, rows, fl["flat"], fl["mask"])
    area = accumulate(w, rows, dr["card"], dr["diag"], dr["pd"])
    return dict(filled=w, area=area, rows=rows, **fl, **dr)
