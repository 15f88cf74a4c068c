"""CPU model of the whole "row order" neighbour search (salva_b200/csrc: phase_grid dims, k_cell_hist_xy, k_neighbors_xy with
arun()), in numpy f32, against a brute-force statement of the reference's rule (contacts.rs:154-400: pairs of the
3 x 3 x 3 cells floor(x / h) +- 1 that pass `(dx*dx + dy*dy) + dz*dz <= h*h`).

The CUDA kernels of this mode could not be run when they were written (no GPU minutes left), so everything that is pure index
arithmetic — bin functions, grid origin / dims with one padding cell, row ranges, run bounds into the exclusive-scanned cell table,
ascending list order — is restated here line by line and checked for random clouds and jittered lattices, with sub-division factors
1 (plain cells), 2 (the mode bench.py probes), 3 and 4 (the largest the engine accepts).
"""
import numpy as np
import pytest

from test_zbin_model import F, abin, arun

# ---- device helpers (sph_kernels.cuh) ------------------------------------------------------------------------------------


def cell_coord(v, h):
    return int(np.floor(F(v) / F(h)))


def accepted(a, b, h):
    d = (a - b).astype(F)
    d2 = F(F(F(d[0] * d[0]) + F(d[1] * d[1])) + F(d[2] * d[2]))      # dist2_exact: no contraction
    return d2 <= F(F(h) * F(h))


# ---- the search as the engine runs it ------------------------------------------------------------------------------------


def row_order_search(pts, h, xysub):
    n = len(pts)
    cells = np.array([[cell_coord(p[a], h) for a in range(3)] for p in pts])
    lo_c, hi_c = cells.min(axis=0), cells.max(axis=0)                 # k_bounds
    dims = hi_c - lo_c + 3                                            # phase_grid: one padding cell each side
    ox, oy, oz = (lo_c[0] - 1) * xysub, (lo_c[1] - 1) * xysub, lo_c[2] - 1
    nx, ny, nz = dims[0] * xysub, dims[1] * xysub, dims[2]
    ncell = nx * ny * nz

    def cell_id(bx, by, bz):
        return ((bx - ox) * ny + (by - oy)) * nz + (bz - oz)

    ids = np.array([cell_id(abin(p[0], h, xysub) if xysub > 1 else cell_coord(p[0], h),
                            abin(p[1], h, xysub) if xysub > 1 else cell_coord(p[1], h), cell_coord(p[2], h)) for p in pts])  # k_cell_hist(_xy)
    assert ids.min() >= 0 and ids.max() < ncell
    order = np.lexsort((np.arange(n), ids))                           # counting sort + canonical in-cell order (ascending id)
    spts = pts[order]
    cstart = np.zeros(ncell + 1, np.int64)
    np.add.at(cstart, ids + 1, 1)
    cstart = np.cumsum(cstart)
    lists = []
    for i in range(n):                                                # k_neighbors(_xy)
        pi = spts[i]
        cx, cy, cz = (cell_coord(pi[a], h) for a in range(3))
        if xysub > 1:
            xlo, xhi = arun(pi[0], cx, h, xysub)
            ylo, yhi = arun(pi[1], cy, h, xysub)
        else:
            xlo, xhi, ylo, yhi = cx - 1, cx + 1, cy - 1, cy + 1
        zlo, zhi = cz - 1, cz + 1
        out = []
        for bx in range(xlo, xhi + 1):
            for by in range(ylo, yhi + 1):
                lo = cell_id(bx, by, zlo)
                hi = lo + (zhi - zlo) + 1
                assert 0 <= lo <= hi <= ncell
                for j in range(cstart[lo], cstart[hi]):
                    if accepted(pi, spts[j], h):
                        out.append(j)
        assert out == sorted(out)                                     # lists stay in ascending index order
        lists.append(set(order[out]))
    res = [None] * n
    for s, i in enumerate(order):
        res[i] = lists[s]
    return res


def brute_force(pts, h):
    n = len(pts)
    cells = np.array([[cell_coord(p[a], h) for a in range(3)] for p in pts])
    res = []
    for i in range(n):
        near = np.nonzero((np.abs(cells - cells[i]).max(axis=1) <= 1))[0]
        res.append({int(j) for j in near if accepted(pts[i], pts[j], h)})
    return res


def _cloud(seed, n, h, extent):
    rng = np.random.default_rng(seed)
    return (rng.uniform(-extent, extent, (n, 3)) * h + rng.uniform(-3, 3, 3) * h).astype(F)


def _lattice(seed, h):
    r = h / 4.0
    g = np.arange(7, dtype=np.float64)
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) * 2 * r + r
    rng = np.random.default_rng(seed)
    return (p + rng.uniform(-0.05 * r, 0.05 * r, p.shape) - 1.3 * h).astype(F)   # marginal neighbours at d ~ h, negative coordinates


@pytest.mark.parametrize("xysub", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["cloud", "lattice"])
def test_row_order_search_finds_exactly_the_reference_contacts(xysub, kind):
    h = 0.1
    pts = _cloud(5 + xysub, 260, h, 1.6) if kind == "cloud" else _lattice(3, h)
    got = row_order_search(pts, h, xysub)
    want = brute_force(pts, h)
    assert got == want
    assert sum(len(s) for s in want) > 4 * len(pts)                   # the scenes do have contacts
