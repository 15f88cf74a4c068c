"""CPU model of the sub-divided bins of the row-order neighbour search (salva_b200/csrc/sph_kernels.cuh: abin(), arun()).

In row order the counting sort splits every cell of width h into `sub` slices along x and y, and the neighbour search cuts each
row of the 27-cell stencil down to the slices within reach of the particle.  The claim that makes this safe — the contact sets
stay EXACTLY the reference's (contacts.rs:285: `(dx*dx + dy*dy) + dz*dz <= h*h` in f32, candidates from the 3 x 3 x 3 cells
floor(x / h) +- 1) — is a statement about f32 arithmetic, so it is checked here along one axis with numpy's IEEE f32 (same
division, same floor, directed rounding emulated through f64 + nextafter):

  * abin is monotone in v and every bin lies inside ONE reference cell (bin // sub == floor(v / h));
  * whenever a pair passes the f32 distance test with its other two coordinate differences zero (the worst case for this axis)
    and sits in adjacent reference cells, the partner's bin lies inside the run [lo, hi] the particle scans.
"""
import numpy as np
import pytest

F = np.float32


def abin(v, h, sub):
    q = F(v) / F(h)                      # __fdiv_rn
    fl = np.floor(q)
    return int(fl) * sub + min(sub - 1, int(F(q - fl) * F(sub)))  # q - floor(q) is exact in f32; the product is rounded, hence the clamp


def _round_dir(x64, up):
    r = F(x64)
    if up and float(r) < x64:
        r = np.nextafter(r, F(np.inf))
    if not up and float(r) > x64:
        r = np.nextafter(r, F(-np.inf))
    return r


def h_reach(h):
    return np.nextafter(F(F(h) * F(1.00001)), F(np.inf))          # fill_static_consts(): Consts::h_reach


def arun(v, c, h, sub):
    lo = max(abin(_round_dir(float(F(v)) - float(h_reach(h)), up=False), h, sub), (c - 1) * sub)   # __fsub_rd
    hi = min(abin(_round_dir(float(F(v)) + float(h_reach(h)), up=True), h, sub), (c + 2) * sub - 1)  # __fadd_ru
    return lo, hi


def accepted(zi, zj, h):
    dz = F(F(zi) - F(zj))
    return F(dz * dz) <= F(F(h) * F(h))                           # dist2_exact with the other two differences zero


@pytest.mark.parametrize("sub", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("h", [0.1, 0.2, 0.37])
def test_zbin_is_monotone_and_nested_in_the_reference_cells(sub, h):
    rng = np.random.default_rng(sub * 7 + int(h * 100))
    z = np.sort(np.concatenate([rng.uniform(-40 * h, 40 * h, 4000), (np.arange(-60, 60) * h).astype(np.float64),
                                np.nextafter((np.arange(-60, 60) * F(h)).astype(F), F(-np.inf)).astype(np.float64)]).astype(F))
    bins = np.array([abin(v, h, sub) for v in z])
    assert np.all(np.diff(bins) >= 0)
    cells = np.floor(z / F(h)).astype(np.int64)
    assert np.array_equal(np.floor_divide(bins, sub), cells)


@pytest.mark.parametrize("sub", [2, 3, 4, 8])
@pytest.mark.parametrize("h", [0.1, 0.2, 0.37])
def test_no_accepted_pair_of_adjacent_cells_is_cut_off(sub, h):
    rng = np.random.default_rng(sub * 13 + int(h * 1000))
    checked = near = 0
    for scale in (1.0, 30.0, 3000.0):                              # far from the origin the f32 grid gets coarse
        zi_all = rng.uniform(-40 * h * scale, 40 * h * scale, 1500).astype(F)
        for zi in zi_all:
            # partners right at the cutoff (a few ulps either side) and anywhere within reach
            cands = [F(zi + s * F(h)) for s in (-1.0, 1.0)]
            for c in list(cands):
                v = c
                for _ in range(4):
                    v = np.nextafter(v, F(np.inf))
                    cands.append(v)
                v = c
                for _ in range(4):
                    v = np.nextafter(v, F(-np.inf))
                    cands.append(v)
            cands += list((zi + rng.uniform(-1.0, 1.0, 6) * h).astype(F))
            czi = int(np.floor(F(zi) / F(h)))
            lo, hi = arun(zi, czi, h, sub)
            assert lo <= abin(zi, h, sub) <= hi
            for zj in cands:
                if not accepted(zi, zj, h):
                    continue
                czj = int(np.floor(F(zj) / F(h)))
                if abs(czj - czi) > 1:
                    continue                                       # the reference's stencil does not look there either
                checked += 1
                near += abs(abs(float(zi) - float(zj)) - h) < 1e-5 * h
                assert lo <= abin(zj, h, sub) <= hi, (zi, zj, lo, hi, abin(zj, h, sub))
    assert checked > 10000 and near > 1000
