"""CPU: the tile grid of tiled detection (mars_b200_tile_rois).  The 3840x2160 known answer, a frame no larger than a tile,
coverage / containment / overlap / order over random sizes, the count-greater-than-cap contract and the -1 cases."""
import numpy as np
import pytest


def test_4k_known_answer(pkg):
    t = pkg.capi.tile_rois(3840, 2160, 640, 640, 128, 128)
    xs, ys = sorted(set(t["x"].tolist())), sorted(set(t["y"].tolist()))
    assert len(t) == 32 and len(xs) == 8 and len(ys) == 4
    assert xs == [0, 512, 1024, 1536, 2048, 2560, 3072, 3200] and ys == [0, 512, 1024, 1520]
    assert (t["w"] == 640).all() and (t["h"] == 640).all() and (t["frame"] == 0).all()
    # row-major
    assert t["y"].tolist() == [y for y in ys for _ in xs] and t["x"].tolist() == xs * len(ys)
    full = pkg.capi.tile_rois(3840, 2160, 640, 640, 128, 128, with_full=True, frame=5)
    assert len(full) == 33 and tuple(full[0]) == (5, 0, 0, 3840, 2160)
    assert full[1:][["x", "y", "w", "h"]].tolist() == t[["x", "y", "w", "h"]].tolist() and (full["frame"] == 5).all()


@pytest.mark.parametrize("w,h", [(640, 640), (100, 37), (1, 1), (640, 200)])
def test_one_region_when_the_frame_fits_a_tile(pkg, w, h):
    for with_full in (False, True):  # one tile: no extra whole-frame region
        t = pkg.capi.tile_rois(w, h, 640, 640, 128, 128, with_full=with_full, frame=2)
        assert t.tolist() == [(2, 0, 0, w, h)]


def test_one_axis_tiled(pkg):
    t = pkg.capi.tile_rois(1000, 300, 640, 640, 100, 100)
    assert t.tolist() == [(0, 0, 0, 640, 300), (0, 360, 0, 640, 300)]


def test_random_grids(pkg):
    rng = np.random.default_rng(0)
    for _ in range(300):
        w, h = int(rng.integers(1, 3000)), int(rng.integers(1, 3000))
        tw, th = int(rng.integers(1, 800)), int(rng.integers(1, 800))
        ow, oh = int(rng.integers(0, tw)), int(rng.integers(0, th))
        with_full = bool(rng.integers(0, 2))
        t = pkg.capi.tile_rois(w, h, tw, th, ow, oh, with_full=with_full, frame=3)
        assert (t["frame"] == 3).all()
        nx = 1 if w <= tw else -(-(w - tw) // (tw - ow)) + 1
        ny = 1 if h <= th else -(-(h - th) // (th - oh)) + 1
        full = with_full and nx * ny > 1
        assert len(t) == nx * ny + full
        if full:
            assert tuple(t[0]) == (3, 0, 0, w, h)
            t = t[1:]
        assert (t["x"] >= 0).all() and (t["y"] >= 0).all()
        assert (t["x"] + t["w"] <= w).all() and (t["y"] + t["h"] <= h).all()
        assert (t["w"] == min(tw, w)).all() and (t["h"] == min(th, h)).all()
        g = t.reshape(ny, nx)
        assert (g["y"] == g["y"][:, :1]).all() and (g["x"] == g["x"][:1, :]).all()  # row-major grid
        x0, y0 = g["x"][0], g["y"][:, 0]
        assert (np.diff(x0) > 0).all() and (np.diff(y0) > 0).all()
        # neighbours overlap by at least the overlap (the last one more when it is pulled flush with the edge)
        assert (x0[:-1] + min(tw, w) - x0[1:] >= ow).all() and (y0[:-1] + min(th, h) - y0[1:] >= oh).all()
        if w * h <= 1 << 20:  # every pixel covered
            cov = np.zeros((h, w), bool)
            for r in t:
                cov[r["y"]: r["y"] + r["h"], r["x"]: r["x"] + r["w"]] = True
            assert cov.all()
        else:
            assert x0[0] == 0 and x0[-1] + min(tw, w) == w and y0[0] == 0 and y0[-1] + min(th, h) == h


def test_cap_and_rejections(pkg):
    L, capi = pkg.lib(), pkg.capi
    out = np.full(40, -7, dtype=capi.ROI_DTYPE)
    assert L.mars_b200_tile_rois(0, 3840, 2160, 640, 640, 128, 128, 1, out.ctypes.data, 32) == 33
    assert (out["x"] == -7).all()  # more than cap: nothing written
    assert L.mars_b200_tile_rois(0, 3840, 2160, 640, 640, 128, 128, 1, None, 0) == 33
    assert L.mars_b200_tile_rois(0, 3840, 2160, 640, 640, 128, 128, 1, out.ctypes.data, 33) == 33
    assert (out["x"][33:] == -7).all() and tuple(out[0]) == (0, 0, 0, 3840, 2160)
    bad = [(0, 10, 640, 640, 0, 0), (10, -1, 640, 640, 0, 0), (10, 10, 0, 640, 0, 0), (10, 10, 640, -5, 0, 0),
           (10, 10, 640, 640, -1, 0), (10, 10, 640, 640, 0, -1), (10, 10, 640, 640, 640, 0), (10, 10, 640, 640, 0, 700)]
    for b in bad:
        assert L.mars_b200_tile_rois(0, *b, 0, out.ctypes.data, 40) == -1, b
        with pytest.raises(ValueError):
            capi.tile_rois(*b)
