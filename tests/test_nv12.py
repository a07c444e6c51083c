"""CPU: the NV12 -> RGB8 conversion of the letterbox.  The numpy restatement (nv12_ref) against the exact colour matrix over
every (Y, U, V), known answers, and the library's constant table (mars_b200_yuv_coefficients) against the restatement."""
import numpy as np
import pytest

from nv12_ref import coefficients, exact_matrix, nv12_to_rgb, yuv_to_rgb


@pytest.mark.parametrize("colour", [0, 1, 2, 3])
def test_fixed_point_is_within_half_a_step_of_the_exact_matrix(colour):
    """every channel of all 2^24 (Y, U, V) within 0.5 + 2^-8 of the clamped exact conversion; the accumulator fits int32"""
    y0, ys, cs, (kr, kb) = exact_matrix(colour)
    kg = 1.0 - kr - kb
    U, V = np.meshgrid(np.arange(256, dtype=np.float64), np.arange(256, dtype=np.float64), indexing="ij")
    u, v = U - 128, V - 128
    _, cy, crv, cgu, cgv, cbu = coefficients(colour)
    worst = 0.0
    for Y in range(256):
        y = ys * (Y - y0)
        exact = [y + cs * 2 * (1 - kr) * v, y - cs * 2 * (kb * (1 - kb) * u + kr * (1 - kr) * v) / kg, y + cs * 2 * (1 - kb) * u]
        got = yuv_to_rgb(Y, U.astype(np.int64), V.astype(np.int64), colour)
        for e, g in zip(exact, got):
            worst = max(worst, float(np.abs(np.clip(e, 0, 255) - g).max()))
        acc = np.abs(cy * (Y - y0)) + np.abs(crv * u) + np.abs(cgu * u) + np.abs(cgv * v) + np.abs(cbu * u) + 32768
        assert acc.max() < 2 ** 26
    assert worst <= 0.5 + 2 ** -8, worst


@pytest.mark.parametrize("colour", [0, 1, 2, 3])
def test_known_answers(colour):
    lim = colour in (0, 1)
    black, white = (16, 235) if lim else (0, 255)
    assert [int(c) for c in yuv_to_rgb(black, 128, 128, colour)] == [0, 0, 0]
    assert [int(c) for c in yuv_to_rgb(white, 128, 128, colour)] == [255, 255, 255]
    gray = yuv_to_rgb(126 if lim else 128, 128, 128, colour)
    assert len({int(c) for c in gray}) == 1 and abs(int(gray[0]) - 128) <= 1
    if lim:  # limited-range values outside [16, 235] clamp
        assert [int(c) for c in yuv_to_rgb(0, 128, 128, colour)] == [0, 0, 0]
        assert [int(c) for c in yuv_to_rgb(255, 128, 128, colour)] == [255, 255, 255]
    # saturated chroma clamps instead of wrapping
    r, g, b = yuv_to_rgb(white, 255, 255, colour)
    assert int(r) == 255 and int(b) == 255 and 0 <= int(g) <= 255
    r, g, b = yuv_to_rgb(black, 0, 0, colour)
    assert int(r) == 0 and int(b) == 0


def test_chroma_is_replicated_over_each_2x2_block():
    """odd sizes: ceil(h/2) x ceil(w/2) pairs, the last row / column of pairs serves one pixel row / column"""
    y = np.full((3, 5), 120, np.uint8)
    uv = np.arange(2 * 3 * 2, dtype=np.uint8).reshape(2, 3, 2) * 20
    rgb = nv12_to_rgb(y, uv, 0)
    for r in range(3):
        for c in range(5):
            want = yuv_to_rgb(120, uv[r // 2, c // 2, 0], uv[r // 2, c // 2, 1], 0)
            assert [int(v) for v in rgb[r, c]] == [int(v) for v in want], (r, c)


def test_library_table_equals_the_restatement(pkg):
    for colour in range(4):
        assert pkg.capi.yuv_coefficients(colour).tolist() == coefficients(colour).tolist(), colour
    out = np.zeros(6, np.int32)
    for bad in (4, -1):
        assert pkg.lib().mars_b200_yuv_coefficients(bad, out.ctypes.data) == -1
    # the values the header documents
    assert coefficients(0).tolist() == [16, 76309, 104597, 25675, 53279, 132201]
    assert coefficients(3).tolist() == [0, 65536, 103206, 12276, 30679, 121609]
