"""numpy restatement of the NV12 -> RGB8 conversion of the letterbox (include/mars_b200.h, MARS_B200_YUV_*): 16.16 fixed point,
constants from (Kr, Kb) and the range, no chroma interpolation (the U,V pair of a 2 x 2 block serves all four pixels)."""
import numpy as np

# variant -> ((Kr, Kb), full range)
VARIANTS = {0: ((0.299, 0.114), False), 1: ((0.2126, 0.0722), False), 2: ((0.299, 0.114), True), 3: ((0.2126, 0.0722), True)}


def coefficients(colour):
    """[y0, cy, crv, cgu, cgv, cbu]: each constant floor(c * 65536 + 0.5) in double"""
    (kr, kb), full = VARIANTS[colour]
    kg = 1.0 - kr - kb
    ys, cs, y0 = (1.0, 1.0, 0) if full else (255.0 / 219.0, 255.0 / 224.0, 16)
    c = [ys, cs * 2 * (1 - kr), cs * 2 * kb * (1 - kb) / kg, cs * 2 * kr * (1 - kr) / kg, cs * 2 * (1 - kb)]
    return np.array([y0] + [int(np.floor(v * 65536 + 0.5)) for v in c], dtype=np.int64)


def exact_matrix(colour):
    """(y0, ys, cs, (Kr, Kb)) of the exact float conversion the fixed point approximates"""
    (kr, kb), full = VARIANTS[colour]
    return (0, 1.0, 1.0, (kr, kb)) if full else (16, 255.0 / 219.0, 255.0 / 224.0, (kr, kb))


def yuv_to_rgb(Y, U, V, colour):
    """integer conversion of broadcastable Y, U, V arrays -> R, G, B int64 arrays in [0, 255]"""
    y0, cy, crv, cgu, cgv, cbu = coefficients(colour)
    y = cy * (np.asarray(Y, np.int64) - y0) + 32768
    u, v = np.asarray(U, np.int64) - 128, np.asarray(V, np.int64) - 128
    return (np.clip((y + crv * v) >> 16, 0, 255), np.clip((y - cgu * u - cgv * v) >> 16, 0, 255),
            np.clip((y + cbu * u) >> 16, 0, 255))


def nv12_to_rgb(y, uv, colour):
    """[h, w] luma and [ceil(h/2), ceil(w/2), 2] U,V planes -> [h, w, 3] uint8 RGB frame"""
    h, w = y.shape
    c = np.asarray(uv).repeat(2, axis=0).repeat(2, axis=1)[:h, :w]
    r, g, b = yuv_to_rgb(y, c[..., 0], c[..., 1], colour)
    return np.stack([r, g, b], axis=-1).astype(np.uint8)


def nv12_frame(w, h, seed):
    """a random NV12 frame: (y [h, w], uv [ceil(h/2), ceil(w/2), 2]) uint8"""
    rng = np.random.default_rng(seed)
    return (rng.integers(0, 256, (h, w), dtype=np.uint8), rng.integers(0, 256, ((h + 1) // 2, (w + 1) // 2, 2), dtype=np.uint8))
