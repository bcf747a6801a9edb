"""Hand-built splat scenes for the raster reference tests (tests/test_f2b_reference.py on the CPU,
tests/test_raster_reference_gpu.py on the GPU).

The camera is an identity model-view and a projection with w = -z, so a splat at depth z = -zd lands at window pixel
(cx, cy) = ((x/zd * .5 + .5) W, (-y/zd * .5 + .5) H), and its screen covariance (before the shader adds 0.3,
index.js:139-141) is (focal/zd)^2 [[S00, -S01], [-S01, S11]] of its world covariance: each case states its footprint
in pixels directly.  The covariance is quantised to the int16 record the pack produces (index.js:384-387), so what
the renderer sees is only close to the requested footprint; the references take the packed record as given."""
import numpy as np

FOCAL = 200.0
VIEW = np.array([0.0, 0.0, 1.0, 0.0], np.float32)  # row 2 of the identity model-view: sort depth = z
N_Q8 = 6  # needle_scene: leading splats that vanish


def camera():
    P = np.zeros(16, np.float32)
    P[0] = 1.0; P[5] = -1.0; P[10] = -1.0; P[11] = -1.0; P[14] = -0.02
    MV = np.eye(4, dtype=np.float32).reshape(16)
    return P, MV


def _q16(v):
    return np.int16(v).view(np.uint16).astype(np.uint32)


def splats(W, H, cx, cy, s00, s01, s11, rgba, zd=None):
    """Packed records (center_scale, cov_color, size_alpha) of splats centred on window pixel (cx, cy) with screen
    covariance [[s00, s01], [s01, s11]] px^2 (before + 0.3).  Arrays broadcast; zd (distance, default 5 + 1e-3 i)
    makes the back-to-front draw order the index order reversed, i.e. nearest first is index order."""
    cx, cy, s00, s01, s11 = np.broadcast_arrays(*(np.atleast_1d(np.asarray(a, np.float64)) for a in (cx, cy, s00, s01, s11)))
    n = cx.shape[0]
    rgba = np.broadcast_to(np.asarray(rgba, np.uint32).reshape(-1, 4), (n, 4))
    zd = 5.0 + 1e-3 * np.arange(n) if zd is None else np.broadcast_to(np.asarray(zd, np.float64), (n,))
    k = (FOCAL / zd) ** 2
    sig = np.stack([s00 / k, -s01 / k, s11 / k], 1)  # world Sigma00, Sigma01, Sigma11 (Sigma_2x = 0)
    mx = np.abs(sig).max(1)
    scale = (mx / 32767.0).astype(np.float32)
    q = np.rint(sig / np.where(scale > 0, scale, 1.0)[:, None]).clip(-32767, 32767).astype(np.int64)
    cs = np.zeros((n, 4), np.float32)
    cs[:, 0] = (cx / W * 2.0 - 1.0) * zd
    cs[:, 1] = -(cy / H * 2.0 - 1.0) * zd
    cs[:, 2] = -zd
    cs[:, 3] = scale
    cc = np.zeros((n, 4), np.uint32)
    cc[:, 0] = _q16(q[:, 0]) | (_q16(q[:, 1]) << 16)
    cc[:, 1] = _q16(q[:, 2]) << 16
    cc[:, 3] = rgba[:, 0] | (rgba[:, 1] << 8) | (rgba[:, 2] << 16) | (rgba[:, 3] << 24)
    return cs, cc, np.ones(n, np.float32)


def cat(*parts):
    """Concatenate (cs, cc, sa) triples; later parts get larger distances only if their zd says so."""
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


def colours(rng, n, alpha):
    c = rng.integers(0, 256, (n, 4)).astype(np.uint32)
    c[:, 3] = alpha
    return c


def sweep_scene(rng):
    """Centres swept in 1/8 px steps across the tile edge x = 96 (also a bin edge) and the tile edge y = 32, with an
    axis-aligned footprint whose r = 2 half-extents are exactly 3 px (x) and 6 px (y): every eighth centre puts a pixel
    centre exactly on the r^2 = 4 contour, others just inside or outside it."""
    W, H = 200, 120
    i = np.arange(128)
    s00 = 9.0 / 8.0 - 0.3   # lambda2 = 1.125: 2 sqrt(2 lambda2) = 3
    s11 = 4.5 - 0.3         # lambda1 = 4.5:   2 sqrt(2 lambda1) = 6
    a = splats(W, H, 88.5 + i / 8.0, 26.5 + (i % 32) / 8.0, s00, 0.0, s11, colours(rng, 128, 96))
    b = splats(W, H, 40.0 + (i % 16) / 16.0, 20.5 + i / 8.0, s00, 0.0, s11, colours(rng, 128, 96), zd=6.0 + 1e-3 * i)
    c = splats(W, H, 186.5 + i / 16.0, 90.0 + i / 16.0, s00, 0.0, s11, colours(rng, 128, 96), zd=7.0 + 1e-3 * i)
    return W, H, cat(a, b, c)


def needle_scene(rng):
    """Needles: minor axis at the 0.1 eigenvalue floor (a negative quantised minor variance), major axis 20 px or at the
    1024 px clamp, at angles 0, 1e-3 rad, 45 deg and 90 deg, three sub-pixel offsets each.  The first N_Q8 = 6 are
    exactly axis-aligned with Sigma00 >= Sigma11: normalize(vec2(0)) is NaN and they vanish (quirk Q8)."""
    W, H = 160, 130
    parts = []
    k = 0
    for major in (400.0, 2.0e6):
        for th in (0.0, 1e-3, np.pi / 4, np.pi / 2):
            c, s = np.cos(th), np.sin(th)
            minor = -1e-3 * major
            S = np.array([[c, -s], [s, c]]) @ np.diag([major, minor]) @ np.array([[c, s], [-s, c]])
            s01 = 0.0 if th in (0.0, np.pi / 2) else S[0, 1]
            s00, s11 = (major, minor) if th == 0.0 else ((minor, major) if th == np.pi / 2 else (S[0, 0], S[1, 1]))
            for dx in (0.0, 0.3, 0.5):
                parts.append((60.0 + 7 * k + dx, 64.5 + 0.25 * k + dx, s00, s01, s11))
            k += 1
    p = np.array(parts)
    # the angle-0 (Q8) needles first
    first = np.argsort([0 if (r[3] == 0.0 and r[2] >= r[4]) else 1 for r in p], kind="stable")
    p = p[first]
    return W, H, splats(W, H, p[:, 0], p[:, 1], p[:, 2], p[:, 3], p[:, 4], colours(rng, len(p), 160))


def offscreen_scene(rng):
    """Frame-covering splats whose centre is off screen but inside the 1.2 clip bound (|x/w| <= 1.2), plus two just
    outside it (clipped)."""
    W, H = 300, 200
    cx = np.array([1.08 * W, -0.08 * W, 0.5 * W, 1.09 * W, -0.09 * W, 1.11 * W, 0.4 * W])
    cy = np.array([0.5 * H, -0.08 * H, 1.09 * H, 1.09 * H, 1.05 * H, 0.5 * H, -0.11 * H])
    return W, H, splats(W, H, cx, cy, 5.0e4, 1.0e4, 6.0e4, colours(rng, 7, 60))


def stack_scene(rng, n=1500, opaque_from=None):
    """n splats centred on tile (1, 1) of a 64 x 64 frame (one bin), alpha byte 1: the bin holds n records, so the
    raster's ring of chunks wraps several times while the transmittance stays near exp(-n/255).  With opaque_from=k
    the k nearest splats keep alpha byte 2 and every farther one is a huge opaque splat (alpha ~0.997 on the whole
    frame): every pixel dies at the second opaque record, i.e. after nearest-first record k + 1."""
    W, H = 64, 64
    cx = 24.0 + rng.uniform(-2, 2, n)
    cy = 24.0 + rng.uniform(-2, 2, n)
    alpha = np.ones(n, np.uint32)
    s = np.full(n, 60.0)
    if opaque_from is not None:  # distance grows with the index: nearest first is index order
        alpha[:] = 2
        alpha[opaque_from:] = 255
        s[opaque_from:] = 2.0e4
    return W, H, splats(W, H, cx, cy, s, 0.3 * s, 1.1 * s, colours(rng, n, alpha))
