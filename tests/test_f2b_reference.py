"""CPU tests of the front-to-back raster reference (orc_render_f2b in oracle/gs_oracle.c), which restates the CUDA
raster's numeric model (DESIGN.md §3) and brackets its early stop.  Pinned here by: the back-to-front oracle (with
the stop disabled the two composite the same pairs, and front-to-back equals back-to-front algebraically, SURVEY A.5),
an independent brute-force numpy restatement, the bracket's own invariants and an analytic single splat."""
import os

import numpy as np
import pytest

import splat_cases as S
from conftest import scene_inputs

GOLD = os.path.join(os.path.dirname(__file__), "golden")
T_STOP = 3e-4


def _composite(f2b, bg):
    """{R, G, B, T} + background -> RGBA, as the kernel's store: out = C + bg T, A = 1 - T + bg.a T."""
    T = f2b[..., 3:4]
    bg = np.asarray(bg, np.float64)
    return np.concatenate([f2b[..., :3] + bg[:3] * T, 1.0 - T + bg[3] * T], axis=-1)


def _no_stop_matches_back_to_front(orc, cs, cc, order, fr, w, h, bg=(0, 0, 0, 0), depth=None):
    exp, st = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=bg, depth_in=depth)
    e, l, fs = orc.render_f2b(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, t_stop=0.0, depth_in=depth)
    assert np.array_equal(e, l) and fs["hits_eager"] == fs["hits_lazy"] and fs["n_differ"] == 0
    assert fs["hits_eager"] == st["fragments"] > 0
    err = np.abs(_composite(e, bg) - exp).max()
    assert err <= 1e-5, err
    return st


def test_no_stop_equals_back_to_front_golden(gs, orc):
    g = np.load(os.path.join(GOLD, "scene64.npz"))
    cs, cc, m = orc.pack(g["rows"])
    fr = gs.FrameInputs(proj=g["proj"], modelview=g["modelview"], view=g["view"], width=int(g["width"]),
                        height=int(g["height"]), focal=float(g["focal"]))
    _no_stop_matches_back_to_front(orc, cs, cc, g["order"], fr, fr.width, fr.height)
    g2 = np.load(os.path.join(GOLD, "scene20k.npz"))
    cs, cc, m = orc.pack(gs.synth_splats(int(g2["n"]), int(g2["seed"])))
    fr2 = gs.FrameInputs(proj=g2["proj"], modelview=g2["modelview"], view=g2["view"], width=int(g2["width"]),
                         height=int(g2["height"]), focal=float(g2["focal"]))
    _no_stop_matches_back_to_front(orc, cs, cc, g2["order"], fr2, fr2.width, fr2.height)


def test_no_stop_equals_back_to_front_depth_and_background(gs, orc):
    w, h = 200, 120
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 8000, 91, w, h)
    order = orc.sort(m, fr.view)
    _no_stop_matches_back_to_front(orc, cs, cc, order, fr, w, h, bg=(0.25, 0.5, 0.75, 0.5))
    p = orc.project(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal)
    zw = (p["zndc"][p["visible"] == 1] * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    depth = np.empty((h, w), np.float32)
    depth[:, : w // 2] = np.median(zw)
    depth[:, w // 2:] = np.linspace(zw.min(), zw.max(), w - w // 2, dtype=np.float32)[None, :]
    st = _no_stop_matches_back_to_front(orc, cs, cc, order, fr, w, h, bg=(0.1, 0.2, 0.3, 1.0), depth=depth)
    _, st_all = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal)
    assert st["fragments"] < st_all["fragments"]


# ---- brute-force numpy restatement: every splat against every pixel, nearest first ----

def _fma32(a, b, c):
    """fmaf on float32 arrays: a*b is exact in fp64; the fp64 sum is corrected to one rounding with TwoSum."""
    a, b, c = (np.asarray(v, np.float32).astype(np.float64) for v in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)  # exact: p + c = s + err
    r = s.astype(np.float32)
    # s rounds to fp32 like p + c unless s sits exactly halfway between two floats and err breaks the tie
    toward = np.where(s > r.astype(np.float64), np.float32(np.inf), np.float32(-np.inf)).astype(np.float32)
    nb = np.nextafter(r, toward)
    half = (r.astype(np.float64) + nb.astype(np.float64)) * 0.5 == s
    tie = half & (err != 0)
    up = np.maximum(r, nb)
    dn = np.minimum(r, nb)
    return np.where(tie, np.where(err > 0, up, dn), r).astype(np.float32)


def _np_f2b(recs, rgba, w, h, t_stop, depth=None, exact=False):
    """recs: oracle records in draw order (back to front); rgba: their packed colour words."""
    u = 2.0 ** -24 + 2.0 ** -50
    s = float(np.float32(t_stop))
    ys, xs = np.mgrid[0:h, 0:w]
    fx = xs.astype(np.float32) + np.float32(0.5)
    fy = ys.astype(np.float32) + np.float32(0.5)
    state = {k: np.zeros((h, w, 4)) for k in ("e", "l")}
    for k in state:
        state[k][..., 3] = 1.0
    hits = {k: np.zeros((h, w), np.int64) for k in ("e", "l")}
    live = {k: np.ones((h, w), bool) for k in ("e", "l")}
    M = np.zeros((h, w))
    for j in range(len(recs) - 1, -1, -1):
        r = recs[j]
        if r["visible"] != 1:
            continue
        dx = (fx - r["cx"]).astype(np.float32)
        dy = (fy - r["cy"]).astype(np.float32)
        px = _fma32(dy, r["a2y"], (dx * r["a2x"]).astype(np.float32))
        py = _fma32(dy, r["a1y"], (dx * r["a1x"]).astype(np.float32))
        r2 = _fma32(py, py, (px * px).astype(np.float32))
        cov = (r2 <= np.float32(4.0)) & live["l"]
        if depth is not None:
            cov &= np.float32(r["zndc"] * np.float32(0.5) + np.float32(0.5)) <= depth
        if not cov.any():
            continue
        c = np.array([(rgba[j] >> (8 * i)) & 255 for i in range(4)], np.float64) / 255.0
        a = np.exp(-r2.astype(np.float64)) * c[3]
        for k in ("l", "e"):
            m = cov & live[k]
            wgt = a * state[k][..., 3]
            for ch in range(3):
                state[k][..., ch] = np.where(m, state[k][..., ch] + c[ch] * wgt, state[k][..., ch])
            state[k][..., 3] = np.where(m, state[k][..., 3] - wgt, state[k][..., 3])
            hits[k] += m
        if t_stop <= 0:
            continue
        if not exact:
            ex = (2.0 + np.floor(1.173 * r2.astype(np.float64))) * 2.0 * u
            eta = (1.0 + ex) * (1.0 + u) ** 3 - 1.0
            with np.errstate(divide="ignore", invalid="ignore"):
                Mn = np.where(a >= 1.0, np.inf, (1.0 + M) * (1.0 + a * eta / (1.0 - a)) * (1.0 + u) - 1.0)
            M = np.where(cov, Mn, M)
        with np.errstate(divide="ignore"):
            live["e"] &= ~(cov & ((M >= 1.0) | (state["l"][..., 3] < s / (1.0 - M))))
        live["l"] &= ~(cov & (state["l"][..., 3] < s / (1.0 + M)))
    return state["e"], state["l"], int(hits["e"].sum()), int(hits["l"].sum()), int((hits["e"] != hits["l"]).sum())


def _small_scenes(gs, orc):
    rng = np.random.default_rng(7)
    P, MV = S.camera()
    # a deep opaque stack over half of the frame, a translucent stack, and needles / tangent footprints around it
    n = 200
    W, H = 64, 48
    deep = S.splats(W, H, 30.0 + rng.uniform(-3, 3, n), 24.0 + rng.uniform(-3, 3, n), 40.0, 8.0, 50.0,
                    S.colours(rng, n, rng.integers(200, 256, n)), zd=5.0 + 1e-3 * np.arange(n))
    thin = S.splats(W, H, rng.uniform(0, W, 150), rng.uniform(0, H, 150), rng.uniform(1, 30, 150), rng.uniform(-5, 5, 150),
                    rng.uniform(2, 40, 150), S.colours(rng, 150, rng.integers(1, 60, 150)), zd=4.0 + 1e-3 * np.arange(150))
    tang = S.splats(W, H, 5.5 + np.arange(40) / 8.0, 40.5 - np.arange(40) / 8.0, 9 / 8 - 0.3, 0.0, 4.2,
                    S.colours(rng, 40, 128), zd=4.5 + 1e-3 * np.arange(40))
    cs, cc, sa = S.cat(deep, thin, tang)
    order = orc.sort_compact(cs, sa, S.VIEW)
    yield "deep_stack", cs, cc, order, P, MV, W, H, S.FOCAL
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 500, 4242, 48, 40)
    yield "synth500", cs, cc, orc.sort(m, fr.view), fr.proj, fr.modelview, 48, 40, fr.focal


@pytest.mark.parametrize("t_stop,exact", [(T_STOP, False), (T_STOP, True), (0.0, False), (0.02, False)])
def test_matches_brute_force_numpy(gs, orc, t_stop, exact):
    for name, cs, cc, order, P, MV, W, H, focal in _small_scenes(gs, orc):
        recs = orc.project(cs, cc, order, P, MV, W, H, focal)
        rgba = cc[order, 3]
        ne, nl, nhe, nhl, ndiff = _np_f2b(recs, rgba, W, H, t_stop, exact=exact)
        e, l, st = orc.render_f2b(cs, cc, order, P, MV, W, H, focal, t_stop=t_stop, exact=exact)
        assert (st["hits_eager"], st["hits_lazy"], st["n_differ"]) == (nhe, nhl, ndiff), name
        assert np.abs(e - ne).max() <= 1e-12 and np.abs(l - nl).max() <= 1e-12, name
        if t_stop == T_STOP and name == "deep_stack":
            assert (ne[..., 3] < T_STOP).any()  # the stop acts in this scene


def test_brute_force_with_depth(gs, orc):
    name, cs, cc, order, P, MV, W, H, focal = next(_small_scenes(gs, orc))
    recs = orc.project(cs, cc, order, P, MV, W, H, focal)
    zw = (recs["zndc"] * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    depth = np.full((H, W), np.median(zw[recs["visible"] == 1]), np.float32)
    depth[:, W // 2:] = np.nextafter(depth[:, W // 2:], np.float32(0))
    ne, nl, nhe, nhl, ndiff = _np_f2b(recs, cc[order, 3], W, H, T_STOP, depth=depth)
    e, l, st = orc.render_f2b(cs, cc, order, P, MV, W, H, focal, depth_in=depth)
    assert (st["hits_eager"], st["hits_lazy"]) == (nhe, nhl) and np.abs(e - ne).max() <= 1e-12


@pytest.mark.parametrize("case", ["synth", "stack", "opaque_stack", "needles", "offscreen"])
def test_bracket_invariants(gs, orc, case):
    """eager <= lazy; the exact fp64 stop rule lies between them; C grows and T shrinks from the no-stop frame's view."""
    rng = np.random.default_rng(11)
    P, MV = S.camera()
    focal = S.FOCAL
    if case == "synth":
        w, h = 320, 180
        rows, cs, cc, m, fr = scene_inputs(gs, orc, 30000, 12, w, h)
        order, P, MV, focal = orc.sort(m, fr.view), fr.proj, fr.modelview, fr.focal
    else:
        w, h, (cs, cc, sa) = {"stack": lambda: S.stack_scene(rng, 400), "opaque_stack": lambda: S.stack_scene(rng, 400, 126),
                              "needles": lambda: S.needle_scene(rng), "offscreen": lambda: S.offscreen_scene(rng)}[case]()
        order = orc.sort_compact(cs, sa, S.VIEW)
    e, l, st = orc.render_f2b(cs, cc, order, P, MV, w, h, focal)
    x, x2, xs = orc.render_f2b(cs, cc, order, P, MV, w, h, focal, exact=True)
    full, _, fst = orc.render_f2b(cs, cc, order, P, MV, w, h, focal, t_stop=0.0)
    assert np.array_equal(x, x2) and xs["hits_eager"] == xs["hits_lazy"]
    assert st["hits_eager"] <= xs["hits_eager"] <= st["hits_lazy"] <= fst["hits_eager"]
    assert st["n_differ"] <= max(4, 1e-3 * w * h)
    for lo, mid, hi in ((e, x, l), (l, full, full)):
        assert np.all(lo[..., :3] <= mid[..., :3] + 1e-12) and np.all(mid[..., :3] <= hi[..., :3] + 1e-12)
        assert np.all(lo[..., 3] >= mid[..., 3] - 1e-12) and np.all(mid[..., 3] >= hi[..., 3] - 1e-12)
    # lazy stops only below the threshold, so what it leaves out (at most its T per channel) is below it too
    assert np.abs(l - full).max() <= float(np.float32(T_STOP))
    assert np.all(l[..., 3] >= 0) and np.all(e[..., :3] >= 0)


def test_single_splat_analytic_fp64(orc):
    """One axis-aligned splat (as test_render_single_splat_analytic): the reference's alpha is exp(-r2) * a computed
    from the fp32 r2 the kernel evaluates, so away from the r2 = 4 contour it equals the analytic Gaussian to the
    quantisation of the packed covariance and fp32 geometry (~1e-6), 200x tighter than the fp32 oracle's check."""
    W, H = 64, 64
    scale = np.float32(0.01 / 32767.0)
    cs = np.array([[0, 0, -5.0, scale]], np.float32)
    q = lambda v: np.uint32(np.int16(v).view(np.uint16))
    s00 = 20970
    cc = np.zeros((1, 4), np.uint32)
    cc[0, 0] = q(s00)
    cc[0, 1] = q(32767) << 16
    cc[0, 2] = q(32767) << 16
    cc[0, 3] = 255 | (128 << 8) | (0 << 16) | (255 << 24)
    P = np.zeros(16, np.float32); P[0] = 1.0; P[5] = -1.0; P[10] = -1.0; P[11] = -1.0; P[14] = -0.02
    MV = np.eye(4, dtype=np.float32).reshape(16)
    focal = 200.0
    e, l, st = orc.render_f2b(cs, cc, np.array([0], np.uint32), P, MV, W, H, focal)
    k = (focal / 5.0) ** 2
    sx2 = float(np.float32(s00) * scale) * k + 0.3
    sy2 = float(np.float32(32767) * scale) * k + 0.3
    ys, xs = np.mgrid[0:H, 0:W]
    r2 = (xs + 0.5 - 32.0) ** 2 / (2 * sx2) + (ys + 0.5 - 32.0) ** 2 / (2 * sy2)
    exp_a = np.where(r2 <= 4.0, np.exp(-r2), 0.0)
    safe = np.abs(r2 - 4.0) > 1e-4  # pixels on the r2 == 4 contour may flip under fp32 rounding
    assert np.array_equal(e, l) and st["hits_eager"] == st["hits_lazy"] and st["n_differ"] == 0
    assert int((r2 <= 4.0)[safe].sum()) <= st["hits_eager"] <= int(((r2 <= 4.0) | ~safe).sum())
    assert np.abs(1.0 - e[..., 3] - exp_a)[safe].max() <= 2e-6
    assert np.abs(e[..., 0] - exp_a)[safe].max() <= 2e-6
    assert np.abs(e[..., 1] - exp_a * (128 / 255))[safe].max() <= 2e-6
    assert np.all(e[..., 2] == 0)
