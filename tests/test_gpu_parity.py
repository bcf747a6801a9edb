"""GPU parity tests (run with -m gpu on a B200): every call goes through the C ABI (ctypes ->
libgsplat_b200.so) and is compared with the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.md "Parity gate"):
  sort / pack  : bit-exact (uint32 index array, packed records)
  projection   : bit-exact on centre and footprint basis (same fp32 op order, no FMA contraction)
  frames       : per-channel abs error <= 1e-3 on float RGBA in [0,1]; <= 1 LSB on >= 99.9 % of RGBA8 pixels
                 and <= 2 LSB everywhere
"""
import os

import numpy as np
import pytest

from conftest import scene_inputs

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
FRAME_TOL = 1e-3


def _load(ctx, cs, cc, m):
    ctx.clear()
    ctx.push_packed(cs, cc, m[:, 15])


def test_pack_exact(gs, orc, ctx):
    rows = gs.synth_splats(300000, 31)
    cs, cc, m = orc.pack(rows)
    ctx.clear()
    ctx.push_splats(rows[:100000])
    ctx.push_splats(rows[100000:])  # progressive push (index.js:259-298)
    assert ctx.num_splats == len(rows)
    gcs, gcc, gsa = ctx.read_packed()
    assert np.array_equal(gcs.view(np.uint32), cs.view(np.uint32))
    assert np.array_equal(gcc, cc)
    assert np.array_equal(gsa.view(np.uint32), m[:, 15].view(np.uint32))


def test_pack_quirks_exact(orc, ctx):
    """Q1 non-unit quaternions, Q2 parseInt exponent form, Q3 truncation, zero scales -> NaN -> 0."""
    rng = np.random.default_rng(5)
    n = 4096
    rows = np.zeros((n, 32), np.uint8)
    f = np.zeros((n, 6), np.float32)
    f[:, :3] = rng.normal(size=(n, 3))
    f[:, 3:] = np.exp(rng.normal(-3, 2, size=(n, 3)))
    f[:64, 3:] = 0.0            # all-zero scales
    f[64:128, 3:] = 0.05        # isotropic: off-diagonals cancel to ~1e-19 residues -> exponent-form strings
    rows[:, :24] = f.view(np.uint8).reshape(n, 24)
    rows[:, 24:32] = rng.integers(0, 256, size=(n, 8), dtype=np.uint8)
    rows[128:192, 28:32] = [255, 128, 128, 128]  # identity-ish rotation
    cs, cc, m = orc.pack(rows)
    ctx.clear()
    ctx.push_splats(rows)
    gcs, gcc, gsa = ctx.read_packed()
    assert np.array_equal(gcs.view(np.uint32), cs.view(np.uint32))
    assert np.array_equal(gcc, cc)
    assert np.array_equal(gsa.view(np.uint32), m[:, 15].view(np.uint32))


@pytest.mark.parametrize("n,cutout", [(1, False), (37, False), (4096, False), (4097, True), (250000, False), (250000, True)])
def test_sort_exact(gs, orc, ctx, n, cutout):
    rows, cs, cc, m, fr = scene_inputs(gs, orc, n, 100 + n, 1920, 1080, cutout=cutout)
    _load(ctx, cs, cc, m)
    got = ctx.sort(fr.view, fr.cutout)
    exp = orc.sort(m, fr.view, fr.cutout)
    assert got.dtype == np.uint32 and len(got) == len(exp)
    assert np.array_equal(got, exp)
    st = ctx.stats()
    assert st["n_sorted"] == len(exp) and st["n_splats"] == n


def test_sort_exact_orbit_and_ties(gs, orc, ctx):
    """Per-frame re-sort around an orbit (config 3) + a scene with massive key ties (stability by index)."""
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 120000, 7, 1920, 1080)
    _load(ctx, cs, cc, m)
    sc = gs.scenes
    for step in (0, 13, 45, 77, 119):
        f = sc.make_frame(sc.orbit_camera(1920, 1080, step), sc.demo_object(), 1920, 1080)
        assert np.array_equal(ctx.sort(f.view), orc.sort(m, f.view)), step
    # 200k splats on only 5 distinct depths -> huge buckets, order inside a bucket must be the index order
    n = 200000
    m2 = np.zeros((n, 16), np.float32)
    m2[:, 12:14] = np.random.default_rng(1).normal(size=(n, 2))
    m2[:, 14] = -1.0 - (np.arange(n) % 5)
    m2[:, 15] = 1.0
    cs2 = np.zeros((n, 4), np.float32); cs2[:, :3] = m2[:, 12:15]
    ctx.clear(); ctx.push_packed(cs2, np.zeros((n, 4), np.uint32), m2[:, 15])
    v = np.array([0, 0, 1, 0], np.float32)
    assert np.array_equal(ctx.sort(v), orc.sort(m2, v))


def test_sort_edge_cases(orc, ctx):
    view = np.array([0, 0, 1, 0], np.float32)

    def run(z, size=1.0, view=view, cut=None, xy=None):
        z = np.asarray(z, np.float32)
        m = np.zeros((len(z), 16), np.float32)
        m[:, 14] = z; m[:, 15] = size
        if xy is not None:
            m[:, 12:14] = xy
        cs = np.zeros((len(z), 4), np.float32); cs[:, :3] = m[:, 12:15]
        ctx.clear(); ctx.push_packed(cs, np.zeros((len(z), 4), np.uint32), m[:, 15])
        got, exp = ctx.sort(view, cut), orc.sort(m, view, cut)
        assert np.array_equal(got, exp), (z[:8], got[:8], exp[:8])
        return got

    assert len(run([1.0, 2.0])) == 0               # Q6: V = 0
    assert np.array_equal(run([-1.0]), [0])        # Q6: V = 1 (depthInv = inf, key NaN -> 0)
    run([-2.0, -2.0, -2.0])                        # all equal
    run([-1.0, -3.0, -2.0, 0.0, -0.0, 1e-30, -1e-30, np.nan, -np.inf])
    run([-1.0, -1.0, -1.0], size=np.array([0.0001, 0.00010001, 0.0], np.float32))
    # Q5: depth range below f32 resolution -> keys outside [0, 65535] are dropped, tail stays 0
    z = -1000.0 - np.arange(4096, dtype=np.float64) * 1e-5
    got = run(z, view=np.array([0, 0, 1, 1e-4], np.float32))
    assert ctx.stats()["n_dropped"] >= 0
    # Q12 cutout faces inclusive, y negated
    cut = np.eye(4, dtype=np.float32).reshape(16)
    run([-0.25] * 4, view=np.array([0, 0, 1, -1], np.float32), cut=cut,
        xy=np.array([[0.5, 0.0], [0.5000001, 0.0], [-0.5, 0.0], [0.0, 0.6]], np.float32))
    # empty context -> GS_ERR_EMPTY (quirk Q7 is not reproduced)
    ctx.clear()
    with pytest.raises(Exception):
        ctx.sort(view)


def _check_projection(gs, orc, ctx, cs, cc, fr, order):
    g = ctx.read_projected()
    ref = orc.project(cs, cc, None, fr.proj, fr.modelview, fr.width, fr.height, fr.focal)
    rect = g[:, 7].copy().view(np.uint32)
    in_order = np.zeros(len(cs), bool)
    in_order[order] = True
    drawn = rect != 0xFFFFFFFF
    # every splat the GPU binned is visible in the oracle and part of the draw order
    assert np.all(ref["visible"][drawn] == 1) and np.all(in_order[drawn] | (np.nonzero(drawn)[0] == 0))
    # visible splats the GPU did not bin have a footprint that misses every pixel centre of the frame
    missing = in_order & (ref["visible"] == 1) & ~drawn
    if missing.any():
        r = ref[missing]
        ex = 2 * np.hypot(r["v1x"], r["v2x"]); ey = 2 * np.hypot(r["v1y"], r["v2y"])
        off = (r["cx"] + ex < 0.5) | (r["cx"] - ex > fr.width - 0.5) | (r["cy"] + ey < 0.5) | (r["cy"] - ey > fr.height - 0.5)
        tiny = (np.ceil(r["cx"] - ex - 0.5) > np.floor(r["cx"] + ex - 0.5)) | (np.ceil(r["cy"] - ey - 0.5) > np.floor(r["cy"] + ey - 0.5))
        assert np.all(off | tiny)
    for k, col in (("cx", 0), ("cy", 1), ("a1x", 2), ("a1y", 3), ("a2x", 4), ("a2y", 5)):
        assert np.array_equal(g[drawn, col].view(np.uint32), ref[k][drawn].view(np.uint32)), k
    return drawn.sum()


@pytest.mark.parametrize("n,w,h,cutout,fmt", [
    (64, 256, 144, False, "f32"), (20000, 256, 144, False, "f32"), (20000, 250, 141, True, "f32"),
    (4099, 250, 141, True, "f32"),  # sparse-frame projection path (cutout keeps < half), chunk tail not a multiple of 4
    (150000, 1920, 1080, False, "f32"), (150000, 1920, 1080, False, "u8"), (60000, 3840, 2160, True, "u8"),
])
def test_render_parity(gs, orc, ctx, n, w, h, cutout, fmt):
    rows, cs, cc, m, fr = scene_inputs(gs, orc, n, 500 + n, w, h, cutout=cutout)
    _load(ctx, cs, cc, m)
    bg = (0.1, 0.2, 0.3, 0.5)
    order = orc.sort(m, fr.view, fr.cutout)
    exp, est = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=bg)
    if fmt == "f32":
        got = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F)
        err = np.abs(got - exp)
        assert err.max() <= FRAME_TOL, (err.max(), np.unravel_index(err.argmax(), err.shape))
    else:
        got = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA8)
        e8 = np.floor(np.clip(exp, 0, 1) * 255.0 + 0.5).astype(np.int32)
        d = np.abs(got.astype(np.int32) - e8)
        assert d.max() <= 2 and (d <= 1).mean() >= 0.999
        assert (d == 0).mean() > 0.98
    st = ctx.stats()
    assert st["n_sorted"] == len(order) and st["n_instances"] > 0
    assert st["width"] == w and st["height"] == h and st["n_tiles"] == ((w + 15) // 16) * ((h + 15) // 16)
    # V2 counts the draw-order entries with a bin rectangle: the splats the GPU binned, no more than the oracle's visible
    assert st["n_dropped"] == 0 and st["n_visible"] == _check_projection(gs, orc, ctx, cs, cc, fr, order) <= est["n_visible"]


def test_render_golden(gs, orc, ctx):
    g = np.load(os.path.join(GOLD, "scene64.npz"))
    ctx.clear(); ctx.push_splats(g["rows"])
    fr = gs.FrameInputs(proj=g["proj"], modelview=g["modelview"], view=g["view"], width=int(g["width"]), height=int(g["height"]),
                        focal=float(g["focal"]))
    assert np.array_equal(ctx.sort(g["view"]), g["order"])
    assert np.array_equal(ctx.sort(g["view"], g["cutout"]), g["order_cutout"])
    got = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F)
    assert np.abs(got - g["frame"]).max() <= FRAME_TOL
    g2 = np.load(os.path.join(GOLD, "scene20k.npz"))
    ctx.clear(); ctx.push_splats(gs.synth_splats(int(g2["n"]), int(g2["seed"])))
    fr2 = gs.FrameInputs(proj=g2["proj"], modelview=g2["modelview"], view=g2["view"], width=int(g2["width"]), height=int(g2["height"]),
                         focal=float(g2["focal"]))
    assert np.array_equal(ctx.sort(g2["view"]), g2["order"])
    got = ctx.render(fr2, fmt=gs.GS_FORMAT_RGBA32F)
    assert np.abs(got - g2["frame"].astype(np.float32)).max() <= FRAME_TOL + 1e-3  # golden frame stored as float16


def test_render_q5_tail_zero_draws_splat0(gs, orc, ctx):
    """Q5 in the draw: dropped keys leave zeros at the END of sortedIndexes, so the reference draws splat 0 again,
    front-most.  The GPU path must composite the same thing."""
    n = 512
    rng = np.random.default_rng(3)
    cs = np.zeros((n, 4), np.float32)
    cs[:, 0] = rng.uniform(-0.3, 0.3, n); cs[:, 1] = rng.uniform(-0.2, 0.2, n)
    cs[:, 2] = (-1000.0 - np.arange(n, dtype=np.float64) * 1e-5).astype(np.float32)
    cs[:, 3] = 30.0 / 32767.0
    cc = np.zeros((n, 4), np.uint32)
    q = lambda v: np.uint32(np.int16(v).view(np.uint16))
    cc[:, 0] = q(20000); cc[:, 1] = q(32767) << 16; cc[:, 2] = q(32767) << 16
    cc[:, 3] = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32) | np.uint32(0x60000000)
    sa = np.ones(n, np.float32)
    m = np.zeros((n, 16), np.float32); m[:, 12:15] = cs[:, :3]; m[:, 15] = sa
    W, H = 128, 96
    P = np.zeros(16, np.float32); P[0] = 1.0; P[5] = -1.3; P[10] = -1.0; P[11] = -1.0; P[14] = -0.02
    MV = np.eye(4, dtype=np.float32).reshape(16); MV[14] = 1e-4
    view = np.array([MV[2], MV[6], MV[10], MV[14]], np.float32)
    order = orc.sort(m, view)
    ctx.clear(); ctx.push_packed(cs, cc, sa)
    assert np.array_equal(ctx.sort(view), order)
    fr = gs.FrameInputs(proj=P, modelview=MV, view=view, width=W, height=H, focal=400.0)
    exp, _ = orc.render(cs, cc, order, P, MV, W, H, 400.0)
    got = ctx.render(fr, fmt=1)
    assert ctx.stats()["n_dropped"] > 0 and (order == 0).sum() >= 2  # zero tail present
    assert np.abs(got - exp).max() <= FRAME_TOL


def test_render_reuse_sort_and_stale_order(gs, orc, ctx):
    """GS_RENDER_REUSE_SORT draws with the previous order (index.js:206,439-440: the draw may use a stale sort)."""
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 30000, 9, 512, 288)
    _load(ctx, cs, cc, m)
    sc = gs.scenes
    fr2 = sc.make_frame(sc.orbit_camera(512, 288, 3), sc.demo_object(), 512, 288)
    order1 = ctx.sort(fr.view)  # sort with camera 1 ...
    got = ctx.render(fr2, fmt=gs.GS_FORMAT_RGBA32F, reuse_sort=True)  # ... draw with camera 2
    exp, _ = orc.render(cs, cc, order1, fr2.proj, fr2.modelview, 512, 288, fr2.focal)
    assert np.abs(got - exp).max() <= FRAME_TOL
    got_sync = ctx.render(fr2, fmt=gs.GS_FORMAT_RGBA32F)
    exp_sync, _ = orc.render(cs, cc, orc.sort(m, fr2.view), fr2.proj, fr2.modelview, 512, 288, fr2.focal)
    assert np.abs(got_sync - exp_sync).max() <= FRAME_TOL


def test_render_async_pipeline(gs, orc, ctx):
    """gs_render_async / gs_wait: two frames in flight, different cameras, pinned and pageable destinations; every
    frame must equal the synchronous gs_render of the same inputs bit for bit (same kernels, same order)."""
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 40000, 10, 640, 360)
    _load(ctx, cs, cc, m)
    sc = gs.scenes
    frames = [sc.make_frame(sc.orbit_camera(640, 360, s), sc.demo_object(), 640, 360) for s in (0, 7, 31, 64, 90)]
    ref = [ctx.render(f, fmt=gs.GS_FORMAT_RGBA8).copy() for f in frames]
    outs = [ctx.pinned_array((360, 640, 4), np.uint8) if i % 2 == 0 else np.empty((360, 640, 4), np.uint8) for i in range(len(frames))]
    tickets = []
    for i, f in enumerate(frames):
        outs[i][...] = 0
        tickets.append(ctx.render_async(ctx.make_params(f, fmt=gs.GS_FORMAT_RGBA8), outs[i].ctypes.data))
        if i >= 1:
            st = ctx.wait(tickets[i - 1])
            bs = ctx._lib.gs_bin_size()
            n_bins = -(-640 // bs) * -(-360 // bs)
            by_entry = os.environ.get("GS_EMIT", "entries") != "windows"  # emission by entry adds k_radix_hist<T1>
            assert st.n_sorted > 0 and st.kernel_launches == (13 if n_bins <= 256 else 17) + (1 if by_entry else 0)
            assert np.array_equal(outs[i - 1], ref[i - 1])
    ctx.wait(tickets[-1])
    assert np.array_equal(outs[-1], ref[-1])
    # a third submit without waiting recycles the oldest slot implicitly
    t0 = ctx.render_async(ctx.make_params(frames[0], fmt=gs.GS_FORMAT_RGBA8), outs[0].ctypes.data)
    t1 = ctx.render_async(ctx.make_params(frames[1], fmt=gs.GS_FORMAT_RGBA8), outs[1].ctypes.data)
    t2 = ctx.render_async(ctx.make_params(frames[2], fmt=gs.GS_FORMAT_RGBA8), outs[2].ctypes.data)
    for t in (t0, t1, t2):
        ctx.wait(t)
    assert all(np.array_equal(outs[i], ref[i]) for i in range(3))
    with pytest.raises(Exception):
        ctx.wait(t2 + 5)
    # four tickets open at once (sort | bin | raster | copy to the host); a fifth and sixth submit recycle the oldest
    # slots implicitly, and waiting on a ticket retired that way still returns GS_OK with the frame in place
    for o in outs:
        o[...] = 0
    ts = [ctx.render_async(ctx.make_params(frames[i], fmt=gs.GS_FORMAT_RGBA8), outs[i].ctypes.data) for i in range(5)]
    extra = ctx.pinned_array((360, 640, 4), np.uint8)
    ts.append(ctx.render_async(ctx.make_params(frames[2], fmt=gs.GS_FORMAT_RGBA8), extra.ctypes.data))
    for t in reversed(ts):
        ctx.wait(t)
    assert all(np.array_equal(outs[i], ref[i]) for i in range(5)) and np.array_equal(extra, ref[2])
    # the oracle agrees with what the pipeline produced
    exp, _ = orc.render(cs, cc, orc.sort(m, frames[3].view), frames[3].proj, frames[3].modelview, 640, 360, frames[3].focal)
    e8 = np.floor(np.clip(exp, 0, 1) * 255.0 + 0.5).astype(np.int32)
    assert np.abs(outs[3].astype(np.int32) - e8).max() <= 2


def test_render_instance_overflow_regrows(gs, orc, ctx, monkeypatch):
    """Huge splats touch every tile: the instance buffer overflows, is regrown and the frame re-run."""
    n = 8000
    rows = gs.synth_splats(n, 77, log_scale_mean=-0.5)
    cs, cc, m = orc.pack(rows)
    monkeypatch.setenv("GS_INST_CAP", "50000")  # initial instance capacity (read when the first frame sizes its buffers)
    with gs.SplatContext(0) as c2:
        c2.push_packed(cs, cc, m[:, 15])
        sc = gs.scenes
        fr = sc.make_frame(sc.fixed_camera(1920, 1080), sc.demo_object(), 1920, 1080)
        got = c2.render(fr, fmt=gs.GS_FORMAT_RGBA32F)
        st = c2.stats()
        assert st["n_instances"] > 50000
        exp, _ = orc.render(cs, cc, orc.sort(m, fr.view), fr.proj, fr.modelview, 1920, 1080, fr.focal)
        assert np.abs(got - exp).max() <= FRAME_TOL


def test_async_overflow_three_in_flight(gs, orc, monkeypatch):
    """ADVICE r1: three frames in flight all see the too-small instance buffer.  The first gs_wait must regrow ONCE to
    the measured demand, the frames must be re-run in submission order, and every frame must equal its synchronous
    render; a following REUSE_SORT frame must use the LAST submitted frame's order."""
    n = 8000
    rows = gs.synth_splats(n, 78, log_scale_mean=-0.5)
    cs, cc, m = orc.pack(rows)
    sc = gs.scenes
    W, H = 1920, 1080
    frames = [sc.make_frame(sc.orbit_camera(W, H, s), sc.demo_object(), W, H) for s in (0, 3, 6)]
    with gs.SplatContext(0) as ref:
        ref.push_packed(cs, cc, m[:, 15])
        exp = [ref.render(f, fmt=gs.GS_FORMAT_RGBA8).copy() for f in frames]
        demand = ref.stats()["n_instances"]
        exp_reuse = ref.render(frames[0], fmt=gs.GS_FORMAT_RGBA8, reuse_sort=True).copy()  # camera 0 drawn with frame 2's order
    assert demand > 100000
    monkeypatch.setenv("GS_INST_CAP", "50000")
    with gs.SplatContext(0) as c2:
        c2.push_packed(cs, cc, m[:, 15])
        outs = [c2.pinned_array((H, W, 4), np.uint8) for _ in frames]
        tickets = [c2.render_async(c2.make_params(f, fmt=gs.GS_FORMAT_RGBA8), o.ctypes.data) for f, o in zip(frames, outs)]
        for t in tickets:
            st = c2.wait(t)
        assert st.n_instances > 50000
        for o, e in zip(outs, exp):
            assert np.array_equal(o, e)
        got_reuse = c2.render(frames[0], fmt=gs.GS_FORMAT_RGBA8, reuse_sort=True)
        assert np.array_equal(got_reuse, exp_reuse)
        # waiting out of order works too (the older frames are finished first)
        tickets = [c2.render_async(c2.make_params(f, fmt=gs.GS_FORMAT_RGBA8), o.ctypes.data) for f, o in zip(frames, outs)]
        c2.wait(tickets[2]); c2.wait(tickets[0]); c2.wait(tickets[1])
        for o, e in zip(outs, exp):
            assert np.array_equal(o, e)


def test_full_size_properties(gs, ctx):
    """BASELINE config sizes (1 M splats, 1920x1080): size-independent properties instead of an oracle run."""
    n = 1_000_000
    rows = gs.synth_splats(n, 0x5EED0002)
    ctx.clear(); ctx.push_splats(rows)
    sc = gs.scenes
    fr = sc.make_frame(sc.fixed_camera(1920, 1080), sc.demo_object(), 1920, 1080)
    order = ctx.sort(fr.view)
    cs, cc, sa = ctx.read_packed()
    # (a) the order is a set of distinct valid indices, (b) keys non-decreasing, (c) ties in index order,
    # (d) exactly the splats passing the filter are present
    assert len(np.unique(order)) == len(order) and order.max() < n
    v = fr.view.astype(np.float64)
    depth_all = ((v[0] * cs[:, 0].astype(np.float64) + v[1] * cs[:, 1]) + v[2] * cs[:, 2]) + v[3]
    keep = (depth_all < 0) & (sa.astype(np.float64) > -0.0001 * depth_all)
    assert len(order) == int(keep.sum()) and np.all(keep[order])
    d = depth_all[order]
    key = np.trunc((d.astype(np.float32).astype(np.float64) - d.min()) * (65535.0 / (d.max() - d.min()))).astype(np.int64)
    assert np.all(np.diff(key) >= 0)
    assert np.all(np.diff(order.astype(np.int64))[np.diff(key) == 0] > 0)
    # (e) idempotence + (f) alpha/colour bounds of the composite, (g) RGBA8 == quantised RGBA32F within 1 LSB
    f32 = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F)
    f32b = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F)
    assert np.array_equal(f32, f32b)
    assert f32.min() >= 0 and f32.max() <= 1.0 + 1e-5
    u8 = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA8)
    assert np.abs(u8.astype(np.int32) - np.floor(np.clip(f32, 0, 1) * 255 + 0.5).astype(np.int32)).max() <= 1
    # (h) compositing over a background is affine in the background: frame(bg) = frame(0) + bg * (1 - alpha)
    fb = ctx.render(fr, bg=(1.0, 0.5, 0.25, 1.0), fmt=gs.GS_FORMAT_RGBA32F)
    T = 1.0 - f32[..., 3]
    assert np.allclose(fb[..., 0], f32[..., 0] + T, atol=2e-6) and np.allclose(fb[..., 3], 1.0, atol=2e-6)
    st = ctx.stats()
    assert st["n_splats"] == n and st["n_instances"] > st["n_visible"] > 0


def test_sort_exact_random_regimes(orc, ctx):
    """Bit-exact sort over the regimes that stress the fp64 / ToInt32 restatement: heavy ties, depth ranges below f32
    resolution (keys wrap or leave [0, 65535], quirk Q5), 40 decades of magnitudes, tricky view vectors, cutouts."""
    tricky = [0.0, -0.0, 1e-30, -1e-30, 1e-45, 1.0, -1.0, 3.4e38, -3.4e38, 1e-6, 65535.0, 0.5]
    for seed in range(24):
        rng = np.random.default_rng(1000 + seed)
        n = int(rng.integers(1, 30000))
        mode = ["random", "ties", "narrow", "wide"][seed % 4]
        m = np.zeros((n, 16), np.float32)
        if mode == "random":
            m[:, 12:15] = rng.normal(0, 5, (n, 3))
        elif mode == "ties":
            m[:, 12:15] = rng.integers(-2, 3, (n, 3))
        elif mode == "narrow":
            m[:, 12:15] = 1000.0 + rng.normal(0, 1e-5, (n, 3))
        else:
            m[:, 12:15] = rng.normal(0, 1, (n, 3)) * 10.0 ** rng.integers(-20, 20, (n, 1))
        m[:, 15] = np.abs(rng.normal(0, 1, n)) * rng.integers(0, 2, n)
        view = rng.normal(0, 1, 4).astype(np.float32)
        if seed % 3 == 0:
            view[rng.integers(0, 4)] = tricky[seed % len(tricky)]
        cut = None
        if seed % 2:
            c = np.eye(4, dtype=np.float32)
            c[:3, :3] *= rng.uniform(0.05, 2.0, 3).astype(np.float32)
            c[3, :3] = rng.normal(0, 1, 3)
            cut = c.reshape(16)
        cs = np.zeros((n, 4), np.float32); cs[:, :3] = m[:, 12:15]
        ctx.clear(); ctx.push_packed(cs, np.zeros((n, 4), np.uint32), m[:, 15])
        got, exp = ctx.sort(view, cut), orc.sort(m, view, cut)
        assert np.array_equal(got, exp), (seed, mode, n, len(got), len(exp))
