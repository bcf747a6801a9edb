"""GPU tests of the draw's optional features through the C ABI: depth interop (index.js:179-180), the two pixel loops
of the raster (packed fp32x2 / scalar) producing identical frames, and the GS_RENDER_STATS counters."""
import os

import numpy as np
import pytest

from conftest import scene_inputs

pytestmark = pytest.mark.gpu
FRAME_TOL = 1e-3


def _depth_plane(orc, cs, cc, order, fr, w, h):
    """A depth buffer that splits the scene: left half at the median splat depth, a ramp on the right, far plane in a
    corner block (so that all three regimes - everything rejected, partially rejected, nothing rejected - occur)."""
    p = orc.project(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal)
    zw = (p["zndc"][p["visible"] == 1] * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    lo, mid, hi = np.percentile(zw, [5, 50, 95]).astype(np.float32)
    d = np.empty((h, w), np.float32)
    d[:, : w // 2] = mid
    d[:, w // 2:] = np.linspace(lo, hi, w - w // 2, dtype=np.float32)[None, :]
    d[: h // 4, : w // 4] = 1.0
    d[-h // 4:, -w // 4:] = 0.0
    return d


@pytest.mark.parametrize("n,w,h", [(20000, 256, 144), (120000, 1000, 562)])
def test_depth_interop_parity(gs, orc, ctx, n, w, h):
    rows, cs, cc, m, fr = scene_inputs(gs, orc, n, 900 + n, w, h)
    ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
    order = orc.sort(m, fr.view)
    depth = _depth_plane(orc, cs, cc, order, fr, w, h)
    bg = (0.3, 0.2, 0.1, 1.0)
    exp, est = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=bg, depth_in=depth)
    base, bst = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=bg)
    assert 0 < est["fragments"] < bst["fragments"]
    got = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F, depth_in=depth)
    err = np.abs(got - exp)
    assert err.max() <= FRAME_TOL, (float(err.max()), np.unravel_index(err.argmax(), err.shape))
    # the block at depth 0 shows only the background, the block at depth 1 equals the frame without a depth buffer
    assert np.allclose(got[-h // 4:, -w // 4:], bg, atol=1e-6)
    plain = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F)
    assert np.array_equal(got[: h // 4, : w // 4], plain[: h // 4, : w // 4])
    # device-resident depth buffer (GS_RENDER_DEPTH_DEVICE) gives the same frame
    import torch
    t = torch.from_numpy(depth).cuda()
    torch.cuda.synchronize()
    p = ctx.make_params(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F, flags=gs.GS_RENDER_DEPTH_DEVICE)
    p.depth_in = t.data_ptr()
    out = np.empty((h, w, 4), np.float32)
    ctx.render_raw(p, out.ctypes.data)
    assert np.array_equal(out, got)
    # RGBA8 output of the depth-tested frame
    got8 = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA8, depth_in=depth)
    e8 = np.floor(np.clip(exp, 0, 1) * 255.0 + 0.5).astype(np.int32)
    assert np.abs(got8.astype(np.int32) - e8).max() <= 2


def test_packed_and_scalar_pixel_loops_agree(gs, orc):
    """GS_RASTER=scalar selects the one-pixel-per-lane loop; the default is the packed fp32x2 loop.  Same operations in
    the same order per pixel -> bit-identical frames (float and RGBA8, with and without a depth buffer)."""
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 150000, 4321, 1000, 562)
    order = orc.sort(m, fr.view)
    depth = _depth_plane(orc, cs, cc, order, fr, 1000, 562)
    frames = {}
    old = os.environ.get("GS_RASTER")
    try:
        for mode in ("scalar", "packed"):
            os.environ["GS_RASTER"] = mode
            with gs.SplatContext(0) as c:
                c.push_packed(cs, cc, m[:, 15])
                frames[mode] = (c.render(fr, fmt=gs.GS_FORMAT_RGBA32F, bg=(0.1, 0.2, 0.3, 0.4)).copy(),
                                c.render(fr, fmt=gs.GS_FORMAT_RGBA8).copy(),
                                c.render(fr, fmt=gs.GS_FORMAT_RGBA32F, depth_in=depth).copy())
    finally:
        if old is None:
            os.environ.pop("GS_RASTER", None)
        else:
            os.environ["GS_RASTER"] = old
    for a, b in zip(frames["scalar"], frames["packed"]):
        assert np.array_equal(a, b)
    exp, _ = orc.render(cs, cc, order, fr.proj, fr.modelview, 1000, 562, fr.focal, bg=(0.1, 0.2, 0.3, 0.4))
    assert np.abs(frames["packed"][0] - exp).max() <= FRAME_TOL


def test_stats_frame_counts(gs, orc, ctx):
    """GS_RENDER_STATS: D = number of (splat, 16x16 tile) pairs whose tile meets the r<=2 footprint, and the pair
    counters.  Checked against counts derived from the oracle's projection on the host."""
    w, h = 640, 360
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 30000, 77, w, h)
    ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
    order = orc.sort(m, fr.view)
    plain = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F).copy()
    st0 = ctx.stats()
    assert st0["n_tile_instances"] == 0 and st0["n_pair_tests"] == 0  # only filled by a STATS frame
    got = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F, stats=True)
    st = ctx.stats()
    assert np.array_equal(got, plain)  # the statistics frame renders the same picture
    # host count: tiles (of the visible splats in the draw order) containing at least one covered pixel centre
    p = orc.project(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal)
    exact = 0
    pairs = 0
    for s in p[p["visible"] == 1]:
        ex = 2 * np.hypot(s["v1x"], s["v2x"]) + 1; ey = 2 * np.hypot(s["v1y"], s["v2y"]) + 1
        x0 = max(0, int(np.floor(s["cx"] - ex))); x1 = min(w - 1, int(np.ceil(s["cx"] + ex)))
        y0 = max(0, int(np.floor(s["cy"] - ey))); y1 = min(h - 1, int(np.ceil(s["cy"] + ey)))
        if x0 > x1 or y0 > y1:
            continue
        dx = (np.arange(x0, x1 + 1, dtype=np.float32) + np.float32(0.5)) - s["cx"]
        dy = (np.arange(y0, y1 + 1, dtype=np.float32) + np.float32(0.5)) - s["cy"]
        DX, DY = np.meshgrid(dx, dy)
        px = DX * s["a2x"] + DY * s["a2y"]; py = DX * s["a1x"] + DY * s["a1y"]
        msk = (px * px + py * py) <= 4.0
        if not msk.any():
            continue
        yy, xx = np.nonzero(msk)
        exact += len(np.unique(((yy + y0) >> 4) * 4096 + ((xx + x0) >> 4)))
        pairs += int(msk.sum())
    # the cull is conservative (0.5 % slack, closest point on the tile box): it may keep a few tiles no pixel centre covers
    assert exact <= st["n_tile_instances"] <= exact * 1.05 + 16
    assert st["n_instances_kept"] < st["n_tile_instances"]            # bins are coarser than tiles: fewer instances
    assert st["n_records_streamed"] >= st["n_tile_instances"]
    assert 0 < st["n_pair_hits"] <= st["n_pair_tests"]
    assert st["n_pair_hits"] <= pairs * 1.001 + 16                     # early-stopped pixels skip pairs, never add any
    # exact: every covered pair at a live pixel is blended; the front-to-back reference brackets where pixels stop
    _, _, f2b = orc.render_f2b(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal)
    assert f2b["hits_eager"] <= st["n_pair_hits"] <= f2b["hits_lazy"]


def _eye_cameras(gs, w, h, ipd=0.064):
    """Two eye cameras around the fixed head camera (same orientation, +-ipd/2 along x)."""
    tm = gs.three_math
    head = gs.scenes.fixed_camera(w, h)
    eyes = []
    for sx in (-0.5, 0.5):
        eyes.append(tm.PerspectiveCamera(fov=80.0, aspect=w / h, near=0.005, far=10000.0,
                                         position=(head.position[0] + sx * ipd, head.position[1], head.position[2])))
    return head, eyes


def test_stereo_one_sort_two_eyes(gs, orc, ctx):
    """gs_render_stereo (index.js:184-195 per-eye onBeforeRender + one tick() sort): both eyes are drawn with the HEAD
    camera's order; each eye frame equals the oracle's frame for (head order, eye matrices)."""
    w, h = 640, 400
    rows, cs, cc, m, fr_head = scene_inputs(gs, orc, 60000, 2024, w, h)
    ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
    sc = gs.scenes
    head, eye_cams = _eye_cameras(gs, w, h)
    fr_head = sc.make_frame(head, sc.demo_object(), w, h)
    eyes = [sc.make_frame(c, sc.demo_object(), w, h) for c in eye_cams]
    order = orc.sort(m, fr_head.view)
    got = ctx.render_stereo(fr_head.view, eyes, fmt=gs.GS_FORMAT_RGBA32F, bg=(0.0, 0.1, 0.2, 1.0))
    for e, g in zip(eyes, got):
        exp, _ = orc.render(cs, cc, order, e.proj, e.modelview, w, h, e.focal, bg=(0.0, 0.1, 0.2, 1.0))
        assert np.abs(g - exp).max() <= FRAME_TOL
    assert not np.array_equal(got[0], got[1])
    st = ctx.last_stereo_stats
    assert st[0].n_sorted == st[1].n_sorted == len(order) and st[0].ms_sort > 0 and st[1].ms_sort == 0
    # with a cutout the cull acts in the one sort
    cut_fr = sc.make_frame(head, sc.demo_object(), w, h, sc.demo_cutout())
    order_c = orc.sort(m, cut_fr.view, cut_fr.cutout)
    got = ctx.render_stereo(cut_fr.view, eyes, cutout=cut_fr.cutout, fmt=gs.GS_FORMAT_RGBA32F)
    exp, _ = orc.render(cs, cc, order_c, eyes[1].proj, eyes[1].modelview, w, h, eyes[1].focal)
    assert len(order_c) < len(order) and np.abs(got[1] - exp).max() <= FRAME_TOL


def test_component_render_xr(gs, orc):
    """The component mirror: xrPixelRatio scales the eye viewports (index.js:13-15), tick()'s camera sorts."""
    sc = gs.scenes
    rows = gs.synth_splats(30000, 11)
    cs, cc, m = orc.pack(rows)
    w, h = 800, 450
    head, eye_cams = _eye_cameras(gs, w, h)
    comp = gs.GaussianSplattingComponent({"src": rows.tobytes(), "xrPixelRatio": 0.5})
    comp.init(head, sc.demo_object())
    try:
        left, right = comp.render_xr(eye_cams, w, h, fmt=gs.GS_FORMAT_RGBA32F)
        assert left.shape == (225, 400, 4) and right.shape == (225, 400, 4)
        fr_head = sc.make_frame(head, sc.demo_object(), 400, 225)
        order = orc.sort(m, fr_head.view)
        e = sc.make_frame(eye_cams[0], sc.demo_object(), 400, 225)
        exp, _ = orc.render(cs, cc, order, e.proj, e.modelview, 400, 225, e.focal)
        assert np.abs(left - exp).max() <= FRAME_TOL
    finally:
        comp.renderer.close()


def test_progressive_push_while_rendering(gs, orc):
    """index.js:259-298: rows are pushed as they arrive while the scene is drawn.  Pushes are interleaved with
    gs_render_async; every frame must equal the oracle's frame of the prefix that was resident when it was submitted."""
    w, h = 640, 360
    n, chunk = 240000, 40000
    rows = gs.synth_splats(n, 555)
    cs, cc, m = orc.pack(rows)
    sc = gs.scenes
    fr = sc.make_frame(sc.fixed_camera(w, h), sc.demo_object(), w, h)
    with gs.SplatContext(0) as c:
        c.reserve(n)  # initGL(numVertexes): no growth (hence no pipeline wait) during the load
        outs, tickets, prefixes = [], [], []
        for first in range(0, n, chunk):
            c.push_splats(rows[first:first + chunk])
            out = c.pinned_array((h, w, 4), np.float32)
            out[...] = -1.0
            t = c.render_async(c.make_params(fr, fmt=gs.GS_FORMAT_RGBA32F), out.ctypes.data)
            outs.append(out); tickets.append(t); prefixes.append(first + chunk)
            if len(tickets) >= 3:  # keep three frames in flight across the pushes
                st = c.wait(tickets[-3])
                assert st.n_splats == prefixes[-3]
        for t, k in zip(tickets[-2:], prefixes[-2:]):
            assert c.wait(t).n_splats == k
        for out, k in zip(outs, prefixes):
            order = orc.sort(m[:k], fr.view)
            exp, _ = orc.render(cs[:k], cc[:k], order, fr.proj, fr.modelview, w, h, fr.focal)
            assert np.abs(out - exp).max() <= FRAME_TOL, k
        assert c.num_splats == n
        # without gs_reserve the table grows geometrically; frames stay correct across the growth
    with gs.SplatContext(0) as c:
        outs, tickets, prefixes = [], [], []
        for first in range(0, n, chunk):
            c.push_splats(rows[first:first + chunk])
            out = np.empty((h, w, 4), np.float32)
            tickets.append(c.render_async(c.make_params(fr, fmt=gs.GS_FORMAT_RGBA32F), out.ctypes.data))
            outs.append(out); prefixes.append(first + chunk)
        for t in tickets[-3:]:
            c.wait(t)
        for out, k in zip(outs[::2], prefixes[::2]):
            order = orc.sort(m[:k], fr.view)
            exp, _ = orc.render(cs[:k], cc[:k], order, fr.proj, fr.modelview, w, h, fr.focal)
            assert np.abs(out - exp).max() <= FRAME_TOL, k


def _slab_ctx(gs, monkeypatch, slab_min, first):
    monkeypatch.setenv("GS_SLAB_MIN", str(slab_min))
    monkeypatch.setenv("GS_SLAB_FIRST", str(first))
    return gs.SplatContext(0)


@pytest.mark.parametrize("n,w,h,first", [(300000, 1000, 562, 20000), (60000, 640, 360, 3000), (500000, 1920, 1080, 50000)])
def test_slab_path_equals_one_pass(gs, orc, ctx, monkeypatch, n, w, h, first):
    """Front-to-back slab path (large scenes; forced here with GS_SLAB_MIN / GS_SLAB_FIRST): same frame as the one-pass
    path BIT FOR BIT (a dead pixel ignores a splat whether or not it was binned), float / RGBA8 / depth-tested, and
    within tolerance of the oracle."""
    rows, cs, cc, m, fr = scene_inputs(gs, orc, n, 31337 + n, w, h)
    order = orc.sort(m, fr.view)
    depth = _depth_plane(orc, cs, cc, order, fr, w, h)
    bg = (0.25, 0.5, 0.75, 0.5)
    ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
    ref32 = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F).copy()
    ref8 = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA8).copy()
    refd = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F, depth_in=depth).copy()
    st_ref = ctx.stats()
    with _slab_ctx(gs, monkeypatch, 1000, first) as c:
        c.push_packed(cs, cc, m[:, 15])
        got32 = c.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F)
        st = c.stats()
        assert np.array_equal(got32, ref32)
        assert np.array_equal(c.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA8), ref8)
        assert np.array_equal(c.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F, depth_in=depth), refd)
        assert st["n_sorted"] == len(order) == st_ref["n_sorted"] and st["n_splats"] == n
        assert st["kernel_launches"] > 40  # several slabs were scheduled
        assert 1 <= st["n_slabs_run"] <= st["n_slabs"] <= 12 and st_ref["n_slabs"] == 0
        # every slab that ran was compacted, sorted and projected: at least the nearest slab, at most the whole sort
        assert min(first, len(order)) * 0.5 <= st["n_slab_entries"] <= len(order) + st["n_dropped"]
        # pipelined: three slab frames in flight, different cameras
        sc = gs.scenes
        frames = [sc.make_frame(sc.orbit_camera(w, h, s), sc.demo_object(), w, h) for s in (0, 9, 33, 77)]
        ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
        exp = [ctx.render(f, fmt=gs.GS_FORMAT_RGBA8).copy() for f in frames]
        outs = [c.pinned_array((h, w, 4), np.uint8) for _ in frames]
        ts = [c.render_async(c.make_params(f, fmt=gs.GS_FORMAT_RGBA8), o.ctypes.data) for f, o in zip(frames[:3], outs[:3])]
        c.wait(ts[0])
        ts.append(c.render_async(c.make_params(frames[3], fmt=gs.GS_FORMAT_RGBA8), outs[3].ctypes.data))
        for t in ts[1:]:
            c.wait(t)
        for o, e in zip(outs, exp):
            assert np.array_equal(o, e)
        # gs_sort and a stale-order draw still work on a slab-sized scene (they take the one-pass path)
        assert np.array_equal(c.sort(fr.view), order)
        stale = c.render(frames[1], fmt=gs.GS_FORMAT_RGBA8, reuse_sort=True)  # camera 1 drawn with fr's order
        ctx.sort(fr.view, readback=False)
        assert np.array_equal(stale, ctx.render(frames[1], fmt=gs.GS_FORMAT_RGBA8, reuse_sort=True))
    exp32, _ = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=bg)
    assert np.abs(ref32 - exp32).max() <= FRAME_TOL


def test_slab_path_quirk_q5_and_sharding(gs, orc, ctx, monkeypatch):
    """Slab path corner cases: (1) quirk Q5 - dropped keys become repeats of splat 0 in front of everything; (2) the frame
    sharded over emulated ranks (bin-column ownership) assembles to the unsharded frame."""
    # (1) the Q5 scene of test_render_q5_tail_zero_draws_splat0
    n = 4096
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
    mm = np.zeros((n, 16), np.float32); mm[:, 12:15] = cs[:, :3]; mm[:, 15] = sa
    W, H = 128, 96
    P = np.zeros(16, np.float32); P[0] = 1.0; P[5] = -1.3; P[10] = -1.0; P[11] = -1.0; P[14] = -0.02
    MV = np.eye(4, dtype=np.float32).reshape(16); MV[14] = 1e-4
    view = np.array([MV[2], MV[6], MV[10], MV[14]], np.float32)
    order = orc.sort(mm, view)
    fr = gs.FrameInputs(proj=P, modelview=MV, view=view, width=W, height=H, focal=400.0)
    exp, _ = orc.render(cs, cc, order, P, MV, W, H, 400.0)
    with _slab_ctx(gs, monkeypatch, 100, 500) as c:
        c.push_packed(cs, cc, sa)
        got = c.render(fr, fmt=gs.GS_FORMAT_RGBA32F)
        st = c.stats()
        assert st["n_dropped"] > 0 and (order == 0).sum() >= 2 and st["n_sorted"] == len(order)
        assert np.abs(got - exp).max() <= FRAME_TOL
    # (2) sharded slab frames
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 120000, 2222, 1000, 562)
    ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
    ctx.set_shard(0, 1)
    ref = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA8, bg=(0.2, 0.1, 0.0, 0.3)).copy()
    with _slab_ctx(gs, monkeypatch, 1000, 10000) as c:
        c.push_packed(cs, cc, m[:, 15])
        world = 3
        sh = gs.dist.TileSharding(fr.width, fr.height, world)
        tpr = sh.tiles_per_rank
        tiles = []
        for r in range(world):
            c.set_shard(r, world)
            p = c.make_params(fr, bg=(0.2, 0.1, 0.0, 0.3), fmt=gs.GS_FORMAT_RGBA8, flags=gs.GS_RENDER_OUT_TILED)
            t = np.zeros((tpr, 256, 4), np.uint8)
            c.render_raw(p, t.ctypes.data)
            tiles.append(t)
        assert np.array_equal(sh.assemble(np.stack(tiles)), ref)


def test_slab_path_random_regimes(gs, orc, ctx, monkeypatch):
    """Slab path vs one-pass path over random regimes: tiny scenes, nothing visible, one visible splat, cutouts, odd frame
    sizes, different slab sizes.  Frames must be identical bit for bit; sampled cases are also compared with the oracle."""
    sc = gs.scenes
    rng = np.random.default_rng(2025)
    cases = [(1, 64, 48, 1000), (37, 250, 141, 5), (4097, 333, 200, 700), (90000, 803, 451, 8000), (250000, 1280, 720, 100000)]
    for k, (n, w, h, first) in enumerate(cases):
        rows = gs.synth_splats(n, 9000 + k)
        cs, cc, m = orc.pack(rows)
        for variant in ("plain", "cutout", "behind"):
            if variant == "behind":  # camera looks away from the scene: nothing passes the worker filter or the clip
                cam = gs.three_math.PerspectiveCamera(fov=80.0, aspect=w / h, near=0.005, far=10000.0, position=(0.0, 1.6, 40.0),
                                                      quaternion=gs.three_math.yaw_quaternion(np.pi))
                fr = sc.make_frame(cam, sc.demo_object(), w, h)
            else:
                cam = sc.orbit_camera(w, h, int(rng.integers(0, 120)))
                fr = sc.make_frame(cam, sc.demo_object(), w, h, sc.demo_cutout() if variant == "cutout" else None)
            ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
            bg = tuple(float(x) for x in rng.uniform(0, 1, 4))
            ref = ctx.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F).copy()
            nsort = ctx.stats()["n_sorted"]
            with _slab_ctx(gs, monkeypatch, 0, first) as c:
                c.push_packed(cs, cc, m[:, 15])
                got = c.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F)
                st = c.stats()
                assert np.array_equal(got, ref), (n, variant)
                assert st["n_sorted"] == nsort and st["kernel_launches"] >= 20
                got2 = c.render(fr, bg=bg, fmt=gs.GS_FORMAT_RGBA32F)  # second frame: same path, same picture
                assert np.array_equal(got2, ref)
            if k in (1, 3):
                order = orc.sort(m, fr.view, fr.cutout)
                exp, _ = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=bg)
                assert len(order) == nsort and np.abs(ref - exp).max() <= FRAME_TOL


def test_largest_frame_4096(gs, orc, ctx):
    """4096 x 4096 is the largest frame the ABI accepts: 65 536 tiles, 43 x 43 bins (two bin passes), frame compared with
    the oracle on a band of rows and on the RGBA8 / float consistency of the rest."""
    w = h = 4096
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 40000, 4096, w, h)
    ctx.clear(); ctx.push_packed(cs, cc, m[:, 15])
    order = orc.sort(m, fr.view)
    got = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F, bg=(0.0, 0.0, 0.0, 1.0))
    st = ctx.stats()
    assert st["n_tiles"] == 256 * 256 and st["width"] == w
    band = (h // 2 - 64, h // 2 + 64)
    exp, _ = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, bg=(0.0, 0.0, 0.0, 1.0), rows=band)
    assert np.abs(got[band[0]:band[1]] - exp[band[0]:band[1]]).max() <= FRAME_TOL
    got8 = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA8, bg=(0.0, 0.0, 0.0, 1.0))
    assert np.abs(got8.astype(np.int32) - np.floor(np.clip(got, 0, 1) * 255 + 0.5).astype(np.int32)).max() <= 1
    with pytest.raises(Exception):
        ctx.render(gs.FrameInputs(proj=fr.proj, modelview=fr.modelview, view=fr.view, width=4097, height=16, focal=fr.focal))
