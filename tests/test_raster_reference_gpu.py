"""GPU raster against the front-to-back fp64 reference (orc_render_f2b, tests/test_f2b_reference.py pins it).

The kernel's coverage and depth decisions are exact fp32 and the reference reproduces them; only where a pixel stops
is uncertain, and the reference brackets it (eager / lazy stop).  Per case:
  - RGBA32F over a background of alpha 0, so T = 1 - A and C = out - bg T: C and T lie in the hull of the eager and
    the lazy result within TOL;
  - the RGBA8 frame lies between the kernel's to_u8 of the hull ends;
  - a STATS frame: hits_eager <= n_pair_hits <= hits_lazy, so a covered pair that the bin emission or the tile cull
    drops at a live pixel fails exactly, whatever its weight;
  - the projected records of the drawn splats are bit-exact with the oracle (a projection error is reported as one).
Each case prints its measured distance outside the hull (run with -s to see it)."""
import numpy as np
import pytest

import splat_cases as S
from conftest import scene_inputs
from test_gpu_parity import _check_projection

pytestmark = pytest.mark.gpu
TOL = 1e-5  # fp32 accumulation + ex2.approx; the per-case maxima measured on a B200 are in DESIGN.md §3
BG = (0.2, 0.45, 0.7, 0.0)


def _to_u8(v):
    """gs_raster.cu to_u8: clamp to [0, 1], fp32 v * 255 + 0.5, truncate."""
    v = np.clip(np.asarray(v, np.float64), 0.0, 1.0).astype(np.float32)
    return (v * np.float32(255.0) + np.float32(0.5)).astype(np.uint32)


def _inputs(ctx, cs, cc, sa, fr):
    ctx.clear()
    ctx.push_packed(cs, cc, sa)
    return ctx.sort(fr.view, fr.cutout)


def _bracket(name, gs, orc, ctx, cs, cc, sa, fr, order, depth=None, stats=True, projection=True, tol=TOL):
    w, h = fr.width, fr.height
    e, l, st = orc.render_f2b(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, depth_in=depth)
    got = ctx.render(fr, bg=BG, fmt=gs.GS_FORMAT_RGBA32F, depth_in=depth).astype(np.float64)
    drawn = _check_projection(gs, orc, ctx, cs, cc, fr, order) if projection else None
    bg = np.array(BG[:3])
    T = 1.0 - got[..., 3]
    C = got[..., :3] - bg * T[..., None]
    out_c = np.maximum(np.maximum(e[..., :3] - C, C - l[..., :3]), 0.0).max(initial=0.0)
    out_t = np.maximum(np.maximum(l[..., 3] - T, T - e[..., 3]), 0.0).max(initial=0.0)
    got8 = ctx.render(fr, bg=BG, fmt=gs.GS_FORMAT_RGBA8, depth_in=depth).astype(np.int64)
    lo = np.concatenate([e[..., :3] + bg * l[..., 3:4], 1.0 - e[..., 3:4]], -1) - tol
    hi = np.concatenate([l[..., :3] + bg * e[..., 3:4], 1.0 - l[..., 3:4]], -1) + tol
    bad8 = int(((got8 < _to_u8(lo)) | (got8 > _to_u8(hi))).sum())
    hits = None
    if stats:
        ctx.render(fr, bg=BG, fmt=gs.GS_FORMAT_RGBA32F, depth_in=depth, stats=True)
        hits = ctx.stats()["n_pair_hits"]
    print(f"[f2b] {name}: {w}x{h} max|C| outside hull {out_c:.2e}, max|T| outside hull {out_t:.2e}, tol {tol:.0e}, "
          f"eager/lazy differ at {st['n_differ']} px, hits {st['hits_eager']} <= {hits} <= {st['hits_lazy']}, "
          f"max M {st['max_m']:.1e}, drawn {drawn}")
    assert out_c <= tol and out_t <= tol, (name, out_c, out_t)
    assert bad8 == 0, (name, bad8)
    if stats:
        assert st["hits_eager"] <= hits <= st["hits_lazy"], (name, st, hits)
    assert st["n_differ"] <= max(4, 1e-3 * w * h), (name, st)
    return st


def _built(ctx, gs, orc, W, H, parts):
    cs, cc, sa = parts
    P, MV = S.camera()
    fr = gs.FrameInputs(proj=P, modelview=MV, view=S.VIEW, width=W, height=H, focal=S.FOCAL)
    order = _inputs(ctx, cs, cc, sa, fr)
    assert np.array_equal(order, orc.sort_compact(cs, sa, S.VIEW))
    return cs, cc, sa, fr, order


BUILT = {
    "sweep": lambda rng: S.sweep_scene(rng),
    "needles": lambda rng: S.needle_scene(rng),
    "offscreen": lambda rng: S.offscreen_scene(rng),
    "stack1500": lambda rng: S.stack_scene(rng),
    "opaque_at_126": lambda rng: S.stack_scene(rng, opaque_from=126),  # dies at record 127: packed chunk boundary
    "opaque_at_190": lambda rng: S.stack_scene(rng, opaque_from=190),  # mid-chunk
    "opaque_at_254": lambda rng: S.stack_scene(rng, opaque_from=254),  # scalar chunk boundary
}


@pytest.mark.parametrize("case", list(BUILT))
def test_built_edge_scenes(gs, orc, ctx, case):
    W, H, parts = BUILT[case](np.random.default_rng(100))
    cs, cc, sa, fr, order = _built(ctx, gs, orc, W, H, parts)
    _bracket(case, gs, orc, ctx, cs, cc, sa, fr, order)
    if case == "needles":  # the angle-0 needles vanish on both sides (quirk Q8)
        rect = ctx.read_projected()[:, 7].copy().view(np.uint32)
        ref = orc.project(cs, cc, None, fr.proj, fr.modelview, W, H, fr.focal)
        assert np.all(rect[:S.N_Q8] == 0xFFFFFFFF) and np.all(ref["visible"][:S.N_Q8] == 0)
        assert np.all(ref["visible"][S.N_Q8:] == 1)


def test_low_alpha_everywhere(gs, orc, ctx):
    """Alpha bytes 1-3 on every splat: contributions of a few 1e-4 that the 1e-3 frame gate cannot see."""
    w, h = 256, 144
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 20000, 31, w, h)
    cc = cc.copy()
    cc[:, 3] = (cc[:, 3] & 0x00FFFFFF) | (np.random.default_rng(3).integers(1, 4, len(cc)).astype(np.uint32) << 24)
    order = _inputs(ctx, cs, cc, m[:, 15], fr)
    _bracket("alpha_1_3", gs, orc, ctx, cs, cc, m[:, 15], fr, order)


def test_depth_exactly_at_window_depth(gs, orc, ctx):
    """depth_in equal to a splat's fp32 window depth keeps it (LEQUAL); one ulp nearer rejects it."""
    W, H, parts = S.sweep_scene(np.random.default_rng(5))
    cs, cc, sa, fr, order = _built(ctx, gs, orc, W, H, parts)
    p = orc.project(cs, cc, order, fr.proj, fr.modelview, W, H, fr.focal)
    zw = (p["zndc"] * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    z = zw[len(zw) // 2]
    depth = np.full((H, W), z, np.float32)
    depth[:, W // 2:] = np.nextafter(z, np.float32(0))
    st = _bracket("depth_eq", gs, orc, ctx, cs, cc, sa, fr, order, depth=depth)
    e_left, _, s_left = orc.render_f2b(cs, cc, order, fr.proj, fr.modelview, W, H, fr.focal, depth_in=np.full((H, W), z, np.float32))
    e_right, _, s_right = orc.render_f2b(cs, cc, order, fr.proj, fr.modelview, W, H, fr.focal,
                                         depth_in=np.full((H, W), np.nextafter(z, np.float32(0)), np.float32))
    assert s_left["hits_eager"] > s_right["hits_eager"] > 0 and st["hits_eager"] > 0


SIZES = [(1, 1), (15, 17), (95, 97), (96, 96), (97, 95), (1536, 1536), (1537, 1536), (4096, 16)]


@pytest.mark.parametrize("w,h", SIZES)
def test_frame_sizes(gs, orc, ctx, w, h):
    """Odd tile/bin remainders, one bin row / column, 256 bins (one bin-sort pass) and 272 (two passes), the widest
    frame the ABI takes."""
    n = 60000 if w * h > 1 << 20 else 20000
    rows, cs, cc, m, fr = scene_inputs(gs, orc, n, 7000 + w + h, w, h)
    order = _inputs(ctx, cs, cc, m[:, 15], fr)
    _bracket(f"size_{w}x{h}", gs, orc, ctx, cs, cc, m[:, 15], fr, order)


@pytest.mark.parametrize("n,w,h,cutout,lsm", [(150000, 1920, 1080, False, None), (20000, 250, 141, True, None),
                                              (8000, 1920, 1080, False, -0.5)])
def test_synthetic_scenes(gs, orc, ctx, n, w, h, cutout, lsm):
    rows = gs.synth_splats(n, 500 + n, log_scale_mean=lsm) if lsm is not None else gs.synth_splats(n, 500 + n)
    cs, cc, m = orc.pack(rows)
    sc = gs.scenes
    fr = sc.make_frame(sc.fixed_camera(w, h), sc.demo_object(), w, h, sc.demo_cutout() if cutout else None)
    order = _inputs(ctx, cs, cc, m[:, 15], fr)
    assert np.array_equal(order, orc.sort(m, fr.view, fr.cutout))
    _bracket(f"synth_{n}_{w}x{h}{'_cutout' if cutout else ''}{'_large' if lsm else ''}", gs, orc, ctx, cs, cc, m[:, 15], fr, order)


def _other_case(gs, orc, which):
    rng = np.random.default_rng(100)
    P, MV = S.camera()
    if which in BUILT:
        W, H, (cs, cc, sa) = BUILT[which](rng)
        return cs, cc, sa, gs.FrameInputs(proj=P, modelview=MV, view=S.VIEW, width=W, height=H, focal=S.FOCAL)
    rows, cs, cc, m, fr = scene_inputs(gs, orc, 150000, 4321, 1000, 562)
    return cs, cc, m[:, 15], fr


@pytest.mark.parametrize("which", ["sweep", "needles", "opaque_at_254", "stack1500", "synth"])
def test_scalar_pixel_loop(gs, orc, monkeypatch, which):
    cs, cc, sa, fr = _other_case(gs, orc, which)
    monkeypatch.setenv("GS_RASTER", "scalar")
    with gs.SplatContext(0) as c:
        order = _inputs(c, cs, cc, sa, fr)
        _bracket(f"scalar_{which}", gs, orc, c, cs, cc, sa, fr, order)


@pytest.mark.parametrize("which", ["sweep", "opaque_at_126", "stack1500", "synth"])
def test_slab_path(gs, orc, monkeypatch, which):
    """The depth-slab path (forced; it keeps no STATS counters and stores records by draw-order entry)."""
    cs, cc, sa, fr = _other_case(gs, orc, which)
    monkeypatch.setenv("GS_SLAB_MIN", "0")
    monkeypatch.setenv("GS_SLAB_FIRST", "1024")
    with gs.SplatContext(0) as c:
        order = _inputs(c, cs, cc, sa, fr)
        _bracket(f"slab_{which}", gs, orc, c, cs, cc, sa, fr, order, stats=False, projection=False)
        assert c.stats()["n_slabs_run"] >= 1


@pytest.mark.parametrize("which", ["stack1500", "synth"])
def test_depth_in(gs, orc, ctx, which):
    cs, cc, sa, fr = _other_case(gs, orc, which)
    order = _inputs(ctx, cs, cc, sa, fr)
    p = orc.project(cs, cc, order, fr.proj, fr.modelview, fr.width, fr.height, fr.focal)
    zw = np.sort((p["zndc"][p["visible"] == 1] * np.float32(0.5) + np.float32(0.5)).astype(np.float32))
    depth = np.empty((fr.height, fr.width), np.float32)
    depth[:, : fr.width // 2] = zw[len(zw) // 2]
    depth[:, fr.width // 2:] = np.linspace(zw[0], zw[-1], fr.width - fr.width // 2, dtype=np.float32)[None, :]
    _bracket(f"depth_{which}", gs, orc, ctx, cs, cc, sa, fr, order, depth=depth)
