"""ctypes wrapper of oracle/libgs_oracle.so — TEST INFRASTRUCTURE ONLY (see gs_oracle.c header).

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg.
PARITY UNPINNED: the reference has no tests or golden vectors; this oracle restates index.js.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgs_oracle.so")


def stale(out: str = LIB_PATH) -> bool:
    return not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(os.path.join(HERE, "gs_oracle.c"))


def build(force: bool = False, out: str = LIB_PATH) -> str:
    """Compile libgs_oracle.so to `out`, by default next to this file."""
    if force or stale(out):
        res = subprocess.run(["make", "-C", HERE, "-B" if force else "-s", f"OUT={os.path.abspath(out)}"], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("oracle build failed:\n" + res.stdout + res.stderr)
    return out


class ProjRec(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("cx", "cy", "v1x", "v1y", "v2x", "v2y", "a1x", "a1y", "a2x", "a2y", "r", "g", "b", "a", "zndc")] + [("visible", C.c_uint32)]


PROJ_DTYPE = np.dtype([(k, np.float32) for k in ("cx", "cy", "v1x", "v1y", "v2x", "v2y", "a1x", "a1y", "a2x", "a2y", "r", "g", "b", "a", "zndc")] + [("visible", np.uint32)])


class RenderStats(C.Structure):
    _fields_ = [("n_order", C.c_uint32), ("n_visible", C.c_uint32), ("fragments", C.c_uint64)]


class F2bStats(C.Structure):
    _fields_ = [("hits_eager", C.c_uint64), ("hits_lazy", C.c_uint64), ("n_differ", C.c_uint64), ("max_m", C.c_double)]


_lib = None


def lib(path: str | None = None):
    """The loaded oracle library: `path`, or the in-tree build (compiled first when stale).  The first call decides."""
    global _lib
    if _lib is None:
        L = C.CDLL(build() if path is None else path)
        L.orc_pack.restype = C.c_int
        L.orc_sort.restype = C.c_int
        L.orc_sort_compact.restype = C.c_int
        L.orc_project.restype = C.c_int
        L.orc_render.restype = C.c_int
        L.orc_render_rows.restype = C.c_int
        L.orc_render_ex.restype = C.c_int
        L.orc_render_f2b.restype = C.c_int
        L.orc_coverage_check.restype = C.c_int
        L.orc_set_affinity.restype = None
        L.orc_ply_to_splat.restype = C.c_int64
        L.orc_ply_to_splat.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.orc_sizeof_proj.restype = C.c_int
        L.orc_version.restype = C.c_char_p
        assert L.orc_sizeof_proj() == PROJ_DTYPE.itemsize == C.sizeof(ProjRec)
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pack(rows: np.ndarray, threads: int | None = None):
    """pushDataBuffer (index.js:343-402) -> (center_scale (n,4) f32, cov_color (n,4) u32, matrices (n,16) f32).
    Rows are independent, so large inputs are packed in chunks on a thread pool (the C call releases the GIL)."""
    rows = np.ascontiguousarray(rows, np.uint8).reshape(-1, 32)
    n = rows.shape[0]
    cs = np.zeros((n, 4), np.float32)
    cc = np.zeros((n, 4), np.uint32)
    m = np.zeros((n, 16), np.float32)
    L = lib()
    chunk = 1 << 18
    if threads is None:
        threads = min(32, os.cpu_count() or 1)

    def one(first):
        cnt = min(chunk, n - first)
        return L.orc_pack(_p(rows[first:]), C.c_uint32(cnt), _p(cs[first:]), _p(cc[first:]), _p(m[first:]))

    starts = list(range(0, n, chunk))
    if threads > 1 and len(starts) > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(threads) as ex:
            rcs = list(ex.map(one, starts))
    else:
        rcs = [one(f) for f in starts]
    assert all(r == 0 for r in rcs)
    return cs, cc, m


def sort(matrices: np.ndarray, view: np.ndarray, cutout: np.ndarray | None = None) -> np.ndarray:
    """sortSplats (index.js:507-570) on the worker's 64 B/row table."""
    matrices = np.ascontiguousarray(matrices, np.float32).reshape(-1, 16)
    n = matrices.shape[0]
    view = np.ascontiguousarray(view, np.float32)
    cu = None if cutout is None else np.ascontiguousarray(cutout, np.float32)
    out = np.zeros((max(n, 1),), np.uint32)
    cnt = C.c_uint32()
    rc = lib().orc_sort(_p(matrices), C.c_uint32(n), _p(view), _p(cu), _p(out), C.byref(cnt))
    assert rc == 0
    return out[:cnt.value].copy()


def sort_compact(center_scale, size_alpha, view, cutout=None) -> np.ndarray:
    cs = np.ascontiguousarray(center_scale, np.float32).reshape(-1, 4)
    sa = np.ascontiguousarray(size_alpha, np.float32).reshape(-1)
    n = cs.shape[0]
    view = np.ascontiguousarray(view, np.float32)
    cu = None if cutout is None else np.ascontiguousarray(cutout, np.float32)
    out = np.zeros((max(n, 1),), np.uint32)
    cnt = C.c_uint32()
    rc = lib().orc_sort_compact(_p(cs), _p(sa), C.c_uint32(n), _p(view), _p(cu), _p(out), C.byref(cnt))
    assert rc == 0
    return out[:cnt.value].copy()


def project(center_scale, cov_color, order, proj, mv, width, height, focal) -> np.ndarray:
    """Vertex shader (index.js:101-164) for the splats listed in `order` (None = all, index order)."""
    cs = np.ascontiguousarray(center_scale, np.float32).reshape(-1, 4)
    cc = np.ascontiguousarray(cov_color, np.uint32).reshape(-1, 4)
    o = None if order is None else np.ascontiguousarray(order, np.uint32)
    count = cs.shape[0] if o is None else o.shape[0]
    out = np.zeros((max(count, 1),), PROJ_DTYPE)
    rc = lib().orc_project(_p(cs), _p(cc), _p(o), C.c_uint32(count), _p(np.ascontiguousarray(proj, np.float32)),
                           _p(np.ascontiguousarray(mv, np.float32)), C.c_float(width), C.c_float(height), C.c_float(focal), _p(out))
    assert rc == 0
    return out[:count]


def physical_cpus() -> list:
    """One logical CPU per physical core, restricted to this process's affinity mask (thread pinning for the
    bench's CPU arm: hyper-thread siblings and unpinned workers made its timing host-dependent)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))
    seen, cpus = set(), []
    for c in allowed:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                sib = f.read().strip()
        except OSError:
            sib = str(c)
        if sib in seen:
            continue
        seen.add(sib)
        cpus.append(c)
    return cpus or allowed


def set_affinity(cpus) -> None:
    """Pin raster worker t to logical CPU cpus[t % len(cpus)] (empty list = no pinning)."""
    arr = (C.c_int * max(1, len(cpus)))(*cpus)
    lib().orc_set_affinity(arr, len(cpus))


def render(center_scale, cov_color, order, proj, mv, width, height, focal, bg=(0, 0, 0, 0), nthreads=None, unorm8=False,
           rows=None, depth_in=None):
    """Fragment shader + blend (index.js:170-181) -> ((H,W,4) f32 frame, row 0 = bottom; stats dict).
    depth_in: optional (H, W) f32 window-space depth of foreign geometry; fragments are depth-tested LEQUAL against
    it and never write it (index.js:179-180)."""
    cs = np.ascontiguousarray(center_scale, np.float32).reshape(-1, 4)
    cc = np.ascontiguousarray(cov_color, np.uint32).reshape(-1, 4)
    o = np.ascontiguousarray(order, np.uint32)
    out = np.zeros((height, width, 4), np.float32)
    bgv = np.asarray(bg, np.float32)
    st = RenderStats()
    if nthreads is None:
        nthreads = os.cpu_count() or 1
    d = None if depth_in is None else np.ascontiguousarray(depth_in, np.float32).reshape(height, width)
    r0, r1 = (0, height) if rows is None else rows  # rows=(y0, y1): shade only that band (bounded-sample timing)
    rc = lib().orc_render_ex(_p(cs), _p(cc), _p(o), C.c_uint32(o.shape[0]), _p(np.ascontiguousarray(proj, np.float32)),
                             _p(np.ascontiguousarray(mv, np.float32)), C.c_uint32(width), C.c_uint32(height), C.c_float(focal),
                             _p(bgv), _p(out), C.c_int(nthreads), C.c_int(1 if unorm8 else 0), C.byref(st),
                             C.c_uint32(r0), C.c_uint32(r1), _p(d))
    assert rc == 0
    return out, {"n_order": st.n_order, "n_visible": st.n_visible, "fragments": st.fragments}


def render_f2b(center_scale, cov_color, order, proj, mv, width, height, focal, t_stop=3e-4, exact=False, depth_in=None,
               nthreads=None):
    """Front-to-back fp64 reference of the CUDA raster with its stop rule bracketed (orc_render_f2b in gs_oracle.c).
    Returns (eager, lazy, stats): two (H, W, 4) float64 frames {R, G, B, T} (row 0 = bottom, no background) and
    {"hits_eager", "hits_lazy", "n_differ", "max_m"}.  t_stop=0 disables the stop; exact=True applies the stop rule to
    the fp64 transmittance without an error margin (then eager == lazy)."""
    cs = np.ascontiguousarray(center_scale, np.float32).reshape(-1, 4)
    cc = np.ascontiguousarray(cov_color, np.uint32).reshape(-1, 4)
    o = np.ascontiguousarray(order, np.uint32)
    eager = np.zeros((height, width, 4), np.float64)
    lazy = np.zeros((height, width, 4), np.float64)
    st = F2bStats()
    if nthreads is None:
        nthreads = os.cpu_count() or 1
    d = None if depth_in is None else np.ascontiguousarray(depth_in, np.float32).reshape(height, width)
    rc = lib().orc_render_f2b(_p(cs), _p(cc), _p(o), C.c_uint32(o.shape[0]), _p(np.ascontiguousarray(proj, np.float32)),
                              _p(np.ascontiguousarray(mv, np.float32)), C.c_uint32(width), C.c_uint32(height), C.c_float(focal),
                              _p(d), C.c_double(t_stop), C.c_int(1 if exact else 0), _p(eager), _p(lazy), C.byref(st),
                              C.c_int(nthreads))
    assert rc == 0
    return eager, lazy, {"hits_eager": st.hits_eager, "hits_lazy": st.hits_lazy, "n_differ": st.n_differ, "max_m": st.max_m}


def coverage_check(center_scale, cov_color, order, proj, mv, width, height, focal, nthreads=None) -> dict:
    """Compare the affine vPosition evaluation used by the rasters with GL's barycentric interpolation over the two
    triangles of the quad (see orc_coverage_check in gs_oracle.c)."""
    cs = np.ascontiguousarray(center_scale, np.float32).reshape(-1, 4)
    cc = np.ascontiguousarray(cov_color, np.uint32).reshape(-1, 4)
    o = np.ascontiguousarray(order, np.uint32)
    out = (C.c_uint64 * 4)()
    md, mf = C.c_double(), C.c_double()
    if nthreads is None:
        nthreads = os.cpu_count() or 1
    rc = lib().orc_coverage_check(_p(cs), _p(cc), _p(o), C.c_uint32(o.shape[0]), _p(np.ascontiguousarray(proj, np.float32)),
                                  _p(np.ascontiguousarray(mv, np.float32)), C.c_uint32(width), C.c_uint32(height),
                                  C.c_float(focal), C.c_int(nthreads), out, C.byref(md), C.byref(mf))
    assert rc == 0
    return {"pairs_affine": int(out[0]), "pairs_gl": int(out[1]), "pairs_differ": int(out[2]), "pairs_in_quad": int(out[3]),
            "max_dalpha_common": md.value, "max_alpha_flipped": mf.value}


def ply_to_splat(ply_bytes: bytes) -> np.ndarray:
    """processPlyBuffer (index.js:600-745) -> (n, 32) uint8 rows."""
    buf = np.frombuffer(ply_bytes, np.uint8)
    n = lib().orc_ply_to_splat(_p(buf), buf.size, None)
    if n < 0:
        raise ValueError("Unable to read .ply file header")
    out = np.zeros((max(n, 1), 32), np.uint8)
    n2 = lib().orc_ply_to_splat(_p(buf), buf.size, _p(out))
    assert n2 == n
    return out[:n]


def camera_matrices(camera_world, camera_projection, object_world):
    """getProjectionMatrix / getModelViewMatrix (index.js:456-487) in fp64 -> (proj16, mv16) float64 arrays."""
    cw = np.ascontiguousarray(camera_world, np.float64)
    cp = np.ascontiguousarray(camera_projection, np.float64)
    ow = np.ascontiguousarray(object_world, np.float64)
    proj = np.zeros(16, np.float64)
    mv = np.zeros(16, np.float64)
    lib().orc_get_projection_matrix(_p(cp), _p(proj))
    lib().orc_get_model_view_matrix(_p(cw), _p(ow), _p(mv))
    return proj, mv


def world_to_cutout(cutout_world, object_world):
    out = np.zeros(16, np.float64)
    lib().orc_world_to_cutout(_p(np.ascontiguousarray(cutout_world, np.float64)), _p(np.ascontiguousarray(object_world, np.float64)), _p(out))
    return out
