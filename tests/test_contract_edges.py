"""Edges of the pixel contract that the rest of the suite compares only between two implementations sharing the same
arithmetic, or never launches at all:

* the flat-texel ray direction (DESIGN.md C8) on low, wide views, where n * invF leaves 64 bits: checked against a
  big-integer restatement of C8 (product through tests/hostcheck, oracle, and every flat pixel of CPU and GPU frames);
* the walk kernel's persistent grid (b2d_walk_device with more than 148 frames: a CTA loops over frames and reuses its
  shared memory), frames against the oracle and worklists against hostcheck;
* every instantiation of the raster kernel launch_raster can select, named by the kernel the profiler saw, plus the
  A/B switches read at renderer creation (B2D_TUNE, B2D_NO_VMM) and B2D_RASTER_GENERIC_W;
* poses the random pose generators do not aim at (octant boundaries, an eye on a partition line / a vertex / a plane,
  far above or below every plane, against a one-sided wall).
"""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import render
from oracle import scene as S
from tests.conftest import sample_poses

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAM_OCTANT = 1 << 29


# ---- C8 restated with unbounded integers --------------------------------------------------------------------------
def c8_dirs(cosq: int, sinq: int, W: int, F: int):
    """Exact Q18 ray direction of every column: ((cos*F + sin*c2) >> 4) * floor(2^32/F) >> 40, c2 = 2x+1-W, no wrap."""
    invF = (1 << 32) // F
    ax = [(((cosq * F + sinq * (2 * x + 1 - W)) >> 4) * invF) >> 40 for x in range(W)]
    ay = [(((sinq * F - cosq * (2 * x + 1 - W)) >> 4) * invF) >> 40 for x in range(W)]
    return np.array(ax, dtype=np.int64), np.array(ay, dtype=np.int64)


def light_row(b: int, z8: np.ndarray) -> np.ndarray:
    """C9: clamp(floor(64(255-b)/255 - 2880/(z+90)), 0, 31) on z8 = depth in 1/8 map units."""
    Z = z8.astype(np.int64) + 720
    num = 64 * (255 - b) * Z - 5875200
    return np.clip(np.where(num <= 0, 0, num // (255 * Z)), 0, 31)


def bam(deg: float) -> int:
    return int(round(deg / 360.0 * 4294967296.0)) & 0xFFFFFFFF


def angles_at_octants(seed: int, n_random: int):
    rng = np.random.default_rng(seed)
    out = [((k * BAM_OCTANT) + d) & 0xFFFFFFFF for k in range(8) for d in (-1, 0, 1)]
    return out + [int(a) for a in rng.integers(0, 1 << 32, n_random, dtype=np.uint64)]


def oracle_view(v) -> render.View:
    return render.View(v.width, v.height, v.F, v.FY2)


# ---- 1. exact flat direction ----------------------------------------------------------------------------------------
def _accepted_views(b2d):
    """(name, product view): W/F from 1 to 2048, H = 2, fields of view near both limits, and views b2d_renderer_create
    accepts that b2d_view_init never makes (F = 2 at full width, F far above W)."""
    from rust_doom_b200 import _lib
    out = []
    for (w, h, fov) in ((320, 200, 65), (1920, 1080, 65), (3840, 2160, 65), (1920, 64, 110), (1300, 30, 110),
                        (1000, 10, 65), (640, 40, 100), (333, 2, 65), (4096, 2, 65), (4096, 2, 95.5), (4096, 2, 1.01),
                        (4096, 2160, 169.9), (4096, 2160, 1.01), (64, 48, 169.9), (1, 2, 65)):
        out.append(("%dx%d@%g" % (w, h, fov), b2d.make_view(w, h, fov)))
    for (w, h, F, FY2) in ((4096, 2160, 2, 2), (4096, 2, 2, 3), (4096, 300, 4096, 300), (2048, 8, (1 << 31) - 1, 2),
                           (3, 2, 2, 2)):
        out.append(("%dx%d F=%d" % (w, h, F), _lib.View(w, h, F, FY2)))
    return out


def test_plane_dir_is_exact_at_every_accepted_view(b2d, hostcheck):
    """Product (b2d_math.cuh plane_dir, run through hostcheck) and oracle give the exact C8 direction for every column at
    every octant boundary +-1 BAM and random yaws; the exact value always fits the int32 the texel rule multiplies."""
    import ctypes
    lib = hostcheck.lib
    pose = np.zeros(1, dtype=b2d.POSE_DTYPE)
    worst = 0
    for name, v in _accepted_views(b2d):
        W, F = v.width, v.F
        for angle in angles_at_octants(len(name) * 131 + W, 8):
            pose["angle"] = angle
            cosq, sinq = render.sincos_q30(angle)
            ax, ay = c8_dirs(cosq, sinq, W, F)
            worst = max(worst, int(np.abs(ax).max()), int(np.abs(ay).max()))
            prod = np.zeros((W, 2), dtype=np.int32)
            lib.hostcheck_plane_dirs(ctypes.byref(v), ctypes.c_void_p(pose.ctypes.data), ctypes.c_void_p(prod.ctypes.data))
            orc = render.plane_dirs(oracle_view(v), angle)
            for who, got in (("product", prod), ("oracle", orc)):
                bad = np.nonzero((got[:, 0] != ax) | (got[:, 1] != ay))[0]
                assert len(bad) == 0, "%s, %s, angle %#x: %d columns differ from exact C8, first x=%d (%s vs %d,%d)" % (
                    who, name, angle, len(bad), bad[0], got[bad[0]].tolist(), ax[bad[0]], ay[bad[0]])
    assert worst < (1 << 30)


# ---- 2. flat pixels on wide views ----------------------------------------------------------------------------------
ROOM = 16384          # half-extent of the flats level, map units


def flats_level() -> bytes:
    """Two rooms A (x in [-ROOM, 0]) and B (x in [0, ROOM]), y in [0, ROOM], sharing an untextured two-sided line at x=0;
    same heights (floor 0, ceiling 256), different floor and ceiling flats, static light.  Everything inside the
    rectangle is floor or ceiling, so which flat a pixel shows follows from where its ray meets the plane."""
    import struct
    from rust_doom_b200 import synthwad as G
    rng = G.SplitMix64(9)
    playpal = G.make_playpal()
    patches, tex, flats = G.make_graphics(rng)
    pn, t1 = G.make_pnames_texture1(list(patches.keys()), tex)
    R = ROOM
    V = [(-R, 0), (0, 0), (0, R), (-R, R), (R, 0), (R, R)]
    secs = [G.Sector(0, 256, "FLOOR1", "CEIL1", 160), G.Sector(0, 256, "FLOOR4", "CEIL3", 200)]
    sides = [G.Sidedef(0, 0, "-", "-", "BRICK1", 0) for _ in range(3)] + \
            [G.Sidedef(0, 0, "-", "-", "BRICK1", 1) for _ in range(3)] + \
            [G.Sidedef(0, 0, "-", "-", "-", 0), G.Sidedef(0, 0, "-", "-", "-", 1)]
    L = [G.Linedef(0, 3, 1, 0, 0, 0, -1), G.Linedef(3, 2, 1, 0, 0, 1, -1), G.Linedef(1, 0, 1, 0, 0, 2, -1),
         G.Linedef(2, 5, 1, 0, 0, 3, -1), G.Linedef(5, 4, 1, 0, 0, 4, -1), G.Linedef(4, 1, 1, 0, 0, 5, -1),
         G.Linedef(2, 1, 0x0004, 0, 0, 6, 7)]
    segsA = [(0, 3, 0, 0), (3, 2, 1, 0), (1, 0, 2, 0), (2, 1, 6, 0)]
    segsB = [(2, 5, 3, 0), (5, 4, 4, 0), (4, 1, 5, 0), (1, 2, 6, 1)]
    lb = struct.pack
    lumps = [("PLAYPAL", playpal), ("COLORMAP", G.make_colormap(playpal)), ("E1M1", b""),
             ("THINGS", lb("<hhhHH", -R // 2, R // 2, 0, 1, 7)),
             ("LINEDEFS", b"".join(lb("<HHHHHhh", l.v1, l.v2, l.flags, 0, 0, l.right, l.left) for l in L)),
             ("SIDEDEFS", b"".join(lb("<hh8s8s8sH", s.xoff, s.yoff, G._name8(s.upper), G._name8(s.lower), G._name8(s.middle), s.sector) for s in sides)),
             ("VERTEXES", b"".join(lb("<hh", *v) for v in V)),
             ("SEGS", b"".join(lb("<HHHHHH", a, b, 0, l, d, 0) for (a, b, l, d) in segsA + segsB)),
             ("SSECTORS", lb("<HH", 4, 0) + lb("<HH", 4, 4)),
             ("NODES", lb("<hhhh4h4hHH", 0, 0, 0, R, R, 0, 0, R, R, 0, -R, 0, 0x8001, 0x8000)),
             ("SECTORS", b"".join(lb("<hh8s8shHH", s.floor, s.ceil, G._name8(s.floor_flat), G._name8(s.ceil_flat), s.light, 0, 0) for s in secs)),
             ("TEXTURE1", t1), ("PNAMES", pn)] + list(patches.items()) + \
            [("S_START", b""), ("S_END", b""), ("F_START", b"")] + list(flats.items()) + [("F_END", b"")]
    return G.assemble_wad(lumps)


def flats_poses():
    R = ROOM
    P = [(-R / 2, R / 2, 41, 0.0), (-R / 2, R / 2, 41, 45.0), (-R / 3, R / 4, 41, 90.0 + 360.0 / 2 ** 32),
         (-100, R / 2, 41, 3.7), (-100, R / 2, 200, 183.2), (R / 3, R / 3, 0.5, 300.0), (R / 2, 2 * R / 3, 255.75, 222.0),
         (-R / 4, R / 5, 128, 135.0)]
    out = np.zeros(len(P), dtype=render.POSE)
    for i, (x, y, z, a) in enumerate(P):
        out[i] = (int(round(x * 65536)), int(round(y * 65536)), int(round(z * 65536)), bam(a))
    return out


FLAT_VIEWS = [(1000, 10, 65.0), (1920, 64, 110.0), (4096, 30, 65.0), (333, 2, 65.0), (4096, 2, 95.5), (320, 200, 65.0)]


def c8_flat_pixels(blob: bytes, view: render.View, pose):
    """(mask, expected) for one frame of flats_level(): every pixel whose floor / ceiling sample point lies clearly
    inside one of the two rooms (2 % + 2 units away from every wall and from the shared line), with the colour the C8
    texel rule and the C9 light rule give it, computed here with exact integers."""
    h = S.header(blob)
    flats = np.frombuffer(blob, dtype=np.uint8, count=h[S.H_NFLATS] * 4096, offset=h[S.H_OFF_FLATS])
    cmap = np.frombuffer(blob, dtype=np.uint8, count=32 * 256, offset=h[S.H_OFF_COLORMAP])
    sectors = S.section(blob, "sectors")
    W, H, F, FY2 = view.W, view.H, view.F, view.FY2
    px, py, pz, angle = int(pose["x"]), int(pose["y"]), int(pose["z"]), int(pose["angle"])
    cosq, sinq = render.sincos_q30(angle)
    ax, ay = c8_dirs(cosq, sinq, W, F)
    mask = np.zeros((H, W), dtype=bool)
    want = np.zeros((H, W), dtype=np.uint8)
    ex, ey = px / 65536.0, py / 65536.0
    assert all(int(sec[0]) == 0 and int(sec[1]) == 256 for sec in sectors)
    lrows = [None, None]
    for y in range(H):
        r2 = 2 * y + 1 - H
        if r2 == 0:
            continue
        floor = r2 > 0                               # below the horizon: floor, above: ceiling
        hgt = 0 if floor else 256
        if floor != ((hgt << 16) < pz):              # the eye is on the far side of that plane: not drawn on this row
            continue
        hrel = max(-(1 << 27), min(1 << 27, (hgt << 16) - pz))
        yslope = (FY2 << 16) // abs(r2)
        z16 = min((abs(hrel) * yslope) >> 16, 0x7FFFFFFF)
        z8q, z8 = z16 >> 8, min(z16 >> 13, 65535)
        U = (px << 10) + z8q * ax                   # Q26, unwrapped: the sample point itself
        V = (py << 10) + z8q * ay
        wx, wy = U / 2.0 ** 26, V / 2.0 ** 26
        margin = 0.02 * np.hypot(wx - ex, wy - ey) + 2.0
        inside = (wx > -ROOM + margin) & (wx < ROOM - margin) & (wy > margin) & (wy < ROOM - margin) & (np.abs(wx) > margin)
        sec = (wx > 0).astype(np.int64)              # room A = sector 0, room B = sector 1
        flat_id = sectors[sec, 2 if floor else 3].astype(np.int64)
        for k in range(2):
            lrows[k] = int(light_row(int(sectors[k, 4]), np.array([z8]))[0])
        rows = np.where(sec == 0, lrows[0], lrows[1])
        Uw, Vw = U & 0xFFFFFFFF, V & 0xFFFFFFFF
        texel = flats[flat_id * 4096 + (((Uw >> 26) << 6) | (Vw >> 26))].astype(np.int64)
        mask[y] = inside
        want[y] = cmap[rows * 256 + texel]
    return mask, want


def assert_flats_follow_c8(blob, view, poses, frames, who):
    checked = 0
    for i in range(len(poses)):
        mask, want = c8_flat_pixels(blob, view, poses[i])
        bad = mask & (frames[i] != want)
        assert not bad.any(), "%s %dx%d F=%d pose %d: %d of %d flat pixels differ from C8, first (y, x) = %s" % (
            who, view.W, view.H, view.F, i, int(bad.sum()), int(mask.sum()), np.argwhere(bad)[0].tolist())
        checked += int(mask.sum())
    assert checked >= view.W, "too few flat pixels checked (%d)" % checked


@pytest.fixture(scope="module")
def flats_blob(b2d):
    data = flats_level()
    blob = b2d.Scene(b2d.Archive.from_bytes(data), 0).blob
    from tests.conftest import oracle_blob
    assert blob == oracle_blob(data, 0)
    assert S.header(blob)[S.H_NANIM] == 0
    return blob


@pytest.mark.parametrize("w,h,fov", FLAT_VIEWS, ids=["%dx%d@%g" % v for v in FLAT_VIEWS])
def test_flat_pixels_follow_c8_at_wide_views_cpu(b2d, hostcheck, flats_blob, w, h, fov):
    """Oracle frames and the product's maths (hostcheck) at low, wide views: every clear floor / ceiling pixel equals the
    big-integer C8 texel rule -- the check that does not rest on the two sharing an expression."""
    poses = flats_poses()
    oview = render.make_view(w, h, fov)
    ofb = render.render(flats_blob, oview, poses, threads=4)
    assert_flats_follow_c8(flats_blob, oview, poses, ofb, "oracle")
    hfb, _, _ = hostcheck(flats_blob, b2d.make_view(w, h, fov), poses)
    assert_flats_follow_c8(flats_blob, oview, poses, hfb, "hostcheck")
    assert np.array_equal(hfb, ofb)


@pytest.mark.gpu
def test_gpu_flat_pixels_follow_c8_at_wide_views(b2d, flats_blob):
    sc = b2d.Scene(b2d.Archive.from_bytes(flats_level()), 0)
    poses = flats_poses()
    for (w, h, fov) in FLAT_VIEWS:
        oview = render.make_view(w, h, fov)
        gfb = b2d.Renderer(sc, b2d.make_view(w, h, fov), max_batch=len(poses)).render(poses)
        _assert_same(render.render(flats_blob, oview, poses, threads=8), gfb, "%dx%d" % (w, h))
        assert_flats_follow_c8(flats_blob, oview, poses, gfb, "GPU")


# ---- shared helpers of the GPU tests -------------------------------------------------------------------------------
def _assert_same(ofb, gfb, what=""):
    bad = [(i, int((ofb[i] != gfb[i]).sum())) for i in range(len(ofb)) if not np.array_equal(ofb[i], gfb[i])]
    assert not bad, "%s: frames differ (index, pixels): %s" % (what, bad[:6])


def _threads():
    return len(os.sched_getaffinity(0))


def _rich_level(b2d, seed=5):
    """Masked middles, sprites, animation, scrolling, odd texture sizes."""
    from rust_doom_b200 import synthwad
    cfg = synthwad.SynthConfig(mid_pct=30, thing_pct=50, anim=True, odd_tex=True)
    return b2d.Scene(b2d.Archive.from_bytes(synthwad.build_iwad(seed, ("E1M1",), cfg=cfg)), 0)


class _env:
    """Environment variables set for the duration of a block (the renderer reads its A/B switches at creation)."""

    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        os.environ.update(self.kv)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ---- 3. the walk's persistent grid ---------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_persistent_walk_grid(b2d, hostcheck):
    """b2d_walk_device with n > 148 runs 148 CTAs that loop over frames, reusing their shared memory (column mask, stack,
    list, count) and waiting on the bulk copy of the traversal tables only for their first frame.  Two batches in flight
    on a walk and a raster stream, at n = 148 (one frame per CTA), 149, 297 (three frames for CTA 0) and 1000: every frame
    equals the oracle, the last batch's worklists equal hostcheck's, and a renderer without the persistent grid
    (B2D_TUNE=4: a CTA per frame) gives the same worklists and frames."""
    import torch
    sc = _rich_level(b2d)
    tics = 1234
    poses = sample_poses(b2d, sc, 1000, 71)
    view, oview = b2d.make_view(320, 200), render.make_view(320, 200)
    ofb = render.render(sc.blob, oview, poses, threads=_threads(), tics=tics)
    _, hcounts, hids = hostcheck(sc.blob, view, poses, tics=tics)
    assert (hcounts > 0).all() and any((hids[i, :hcounts[i]] < 0).any() for i in range(1000)), "no sprite entries"
    dp_all = torch.from_numpy(poses.view(np.int32).reshape(-1, 4).copy()).cuda()
    results = {}
    for tune in ("0", "4"):
        with _env(B2D_TUNE=tune):
            r = b2d.Renderer(sc, view, max_batch=1000)
        r.set_time(tics)
        s_walk, s_raster = torch.cuda.Stream(priority=-1), torch.cuda.Stream()
        for n in (148, 149, 297, 1000):
            idx = [(np.arange(n) + off) % 1000 for off in (1000 - n, 337)]          # batches A and B
            dps = [dp_all[torch.from_numpy(i).cuda()].contiguous() for i in idx]
            outs = [torch.full((n, 200, 320), 0xAB, dtype=torch.uint8, device="cuda") for _ in idx]
            torch.cuda.synchronize()
            ta = r.walk_device(dps[0].data_ptr(), n, s_walk.cuda_stream)
            tb = r.walk_device(dps[1].data_ptr(), n, s_walk.cuda_stream)           # walks while A rasters
            r.raster_device(ta, outs[0].data_ptr(), 0, s_raster.cuda_stream)
            r.raster_device(tb, outs[1].data_ptr(), 0, s_raster.cuda_stream)
            torch.cuda.synchronize()
            assert r.status() == 0
            counts, ids = r.worklist(n)                                              # batch B (last walked)
            ib = idx[1]
            assert counts.tolist() == hcounts[ib].tolist(), "B2D_TUNE=%s n=%d: worklist lengths" % (tune, n)
            for k in range(n):
                assert ids[k, :counts[k]].tolist() == hids[ib[k], :hcounts[ib[k]]].tolist(), \
                    "B2D_TUNE=%s n=%d frame %d (pose %d): worklist" % (tune, n, k, ib[k])
            frames = [o.cpu().numpy() for o in outs]
            for j in range(2):
                _assert_same(ofb[idx[j]], frames[j], "B2D_TUNE=%s n=%d batch %s" % (tune, n, "AB"[j]))
            results[(tune, n)] = (counts, ids, frames)
    for n in (148, 149, 297, 1000):
        c0, i0, f0 = results[("0", n)]
        c4, i4, f4 = results[("4", n)]
        assert np.array_equal(c0, c4) and np.array_equal(i0, i4)
        assert all(np.array_equal(a, b) for a, b in zip(f0, f4))


# ---- 4. raster instantiations --------------------------------------------------------------------------------------
_KERNEL = re.compile(r"b2d_raster_kernel<(true|false), *\d+, *(\d+), *\d+, *(true|false)>")


def expected_instantiation(width: int, rgba: bool, masked: bool, generic_w: bool = False):
    """launch_raster's choice: (rgba, compile-time width or 0, masked)."""
    kw = 0
    if not generic_w and width == 1920:
        kw = 1920
    elif not generic_w and width == 3840 and not rgba:
        kw = 3840
    return (rgba, kw, masked)


def launched_instantiations(fn):
    """Run fn() under the CUDA profiler; the raster kernel instantiations it launched, from their demangled names."""
    import json
    import tempfile
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:          # the raw trace lists every kernel, with or without a torch op
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    names = {e.get("name", "") for e in events if "b2d_raster_kernel" in e.get("name", "")}
    got = set()
    for nm in names:
        m = _KERNEL.search(nm)
        assert m, "cannot read the instantiation from kernel name %r" % nm
        got.add((m.group(1) == "true", int(m.group(2)), m.group(3) == "true"))
    return got


def _matrix_scenes(b2d):
    from rust_doom_b200 import synthwad
    plain = b2d.Scene(b2d.Archive.from_bytes(synthwad.build_iwad(1, ("E1M1",))), 0)
    masked = b2d.Scene(b2d.Archive.from_bytes(synthwad.build_iwad(3, ("E1M1",), cfg=synthwad.SynthConfig(mid_pct=35, thing_pct=40))), 0)
    assert plain.info.n_masked_mids == 0 and plain.info.n_sprites == 0
    assert masked.info.n_masked_mids > 0 and masked.info.n_sprites > 0
    return {"plain": plain, "masked": masked}


def _check_case(b2d, sc, w, h, rgba, poses, what):
    r = b2d.Renderer(sc, b2d.make_view(w, h), max_batch=len(poses))
    out = {}
    got = launched_instantiations(lambda: out.setdefault("fb", r.render(poses, rgba=rgba)))
    res = render.render(sc.blob, render.make_view(w, h), poses, rgba=rgba, threads=_threads())
    if rgba:
        _assert_same(res[0], out["fb"][0], what)
        assert np.array_equal(res[1], out["fb"][1]), what + ": RGBA"
    else:
        _assert_same(res, out["fb"], what)
    return got


MATRIX = [(w, h, rgba) for (w, h) in ((1920, 1080), (3840, 2160), (640, 400)) for rgba in (False, True)
          if not (w == 3840 and rgba)]


@pytest.mark.gpu
def test_gpu_every_raster_instantiation_matches_oracle(b2d):
    """All 10 instantiations: {index, RGBA} x {1920, 3840 (index only), generic width} x {plain, masked}, each run with
    3 poses against the oracle; the instantiation that ran is read from the profiler's kernel name."""
    scenes = _matrix_scenes(b2d)
    seen = set()
    for kind, sc in scenes.items():
        poses = sample_poses(b2d, sc, 3, 211)
        for (w, h, rgba) in MATRIX:
            want = expected_instantiation(w, rgba, kind == "masked")
            got = _check_case(b2d, sc, w, h, rgba, poses, "%s %dx%d %s" % (kind, w, h, "rgba" if rgba else "index"))
            assert got == {want}, "%s %dx%d rgba=%s ran %s" % (kind, w, h, rgba, got)
            seen.add(want)
    assert len(seen) == 10


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"B2D_TUNE": "1"}, {"B2D_TUNE": "2"}, {"B2D_NO_VMM": "1"}],
                         ids=["tune1_general_wall_paths", "tune2_8row_fast_loop", "no_vmm_flats"])
def test_gpu_raster_switches_match_oracle(b2d, env):
    """The wall paths the incremental 16-row loop normally shadows (B2D_TUNE=1: re-anchored word and byte-load forms;
    B2D_TUNE=2: 8-row batches), and the plain 4 GiB-over-allocation behind the pre-lit flats (B2D_NO_VMM=1), at 1080p and
    4K on the masked level, index and RGBA."""
    sc = _matrix_scenes(b2d)["masked"]
    poses = sample_poses(b2d, sc, 3, 223)
    for (w, h, rgba) in ((1920, 1080, False), (1920, 1080, True), (3840, 2160, False)):
        with _env(**env):
            r = b2d.Renderer(sc, b2d.make_view(w, h), max_batch=3)
        got = r.render(poses, rgba=rgba)
        want = render.render(sc.blob, render.make_view(w, h), poses, rgba=rgba, threads=_threads())
        what = "%s %dx%d rgba=%s" % (env, w, h, rgba)
        if rgba:
            _assert_same(want[0], got[0], what)
            assert np.array_equal(want[1], got[1]), what
        else:
            _assert_same(want, got, what)


_GENERIC_W_CHILD = r"""
import sys
sys.path.insert(0, sys.argv[1])
import rust_doom_b200 as b2d
from tests import test_contract_edges as T
scenes = T._matrix_scenes(b2d)
for kind, sc in scenes.items():
    poses = T.sample_poses(b2d, sc, 2, 227)
    for (w, h, rgba) in T.MATRIX:
        if w == 640:
            continue
        got = T._check_case(b2d, sc, w, h, rgba, poses, "generic-width %s %dx%d rgba=%s" % (kind, w, h, rgba))
        assert got == {T.expected_instantiation(w, rgba, kind == "masked", generic_w=True)}, got
print("generic width ok")
"""


@pytest.mark.gpu
def test_gpu_raster_generic_width_switch():
    """B2D_RASTER_GENERIC_W (cached once per process): 1080p and 4K through the generic-width instantiations."""
    env = dict(os.environ, B2D_RASTER_GENERIC_W="1")
    res = subprocess.run([sys.executable, "-c", _GENERIC_W_CHILD, ROOT], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    assert "generic width ok" in res.stdout


# ---- 5. adversarial poses ------------------------------------------------------------------------------------------
def adversarial_poses(sc) -> np.ndarray:
    """Poses the random generators do not aim at, all inside the level: yaw at each octant boundary and +-1 BAM; the
    eye exactly on a BSP partition line and on a vertex; 1/65536 above a floor and below a ceiling; more than 2048
    units above or below every plane (the +-2^27 clamps of wall_hrel / plane_habs); standing against a one-sided wall
    (near clamp, scale cap)."""
    blob = sc.blob
    verts = S.section(blob, "verts")
    nodes = S.section(blob, "nodes")
    segs = S.section(blob, "segs")
    out = []

    def add(x16, y16, z16, angle):
        out.append((int(x16), int(y16), int(z16), int(angle) & 0xFFFFFFFF))

    def floor_ceil(x16, y16):
        sec, fl, cl = sc.sector_at(x16 / 65536.0, y16 / 65536.0)
        return (fl, cl) if sec >= 0 and fl < cl else None

    base = sc.start_pose[0]
    bx, by = int(base["x"]), int(base["y"])
    fc = floor_ceil(bx, by)
    assert fc is not None
    for k in range(8):
        for d in (-1, 0, 1):
            add(bx, by, (fc[0] + 41) << 16, k * BAM_OCTANT + d)
    on_line = 0
    for nd in nodes:                      # partition start point and midpoint, looking along and across the line
        x, y, dx, dy = (int(v) for v in nd[:4])
        for (px, py) in ((x << 16, y << 16), ((x << 16) + (dx << 15), (y << 16) + (dy << 15))):
            fcp = floor_ceil(px, py)
            if fcp is None or on_line >= 6:
                continue
            a = bam(math.degrees(math.atan2(dy, dx)))
            add(px, py, (fcp[0] + 41) << 16, a)
            add(px, py, (fcp[0] + 41) << 16, a + (1 << 30))
            on_line += 1
    on_vertex = 0
    for v in verts:
        fcv = floor_ceil(int(v[0]) << 16, int(v[1]) << 16)
        if fcv is None or on_vertex >= 4:
            continue
        add(int(v[0]) << 16, int(v[1]) << 16, (fcv[0] + 30) << 16, bam(37.0 + 90 * on_vertex))
        on_vertex += 1
    assert on_line >= 2 and on_vertex >= 2
    add(bx, by, (fc[0] << 16) + 1, bam(10.0))
    add(bx, by, (fc[1] << 16) - 1, bam(190.0))
    assert -3000 < sc.info.min_height <= sc.info.max_height < 3000
    add(bx, by, (sc.info.max_height + 2100) << 16, bam(75.0))
    add(bx, by, (sc.info.min_height - 2100) << 16, bam(255.0))
    walls = 0
    for s in segs:                        # one-sided walls, from 1/65536 and 1/16 units in front, facing them and along them
        if int(s[3]) & (S.SEG_TWO_SIDED | S.SEG_INVALID) or walls >= 4:
            continue
        (x1, y1), (x2, y2) = verts[int(s[0])], verts[int(s[1])]
        dx, dy = int(x2) - int(x1), int(y2) - int(y1)
        ln = math.hypot(dx, dy)
        if ln < 64:
            continue
        for eps in (1.0 / 65536, 1.0 / 16):
            mx = (int(x1) + int(x2)) / 2.0 + eps * dy / ln            # the front (right) side of v1 -> v2
            my = (int(y1) + int(y2)) / 2.0 - eps * dx / ln
            fcw = floor_ceil(round(mx * 65536), round(my * 65536))
            if fcw is None:
                break
            face = bam(math.degrees(math.atan2(dx, -dy)))
            add(round(mx * 65536), round(my * 65536), (fcw[0] + 41) << 16, face)
            add(round(mx * 65536), round(my * 65536), (fcw[0] + 41) << 16, bam(math.degrees(math.atan2(dy, dx))) + 7)
        else:
            walls += 1
    assert walls >= 2
    return np.array(out, dtype=render.POSE)


ADV_VIEWS = [(320, 200), (1920, 1080)]


@pytest.mark.parametrize("w,h", ADV_VIEWS, ids=["%dx%d" % v for v in ADV_VIEWS])
def test_adversarial_poses_hostcheck_matches_oracle(b2d, hostcheck, w, h):
    sc = _rich_level(b2d, 6)
    poses = adversarial_poses(sc)
    hfb, hcounts, _ = hostcheck(sc.blob, b2d.make_view(w, h), poses, tics=77)
    assert (hcounts >= 0).all()
    _assert_same(render.render(sc.blob, render.make_view(w, h), poses, threads=_threads(), tics=77), hfb, "hostcheck")


@pytest.mark.gpu
def test_gpu_adversarial_poses(b2d, hostcheck):
    import torch
    sc = _rich_level(b2d, 6)
    poses = adversarial_poses(sc)
    n = len(poses)
    for (w, h) in ADV_VIEWS:
        view = b2d.make_view(w, h)
        r = b2d.Renderer(sc, view, max_batch=n)
        r.set_time(77)
        dp = torch.from_numpy(poses.view(np.int32).reshape(-1, 4).copy()).cuda()
        out = torch.full((n, h, w), 0xAB, dtype=torch.uint8, device="cuda")
        r.render_device(dp.data_ptr(), n, out.data_ptr())
        torch.cuda.synchronize()
        assert r.status() == 0
        counts, ids = r.worklist(n)
        _, hcounts, hids = hostcheck(sc.blob, view, poses, tics=77)
        assert counts.tolist() == hcounts.tolist()
        for i in range(n):
            assert ids[i, :counts[i]].tolist() == hids[i, :hcounts[i]].tolist(), "%dx%d pose %d" % (w, h, i)
        _assert_same(render.render(sc.blob, render.make_view(w, h), poses, threads=_threads(), tics=77),
                     out.cpu().numpy(), "%dx%d" % (w, h))
