"""gsb_render_aux: the per-pixel (opacity, expected depth) planes of a frame, against the CPU reference (tests/aux_oracle.c) and
against gsb_render.  EXACT mode: both planes bit-identical to the oracle's shared-definition exp (mode 1) and the colour
bit-identical to gsb_render's, at every tile-cull level, with and without the captured graph, in every output memory."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import aux_oracle
import scenes

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
CAMS = ["c1", "inside", "odd_size", "tiny", "wide", "away"]


def oracle_aux(o, vtx, u, exp_mode=1, rows=None, probed=False):
    return aux_oracle.render_frame(vtx, u, rows, exp_mode=exp_mode, probed=probed)


def z_max(f):
    live = f["tiles"] > 0
    return float(f["attr"]["depth"][live].max()) if live.any() else 1.0


class Pinned:
    """gsb_host_alloc buffer viewed as a numpy array."""

    def __init__(self, gs, shape, dtype, fill=0):
        self.gs, self.p = gs, C.c_void_p()
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        assert gs.lib.gsb_host_alloc(C.byref(self.p), nbytes) == 0
        self.a = np.frombuffer((C.c_char * nbytes).from_address(self.p.value), dtype).reshape(shape)
        self.a.view(np.uint8)[...] = fill

    def free(self):
        self.gs.lib.gsb_host_free(self.p)


@pytest.mark.parametrize("cam", CAMS)
def test_aux_exact_matches_oracle_and_keeps_the_colour(gs, oracle, ctx, cam):
    _, vtx, _ = scenes.c1()
    u = scenes.camera(cam)
    ctx.set_mode(gs.MODE_EXACT)
    ctx.set_debug(True)
    ctx.upload(vtx)
    try:
        img = ctx.render(u, gs.FORMAT_RGBA32F)
        consumed = ctx.stats().blend_consumed
        img_a, aux = ctx.render_aux(u, gs.FORMAT_RGBA32F)
        st = ctx.stats()
    finally:
        ctx.set_debug(False)
    ref = oracle_aux(oracle, vtx, u)
    assert aux.shape == (u.height, u.width, 2) and aux.dtype == np.float32
    assert np.array_equal(aux, ref["aux"]), cam
    assert np.array_equal(img_a, img) and np.array_equal(img_a, ref["rgba"]), cam
    assert st.blend_consumed == consumed == int(ref["consumed"].sum()), cam


def test_aux_is_identical_across_cull_levels_graph_and_formats(gs, oracle, ctx):
    _, vtx, _ = scenes.c1()
    ctx.set_mode(gs.MODE_EXACT)
    ctx.upload(vtx)
    for cam in ("c1", "odd_size", "wide"):
        u = scenes.camera(cam)
        ref = oracle_aux(oracle, vtx, u)["aux"]
        try:
            ctx.set_timers(False)  # the captured middle graph is used only with timers and debug off
            for level in (0, 1, 2):
                ctx.set_tile_cull(level)
                for graph in (True, False):
                    ctx.set_graph(graph)
                    for fmt in (gs.FORMAT_RGBA32F, gs.FORMAT_BGRA8):
                        img, aux = ctx.render_aux(u, fmt)
                        assert np.array_equal(aux, ref), (cam, level, graph, fmt)
                        assert np.array_equal(img, ctx.render(u, fmt)), (cam, level, graph, fmt)
        finally:
            ctx.set_tile_cull(0)
            ctx.set_graph(True)
            ctx.set_timers(True)


def test_aux_fast_mode_within_tolerance(gs, oracle, ctx):
    _, vtx, _ = scenes.c1()
    ctx.upload(vtx)
    for cam in ("c1", "inside", "odd_size"):
        u = scenes.camera(cam)
        ctx.set_mode(gs.MODE_FAST)
        try:
            _, aux = ctx.render_aux(u, gs.FORMAT_RGBA32F)
        finally:
            ctx.set_mode(gs.MODE_EXACT)
        ref, near_step = oracle_aux(oracle, vtx, u, exp_mode=0, probed=True)
        keep = ~near_step
        assert near_step.mean() < 0.05
        assert np.abs(aux[..., 0] - ref["aux"][..., 0])[keep].max() <= 1e-4, cam
        assert np.abs(aux[..., 1] - ref["aux"][..., 1])[keep].max() <= 1e-4 * z_max(ref), cam


def test_aux_bands_concatenate_to_the_frame(gs, oracle, ctx):
    _, vtx, u = scenes.c1()
    ctx.set_mode(gs.MODE_EXACT)
    ctx.upload(vtx)
    full_img, full = ctx.render_aux(u)
    tiles_y = (u.height + 15) // 16
    for parts in (2, 3, 4):
        rows = [(tiles_y * k // parts, tiles_y * (k + 1) // parts) for k in range(parts)]
        bands = [ctx.render_aux(u, rows=r) for r in rows]
        assert np.array_equal(np.concatenate([b[1] for b in bands], axis=0), full), parts
        assert np.array_equal(np.concatenate([b[0] for b in bands], axis=0), full_img), parts
    r = (tiles_y // 3, 2 * tiles_y // 3)
    _, band = ctx.render_aux(u, rows=r)
    ref = oracle_aux(oracle, vtx, u, rows=r)
    assert np.array_equal(band, ref["aux"][r[0] * 16:min(u.height, r[1] * 16)])


@pytest.mark.parametrize("fmt_name", ["FORMAT_RGBA32F", "FORMAT_BGRA8"])
def test_aux_output_memory(gs, ctx, fmt_name):
    """Device, pageable host and page-locked host buffers give the same planes; a padded aux pitch leaves the padding
    alone; a page-locked colour buffer with a pageable aux plane works, and the reverse."""
    import torch
    fmt = getattr(gs, fmt_name)
    _, vtx, _ = scenes.c1()
    ctx.set_mode(gs.MODE_EXACT)
    ctx.upload(vtx)
    for cam in ("c1", "odd_size", "tiny"):
        u = scenes.camera(cam)
        H, W = u.height, u.width
        dt = np.float32 if fmt == gs.FORMAT_RGBA32F else np.uint8
        tdt = torch.float32 if fmt == gs.FORMAT_RGBA32F else torch.uint8
        dev_img = torch.zeros((H, W, 4), dtype=tdt, device="cuda:0")
        dev_aux = torch.zeros((H, W, 2), dtype=torch.float32, device="cuda:0")
        ctx.render_aux_into(u, dev_img.data_ptr(), dev_aux.data_ptr(), fmt)
        torch.cuda.synchronize()
        ref_img, ref_aux = dev_img.cpu().numpy(), dev_aux.cpu().numpy()
        assert np.array_equal(ref_img, ctx.render(u, fmt)), cam
        img, aux = ctx.render_aux(u, fmt)  # pageable numpy buffers
        assert np.array_equal(img, ref_img) and np.array_equal(aux, ref_aux), cam
        # page-locked colour and aux; aux rows padded by 40 bytes that must stay untouched
        pitch_f = W * 2 + 10  # floats per padded aux row (a multiple of 8 bytes)
        p_img, p_aux = Pinned(gs, (H, W, 4), dt), Pinned(gs, (H, pitch_f), np.float32, fill=0xAB)
        try:
            ctx._ck(gs.lib.gsb_render_aux(ctx.h, C.byref(u), 0, gs.ALL_ROWS, p_img.p, 0, p_aux.p, pitch_f * 4, gs.MEM_HOST, fmt,
                                          None))
            assert np.array_equal(p_img.a, ref_img), cam
            assert np.array_equal(p_aux.a[:, :W * 2].reshape(H, W, 2), ref_aux), cam
            assert np.all(p_aux.a[:, W * 2:].view(np.uint8) == 0xAB), cam
            # page-locked colour + pageable aux, and pageable colour + page-locked aux
            np_aux = np.full((H, W, 2), -1.0, np.float32)
            p_img.a[...] = 0
            ctx._ck(gs.lib.gsb_render_aux(ctx.h, C.byref(u), 0, gs.ALL_ROWS, p_img.p, 0, np_aux.ctypes.data, 0, gs.MEM_HOST, fmt,
                                          None))
            assert np.array_equal(p_img.a, ref_img) and np.array_equal(np_aux, ref_aux), cam
            np_img = np.zeros((H, W, 4), dt)
            p_aux.a.view(np.uint8)[...] = 0xAB
            ctx._ck(gs.lib.gsb_render_aux(ctx.h, C.byref(u), 0, gs.ALL_ROWS, np_img.ctypes.data, 0, p_aux.p, pitch_f * 4,
                                          gs.MEM_HOST, fmt, None))
            assert np.array_equal(np_img, ref_img) and np.array_equal(p_aux.a[:, :W * 2].reshape(H, W, 2), ref_aux), cam
            assert np.all(p_aux.a[:, W * 2:].view(np.uint8) == 0xAB), cam
        finally:
            p_img.free()
            p_aux.free()
        # padded aux pitch in device memory too
        dev_pad = torch.full((H, pitch_f), float("nan"), dtype=torch.float32, device="cuda:0")
        ctx.render_aux_into(u, dev_img.data_ptr(), dev_pad.data_ptr(), fmt, aux_row_pitch=pitch_f * 4)
        torch.cuda.synchronize()
        pad = dev_pad.cpu().numpy()
        assert np.array_equal(pad[:, :W * 2].reshape(H, W, 2), ref_aux) and np.isnan(pad[:, W * 2:]).all(), cam


def test_aux_arena_regrow(gs, oracle):
    _, vtx, u = scenes.c1(n=3000)
    small, roomy = gs.Context(0), gs.Context(0)
    try:
        small.upload(vtx)  # the arena starts at max(N, 1024) = 3000 < M
        roomy.upload(vtx)
        roomy.reserve(1 << 20)
        img, aux = small.render_aux(u)
        st = small.stats()
        img_r, aux_r = roomy.render_aux(u)
        assert st.regrow_count >= 1 and roomy.stats().regrow_count == 0
        assert np.array_equal(aux, aux_r) and np.array_equal(img, img_r)
        assert np.array_equal(aux, oracle_aux(oracle, vtx, u)["aux"])
    finally:
        small.close()
        roomy.close()


def test_aux_errors(gs):
    c = gs.Context(0)
    try:
        u = scenes.camera("c1")
        img = np.zeros((u.height, u.width, 4), np.float32)
        aux = np.zeros((u.height, u.width + 1, 2), np.float32)

        def call(aux_ptr, aux_pitch):
            return gs.lib.gsb_render_aux(c.h, C.byref(u), 0, gs.ALL_ROWS, img.ctypes.data, 0, aux_ptr, aux_pitch, gs.MEM_HOST,
                                         gs.FORMAT_RGBA32F, None)

        assert call(aux.ctypes.data, 0) == gs.ERR_NO_SCENE
        c.upload(scenes.c1(n=10)[1])
        assert call(None, 0) == gs.ERR_INVALID
        assert call(aux.ctypes.data, 8 * u.width - 8) == gs.ERR_INVALID  # shorter than a row
        assert call(aux.ctypes.data, 8 * u.width + 4) == gs.ERR_INVALID  # not a multiple of 8
        assert call(aux.ctypes.data, 8 * u.width + 8) == gs.OK
        assert call(aux.ctypes.data, 0) == gs.OK
    finally:
        c.close()
    g = gs.Group([0, 0])
    try:
        g.upload(scenes.c1(n=100)[1])
        r0 = g.context(0)
        with pytest.raises(gs.GsbError) as e:
            r0.render_aux(scenes.camera("c1"))
        assert e.value.code == gs.ERR_INVALID
    finally:
        g.close()


def test_aux_full_size_garden_bands_match_oracle(gs, oracle):
    """bench.py's headline workload (garden stand-in, pose 3) with coarse bins: the list lengths of a real frame through
    the coarse-bin / TMA staging path.  Three oracle bands: top, densest middle, bottom."""
    sys.path.insert(0, str(ROOT))
    import bench
    wl = bench.WORKLOADS["garden-standin"]
    vtx = bench.make_scene(gs, wl)
    u = bench.cameras(gs, wl)[3]
    cov = oracle.cov3d(vtx)
    tiles_y = (wl["h"] + 15) // 16
    c = gs.Context(0)
    try:
        c.set_mode(gs.MODE_EXACT)
        c.set_tile_cull(2)
        c.upload(vtx)
        for rows in [(1, 2), (tiles_y // 2 - 1, tiles_y // 2 + 1), (tiles_y - 2, tiles_y - 1)]:
            oracle.set_exp_mode(1)
            try:
                ref = oracle.render_frame(vtx, cov, u, rows=rows)
            finally:
                oracle.set_exp_mode(0)
            _, ref["aux"] = aux_oracle.blend(ref["attr"], ref["vals"], ref["ranges"], u.width, u.height, rows, exp_mode=1)
            sl = slice(rows[0] * 16, min(u.height, rows[1] * 16))
            img, aux = c.render_aux(u, rows=rows)
            assert np.array_equal(aux, ref["aux"][sl]), rows
            assert np.array_equal(img, ref["rgba"][sl]), rows
            assert (aux[..., 0] > 0).any(), rows  # the band is not empty
    finally:
        c.close()


@pytest.fixture(scope="module")
def ply(gs, tmp_path_factory):
    rec = gs.synth_records(42, 10_000)
    path = tmp_path_factory.mktemp("scene") / "c1.ply"
    gs.write_ply(path, rec)
    return path, gs.activate_records(rec)


def test_host_renderer_render_aux(gs, oracle, ply, ctx):
    path, vtx = ply
    r = gs.HostRenderer(path, device=0, width=640, height=480, fmt=gs.FORMAT_BGRA8)
    try:
        r.set_camera([0, 0, 5], [1, 0, 0, 0])
        img, aux = r.render_aux(640, 480, gs.FORMAT_RGBA32F)
    finally:
        r.close()
    u = gs.uniforms_from_camera([0, 0, 5], [1, 0, 0, 0], 45.0, 0.1, 1000.0, 640, 480)
    ctx.set_mode(gs.MODE_EXACT)
    ctx.upload(vtx)
    img_c, aux_c = ctx.render_aux(u)
    assert np.array_equal(aux, aux_c) and np.array_equal(img, img_c)


def test_headless_viewer_alpha_and_depth_out(gs, oracle, ply, tmp_path):
    path, vtx = ply
    exe = ROOT / "3dgs.cpp_b200" / "gs_viewer_headless"
    alpha, depth = tmp_path / "alpha.pfm", tmp_path / "depth.pfm"
    r = subprocess.run([str(exe), "-w", "640", "-h", "480", "--camera", "0,0,5", "--alpha-out", str(alpha), "--depth-out", str(depth),
                        str(path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1])["gaussians"] == 10_000
    ref = oracle_aux(oracle, vtx, gs.uniforms_from_camera([0, 0, 5], [1, 0, 0, 0], 45.0, 0.1, 1000.0, 640, 480))["aux"]
    head = b"Pf\n640 480\n-1.0\n"
    for f, plane in ((alpha, 0), (depth, 1)):
        blob = f.read_bytes()
        assert blob.startswith(head) and len(blob) == len(head) + 640 * 480 * 4
        got = np.frombuffer(blob[len(head):], "<f4").reshape(480, 640)[::-1]
        assert np.array_equal(got, ref[..., plane]), f.name
