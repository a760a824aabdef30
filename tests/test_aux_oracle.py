"""CPU reference of gsb_render_aux's per-pixel planes (tests/aux_oracle.c): aux[..., 0] = opacity = 1 - T_end,
aux[..., 1] = the un-normalised expected depth D = sum (depth_i * alpha_i) * T_i over the Gaussians that reach
render.comp:87."""
import math

import numpy as np
import pytest

import aux_oracle
import scenes


def oracle_aux(o, vtx, u, exp_mode=0, rows=None, probed=False):
    return aux_oracle.render_frame(vtx, u, rows, exp_mode=exp_mode, probed=probed)


def numpy_aux_pixel(f, px, py):
    """The definition restated: the shader's tests in fp32 (as test_oracle.numpy_blend_pixel), T and D carried in float64."""
    t = (px // 16) + (py // 16) * f["tiles_x"]
    s, e = f["ranges"][t]
    T32, T, D = np.float32(1.0), 1.0, 0.0
    for i in range(s, e):
        a = f["attr"][f["vals"][i]]
        dx, dy = np.float32(a["uv"][0] - np.float32(px)), np.float32(a["uv"][1] - np.float32(py))
        co = a["conic_opacity"]
        power = np.float32(-0.5) * (co[0] * dx * dx + co[2] * dy * dy) - co[1] * dx * dy
        if power > 0:
            continue
        alpha = min(np.float32(0.99), np.float32(co[3] * np.float32(math.exp(power))))
        if alpha < np.float32(1.0 / 255.0):
            continue
        test_T = np.float32(T32 * (np.float32(1) - alpha))
        if test_T < np.float32(0.0001):
            break
        D += float(a["depth"]) * float(alpha) * T
        T *= 1.0 - float(alpha)
        T32 = test_T
    return np.array([1.0 - T, D])


@pytest.mark.parametrize("cam", list(scenes.CAMERAS))
def test_aux_blend_keeps_the_colour(gs, oracle, cam):
    """The reference's colour is gso_blend's, bit for bit, in both exp modes, full frame and band."""
    _, vtx, _ = scenes.c1(n=3000)
    u = scenes.camera(cam)
    tiles_y = (u.height + 15) // 16
    for mode in (0, 1):
        for rows in (None, (tiles_y // 3, tiles_y)):
            f = oracle_aux(oracle, vtx, u, exp_mode=mode, rows=rows)
            assert np.array_equal(f["rgba_aux"], f["rgba"]), (cam, mode, rows)


def test_aux_matches_numpy_on_sampled_pixels(gs, oracle):
    _, vtx, u = scenes.c1(n=3000)
    f = oracle_aux(oracle, vtx, u)
    rng = np.random.default_rng(3)
    covered = 0
    for _ in range(60):
        px, py = int(rng.integers(0, u.width)), int(rng.integers(0, u.height))
        want = numpy_aux_pixel(f, px, py)
        covered += want[0] > 0
        assert np.allclose(f["aux"][py, px], want, rtol=1e-5, atol=2e-6), (px, py, f["aux"][py, px], want)
    assert covered >= 30  # the sample actually exercises covered pixels


@pytest.mark.parametrize("cam", list(scenes.CAMERAS))
def test_aux_invariants(gs, oracle, cam):
    _, vtx, _ = scenes.c1()
    u = scenes.camera(cam)
    f = oracle_aux(oracle, vtx, u, exp_mode=1)
    a, D = f["aux"][..., 0], f["aux"][..., 1]
    assert np.isfinite(f["aux"]).all()
    assert a.min() >= 0.0 and a.max() <= np.float32(0.9999)
    empty = a == 0
    assert np.all(D[empty] == 0) and np.all(f["rgba"][empty][:, :3] == 0)
    live = f["tiles"] > 0
    if not live.any():
        assert np.all(a == 0)
        return
    z = f["attr"]["depth"][live].astype(np.float64)
    z_min, z_max = z.min(), z.max()
    assert z_min > 0
    # D and aux.x are both sums of the same weights alpha_i * T_i, rounded differently in fp32: D carries one rounding
    # per product and per add, 1 - T_end one per transmittance step.  Over the at most ~2350 accumulated Gaussians of a
    # pixel (T >= 1e-4, alpha >= 1/255) that stays far below 1e-4 relative; the slack is that, times z_max.
    slack = 1e-4 * z_max
    a64, D64 = a.astype(np.float64), D.astype(np.float64)
    assert np.all(D64 >= a64 * z_min - slack), (D64 - a64 * z_min).min()
    assert np.all(D64 <= a64 * z_max + slack), (D64 - a64 * z_max).max()


def test_aux_bands_reproduce_the_full_frame(gs, oracle):
    _, vtx, u = scenes.c1(n=3000)
    full = oracle_aux(oracle, vtx, u, exp_mode=1)
    tiles_y = full["tiles_y"]
    for rb, re in [(0, 7), (7, 19), (19, tiles_y)]:
        band = oracle_aux(oracle, vtx, u, exp_mode=1, rows=(rb, re))
        r0, r1 = rb * 16, min(u.height, re * 16)
        assert np.array_equal(band["aux"][r0:r1], full["aux"][r0:r1])
        assert np.array_equal(band["rgba"][r0:r1], full["rgba"][r0:r1])


@pytest.mark.parametrize("cam", ["c1", "inside", "odd_size"])
def test_aux_exp_modes_agree_within_tolerance(gs, oracle, cam):
    """libm exp vs the shared-definition exp, away from the pixels whose step functions sit on a threshold."""
    _, vtx, _ = scenes.c1()
    u = scenes.camera(cam)
    f0, m0 = oracle_aux(oracle, vtx, u, exp_mode=0, probed=True)
    f1, m1 = oracle_aux(oracle, vtx, u, exp_mode=1, probed=True)
    keep = ~(m0 | m1)
    live = f0["tiles"] > 0
    z_max = float(f0["attr"]["depth"][live].max()) if live.any() else 1.0
    assert np.abs(f0["aux"][..., 0] - f1["aux"][..., 0])[keep].max() <= 1e-4
    assert np.abs(f0["aux"][..., 1] - f1["aux"][..., 1])[keep].max() <= 1e-4 * z_max
