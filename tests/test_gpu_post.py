"""GPU parity tests of the stages SURVEY section 8f row N4 names besides multi-channel: the regridding of a
FINER field (oct_zoom_out_float, reference src/oct_zoom.cc:51) and the -srsal post-smoother (oct_srsal_cu,
reference src/oct_srsal_cuda.cu:73), called through the C ABI and compared with the CPU oracle, with the
reference's own CPU object (zoom-out) and with fixtures the reference's CUDA kernel produced (srsal)."""
import numpy as np
import pytest

import cases
import octane_b200 as ob
from conftest import load_golden

pytestmark = pytest.mark.gpu

# srsal: double accumulators narrowed to float; CUDA's exp() and glibc's may differ in the last double bit,
# which moves a result across a float rounding boundary now and then: one float ulp
SRSAL_TOL = dict(rtol=3e-7, atol=1e-7)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("name", sorted(cases.ZOOMOUT))
def test_zoom_out_float_is_bit_identical_to_oracle_and_reference(ctx, oracle, name):
    field, factor = cases.zoomout_input(name)
    got = ctx.oct_zoom_out_float(field, factor)
    want = oracle.zoom_out_float(field, factor)
    assert got.shape == want.shape
    assert np.array_equal(got, want), np.abs(got - want).max()      # explicitly rounded double arithmetic: exact
    got_dev = ctx.oct_zoom_out_float(dev(field), factor)        # stream-ordered by the wrapper, no synchronize
    assert np.array_equal(got_dev.cpu().numpy(), got)
    assert np.array_equal(got, cases.zoomout_reference(oracle, name, field, factor))


@pytest.mark.parametrize("factor", [0.5, 0.25, 0.125])
def test_zoom_out_equals_the_reference_cpu_pyramid_stage_on_config_1(ctx, oracle, factor):
    """BASELINE config 1: the 500 x 500 texture through the reference's CPU pyramid stage oct_zoom_out (double,
    src/oct_zoom.cc:17) -- the kernel's float output is that double result rounded once"""
    from octane_b200 import synthetic as S
    i1, _, _, _ = S.make_pair(500, 500, seed=1, kind="shift", drift=(2.0, -1.0))
    got = ctx.oct_zoom_out_float(i1, factor)
    assert np.array_equal(got, cases.zoomout_reference(oracle, f"config1_{factor}", i1, factor, pyramid=True))


def test_zoom_out_float_large_field_properties(ctx):
    """a 0.5 km mesoscale channel (2000 x 2000) down to the 2 km grid: constant in -> the same constant scale
    everywhere (dropped tap), and blur + decimation commutes with a shift by whole output pixels in the interior"""
    n = 2000
    rng = np.random.default_rng(3)
    f = (rng.standard_normal((n, n)) * 10 + 100).astype(np.float32)
    out = ctx.oct_zoom_out_float(f, 0.25)
    assert out.shape == (500, 500) and np.isfinite(out).all()
    shifted = ctx.oct_zoom_out_float(np.roll(f, (8, 12), axis=(0, 1)), 0.25)
    assert np.array_equal(shifted[10:-10, 10:-10], np.roll(out, (2, 3), axis=(0, 1))[10:-10, 10:-10])
    const = ctx.oct_zoom_out_float(np.full((n, n), 7.0, np.float32), 0.25)
    assert np.ptp(const) == 0


def test_zoom_out_float_rejects_bad_arguments(ctx):
    f = np.zeros((10, 10), np.float32)
    for factor in (0.0, -0.5, 1.5, float("nan")):
        with pytest.raises(ob.OctaneError):
            ctx.oct_zoom_out_float(f, factor)
    with pytest.raises(ob.OctaneError):
        ctx.oct_zoom_out_float(np.zeros((4000, 4000), np.float32), 0.01)     # blur radius beyond the supported 32


@pytest.mark.parametrize("name", sorted(cases.SRSAL))
def test_srsal_matches_oracle(ctx, oracle, name):
    u, v, cth = cases.srsal_inputs(cases.SRSAL[name])
    wu, wv = oracle.srsal(u, v, cth)
    gu, gv = ctx.oct_srsal_cu(u.copy(), v.copy(), cth)
    np.testing.assert_allclose(gu, wu, **SRSAL_TOL)
    np.testing.assert_allclose(gv, wv, **SRSAL_TOL)
    du, dv = dev(u), dev(v)
    ctx.oct_srsal_cu(du, dv, dev(cth))                          # stream-ordered by the wrapper, no synchronize
    assert np.array_equal(du.cpu().numpy(), gu) and np.array_equal(dv.cpu().numpy(), gv)


@pytest.mark.parametrize("name", sorted(cases.SRSAL))
def test_srsal_matches_reference_fixture(ctx, name):
    g = load_golden(name)
    u, v, cth = cases.srsal_inputs(cases.SRSAL[name])
    gu, gv = ctx.oct_srsal_cu(u.copy(), v.copy(), cth)
    np.testing.assert_allclose(gu, g["u"], **SRSAL_TOL)
    np.testing.assert_allclose(gv, g["v"], **SRSAL_TOL)


def test_srsal_partial_tiles_and_rejects_small_scenes(ctx, oracle):
    """scene sizes that are not multiples of the 32 x 8 tile; nx or ny <= 18 is refused (the reference's reflected
    index leaves the array there)"""
    rng = np.random.default_rng(9)
    for ny, nx in ((19, 19), (33, 45), (41, 130)):
        u = rng.standard_normal((ny, nx)).astype(np.float32)
        v = rng.standard_normal((ny, nx)).astype(np.float32)
        cth = (5000 + 25 * rng.standard_normal((ny, nx))).astype(np.float32)
        wu, wv = oracle.srsal(u, v, cth)
        gu, gv = ctx.oct_srsal_cu(u.copy(), v.copy(), cth)
        np.testing.assert_allclose(gu, wu, **SRSAL_TOL)
        np.testing.assert_allclose(gv, wv, **SRSAL_TOL)
    z = np.zeros((18, 64), np.float32)
    with pytest.raises(ob.OctaneError):
        ctx.oct_srsal_cu(z.copy(), z.copy(), z)


def test_dispatcher_with_srsal_smooths_only_the_pixel_displacements(ctx, oracle):
    """oct_optical_flow.cc:91-105: the navigation runs on the raw flow, then -srsal replaces uPix / vPix"""
    g = load_golden("dispatch_cth_ir0")
    kw, extra, t1, t2, flags = cases.nav_constants(cases.NAVIGATION["nav_goes_meso"])
    nav = ob.goes_nav(**kw)
    plain = ctx.oct_optical_flow(g["img1"], g["img2"], nav, t1, t2, ob.default_params(doCTH=1), cth=g["cth"])
    smooth = ctx.oct_optical_flow(g["img1"], g["img2"], nav, t1, t2, ob.default_params(doCTH=1, dosrsal=1), cth=g["cth"])
    for k in ("uVal", "vVal", "uVal2", "vVal2", "CTP"):
        assert np.array_equal(plain[k], smooth[k])
    wu, wv = oracle.srsal(plain["uPix"], plain["vPix"], g["cth"])
    np.testing.assert_allclose(smooth["uPix"], wu, **SRSAL_TOL)
    np.testing.assert_allclose(smooth["vPix"], wv, **SRSAL_TOL)
    # device-buffer dispatcher
    import torch
    ny, nx = g["img1"].shape
    mk = lambda dt: torch.zeros((ny, nx), dtype=dt, device="cuda")      # noqa: E731
    up, vp = mk(torch.float32), mk(torch.float32)
    sh = [mk(torch.int16) for _ in range(5)]
    ctx.oct_optical_flow_dev(dev(g["img1"]), dev(g["img2"]), nav, t1, t2, ob.default_params(doCTH=1, dosrsal=1), up, vp,
                             sh[0], sh[1], sh[2], sh[3], cth=dev(g["cth"]), ctp=sh[4])
    ctx.synchronize()
    assert np.array_equal(up.cpu().numpy(), smooth["uPix"]) and np.array_equal(vp.cpu().numpy(), smooth["vPix"])
    assert np.array_equal(sh[0].cpu().numpy(), plain["uVal"])
    with pytest.raises(ob.OctaneError):
        ctx.oct_optical_flow(g["img1"], g["img2"], nav, t1, t2, ob.default_params(dosrsal=1))      # no heights


def test_reference_signatures_of_regridding_and_srsal_drop_in(oracle):
    """oct_zoom_in_float / oct_zoom_out_float / oct_srsal_cu with the reference's own C++ signatures, provided by the
    shim on top of liboctane_b200.so (oracle/_ref/libref_shim.so: the reference's two regridders are weakened in its
    copy of oct_zoom.o and its oct_srsal_cuda.o is not linked), against the reference's CPU object and the oracle."""
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.exists(os.path.join(root, "oracle", "_ref", "libref_shim.so")):
        pytest.skip("oracle/_ref/libref_shim.so not built (reference tree absent at build time)")
    S = oracle.ref_shim()
    field, factor = cases.zoomout_input("third")
    assert np.array_equal(oracle.ref_zoom_out_float(field, factor, L=S), oracle.ref_zoom_out_float(field, factor))
    raw = oracle.ref_zoom_out_float(field, 0.5, cnum=1, L=S)                 # the element offset of :84 is kept
    assert raw[0] == 0 and np.array_equal(raw[1:], oracle.zoom_out_float(field, 0.5).ravel())
    coarse = field[:30, :40]
    up = oracle.ref_zoom_in_float(coarse, 120, 90, 1, L=S)
    assert np.abs(up - oracle.ref_zoom_in_float(coarse, 120, 90, 1)).max() <= 1e-3
    u, v, cth = cases.srsal_inputs(cases.SRSAL["srsal_96x80_deck"])
    su, sv = oracle.ref_srsal(u, v, cth, L=S)
    wu, wv = oracle.srsal(u, v, cth)
    np.testing.assert_allclose(su, wu, **SRSAL_TOL)
    np.testing.assert_allclose(sv, wv, **SRSAL_TOL)


def test_band_first_guess_entry_point_on_one_gpu(ctx):
    """octane_variational_flow_band_fg_dev at world size 1 (band == scene): separate first-guess input and flow output
    buffers give the bits of the in/out entry point (the multi-GPU case is tests/test_gpu_band.py)"""
    import torch
    c = cases.VARIATIONAL["var_160x120_fg"]
    img1, img2, u0, v0 = cases.variational_inputs(c)
    ny, nx = img1.shape
    p = ob.default_params(first_guess=1, **c["params"])
    u, v = u0.copy(), v0.copy()
    ctx.oct_variational_optical_flow(img1, img2, u, v, p)
    ub = torch.zeros((ny, nx), device="cuda"); vb = torch.zeros_like(ub)
    fgu, fgv = dev(u0), dev(v0)
    ctx.oct_variational_optical_flow_band(dev(img1), dev(img2), ub, vb, nx, ny, p, fg_u_band=fgu, fg_v_band=fgv)
    ctx.synchronize()
    assert np.array_equal(ub.cpu().numpy(), u) and np.array_equal(vb.cpu().numpy(), v)
    assert np.array_equal(fgu.cpu().numpy(), u0)            # the first guess is an input only
    g = load_golden("var_160x120_fg")
    assert np.abs(u - g["u"]).max() < 1e-2
