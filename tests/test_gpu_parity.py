"""GPU parity tests: the CUDA path, called through the C ABI, against
(1) fixtures produced by the reference itself (tests/golden), (2) the CPU
oracle on the same seeded inputs, (3) size-independent properties at the
BASELINE.json sizes.

Tolerances (BASELINE.json north_star): pyramid dimensions and indexing
bit-exact; fp32 flow mean |du,dv| <= 1e-3 px, max <= 1e-2 px; navigated speed
within 0.01 m/s (= 1 count of the short outputs)."""
import ctypes as C
import os

import numpy as np
import pytest

import cases
import octane_b200 as ob
from conftest import load_golden
from octane_b200 import synthetic as S

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEAN_TOL, MAX_TOL = 1e-3, 1e-2


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def solve(ctx, c, img1, img2, u0, v0):
    ny, nx = img1.shape[-2:]
    p = ob.default_params(first_guess=int(u0 is not None), **c.get("params", {}))
    u = np.zeros((ny, nx), np.float32) if u0 is None else u0.copy()
    v = np.zeros((ny, nx), np.float32) if v0 is None else v0.copy()
    ctx.oct_variational_optical_flow(img1, img2, u, v, p, nc=c.get("nc", 1))
    return u, v, p


@pytest.mark.parametrize("name", sorted(cases.VARIATIONAL))
def test_flow_matches_reference_fixture(ctx, name):
    c = cases.VARIATIONAL[name]
    g = load_golden(name)
    img1, img2, u0, v0 = cases.variational_inputs(c)
    u, v, _ = solve(ctx, c, img1, img2, u0, v0)
    du, dv = np.abs(u - g["u"]), np.abs(v - g["v"])
    assert du.mean() < MEAN_TOL and dv.mean() < MEAN_TOL
    assert du.max() < MAX_TOL and dv.max() < MAX_TOL
    assert max(du.max(), dv.max()) < max(20 * float(g["spread"].max()), 2e-4)


@pytest.mark.parametrize("name", sorted(cases.VARIATIONAL))
def test_flow_matches_oracle(ctx, oracle, name):
    c = cases.VARIATIONAL[name]
    img1, img2, u0, v0 = cases.variational_inputs(c)
    u, v, p = solve(ctx, c, img1, img2, u0, v0)
    st = ctx.stats()
    uo, vo, its = oracle.variational_flow(img1, img2, oracle.params(**c.get("params", {})), u0, v0, nc=c.get("nc", 1))
    assert np.abs(u - uo).mean() < 1e-4 and np.abs(v - vo).mean() < 1e-4
    assert np.abs(u - uo).max() < 2e-3 and np.abs(v - vo).max() < 2e-3
    assert list(st.cg_iterations[:st.n_solves]) == list(its)
    assert st.kernel_launches > 0
    dims = [(st.level_nx[k], st.level_ny[k]) for k in range(st.n_levels)]
    assert dims == oracle.level_dims(c["nx"], c["ny"], kiters=p.kiters)       # bit-exact pyramid geometry


@pytest.mark.parametrize("name", sorted(cases.NAVIGATION))
def test_navigation_matches_reference_fixture(ctx, name):
    c = cases.NAVIGATION[name]
    g = load_golden(name)
    kw, extra, t1, t2, flags = cases.nav_constants(c)
    nav = ob.goes_nav(**kw)
    for k, val in extra.items():
        setattr(nav, k, val)
    p = ob.default_params(**flags)
    ny, nx = g["u"].shape
    outs = [np.full((ny, nx), 7, np.int16) for _ in range(4)]
    dT, moved = ctx.oct_pix2uv_cuda(nav, t1, t2, g["u"], g["v"], *outs, p)
    assert moved == bool(c.get("moved")) and abs(dT - float(g["dT"])) < 1e-6
    U, V, U2, V2 = outs
    # same CUDA libm, same expression order: identical shorts
    assert np.array_equal(U, g["U"]) and np.array_equal(V, g["V"])
    if not flags["pixuv"]:
        assert np.array_equal(U2, g["U_raw"]) and np.array_equal(V2, g["V_raw"])
    else:   # documented deviation: the reference leaves U_raw/V_raw unwritten with -pd; we write 100*u
        assert np.array_equal(U2, U) and np.array_equal(V2, V)


@pytest.mark.parametrize("ir", [0, 1])
def test_dispatcher_with_cloud_top_heights(ctx, ir):
    g = load_golden(f"dispatch_cth_ir{ir}")
    kw, extra, t1, t2, flags = cases.nav_constants(cases.NAVIGATION["nav_goes_meso"])
    p = ob.default_params(doCTH=1, ir=ir)
    out = ctx.oct_optical_flow(g["img1"], g["img2"], ob.goes_nav(**kw), t1, t2, p, cth=g["cth"])
    assert np.abs(out["uPix"] - g["uPix"]).max() < 2e-4 and np.abs(out["vPix"] - g["vPix"]).max() < 2e-4
    assert np.array_equal(out["CTP"], g["CTP"])
    # The flow differs from the fixture by the reference's own run-to-run noise (~1e-5 px), and
    # the reference quantises its speeds through a float-narrowed lat/lon (steps of ~1.4 counts
    # at dt = 60 s, SURVEY.md P13), so a few pixels land on the neighbouring quantum.
    for a, b in (("uVal", "U"), ("vVal", "V")):
        d = np.abs(out[a].astype(int) - g[b])
        assert d.max() <= 2 and (d > 0).mean() < 0.02
    for a, b in (("uVal2", "U_raw"), ("vVal2", "V_raw")):
        assert np.abs(out[a].astype(int) - g[b]).max() <= 1
    assert abs(out["dT"] - float(g["dT"])) < 1e-6


@pytest.mark.parametrize("ir", [0, 1])
def test_reference_dispatcher_drops_in_on_our_kernels(oracle, ir):
    """The reference's unmodified oct_optical_flow() object, linked against the shim
    (octane_b200/shim/oct_b200_shim.cc) + liboctane_b200.so instead of the reference's two .cu
    objects, must reproduce the fixture the reference's own CUDA build produced."""
    so = os.path.join(ROOT, "oracle", "_ref", "libref_shim.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref/libref_shim.so not built (reference tree absent at build time)")
    g = load_golden(f"dispatch_cth_ir{ir}")
    kw, extra, t1, t2, flags = cases.nav_constants(cases.NAVIGATION["nav_goes_meso"])
    nav = oracle.goes_nav(**kw)
    out = oracle.ref_dispatch(oracle.ref_shim(), g["img1"], g["img2"], nav, t1, t2,
                              oracle.ref_params(doCTH=1, ir=ir), cth=g["cth"])
    assert np.abs(out["uPix"] - g["uPix"]).max() < 2e-4 and np.abs(out["vPix"] - g["vPix"]).max() < 2e-4
    assert np.array_equal(out["CTP"], g["CTP"])
    for k in ("U", "V"):
        d = np.abs(out[k].astype(int) - g[k])
        assert d.max() <= 2 and (d > 0).mean() < 0.02
    for k in ("U_raw", "V_raw"):
        assert np.abs(out[k].astype(int) - g[k]).max() <= 1
    assert abs(out["dT"] - float(g["dT"])) < 1e-6


# ---- stage-level parity against the oracle --------------------------------------------
@pytest.mark.parametrize("shape", [(96, 80), (257, 131), (500, 500)])
@pytest.mark.parametrize("factor", [0.5, 0.25, 0.125])
def test_stage_blur_decimate(ctx, oracle, shape, factor):
    import torch
    nx, ny = shape
    img = S.texture(nx, ny, 21)
    nxx, nyy = int(nx * factor + 0.5), int(ny * factor + 0.5)
    want = np.zeros((nyy, nxx), np.float32)
    oracle.lib().oracle_blur_decimate(img, nx, ny, 1, factor, want)
    got = torch.zeros((nyy, nxx), device="cuda")
    ctx.stage_blur_decimate(dev(img), nx, ny, 1, factor, got)
    got = got.cpu().numpy()
    assert got.shape == want.shape                                # dims bit-exact
    # taps come from CUDA expf vs glibc expf (<= 1 ulp): values to 1e-6 relative
    assert np.abs(got - want).max() <= 1e-6 * 255 * 4


@pytest.mark.parametrize("shape", [(96, 80), (257, 131), (33, 17), (260, 70), (4, 5), (3, 9), (132, 64)])
def test_stage_gradient_bit_exact(ctx, oracle, shape):
    import torch
    nx, ny = shape
    img = S.texture(nx, ny, 22)
    gx, gy = np.zeros_like(img), np.zeros_like(img)
    oracle.lib().oracle_gradient(img, gx, gy, nx, ny, 1)
    dgx, dgy = torch.zeros((ny, nx), device="cuda"), torch.zeros((ny, nx), device="cuda")
    ctx.stage_gradient(dev(img), nx, ny, 1, dgx, dgy)
    assert np.array_equal(dgx.cpu().numpy(), gx) and np.array_equal(dgy.cpu().numpy(), gy)


@pytest.mark.parametrize("dims", [((63, 63), (125, 125)), ((125, 125), (250, 250)), ((16, 18), (32, 35)), ((40, 30), (81, 59)),
                                  ((150, 20), (300, 41)), ((129, 9), (259, 17)), ((200, 12), (230, 13))])
def test_stage_zoom_in_bit_exact(ctx, oracle, dims):
    import torch
    (nx, ny), (nxx, nyy) = dims
    u, _ = S.flow_field(nx, ny)
    u = u.astype(np.float32)
    want = np.zeros((nyy, nxx), np.float32)
    oracle.lib().oracle_zoom_in(u, want, nx, ny, nxx, nyy, 0.5)
    got = torch.zeros((nyy, nxx), device="cuda")
    ctx.stage_zoom_in(dev(u), nx, ny, nxx, nyy, 0.5, got)
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("gnc", [0, 1, 2])
@pytest.mark.parametrize("nc", [1, 2, 3])
def test_stage_build_and_pcg(ctx, oracle, gnc, nc):
    import torch
    nx, ny = 150, 110
    chans1, chans2 = [], []
    for ch in range(nc):
        a, b, ut, vt = S.make_pair(nx, ny, 30 + ch)
        chans1.append(a); chans2.append(b)
    g1 = np.ascontiguousarray(np.stack(chans1)); g2 = np.ascontiguousarray(np.stack(chans2))
    u = (0.7 * ut).astype(np.float32); v = (0.7 * vt).astype(np.float32)
    uh = (0.5 * ut).astype(np.float32); vh = (0.5 * vt).astype(np.float32)
    p = ob.default_params()
    lambdac = 0.25
    # oracle: gradients then build
    L = oracle.lib()
    n = nx * ny
    f = {k: np.zeros((nc, ny, nx), np.float32) for k in ("g1x", "g1y", "g2x", "g2y", "g2xx", "g2xy", "g2yy")}
    L.oracle_gradient(g1, f["g1x"], f["g1y"], nx, ny, nc)
    L.oracle_gradient(g2, f["g2x"], f["g2y"], nx, ny, nc)
    L.oracle_gradient(f["g2x"], f["g2xx"], f["g2xy"], nx, ny, nc)
    L.oracle_gradient(f["g2y"], f["g2xy"], f["g2yy"], nx, ny, nc)
    coef = np.zeros((7, ny, nx), np.float32); bu = np.zeros((ny, nx), np.float32); bv = np.zeros((ny, nx), np.float32)
    L.oracle_build(u, v, uh.ctypes.data, vh.ctypes.data, g1, f["g1x"], f["g1y"], g2, f["g2x"], f["g2y"], f["g2xx"],
                   f["g2xy"], f["g2yy"], nx, ny, nc, p.alpha, p.lambda_ / p.alpha, lambdac, gnc, 1, coef, bu, bv)
    dcoef = torch.zeros((7, ny, nx), device="cuda"); dbu = torch.zeros((ny, nx), device="cuda"); dbv = torch.zeros((ny, nx), device="cuda")
    ctx.stage_build(dev(u), dev(v), dev(uh), dev(vh), dev(g1), dev(g2), nx, ny, nc, p, lambdac, gnc, dcoef, dbu, dbv)
    gc, gbu, gbv = dcoef.cpu().numpy(), dbu.cpu().numpy(), dbv.cpu().numpy()
    scale = np.abs(coef).max(axis=(1, 2), keepdims=True)
    # FMA contraction differences only -- except where a robust weight 1/sqrt(x + 1e-6) sits on
    # x ~ 0 (psi up to 1000): there a 1-ulp change of x moves the coefficient by up to ~0.2 %
    err = np.abs(gc - coef) / scale
    assert np.quantile(err, 0.999) < 2e-5 and err.max() < 5e-3
    # the rhs holds sum_k psi_k u_k - (sum_k psi_k) u with psi up to 1000: its absolute rounding noise
    # scales with the diagonal, not with |b|
    for got, want in ((gbu, bu), (gbv, bv)):
        e = np.abs(got - want)
        assert np.quantile(e, 0.999) < 1e-4 * max(1.0, np.abs(want).max()) and e.max() < 2e-6 * scale[0].max()
    # boundary-merged entries: absent neighbours are exactly zero
    assert np.all(gc[3][:, 0] == 0) and np.all(gc[5][:, -1] == 0) and np.all(gc[4][0, :] == 0) and np.all(gc[6][-1, :] == 0)
    # PCG on the oracle's system: same iterate after the same number of iterations
    for iters in (1, 7, 30):
        b1, b2 = bu.copy(), bv.copy()
        xu, xv = np.zeros((ny, nx), np.float32), np.zeros((ny, nx), np.float32)
        work = np.zeros(8 * n, np.float32)
        its = L.oracle_pcg(coef, b1, b2, xu, xv, nx, ny, iters, 1e-8, work)
        dxu, dxv = torch.zeros((ny, nx), device="cuda"), torch.zeros((ny, nx), device="cuda")
        got_its = ctx.stage_pcg(dev(coef), dev(bu), dev(bv), nx, ny, iters, 1e-8, dxu, dxv)
        assert got_its == its
        tol = 5e-5 * max(1.0, np.abs(xu).max())
        assert np.abs(dxu.cpu().numpy() - xu).max() < tol and np.abs(dxv.cpu().numpy() - xv).max() < tol


def test_pcg_stop_rule_and_zero_rhs(ctx):
    import torch
    nx, ny = 64, 48
    coef = np.zeros((7, ny, nx), np.float32)
    coef[0] = 9; coef[2] = 9
    for k in (3, 4, 5, 6):
        coef[k] = -1
    # mirror-merged edges as the build produces them (:929-1077): the absent neighbour's entry is
    # zero and its weight is added to the opposite one
    coef[3][:, 0] = 0; coef[5][:, -1] = 0; coef[4][0, :] = 0; coef[6][-1, :] = 0
    coef[3][:, -1] = -2; coef[5][:, 0] = -2; coef[4][-1, :] = -2; coef[6][0, :] = -2
    z = np.zeros((ny, nx), np.float32)
    dxu, dxv = torch.ones((ny, nx), device="cuda"), torch.ones((ny, nx), device="cuda")
    assert ctx.stage_pcg(dev(coef), dev(z), dev(z), nx, ny, 30, 1e-8, dxu, dxv) == 0     # ||b||^2 <= tol: no iteration
    assert float(dxu.abs().max()) == 0 and float(dxv.abs().max()) == 0
    b = np.random.default_rng(1).standard_normal((ny, nx)).astype(np.float32)
    its = ctx.stage_pcg(dev(coef), dev(b), dev(b), nx, ny, 200, 1e-8, dxu, dxv)
    assert 0 < its < 200                                                               # converges before the cap


# ---- size-independent properties at the BASELINE sizes ----------------------------------
def test_meso_2000_matches_oracle(ctx, oracle):
    nx = ny = 2000
    import torch
    a, b = S.make_pair_torch(nx, ny, 2, "cuda")
    i1, i2 = a.cpu().numpy(), b.cpu().numpy()
    u, v = np.zeros((ny, nx), np.float32), np.zeros((ny, nx), np.float32)
    ctx.oct_variational_optical_flow(i1, i2, u, v, ob.default_params())
    uo, vo, its = oracle.variational_flow(i1, i2)
    assert np.abs(u - uo).mean() < MEAN_TOL and np.abs(v - vo).mean() < MEAN_TOL
    assert np.abs(u - uo).max() < MAX_TOL and np.abs(v - vo).max() < MAX_TOL
    st = ctx.stats()
    assert list(st.cg_iterations[:st.n_solves]) == list(its)


@pytest.mark.parametrize("workload", ["conus", "fulldisk"])
def test_large_scene_properties(ctx, workload):
    """CONUS 10000x6000 and full disk 21696x21696 (beyond the reference's int CSR limit):
    bit-exact pyramid dims, run-to-run bit-reproducibility, recovery of the known
    displacement, navigation round trip of the recovered flow."""
    import torch
    nx, ny, sector, taper = {"conus": (10000, 6000, "conus_0.5km", False),
                             "fulldisk": (21696, 21696, "fulldisk_0.5km", True)}[workload]
    a, b = S.make_pair_torch(nx, ny, 4, "cuda", limb_taper=taper)
    u = torch.zeros((ny, nx), device="cuda"); v = torch.zeros_like(u)
    p = ob.default_params()
    ctx.oct_variational_optical_flow(a, b, u, v, p)
    ctx.synchronize()
    st = ctx.stats()
    dims = [(st.level_nx[k], st.level_ny[k]) for k in range(st.n_levels)]
    assert dims == [(int(nx * f + 0.5), int(ny * f + 0.5)) for f in (0.125, 0.25, 0.5, 1.0)]
    assert all(0 < i <= 30 for i in st.cg_iterations[:st.n_solves])
    assert bool(torch.isfinite(u).all()) and bool(torch.isfinite(v).all())
    # known flow: drift (0.8,-0.4) + vortex of peak 2 px; compare on a central window away from the limb
    ys, xs = slice(ny // 2 - 1500, ny // 2 + 1500), slice(nx // 2 - 1500, nx // 2 + 1500)
    ut, vt = S.flow_field(nx, ny)
    eu = (u[ys, xs].cpu().numpy() - ut[ys, xs]); ev = (v[ys, xs].cpu().numpy() - vt[ys, xs])
    assert np.abs(eu).mean() < 0.05 and np.abs(ev).mean() < 0.05
    # determinism: fixed-order reductions make a second run bit-identical
    u2 = torch.zeros_like(u); v2 = torch.zeros_like(v)
    ctx.oct_variational_optical_flow(a, b, u2, v2, p)
    ctx.synchronize()
    assert torch.equal(u, u2) and torch.equal(v, v2)
    # navigation of the whole scene: U_raw is exactly (short)(100*u), fill/limb pixels are 0
    xsc, ysc, xo, yo, dt = S.SECTORS[sector]
    outs = [torch.zeros((ny, nx), dtype=torch.int16, device="cuda") for _ in range(4)]
    ctx.oct_pix2uv_cuda(ob.goes_nav(xsc, ysc, xo, yo), 0.0, dt, u, v, *outs, p)
    ctx.synchronize()
    assert torch.equal(outs[2], (100 * u).to(torch.int32).to(torch.int16))
    if taper:
        assert int(outs[0][0, 0]) == 0 and int(outs[1][0, 0]) == 0          # off-earth corner
    # speed = displacement * ~500 m / dt: centre pixel within 5 %
    cy, cx = ny // 2, nx // 2
    ms = float(outs[0][cy, cx]) / 100.0
    px = float(u[cy, cx])
    gsd = 35786023.0 * 1.4e-5
    if abs(px) > 0.2:
        assert abs(ms - px * gsd / dt) < 0.08 * abs(px * gsd / dt) + 0.02


def test_errors_are_codes_not_exits(ctx):
    img = np.zeros((8, 8), np.float32)
    u = np.zeros((8, 8), np.float32)
    with pytest.raises(ob.OctaneError) as e:       # level smaller than 4 pixels
        ctx.oct_variational_optical_flow(img, img, u, u.copy(), ob.default_params())
    assert e.value.code == -2
    with pytest.raises(ob.OctaneError):
        ctx.oct_variational_optical_flow(img, img, u, u.copy(), ob.default_params(kiters=1, alpha=0.0))
    c2 = ob.Context(99)          # out-of-range device -> device 0, as the reference (:1260-1264)
    c2.close()


def test_graph_and_plain_launch_paths_agree(ctx):
    i1, i2, _, _ = S.make_pair(300, 220, 40)
    p = ob.default_params()
    u1, v1 = np.zeros((220, 300), np.float32), np.zeros((220, 300), np.float32)
    ctx.oct_variational_optical_flow(i1, i2, u1, v1, p)
    ctx.set_graphs(False)
    u2, v2 = np.zeros_like(u1), np.zeros_like(v1)
    ctx.oct_variational_optical_flow(i1, i2, u2, v2, p)
    ctx.set_graphs(True)
    ctx.set_profile(True)
    u3, v3 = np.zeros_like(u1), np.zeros_like(v1)
    ctx.oct_variational_optical_flow(i1, i2, u3, v3, p)
    st = ctx.stats()
    ctx.set_profile(False)
    assert np.array_equal(u1, u2) and np.array_equal(v1, v2) and np.array_equal(u1, u3)
    # a scene this small runs every solve as ONE cooperative launch (k_pcg_coop): timed as a whole, no per-iteration figures
    assert st.ms_pcg_pass1 > 0 and st.kernel_launches < 400 and st.finest_pass2_ms == 0


# ---- ingest (oct_navcal_cuda) and first-guess conversion (oct_uv2pix) --------------------------
def _ingest(oracle, name):
    c = cases.INGEST[name]
    rad, xc, yc, kw, dt = cases.ingest_inputs(c)
    onav = oracle.goes_nav(**kw)
    ocal = oracle.goes_cal(onav, c["radScale"], c["radOffset"], c["maxin"], c["minin"], donav=c.get("donav", 1))
    nav = ob.goes_nav(**kw)
    cal = ob.goes_cal(c["radScale"], c["radOffset"], band=c["band"], donav=c.get("donav", 1))
    return rad, xc, yc, onav, ocal, nav, cal, dt


def _check_ingest(got, want, r2, tol_data=5e-5):
    data, lat, lon = got
    wd, wlat, wlon = want
    assert np.abs(data - wd).max() <= tol_data
    assert np.array_equal(data == 0, wd == 0)
    cases.check_latlon(lat, lon, wlat, wlon, r2)


@pytest.mark.parametrize("name", sorted(cases.INGEST))
def test_navcal_matches_oracle_and_reference(ctx, oracle, name):
    rad, xc, yc, onav, ocal, nav, cal, dt = _ingest(oracle, name)
    r2 = cases.ingest_r2(cases.INGEST[name])
    got = ctx.oct_navcal_cuda(rad, xc, yc, nav, cal)                    # host entry point
    _check_ingest(got, oracle.navcal(rad, xc, yc, ocal), r2)
    got_dev = ctx.oct_navcal_cuda(dev(rad), dev(xc), dev(yc), nav, cal)  # device entry point; no explicit
    # synchronisation: the wrapper orders torch's stream after the context's, which the .cpu() below relies on
    for a, b in zip(got, got_dev):
        assert np.array_equal(a, b.cpu().numpy(), equal_nan=True)
    g = load_golden(name)
    _check_ingest(got, (g["data"], g["lat"], g["lon"]), r2)


@pytest.mark.parametrize("name", sorted(cases.UV2PIX))
def test_uv2pix_matches_oracle_and_reference(ctx, oracle, name):
    c = cases.UV2PIX[name]
    rad, xc, yc, onav, ocal, nav, cal, dt = _ingest(oracle, c["ingest"])
    _, lat, lon = oracle.navcal(rad, xc, yc, ocal)
    if c.get("moved"):
        onav.g2xOffset = onav.xOffset + np.float32(0.001)
        nav.g2xOffset = nav.xOffset + np.float32(0.001)
    u0, v0 = cases.uv2pix_winds(len(xc), len(yc))
    wu, wv, wrc = oracle.uv2pix(onav, 1000.0, 1000.0 + dt, lat, lon, xc, yc, u0, v0)
    u, v = u0.copy(), v0.copy()
    rc = ctx.oct_uv2pix(nav, 1000.0, 1000.0 + dt, lat, lon, xc, yc, u, v)
    assert rc == wrc == int(bool(c.get("moved")))
    assert np.array_equal(np.isnan(u), np.isnan(wu))
    ok = ~np.isnan(u)
    assert np.abs(u - wu)[ok].max(initial=0) <= 1e-4 and np.abs(v - wv)[ok].max(initial=0) <= 1e-4
    g = load_golden(name)
    gi = load_golden(c["ingest"])
    u, v = g["u"].copy(), g["v"].copy()
    ctx.oct_uv2pix(nav, 1000.0, 1000.0 + dt, gi["lat"], gi["lon"], xc, yc, u, v)
    ok = ~np.isnan(g["upix"])
    assert np.array_equal(np.isnan(u), ~ok)
    assert np.abs(u - g["upix"])[ok].max(initial=0) <= 1e-4 and np.abs(v - g["vpix"])[ok].max(initial=0) <= 1e-4


def test_reference_signatures_of_ingest_drop_in(oracle):
    """oct_navcal_cuda / oct_uv2pix with the reference's own C++ signatures, provided by the shim on
    top of liboctane_b200.so (oracle/_ref/libref_shim.so links no reference .cu object for them)."""
    so = os.path.join(ROOT, "oracle", "_ref", "libref_shim.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref/libref_shim.so not built (reference tree absent at build time)")
    name = "ingest_limb_b13"
    rad, xc, yc, onav, ocal, nav, cal, dt = _ingest(oracle, name)
    r2 = cases.ingest_r2(cases.INGEST[name])
    got = oracle.ref_navcal(rad, xc, yc, ocal, L=oracle.ref_shim())
    _check_ingest(got, oracle.navcal(rad, xc, yc, ocal), r2)
    g = load_golden(name)
    _check_ingest(got, (g["data"], g["lat"], g["lon"]), r2)
    u0, v0 = cases.uv2pix_winds(len(xc), len(yc))
    u, v = oracle.ref_uv2pix(onav, 1000.0, 1000.0 + dt, g["lat"], g["lon"], xc, yc, u0, v0, L=oracle.ref_shim())
    gu = load_golden("uv2pix_limb")
    ok = ~np.isnan(gu["upix"])
    assert np.abs(u - gu["upix"])[ok].max(initial=0) <= 1e-4 and np.abs(v - gu["vpix"])[ok].max(initial=0) <= 1e-4


@pytest.mark.parametrize("dims", [((50, 60), (200, 240)), ((37, 41), (111, 123)), ((64, 64), (64, 64)), ((30, 45), (75, 113))])
@pytest.mark.parametrize("interp", [1, 0])
def test_zoom_in_float_matches_oracle_and_reference(ctx, oracle, dims, interp):
    """oct_zoom_in_float (reference src/oct_zoom.cc:180): the regridding of cloud-top heights / extra
    channels.  Checked against the CPU restatement and against the reference's own CPU object."""
    (ny, nx), (nyy, nxx) = dims
    f = (np.random.default_rng(nx * 7 + ny).standard_normal((ny, nx)) * 1000 + 5000).astype(np.float32)
    got = ctx.oct_zoom_in_float(f, nxx, nyy, interp)
    want = oracle.zoom_in_float(f, nxx, nyy, interp)
    if interp == 0:
        assert np.array_equal(got, want)                       # nearest neighbour: index arithmetic only
    else:
        assert np.abs(got - want).max() <= 1e-3                # values ~5000: one float ulp (FMA contraction in double)
    got_dev = ctx.oct_zoom_in_float(dev(f), nxx, nyy, interp)       # stream-ordered by the wrapper, no synchronize
    assert np.array_equal(got_dev.cpu().numpy(), got)
    try:
        ref = oracle.ref_zoom_in_float(f, nxx, nyy, interp)
    except OSError:
        pytest.skip("oracle/_ref/libref_cpu.so not built")
    assert np.abs(got - ref).max() <= (0 if interp == 0 else 1e-3)


@pytest.mark.parametrize("name", sorted(cases.GRIDNAV))
def test_gridnav_matches_oracle_and_reference(ctx, oracle, name):
    c = cases.GRIDNAV[name]
    data, xc, yc = cases.gridnav_inputs(c)
    nav = ob.goes_nav(c["xScale"], c["yScale"], c["xOffset"], c["yOffset"])
    nav.R = c["R"]; nav.lon0 = c["lon0"]; nav.lon1 = c["lon0"]; nav.lat1 = c["lat1"]
    got = ctx.oct_navcal_grid(c["grid"], data, xc, yc, nav, c.get("donav", 1))
    want = oracle.navcal_grid(c["grid"], data, xc, yc, c["xScale"], c["xOffset"], c["yScale"], c["yOffset"], c["R"], c["lon0"],
                              c["lat1"], c.get("donav", 1))
    refs = [want]
    g = load_golden(name)
    refs.append((g["data"], g["lat"], g["lon"]))
    so = os.path.join(ROOT, "oracle", "_ref", "libref_shim.so")
    if os.path.exists(so):     # the reference's own C++ signatures, provided by the shim on top of the library
        shim = oracle.ref_navcal_grid(c["grid"], data, xc, yc, c["xScale"], c["xOffset"], c["yScale"], c["yOffset"], c["R"],
                                      c["lon0"], c["lat1"], c.get("donav", 1), L=oracle.ref_shim())
        for a, b in zip(shim, got):
            assert np.array_equal(a, b, equal_nan=True)
    for wd, wlat, wlon in refs:
        assert np.array_equal(got[0], wd)
        assert np.array_equal(np.isnan(got[1]), np.isnan(wlat))
        ok = ~np.isnan(wlat)
        assert np.abs(got[1] - wlat)[ok].max(initial=0) <= 3.1e-5 and np.abs(got[2] - wlon)[ok].max(initial=0) <= 3.1e-5


def test_pairs_in_flight_on_several_contexts_match_sequential(ctx):
    """BASELINE config 5 (independent pairs): the device-buffer dispatcher on three contexts with pairs in flight
    concurrently gives, bit for bit, what one context gives pair after pair -- and the CTP pack rides along."""
    import torch
    nx, ny, npairs = 200, 160, 6
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(doCTH=1)
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = (7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)
    pairs = [S.make_pair(nx, ny, 200 + k)[:2] for k in range(npairs)]
    seq = [ctx.oct_optical_flow(a, b, nav, 0.0, dt, p, cth=cth) for a, b in pairs]
    ctxs = [ob.Context(0) for _ in range(3)]
    d_cth = dev(cth)
    d_pairs = [(dev(a), dev(b)) for a, b in pairs]
    outs = [dict(u=torch.zeros((ny, nx), device="cuda"), v=torch.zeros((ny, nx), device="cuda"),
                 s=[torch.zeros((ny, nx), dtype=torch.int16, device="cuda") for _ in range(5)]) for _ in pairs]
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(d_pairs):
        o = outs[i]
        ctxs[i % 3].oct_optical_flow_dev(a, b, nav, 0.0, dt, p, o["u"], o["v"], *o["s"][:4], cth=d_cth, ctp=o["s"][4],
                                         sync_torch=False)
    for c in ctxs:
        c.synchronize()
    for i, want in enumerate(seq):
        o = outs[i]
        assert np.array_equal(o["u"].cpu().numpy(), want["uPix"]) and np.array_equal(o["v"].cpu().numpy(), want["vPix"])
        for k, key in enumerate(("uVal", "vVal", "uVal2", "vVal2", "CTP")):
            assert np.array_equal(o["s"][k].cpu().numpy(), want[key]), key
    for c in ctxs:
        c.close()


def test_pipelined_dispatcher_matches_blocking_calls(ctx):
    """octane_stream_submit / octane_stream_wait over a sequence of pairs, two in flight: every pair's outputs are,
    bit for bit, what the blocking dispatcher returns for it (same kernels, only the copies overlap)."""
    import torch
    nx, ny, npairs = 640, 200, 5
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(doCTH=1, kiters=3)
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = (7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)
    pairs = [S.make_pair(nx, ny, 300 + k)[:2] for k in range(npairs)]
    want = [ctx.oct_optical_flow(a, b, nav, 0.0, dt, p, cth=cth) for a, b in pairs]

    def pinned(dtype):
        return torch.zeros((ny, nx), dtype=dtype, pin_memory=True).numpy()

    outs = [dict(uPix=pinned(torch.float32), vPix=pinned(torch.float32), uVal=pinned(torch.int16), vVal=pinned(torch.int16),
                 uVal2=pinned(torch.int16), vVal2=pinned(torch.int16), CTP=pinned(torch.int16)) for _ in range(2)]
    hin = [(torch.from_numpy(a).pin_memory().numpy(), torch.from_numpy(b).pin_memory().numpy()) for a, b in pairs]
    hcth = torch.from_numpy(cth).pin_memory().numpy()
    got = []
    for k in range(npairs):
        ctx.stream_submit(k % 2, hin[k][0], hin[k][1], nav, 0.0, dt, p, outs[k % 2], nx, ny, cth=hcth)
        if k > 0:
            ctx.stream_wait((k - 1) % 2)
            got.append({key: val.copy() for key, val in outs[(k - 1) % 2].items()})
    ctx.stream_wait((npairs - 1) % 2)
    got.append({key: val.copy() for key, val in outs[(npairs - 1) % 2].items()})
    for k in range(npairs):
        for key in ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2", "CTP"):
            assert np.array_equal(got[k][key], want[k][key]), (k, key)
    # without the pixel displacements (the reference writes them only with -pd)
    o = {key: outs[0][key] for key in ("uVal", "vVal", "uVal2", "vVal2")}
    ctx.stream_submit(0, hin[0][0], hin[0][1], nav, 0.0, dt, ob.default_params(kiters=3), o, nx, ny)
    ctx.stream_wait(0)
    assert np.array_equal(o["uVal"], want[0]["uVal"]) and np.array_equal(o["vVal2"], want[0]["vVal2"])
    with pytest.raises(ob.OctaneError):
        ctx.stream_submit(0, hin[0][0], hin[0][1], nav, 0.0, dt, ob.default_params(dosrsal=1), o, nx, ny, cth=hcth)


def test_fresh_context_first_call_is_the_pipelined_dispatcher():
    """A context whose very first call is octane_stream_submit (navigation tables, staging slots and the copy-in stream are
    all created inside it), then a larger scene through the same context while the other slot is still in flight:
    nothing a live slot uses may be released by that growth."""
    import torch
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(kiters=3)
    sizes = [(640, 200), (704, 320)]
    pairs = [S.make_pair(nx, ny, 410 + i)[:2] for i, (nx, ny) in enumerate(sizes)]
    ref = ob.Context(0)
    try:
        want = [ref.oct_optical_flow(a, b, nav, 0.0, dt, p) for a, b in pairs]
    finally:
        ref.close()
    c = ob.Context(0)
    try:
        outs, keep = [], []
        for i, (nx, ny) in enumerate(sizes):
            o = {k: torch.zeros((ny, nx), dtype=(torch.float32 if k.endswith("Pix") else torch.int16), pin_memory=True).numpy()
                 for k in ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")}
            a, b = (torch.from_numpy(x).pin_memory().numpy() for x in pairs[i])
            keep.append((a, b))
            c.stream_submit(i, a, b, nav, 0.0, dt, p, o, nx, ny)      # slot 1 is submitted while slot 0 is in flight
            outs.append(o)
        for i in range(2):
            c.stream_wait(i)
            for k in outs[i]:
                assert np.array_equal(outs[i][k], want[i][k]), (i, k)
    finally:
        c.close()


def test_pipelined_dispatcher_with_deferred_copy_out():
    """Banded contexts hold a pair's copy-out back until the next pair's solve reaches its finest level (DESIGN.md section 5).
    OCTANE_STREAM_DEFER=1 switches that schedule on for a single-GPU context: the two dispatcher tests above must pass
    unchanged under it (the switch is read once per process, hence the child process)."""
    import subprocess
    import sys
    if os.environ.get("OCTANE_STREAM_DEFER"):
        pytest.skip("already inside the child run")
    env = dict(os.environ, OCTANE_STREAM_DEFER="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
                        "-k", "test_pipelined_dispatcher_matches_blocking_calls or test_fresh_context_first_call"],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "2 passed" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
