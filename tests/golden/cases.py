"""Seeded golden cases shared by make_golden.py (which runs the REFERENCE on a
B200 to produce the fixtures) and by the parity tests (which replay the same
inputs through the oracle and through the CUDA path)."""
from __future__ import annotations

import numpy as np

from octane_b200 import synthetic as S

# name: dict(nx, ny, seed, kind, drift, nc, params overrides, first guess)
VARIATIONAL = {
    "var_96x80_shift": dict(nx=96, ny=80, seed=11, kind="shift", drift=(1.5, -0.75)),
    "var_200x160_vortex": dict(nx=200, ny=160, seed=12, kind="vortex"),
    "var_63x70_k3": dict(nx=63, ny=70, seed=13, kind="vortex", params=dict(kiters=3)),
    "var_128x96_nc2": dict(nx=128, ny=96, seed=14, kind="vortex", nc=2),
    "var_160x120_fg": dict(nx=160, ny=120, seed=15, kind="vortex", first_guess=True, params=dict(lambdac=0.5)),
    "var_150x130_brox": dict(nx=150, ny=130, seed=16, kind="vortex",
                             params=dict(dozim=0, alpha=10.0, lambda_=2.0, kiters=3, liters=2)),
    "var_101x67_cg5": dict(nx=101, ny=67, seed=17, kind="shift", drift=(-0.6, 0.9), params=dict(cgiters=5, kiters=2)),
}

NAVIGATION = {
    # GOES fixed grid, mesoscale sector away from the limb
    "nav_goes_meso": dict(kind="goes", sector="meso_0.5km", nx=120, ny=90, minX=0, minY=0),
    # full-disk corner: off-earth pixels (d<0) and the limb cut x^2+y^2 > 0.021
    "nav_goes_limb": dict(kind="goes", sector="fulldisk_0.5km", nx=160, ny=120, minX=2900, minY=2900),
    "nav_goes_2km_offset": dict(kind="goes", sector="meso_2km", nx=100, ny=100, minX=1500, minY=700),
    "nav_polar": dict(kind="polar", nx=90, ny=110),
    "nav_polar_pole": dict(kind="polar", nx=64, ny=64, lat1=90.0),
    "nav_merc": dict(kind="merc", nx=110, ny=70),
    "nav_pixuv": dict(kind="goes", sector="meso_0.5km", nx=80, ny=60, minX=0, minY=0, pixuv=1),
    "nav_moved": dict(kind="goes", sector="meso_0.5km", nx=80, ny=60, minX=0, minY=0, moved=True),
}


def variational_inputs(c):
    nx, ny, nc = c["nx"], c["ny"], c.get("nc", 1)
    i1s, i2s = [], []
    u = v = None
    for ch in range(nc):
        a, b, u, v = S.make_pair(nx, ny, c["seed"] + 100 * ch, kind=c["kind"], drift=c.get("drift", (0.8, -0.4)))
        i1s.append(a); i2s.append(b)
    img1 = np.ascontiguousarray(np.stack(i1s)) if nc > 1 else i1s[0]
    img2 = np.ascontiguousarray(np.stack(i2s)) if nc > 1 else i2s[0]
    u0 = v0 = None
    if c.get("first_guess"):
        y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
        u0 = (0.6 + 0.3 * np.sin(x / 23.0) * np.cos(y / 31.0)).astype(np.float32)
        v0 = (-0.3 + 0.2 * np.cos(x / 19.0 + y / 29.0)).astype(np.float32)
    return img1, img2, u0, v0


def nav_flow(nx, ny, seed=5):
    """A smooth displacement field with a few special values (zero, exact integers, -9999 fill)."""
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
    u = (1.7 * np.sin(x / 17.0) + 0.9 * np.cos(y / 13.0) + 0.4).astype(np.float32)
    v = (-1.1 * np.cos(x / 11.0) * np.sin(y / 19.0) - 0.25).astype(np.float32)
    u[0, 0] = 0.0; v[0, 0] = 0.0
    u[1, 1] = 2.0; v[1, 1] = -3.0
    u[2, 2] = -9999.0; v[2, 2] = -9999.0
    return u, v


def nav_constants(c):
    """kwargs for goes_nav() + (t1, t2) + flag dict."""
    kind = c["kind"]
    if kind == "goes":
        xs, ys, xo, yo, dt = S.SECTORS[c["sector"]]
        kw = dict(xScale=xs, yScale=ys, xOffset=xo, yOffset=yo, minX=c.get("minX", 0), minY=c.get("minY", 0))
        if c.get("moved"):
            kw.update(g2xOffset=xo + 0.001, g2yOffset=yo)
        extra = {}
    elif kind == "polar":
        # orthographic polar grid in metres (1 km pixels), centred near the pole
        kw = dict(xScale=1000.0, yScale=-1000.0, xOffset=-45000.0, yOffset=55000.0)
        extra = dict(lat1=c.get("lat1", 75.0), lon0=-150.0, R=6371228.0)
        dt = 3600.0
    else:
        # spherical Mercator in metres (2 km pixels)
        kw = dict(xScale=2000.0, yScale=-2000.0, xOffset=-110000.0, yOffset=4100000.0)
        extra = dict(lon1=float(np.deg2rad(-95.0)), R=6371228.0)
        dt = 3600.0
    flags = dict(pixuv=c.get("pixuv", 0), dopolar=int(kind == "polar"), domerc=int(kind == "merc"))
    return kw, extra, 1000.0, 1000.0 + dt, flags


# ---- ingest (oct_navcal_cuda) and first-guess conversion (oct_uv2pix) ---------------------------
INGEST = {
    # band-2 mesoscale sector, far from the limb
    "ingest_meso_b2": dict(sector="meso_0.5km", nx=160, ny=120, x0=0, y0=0, band=2, maxin=628.98723908, minin=-20.28991094,
                           radScale=0.1586, radOffset=-20.29),
    # full-disk window straddling the limb taper x^2+y^2 in [0.021, 0.0212) and the off-earth corner
    "ingest_limb_b13": dict(sector="fulldisk_0.5km", nx=480, ny=440, x0=3150, y0=3150, band=13, maxin=185.5699, minin=-1.6443,
                            radScale=0.04572, radOffset=-1.6443),
    # no navigation requested (second file of a pair: donav = 0)
    "ingest_nonav": dict(sector="meso_2km", nx=96, ny=64, x0=40, y0=10, band=2, maxin=628.98723908, minin=-20.28991094,
                         radScale=0.1586, radOffset=-20.29, donav=0),
}

UV2PIX = {
    "uv2pix_meso": dict(ingest="ingest_meso_b2"),
    "uv2pix_limb": dict(ingest="ingest_limb_b13"),
    "uv2pix_moved": dict(ingest="ingest_meso_b2", moved=True),
}


def ingest_inputs(c):
    """(rad counts, x counts, y counts, nav kwargs) of an ingest case; counts are seeded 12-bit radiances"""
    nx, ny = c["nx"], c["ny"]
    rng = np.random.default_rng(sum(map(ord, c["sector"])) + nx)
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
    rad = (2000 + 1500 * np.sin(x / 9.0) * np.cos(y / 7.0) + rng.integers(-200, 200, (ny, nx))).astype(np.int16)
    rad[0, 0] = 0; rad[1, 1] = 4095; rad[2, 2] = -1          # extremes / fill-like value
    xs, ys, xo, yo, dt = S.SECTORS[c["sector"]]
    xc = (np.arange(nx) + c["x0"]).astype(np.int16)
    yc = (np.arange(ny) + c["y0"]).astype(np.int16)
    return rad, xc, yc, dict(xScale=xs, yScale=ys, xOffset=xo, yOffset=yo), dt


def uv2pix_winds(nx, ny):
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
    u = (12.0 * np.sin(x / 31.0) + 6.0 * np.cos(y / 23.0) + 3.0).astype(np.float32)
    v = (-9.0 * np.cos(x / 27.0) * np.sin(y / 19.0) - 2.0).astype(np.float32)
    u[0, 0] = 0.0; v[0, 0] = 0.0
    return u, v


def ingest_r2(c):
    """x^2 + y^2 (rad^2) of every pixel of an ingest case: the limb cut of oct_navcal_cuda.cu:80-91 is at 0.0212"""
    _, xc, yc, kw, _ = ingest_inputs(c)
    xv = xc.astype(np.float64) * kw["xScale"] + kw["xOffset"]
    yv = yc.astype(np.float64) * kw["yScale"] + kw["yOffset"]
    return xv[None, :] ** 2 + yv[:, None] ** 2


def check_latlon(lat, lon, wlat, wlon, r2):
    """lat/lon parity: 2 float ulps (3e-5 deg at |lon| < 256) where the image is used (inside the limb cut);
    between the cut and the earth's edge the fixed-grid inverse is ill-conditioned (sqrt of a vanishing
    discriminant, src/oct_navcal_cuda.cu:41) and last-bit differences of sin/cos grow: 2e-3 deg there.
    Off-earth pixels (NaN) must coincide."""
    assert np.array_equal(np.isnan(lat), np.isnan(wlat)) and np.array_equal(np.isnan(lon), np.isnan(wlon))
    ok = ~np.isnan(lat)
    inner = ok & (r2 < 0.0212)
    outer = ok & ~inner
    for a, b in ((lat, wlat), (lon, wlon)):
        d = np.abs(a - b)
        assert d[inner].max(initial=0) <= 3.1e-5, d[inner].max(initial=0)
        assert d[outer].max(initial=0) <= 2e-3, d[outer].max(initial=0)


# ---- ingest of the projected grids (oct_polar_navcal_cuda / oct_merc_navcal_cuda) ------------------
GRIDNAV = {
    "gridnav_polar": dict(grid=1, nx=90, ny=110, xScale=1000.0, xOffset=-45000.0, yScale=-1000.0, yOffset=55000.0,
                          R=6371228.0, lon0=-150.0, lat1=75.0),
    "gridnav_polar_origin": dict(grid=1, nx=41, ny=41, xScale=1000.0, xOffset=-20000.0, yScale=-1000.0, yOffset=20000.0,
                                 R=6371228.0, lon0=30.0, lat1=90.0),       # passes through rho = 0
    "gridnav_merc": dict(grid=2, nx=110, ny=70, xScale=2000.0, xOffset=-110000.0, yScale=-2000.0, yOffset=4100000.0,
                         R=6371228.0, lon0=-95.0, lat1=0.0),
    "gridnav_merc_nonav": dict(grid=2, nx=32, ny=24, xScale=2000.0, xOffset=0.0, yScale=-2000.0, yOffset=100000.0,
                               R=6371228.0, lon0=10.0, lat1=0.0, donav=0),
}


def gridnav_inputs(c):
    nx, ny = c["nx"], c["ny"]
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
    data = (120.0 + 90.0 * np.sin(x / 7.0) * np.cos(y / 5.0)).astype(np.float32)
    return data, np.arange(nx, dtype=np.int16), np.arange(ny, dtype=np.int16)


# ---- regridding of a finer field (oct_zoom_out_float) and the -srsal post-smoother (oct_srsal_cu) ---
# (ny, nx), factor: integer ratios (the GOES channel pairs: 0.5 km -> 1 km / 2 km), non-integer ratios
# (bicubic between blurred pixels), a blur radius above the minimum of 5 (factor 1/8 -> 9), the copy branch
ZOOMOUT = {
    "half": ((97, 131), 0.5),
    "quarter": ((120, 160), 0.25),
    "third": ((90, 77), 1.0 / 3.0),
    "ragged": ((64, 80), 0.37),
    "eighth": ((200, 240), 0.125),
    "copy": ((50, 50), 1.0),
    "almost_one": ((40, 40), 0.9999995),
    "tiny": ((7, 9), 0.5),
}


def zoomout_input(name):
    (ny, nx), factor = ZOOMOUT[name]
    rng = np.random.default_rng(nx * 7 + ny)
    return (rng.standard_normal((ny, nx)) * 1000 + 5000).astype(np.float32), factor


def zoomout_reference(oracle, key, field, factor, pyramid=False):
    """The reference's oct_zoom_out_float of `field` or, with pyramid=True, its double pyramid stage oct_zoom_out
    rounded to float.  Computed by the reference's own object when oracle/_ref is built, else the stored output
    zoomout_ref.npz[key] (make_golden.py --zoomout-only): keys are the ZOOMOUT names and config1_<factor> for the
    500 x 500 texture of BASELINE config 1."""
    try:
        return oracle.ref_zoom_out(field, factor).astype(np.float32) if pyramid else oracle.ref_zoom_out_float(field, factor)
    except OSError:
        import os
        with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "zoomout_ref.npz")) as z:
            return z[key]


SRSAL = {
    # cloud deck with sharp edges (range weight switches neighbours off) and smooth height variation
    "srsal_96x80_deck": dict(nx=96, ny=80, seed=31, kind="deck"),
    # barely larger than the window radius: every pixel reflects on both sides
    "srsal_23x19_small": dict(nx=23, ny=19, seed=32, kind="smooth"),
    # constant heights: the range weight is 1 and the filter is the plain truncated Gaussian
    "srsal_70x50_flat": dict(nx=70, ny=50, seed=33, kind="flat"),
}


def srsal_inputs(c):
    nx, ny = c["nx"], c["ny"]
    rng = np.random.default_rng(c["seed"])
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
    u = (1.7 * np.sin(x / 17.0) + 0.9 * np.cos(y / 13.0) + 0.4 + 0.3 * rng.standard_normal((ny, nx))).astype(np.float32)
    v = (-1.1 * np.cos(x / 11.0) * np.sin(y / 19.0) - 0.25 + 0.3 * rng.standard_normal((ny, nx))).astype(np.float32)
    if c["kind"] == "flat":
        cth = np.full((ny, nx), 8000.0, np.float32)
    elif c["kind"] == "smooth":
        cth = (6000.0 + 30.0 * np.sin(x / 5.0) * np.cos(y / 4.0)).astype(np.float32)
    else:
        cth = (2000.0 + 15.0 * np.sin(x / 9.0) + 10.0 * np.cos(y / 7.0)).astype(np.float32)
        cth[(x - 0.55 * nx) ** 2 + (y - 0.45 * ny) ** 2 < (0.28 * ny) ** 2] += 9000.0      # a tower
        cth[:, : nx // 5] += 40.0                                                          # a low step (partial weight)
        cth += (5.0 * rng.standard_normal((ny, nx))).astype(np.float32)
    return u, v, cth


# ---- the benchmarked configurations (BASELINE.json configs 2-4) -----------------------------------
# Large enough for the TMA-fed PCG kernels (nx >= 512).  The reference's own sm_100 build is valid up to
# ~178 Mpix (int CSR offsets, src/oct_variational_optical_flow.cu:1222,1293), so the mesoscale sector, CONUS
# and 2048^2 crops of the tapered full-disk scene all have reference outputs; the fixtures keep a strided
# sample of u, v (`stride`), one full-resolution block and global statistics.  Inputs are regenerated at
# test time on the CPU (`S.make_pair_torch(..., "cpu")`), never stored.
FULLDISK = (21696, 21696)
HEADLINE = {
    "ref_1024x768": dict(kind="scene", nx=1024, ny=768, seed=21, stride=3, runs=2),
    "ref_meso_2000": dict(kind="scene", nx=2000, ny=2000, seed=2, stride=5, runs=2),        # config 2
    "ref_conus": dict(kind="scene", nx=10000, ny=6000, seed=4, stride=16, runs=1),          # config 3
    # config 4: crops of the tapered full-disk scene (seed 4, the bench's scene)
    "ref_fd_centre": dict(kind="fdcrop", x0=9824, y0=9824, size=2048, seed=4, stride=8, runs=2),
    # the limb on the equator: disk, the taper band x^2+y^2 in [0.021, 0.0212) and space (all-zero columns)
    "ref_fd_limb": dict(kind="fdcrop", x0=19648, y0=9824, size=2048, seed=4, stride=8, runs=2),
    # towards the corner: space (zeros) in the upper left, the taper band on the diagonal, disk below it
    "ref_fd_corner": dict(kind="fdcrop", x0=2600, y0=2600, size=2048, seed=4, stride=8, runs=2),
}
BLOCK = 128      # edge of the full-resolution block kept in a headline fixture (at the scene centre)


def headline_inputs(c):
    """(img1, img2) float32 numpy arrays of a HEADLINE case, generated on the CPU"""
    if c["kind"] == "scene":
        a, b = S.make_pair_torch(c["nx"], c["ny"], c["seed"], "cpu")
        return a.numpy(), b.numpy()
    nx, ny = FULLDISK
    x0, y0, n = c["x0"], c["y0"], c["size"]
    a, b = S.make_pair_torch(nx, ny, c["seed"], "cpu", limb_taper=True, rows=(y0, y0 + n))
    return a[:, x0:x0 + n].contiguous().numpy(), b[:, x0:x0 + n].contiguous().numpy()


def headline_digest(u, v, stride):
    """what a headline fixture keeps of a flow field: strided sample, centre block, float64 statistics"""
    ny, nx = u.shape
    by, bx = max(0, ny // 2 - BLOCK // 2), max(0, nx // 2 - BLOCK // 2)
    return dict(us=np.ascontiguousarray(u[::stride, ::stride]), vs=np.ascontiguousarray(v[::stride, ::stride]),
                ub=np.ascontiguousarray(u[by:by + BLOCK, bx:bx + BLOCK]), vb=np.ascontiguousarray(v[by:by + BLOCK, bx:bx + BLOCK]),
                stats=np.array([np.abs(u, dtype=np.float64).mean(), np.abs(v, dtype=np.float64).mean(),
                                float(np.abs(u).max()), float(np.abs(v).max()),
                                u.astype(np.float64).sum(), v.astype(np.float64).sum()]))


def input_hash(*arrays):
    import hashlib
    h = hashlib.sha1()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()
