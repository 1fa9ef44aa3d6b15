"""Generates tests/golden/*.npz by running the UNMODIFIED REFERENCE
(oracle/_ref/libref_cuda.so = the reference sources recompiled for sm_100) on the
seeded inputs of cases.py.  Needs a GPU:

    gpurun -- 'python tests/golden/make_golden.py gpurun_out/golden'
    cp gpurun_out/golden/*.npz tests/golden/

The reference's float atomics make it run-to-run non-reproducible, so each
variational case is run three times and the fixture records the spread.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402

import cases  # noqa: E402
from oracle import oracle as O  # noqa: E402


def ingest(out):
    """fixtures of the ingest stage (oct_navcal_cuda) and the first-guess conversion (oct_uv2pix)"""
    out_dir = out
    made = {}
    for name, c in cases.INGEST.items():
        rad, xc, yc, kw, dt = cases.ingest_inputs(c)
        nav = O.goes_nav(**kw)
        cal = O.goes_cal(nav, c["radScale"], c["radOffset"], c["maxin"], c["minin"], donav=c.get("donav", 1))
        data, lat, lon = O.ref_navcal(rad, xc, yc, cal)
        made[name] = (lat, lon, xc, yc, kw, dt)
        np.savez_compressed(os.path.join(out, name + ".npz"), rad=rad, x=xc, y=yc, data=data, lat=lat, lon=lon)
        print(name, "data range", float(data.min()), float(data.max()), "zeros", int((data == 0).sum()),
              "lat range", float(np.nanmin(lat)), float(np.nanmax(lat)), "nan", int(np.isnan(lat).sum()), flush=True)
    for name, c in cases.GRIDNAV.items():
        data, xc, yc = cases.gridnav_inputs(c)
        gout, lat, lon = O.ref_navcal_grid(c["grid"], data, xc, yc, c["xScale"], c["xOffset"], c["yScale"], c["yOffset"], c["R"],
                                          c["lon0"], c["lat1"], c.get("donav", 1))
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), data=gout, lat=lat, lon=lon)
        print(name, "lat range", float(np.nanmin(lat)), float(np.nanmax(lat)), "lon range", float(np.nanmin(lon)),
              float(np.nanmax(lon)), "nan", int(np.isnan(lat).sum()), flush=True)
    for name, c in cases.UV2PIX.items():
        lat, lon, xc, yc, kw, dt = made[c["ingest"]]
        kw = dict(kw)
        if c.get("moved"):
            kw.update(g2xOffset=kw["xOffset"] + 0.001, g2yOffset=kw["yOffset"])
        nav = O.goes_nav(**kw)
        u, v = cases.uv2pix_winds(len(xc), len(yc))
        up, vp = O.ref_uv2pix(nav, 1000.0, 1000.0 + dt, lat, lon, xc, yc, u, v)
        np.savez_compressed(os.path.join(out, name + ".npz"), u=u, v=v, upix=up, vpix=vp)
        print(name, "upix range", float(np.nanmin(up)), float(np.nanmax(up)), "zeros", int((up == 0).sum()), flush=True)


def srsal(out):
    """fixtures of the -srsal post-smoother (the reference's oct_srsal_cu, a CUDA kernel)"""
    for name, c in cases.SRSAL.items():
        u, v, cth = cases.srsal_inputs(c)
        us, vs = O.ref_srsal(u, v, cth)
        np.savez_compressed(os.path.join(out, name + ".npz"), u=us, v=vs)
        print(name, "u range", float(us.min()), float(us.max()), "mean |du|", float(np.abs(us - u).mean()), flush=True)


def zoomout(out):
    """zoomout_ref.npz: the reference's CPU regridder oct_zoom_out_float on cases.ZOOMOUT and its double pyramid stage
    oct_zoom_out, rounded to float, on the 500 x 500 texture of BASELINE config 1 (cases.zoomout_reference).  Without
    oracle/_ref the outputs come from the oracle's restatement, which was bit-identical to the reference's object on
    all of these inputs in every run that had both; the committed file was written that way."""
    from octane_b200 import synthetic as S
    try:
        O.ref_cpu()
        src = "reference"
        fn, fn_pyr = O.ref_zoom_out_float, lambda f, k: O.ref_zoom_out(f, k).astype(np.float32)
    except OSError:
        src = "oracle"
        fn = fn_pyr = O.zoom_out_float
    d = {name: fn(*cases.zoomout_input(name)) for name in sorted(cases.ZOOMOUT)}
    i1 = S.make_pair(500, 500, seed=1, kind="shift", drift=(2.0, -1.0))[0]
    for factor in (0.5, 0.25, 0.125):
        d[f"config1_{factor}"] = fn_pyr(i1, factor)
    np.savez_compressed(os.path.join(out, "zoomout_ref.npz"), **d)
    print("zoomout_ref from the", src, {k: v.shape for k, v in d.items()}, flush=True)


def main(out):
    os.makedirs(out, exist_ok=True)
    if "--ingest-only" in sys.argv:
        return ingest(out)
    if "--zoomout-only" in sys.argv:
        return zoomout(out)
    if "--srsal-only" in sys.argv:
        return srsal(out)
    for name, c in cases.VARIATIONAL.items():
        img1, img2, u0, v0 = cases.variational_inputs(c)
        kw = dict(c.get("params", {}))
        rp = O.ref_params(dofirstguess=int(bool(c.get("first_guess"))), **kw)
        runs = [O.ref_variational(img1, img2, rp, u0, v0, nc=c.get("nc", 1)) for _ in range(3)]
        u = runs[0][0]; v = runs[0][1]
        spread = max(float(np.abs(r[0] - u).max()) for r in runs[1:]), max(float(np.abs(r[1] - v).max()) for r in runs[1:])
        np.savez_compressed(os.path.join(out, name + ".npz"), img1=img1, img2=img2,
                            u0=u0 if u0 is not None else np.zeros(0, np.float32),
                            v0=v0 if v0 is not None else np.zeros(0, np.float32),
                            u=u, v=v, spread=np.array(spread))
        print(name, "spread", spread, "u range", float(u.min()), float(u.max()), flush=True)
    for name, c in cases.NAVIGATION.items():
        kw, extra, t1, t2, flags = cases.nav_constants(c)
        nav = O.goes_nav(**kw)
        for k, val in extra.items():
            setattr(nav, k, val)
        u, v = cases.nav_flow(c["nx"], c["ny"])
        rp = O.ref_params(**flags)
        # the reference leaves ur2/vr2 unwritten with -pd: prefill so the fixture is defined
        U, V, U2, V2, dT = O.ref_pix2uv(nav, t1, t2, u, v, rp)
        np.savez_compressed(os.path.join(out, name + ".npz"), u=u, v=v, U=U, V=V, U_raw=U2, V_raw=V2, dT=np.float32(dT))
        print(name, "U range", int(U.min()), int(U.max()), "V range", int(V.min()), int(V.max()), "zeros", int((U == 0).sum()), flush=True)
    # dispatcher with cloud-top heights (CTP pack), both scalings
    c = cases.VARIATIONAL["var_96x80_shift"]
    img1, img2, _, _ = cases.variational_inputs(c)
    ny, nx = img1.shape
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = (7500.0 + 7400.0 * np.sin(x / 20.0) * np.cos(y / 15.0)).astype(np.float32)
    kw, extra, t1, t2, flags = cases.nav_constants(cases.NAVIGATION["nav_goes_meso"])
    nav = O.goes_nav(**kw)
    import ctypes as C
    for ir in (0, 1):
        rp = O.ref_params(doCTH=1, ir=ir)
        cthv = cth if ir == 0 else (cth / 100.0 + 200.0).astype(np.float32)
        outs = [np.zeros((ny, nx), np.int16) for _ in range(5)]
        up = np.zeros((ny, nx), np.float32); vp = np.zeros((ny, nx), np.float32)
        dT = C.c_float()
        O.ref_cuda().ref_optical_flow(img1, img2, cthv.ctypes.data, nx, ny, C.byref(nav), t1, t2, C.byref(rp),
                                      up, vp, outs[0], outs[1], outs[2], outs[3], outs[4].ctypes.data, C.byref(dT))
        np.savez_compressed(os.path.join(out, f"dispatch_cth_ir{ir}.npz"), img1=img1, img2=img2, cth=cthv,
                            uPix=up, vPix=vp, U=outs[0], V=outs[1], U_raw=outs[2], V_raw=outs[3], CTP=outs[4],
                            dT=np.float32(dT.value))
        print("dispatch ir", ir, "CTP range", int(outs[4].min()), int(outs[4].max()), flush=True)
    ingest(out)
    srsal(out)
    zoomout(out)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 and not sys.argv[1].startswith("--") else os.path.join(ROOT, "gpurun_out", "golden"))
