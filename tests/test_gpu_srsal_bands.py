"""-srsal on row bands (octane_srsal_band_dev) and -srsal / a first guess through the pipelined dispatcher
(octane_stream_submit, octane_stream_submit_fg).

One GPU: the banded entry point at world size 1 is octane_srsal_dev, and the pipelined dispatcher gives, bit for bit,
what the blocking dispatcher gives with the same flags.  Row bands (needs as many GPUs as ranks): the gathered bands are
bit for bit the single-GPU filter of the whole field, the pipelined dispatcher on bands equals the banded device path,
and a refusal or a rank out of memory comes back as an error on every rank (tests/band_post_worker.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
import octane_b200 as ob
from octane_b200 import synthetic as S

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2", "CTP")


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def pinned(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def cloud_tops(nx, ny):
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    return (7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)


def run_pipeline(ctx, pairs, nav, dt, p, nx, ny, cth=None, fg=None, keys=KEYS):
    """submit every pair, two in flight, and return the outputs pair by pair"""
    import torch
    outs = [{k: torch.zeros((ny, nx), dtype=(torch.float32 if k.endswith("Pix") else torch.int16), pin_memory=True).numpy()
             for k in keys} for _ in range(2)]
    kw = {} if fg is None else dict(fg_u_band=fg[0], fg_v_band=fg[1])
    got = []
    for k, (a, b) in enumerate(pairs):
        ctx.stream_submit(k % 2, a, b, nav, 0.0, dt, p, outs[k % 2], nx, ny, cth=cth, **kw)
        if k > 0:
            ctx.stream_wait((k - 1) % 2)
            got.append({key: val.copy() for key, val in outs[(k - 1) % 2].items()})
    ctx.stream_wait((len(pairs) - 1) % 2)
    got.append({key: val.copy() for key, val in outs[(len(pairs) - 1) % 2].items()})
    return got


def test_srsal_band_on_one_gpu_is_the_single_gpu_filter(ctx):
    """world size 1: the band is the scene, octane_srsal_band_dev is octane_srsal_dev (fixture inputs and the sizes
    that leave partial 32 x 8 tiles)"""
    rng = np.random.default_rng(9)
    fields = [cases.srsal_inputs(cases.SRSAL[name]) for name in sorted(cases.SRSAL)]
    for ny, nx in ((19, 19), (33, 45), (41, 130)):
        fields.append((rng.standard_normal((ny, nx)).astype(np.float32), rng.standard_normal((ny, nx)).astype(np.float32),
                       (5000 + 25 * rng.standard_normal((ny, nx))).astype(np.float32)))
    for u, v, cth in fields:
        ny, nx = u.shape
        wu, wv = ctx.oct_srsal_cu(dev(u), dev(v), dev(cth))
        gu, gv = ctx.oct_srsal_band(dev(u), dev(v), dev(cth), nx, ny)
        assert np.array_equal(gu.cpu().numpy(), wu.cpu().numpy()) and np.array_equal(gv.cpu().numpy(), wv.cpu().numpy())
    z = dev(np.zeros((18, 64), np.float32))
    with pytest.raises(ob.OctaneError):
        ctx.oct_srsal_band(z, z.clone(), z.clone(), 64, 18)


def test_pipelined_srsal_matches_blocking_calls(ctx):
    """doCTH + dosrsal with uPix / vPix requested, five pairs, two in flight: every output is the blocking dispatcher's,
    and the navigated and CTP planes are those of the run without -srsal (they come from the unsmoothed flow)"""
    nx, ny = 640, 200
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(doCTH=1, dosrsal=1, kiters=3)
    cth = cloud_tops(nx, ny)
    pairs = [S.make_pair(nx, ny, 300 + k)[:2] for k in range(5)]
    want = [ctx.oct_optical_flow(a, b, nav, 0.0, dt, p, cth=cth) for a, b in pairs]
    plain = [ctx.oct_optical_flow(a, b, nav, 0.0, dt, ob.default_params(doCTH=1, kiters=3), cth=cth) for a, b in pairs]
    got = run_pipeline(ctx, [(pinned(a), pinned(b)) for a, b in pairs], nav, dt, p, nx, ny, cth=pinned(cth))
    for k in range(len(pairs)):
        for key in KEYS:
            assert np.array_equal(got[k][key], want[k][key]), (k, key)
        for key in ("uVal", "vVal", "uVal2", "vVal2", "CTP"):
            assert np.array_equal(got[k][key], plain[k][key]), (k, key)
        assert not np.array_equal(got[k]["uPix"], plain[k]["uPix"])          # the smoother did run


def test_pipelined_first_guess_matches_blocking_calls(ctx):
    """octane_stream_submit_fg with -firstguess -lambdac 0.5: the blocking dispatcher given the same first guess in
    upix / vpix, bit for bit; the first-guess arrays are only read"""
    nx, ny = 640, 200
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(first_guess=1, lambdac=0.5, kiters=3)
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    fgu = (0.6 + 0.3 * np.sin(xx / 23.0) * np.cos(yy / 31.0)).astype(np.float32)
    fgv = (-0.3 + 0.2 * np.cos(xx / 19.0 + yy / 29.0)).astype(np.float32)
    pairs = [S.make_pair(nx, ny, 320 + k)[:2] for k in range(4)]
    want = [ctx.oct_optical_flow(a, b, nav, 0.0, dt, p, upix=fgu.copy(), vpix=fgv.copy()) for a, b in pairs]
    hfg = (pinned(fgu), pinned(fgv))
    keys = ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")
    got = run_pipeline(ctx, [(pinned(a), pinned(b)) for a, b in pairs], nav, dt, p, nx, ny, fg=hfg, keys=keys)
    for k in range(len(pairs)):
        for key in keys:
            assert np.array_equal(got[k][key], want[k][key]), (k, key)
    assert np.array_equal(hfg[0], fgu) and np.array_equal(hfg[1], fgv)
    zero = ctx.oct_optical_flow(*pairs[0], nav, 0.0, dt, ob.default_params(kiters=3))
    assert not np.array_equal(got[0]["uPix"], zero["uPix"])                 # the first guess did steer the solve


def test_pipelined_srsal_and_first_guess_with_deferred_copy_out():
    """the two tests above under the copy-out schedule of banded contexts (OCTANE_STREAM_DEFER=1, read once per process,
    hence the child process): the copy-out of a pair must still read the smoothed displacements"""
    if os.environ.get("OCTANE_STREAM_DEFER"):
        pytest.skip("already inside the child run")
    env = dict(os.environ, OCTANE_STREAM_DEFER="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
                        "-k", "test_pipelined_srsal_matches_blocking_calls or test_pipelined_first_guess_matches_blocking_calls"],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "2 passed" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_pipelined_dispatcher_refusals(ctx):
    """-srsal needs the heights and the pixel displacements it smooths; the first-guess submit needs p.first_guess and
    both first-guess planes, and the plain submit still refuses p.first_guess.  The context works afterwards."""
    nx, ny = 256, 96
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    a, b = S.make_pair(nx, ny, 340)[:2]
    cth = cloud_tops(nx, ny)
    fg = np.zeros((ny, nx), np.float32)
    out = {k: np.zeros((ny, nx), np.float32 if k.endswith("Pix") else np.int16) for k in ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")}
    no_pix = {k: out[k] for k in ("uVal", "vVal", "uVal2", "vVal2")}
    srsal, fgp = ob.default_params(dosrsal=1, kiters=3), ob.default_params(first_guess=1, kiters=3)
    refused = [
        lambda: ctx.stream_submit(0, a, b, nav, 0.0, dt, srsal, out, nx, ny),                         # no heights
        lambda: ctx.stream_submit(0, a, b, nav, 0.0, dt, srsal, no_pix, nx, ny, cth=cth),             # no uPix / vPix
        lambda: ctx.stream_submit(0, a, b, nav, 0.0, dt, ob.default_params(kiters=3), out, nx, ny,
                                  fg_u_band=fg, fg_v_band=fg),                                        # no p.first_guess
        lambda: ctx.stream_submit(0, a, b, nav, 0.0, dt, fgp, out, nx, ny, fg_u_band=fg),              # one plane only
        lambda: ctx.stream_submit(0, a, b, nav, 0.0, dt, fgp, out, nx, ny),                           # plain submit
    ]
    for call in refused:
        with pytest.raises(ob.OctaneError) as e:
            call()
        assert e.value.code == -2
    want = ctx.oct_optical_flow(a, b, nav, 0.0, dt, srsal, cth=cth)
    ctx.stream_submit(0, a, b, nav, 0.0, dt, srsal, out, nx, ny, cth=cth)
    ctx.stream_wait(0)
    for k in out:
        assert np.array_equal(out[k], want[k]), k


# ---- row bands ----------------------------------------------------------------------------------------------------
def run_worker(world, nx, ny, modes):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 30600 + os.getpid() % 1000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "band_post_worker.py"),
           str(nx), str(ny), modes]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("BAND_POST_RESULT ")]
    assert line, out.stdout[-2000:] + out.stderr[-4000:]
    return json.loads(line[0][len("BAND_POST_RESULT "):])


@pytest.mark.parametrize("world,shape", [(2, (1500, 1100)), (4, (1500, 1100)), (2, (100, 36)), (8, (6000, 6000))])
def test_srsal_band_equals_single_gpu(world, shape):
    """the gathered bands are bit for bit the single-GPU filter of the whole field (100 x 36 on two ranks: bands of
    exactly 18 rows, every window reaches the far edge of the neighbour's band)"""
    r = run_worker(world, *shape, "field")
    assert r["field_equal"], r


def test_srsal_band_refusals_and_recovery():
    """ny = 35 on two ranks (a 17-row band): every rank refuses, nothing hangs.  Then one rank cannot allocate its
    staging: every rank gets an error, and the same contexts filter correctly on the next call."""
    r = run_worker(2, 100, 35, "refuse")
    assert r["refused_everywhere"], r
    assert r["oom_everywhere"] and r["oom_codes"][-1] == -3, r
    assert r["recovered"], r


@pytest.mark.parametrize("world,shape", [(2, (1500, 1100)), (4, (4000, 3000))])
def test_pipelined_srsal_on_bands(world, shape):
    """octane_stream_submit with -srsal on bands: bit for bit the banded device path (band solve -> pix2uv_band ->
    oct_srsal_band); against the single-GPU pipeline the gates of test_banded_equals_single_gpu, and -- the filter is a
    convex combination -- no larger a difference after smoothing than before it"""
    r = run_worker(world, *shape, "stream")
    assert r["stream_equal"], r
    assert r["du_mean"] < 1e-4 and r["dv_mean"] < 1e-4 and r["du_max"] < 2e-3 and r["dv_max"] < 2e-3, r
    assert r["nav_max"] <= 2, r
    assert r["du_max"] <= r["du_raw_max"] + 1e-6 and r["dv_max"] <= r["dv_raw_max"] + 1e-6, r


@pytest.mark.parametrize("world,shape", [(2, (1500, 1100)), (4, (4000, 3000))])
def test_pipelined_first_guess_on_bands(world, shape):
    """octane_stream_submit_fg on bands: bit for bit octane_variational_flow_band_fg_dev -> pix2uv_band"""
    r = run_worker(world, *shape, "fg")
    assert r["fg_equal"], r
