"""Batched dispatcher (octane_optical_flow_batch_dev): many same-size pairs in one call.

A pair's result must not depend on the other pairs of the call (batch invariance), must meet the single-pair gates
against the CPU oracle and the reference's fixtures, and must agree with the single-pair dispatcher up to the
reordered dot-product sums of the per-pair PCG groups."""
import numpy as np
import pytest

import cases
import octane_b200 as ob
from conftest import load_golden
from octane_b200 import synthetic as S

pytestmark = pytest.mark.gpu
KEYS_F = ("uPix", "vPix")
KEYS_S = ("uVal", "vVal", "uVal2", "vVal2", "CTP")


@pytest.fixture(scope="module")
def bctx():
    c = ob.Context(0)
    yield c
    c.close()


def tdev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_batch(ctx, img1, img2, navs, t1, t2, p, cth=None, nc=1):
    """img1 / img2: numpy [B, (nc,) ny, nx]; returns (dict of numpy [B, ny, nx], moved, its [B, n_solves])"""
    import torch
    B = img1.shape[0]
    ny, nx = img1.shape[-2:]
    out = {k: torch.zeros((B, ny, nx), device="cuda") for k in KEYS_F}
    for k in KEYS_S:
        if k != "CTP" or p.doCTH:
            out[k] = torch.zeros((B, ny, nx), dtype=torch.int16, device="cuda")
    moved = ctx.oct_optical_flow_batch_dev(tdev(img1), tdev(img2), navs, t1, t2, p, out,
                                           cth=None if cth is None else tdev(cth), nc=nc)
    its = ctx.batch_cg_iterations(B, p.kiters * 3 * p.liters)
    return {k: v.cpu().numpy() for k, v in out.items()}, moved, its


def meso_inputs(npairs, n=500, seed0=100):
    """bench.py's batch64 generator: seeded pairs and the same cloud-top-height field for every pair"""
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    yy, xx = np.mgrid[0:n, 0:n].astype(np.float32)
    cth = (7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)
    pairs = [S.make_pair(n, n, seed0 + k)[:2] for k in range(npairs)]
    img1 = np.stack([a for a, _ in pairs]).astype(np.float32)
    img2 = np.stack([b for _, b in pairs]).astype(np.float32)
    return img1, img2, np.stack([cth] * npairs), [nav] * npairs, [0.0] * npairs, [dt] * npairs


def test_batch_invariance(bctx):
    """64 pairs of 500^2 with CTH: one call, a shuffled call and ragged sub-batches give the same bits per pair"""
    img1, img2, cth, navs, t1, t2 = meso_inputs(64)
    p = ob.default_params(doCTH=1)
    full, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
    perm = np.random.default_rng(5).permutation(64)
    shuf, _, its_s = run_batch(bctx, img1[perm], img2[perm], navs, t1, t2, p, cth[perm])
    for k in full:
        assert np.array_equal(shuf[k], full[k][perm]), k
    assert np.array_equal(its_s, its[perm])
    b0 = 0
    for n in (1, 5, 58):
        part, _, its_p = run_batch(bctx, img1[b0:b0 + n], img2[b0:b0 + n], navs[:n], t1[:n], t2[:n], p, cth[b0:b0 + n])
        for k in full:
            assert np.array_equal(part[k], full[k][b0:b0 + n]), (k, n)
        assert np.array_equal(its_p, its[b0:b0 + n])
        b0 += n


VAR_CASES = sorted(k for k, c in cases.VARIATIONAL.items() if not c.get("first_guess") and
                   cases.variational_inputs(c)[2] is None)


@pytest.mark.parametrize("name", VAR_CASES)
def test_batch_matches_oracle_and_fixture(bctx, oracle, name):
    """each of three copies of a pair meets the single-pair gates against the oracle and the reference fixture"""
    c = cases.VARIATIONAL[name]
    nc = c.get("nc", 1)
    img1, img2, _, _ = cases.variational_inputs(c)
    p = ob.default_params(**c.get("params", {}))
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    navs = [ob.goes_nav(xs, ys, xo, yo)] * 3
    out, _, its = run_batch(bctx, np.stack([img1] * 3), np.stack([img2] * 3), navs, [0.0] * 3, [dt] * 3, p, nc=nc)
    uo, vo, its_o = oracle.variational_flow(img1, img2, oracle.params(**c.get("params", {})), None, None, nc=nc)
    g = load_golden(name)
    for b in range(3):
        u, v = out["uPix"][b], out["vPix"][b]
        assert np.abs(u - uo).mean() < 1e-4 and np.abs(v - vo).mean() < 1e-4
        assert np.abs(u - uo).max() < 2e-3 and np.abs(v - vo).max() < 2e-3
        assert list(its[b]) == list(its_o)
        du, dv = np.abs(u - g["u"]), np.abs(v - g["v"])
        assert du.mean() < 1e-3 and dv.mean() < 1e-3 and du.max() < 1e-2 and dv.max() < 1e-2
        assert max(du.max(), dv.max()) < max(20 * float(g["spread"].max()), 2e-4)


def single(ctx, a, b, nav, t1, t2, p, cth):
    import torch
    ny, nx = a.shape[-2:]
    u, v = torch.zeros((ny, nx), device="cuda"), torch.zeros((ny, nx), device="cuda")
    s = [torch.zeros((ny, nx), dtype=torch.int16, device="cuda") for _ in range(5)]
    ctx.oct_optical_flow_dev(tdev(a), tdev(b), nav, t1, t2, p, u, v, *s[:4], cth=tdev(cth), ctp=s[4])
    ctx.synchronize()
    r = dict(uPix=u.cpu().numpy(), vPix=v.cpu().numpy())
    r.update({k: x.cpu().numpy() for k, x in zip(KEYS_S, s)})
    return r


def check_vs_single(out, b, want, tag):
    dmax = max(np.abs(out["uPix"][b] - want["uPix"]).max(), np.abs(out["vPix"][b] - want["vPix"]).max())
    print(f"{tag} pair {b}: max |d uPix, vPix| vs the single-pair dispatcher = {dmax:.3e} px")
    assert dmax < 2e-4
    if "CTP" in out:
        assert np.array_equal(out["CTP"][b], want["CTP"])
    for k in ("uVal", "vVal"):
        d = np.abs(out[k][b].astype(int) - want[k].astype(int))
        assert d.max() <= 2 and (d > 0).mean() < 0.02, k
    for k in ("uVal2", "vVal2"):
        assert np.abs(out[k][b].astype(int) - want[k].astype(int)).max() <= 1, k


@pytest.mark.parametrize("ir", [0, 1])
def test_batch_matches_single_dispatcher_cth(bctx, ir):
    g = load_golden(f"dispatch_cth_ir{ir}")
    kw, extra, t1, t2, flags = cases.nav_constants(cases.NAVIGATION["nav_goes_meso"])
    nav = ob.goes_nav(**kw)
    p = ob.default_params(doCTH=1, ir=ir)
    want = single(bctx, g["img1"], g["img2"], nav, t1, t2, p, g["cth"])
    out, moved, _ = run_batch(bctx, np.stack([g["img1"]] * 2), np.stack([g["img2"]] * 2), [nav] * 2, [t1] * 2, [t2] * 2,
                              p, np.stack([g["cth"]] * 2))
    for b in range(2):
        check_vs_single(out, b, want, f"dispatch_cth_ir{ir}")


def test_batch_matches_single_dispatcher_pairs(bctx):
    """the pairs of the contexts-in-flight test, in one call, with one pair's sector moved"""
    nx, ny, npairs = 200, 160, 6
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    moved_nav = ob.goes_nav(xs, ys, xo, yo)
    moved_nav.g2xOffset = moved_nav.xOffset + 0.001
    navs = [nav] * npairs
    navs[3] = moved_nav
    p = ob.default_params(doCTH=1)
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = (7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)
    pairs = [S.make_pair(nx, ny, 200 + k)[:2] for k in range(npairs)]
    out, moved, _ = run_batch(bctx, np.stack([a for a, _ in pairs]), np.stack([b for _, b in pairs]), navs,
                              [0.0] * npairs, [dt] * npairs, p, np.stack([cth] * npairs))
    assert moved == [3]
    for b, (i1, i2) in enumerate(pairs):
        check_vs_single(out, b, single(bctx, i1, i2, navs[b], 0.0, dt, p, cth), "pairs")


@pytest.mark.parametrize("solver", [1, 0])
def test_batch_large_levels(solver):
    """2000^2 pairs: the finest levels run the single-pair PCG kernels pair by pair, under both solvers"""
    ctx = ob.Context(0)
    try:
        ctx.set_solver(solver)
        img1, img2, cth, navs, t1, t2 = meso_inputs(3, n=2000, seed0=300)
        p = ob.default_params(doCTH=1)
        out, _, its = run_batch(ctx, img1, img2, navs, t1, t2, p, cth)
        for b in range(3):
            check_vs_single(out, b, single(ctx, img1[b], img2[b], navs[b], t1[b], t2[b], p, cth[b]), f"2000^2 solver {solver}")
    finally:
        ctx.close()


def test_batch_launch_count_does_not_grow_with_pairs(bctx):
    """16 pairs of 500^2 take as many launches as one pair (they fit one cooperative launch per solve)"""
    img1, img2, cth, navs, t1, t2 = meso_inputs(16)
    p = ob.default_params(doCTH=1)
    run_batch(bctx, img1[:1], img2[:1], navs[:1], t1[:1], t2[:1], p, cth[:1])
    one = bctx.stats().kernel_launches
    run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
    sixteen = bctx.stats().kernel_launches
    print(f"kernel launches: 1 pair {one}, 16 pairs {sixteen}")
    assert one > 0 and sixteen == one


def test_batch_refusals_leave_context_usable(bctx):
    img1, img2, cth, navs, t1, t2 = meso_inputs(2, n=200)
    p = ob.default_params(doCTH=1)
    want, _, its_want = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)

    def refused(fn):
        with pytest.raises(ob.OctaneError) as e:
            fn()
        assert e.value.code == -2                          # OCTANE_EINVAL
        got, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
        for k in want:
            assert np.array_equal(got[k], want[k]), k
        assert np.array_equal(its, its_want)

    refused(lambda: run_batch(bctx, img1[:0], img2[:0], [], [], [], p, cth[:0]))
    refused(lambda: run_batch(bctx, img1, img2, navs, t1, t2, ob.default_params(doCTH=1, first_guess=1), cth))
    refused(lambda: run_batch(bctx, img1, img2, navs, t1, t2, ob.default_params(doCTH=1, dosrsal=1), cth))
