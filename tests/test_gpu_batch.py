"""Batched dispatcher (octane_optical_flow_batch_dev): many same-size pairs in one call.

A pair's result must not depend on the other pairs of the call (batch invariance), must meet the single-pair gates
against the CPU oracle and the reference's fixtures, and must agree with the single-pair dispatcher up to the
reordered dot-product sums of the per-pair PCG groups.

Every pair of a batch is distinct where the oracle judges it: a kernel that reads pair 0's planes, navigation or
heights for every pair cannot pass.  The cases reach every group size of the cooperative small-level solver
(k_pcg_coop_batch), batches that need several waves and end with a one-pair wave, pairs that stop at the build next
to pairs that reach the iteration cap, every navigation grid and the workspace state kept between calls."""
import numpy as np
import pytest

import cases
import octane_b200 as ob
from conftest import load_golden
from octane_b200 import synthetic as S

pytestmark = pytest.mark.gpu
KEYS_F = ("uPix", "vPix")
KEYS_S = ("uVal", "vVal", "uVal2", "vVal2", "CTP")
COOP_PER_SM = 2        # k_pcg_coop_batch: __launch_bounds__(256, 2), 2 co-resident blocks per SM


@pytest.fixture(scope="module")
def bctx():
    c = ob.Context(0)
    yield c
    c.close()


def tdev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


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


def distinct_inputs(npairs, nx, ny, seed0, nc=1):
    """npairs distinct nx x ny pairs (nc channels: seeds + 100 ch, as cases.variational_inputs), each with its own
    cloud-top heights and times, all on the 2 km mesoscale grid"""
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    img1, img2 = [], []
    for k in range(npairs):
        chans = [S.make_pair(nx, ny, seed0 + k + 100 * ch)[:2] for ch in range(nc)]
        img1.append(np.stack([a for a, _ in chans]) if nc > 1 else chans[0][0])
        img2.append(np.stack([b for _, b in chans]) if nc > 1 else chans[0][1])
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = np.stack([(7500.0 + 7400.0 * np.sin(xx / (30.0 + k) + k) * np.cos(yy / 30.0)).astype(np.float32)
                    for k in range(npairs)])
    t1 = [100.0 * k for k in range(npairs)]
    return (np.stack(img1).astype(np.float32), np.stack(img2).astype(np.float32), cth,
            [ob.goes_nav(xs, ys, xo, yo)] * npairs, t1, [t + dt for t in t1])


def check_vs_oracle(oracle, out, its, b, img1, img2, p_over, nc, tag, want=None):
    """pair b of a batch against its own oracle run (or `want`, a stored one) with the gates of
    test_flow_matches_oracle: mean |d| < 1e-4 px, max < 2e-3 px, equal iteration counts per solve"""
    uo, vo, its_o = want if want is not None else oracle.variational_flow(img1, img2, oracle.params(**p_over), None, None,
                                                                        nc=nc)
    du, dv = np.abs(out["uPix"][b] - uo), np.abs(out["vPix"][b] - vo)
    print(f"{tag} pair {b}: max |d u, v| vs the oracle = {max(du.max(), dv.max()):.3e} px, "
          f"oracle iterations {int(its_o.min())}..{int(its_o.max())}")
    assert du.mean() < 1e-4 and dv.mean() < 1e-4, (tag, b, du.mean(), dv.mean())
    assert du.max() < 2e-3 and dv.max() < 2e-3, (tag, b, du.max(), dv.max())
    bad = [s for s in range(len(its_o)) if its[b][s] != its_o[s]]
    assert not bad, f"{tag} pair {b}: iterations differ at solves {bad}: batch {list(its[b][bad])}, oracle {list(its_o[bad])}"
    return uo, vo, its_o


# ---- small-level solver geometry (mirror of pcg.cu coop_batch_blocks and ctx.cu run_levels_batch) ----------------
def coop_blocks(nx, rows):
    """blocks per pair of k_pcg_coop_batch: one per 8 warp tasks of 128 columns x 8 rows, clamped to 1..8"""
    g = ((nx + 127) // 128 * ((rows + 7) // 8) + 7) // 8
    return min(max(g, 1), 8)


def small_level(nx, rows):
    """a level the batched call solves in cooperative launches (the merged-reduction kernels need nx >= 512 and
    at least 64 rows); the others run the single-pair PCG kernels pair by pair"""
    return nx < 512 or rows < 64


def small_level_groups(oracle, nx, ny, p):
    return [coop_blocks(a, b) for a, b in oracle.level_dims(nx, ny, kiters=p.kiters, scaleF=p.scaleF) if small_level(a, b)]


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
# judged by the oracle alone (no reference fixture): three channels, and the stop after one or two iterations
# (k_pcg_coop_batch's XM_NONE-only and XM_INIT exits, k_update_uv with its = 1 and 2)
EXTRA_VAR_CASES = {
    "var_112x88_nc3": dict(nx=112, ny=88, seed=18, kind="vortex", nc=3),
    "var_96x80_shift_cg1": dict(cases.VARIATIONAL["var_96x80_shift"], params=dict(cgiters=1)),
    "var_96x80_shift_cg2": dict(cases.VARIATIONAL["var_96x80_shift"], params=dict(cgiters=2)),
}


@pytest.mark.parametrize("name", VAR_CASES + sorted(EXTRA_VAR_CASES))
def test_batch_matches_oracle_and_fixture(bctx, oracle, name):
    """four distinct pairs: pair 0 is the case's input, pairs 1-3 the case regenerated with seed + 1000 k; each meets
    the single-pair gates against its own oracle run, and pair 0 also against the reference fixture"""
    c = cases.VARIATIONAL.get(name) or EXTRA_VAR_CASES[name]
    nc = c.get("nc", 1)
    ins = [cases.variational_inputs(dict(c, seed=c["seed"] + 1000 * k))[:2] for k in range(4)]
    p = ob.default_params(**c.get("params", {}))
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    navs = [ob.goes_nav(xs, ys, xo, yo)] * 4
    out, _, its = run_batch(bctx, np.stack([a for a, _ in ins]), np.stack([b for _, b in ins]), navs, [0.0] * 4, [dt] * 4,
                            p, nc=nc)
    for b, (i1, i2) in enumerate(ins):
        check_vs_oracle(oracle, out, its, b, i1, i2, c.get("params", {}), nc, name)
    if name not in cases.VARIATIONAL:
        if "cgiters" in c.get("params", {}):                  # every solve stops at the cap
            assert (its == c["params"]["cgiters"]).all()
        return
    g = load_golden(name)
    du, dv = np.abs(out["uPix"][0] - g["u"]), np.abs(out["vPix"][0] - g["v"])
    assert du.mean() < 1e-3 and dv.mean() < 1e-3 and du.max() < 1e-2 and dv.max() < 1e-2
    assert max(du.max(), dv.max()) < max(20 * float(g["spread"].max()), 2e-4)


# (nx, ny): the small levels of these shapes use every group size 1..8 of k_pcg_coop_batch
GROUP_SHAPES = [(120, 160), (200, 192), (256, 224), (264, 240), (300, 104)]


def test_batch_shapes_cover_every_group_size(oracle):
    p = ob.default_params()
    per_shape = {s: small_level_groups(oracle, *s, p) for s in GROUP_SHAPES}
    covered = sorted(set().union(*per_shape.values()))
    print(f"group sizes per shape (coarsest first): {per_shape}; covered {covered}")
    assert covered == list(range(1, 9))
    assert any(nx % 128 == 0 for nx, _ in GROUP_SHAPES) and any(nx % 128 for nx, _ in GROUP_SHAPES)


@pytest.mark.parametrize("shape", GROUP_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_batch_group_sizes_match_oracle(bctx, oracle, shape):
    """three distinct pairs per shape, each against its own oracle run"""
    nx, ny = shape
    p = ob.default_params()
    img1, img2, _, navs, t1, t2 = distinct_inputs(3, nx, ny, seed0=400 + nx)
    out, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p)
    tag = f"{nx}x{ny} G={small_level_groups(oracle, nx, ny, p)}"
    for b in range(3):
        check_vs_oracle(oracle, out, its, b, img1[b], img2[b], {}, 1, tag)


def test_batch_waves_and_mixed_exits(bctx, oracle):
    """2 floor(2 sm / 8) + 1 distinct 264x240 pairs: the finest level (8 blocks per pair) runs in three waves and
    132x120 (4 blocks) in two, each ending with a one-pair wave.  Pairs with img1 == img2 (zero rhs: no iteration in
    any solve) sit at index 0, at both sides of the first wave boundary and alone in the last wave; the others mostly
    reach the 30-iteration cap"""
    nx, ny = 264, 240
    p = ob.default_params()
    sms = sm_count()
    per8 = sms * COOP_PER_SM // 8
    B = 2 * per8 + 1
    groups = small_level_groups(oracle, nx, ny, p)
    assert groups[-1] == 8 and B % per8 == 1 and B % (sms * COOP_PER_SM // 4) == 1 and 4 in groups
    img1, img2, _, navs, t1, t2 = distinct_inputs(B, nx, ny, seed0=500)
    still = [0, per8 - 1, per8, B - 1]
    for b in still:
        img2[b] = img1[b]
    run_batch(bctx, img1[1:2], img2[1:2], navs[:1], t1[:1], t2[:1], p)
    one = bctx.stats().kernel_launches
    out, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p)
    many = bctx.stats().kernel_launches
    want = sum(3 * p.liters * (-(-B // max(1, sms * COOP_PER_SM // g)) - 1) for g in groups)
    print(f"{B} pairs of {nx}x{ny} on {sms} SMs: group sizes {groups}, kernel launches 1 pair {one}, "
          f"{B} pairs {many}, delta {many - one} (expected {want})")
    assert many - one == want
    capped = 0
    for b in range(B):
        uo, vo, its_o = check_vs_oracle(oracle, out, its, b, img1[b], img2[b], {}, 1, f"waves {nx}x{ny}")
        if b in still:
            assert its_o.max() == 0 and not uo.any() and not vo.any()
            assert not out["uPix"][b].any() and not out["vPix"][b].any()
        capped += int((its_o == p.cgiters).any())
    assert capped > 0


@pytest.fixture(scope="module")
def large_pairs(oracle):
    img1, img2, _, navs, t1, t2 = distinct_inputs(3, 768, 640, seed0=600)
    want = [oracle.variational_flow(img1[b], img2[b], oracle.params()) for b in range(3)]
    return img1, img2, navs, t1, t2, want


@pytest.mark.parametrize("solver", [1, 0])
def test_batch_large_levels_match_oracle(oracle, large_pairs, solver):
    """three distinct 768x640 pairs: the finest level runs the single-pair PCG kernels pair by pair, the coarser ones
    the cooperative solver with 2, 5 and 8 blocks per pair"""
    img1, img2, navs, t1, t2, want = large_pairs
    p = ob.default_params()
    assert small_level_groups(oracle, 768, 640, p) == [2, 5, 8]
    ctx = ob.Context(0)
    try:
        ctx.set_solver(solver)
        out, _, its = run_batch(ctx, img1, img2, navs, t1, t2, p)
        for b in range(3):
            check_vs_oracle(oracle, out, its, b, img1[b], img2[b], {}, 1, f"768x640 solver {solver}", want=want[b])
    finally:
        ctx.close()


def ctp_model(cth, ir):
    """the reference's host packing of CTP (src/oct_optical_flow.cc:71-88): float arithmetic, conversion to int
    (truncation), then to short (16-bit wrap)"""
    f = np.float32
    x = (cth.astype(f) - f(300)) * f(100) if ir else cth.astype(f)
    return x.astype(np.int32).astype(np.int16)


def grid_batch(grid):
    """(navs, t1, t2, moved pairs, flags) of four pairs on one navigation grid, each with its own times"""
    if grid in ("goes", "pixuv"):
        cs = [cases.NAVIGATION[n] for n in ("nav_goes_meso", "nav_goes_limb", "nav_goes_2km_offset", "nav_moved")]
        named = [cases.nav_constants(c) for c in cs]
    elif grid == "polar":
        named = [cases.nav_constants(cases.NAVIGATION[n]) for n in ("nav_polar", "nav_polar_pole")] * 2
    else:
        kw, extra, t1, t2, flags = cases.nav_constants(cases.NAVIGATION["nav_merc"])
        kw2 = dict(kw, xOffset=kw["xOffset"] + 84000.0, yOffset=kw["yOffset"] - 1500000.0)
        named = [(kw, extra, t1, t2, flags), (kw2, extra, t1, t2, flags)] * 2
    navs, t1s, t2s = [], [], []
    for b, (kw, extra, t1, t2, _) in enumerate(named):
        nav = ob.goes_nav(**kw)
        for k, val in extra.items():
            setattr(nav, k, val)
        navs.append(nav)
        t1s.append(t1 + 37.0 * b)
        t2s.append(t1 + 37.0 * b + (t2 - t1) * (1.0 + 0.5 * b))
    flags = dict(pixuv=int(grid == "pixuv"), dopolar=int(grid == "polar"), domerc=int(grid == "merc"))
    moved = [b for b, (kw, *_) in enumerate(named) if "g2xOffset" in kw]
    return navs, t1s, t2s, moved, flags


@pytest.mark.parametrize("ir", [0, 1])
@pytest.mark.parametrize("grid", ["goes", "polar", "merc", "pixuv"])
def test_batch_navigation_and_ctp_per_pair(bctx, grid, ir):
    """every pair navigates with its own nav and times: its four short planes are, bit for bit, what the single-pair
    navigation gives on the batch's own flow; CTP packs each pair's own heights as the reference's host code does"""
    nx, ny = 120, 90
    navs, t1, t2, want_moved, flags = grid_batch(grid)
    B = len(navs)
    img1, img2, cth, _, _, _ = distinct_inputs(B, nx, ny, seed0=700)
    cth[:, 0, :12] = [-50.0, 0.0, 299.99, 300.0, 627.6, 627.7, 655.35, 12000.5, 19999.9, 32767.0, 32768.9, 65535.5]
    cth[:, 1, :3] = [-32768.0, -32769.5, 40000.7]
    p = ob.default_params(doCTH=1, ir=ir, **flags)
    out, moved, _ = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
    assert moved == want_moved
    import torch
    for b in range(B):
        ref = [torch.full((ny, nx), 7, dtype=torch.int16, device="cuda") for _ in range(4)]
        _, mv = bctx.oct_pix2uv_cuda(navs[b], t1[b], t2[b], tdev(out["uPix"][b]), tdev(out["vPix"][b]), *ref, p)
        assert mv == (b in want_moved)
        for k, r in zip(("uVal", "vVal", "uVal2", "vVal2"), ref):
            assert np.array_equal(out[k][b], r.cpu().numpy()), (grid, b, k)
        assert np.array_equal(out["CTP"][b], ctp_model(cth[b], ir)), (grid, ir, b)
    # (the limb sector lies wholly beyond the limb cut: its speeds are zero)
    assert sum(bool(out["uVal"][b].any() and out["vVal"][b].any()) for b in range(B) if b not in want_moved) >= 2


def test_batch_state_across_calls():
    """batches and single-pair calls of several sizes on one context (re-plans, a workspace that grows and drops the
    captured PCG graphs, batch buffers sized by an earlier call) give what a fresh context gives, bit for bit"""
    p = ob.default_params(doCTH=1)
    batches = [distinct_inputs(16, 264, 240, seed0=800), distinct_inputs(5, 200, 192, seed0=820, nc=2),
               distinct_inputs(40, 264, 240, seed0=840)]
    ncs = [1, 2, 1]
    i1, i2, cth, navs, t1, t2 = distinct_inputs(1, 768, 640, seed0=900)

    def batch(ctx, k):
        img1, img2, bcth, bnavs, bt1, bt2 = batches[k]
        return run_batch(ctx, img1, img2, bnavs, bt1, bt2, p, bcth, nc=ncs[k])

    def one(ctx):
        return single(ctx, i1[0], i2[0], navs[0], t1[0], t2[0], p, cth[0])

    ctx = ob.Context(0)
    try:
        got = [batch(ctx, 0), one(ctx), batch(ctx, 1), batch(ctx, 2), one(ctx)]
    finally:
        ctx.close()
    for k, pos in ((0, 0), (1, 2), (2, 3)):
        fresh = ob.Context(0)
        try:
            want = batch(fresh, k)
        finally:
            fresh.close()
        for key in want[0]:
            assert np.array_equal(got[pos][0][key], want[0][key]), (k, key)
        assert got[pos][1] == want[1] and np.array_equal(got[pos][2], want[2]), k
    for key in got[1]:
        assert np.array_equal(got[4][key], got[1][key]), key


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
