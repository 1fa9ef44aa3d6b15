"""Batched dispatcher with a first guess and -srsal (octane_optical_flow_batch_ex_dev).

Per pair, the call must do what octane_optical_flow_dev does with the same flags: the first guess initialises the
coarsest level and, where lambda_c != 0, enters the coefficients as a hint; -srsal smooths uPix / vPix with the pair's
own heights after the CTP pack and the navigation.  Every pair of a batch is distinct where a check judges it: its
images, its first guess (cases.variational_inputs builds one u0 per shape, so it is scaled and shifted by the pair
index), its heights and its times.  A kernel that reads pair 0's hint or heights for every pair cannot pass."""
import numpy as np
import pytest

import cases
import octane_b200 as ob
from conftest import load_golden
from octane_b200 import synthetic as S
from test_gpu_batch import (COOP_PER_SM, KEYS_F, KEYS_S, check_vs_oracle, check_vs_single, distinct_inputs, meso_inputs,
                            run_batch, sm_count, tdev)

pytestmark = pytest.mark.gpu
KEYS_NAV = ("uVal", "vVal", "uVal2", "vVal2")


@pytest.fixture(scope="module")
def bctx():
    c = ob.Context(0)
    yield c
    c.close()


def outputs(B, ny, nx, p):
    import torch
    out = {k: torch.zeros((B, ny, nx), device="cuda") for k in KEYS_F}
    for k in KEYS_S:
        if k != "CTP" or p.doCTH:
            out[k] = torch.zeros((B, ny, nx), dtype=torch.int16, device="cuda")
    return out


def run_ex(ctx, img1, img2, navs, t1, t2, p, cth=None, nc=1, fg=None, alias=False):
    """img1 / img2: numpy [B, (nc,) ny, nx]; fg: (fu, fv) numpy [B, ny, nx] or None.  alias: pass the first guess in
    the uPix / vPix tensors themselves.  Returns (dict of numpy [B, ny, nx], moved, its [B, n_solves])"""
    B = img1.shape[0]
    ny, nx = img1.shape[-2:]
    out = outputs(B, ny, nx, p)
    kw = {}
    if fg is not None:
        if alias:
            out["uPix"].copy_(tdev(fg[0]))
            out["vPix"].copy_(tdev(fg[1]))
            kw = dict(fg_u=out["uPix"], fg_v=out["vPix"])
        else:
            kw = dict(fg_u=tdev(fg[0]), fg_v=tdev(fg[1]))
    moved = ctx.oct_optical_flow_batch_ex_dev(tdev(img1), tdev(img2), navs, t1, t2, p, out,
                                              cth=None if cth is None else tdev(cth), nc=nc, **kw)
    its = ctx.batch_cg_iterations(B, p.kiters * 3 * p.liters)
    return {k: v.cpu().numpy() for k, v in out.items()}, moved, its


def first_guesses(npairs, nx, ny):
    """pair k: the first guess of cases.variational_inputs scaled and shifted by a = k / (npairs - 1) (pair 0 is the
    case's own).  The span is the same for every batch size and keeps the guesses within 3 px, near the scenes' own
    motion: the max |d| against the oracle grows with the size of the guess (to about 0.05 px for 16 px guesses on
    264x240), and check_vs_oracle's gates are for guesses of a few pixels."""
    _, _, u0, v0 = cases.variational_inputs(dict(nx=nx, ny=ny, seed=0, kind="vortex", first_guess=True))
    a = [k / max(npairs - 1, 1) for k in range(npairs)]
    fu = np.stack([u0 * (1.0 + 1.5 * x) + 0.6 * x for x in a]).astype(np.float32)
    fv = np.stack([v0 * (1.0 - 1.2 * x) - 0.3 * x for x in a]).astype(np.float32)
    return fu, fv


def meso_navs(npairs):
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    return [ob.goes_nav(xs, ys, xo, yo)] * npairs, [0.0] * npairs, [dt] * npairs


def same(a, b, tag):
    for k in a:
        assert np.array_equal(a[k], b[k]), (tag, k)


def test_ex_without_flags_is_batch_dev(bctx):
    """the shared body: neither flag gives octane_optical_flow_batch_dev's bits and iteration counts"""
    img1, img2, cth, navs, t1, t2 = distinct_inputs(8, 200, 200, seed0=1100)
    p = ob.default_params(doCTH=1)
    want, moved_w, its_w = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
    got, moved, its = run_ex(bctx, img1, img2, navs, t1, t2, p, cth)
    same(got, want, "no flags")
    assert moved == moved_w and np.array_equal(its, its_w)


FG_CASES = {
    "var_160x120_fg": {},
    "lambdac0": dict(params=dict(lambdac=0.0)),                 # the guess only initialises the coarsest level
    "kiters1": dict(params=dict(lambdac=0.5, kiters=1)),       # the finest level is the first: the hint is uh itself
    "nc2": dict(nc=2),
}


@pytest.mark.parametrize("name", sorted(FG_CASES))
def test_ex_first_guess_matches_oracle_and_fixture(bctx, oracle, name):
    """four distinct pairs with their own first guesses, each against its own oracle run; pair 0 of the base case
    is the fixture's input and also meets test_batch_matches_oracle_and_fixture's gates against the fixture"""
    c = dict(cases.VARIATIONAL["var_160x120_fg"], **FG_CASES[name])
    nc = c.get("nc", 1)
    ins = [cases.variational_inputs(dict(c, seed=c["seed"] + 1000 * k))[:2] for k in range(4)]
    fu, fv = first_guesses(4, c["nx"], c["ny"])
    assert np.array_equal(fu[0], cases.variational_inputs(c)[2])
    p = ob.default_params(first_guess=1, **c["params"])
    navs, t1, t2 = meso_navs(4)
    out, _, its = run_ex(bctx, np.stack([a for a, _ in ins]), np.stack([b for _, b in ins]), navs, t1, t2, p, nc=nc,
                         fg=(fu, fv))
    for b, (i1, i2) in enumerate(ins):
        want = oracle.variational_flow(i1, i2, oracle.params(**c["params"]), fu[b], fv[b], nc=nc)
        check_vs_oracle(oracle, out, its, b, i1, i2, c["params"], nc, f"{name} fg", want=want)
    if name != "var_160x120_fg":
        return
    g = load_golden(name)
    du, dv = np.abs(out["uPix"][0] - g["u"]), np.abs(out["vPix"][0] - g["v"])
    assert du.mean() < 1e-3 and dv.mean() < 1e-3 and du.max() < 1e-2 and dv.max() < 1e-2
    assert max(du.max(), dv.max()) < max(20 * float(g["spread"].max()), 2e-4)


def test_ex_first_guess_waves(bctx, oracle):
    """2 floor(2 sm / 8) + 1 distinct 264x240 pairs with their own first guesses and lambda_c > 0: the finest level
    runs in three waves of the cooperative solver, the last with one pair"""
    nx, ny = 264, 240
    per8 = sm_count() * COOP_PER_SM // 8
    B = 2 * per8 + 1
    img1, img2, _, navs, t1, t2 = distinct_inputs(B, nx, ny, seed0=1200)
    fu, fv = first_guesses(B, nx, ny)
    over = dict(lambdac=0.5)
    p = ob.default_params(first_guess=1, **over)
    out, _, its = run_ex(bctx, img1, img2, navs, t1, t2, p, fg=(fu, fv))
    for b in range(B):
        want = oracle.variational_flow(img1[b], img2[b], oracle.params(**over), fu[b], fv[b])
        check_vs_oracle(oracle, out, its, b, img1[b], img2[b], over, 1, f"fg waves {nx}x{ny}", want=want)


def single(ctx, a, b, nav, t1, t2, p, cth=None, fg=None):
    """octane_optical_flow_dev on one pair; fg: (fu, fv) seeds uPix / vPix (its in/out convention)"""
    import torch
    ny, nx = a.shape[-2:]
    u = tdev(fg[0]) if fg is not None else torch.zeros((ny, nx), device="cuda")
    v = tdev(fg[1]) if fg is not None else torch.zeros((ny, nx), device="cuda")
    s = [torch.zeros((ny, nx), dtype=torch.int16, device="cuda") for _ in range(5)]
    ctx.oct_optical_flow_dev(tdev(a), tdev(b), nav, t1, t2, p, u, v, *s[:4], cth=None if cth is None else tdev(cth),
                             ctp=s[4] if p.doCTH else None)
    ctx.synchronize()
    r = dict(uPix=u.cpu().numpy(), vPix=v.cpu().numpy())
    r.update({k: x.cpu().numpy() for k, x in zip(KEYS_S, s) if k != "CTP" or p.doCTH})
    return r


@pytest.mark.parametrize("solver", [1, 0])
def test_ex_first_guess_large_levels(solver):
    """768x640 pairs with first guesses: the finest level runs the single-pair PCG kernels pair by pair; against the
    single-pair dispatcher with first_guess = 1"""
    ctx = ob.Context(0)
    try:
        ctx.set_solver(solver)
        img1, img2, cth, navs, t1, t2 = distinct_inputs(3, 768, 640, seed0=1300)
        fu, fv = first_guesses(3, 768, 640)
        p = ob.default_params(first_guess=1, lambdac=0.5, doCTH=1)
        out, _, _ = run_ex(ctx, img1, img2, navs, t1, t2, p, cth, fg=(fu, fv))
        for b in range(3):
            want = single(ctx, img1[b], img2[b], navs[b], t1[b], t2[b], p, cth[b], fg=(fu[b], fv[b]))
            check_vs_single(out, b, want, f"768x640 fg solver {solver}")
    finally:
        ctx.close()


def test_ex_first_guess_may_alias_outputs_and_is_only_read(bctx):
    """the first guess passed in uPix / vPix gives the bits of separate buffers, and separate buffers come back
    unchanged"""
    import torch
    img1, img2, cth, navs, t1, t2 = distinct_inputs(4, 160, 120, seed0=1400)
    fu, fv = first_guesses(4, 160, 120)
    p = ob.default_params(first_guess=1, lambdac=0.5, doCTH=1, dosrsal=1)
    out = outputs(4, 120, 160, p)
    gu, gv = tdev(fu), tdev(fv)
    bctx.oct_optical_flow_batch_ex_dev(tdev(img1), tdev(img2), navs, t1, t2, p, out, cth=tdev(cth), fg_u=gu, fg_v=gv)
    torch.cuda.synchronize()
    assert np.array_equal(gu.cpu().numpy(), fu) and np.array_equal(gv.cpu().numpy(), fv)
    sep = {k: v.cpu().numpy() for k, v in out.items()}
    ali, _, _ = run_ex(bctx, img1, img2, navs, t1, t2, p, cth, fg=(fu, fv), alias=True)
    same(ali, sep, "alias")
    assert not np.array_equal(sep["uPix"][0], sep["uPix"][1])


def moved_navs(npairs, moved):
    navs, t1, t2 = [], [], []
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    for b in range(npairs):
        nav = ob.goes_nav(xs, ys, xo, yo)
        if b in moved:
            nav.g2xOffset = nav.xOffset + 0.001
        navs.append(nav)
        t1.append(60.0 * b)
        t2.append(60.0 * b + dt * (1.0 + 0.25 * b))
    return navs, t1, t2


def check_srsal_per_pair(ctx, img1, img2, cth, navs, t1, t2, p_over, moved, nc=1):
    """-srsal off and on, on the same inputs: the short planes and CTP are equal; each pair's uPix / vPix is
    octane_srsal_dev applied with its own heights to its unsmoothed output; moved pairs are smoothed too"""
    import torch
    B = img1.shape[0]
    raw, mv0, its0 = run_ex(ctx, img1, img2, navs, t1, t2, ob.default_params(dosrsal=0, **p_over), cth, nc=nc)
    smo, mv1, its1 = run_ex(ctx, img1, img2, navs, t1, t2, ob.default_params(dosrsal=1, **p_over), cth, nc=nc)
    assert mv0 == mv1 == moved
    assert np.array_equal(its0, its1)
    for k in KEYS_NAV + (("CTP",) if p_over.get("doCTH") else ()):
        assert np.array_equal(raw[k], smo[k]), k
    for b in range(B):
        u, v = tdev(raw["uPix"][b]), tdev(raw["vPix"][b])
        ctx.oct_srsal_cu(u, v, tdev(cth[b]))
        torch.cuda.synchronize()
        assert np.array_equal(smo["uPix"][b], u.cpu().numpy()), b
        assert np.array_equal(smo["vPix"][b], v.cpu().numpy()), b
        assert not np.array_equal(smo["uPix"][b], raw["uPix"][b]), b
        if b in moved:
            assert all(not smo[k][b].any() for k in KEYS_NAV), b
    # the pairs' heights differ, so the smoothing of one pair with another's heights is visible
    u, v = tdev(raw["uPix"][1]), tdev(raw["vPix"][1])
    ctx.oct_srsal_cu(u, v, tdev(cth[0]))
    assert not np.array_equal(smo["uPix"][1], u.cpu().numpy())


@pytest.mark.parametrize("doCTH", [0, 1])
def test_ex_srsal_per_pair(bctx, doCTH):
    """200x150 (partial 32 x 8 tiles in both directions), four pairs with their own heights and times, pair 2's
    sector moved"""
    img1, img2, cth, _, _, _ = distinct_inputs(4, 200, 150, seed0=1500)
    navs, t1, t2 = moved_navs(4, [2])
    check_srsal_per_pair(bctx, img1, img2, cth, navs, t1, t2, dict(doCTH=doCTH), [2])


def test_ex_srsal_at_the_edges(bctx):
    """96x24: every window reflects at the top and the bottom of the scene; a scene 18 pixels wide or high is refused"""
    img1, img2, cth, _, _, _ = distinct_inputs(3, 96, 24, seed0=1600)
    navs, t1, t2 = moved_navs(3, [])
    check_srsal_per_pair(bctx, img1, img2, cth, navs, t1, t2, dict(doCTH=1, kiters=2), [])
    p = ob.default_params(dosrsal=1, kiters=2)
    for nx, ny in ((18, 40), (40, 18)):
        i1, i2, c, _, _, _ = distinct_inputs(2, nx, ny, seed0=1610)
        nv, a, b = moved_navs(2, [])
        with pytest.raises(ob.OctaneError) as e:
            run_ex(bctx, i1, i2, nv, a, b, p, c)
        assert e.value.code == -2


def fg_srsal_inputs(npairs, nx, ny, seed0):
    img1, img2, cth, _, _, _ = distinct_inputs(npairs, nx, ny, seed0=seed0)
    navs, t1, t2 = moved_navs(npairs, [3] if npairs > 3 else [])
    return img1, img2, cth, navs, t1, t2, first_guesses(npairs, nx, ny)


FG_SRSAL = dict(first_guess=1, lambdac=0.5, dosrsal=1, doCTH=1)


def test_ex_invariance(bctx):
    """24 pairs with first guess, lambda_c, -srsal and CTH: whole, shuffled and in ragged sub-batches, the same bits
    and iteration counts per pair"""
    img1, img2, cth, navs, t1, t2, (fu, fv) = fg_srsal_inputs(24, 200, 150, 1700)
    p = ob.default_params(**FG_SRSAL)
    full, moved, its = run_ex(bctx, img1, img2, navs, t1, t2, p, cth, fg=(fu, fv))
    assert moved == [3]
    perm = np.random.default_rng(7).permutation(24)
    shuf, _, its_s = run_ex(bctx, img1[perm], img2[perm], [navs[i] for i in perm], [t1[i] for i in perm],
                            [t2[i] for i in perm], p, cth[perm], fg=(fu[perm], fv[perm]))
    for k in full:
        assert np.array_equal(shuf[k], full[k][perm]), k
    assert np.array_equal(its_s, its[perm])
    b0 = 0
    for n in (1, 5, 18):
        s = slice(b0, b0 + n)
        part, _, its_p = run_ex(bctx, img1[s], img2[s], navs[s], t1[s], t2[s], p, cth[s], fg=(fu[s], fv[s]))
        for k in full:
            assert np.array_equal(part[k], full[k][s]), (k, n)
        assert np.array_equal(its_p, its[s])
        b0 += n


def test_ex_launch_count_does_not_grow_with_pairs(bctx):
    """with first guess and -srsal, 16 pairs of 500^2 take as many kernel launches as one pair"""
    img1, img2, cth, navs, t1, t2 = meso_inputs(16)
    fu, fv = first_guesses(16, 500, 500)
    p = ob.default_params(**FG_SRSAL)
    run_ex(bctx, img1[:1], img2[:1], navs[:1], t1[:1], t2[:1], p, cth[:1], fg=(fu[:1], fv[:1]))
    one = bctx.stats().kernel_launches
    run_ex(bctx, img1, img2, navs, t1, t2, p, cth, fg=(fu, fv))
    sixteen = bctx.stats().kernel_launches
    run_ex(bctx, img1, img2, navs, t1, t2, ob.default_params(doCTH=1), cth)
    plain = bctx.stats().kernel_launches
    print(f"kernel launches with first guess and -srsal: 1 pair {one}, 16 pairs {sixteen}; without: {plain}")
    assert one > 0 and sixteen == one and one > plain


def test_ex_state_across_calls():
    """a plain batch, an fg + srsal batch, a single-pair call, a plain batch of another pair count and the fg batch
    again, on one context (re-plans whose pair stride grows and shrinks): each call equals a fresh context's"""
    plain16 = distinct_inputs(16, 264, 240, seed0=1800)
    plain40 = distinct_inputs(40, 264, 240, seed0=1840)
    fgb = fg_srsal_inputs(12, 264, 240, 1820)
    i1, i2, c1, n1, a1, b1 = distinct_inputs(1, 768, 640, seed0=1900)
    plain, fgp = ob.default_params(doCTH=1), ob.default_params(**FG_SRSAL)

    def call(ctx, k):
        if k == "plain16":
            return run_ex(ctx, *plain16[:2], *plain16[3:], plain, plain16[2])
        if k == "plain40":
            return run_ex(ctx, *plain40[:2], *plain40[3:], plain, plain40[2])
        if k == "fg":
            img1, img2, cth, navs, t1, t2, fg = fgb
            return run_ex(ctx, img1, img2, navs, t1, t2, fgp, cth, fg=fg)
        fg = first_guesses(1, 768, 640)
        return single(ctx, i1[0], i2[0], n1[0], a1[0], b1[0], fgp, c1[0], fg=(fg[0][0], fg[1][0]))

    order = ["plain16", "fg", "single", "plain40", "fg"]
    ctx = ob.Context(0)
    try:
        got = [call(ctx, k) for k in order]
    finally:
        ctx.close()
    for pos, k in enumerate(order):
        fresh = ob.Context(0)
        try:
            want = call(fresh, k)
        finally:
            fresh.close()
        if k == "single":
            same(got[pos], want, k)
            continue
        same(got[pos][0], want[0], (pos, k))
        assert got[pos][1] == want[1] and np.array_equal(got[pos][2], want[2]), (pos, k)


def test_ex_refusals_leave_context_usable(bctx):
    """each refusal is OCTANE_EINVAL, and a valid first guess + -srsal call then returns the bits it returned before"""
    img1, img2, cth, navs, t1, t2, (fu, fv) = fg_srsal_inputs(2, 200, 200, 2000)
    p = ob.default_params(**FG_SRSAL)
    want, _, its_want = run_ex(bctx, img1, img2, navs, t1, t2, p, cth, fg=(fu, fv))

    def refused(fn):
        with pytest.raises(ob.OctaneError) as e:
            fn()
        assert e.value.code == -2                          # OCTANE_EINVAL
        got, _, its = run_ex(bctx, img1, img2, navs, t1, t2, p, cth, fg=(fu, fv))
        same(got, want, "after a refusal")
        assert np.array_equal(its, its_want)

    def raw(p, cth=cth, fg_u=None, fg_v=None, ctp=True, img=(img1, img2)):
        out = outputs(img[0].shape[0], *img[0].shape[-2:], p)
        if not ctp:
            out.pop("CTP", None)
        return bctx.oct_optical_flow_batch_ex_dev(tdev(img[0]), tdev(img[1]), navs[:len(img[0])], t1[:len(img[0])],
                                                  t2[:len(img[0])], p, out, cth=None if cth is None else tdev(cth),
                                                  fg_u=fg_u, fg_v=fg_v)

    refused(lambda: run_ex(bctx, img1[:0], img2[:0], [], [], [], p, cth[:0], fg=(fu[:0], fv[:0])))     # npairs 0
    refused(lambda: raw(p))                                                                       # no first guess
    refused(lambda: raw(p, fg_u=tdev(fu)))                                                         # one plane only
    refused(lambda: raw(ob.default_params(dosrsal=1), cth=None))                                  # -srsal, no heights
    small = distinct_inputs(2, 200, 18, seed0=2010)
    refused(lambda: raw(ob.default_params(dosrsal=1), cth=small[2], img=small[:2]))               # 18 rows
    refused(lambda: raw(ob.default_params(doCTH=1), cth=None))                                    # doCTH, no cth
    refused(lambda: raw(ob.default_params(doCTH=1), ctp=False))                                   # doCTH, no ctp
