"""Batched dispatcher on large levels (nx >= 512, >= 64 rows) under the merged-reduction solver.

There one k_pcg_fused launch per iteration serves every pair of the batch: each pair runs on the grid and tiling it
would get alone, with its own scalars, partial sums, ticket and stop rule, and the loop is replayed from a CUDA graph
captured for the call's number of pairs.  A pair's bits must therefore be those of the same pair solved alone, in any
order and next to any other pairs; pairs that stop at different iterations must share one launch; the launch count
must not grow with the pairs; and the captured graphs must follow npairs, re-plans and a workspace that grows.
768x640 has one large level (the finest), 1024x1024 two."""
import numpy as np
import pytest

import octane_b200 as ob
from test_gpu_batch import check_vs_oracle, distinct_inputs, run_batch, single
from test_gpu_batch_fg_srsal import FG_SRSAL, first_guesses, run_ex

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bctx():
    c = ob.Context(0)
    yield c
    c.close()


def alone(ctx, img1, img2, navs, t1, t2, p, cth, b, runner=run_batch, fg=None):
    """pair b solved in a batch of one"""
    s = slice(b, b + 1)
    kw = {} if fg is None else dict(fg=(fg[0][s], fg[1][s]))
    return runner(ctx, img1[s], img2[s], navs[s], t1[s], t2[s], p, cth[s], **kw)


def assert_pair_is(got, its, b, want, its_want, tag):
    for k in want[0]:
        assert np.array_equal(got[k][b], want[0][k][0]), (tag, b, k)
    assert np.array_equal(its[b], its_want[0]), (tag, b)


@pytest.mark.parametrize("nx,ny,B", [(768, 640, 5), (768, 640, 9), (1024, 1024, 5), (1024, 1024, 10)])
def test_large_batch_pairs_are_independent(bctx, nx, ny, B):
    """every pair of a batch (and of the same batch shuffled) is, bit for bit, the pair solved alone: uPix, vPix, the
    four navigated short planes, CTP and the iteration count of every solve"""
    img1, img2, cth, navs, t1, t2 = distinct_inputs(B, nx, ny, seed0=3000 + nx)
    p = ob.default_params(doCTH=1)
    out, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
    for b in range(B):
        want, _, its_w = alone(bctx, img1, img2, navs, t1, t2, p, cth, b)
        assert_pair_is(out, its, b, (want,), its_w, f"{nx}x{ny} B={B}")
    perm = np.random.default_rng(B).permutation(B)
    shuf, _, its_s = run_batch(bctx, img1[perm], img2[perm], [navs[i] for i in perm], [t1[i] for i in perm],
                               [t2[i] for i in perm], p, cth[perm])
    for k in out:
        assert np.array_equal(shuf[k], out[k][perm]), k
    assert np.array_equal(its_s, its[perm])


@pytest.mark.parametrize("cgiters", [1, 2, 3, 30])
def test_large_batch_mixed_exits_match_oracle(bctx, oracle, cgiters):
    """one call with a pair whose images are identical (zero right-hand side: done after the build) and ordinary
    pairs that run to the cap; cgiters 1, 2, 3 and 30 end each solve on each launch mode of k_pcg_fused (the first
    iteration, the one that starts x, an even and an odd one).  Each pair meets its own oracle run"""
    nx, ny = 768, 640
    img1, img2, _, navs, t1, t2 = distinct_inputs(3, nx, ny, seed0=3100)
    img2[1] = img1[1]
    p_over = dict(cgiters=cgiters)
    p = ob.default_params(**p_over)
    out, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p)
    capped = 0
    for b in range(3):
        uo, vo, its_o = check_vs_oracle(oracle, out, its, b, img1[b], img2[b], p_over, 1, f"cgiters={cgiters}")
        if b == 1:
            assert its_o.max() == 0 and not out["uPix"][b].any() and not out["vPix"][b].any()
        else:
            capped += int((its_o == cgiters).any())
    assert capped == 2


@pytest.mark.parametrize("nx,ny", [(768, 640), (1024, 1024)])
def test_large_batch_launch_count_does_not_grow_with_pairs(nx, ny):
    """solver 1: 8 pairs take as many kernel launches as one; solver 0 (the two-pass kernels, still pair by pair on
    large levels) is only reported"""
    img1, img2, cth, navs, t1, t2 = distinct_inputs(8, nx, ny, seed0=3200)
    p = ob.default_params(doCTH=1)
    counts = {}
    for solver in (1, 0):
        ctx = ob.Context(0)
        try:
            ctx.set_solver(solver)
            run_batch(ctx, img1[:1], img2[:1], navs[:1], t1[:1], t2[:1], p, cth[:1])
            one = ctx.stats().kernel_launches
            run_batch(ctx, img1, img2, navs, t1, t2, p, cth)
            counts[solver] = (one, ctx.stats().kernel_launches)
        finally:
            ctx.close()
    print(f"{nx}x{ny} kernel launches (1 pair, 8 pairs): solver 1 {counts[1]}, solver 0 {counts[0]}")
    assert counts[1][0] > 0 and counts[1][0] == counts[1][1]


def test_large_batch_graphs_follow_npairs_replans_and_workspace():
    """one context: npairs 3, 5, 3, a single-pair call, npairs 3 at another size (re-plan), npairs 12 (the workspace
    grows), then 14 pairs of the first size (re-plan; the per-pair scalars, partials and tickets grow, the workspace
    does not) and a single-pair call; every result is what a fresh context gives, bit for bit, with graphs and again
    with profiling on"""
    p = ob.default_params(doCTH=1)
    a = distinct_inputs(14, 768, 640, seed0=3300)
    b = distinct_inputs(12, 1024, 1024, seed0=3400)
    calls = [("batch", a, 3), ("batch", a, 5), ("batch", a, 3), ("single", a, 1), ("batch", b, 3), ("batch", b, 12),
             ("batch", a, 14), ("single", a, 1)]

    def run(ctx, call):
        kind, (img1, img2, cth, navs, t1, t2), n = call
        if kind == "single":
            r = single(ctx, img1[0], img2[0], navs[0], t1[0], t2[0], p, cth[0])
            return r, None
        out, _, its = run_batch(ctx, img1[:n], img2[:n], navs[:n], t1[:n], t2[:n], p, cth[:n])
        return out, its

    fresh = []
    for call in calls:
        ctx = ob.Context(0)
        try:
            fresh.append(run(ctx, call))
        finally:
            ctx.close()
    for profile in (False, True):
        ctx = ob.Context(0)
        try:
            ctx.set_profile(profile)
            got = [run(ctx, call) for call in calls]
        finally:
            ctx.close()
        for i, ((out, its), (want, its_w)) in enumerate(zip(got, fresh)):
            for k in want:
                assert np.array_equal(out[k], want[k]), (profile, i, k)
            if its_w is not None:
                assert np.array_equal(its, its_w), (profile, i)


def test_large_batch_ex_first_guess_and_srsal(bctx):
    """first guess (lambda_c = 0.5) and -srsal at 768x640: each pair is its batch of one, bit for bit"""
    nx, ny, B = 768, 640, 4
    img1, img2, cth, navs, t1, t2 = distinct_inputs(B, nx, ny, seed0=3500)
    fg = first_guesses(B, nx, ny)
    p = ob.default_params(**FG_SRSAL)
    out, _, its = run_ex(bctx, img1, img2, navs, t1, t2, p, cth, fg=fg)
    for b in range(B):
        want, _, its_w = alone(bctx, img1, img2, navs, t1, t2, p, cth, b, runner=run_ex, fg=fg)
        assert_pair_is(out, its, b, (want,), its_w, "ex")


def test_large_batch_refusal_leaves_context_usable(bctx):
    """refused batched calls (OCTANE_EINVAL) between two runs of a large batch change nothing"""
    img1, img2, cth, navs, t1, t2 = distinct_inputs(3, 768, 640, seed0=3600)
    p = ob.default_params(doCTH=1)
    want, _, its_want = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
    for bad in (lambda: run_batch(bctx, img1[:0], img2[:0], [], [], [], p, cth[:0]),
                lambda: run_batch(bctx, img1, img2, navs, t1, t2, ob.default_params(doCTH=1, first_guess=1), cth)):
        with pytest.raises(ob.OctaneError) as e:
            bad()
        assert e.value.code == -2                          # OCTANE_EINVAL
        got, _, its = run_batch(bctx, img1, img2, navs, t1, t2, p, cth)
        for k in want:
            assert np.array_equal(got[k], want[k]), k
        assert np.array_equal(its, its_want)
