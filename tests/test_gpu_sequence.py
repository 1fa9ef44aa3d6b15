"""Sequences of frames in one call (octane_optical_flow_sequence_dev).

Pair k of a sequence is (frame k, frame k + 1).  The call prepares each frame once (copy-in, blur / decimation and
first gradients) where a batch of the same pairs prepares every inner frame twice; the per-pixel kernels involved
have no atomics, so every output must be octane_optical_flow_batch_ex_dev's on frames[:-1], frames[1:], bit for bit:
uPix, vPix, the four navigated short planes, CTP, the moved flags and every pair's iteration counts.  The frames of
a sequence move: frame k + 1 is frame k warped by a vortex, so consecutive pairs see the same motion on new
texture."""
import ctypes as C

import numpy as np
import pytest

import octane_b200 as ob
from octane_b200 import synthetic as S
from test_gpu_batch import COOP_PER_SM, check_vs_oracle, sm_count, tdev
from test_gpu_batch_fg_srsal import outputs, run_ex

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sctx():
    c = ob.Context(0)
    yield c
    c.close()


def make_sequence(nframes, nx, ny, seed, nc=1):
    """[nframes, (nc,) ny, nx] frames, cloud-top heights [nframes - 1, ny, nx] (image 1's of each pair), navigations
    and nframes times 60 s apart on the 2 km mesoscale grid"""
    xs, ys, xo, yo, _ = S.SECTORS["meso_2km"]
    u, v = S.flow_field(nx, ny, "vortex")
    chans = []
    for ch in range(nc):
        f = [S.texture(nx, ny, seed + 100 * ch)]
        for _ in range(nframes - 1):
            f.append(S.warp_pair(f[-1], u, v))
        chans.append(np.stack(f))
    frames = (np.stack(chans, axis=1) if nc > 1 else chans[0]).astype(np.float32)
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = np.stack([(7500.0 + 7400.0 * np.sin(xx / (30.0 + k) + k) * np.cos(yy / 30.0)).astype(np.float32)
                    for k in range(nframes - 1)])
    return frames, cth, [ob.goes_nav(xs, ys, xo, yo)] * (nframes - 1), [60.0 * k for k in range(nframes)]


def run_seq(ctx, frames, navs, t, p, cth=None, nc=1, fg=None):
    """returns (dict of numpy [N, ny, nx], moved, its [N, n_solves], kernel launches)"""
    N = frames.shape[0] - 1
    ny, nx = frames.shape[-2:]
    out = outputs(N, ny, nx, p)
    kw = {} if fg is None else dict(fg_u=tdev(fg[0]), fg_v=tdev(fg[1]))
    moved = ctx.oct_optical_flow_sequence_dev(tdev(frames), navs, t, p, out, cth=None if cth is None else tdev(cth),
                                              nc=nc, **kw)
    launches = ctx.stats().kernel_launches
    its = ctx.batch_cg_iterations(N, p.kiters * 3 * p.liters)
    return {k: v.cpu().numpy() for k, v in out.items()}, moved, its, launches


def run_pairs(ctx, frames, navs, t, p, cth=None, nc=1, fg=None):
    """the same pairs through octane_optical_flow_batch_ex_dev: (outputs, moved, its, kernel launches)"""
    out, moved, its = run_ex(ctx, frames[:-1], frames[1:], navs, t[:-1], t[1:], p, cth, nc=nc, fg=fg)
    return out, moved, its, ctx.stats().kernel_launches


def assert_same(seq, pairs, tag):
    out_s, moved_s, its_s, _ = seq
    out_p, moved_p, its_p, _ = pairs
    assert sorted(out_s) == sorted(out_p), tag
    for k in out_p:
        assert np.array_equal(out_s[k], out_p[k]), (tag, k)
    assert moved_s == moved_p, tag
    assert np.array_equal(its_s, its_p), tag


def check(ctx, frames, navs, t, p, tag, cth=None, nc=1, fg=None):
    seq = run_seq(ctx, frames, navs, t, p, cth, nc, fg)
    pairs = run_pairs(ctx, frames, navs, t, p, cth, nc, fg)
    print(f"{tag}: {frames.shape[0]} frames, kernel launches sequence {seq[3]}, pairs {pairs[3]}, "
          f"iterations {int(seq[2].min())}..{int(seq[2].max())}")
    assert_same(seq, pairs, tag)
    assert seq[2].max() > 0
    return seq, pairs


@pytest.mark.parametrize("nframes", [2, 3, 9])
def test_sequence_small_levels(sctx, nframes):
    """200x200: every level small (cooperative PCG launches); nframes = 2 is a sequence of one pair"""
    frames, cth, navs, t = make_sequence(nframes, 200, 200, seed=4000 + nframes)
    check(sctx, frames, navs, t, ob.default_params(doCTH=1), f"200x200 x{nframes}", cth)


def test_sequence_waves(sctx):
    """2 floor(2 sm / 8) + 2 frames of 264x240: the finest level (8 blocks per pair) runs in three waves of
    cooperative launches and 132x120 (4 blocks per pair) in two, each ending with a one-pair wave"""
    per8 = sm_count() * COOP_PER_SM // 8
    frames, cth, navs, t = make_sequence(2 * per8 + 2, 264, 240, seed=4100)
    check(sctx, frames, navs, t, ob.default_params(), f"264x240 waves, {per8} pairs per wave")


@pytest.mark.parametrize("solver,graphs", [(1, True), (1, False), (0, True)])
def test_sequence_large_levels(solver, graphs):
    """768x640 (finest level large: nx >= 512, >= 64 rows) and 1024^2 (two large levels): the merged-recurrence
    launch for every pair, replayed from graphs or not, and the two-pass kernels pair by pair"""
    ctx = ob.Context(0)
    try:
        ctx.set_solver(solver)
        ctx.set_graphs(graphs)
        for nx, ny, n in ((768, 640, 5), (1024, 1024, 4)):
            frames, cth, navs, t = make_sequence(n, nx, ny, seed=4200 + nx)
            check(ctx, frames, navs, t, ob.default_params(doCTH=1), f"{nx}x{ny} solver {solver} graphs {graphs}", cth)
    finally:
        ctx.close()


def test_sequence_first_guess(sctx):
    """a first guess per pair with lambda_c = 0.5 (the hint term on every level) and lambda_c = 0"""
    nx, ny, n = 160, 120, 6
    frames, _, navs, t = make_sequence(n, nx, ny, seed=4300)
    u, v = S.flow_field(nx, ny, "vortex")
    fu = np.stack([u * (0.8 + 0.1 * k) + 0.2 for k in range(n - 1)]).astype(np.float32)
    fv = np.stack([v * (1.1 - 0.1 * k) - 0.1 for k in range(n - 1)]).astype(np.float32)
    for lc in (0.5, 0.0):
        check(sctx, frames, navs, t, ob.default_params(first_guess=1, lambdac=lc), f"first guess lambdac={lc}",
              fg=(fu, fv))


@pytest.mark.parametrize("ir", [0, 1])
def test_sequence_srsal(sctx, ir):
    """-srsal with each pair's own heights, doCTH with ir 0 / 1"""
    frames, cth, navs, t = make_sequence(5, 200, 150, seed=4400 + ir)
    check(sctx, frames, navs, t, ob.default_params(dosrsal=1, doCTH=1, ir=ir), f"srsal ir={ir}", cth)


def test_sequence_two_channels(sctx):
    frames, cth, navs, t = make_sequence(5, 264, 240, seed=4500, nc=2)
    assert frames.shape == (5, 2, 240, 264)
    check(sctx, frames, navs, t, ob.default_params(doCTH=1), "nc=2", cth, nc=2)


def test_sequence_moved_sector_in_the_middle(sctx):
    """pair 2 of 5 has a frame 3 from a sector that moved: its four short planes are zero, the others are not"""
    frames, cth, navs, t = make_sequence(6, 200, 200, seed=4600)
    xs, ys, xo, yo, _ = S.SECTORS["meso_2km"]
    navs = list(navs)
    navs[2] = ob.goes_nav(xs, ys, xo, yo, g2xOffset=xo + 1e-3)
    seq, _ = check(sctx, frames, navs, t, ob.default_params(doCTH=1), "moved sector", cth)
    assert seq[1] == [2]
    assert not seq[0]["uVal"][2].any() and not seq[0]["vVal2"][2].any()
    assert seq[0]["uVal"][1].any() and seq[0]["uVal"][3].any()


def test_sequence_pair_matches_oracle(sctx, oracle):
    """pair 3 of a 6-frame sequence against its own oracle run, with the batch tests' gates"""
    frames, _, navs, t = make_sequence(6, 160, 120, seed=4700)
    out, _, its, _ = run_seq(sctx, frames, navs, t, ob.default_params())
    check_vs_oracle(oracle, out, its, 3, frames[3], frames[4], {}, 1, "sequence")


def test_sequence_launches(sctx):
    """K levels: the sequence makes the batch's launches less the K - 1 coarse-level blurs and the K first-gradient
    launches of the second image run"""
    p = ob.default_params(doCTH=1)
    frames, cth, navs, t = make_sequence(9, 500, 500, seed=4800)
    seq, pairs = check(sctx, frames, navs, t, p, "launches", cth)
    K = p.kiters
    assert seq[3] == pairs[3] - (K - 1) - K, (seq[3], pairs[3], K)


def test_sequence_state_across_calls(sctx):
    """a sequence, a batch of another size, a single-pair call and a sequence of another length on one context
    (every one lays the workspace out differently): the first sequence's bits come back"""
    frames, cth, navs, t = make_sequence(5, 200, 200, seed=4900)
    p = ob.default_params(doCTH=1)
    want = run_seq(sctx, frames, navs, t, p, cth)
    f2, c2, n2, t2 = make_sequence(8, 200, 200, seed=4950)
    run_pairs(sctx, f2, n2, t2, p, c2)
    import torch
    z = [torch.zeros((200, 200), device="cuda") for _ in range(2)]
    s = [torch.zeros((200, 200), dtype=torch.int16, device="cuda") for _ in range(5)]
    sctx.oct_optical_flow_dev(tdev(f2[0]), tdev(f2[1]), n2[0], t2[0], t2[1], p, *z, *s[:4], cth=tdev(c2[0]), ctp=s[4])
    run_seq(sctx, f2, n2, t2, p, c2)
    assert_same(run_seq(sctx, frames, navs, t, p, cth), want, "after mixed calls")


def call_raw(ctx, nframes, frames, p, out, cth=None, fg=None, nx=200, ny=200):
    """octane_optical_flow_sequence_dev with the arguments as given (no wrapper checks)"""
    npairs = max(nframes - 1, 1)
    xs, ys, xo, yo, _ = S.SECTORS["meso_2km"]
    navs = (ob.Nav * npairs)(*([ob.goes_nav(xs, ys, xo, yo)] * npairs))
    t = (C.c_double * (npairs + 1))(*[60.0 * k for k in range(npairs + 1)])
    moved = (C.c_int * npairs)()
    ptr = lambda a: None if a is None else C.c_void_p(a.data_ptr())
    fu, fv = (None, None) if fg is None else fg
    return ctx._L.octane_optical_flow_sequence_dev(
        ctx._h, nframes, ptr(frames), ptr(fu), ptr(fv), ptr(cth), nx, ny, 1, navs, t, C.byref(p), ptr(out["uPix"]),
        ptr(out["vPix"]), ptr(out["uVal"]), ptr(out["vVal"]), ptr(out["uVal2"]), ptr(out["vVal2"]), ptr(out.get("CTP")),
        moved)


def test_sequence_refusals_leave_context_usable(sctx):
    """nframes < 2, a first guess without its planes, doCTH / -srsal without heights and a request larger than the
    device (OCTANE_ENOMEM, refused before anything is enqueued) each fail, and the next call gives the same bits.
    (The banded-context refusal needs a multi-GPU communicator and is not exercised here.)"""
    import torch
    frames, cth, navs, t = make_sequence(4, 200, 200, seed=5000)
    p = ob.default_params(doCTH=1)
    want = run_seq(sctx, frames, navs, t, p, cth)
    d_frames, d_cth = tdev(frames), tdev(cth)
    out = outputs(3, 200, 200, p)
    EINVAL, ENOMEM = -2, -3
    refusals = {
        "nframes 1": (1, p, d_cth, None),
        "nframes 0": (0, p, d_cth, None),
        "first guess without planes": (4, ob.default_params(first_guess=1), d_cth, None),
        "first guess without fg_v": (4, ob.default_params(first_guess=1), d_cth, (out["uPix"], None)),
        "doCTH without heights": (4, p, None, None),
        "srsal without heights": (4, ob.default_params(dosrsal=1), None, None),
    }
    for tag, (nf, q, c, fg) in refusals.items():
        assert call_raw(sctx, nf, d_frames, q, out, c, fg=fg) == EINVAL, tag
        assert_same(run_seq(sctx, frames, navs, t, p, cth), want, f"after refusal: {tag}")
    # 4000^2 frames, as many as it takes to need twice the device's memory: the single-pair plan fits, the
    # sequence's workspace cannot be allocated, and nothing is read from the (small) buffers passed
    total = torch.cuda.get_device_properties(0).total_memory
    per = ob.batch_workspace_bytes(2, 4000, 4000, 1, p, sequence=True) - ob.batch_workspace_bytes(1, 4000, 4000, 1, p,
                                                                                                    sequence=True)
    n = 2 * total // per + 2
    assert ob.batch_workspace_bytes(n - 1, 4000, 4000, 1, p, sequence=True) > 2 * total
    assert call_raw(sctx, n, d_frames, p, out, d_cth, nx=4000, ny=4000) == ENOMEM
    print("ENOMEM:", sctx._L.octane_last_error().decode())
    assert_same(run_seq(sctx, frames, navs, t, p, cth), want, "after ENOMEM")
