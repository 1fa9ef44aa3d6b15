"""Multi-GPU worker (launched by torch.distributed.run, one rank per GPU) for -srsal on row bands and for -srsal / a
first guess through the pipelined dispatcher on bands.  argv: nx ny modes (comma-separated: field, refuse, stream, fg).
Prints one line `BAND_POST_RESULT {...json...}` on rank 0."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import octane_b200 as ob  # noqa: E402
from octane_b200 import synthetic as S  # noqa: E402


def own_rows(ny, rank, world):
    """the rows octane_srsal_band_dev filters on `rank`: the finest level's rule of the band plan"""
    return rank * ny // world, (rank + 1) * ny // world


def seeded_field(nx, ny, seed):
    """u, v, cth of the whole scene, the same on every rank: noisy displacements over a cloud deck with steps"""
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((ny, nx)).astype(np.float32)
    v = rng.standard_normal((ny, nx)).astype(np.float32)
    yy, xx = np.mgrid[0:ny, 0:nx]
    deck = np.where((xx // 37 + yy // 23) % 3 == 0, 9000.0, 4000.0) + 30.0 * rng.standard_normal((ny, nx))
    return u, v, deck.astype(np.float32)


def cloud_tops(nx, r0, r1):
    yy, xx = np.mgrid[r0:r1, 0:nx].astype(np.float32)
    return (7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)


def first_guess(nx, r0, r1):
    """smooth displacement field close to the true drift, rows [r0, r1) (as tests/band_worker.py)"""
    yy, xx = np.mgrid[r0:r1, 0:nx].astype(np.float32)
    return ((0.6 + 0.3 * np.sin(xx / 23.0) * np.cos(yy / 31.0)).astype(np.float32),
            (-0.3 + 0.2 * np.cos(xx / 19.0 + yy / 29.0)).astype(np.float32))


def pinned(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def gather_rows(world, own0, *planes):
    """every rank's owned rows of each plane, concatenated in row order (on every rank)"""
    parts = [None] * world
    dist.all_gather_object(parts, (own0,) + tuple(planes))
    parts.sort(key=lambda t: t[0])
    return [np.concatenate([t[1 + i] for t in parts]) for i in range(len(planes))]


def all_ranks(flag, world):
    flags = [None] * world
    dist.all_gather_object(flags, bool(flag))
    return all(flags)


def banded_srsal_equals_single(ctx, nx, ny, seed, rank, world, dev, local):
    u, v, cth = seeded_field(nx, ny, seed)
    o0, o1 = own_rows(ny, rank, world)
    du, dv = torch.from_numpy(u[o0:o1].copy()).to(dev), torch.from_numpy(v[o0:o1].copy()).to(dev)
    ctx.oct_srsal_band(du, dv, torch.from_numpy(cth[o0:o1].copy()).to(dev), nx, ny)
    ctx.synchronize()
    U, V = gather_rows(world, o0, du.cpu().numpy(), dv.cpu().numpy())
    ok = True
    if rank == 0:                      # single-GPU filter of the whole field with a fresh, un-banded context
        c1 = ob.Context(local)
        wu, wv = c1.oct_srsal_cu(torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev), torch.from_numpy(cth).to(dev))
        c1.synchronize()
        ok = np.array_equal(U, wu.cpu().numpy()) and np.array_equal(V, wv.cpu().numpy())
        c1.close()
    return all_ranks(ok, world)


def run_pipeline(ctx, submits, nav, dt, p, nx, ny, rows, img1, img2, cth=None, fg=None, keys=("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")):
    """`submits` submits of the same pair, two in flight; returns the outputs of every submit (rows [own0,own1))"""
    outs = [{k: torch.zeros((rows, nx), dtype=(torch.float32 if k.endswith("Pix") else torch.int16), pin_memory=True).numpy()
             for k in keys} for _ in range(2)]
    kw = {} if fg is None else dict(fg_u_band=fg[0], fg_v_band=fg[1])
    got = []
    for k in range(submits):
        ctx.stream_submit(k % 2, img1, img2, nav, 0.0, dt, p, outs[k % 2], nx, ny, cth=cth, **kw)
        if k > 0:
            ctx.stream_wait((k - 1) % 2)
            got.append({key: val.copy() for key, val in outs[(k - 1) % 2].items()})
    ctx.stream_wait((submits - 1) % 2)
    got.append({key: val.copy() for key, val in outs[(submits - 1) % 2].items()})
    return got


def main():
    nx, ny, modes = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3].split(",")
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ctx = ob.Context(local)
    ids = [ob.Context.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    ctx.comm_init(ids[0], rank, world)
    res = dict(world=world, nx=nx, ny=ny)
    xs, ys, xo, yo, dt = S.SECTORS["conus_0.5km"]
    nav = ob.goes_nav(xs, ys, xo, yo)

    if "field" in modes:
        res["field_equal"] = banded_srsal_equals_single(ctx, nx, ny, 21, rank, world, dev, local)

    if "refuse" in modes:
        # a band thinner than the window's reach: every rank computes the same refusal before any exchange
        o0, o1 = own_rows(ny, rank, world)
        z = torch.zeros((o1 - o0, nx), device=dev)
        code = 0
        try:
            ctx.oct_srsal_band(z, z.clone(), z.clone(), nx, ny)
        except ob.OctaneError as e:
            code = e.code
        codes = [None] * world
        dist.all_gather_object(codes, code)
        res["refused_everywhere"] = all(c_ == -2 for c_ in codes)
        # a call that succeeds first: the NCCL all-reduce and send / receive paths are set up before memory runs short
        warm = banded_srsal_equals_single(ctx, nx, 4 * ny, 22, rank, world, dev, local)
        # one rank cannot allocate its staging (the three extended planes of a 3000 x 3000 scene, ~55 MB per rank):
        # the vote turns that into an error on every rank
        n2 = 3000
        b0, b1 = own_rows(n2, rank, world)
        bu = torch.ones((b1 - b0, n2), device=dev); bv = torch.ones_like(bu); bc = torch.ones_like(bu)
        hog = None
        if rank == world - 1:
            torch.cuda.synchronize(dev)
            torch.cuda.empty_cache()
            free, _ = torch.cuda.mem_get_info(dev)
            hog = torch.empty(max(free - (8 << 20), 0), dtype=torch.uint8, device=dev)
        code = 0
        try:
            ctx.oct_srsal_band(bu, bv, bc, n2, n2)
            ctx.synchronize()
        except ob.OctaneError as e:
            code = e.code
        codes = [None] * world
        dist.all_gather_object(codes, code)
        del hog, bu, bv, bc
        torch.cuda.empty_cache()
        res["oom_codes"] = codes
        res["oom_everywhere"] = all(c_ != 0 for c_ in codes)
        # the same contexts on a scene the ranks can filter
        res["recovered"] = warm and banded_srsal_equals_single(ctx, nx, 4 * ny, 22, rank, world, dev, local)

    if "stream" in modes or "fg" in modes:
        with_fg = "fg" in modes
        p = ob.default_params(max_disp=16, first_guess=int(with_fg), lambdac=0.5 if with_fg else 0.0,
                              dosrsal=0 if with_fg else 1)
        own0, own1, in0, in1 = ob.band_plan(nx, ny, p, rank, world)
        rows = own1 - own0
        img1, img2 = S.make_pair_torch(nx, ny, 9, dev, rows=(in0, in1))
        cth = cloud_tops(nx, own0, own1)
        fgu, fgv = first_guess(nx, in0, in1)
        # the banded device path
        u = torch.zeros((rows, nx), device=dev); v = torch.zeros_like(u)
        if with_fg:
            ctx.oct_variational_optical_flow_band(img1, img2, u, v, nx, ny, p, fg_u_band=torch.from_numpy(fgu).to(dev),
                                                  fg_v_band=torch.from_numpy(fgv).to(dev))
        else:
            ctx.oct_variational_optical_flow_band(img1, img2, u, v, nx, ny, p)
        sh = [torch.zeros((rows, nx), dtype=torch.int16, device=dev) for _ in range(4)]
        ctx.oct_pix2uv_band(nav, 0.0, dt, u, v, nx, own0, rows, *sh, p)
        raw_u, raw_v = u.cpu().numpy(), v.cpu().numpy()
        if not with_fg:
            ctx.oct_srsal_band(u, v, torch.from_numpy(cth).to(dev), nx, ny)
        ctx.synchronize()
        want = dict(uPix=u.cpu().numpy(), vPix=v.cpu().numpy(), uVal=sh[0].cpu().numpy(), vVal=sh[1].cpu().numpy(),
                    uVal2=sh[2].cpu().numpy(), vVal2=sh[3].cpu().numpy())
        # the pipelined dispatcher on the same band
        h1 = pinned(img1.cpu().numpy()); h2 = pinned(img2.cpu().numpy())
        hfg = (pinned(fgu), pinned(fgv)) if with_fg else None
        got = run_pipeline(ctx, 3, nav, dt, p, nx, ny, rows, h1, h2, cth=None if with_fg else pinned(cth), fg=hfg)
        ok = all(np.array_equal(g[k], want[k]) for g in got for k in want)
        if with_fg:
            ok = ok and np.array_equal(hfg[0], fgu) and np.array_equal(hfg[1], fgv)
            res["fg_equal"] = all_ranks(ok, world)
        else:
            res["stream_equal"] = all_ranks(ok, world)
            U, V, RU, RV, SU = gather_rows(world, own0, got[-1]["uPix"], got[-1]["vPix"], raw_u, raw_v, got[-1]["uVal"])
            if rank == 0:          # the single-GPU pipeline with -srsal, and the single-GPU flow before smoothing
                c1 = ob.Context(local)
                a, b = S.make_pair_torch(nx, ny, 9, dev)
                ha, hb = pinned(a.cpu().numpy()), pinned(b.cpu().numpy())
                one = run_pipeline(c1, 1, nav, dt, p, nx, ny, ny, ha, hb, cth=pinned(cloud_tops(nx, 0, ny)))[0]
                u1 = torch.zeros((ny, nx), device=dev); v1 = torch.zeros_like(u1)
                c1.oct_variational_optical_flow(a, b, u1, v1, p)
                c1.synchronize()
                du, dv = np.abs(U - one["uPix"]), np.abs(V - one["vPix"])
                res.update(du_mean=float(du.mean()), du_max=float(du.max()), dv_mean=float(dv.mean()), dv_max=float(dv.max()),
                           du_raw_max=float(np.abs(RU - u1.cpu().numpy()).max()),
                           dv_raw_max=float(np.abs(RV - v1.cpu().numpy()).max()),
                           nav_max=int(np.abs(SU.astype(int) - one["uVal"].astype(int)).max()))
                c1.close()

    if rank == 0:
        print("BAND_POST_RESULT " + json.dumps(res), flush=True)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
