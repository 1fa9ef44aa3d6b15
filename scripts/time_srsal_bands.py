"""Times -srsal on the full disk (21696 x 21696, 0.5 km) on 1 or more GPUs, one rank per GPU:

  * srsal alone: octane_srsal_band_dev on each rank's owned rows (staging vote, 18-row exchange and the filter), CUDA
    events on the context's stream, the maximum over ranks;
  * the pipelined dispatcher end to end (octane_stream_submit / octane_stream_wait, pinned host buffers, two pairs in
    flight, every copy inside the timed region), ms per pair, with -pd (pixel displacements returned) with and
    without -srsal.

Writes <out>/r03_srsal_bands_n<world>.json with the card's name and power limit read in the same run.
Usage: python scripts/time_srsal_bands.py [--out DIR]                         (one GPU)
       python -m torch.distributed.run --nproc-per-node=N scripts/time_srsal_bands.py [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import octane_b200 as ob  # noqa: E402
from octane_b200 import synthetic as S  # noqa: E402


def card(local):
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(local)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--nx", type=int, default=21696)
    ap.add_argument("--ny", type=int, default=21696)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--srsal-reps", type=int, default=3)
    args = ap.parse_args()
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    nx, ny = args.nx, args.ny
    ctx = ob.Context(local)
    if world > 1:
        ids = [ob.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(ids[0], rank, world)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr, device=dev)

    def max_over_ranks(ms):
        if dist:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def timed(fn, reps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / reps)

    xs, ys, xo, yo, dt = S.SECTORS["fulldisk_0.5km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p_pd = ob.default_params(max_disp=64, pixuv=1)
    p_sr = ob.default_params(max_disp=64, pixuv=1, dosrsal=1)
    own0, own1, in0, in1 = ob.band_plan(nx, ny, p_pd, rank, world)
    nown = own1 - own0
    res = dict(world=world, nx=nx, ny=ny, own_rows=[own0, own1], card=card(local) if rank == 0 else None)

    # ---- srsal alone on the owned rows (a smooth cloud deck with noise; the filter's cost does not depend on the values)
    g = torch.Generator(device=dev).manual_seed(11 + rank)
    u = torch.randn((nown, nx), device=dev, generator=g)
    v = torch.randn((nown, nx), device=dev, generator=g)
    yy = torch.arange(own0, own1, device=dev, dtype=torch.float32)[:, None]
    xx = torch.arange(nx, device=dev, dtype=torch.float32)[None, :]
    cth = (7500.0 + 7400.0 * torch.sin(xx / 40.0) * torch.cos(yy / 30.0) + 30.0 * torch.randn((nown, nx), device=dev, generator=g)).contiguous()
    ctx.oct_srsal_band(u, v, cth, nx, ny)                   # staging, NCCL set-up
    res["srsal_ms"] = timed(lambda: ctx.oct_srsal_band(u, v, cth, nx, ny), args.srsal_reps)
    res["srsal_Mpix_per_s"] = nx * ny / 1e3 / res["srsal_ms"]
    del u, v

    # ---- the pipelined dispatcher, -pd, with and without -srsal
    img1, img2 = S.make_pair_torch(nx, ny, 4, dev, limb_taper=True, rows=(in0, in1))
    h1 = torch.empty(img1.shape, dtype=torch.float32, pin_memory=True); h1.copy_(img1)
    h2 = torch.empty(img2.shape, dtype=torch.float32, pin_memory=True); h2.copy_(img2)
    hc = torch.empty(cth.shape, dtype=torch.float32, pin_memory=True); hc.copy_(cth)
    del img1, img2, cth
    torch.cuda.empty_cache()
    outs = [{k: torch.zeros((nown, nx), dtype=(torch.float32 if k.endswith("Pix") else torch.int16), pin_memory=True).numpy()
             for k in ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")} for _ in range(2)]

    def pipelined(p, steps):
        def run(n):
            for k in range(n):
                ctx.stream_submit(k % 2, h1.numpy(), h2.numpy(), nav, 0.0, dt, p, outs[k % 2], nx, ny, cth=hc.numpy())
                if k > 0:
                    ctx.stream_wait((k - 1) % 2)
            ctx.stream_wait((n - 1) % 2)
        run(2)                                              # warm-up: plan, graphs, staging slots
        return timed(lambda: run(steps), 1) / steps

    for name, p in (("pd", p_pd), ("pd_srsal", p_sr)):
        ms = pipelined(p, args.steps)
        res[f"e2e_ms_per_pair_{name}"] = ms
        res[f"e2e_Mpix_per_s_{name}"] = nx * ny / 1e3 / ms
    res["e2e_srsal_share"] = 1.0 - res["e2e_ms_per_pair_pd"] / res["e2e_ms_per_pair_pd_srsal"]
    res["note"] = ("srsal_ms: CUDA events on the context's stream around octane_srsal_band_dev (staging vote, 18-row NCCL "
                   "exchange, filter), max over ranks; e2e: octane_stream_submit / _wait over the pairs, pinned host buffers, "
                   f"{args.steps} pairs after 2 warm-up pairs, max over ranks")
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, f"r03_srsal_bands_n{world}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res), flush=True)
    barrier()
    del outs, h1, h2, hc              # pinned blocks carry events of the context's stream: release them before it
    ctx.close()
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
