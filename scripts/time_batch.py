"""Time the batched dispatcher (octane_optical_flow_batch_dev) against contexts in flight.

Two workloads: 64 x 500^2 with cloud-top heights and m/s output (BASELINE config 5, bench.py --workload batch64), and
8 x 2000^2, whose finest levels run the single-pair PCG kernels pair by pair.  Arms, alternated on the same inputs in
one run: one batched call per step, and the contexts-in-flight loop of bench.py's batch_arm with K = 8 and 16
contexts.  Reports device ms per step (CUDA events), Mpix/s and kernel launches per step, with the card's name and
power limit.  Writes --out (JSON).

--first-guess (with lambda_c = 0.5) and --srsal time the same workloads with those flags: the batch arm calls
octane_optical_flow_batch_ex_dev, the contexts arms pass the same flags to octane_optical_flow_dev, and with --srsal a
second batch arm without -srsal gives the cost of the smoother.  The default output is then
profiles/r03_batch_fg_srsal_n1.json.

--sequence times octane_optical_flow_sequence_dev on npairs + 1 frames against octane_optical_flow_batch_ex_dev on
the same pairs (frames[:-1], frames[1:]), alternated, for 64 x 500^2 (65 frames) and 8 x 2000^2 (9 frames).  The
frames alternate the two images of a synthetic pair, so every pair has real motion.  It also reports the device
bytes each call allocates (octane_batch_workspace_bytes) and whether the two arms' outputs are bit-identical.  The
default output is then profiles/r04_sequence_n1.json."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def workload(n, npairs, seed0, rounds, steps, warmup, fg=False, srsal=False):
    import torch

    import octane_b200 as ob
    from octane_b200 import synthetic as S

    dev = torch.device("cuda", 0)
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    flags = dict(first_guess=1, lambdac=0.5) if fg else {}
    p = ob.default_params(doCTH=1, dosrsal=int(srsal), **flags)
    yy, xx = np.mgrid[0:n, 0:n].astype(np.float32)
    cth1 = torch.from_numpy((7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)).to(dev)
    pairs = [S.make_pair_torch(n, n, seed0 + k, dev) for k in range(npairs)]
    img1 = torch.stack([a for a, _ in pairs]).contiguous()
    img2 = torch.stack([b for _, b in pairs]).contiguous()
    cth = cth1.expand(npairs, n, n).contiguous()
    bout = {k: torch.zeros((npairs, n, n), device=dev) for k in ("uPix", "vPix")}
    for k in ("uVal", "vVal", "uVal2", "vVal2", "CTP"):
        bout[k] = torch.zeros((npairs, n, n), dtype=torch.int16, device=dev)
    bctx = ob.Context(0)
    if fg:                                       # a smooth first guess, scaled per pair
        u0 = torch.from_numpy(0.6 + 0.3 * np.sin(xx / 23.0) * np.cos(yy / 31.0)).to(dev)
        v0 = torch.from_numpy(-0.3 + 0.2 * np.cos(xx / 19.0 + yy / 29.0)).to(dev)
        scale = torch.linspace(0.8, 1.2, npairs, device=dev).view(npairs, 1, 1)
        fgu, fgv = (u0 * scale).contiguous(), (v0 * scale).contiguous()
    ex = dict(fg_u=fgu, fg_v=fgv) if fg else {}

    def batch_step(p=p, bout=bout):
        if fg or srsal:
            bctx.oct_optical_flow_batch_ex_dev(img1, img2, [nav] * npairs, [0.0] * npairs, [dt] * npairs, p, bout,
                                               cth=cth, **ex)
        else:
            bctx.oct_optical_flow_batch_dev(img1, img2, [nav] * npairs, [0.0] * npairs, [dt] * npairs, p, bout, cth=cth)

    arms = {"batch": ([bctx], batch_step)}
    if srsal:                                    # the same call without -srsal, on its own outputs
        p0 = ob.default_params(doCTH=1, **flags)
        bout0 = {k: torch.zeros_like(a) for k, a in bout.items()}
        arms["batch_no_srsal"] = ([bctx], lambda: batch_step(p0, bout0))
    for K in (8, 16):
        ctxs = [ob.Context(0) for _ in range(K)]
        outs = [dict(u=torch.zeros((n, n), device=dev), v=torch.zeros((n, n), device=dev),
                     s=[torch.zeros((n, n), dtype=torch.int16, device=dev) for _ in range(5)]) for _ in pairs]

        def step(ctxs=ctxs, outs=outs, K=K):
            for i, (a, b) in enumerate(pairs):
                o = outs[i]
                if fg:                           # octane_optical_flow_dev reads its first guess from uPix / vPix
                    with torch.cuda.stream(ctxs[i % K]._ext_stream()):
                        o["u"].copy_(fgu[i])
                        o["v"].copy_(fgv[i])
                ctxs[i % K].oct_optical_flow_dev(a, b, nav, 0.0, dt, p, o["u"], o["v"], *o["s"][:4], cth=cth1,
                                                 ctp=o["s"][4], sync_torch=False)
        arms[f"contexts_{K}"] = (ctxs, step)
        if K == 8:
            outs8 = outs

    def timed(ctxs, fn):
        for c in ctxs:
            c.synchronize()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for c in ctxs:
            c._after_torch()
        for _ in range(steps):
            fn()
        for c in ctxs:
            c._before_torch()
        e1.record()
        for c in ctxs:
            c.synchronize()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for ctxs, fn in arms.values():
        for _ in range(warmup):
            fn()
    ms = {k: [] for k in arms}
    for _ in range(rounds):                       # alternate the arms
        for k, (ctxs, fn) in arms.items():
            ms[k].append(timed(ctxs, fn))
    res = {}
    mpix = npairs * n * n / 1e6
    for k, (ctxs, fn) in arms.items():
        if srsal and k.startswith("batch"):      # the two batch arms share a context: its counters hold the last call
            fn()
        launches = sum(int(c.stats().kernel_launches) for c in ctxs)
        if k.startswith("contexts"):
            used = min(len(ctxs), npairs)                 # every used context's last call was one pair
            launches = launches // used * npairs
        best = min(ms[k])
        res[k] = {"ms_per_step": best, "ms_per_step_all": ms[k], "mpix_per_s": mpix / (best / 1e3),
                  "kernel_launches_per_step": launches}
    # the batched flow against the single-pair dispatcher on the same inputs
    torch.cuda.synchronize()
    u8 = torch.stack([o["u"] for o in outs8])
    res["batch_vs_contexts_max_abs_px"] = float((bout["uPix"] - u8).abs().max())
    if fg or srsal:
        v8 = torch.stack([o["v"] for o in outs8])
        res["batch_vs_contexts_max_abs_px_v"] = float((bout["vPix"] - v8).abs().max())
    for name, (ctxs, _) in arms.items():
        if name.startswith("contexts"):
            for c in ctxs:
                c.close()
    bctx.close()
    if srsal:
        res["srsal_ms_per_step"] = res["batch"]["ms_per_step"] - res["batch_no_srsal"]["ms_per_step"]
    if fg:
        res["first_guess_note"] = ("the contexts arms copy each pair's first guess into its uPix / vPix on the "
                                   "context's stream before each call (two device copies per pair, timed); the batch "
                                   "arm reads fg_u / fg_v directly")
    return {"pairs": npairs, "size": n, "doCTH": 1, "output": "m/s", **({"first_guess": 1, "lambdac": 0.5} if fg else {}),
            **({"dosrsal": 1} if srsal else {}), **res}


def sequence_workload(n, npairs, seed, rounds, steps, warmup):
    import torch

    import octane_b200 as ob
    from octane_b200 import synthetic as S

    dev = torch.device("cuda", 0)
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(doCTH=1)
    a, b = S.make_pair_torch(n, n, seed, dev)
    frames = torch.stack([a if k % 2 == 0 else b for k in range(npairs + 1)]).contiguous()
    t = [dt * k for k in range(npairs + 1)]
    yy, xx = np.mgrid[0:n, 0:n].astype(np.float32)
    cth1 = torch.from_numpy((7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)).to(dev)
    cth = cth1.expand(npairs, n, n).contiguous()

    def outputs():
        o = {k: torch.zeros((npairs, n, n), device=dev) for k in ("uPix", "vPix")}
        for k in ("uVal", "vVal", "uVal2", "vVal2", "CTP"):
            o[k] = torch.zeros((npairs, n, n), dtype=torch.int16, device=dev)
        return o

    ctx = ob.Context(0)
    outs = {"sequence": outputs(), "batch": outputs()}
    navs = [nav] * npairs
    arms = {
        "sequence": lambda: ctx.oct_optical_flow_sequence_dev(frames, navs, t, p, outs["sequence"], cth=cth),
        "batch": lambda: ctx.oct_optical_flow_batch_ex_dev(frames[:-1], frames[1:], navs, t[:-1], t[1:], p,
                                                           outs["batch"], cth=cth),
    }

    def timed(fn):
        ctx.synchronize()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx._after_torch()
        for _ in range(steps):
            fn()
        ctx._before_torch()
        e1.record()
        ctx.synchronize()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for fn in arms.values():
        for _ in range(warmup):
            fn()
    ms = {k: [] for k in arms}
    for _ in range(rounds):                       # alternate the arms
        for k, fn in arms.items():
            ms[k].append(timed(fn))
    res = {}
    mpix = npairs * n * n / 1e6
    for k, fn in arms.items():
        fn()
        best = min(ms[k])
        res[k] = {"ms_per_step": best, "ms_per_step_all": ms[k], "mpix_per_s": mpix / (best / 1e3),
                  "kernel_launches_per_step": int(ctx.stats().kernel_launches)}
    torch.cuda.synchronize()
    res["outputs_bit_identical"] = all(torch.equal(outs["sequence"][k], outs["batch"][k]) for k in outs["batch"])
    res["workspace_bytes"] = {"sequence": ob.batch_workspace_bytes(npairs, n, n, 1, p, sequence=True),
                              "batch": ob.batch_workspace_bytes(npairs, n, n, 1, p)}
    ctx.close()
    return {"pairs": npairs, "frames": npairs + 1, "size": n, "doCTH": 1, "output": "m/s", **res}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--first-guess", action="store_true", help="solve with a first guess and lambda_c = 0.5")
    ap.add_argument("--srsal", action="store_true", help="run the -srsal post-smoother")
    ap.add_argument("--sequence", action="store_true", help="time the sequence call against the batch on the same frames")
    a = ap.parse_args()
    if a.sequence and (a.first_guess or a.srsal):
        ap.error("--sequence times the plain call")
    name = ("r04_sequence_n1.json" if a.sequence else
            "r03_batch_fg_srsal_n1.json" if a.first_guess or a.srsal else "r03_batch_n1.json")
    a.out = a.out or os.path.join(ROOT, "profiles", name)
    flags = dict(fg=a.first_guess, srsal=a.srsal)
    res = {"card": card(), "what": "device ms per step over CUDA events, best of the alternated rounds"}
    if a.sequence:
        res["workloads"] = [sequence_workload(500, 64, 100, a.rounds, a.steps, a.warmup),
                            sequence_workload(2000, 8, 300, a.rounds, a.steps, a.warmup)]
    else:
        res["workloads"] = [workload(500, 64, 100, a.rounds, a.steps, a.warmup, **flags),
                            workload(2000, 8, 300, a.rounds, a.steps, a.warmup, **flags)]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
