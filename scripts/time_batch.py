"""Time the batched dispatcher (octane_optical_flow_batch_dev) against contexts in flight.

Two workloads: 64 x 500^2 with cloud-top heights and m/s output (BASELINE config 5, bench.py --workload batch64), and
8 x 2000^2, whose finest levels run the single-pair PCG kernels pair by pair.  Arms, alternated on the same inputs in
one run: one batched call per step, and the contexts-in-flight loop of bench.py's batch_arm with K = 8 and 16
contexts.  Reports device ms per step (CUDA events), Mpix/s and kernel launches per step, with the card's name and
power limit.  Writes --out (JSON)."""
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


def workload(n, npairs, seed0, rounds, steps, warmup):
    import torch

    import octane_b200 as ob
    from octane_b200 import synthetic as S

    dev = torch.device("cuda", 0)
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(doCTH=1)
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

    def batch_step():
        bctx.oct_optical_flow_batch_dev(img1, img2, [nav] * npairs, [0.0] * npairs, [dt] * npairs, p, bout, cth=cth)

    arms = {"batch": ([bctx], batch_step)}
    for K in (8, 16):
        ctxs = [ob.Context(0) for _ in range(K)]
        outs = [dict(u=torch.zeros((n, n), device=dev), v=torch.zeros((n, n), device=dev),
                     s=[torch.zeros((n, n), dtype=torch.int16, device=dev) for _ in range(5)]) for _ in pairs]

        def step(ctxs=ctxs, outs=outs, K=K):
            for i, (a, b) in enumerate(pairs):
                o = outs[i]
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
        launches = sum(int(c.stats().kernel_launches) for c in ctxs)
        if k != "batch":
            used = min(len(ctxs), npairs)                 # every used context's last call was one pair
            launches = launches // used * npairs
        best = min(ms[k])
        res[k] = {"ms_per_step": best, "ms_per_step_all": ms[k], "mpix_per_s": mpix / (best / 1e3),
                  "kernel_launches_per_step": launches}
    # the batched flow against the single-pair dispatcher on the same inputs
    torch.cuda.synchronize()
    u8 = torch.stack([o["u"] for o in outs8])
    res["batch_vs_contexts_max_abs_px"] = float((bout["uPix"] - u8).abs().max())
    for name, (ctxs, _) in arms.items():
        if name != "batch":
            for c in ctxs:
                c.close()
    bctx.close()
    return {"pairs": npairs, "size": n, "doCTH": 1, "output": "m/s", **res}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_batch_n1.json"))
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    res = {"card": card(), "what": "device ms per step over CUDA events, best of the alternated rounds",
           "workloads": [workload(500, 64, 100, a.rounds, a.steps, a.warmup),
                         workload(2000, 8, 300, a.rounds, a.steps, a.warmup)]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
