#!/usr/bin/env python
"""bench.py -- flow Mpix/s of the dense variational optical-flow path.

    python bench.py --gpus N --steps K --warmup W [--workload fulldisk|conus|meso] [--dump-outputs DIR]
    python bench.py --impl reference ...          # the reference's own CPU flow path

One "step" = one pass of the hot path over one synthetic image pair:
pyramid -> (build + Jacobi-PCG) x kiters*3*liters -> prolongation -> pix2uv
navigation.  `value` is timed with the pair already resident in HBM (CUDA
events on the context's stream); `e2e` is the same metric through the C-ABI
host-buffer entry point octane_optical_flow (pinned host inputs, H2D and D2H
inside the timed region).  N > 1 shards the pair across ranks as row bands
(halo exchange + scalar all-reduce over NCCL): total work is fixed -> "strong".
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (nx, ny, sector, limb taper)
    "fulldisk": (21696, 21696, "fulldisk_0.5km", True),
    "conus": (10000, 6000, "conus_0.5km", False),
    "meso": (2000, 2000, "meso_0.5km", False),
    "meso500": (500, 500, "meso_2km", False),
}
METRIC = "flow Mpix/s"
# algorithmic bytes per pixel per launch (DESIGN.md section 4): pass 1 reads r, p, x, a1, a2, a4, W, N
# and writes p, q, x (68 B; 44 B in iteration 0 and 60 B in iteration 1 of a solve, where p / x do not
# exist yet); pass 2 reads q, r, a1, a4 and writes r (32 B)
B_PASS1, B_PASS1_IT0, B_PASS1_IT1, B_PASS2 = 68.0, 44.0, 60.0, 32.0


def pass1_bytes(its):
    """average pass-1 bytes per pixel per working launch over solves with `its` iterations each"""
    tot = sum((B_PASS1_IT0 if n >= 1 else 0) + (B_PASS1_IT1 if n >= 2 else 0) + B_PASS1 * max(n - 2, 0) for n in its)
    return tot / max(sum(its), 1)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.proc.terminate()
        self.t.join(timeout=5)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            try:
                pw.append(float(c[2]))
            except ValueError:
                pass
            for nm, val in zip(names, c[3:7]):
                if val == "Active":
                    reasons.add(nm)
        # samples under load only (idle samples at the edges read the idle clock)
        load = [x for x in sm if x > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


def cpu_sample(nx, ny, sector, seed, size):
    """Bounded sample for the CPU arms: a size x size crop at the scene centre (same generator)."""
    import torch

    from octane_b200 import synthetic as S
    sx, sy = min(size, nx), min(size, ny)
    r0 = (ny - sy) // 2
    a, b = S.make_pair_torch(nx, ny, seed, "cpu", rows=(r0, r0 + sy), limb_taper=False)
    c0 = (nx - sx) // 2
    i1 = a[:, c0:c0 + sx].contiguous().numpy()
    i2 = b[:, c0:c0 + sx].contiguous().numpy()
    return i1, i2, c0, r0


def run_cpu_port(nx, ny, sector, seed, size=2048):
    """cpu_baseline kind 'port': the CPU oracle (OpenMP, all host cores) on a bounded sample."""
    import numpy as np

    from octane_b200 import synthetic as S
    from oracle import oracle as O
    i1, i2, c0, r0 = cpu_sample(nx, ny, sector, seed, size)
    xs, ys, xo, yo, dt = S.SECTORS[sector]
    nav = O.goes_nav(xs, ys, xo, yo, minX=c0, minY=r0)
    t = time.perf_counter()
    u, v, _ = O.variational_flow(i1, i2)
    O.pix2uv(nav, 0.0, dt, u, v)
    sec = time.perf_counter() - t
    n = i1.shape[0] * i1.shape[1]
    return {"value": n / sec / 1e6, "unit": "Mpix/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"{i1.shape[1]}x{i1.shape[0]} centre crop of the workload, 1 pair, variational oracle + pix2uv, OpenMP",
            "seconds": sec}


def run_ref_cuda(nx, ny, sector, seed, size=2000):
    """The reference's own CUDA path recompiled for sm_100 (oracle/_ref), bounded sample, 1 host thread."""
    from octane_b200 import synthetic as S
    from oracle import oracle as O
    import numpy as np
    i1, i2, c0, r0 = cpu_sample(nx, ny, sector, seed, size)
    xs, ys, xo, yo, dt = S.SECTORS[sector]
    nav = O.goes_nav(xs, ys, xo, yo, minX=c0, minY=r0)
    sy, sx = i1.shape
    L = O.ref_cuda()
    import ctypes as C
    outs = [np.zeros((sy, sx), np.int16) for _ in range(4)]
    up = np.zeros((sy, sx), np.float32); vp = np.zeros((sy, sx), np.float32)
    dT = C.c_float()
    rp = O.ref_params()
    best = None
    for _ in range(2):       # first call pays CUDA context + managed-memory setup
        t = time.perf_counter()
        L.ref_optical_flow(i1, i2, None, sx, sy, C.byref(nav), 0.0, dt, C.byref(rp), up, vp, *outs, None, C.byref(dT))
        sec = time.perf_counter() - t
        best = sec if best is None else min(best, sec)
    res = {"value": sx * sy / best / 1e6, "unit": "Mpix/s", "sample": f"{sx}x{sy} centre crop, best of 2, whole oct_optical_flow() "
           "call (managed-memory migration and host loops included)", "seconds": best, "host_threads": 1}
    # the same crop through this repo's dispatcher (host buffers in and out, like the reference's call): its rate, and
    # the difference between the two results -- the reference's output is a parity check here, not only a timing
    try:
        import octane_b200 as ob
        ctx = ob.Context(0)
        onav = ob.goes_nav(xs, ys, xo, yo, minX=c0, minY=r0)
        ours = None
        obest = None
        for _ in range(2):
            t = time.perf_counter()
            ours = ctx.oct_optical_flow(i1, i2, onav, 0.0, dt, ob.default_params())
            sec = time.perf_counter() - t
            obest = sec if obest is None else min(obest, sec)
        ctx.close()
        du, dv = np.abs(ours["uPix"] - up), np.abs(ours["vPix"] - vp)
        dU = np.abs(ours["uVal"].astype(np.int32) - outs[0]); dV = np.abs(ours["vVal"].astype(np.int32) - outs[1])
        res["ours_same_crop"] = {"value": sx * sy / obest / 1e6, "unit": "Mpix/s", "seconds": obest,
                                 "api": "octane_optical_flow (pageable host buffers, best of 2)"}
        res["delta_vs_ours"] = {"mean_abs_du_px": float(du.mean()), "mean_abs_dv_px": float(dv.mean()),
                                "max_abs_du_px": float(du.max()), "max_abs_dv_px": float(dv.max()),
                                "max_abs_dU_counts": int(dU.max()), "max_abs_dV_counts": int(dV.max()),
                                "frac_U_or_V_differs": float(((dU > 0) | (dV > 0)).mean()),
                                "within_gates": bool(max(du.mean(), dv.mean()) <= 1e-3 and max(du.max(), dv.max()) <= 1e-2)}
    except Exception as e:
        res["delta_vs_ours"] = {"unavailable": str(e)[:160]}
    return res


DIGEST_STRIDE = 64


def flow_check(u, v, own0, nx, ny, workload, dist, write):
    """In-run result check: a strided sample (every 64th row and column) of the flow this run produced, gathered
    over the ranks and compared with the digest a single-GPU run of the same workload stored under
    tests/golden/digest_<workload>.npz (`--write-digest`, N = 1).  Collective: every rank calls it."""
    import numpy as np
    import torch
    s = DIGEST_STRIDE
    rows = [j for j in range(own0, own0 + u.shape[0]) if j % s == 0]
    idx = torch.tensor([j - own0 for j in rows], device=u.device, dtype=torch.long)
    mine = (rows, u.index_select(0, idx)[:, ::s].cpu().numpy(), v.index_select(0, idx)[:, ::s].cpu().numpy())
    parts = [mine]
    if dist:
        parts = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
        dist.gather_object(mine, parts, dst=0)
        if dist.get_rank() != 0:
            return None
    parts.sort(key=lambda t: t[0][0] if t[0] else 1 << 30)
    us = np.concatenate([t[1] for t in parts if t[0]]); vs = np.concatenate([t[2] for t in parts if t[0]])
    path = os.path.join(ROOT, "tests", "golden", f"digest_{workload}.npz")
    if write:
        np.savez_compressed(path, us=us, vs=vs, stride=np.int32(s), nx=np.int32(nx), ny=np.int32(ny))
        return {"digest": os.path.relpath(path, ROOT), "written": True, "samples": int(us.size)}
    if not os.path.exists(path):
        return {"digest": None, "note": "no stored single-GPU digest for this workload"}
    d = np.load(path)
    if d["us"].shape != us.shape:
        return {"digest": os.path.relpath(path, ROOT), "note": "digest shape differs"}
    du, dv = np.abs(us - d["us"]), np.abs(vs - d["vs"])
    return {"digest": os.path.relpath(path, ROOT), "what": "strided sample of u, v against the stored single-GPU result",
            "samples": int(us.size), "max_abs_du": float(du.max()), "max_abs_dv": float(dv.max()),
            "mean_abs_du": float(du.mean()), "mean_abs_dv": float(dv.mean()),
            "finite": bool(np.isfinite(us).all() and np.isfinite(vs).all()),
            "within_gates": bool(max(du.mean(), dv.mean()) <= 1e-3 and max(du.max(), dv.max()) <= 1e-2)}


DUMP_NAMES = ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")
DUMP_PIXELS = 1 << 21      # per plane: six float32 planes of at most 8 MB each
DUMP_SEED = 20241020


def dump_positions(nx, ny):
    """Flat row-major pixel indices (ascending) that --dump-outputs samples, or None when the scene is written whole.
    Fixed seed: every run of the same scene size samples the same pixels."""
    import numpy as np
    if nx * ny <= DUMP_PIXELS:
        return None
    idx = np.random.default_rng(DUMP_SEED).choice(nx * ny, DUMP_PIXELS, replace=False, shuffle=False)
    idx.sort()
    return idx


def dump_outputs(out_dir, nx, ny, own0, planes, dist):
    """--dump-outputs: the planes the timed path hands its caller (pixel displacements u, v and the four navigated
    short planes of pix2uv) as float32 <out_dir>/<name>.npy; ny x nx when the scene has at most DUMP_PIXELS pixels,
    else the values at dump_positions(nx, ny).  Collective: every rank calls it with the rows it owns."""
    import numpy as np
    import torch
    nown = planes[0].shape[0]
    idx = dump_positions(nx, ny)
    if idx is None:
        mine = [p.float().cpu().numpy() for p in planes]
    else:
        sel = idx[(idx >= own0 * nx) & (idx < (own0 + nown) * nx)] - own0 * nx
        t = torch.from_numpy(sel).to(planes[0].device)
        mine = [p.reshape(-1).index_select(0, t).float().cpu().numpy() for p in planes]
    parts = [(own0, mine)]
    if dist:
        parts = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
        dist.gather_object((own0, mine), parts, dst=0)
        if dist.get_rank() != 0:
            return
    parts.sort(key=lambda t: t[0])
    os.makedirs(out_dir, exist_ok=True)
    for k, name in enumerate(DUMP_NAMES):
        np.save(os.path.join(out_dir, name + ".npy"), np.concatenate([m[k] for _, m in parts]))


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the flow path
    (oct_patch_match_optical_flow, its -sosm solver, compiled unmodified into
    oracle/_ref/libref_cpu.so) on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nx, ny, sector, _ = WORKLOADS[args.workload]
    import numpy as np

    from concurrent.futures import ThreadPoolExecutor

    import torch

    from octane_b200 import synthetic as S
    from oracle import oracle as O
    size = args.ref_size
    kind = "reference"
    try:
        O.ref_cpu()
        have_ref = True
    except OSError:
        have_ref = False
    if have_ref:
        # The reference's CPU solver is single-threaded code without global state (ctypes releases the GIL
        # around the call), so "all the host threads it can use" = one crop of the scene per host thread,
        # solved concurrently: T windows of size x size spread across a band of rows at the scene centre.
        T = max(1, min(os.cpu_count() or 1, 64, nx // size))
        sy = min(size, ny); sx = min(size, nx)
        r0 = (ny - sy) // 2
        a, b = S.make_pair_torch(nx, ny, args.seed, "cpu", rows=(r0, r0 + sy), limb_taper=False)
        cols = [int(round(k * (nx - sx) / max(T - 1, 1))) for k in range(T)] if T > 1 else [(nx - sx) // 2]
        crops = [(a[:, c:c + sx].contiguous().numpy(), b[:, c:c + sx].contiguous().numpy()) for c in cols]
        del a, b
        n = T * sx * sy
        pool = ThreadPoolExecutor(T)
        fn = lambda: list(pool.map(lambda ab: O.ref_patch_match(ab[0], ab[1]), crops))      # noqa: E731
        what = (f"{T} concurrent {sx}x{sy} crops per step, one per host thread; oct_patch_match_optical_flow rad=2 srad=2 "
                "(reference objects; the code itself is single-threaded)")
        cores = T
        sample = f"{T} x {sx}x{sy} crops across the centre rows"
    else:
        kind = "port"
        i1, i2, c0, r0 = cpu_sample(nx, ny, sector, args.seed, size)
        n = i1.shape[0] * i1.shape[1]
        fn = lambda: O.variational_flow(i1, i2)                # noqa: E731
        what = f"{i1.shape[1]}x{i1.shape[0]} centre crop per step; variational CPU oracle, OpenMP (reference objects absent)"
        cores = os.cpu_count()
        sample = f"{i1.shape[1]}x{i1.shape[0]} centre crop"
    torch.set_num_threads(1)
    for _ in range(args.warmup):
        fn()
    t = time.perf_counter()
    for _ in range(args.steps):
        fn()
    sec = (time.perf_counter() - t) / args.steps
    v = n / sec / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mpix/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.workload} {nx}x{ny}" + (", patch-match solver (-sosm): the reference's only CPU flow path, "
                                   "a different and cheaper algorithm than the variational solve" if have_ref else ""),
                       "sample": sample, "same_algorithm": not have_ref},
            "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": cores, "kind": kind, "sample": what},
            "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "host_cores_available": os.cpu_count()}
    if have_ref:
        line["cpu_stages"] = ref_cpu_stages(args.seed)
    if args.ref_cuda:
        try:
            line["ref_cuda_sm100"] = run_ref_cuda(nx, ny, sector, args.seed)
        except Exception as e:   # no GPU / library absent
            line["ref_cuda_sm100"] = {"unavailable": str(e)[:120]}
    print(json.dumps(line), flush=True)


def ref_cuda_child(args):
    """run_ref_cuda in a child process with a time limit; any failure becomes {"unavailable": why}"""
    import subprocess
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_cuda.so")):
        return {"unavailable": "oracle/_ref/libref_cuda.so not built"}
    try:
        cmd = [sys.executable, os.path.abspath(__file__), "--ref-cuda-only", "--workload", args.workload, "--seed", str(args.seed)]
        if args.size:
            cmd += ["--size", args.size]
        env = dict(os.environ)
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
            env.pop(k, None)
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=180, env=env)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"unavailable": ("exit %d: " % r.returncode) + (r.stderr.strip().splitlines() or r.stdout.strip().splitlines() or ["no output"])[-1][:160]}
        return json.loads(lines[-1])
    except Exception as e:      # timeout, unparsable output, ...
        return {"unavailable": str(e)[:160]}


def ref_cpu_stages(seed):
    """The reference's CPU pyramid / resampling stages (oct_zoom_out = oct_gaussian + oct_bicubic, oct_zoom_in;
    src/oct_zoom.cc:17,154) on the 500 x 500 texture of BASELINE config 1 and on a 2000 x 2000 one: single-threaded
    code, best of 3, one host core."""
    from octane_b200 import synthetic as S
    from oracle import oracle as O
    out = {"cores": 1, "unit": "ms", "what": "reference objects (g++ -O3), best of 3"}
    for n in (500, 2000):
        img = S.make_pair(n, n, seed)[0].astype("float64")
        for f in (0.5, 0.25, 0.125):
            best = min(_timed(lambda: O.ref_zoom_out(img, f)) for _ in range(3))
            out[f"oct_zoom_out_{n}_f{f}"] = round(best * 1e3, 2)
        best = min(_timed(lambda: O.ref_zoom_in(img, 2 * n, 2 * n)) for _ in range(3))
        out[f"oct_zoom_in_{n}_x2"] = round(best * 1e3, 2)
    return out


def _timed(fn):
    t = time.perf_counter()
    fn()
    return time.perf_counter() - t


def batch_arm(args):
    """--workload batch64 (BASELINE config 5): 64 independent 1-minute mesoscale band-13 pairs (500x500, 2 km) with a
    cloud-top-height field and m/s output.  Pairs shard trivially: rank r takes pairs r, r+N, ...; on each GPU
    `--streams` contexts (stream + workspace each) keep that many pairs in flight, because one 500x500 pair is
    launch-latency bound.  No collective on the data path."""
    import numpy as np
    import torch

    import octane_b200 as ob
    from octane_b200 import synthetic as S

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    nx = ny = 500
    npairs = 64
    xs, ys, xo, yo, dt = S.SECTORS["meso_2km"]
    nav = ob.goes_nav(xs, ys, xo, yo)
    p = ob.default_params(doCTH=1)
    mine = list(range(rank, npairs, world))
    K = max(1, min(args.streams, len(mine)))
    ctxs = [ob.Context(local) for _ in range(K)]
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float32)
    cth = torch.from_numpy((7500.0 + 7400.0 * np.sin(xx / 40.0) * np.cos(yy / 30.0)).astype(np.float32)).to(dev)
    pairs = []
    for k in mine:
        a, b = S.make_pair_torch(nx, ny, 100 + k, dev)
        pairs.append((a, b))
    outs = [dict(u=torch.zeros((ny, nx), device=dev), v=torch.zeros((ny, nx), device=dev),
                 s=[torch.zeros((ny, nx), dtype=torch.int16, device=dev) for _ in range(5)]) for _ in mine]
    torch.cuda.synchronize()

    def step():
        for i, (a, b) in enumerate(pairs):
            o = outs[i]
            ctxs[i % K].oct_optical_flow_dev(a, b, nav, 0.0, dt, p, o["u"], o["v"], o["s"][0], o["s"][1], o["s"][2], o["s"][3],
                                             cth=cth, ctp=o["s"][4], sync_torch=False)

    def barrier():
        for c in ctxs:
            c.synchronize()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for c in ctxs:                       # every context's stream starts after e0 ...
            c._after_torch()
        for _ in range(steps):
            fn()
        for c in ctxs:                       # ... and e1 is recorded after all of them
            c._before_torch()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step = timed(step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    launches = sum(int(c.stats().kernel_launches) for c in ctxs) // K * len(mine)
    # end to end: pinned host frames in, U/V/CTP shorts and pixel displacements out, per pair
    hp = [(torch.empty((ny, nx), pin_memory=True).copy_(a), torch.empty((ny, nx), pin_memory=True).copy_(b)) for a, b in pairs]
    ho = [dict(u=torch.empty((ny, nx), pin_memory=True), v=torch.empty((ny, nx), pin_memory=True),
               s=[torch.empty((ny, nx), dtype=torch.int16, pin_memory=True) for _ in range(5)]) for _ in mine]

    def e2e_step():
        for i, (a, b) in enumerate(pairs):
            c = ctxs[i % K]
            with torch.cuda.stream(c._ext_stream()):
                a.copy_(hp[i][0], non_blocking=True); b.copy_(hp[i][1], non_blocking=True)
                o = outs[i]
                c.oct_optical_flow_dev(a, b, nav, 0.0, dt, p, o["u"], o["v"], o["s"][0], o["s"][1], o["s"][2], o["s"][3],
                                       cth=cth, ctp=o["s"][4], sync_torch=False)
                ho[i]["u"].copy_(o["u"], non_blocking=True); ho[i]["v"].copy_(o["v"], non_blocking=True)
                for x, y in zip(ho[i]["s"], o["s"]):
                    x.copy_(y, non_blocking=True)

    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    del hp, ho
    mpix = npairs * nx * ny / 1e6
    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": mpix / (ms_step / 1e3), "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "batch of 64 mesoscale band-13-like pairs 500x500 (2 km) with cloud-top heights, m/s output",
                           "pairs_per_gpu": len(mine), "contexts_per_gpu": K, "parallelism": f"pairs x{world}, no data-path collective",
                           "l2": "a pair's working set fits L2; every step runs all pairs, 200 MB of inputs per GPU"},
                "clocks": clocks, "gpu_launches": launches * args.steps * world,
                "e2e": {"value": mpix / (ms_e2e / 1e3), "unit": "Mpix/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": npairs * 2 * nx * ny * 4, "d2h_bytes_per_step": npairs * nx * ny * (8 + 10),
                        "api": "pinned frames -> octane_optical_flow_dev -> pinned outputs, per pair, contexts in flight"}}
        print(json.dumps(line), flush=True)
    del pairs, outs, cth
    for c in ctxs:
        c.synchronize()
    if dist:
        dist.barrier()
    for c in ctxs:
        c.close()
    if dist:
        dist.destroy_process_group()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="fulldisk", choices=sorted(WORKLOADS) + ["custom", "batch64"])
    ap.add_argument("--streams", type=int, default=8, help="batch64: contexts (pairs in flight) per GPU")
    ap.add_argument("--size", default=None, help="developer: NXxNY scene instead of a named workload (conus sector)")
    ap.add_argument("--seed", type=int, default=4)
    ap.add_argument("--ref-size", type=int, default=1000, help="crop edge of the --impl reference sample")
    ap.add_argument("--ref-cuda", action="store_true", help="also time the reference CUDA build (sm_100 recompile)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-cuda-only", action="store_true", help=argparse.SUPPRESS)   # child process of the baseline leg
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--max-disp", type=int, default=64)
    ap.add_argument("--solver", type=int, default=1, choices=[0, 1],
                    help="PCG kernels of the large levels: 1 merged reduction (default), 0 the reference's loop literally")
    ap.add_argument("--taper", type=int, default=None, help="developer: force the limb taper on (1) / off (0)")
    ap.add_argument("--noise-floor", type=float, default=0.0, help="developer: add uniform noise of this amplitude to both frames")
    ap.add_argument("--empty-cache", action="store_true", help="developer: release torch's cached blocks before the first solve")
    ap.add_argument("--write-digest", action="store_true",
                    help="N = 1: store the strided sample of this run's flow that later runs (any N) are checked against")
    ap.add_argument("--rank-stats", action="store_true",
                    help="developer (N > 1): add every rank's per-stage CUDA-event times of the profiled step to the line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (u, v and the four short planes) as float32 DIR/<name>.npy: "
                         f"whole planes up to {DUMP_PIXELS} pixels, else the same seeded sample of that many pixels every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "batch64"):
        ap.error("--dump-outputs writes the flow workloads of --impl ours")
    if args.size:
        sx, sy = (int(t) for t in args.size.split("x"))
        WORKLOADS["custom"] = (sx, sy, "conus_0.5km", False)
        args.workload = "custom"
    if args.ref_cuda_only:
        nx_, ny_, sector_, _ = WORKLOADS[args.workload]
        print(json.dumps(run_ref_cuda(nx_, ny_, sector_, args.seed)), flush=True)
        return
    if args.impl == "reference":
        if args.workload == "batch64":
            args.workload = "meso500"
        return reference_arm(args)
    if args.workload == "batch64":
        return batch_arm(args)

    import numpy as np
    import torch

    import octane_b200 as ob
    from octane_b200 import synthetic as S

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    nx, ny, sector, taper = WORKLOADS[args.workload]
    if args.taper is not None:
        taper = bool(args.taper)
        if taper:
            sector = "fulldisk_0.5km"
    xs, ys, xo, yo, dt = S.SECTORS[sector]
    p = ob.default_params(max_disp=args.max_disp)
    ctx = ob.Context(local)
    if os.environ.get("OCTANE_NO_GRAPHS"):      # profiling under ncu: plain launches
        ctx.set_graphs(False)
    ctx.set_solver(args.solver)
    if world > 1:
        ids = [ob.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(ids[0], rank, world)
    own0, own1, in0, in1 = ob.band_plan(nx, ny, p, rank, world)
    nav = ob.goes_nav(xs, ys, xo, yo)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr, device=dev)

    # ---- synthetic inputs, resident in HBM (band rows [in0,in1) of the scene)
    img1, img2 = S.make_pair_torch(nx, ny, args.seed, dev, limb_taper=taper, rows=(in0, in1))
    if args.noise_floor > 0:
        g = torch.Generator(device=dev); g.manual_seed(1)
        for im in (img1, img2):
            for j0 in range(0, im.shape[0], 1024):
                blk = im[j0:j0 + 1024]
                blk.add_(torch.rand(blk.shape, device=dev, generator=g) * args.noise_floor)
    if args.empty_cache:
        torch.cuda.empty_cache()
    nown = own1 - own0
    u = torch.zeros((nown, nx), dtype=torch.float32, device=dev)
    v = torch.zeros_like(u)
    shorts = [torch.zeros((nown, nx), dtype=torch.int16, device=dev) for _ in range(4)]
    torch.cuda.synchronize()

    def step():
        if world > 1:
            ctx.oct_variational_optical_flow_band(img1, img2, u, v, nx, ny, p)
            ctx.oct_pix2uv_band(nav, 0.0, dt, u, v, nx, own0, nown, *shorts, p)
        else:
            ctx.oct_variational_optical_flow(img1, img2, u, v, p)
            ctx.oct_pix2uv_cuda(nav, 0.0, dt, u, v, *shorts, p)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if dist:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step = timed(step, args.steps)
    if args.dump_outputs:       # before the profiled step below runs the path again
        dump_outputs(args.dump_outputs, nx, ny, own0, [u, v, *shorts], dist)
    # one more step of the same loop with per-launch CUDA events around the finest level's
    # PCG kernels (that level runs un-graphed for it): the roofline's kernel durations
    ctx.set_profile(True)
    ms_prof = timed(step, 1)
    st = ctx.stats()
    ctx.set_profile(False)
    clocks = sampler.stop() if rank == 0 else None
    launches = int(st.kernel_launches)
    mpix = nx * ny / 1e6

    # ---- end to end through the host-buffer C-ABI entry point (N = 1) or its band equivalent.
    # A function of its own: the pinned buffers must be released while the context's stream is still
    # alive (torch's host allocator records an event on every stream a pinned block was used on).
    def run_e2e():
        """End to end through the C ABI with pinned HOST buffers: every pair's band goes host -> device, its pixel
        displacements (float) and the four short planes come back, all inside the timed region.
        N = 1, `latency`: octane_optical_flow, one blocking call per pair (copy-in, solve, navigation, copy-out in sequence,
        the copy-out of the displacements overlapping the navigation).
        `value`: the pipelined dispatcher octane_stream_submit / octane_stream_wait over the sequence of pairs of the
        timed region -- two pairs in flight, so the copies of pair k+1 and k-1 run under the solve of pair k.  It is the
        loop an archive reprocessing run makes; per-pair latency is reported beside it."""
        nin = in1 - in0
        h1 = torch.empty((nin, nx), dtype=torch.float32, pin_memory=True); h1.copy_(img1)
        h2 = torch.empty((nin, nx), dtype=torch.float32, pin_memory=True); h2.copy_(img2)
        n1, n2 = h1.numpy(), h2.numpy()
        outs = [{k: torch.zeros((nown, nx), dtype=(torch.float32 if k.endswith("Pix") else torch.int16), pin_memory=True).numpy()
                 for k in ("uPix", "vPix", "uVal", "vVal", "uVal2", "vVal2")} for _ in range(2)]
        state = {"k": 0}
        host = {"submit": 0.0, "wait": 0.0, "n": 0}      # host time inside the two calls (ms): submit must not block

        def submit_next():
            k = state["k"]
            t0 = time.perf_counter()
            ctx.stream_submit(k % 2, n1, n2, nav, 0.0, dt, p, outs[k % 2], nx, ny)
            t1 = time.perf_counter()
            if k > 0:
                ctx.stream_wait((k - 1) % 2)
            t2 = time.perf_counter()
            host["submit"] += (t1 - t0) * 1e3; host["wait"] += (t2 - t1) * 1e3; host["n"] += 1
            state["k"] = k + 1

        def drain():
            if state["k"] > 0:
                ctx.stream_wait((state["k"] - 1) % 2)

        def pipelined(steps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                submit_next()
            drain()                               # the last pair's outputs are in host memory
            e1.record(stream)
            barrier()
            ms = e0.elapsed_time(e1)
            if dist:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms / steps

        for _ in range(max(2, min(args.warmup, 3))):
            submit_next()
        drain()
        host.update(submit=0.0, wait=0.0, n=0)
        ms_e2e = pipelined(args.steps)
        # per-pair latency: one pair at a time through the same entry points
        def one():
            ctx.stream_submit(0, n1, n2, nav, 0.0, dt, p, outs[0], nx, ny)
            ctx.stream_wait(0)
        ms_lat = timed(one, min(args.steps, 3))
        res = {"value": mpix / (ms_e2e / 1e3), "unit": "Mpix/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": 2 * nx * nin * 4, "d2h_bytes_per_step": nx * nown * (2 * 4 + 4 * 2),
               "api": "octane_stream_submit / octane_stream_wait (pinned host buffers; two pairs in flight: the copies of one "
                      "pair run under the solve of the other; every pair's H2D and D2H are inside the timed region)",
               "host_ms_in_submit": host["submit"] / max(host["n"], 1), "host_ms_in_wait": host["wait"] / max(host["n"], 1),
               "latency_ms_per_pair": ms_lat, "latency_Mpix/s": mpix / (ms_lat / 1e3),
               "latency_api": "one pair at a time: submit + wait (copy-in, solve, navigation, copy-out in sequence)"}
        if world == 1:
            hs = {k: outs[1][k] for k in ("uVal", "vVal", "uVal2", "vVal2")}

            def blocking():
                ctx.oct_optical_flow(n1, n2, nav, 0.0, dt, p, upix=outs[1]["uPix"], vpix=outs[1]["vPix"], out=hs)

            blocking()
            ms_blk = timed(blocking, min(args.steps, 3))
            res["blocking_call"] = {"api": "octane_optical_flow (host buffers, pinned)", "ms_per_step": ms_blk,
                                    "Mpix/s": mpix / (ms_blk / 1e3)}
        return res

    # the flow of the last timed step, checked against the stored single-GPU digest (every rank contributes its rows)
    check = flow_check(u, v, own0, nx, ny, args.workload, dist, args.write_digest and world == 1)

    e2e = None if args.no_e2e else run_e2e()
    torch.cuda.synchronize()

    def shutdown():
        # every rank's kernels are done before anybody frees memory a neighbour has mapped
        ctx.synchronize()
        if dist:
            dist.barrier()
        ctx.close()
        if dist:
            dist.destroy_process_group()
            # multi-process runs: skip interpreter finalisation, where torch / NCCL / CUDA-IPC objects
            # are torn down in no particular order (seen as "context is destroyed" aborts after the result line)
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(0)

    per_rank = None
    if args.rank_stats and dist:
        # where the scaling loss sits: per-rank stage times and finest-level pass durations of the profiled step
        mine = {"rank": rank, "rows": [own0, own1], "pyramid": st.ms_pyramid, "build": st.ms_build,
                "pcg_pass1": st.ms_pcg_pass1, "pcg_pass2": st.ms_pcg_pass2, "update": st.ms_update, "nav": st.ms_nav,
                "finest_pass1_ms": st.finest_pass1_ms, "finest_pass2_ms": st.finest_pass2_ms}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    if rank != 0:
        del img1, img2, u, v, shorts
        shutdown()
        return

    # ---- roofline of the dominant kernel (finest-level PCG passes, timed live above)
    peak, peak_src = peaks()
    its = list(st.cg_iterations[:st.n_solves])
    fused = int(st.pcg_solver) == 1
    # algorithmic bytes per pixel of the launches the average duration was taken over (the library counts them per
    # launch: which vectors exist yet, whether the constant W / N planes are skipped; DESIGN.md section 4)
    b1 = float(st.finest_pass1_bytes_per_px) or pass1_bytes(its[-3 * p.liters:])
    k1 = b1 * st.finest_pixels / (st.finest_pass1_ms * 1e-3) / 1e9 if st.finest_pass1_ms > 0 else 0.0
    k2 = B_PASS2 * st.finest_pixels / (st.finest_pass2_ms * 1e-3) / 1e9 if st.finest_pass2_ms > 0 else 0.0
    if fused:
        dom = "pcg_fused"          # one kernel per iteration: the library times it in the pass-1 slot
    else:
        dom = "pcg_pass2" if st.ms_pcg_pass2 >= st.ms_pcg_pass1 else "pcg_pass1"
    ach = k2 if dom == "pcg_pass2" else k1
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            # one ncu --set full capture per workload AND rank count (see the file's note); absent -> null
            ent = json.load(f).get(args.workload, {}).get(f"n{world}", {}).get(dom)
        if ent and "ratio_to_algorithmic" in ent:
            traffic = ent["ratio_to_algorithmic"] * (B_PASS2 if dom == "pcg_pass2" else b1) * float(st.finest_pixels)
            traffic_src = f"{ent['capture']}: measured DRAM bytes / algorithmic bytes of the captured launches = {ent['ratio_to_algorithmic']}"
        elif ent:
            traffic, traffic_src = ent["bytes"], ent["capture"]
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": mpix / (ms_step / 1e3), "unit": "Mpix/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload} {nx}x{ny} band-2-like pair, {sector}", "nc": 1, "solver": args.solver,
                   "alpha": p.alpha, "lambda": p.lambda_, "kiters": p.kiters, "liters": p.liters, "cgiters": p.cgiters,
                   "parallelism": f"row bands x{world}" if world > 1 else "single GPU",
                   "l2": "inputs and every level-3 plane are larger than L2 (no flush needed)" if nx * ny * 4 > 130e6
                         else "working set of the coarse levels fits L2; inputs re-read from HBM each step"},
        "clocks": clocks, "gpu_launches": launches * args.steps,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                     "frac": ach / peak, "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu)", "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": (B_PASS2 if dom == "pcg_pass2" else b1) * float(st.finest_pixels),
                     "peak_source": peak_src,
                     "bytes_per_pixel_per_launch": B_PASS2 if dom == "pcg_pass2" else b1,
                     "pixels_per_launch": int(st.finest_pixels),
                     ("fused" if fused else "pass1"): {"GB/s": k1, "avg_ms": st.finest_pass1_ms, "bytes_per_pixel": b1},
                     "pass2": {"GB/s": k2, "avg_ms": st.finest_pass2_ms} if not fused else None,
                     "solver": "merged reduction: one launch per PCG iteration" if fused else "two launches per PCG iteration",
                     "whole_step": {"algorithmic_GB": st.algorithmic_bytes * world / 1e9,
                                    "GB/s_per_gpu": st.algorithmic_bytes / (ms_step * 1e-3) / 1e9,
                                    "frac": st.algorithmic_bytes / (ms_step * 1e-3) / 1e9 / peak}},
        "stage_ms": {"pyramid": st.ms_pyramid, "build": st.ms_build,
                     ("pcg_fused_and_small_pass1" if fused else "pcg_pass1"): st.ms_pcg_pass1,
                     "pcg_pass2": st.ms_pcg_pass2, "update": st.ms_update, "nav": st.ms_nav,
                     "profiled_step_ms": ms_prof,
                     "note": "from one extra step with per-launch events; PCG passes timed at the finest level only"},
        "cg_iterations": {"min": min(its), "max": max(its), "sum": sum(its)},
    }
    if e2e:
        line["e2e"] = e2e
    if check:
        line["check"] = check
    if per_rank:
        line["per_rank_stage_ms"] = per_rank
    if not args.no_cpu_baseline and world == 1:        # the CPU arm is timed at N = 1 only (the other ranks would wait for it)
        line["cpu_baseline"] = run_cpu_port(nx, ny, sector, args.seed)
        # the second baseline BASELINE.json names: the reference's own CUDA build recompiled for sm_100 (oracle/_ref),
        # on a 2000 x 2000 crop, in a child process (the reference exit()s on errors and leaks device memory)
        line["cpu_baseline"]["ref_cuda_sm100"] = ref_cuda_child(args)
        line["ref_cuda_sm100"] = line["cpu_baseline"]["ref_cuda_sm100"]      # same record at top level
    if args.ref_cuda:
        try:
            line["ref_cuda_sm100"] = run_ref_cuda(nx, ny, sector, args.seed)
        except Exception as e:
            line["ref_cuda_sm100"] = {"unavailable": str(e)[:120]}
    print(json.dumps(line), flush=True)
    del img1, img2, u, v, shorts
    shutdown()


if __name__ == "__main__":
    main()
