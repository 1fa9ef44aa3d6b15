"""bench.py contract pieces that run without a GPU: the reference arm (`--impl reference`, the reference's own CPU
flow solver from oracle/_ref on the host cores) prints one JSON line with the agreed keys; ranks other than 0 print
nothing and exit 0; the arguments bench.py refuses.  On a GPU: what --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, *args):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                           "--ref-size", "200", "--workload", "meso", *args], capture_output=True, text=True, timeout=600, env=env)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "flow Mpix/s" and d["unit"] == "Mpix/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    if cb["kind"] == "reference":      # the reference's CPU pyramid stages are timed beside its solver
        st = d["cpu_stages"]
        assert st["cores"] == 1 and st["oct_zoom_out_500_f0.5"] > 0 and st["oct_zoom_in_2000_x2"] > st["oct_zoom_in_500_x2"]


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_positions_are_a_fixed_sample():
    import bench
    assert bench.dump_positions(2000, 1000) is None                  # 2 Mpix: written whole
    nx, ny = 21696, 21696
    idx = bench.dump_positions(nx, ny)
    assert idx.shape == (bench.DUMP_PIXELS,) and idx[0] >= 0 and idx[-1] < nx * ny
    assert (np.diff(idx) > 0).all()                                  # ascending, no pixel twice
    assert np.array_equal(idx, bench.dump_positions(nx, ny))
    assert 4 * bench.DUMP_PIXELS * len(bench.DUMP_NAMES) <= 64 << 20


def test_bench_refuses_bad_step_counts_and_dumps_it_cannot_make(tmp_path):
    r = _run(None, "--steps", "0")
    assert r.returncode != 0 and "--steps" in r.stderr
    r = _run(None, "--dump-outputs", str(tmp_path))
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dumped_outputs_are_what_the_path_computes(tmp_path):
    """--dump-outputs on a scene above DUMP_PIXELS (sampled) against the same pair solved directly through the library"""
    import torch

    import bench
    import octane_b200 as ob
    from octane_b200 import synthetic as S
    nx, ny = 2100, 1000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", f"{nx}x{ny}", "--steps", "2", "--warmup", "1",
                        "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {k: np.load(tmp_path / f"{k}.npy") for k in bench.DUMP_NAMES}
    assert sorted(os.listdir(tmp_path)) == sorted(f"{k}.npy" for k in bench.DUMP_NAMES)
    assert all(a.dtype == np.float32 and a.shape == (bench.DUMP_PIXELS,) for a in got.values())

    xs, ys, xo, yo, dt = S.SECTORS["conus_0.5km"]
    ctx = ob.Context(0)
    ctx.set_solver(1)
    p = ob.default_params(max_disp=64)
    img1, img2 = S.make_pair_torch(nx, ny, 4, "cuda")
    u = torch.zeros((ny, nx), device="cuda"); v = torch.zeros_like(u)
    shorts = [torch.zeros((ny, nx), dtype=torch.int16, device="cuda") for _ in range(4)]
    ctx.oct_variational_optical_flow(img1, img2, u, v, p)
    ctx.oct_pix2uv_cuda(ob.goes_nav(xs, ys, xo, yo), 0.0, dt, u, v, *shorts, p)
    ctx.synchronize()
    idx = torch.from_numpy(bench.dump_positions(nx, ny)).cuda()
    want = dict(zip(bench.DUMP_NAMES, (t.reshape(-1).index_select(0, idx).float().cpu().numpy() for t in [u, v, *shorts])))
    ctx.close()
    for k in ("uPix", "vPix"):
        d = np.abs(got[k] - want[k])
        assert d.mean() <= 1e-3 and d.max() <= 1e-2, (k, d.mean(), d.max())
    for k in ("uVal", "vVal", "uVal2", "vVal2"):
        assert np.abs(got[k] - want[k]).max() <= 1, k
