"""CPU tests (no GPU) of the two stages either side of the flow path that SURVEY section 8f row N4 names:
the regridding of a FINER field (oct_zoom_out_float, reference src/oct_zoom.cc:51) and the -srsal
post-smoother (oct_srsal_cu, reference src/oct_srsal_cuda.cu:73).

oct_zoom_out_float is CPU code in the reference: the oracle is pinned bit for bit on the reference's own
object (oracle/_ref/libref_cpu.so, built from the sources where they lie) or, without it, on stored values of
its output (tests/golden/zoomout_ref.npz; make_golden.py zoomout says how they were written).  oct_srsal_cu is a
CUDA kernel:
the oracle is pinned on fixtures the reference produced on a B200 (tests/golden/srsal_*.npz) and on an
independent numpy evaluation of the case where the filter degenerates to a plain Gaussian."""
import numpy as np
import pytest

import cases
import octane_b200 as ob
from conftest import load_golden


def _ref_or_skip(oracle):
    try:
        return oracle.ref_cpu()
    except OSError:
        pytest.skip("oracle/_ref/libref_cpu.so not built (reference tree absent at build time)")


@pytest.mark.parametrize("name", sorted(cases.ZOOMOUT))
def test_zoom_out_oracle_is_bit_identical_to_reference(oracle, name):
    field, factor = cases.zoomout_input(name)
    want = cases.zoomout_reference(oracle, name, field, factor)
    got = oracle.zoom_out_float(field, factor)
    assert got.shape == want.shape
    assert np.array_equal(got, want)
    ny, nx = field.shape
    assert got.shape == (int(ny * factor + 0.5), int(nx * factor + 0.5))
    assert ob.api.zoom_out_size(nx, ny, factor) == (got.shape[1], got.shape[0])      # host side of the C ABI


def test_zoom_out_reference_channel_offset_is_an_element_offset(oracle):
    """src/oct_zoom.cc:84 stores pixel k of channel `cnum` at imageout[k + cnum] (not + cnum * plane):
    the C ABI returns the dense plane and leaves its placement to the caller."""
    _ref_or_skip(oracle)
    field, factor = cases.zoomout_input("half")
    plane = oracle.zoom_out_float(field, factor)
    raw = oracle.ref_zoom_out_float(field, factor, cnum=2)
    assert np.array_equal(raw[2:], plane.ravel()) and np.all(raw[:2] == 0)


def test_zoom_out_integer_ratio_is_blur_then_decimation(oracle):
    """at integer ratios the bicubic is evaluated at integer coordinates and returns the blurred pixel itself"""
    field, _ = cases.zoomout_input("quarter")
    out = oracle.zoom_out_float(field, 0.25)
    smooth = oracle.zoom_out_float(np.full_like(field, 123.25), 0.25)
    # the taps are normalised over 2R+1 but the +R one is dropped: a constant comes out scaled by the same
    # factor at every pixel, twice (two passes)
    assert np.ptp(smooth) == 0 and 0.9 < smooth[0, 0] / 123.25 < 1.0
    assert out.shape == (30, 40) and np.isfinite(out).all()


@pytest.mark.parametrize("factor", [0.5, 0.25, 0.125])
def test_zoom_out_equals_the_reference_cpu_pyramid_stage_on_config_1(oracle, factor):
    """BASELINE config 1 (500 x 500 cloud texture through the reference's CPU pyramid / zoom): oct_zoom_out (double,
    src/oct_zoom.cc:17) and oct_zoom_out_float are the same arithmetic; on float input the float restatement is the
    double result rounded once"""
    from octane_b200 import synthetic as S
    i1, _, _, _ = S.make_pair(500, 500, seed=1, kind="shift", drift=(2.0, -1.0))
    want = cases.zoomout_reference(oracle, f"config1_{factor}", i1, factor, pyramid=True)
    got = oracle.zoom_out_float(i1, factor)
    assert got.shape == (int(500 * factor + 0.5),) * 2 and np.array_equal(got, want)


def _reflect(x, n):
    x = np.where(x < 0, -x, x)
    return np.where(x >= n, n - (x - n + 1), x)


def _gauss_numpy(f, R=18, sigma=9.0):
    ny, nx = f.shape
    k = np.arange(-R, R + 1, dtype=np.float64)
    w = np.exp(-(k * k) / (2 * sigma * sigma))
    w /= w.sum()
    f = f.astype(np.float64)
    ix = _reflect(np.arange(nx)[:, None] + k[None, :].astype(int), nx)      # (nx, 37)
    iy = _reflect(np.arange(ny)[:, None] + k[None, :].astype(int), ny)
    h = (f[:, ix] * w).sum(-1)                                               # along x
    return (h[iy, :] * w[None, :, None]).sum(1)                              # along y


def test_srsal_with_flat_heights_is_the_truncated_gaussian(oracle):
    c = cases.SRSAL["srsal_70x50_flat"]
    u, v, cth = cases.srsal_inputs(c)
    us, vs = oracle.srsal(u, v, cth)
    assert np.abs(us - _gauss_numpy(u)).max() < 2e-6 and np.abs(vs - _gauss_numpy(v)).max() < 2e-6
    assert not np.shares_memory(us, u) and np.abs(us - u).mean() > 0.05      # it did smooth


def test_srsal_keeps_constants_and_respects_cloud_edges(oracle):
    c = cases.SRSAL["srsal_96x80_deck"]
    u, v, cth = cases.srsal_inputs(c)
    one = np.full_like(u, 3.5)
    us, vs = oracle.srsal(one, -one, cth)
    assert np.abs(us - 3.5).max() < 1e-6 and np.abs(vs + 3.5).max() < 1e-6
    # a flow that differs between the tower (cth + 9000) and the deck is not mixed across the edge:
    # exp(-(9000^2)/800) underflows to zero
    tower = cth > 8000
    assert 100 < tower.sum() < tower.size - 100
    step = np.where(tower, 5.0, -5.0).astype(np.float32)
    us, _ = oracle.srsal(step, step, cth)
    assert np.abs(us[tower] - 5.0).max() < 1e-5 and np.abs(us[~tower] + 5.0).max() < 1e-5


def test_srsal_rejects_scenes_smaller_than_the_window(oracle):
    L = oracle.lib()
    import ctypes as C
    a = np.zeros((18, 40), np.float32)
    L.oracle_srsal.argtypes = [np.ctypeslib.ndpointer(np.float32)] * 3 + [C.c_int, C.c_int]
    assert L.oracle_srsal(a, a.copy(), a.copy(), 40, 18) != 0


@pytest.mark.parametrize("name", sorted(cases.SRSAL))
def test_srsal_oracle_matches_reference_fixture(oracle, name):
    g = load_golden(name)
    u, v, cth = cases.srsal_inputs(cases.SRSAL[name])
    us, vs = oracle.srsal(u, v, cth)
    # double accumulation narrowed to float: identical up to the last float bit (libm exp vs CUDA exp)
    np.testing.assert_allclose(us, g["u"], rtol=3e-7, atol=1e-7)
    np.testing.assert_allclose(vs, g["v"], rtol=3e-7, atol=1e-7)
