"""CPU tests of the sequence interface: the workspace arithmetic of octane_batch_workspace_bytes and the host-side
checks of Context.oct_optical_flow_sequence_dev (no device is touched)."""
import numpy as np
import pytest

import octane_b200 as ob


def align(nfloats):
    """arena_layout's allocation unit: 256 bytes"""
    return (nfloats * 4 + 255) // 256 * 256


def planes(nx, ny, nc, p):
    """(P, Pc): the finest plane and the largest coarse plane in floats, rows pitched to 32 columns"""
    dims = ob.level_dims(nx, ny, p)
    pitched = [((a + 31) // 32 * 32) * b for a, b in dims]
    return pitched[-1], max(pitched[:-1], default=0)


def slot_bytes(nx, ny, nc, p):
    """one image slot: the finest image, its coarse-level plane and that level's two gradients (nc planes each)"""
    P, Pc = planes(nx, ny, nc, p)
    return 3 * align(P * nc) + align(Pc * nc)


def state_bytes(nx, ny, nc, p):
    """one pair's state: second derivatives (nc planes each), u, v, ut, vt, the hint planes with a first guess, five
    coefficient planes and ten PCG planes"""
    P, Pc = planes(nx, ny, nc, p)
    hint = 2 * align(P) + 2 * align(Pc) if p.first_guess else 0
    return 3 * align(P * nc) + 2 * align(P) + 2 * align(Pc) + hint + 5 * align(P) + 10 * align(P)


SHAPES = [(500, 500, 1, {}), (2000, 2000, 1, {}), (264, 240, 2, {}), (160, 120, 1, dict(first_guess=1, lambdac=0.5)),
          (768, 640, 1, dict(dosrsal=1, doCTH=1)), (96, 80, 3, dict(kiters=1))]


@pytest.mark.parametrize("nx,ny,nc,over", SHAPES, ids=lambda x: str(x))
def test_sequence_saves_exactly_the_duplicate_image_slots(nx, ny, nc, over):
    p = ob.default_params(**over)
    slot = slot_bytes(nx, ny, nc, p)
    single = ob._lib.load().octane_workspace_bytes(nx, ny, nc, p)
    assert single == 2 * slot + state_bytes(nx, ny, nc, p)
    for n in (1, 2, 7, 64):
        batch = ob.batch_workspace_bytes(n, nx, ny, nc, p)
        seq = ob.batch_workspace_bytes(n, nx, ny, nc, p, sequence=True)
        assert batch > 0 and seq == batch - (n - 1) * slot, (n, batch, seq, slot)


@pytest.mark.parametrize("nx,ny,nc,over", SHAPES, ids=lambda x: str(x))
def test_batch_workspace_is_one_single_pair_workspace_per_pair(nx, ny, nc, over):
    """a batch of N pairs allocates N single-pair workspaces and N pairs' scalars, partials and navigation tables:
    as much as before the workspace was split into image slots and pair states"""
    p = ob.default_params(**over)
    single = ob._lib.load().octane_workspace_bytes(nx, ny, nc, p)
    one = ob.batch_workspace_bytes(1, nx, ny, nc, p)
    extra = one - single
    assert 0 < extra < single
    for n in (2, 7, 64):
        srsal = 2 * align(n * nx * ny) - n * 2 * align(nx * ny) if p.dosrsal else 0
        assert ob.batch_workspace_bytes(n, nx, ny, nc, p) == n * one + srsal


def test_workspace_bytes_refuses_invalid_arguments():
    p = ob.default_params()
    assert ob.batch_workspace_bytes(0, 500, 500, 1, p) == 0
    assert ob.batch_workspace_bytes(0, 500, 500, 1, p, sequence=True) == 0
    assert ob.batch_workspace_bytes(4, 2, 2, 1, p) == 0
    assert ob.batch_workspace_bytes(4, 500, 500, 4, p) == 0


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name}) although the arguments were inconsistent")


def _unbound_context():
    ctx = ob.Context.__new__(ob.Context)
    ctx._L = _NoLibrary()
    ctx._h = None
    return ctx


def test_sequence_wrapper_checks_frames_times_and_navs_first():
    ctx = _unbound_context()
    nav = ob.goes_nav(5.6e-5, -5.6e-5, -0.1, 0.1)
    frames = np.zeros((4, 8, 8), np.float32)
    out = {}
    p = ob.default_params()
    with pytest.raises(ValueError, match="one time per frame"):
        ctx.oct_optical_flow_sequence_dev(frames, [nav] * 3, [0.0, 60.0, 120.0], p, out)
    with pytest.raises(ValueError, match="one time per frame"):
        ctx.oct_optical_flow_sequence_dev(frames, [nav] * 3, [0.0] * 5, p, out)
    with pytest.raises(ValueError, match="one entry per pair"):
        ctx.oct_optical_flow_sequence_dev(frames, [nav] * 4, [0.0] * 4, p, out)
    with pytest.raises(ValueError, match="one entry per pair"):
        ctx.oct_optical_flow_sequence_dev(frames, [nav] * 2, [0.0] * 4, p, out)
    with pytest.raises(TypeError, match="device-pointer"):           # consistent, but host memory
        ctx.oct_optical_flow_sequence_dev(frames, [nav] * 3, [0.0] * 4, p, out)
