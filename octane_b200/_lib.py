"""ctypes binding of liboctane_b200.so (include/octane_b200.h).

The library is the product; this module only loads it.  There is no Python or
CPU fallback: if the shared object is missing the import of any compute entry
point raises, and without a CUDA device `Context()` raises OctaneError(ENODEV).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# OCTANE_B200_LIB: load another build of the same C ABI (A/B comparisons of kernel revisions)
LIB_PATH = os.environ.get("OCTANE_B200_LIB") or os.path.join(HERE, "lib", "liboctane_b200.so")

OCTANE_MAX_SOLVES = 256
EXPECTED_ABI = 3          # include/octane_b200.h: OCTANE_ABI_VERSION the struct mirrors below were written against


class Params(C.Structure):
    """octane_params: the OFFlags fields the path reads (reference include/offlags.h:4-72)."""
    _fields_ = [("alpha", C.c_double), ("lambda_", C.c_double), ("lambdac", C.c_double),
                ("scaleF", C.c_double), ("scsig", C.c_double),
                ("kiters", C.c_int), ("liters", C.c_int), ("cgiters", C.c_int), ("dozim", C.c_int),
                ("setdevice", C.c_int), ("pixuv", C.c_int), ("dopolar", C.c_int), ("domerc", C.c_int),
                ("first_guess", C.c_int), ("max_disp", C.c_int), ("doCTH", C.c_int), ("ir", C.c_int),
                ("dosrsal", C.c_int)]


class Nav(C.Structure):
    """octane_nav: GOESNAVVar subset (reference include/goesread.h:3-14)."""
    _fields_ = [("pph", C.c_double), ("req", C.c_double), ("rpol", C.c_double), ("lam0", C.c_double),
                ("xScale", C.c_float), ("xOffset", C.c_float), ("yScale", C.c_float), ("yOffset", C.c_float),
                ("g2xOffset", C.c_float), ("g2yOffset", C.c_float),
                ("lat1", C.c_float), ("lon1", C.c_float), ("lon0", C.c_float), ("R", C.c_float),
                ("minX", C.c_int), ("minY", C.c_int)]


class Cal(C.Structure):
    """octane_cal: the scalar arguments of oct_navcal_cuda (reference src/oct_navcal_cuda.cu:100-107)."""
    _fields_ = [("radScale", C.c_float), ("radOffset", C.c_float),
                ("fk1", C.c_float), ("fk2", C.c_float), ("bc1", C.c_float), ("bc2", C.c_float), ("kap1", C.c_float),
                ("maxin", C.c_float), ("minin", C.c_float), ("maxout", C.c_float), ("minout", C.c_float),
                ("H", C.c_float), ("cal", C.c_int), ("donav", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("n_levels", C.c_int), ("n_solves", C.c_int),
                ("level_nx", C.c_int * 16), ("level_ny", C.c_int * 16),
                ("cg_iterations", C.c_int * OCTANE_MAX_SOLVES),
                ("kernel_launches", C.c_longlong), ("algorithmic_bytes", C.c_double),
                ("ms_total", C.c_double), ("ms_pyramid", C.c_double), ("ms_build", C.c_double),
                ("ms_pcg_pass1", C.c_double), ("ms_pcg_pass2", C.c_double), ("ms_update", C.c_double),
                ("ms_nav", C.c_double), ("n_pcg_pass1", C.c_longlong), ("n_pcg_pass2", C.c_longlong),
                ("finest_pass1_ms", C.c_double), ("finest_pass2_ms", C.c_double),
                ("finest_pixels", C.c_longlong), ("pcg_solver", C.c_int), ("finest_pass1_bytes_per_px", C.c_double)]


# every symbol include/octane_b200.h declares (tests check the library exports them all)
EXPORTS = [
    "octane_abi_version", "octane_last_error", "octane_device_count", "octane_params_default",
    "octane_ctx_create", "octane_ctx_destroy", "octane_ctx_set_profile", "octane_ctx_set_graphs", "octane_ctx_set_solver",
    "octane_get_stats", "octane_ctx_synchronize", "octane_ctx_stream", "octane_workspace_bytes", "octane_level_dims",
    "octane_variational_flow", "octane_pix2uv", "octane_optical_flow",
    "octane_variational_flow_dev", "octane_pix2uv_dev", "octane_optical_flow_dev",
    "octane_navcal", "octane_navcal_dev", "octane_band_minmax", "octane_uv2pix", "octane_uv2pix_dev",
    "octane_zoom_in_float", "octane_zoom_in_float_dev", "octane_navcal_grid",
    "octane_zoom_out_size", "octane_zoom_out_float", "octane_zoom_out_float_dev", "octane_srsal", "octane_srsal_dev",
    "octane_stage_blur_decimate", "octane_stage_gradient", "octane_stage_zoom_in",
    "octane_stage_build", "octane_stage_pcg",
    "octane_band_plan", "octane_comm_unique_id", "octane_comm_init", "octane_comm_rank",
    "octane_variational_flow_band_dev", "octane_variational_flow_band_fg_dev", "octane_pix2uv_band_dev",
    "octane_srsal_band_dev", "octane_stream_submit", "octane_stream_submit_fg", "octane_stream_wait",
    "octane_optical_flow_batch_dev", "octane_optical_flow_batch_ex_dev", "octane_batch_cg_iterations",
    "octane_optical_flow_sequence_dev", "octane_batch_workspace_bytes",
]

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(octane_b200 has no fallback path)")
    L = C.CDLL(LIB_PATH)
    L.octane_abi_version.restype = C.c_int
    if L.octane_abi_version() != EXPECTED_ABI:
        # a library and mirror that disagree would read / write past the ctypes structs silently
        raise ImportError(f"{LIB_PATH} has ABI version {L.octane_abi_version()}, this package mirrors version {EXPECTED_ABI}")
    vp, ip, fp = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float)
    PP, NP = C.POINTER(Params), C.POINTER(Nav)
    i, d, f = C.c_int, C.c_double, C.c_float
    L.octane_abi_version.restype = i
    L.octane_last_error.restype = C.c_char_p
    L.octane_device_count.restype = i
    L.octane_params_default.argtypes = [PP]
    L.octane_params_default.restype = None
    L.octane_ctx_create.argtypes = [C.POINTER(vp), i]
    L.octane_ctx_destroy.argtypes = [vp]
    L.octane_ctx_destroy.restype = None
    L.octane_ctx_set_profile.argtypes = [vp, i]
    L.octane_ctx_set_graphs.argtypes = [vp, i]
    L.octane_ctx_set_solver.argtypes = [vp, i]
    L.octane_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.octane_ctx_synchronize.argtypes = [vp]
    L.octane_ctx_stream.argtypes = [vp]
    L.octane_ctx_stream.restype = vp
    L.octane_workspace_bytes.argtypes = [i, i, i, PP]
    L.octane_workspace_bytes.restype = C.c_size_t
    L.octane_level_dims.argtypes = [i, i, PP, i, ip, ip]
    L.octane_variational_flow.argtypes = [vp, vp, vp, i, i, i, PP, vp, vp]
    L.octane_pix2uv.argtypes = [vp, NP, d, d, vp, vp, i, i, PP, vp, vp, vp, vp, fp]
    L.octane_optical_flow.argtypes = [vp, vp, vp, vp, i, i, i, NP, d, d, PP, vp, vp, vp, vp, vp, vp, vp, fp]
    L.octane_variational_flow_dev.argtypes = [vp, vp, vp, i, i, i, PP, vp, vp]
    L.octane_pix2uv_dev.argtypes = [vp, NP, d, d, vp, vp, i, i, PP, vp, vp, vp, vp]
    L.octane_optical_flow_dev.argtypes = [vp, vp, vp, vp, i, i, i, NP, d, d, PP, vp, vp, vp, vp, vp, vp, vp]
    L.octane_optical_flow_batch_dev.argtypes = [vp, i, vp, vp, vp, i, i, i, NP, C.POINTER(d), C.POINTER(d), PP,
                                                vp, vp, vp, vp, vp, vp, vp, ip]
    L.octane_optical_flow_batch_ex_dev.argtypes = [vp, i, vp, vp, vp, vp, vp, i, i, i, NP, C.POINTER(d), C.POINTER(d),
                                                   PP, vp, vp, vp, vp, vp, vp, vp, ip]
    L.octane_batch_cg_iterations.argtypes = [vp, ip, i]
    L.octane_optical_flow_sequence_dev.argtypes = [vp, i, vp, vp, vp, vp, i, i, i, NP, C.POINTER(d), PP,
                                                   vp, vp, vp, vp, vp, vp, vp, ip]
    L.octane_batch_workspace_bytes.argtypes = [i, i, i, i, i, PP]
    L.octane_batch_workspace_bytes.restype = C.c_size_t
    CP = C.POINTER(Cal)
    L.octane_navcal.argtypes = [vp, vp, vp, vp, i, i, NP, CP, vp, vp, vp]
    L.octane_navcal_dev.argtypes = [vp, vp, vp, vp, i, i, NP, CP, vp, vp, vp]
    L.octane_band_minmax.argtypes = [i, fp, fp]
    L.octane_uv2pix.argtypes = [vp, NP, d, d, vp, vp, vp, vp, i, i, PP, vp, vp]
    L.octane_uv2pix_dev.argtypes = [vp, NP, d, d, vp, vp, vp, vp, i, i, PP, vp, vp]
    L.octane_navcal_grid.argtypes = [vp, i, vp, vp, vp, i, i, NP, i, vp, vp, vp]
    L.octane_zoom_in_float.argtypes = [vp, vp, i, i, vp, i, i, i]
    L.octane_zoom_in_float_dev.argtypes = [vp, vp, i, i, vp, i, i, i]
    L.octane_zoom_out_size.argtypes = [i, i, d, ip, ip]
    L.octane_zoom_out_float.argtypes = [vp, vp, i, i, vp, d]
    L.octane_zoom_out_float_dev.argtypes = [vp, vp, i, i, vp, d]
    L.octane_srsal.argtypes = [vp, vp, vp, vp, i, i]
    L.octane_srsal_dev.argtypes = [vp, vp, vp, vp, i, i]
    L.octane_stage_blur_decimate.argtypes = [vp, vp, i, i, i, f, vp]
    L.octane_stage_gradient.argtypes = [vp, vp, i, i, i, vp, vp]
    L.octane_stage_zoom_in.argtypes = [vp, vp, i, i, i, i, f, vp]
    L.octane_stage_build.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, PP, f, i, vp, vp, vp]
    L.octane_stage_pcg.argtypes = [vp, vp, vp, vp, i, i, i, f, vp, vp, ip]
    L.octane_band_plan.argtypes = [i, i, PP, i, i, ip, ip, ip, ip]
    L.octane_comm_unique_id.argtypes = [C.c_char_p]
    L.octane_comm_init.argtypes = [vp, C.c_char_p, i, i]
    L.octane_comm_rank.argtypes = [vp, ip, ip]
    L.octane_variational_flow_band_dev.argtypes = [vp, vp, vp, i, i, i, PP, vp, vp]
    L.octane_variational_flow_band_fg_dev.argtypes = [vp, vp, vp, vp, vp, i, i, i, PP, vp, vp]
    L.octane_pix2uv_band_dev.argtypes = [vp, NP, d, d, vp, vp, i, i, i, PP, vp, vp, vp, vp]
    L.octane_srsal_band_dev.argtypes = [vp, vp, vp, vp, i, i]
    L.octane_stream_submit.argtypes = [vp, i, vp, vp, vp, i, i, i, NP, d, d, PP, vp, vp, vp, vp, vp, vp, vp]
    L.octane_stream_submit_fg.argtypes = [vp, i, vp, vp, vp, vp, vp, i, i, i, NP, d, d, PP, vp, vp, vp, vp, vp, vp, vp]
    L.octane_stream_wait.argtypes = [vp, i]
    _lib = L
    return L
