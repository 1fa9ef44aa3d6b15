"""Host-side mirror of the reference's operator surface for the hot path.

The reference exposes three C++ functions on this path (no library, no Python):

    oct_variational_optical_flow(Image, Image, float* CTH, float* u, float* v, nx, ny, nc, OFFlags)
        src/oct_variational_optical_flow.cu:1213
    oct_pix2uv_cuda(GOESVar&, double t2, float* u, float* v, short* ur, short* vr,
                    short* ur2, short* vr2, OFFlags)              src/oct_pix2uv_cuda.cu:265
    oct_optical_flow(GOESVar&, GOESVar&, OFFlags&)                src/oct_optical_flow.cc:21

`Context` binds their C-ABI replacements (include/octane_b200.h) with the same
names, argument meaning (u, v are in/out: first guess in, flow out) and error
behaviour turned into exceptions.  numpy arrays go through the host-buffer
entry points (copies inside the call); torch CUDA tensors go through the
device-pointer entry points on the context's stream.  torch is used only for
device memory and process-group bootstrap, never for compute.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from ._lib import Cal, Nav, Params, Stats

ERRORS = {-1: "ENODEV", -2: "EINVAL", -3: "ENOMEM", -4: "ECUDA", -5: "EHALO", -6: "ECOMM"}


class OctaneError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"octane_b200 {ERRORS.get(code, code)}: {msg}")
        self.code = code


def default_params(**kw) -> Params:
    """OFFlags defaults of src/main.cc:53-108, overridable by flag name
    (alpha, lambda_, lambdac, kiters, liters, cgiters, dozim, pixuv, ...)."""
    p = Params()
    _lib.load().octane_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown parameter {k}")
        setattr(p, k, v)
    return p


def goes_nav(xScale, yScale, xOffset, yOffset, pph=35786023.0, req=6378137.0, rpol=6356752.31414,
             lon0_deg=-75.0, minX=0, minY=0, g2xOffset=None, g2yOffset=None) -> Nav:
    lam0 = lon0_deg * (3.14159265 / 180.0)
    return Nav(pph, req, rpol, lam0, xScale, xOffset, yScale, yOffset,
               xOffset if g2xOffset is None else g2xOffset, yOffset if g2yOffset is None else g2yOffset,
               0.0, 0.0, 0.0, 6371000.0, minX, minY)


def band_minmax(band: int):
    """(maxch, minch) radiance range of ABI band 1..16 -- oct_bandminmax, src/oct_normalize_geo.cc:9."""
    L = _lib.load()
    a, b = C.c_float(), C.c_float()
    rc = L.octane_band_minmax(band, C.byref(a), C.byref(b))
    if rc < 0:
        raise OctaneError(rc, L.octane_last_error().decode())
    return a.value, b.value


def goes_cal(radScale, radOffset, band=2, fk1=0.0, fk2=0.0, bc1=0.0, bc2=1.0, kap1=0.0, cal=0, donav=1,
             maxin=None, minin=None) -> Cal:
    """Calibration block as oct_goesread assembles it (src/oct_fileread.cc:341-388): band range from the
    table, output range 0..255, cal "RAW"."""
    mx, mn = band_minmax(band)
    return Cal(radScale, radOffset, fk1, fk2, bc1, bc2, kap1, mx if maxin is None else maxin,
               mn if minin is None else minin, 255.0, 0.0, 0.0, cal, donav)


def level_dims(nx: int, ny: int, p: Optional[Params] = None):
    p = p or default_params()
    L = _lib.load()
    out = []
    for k in range(p.kiters):
        a, b = C.c_int(), C.c_int()
        L.octane_level_dims(nx, ny, C.byref(p), k, C.byref(a), C.byref(b))
        out.append((a.value, b.value))
    return out


def batch_workspace_bytes(npairs: int, nx: int, ny: int, nc: int = 1, p: Optional[Params] = None,
                          sequence: bool = False) -> int:
    """device bytes a batched call (or, with sequence=True, a sequence call) of npairs pairs allocates on a fresh
    context (octane_batch_workspace_bytes); 0 for invalid arguments"""
    p = p or default_params()
    return int(_lib.load().octane_batch_workspace_bytes(npairs, int(sequence), nx, ny, nc, C.byref(p)))


def zoom_out_size(nx: int, ny: int, factor: float):
    """(nxx, nyy) of oct_zoom_size, src/oct_zoom.cc:12"""
    L = _lib.load()
    a, b = C.c_int(), C.c_int()
    rc = L.octane_zoom_out_size(nx, ny, factor, C.byref(a), C.byref(b))
    if rc < 0:
        raise OctaneError(rc, L.octane_last_error().decode())
    return a.value, b.value


def band_plan(nx: int, ny: int, p: Params, rank: int, world: int):
    """(own0, own1, in0, in1): finest rows solved by `rank`, full-res input rows it needs."""
    L = _lib.load()
    v = [C.c_int() for _ in range(4)]
    rc = L.octane_band_plan(nx, ny, C.byref(p), rank, world, *[C.byref(x) for x in v])
    if rc < 0:
        raise OctaneError(rc, L.octane_last_error().decode())
    return tuple(x.value for x in v)


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


_NP = {"float32": np.float32, "int16": np.int16}


def _require(what: str, a, dtype: str, cuda: Optional[bool] = None):
    """The C ABI takes raw pointers: refuse anything that is not a C-contiguous array / tensor of the expected
    element type (a float64 or strided array would be read as garbage, not converted).  cuda=True / False also pins
    where a torch tensor lives (device-pointer vs host-buffer entry points).  None passes (optional arguments)."""
    if a is None:
        return
    if _is_torch(a):
        ok = str(a.dtype) == "torch." + dtype and a.is_contiguous()
        where = "cuda" if a.is_cuda else "cpu"
        if ok and cuda is not None and a.is_cuda != cuda:
            raise TypeError(f"{what}: tensor lives on the {where}, this entry point needs {'CUDA' if cuda else 'host'} memory")
    else:
        ok = isinstance(a, np.ndarray) and a.dtype == _NP[dtype] and a.flags["C_CONTIGUOUS"]
        if ok and cuda:
            raise TypeError(f"{what}: numpy array given to a device-pointer entry point")
    if not ok:
        raise TypeError(f"{what}: expected a C-contiguous {dtype} array, got {type(a).__name__} "
                        f"{getattr(a, 'dtype', '?')}{'' if getattr(a, 'ndim', 0) == 0 else ' (strided?)'}")


def _ptr(x):
    if x is None:
        return None
    if _is_torch(x):
        return C.c_void_p(x.data_ptr())
    return C.c_void_p(x.ctypes.data)


class Context:
    """octane_ctx: a CUDA stream plus a reusable device workspace."""

    def __init__(self, device: int = 0):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.octane_ctx_create(C.byref(h), device)
        if rc < 0:
            raise OctaneError(rc, self._L.octane_last_error().decode())
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._L.octane_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise OctaneError(rc, self._L.octane_last_error().decode())
        return rc

    # ---- knobs / stats
    def set_profile(self, on: bool):
        self._check(self._L.octane_ctx_set_profile(self._h, int(on)))

    def set_graphs(self, on: bool):
        self._check(self._L.octane_ctx_set_graphs(self._h, int(on)))

    def set_solver(self, solver: int):
        """1 (default): merged-reduction PCG kernels on the large levels; 0: the reference's recurrence literally"""
        self._check(self._L.octane_ctx_set_solver(self._h, int(solver)))

    def synchronize(self):
        self._check(self._L.octane_ctx_synchronize(self._h))

    @property
    def stream_ptr(self) -> int:
        """cudaStream_t (as int) that every call of this context is ordered on."""
        return int(self._L.octane_ctx_stream(self._h) or 0)

    def stats(self) -> Stats:
        s = Stats()
        self._check(self._L.octane_get_stats(self._h, C.byref(s)))
        return s

    # ---- multi-GPU bootstrap (one process per GPU)
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        self._check(self._L.octane_comm_init(self._h, unique_id, rank, world))

    @staticmethod
    def comm_unique_id() -> bytes:
        L = _lib.load()
        buf = C.create_string_buffer(128)
        rc = L.octane_comm_unique_id(buf)
        if rc < 0:
            raise OctaneError(rc, L.octane_last_error().decode())
        return buf.raw

    # ---- stream ordering with the host framework (device-pointer entry points only)
    def _ext_stream(self):
        import torch
        if getattr(self, "_ext", None) is None:
            self._ext = torch.cuda.ExternalStream(self.stream_ptr, device=torch.device("cuda", self.device))
        return self._ext

    def _after_torch(self):
        """our stream waits for work already queued on torch's current stream (tensor producers)"""
        import torch
        self._ext_stream().wait_stream(torch.cuda.current_stream(self.device))

    def _before_torch(self):
        """torch's current stream waits for our stream (tensor consumers)"""
        import torch
        torch.cuda.current_stream(self.device).wait_stream(self._ext_stream())

    # ---- the reference's operators
    def oct_variational_optical_flow(self, geo1, geo2, u, v, p: Optional[Params] = None, nc: int = 1):
        """u, v in/out (ny x nx float32).  numpy -> host entry point; torch CUDA -> device entry point."""
        p = p or default_params()
        ny, nx = geo1.shape[-2:]
        dev = _is_torch(geo1)
        for name, a in (("geo1", geo1), ("geo2", geo2), ("u", u), ("v", v)):
            _require(name, a, "float32", cuda=dev)
        if dev:
            fn = self._L.octane_variational_flow_dev
            self._after_torch()
        else:
            fn = self._L.octane_variational_flow
        self._check(fn(self._h, _ptr(geo1), _ptr(geo2), nx, ny, nc, C.byref(p), _ptr(u), _ptr(v)))
        if dev:
            self._before_torch()
        return u, v

    def oct_variational_optical_flow_band(self, geo1_band, geo2_band, u_band, v_band, nx, ny, p: Params, nc: int = 1,
                                          fg_u_band=None, fg_v_band=None):
        """row-band solve (collective).  geo*_band and the optional first guess fg_*_band hold rows [in0,in1) of
        band_plan(); u_band / v_band receive rows [own0,own1)."""
        for name, a in (("geo1_band", geo1_band), ("geo2_band", geo2_band), ("u_band", u_band), ("v_band", v_band),
                        ("fg_u_band", fg_u_band), ("fg_v_band", fg_v_band)):
            _require(name, a, "float32", cuda=True)
        self._after_torch()
        if p.first_guess and fg_u_band is not None:
            self._check(self._L.octane_variational_flow_band_fg_dev(self._h, _ptr(geo1_band), _ptr(geo2_band),
                                                                    _ptr(fg_u_band), _ptr(fg_v_band), nx, ny, nc,
                                                                    C.byref(p), _ptr(u_band), _ptr(v_band)))
        else:
            self._check(self._L.octane_variational_flow_band_dev(self._h, _ptr(geo1_band), _ptr(geo2_band), nx, ny, nc,
                                                                 C.byref(p), _ptr(u_band), _ptr(v_band)))
        self._before_torch()
        return u_band, v_band

    def oct_pix2uv_cuda(self, nav: Nav, t1: float, t2: float, u, v, ur, vr, ur2, vr2, p: Optional[Params] = None):
        """Returns (dT, moved): moved=True when the sector-moved guard zeroed the outputs."""
        p = p or default_params()
        ny, nx = u.shape
        dev = _is_torch(u)
        for name, a in (("u", u), ("v", v)):
            _require(name, a, "float32", cuda=dev)
        for name, a in (("ur", ur), ("vr", vr), ("ur2", ur2), ("vr2", vr2)):
            _require(name, a, "int16", cuda=dev)
        if dev:
            self._after_torch()
            rc = self._check(self._L.octane_pix2uv_dev(self._h, C.byref(nav), t1, t2, _ptr(u), _ptr(v), nx, ny,
                                                       C.byref(p), _ptr(ur), _ptr(vr), _ptr(ur2), _ptr(vr2)))
            self._before_torch()
            return float(np.float32(t2 - t1)), rc == 1
        dT = C.c_float()
        rc = self._check(self._L.octane_pix2uv(self._h, C.byref(nav), t1, t2, _ptr(u), _ptr(v), nx, ny, C.byref(p),
                                               _ptr(ur), _ptr(vr), _ptr(ur2), _ptr(vr2), C.byref(dT)))
        return dT.value, rc == 1

    def oct_pix2uv_band(self, nav: Nav, t1, t2, u, v, nx, row0, nrows, ur, vr, ur2, vr2, p: Params):
        for name, a in (("u", u), ("v", v)):
            _require(name, a, "float32", cuda=True)
        for name, a in (("ur", ur), ("vr", vr), ("ur2", ur2), ("vr2", vr2)):
            _require(name, a, "int16", cuda=True)
        self._after_torch()
        rc = self._check(self._L.octane_pix2uv_band_dev(self._h, C.byref(nav), t1, t2, _ptr(u), _ptr(v), nx, row0,
                                                        nrows, C.byref(p), _ptr(ur), _ptr(vr), _ptr(ur2), _ptr(vr2)))
        self._before_torch()
        return rc

    def oct_srsal_band(self, u_own, v_own, cth_own, nx: int, ny: int):
        """-srsal on row bands (collective), in place on torch CUDA tensors holding the owned rows [own0,own1) of
        band_plan(); cth_own: the same rows of the cloud-top heights.  At world size 1: oct_srsal_cu."""
        for name, a in (("u_own", u_own), ("v_own", v_own), ("cth_own", cth_own)):
            _require(name, a, "float32", cuda=True)
        self._after_torch()
        self._check(self._L.octane_srsal_band_dev(self._h, _ptr(u_own), _ptr(v_own), _ptr(cth_own), nx, ny))
        self._before_torch()
        return u_own, v_own

    def oct_optical_flow(self, geo1, geo2, nav: Nav, t1: float, t2: float, p: Optional[Params] = None,
                         cth=None, upix=None, vpix=None, nc: int = 1, out=None):
        """Dispatcher (host arrays): returns dict(uPix, vPix, uVal, vVal, uVal2, vVal2, CTP, dT).
        `out` may carry preallocated (e.g. pinned) int16 arrays under the same keys."""
        p = p or default_params()
        ny, nx = geo1.shape[-2:]
        upix = np.zeros((ny, nx), np.float32) if upix is None else upix
        vpix = np.zeros((ny, nx), np.float32) if vpix is None else vpix
        out = dict(out) if out else {}
        for k in ("uVal", "vVal", "uVal2", "vVal2"):
            if k not in out:
                out[k] = np.zeros((ny, nx), np.int16)
        ctp = out.get("CTP") if p.doCTH else None
        if p.doCTH and ctp is None:
            ctp = np.zeros((ny, nx), np.int16)
        for name, a in (("geo1", geo1), ("geo2", geo2), ("cth", cth), ("upix", upix), ("vpix", vpix)):
            _require(name, a, "float32", cuda=False)
        for name in ("uVal", "vVal", "uVal2", "vVal2"):
            _require(name, out[name], "int16", cuda=False)
        _require("CTP", ctp, "int16", cuda=False)
        dT = C.c_float()
        self._check(self._L.octane_optical_flow(self._h, _ptr(geo1), _ptr(geo2), _ptr(cth), nx, ny, nc, C.byref(nav),
                                                t1, t2, C.byref(p), _ptr(upix), _ptr(vpix), _ptr(out["uVal"]),
                                                _ptr(out["vVal"]), _ptr(out["uVal2"]), _ptr(out["vVal2"]),
                                                _ptr(ctp), C.byref(dT)))
        out.update(uPix=upix, vPix=vpix, CTP=ctp, dT=dT.value)
        return out

    def oct_optical_flow_dev(self, geo1, geo2, nav: Nav, t1: float, t2: float, p: Params, upix, vpix, ur, vr, ur2, vr2,
                             cth=None, ctp=None, nc: int = 1, sync_torch: bool = True) -> int:
        """Dispatcher on torch CUDA tensors, stream-ordered on the context's stream, no host synchronisation.
        sync_torch=False skips the ordering against torch's current stream (the caller keeps several contexts
        in flight and orders them itself: batch mode)."""
        ny, nx = geo1.shape[-2:]
        for name, a in (("geo1", geo1), ("geo2", geo2), ("cth", cth), ("upix", upix), ("vpix", vpix)):
            _require(name, a, "float32", cuda=True)
        for name, a in (("ur", ur), ("vr", vr), ("ur2", ur2), ("vr2", vr2), ("ctp", ctp)):
            _require(name, a, "int16", cuda=True)
        if sync_torch:
            self._after_torch()
        rc = self._check(self._L.octane_optical_flow_dev(self._h, _ptr(geo1), _ptr(geo2), _ptr(cth), nx, ny, nc, C.byref(nav),
                                                         t1, t2, C.byref(p), _ptr(upix), _ptr(vpix), _ptr(ur), _ptr(vr),
                                                         _ptr(ur2), _ptr(vr2), _ptr(ctp)))
        if sync_torch:
            self._before_torch()
        return rc

    def _batch_args(self, geo1, geo2, nav_list, t1_list, t2_list, out: dict, cth, fg_u=None, fg_v=None):
        """the checks and ctypes arguments both batched calls share: (B, nx, ny, navs, t1, t2, moved)"""
        B = int(geo1.shape[0])
        ny, nx = geo1.shape[-2:]
        for name, a in (("geo1", geo1), ("geo2", geo2), ("cth", cth), ("uPix", out.get("uPix")), ("vPix", out.get("vPix")),
                        ("fg_u", fg_u), ("fg_v", fg_v)):
            _require(name, a, "float32", cuda=True)
        for name in ("uVal", "vVal", "uVal2", "vVal2", "CTP"):
            _require(name, out.get(name), "int16", cuda=True)
        arrays = [a for a in (geo2, cth, fg_u, fg_v, *out.values()) if a is not None]
        shapes = {tuple(a.shape[-2:]) for a in arrays}
        if shapes != {(ny, nx)} or any(int(a.shape[0]) != B for a in arrays):
            raise ValueError("every array must be [B, ny, nx] (images [B, nc, ny, nx]) with the same B, ny, nx")
        if not (len(nav_list) == len(t1_list) == len(t2_list) == B):
            raise ValueError("nav_list, t1_list and t2_list need one entry per pair")
        navs = (Nav * max(B, 1))(*nav_list)
        t1 = (C.c_double * max(B, 1))(*t1_list)
        t2 = (C.c_double * max(B, 1))(*t2_list)
        moved = (C.c_int * max(B, 1))()
        return B, nx, ny, navs, t1, t2, moved

    def oct_optical_flow_batch_dev(self, geo1, geo2, nav_list, t1_list, t2_list, p: Params, out: dict, cth=None,
                                   nc: int = 1):
        """Many same-size pairs in one call, on torch CUDA tensors shaped [B, ny, nx] (or [B, nc, ny, nx] for the
        images).  `out` holds [B, ny, nx] tensors under uPix, vPix (float32), uVal, vVal, uVal2, vVal2 and, with
        doCTH, CTP (int16).  Stream-ordered like oct_optical_flow_dev.  Returns the list of pairs whose sector moved
        (their four navigated planes are zero); cg_iterations() gives the per-pair iteration counts."""
        B, nx, ny, navs, t1, t2, moved = self._batch_args(geo1, geo2, nav_list, t1_list, t2_list, out, cth)
        self._after_torch()
        self._check(self._L.octane_optical_flow_batch_dev(
            self._h, B, _ptr(geo1), _ptr(geo2), _ptr(cth), nx, ny, nc, navs, t1, t2, C.byref(p), _ptr(out["uPix"]),
            _ptr(out["vPix"]), _ptr(out["uVal"]), _ptr(out["vVal"]), _ptr(out["uVal2"]), _ptr(out["vVal2"]),
            _ptr(out.get("CTP")), moved))
        self._before_torch()
        return [b for b in range(B) if moved[b]]

    def oct_optical_flow_batch_ex_dev(self, geo1, geo2, nav_list, t1_list, t2_list, p: Params, out: dict, cth=None,
                                      nc: int = 1, *, fg_u=None, fg_v=None):
        """oct_optical_flow_batch_dev with a first guess (p.first_guess: fg_u / fg_v, [B, ny, nx] float32 CUDA
        tensors, only read; they may be out["uPix"] / out["vPix"]) and -srsal (p.dosrsal: each pair's uPix / vPix
        smoothed with its own heights cth after the navigation).  Returns the list of pairs whose sector moved."""
        B, nx, ny, navs, t1, t2, moved = self._batch_args(geo1, geo2, nav_list, t1_list, t2_list, out, cth, fg_u, fg_v)
        self._after_torch()
        self._check(self._L.octane_optical_flow_batch_ex_dev(
            self._h, B, _ptr(geo1), _ptr(geo2), _ptr(fg_u), _ptr(fg_v), _ptr(cth), nx, ny, nc, navs, t1, t2, C.byref(p),
            _ptr(out["uPix"]), _ptr(out["vPix"]), _ptr(out["uVal"]), _ptr(out["vVal"]), _ptr(out["uVal2"]),
            _ptr(out["vVal2"]), _ptr(out.get("CTP")), moved))
        self._before_torch()
        return [b for b in range(B) if moved[b]]

    def oct_optical_flow_sequence_dev(self, frames, nav_list, t_list, p: Params, out: dict, cth=None, nc: int = 1, *,
                                      fg_u=None, fg_v=None):
        """The consecutive pairs (frames[k], frames[k + 1]) of a sequence of N + 1 frames ([N + 1, ny, nx] or
        [N + 1, nc, ny, nx] float32 CUDA tensor, t_list: N + 1 times, nav_list: N navigations) in one call, each frame
        prepared once.  `out`, cth, fg_u and fg_v are [N, ny, nx] as in oct_optical_flow_batch_ex_dev, whose results
        this gives bit for bit on frames[:-1], frames[1:].  Returns the list of pairs whose sector moved."""
        nframes = int(frames.shape[0])
        if len(t_list) != nframes:
            raise ValueError(f"t_list needs one time per frame: {len(t_list)} for {nframes} frames")
        if len(nav_list) != nframes - 1:
            raise ValueError(f"nav_list needs one entry per pair: {len(nav_list)} for {nframes} frames")
        _require("frames", frames, "float32", cuda=True)
        B, nx, ny, navs, _, _, moved = self._batch_args(frames[:-1], frames[1:], nav_list, t_list[:-1], t_list[1:], out,
                                                        cth, fg_u, fg_v)
        t = (C.c_double * nframes)(*t_list)
        self._after_torch()
        self._check(self._L.octane_optical_flow_sequence_dev(
            self._h, nframes, _ptr(frames), _ptr(fg_u), _ptr(fg_v), _ptr(cth), nx, ny, nc, navs, t, C.byref(p),
            _ptr(out["uPix"]), _ptr(out["vPix"]), _ptr(out["uVal"]), _ptr(out["vVal"]), _ptr(out["uVal2"]),
            _ptr(out["vVal2"]), _ptr(out.get("CTP")), moved))
        self._before_torch()
        return [b for b in range(B) if moved[b]]

    def batch_cg_iterations(self, npairs: int, n_solves: int) -> np.ndarray:
        """[npairs, n_solves] PCG iterations of the last batched call (synchronises the context's stream)"""
        its = np.zeros((npairs, n_solves), np.int32)
        self._check(self._L.octane_batch_cg_iterations(self._h, its.ctypes.data_as(C.POINTER(C.c_int)), npairs))
        return its

    # ---- pipelined dispatcher over a sequence of pairs (host buffers, ideally pinned)
    def stream_submit(self, slot: int, geo1_band, geo2_band, nav: Nav, t1: float, t2: float, p: Params, out: dict,
                      nx: int, ny: int, cth=None, nc: int = 1, *, fg_u_band=None, fg_v_band=None) -> int:
        """enqueue copy-in -> solve -> navigation (-> -srsal) -> copy-out of one pair and return.  geo*_band: rows
        [in0,in1) of band_plan() (the whole scene on one GPU); `out`: host arrays for rows [own0,own1) under the keys
        uVal, vVal, uVal2, vVal2 (int16) and optionally uPix, vPix (float32), CTP (int16).  cth: rows [own0,own1) of the
        cloud-top heights (doCTH, dosrsal; dosrsal also needs uPix / vPix).  fg_u_band / fg_v_band: rows [in0,in1) of a
        first guess (p.first_guess), only read.  The arrays must stay alive and untouched until stream_wait(slot)."""
        for name, a in (("geo1_band", geo1_band), ("geo2_band", geo2_band), ("cth", cth), ("uPix", out.get("uPix")),
                        ("vPix", out.get("vPix")), ("fg_u_band", fg_u_band), ("fg_v_band", fg_v_band)):
            _require(name, a, "float32", cuda=False)
        for name in ("uVal", "vVal", "uVal2", "vVal2"):
            _require(name, out[name], "int16", cuda=False)
        _require("CTP", out.get("CTP"), "int16", cuda=False)
        tail = (nx, ny, nc, C.byref(nav), t1, t2, C.byref(p), _ptr(out.get("uPix")), _ptr(out.get("vPix")),
                _ptr(out["uVal"]), _ptr(out["vVal"]), _ptr(out["uVal2"]), _ptr(out["vVal2"]), _ptr(out.get("CTP")))
        if fg_u_band is not None or fg_v_band is not None:
            return self._check(self._L.octane_stream_submit_fg(self._h, slot, _ptr(geo1_band), _ptr(geo2_band),
                                                               _ptr(fg_u_band), _ptr(fg_v_band), _ptr(cth), *tail))
        return self._check(self._L.octane_stream_submit(self._h, slot, _ptr(geo1_band), _ptr(geo2_band), _ptr(cth), *tail))

    def stream_wait(self, slot: int):
        self._check(self._L.octane_stream_wait(self._h, slot))

    # ---- stage entry points (device pointers; parity tests)
    def stage_blur_decimate(self, d_img, nx, ny, nc, factor, d_out):
        self._after_torch()
        self._check(self._L.octane_stage_blur_decimate(self._h, _ptr(d_img), nx, ny, nc, factor, _ptr(d_out)))
        self._before_torch()

    def stage_gradient(self, d_f, xi, yi, nc, d_gx, d_gy):
        self._after_torch()
        self._check(self._L.octane_stage_gradient(self._h, _ptr(d_f), xi, yi, nc, _ptr(d_gx), _ptr(d_gy)))
        self._before_torch()

    def stage_zoom_in(self, d_flow, nx, ny, nxx, nyy, sf, d_out):
        self._after_torch()
        self._check(self._L.octane_stage_zoom_in(self._h, _ptr(d_flow), nx, ny, nxx, nyy, sf, _ptr(d_out)))
        self._before_torch()

    # ---- ingest (src/oct_navcal_cuda.cu:100) and first-guess conversion (src/oct_pix2uv_cuda.cu:372)
    def oct_navcal_cuda(self, rad, x, y, nav: Nav, cal: Cal, data=None, lat=None, lon=None):
        """rad: ny x nx int16 counts, x: nx, y: ny int16 fixed-grid counts.  numpy in -> numpy out
        (host entry point); torch CUDA tensors -> device entry point.  Returns (data, lat, lon)."""
        ny, nx = rad.shape
        if _is_torch(rad):
            import torch
            mk = lambda: torch.empty((ny, nx), dtype=torch.float32, device=rad.device)   # noqa: E731
            data = mk() if data is None else data
            lat = mk() if lat is None else lat
            lon = mk() if lon is None else lon
            for name, arr in (("rad", rad), ("x", x), ("y", y)):
                _require(name, arr, "int16", cuda=True)
            for name, arr in (("data", data), ("lat", lat), ("lon", lon)):
                _require(name, arr, "float32", cuda=True)
            self._after_torch()
            self._check(self._L.octane_navcal_dev(self._h, _ptr(rad), _ptr(x), _ptr(y), nx, ny, C.byref(nav),
                                                  C.byref(cal), _ptr(data), _ptr(lat), _ptr(lon)))
            self._before_torch()       # the outputs were allocated on torch's stream: order it after our kernel
            return data, lat, lon
        rad = np.ascontiguousarray(rad, np.int16); x = np.ascontiguousarray(x, np.int16); y = np.ascontiguousarray(y, np.int16)
        data = np.empty((ny, nx), np.float32) if data is None else data
        lat = np.empty((ny, nx), np.float32) if lat is None else lat
        lon = np.empty((ny, nx), np.float32) if lon is None else lon
        for name, arr in (("data", data), ("lat", lat), ("lon", lon)):
            _require(name, arr, "float32", cuda=False)
        self._check(self._L.octane_navcal(self._h, _ptr(rad), _ptr(x), _ptr(y), nx, ny, C.byref(nav), C.byref(cal),
                                          _ptr(data), _ptr(lat), _ptr(lon)))
        return data, lat, lon

    def oct_navcal_grid(self, grid: int, data, x, y, nav: Nav, donav: int = 1):
        """ingest of a -Polar (grid 1) / -Merc (grid 2) file: oct_polar_navcal_cuda / oct_merc_navcal_cuda.
        Returns (data, lat, lon)."""
        data = np.ascontiguousarray(data, np.float32); x = np.ascontiguousarray(x, np.int16); y = np.ascontiguousarray(y, np.int16)
        ny, nx = data.shape
        out = np.empty((ny, nx), np.float32); lat = np.empty((ny, nx), np.float32); lon = np.empty((ny, nx), np.float32)
        self._check(self._L.octane_navcal_grid(self._h, grid, _ptr(data), _ptr(x), _ptr(y), nx, ny, C.byref(nav), donav,
                                               _ptr(out), _ptr(lat), _ptr(lon)))
        return out, lat, lon

    def oct_zoom_in_float(self, field, nxx: int, nyy: int, interp: int = 1):
        """regrid a coarser field onto an nyy x nxx grid (oct_zoom_in_float, src/oct_zoom.cc:180)"""
        ny, nx = field.shape
        if _is_torch(field):
            import torch
            _require("field", field, "float32", cuda=True)
            out = torch.empty((nyy, nxx), dtype=torch.float32, device=field.device)
            self._after_torch()
            self._check(self._L.octane_zoom_in_float_dev(self._h, _ptr(field), nx, ny, _ptr(out), nxx, nyy, interp))
            self._before_torch()
            return out
        field = np.ascontiguousarray(field, np.float32)
        out = np.empty((nyy, nxx), np.float32)
        self._check(self._L.octane_zoom_in_float(self._h, _ptr(field), nx, ny, _ptr(out), nxx, nyy, interp))
        return out

    def oct_zoom_out_float(self, field, factor: float):
        """regrid a FINER field down by `factor` <= 1 (oct_zoom_out_float, src/oct_zoom.cc:51); the output is
        the dense (nyy, nxx) plane of zoom_out_size"""
        ny, nx = field.shape
        nxx, nyy = zoom_out_size(nx, ny, factor)
        if _is_torch(field):
            import torch
            _require("field", field, "float32", cuda=True)
            out = torch.empty((nyy, nxx), dtype=torch.float32, device=field.device)
            self._after_torch()
            self._check(self._L.octane_zoom_out_float_dev(self._h, _ptr(field), nx, ny, _ptr(out), factor))
            self._before_torch()
            return out
        field = np.ascontiguousarray(field, np.float32)
        out = np.empty((nyy, nxx), np.float32)
        self._check(self._L.octane_zoom_out_float(self._h, _ptr(field), nx, ny, _ptr(out), factor))
        return out

    def oct_srsal_cu(self, upix, vpix, cth):
        """-srsal bilateral post-smoother, in place on upix / vpix (oct_srsal_cu, src/oct_srsal_cuda.cu:73)"""
        ny, nx = upix.shape
        dev = _is_torch(upix)
        _require("upix", upix, "float32", cuda=dev)
        _require("vpix", vpix, "float32", cuda=dev)
        if dev:
            _require("cth", cth, "float32", cuda=True)
            self._after_torch()
            self._check(self._L.octane_srsal_dev(self._h, _ptr(upix), _ptr(vpix), _ptr(cth), nx, ny))
            self._before_torch()
            return upix, vpix
        cth = np.ascontiguousarray(cth, np.float32)
        self._check(self._L.octane_srsal(self._h, _ptr(upix), _ptr(vpix), _ptr(cth), nx, ny))
        return upix, vpix

    def oct_uv2pix(self, nav: Nav, t1: float, t2: float, lat, lon, x, y, u, v, p: Optional[Params] = None) -> int:
        """u, v: first-guess winds (m/s) in, pixel displacements out (in place).  Returns 1 when the
        sector-moved guard zeroed them."""
        p = p or default_params()
        ny, nx = u.shape
        dev = _is_torch(u)
        for name, arr in (("lat", lat), ("lon", lon), ("u", u), ("v", v)):
            _require(name, arr, "float32", cuda=dev)
        for name, arr in (("x", x), ("y", y)):
            _require(name, arr, "int16", cuda=dev)
        if dev:
            self._after_torch()
            rc = self._check(self._L.octane_uv2pix_dev(self._h, C.byref(nav), t1, t2, _ptr(lat), _ptr(lon), _ptr(x),
                                                       _ptr(y), nx, ny, C.byref(p), _ptr(u), _ptr(v)))
            self._before_torch()
            return rc
        return self._check(self._L.octane_uv2pix(self._h, C.byref(nav), t1, t2, _ptr(lat), _ptr(lon), _ptr(x), _ptr(y),
                                                 nx, ny, C.byref(p), _ptr(u), _ptr(v)))

    def stage_build(self, d_u, d_v, d_uh, d_vh, d_g1, d_g2, xi, yi, nc, p, lambdac, gnc, d_coef, d_bu, d_bv):
        self._after_torch()
        self._check(self._L.octane_stage_build(self._h, _ptr(d_u), _ptr(d_v), _ptr(d_uh), _ptr(d_vh), _ptr(d_g1),
                                               _ptr(d_g2), xi, yi, nc, C.byref(p), lambdac, gnc, _ptr(d_coef),
                                               _ptr(d_bu), _ptr(d_bv)))
        self._before_torch()

    def stage_pcg(self, d_coef, d_bu, d_bv, xi, yi, iters, tol, d_xu, d_xv) -> int:
        its = C.c_int()
        self._after_torch()
        self._check(self._L.octane_stage_pcg(self._h, _ptr(d_coef), _ptr(d_bu), _ptr(d_bv), xi, yi, iters, tol,
                                             _ptr(d_xu), _ptr(d_xv), C.byref(its)))
        self._before_torch()
        return its.value
