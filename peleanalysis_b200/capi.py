"""ctypes binding of the C ABI (include/pele_stencil_b200.h) -- the same calls a C++ host shell makes.

No compute happens in Python and nothing here falls back to a CPU path: if the CUDA library is missing or no
device is usable the calls raise PaError.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libpelestencil_b200.so")


class PaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("pa error %d: %s" % (code, msg))
        self.code = code


class LevelDesc(C.Structure):
    _fields_ = [("domain_lo", C.c_int * 3), ("domain_hi", C.c_int * 3), ("dx", C.c_double * 3),
                ("nboxes", C.c_int), ("boxes", C.POINTER(C.c_int)), ("owner", C.POINTER(C.c_int))]


class CurvOpts(C.Structure):
    _fields_ = [("prog_min", C.c_double), ("prog_max", C.c_double), ("do_threshold", C.c_int),
                ("threshold", C.c_double), ("do_gauss", C.c_int), ("do_strain", C.c_int),
                ("get_strain_tensor", C.c_int), ("do_velnormal", C.c_int), ("reserved", C.c_int * 8)]


class SmoothOpts(C.Structure):
    """pa_smooth_opts: smoothing_time (>= 0), tol_rel (0 = 1e-10), max_iter (0 = 1000), precond (PA_SMOOTH_PRECOND_*, 0 = Jacobi)."""
    _fields_ = [("smoothing_time", C.c_double), ("tol_rel", C.c_double), ("max_iter", C.c_int), ("precond", C.c_int),
                ("reserved", C.c_int * 7)]


PA_ERR_UNSUPPORTED, PA_ERR_NOCONV = -4, -6
PA_SMOOTH_PRECOND_JACOBI, PA_SMOOTH_PRECOND_MG = 0, 1
SMOOTH_PRECONDS = {"jacobi": PA_SMOOTH_PRECOND_JACOBI, "mg": PA_SMOOTH_PRECOND_MG}


# every symbol include/pele_stencil_b200.h declares: (restype, argtypes)
_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
SYMBOLS = {
    "pa_init": (_i, [_i]), "pa_finalize": (_i, []), "pa_last_error": (C.c_char_p, []), "pa_version": (C.c_char_p, []),
    "pa_set_stream": (_i, [_vp]), "pa_sync": (_i, []),
    "pa_host_alloc": (_i, [C.POINTER(_vp), C.c_size_t]), "pa_host_free": (_i, [_vp]),
    "pa_host_register": (_i, [_vp, C.c_size_t]), "pa_host_unregister": (_i, [_vp]),
    "pa_hier_create": (_i, [C.POINTER(_vp), _i, C.POINTER(LevelDesc), C.POINTER(_i), C.POINTER(_i), _i, _i]),
    "pa_hier_create2": (_i, [C.POINTER(_vp), _i, C.POINTER(LevelDesc), C.POINTER(_i), C.POINTER(_i), _i, _i, C.c_uint]),
    "pa_field_ipc_handle": (_i, [_vp, _i, _vp]), "pa_field_map_peer": (_i, [_vp, _i, _i, _vp]),
    "pa_enable_peer_access": (_i, [_i]), "pa_field_slab": (_i, [_vp, _i, C.POINTER(_vp)]),
    "pa_field_map_peer_ptr": (_i, [_vp, _i, _i, _vp]), "pa_copy_async": (_i, [_vp, _vp, _i64]),
    "pa_hier_destroy": (_i, [_vp]), "pa_hier_num_levels": (_i, [_vp]), "pa_hier_num_boxes": (_i, [_vp, _i]),
    "pa_hier_num_cells": (_i64, [_vp, _i]), "pa_hier_num_local_cells": (_i64, [_vp, _i]),
    "pa_hier_box_owner": (_i, [_vp, _i, _i]),
    "pa_sfc_distribute": (_i, [_i, C.POINTER(_i), _i, C.POINTER(_i)]),
    "pa_field_alloc": (_i, [_vp, _i, _i, C.POINTER(_vp)]), "pa_field_free": (_i, [_vp]),
    "pa_field_ncomp": (_i, [_vp]), "pa_field_nghost": (_i, [_vp]), "pa_field_bytes": (_i64, [_vp]),
    "pa_field_upload": (_i, [_vp, _i, _i, _i, _vp]), "pa_field_download": (_i, [_vp, _i, _i, _i, _vp]),
    "pa_field_upload_level": (_i, [_vp, _i, _i, _vp]), "pa_field_download_level": (_i, [_vp, _i, _i, _vp]),
    "pa_field_set_val": (_i, [_vp, _i, _i, _d]),
    "pa_field_hash": (_i, [_vp, _i, _i, C.POINTER(C.c_uint64)]),
    "pa_fill_boundary": (_i, [_vp, _i, _i, _i]), "pa_fill_ghosts": (_i, [_vp, _i, _i, _i, _i]),
    "pa_grad": (_i, [_vp, _i, _i, _vp, _i]), "pa_grad_phases": (_i, [_vp, _i, _i, _vp, _i, _i]),
    "pa_curvature": (_i, [_vp, _i, _i, C.POINTER(CurvOpts), _vp, _i]),
    "pa_curvature_num_outputs": (_i, [C.POINTER(CurvOpts)]),
    "pa_debug_selftest_math": (C.c_int64, [C.c_int64, C.c_uint64]),
    "pa_debug_normal_math": (C.c_int, []),
    "pa_debug_curv_fused": (C.c_int, [_vp]),
    "pa_debug_curv_fused_launches": (C.c_int64, []),
    "pa_curvature_phases": (_i, [_vp, _i, _i, C.POINTER(CurvOpts), _vp, _i, _i]),
    "pa_curvature_steps": (_i, [_vp, _i, _i, C.POINTER(CurvOpts), _vp, _i, _i, _i, _i]),
    "pa_curvature_scratch": (_i, [_vp, _i, C.POINTER(_vp)]),
    "pa_exchange_counts": (_i, [_vp, _i, _i, C.POINTER(_i64), C.POINTER(_i64)]),
    "pa_exchange_buffers": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64)]),
    "pa_exchange_pack": (_i, [_vp, _i, _i]), "pa_exchange_mark_received": (_i, [_vp, _i, _i]),
    "pa_kernel_launches": (_i64, []), "pa_hier_build_seconds": (_i, [_vp, C.POINTER(_d)]),
    "pa_debug_device_bytes": (_i, [C.POINTER(_i64)]),
    "pa_algorithmic_bytes": (_i64, [_vp, _i]),
    "pa_debug_download_grown": (_i, [_vp, _i, _i, _i, _vp]),
    "pa_debug_fb_source_map": (_i, [_vp, _i, _i, _i, _vp, _i64]),
    "pa_debug_face_flags": (_i64, [_vp, _i, _i, _i, _vp, _i64]),
    "pa_debug_exchange_ids": (_i64, [_vp, _i, _vp, _i64]),
    "pa_debug_links": (_i, [_vp, _i, _i, C.POINTER(_i)]),
    "pa_debug_face_coef": (_i, [_vp, _i, _i, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_d)]),
    "pa_debug_fp64_rate": (_i, [C.POINTER(_d)]),
    "pa_filter_weights": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_d), _i]),
    "pa_boxes_max_size": (_i, [_i, C.POINTER(_i), _i, C.POINTER(_i), _i]),
    "pa_fill_patch": (_i, [_vp, _i, _i, _i, _i, _i]),
    "pa_fill_patch_exchange_buffers": (_i, [_vp, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64)]),
    "pa_fill_patch_pack": (_i, [_vp, _i, _i, _i, _i, _i]), "pa_fill_patch_mark_received": (_i, [_vp, _i, _i, _i, _i, _i]),
    "pa_debug_fill_patch_exchange_ids": (_i64, [_vp, _i, _i, _i, _i, _vp, _i64]),
    "pa_filter": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i]),
    "pa_smooth": (_i, [_vp, _i, _d, _d, C.POINTER(SmoothOpts), _vp, _i, _i, C.POINTER(_i), C.POINTER(_d)]),
    "pa_debug_smooth_vcycle": (_i, [_vp, _i, _d, _d, C.POINTER(SmoothOpts), _vp, _i, _i, _i, C.POINTER(_d), C.POINTER(_i)]),
}

_lib = None


def lib():
    """Load the CUDA library.  Raises if it has not been built (python -m peleanalysis_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PaError(-2, "CUDA library %s is missing: run __graft_entry__.build() (there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise PaError(code, lib().pa_last_error().decode())


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def init(device: int = 0) -> None:
    check(lib().pa_init(device))


def set_stream(stream_ptr: int) -> None:
    check(lib().pa_set_stream(C.c_void_p(stream_ptr)))


def sync() -> None:
    check(lib().pa_sync())


def kernel_launches() -> int:
    return int(lib().pa_kernel_launches())


def device_bytes() -> int:
    """Device memory the library holds on the current device (pa_debug_device_bytes)."""
    v = _i64()
    check(lib().pa_debug_device_bytes(C.byref(v)))
    return int(v.value)


def curv_fused_launches() -> int:
    return int(lib().pa_debug_curv_fused_launches())


def sfc_distribute(boxes: Sequence[tuple], nranks: int) -> np.ndarray:
    bx = np.array([list(lo) + list(hi) for lo, hi in boxes], dtype=np.int32)
    out = np.zeros(len(boxes), dtype=np.int32)
    check(lib().pa_sfc_distribute(len(boxes), bx.ctypes.data_as(C.POINTER(C.c_int)), nranks, out.ctypes.data_as(C.POINTER(C.c_int))))
    return out


class PinnedArray:
    """float64 numpy view over cudaHostAlloc'ed memory."""

    def __init__(self, n: int):
        self.ptr = C.c_void_p()
        self.n = int(n)
        check(lib().pa_host_alloc(C.byref(self.ptr), max(self.n, 1) * 8))
        buf = (C.c_double * max(self.n, 1)).from_address(self.ptr.value)
        self.array = np.frombuffer(buf, dtype=np.float64, count=self.n)

    def free(self):
        if self.ptr:
            self.array = None
            lib().pa_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Hierarchy:
    """Geometry + BoxArray + DistributionMapping of all levels and the descriptor tables built from them."""

    def __init__(self, levels, is_per=(1, 1, 1), sym_dir=(0, 0, 0), rank: int = 0, nranks: int = 1,
                 owners: Optional[List[np.ndarray]] = None, flags: int = 0):
        """levels: objects with domain_lo, domain_hi, dx, boxes (e.g. plotfile.Level)."""
        self.levels = levels
        self.rank, self.nranks = rank, nranks
        nlev = len(levels)
        descs = (LevelDesc * nlev)()
        self._keep = []
        self.owners = []
        for l, lv in enumerate(levels):
            d = descs[l]
            d.domain_lo[:] = list(lv.domain_lo)
            d.domain_hi[:] = list(lv.domain_hi)
            d.dx[:] = list(lv.dx)
            bx = np.ascontiguousarray([list(lo) + list(hi) for lo, hi in lv.boxes], dtype=np.int32)
            d.nboxes = len(lv.boxes)
            d.boxes = bx.ctypes.data_as(C.POINTER(C.c_int))
            if owners is not None:
                ow = np.ascontiguousarray(owners[l], dtype=np.int32)
            elif nranks > 1:
                ow = sfc_distribute(lv.boxes, nranks)
            else:
                ow = np.zeros(len(lv.boxes), dtype=np.int32)
            d.owner = ow.ctypes.data_as(C.POINTER(C.c_int))
            self._keep += [bx, ow]
            self.owners.append(ow)
        per = (C.c_int * 3)(*[int(v) for v in is_per])
        bck = (C.c_int * 3)(*[int(v) for v in sym_dir])
        self.h = C.c_void_p()
        self.flags = flags
        check(lib().pa_hier_create2(C.byref(self.h), nlev, descs, per, bck, rank, nranks, flags))
        self.nlev = nlev
        self.local_boxes = [[b for b in range(len(lv.boxes)) if self.owners[l][b] == rank] for l, lv in enumerate(levels)]
        self.local_cells = [sum(int(np.prod([hi[d] - lo[d] + 1 for d in range(3)])) for b in self.local_boxes[l]
                                for lo, hi in [lv.boxes[b]]) for l, lv in enumerate(levels)]

    def __del__(self):
        try:
            if self.h:
                lib().pa_hier_destroy(self.h)
                self.h = None
        except Exception:
            pass

    @property
    def num_cells(self) -> int:
        return int(lib().pa_hier_num_cells(self.h, -1))

    @property
    def num_local_cells(self) -> int:
        return int(lib().pa_hier_num_local_cells(self.h, -1))

    @property
    def build_seconds(self) -> float:
        s = C.c_double()
        check(lib().pa_hier_build_seconds(self.h, C.byref(s)))
        return s.value

    def algorithmic_bytes(self, nout: int) -> int:
        return int(lib().pa_algorithmic_bytes(self.h, nout))

    # ---- debug / parity tables -----------------------------------------------------------------------
    def fb_source_map(self, lev: int, ng: int = 1, cross: bool = True):
        lv = self.levels[lev]
        sizes = [int(np.prod([hi[d] - lo[d] + 1 + 2 * ng for d in range(3)])) for b in self.local_boxes[lev] for lo, hi in [lv.boxes[b]]]
        out = np.empty(sum(sizes), dtype=np.int64)
        check(lib().pa_debug_fb_source_map(self.h, lev, ng, int(cross), _ptr(out), out.size))
        res, o = [], 0
        for b, m in zip(self.local_boxes[lev], sizes):
            lo, hi = lv.boxes[b]
            n = [hi[d] - lo[d] + 1 + 2 * ng for d in range(3)]
            res.append(out[o:o + m].reshape(n[2], n[1], n[0]))
            o += m
        return res

    def exchange_ids(self, which: int) -> np.ndarray:
        n = lib().pa_debug_exchange_ids(self.h, which, None, 0)
        out = np.empty(n, dtype=np.int64)
        lib().pa_debug_exchange_ids(self.h, which, _ptr(out) if n else None, n)
        return out

    def fill_patch_exchange_ids(self, lev: int, nghost: int, interp_type: int, which: int) -> np.ndarray:
        """pa_fill_patch's exchange plan: identity of the cell in every send- (which=0) / recv-slab (1) slot."""
        n = lib().pa_debug_fill_patch_exchange_ids(self.h, lev, nghost, interp_type, which, None, 0)
        if n < 0:
            check(int(n))
        out = np.empty(n, dtype=np.int64)
        lib().pa_debug_fill_patch_exchange_ids(self.h, lev, nghost, interp_type, which, _ptr(out) if n else None, n)
        return out

    def exchange_prefix(self, ncomp: int = 1):
        """(send_counts, recv_counts) per peer, in doubles for ncomp components."""
        s = (C.c_int64 * self.nranks)()
        r = (C.c_int64 * self.nranks)()
        check(lib().pa_exchange_counts(self.h, 1, ncomp, s, r))
        return np.array(list(s)), np.array(list(r))

    def face_flags(self, lev: int, box: int, face: int):
        n = lib().pa_debug_face_flags(self.h, lev, box, face, None, 0)
        if n <= 0:
            return None
        out = np.empty(n, dtype=np.uint16)
        lib().pa_debug_face_flags(self.h, lev, box, face, _ptr(out), n)
        lo, hi = self.levels[lev].boxes[box]
        d = face % 3
        t1 = 1 if d == 0 else 0
        t2 = 1 if d == 2 else 2
        return out.reshape(hi[t2] - lo[t2] + 1, hi[t1] - lo[t1] + 1)

    def links(self, lev: int, box: int) -> np.ndarray:
        """[6,5] ints per face: neighbour global box (-1 = no link), its owner rank, rel[3]."""
        out = np.zeros(30, dtype=np.int32)
        check(lib().pa_debug_links(self.h, lev, box, out.ctypes.data_as(C.POINTER(C.c_int))))
        return out.reshape(6, 5)

    def face_coef(self, lev: int, box: int, face: int):
        kind, nx = C.c_int(), C.c_int()
        coef = (C.c_double * 4)()
        check(lib().pa_debug_face_coef(self.h, lev, box, face, C.byref(kind), C.byref(nx), coef))
        return kind.value, nx.value, list(coef)


class Field:
    """Device-resident MultiFab: ncomp components with nghost ghost layers on every level of a Hierarchy."""

    def __init__(self, hier: Hierarchy, ncomp: int, nghost: int):
        self.hier = hier
        self.ncomp, self.nghost = ncomp, nghost
        self.f = C.c_void_p()
        check(lib().pa_field_alloc(hier.h, ncomp, nghost, C.byref(self.f)))

    def free(self):
        if self.f:
            lib().pa_field_free(self.f)
            self.f = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @property
    def nbytes(self) -> int:
        return int(lib().pa_field_bytes(self.f))

    def upload_level(self, lev: int, comp: int, host: np.ndarray) -> None:
        """host: this rank's boxes of the level concatenated (float64, C-contiguous; pinned for async DMA)."""
        assert host.dtype == np.float64 and host.flags.c_contiguous and host.size == self.hier.local_cells[lev]
        check(lib().pa_field_upload_level(self.f, lev, comp, _ptr(host)))

    def download_level(self, lev: int, comp: int, host: np.ndarray) -> None:
        assert host.dtype == np.float64 and host.flags.c_contiguous and host.size == self.hier.local_cells[lev]
        check(lib().pa_field_download_level(self.f, lev, comp, _ptr(host)))

    def upload_box(self, lev: int, box: int, comp: int, host: np.ndarray) -> None:
        host = np.ascontiguousarray(host, dtype=np.float64)
        check(lib().pa_field_upload(self.f, lev, box, comp, _ptr(host)))
        sync()

    def download_box(self, lev: int, box: int, comp: int) -> np.ndarray:
        lo, hi = self.hier.levels[lev].boxes[box]
        out = np.empty((hi[2] - lo[2] + 1, hi[1] - lo[1] + 1, hi[0] - lo[0] + 1))
        check(lib().pa_field_download(self.f, lev, box, comp, _ptr(out)))
        sync()
        return out

    def download_grown(self, lev: int, box: int, comp: int) -> np.ndarray:
        lo, hi = self.hier.levels[lev].boxes[box]
        g = self.nghost
        out = np.empty((hi[2] - lo[2] + 1 + 2 * g, hi[1] - lo[1] + 1 + 2 * g, hi[0] - lo[0] + 1 + 2 * g))
        check(lib().pa_debug_download_grown(self.f, lev, box, comp, _ptr(out)))
        return out

    def upload_fabs(self, comp: int, fabs_per_level: List[List[np.ndarray]]) -> None:
        """fabs_per_level[l][b]: [nz,ny,nx] array of GLOBAL box b (only this rank's boxes are read)."""
        for l, fabs in enumerate(fabs_per_level):
            if not self.hier.local_boxes[l]:
                continue
            host = np.concatenate([np.ascontiguousarray(fabs[b], dtype=np.float64).ravel() for b in self.hier.local_boxes[l]])
            self.upload_level(l, comp, host)
            sync()

    def download_fabs(self, comp: int) -> List[List[Optional[np.ndarray]]]:
        out = []
        for l, lv in enumerate(self.hier.levels):
            res: List[Optional[np.ndarray]] = [None] * len(lv.boxes)
            if self.hier.local_boxes[l]:
                host = np.empty(self.hier.local_cells[l])
                self.download_level(l, comp, host)
                sync()
                o = 0
                for b in self.hier.local_boxes[l]:
                    lo, hi = lv.boxes[b]
                    n = [hi[d] - lo[d] + 1 for d in range(3)]
                    m = n[0] * n[1] * n[2]
                    res[b] = host[o:o + m].reshape(n[2], n[1], n[0])
                    o += m
            out.append(res)
        return out

    def ipc_handles(self) -> bytes:
        """64-byte CUDA IPC handle of every level's slab, concatenated (zeros where this rank owns no box)."""
        buf = (C.c_ubyte * (64 * self.hier.nlev))()
        for l in range(self.hier.nlev):
            check(lib().pa_field_ipc_handle(self.f, l, C.byref(buf, 64 * l)))
        return bytes(buf)

    def map_peer(self, peer_rank: int, handles: bytes) -> None:
        for l in range(self.hier.nlev):
            h = (C.c_ubyte * 64).from_buffer_copy(handles[64 * l:64 * l + 64])
            check(lib().pa_field_map_peer(self.f, l, peer_rank, h))

    def set_val(self, v: float, comp: int = 0, ncomp: Optional[int] = None) -> None:
        check(lib().pa_field_set_val(self.f, comp, ncomp or self.ncomp - comp, v))

    def hash(self, comp: int = 0, ncomp: Optional[int] = None) -> int:
        """Order-independent fingerprint of this rank's valid cells (pa_field_hash); add the ranks' values mod 2^64."""
        v = C.c_uint64(0)
        check(lib().pa_field_hash(self.f, comp, ncomp or self.ncomp - comp, C.byref(v)))
        return int(v.value)

    def fill_boundary(self, comp: int = 0, ncomp: int = 1, cross: bool = False) -> None:
        check(lib().pa_fill_boundary(self.f, comp, ncomp, int(cross)))

    def fill_ghosts(self, comp: int = 0, ncomp: int = 1, lev_lo: int = 0, lev_hi: int = -1) -> None:
        check(lib().pa_fill_ghosts(self.f, comp, ncomp, lev_lo, lev_hi))


PEER_LINKS, NO_LINKS, FILTER_ONLY = 1, 2, 4


def grad(inp: Field, comp_in: int, nvar: int, out: Field, comp_out: int, phases: int = 3) -> None:
    check(lib().pa_grad_phases(inp.f, comp_in, nvar, out.f, comp_out, phases))


def curvature(state: Field, comp_S: int, comp_vel: int, opts: CurvOpts, out: Field, comp_out: int = 0) -> None:
    check(lib().pa_curvature(state.f, comp_S, comp_vel, C.byref(opts), out.f, comp_out))


def curvature_phases(state: Field, comp_S: int, comp_vel: int, opts: CurvOpts, out: Field, comp_out: int, phases: int) -> None:
    check(lib().pa_curvature_phases(state.f, comp_S, comp_vel, C.byref(opts), out.f, comp_out, phases))


CURV_PASS1, CURV_DIV, CURV_GAUSS, CURV_STRAIN, CURV_VELN, CURV_CLIP = 1, 2, 4, 8, 16, 32


def curvature_steps(state: Field, comp_S: int, comp_vel: int, opts: CurvOpts, out: Field, comp_out: int, steps: int,
                    lev_lo: int = -1, lev_hi: int = -1) -> None:
    check(lib().pa_curvature_steps(state.f, comp_S, comp_vel, C.byref(opts), out.f, comp_out, steps, lev_lo, lev_hi))


class ScratchField(Field):
    """The curvature tool's internal un-normalised gradient field (owned by the hierarchy: never freed from here)."""

    def __init__(self, hier: Hierarchy, which: int = 0):
        self.hier = hier
        self.ncomp, self.nghost = 3, 1
        self.f = C.c_void_p()
        check(lib().pa_curvature_scratch(hier.h, which, C.byref(self.f)))

    def free(self):
        self.f = None


# ---- filterPlt path (Src/filterPlt.cpp): one Python call per C entry point
def filter_weights(filter_type: int, fgr: int):
    """(ngrow, weights) of Filter(filter_type, fgr)."""
    n = lib().pa_filter_weights(filter_type, fgr, None, None, 0)
    if n < 0:
        check(n)
    w = np.zeros(n)
    ng = C.c_int(0)
    n2 = lib().pa_filter_weights(filter_type, fgr, C.byref(ng), w.ctypes.data_as(C.POINTER(C.c_double)), n)
    if n2 < 0:
        check(n2)
    return int(ng.value), w


def boxes_max_size(boxes: Sequence[tuple], max_grid_size: int) -> List[tuple]:
    """BoxArray::maxSize on [(lo, hi), ...]."""
    bx = np.array([list(lo) + list(hi) for lo, hi in boxes], dtype=np.int32).reshape(-1, 6)
    p = bx.ctypes.data_as(C.POINTER(C.c_int))
    n = lib().pa_boxes_max_size(len(boxes), p, max_grid_size, None, 0)
    if n < 0:
        check(n)
    out = np.zeros((n, 6), dtype=np.int32)
    n2 = lib().pa_boxes_max_size(len(boxes), p, max_grid_size, out.ctypes.data_as(C.POINTER(C.c_int)), n)
    if n2 < 0:
        check(n2)
    return [(tuple(int(v) for v in b[:3]), tuple(int(v) for v in b[3:])) for b in out]


def fp64_rate_gops() -> float:
    """measured FP64 rate for separate multiplies and adds (no FMA), Gop/s"""
    v = C.c_double(0.0)
    check(lib().pa_debug_fp64_rate(C.byref(v)))
    return float(v.value)


def fill_patch(f: Field, comp: int, ncomp: int, lev: int, nghost: int, interp_type: int = 1) -> None:
    check(lib().pa_fill_patch(f.f, comp, ncomp, lev, nghost, interp_type))


def fill_patch_exchange_buffers(f: Field, ncomp: int, lev: int, nghost: int, interp_type: int = 1):
    """(send slab pointer, recv slab pointer, send offsets, recv offsets) of pa_fill_patch's exchange, offsets in doubles"""
    n = f.hier.nranks
    sp, rp = C.c_void_p(), C.c_void_p()
    so, ro = (C.c_int64 * (n + 1))(), (C.c_int64 * (n + 1))()
    check(lib().pa_fill_patch_exchange_buffers(f.f, ncomp, lev, nghost, interp_type, C.byref(sp), C.byref(rp), so, ro))
    return sp.value, rp.value, list(so), list(ro)


def fill_patch_pack(f: Field, comp: int, ncomp: int, lev: int, nghost: int, interp_type: int = 1) -> None:
    check(lib().pa_fill_patch_pack(f.f, comp, ncomp, lev, nghost, interp_type))


def fill_patch_mark_received(f: Field, comp: int, ncomp: int, lev: int, nghost: int, interp_type: int = 1) -> None:
    check(lib().pa_fill_patch_mark_received(f.f, comp, ncomp, lev, nghost, interp_type))


def filter_level(inp: Field, comp_in: int, out: Field, comp_out: int, ncomp: int, lev: int, filter_type: int, fgr: int) -> None:
    check(lib().pa_filter(inp.f, comp_in, out.f, comp_out, ncomp, lev, filter_type, fgr))


def smooth(state: Field, comp_S: int, prog_min: float, prog_max: float, opts: SmoothOpts, out: Field, comp_c: int, comp_phi: int):
    """curvature's do_smooth (curvature.cpp:328-406): c = (S - prog_min) / (prog_max - prog_min) into out[comp_c], the solution
    phi of phi - smoothing_time * div(grad phi) = c on the composite hierarchy into out[comp_phi].  Returns (iterations,
    relative residual); raises PaError (code PA_ERR_NOCONV) if the solve does not converge."""
    it, res = C.c_int(0), C.c_double(0.0)
    check(lib().pa_smooth(state.f, comp_S, prog_min, prog_max, C.byref(opts), out.f, comp_c, comp_phi, C.byref(it), C.byref(res)))
    return it.value, res.value


def smooth_precond(name: str) -> int:
    """PA_SMOOTH_PRECOND_* of a preconditioner name ("jacobi" or "mg"); ValueError for any other name"""
    if name not in SMOOTH_PRECONDS:
        raise ValueError("smooth_precond must be one of %s (got %r)" % ("|".join(SMOOTH_PRECONDS), name))
    return SMOOTH_PRECONDS[name]


def debug_smooth_vcycle(state: Field, comp_S: int, prog_min: float, prog_max: float, opts: SmoothOpts, out: Field, comp_c: int,
                        comp_phi: int, ncycles: int):
    """pa_debug_smooth_vcycle: ncycles steps of phi <- phi + B (c - A phi) from phi = c, B one V-cycle of pa_smooth's multigrid
    preconditioner.  Returns (relative residuals: [0] before the first step, [n] after step n; number of MG levels of level 0)."""
    res = np.zeros(max(ncycles, 0) + 1, dtype=np.float64)
    nmg = C.c_int(0)
    check(lib().pa_debug_smooth_vcycle(state.f, comp_S, prog_min, prog_max, C.byref(opts), out.f, comp_c, comp_phi, ncycles,
                                       res.ctypes.data_as(C.POINTER(C.c_double)), C.byref(nmg)))
    return res, nmg.value


def curvature_num_outputs(opts: CurvOpts) -> int:
    return int(lib().pa_curvature_num_outputs(C.byref(opts)))
