"""One-process-per-GPU plumbing above the C ABI: torch.distributed moves what has to move between processes --
CUDA-IPC handles once per field (peer links), and the packed ghost slabs of whatever is NOT peer-linked per fill.
No compute happens here."""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import capi


class _DevArray:
    """Raw device pointer -> torch tensor (via __cuda_array_interface__)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<f8", "data": (int(ptr), False), "version": 2}


def _wrap_device(ptr: int, n: int) -> torch.Tensor:
    """The library's send / recv slab (a raw device pointer) as a CUDA tensor NCCL can send from / receive into."""
    return torch.as_tensor(_DevArray(ptr, n), device="cuda")


def map_peers(field: capi.Field) -> None:
    """Collective: every rank maps every other rank's slabs of `field` (PA_HIER_PEER_LINKS hierarchies)."""
    H = field.hier
    if H.nranks == 1 or getattr(field, "_peers_mapped", False):
        return
    field._peers_mapped = True
    mine = field.ipc_handles()
    got = [None] * H.nranks
    dist.all_gather_object(got, mine)
    for r, h in enumerate(got):
        if r != H.rank:
            field.map_peer(r, h)
    dist.barrier()


def stream_barrier() -> None:
    """Cross-rank ordering point on the current CUDA stream without a host sync: a 1-element all-reduce.  Peers'
    writes enqueued before it are visible to kernels this rank enqueues after it."""
    if dist.is_initialized() and dist.get_world_size() > 1:
        t = torch.zeros(1, device="cuda")
        dist.all_reduce(t)


class SlabExchange:
    """NCCL send/recv of the packed ghost slabs for ncomp components of one field (everything the neighbour links do
    not cover: ragged same-level neighbours and coarse cells of coarse-fine faces owned by other ranks)."""

    def __init__(self, field: capi.Field, ncomp: int, wrap=_wrap_device):
        """wrap(ptr, n): raw slab pointer -> tensor for the process group's backend (CUDA tensors for NCCL)."""
        H = field.hier
        self.field, self.ncomp, self.rank, self.world = field, ncomp, H.rank, H.nranks
        self.soff = self.roff = [0]
        self.empty = True
        if self.world == 1:
            return
        sp, rp = C.c_void_p(), C.c_void_p()
        so = (C.c_int64 * (self.world + 1))()
        ro = (C.c_int64 * (self.world + 1))()
        capi.check(capi.lib().pa_exchange_buffers(field.f, ncomp, C.byref(sp), C.byref(rp), so, ro))
        self.soff, self.roff = list(so), list(ro)
        self.send_t = wrap(sp.value, max(self.soff[-1], 1))
        self.recv_t = wrap(rp.value, max(self.roff[-1], 1))
        # a rank with nothing to send or receive still takes part if any peer does (batch_isend_irecv is pairwise)
        self.empty = (self.soff[-1] == 0 and self.roff[-1] == 0)

    def run(self, comp: int = 0) -> None:
        if self.world == 1 or self.empty:
            return
        f = self.field
        capi.check(capi.lib().pa_exchange_pack(f.f, comp, self.ncomp))
        ops = []
        for p in range(self.world):
            if p == self.rank:
                continue
            if self.roff[p + 1] > self.roff[p]:
                ops.append(dist.P2POp(dist.irecv, self.recv_t[self.roff[p]:self.roff[p + 1]], p))
            if self.soff[p + 1] > self.soff[p]:
                ops.append(dist.P2POp(dist.isend, self.send_t[self.soff[p]:self.soff[p + 1]], p))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        capi.check(capi.lib().pa_exchange_mark_received(f.f, comp, self.ncomp))


class FillPatchExchange:
    """NCCL send/recv of the packed slabs of one pa_fill_patch(lev, nghost, interp_type) on ncomp components of a field: the
    same-level neighbours and coarse-patch cells owned by another rank than the box they fill.  pack -> send/recv -> mark;
    then capi.fill_patch with the same arguments reads the recv slab.  The slabs are shared by every fill of the hierarchy and
    grow to the largest plan, so their pointers are taken afresh at every run."""

    def __init__(self, field: capi.Field, ncomp: int, lev: int, nghost: int, interp_type: int = 1, wrap=_wrap_device):
        """wrap(ptr, n): raw slab pointer -> tensor for the process group's backend (CUDA tensors for NCCL)."""
        H = field.hier
        self.field, self.ncomp, self.lev, self.nghost, self.interp_type = field, ncomp, lev, nghost, interp_type
        self.rank, self.world, self.wrap = H.rank, H.nranks, wrap
        # the plan (and the nesting verdict, the same on every rank) is built here, before any communication
        _, _, self.soff, self.roff = capi.fill_patch_exchange_buffers(field, ncomp, lev, nghost, interp_type)
        self.bytes_sent = 8 * self.soff[-1]

    def run(self, comp: int = 0) -> None:
        if self.world == 1:
            return
        f, a = self.field, (self.lev, self.nghost, self.interp_type)
        sp, rp, so, ro = capi.fill_patch_exchange_buffers(f, self.ncomp, *a)
        capi.fill_patch_pack(f, comp, self.ncomp, *a)
        ops = []
        for p in range(self.world):
            if p == self.rank:
                continue
            if ro[p + 1] > ro[p]:
                ops.append(dist.P2POp(dist.irecv, self.wrap(rp + 8 * ro[p], ro[p + 1] - ro[p]), p))
            if so[p + 1] > so[p]:
                ops.append(dist.P2POp(dist.isend, self.wrap(sp + 8 * so[p], so[p + 1] - so[p]), p))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        capi.fill_patch_mark_received(f, comp, self.ncomp, *a)


class Curvature:
    """The curvature tool on a multi-rank hierarchy: its steps (pa_curvature_steps) with the cross-rank step each one needs
    in front of it.

        [barrier]  exchange S            ->  PASS1   ghost fill of S, Progress, flame normal (+ un-normalised gradient G)
        [barrier]  exchange n            ->  DIV     ghost fill of n, MeanCurvature    -- threshold_prog: once per level, in
                                                     order, because level l reads the CLIPPED normal of level l-1
        [barrier]                        ->  CLIP    (threshold_prog, per level) zeroes n in place: only after every rank's
                                                     DIV of the level, which reads the unclipped normal of its peers
        [barrier]  exchange G            ->  GAUSS   (do_gaussCurv)      G is an internal field of the library
        [barrier]  exchange velocities   ->  STRAIN  (do_strain)
                                             VELN    (do_velnormal; pointwise)

    The barriers (1-element all-reduce on the stream) are only needed with peer links, where a rank's kernels read the
    other ranks' slabs in place: a step must not start before every peer finished writing what it reads, and the next
    run's PASS1 must not overwrite n while a peer still reads it.  The reference reaches the same ordering through MPI
    inside FillBoundary / ParallelCopy (Src/curvature.cpp:322, 487-502, 514-520, 686-717)."""

    def __init__(self, state: capi.Field, comp_S: int, opts: capi.CurvOpts, out: capi.Field, comp_out: int = 0, comp_vel: int = 0,
                 wrap=_wrap_device):
        self.state, self.comp_S, self.opts, self.out, self.comp_out, self.comp_vel = state, comp_S, opts, out, comp_out, comp_vel
        H = state.hier
        self.nlev = H.nlev
        self.peer = bool(H.flags & capi.PEER_LINKS) and H.nranks > 1
        self.scratch = capi.ScratchField(H) if opts.do_gauss else None
        # the 3-component exchanges first: the library grows its slabs to the largest request, and the tensors below
        # wrap raw slab pointers
        self.Xn = SlabExchange(out, 3, wrap)
        self.Xg = SlabExchange(self.scratch, 3, wrap) if self.scratch is not None else None
        self.Xv = SlabExchange(state, 3, wrap) if opts.do_strain else None
        self.Xs = SlabExchange(state, 1, wrap)
        if self.peer:
            map_peers(state)
            map_peers(out)
            if self.scratch is not None:
                map_peers(self.scratch)

    def _step(self, steps: int, lo: int = -1, hi: int = -1) -> None:
        capi.curvature_steps(self.state, self.comp_S, self.comp_vel, self.opts, self.out, self.comp_out, steps, lo, hi)

    def _barrier(self) -> None:
        if self.peer:
            stream_barrier()

    def run(self) -> None:
        o, cN = self.opts, self.comp_out + 2
        self._barrier()
        self.Xs.run(self.comp_S)
        self._step(capi.CURV_PASS1)
        if o.do_threshold:
            for l in range(self.nlev):
                self._barrier()
                self.Xn.run(cN)
                self._step(capi.CURV_DIV, l, l)
                self._barrier()             # every rank's DIV(l) has read its peers' UNCLIPPED n(l) (curvature.cpp:487-567)
                self._step(capi.CURV_CLIP, l, l)
        else:
            self._barrier()
            self.Xn.run(cN)
            self._step(capi.CURV_DIV)
        if o.do_gauss:
            self._barrier()
            self.Xg.run(0)
            self._step(capi.CURV_GAUSS)
        if o.do_strain:
            self._barrier()
            self.Xv.run(self.comp_vel)
            self._step(capi.CURV_STRAIN)
        if o.do_velnormal:
            self._step(capi.CURV_VELN)      # reads this rank's own cells only
