"""Host-side mirror of the reference's public API for the dense-grid integration path.

Julia is not installed in this image, so the host side that the reference writes in Julia
(``meshes.jl``, ``boundaryconditions.jl``, ``meshfield.jl``, ``levelsetterms.jl``,
``timestepping.jl``, ``levelsetequation.jl``) is mirrored here in Python over the same C ABI the
Julia glue (``julia/LSMB200.jl``) binds.  Names, argument meaning and error behaviour follow the
reference; every class/function cites the reference lines it mirrors.  Node indices are 1-based,
like the reference, wherever an index is part of the API (``getnode``, ``phi[I]``).

All arithmetic on field data happens on the GPU through ``liblsm_b200.so``; this module only
marshals data and runs the host control flow of ``integrate!``.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import re
from typing import Callable, NamedTuple, Optional, Sequence

import numpy as np

from . import _lib as L

inf = float("inf")


# =================================================================================================
# context
# =================================================================================================
class Context:
    """One process == one GPU == one rank (``lsm_ctx``)."""

    def __init__(self, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: Optional[bytes] = None):
        self.handle = C.c_void_p()
        self.rank, self.nranks, self.device = rank, nranks, device
        if nranks == 1:
            L.check(L.lib().lsm_ctx_create(device, C.byref(self.handle)))
        else:
            buf = C.create_string_buffer(nccl_id, 128)
            L.check(L.lib().lsm_ctx_create_rank(device, rank, nranks, buf, C.byref(self.handle)))

    @classmethod
    def _wrap(cls, handle, device: int, rank: int, nranks: int) -> "Context":
        c = cls.__new__(cls)
        c.handle, c.rank, c.nranks, c.device = C.c_void_p(handle), rank, nranks, device
        return c

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        L.check(L.lib().lsm_nccl_unique_id(buf))
        return buf.raw

    @classmethod
    def from_torch_distributed(cls, device: Optional[int] = None) -> "Context":
        """Build the rank's context from an initialised ``torch.distributed`` process group: rank 0
        makes the NCCL id and broadcasts its 128 bytes (plumbing only)."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", rank))
        if world == 1:
            return cls(device)
        ident = [cls.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        return cls(device, rank, world, ident[0])

    def sync(self):
        L.check(L.lib().lsm_sync(self.handle))

    def set_option(self, opt: int, value: int):
        L.check(L.lib().lsm_set_option(self.handle, opt, value))

    def counters(self) -> dict:
        c = L.lsm_counters()
        L.check(L.lib().lsm_get_counters(self.handle, C.byref(c)))
        return {k: getattr(c, k) for k, _ in c._fields_}

    def reset_counters(self):
        L.check(L.lib().lsm_reset_counters(self.handle))

    def event_record(self, slot: int):
        L.check(L.lib().lsm_event_record(self.handle, slot))

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_double()
        L.check(L.lib().lsm_event_elapsed_ms(self.handle, a, b, C.byref(ms)))
        return ms.value

    def slab(self, n_last: int):
        """(first, count) of the planes of the last dimension this rank owns (0-based first)."""
        f, c = C.c_int32(), C.c_int32()
        L.check(L.lib().lsm_slab_plan(n_last, self.nranks, self.rank, C.byref(f), C.byref(c)))
        return f.value, c.value

    def close(self):
        if self.handle:
            L.lib().lsm_ctx_destroy(self.handle)
            self.handle = C.c_void_p()


_default_ctx: Optional[Context] = None


class MultiContext:
    """All GPUs of a box driven from ONE process / thread (``lsm_ctx_create_multi``: ncclCommInitAll, one rank per device).
    ``ranks[r]`` is an ordinary :class:`Context` (rank r of n): build the per-rank slabs with ``MeshField(global_array, grid,
    ctx=mc.ranks[r])`` (or the device generators), then advance all of them together with :func:`integrate_multi`."""

    def __init__(self, device_ids: Sequence[int]):
        n = len(device_ids)
        hs = (C.c_void_p * n)()
        L.check(L.lib().lsm_ctx_create_multi(n, (C.c_int32 * n)(*device_ids), hs))
        self.ranks = [Context._wrap(hs[r], int(device_ids[r]), r, n) for r in range(n)]

    def __len__(self):
        return len(self.ranks)

    def close(self):
        for c in self.ranks:
            c.close()

    @staticmethod
    def gather(fields: Sequence["MeshField"]) -> np.ndarray:
        """The global array from the per-rank slabs (concatenated along the decomposed, last axis)."""
        return np.concatenate([np.asarray(f.peek()) for f in fields], axis=-1)


def compute_cfl_multi(mc: MultiContext, terms_per_rank, phis, t: float) -> float:
    n = len(mc)
    lows = [_Lowered(terms_per_rank[r], phis[r], t) for r in range(n)]
    dt = C.c_double()
    L.check(L.lib().lsm_multi_compute_cfl(
        n, (C.c_void_p * n)(*[c.handle for c in mc.ranks]), (C.c_void_p * n)(*[phis[r].device() for r in range(n)]),
        (C.POINTER(L.lsm_term) * n)(*[C.cast(lw.arr, C.POINTER(L.lsm_term)) for lw in lows]), len(terms_per_rank[0]), float(t),
        lows[0].gscale, C.byref(dt)))
    return dt.value


def integrate_multi(mc: MultiContext, eqs, tf: float, dt: float = inf):
    """``integrate!`` of the same equation on every rank's slab, from one thread: ``eqs[r]`` is the rank's
    :class:`LevelSetEquation` (device-only terms: stored / separable / constant coefficients, default hooks)."""
    n = len(mc)
    lows = [_Lowered(eqs[r].terms, eqs[r].state, eqs[r].t) for r in range(n)]
    if not all(lw.device_only for lw in lows):
        raise NotImplementedError("integrate_multi supports device-resident coefficients and default hooks")
    t_out, st = C.c_double(), C.c_int64()
    L.check(L.lib().lsm_multi_integrate(
        n, (C.c_void_p * n)(*[c.handle for c in mc.ranks]), eqs[0].integrator.code, float(eqs[0].integrator.cfl),
        (C.c_void_p * n)(*[eqs[r].state.device() for r in range(n)]),
        (C.POINTER(L.lsm_term) * n)(*[C.cast(lw.arr, C.POINTER(L.lsm_term)) for lw in lows]), len(eqs[0].terms),
        float(eqs[0].t), float(tf), float(dt), -1, C.byref(t_out), C.byref(st)))
    for e in eqs:
        e.state._mark_device_advanced()
        e.t = t_out.value
        e.steps_taken += st.value
    return eqs


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(int(os.environ.get("LSM_B200_DEVICE", os.environ.get("LOCAL_RANK", "0"))))
    return _default_ctx


def set_default_context(ctx: Optional[Context]):
    global _default_ctx
    _default_ctx = ctx


# =================================================================================================
# meshes.jl
# =================================================================================================
class CartesianGrid:
    """``CartesianGrid(lc, hc, n)`` / ``CartesianGrid(lc, hc; meshsize)`` (meshes.jl:1-5,34-42,69-83)."""

    def __init__(self, lc, hc, n=None, *, meshsize=None):
        lc, hc = tuple(float(x) for x in lc), tuple(float(x) for x in hc)
        if len(lc) != len(hc):
            raise ValueError("lc and hc must have the same length")
        N = len(lc)
        if n is None:
            if meshsize is None:
                raise ValueError("give the node counts n or a meshsize")
            h = (meshsize,) * N if np.isscalar(meshsize) else tuple(meshsize)
            if len(h) != N:
                raise ValueError("meshsize must be a scalar or have one entry per dimension")
            if not all(x > 0 for x in h):
                raise ValueError("meshsize must be positive in every dimension")
            if not all(hc[d] > lc[d] for d in range(N)):
                raise ValueError("hc must be strictly greater than lc in every dimension")
            n = tuple(int(math.ceil((hc[d] - lc[d]) / h[d])) + 1 for d in range(N))
        if len(n) != N:
            raise ValueError("all arguments must have the same length")
        self.lc, self.hc, self.n = lc, hc, tuple(int(x) for x in n)

    def __len__(self):
        return int(np.prod(self.n))

    @property
    def ndim(self):
        return len(self.n)

    size = property(lambda self: self.n)

    def meshsize(self, dim: Optional[int] = None):
        """meshes.jl:109-110 — (hc - lc) / (n - 1); ``dim`` is 1-based."""
        if dim is None:
            return tuple((self.hc[d] - self.lc[d]) / (self.n[d] - 1) for d in range(self.ndim))
        return (self.hc[dim - 1] - self.lc[dim - 1]) / (self.n[dim - 1] - 1)

    def getnode(self, *I):
        """meshes.jl:126-130 — coordinates of node ``I`` (1-based); lc + (I-1)*h."""
        if len(I) == 1 and not np.isscalar(I[0]):
            I = tuple(I[0])
        if not all(1 <= I[d] <= self.n[d] for d in range(self.ndim)):
            raise ValueError(f"{I} is not a valid node index for this grid")
        h = self.meshsize()
        return tuple(self.lc[d] + (I[d] - 1) * h[d] for d in range(self.ndim))

    def coords(self, first_last: int = 0, count_last: Optional[int] = None):
        """Broadcastable coordinate arrays of the (slab of the) grid: lc + (I-1)*h."""
        out, h = [], self.meshsize()
        for d in range(self.ndim):
            n, off = self.n[d], 0
            if d == self.ndim - 1 and count_last is not None:
                n, off = count_last, first_last
            x = self.lc[d] + (np.arange(n, dtype=np.float64) + off) * h[d]
            shape = [1] * self.ndim
            shape[d] = n
            out.append(x.reshape(shape))
        return out

    def __repr__(self):
        return f"CartesianGrid(lc={self.lc}, hc={self.hc}, n={self.n})"


# =================================================================================================
# boundaryconditions.jl
# =================================================================================================
class BoundaryCondition:
    kind, P = L.BC_NONE, 0

    def __eq__(self, other):
        return isinstance(other, BoundaryCondition) and (self.kind, self.P) == (other.kind, other.P)

    def __hash__(self):
        return hash((self.kind, self.P))


class PeriodicBC(BoundaryCondition):
    """boundaryconditions.jl:27 — node n duplicates node 1 (period is n-1 cells)."""
    kind = L.BC_PERIODIC

    def __repr__(self):
        return "Periodic"


class ExtrapolationBC(BoundaryCondition):
    """boundaryconditions.jl:40-47 — degree-P one-sided polynomial extrapolation."""
    kind = L.BC_EXTRAP

    def __init__(self, P: int = 0):
        if P < 0:
            raise ValueError("extrapolation order P must be at least 0")
        self.P = int(P)

    def __repr__(self):
        return {0: "Neumann", 1: "Linear extrapolation"}.get(self.P, f"Degree {self.P} extrapolation")


def NeumannBC():
    """boundaryconditions.jl:56 — ``ExtrapolationBC{0}``."""
    return ExtrapolationBC(0)


def LinearExtrapolationBC():
    """boundaryconditions.jl:64 — ``ExtrapolationBC{1}``."""
    return ExtrapolationBC(1)


class SymmetryBC(BoundaryCondition):
    """boundaryconditions.jl:74 — reflection about the boundary node."""
    kind = L.BC_SYMMETRY

    def __repr__(self):
        return "Symmetry"


def _normalize_bc(bc, dim: int):
    """boundaryconditions.jl:166-188 — tuple of (left, right) per dimension."""
    if isinstance(bc, BoundaryCondition):
        return tuple((bc, bc) for _ in range(dim))
    if len(bc) != dim:
        raise ValueError("invalid number of boundary conditions")
    out = []
    for i, b in enumerate(bc):
        if isinstance(b, BoundaryCondition):
            out.append((b, b))
            continue
        if not (len(b) == 2 and all(isinstance(x, BoundaryCondition) for x in b)):
            raise ValueError(f"invalid boundary condition for dimension {i + 1}")
        l, r = b
        if isinstance(l, PeriodicBC) != isinstance(r, PeriodicBC):
            raise ValueError(f"periodic boundary conditions cannot be mixed with others in dimension {i + 1}")
        out.append((l, r))
    return tuple(out)


# =================================================================================================
# meshfield.jl (dense half)
# =================================================================================================
class MeshField:
    """``MeshField(vals_or_f, grid; bc)`` (meshfield.jl:51-55,178-211).

    ``vals`` is the host array (column-major, like the Julia ``Array{V,N}``); a device mirror is
    created on first use by the engine and the two are kept coherent lazily: reading ``.vals`` after
    the device advanced downloads, handing the field to the engine after ``.vals`` was touched
    uploads.  Vector-valued fields (velocities) have shape ``(N, n1, .., nN)``.
    With a multi-rank context the field holds this rank's slab of the last dimension.
    """

    def __init__(self, vals, grid: CartesianGrid, bc=None, dtype=None, ctx: Optional[Context] = None):
        self.mesh = grid
        self.ctx = ctx
        N = grid.ndim
        c = ctx if ctx is not None else (_default_ctx if _default_ctx is not None else None)
        nr = c.nranks if c is not None else 1
        self._first, self._count = (c.slab(grid.n[-1]) if nr > 1 else (0, grid.n[-1]))
        local = tuple(grid.n[:-1]) + (self._count,)
        if callable(vals):
            X = grid.coords(self._first, self._count)
            v = vals(tuple(X))
            if isinstance(v, (tuple, list)):
                v = np.stack([np.broadcast_to(np.asarray(c_, dtype=np.float64), local) for c_ in v], axis=0)
            else:
                v = np.broadcast_to(np.asarray(v, dtype=np.float64), local)
            vals = v
        vals = np.asarray(vals)
        if dtype is None:
            dtype = vals.dtype if vals.dtype in (np.float32, np.float64) else np.float64
        if vals.shape == tuple(grid.n) and nr > 1:
            vals = vals[..., self._first:self._first + self._count]
        elif vals.shape == (N,) + tuple(grid.n) and nr > 1:
            vals = vals[..., self._first:self._first + self._count]
        if vals.shape == local:
            self.ncomp = 1
        elif vals.shape == (N,) + local:
            self.ncomp = N
        else:
            raise ValueError(f"values of shape {vals.shape} do not match the grid {grid.n}")
        self._vals = np.array(vals, dtype=dtype, order="F", copy=True)
        self._shape, self._dtype = self._vals.shape, self._vals.dtype
        self.bcs = None if bc is None else _normalize_bc(bc, N)
        self._dev = None          # lsm_field handle
        self._dev_bcs = None
        self._host_fresh, self._dev_fresh = True, False
        self._borrowed = False

    # --- fields generated on the device (no host array until someone asks for the values) ---
    @classmethod
    def _device_only(cls, grid: CartesianGrid, ncomp: int, bc, dtype, ctx: Optional[Context]) -> "MeshField":
        f = cls.__new__(cls)
        f.mesh, f.ctx = grid, (ctx if ctx is not None else default_context())
        nr = f.ctx.nranks
        f._first, f._count = (f.ctx.slab(grid.n[-1]) if nr > 1 else (0, grid.n[-1]))
        local = tuple(grid.n[:-1]) + (f._count,)
        f.ncomp = ncomp
        f._shape = local if ncomp == 1 else (ncomp,) + local
        f._dtype = np.dtype(dtype or np.float64)
        f._vals = None
        f.bcs = None if bc is None else _normalize_bc(bc, grid.ndim)
        f._dev, f._dev_bcs, f._borrowed = None, None, False
        f._host_fresh, f._dev_fresh = False, True
        f._create_device()
        return f

    @classmethod
    def from_shape(cls, grid: CartesianGrid, shape: str, params, bc=None, dtype=None, ctx: Optional[Context] = None) -> "MeshField":
        """Engine extension: ``MeshField(f, grid)`` for an analytic ``f`` evaluated on the DEVICE (``lsm_field_fill_shape``):
        ``"sphere"`` (centre..., radius), ``"box"`` (centre..., widths...), ``"plane"`` (normal..., offset), ``"const"`` (value)."""
        code = {"sphere": L.SHAPE_SPHERE, "box": L.SHAPE_BOX, "plane": L.SHAPE_PLANE, "const": L.SHAPE_CONST}[shape]
        p = [float(v) for v in np.ravel(np.asarray(params, dtype=np.float64))]
        f = cls._device_only(grid, len(p) if (shape == "const" and len(p) > 1) else 1, bc, dtype, ctx)
        L.check(L.lib().lsm_field_fill_shape(f._dev, code, (C.c_double * len(p))(*p), len(p)))
        return f

    @classmethod
    def from_separable(cls, sep: "SeparableVelocity", dtype=None, ctx: Optional[Context] = None) -> "MeshField":
        """Engine extension: the stored velocity field ``u_d = ((s_d X_d[i]) Y_d[j]) Z_d[k]`` of a :class:`SeparableVelocity`,
        materialised on the device (``lsm_field_fill_separable``) — bit-identical to building it with NumPy and uploading."""
        ctx = ctx if ctx is not None else (sep.ctx or default_context())
        if sep.ctx is None:
            sep.ctx = ctx
        f = cls._device_only(sep.grid, sep.grid.ndim, None, dtype, ctx)
        L.check(L.lib().lsm_field_fill_separable(f._dev, sep.device()))
        return f

    @classmethod
    def from_expr(cls, grid: CartesianGrid, expr, bc=None, dtype=None, ctx: Optional[Context] = None) -> "MeshField":
        """Engine extension: ``MeshField(f, grid)`` (meshfield.jl:208-211) for any ``f`` written as a :class:`DeviceExpr` (or its
        expression strings), evaluated on the device at ``t = 0`` (``lsm_field_fill_expr``)."""
        expr = expr if isinstance(expr, DeviceExpr) else DeviceExpr(expr)
        f = cls._device_only(grid, expr.ncomp, bc, dtype, ctx)
        L.check(L.lib().lsm_field_set_expr(f._dev, expr._carray()))
        L.check(L.lib().lsm_field_fill_expr(f._dev, 0.0))
        return f

    def _host(self) -> np.ndarray:
        if self._vals is None:
            self._vals = np.empty(self._shape, dtype=self._dtype, order="F")
        return self._vals

    # --- getters (meshfield.jl:58-64) ---
    @property
    def vals(self) -> np.ndarray:
        """``values(phi)``.  Syncs from the device if it is ahead; the caller may mutate the array."""
        if not self._host_fresh:
            L.check(L.lib().lsm_field_download(self._dev, self._host().ctypes.data))
            self._host_fresh = True
        self._dev_fresh = False      # conservative: the caller may write through the returned array
        return self._vals

    values = vals

    def peek(self) -> np.ndarray:
        """Read-only look at the current values (does not invalidate the device copy)."""
        if not self._host_fresh:
            L.check(L.lib().lsm_field_download(self._dev, self._host().ctypes.data))
            self._host_fresh = True
        v = self._vals.view()
        v.flags.writeable = False
        return v

    @property
    def ndim(self):
        return self.mesh.ndim

    @property
    def valtype(self):
        return self._dtype

    def has_boundary_conditions(self):
        return self.bcs is not None

    def boundary_conditions(self):
        return self.bcs

    def meshsize(self, dim=None):
        return self.mesh.meshsize(dim)

    def getnode(self, *I):
        return self.mesh.getnode(*I)

    @property
    def local_range(self):
        return self._first, self._count

    # --- device residency ---
    def _context(self) -> Context:
        if self.ctx is None:
            self.ctx = default_context()
        return self.ctx

    def _create_device(self):
        lib, ctx = L.lib(), self._context()
        h = C.c_void_p()
        g = self.mesh
        n = (C.c_int32 * 3)(*g.n, *([1] * (3 - g.ndim)))
        lc = (C.c_double * 3)(*g.lc, *([0.0] * (3 - g.ndim)))
        hc = (C.c_double * 3)(*g.hc, *([1.0] * (3 - g.ndim)))
        dt = L.F32 if self._dtype == np.float32 else L.F64
        L.check(lib.lsm_field_create(ctx.handle, g.ndim, n, dt, self.ncomp, lc, hc, C.byref(h)))
        self._dev = h

    def device(self):
        """The up-to-date ``lsm_field`` handle (creating / uploading as needed)."""
        lib = L.lib()
        if self._dev is None:
            self._create_device()
        if self.bcs is not None and self._dev_bcs != self.bcs:
            arr = (L.lsm_bc * 6)()
            for d, (l, r) in enumerate(self.bcs):
                arr[2 * d].kind, arr[2 * d].P = l.kind, l.P
                arr[2 * d + 1].kind, arr[2 * d + 1].P = r.kind, r.P
            L.check(lib.lsm_field_set_bc(self._dev, arr))
            self._dev_bcs = self.bcs
        if not self._dev_fresh:
            L.check(lib.lsm_field_upload(self._dev, self._vals.ctypes.data))
            self._dev_fresh = True
        return self._dev

    def _mark_device_advanced(self):
        self._dev_fresh, self._host_fresh = True, False

    @classmethod
    def _borrow(cls, handle, like: "MeshField") -> "MeshField":
        """Wrap a library-owned handle (an RK stage buffer) as a MeshField sharing ``like``'s grid/BCs."""
        f = cls.__new__(cls)
        f.mesh, f.ctx, f.ncomp, f.bcs = like.mesh, like.ctx, 1, like.bcs
        f._first, f._count = like._first, like._count
        f._vals, f._shape, f._dtype = None, like._shape, like._dtype      # host array allocated on first read
        f._dev, f._dev_bcs = handle, like.bcs
        f._host_fresh, f._dev_fresh, f._borrowed = False, True, True
        return f

    # --- indexing (meshfield.jl:213-260) ---
    def __getitem__(self, I):
        """``phi[I]`` with a 1-based index that may lie outside the grid (resolved through the BCs on
        the device, by the same ghost-cell code the stencil kernels use)."""
        if not isinstance(I, tuple):
            I = (I,)
        if self.ncomp != 1:
            return self.peek()[(slice(None),) + tuple(i - 1 for i in I)]
        idx = (C.c_int32 * len(I))(*[int(i) for i in I])
        out = C.c_double()
        L.check(L.lib().lsm_field_getindex(self.device(), idx, 1, C.byref(out)))
        return float(out.value) if self._dtype == np.float64 else float(np.float32(out.value))

    def __setitem__(self, I, val):
        if not isinstance(I, tuple):
            I = (I,)
        self.vals[tuple(i - 1 for i in I)] = val

    # --- copy / copy! / map (meshfield.jl:161-169,275-278) ---
    def copy(self) -> "MeshField":
        if self._vals is None or not self._host_fresh:
            # the device holds the current values (device-generated or advanced by the engine): copy there, no host round trip
            f = MeshField._device_only(self.mesh, self.ncomp, self.bcs, self._dtype, self.ctx)
            L.check(L.lib().lsm_field_copy(f._dev, self.device()))
            return f
        return MeshField(self.peek().copy(order="F"), self.mesh, bc=None if self.bcs is None else self.bcs, ctx=self.ctx)

    def copy_from(self, src: "MeshField") -> "MeshField":
        """``copy!(dest, src)``."""
        self.vals[...] = src.peek()
        return self

    def map(self, f: Callable) -> "MeshField":
        return MeshField(f(self.peek()), self.mesh, bc=self.bcs, ctx=self.ctx)

    def __del__(self):
        try:
            if self._dev is not None and not self._borrowed and self.ctx is not None and self.ctx.handle:
                L.lib().lsm_field_destroy(self._dev)
        except Exception:
            pass

    def __repr__(self):
        return f"MeshField on {self.mesh!r}, valtype={self._dtype}, bc={self.bcs}"


def _add_boundary_conditions(phi: MeshField, bc) -> MeshField:
    """meshfield.jl:150-153 — same data, new BCs (the data is aliased)."""
    out = MeshField.__new__(MeshField)
    out.__dict__.update(phi.__dict__)
    out.bcs = _normalize_bc(bc, phi.ndim)
    out._dev, out._dev_bcs, out._dev_fresh, out._borrowed = None, None, False, False
    out._host_fresh = True
    out._vals = phi.vals          # aliased, like the reference
    return out


# =================================================================================================
# derivatives.jl tags, levelsetterms.jl terms
# =================================================================================================
class Upwind:
    code = L.UPWIND


class WENO5:
    code = L.WENO5


class TimeScaled:
    """Engine extension: coefficient = ``base * g(t)`` with ``base`` a MeshField or constant and ``g`` a
    Python callable evaluated on the host at stage times, or ``("cos", T)`` for ``cos(pi t / T)`` evaluated
    inside the library (so the whole step loop stays on the device)."""

    def __init__(self, base, g):
        if isinstance(base, DeviceExpr):
            raise ValueError("TimeScaled(DeviceExpr(...)): write the time factor into the expression, which already sees t")
        self.base, self.g = base, g


class DeviceExpr:
    """Engine extension: a function-valued coefficient ``f(x, t)`` (levelsetterms.jl:42-43) evaluated on the DEVICE.  ``exprs`` is
    one CUDA C++ expression (a speed or ``b``) or a tuple of ``N`` (a velocity) in ``x1 .. xN``, ``t``, ``pi`` and CUDA's double
    math functions, e.g. ``AdvectionTerm(DeviceExpr(("-x2", "x1")))`` for ``(x, t) -> SVector(-x[2], x[1])``.  The expressions are
    checked and compiled (NVRTC, sm_100a, once per process) here, so a bad one fails before any GPU work; the engine then
    materialises the coefficient in HBM at every time the reference would call ``f``.  Without ``t`` the coefficient is
    materialised once and runs exactly like a stored field."""

    def __init__(self, exprs):
        self.exprs = (exprs,) if isinstance(exprs, str) else tuple(exprs)
        if not all(isinstance(e, str) for e in self.exprs):
            raise TypeError("DeviceExpr takes a string or a tuple of strings")
        self.ncomp = len(self.exprs)
        # a velocity has one component per dimension; a scalar is checked for the highest coordinate it names
        used = [int(k) for e in self.exprs for k in re.findall(r"\bx([1-3])\b", e)]
        ndim = self.ncomp if self.ncomp > 1 else max(used, default=1)
        L.check(L.lib().lsm_expr_check(ndim, self.ncomp, self._carray()))
        self._fields = {}         # (context, grid, dtype) -> MeshField carrying these expressions

    def _carray(self):
        return (C.c_char_p * (self.ncomp + 1))(*[e.encode() for e in self.exprs], None)

    def _field(self, phi: MeshField, ncomp: int) -> MeshField:
        """The device field of this coefficient for ``phi``'s context, grid and dtype (created on first use)."""
        if ncomp != self.ncomp:
            raise ValueError(f"this coefficient needs {ncomp} expression(s), the DeviceExpr has {self.ncomp}")
        ctx, g = phi._context(), phi.mesh
        key = (ctx, g.lc, g.hc, g.n, np.dtype(phi.valtype).str)
        f = self._fields.get(key)
        if f is None:
            f = MeshField._device_only(g, ncomp, None, phi.valtype, ctx)
            L.check(L.lib().lsm_field_set_expr(f._dev, self._carray()))
            self._fields[key] = f
        return f

    def __repr__(self):
        return f"DeviceExpr({self.exprs!r})"


class SeparableVelocity:
    """Engine extension: rank-1 separable velocity ``u_d = scale[d] * X_d[i1] * Y_d[i2] * Z_d[i3]``
    evaluated in-kernel from tiny per-axis tables (no velocity traffic from HBM)."""

    def __init__(self, grid: CartesianGrid, scales: Sequence[float], tabs, ctx: Optional[Context] = None):
        self.grid, self.ctx = grid, ctx
        N = grid.ndim
        self.scales = tuple(float(s) for s in scales)
        self.tabs = [[np.ascontiguousarray(tabs[d][a], dtype=np.float64) for a in range(N)] for d in range(N)]
        for d in range(N):
            for a in range(N):
                assert self.tabs[d][a].shape == (grid.n[a],)
        self._dev = None

    def device(self):
        if self._dev is None:
            ctx = self.ctx or default_context()
            self.ctx = ctx
            g, N = self.grid, self.grid.ndim
            flat = np.concatenate([self.tabs[d][a] for d in range(N) for a in range(N)])
            h = C.c_void_p()
            L.check(L.lib().lsm_field_create_separable(
                ctx.handle, N, (C.c_int32 * 3)(*g.n, *([1] * (3 - N))), (C.c_double * 3)(*g.lc, *([0.0] * (3 - N))),
                (C.c_double * 3)(*g.hc, *([1.0] * (3 - N))), (C.c_double * 3)(*self.scales, *([0.0] * (3 - N))),
                flat.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h)))
            self._dev = h
        return self._dev


_noop = None


class LevelSetTerm:
    update_func = None

    def _coef(self):
        raise NotImplementedError


class AdvectionTerm(LevelSetTerm):
    """``AdvectionTerm(u[, scheme = WENO5(), update_func])`` — ``u . grad(phi)`` (levelsetterms.jl:45-63)."""
    kind = L.TERM_ADVECTION

    def __init__(self, velocity, scheme=None, update_func=None):
        self.velocity, self.scheme, self.update_func = velocity, scheme or WENO5(), update_func

    def _coef(self):
        return self.velocity

    def __repr__(self):
        return "u . grad(phi)"


class CurvatureTerm(LevelSetTerm):
    """``CurvatureTerm(b)`` — ``b kappa |grad(phi)|`` (levelsetterms.jl:104-106)."""
    kind = L.TERM_CURVATURE

    def __init__(self, b):
        self.b = b

    def _coef(self):
        return self.b

    def __repr__(self):
        return "b kappa |grad(phi)|"


class NormalMotionTerm(LevelSetTerm):
    """``NormalMotionTerm(v[, update_func])`` — ``v |grad(phi)|`` (levelsetterms.jl:139-146)."""
    kind = L.TERM_NORMAL

    def __init__(self, speed, update_func=None):
        self.speed, self.update_func = speed, update_func

    def _coef(self):
        return self.speed

    def __repr__(self):
        return "v |grad(phi)|"


class EikonalReinitializationTerm(LevelSetTerm):
    """``EikonalReinitializationTerm(phi0)`` (frozen sign, O&F 7.5) / ``EikonalReinitializationTerm()``
    (live sign, 7.6) — levelsetterms.jl:211-222.  ``S0`` is computed on the device."""
    kind = L.TERM_EIKONAL

    def __init__(self, phi0: Optional[MeshField] = None):
        self.S0 = None
        if phi0 is not None:
            # S0 = v / sqrt(v^2 + dx^2) promotes to Float64 in the reference even for a Float32 phi0
            s0 = MeshField(np.zeros(phi0.peek().shape, dtype=np.float64), phi0.mesh, bc=phi0.bcs, ctx=phi0.ctx)
            L.check(L.lib().lsm_eikonal_s0(s0.device(), phi0.device()))
            s0._mark_device_advanced()
            self.S0 = s0

    def _coef(self):
        return self.S0

    def __repr__(self):
        return "sign(phi) (|grad(phi)| - 1)" if self.S0 is None else "sign(phi0) (|grad(phi)| - 1)"


def update_term(term: LevelSetTerm, phi: MeshField, t: float):
    """``update_term!`` (levelsetterms.jl:14,65-69,148-152): call the user hook as ``f(coeff, phi, t)``."""
    f = term.update_func
    if f is not None:
        return f(term._coef(), phi, t)
    return None


class _Lowered:
    """Terms lowered to the C descriptors for one stage time; keeps temporaries alive."""

    def __init__(self, terms, phi: MeshField, t: float):
        self.keep = []
        n = len(terms)
        if n > L.MAX_TERMS:
            raise ValueError(f"at most {L.MAX_TERMS} terms are supported")
        self.arr = (L.lsm_term * n)()
        self.gscale = (C.c_double * n)(*([1.0] * n))
        self.device_only = True       # no host evaluation needed at other times
        for k, term in enumerate(terms):
            self._lower(k, term, phi, t)

    def _lower(self, k, term, phi, t):
        d = self.arr[k]
        d.kind = term.kind
        d.scheme = term.scheme.code if isinstance(term, AdvectionTerm) else 0
        d.tscale_kind, d.tparam, d.field = L.TS_NONE, 1.0, None
        coef = term._coef()
        ncomp = phi.ndim if isinstance(term, AdvectionTerm) else 1
        if isinstance(coef, TimeScaled):
            if isinstance(coef.g, tuple) and coef.g[0] == "cos":
                d.tscale_kind, d.tparam = L.TS_COS, float(coef.g[1])
            else:
                d.tscale_kind = L.TS_HOST
                self.gscale[k] = float(coef.g(t))
                self.device_only = False
            coef = coef.base
        if term.update_func is not None:
            self.device_only = False
        if coef is None:
            d.coef_kind = L.COEF_NONE
        elif isinstance(coef, MeshField):
            d.coef_kind, d.field = L.COEF_FIELD, coef.device()
            self.keep.append(coef)
        elif isinstance(coef, SeparableVelocity):
            d.coef_kind, d.field = L.COEF_SEPARABLE, coef.device()
            self.keep.append(coef)
        elif isinstance(coef, DeviceExpr):
            # f(x, t) on the device: materialised by the library at the CFL and stage times (no host evaluation)
            f = coef._field(phi, ncomp)
            d.coef_kind, d.field = L.COEF_EXPR, f.device()
            self.keep.append(f)
        elif callable(coef):
            # Function-valued coefficient f(x, t) (levelsetterms.jl:43): evaluated on the HOST at the
            # stage time (slow path, like every host callback).  A result that does not depend on x
            # (e.g. (x,t) -> SVector(1.0)) lowers to a constant.
            self.device_only = False
            X = phi.mesh.coords(*phi.local_range)
            v = coef(tuple(X), t)
            comps = list(v) if isinstance(v, (tuple, list)) else [v]
            if all(np.ndim(c_) == 0 for c_ in comps):
                d.coef_kind = L.COEF_CONST
                for i, c_ in enumerate(comps):
                    d.cval[i] = float(c_)
            else:
                local = phi.peek().shape
                arr = np.stack([np.broadcast_to(np.asarray(c_, dtype=np.float64), local) for c_ in comps], axis=0)
                arr = arr if ncomp > 1 else arr[0]
                f = MeshField(arr.astype(phi.valtype), phi.mesh, ctx=phi.ctx)
                d.coef_kind, d.field = L.COEF_FIELD, f.device()
                self.keep.append(f)
        else:
            d.coef_kind = L.COEF_CONST
            vals = list(coef) if isinstance(coef, (tuple, list, np.ndarray)) else [coef]
            if len(vals) != ncomp:
                raise ValueError(f"constant coefficient needs {ncomp} component(s)")
            for i, c_ in enumerate(vals):
                d.cval[i] = float(c_)


def step_plan(t0: float, tf: float, dt_max: float, cfl: float, dt_cfl: float, max_steps: int = -1):
    """The step sizes ``_integrate!`` takes when the CFL step is constant (timestepping.jl:104-118), run-length encoded:
    ``(runs, steps, t_reached)`` with ``runs = [(dt, count), ...]``.  Pure host function (``lsm_step_plan``); this is the sequence
    ``lsm_integrate`` hands to the resident cluster kernel of small 2-D grids."""
    lib = L.lib()
    nr, st, tt = C.c_int32(), C.c_int64(), C.c_double()
    L.check(lib.lsm_step_plan(t0, tf, dt_max, cfl, dt_cfl, max_steps, 0, None, None, C.byref(nr), C.byref(st), C.byref(tt)))
    dts, cnt = (C.c_double * max(nr.value, 1))(), (C.c_int64 * max(nr.value, 1))()
    L.check(lib.lsm_step_plan(t0, tf, dt_max, cfl, dt_cfl, max_steps, nr.value, dts, cnt, C.byref(nr), C.byref(st), C.byref(tt)))
    return [(dts[i], cnt[i]) for i in range(nr.value)], st.value, tt.value


def compute_cfl(terms, phi: MeshField, t: float) -> float:
    """``compute_cfl(terms, phi, t)`` (levelsetterms.jl:22-38); raises :class:`CFLError` unless ``dt > 0``."""
    low = _Lowered(terms, phi, t)
    dt = C.c_double()
    ctx = phi._context()
    L.check(L.lib().lsm_compute_cfl(ctx.handle, phi.device(), low.arr, len(terms), float(t), low.gscale, C.byref(dt)))
    return dt.value


# =================================================================================================
# timestepping.jl
# =================================================================================================
class TimeIntegrator:
    code, nstages = -1, 0

    def __init__(self, cfl: float = 0.5):
        self.cfl = float(cfl)


class ForwardEuler(TimeIntegrator):
    """timestepping.jl:26-28"""
    code, nstages = L.FORWARD_EULER, 1


class RK2(TimeIntegrator):
    """timestepping.jl:46-48 (Heun)"""
    code, nstages = L.RK2, 2


class RK3(TimeIntegrator):
    """timestepping.jl:65-67 (Shu–Osher TVD)"""
    code, nstages = L.RK3, 3


def _stage_times(integ: TimeIntegrator, tc: float, dt: float):
    if isinstance(integ, ForwardEuler):
        return [tc]
    if isinstance(integ, RK2):
        return [tc, tc + dt]
    return [tc, tc + dt, tc + 0.5 * dt]


def _stage_inputs(integ: TimeIntegrator, phi: MeshField):
    """The field each stage differentiates (what ``update_term!`` receives, timestepping.jl:131,146,157,173,186,197)."""
    if isinstance(integ, ForwardEuler):
        return [phi]
    h1, h2 = C.c_void_p(), C.c_void_p()
    L.check(L.lib().lsm_field_stage_buffer(phi.device(), 1, C.byref(h1)))
    L.check(L.lib().lsm_field_stage_buffer(phi.device(), 2, C.byref(h2)))
    b1, b2 = MeshField._borrow(h1, phi), MeshField._borrow(h2, phi)
    return [phi, b1] if isinstance(integ, RK2) else [phi, b1, b2]


def _advance(integ: TimeIntegrator, phi: MeshField, terms, tc: float, dt: float):
    """``_advance!`` stage by stage, running ``update_term!`` before each stage like the reference."""
    ctx = phi._context()
    times = _stage_times(integ, tc, dt)
    inputs = _stage_inputs(integ, phi) if any(t.update_func is not None for t in terms) else [phi] * len(times)
    for s, ts in enumerate(times, start=1):
        for term in terms:
            update_term(term, inputs[s - 1], ts)
        low = _Lowered(terms, phi, ts)
        L.check(L.lib().lsm_stage(ctx.handle, integ.code, s, phi.device(), low.arr, len(terms), float(tc), float(dt),
                                  low.gscale))
        phi._mark_device_advanced()


def _eps(x: float) -> float:
    return float(np.spacing(abs(x)))


def _integrate(ls, phi: MeshField, integ: TimeIntegrator, terms, tc, tf, dt_max, prehook, posthook):
    """``_integrate!`` (timestepping.jl:101-122)."""
    ctx = phi._context()
    low = _Lowered(terms, phi, tc)
    if prehook is None and posthook is None and low.device_only:
        # no host callbacks: the whole loop runs inside the library
        t_out, steps = C.c_double(), C.c_int64()
        dev = phi.device()
        rc = L.lib().lsm_integrate(ctx.handle, integ.code, integ.cfl, dev, low.arr, len(terms), float(tc), float(tf),
                                   float(dt_max), -1, C.byref(t_out), C.byref(steps))
        phi._mark_device_advanced()
        ls.t = t_out.value
        ls.steps_taken = steps.value
        L.check(rc)
        return
    alpha = integ.cfl
    steps = 0
    while tc <= tf - _eps(tc):
        if prehook is not None:
            prehook(ls)
        for term in terms:
            update_term(term, phi, tc)
        dt = min(dt_max, alpha * compute_cfl(terms, phi, tc), tf - tc)
        _advance(integ, phi, terms, tc, dt)
        tc += dt
        ls.t = tc
        steps += 1
        if posthook is not None:
            posthook(ls)
    ls.t = float(tf)
    ls.steps_taken = steps


# =================================================================================================
# levelsetequation.jl
# =================================================================================================
class LevelSetEquation:
    """``LevelSetEquation(; terms, ic, bc, t = 0, integrator = RK2())`` (levelsetequation.jl:59-78)."""

    def __init__(self, *, terms, ic: MeshField, bc=None, t: float = 0.0, integrator: Optional[TimeIntegrator] = None):
        if isinstance(terms, LevelSetTerm):
            terms = (terms,)
        if not (isinstance(terms, tuple) and all(isinstance(x, LevelSetTerm) for x in terms)):
            raise ValueError(f"terms must be a LevelSetTerm or a tuple of them, got {type(terms)}")
        self.terms = terms
        self.integrator = integrator if integrator is not None else RK2()
        if bc is None:
            if not ic.has_boundary_conditions():
                raise L.BCError(L.ERR_BC, "no boundary conditions: pass `bc` or build `ic` with one")
            state = ic.copy()
        else:
            state = ic.copy()
            state.bcs = _normalize_bc(bc, ic.ndim)
        self.state = state
        self.t = float(t)
        self.steps_taken = 0

    def __repr__(self):
        return f"LevelSetEquation(phi_t + {' + '.join(map(repr, self.terms))} = 0, t={self.t})"


def volume(phi) -> float:
    """``volume(phi)`` (levelsetops.jl:27-33) — measure of {phi <= 0}, reduced on the device (no download of the field)."""
    phi = current_state(phi)
    out = C.c_double()
    L.check(L.lib().lsm_volume(phi._context().handle, phi.device(), C.byref(out)))
    return out.value


def perimeter(phi) -> float:
    """``perimeter(phi)`` (levelsetops.jl:139-149) — measure of {phi = 0}, reduced on the device."""
    phi = current_state(phi)
    out = C.c_double()
    L.check(L.lib().lsm_perimeter(phi._context().handle, phi.device(), C.byref(out)))
    return out.value


class InterfaceMesh(NamedTuple):
    """The zero level set as a piecewise-linear mesh (``lsm_interface_extract``): ``vertices`` (nv, N) float64, ``faces`` (np, N)
    int32 0-based vertex indices (triangles in 3-D, segments in 2-D, points in 1-D), and ``keys`` (nv,) int64, the global id of
    the lattice edge each vertex lies on (sorted; what :func:`merge_interfaces` welds on)."""
    vertices: np.ndarray
    faces: np.ndarray
    keys: np.ndarray


def _fetch_interface(ctx: Context, ndim: int, nv: int, nf: int) -> InterfaceMesh:
    V = np.empty((nv, ndim), dtype=np.float64)
    K = np.empty(nv, dtype=np.int64)
    F = np.empty((nf, ndim), dtype=np.int32)
    ptr = lambda a, t: C.cast(a.ctypes.data, C.POINTER(t)) if a.size else None
    L.check(L.lib().lsm_interface_fetch(ctx.handle, ptr(V, C.c_double), ptr(K, C.c_int64), ptr(F, C.c_int32)))
    return InterfaceMesh(V, F, K)


def extract_interface(phi, level: float = 0.0) -> InterfaceMesh:
    """Engine extension: the interface {phi = level} extracted on the device (marching simplices on the Freudenthal–Kuhn
    triangulation, include/lsm_b200.h); only the mesh is copied to the host, not the field.  Triangles are oriented so that their
    normal points toward phi > level; segments have phi <= level on their left.  The reference draws the interface from
    ``values(phi)`` (ext/MakieExt.jl)."""
    phi = current_state(phi)
    ctx = phi._context()
    nv, nf = C.c_int64(), C.c_int64()
    L.check(L.lib().lsm_interface_extract(ctx.handle, phi.device(), float(level), C.byref(nv), C.byref(nf)))
    return _fetch_interface(ctx, phi.ndim, nv.value, nf.value)


def merge_interfaces(pieces: Sequence[InterfaceMesh]) -> InterfaceMesh:
    """Weld the per-rank pieces of an extraction (in rank order) into one mesh: vertices with the same key are one vertex.  The
    result equals the single-GPU extraction of the whole field."""
    if not pieces:
        raise ValueError("merge_interfaces needs at least one piece")
    keys = np.concatenate([p.keys for p in pieces])
    uniq, first, inv = np.unique(keys, return_index=True, return_inverse=True)
    V = np.concatenate([p.vertices for p in pieces], axis=0)[first]
    base = np.cumsum([0] + [len(p.keys) for p in pieces[:-1]])
    F = np.concatenate([inv[p.faces.astype(np.int64) + b] for p, b in zip(pieces, base)], axis=0).astype(np.int32)
    return InterfaceMesh(V, F.reshape(-1, pieces[0].faces.shape[1]), uniq.astype(np.int64))


def extract_interface_multi(mc: MultiContext, phis, level: float = 0.0) -> InterfaceMesh:
    """:func:`extract_interface` of a field slab-decomposed over ``mc`` (collective): each rank extracts the cells it owns, and the
    pieces are welded on the host (:func:`merge_interfaces`)."""
    n = len(mc)
    phis = [current_state(p) for p in phis]
    nv, nf = (C.c_int64 * n)(), (C.c_int64 * n)()
    L.check(L.lib().lsm_multi_interface_extract(
        n, (C.c_void_p * n)(*[c.handle for c in mc.ranks]), (C.c_void_p * n)(*[p.device() for p in phis]), float(level), nv, nf))
    return merge_interfaces([_fetch_interface(mc.ranks[r], phis[r].ndim, nv[r], nf[r]) for r in range(n)])


def redistance(phi, band: int = 3, order: int = 1):
    """Engine extension: replace phi, in place on the device, by the signed distance to its zero level set (``lsm_redistance``).

    The interface is the piecewise-linear mesh :func:`extract_interface` returns, but the mesh is never built: nodes within ``band``
    cells of it scan the nearby primitives for their exact closest point, and jump flooding carries closest points to the rest of
    the grid.  Every node keeps its inside / outside classification, so the interface does not move beyond the linear
    reconstruction; NaN nodes stay NaN and a field without an interface is left unchanged.  No boundary conditions are needed,
    nothing is copied to the host and the call does not synchronise, so it fits a ``prehook``:
    ``integrate(eq, tf, prehook=lambda ls: redistance(ls.state))``.

    ``order=3`` (``lsm_redistance_cubic``) refines every closest point by Newton's method on the zero set of the cubic interpolant
    of phi (:func:`interpolate`), as the reference's ``reinitialize!`` does on its Bernstein patches (reinitializer.jl:12-42):
    third-order accurate instead of second, at the price of one more pass.  A node where Newton does not converge keeps the linear
    closest point.  The seeds (the linear mesh here, a KD-tree there) and the one-sided stencils at the box faces differ from the
    reference, so the two agree in idea, not bit for bit; unlike :func:`eikonal_reinitialize` either order is exact to its
    interface after one call.  ``phi`` is a field or an equation (its ``current_state``); returns the field.  Any other ``order``
    raises ``ValueError``."""
    if order not in (1, 3):
        raise ValueError(f"redistance: order must be 1 or 3 (got {order!r})")
    phi = current_state(phi)
    if order == 1:
        L.check(L.lib().lsm_redistance(phi._context().handle, phi.device(), int(band), None))
    else:
        L.check(L.lib().lsm_redistance_cubic(phi._context().handle, phi.device(), int(band), None, None))
    phi._mark_device_advanced()
    return phi


class CubicInterpolation(NamedTuple):
    """The cubic interpolant of a field at points (:func:`interpolate`): ``values`` (npts,), ``gradients`` (npts, N) and
    ``hessians`` (npts, N, N), float64, NaN at points outside the grid."""
    values: np.ndarray
    gradients: np.ndarray
    hessians: np.ndarray


def interpolate(phi, X) -> CubicInterpolation:
    """Engine extension: the tensor-product cubic interpolant of ``phi`` (``lsm_interpolate_cubic``), its gradient and its Hessian
    at the points ``X`` ((npts, N) or (N,) array-like of coordinates), evaluated on the device.

    Each cell uses the degree-3 polynomial through the 4^N surrounding nodes (one-sided at the faces of the grid, so no boundary
    conditions are involved): the same polynomial as the reference's Bernstein patch of an ``InterpolatedField``
    (interpolation.jl, bernstein.jl), not the same bits.  Node values are reproduced exactly; points outside the grid get NaN.
    This is the surface ``redistance(phi, order=3)`` measures distances to.  ``phi`` is a scalar field or an equation (its
    ``current_state``) with at least 4 nodes along every dimension."""
    phi = current_state(phi)
    X = np.asarray(X, dtype=np.float64)
    N = phi.ndim
    if X.ndim == 1 and X.shape[0] == N:
        X = X[None, :]
    if X.ndim != 2 or X.shape[1] != N:
        raise ValueError(f"interpolate: X must have shape (npts, {N}), got {X.shape}")
    X = np.ascontiguousarray(X)
    n = X.shape[0]
    val, grad, hess = np.empty(n), np.empty((n, N)), np.empty((n, N, N))
    ptr = lambda a: C.cast(a.ctypes.data, C.POINTER(C.c_double))
    L.check(L.lib().lsm_interpolate_cubic(phi._context().handle, phi.device(), n, ptr(X), ptr(val), ptr(grad), ptr(hess)))
    return CubicInterpolation(val, grad, hess)


def extend_closest_point(F: MeshField, phi, band: int = 3, redistance: bool = False) -> MeshField:
    """Engine extension: give every node of ``F``, in place on the device, the value of ``F`` at its closest point on the zero level
    set of ``phi`` (``lsm_extend_closest_point``): a speed known on or near the interface becomes constant along the normals, so a
    ``NormalMotionTerm(F)`` moves the interface with it.

    The closest points are exactly those :func:`redistance` finds (the piecewise-linear mesh of :func:`extract_interface`, never
    built); ``F`` there is interpolated linearly on the mesh from its values at the lattice nodes, so a constant ``F`` comes back
    unchanged.  NaN nodes of ``phi`` keep their ``F``, and so does every node when ``phi`` has no interface.  With
    ``redistance=True`` the same call also replaces ``phi`` by its signed distance, bit for bit what :func:`redistance` writes, so
    ``integrate(eq, tf, prehook=lambda ls: extend_closest_point(v, ls.state, redistance=True))`` reinitialises and extends in one
    scan.  No boundary conditions are needed, nothing is copied to the host and the call does not synchronise.

    Unlike :func:`extend_along_normals` (the reference's upwind pseudo-time PDE, velocityextension.jl:20-78) the result does not
    depend on a number of iterations and is not smeared at the interface.  ``phi`` is a field or an equation (its
    ``current_state``); ``F`` is a scalar field on the same grid, of either dtype; returns ``F``."""
    phi = current_state(phi)
    L.check(L.lib().lsm_extend_closest_point(phi._context().handle, F.device(), phi.device(), int(band), int(bool(redistance)), None))
    F._mark_device_advanced()
    if redistance:
        phi._mark_device_advanced()
    return F


class LevelSetIntegrals(NamedTuple):
    """What :func:`level_set_integrals` returns: the measures of the region {phi <= level} (``inside``: area in 2-D, volume in 3-D)
    and of the interface {phi = level} (``interface``: length in 2-D, area in 3-D, the number of points in 1-D), and the integrals of
    F over them (``None`` without F)."""
    inside: float
    interface: float
    F_inside: Optional[float]
    F_interface: Optional[float]


def _integrals(out, with_F: bool) -> LevelSetIntegrals:
    return LevelSetIntegrals(out[0], out[1], out[2] if with_F else None, out[3] if with_F else None)


def level_set_integrals(phi, F: Optional[MeshField] = None, level: float = 0.0) -> LevelSetIntegrals:
    """Engine extension: the measures of {phi <= level} and {phi = level}, and the integrals of ``F`` over both, on the device
    (``lsm_level_set_integrals``); only 32 bytes reach the host.

    The geometry is the sharp piecewise-linear interface of :func:`extract_interface` (the interface measure equals the measure of
    that mesh) and the region it bounds, with ``F`` interpolated linearly; both integrals are exact for a linear ``F``.  This
    differs from :func:`volume` and :func:`perimeter`, which are the reference's smoothed-Heaviside and smoothed-delta sums and
    depend on the smoothing width.  Typical uses: the area or volume lost by the enclosed region in the Zalesak and Enright
    benchmarks, shape functionals such as the integral of a speed from :func:`extend_closest_point` over the interface, and
    moments: with ``F = MeshField.from_expr(grid, "x1")`` the region's first moment along x1 is ``F_inside``, so its centroid is
    ``F_inside / inside``.

    ``phi`` is a scalar field or an equation (its ``current_state``); ``F`` is a scalar field on the same grid, of either dtype, and
    may be ``phi`` itself.  NaN nodes of ``phi`` drop the simplices they touch; no boundary conditions are used."""
    phi = current_state(phi)
    out = (C.c_double * 4)()
    L.check(L.lib().lsm_level_set_integrals(phi._context().handle, phi.device(), None if F is None else F.device(), float(level),
                                            out))
    return _integrals(out, F is not None)


def level_set_integrals_multi(mc: MultiContext, phis, Fs=None, level: float = 0.0) -> LevelSetIntegrals:
    """:func:`level_set_integrals` of a field slab-decomposed over ``mc`` (collective): each rank integrates the cells it owns and
    the per-plane partials are all-reduced, so the result equals the single-GPU call bit for bit.  ``Fs`` is None or one field per
    rank."""
    n = len(mc)
    phis = [current_state(p) for p in phis]
    out = (C.c_double * 4)()
    fs = None if Fs is None else (C.c_void_p * n)(*[f.device() for f in Fs])
    L.check(L.lib().lsm_multi_level_set_integrals(
        n, (C.c_void_p * n)(*[c.handle for c in mc.ranks]), (C.c_void_p * n)(*[p.device() for p in phis]), fs, float(level), out))
    return _integrals(out, Fs is not None)


def _csg(dst: MeshField, src: Optional[MeshField], op: int) -> MeshField:
    for f in (dst, src):
        if f is not None and f.ncomp != 1:
            raise ValueError("set operations need real-valued level-set fields")
    if src is not None and src.mesh.n != dst.mesh.n:
        raise ValueError("set operation between fields of different size")
    ctx = dst._context()
    L.check(L.lib().lsm_field_csg(ctx.handle, dst.device(), None if src is None else src.device(), op))
    dst._mark_device_advanced()
    return dst


def union_(phi1: MeshField, phi2: MeshField) -> MeshField:
    """``union!(phi1, phi2)``: phi1 = min(phi1, phi2) on the device (levelsetops.jl:253-259)."""
    return _csg(phi1, phi2, 0)


def intersect_(phi1: MeshField, phi2: MeshField) -> MeshField:
    """``intersect!(phi1, phi2)``: phi1 = max(phi1, phi2) (levelsetops.jl:273-279)."""
    return _csg(phi1, phi2, 1)


def setdiff_(phi1: MeshField, phi2: MeshField) -> MeshField:
    """``setdiff!(phi1, phi2)``: phi1 = max(phi1, -phi2) (levelsetops.jl:311-317)."""
    return _csg(phi1, phi2, 2)


def complement_(phi: MeshField) -> MeshField:
    """``complement!(phi)``: phi = -phi (levelsetops.jl:293-298)."""
    return _csg(phi, None, 3)


def union(phi1: MeshField, phi2: MeshField) -> MeshField:
    return union_(phi1.copy(), phi2)


def intersect(phi1: MeshField, phi2: MeshField) -> MeshField:
    return intersect_(phi1.copy(), phi2)


def setdiff(phi1: MeshField, phi2: MeshField) -> MeshField:
    return setdiff_(phi1.copy(), phi2)


def complement(phi: MeshField) -> MeshField:
    return complement_(phi.copy())


def extend_along_normals(F: MeshField, phi: MeshField, nb_iters: int = 50, cfl: float = 0.45, frozen=None,
                         interface_band: float = 1.5, min_norm: float = 1.0e-14) -> MeshField:
    """``extend_along_normals!(F, phi; nb_iters, cfl, frozen, interface_band, min_norm)`` (velocityextension.jl:20-78) on the
    device: extends the speed field `F` off the interface of `phi` along its normals.  Mutates and returns `F`."""
    if F.mesh.n != phi.mesh.n:
        raise ValueError("F and phi must be defined on the same mesh")
    if nb_iters < 0:
        raise ValueError("nb_iters must be non-negative")
    if not cfl > 0:
        raise ValueError("cfl must be strictly positive")
    fr = None
    if frozen is not None:
        fr = frozen.peek() if isinstance(frozen, MeshField) else np.asarray(frozen)
        if fr.shape != phi.peek().shape:
            raise ValueError("frozen mask must have the same size as phi")
        if fr.dtype != np.bool_:
            raise ValueError("frozen mask must contain Bool values")
        fr = np.asfortranarray(fr.astype(np.uint8))
    ctx = phi._context()
    L.check(L.lib().lsm_extend_along_normals(ctx.handle, F.device(), phi.device(), int(nb_iters), float(cfl),
                                             None if fr is None else fr.ctypes.data, float(interface_band), float(min_norm)))
    F._mark_device_advanced()
    return F


def eikonal_reinitialize(phi: MeshField, iterations: int = 20, integrator: Optional["TimeIntegrator"] = None, frozen: bool = True):
    """Device-side alternative to the reference's Newton ``reinitialize!`` (reinitializer.jl:12-42, which stays on the host):
    `iterations` pseudo-time steps of ``phi_t + sign(phi0)(|grad phi| - 1) = 0`` (EikonalReinitializationTerm, levelsetterms.jl:211-265)
    applied in place to `phi` — usable as a prehook without leaving the GPU (SURVEY.md §8f row 3)."""
    if not phi.has_boundary_conditions():
        raise L.BCError(L.ERR_BC, "reinitialization needs boundary conditions on the field")
    term = EikonalReinitializationTerm(phi if frozen else None)
    integ = integrator if integrator is not None else RK2()
    eq = LevelSetEquation.__new__(LevelSetEquation)
    eq.terms, eq.integrator, eq.state, eq.t, eq.steps_taken = (term,), integ, phi, 0.0, 0
    dt = integ.cfl * compute_cfl(eq.terms, phi, 0.0)
    integrate(eq, dt * iterations * (1 - 1e-12))
    return phi


def current_state(eq):
    return eq.state if isinstance(eq, LevelSetEquation) else eq


def current_time(eq: LevelSetEquation):
    return eq.t


def integrate(ls: LevelSetEquation, tf, dt=inf, *, prehook=None, posthook=None) -> LevelSetEquation:
    """``integrate!(ls, tf, dt = Inf; prehook, posthook)`` (levelsetequation.jl:194-203)."""
    tc = current_time(ls)
    if not tf >= tc:
        raise L.TimeError(L.ERR_TIME, f"final time {tf} must be >= initial time {tc}: the level-set equation cannot "
                                      "be solved back in time")
    _integrate(ls, ls.state, ls.integrator, ls.terms, tc, float(tf), float(dt), prehook, posthook)
    return ls


integrate_bang = integrate
