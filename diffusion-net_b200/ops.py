"""Host glue between torch tensors and the C-ABI kernels: operator prep (COO -> shared-pattern
CSR, cached on tensor identity), workspace, and the autograd Functions of the hot path.

PyTorch is plumbing only here (device memory, streams, autograd graph); every arithmetic step
of the path runs in the hand-written kernels behind ``include/diffusion_net_b200.h``.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import torch

from . import _lib

_ENGINES = {"simt": _lib.ENGINE_SIMT, "tc3x": _lib.ENGINE_TC3X, "tc1x": _lib.ENGINE_TC1X, "bf16": _lib.ENGINE_BF16}
_engine = _ENGINES[os.environ.get("DN_B200_ENGINE", "tc3x")]


def set_engine(name: str):
    """'tc3x' (default: tcgen05, error-compensated 3xTF32, fp32-grade), 'tc1x' (single-pass
    TF32), 'bf16' (single-pass bf16 tensor-core arithmetic, fp32 tensors in HBM; ~1e-2) or 'simt'
    (exact fp32 FFMA).  Shapes outside the tcgen05 kernels' envelope always run the exact SIMT kernels."""
    global _engine
    _engine = _ENGINES[name]


def get_engine() -> str:
    return {v: k for k, v in _ENGINES.items()}[_engine]


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("diffusion_net_b200 runs on CUDA tensors only (there is no CPU fallback); "
                               "got a tensor on {}".format(t.device))


def _f32c(t):
    if t.dtype != torch.float32:
        raise RuntimeError("diffusion_net_b200 computes in float32; got {}".format(t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _on(t):
    """Context manager making ``t``'s device current for a C-ABI call: kernel attributes, the current stream and the
    workspace are all per device (a model on cuda:1 while cuda:0 is current must launch on cuda:1)."""
    return torch.cuda.device(t.device)


_workspaces = {}
_retired_workspaces = []
pin_workspaces = False      # set by graphs.GraphedNet: never free a workspace a graph may point into


def workspace(V, K, C_, device, extra=0):
    """Scratch for the C-ABI calls, one buffer per (device, stream): calls on different streams
    (graphs.GraphedNet replays meshes concurrently) never share scratch.  ``extra``: bytes on top of
    dn_workspace_bytes (mesh batches: one packed spectral multiplier per mesh)."""
    need = _lib.load().dn_workspace_bytes(int(V), int(K), int(C_)) + int(extra) + 4096
    dev_index = device.index if device.index is not None else torch.cuda.current_device()
    key = (dev_index, torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < need:
        if ws is not None and pin_workspaces:
            _retired_workspaces.append(ws)     # captured CUDA graphs hold raw pointers into it
        ws = torch.empty(need, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


class GradOperators:
    """Shared-pattern CSR of (gradX, gradY) for one mesh, plus (lazily) its transpose."""

    def __init__(self, gradX, gradY):
        _require_cuda(gradX, gradY)
        gx = gradX if gradX.is_coalesced() else gradX.coalesce()
        gy = gradY if gradY.is_coalesced() else gradY.coalesce()
        if gx.dim() != 2 or gx.shape[0] != gx.shape[1] or gx.shape != gy.shape:
            raise ValueError("gradX/gradY must be square sparse matrices of equal shape")
        self.V = int(gx.shape[0])
        ix, iy = gx.indices(), gy.indices()
        if ix.shape == iy.shape and torch.equal(ix, iy):
            idx, vx, vy = ix, gx.values(), gy.values()
        else:  # general case: union pattern (index plumbing only)
            z = torch.zeros_like
            both = torch.sparse_coo_tensor(
                torch.cat((ix, iy), dim=1),
                torch.cat((torch.stack((gx.values(), z(gx.values())), -1),
                           torch.stack((z(gy.values()), gy.values()), -1)), dim=0),
                (self.V, self.V, 2)).coalesce()
            idx, vx, vy = both.indices(), both.values()[:, 0].contiguous(), both.values()[:, 1].contiguous()
        self.device = gx.device
        self._coo = (idx[0].contiguous(), idx[1].contiguous(), _f32c(vx), _f32c(vy))
        self.nnz = int(idx.shape[1])
        self.csr = self._build(*self._coo)
        self._csr_t = None

    def _build(self, rows, cols, vx, vy):
        lib = _lib.load()
        rowptr = torch.empty(self.V + 1, dtype=torch.int32, device=self.device)
        colidx = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=self.device)
        vals = torch.empty(2 * max(self.nnz, 1), dtype=torch.float32, device=self.device)
        _lib.check(lib.dn_csr_from_coo(rows.data_ptr(), cols.data_ptr(), vx.data_ptr(), vy.data_ptr(),
                                       self.nnz, self.V, rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(),
                                       _stream()), "dn_csr_from_coo")
        st = _lib.dn_csr(rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), self.nnz)
        return (st, rowptr, colidx, vals)   # keep the tensors alive next to the struct

    @classmethod
    def from_csc(cls, V, indptr, indices, data_x, data_y, device):
        """Straight from the reference's on-disk cache (scipy CSC arrays, geometry.py:548-568): the CSC arrays ARE
        the transposed CSR the backward pass needs; the forward CSR comes from one ``dn_csr_transpose`` call.
        No COO expansion, no coalesce, no int64 indices.  ``data_x``/``data_y`` share (indptr, indices)."""
        self = cls.__new__(cls)
        self.V, self.device = int(V), torch.device(device)
        dev = self.device
        rowptr_t = torch.as_tensor(indptr, dtype=torch.int32).to(dev)
        self.nnz = int(len(indices))
        colidx_t = torch.as_tensor(indices, dtype=torch.int32).to(dev) if self.nnz else \
            torch.empty(1, dtype=torch.int32, device=dev)
        vals_t = torch.empty(2 * max(self.nnz, 1), dtype=torch.float32, device=dev)
        if self.nnz:
            vals_t[0:2 * self.nnz:2] = torch.as_tensor(data_x, dtype=torch.float32).to(dev)
            vals_t[1:2 * self.nnz:2] = torch.as_tensor(data_y, dtype=torch.float32).to(dev)
        st_t = _lib.dn_csr(rowptr_t.data_ptr(), colidx_t.data_ptr(), vals_t.data_ptr(), self.nnz)
        self._csr_t = (st_t, rowptr_t, colidx_t, vals_t)
        rowptr = torch.empty(self.V + 1, dtype=torch.int32, device=dev)
        colidx = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
        vals = torch.empty(2 * max(self.nnz, 1), dtype=torch.float32, device=dev)
        scratch = torch.empty(max(self.V, 1), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().dn_csr_transpose(C.byref(st_t), self.V, rowptr.data_ptr(), colidx.data_ptr(),
                                                    vals.data_ptr(), scratch.data_ptr(), 4 * scratch.numel(),
                                                    _stream()), "dn_csr_transpose")
        self.csr = (_lib.dn_csr(rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), self.nnz),
                    rowptr, colidx, vals)
        self._coo = None
        return self

    @classmethod
    def from_csr(cls, V, rowptr, colidx, vals_xy):
        """Wrap an already-built shared-pattern CSR that lives on the device: ``rowptr`` int32 (V+1), ``colidx`` int32
        (nnz), ``vals_xy`` float32 (nnz, 2) = (gradX, gradY) values interleaved.  No kernel runs and nothing is copied:
        this is the cheapest way to hand per-step uploaded operators to the layers (12 B/nnz on the host link instead
        of the reference's 40 B/nnz of int64 COO).  ``to_host_csr()`` produces the matching host arrays."""
        self = cls.__new__(cls)
        _require_cuda(rowptr, colidx, vals_xy)
        if rowptr.dtype != torch.int32 or colidx.dtype != torch.int32 or vals_xy.dtype != torch.float32:
            raise RuntimeError("from_csr expects int32 rowptr/colidx and float32 values")
        self.V, self.device = int(V), rowptr.device
        self.nnz = int(colidx.numel())
        rowptr, colidx, vals = rowptr.contiguous(), colidx.contiguous(), vals_xy.contiguous().view(-1)
        if self.nnz == 0:
            colidx = torch.empty(1, dtype=torch.int32, device=self.device)
            vals = torch.empty(2, dtype=torch.float32, device=self.device)
        self.csr = (_lib.dn_csr(rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), self.nnz), rowptr, colidx, vals)
        self._coo = None
        self._csr_t = None
        return self

    def to_host_csr(self):
        """(rowptr int32, colidx int32, vals (nnz,2) float32) as pinned host tensors (see ``from_csr``)."""
        _, rowptr, colidx, vals = self.csr
        pin = lambda t: t.cpu().contiguous().pin_memory()
        return pin(rowptr), pin(colidx[:self.nnz]), pin(vals[:2 * self.nnz].view(-1, 2))

    def locality(self):
        """Share of entries whose column lies within 8 rows of their row: a proxy for how much of a row's gather the
        neighbouring warps of a CTA (8 consecutive rows) have already pulled into L1.  0.43 on a row-major grid
        mesh, ~0.15 on a randomly permuted one (the diagonal stays).  (Index plumbing on the device.)"""
        if self.nnz == 0:
            return 1.0
        _, rowptr, colidx, _ = self.csr
        counts = (rowptr[1:] - rowptr[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(self.V, device=self.device), counts)
        return float(((colidx[:self.nnz].long() - rows).abs() <= 8).float().mean())

    def build_patches(self, max_targets=None, max_src=None):
        """Locality structure for the fused gradient-features kernel (``dn_patches``): rows are clustered into patches of
        graph-adjacent vertices (host side, ``dn_patch_build``) so the kernel stages each patch's distinct neighbour
        rows in shared memory once.  Worth its one-off cost (a D2H of the pattern, the clustering, an H2D) only for
        operators that stay resident, so ``prepare_operators`` calls it on the SECOND use of the same tensors.
        Default 32 rows / 72 distinct source rows per patch: 72 x (C + 2C) floats = 108 KiB of shared memory at
        C = 128, two CTAs per SM (measured best of the shapes tried, tools/ab_patch.py)."""
        if getattr(self, "_patches", None) is not None or self.nnz == 0:
            return self
        import numpy as np
        max_targets = int(os.environ.get("DN_PATCH_T", 32)) if max_targets is None else max_targets
        max_src = int(os.environ.get("DN_PATCH_R", 72)) if max_src is None else max_src
        st, rowptr, colidx, vals = self.csr
        rp = rowptr.cpu().numpy()
        ci = colidx[:self.nnz].cpu().numpy()
        V, nnz = self.V, self.nnz
        tgt_ptr, src_ptr, ent_ptr = (np.empty(V + 1, np.int32) for _ in range(3))
        tgt = np.empty(V, np.int32)
        src_rows, perm = np.empty(nnz, np.int32), np.empty(nnz, np.int32)
        lcol = np.empty(nnz, np.uint8)
        worst = np.zeros(1, np.int32)
        hp = lambda a: C.c_void_p(a.ctypes.data)
        n = _lib.load().dn_patch_build(V, hp(rp), hp(ci), int(max_targets), int(max_src), hp(tgt_ptr), hp(tgt),
                                       hp(src_ptr), hp(src_rows), hp(ent_ptr), hp(lcol), hp(perm), hp(worst))
        if n == -2:                     # a row with more than max_src entries: the plain kernel keeps serving it
            self._patches = False
            return self
        if n < 0:
            _lib.check(int(n), "dn_patch_build")
        n = int(n)
        dev = self.device
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        d = dict(tgt_ptr=up(tgt_ptr[:n + 1]), tgt=up(tgt), src_ptr=up(src_ptr[:n + 1]),
                 src_rows=up(src_rows[:int(src_ptr[n])]), ent_ptr=up(ent_ptr), lcol=up(lcol))
        d["vals"] = vals.view(-1, 2)[:nnz][up(perm).long()].contiguous().view(-1)
        pst = _lib.dn_patches(n, int(worst[0]), d["tgt_ptr"].data_ptr(), d["tgt"].data_ptr(), d["src_ptr"].data_ptr(),
                              d["src_rows"].data_ptr(), d["ent_ptr"].data_ptr(), d["lcol"].data_ptr(),
                              d["vals"].data_ptr())
        self._patches = (pst, d)        # keep the device arrays alive next to the struct
        st.patches = C.pointer(pst)
        self.patch_stats = dict(n_patches=n, max_src=int(worst[0]), src_per_row=float(src_ptr[n]) / max(V, 1))
        return self

    def to_sparse_coo(self):
        """(gradX, gradY) as the coalesced int64 COO tensors the reference hands around (utils.py:50-55), built from
        the forward CSR (index plumbing only; rows are sorted and unique, so no coalesce pass is needed)."""
        _, rowptr, colidx, vals = self.csr
        counts = (rowptr[1:] - rowptr[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(self.V, device=self.device), counts)
        idx = torch.stack((rows, colidx[:self.nnz].long()), 0)
        mk = lambda v: torch.sparse_coo_tensor(idx, v.contiguous(), (self.V, self.V), is_coalesced=True)
        return mk(vals[0:2 * self.nnz:2]), mk(vals[1:2 * self.nnz:2])

    @property
    def csr_t(self):
        """CSR of the transposed pattern (backward pass); index sort is prep-time plumbing."""
        if self._csr_t is None and self._coo is None:      # built by from_csr: transpose on the device
            _, rowptr, colidx, vals = self.csr
            rt = torch.empty(self.V + 1, dtype=torch.int32, device=self.device)
            ct = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=self.device)
            vt = torch.empty(2 * max(self.nnz, 1), dtype=torch.float32, device=self.device)
            scratch = torch.empty(max(self.V, 1), dtype=torch.int32, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(_lib.load().dn_csr_transpose(C.byref(self.csr[0]), self.V, rt.data_ptr(), ct.data_ptr(),
                                                        vt.data_ptr(), scratch.data_ptr(), 4 * scratch.numel(),
                                                        _stream()), "dn_csr_transpose")
            self._csr_t = (_lib.dn_csr(rt.data_ptr(), ct.data_ptr(), vt.data_ptr(), self.nnz), rt, ct, vt)
        if self._csr_t is None:
            rows, cols, vx, vy = self._coo
            order = torch.argsort(cols * self.V + rows)
            self._csr_t = self._build(cols[order].contiguous(), rows[order].contiguous(),
                                      vx[order].contiguous(), vy[order].contiguous())
        return self._csr_t


_prep_cache = {}
# dn_patches policy on the SECOND use of an operator pair (= the operators are resident): "auto" (default) builds the
# structure only for poorly ordered meshes, "1" always, "0" never.  Measured on B200 (tools/ab_patch.py, V = 200k,
# C = 128): the staged gather takes ~206 us whatever the vertex order; the plain gather takes 179 us on a mesh whose
# order has locality (47 % L1 hits) and 346 us on a randomly permuted one.
auto_patch = os.environ.get("DN_SPMM_PATCH", "auto")
PATCH_LOCALITY_THRESHOLD = 0.25


def _maybe_patch(ops):
    if auto_patch == "0" or getattr(ops, "_patches", None) is not None:
        return
    if torch.cuda.is_current_stream_capturing():     # the decision needs host round trips: not inside a graph capture
        return
    if auto_patch == "1" or ops.locality() < PATCH_LOCALITY_THRESHOLD:
        ops.build_patches()
    else:
        ops._patches = False            # decided: the vertex order already has locality


_prep_sweep_at = 256


def _sweep_prep_cache():
    """Drop entries whose sparse tensors died.  Live entries are never evicted: a dataset keeps its operator
    tensors for the whole run (SURVEY.md 8b 'Ownership') and their CSR must stay resident with them."""
    global _prep_sweep_at
    if len(_prep_cache) > _prep_sweep_at:
        for k in [k for k, v in _prep_cache.items() if v[0]() is None or v[1]() is None]:
            del _prep_cache[k]
        _prep_sweep_at = max(256, 2 * len(_prep_cache))


def _evict_when_dead(key, *tensors):
    """Drop a memoised entry (device CSR, transposed CSR, patches: ~17 MB per mesh at V = 200k) as soon as one of the
    user's sparse tensors it was built from dies.  Training loops that re-upload the operators every step
    (``gradX.to(device)``, as the reference's experiments do) would otherwise pile up dead entries."""
    for t in tensors:
        weakref.finalize(t, _prep_cache.pop, key, None)


def prepare_operators(gradX, gradY):
    """Memoised on the identity (+ version) of the user's sparse tensors: the reference reuses the
    same operator tensors across blocks and epochs (SURVEY.md section 8b 'Ownership').  Keep the operators
    resident on the device: a fresh ``.to(device)`` copy every step is a cache miss (CSR rebuild + one host sync)."""
    key = (id(gradX), id(gradY))
    hit = _prep_cache.get(key)
    if hit is not None:
        rx, ry, ver, ops = hit
        if rx() is gradX and ry() is gradY and ver == (gradX._version, gradY._version):
            _maybe_patch(ops)           # second use of the same operator tensors: they are resident
            return ops
    ops = GradOperators(gradX, gradY)
    _sweep_prep_cache()
    _prep_cache[key] = (weakref.ref(gradX), weakref.ref(gradY), (gradX._version, gradY._version), ops)
    _evict_when_dead(key, gradX, gradY)
    return ops


def register_prepared(gradX, gradY, ops):
    """Attach an already-built GradOperators to the sparse tensors a caller will pass to the layers
    (geometry.get_operators builds the CSR straight from the cache file)."""
    key = (id(gradX), id(gradY))
    _prep_cache[key] = (weakref.ref(gradX), weakref.ref(gradY), (gradX._version, gradY._version), ops)
    _evict_when_dead(key, gradX, gradY)
    _sweep_prep_cache()


def prepare_operators_batched(gradX, gradY):
    """For the reference's stacked (B,V,V) sparse operators: one GradOperators per mesh."""
    key = (id(gradX), id(gradY), "batched")
    hit = _prep_cache.get(key)
    if hit is not None:
        rx, ry, ver, ops = hit
        if rx() is gradX and ry() is gradY and ver == (gradX._version, gradY._version):
            for o in ops:
                _maybe_patch(o)
            return ops
    ops = [GradOperators(gradX[b], gradY[b]) for b in range(gradX.shape[0])]
    _sweep_prep_cache()
    _prep_cache[key] = (weakref.ref(gradX), weakref.ref(gradY), (gradX._version, gradY._version), ops)
    _evict_when_dead(key, gradX, gradY)
    return ops


# ------------------------------------------------------------------------------------------------
# thin wrappers (no autograd)
# ------------------------------------------------------------------------------------------------
def to_basis_raw(values, basis, massvec):
    _require_cuda(values, basis, massvec)
    values, basis = _f32c(values), _f32c(basis)
    V, K = basis.shape
    Cc = values.shape[-1]
    out = torch.empty(K, Cc, dtype=torch.float32, device=values.device)
    mv = _f32c(massvec) if massvec is not None else None
    with _on(values):
        ws = workspace(V, K, Cc, values.device)
        _lib.check(_lib.load().dn_to_basis(values.data_ptr(), basis.data_ptr(),
                                           mv.data_ptr() if mv is not None else None, V, K, Cc,
                                           out.data_ptr(), ws.data_ptr(), ws.numel(), _engine, _stream()),
                   "dn_to_basis")
    return out


def from_basis_raw(values, basis, row_scale=None):
    _require_cuda(values, basis, row_scale)
    values, basis = _f32c(values), _f32c(basis)
    V, K = basis.shape
    Cc = values.shape[-1]
    out = torch.empty(V, Cc, dtype=torch.float32, device=values.device)
    rs = _f32c(row_scale) if row_scale is not None else None
    with _on(values):
        ws = workspace(V, K, Cc, values.device)
        _lib.check(_lib.load().dn_from_basis(values.data_ptr(), basis.data_ptr(),
                                             rs.data_ptr() if rs is not None else None, V, K, Cc, out.data_ptr(),
                                             ws.data_ptr(), ws.numel(), _engine, _stream()), "dn_from_basis")
    return out


def _device_guard(fn):
    """Run an autograd Function's forward/backward with the device of its first tensor argument current."""
    import functools

    @functools.wraps(fn)
    def wrapped(ctx, *a):
        t = next((x for x in a if torch.is_tensor(x)), None)
        if t is None or not t.is_cuda:
            return fn(ctx, *a)
        with torch.cuda.device(t.device):
            return fn(ctx, *a)
    return wrapped


def _no_operator_grads(*named):
    for name, t in named:
        if t is not None and t.requires_grad:
            raise RuntimeError("diffusion_net_b200: gradients w.r.t. the operator tuple ({}) are not provided "
                               "(the operators are data, SURVEY.md section 8a)".format(name))


class ToBasisFn(torch.autograd.Function):
    """geometry.py:572-583, differentiable in ``values``: d values = mass * (basis @ g)."""

    @staticmethod
    def forward(ctx, values, basis, massvec):
        ctx.save_for_backward(basis, massvec)
        return to_basis_raw(values, basis, massvec)

    @staticmethod
    def backward(ctx, g):
        basis, massvec = ctx.saved_tensors
        return from_basis_raw(_f32c(g), basis, row_scale=massvec), None, None


class FromBasisFn(torch.autograd.Function):
    """geometry.py:586-598 (real branch), differentiable in ``values``: d values = basis^T g."""

    @staticmethod
    def forward(ctx, values, basis):
        ctx.save_for_backward(basis)
        return from_basis_raw(values, basis)

    @staticmethod
    def backward(ctx, g):
        (basis,) = ctx.saved_tensors
        return to_basis_raw(_f32c(g), basis, None), None


def to_basis(values, basis, massvec):
    if torch.is_grad_enabled():
        _no_operator_grads(("basis", basis), ("massvec", massvec))
        if values.requires_grad:
            return ToBasisFn.apply(values, basis, massvec)
    return to_basis_raw(values, basis, massvec)


def from_basis(values, basis):
    if torch.is_grad_enabled():
        _no_operator_grads(("basis", basis))
        if values.requires_grad:
            return FromBasisFn.apply(values, basis)
    return from_basis_raw(values, basis)


def compute_hks_raw(evals, evecs, scales):
    _require_cuda(evals, evecs, scales)
    evals, evecs, scales = _f32c(evals), _f32c(evecs), _f32c(scales)
    V, K = evecs.shape
    if evals.shape != (K,) or scales.dim() != 1:
        raise ValueError("compute_hks expects evals (K), evecs (V,K), scales (S)")
    S = scales.shape[0]
    out = torch.empty(V, S, dtype=torch.float32, device=evecs.device)
    with torch.cuda.device(evecs.device):
        _lib.check(_lib.load().dn_compute_hks(evals.data_ptr(), evecs.data_ptr(), scales.data_ptr(), V, K, S,
                                              out.data_ptr(), _stream()), "dn_compute_hks")
    return out


def grad_spmm_raw(ops: GradOperators, x):
    x = _f32c(x)
    V, Cc = x.shape
    out = torch.empty(V, Cc, 2, dtype=torch.float32, device=x.device)
    with _on(x):
        _lib.check(_lib.load().dn_grad_spmm(C.byref(ops.csr[0]), x.data_ptr(), V, Cc, out.data_ptr(), _stream()),
                   "dn_grad_spmm")
    return out


def spatial_gradient_features_raw(vectors, A_re, A_im):
    vectors = _f32c(vectors)
    V, Cc, _ = vectors.shape
    out = torch.empty(V, Cc, dtype=torch.float32, device=vectors.device)
    a_re = _f32c(A_re)                                  # contiguous copies stay referenced until the call returns
    a_im = _f32c(A_im) if A_im is not None else None
    with _on(vectors):
        ws = workspace(V, Cc, Cc, vectors.device)
        _lib.check(_lib.load().dn_spatial_gradient_features_fwd(
            vectors.data_ptr(), a_re.data_ptr(), a_im.data_ptr() if a_im is not None else None,
            1 if a_im is not None else 0, V, Cc, out.data_ptr(), ws.data_ptr(), ws.numel(), _engine, _stream()),
            "dn_spatial_gradient_features_fwd")
    return out


class HeadNotFused(RuntimeError):
    """The linear head cannot ride in this block's MiniMLP epilogue (shape / engine outside the fused chain)."""


PROFILE_STAGES = ("to_basis", "spectral_scale", "pack_weights", "from_basis_pq", "grad_features_gather", "mlp")


def head_fusable(n_out):
    """``DiffusionNet.last_lin`` can ride in the last block's MiniMLP epilogue (dn_block_fwd_ex) for up to 8 outputs."""
    return 1 <= int(n_out) <= 8


def block_forward_raw(x_in, mass, evals, evecs, ops, time, A_re, A_im, weights, biases, with_features,
                      profile=None, head=None, batch_desc=None):
    """Fused inference forward of one block on one mesh (dn_block_fwd).  ``profile``: a list that receives the
    per-stage device times in ms (``PROFILE_STAGES`` order; dn_block_fwd_profile, synchronises).
    ``head=(weight, bias)``: a linear head (``DiffusionNet.last_lin``) fused behind the block -- the return value is then
    the (V, n_out) head output and the block output is never written; raises ``HeadNotFused`` when the MiniMLP is not
    on the fused tensor-core chain (the caller applies the head separately).  ``batch_desc``: a ``_lib.dn_mesh_batch``
    (see batch.MeshBatch) when ``x_in`` / the operators are a batch laid out as one vertex range."""
    lib = _lib.load()
    x_in, mass, evals, evecs = _f32c(x_in), _f32c(mass), _f32c(evals), _f32c(evecs)
    V, Cc = x_in.shape
    K = evecs.shape[1]
    out = torch.empty_like(x_in)
    dims = [weights[0].shape[1]] + [w.shape[0] for w in weights]
    # contiguous copies (if any were needed) must outlive the launch: keep them in locals, not temporaries
    wc = [_f32c(w) for w in weights]
    bc = [_f32c(b) if b is not None else None for b in biases]
    a_re = _f32c(A_re) if A_re is not None else None
    a_im = _f32c(A_im) if A_im is not None else None
    wp = _lib.ptr_array([w.data_ptr() for w in wc])
    bp = _lib.ptr_array([b.data_ptr() if b is not None else None for b in bc])
    dm = _lib.int_array(dims)
    prm = _lib.dn_block_params(
        time.data_ptr(), a_re.data_ptr() if a_re is not None else None,
        a_im.data_ptr() if a_im is not None else None, 1 if with_features else 0,
        1 if a_im is not None else 0, len(weights), wp, bp, dm)
    csr = C.byref(ops.csr[0]) if ops is not None else None
    with _on(x_in):
        # the unfused MLP route carves 2 x V x max(hidden) floats: size the scratch by the widest layer
        extra = 0 if batch_desc is None else int(batch_desc.n_meshes) * K * Cc * 8
        ws = workspace(V, K, max(Cc, max(dims[1:])), x_in.device, extra=extra)
        if head is not None or batch_desc is not None:
            hd, hout = None, None
            if head is not None:
                hw = _f32c(head[0])
                hb = _f32c(head[1]) if head[1] is not None else None
                hout = torch.empty(V, hw.shape[0], dtype=torch.float32, device=x_in.device)
                hd = _lib.dn_head(hw.data_ptr(), hb.data_ptr() if hb is not None else None, int(hw.shape[0]),
                                  hout.data_ptr(), int(hw.shape[0]))
            rc = lib.dn_block_fwd_ex(x_in.data_ptr(), mass.data_ptr(), evals.data_ptr(), evecs.data_ptr(), csr, C.byref(prm),
                                     C.byref(batch_desc) if batch_desc is not None else None,
                                     C.byref(hd) if hd is not None else None, V, K, Cc,
                                     None if head is not None else out.data_ptr(), ws.data_ptr(), ws.numel(), _engine,
                                     _stream())
            if rc == -2 and head is not None:      # DN_ERR_UNSUPPORTED: the chain that would carry the head is not available
                raise HeadNotFused()
            _lib.check(rc, "dn_block_fwd_ex")
            return hout if head is not None else out
        if profile is not None:
            ms = (C.c_float * 6)()
            _lib.check(lib.dn_block_fwd_profile(x_in.data_ptr(), mass.data_ptr(), evals.data_ptr(), evecs.data_ptr(),
                                                csr, C.byref(prm), V, K, Cc, out.data_ptr(), ws.data_ptr(),
                                                ws.numel(), _engine, _stream(), ms), "dn_block_fwd_profile")
            profile[:] = [float(v) for v in ms]
            return out
        _lib.check(lib.dn_block_fwd(x_in.data_ptr(), mass.data_ptr(), evals.data_ptr(), evecs.data_ptr(), csr,
                                    C.byref(prm), V, K, Cc, out.data_ptr(), ws.data_ptr(), ws.numel(), _engine,
                                    _stream()), "dn_block_fwd")
    return out


# ------------------------------------------------------------------------------------------------
# autograd Functions (one mesh each; gradients only w.r.t. features and parameters -- the operator
# tuple is data, SURVEY.md section 8a)
# ------------------------------------------------------------------------------------------------
class DiffusionFn(torch.autograd.Function):
    """layers.py:44-67 spectral LearnedTimeDiffusion on one mesh."""

    @staticmethod
    @_device_guard
    def forward(ctx, x, time, mass, evals, evecs):
        lib = _lib.load()
        x, mass, evals, evecs = _f32c(x), _f32c(mass), _f32c(evals), _f32c(evecs)
        V, Cc = x.shape
        K = evecs.shape[1]
        xd = torch.empty_like(x)
        x_spec = torch.empty(K, Cc, dtype=torch.float32, device=x.device)
        ws = workspace(V, K, Cc, x.device)
        # the kernel clamps `time` in place, as the reference does on the Parameter (layers.py:48-49)
        _lib.check(lib.dn_learned_time_diffusion_fwd(x.data_ptr(), mass.data_ptr(), evals.data_ptr(),
                                                     evecs.data_ptr(), time.data_ptr(), V, K, Cc, xd.data_ptr(),
                                                     x_spec.data_ptr(), ws.data_ptr(), ws.numel(), _engine,
                                                     _stream()), "dn_learned_time_diffusion_fwd")
        ctx.save_for_backward(mass, evals, evecs, time.detach().clone(), x_spec)
        return xd

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        lib = _lib.load()
        mass, evals, evecs, time, x_spec = ctx.saved_tensors
        g = _f32c(g)
        V, Cc = g.shape
        K = evecs.shape[1]
        gx = torch.empty_like(g)
        gt = torch.zeros_like(time)
        ws = workspace(V, K, Cc, g.device)
        _lib.check(lib.dn_learned_time_diffusion_bwd(g.data_ptr(), mass.data_ptr(), evals.data_ptr(),
                                                     evecs.data_ptr(), time.data_ptr(), x_spec.data_ptr(), V, K, Cc,
                                                     gx.data_ptr(), gt.data_ptr(), ws.data_ptr(), ws.numel(),
                                                     _engine, _stream()), "dn_learned_time_diffusion_bwd")
        return gx, gt, None, None, None


class _BatchUnsupported(Exception):
    """dn_learned_time_diffusion_*_batched refused the shape / engine (DN_ERR_UNSUPPORTED, nothing enqueued)."""


def _batched_ws(batch, K, Cc, device):
    # per-mesh packed multipliers (2 K C floats each) + the backward's per-mesh grad_time partials (K C / 4 floats each)
    return workspace(batch.V, K, Cc, device, extra=int(batch.n_meshes) * K * Cc * 12)


class BatchedDiffusionFn(torch.autograd.Function):
    """layers.py:44-67 spectral LearnedTimeDiffusion over every mesh of a ``batch.MeshBatch`` (``x`` in the batch layout):
    grouped to_basis, one packed multiplier per mesh and a from_basis chain that picks its weights per tile, forward and
    backward each a fixed launch sequence whatever the number of meshes (dn_learned_time_diffusion_{fwd,bwd}_batched).
    Use ``batched_diffusion``, which takes the per-mesh route where these kernels do not apply."""

    @staticmethod
    @_device_guard
    def forward(ctx, x, time, batch):
        lib = _lib.load()
        x = _f32c(x)
        V, Cc = x.shape
        K = batch.K
        B = batch.n_meshes
        xd = torch.empty_like(x)
        x_spec = torch.empty(B, K, Cc, dtype=torch.float32, device=x.device)
        ws = _batched_ws(batch, K, Cc, x.device)
        # the kernel clamps `time` in place, as the reference does on the Parameter (layers.py:48-49)
        rc = lib.dn_learned_time_diffusion_fwd_batched(x.data_ptr(), batch.mass.data_ptr(), batch.evals.data_ptr(),
                                                       batch.evecs.data_ptr(), time.data_ptr(), C.byref(batch.desc), V, K,
                                                       Cc, xd.data_ptr(), x_spec.data_ptr(), ws.data_ptr(), ws.numel(),
                                                       _engine, _stream())
        if rc == -2:                    # DN_ERR_UNSUPPORTED
            raise _BatchUnsupported()
        _lib.check(rc, "dn_learned_time_diffusion_fwd_batched")
        ctx.batch = batch
        ctx.save_for_backward(time.detach().clone(), x_spec)
        return xd

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        lib = _lib.load()
        time, x_spec = ctx.saved_tensors
        batch = ctx.batch
        g = _f32c(g)
        V, Cc = g.shape
        K = batch.K
        gx = torch.empty_like(g)
        gt = torch.zeros_like(time)
        ws = _batched_ws(batch, K, Cc, g.device)
        _lib.check(lib.dn_learned_time_diffusion_bwd_batched(g.data_ptr(), batch.mass.data_ptr(), batch.evals.data_ptr(),
                                                             batch.evecs.data_ptr(), time.data_ptr(), x_spec.data_ptr(),
                                                             C.byref(batch.desc), V, K, Cc, gx.data_ptr(), gt.data_ptr(),
                                                             ws.data_ptr(), ws.numel(), _engine, _stream()),
                   "dn_learned_time_diffusion_bwd_batched")
        return gx, gt, None


def batched_diffusion(x, time, batch):
    """Differentiable learned-time diffusion over a mesh batch (``x``: (batch.V, C) in the batch layout).  Shapes and
    engines outside the grouped kernels (the SIMT engine, K not a multiple of 64, ...) run ``DiffusionFn`` on each mesh's
    rows instead; padding rows are zero either way."""
    _require_cuda(x, time)
    if x.shape[0] != batch.V:
        raise ValueError("x is not in this batch's layout ({} rows, expected {})".format(x.shape[0], batch.V))
    try:
        return BatchedDiffusionFn.apply(x, time, batch)
    except _BatchUnsupported:
        pass
    pieces = []
    for b in range(batch.n_meshes):
        r0, n = batch.row_begin[b], batch.n_rows[b]
        pieces.append(DiffusionFn.apply(x[r0:r0 + n], time, batch.mass[r0:r0 + n], batch.evals[b], batch.evecs[r0:r0 + n]))
        pad = batch.row_begin[b + 1] - r0 - n
        if pad:
            pieces.append(x.new_zeros(pad, x.shape[1]))
    return torch.cat(pieces, dim=0)


class GradFeaturesFn(torch.autograd.Function):
    """layers.py:216-226: sparse tangent gradient + SpatialGradientFeatures, fused."""

    @staticmethod
    @_device_guard
    def forward(ctx, xd, A_re, A_im, ops):
        lib = _lib.load()
        xd, A_re = _f32c(xd), _f32c(A_re)
        A_im = _f32c(A_im) if A_im is not None else None
        V, Cc = xd.shape
        rot = A_im is not None
        feat = torch.empty_like(xd)
        pq = torch.empty(V, (2 if rot else 1) * Cc, dtype=torch.float32, device=xd.device)
        ws = workspace(V, Cc, Cc, xd.device)
        _lib.check(lib.dn_gradient_features_fwd(C.byref(ops.csr[0]), xd.data_ptr(), A_re.data_ptr(),
                                                A_im.data_ptr() if rot else None, 1 if rot else 0, V, Cc,
                                                feat.data_ptr(), pq.data_ptr(), ws.data_ptr(), ws.numel(), _engine,
                                                _stream()), "dn_gradient_features_fwd")
        ctx.ops = ops
        ctx.rot = rot
        ctx.save_for_backward(xd, pq, feat, A_re, A_im if rot else A_re)
        return feat

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        lib = _lib.load()
        xd, pq, feat, A_re, A_im = ctx.saved_tensors
        ops, rot = ctx.ops, ctx.rot
        g = _f32c(g)
        V, Cc = xd.shape
        gx = torch.empty_like(xd)
        gAre = torch.zeros_like(A_re)
        gAim = torch.zeros_like(A_im) if rot else None
        ws = workspace(V, Cc, Cc, xd.device)
        _lib.check(lib.dn_gradient_features_bwd(
            C.byref(ops.csr[0]), C.byref(ops.csr_t[0]), g.data_ptr(), xd.data_ptr(), pq.data_ptr(), feat.data_ptr(),
            A_re.data_ptr(), A_im.data_ptr() if rot else None, 1 if rot else 0, V, Cc, gx.data_ptr(),
            gAre.data_ptr(), gAim.data_ptr() if rot else None, ws.data_ptr(), ws.numel(), _engine, _stream()),
            "dn_gradient_features_bwd")
        return gx, gAre, gAim, None


class MLPFn(torch.autograd.Function):
    """cat(srcs) -> [Linear, ReLU, (Dropout)]* -> Linear (+ residual): layers.py:133-164, 229-239.

    Call as ``MLPFn.apply(n_src, n_layers, has_residual, drop_p, *srcs, *weights, *biases[, residual])``
    (a bias slot may be None)."""

    @staticmethod
    @_device_guard
    def forward(ctx, n_src, n_layers, has_res, drop_p, *t):
        lib = _lib.load()
        srcs = [_f32c(s) for s in t[:n_src]]
        weights = [_f32c(w) for w in t[n_src:n_src + n_layers]]
        biases = [(_f32c(b) if b is not None else None) for b in t[n_src + n_layers:n_src + 2 * n_layers]]
        residual = _f32c(t[n_src + 2 * n_layers]) if has_res else None
        V = srcs[0].shape[0]
        dev = srcs[0].device
        dims = [sum(s.shape[1] for s in srcs)] + [w.shape[0] for w in weights]
        for l, w in enumerate(weights):
            if w.shape[1] != dims[l]:
                raise ValueError("MiniMLP layer {} expects {} inputs, got {}".format(l, w.shape[1], dims[l]))
        need_grad = any(ctx.needs_input_grad)
        hidden = [torch.empty(V, dims[l + 1], dtype=torch.float32, device=dev) for l in range(n_layers - 1)] \
            if need_grad else []
        masks = []
        if drop_p > 0.0:
            # mask generation is RNG plumbing; applying it is fused into the layer epilogue
            masks = [torch.empty(V, dims[l + 1], dtype=torch.float32, device=dev).bernoulli_(1.0 - drop_p)
                     .mul_(1.0 / (1.0 - drop_p)) for l in range(n_layers - 1)]
        out = torch.empty(V, dims[-1], dtype=torch.float32, device=dev)
        ws = workspace(V, max(dims[1:]), max(max(dims[1:]), (max(dims) + 2) // 3), dev)
        _lib.check(lib.dn_mini_mlp_fwd(
            _lib.ptr_array([s.data_ptr() for s in srcs]), _lib.int_array([s.shape[1] for s in srcs]), n_src,
            _lib.ptr_array([w.data_ptr() for w in weights]),
            _lib.ptr_array([b.data_ptr() if b is not None else None for b in biases]), _lib.int_array(dims),
            n_layers, _lib.ptr_array([m.data_ptr() for m in masks]) if masks else None,
            residual.data_ptr() if residual is not None else None, V,
            _lib.ptr_array([h.data_ptr() for h in hidden]) if hidden else None, out.data_ptr(), ws.data_ptr(),
            ws.numel(), _engine, _stream()), "dn_mini_mlp_fwd")
        ctx.meta = (n_src, n_layers, has_res, dims, [b is not None for b in biases])
        ctx.save_for_backward(*srcs, *weights, *hidden, *masks)
        ctx.n_hidden, ctx.n_masks = len(hidden), len(masks)
        return out

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        lib = _lib.load()
        n_src, n_layers, has_res, dims, has_bias = ctx.meta
        sv = ctx.saved_tensors
        srcs = sv[:n_src]
        weights = sv[n_src:n_src + n_layers]
        hidden = sv[n_src + n_layers:n_src + n_layers + ctx.n_hidden]
        masks = sv[n_src + n_layers + ctx.n_hidden:]
        g = _f32c(g)
        V = g.shape[0]
        dev = g.device
        gs = [torch.empty_like(s) for s in srcs]
        gw = [torch.zeros_like(w) for w in weights]
        gb = [torch.zeros(w.shape[0], dtype=torch.float32, device=dev) if hb else None
              for w, hb in zip(weights, has_bias)]
        ws = workspace(V, max(dims[1:]), max(max(dims[1:]), (max(dims) + 2) // 3), dev)
        _lib.check(lib.dn_mini_mlp_bwd(
            g.data_ptr(), _lib.ptr_array([s.data_ptr() for s in srcs]),
            _lib.int_array([s.shape[1] for s in srcs]), n_src, _lib.ptr_array([w.data_ptr() for w in weights]),
            _lib.int_array(dims), n_layers, _lib.ptr_array([h.data_ptr() for h in hidden]) if hidden else None,
            _lib.ptr_array([m.data_ptr() for m in masks]) if masks else None, V,
            _lib.ptr_array([x.data_ptr() for x in gs]), _lib.ptr_array([x.data_ptr() for x in gw]),
            _lib.ptr_array([x.data_ptr() if x is not None else None for x in gb]), ws.data_ptr(), ws.numel(),
            _engine, _stream()), "dn_mini_mlp_bwd")
        res = (g,) if has_res else ()
        return (None, None, None, None, *gs, *gw, *gb, *res)


def mlp_apply(srcs, weights, biases, residual=None, drop_p=0.0):
    args = list(srcs) + list(weights) + list(biases) + ([residual] if residual is not None else [])
    return MLPFn.apply(len(srcs), len(weights), residual is not None, float(drop_p), *args)
