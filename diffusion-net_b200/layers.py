"""Drop-in mirror of ``diffusion_net.layers`` (reference ``src/diffusion_net/layers.py``) whose
per-block hot path runs the hand-written sm_100a kernels behind the C-ABI.

Same class names, constructor kwargs, forward signatures, exceptions and state_dict keys as the
reference (SURVEY.md section 8b), so shipped ``.pth`` checkpoints load with ``strict=True`` and
experiment scripts only change their import.  CUDA float32 tensors only -- there is no CPU path.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops


class LearnedTimeDiffusion(nn.Module):
    """Per-channel learned-time heat diffusion (reference layers.py:17-90).

    ``spectral``: ``evecs @ (exp(-evals t^T) * (evecs^T (mass * x)))``.  ``implicit_dense`` (a dense
    O(C V^3) Cholesky solve, toy sizes only) is outside the accelerated path and not provided."""

    def __init__(self, C_inout, method='spectral'):
        super(LearnedTimeDiffusion, self).__init__()
        self.C_inout = C_inout
        self.diffusion_time = nn.Parameter(torch.Tensor(C_inout))  # (C), reference layers.py:38
        self.method = method  # one of ['spectral', 'implicit_dense']
        nn.init.constant_(self.diffusion_time, 0.0)

    def forward(self, x, L, mass, evals, evecs):
        if x.shape[-1] != self.C_inout:  # reference layers.py:51-54
            raise ValueError(
                "Tensor has wrong shape = {}. Last dim shape should have number of channels = {}".format(
                    x.shape, self.C_inout))
        if self.method == 'spectral':
            ops._require_cuda(x, mass, evals, evecs, self.diffusion_time)
            # the clamp of layers.py:48-49 happens inside the kernel, in place on the Parameter's storage
            if x.dim() == 2:
                return ops.DiffusionFn.apply(x, self.diffusion_time, mass, evals, evecs)
            return torch.stack([ops.DiffusionFn.apply(x[b], self.diffusion_time, mass[b], evals[b], evecs[b])
                                for b in range(x.shape[0])], dim=0)
        elif self.method == 'implicit_dense':
            raise NotImplementedError("diffusion_method='implicit_dense' is outside the B200 hot path "
                                      "(dense Cholesky per channel; use the reference for toy sizes)")
        else:
            raise ValueError("unrecognized method")


class SpatialGradientFeatures(nn.Module):
    """tanh(Re(conj(z) * A z)) with a learned complex-linear A (reference layers.py:93-130).

    Input ``vectors`` (..., V, C, 2); output (..., V, C)."""

    def __init__(self, C_inout, with_gradient_rotations=True):
        super(SpatialGradientFeatures, self).__init__()
        self.C_inout = C_inout
        self.with_gradient_rotations = with_gradient_rotations
        if self.with_gradient_rotations:
            self.A_re = nn.Linear(self.C_inout, self.C_inout, bias=False)
            self.A_im = nn.Linear(self.C_inout, self.C_inout, bias=False)
        else:
            self.A = nn.Linear(self.C_inout, self.C_inout, bias=False)

    def weights(self):
        if self.with_gradient_rotations:
            return self.A_re.weight, self.A_im.weight
        return self.A.weight, None

    def forward(self, vectors):
        ops._require_cuda(vectors)
        A_re, A_im = self.weights()
        lead = vectors.shape[:-3]
        v = vectors.reshape((-1,) + tuple(vectors.shape[-3:]))
        needs_grad = torch.is_grad_enabled() and (vectors.requires_grad or A_re.requires_grad or
                                                  (A_im is not None and A_im.requires_grad))
        outs = []
        for b in range(v.shape[0]):
            if not needs_grad:
                outs.append(ops.spatial_gradient_features_raw(v[b], A_re, A_im))
            else:
                # standalone differentiable route: dense maps through the row-GEMM kernels,
                # the per-element product/tanh as autograd glue (the block itself uses the fused path)
                g0, g1 = v[b][..., 0].contiguous(), v[b][..., 1].contiguous()
                lin = lambda w, g: ops.mlp_apply([g], [w], [None])
                if A_im is not None:
                    b_re = lin(A_re, g0) - lin(A_im, g1)
                    b_im = lin(A_re, g1) + lin(A_im, g0)
                else:
                    b_re, b_im = lin(A_re, g0), lin(A_re, g1)
                outs.append(torch.tanh(g0 * b_re + g1 * b_im))
        return torch.stack(outs, 0).reshape(lead + outs[0].shape)


FUSE_HEAD = True     # DiffusionNet: compute last_lin in the last block's MiniMLP epilogue when possible (inference)


class MiniMLP(nn.Sequential):
    """[Linear, ReLU, (Dropout .5)]* Linear, with the reference submodule names (layers.py:133-164)."""

    def __init__(self, layer_sizes, dropout=False, activation=nn.ReLU, name="miniMLP"):
        super(MiniMLP, self).__init__()
        self._fused_ok = activation is nn.ReLU
        self._uses_dropout = bool(dropout)
        self._linear_names = []
        for i in range(len(layer_sizes) - 1):
            is_last = (i + 2 == len(layer_sizes))
            if dropout and i > 0:
                self.add_module(name + "_mlp_layer_dropout_{:03d}".format(i), nn.Dropout(p=.5))
            self.add_module(name + "_mlp_layer_{:03d}".format(i), nn.Linear(layer_sizes[i], layer_sizes[i + 1]))
            self._linear_names.append(name + "_mlp_layer_{:03d}".format(i))
            if not is_last:
                self.add_module(name + "_mlp_act_{:03d}".format(i), activation())

    def linears(self):
        return [getattr(self, n) for n in self._linear_names]

    def forward_sources(self, srcs, residual=None):
        """cat(srcs, -1) -> MLP (+ residual) on one mesh, the concat never materialised."""
        lins = self.linears()
        if not self._fused_ok:
            x = torch.cat(srcs, dim=-1)
            for m in self:
                x = ops.mlp_apply([x], [m.weight], [m.bias]) if isinstance(m, nn.Linear) else m(x)
            return x if residual is None else x + residual
        drop_p = 0.5 if (self._uses_dropout and self.training) else 0.0
        return ops.mlp_apply(srcs, [l.weight for l in lins], [l.bias for l in lins], residual=residual,
                             drop_p=drop_p)

    def forward(self, x):
        ops._require_cuda(x)
        lead = x.shape[:-1]
        y = self.forward_sources([x.reshape(-1, x.shape[-1])])
        return y.reshape(lead + (y.shape[-1],))


class DiffusionNetBlock(nn.Module):
    """diffusion -> tangent-gradient features -> MiniMLP -> skip (reference layers.py:167-241)."""

    def __init__(self, C_width, mlp_hidden_dims, dropout=True, diffusion_method='spectral',
                 with_gradient_features=True, with_gradient_rotations=True):
        super(DiffusionNetBlock, self).__init__()
        self.C_width = C_width
        self.mlp_hidden_dims = mlp_hidden_dims
        self.dropout = dropout
        self.with_gradient_features = with_gradient_features
        self.with_gradient_rotations = with_gradient_rotations
        self.diffusion = LearnedTimeDiffusion(self.C_width, method=diffusion_method)
        self.MLP_C = 2 * self.C_width
        if self.with_gradient_features:
            self.gradient_features = SpatialGradientFeatures(
                self.C_width, with_gradient_rotations=self.with_gradient_rotations)
            self.MLP_C += self.C_width
        self.mlp = MiniMLP([self.MLP_C] + self.mlp_hidden_dims + [self.C_width], dropout=self.dropout)

    def _forward_mesh(self, x_in, mass, evals, evecs, gops, fused, head=None):
        A_re = A_im = None
        if self.with_gradient_features:
            A_re, A_im = self.gradient_features.weights()
        if fused:  # inference: one C-ABI call, nothing saved (dn_block_fwd)
            lins = self.mlp.linears()
            return ops.block_forward_raw(x_in, mass, evals, evecs, gops, self.diffusion.diffusion_time, A_re, A_im,
                                         [l.weight for l in lins], [l.bias for l in lins],
                                         self.with_gradient_features, head=head)
        if head is not None:
            raise ops.HeadNotFused()
        x_diffuse = self.diffusion(x_in, None, mass, evals, evecs)
        srcs = [x_in, x_diffuse]
        if self.with_gradient_features:
            srcs.append(ops.GradFeaturesFn.apply(x_diffuse, A_re, A_im, gops))
        return self.mlp.forward_sources(srcs, residual=x_in)   # layers.py:229-239

    def forward(self, x_in, mass, L, evals, evecs, gradX, gradY, head=None):
        """Reference signature (layers.py:200); ``head=(weight, bias)`` is this package's extension: a linear head fused
        behind the block in inference (returns the head's output; raises ops.HeadNotFused when it cannot be fused)."""
        B = x_in.shape[0]
        if x_in.shape[-1] != self.C_width:  # reference layers.py:204-207
            raise ValueError(
                "Tensor has wrong shape = {}. Last dim shape should have number of channels = {}".format(
                    x_in.shape, self.C_width))
        ops._require_cuda(x_in, mass, evals, evecs)
        if self.diffusion.method != 'spectral':
            self.diffusion(x_in, L, mass, evals, evecs)   # raises like the reference would route
        gops = [None] * B
        if self.with_gradient_features:
            if isinstance(gradX, (list, tuple)):           # pre-split per-mesh operators
                # an element may already be a prepared ops.GradOperators (geometry.get_operators /
                # GradOperators.from_csr): it then stands for the (gradX, gradY) pair and gradY[b] is ignored
                gys = gradY if gradY is not None else [None] * len(gradX)
                gops = [gx if isinstance(gx, ops.GradOperators) else ops.prepare_operators(gx, gy)
                        for gx, gy in zip(gradX, gys)]
            else:
                gops = ops.prepare_operators_batched(gradX, gradY)
        params_need_grad = any(p.requires_grad for p in self.parameters())
        needs_grad = torch.is_grad_enabled() and (x_in.requires_grad or params_need_grad)
        fused = (not needs_grad) and self.mlp._fused_ok and not (self.training and self.dropout)
        if head is not None and not fused:
            raise ops.HeadNotFused()
        outs = [self._forward_mesh(x_in[b], mass[b], evals[b], evecs[b], gops[b], fused, head) for b in range(B)]
        return torch.stack(outs, dim=0)

    def forward_batch(self, batch, x_in):
        """Differentiable block over every mesh of a ``batch.MeshBatch`` (``x_in``: (batch.V, C_width) in the batch
        layout): batched spectral diffusion, the gradient features on the block-diagonal CSR and the MiniMLP, each one
        launch sequence over all meshes.  Training-mode dropout applies (MiniMLP masks)."""
        if self.diffusion.method != 'spectral':
            raise NotImplementedError("forward_batch: spectral diffusion only")
        x_diffuse = ops.batched_diffusion(x_in, self.diffusion.diffusion_time, batch)
        srcs = [x_in, x_diffuse]
        if self.with_gradient_features:
            A_re, A_im = self.gradient_features.weights()
            srcs.append(ops.GradFeaturesFn.apply(x_diffuse, A_re, A_im, batch.gops))
        return self.mlp.forward_sources(srcs, residual=x_in)   # layers.py:229-239


class DiffusionNet(nn.Module):

    def __init__(self, C_in, C_out, C_width=128, N_block=4, last_activation=None, outputs_at='vertices',
                 mlp_hidden_dims=None, dropout=True, with_gradient_features=True, with_gradient_rotations=True,
                 diffusion_method='spectral'):
        """Same parameters as the reference ``DiffusionNet`` (layers.py:246-263)."""
        super(DiffusionNet, self).__init__()
        self.C_in = C_in
        self.C_out = C_out
        self.C_width = C_width
        self.N_block = N_block
        self.last_activation = last_activation
        self.outputs_at = outputs_at
        if outputs_at not in ['vertices', 'edges', 'faces', 'global_mean']:
            raise ValueError("invalid setting for outputs_at")
        if mlp_hidden_dims == None:
            mlp_hidden_dims = [C_width, C_width]
        self.mlp_hidden_dims = mlp_hidden_dims
        self.dropout = dropout
        self.diffusion_method = diffusion_method
        if diffusion_method not in ['spectral', 'implicit_dense']:
            raise ValueError("invalid setting for diffusion_method")
        self.with_gradient_features = with_gradient_features
        self.with_gradient_rotations = with_gradient_rotations

        self.first_lin = nn.Linear(C_in, C_width)
        self.last_lin = nn.Linear(C_width, C_out)
        self.blocks = []
        for i_block in range(self.N_block):
            block = DiffusionNetBlock(C_width=C_width, mlp_hidden_dims=mlp_hidden_dims, dropout=dropout,
                                      diffusion_method=diffusion_method,
                                      with_gradient_features=with_gradient_features,
                                      with_gradient_rotations=with_gradient_rotations)
            self.blocks.append(block)
            self.add_module("block_" + str(i_block), self.blocks[-1])

    def _linear(self, lin, x):
        B = x.shape[0]
        return torch.stack([ops.mlp_apply([x[b]], [lin.weight], [lin.bias]) for b in range(B)], 0)

    def forward_batch(self, batch, xs, edges=None, faces=None):
        """The network over a ``batch.MeshBatch`` of independent meshes in ONE launch sequence (BASELINE configs 4 and
        5): the reference's per-mesh loop (layers.py:217-222, 366-401) with every stage of every block launched once over
        all meshes.  ``xs``: list of per-mesh (V_b, C_in) features, or one tensor already in the batch layout.
        ``edges`` / ``faces``: lists of per-mesh (E_b, 2) / (F_b, 3) vertex indices local to each mesh, for
        ``outputs_at`` 'edges' / 'faces'.  Returns the list of per-mesh outputs.  Equal to ``[self(x_b, mass_b, ...) for
        b]`` (tests/test_gpu_parity.py, tests/test_gpu_batch_train.py).

        Under ``torch.no_grad()`` (or with nothing to differentiate) this is the fused inference route
        (``dn_block_fwd_batched``, last_lin fused when possible).  With autograd on it is differentiable: first_lin ->
        per block ``DiffusionNetBlock.forward_batch`` -> last_lin over the whole range, so a training step over any
        number of meshes is one fixed launch sequence (and can be captured as one graph, graphs.GraphedTrainStep)."""
        if self.diffusion_method != 'spectral':
            raise NotImplementedError("forward_batch: spectral diffusion only")
        elems = None
        if self.outputs_at in ('edges', 'faces'):
            elems = edges if self.outputs_at == 'edges' else faces
            if elems is None or len(elems) != batch.n_meshes:
                raise ValueError("forward_batch with outputs_at='{}' needs one index tensor per mesh in `{}`".format(
                    self.outputs_at, self.outputs_at))
        x = xs if torch.is_tensor(xs) else batch.pack(xs)
        if x.shape[-1] != self.C_in:
            raise ValueError("DiffusionNet was constructed with C_in={}, but x_in has last dim={}".format(
                self.C_in, x.shape[-1]))
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            _ = batch.gops.csr_t           # the gather's backward needs the transposed CSR: build it now, not mid-capture
            x = ops.mlp_apply([x], [self.first_lin.weight], [self.first_lin.bias])
            for blk in self.blocks:
                x = blk.forward_batch(batch, x)
            x = ops.mlp_apply([x], [self.last_lin.weight], [self.last_lin.bias])
        else:
            x = self._forward_batch_fused(batch, x)
        outs = batch.unpack(x)
        if elems is not None:
            # mean of the per-vertex outputs over each element's corners, as ``forward`` does
            outs = [o[e].mean(dim=1) for o, e in zip(outs, elems)]
        elif self.outputs_at == 'global_mean':
            res = []
            for b, o in enumerate(outs):
                m = batch.mass[batch.row_begin[b]:batch.row_begin[b] + batch.n_rows[b]]
                res.append((o * (m / m.sum()).unsqueeze(-1)).sum(dim=-2))
            outs = res
        if self.last_activation != None:
            outs = [self.last_activation(o) for o in outs]
        return outs

    def _forward_batch_fused(self, batch, x):
        """Inference route of ``forward_batch``: batch-layout input -> per-vertex outputs (V, C_out), batch layout."""
        from . import batch as _batch
        x = ops.mlp_apply([x], [self.first_lin.weight], [self.first_lin.bias])
        fuse_head = FUSE_HEAD and ops.head_fusable(self.C_out)
        head_done = False
        for i_b, blk in enumerate(self.blocks):
            if blk.training and blk.dropout:
                raise RuntimeError("forward_batch under no_grad: eval mode only (dropout); training-mode dropout runs "
                                   "with autograd on")
            A_re = A_im = None
            if blk.with_gradient_features:
                A_re, A_im = blk.gradient_features.weights()
            lins = blk.mlp.linears()
            args = (batch, x, blk.diffusion.diffusion_time, A_re, A_im, [l.weight for l in lins], [l.bias for l in lins],
                    blk.with_gradient_features)
            if fuse_head and i_b + 1 == len(self.blocks):
                try:
                    x = _batch.block_forward_batched_raw(*args, head=(self.last_lin.weight, self.last_lin.bias))
                    head_done = True
                    break
                except ops.HeadNotFused:
                    pass
            x = _batch.block_forward_batched_raw(*args)
        if not head_done:
            x = ops.mlp_apply([x], [self.last_lin.weight], [self.last_lin.bias])
        return x

    def forward(self, x_in, mass, L=None, evals=None, evecs=None, gradX=None, gradY=None, edges=None, faces=None):
        """[N,C] or [B,N,C] in, [N,C_out] or [B,N,C_out] out (reference layers.py:314-407)."""
        if x_in.shape[-1] != self.C_in:
            raise ValueError("DiffusionNet was constructed with C_in={}, but x_in has last dim={}".format(
                self.C_in, x_in.shape[-1]))
        if len(x_in.shape) not in (2, 3):
            raise ValueError("x_in should be tensor with shape [N,C] or [B,N,C]")
        ops._require_cuda(x_in, mass)
        if len(x_in.shape) == 2:
            appended_batch_dim = True
            x_in = x_in.unsqueeze(0)
            mass = mass.unsqueeze(0)
            if evals != None: evals = evals.unsqueeze(0)
            if evecs != None: evecs = evecs.unsqueeze(0)
            # sparse operators stay un-batched: wrapping them in 1-element lists keeps the user's
            # tensor objects (and the CSR prepared from them) alive across blocks and epochs
            if gradX != None: gradX = [gradX]
            if gradY != None: gradY = [gradY]
            if edges != None: edges = edges.unsqueeze(0)
            if faces != None: faces = faces.unsqueeze(0)
        else:
            appended_batch_dim = False

        x = self._linear(self.first_lin, x_in)
        # last_lin rides in the last block's MiniMLP epilogue when it can (inference, <= 8 outputs, fused tensor-core chain):
        # the C_width-wide output of the last block is then never written (SURVEY.md 8f-1)
        fuse_head = FUSE_HEAD and len(self.blocks) > 0 and ops.head_fusable(self.C_out) and not torch.is_grad_enabled()
        for i_b, b in enumerate(self.blocks):
            if fuse_head and i_b + 1 == len(self.blocks):
                try:
                    x = b(x, mass, L, evals, evecs, gradX, gradY, head=(self.last_lin.weight, self.last_lin.bias))
                    break
                except ops.HeadNotFused:
                    fuse_head = False
            x = b(x, mass, L, evals, evecs, gradX, gradY)
        if not fuse_head:
            x = self._linear(self.last_lin, x)

        # remap to edges / faces / global mean: callers' side of the hot path (SURVEY.md 8f row 1)
        if self.outputs_at in ('edges', 'faces'):
            # mean of the per-vertex outputs over each element's corners
            elems = edges if self.outputs_at == 'edges' else faces
            x_out = torch.stack([x[b][elems[b]].mean(dim=1) for b in range(x.shape[0])], dim=0)
        elif self.outputs_at == 'global_mean':
            # area-weighted mean (discretisation invariant)
            w = mass / mass.sum(dim=-1, keepdim=True)
            x_out = (x * w.unsqueeze(-1)).sum(dim=-2)
        else:
            x_out = x

        if self.last_activation != None:
            x_out = self.last_activation(x_out)
        if appended_batch_dim:
            x_out = x_out.squeeze(0)
        return x_out
