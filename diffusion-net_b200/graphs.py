"""CUDA-graph replay of whole-network forwards for launch-bound (small-mesh) workloads.

A 4-block DiffusionNet forward on a ~2k-vertex mesh is ~30 kernel launches of a few microseconds each;
issued eagerly from Python the GPU idles between them (BASELINE config 4: 32 such meshes).  ``GraphedNet``
captures the launch sequence of each (network, mesh) pair once into a CUDA graph and replays it; different
meshes are independent, so their graphs are replayed round-robin on several streams and overlap on the GPU.

Semantics: inference only (no autograd); the returned tensors are the graphs' static output buffers and are
overwritten by the next ``forward_batch`` on the same mesh; parameters are read at replay time, so weight
updates between calls are seen.  Graphs are keyed on the identity of the input tensors.
"""
from __future__ import annotations

import torch

from . import ops


class GraphedNet:
    def __init__(self, net, n_streams=4):
        self.net = net
        self.device = next(net.parameters()).device
        self.streams = [torch.cuda.Stream(device=self.device) for _ in range(n_streams)]
        self.cache = {}
        ops.pin_workspaces = True

    def _key(self, kw):
        return tuple((k, id(v)) for k, v in sorted(kw.items()) if v is not None)

    def _capture(self, kw, stream):
        cur = torch.cuda.current_stream(self.device)
        stream.wait_stream(cur)
        with torch.cuda.stream(stream), torch.no_grad():
            for _ in range(2):                       # warm-up: operator prep cache, workspace, allocator
                self.net(**kw)
        stream.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(g, stream=stream):
            out = self.net(**kw)
        return {"graph": g, "out": out, "stream": stream, "keep": kw}

    def forward_batch(self, items):
        """``items``: list of kwargs dicts for ``net.forward`` (x_in, mass, evals, evecs, gradX, gradY, ...)."""
        cur = torch.cuda.current_stream(self.device)
        outs, used = [], set()
        for i, kw in enumerate(items):
            key = self._key(kw)
            ent = self.cache.get(key)
            if ent is None:
                ent = self._capture(kw, self.streams[i % len(self.streams)])
                self.cache[key] = ent
            st = ent["stream"]
            if st not in used:
                st.wait_stream(cur)
                used.add(st)
            with torch.cuda.stream(st):
                ent["graph"].replay()
            outs.append(ent["out"])
        for st in used:
            cur.wait_stream(st)
        return outs


class GraphedBatch:
    """One CUDA graph for ``net.forward_batch(batch, x)`` over a ``batch.MeshBatch``: the ~27 launches of a 4-block
    net over ALL meshes of the batch replay as one graph launch (BASELINE config 4).  ``forward(x)`` copies ``x``
    (batch layout, or a per-mesh list) into the graph's static input and replays; the returned per-mesh outputs are
    views of the static output buffer (overwritten by the next call).  Inference only."""

    def __init__(self, net, batch):
        self.net, self.batch = net, batch
        self.device = batch.device
        ops.pin_workspaces = True
        self.x = torch.zeros(batch.V, net.C_in, dtype=torch.float32, device=self.device)
        self.graph = None
        self.outs = None

    def _capture(self):
        st = torch.cuda.Stream(device=self.device)
        st.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(st), torch.no_grad():
            for _ in range(2):
                self.net.forward_batch(self.batch, self.x)
        st.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(g, stream=st):
            outs = self.net.forward_batch(self.batch, self.x)
        self.graph, self.outs, self._stream = g, outs, st

    def forward(self, xs):
        x = xs if torch.is_tensor(xs) else self.batch.pack(xs)
        self.x.copy_(x)
        if self.graph is None:
            self._capture()
        self.graph.replay()
        return self.outs


class GraphedTrainStep:
    """Forward + backward of ``loss_fn(net, *inputs)`` for one fixed set of input tensors (one mesh, or a whole
    ``batch.MeshBatch`` when ``loss_fn`` calls ``net.forward_batch``) as ONE CUDA graph.

    A 4-block DiffusionNet training step on a human-seg-sized mesh is ~190 launches of 5-20 us each: eager autograd is
    launch-bound (BASELINE configs 2 and 5).  The graph is captured once per mesh (PyTorch's whole-network capture
    recipe: warm-up on a side stream, ``.grad`` buffers allocated before capture) and replayed every step; gradients
    ACCUMULATE into the parameters' ``.grad`` exactly like eager ``backward()`` does, so a data-parallel step is
    ``zero_grads(); for g in graphs: g.replay(); all-reduce; optimizer.step()``.  The inputs are the tensors passed at
    construction (update them in place to change the data); dropout must be off (the mask generation is host RNG
    plumbing, see layers.MiniMLP)."""

    def __init__(self, net, loss_fn, inputs, warmup=3):
        self.net, self.loss_fn, self.inputs = net, loss_fn, inputs
        dev = next(net.parameters()).device
        ops.pin_workspaces = True
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):                       # allocates .grad, workspaces, operator prep caches
                loss_fn(net, *inputs).backward()
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        saved = [p.grad.clone() if p.grad is not None else None for p in net.parameters()]
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = loss_fn(net, *inputs)
            self.loss.backward()
        # capture does not execute: restore what the warm-up accumulated so that the caller's zero_grad decides
        for p, g in zip(net.parameters(), saved):
            if g is not None:
                p.grad.copy_(g)

    def replay(self):
        self.graph.replay()
        return self.loss

    @staticmethod
    def zero_grads(net):
        for p in net.parameters():
            if p.grad is not None:
                p.grad.zero_()
