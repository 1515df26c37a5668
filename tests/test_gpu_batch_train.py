"""Training over mesh batches: ``DiffusionNet.forward_batch`` with autograd on (ops.BatchedDiffusionFn and the grouped
spectral forward / backward kernels, dn_learned_time_diffusion_{fwd,bwd}_batched) against the per-mesh eager route, the
fp64 restatement of the reference, the per-mesh fallback, launch counts, padding rows, and one-graph capture."""
import ctypes
import os
import sys

import pytest
import torch

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))

pytestmark = pytest.mark.gpu

# ragged batches: (n, m) torus grids of V = n * m vertices; the K = 64 set has meshes below one 128-row tile
SHAPES = {128: [(36, 50), (12, 11), (44, 50), (16, 8), (40, 51)],
          64: [(36, 50), (9, 8), (44, 50), (10, 10), (40, 51)],
          32: [(36, 50), (9, 8), (44, 50), (10, 10), (40, 51)]}
C_IN, C_OUT = 16, 8


@pytest.fixture(scope="module")
def dn():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import diffusion_net_b200 as d
    d._lib.load()
    return d


def rel_err(a, ref):
    return float((a - ref).abs().max() / (ref.abs().max() + 1e-30))


def make_net(dn, C, outputs_at="vertices", N_block=2, seed=0, C_in=C_IN, C_out=C_OUT, mlp_hidden_dims=None):
    torch.manual_seed(seed)
    net = dn.DiffusionNet(C_in=C_in, C_out=C_out, C_width=C, N_block=N_block, dropout=False, outputs_at=outputs_at,
                          mlp_hidden_dims=mlp_hidden_dims).cuda().train()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if n_.endswith("diffusion_time"):
                p_.uniform_(1e-3, 0.3)
    return net


def make_meshes(dn, K, shapes, C_in=C_IN):
    meshes = []
    for i, (n, m) in enumerate(shapes):
        mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(n, m, K, seed=i, device="cuda")
        faces = dn.synthetic.torus_mesh(n, m, seed=i)[1].cuda()
        x = torch.randn(n * m, C_in, generator=torch.Generator().manual_seed(i)).cuda()
        meshes.append(dict(mass=mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY, faces=faces, x=x))
    return meshes


def batch_of(dn, meshes):
    return dn.MeshBatch([{k: m[k] for k in ("mass", "evals", "evecs", "gradX", "gradY")} for m in meshes])


def loss_weights(outs):
    return [torch.randn(o.shape, generator=torch.Generator().manual_seed(100 + b)).cuda() for b, o in enumerate(outs)]


def per_mesh_step(net, meshes):
    """Reference route: eager per-mesh ``net(...)``, gradients accumulated over the meshes."""
    for p_ in net.parameters():
        p_.grad = None
    outs, xgrads = [], []
    for m in meshes:
        x = m["x"].clone().requires_grad_(True)
        outs.append(net(x, m["mass"], evals=m["evals"], evecs=m["evecs"], gradX=m["gradX"], gradY=m["gradY"],
                        faces=m["faces"]))
        xgrads.append(x)
    ws = loss_weights(outs)
    sum((o * w).sum() for o, w in zip(outs, ws)).backward()
    return ([o.detach().clone() for o in outs], {n_: p_.grad.clone() for n_, p_ in net.named_parameters()},
            [x.grad.clone() for x in xgrads])


def batched_step(net, mb, meshes):
    """``forward_batch`` with autograd on, the same per-mesh-summed loss."""
    for p_ in net.parameters():
        p_.grad = None
    xp = mb.pack([m["x"] for m in meshes]).requires_grad_(True)
    outs = net.forward_batch(mb, xp, faces=[m["faces"] for m in meshes])
    ws = loss_weights(outs)
    sum((o * w).sum() for o, w in zip(outs, ws)).backward()
    return ([o.detach().clone() for o in outs], {n_: p_.grad.clone() for n_, p_ in net.named_parameters()}, xp.grad)


def assert_routes_agree(net, mb, meshes, tol=2e-5):
    ref_out, ref_g, ref_x = per_mesh_step(net, meshes)
    out, g, xg = batched_step(net, mb, meshes)
    for o, r in zip(out, ref_out):
        assert o.shape == r.shape
        assert rel_err(o, r) < tol
    for name, r in ref_g.items():
        assert torch.isfinite(g[name]).all(), name
        assert rel_err(g[name], r) < tol, (name, rel_err(g[name], r))
    for b, r in enumerate(ref_x):
        assert rel_err(mb.unpack(xg)[b], r) < tol, b
    return xg


# MiniMLP hidden layers of the compared nets.  "default" is [C, C] with ReLUs.  The gradient of ReLU jumps at 0, and a
# hidden pre-activation of order 1e-7 lands on either side depending on fp32 summation order (DESIGN.md section 2): at
# C = K = 64 on these meshes that moves first_lin / diffusion_time gradients by 1e-4 between ANY two fp32 routes (the
# per-mesh loop on the exact SIMT engine vs on tc3x included).  "linear" (mlp_hidden_dims=[]: one Linear per block, no
# kink anywhere in the net) makes the 2e-5 comparison well posed at every shape.
MLPS = {"default": None, "linear": []}


@pytest.mark.parametrize("C,K,mlp", [(128, 128, "default"), (128, 128, "linear"), (64, 64, "linear")])
@pytest.mark.parametrize("outputs_at", ["vertices", "global_mean", "faces"])
def test_batched_gradients_equal_per_mesh(dn, C, K, mlp, outputs_at):
    """Every parameter's gradient, the input gradient and the outputs of ``forward_batch`` (autograd on, tc3x) match the
    per-mesh eager loop: grad_time summed over meshes by the batched backward equals the per-mesh accumulation."""
    dn.set_engine("tc3x")
    meshes = make_meshes(dn, K, SHAPES[K])
    mb = batch_of(dn, meshes)
    net = make_net(dn, C, outputs_at, mlp_hidden_dims=MLPS[mlp])
    assert_routes_agree(net, mb, meshes)


def test_batched_gradients_vs_fp64_gold(dn):
    """At a grouped-route shape (K = 64), the batched training step's gradients equal fp64 autograd through the torch
    restatement of the reference net (oracle/dn_oracle_torch.py), summed over the meshes."""
    import dn_oracle_torch as T
    dn.set_engine("tc3x")
    C, K, NB, C_in, C_out = 64, 64, 2, 3, 4
    net = make_net(dn, C, N_block=NB, C_in=C_in, C_out=C_out)
    meshes = make_meshes(dn, K, SHAPES[64][:3], C_in=C_in)
    mb = batch_of(dn, meshes)
    ys = [torch.randint(0, C_out, (m["x"].shape[0],), generator=torch.Generator().manual_seed(20 + i)).cuda()
          for i, m in enumerate(meshes)]
    for p_ in net.parameters():
        p_.grad = None
    outs = net.forward_batch(mb, [m["x"] for m in meshes])
    sum(torch.nn.functional.cross_entropy(o, y) for o, y in zip(outs, ys)).backward()
    d = torch.float64
    prm = {k: v.detach().cpu().to(d).requires_grad_(True) for k, v in net.state_dict().items()}
    for m, y in zip(meshes, ys):
        h = torch.addmm(prm["first_lin.bias"], m["x"].cpu().to(d), prm["first_lin.weight"].t()).unsqueeze(0)
        for b in range(NB):
            bp = {k[len("block_%d." % b):]: v for k, v in prm.items() if k.startswith("block_%d." % b)}
            h = T.block_forward(h, m["mass"].cpu().to(d).unsqueeze(0), m["evals"].cpu().to(d).unsqueeze(0),
                                m["evecs"].cpu().to(d).unsqueeze(0), [m["gradX"].cpu().to(d)], [m["gradY"].cpu().to(d)], bp)
        logits = torch.addmm(prm["last_lin.bias"], h[0], prm["last_lin.weight"].t())
        torch.nn.functional.cross_entropy(logits, y.cpu()).backward()
    for name, p_ in net.named_parameters():
        assert p_.grad is not None, name
        assert rel_err(p_.grad.cpu().double(), prm[name].grad) < 5e-5, name


def _raw_fwd_rc(dn, mb, C):
    """Return code of the batched forward entry point on zeros, and the kernels it launched."""
    lib = dn._lib.load()
    x = torch.zeros(mb.V, C, device="cuda")
    t = torch.full((C,), 0.1, device="cuda")
    xd = torch.empty_like(x)
    ws = dn.ops.workspace(mb.V, mb.K, C, x.device, extra=mb.n_meshes * mb.K * C * 12)
    n0 = lib.dn_kernel_launch_count()
    rc = lib.dn_learned_time_diffusion_fwd_batched(x.data_ptr(), mb.mass.data_ptr(), mb.evals.data_ptr(),
                                                   mb.evecs.data_ptr(), t.data_ptr(), ctypes.byref(mb.desc),
                                                   mb.V, mb.K, C, xd.data_ptr(), None, ws.data_ptr(), ws.numel(),
                                                   dn.ops._engine, dn.ops._stream())
    return rc, lib.dn_kernel_launch_count() - n0


@pytest.mark.parametrize("engine,C,K", [("simt", 64, 64), ("tc3x", 64, 32)])
def test_fallback_route_agrees(dn, engine, C, K):
    """The SIMT engine and K = 32 (outside the grouped chain) are refused by the batched entry points with nothing
    enqueued; ``forward_batch`` then runs the per-mesh DiffusionFn route and agrees with the per-mesh eager loop (same
    engine) and with the tensor-core per-mesh reference of the grouped-route test."""
    meshes = make_meshes(dn, K, SHAPES[K])
    mb = batch_of(dn, meshes)
    net = make_net(dn, C, "faces", mlp_hidden_dims=MLPS["linear"])
    dn.set_engine("tc3x")
    tc_ref = per_mesh_step(net, meshes)
    dn.set_engine(engine)
    try:
        rc, launched = _raw_fwd_rc(dn, mb, C)
        assert rc == -2 and launched == 0
        xg = assert_routes_agree(net, mb, meshes)
        out, g, _ = batched_step(net, mb, meshes)
    finally:
        dn.set_engine("tc3x")
    ref_out, ref_g, ref_x = tc_ref
    for o, r in zip(out, ref_out):
        assert rel_err(o, r) < 5e-5
    for name, r in ref_g.items():
        assert rel_err(g[name], r) < 5e-5, name
    for b, r in enumerate(ref_x):
        assert rel_err(mb.unpack(xg)[b], r) < 5e-5, b


def test_launches_per_step_do_not_grow_with_meshes(dn):
    """A batched training step (forward + backward) launches the same number of kernels for 2 and 5 meshes, and fewer
    than the per-mesh loop over the 5 meshes."""
    dn.set_engine("tc3x")
    lib = dn._lib.load()
    meshes = make_meshes(dn, 64, SHAPES[64])
    net = make_net(dn, 64, "vertices")

    def count(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        n0 = lib.dn_kernel_launch_count()
        fn()
        torch.cuda.synchronize()
        return lib.dn_kernel_launch_count() - n0

    counts = {}
    for nb in (2, 5):
        mb = batch_of(dn, meshes[:nb])
        counts[nb] = count(lambda: batched_step(net, mb, meshes[:nb]))
    loop = count(lambda: per_mesh_step(net, meshes))
    assert counts[2] == counts[5], counts
    assert counts[5] < loop, (counts, loop)


def test_padding_rows_and_time_clamp(dn):
    """The gradient w.r.t. the packed input is exactly 0 on padding rows and every gradient is finite; a negative
    diffusion_time is clamped to 1e-8 in place by the batched forward."""
    dn.set_engine("tc3x")
    meshes = make_meshes(dn, 64, SHAPES[64])
    mb = batch_of(dn, meshes)
    net = make_net(dn, 64, "vertices")
    t = net.blocks[0].diffusion.diffusion_time
    with torch.no_grad():
        t[:5] = -0.25
    out, g, xg = batched_step(net, mb, meshes)
    assert torch.equal(t[:5], torch.full_like(t[:5], 1e-8))
    assert float(t[5:].detach().min()) >= 1e-3
    pad = torch.ones(mb.V, dtype=torch.bool, device="cuda")
    for b in range(mb.n_meshes):
        pad[mb.row_begin[b]:mb.row_begin[b] + mb.n_rows[b]] = False
    assert bool(pad.any())
    assert bool((xg[pad] == 0).all())
    assert all(torch.isfinite(v).all() for v in g.values()) and torch.isfinite(xg).all()


def test_graphed_train_step_over_a_batch(dn):
    """graphs.GraphedTrainStep around a loss that calls ``forward_batch`` on a fixed MeshBatch: one graph for the whole
    step, whose replays give ``.grad`` bit-equal to the eager batched backward (and 2x without zeroing).  Three meshes
    below 128 vertices keep the bias gradients' column sums (cross-block float atomics, order-independent for up to two
    256-row blocks) bit-reproducible, so the comparison is exact."""
    dn.set_engine("tc3x")
    meshes = make_meshes(dn, 64, [(9, 8), (10, 10), (8, 11)])
    mb = batch_of(dn, meshes)
    assert mb.V <= 512
    net = make_net(dn, 64, "vertices")
    x = mb.pack([m["x"] for m in meshes])
    ys = [torch.randint(0, C_OUT, (m["x"].shape[0],), generator=torch.Generator().manual_seed(30 + i)).cuda()
          for i, m in enumerate(meshes)]

    def loss_fn(net_, x_, *ys_):
        outs = net_.forward_batch(mb, x_)
        return sum(torch.nn.functional.cross_entropy(o, y) for o, y in zip(outs, ys_))

    for p_ in net.parameters():
        p_.grad = None
    loss_fn(net, x, *ys).backward()
    ref = [p_.grad.clone() for p_ in net.parameters()]
    lib = dn._lib.load()
    gts = dn.graphs.GraphedTrainStep(net, loss_fn, (x, *ys))
    for _ in range(2):
        dn.graphs.GraphedTrainStep.zero_grads(net)
        n0 = lib.dn_kernel_launch_count()
        loss = gts.replay()
        torch.cuda.synchronize()
        assert lib.dn_kernel_launch_count() == n0          # replays launch the graph, not the library's kernels
        assert torch.isfinite(loss)
        for p_, r in zip(net.parameters(), ref):
            assert torch.equal(p_.grad, r)
    gts.replay()
    torch.cuda.synchronize()
    for p_, r in zip(net.parameters(), ref):
        assert torch.allclose(p_.grad, 2 * r, rtol=1e-6, atol=0)
