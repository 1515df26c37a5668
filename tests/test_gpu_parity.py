"""Parity of the CUDA path (through the C-ABI) with the fp64 gold of the unmodified reference
(tests/golden, written by oracle/make_golden.py) and with the numpy oracle on seeded inputs.

Tolerance: north_star asks for 1e-5 relative fp32; the metric is max|ours - gold| / max|gold|
(SURVEY.md section 8c).  TOL below is that bound; the exact-fp32 SIMT engine is held to 2e-6.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import load_golden, golden_params, ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import dn_oracle as O  # noqa: E402  (checker only)

pytestmark = pytest.mark.gpu

TOL = {"tc3x": 1e-5, "simt": 3e-6}
ENGINES = ["simt", "tc3x"]


@pytest.fixture(scope="module")
def dn():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import diffusion_net_b200 as d
    d._lib.load()
    return d


def dev(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


def sparse_pair(fx, prefix=""):
    V = fx[prefix + "mass"].shape[0]
    idx = torch.from_numpy(np.stack((fx[prefix + "g_rows"], fx[prefix + "g_cols"])).astype(np.int64))
    gx = torch.sparse_coo_tensor(idx, torch.from_numpy(fx[prefix + "gx_vals"]), (V, V)).coalesce().cuda()
    gy = torch.sparse_coo_tensor(idx, torch.from_numpy(fx[prefix + "gy_vals"]), (V, V)).coalesce().cuda()
    return gx, gy


def oracle_ops(fx, prefix=""):
    V = fx[prefix + "mass"].shape[0]
    r, c = fx[prefix + "g_rows"].astype(np.int64), fx[prefix + "g_cols"].astype(np.int64)
    f = np.float64
    return (fx[prefix + "mass"].astype(f), fx[prefix + "evals"].astype(f), fx[prefix + "evecs"].astype(f),
            O.coo_to_csr(r, c, fx[prefix + "gx_vals"].astype(f), (V, V)),
            O.coo_to_csr(r, c, fx[prefix + "gy_vals"].astype(f), (V, V)))


def make_block(dn, C, params, **kw):
    blk = dn.DiffusionNetBlock(C_width=C, mlp_hidden_dims=[C, C], dropout=False, **kw)
    blk.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in params.items()}, strict=True)
    return blk.cuda().eval()


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name,kw", [("block_small", {}), ("block_norot", {"with_gradient_rotations": False}),
                                     ("block_nograd", {"with_gradient_features": False})])
def test_block_forward_golden(dn, engine, name, kw):
    dn.set_engine(engine)
    base = load_golden("block_small")
    fx = load_golden(name)
    C = fx["x_in"].shape[1]
    blk = make_block(dn, C, golden_params(fx), **kw)
    gx, gy = sparse_pair(base)
    b = lambda a: dev(a).unsqueeze(0)
    with torch.no_grad():
        out = blk(b(fx["x_in"]), b(base["mass"]), None, b(base["evals"]), b(base["evecs"]),
                  gx.unsqueeze(0), gy.unsqueeze(0))
    assert out.shape == (1,) + fx["x_in"].shape
    assert O.rel_err(out[0].cpu().numpy(), fx["out_f64"]) < TOL[engine]
    # in-place clamp side effect on the Parameter (layers.py:48-49)
    np.testing.assert_array_equal(blk.diffusion.diffusion_time.detach().cpu().numpy(), fx["time_after_f32"])
    assert isinstance(blk.diffusion.diffusion_time, torch.nn.Parameter)


@pytest.mark.parametrize("engine", ENGINES)
def test_block_k128_golden(dn, engine):
    dn.set_engine(engine)
    fx = load_golden("block_k128")
    blk = make_block(dn, 128, golden_params(fx))
    gx, gy = sparse_pair(fx)
    b = lambda a: dev(a).unsqueeze(0)
    with torch.no_grad():
        xd = blk.diffusion(b(fx["x_in"]), None, b(fx["mass"]), b(fx["evals"]), b(fx["evecs"]))
        out = blk(b(fx["x_in"]), b(fx["mass"]), None, b(fx["evals"]), b(fx["evecs"]), gx.unsqueeze(0),
                  gy.unsqueeze(0))
    assert O.rel_err(xd[0].cpu().numpy(), fx["x_diffuse_f64_as32"]) < TOL[engine]
    assert O.rel_err(out[0].cpu().numpy(), fx["out_f64_as32"]) < TOL[engine]


@pytest.mark.parametrize("engine", ENGINES)
def test_components_vs_oracle(dn, engine):
    """to_basis / from_basis / grad spmm / SpatialGradientFeatures / MiniMLP, each through its C-ABI call."""
    dn.set_engine(engine)
    fx = load_golden("block_small")
    p = golden_params(fx, np.float64)
    mass, evals, evecs, gX, gY = oracle_ops(fx)
    x64 = fx["x_in"].astype(np.float64)
    x = dev(fx["x_in"])
    spec = dn.to_basis(x, dev(fx["evecs"]), dev(fx["mass"]))
    assert O.rel_err(spec.cpu().numpy(), O.to_basis(x64, evecs, mass)) < TOL[engine]
    back = dn.from_basis(spec, dev(fx["evecs"]))
    assert O.rel_err(back.cpu().numpy(), O.from_basis(spec.double().cpu().numpy(), evecs)) < TOL[engine]
    # batched signatures
    specb = dn.to_basis(x.unsqueeze(0), dev(fx["evecs"]).unsqueeze(0), dev(fx["mass"]).unsqueeze(0))
    assert specb.shape == (1,) + spec.shape
    gx, gy = sparse_pair(fx)
    gops = dn.prepare_operators(gx, gy)
    xd = dev(fx["x_diffuse_f32"])
    vc2 = dn.ops.grad_spmm_raw(gops, xd)
    ref_vc2 = O.grad_spmm(gX, gY, fx["x_diffuse_f32"].astype(np.float64))
    assert O.rel_err(vc2.cpu().numpy(), ref_vc2) < TOL[engine]
    sgf = dn.SpatialGradientFeatures(32).cuda()
    sgf.load_state_dict({"A_re.weight": torch.from_numpy(fx["p:gradient_features.A_re.weight"]),
                         "A_im.weight": torch.from_numpy(fx["p:gradient_features.A_im.weight"])})
    with torch.no_grad():
        f = sgf(vc2)
    ref_f = O.spatial_gradient_features(vc2.double().cpu().numpy(), A_re=p["gradient_features.A_re.weight"],
                                        A_im=p["gradient_features.A_im.weight"])
    assert O.rel_err(f.cpu().numpy(), ref_f) < TOL[engine]
    mlp = dn.MiniMLP([96, 32, 32, 32]).cuda()
    mlp.load_state_dict({k[len("mlp."):]: torch.from_numpy(v) for k, v in golden_params(fx).items()
                         if k.startswith("mlp.")})
    comb = np.concatenate((fx["x_in"], fx["x_diffuse_f32"], fx["x_grad_features_f32"]), axis=-1)
    with torch.no_grad():
        y = mlp(dev(comb))
    ws = [p["mlp.miniMLP_mlp_layer_{:03d}.weight".format(i)] for i in range(3)]
    bs = [p["mlp.miniMLP_mlp_layer_{:03d}.bias".format(i)] for i in range(3)]
    assert O.rel_err(y.cpu().numpy(), O.mini_mlp(comb.astype(np.float64), ws, bs)) < TOL[engine]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("mode", ["vertices", "edges", "faces", "global_mean"])
def test_net_golden(dn, engine, mode):
    dn.set_engine(engine)
    fx = load_golden("net_small")
    net = dn.DiffusionNet(C_in=3, C_out=8, C_width=32, N_block=2, dropout=False, outputs_at=mode)
    net.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in golden_params(fx).items()}, strict=True)
    net = net.cuda().eval()
    gx, gy = sparse_pair(fx, "m0_")
    with torch.no_grad():
        out = net(dev(fx["verts0"]), dev(fx["m0_mass"]), L=None, evals=dev(fx["m0_evals"]),
                  evecs=dev(fx["m0_evecs"]), gradX=gx, gradY=gy,
                  edges=dev(fx["edges"], torch.int64), faces=dev(fx["faces"], torch.int64))
    gold = fx["out_{}_f64".format(mode)]
    assert out.shape == gold.shape
    assert O.rel_err(out.cpu().numpy(), gold) < TOL[engine] * 3   # 2 blocks + 2 linears deep


def test_net_batched_sparse(dn):
    """The reference's stacked (B,V,V) sparse operators (B=2) equal per-mesh results."""
    dn.set_engine("tc3x")
    fx = load_golden("net_small")
    net = dn.DiffusionNet(C_in=3, C_out=8, C_width=32, N_block=2, dropout=False)
    net.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in golden_params(fx).items()}, strict=True)
    net = net.cuda().eval()
    g0x, g0y = sparse_pair(fx, "m0_")
    g1x, g1y = sparse_pair(fx, "m1_")
    st = lambda a, b: torch.stack((dev(fx[a]), dev(fx[b])), 0)
    with torch.no_grad():
        out = net(st("verts0", "verts1"), st("m0_mass", "m1_mass"), L=None, evals=st("m0_evals", "m1_evals"),
                  evecs=st("m0_evecs", "m1_evecs"), gradX=torch.stack((g0x, g1x), 0),
                  gradY=torch.stack((g0y, g1y), 0))
    assert O.rel_err(out.cpu().numpy(), fx["out_batch2_f64"]) < 3e-5


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name,kw", [("block_small", {}), ("block_norot", {"with_gradient_rotations": False}),
                                     ("block_nograd", {"with_gradient_features": False})])
def test_block_backward_golden(dn, engine, name, kw):
    """Gradients of sum(out*R) w.r.t. x_in and every parameter vs the reference's own autograd (fp64)."""
    dn.set_engine(engine)
    base = load_golden("block_small")
    fx = load_golden(name)
    C = fx["x_in"].shape[1]
    blk = make_block(dn, C, golden_params(fx), **kw).train()   # dropout=False => train == eval numerics
    gx, gy = sparse_pair(base)
    b = lambda a: dev(a).unsqueeze(0)
    x = b(fx["x_in"]).requires_grad_(True)
    out = blk(x, b(base["mass"]), None, b(base["evals"]), b(base["evecs"]), gx.unsqueeze(0), gy.unsqueeze(0))
    assert O.rel_err(out[0].detach().cpu().numpy(), fx["out_f64"]) < TOL[engine]
    (out[0] * dev(fx["loss_R"])).sum().backward()
    assert O.rel_err(x.grad[0].cpu().numpy(), fx["g:x_in"]) < 2e-5
    for n, prm in blk.named_parameters():
        assert prm.grad is not None, n
        assert O.rel_err(prm.grad.cpu().numpy(), fx["g:" + n]) < 5e-5, n


@pytest.mark.parametrize("engine", ENGINES)
def test_block_backward_config2_shape_vs_oracle_autograd(dn, engine):
    """BASELINE config 2 shape (human-seg class: V ~ 7k, K = 128, C = 128): forward + backward of one block against
    fp64 autograd through the torch restatement of the reference block (oracle/dn_oracle_torch.py, itself pinned to
    the live reference by tests/test_oracle.py).  This is the shape the tensor-core backward (rows_chain3 dX layers,
    split-V tcgen05 weight gradients) is built for.  Tolerances as in the golden backward test."""
    import dn_oracle_torch as T
    dn.set_engine(engine)
    n, m, K, C = 84, 84, 128, 128
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(n, m, K, seed=3, device="cuda")
    V = n * m
    params = dn.synthetic.block_weights(C, seed=3)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(V, C, generator=g)
    R = torch.randn(V, C, generator=g)
    blk = dn.DiffusionNetBlock(C_width=C, mlp_hidden_dims=[C, C], dropout=False)
    blk.load_state_dict(params, strict=True)
    blk = blk.cuda().train()
    xg = x.cuda().unsqueeze(0).requires_grad_(True)
    out = blk(xg, mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gX], [gY])
    # gold: fp64 on the CPU.  ReLU's gradient is discontinuous at 0: a hidden pre-activation of order 1e-7 may land
    # on the other side of the kink in an fp32 forward (ours or the reference's own), which changes a whole row of the
    # input gradient.  So (1) our activation pattern may differ from the fp64 one only where the fp64 pre-activation
    # is within fp32 rounding of 0, and (2) the gradients are compared under OUR activation pattern.
    node, stack = None, [out.grad_fn]
    while stack and node is None:
        f = stack.pop()
        if f is None:
            continue
        if "MLPFn" in type(f).__name__:
            node = f
        stack.extend(nf for nf, _ in f.next_functions)
    assert node is not None, "the MiniMLP autograd node was not found"
    ours_hidden = [h for h in node.saved_tensors[6:8]]      # 3 sources, 3 weights, then the 2 hidden activations
    assert [tuple(h.shape) for h in ours_hidden] == [(V, C), (V, C)]
    masks = [(h > 0).cpu() for h in ours_hidden]
    (out[0] * R.cuda()).sum().backward()
    d = torch.float64
    prm = {k: v.to(d).requires_grad_(True) for k, v in params.items()}
    x64 = x.to(d).unsqueeze(0).requires_grad_(True)
    gxc, gyc = gX.cpu().to(d), gY.cpu().to(d)
    pre = []
    gold = T.block_forward(x64, mass.cpu().to(d).unsqueeze(0), evals.cpu().to(d).unsqueeze(0),
                           evecs.cpu().to(d).unsqueeze(0), [gxc], [gyc], prm, relu_masks=masks, pre_acts=pre)
    (gold[0] * R.to(d)).sum().backward()
    for mk, pa in zip(masks, pre):
        pa = pa.reshape(mk.shape)
        flips = mk != (pa > 0)
        assert int(flips.sum()) <= 8
        assert float(pa[flips].abs().max() if flips.any() else 0.0) < 1e-5 * float(pa.abs().max())
    assert O.rel_err(out[0].detach().cpu().numpy(), gold[0].detach().numpy()) < TOL[engine]
    assert O.rel_err(xg.grad[0].cpu().numpy(), x64.grad[0].numpy()) < 2e-5
    for name, p_ in blk.named_parameters():
        assert p_.grad is not None, name
        assert O.rel_err(p_.grad.cpu().numpy(), prm[name].grad.numpy()) < 5e-5, name


def test_errors_and_no_cpu_fallback(dn):
    blk = dn.DiffusionNetBlock(C_width=32, mlp_hidden_dims=[32, 32], dropout=False)
    x = torch.zeros(1, 10, 32)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        blk(x, torch.ones(1, 10), None, torch.zeros(1, 4), torch.zeros(1, 10, 4), None, None)
    with pytest.raises(ValueError, match="wrong shape"):
        blk.cuda()(torch.zeros(1, 10, 5).cuda(), torch.ones(1, 10).cuda(), None, torch.zeros(1, 4).cuda(),
                   torch.zeros(1, 10, 4).cuda(), None, None)
    with pytest.raises(ValueError):
        dn.DiffusionNet(3, 4, outputs_at="nowhere")
    with pytest.raises(ValueError, match="C_in=3"):
        dn.DiffusionNet(3, 4, C_width=32).cuda()(torch.zeros(10, 4).cuda(), torch.ones(10).cuda())


_NOT_SM100_SCRIPT = r'''
import ctypes as C, sys, types
sys.path.insert(0, %r)
import torch
import diffusion_net_b200 as dn
from diffusion_net_b200 import _lib, ops
lib = _lib.load()
assert dn.get_engine() == "tc3x"
K = W = 64
mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(12, 16, K, seed=0, device="cuda")
V = mass.shape[0]
g = torch.Generator().manual_seed(0)
rnd = lambda *s: torch.randn(*s, generator=g).cuda()
x, spec, time = rnd(V, W), rnd(K, W), torch.full((W,), 0.1, device="cuda")
A_re, A_im, pq, hidden = rnd(W, W), rnd(W, W), rnd(V, 2 * W), [rnd(V, W), rnd(V, W)]
wts, bias = [rnd(W, 3 * W), rnd(W, W), rnd(W, W)], [rnd(W), rnd(W), rnd(W)]
head = (rnd(4, W), rnd(4))
gops = ops.GradOperators(gX, gY)
gops.csr_t
mb = dn.MeshBatch([dict(mass=mass, evals=evals, evecs=evecs, gradX=gops)] * 2)
xb, specb = rnd(mb.V, W), rnd(2, K, W)
out, gA_re, gA_im = torch.empty_like(x), rnd(W, W), rnd(W, W)
outb = torch.empty_like(xb)
ws = ops.workspace(mb.V, K, 3 * W, x.device, extra=2 * K * W * 12)
prm = _lib.dn_block_params(time.data_ptr(), A_re.data_ptr(), A_im.data_ptr(), 1, 1, 3,
                           _lib.ptr_array([w.data_ptr() for w in wts]), _lib.ptr_array([b.data_ptr() for b in bias]),
                           _lib.int_array([3 * W, W, W, W]))
ctx = types.SimpleNamespace
calls = {
    "dn_to_basis": lambda: ops.to_basis_raw(x, evecs, mass),
    "dn_from_basis": lambda: ops.from_basis_raw(spec, evecs),
    "dn_learned_time_diffusion_fwd": lambda: ops.DiffusionFn.apply(x, time, mass, evals, evecs),
    "dn_learned_time_diffusion_bwd": lambda: ops.DiffusionFn.backward(ctx(saved_tensors=(mass, evals, evecs, time, spec)), x),
    "dn_learned_time_diffusion_fwd_batched": lambda: ops.BatchedDiffusionFn.apply(xb, time, mb),
    "dn_learned_time_diffusion_bwd_batched": lambda: ops.BatchedDiffusionFn.backward(
        ctx(batch=mb, saved_tensors=(time, specb)), xb),
    "dn_gradient_features_fwd": lambda: ops.GradFeaturesFn.apply(x, A_re, A_im, gops),
    "dn_gradient_features_bwd": lambda: _lib.check(lib.dn_gradient_features_bwd(
        C.byref(gops.csr[0]), C.byref(gops.csr_t[0]), x.data_ptr(), x.data_ptr(), pq.data_ptr(), x.data_ptr(),
        A_re.data_ptr(), A_im.data_ptr(), 1, V, W, out.data_ptr(), gA_re.data_ptr(), gA_im.data_ptr(), ws.data_ptr(),
        ws.numel(), ops._engine, ops._stream()), "dn_gradient_features_bwd"),
    "dn_mini_mlp_fwd": lambda: ops.mlp_apply([x, x, x], wts, bias, residual=x),
    "dn_mini_mlp_bwd": lambda: ops.MLPFn.backward(ctx(meta=(3, 3, True, [3 * W, W, W, W], [True] * 3),
                                                      saved_tensors=(x, x, x, *wts, *hidden), n_hidden=2, n_masks=0), x),
    "dn_block_fwd": lambda: ops.block_forward_raw(x, mass, evals, evecs, gops, time, A_re, A_im, wts, bias, True),
    "dn_block_fwd_profile": lambda: ops.block_forward_raw(x, mass, evals, evecs, gops, time, A_re, A_im, wts, bias, True,
                                                          profile=[]),
    "dn_block_fwd_ex (head)": lambda: ops.block_forward_raw(x, mass, evals, evecs, gops, time, A_re, A_im, wts, bias,
                                                            True, head=head),
    "dn_block_fwd_ex (batch)": lambda: dn.batch.block_forward_batched_raw(mb, xb, time, A_re, A_im, wts, bias, True),
    "dn_block_fwd_batched": lambda: _lib.check(lib.dn_block_fwd_batched(
        xb.data_ptr(), mb.mass.data_ptr(), mb.evals.data_ptr(), mb.evecs.data_ptr(), C.byref(mb.gops.csr[0]),
        C.byref(prm), C.byref(mb.desc), mb.V, K, W, outb.data_ptr(), ws.data_ptr(), ws.numel(), ops._engine,
        ops._stream()), "dn_block_fwd_batched"),
}
torch.cuda.synchronize()
bad = []
for name, fn in calls.items():
    n0 = lib.dn_kernel_launch_count()
    try:
        fn()
        err = "returned normally"
    except RuntimeError as e:
        err = repr(e)
    launched = lib.dn_kernel_launch_count() - n0
    if "(-4)" not in err or launched:
        bad.append("{}: {}, {} kernels enqueued".format(name, err, launched))
print("\n".join(bad) if bad else "ALL_NOT_SM100")
'''


def test_tensor_core_engine_on_unsupported_device_enqueues_nothing(dn):
    """With tcgen05 unavailable (DN_TC_DISABLE=1), every tensor-core-capable entry point under the tc3x engine fails
    with DN_ERR_NOT_SM100 before it enqueues a kernel: no silent SIMT fallback and no partial work on the stream."""
    env = dict(os.environ, DN_TC_DISABLE="1", DN_B200_ENGINE="tc3x")
    r = subprocess.run([sys.executable, "-c", _NOT_SM100_SCRIPT % ROOT], capture_output=True, text=True, timeout=600,
                       env=env)
    assert r.returncode == 0 and r.stdout.strip().endswith("ALL_NOT_SM100"), r.stdout + r.stderr


def _structural_case(dn, n, m, K, C, seed=0, **kw):
    ops_t = dn.synthetic.structural_operators(n, m, K, seed=seed, device="cuda", **kw)
    params = dn.synthetic.block_weights(C, seed=seed)
    x = torch.randn(n * m, C, generator=torch.Generator().manual_seed(seed)).cuda()
    return ops_t, params, x


def _oracle_block(ops_t, params, x):
    mass, L, evals, evecs, gradX, gradY = ops_t
    gxc, gyc = gradX.coalesce().cpu(), gradY.coalesce().cpu()
    V = mass.shape[0]
    f = np.float64
    gX = O.coo_to_csr(gxc.indices()[0].numpy(), gxc.indices()[1].numpy(), gxc.values().numpy().astype(f), (V, V))
    gY = O.coo_to_csr(gyc.indices()[0].numpy(), gyc.indices()[1].numpy(), gyc.values().numpy().astype(f), (V, V))
    p64 = {k: v.numpy().astype(f) for k, v in params.items()}
    return O.diffusion_net_block(x.cpu().numpy().astype(f), mass.cpu().numpy().astype(f),
                                 evals.cpu().numpy().astype(f), evecs.cpu().numpy().astype(f), gX, gY, p64)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("n,m,K,C,kw", [
    (40, 50, 64, 32, {}),                 # BASELINE config 1 shape (V=2000,K=64,C=32)
    (5, 10, 8, 16, {}),                   # V=50 < one row tile
    (23, 31, 40, 64, {"permute": True}),  # ragged V, K not a power of two, scattered gathers
    (20, 25, 128, 256, {}),               # C_width=256 (BASELINE config 3 width)
    (60, 83, 128, 256, {}),               # C_width=256, ragged tiles: two-slice to_basis, split P / Q layers
    (70, 100, 128, 128, {}),              # human-seg shape (config 2)
])
def test_block_vs_oracle_shapes(dn, engine, n, m, K, C, kw):
    dn.set_engine(engine)
    ops_t, params, x = _structural_case(dn, n, m, K, C, **kw)
    mass, L, evals, evecs, gradX, gradY = ops_t
    blk = make_block(dn, C, {k: v.numpy() for k, v in params.items()})
    with torch.no_grad():
        out = blk(x.unsqueeze(0), mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY])
    gold = _oracle_block(ops_t, params, x)
    assert O.rel_err(out[0].cpu().numpy(), gold) < TOL[engine]


def test_empty_rows_and_union_pattern(dn):
    """A vertex with no gradient entries, and gradX/gradY with different sparsity patterns."""
    dn.set_engine("tc3x")
    V, C = 64, 16
    g = torch.Generator().manual_seed(5)
    rows = torch.randint(1, V, (300,), generator=g)       # row 0 stays empty
    cols = torch.randint(0, V, (300,), generator=g)
    gx = torch.sparse_coo_tensor(torch.stack((rows, cols)), torch.randn(300, generator=g), (V, V)).coalesce().cuda()
    rows2 = torch.randint(1, V, (200,), generator=g)
    cols2 = torch.randint(0, V, (200,), generator=g)
    gy = torch.sparse_coo_tensor(torch.stack((rows2, cols2)), torch.randn(200, generator=g), (V, V)).coalesce().cuda()
    gops = dn.prepare_operators(gx, gy)
    x = torch.randn(V, C, generator=g).cuda()
    out = dn.ops.grad_spmm_raw(gops, x)
    ref = torch.stack((torch.sparse.mm(gx, x), torch.sparse.mm(gy, x)), -1)
    assert torch.allclose(out, ref, rtol=1e-5, atol=1e-5)
    assert torch.all(out[0] == 0)


@pytest.mark.parametrize("engine", ENGINES)
def test_full_size_properties(dn, engine):
    """BASELINE metric size (V=200k,K=128,C=128): oracle check plus size-independent properties."""
    dn.set_engine(engine)
    n, m, K, C = 400, 500, 128, 128
    ops_t, params, x = _structural_case(dn, n, m, K, C, seed=1)
    mass, L, evals, evecs, gradX, gradY = ops_t
    blk = make_block(dn, C, {k: v.numpy() for k, v in params.items()})
    b = lambda t: t.unsqueeze(0)
    with torch.no_grad():
        out = blk(b(x), b(mass), None, b(evals), b(evecs), [gradX], [gradY])
        # linearity of the spectral diffusion in x
        x2 = torch.randn_like(x)
        d = lambda t: blk.diffusion(b(t), None, b(mass), b(evals), b(evecs))[0]
        lhs = d(2.0 * x + 3.0 * x2)
        rhs = 2.0 * d(x) + 3.0 * d(x2)
        assert O.rel_err(lhs.cpu().numpy(), rhs.cpu().numpy()) < 2e-5
        # t -> 0: diffusion is the M-orthogonal projection onto span(evecs), hence idempotent
        blk.diffusion.diffusion_time.data.fill_(0.0)
        p1 = d(x)
        p2 = d(p1)
        assert float(blk.diffusion.diffusion_time.min()) == pytest.approx(1e-8)
        assert O.rel_err(p2.cpu().numpy(), p1.cpu().numpy()) < 2e-5
    gold = _oracle_block(ops_t, params, x)
    assert O.rel_err(out[0].cpu().numpy(), gold) < TOL[engine]


# DN_ENGINE_BF16 (BASELINE config 3's arithmetic): one bf16 tensor-core pass, fp32 accumulate.  SURVEY.md 8c exempts
# bf16 mode from the 1e-5 bound and asks for its own stated one: 2e-2 of max|gold| (measured 3e-4 .. 1.5e-2).
BF16_TOL = 2e-2


@pytest.mark.parametrize("n,m,K,C", [(70, 100, 128, 128), (60, 83, 128, 256), (20, 25, 128, 256), (40, 50, 64, 32),
                                     (5, 10, 8, 16)])
def test_bf16_engine_block_vs_oracle(dn, n, m, K, C):
    dn.set_engine("bf16")
    try:
        ops_t, params, x = _structural_case(dn, n, m, K, C)
        mass, L, evals, evecs, gradX, gradY = ops_t
        blk = make_block(dn, C, {k: v.numpy() for k, v in params.items()})
        with torch.no_grad():
            out = blk(x.unsqueeze(0), mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY])
            out2 = blk(x.unsqueeze(0), mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY])
        assert torch.equal(out, out2)                      # deterministic (no hand-off race)
        gold = _oracle_block(ops_t, params, x)
        assert O.rel_err(out[0].cpu().numpy(), gold) < BF16_TOL
        # the training route (autograd Functions, hidden activations written by the chain) under the same engine
        blk.train()
        xg = x.unsqueeze(0).clone().requires_grad_(True)
        y = blk(xg, mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY])
        assert O.rel_err(y[0].detach().cpu().numpy(), gold) < BF16_TOL
        y.square().mean().backward()
        dn.set_engine("simt")
        blk.zero_grad()
        xs = x.unsqueeze(0).clone().requires_grad_(True)
        blk(xs, mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY]).square().mean().backward()
        assert O.rel_err(xg.grad.cpu().numpy(), xs.grad.cpu().numpy()) < 5e-2
    finally:
        dn.set_engine("tc3x")


def test_config3_full_size_bf16(dn):
    """BASELINE config 3's block: V = 200k, K = 128, C_width = 256, bf16 engine, against the fp64 oracle."""
    dn.set_engine("bf16")
    try:
        ops_t, params, x = _structural_case(dn, 400, 500, 128, 256, seed=2)
        mass, L, evals, evecs, gradX, gradY = ops_t
        blk = make_block(dn, 256, {k: v.numpy() for k, v in params.items()})
        with torch.no_grad():
            out = blk(x.unsqueeze(0), mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY])
        gold = _oracle_block(ops_t, params, x)
        assert O.rel_err(out[0].cpu().numpy(), gold) < BF16_TOL
    finally:
        dn.set_engine("tc3x")


@pytest.mark.parametrize("engine,C", [("tc3x", 128), ("tc3x", 64), ("bf16", 128)])
def test_forward_batch_equals_per_mesh(dn, engine, C):
    """BASELINE config 4: a ragged batch of meshes run as ONE launch sequence (MeshBatch + dn_block_fwd_batched)
    equals the reference-style per-mesh loop."""
    dn.set_engine(engine)
    try:
        K = 128 if C == 128 else 64
        net = dn.DiffusionNet(C_in=16, C_out=8, C_width=C, N_block=2, dropout=False).cuda().eval()
        with torch.no_grad():
            for n_, p_ in net.named_parameters():
                if n_.endswith("diffusion_time"):
                    p_.uniform_(1e-3, 0.3)
        items, xs, refs = [], [], []
        for i, (n, m) in enumerate([(36, 50), (12, 11), (44, 50), (16, 8), (40, 51)]):
            mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(n, m, K, seed=i, device="cuda")
            x = torch.randn(n * m, 16, generator=torch.Generator().manual_seed(i)).cuda()
            items.append(dict(mass=mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY))
            xs.append(x)
            with torch.no_grad():
                refs.append(net(x, mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY).clone())
        mb = dn.MeshBatch(items)
        assert mb.V % 128 == 0 and mb.n_meshes == 5
        with torch.no_grad():
            outs = net.forward_batch(mb, xs)
            outs2 = net.forward_batch(mb, mb.pack(xs))
            if engine == "tc3x" and C == 128:                  # one CUDA graph for the whole batched forward
                gb = dn.graphs.GraphedBatch(net, mb)
                for _ in range(2):
                    og = gb.forward(xs)
                    torch.cuda.synchronize()
                    assert all(torch.equal(a, b) for a, b in zip(og, outs))
        tol = 2e-5 if engine == "tc3x" else BF16_TOL
        for o, o2, r in zip(outs, outs2, refs):
            assert o.shape == r.shape
            assert torch.equal(o, o2)
            assert O.rel_err(o.cpu().numpy(), r.cpu().numpy()) < tol
    finally:
        dn.set_engine("tc3x")


def test_build_grad_on_device_vs_reference(dn):
    """SURVEY 8f-4: dn_build_grad (edge_tangent_vectors + build_grad, geometry.py:198-273) against the gradX / gradY the
    live reference produced (tests/golden/geom_small.npz) and against the oracle restatement on a larger mesh."""
    import scipy.sparse as sp
    fx = load_golden("geom_small")
    V = fx["verts"].shape[0]
    edges = torch.from_numpy(np.stack((fx["L_rows"], fx["L_cols"])).astype(np.int64))
    g = dn.geometry.build_grad_operators(dev(fx["verts"]), dev(fx["frames"]), edges)
    rowptr, colidx, vals = (np.asarray(a) for a in g.to_host_csr())
    for k, name in enumerate(("gradX", "gradY")):
        ref = sp.coo_matrix((fx[name + "_vals"], (fx[name + "_rows"], fx[name + "_cols"])), shape=(V, V)).tocsr()
        ref.sort_indices()
        assert np.array_equal(rowptr, ref.indptr) and np.array_equal(colidx, ref.indices)
        assert np.abs(vals[:, k] - ref.data).max() <= 2e-6 * np.abs(ref.data).max()
    # the reference-signature mirror (numpy in, scipy complex CSC out) with precomputed tangent vectors
    et = O.edge_tangent_vectors(fx["verts"], fx["frames"], edges.numpy())
    M = dn.geometry.build_grad(fx["verts"], edges.numpy(), et).tocsr()
    M.sort_indices()
    assert np.array_equal(M.indices, colidx) and np.abs(np.real(M.data) - vals[:, 0]).max() <= 1e-6 * np.abs(vals).max()
    # a larger, irregular case: random frames / neighbour lists of varying length (incl. a vertex with no edges, a self
    # loop, unsorted edge order) vs the fp64 oracle
    rng = np.random.RandomState(3)
    V2 = 5000
    verts = rng.randn(V2, 3).astype(np.float32)
    q = np.linalg.qr(rng.randn(V2, 3, 3))[0].astype(np.float32)
    tails = np.repeat(np.arange(1, V2), rng.randint(3, 12, V2 - 1))          # vertex 0 has no outgoing edge
    tips = rng.randint(0, V2, tails.shape[0])
    keep = np.ones(tails.shape[0], bool)
    seen = set()
    for i, (a, b) in enumerate(zip(tails, tips)):                            # unique (tail, tip) pairs
        keep[i] = (a, b) not in seen
        seen.add((a, b))
    e2 = np.stack((tails[keep], tips[keep]))
    e2 = e2[:, rng.permutation(e2.shape[1])]
    e2[1, 7] = e2[0, 7]                                                      # one self loop: skipped (geometry.py:228)
    g2 = dn.geometry.build_grad_operators(dev(verts), dev(q), torch.from_numpy(e2))
    rp2, ci2, va2 = (np.asarray(a) for a in g2.to_host_csr())
    gold = O.build_grad(V2, e2, O.edge_tangent_vectors(verts, q, e2))     # fp32 tangent vectors like the torch ops
    gold.sum_duplicates(); gold.sort_indices()
    assert np.array_equal(rp2, gold.indptr) and np.array_equal(ci2, gold.indices)
    scale = np.abs(gold.data).max()
    assert np.abs(va2[:, 0] - np.real(gold.data)).max() <= 2e-5 * scale
    assert np.abs(va2[:, 1] - np.imag(gold.data)).max() <= 2e-5 * scale


@pytest.mark.parametrize("C,K,C_out,outputs_at", [(128, 128, 8, "vertices"), (64, 64, 5, "faces"), (128, 64, 1, "global_mean")])
def test_last_lin_fused_into_last_block(dn, C, K, C_out, outputs_at):
    """SURVEY 8f-1: DiffusionNet.last_lin (layers.py:366-370) computed in the epilogue of the last block's MiniMLP chain
    (dn_block_fwd_ex, exact fp32 head) equals the separate linear layer, single mesh and batched, and the fp64 oracle
    composition of blocks + linear."""
    dn.set_engine("tc3x")
    net = dn.DiffusionNet(C_in=16, C_out=C_out, C_width=C, N_block=2, dropout=False, outputs_at=outputs_at).cuda().eval()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if n_.endswith("diffusion_time"):
                p_.uniform_(1e-3, 0.3)
    n, m = 30, 41
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(n, m, K, seed=5, device="cuda")
    V = n * m
    g = torch.Generator().manual_seed(6)
    x = torch.randn(V, 16, generator=g).cuda()
    faces = torch.randint(0, V, (50, 3), generator=g).cuda()
    kw = dict(mass=mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY, faces=faces)
    try:
        with torch.no_grad():
            net(x, **kw)                                            # (operator prep happens on the first call)
            l0 = dn._lib.load().dn_kernel_launch_count()
            dn.layers.FUSE_HEAD = True
            y1 = net(x, **kw)
            l1 = dn._lib.load().dn_kernel_launch_count()
            dn.layers.FUSE_HEAD = False
            y0 = net(x, **kw)
            l2 = dn._lib.load().dn_kernel_launch_count()
            assert (l2 - l1) == (l1 - l0) + 1                       # the fused route saves exactly the last_lin launch
            assert y1.shape == y0.shape
            assert O.rel_err(y1.cpu().numpy(), y0.cpu().numpy()) < 2e-6
            if outputs_at == "vertices":
                mb = dn.MeshBatch([dict(mass=mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY)] * 2)
                dn.layers.FUSE_HEAD = True
                b1 = net.forward_batch(mb, [x, x])
                dn.layers.FUSE_HEAD = False
                b0 = net.forward_batch(mb, [x, x])
                for a, b_ in zip(b1, b0):
                    assert O.rel_err(a.cpu().numpy(), b_.cpu().numpy()) < 2e-6
                assert O.rel_err(b1[0].cpu().numpy(), y1.cpu().numpy()) < 2e-5
    finally:
        dn.layers.FUSE_HEAD = True


def test_graphed_net_and_streamed_forward(dn):
    """CUDA-graph replay (launch-bound small meshes) and the host-streaming helper reproduce the eager forward."""
    dn.set_engine("tc3x")
    C, K = 32, 32
    net = dn.DiffusionNet(C_in=3, C_out=5, C_width=C, N_block=2, dropout=False).cuda().eval()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if n_.endswith("diffusion_time"):
                p_.uniform_(1e-3, 0.3)
    items, refs = [], []
    for i in range(5):
        mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(12 + i, 16, K, seed=i, device="cuda")
        x = torch.randn((12 + i) * 16, 3, generator=torch.Generator().manual_seed(i)).cuda()
        items.append(dict(x_in=x, mass=mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY))
        with torch.no_grad():
            refs.append(net(**items[-1]).clone())
    gn = dn.graphs.GraphedNet(net, n_streams=2)
    for _ in range(2):                                   # capture, then pure replay
        outs = gn.forward_batch(items)
        torch.cuda.synchronize()
        for o, r in zip(outs, refs):
            assert torch.equal(o, r)
    # host pipeline: same result as the eager call on device tensors
    host = {k: v.cpu().pin_memory() for k, v in items[0].items() if not v.is_sparse}
    gX, gY = items[0]["gradX"], items[0]["gradY"]
    def fn(x_in, mass, evals, evecs):
        with torch.no_grad():
            return net(x_in, mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY)
    pipe = dn.streaming.StreamedForward(fn, torch.device("cuda", 0), depth=2)
    tickets = [pipe.submit(host) for _ in range(3)]
    for t in tickets:
        assert torch.equal(pipe.result(t), refs[0].cpu())
    assert pipe.h2d_bytes == 3 * sum(v.numel() * v.element_size() for v in host.values())


def test_training_mode_dropout_matches_manual_masks(dn):
    """MiniMLP in train() mode: Dropout(p=.5) after each hidden ReLU (layers.py:143-147).  The masks come from
    torch's generator, so re-seeding reproduces them; forward and all gradients must match a plain-torch fp64
    evaluation with the same masks."""
    dn.set_engine("tc3x")
    V, C = 300, 32
    g = torch.Generator().manual_seed(3)
    mlp = dn.MiniMLP([3 * C, C, C, C], dropout=True).cuda().train()
    x = torch.randn(V, 3 * C, generator=g).cuda().requires_grad_(True)
    R = torch.randn(V, C, generator=g).cuda()
    torch.manual_seed(1234)
    y = mlp(x)
    (y * R).sum().backward()
    # replay the mask draws (same order/shapes as ops.MLPFn.forward)
    torch.manual_seed(1234)
    masks = [torch.empty(V, C, device="cuda").bernoulli_(0.5).mul_(2.0) for _ in range(2)]
    lins = mlp.linears()
    xr = x.detach().double().requires_grad_(True)
    ws = [l.weight.detach().double().requires_grad_(True) for l in lins]
    bs = [l.bias.detach().double().requires_grad_(True) for l in lins]
    h = xr
    for i in range(3):
        h = h @ ws[i].t() + bs[i]
        if i < 2:
            h = torch.relu(h) * masks[i].double()
    (h * R.double()).sum().backward()
    assert O.rel_err(y.detach().cpu().numpy(), h.detach().cpu().numpy()) < 1e-5
    assert O.rel_err(x.grad.cpu().numpy(), xr.grad.cpu().numpy()) < 2e-5
    for i, l in enumerate(lins):
        assert O.rel_err(l.weight.grad.cpu().numpy(), ws[i].grad.cpu().numpy()) < 5e-5
        assert O.rel_err(l.bias.grad.cpu().numpy(), bs[i].grad.cpu().numpy()) < 5e-5


def test_net_training_step_and_gradient_allreduce(dn):
    """One optimiser step of a 2-block net on two meshes with gradients accumulated and averaged through
    dist.allreduce_gradients (world size 1 here; the collective itself is covered by the gloo test)."""
    dn.set_engine("tc3x")
    net = dn.DiffusionNet(C_in=3, C_out=4, C_width=32, N_block=2, dropout=True).cuda().train()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if n_.endswith("diffusion_time"):
                p_.uniform_(1e-3, 0.3)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    before = [p_.detach().clone() for p_ in net.parameters()]
    opt.zero_grad()
    for i in range(2):
        mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(14 + i, 16, 32, seed=i, device="cuda")
        x = torch.randn((14 + i) * 16, 3, generator=torch.Generator().manual_seed(i)).cuda()
        out = net(x, mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY)
        target = torch.randint(0, 4, (out.shape[0],), generator=torch.Generator().manual_seed(10 + i)).cuda()
        torch.nn.functional.cross_entropy(out, target).backward()
    dn.dist.allreduce_gradients(list(net.parameters()), n_global_meshes=2)
    assert all(p_.grad is not None and torch.isfinite(p_.grad).all() for p_ in net.parameters())
    opt.step()
    assert any(not torch.equal(a, b) for a, b in zip(before, [p_.detach() for p_ in net.parameters()]))
    assert float(min(b.diffusion.diffusion_time.min() for b in net.blocks)) >= 0.0


def test_data_parallel_step_gradients_vs_oracle_accumulation(dn):
    """BASELINE config 5 semantics: gradients of a 2-block net accumulated over the rank's meshes and averaged by
    dist.allreduce_gradients (world size 1 here; the NCCL / gloo collective itself is covered by tests/test_host.py and
    the multi-GPU bench logs) equal the mean over the same meshes of the reference's autograd gradients -- fp64 autograd
    through the torch restatement of the reference net (oracle/dn_oracle_torch.py blocks + the two Linear layers,
    layers.py:362-370), i.e. the reference run with gradients accumulated over the batch (SURVEY.md 8e)."""
    import dn_oracle_torch as T
    dn.set_engine("tc3x")
    C, K, C_in, C_out, NB = 32, 32, 3, 4, 2
    net = dn.DiffusionNet(C_in=C_in, C_out=C_out, C_width=C, N_block=NB, dropout=False).cuda().train()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if n_.endswith("diffusion_time"):
                p_.uniform_(1e-3, 0.3)
    meshes = []
    for i in range(2):
        ops_t = dn.synthetic.structural_operators(14 + i, 16, K, seed=i, device="cuda")
        g = torch.Generator().manual_seed(20 + i)
        V = (14 + i) * 16
        meshes.append((torch.randn(V, C_in, generator=g).cuda(), torch.randint(0, C_out, (V,), generator=g).cuda(), ops_t))
    for p_ in net.parameters():
        p_.grad = None
    for x, y, (mass, L, evals, evecs, gX, gY) in meshes:
        out = net(x, mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY)
        torch.nn.functional.cross_entropy(out, y).backward()
    dn.dist.allreduce_gradients(list(net.parameters()), n_global_meshes=len(meshes))
    # gold: fp64, CPU, the reference's composition; mean of the per-mesh gradients
    d = torch.float64
    prm = {k: v.detach().cpu().to(d).requires_grad_(True) for k, v in net.state_dict().items()}
    for x, y, (mass, L, evals, evecs, gX, gY) in meshes:
        h = torch.addmm(prm["first_lin.bias"], x.cpu().to(d), prm["first_lin.weight"].t()).unsqueeze(0)
        for b in range(NB):
            bp = {k[len("block_%d." % b):]: v for k, v in prm.items() if k.startswith("block_%d." % b)}
            h = T.block_forward(h, mass.cpu().to(d).unsqueeze(0), evals.cpu().to(d).unsqueeze(0),
                                evecs.cpu().to(d).unsqueeze(0), [gX.cpu().to(d)], [gY.cpu().to(d)], bp)
        logits = torch.addmm(prm["last_lin.bias"], h[0], prm["last_lin.weight"].t())
        (torch.nn.functional.cross_entropy(logits, y.cpu()) / len(meshes)).backward()
    for name, p_ in net.named_parameters():
        assert p_.grad is not None, name
        assert O.rel_err(p_.grad.cpu().numpy(), prm[name].grad.numpy()) < 5e-5, name


def test_graphed_train_step_matches_eager_autograd(dn):
    """graphs.GraphedTrainStep: forward + backward of a net on one mesh replayed as one CUDA graph accumulates the same
    gradients as eager autograd (BASELINE configs 2 / 5 are launch-bound in eager mode)."""
    dn.set_engine("tc3x")
    net = dn.DiffusionNet(C_in=16, C_out=4, C_width=64, N_block=2, dropout=False).cuda().train()
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if n_.endswith("diffusion_time"):
                p_.uniform_(1e-3, 0.3)
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(20, 24, 64, seed=1, device="cuda")
    g = torch.Generator().manual_seed(2)
    x = torch.randn(480, 16, generator=g).cuda()
    y = torch.randint(0, 4, (480,), generator=g).cuda()

    def loss_fn(net_, x_, y_):
        return torch.nn.functional.cross_entropy(net_(x_, mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY), y_)

    for p_ in net.parameters():
        p_.grad = None
    loss_fn(net, x, y).backward()
    ref = [p_.grad.clone() for p_ in net.parameters()]
    gts = dn.graphs.GraphedTrainStep(net, loss_fn, (x, y))
    for rep in range(2):
        dn.graphs.GraphedTrainStep.zero_grads(net)
        loss = gts.replay()
        torch.cuda.synchronize()
        assert torch.isfinite(loss)
        for p_, r in zip(net.parameters(), ref):
            assert torch.equal(p_.grad, r)
    gts.replay()                                            # a second replay without zeroing accumulates: 2 x the gradient
    torch.cuda.synchronize()
    for p_, r in zip(net.parameters(), ref):
        assert torch.allclose(p_.grad, 2 * r, rtol=1e-6, atol=0)


# ---- data-side neighbours of the block (SURVEY.md 8f items 2-3) ------------------------------------------------
GEOM_CACHE = os.path.join(ROOT, "tests", "golden", "op_cache")


def _csr_np(st):
    _, rowptr, colidx, vals = st
    return rowptr.cpu().numpy(), colidx.cpu().numpy(), vals.cpu().numpy()


def test_operator_cache_to_device_matches_reference_hit_branch(dn):
    """geometry.get_operators on the cache entry the reference wrote: every tensor of the tuple equals what the
    reference's own cache-hit branch returned (bit-exact), and the CSR/CSR^T built straight from the file's CSC
    arrays equal the ones the generic COO path builds."""
    fx = load_golden("geom_small")
    verts, faces = torch.from_numpy(fx["verts"]), torch.from_numpy(fx["faces"])
    frames, mass, L, evals, evecs, gradX, gradY = dn.geometry.get_operators(verts, faces, 16, GEOM_CACHE,
                                                                            device="cuda")
    for got, key in ((frames, "frames"), (mass, "mass"), (evals, "evals"), (evecs, "evecs")):
        assert got.is_cuda and got.dtype == torch.float32
        assert np.array_equal(got.cpu().numpy(), fx[key]), key
    for got, pre in ((L, "L"), (gradX, "gradX"), (gradY, "gradY")):
        assert got.is_sparse and got.is_coalesced() and got.indices().dtype == torch.int64     # utils.py:55
        assert np.array_equal(got.indices()[0].cpu().numpy(), fx[pre + "_rows"]), pre
        assert np.array_equal(got.indices()[1].cpu().numpy(), fx[pre + "_cols"]), pre
        assert np.array_equal(got.values().cpu().numpy(), fx[pre + "_vals"]), pre
    pre_built = dn.ops.prepare_operators(gradX, gradY)
    assert pre_built._coo is None            # the registered from_csc object, not a rebuild through COO
    generic = dn.ops.GradOperators(gradX, gradY)
    for a, b in zip(_csr_np(pre_built.csr), _csr_np(generic.csr)):
        assert np.array_equal(a, b)
    for a, b in zip(_csr_np(pre_built.csr_t), _csr_np(generic.csr_t)):
        assert np.array_equal(a, b)
    e12, v12 = dn.geometry.get_operators(verts, faces, 12, GEOM_CACHE, device="cuda")[3:5]
    assert np.array_equal(e12.cpu().numpy(), fx["evals12"]) and np.array_equal(v12.cpu().numpy(), fx["evecs12"])
    lists = dn.geometry.get_all_operators([verts, verts], [faces, faces], 16, GEOM_CACHE, device="cuda")
    assert len(lists) == 7 and all(len(l) == 2 for l in lists)


def test_hks_matches_reference(dn):
    fx = load_golden("geom_small")
    evals, evecs = dev(fx["evals"]), dev(fx["evecs"])
    got = dn.geometry.compute_hks_autoscale(evals, evecs, 16)          # K=16: generic kernel
    assert got.shape == (evecs.shape[0], 16)
    assert O.rel_err(got.cpu().numpy(), fx["hks_f64"]) < 1e-5
    got3 = dn.geometry.compute_hks(evals, evecs, dev(fx["hks3_scales"]))
    assert O.rel_err(got3.cpu().numpy(), fx["hks3_f64"]) < 1e-5
    gb = dn.geometry.compute_hks(torch.stack((evals, evals)), torch.stack((evecs, evecs)),
                                 torch.stack((dev(fx["hks3_scales"]),) * 2))        # batched form, geometry.py:611-616
    assert gb.shape == (2, evecs.shape[0], 3) and torch.equal(gb[0], got3) and torch.equal(gb[1], got3)


@pytest.mark.parametrize("K,S", [(32, 16), (64, 16), (96, 5), (128, 16), (256, 16), (128, 17), (160, 16), (40, 1)])
def test_hks_shapes_against_oracle(dn, K, S):
    """warp-per-row register kernel (K in {32,64,96,128,256}, S<=16) and the generic one, vs the fp64 oracle."""
    V = 3001
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(60, 50, K, seed=K + S, device="cuda")
    evecs = evecs[:V].contiguous()
    scales = torch.logspace(-2, 0.3, S, device="cuda")
    got = dn.geometry.compute_hks(evals, evecs, scales).cpu().numpy()
    want = O.compute_hks(evals.double().cpu().numpy(), evecs.double().cpu().numpy(), scales.double().cpu().numpy())
    assert O.rel_err(got, want) < 2e-6


def test_cache_to_hks_to_net_pipeline_matches_reference(dn):
    """The experiments' data path end to end (human_segmentation_original.py:111-126): cache entry -> operators on
    the device -> HKS input features -> DiffusionNet, against the reference's fp64 output."""
    fx = load_golden("geom_small")
    verts, faces = torch.from_numpy(fx["verts"]), torch.from_numpy(fx["faces"])
    frames, mass, L, evals, evecs, gradX, gradY = dn.geometry.get_operators(verts, faces, 16, GEOM_CACHE,
                                                                            device="cuda")
    feats = dn.geometry.compute_hks_autoscale(evals, evecs, 16)
    for eng in ENGINES:
        dn.set_engine(eng)
        net = dn.DiffusionNet(C_in=16, C_out=6, C_width=32, N_block=2, dropout=False)
        net.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in golden_params(fx).items()}, strict=True)
        net = net.cuda().eval()
        with torch.no_grad():
            out = net(feats, mass, L=L, evals=evals, evecs=evecs, gradX=gradX, gradY=gradY)
        assert O.rel_err(out.cpu().numpy(), fx["net_out_f64"]) < TOL[eng], eng
    dn.set_engine("tc3x")


def test_full_size_hks_and_transpose_properties(dn):
    """V=200k (BASELINE size): (1) Phi^T M Phi = I  =>  sum_v mass[v] hks[v,s] = sum_k exp(-evals[k] t_s);
    (2) transposing the CSR twice is the identity, bit for bit, and every row comes out column-sorted."""
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(400, 500, 128, seed=0, device="cuda")
    V = mass.shape[0]
    scales = torch.logspace(-2, 0, 16, device="cuda")
    hks = dn.geometry.compute_hks(evals, evecs, scales)
    lhs = (hks.double() * mass.double()[:, None]).sum(0)
    rhs = torch.exp(-evals.double()[None, :] * scales.double()[:, None]).sum(1)
    assert float(((lhs - rhs).abs() / rhs).max()) < 1e-4
    g = dn.ops.prepare_operators(gX, gY)
    st, rowptr, colidx, vals = g.csr
    rp, ci, va = rowptr.cpu().numpy(), colidx.cpu().numpy(), vals.cpu().numpy()
    t = dn.ops.GradOperators.from_csc(V, rp, ci, va[0::2], va[1::2], "cuda")      # treats csr as the CSC of A^T
    # t.csr_t is the input verbatim; t.csr = its transpose = CSR of A^T
    tt = dn.ops.GradOperators.from_csc(V, *[a.cpu().numpy() for a in t.csr[1:3]],
                                       t.csr[3][0::2].cpu().numpy(), t.csr[3][1::2].cpu().numpy(), "cuda")
    for a, b in zip(_csr_np(tt.csr), (rp, ci, va)):
        assert np.array_equal(a, b)
    trp, tci = t.csr[1].cpu().numpy(), t.csr[2].cpu().numpy()
    assert trp[0] == 0 and trp[-1] == g.nnz
    key = np.repeat(np.arange(V, dtype=np.int64), np.diff(trp)) * V + tci[:g.nnz]
    assert np.all(np.diff(key) > 0)                       # rows ascending, columns strictly ascending inside a row
    # and it matches the argsort-based transpose of the generic path
    for a, b in zip(_csr_np(t.csr), _csr_np(g.csr_t)):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("permute", [False, True])
@pytest.mark.parametrize("rot", [True, False])
def test_patched_gather_is_bit_identical_and_patch_policy(dn, permute, rot):
    """dn_patches (shared-memory staged gather) vs the plain gather kernel: same entries, same order, same arithmetic;
    and prepare_operators builds the structure on the second use exactly when the vertex order lacks locality."""
    dn.set_engine("tc3x")
    C = 128
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(60, 70, 32, seed=2, device="cuda", permute=permute)
    V = mass.shape[0]
    g = torch.Generator().manual_seed(4)
    xd = torch.randn(V, C, generator=g).cuda()
    A_re = (torch.randn(C, C, generator=g) / C ** 0.5).cuda()
    A_im = (torch.randn(C, C, generator=g) / C ** 0.5).cuda() if rot else None
    plain = dn.ops.GradOperators(gX, gY)
    with torch.no_grad():
        ref = dn.ops.GradFeaturesFn.apply(xd, A_re, A_im, plain)
        for T, R in ((64, 144), (32, 72), (7, 16)):
            patched = dn.ops.GradOperators(gX, gY).build_patches(T, R)
            assert patched._patches and patched.patch_stats["max_src"] <= R
            out = dn.ops.GradFeaturesFn.apply(xd, A_re, A_im, patched)
            assert torch.equal(out, ref), (T, R)
    # second use of the same operator tensors: the structure is built only when the vertex order lacks locality
    o1 = dn.ops.prepare_operators(gX, gY)
    assert getattr(o1, "_patches", None) is None
    o2 = dn.ops.prepare_operators(gX, gY)
    assert o2 is o1
    # (a symmetric permutation keeps the diagonal entry on the diagonal: 1/7 of the entries stay 'local')
    assert (o2.locality() < 0.2 and o2._patches) if permute else (o2.locality() > 0.3 and o2._patches is False)
    with torch.no_grad():
        assert torch.equal(dn.ops.GradFeaturesFn.apply(xd, A_re, A_im, o2), ref)
