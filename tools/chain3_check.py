"""Round-2 bring-up of rows_chain3_kernel (dn_chain.cu): parity against the exact SIMT engine and device time,
for the two fused chains of the block (from_basis + [P|Q]; MiniMLP + skip) and single layers, at several V
(ragged last tile, V < 128, one tile, many tiles per CTA), repeated calls to catch hand-off races.

    python tools/chain3_check.py
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import diffusion_net_b200 as dn

C = 128
torch.manual_seed(0)


def t_us(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return 1e3 * a.elapsed_time(b) / n


def rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


def check(V, reps=4, timing=False):
    g = torch.Generator().manual_seed(V)
    x, xd, ft = (torch.randn(V, C, generator=g).cuda() for _ in range(3))
    p = dn.synthetic.block_weights(C, seed=0)
    ws = [p["mlp.miniMLP_mlp_layer_{:03d}.weight".format(i)].cuda() for i in range(3)]
    bs = [p["mlp.miniMLP_mlp_layer_{:03d}.bias".format(i)].cuda() for i in range(3)]
    A_re, A_im = p["gradient_features.A_re.weight"].cuda(), p["gradient_features.A_im.weight"].cuda()
    evecs = torch.randn(V, 128, generator=g).cuda() / 30.0
    spec = torch.randn(128, C, generator=g).cuda()
    out = {}
    with torch.no_grad():
        dn.set_engine("simt")
        y0 = dn.ops.mlp_apply([x, xd, ft], ws, bs, residual=x)
        f0 = dn.ops.from_basis_raw(spec, evecs)
        l0 = dn.ops.mlp_apply([x], [ws[1]], [bs[1]])
        r0 = dn.ops.mlp_apply([x], [ws[1]], [bs[1]], residual=xd)
        n0 = dn.ops.mlp_apply([x, xd, ft], ws, bs)
        dn.set_engine("tc3x")
        worst = 0.0
        for it in range(reps):
            y = dn.ops.mlp_apply([x, xd, ft], ws, bs, residual=x)
            f = dn.ops.from_basis_raw(spec, evecs)
            l1 = dn.ops.mlp_apply([x], [ws[1]], [bs[1]])
            r1 = dn.ops.mlp_apply([x], [ws[1]], [bs[1]], residual=xd)
            n1 = dn.ops.mlp_apply([x, xd, ft], ws, bs)
            torch.cuda.synchronize()
            e = max(rel(y, y0), rel(f, f0), rel(l1, l0), rel(r1, r0), rel(n1, n0))
            worst = max(worst, e)
            if e > 1e-5:
                bad = ((y - y0).abs() > 1e-4 * y0.abs().max()).any(1).nonzero().flatten()
                print("   V={} call {}: mlp {:.2e} from_basis {:.2e} single {:.2e} single+res {:.2e} mlp-nores {:.2e}; bad mlp rows {} first {}".format(
                    V, it, rel(y, y0), rel(f, f0), rel(l1, l0), rel(r1, r0), rel(n1, n0), bad.numel(), bad[:8].tolist()), flush=True)
        out["err"] = worst
        if timing:
            out["mlp_us"] = t_us(lambda: dn.ops.mlp_apply([x, xd, ft], ws, bs, residual=x))
            out["from_basis_us"] = t_us(lambda: dn.ops.from_basis_raw(spec, evecs))
    return out


def check_block(V_n, V_m, reps=3, timing=False):
    """Whole fused block forward (dn_block_fwd: to_basis, scale, from_basis+[P|Q] chain, gather, MiniMLP chain)."""
    ops_t = dn.synthetic.structural_operators(V_n, V_m, 128, seed=0, device="cuda")
    mass, L, evals, evecs, gradX, gradY = ops_t
    V = V_n * V_m
    params = dn.synthetic.block_weights(C, seed=0)
    x = torch.randn(V, C, generator=torch.Generator().manual_seed(1)).cuda()
    blk = dn.DiffusionNetBlock(C_width=C, mlp_hidden_dims=[C, C], dropout=False)
    blk.load_state_dict(params, strict=True)
    blk = blk.cuda().eval()
    args = (x.unsqueeze(0), mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gradX], [gradY])
    with torch.no_grad():
        dn.set_engine("simt")
        y0 = blk(*args)
        dn.set_engine("tc3x")
        worst = 0.0
        for _ in range(reps):
            y = blk(*args)
            torch.cuda.synchronize()
            worst = max(worst, rel(y, y0))
        res = {"err": worst}
        if timing:
            res["block_us"] = t_us(lambda: blk(*args))
            gops = dn.ops.prepare_operators(gradX, gradY)
            A_re, A_im = blk.gradient_features.weights()
            lins = blk.mlp.linears()
            acc = [0.0] * 6
            for _ in range(5):
                prof = []
                dn.ops.block_forward_raw(x, mass, evals, evecs, gops, blk.diffusion.diffusion_time, A_re, A_im,
                                         [l.weight for l in lins], [l.bias for l in lins], True, profile=prof)
                acc = [a + b for a, b in zip(acc, prof)]
            res["stages_us"] = {n: round(1e3 * a / 5, 1) for n, a in zip(dn.ops.PROFILE_STAGES, acc)}
    return res


def check_shapes(V=5000):
    """Envelope sweep: chains of Linear(+ReLU) with random weights, tc3x vs the exact SIMT engine."""
    g = torch.Generator().manual_seed(11)
    for dims in ([128, 256], [128, 128], [128, 64], [128, 32], [64, 128], [256, 128], [256, 256], [192, 96],
                 [128, 128, 256], [128, 64, 128], [384, 128, 128, 128], [64, 64, 64, 64, 64], [128, 128, 128, 128, 128, 128, 128]):
        x = torch.randn(V, dims[0], generator=g).cuda()
        ws = [((torch.rand(dims[i + 1], dims[i], generator=g) * 2 - 1) / dims[i] ** 0.5).cuda() for i in range(len(dims) - 1)]
        bs = [((torch.rand(dims[i + 1], generator=g) * 2 - 1) / dims[i] ** 0.5).cuda() for i in range(len(dims) - 1)]
        with torch.no_grad():
            dn.set_engine("simt"); y0 = dn.ops.mlp_apply([x], ws, bs)
            dn.set_engine("tc3x"); y1 = dn.ops.mlp_apply([x], ws, bs)
        print("   dims {}: rel err {:.2e}".format(dims, rel(y1, y0)), flush=True)


if __name__ == "__main__":
    check_shapes()
    for V in (100, 128, 129, 1000, 18944, 18945, 40000):
        print("V={:6d}: {}".format(V, check(V)), flush=True)
    print("V=200000:", check(200000, reps=6, timing=True), flush=True)
    print("block 30x40:", check_block(30, 40), flush=True)
    print("block 400x500:", check_block(400, 500, timing=True), flush=True)
