"""Tensor-core gradient-features route (C_width = 128 with rotations): per-stage times of the fused block at V=200k, the x-only gather's
share of stage [4], parity vs the exact engine, repeatability."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import diffusion_net_b200 as dn
lib = dn._lib.load()
lib.dn_debug_gf_gather_ms.restype = ctypes.c_float
C = 128
for permute in (False, True):
    mass, L, evals, evecs, gX, gY = dn.synthetic.structural_operators(400, 500, 128, seed=0, device="cuda", permute=permute)
    V = mass.shape[0]
    params = dn.synthetic.block_weights(C, seed=0)
    x = torch.randn(V, C, generator=torch.Generator().manual_seed(1)).cuda()
    blk = dn.DiffusionNetBlock(C_width=C, mlp_hidden_dims=[C, C], dropout=False)
    blk.load_state_dict(params, strict=True)
    blk = blk.cuda().eval()
    gops = dn.ops.GradOperators(gX, gY)
    A_re, A_im = blk.gradient_features.weights()
    lins = blk.mlp.linears()
    run = lambda prof=None: dn.ops.block_forward_raw(x, mass, evals, evecs, gops, blk.diffusion.diffusion_time, A_re, A_im,
                                                     [l.weight for l in lins], [l.bias for l in lins], True, profile=prof)
    with torch.no_grad():
        dn.set_engine("simt"); y0 = run(); dn.set_engine("tc3x")
        y = run(); torch.cuda.synchronize()
        rep = all(torch.equal(y, run()) for _ in range(4))
        acc, gat = [0.0] * 6, 0.0
        for it in range(12):
            prof = []; run(prof)
            if it >= 2:
                acc = [a + b for a, b in zip(acc, prof)]; gat += lib.dn_debug_gf_gather_ms()
    print("permute={} err {:.2e} repeatable={} stages_us {} (x-only gather {:.1f} us of the gradient stage)".format(
        permute, float((y - y0).abs().max() / y0.abs().max()), rep, {n: round(100 * a, 1) for n, a in zip(dn.ops.PROFILE_STAGES, acc)},
        100 * gat), flush=True)
