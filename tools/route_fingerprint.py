"""Route fingerprint: a fixed, seeded matrix of calls through the public API, with every output and the number of
kernels each call launched (dn_kernel_launch_count), written to one .npz.  Two builds that take the same kernel routes
with the same arithmetic write identical files.

    python tools/route_fingerprint.py OUT.npz
    python tools/route_fingerprint.py --compare A.npz B.npz     # exit status 1 when any entry differs

Per engine (simt, tc3x, tc1x, bf16) and C_width x K in {128, 256, 48, 8} x {128, 64, 32} (rows_chain3, the two-slice
to_basis, the round-1 chain kernels, the SIMT fallbacks), with and without gradient rotations, on a randomly permuted
mesh: the fused block forward on plain and on patched operators, with a fused linear head, and a block's training
forward + backward.  Per engine and a few (C_width, K): a DiffusionNet training step with dropout, and MeshBatch
inference and training.  Meshes stay at or below 512 rows so that the bias gradients (column sums with float atomics
across 256-row blocks) are reproducible bit for bit.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def compare(path_a, path_b):
    a, b = np.load(path_a), np.load(path_b)
    bad = sorted(set(a.files) ^ set(b.files)) + [k for k in a.files if k in b.files and not np.array_equal(a[k], b[k])]
    print("{} entries, {} differ".format(len(a.files), len(bad)))
    for k in bad[:40]:
        print("  ", k)
    return 1 if bad else 0


def run(out_path):
    import torch
    import diffusion_net_b200 as dn
    from diffusion_net_b200 import ops

    lib = dn._lib.load()
    rec = {}

    def call(name, fn):
        torch.cuda.synchronize()
        n0 = lib.dn_kernel_launch_count()
        try:
            res = fn()
        except RuntimeError as e:                 # a refusal (HeadNotFused, DN_ERR_*) is part of the fingerprint
            res = np.array("{}: {}".format(type(e).__name__, e))
        torch.cuda.synchronize()
        rec[name + "/launches"] = np.array(lib.dn_kernel_launch_count() - n0)
        for i, t in enumerate(res if isinstance(res, (list, tuple)) else [res]):
            rec["{}/{}".format(name, i)] = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(str(t))

    def grads(module, *tensors):
        return [t.grad for t in tensors] + [p.grad for p in module.parameters()]

    meshes = {}                                   # K -> [(mass, evals, evecs, plain ops, patched ops)]
    for K in (128, 64, 32):
        meshes[K] = []
        for i, (n, m) in enumerate([(19, 23), (8, 16), (9, 15), (16, 8)]):
            mass, _, evals, evecs, gX, gY = dn.synthetic.structural_operators(n, m, K, seed=i, device="cuda", permute=True)
            plain = ops.GradOperators(gX, gY)
            meshes[K].append((mass, evals, evecs, plain, ops.GradOperators(gX, gY).build_patches()))
            _ = plain.csr_t
    for engine in ("simt", "tc3x", "tc1x", "bf16"):
        dn.set_engine(engine)
        for C in (128, 256, 48, 8):
            for K in (128, 64, 32):
                mass, evals, evecs, plain, patched = meshes[K][0]
                V = mass.shape[0]
                b = lambda t: t.unsqueeze(0)
                for rot in (True, False):
                    tag = "{}/C{}/K{}/rot{}".format(engine, C, K, int(rot))
                    torch.manual_seed(C + K + rot)
                    blk = dn.DiffusionNetBlock(C, [C, C], dropout=False, with_gradient_rotations=rot).cuda().eval()
                    with torch.no_grad():
                        blk.diffusion.diffusion_time.uniform_(1e-3, 0.3)
                    g = torch.Generator().manual_seed(C * K)
                    x = torch.randn(V, C, generator=g).cuda()
                    R = torch.randn(V, C, generator=g).cuda()
                    head = (torch.randn(5, C, generator=g).cuda(), torch.randn(5, generator=g).cuda())
                    fwd = lambda xin, gops, **kw: blk(xin, b(mass), None, b(evals), b(evecs), [gops], None, **kw)
                    with torch.no_grad():
                        call(tag + "/block", lambda: fwd(b(x), plain))
                        call(tag + "/block_patched", lambda: fwd(b(x), patched))
                        call(tag + "/block_head", lambda: fwd(b(x), plain, head=head))

                    def train_block():
                        blk.train()
                        xg = b(x).clone().requires_grad_(True)
                        y = fwd(xg, plain)
                        (y[0] * R).sum().backward()
                        return [y] + grads(blk, xg)
                    call(tag + "/block_train", train_block)
        for C, K in ((128, 128), (256, 128), (48, 64), (8, 32), (128, 32)):
            tag = "{}/net/C{}/K{}".format(engine, C, K)
            torch.manual_seed(7 * C + K)
            net = dn.DiffusionNet(C_in=16, C_out=5, C_width=C, N_block=2, dropout=True).cuda()
            with torch.no_grad():
                for n_, p_ in net.named_parameters():
                    if n_.endswith("diffusion_time"):
                        p_.uniform_(1e-3, 0.3)
            g = torch.Generator().manual_seed(C + K)
            xs = [torch.randn(mesh[0].shape[0], 16, generator=g).cuda() for mesh in meshes[K]]
            ys = [torch.randint(0, 5, (mesh[0].shape[0],), generator=g).cuda() for mesh in meshes[K]]

            def train_net():
                net.train()
                net.zero_grad(set_to_none=True)
                mass, evals, evecs, plain, _ = meshes[K][0]
                torch.manual_seed(11)
                out = net(xs[0], mass, evals=evals, evecs=evecs, gradX=plain)
                torch.nn.functional.cross_entropy(out, ys[0]).backward()
                return [out] + grads(net)
            call(tag + "/train", train_net)
            mb = dn.MeshBatch([dict(mass=m_, evals=e_, evecs=v_, gradX=p_) for m_, e_, v_, p_, _ in meshes[K][1:]])

            def batch_infer():
                net.eval()
                with torch.no_grad():
                    return net.forward_batch(mb, xs[1:])
            call(tag + "/batch_infer", batch_infer)

            def batch_train():
                net.train()
                net.zero_grad(set_to_none=True)
                torch.manual_seed(13)
                outs = net.forward_batch(mb, xs[1:])
                sum(torch.nn.functional.cross_entropy(o, y) for o, y in zip(outs, ys[1:])).backward()
                return outs + grads(net)
            call(tag + "/batch_train", batch_train)
    dn.set_engine("tc3x")
    np.savez_compressed(out_path, **rec)
    refused = sum(1 for k, v in rec.items() if v.dtype.kind == "U")
    print("{} entries ({} refusals) -> {}".format(len(rec), refused, out_path))


if __name__ == "__main__":
    if len(sys.argv) == 4 and sys.argv[1] == "--compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    run(sys.argv[1])
