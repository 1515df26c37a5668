"""Generate tests/golden/*.npz by running the UNMODIFIED reference here.

Run in the build container only (needs /root/reference):

    python oracle/make_golden.py [FILE ...]      # e.g. block_k128.npz: rewrite only the named fixtures

Each fixture stores seeded inputs in the reference's own layout (operator tuple
from the reference's ``get_operators``; parameters under the reference
state_dict names) plus the reference module outputs in fp32 and fp64
(``.double()`` on module and inputs = gold, SURVEY.md section 8c).  The fixtures are
what pins ``oracle/dn_oracle.py`` and what the GPU parity tests compare with on
the GPU box, where /root/reference does not exist.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from ref_import import import_reference, reference_src  # noqa: E402
import diffusion_net_b200.synthetic as syn  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def ref_operators(dn, n, m, k_eig, seed):
    verts, faces = syn.torus_mesh(n, m, seed=seed)
    verts = dn.geometry.normalize_positions(verts)
    frames, mass, L, evals, evecs, gradX, gradY = dn.geometry.get_operators(verts, faces, k_eig=k_eig)
    return verts, faces, mass, L, evals, evecs, gradX, gradY


def pack_ops(prefix, mass, evals, evecs, gradX, gradY):
    gx, gy = gradX.coalesce(), gradY.coalesce()
    assert torch.equal(gx.indices(), gy.indices())
    return {
        prefix + "mass": mass.numpy(), prefix + "evals": evals.numpy(), prefix + "evecs": evecs.numpy(),
        prefix + "g_rows": gx.indices()[0].numpy().astype(np.int32),
        prefix + "g_cols": gx.indices()[1].numpy().astype(np.int32),
        prefix + "gx_vals": gx.values().numpy(), prefix + "gy_vals": gy.values().numpy(),
    }


def load_params(module, params, prefix=""):
    sd = {prefix + k: v.clone() for k, v in params.items()}
    module.load_state_dict(sd, strict=True)


def run_block(dn, C, params, x, ops, **kw):
    """Reference DiffusionNetBlock in fp32 and fp64, with intermediates."""
    mass, L, evals, evecs, gradX, gradY = ops
    res = {}
    for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
        blk = dn.layers.DiffusionNetBlock(C_width=C, mlp_hidden_dims=[C, C], dropout=False, **kw).to(dt)
        load_params(blk, {k: v.to(dt) for k, v in params.items()})
        blk.eval()
        cast = lambda t: t.to(dt).unsqueeze(0)
        with torch.no_grad():
            xb = cast(x)
            xd = blk.diffusion(xb, None, cast(mass), cast(evals), cast(evecs))
            out = blk(xb, cast(mass), None, cast(evals), cast(evecs), cast(gradX), cast(gradY))
            res["x_diffuse_" + tag] = xd[0].numpy()
            if kw.get("with_gradient_features", True):
                gxv = torch.mm(gradX.to(dt), xd[0])
                gyv = torch.mm(gradY.to(dt), xd[0])
                feats = blk.gradient_features(torch.stack((gxv, gyv), dim=-1))
                res["x_grad_features_" + tag] = feats.numpy()
            res["out_" + tag] = out[0].numpy()
            res["time_after_" + tag] = blk.diffusion.diffusion_time.detach().numpy().copy()
        if tag == "f64":
            # gradients of loss = sum(out * R) through the reference's own autograd (fp64 gold)
            R = torch.randn(x.shape, generator=torch.Generator().manual_seed(21), dtype=torch.float64)
            xg = x.to(dt).unsqueeze(0).clone().requires_grad_(True)
            out = blk(xg, cast(mass), None, cast(evals), cast(evecs), cast(gradX), cast(gradY))
            (out[0] * R).sum().backward()
            res["loss_R"] = R.numpy()
            res["g:x_in"] = xg.grad[0].numpy()
            for n, prm in blk.named_parameters():
                res["g:" + n] = prm.grad.numpy()
    return res


def main(only=()):
    """Writes every fixture, or only the files named in `only`.  Every section runs either way: the reference's
    module constructors draw from the global torch generator, so later fixtures depend on the sections before them."""
    os.makedirs(OUT, exist_ok=True)

    def save(fname, arrays):
        if not only or fname in only:
            np.savez_compressed(os.path.join(OUT, fname), **arrays)

    dn = import_reference()
    torch.manual_seed(0)

    # ---- 1. small block, real operators, incl. one negative diffusion time (clamp) ----
    C, K = 32, 32
    verts, faces, mass, L, evals, evecs, gradX, gradY = ref_operators(dn, 16, 20, K, seed=0)
    ops = (mass, L, evals, evecs, gradX, gradY)
    x = torch.randn(mass.shape[0], C, generator=torch.Generator().manual_seed(7))
    params = syn.block_weights(C, seed=0)
    params["diffusion.diffusion_time"][3] = -1.6e-5     # a shipped checkpoint has a negative t
    fx = {"x_in": x.numpy(), "faces": faces.numpy().astype(np.int32), "verts": verts.numpy()}
    fx.update(pack_ops("", mass, evals, evecs, gradX, gradY))
    fx.update({"p:" + k: v.numpy() for k, v in params.items()})
    fx.update(run_block(dn, C, params, x, ops))
    save("block_small.npz", fx)

    # ---- 2. no rotations / 3. no gradient features (same operators) ----
    for name, kw in (("block_norot", dict(with_gradient_rotations=False)),
                     ("block_nograd", dict(with_gradient_features=False))):
        p2 = syn.block_weights(C, seed=1, **kw)
        fx2 = {"x_in": x.numpy()}
        fx2.update({"p:" + k: v.numpy() for k, v in p2.items()})
        fx2.update(run_block(dn, C, p2, x, ops, **kw))
        save(name + ".npz", fx2)

    # ---- 4. K=128, C=128 block (human-seg widths on a 12x16 torus: V=192, one full 128-row tile and a ragged one;
    #         the mesh is kept this small so that the fixture stays well under 1 MB) ----
    C4, K4 = 128, 128
    v4, f4, mass4, L4, evals4, evecs4, gX4, gY4 = ref_operators(dn, 12, 16, K4, seed=3)
    x4 = torch.randn(mass4.shape[0], C4, generator=torch.Generator().manual_seed(11))
    p4 = syn.block_weights(C4, seed=2)
    fx4 = {"x_in": x4.numpy()}
    fx4.update(pack_ops("", mass4, evals4, evecs4, gX4, gY4))
    fx4.update({"p:" + k: v.numpy() for k, v in p4.items()})
    r4 = run_block(dn, C4, p4, x4, (mass4, L4, evals4, evecs4, gX4, gY4))
    # gold kept fp32-rounded here to keep the fixture small (adds <=6e-8 relative)
    for k in ("x_diffuse_f64", "out_f64"):
        fx4[k + "_as32"] = r4[k].astype(np.float32)
    save("block_k128.npz", fx4)

    # ---- 5. whole net, 2 blocks, all outputs_at modes, batched B=2 ----
    Cin, Cout, Cw, NB = 3, 8, 32, 2
    verts_b, faces_b, mass_b, L_b, evals_b, evecs_b, gX_b, gY_b = ref_operators(dn, 16, 20, K, seed=5)
    fxn = {"verts0": verts.numpy(), "verts1": verts_b.numpy(), "faces": faces.numpy().astype(np.int32)}
    fxn.update(pack_ops("m0_", mass, evals, evecs, gradX, gradY))
    fxn.update(pack_ops("m1_", mass_b, evals_b, evecs_b, gX_b, gY_b))
    edges = torch.stack((faces[:, 0], faces[:, 1]), dim=-1)
    fxn["edges"] = edges.numpy().astype(np.int32)
    net = dn.layers.DiffusionNet(C_in=Cin, C_out=Cout, C_width=Cw, N_block=NB, dropout=False)
    g = torch.Generator().manual_seed(99)
    with torch.no_grad():
        for name, prm in net.named_parameters():
            if name.endswith("diffusion_time"):
                prm.copy_(1e-3 + 0.3 * torch.rand(prm.shape, generator=g))
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    fxn.update({"p:" + k: v.numpy() for k, v in sd.items()})
    for mode in ("vertices", "edges", "faces", "global_mean"):
        for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
            nt = dn.layers.DiffusionNet(C_in=Cin, C_out=Cout, C_width=Cw, N_block=NB, dropout=False,
                                        outputs_at=mode).to(dt)
            nt.load_state_dict({k: v.to(dt) for k, v in sd.items()})
            nt.eval()
            with torch.no_grad():
                o0 = nt(verts.to(dt), mass.to(dt), L=L.to(dt), evals=evals.to(dt), evecs=evecs.to(dt),
                        gradX=gradX.to(dt), gradY=gradY.to(dt), edges=edges, faces=faces)
                fxn["out_{}_{}".format(mode, tag)] = o0.numpy()
                if mode == "vertices":
                    st = lambda a, b: torch.stack((a.to(dt), b.to(dt)), dim=0)
                    ob = nt(st(verts, verts_b), st(mass, mass_b), L=None, evals=st(evals, evals_b),
                            evecs=st(evecs, evecs_b), gradX=st(gradX, gX_b), gradY=st(gradY, gY_b))
                    fxn["out_batch2_" + tag] = ob.numpy()
    save("net_small.npz", fxn)

    # ---- 6. state_dict manifest of the shipped checkpoints (names/shapes only) ----
    man = {}
    exp = os.path.join(os.path.dirname(reference_src()), "experiments")
    for sub, fn in (("human_segmentation_original", "human_seg_xyz_4x128.pth"),
                    ("human_segmentation_original", "human_seg_hks_4x128.pth"),
                    ("functional_correspondence", "faust_xyz.pth"),
                    ("sampling_invariance", None)):
        d = os.path.join(exp, sub, "pretrained_models")
        if not os.path.isdir(d):
            continue
        for f in sorted(os.listdir(d)):
            if fn is not None and f != fn:
                continue
            sdp = torch.load(os.path.join(d, f), map_location="cpu", weights_only=True)
            man[sub + "/" + f] = {k: list(v.shape) for k, v in sdp.items()}
    if not only or "statedict_manifest.json" in only:
        with open(os.path.join(OUT, "statedict_manifest.json"), "w") as fh:
            json.dump(man, fh, indent=1, sort_keys=True)

    # ---- 7. one shipped checkpoint: every name in file order with its shape, and a seeded sample of 16 values per
    #         tensor (the whole file is 1.9 MB) ----
    ckpt = os.path.join(exp, "human_segmentation_original", "pretrained_models", "human_seg_xyz_4x128.pth")
    if os.path.isfile(ckpt):
        sdp = torch.load(ckpt, map_location="cpu", weights_only=True)
        rs = np.random.RandomState(0)
        fxc = {"names": np.array(list(sdp))}
        for k, v in sdp.items():
            flat = v.reshape(-1).numpy()
            idx = np.sort(rs.choice(flat.size, min(16, flat.size), replace=False)).astype(np.int64)
            fxc.update({"shape:" + k: np.array(v.shape, dtype=np.int64), "idx:" + k: idx, "val:" + k: flat[idx]})
        save("checkpoint_human_seg_xyz_4x128.npz", fxc)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main(sys.argv[1:])
