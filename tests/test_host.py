"""CPU-side checks: the C-ABI library builds, loads and exports every symbol the header declares;
the module mirror keeps the reference's names/keys/errors; host-side sharding and the gradient
all-reduce (gloo, world_size 2).  No GPU compute here."""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from conftest import ROOT, GOLDEN, load_golden

import diffusion_net_b200 as dn


def test_library_builds_and_exports_header_symbols():
    dn._lib.build()
    lib = dn._lib.load()
    hdr = open(os.path.join(ROOT, "include", "diffusion_net_b200.h")).read()
    declared = set(re.findall(r"\b(dn_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(dn._lib.SIGNATURES), declared ^ set(dn._lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.dn_abi_version() == 5
    assert lib.dn_error_string(-3).decode().startswith("diffusion_net_b200: workspace")
    assert lib.dn_workspace_bytes(200000, 128, 128) > 0
    assert lib.dn_workspace_bytes(-1, 128, 128) == -1


def test_sass_is_sm100a_only():
    cuobjdump = os.path.join(os.path.dirname(dn._lib.nvcc()), "cuobjdump")     # beside nvcc, which need not be on PATH
    out = subprocess.run([cuobjdump, "-lelf", dn._lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_state_dict_keys_match_shipped_checkpoints():
    man = json.load(open(os.path.join(GOLDEN, "statedict_manifest.json")))
    assert man
    for name, keys in man.items():
        # the functional-map checkpoints wrap the net as `feature_extractor.` (fmaps_model.py)
        pre = "feature_extractor."
        if all(k.startswith(pre) for k in keys):
            keys = {k[len(pre):]: v for k, v in keys.items()}
        C_in = keys["first_lin.weight"][1]
        C_out = keys["last_lin.weight"][0]
        C_width = keys["first_lin.weight"][0]
        n_block = len([k for k in keys if k.endswith("diffusion.diffusion_time")])
        net = dn.DiffusionNet(C_in=C_in, C_out=C_out, C_width=C_width, N_block=n_block)
        ours = {k: list(v.shape) for k, v in net.state_dict().items()}
        assert ours == keys, name


def test_live_checkpoint_strict_load():
    """The reference's pretrained human-segmentation model (human_seg_xyz_4x128.pth), rebuilt from its stored names,
    order and shapes with a sample of its values (oracle/make_golden.py), loads strictly, and every sampled value lands
    in the parameter of that name."""
    fx = load_golden("checkpoint_human_seg_xyz_4x128")
    names = [str(k) for k in fx["names"]]
    sd = {}
    for k in names:
        t = torch.zeros(tuple(int(s) for s in fx["shape:" + k]))
        t.view(-1)[torch.from_numpy(fx["idx:" + k])] = torch.from_numpy(fx["val:" + k])
        sd[k] = t
    net = dn.DiffusionNet(C_in=3, C_out=8, C_width=128, N_block=4, outputs_at="faces")
    net.load_state_dict(sd, strict=True)
    assert len(net.blocks) == 4 and net.blocks[0] is net.block_0
    ours = net.state_dict()
    assert list(ours) == names
    for k in names:
        assert torch.equal(ours[k].view(-1)[torch.from_numpy(fx["idx:" + k])], torch.from_numpy(fx["val:" + k])), k


def test_variant_keys_and_module_layout():
    b = dn.DiffusionNetBlock(16, [16, 16], with_gradient_rotations=False)
    assert "gradient_features.A.weight" in b.state_dict()
    b2 = dn.DiffusionNetBlock(16, [16, 16], with_gradient_features=False)
    assert b2.state_dict()["mlp.miniMLP_mlp_layer_000.weight"].shape == (16, 32)
    kinds = [type(m).__name__ for m in dn.MiniMLP([48, 16, 16, 16], dropout=True)]
    assert kinds == ["Linear", "ReLU", "Dropout", "Linear", "ReLU", "Dropout", "Linear"]
    assert float(dn.LearnedTimeDiffusion(8).diffusion_time.abs().sum()) == 0.0


def test_errors_match_reference():
    with pytest.raises(ValueError, match="invalid setting for outputs_at"):
        dn.DiffusionNet(3, 4, outputs_at="bad")
    with pytest.raises(ValueError, match="invalid setting for diffusion_method"):
        dn.DiffusionNet(3, 4, diffusion_method="bad")
    net = dn.DiffusionNet(3, 4, C_width=16, N_block=1)
    with pytest.raises(ValueError, match="C_in=3"):
        net(torch.zeros(10, 5), torch.ones(10))
    with pytest.raises(ValueError, match="shape"):
        net(torch.zeros(2, 2, 10, 3), torch.ones(10))
    blk = dn.DiffusionNetBlock(16, [16, 16])
    with pytest.raises(ValueError, match="wrong shape"):
        blk(torch.zeros(1, 10, 5), None, None, None, None, None, None)
    # no CPU fallback: the product path refuses CPU tensors loudly
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        blk(torch.zeros(1, 10, 16), torch.ones(1, 10), None, torch.zeros(1, 4), torch.zeros(1, 10, 4), None, None)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "diffusion-net_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), os.path.join(dirpath, f)


def test_shard_meshes_lpt():
    from diffusion_net_b200.dist import shard_meshes, mesh_cost
    costs = [mesh_cost(1800 + 50 * (i % 9), 128, 128) for i in range(32)]
    for ws in (1, 2, 4, 8):
        shards = shard_meshes(costs, ws)
        flat = sorted(i for s in shards for i in s)
        assert flat == list(range(32))
        loads = [sum(costs[i] for i in s) for s in shards]
        assert max(loads) <= min(loads) * 1.1 + 1
    assert shard_meshes([5, 1, 1, 1], 2) == [[0], [1, 2, 3]]


def test_allreduce_gradients_gloo_world2(tmp_path):
    script = tmp_path / "w.py"
    script.write_text('''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from diffusion_net_b200.dist import allreduce_gradients, shard_meshes
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
torch.manual_seed(0)
lin = torch.nn.Linear(4, 3)
frozen = torch.nn.Parameter(torch.ones(2), requires_grad=False)
for p in lin.parameters():
    p.grad = torch.full_like(p, float(r + 1))
allreduce_gradients(list(lin.parameters()) + [frozen], n_global_meshes=4)
exp = sum(range(1, w + 1)) / 4.0
assert all(torch.allclose(p.grad, torch.full_like(p, exp)) for p in lin.parameters())
assert frozen.grad is None
mine = shard_meshes([3.0, 2.0, 2.0, 1.0], w)[r]
got = [None] * w
dist.all_gather_object(got, mine)
assert sorted(i for s in got for i in s) == [0, 1, 2, 3]
dist.barrier()
if r == 0: print("GLOO_OK")
''' % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0 and "GLOO_OK" in r.stdout, r.stdout + r.stderr


# ---- operator cache, read side (geometry.py:426-519) -- host logic only ---------------------------------------
def _geom():
    import numpy as np
    with np.load(os.path.join(GOLDEN, "geom_small.npz")) as z:
        return {k: z[k] for k in z.files}


def test_cache_probe_uses_the_reference_file_naming():
    fx = _geom()
    cache = os.path.join(GOLDEN, "op_cache")
    verts, faces = torch.from_numpy(fx["verts"]), torch.from_numpy(fx["faces"])
    assert dn.geometry.hash_arrays((fx["verts"], fx["faces"])) + "_0.npz" == str(fx["cache_file"])
    npz = dn.geometry.find_cached_operators(verts, faces, 16, cache)
    assert npz is not None and int(npz["k_eig"].item()) == 16
    assert dn.geometry.find_cached_operators(verts, faces, 12, cache) is not None       # fewer eigenpairs: still a hit
    assert dn.geometry.find_cached_operators(verts, faces, 17, cache) is None           # geometry.py:482-485
    assert dn.geometry.find_cached_operators(verts + 1.0, faces, 16, cache) is None     # other mesh: miss


def test_cache_miss_and_cpu_device_fail_loudly():
    fx = _geom()
    cache = os.path.join(GOLDEN, "op_cache")
    verts, faces = torch.from_numpy(fx["verts"]), torch.from_numpy(fx["faces"])
    with pytest.raises(NotImplementedError, match="populate the cache"):
        dn.geometry.get_operators(verts + 1.0, faces, 16, cache, device="cuda")
    with pytest.raises(NotImplementedError):
        dn.geometry.get_operators(verts, faces, 16, None, device="cuda")
    with pytest.raises(RuntimeError, match="CUDA devices only"):
        dn.geometry.get_operators(verts, faces, 16, cache)            # default device = verts.device = cpu
    bad = verts.clone()
    bad[0, 0] = float("nan")
    with pytest.raises(RuntimeError, match="NaN verts"):              # geometry.py:438-439
        dn.geometry.get_operators(bad, faces, 16, cache)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        dn.geometry.compute_hks(torch.zeros(4), torch.zeros(3, 4), torch.ones(2))


# ---- dn_patch_build: host-side clustering for the gather kernel (include/diffusion_net_b200.h dn_patches) --------
def _patch_build(rp, ci, V, T, R):
    import ctypes as C
    import numpy as np
    nnz = len(ci)
    tgt_ptr, src_ptr, ent_ptr = (np.empty(V + 1, np.int32) for _ in range(3))
    tgt, src_rows, perm = np.empty(V, np.int32), np.empty(max(nnz, 1), np.int32), np.empty(max(nnz, 1), np.int32)
    lcol, worst = np.empty(max(nnz, 1), np.uint8), np.zeros(1, np.int32)
    hp = lambda a: C.c_void_p(a.ctypes.data)
    n = dn._lib.load().dn_patch_build(V, hp(rp), hp(ci), T, R, hp(tgt_ptr), hp(tgt), hp(src_ptr), hp(src_rows),
                                      hp(ent_ptr), hp(lcol), hp(perm), hp(worst))
    return n, tgt_ptr, tgt, src_ptr, src_rows, ent_ptr, lcol, perm, int(worst[0])


@pytest.mark.parametrize("permute", [False, True])
def test_patch_build_covers_every_row_once_and_reproduces_the_spmm(permute):
    import numpy as np
    import scipy.sparse as sp
    n_, m_ = 30, 41
    V = n_ * m_
    rows, cols = (np.asarray(a) for a in dn.synthetic.torus_pattern(n_, m_))
    rng = np.random.default_rng(3)
    A = sp.csr_matrix((rng.standard_normal(len(rows)).astype(np.float32), (rows, cols)), shape=(V, V))
    A = sp.vstack([A[:17], sp.csr_matrix((3, V), dtype=np.float32), A[20:]]).tocsr()    # three empty rows
    if permute:
        pv = rng.permutation(V)
        A = A[pv][:, pv].tocsr()
    A.sort_indices()
    rp, ci = A.indptr.astype(np.int32), A.indices.astype(np.int32)
    for T, R in ((64, 144), (32, 72), (5, 9)):
        n, tgt_ptr, tgt, src_ptr, src_rows, ent_ptr, lcol, perm, worst = _patch_build(rp, ci, V, T, R)
        assert n > 0 and tgt_ptr[n] == V and ent_ptr[V] == A.nnz
        assert np.array_equal(np.sort(tgt), np.arange(V))                      # every row exactly once
        assert np.array_equal(np.sort(perm[:A.nnz]), np.arange(A.nnz))         # every entry exactly once
        sizes, nsrc = np.diff(tgt_ptr[:n + 1]), np.diff(src_ptr[:n + 1])
        assert sizes.min() >= 1 and sizes.max() <= T and nsrc.max() <= R and nsrc.max() == worst
        # emulate the kernel: out[tgt[i]] = sum_e vals_p[e] * x[src_rows[src_ptr[p] + lcol[e]]], entries in CSR order
        x = rng.standard_normal(V)
        out = np.zeros(V)
        vals_p = A.data[perm[:A.nnz]]
        for p_ in range(n):
            src = src_rows[src_ptr[p_]:src_ptr[p_ + 1]]
            assert len(np.unique(src)) == len(src)
            for i in range(tgt_ptr[p_], tgt_ptr[p_ + 1]):
                e0, e1 = ent_ptr[i], ent_ptr[i + 1]
                assert np.array_equal(perm[e0:e1], np.arange(rp[tgt[i]], rp[tgt[i] + 1]))   # row's entries, same order
                out[tgt[i]] = np.dot(vals_p[e0:e1], x[src[lcol[e0:e1]]])
        assert np.allclose(out, A @ x, rtol=1e-12, atol=1e-12)
    assert _patch_build(rp, ci, V, 64, 3)[0] == -2                              # a row longer than max_src


def test_mesh_batch_plan_host():
    """dn_mesh_batch_plan (host-only): 128-aligned mesh starts, tile -> mesh table, to_basis CTAs that tile every
    mesh exactly and never cross one."""
    import ctypes as C
    import numpy as np
    import diffusion_net_b200 as dn
    lib = dn._lib.load()
    for n_rows in ([1800, 2200, 1, 0, 129, 128, 4000], [2000] * 32, [200000], [5] * 300):
        B = len(n_rows)
        nr = np.asarray(n_rows, dtype=np.int32)
        row_begin = np.zeros(B + 1, dtype=np.int32)
        tile_mesh = np.full(sum((v + 127) // 128 for v in n_rows) + 1, -1, dtype=np.int32)
        tb_rows = np.zeros(2048, dtype=np.int32)
        cta_begin = np.zeros(B + 1, dtype=np.int32)
        n = lib.dn_mesh_batch_plan(B, nr.ctypes.data, 148, row_begin.ctypes.data, tile_mesh.ctypes.data,
                                   tb_rows.ctypes.data, cta_begin.ctypes.data)
        assert 1 <= n <= 1024
        assert cta_begin[0] == 0 and cta_begin[B] == n
        for b in range(B):
            assert row_begin[b] % 128 == 0 and row_begin[b + 1] - row_begin[b] == (n_rows[b] + 127) // 128 * 128
            assert (tile_mesh[row_begin[b] // 128:row_begin[b + 1] // 128] == b).all()
            lo, hi = cta_begin[b], cta_begin[b + 1]
            assert hi > lo
            cur = row_begin[b]
            for c in range(lo, hi):
                rb, re = tb_rows[2 * c], tb_rows[2 * c + 1]
                assert rb == cur and (re > rb or n_rows[b] == 0) and (rb - row_begin[b]) % 16 == 0
                cur = re
            assert cur == row_begin[b] + n_rows[b]
    assert lib.dn_mesh_batch_plan(0, None, 148, None, None, None, None) < 0
