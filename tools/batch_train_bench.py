"""Training step over a batch of meshes, one GPU: one CUDA graph per mesh (graphs.GraphedTrainStep around ``net(...)``)
against one graph for the whole batch (graphs.GraphedTrainStep around ``net.forward_batch`` on a MeshBatch).

Both routes run the same 4-block DiffusionNet (K = 128, C = 128, C_in = 16, 8 classes, log_softmax head, dropout off) on
the same meshes with the same per-mesh nll losses, summed over the batch.  Prints one JSON line per configuration:
median ms per step (CUDA events around each step, after warm-up), the library kernels each route launches per step
(counted on an eager step: a graph replays exactly that sequence), the largest relative difference of any parameter's
gradient between the two routes, and the device name and power limit read in the same run.

  python tools/batch_train_bench.py [--config 5|4|all] [--steps 30] [--warmup 5]
    config 5: 8 meshes of 100 x 200 = 20000 vertices (BASELINE config 5, bench.py --workload train)
    config 4: 32 meshes of 36..44 x 50 ~= 2000 vertices (BASELINE config 4, trained instead of inferred)
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import diffusion_net_b200 as dn  # noqa: E402

K, C, C_IN, C_OUT, NB = 128, 128, 16, 8, 4
CONFIGS = {"5": [(100, 200)] * 8, "4": [(36 + i % 9, 50) for i in range(32)]}


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        power = r.stdout.strip() or "unavailable"
    except (OSError, subprocess.SubprocessError):
        power = "unavailable"
    return name, power


def seeded_net(dev):
    net = dn.DiffusionNet(C_in=C_IN, C_out=C_OUT, C_width=C, N_block=NB, dropout=False,
                          last_activation=lambda x: torch.nn.functional.log_softmax(x, dim=-1))
    g = torch.Generator().manual_seed(77)
    sd = net.state_dict()
    for k, v in sd.items():
        if k.endswith("diffusion_time"):
            v.copy_(1e-3 + 0.3 * torch.rand(v.shape, generator=g))
        else:
            fan_in = v.shape[-1] if v.dim() > 1 else C
            v.copy_((torch.rand(v.shape, generator=g) * 2 - 1) / (fan_in ** 0.5))
    net.load_state_dict(sd)
    return net.to(dev).train()


def make_meshes(shapes, dev):
    out = []
    for i, (n, m) in enumerate(shapes):
        ops_t = dn.synthetic.structural_operators(n, m, K, seed=i, device=dev)
        g = torch.Generator().manual_seed(900 + i)
        x = torch.randn(n * m, C_IN, generator=g).to(dev)
        y = torch.randint(0, C_OUT, (n * m,), generator=g).to(dev)
        out.append((x, y, ops_t))
    return out


def mesh_loss(net, x, y, ops_t):
    mass, L, evals, evecs, gX, gY = ops_t
    return torch.nn.functional.nll_loss(net(x, mass, evals=evals, evecs=evecs, gradX=gX, gradY=gY), y)


def run(name, shapes, steps, warmup, dev, lib):
    net = seeded_net(dev)
    meshes = make_meshes(shapes, dev)
    mb = dn.MeshBatch([dict(mass=o[0], evals=o[2], evecs=o[3], gradX=o[4], gradY=o[5]) for _, _, o in meshes])
    xb = mb.pack([x for x, _, _ in meshes])
    ys = [y for _, y, _ in meshes]

    def batch_loss(net_, x_, *ys_):
        return sum(torch.nn.functional.nll_loss(o, y) for o, y in zip(net_.forward_batch(mb, x_), ys_))

    def grads_and_launches(step):
        for p_ in net.parameters():
            p_.grad = None
        torch.cuda.synchronize()
        n0 = lib.dn_kernel_launch_count()
        step()
        torch.cuda.synchronize()
        return [p_.grad.clone() for p_ in net.parameters()], int(lib.dn_kernel_launch_count() - n0)

    def eager_per_mesh():
        for m in meshes:
            mesh_loss(net, *m).backward()

    grads_pm, launches_pm = grads_and_launches(eager_per_mesh)
    grads_b, launches_b = grads_and_launches(lambda: batch_loss(net, xb, *ys).backward())
    grad_diff = max(float((a - b).abs().max() / (b.abs().max() + 1e-30)) for a, b in zip(grads_b, grads_pm))

    g_pm = [dn.graphs.GraphedTrainStep(net, mesh_loss, m) for m in meshes]
    g_b = dn.graphs.GraphedTrainStep(net, batch_loss, (xb, *ys))

    def step_pm():
        dn.graphs.GraphedTrainStep.zero_grads(net)
        for g_ in g_pm:
            g_.replay()

    def step_b():
        dn.graphs.GraphedTrainStep.zero_grads(net)
        g_b.replay()

    def timed(step):
        for _ in range(warmup):
            step()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for a, b in ev:
            a.record()
            step()
            b.record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev]

    # two rounds, alternating the routes so that both see the same machine state; median over all timed steps
    res = {"per_mesh": [], "batched": []}
    for _ in range(2):
        res["per_mesh"] += timed(step_pm)
        res["batched"] += timed(step_b)
    med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
    # graph replays reproduce the eager gradients of their route
    step_b()
    torch.cuda.synchronize()
    graph_vs_eager = max(float((p_.grad - r).abs().max() / (r.abs().max() + 1e-30)) for p_, r in zip(net.parameters(), grads_b))
    dev_name, power = device_info()
    V = sum(x.shape[0] for x, _, _ in meshes)
    return {"config": name, "meshes": len(shapes), "vertices_total": V, "padded_rows": mb.V, "K": K, "C_width": C,
            "n_block": NB, "loss": "sum of per-mesh nll_loss", "engine": dn.get_engine(),
            "ms_per_step_per_mesh_graphs": med["per_mesh"], "ms_per_step_batched_graph": med["batched"],
            "speedup_batched": med["per_mesh"] / med["batched"],
            "ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in res.items()},
            "launches_per_step_per_mesh": launches_pm, "launches_per_step_batched": launches_b,
            "max_rel_grad_diff_batched_vs_per_mesh": grad_diff, "max_rel_grad_diff_batched_graph_vs_eager": graph_vs_eager,
            "steps": steps, "warmup": warmup, "device": dev_name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--config", choices=["5", "4", "all"], default="all")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if not torch.cuda.is_available():
        sys.exit("batch_train_bench.py needs a GPU")
    dn.set_engine(os.environ.get("DN_B200_ENGINE", "tc3x"))
    dev = torch.device("cuda", 0)
    lib = dn._lib.load()
    for name in (["5", "4"] if args.config == "all" else [args.config]):
        print(json.dumps(run("config" + name, CONFIGS[name], args.steps, args.warmup, dev, lib)), flush=True)


if __name__ == "__main__":
    main()
