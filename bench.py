#!/usr/bin/env python
"""DiffusionNetBlock forward throughput (BASELINE.json metric): Mverts/s at V=200k, K=128, C=128.

    python bench.py --gpus 1 --steps 20 --warmup 3            # our arm (one JSON line on rank 0)
    python bench.py --steps 20 --dump-outputs DIR             # ... and DIR/out.npy: sampled output of the last step
    python bench.py --impl reference --steps 5 --warmup 1      # the reference's CPU path (torch-CPU port)
    torchrun ... bench.py --gpus N ...                         # one rank per GPU, one mesh per rank (weak scaling)

A "step" is one DiffusionNetBlock forward (eval, no_grad, fp32) over one synthetic mesh per GPU:
Tier-S operators on a 400x500 torus (V=200000, 7 nnz/row, M-orthonormal random eigenbasis, K=128),
C_width=128, seeded weights (SURVEY.md section 8d).  `value` has all inputs resident in HBM; `e2e`
goes through the public module API from pinned HOST buffers (H2D of features + the whole operator
tuple, CSR prep, forward, D2H of the result inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TORUS, M_TORUS, K_EIG, C_WIDTH = 400, 500, 128, 128
NNZ_ROW = 7
METRIC = "DiffusionNetBlock forward Mverts/sec at V=200k,K=128,C=128; 1/2/4/8 GPU"
WORKLOAD = "block_fwd V=200000 K=128 C=128, 1 mesh per GPU"      # identical in both arms (config.workload)
# --dump-outputs: the whole (V, C) output is 102 MB, so a fixed sample of 2^16 of its rows (32 MB) is written
DUMP_ROWS, DUMP_SEED = 1 << 16, 0


def flops_per_vertex(K, C, r=NNZ_ROW):
    return 4 * K * C + 18 * C * C + 4 * r * C           # SURVEY.md 8d (reference op count)


def bytes_per_vertex(K, C, r=NNZ_ROW, s=4):
    return s * (5 * C + 2 * K) + 12 * r + 8             # SURVEY.md 8d (minimum HBM traffic)


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            m = json.load(fh)
        p.update({k: m[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in m})
        p["source"] = "measured"
    except Exception:
        pass
    return p


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the GPU is under the benchmark load
    (profiling recipe).  Rows are time-stamped on arrival; stop() reports the samples that fell
    inside [t_begin, t_end] (the timed region plus, if that is shorter than a few sampling
    periods, the identical-load extension the caller ran while sampling)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:   # wait for the first sample
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def count_since(self, t_begin):
        return sum(1 for t, _ in self.rows if t >= t_begin)

    def stop(self, t_begin, t_end):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        isnum = lambda x: x.replace(".", "", 1).isdigit()
        rows = [r for t, r in self.rows if t_begin <= t <= t_end and r and isnum(r[0])]
        if not rows:
            return None
        sm = sorted(float(r[0]) for r in rows)
        mx = max(float(r[1]) for r in rows if len(r) > 1 and isnum(r[1]))
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower() == "active"
                                                          for r in rows)]
        pw = [float(r[2]) for r in rows if len(r) > 2 and isnum(r[2])]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm),
                "power_w_max": max(pw) if pw else None}


def make_workload(dn, device, seed):
    import torch
    ops_t = dn.synthetic.structural_operators(N_TORUS, M_TORUS, K_EIG, seed=seed, device="cpu")
    params = dn.synthetic.block_weights(C_WIDTH, seed=seed)
    x = torch.randn(N_TORUS * M_TORUS, C_WIDTH, generator=torch.Generator().manual_seed(100 + seed))
    return ops_t, params, x


def _reference_block(params, device):
    """The reference's own DiffusionNetBlock (oracle/_ref, staged by oracle/stage_ref.py) with our seeded weights,
    or None when no staged copy travelled to this box (then the torch restatement in oracle/ is timed instead)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_import                      # checker/baseline infrastructure; never on the product path
    if not ref_import.reference_available():
        return None
    ref = ref_import.import_reference()
    blk = ref.layers.DiffusionNetBlock(C_width=C_WIDTH, mlp_hidden_dims=[C_WIDTH, C_WIDTH], dropout=False)
    blk.load_state_dict(params, strict=True)
    return blk.to(device).eval()


def make_baseline_step(host, params, device):
    """One reference block forward (eval, fp32) on `device`: the reference module itself when staged (kind
    "reference"), else its torch restatement (kind "port").  Stacked (B,V,V) sparse operators, as
    DiffusionNet.forward hands them to the block."""
    import torch
    mass, L, evals, evecs, gradX, gradY, x = [t.to(device) for t in host]
    xb, mb, eb, vb = x.unsqueeze(0), mass.unsqueeze(0), evals.unsqueeze(0), evecs.unsqueeze(0)
    gxb, gyb = gradX.unsqueeze(0), gradY.unsqueeze(0)
    blk = _reference_block(params, device)
    if blk is not None:
        def step():
            with torch.no_grad():
                return blk(xb, mb, None, eb, vb, gxb, gyb)
        return step, "reference"
    import dn_oracle_torch as T
    prm = {k: v.to(device) for k, v in params.items()}

    def step():
        with torch.no_grad():
            return T.block_forward(xb, mb, eb, vb, gxb, gyb, prm)
    return step, "port"


def time_cpu_baseline(host, params, steps, warmup):
    """The reference's CPU PyTorch path on the host cores.  The thread count is picked by a small sweep (one step
    each): oversubscribing the box (128 logical cores) was 3-4x slower than 8-32 threads in round 1."""
    import torch
    step, kind = make_baseline_step(host, params, "cpu")
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu} or {ncpu})
    sweep = {}
    step()                                           # first-touch / lazy init outside the sweep
    for c in cands:
        torch.set_num_threads(c)
        step()
        t0 = time.perf_counter()
        step()
        sweep[c] = time.perf_counter() - t0
    best = min(sweep, key=sweep.get)
    torch.set_num_threads(best)
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2], best, kind, {str(k): round(v, 3) for k, v in sweep.items()}


def run_reference(args, rank):
    if rank != 0:
        return
    import diffusion_net_b200 as dn
    V = N_TORUS * M_TORUS
    (mass, L, evals, evecs, gradX, gradY), params, x = make_workload(dn, "cpu", 0)
    steps, warm = args.steps, max(1, args.warmup)
    sec, cores, kind, sweep = time_cpu_baseline((mass, L, evals, evecs, gradX, gradY, x), params, steps, warm)
    val = V / sec / 1e6
    sample = "full workload: 1 mesh V={} K={} C={}, {} steps (median), {} warm-up; threads picked by sweep {}".format(
        V, K_EIG, C_WIDTH, steps, warm, sweep)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mverts/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "device": "cpu (the reference's CPU PyTorch path on the host cores)"},
        "cpu_baseline": {"value": val, "unit": "Mverts/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "Mverts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def measure_tf32_peak(dev, secs=1.0):
    """cuBLAS TF32 GEMM (8192^3) on this GPU, burst (best of 10) and sustained (back to back for `secs`): the
    denominator for kind::tf32 tensor-pipe fractions (MEASURED_PEAKS.json only holds the bf16 rate)."""
    import torch
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize(dev)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); a @ b; e1.record(); torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1))
        t0, cnt = time.time(), 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        while time.time() - t0 < secs:
            for _ in range(10):
                a @ b
            cnt += 10
            torch.cuda.synchronize(dev)
        e1.record(); torch.cuda.synchronize(dev)
        f = 2.0 * n ** 3 / 1e12
        return {"tf32_tflops": f / (best * 1e-3), "tf32_tflops_sustained": f / (e0.elapsed_time(e1) / cnt * 1e-3),
                "how": "torch.matmul fp32 8192^3 with allow_tf32 (cuBLAS TF32), in this run"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


# ------------------------------------------------------------------------------------------------
# Auxiliary workloads (BASELINE.json configs 2, 4, 5).  The headline metric and the driver's runs use the default
# `--workload block_fwd`; these print the same kind of JSON line for their own metric.
# ------------------------------------------------------------------------------------------------
def _seeded_net(dn, C_in, C_out, C, n_block, dev, seed=0):
    """4-block DiffusionNet with seeded weights (dropout off: the bench compares numerically identical runs)."""
    import torch
    net = dn.DiffusionNet(C_in=C_in, C_out=C_out, C_width=C, N_block=n_block, dropout=False,
                          last_activation=lambda x: torch.nn.functional.log_softmax(x, dim=-1))
    g = torch.Generator().manual_seed(77 + seed)
    sd = net.state_dict()
    for k, v in sd.items():
        if k.endswith("diffusion_time"):
            v.copy_(1e-3 + 0.3 * torch.rand(v.shape, generator=g))
        else:
            fan_in = v.shape[-1] if v.dim() > 1 else C
            v.copy_((torch.rand(v.shape, generator=g) * 2 - 1) / (fan_in ** 0.5))
    net.load_state_dict(sd)
    return net.to(dev)


def _reference_net(state_dict, C_in, C_out, C, n_block, dev):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_import
    if not ref_import.reference_available():
        return None
    ref = ref_import.import_reference()
    net = ref.layers.DiffusionNet(C_in=C_in, C_out=C_out, C_width=C, N_block=n_block, dropout=False,
                                  last_activation=lambda x: torch.nn.functional.log_softmax(x, dim=-1))
    net.load_state_dict(state_dict, strict=True)
    return net.to(dev)


def _mesh_batch(dn, shapes, K, C_in, dev, seed0=0):
    import torch
    out = []
    for i, (n, m) in enumerate(shapes):
        ops_t = dn.synthetic.structural_operators(n, m, K, seed=seed0 + i, device=dev)
        g = torch.Generator().manual_seed(900 + seed0 + i)
        x = torch.randn(n * m, C_in, generator=g).to(dev)
        y = torch.randint(0, 8, (n * m,), generator=g).to(dev)
        out.append((x, y, ops_t))
    return out


def _net_loss(net, x, y, ops_t):
    import torch
    mass, L, evals, evecs, gX, gY = ops_t
    pred = net(x, mass, L=None, evals=evals, evecs=evecs, gradX=gX, gradY=gY)
    return torch.nn.functional.nll_loss(pred, y)


def run_aux(args, rank, world, local):
    import torch
    import torch.distributed as dist
    import diffusion_net_b200 as dn
    assert torch.cuda.is_available()
    dn.dist.bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dn.set_engine(args.engine)
    lib = dn._lib.load()
    steps, warm = args.steps, max(3, args.warmup)
    K, C, C_in, C_out, NB = 128, 128, 16, 8, 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        for _ in range(warm):
            fn()
        barrier()
        l0 = lib.dn_kernel_launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, int(lib.dn_kernel_launch_count() - l0)

    line = {"unit": "Mverts/s", "n_gpus": world, "steps": steps, "warmup": warm, "higher_is_better": True,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    if args.workload == "fwd_bwd":
        # config 2: human-seg shape, one mesh per GPU, forward + backward of the 4-block net (no optimiser)
        shapes = [(84, 84)]
        net = _seeded_net(dn, C_in, C_out, C, NB, dev, seed=0).train()
        (x, y, ops_t), = _mesh_batch(dn, shapes, K, C_in, dev, seed0=rank)
        V = x.shape[0]

        def step():
            for p_ in net.parameters():
                p_.grad = None
            _net_loss(net, x, y, ops_t).backward()
        ms_eager, launches = timed(step)
        # the same forward + backward as ONE CUDA graph (graphs.GraphedTrainStep): the route the metric is quoted on
        gts = dn.graphs.GraphedTrainStep(net, _net_loss, (x, y, ops_t))

        def gstep():
            dn.graphs.GraphedTrainStep.zero_grads(net)
            gts.replay()
        ms, _ = timed(gstep)
        # the graph reproduces the eager gradients
        step()
        ref_g = [p_.grad.clone() for p_ in net.parameters()]
        gstep()
        torch.cuda.synchronize()
        graph_vs_eager = max(float((p_.grad - r).abs().max() / (r.abs().max() + 1e-30)) for p_, r in zip(net.parameters(), ref_g))
        with torch.no_grad():
            net.eval()
            ms_f, _ = timed(lambda: _net_loss(net, x, y, ops_t))
            net.train()
        gpu_base = None
        if rank == 0 and world == 1:
            try:
                prev = torch.backends.cuda.matmul.allow_tf32
                torch.backends.cuda.matmul.allow_tf32 = False
                rnet = _reference_net(net.state_dict(), C_in, C_out, C, NB, dev)
                if rnet is not None:
                    rnet.train()

                    def rstep():
                        for p_ in rnet.parameters():
                            p_.grad = None
                        _net_loss(rnet, x, y, ops_t).backward()
                    rms, _ = timed(rstep)
                    # gradient parity of the two arms on the same inputs
                    step(); rstep()
                    worst = 0.0
                    for (n1, p1), (n2, p2) in zip(net.named_parameters(), rnet.named_parameters()):
                        worst = max(worst, float((p1.grad - p2.grad).abs().max() / (p2.grad.abs().max() + 1e-30)))
                    gpu_base = {"value": V / (rms * 1e-3) / 1e6, "unit": "Mverts/s", "ms_per_step": rms,
                                "kind": "reference", "how": "reference DiffusionNet, torch eager autograd on this B200, "
                                "fp32 (TF32 off)", "speedup_ours": rms / ms, "max_rel_grad_diff_vs_ours": worst}
                torch.backends.cuda.matmul.allow_tf32 = prev
            except Exception as exc:
                gpu_base = {"unavailable": repr(exc)[:200]}
        line.update({"metric": "DiffusionNet (4 blocks) forward+backward Mverts/sec at V=7056,K=128,C=128",
                     "value": world * V / (ms * 1e-3) / 1e6, "ms_per_step": ms, "scaling": "weak",
                     "config": {"workload": "net_fwd_bwd V=7056 K=128 C=128 4 blocks, 1 mesh per GPU",
                                "engine": args.engine, "forward_only_ms": ms_f, "route": "forward + backward replayed as one "
                                "CUDA graph (graphs.GraphedTrainStep)", "eager_autograd_ms": ms_eager,
                                "graph_vs_eager_max_rel_grad_diff": graph_vs_eager},
                     "gpu_launches": launches, "gpu_baseline": gpu_base})
    elif args.workload == "train":
        # config 5: global batch of 8 meshes (V = 20000 each), data parallel: every rank takes 8 / world meshes, one flat
        # NCCL all-reduce of the gradients (mean over the 8 meshes), one Adam step.  Strong scaling (global work fixed).
        n_global = 8
        shards = dn.dist.shard_meshes([dn.dist.mesh_cost(20000, K, C)] * n_global, world)
        mine = shards[rank]
        net = _seeded_net(dn, C_in, C_out, C, NB, dev, seed=0).train()
        meshes = _mesh_batch(dn, [(100, 200)] * n_global, K, C_in, dev, seed0=0)
        meshes = [meshes[i] for i in mine]
        opt = torch.optim.Adam(net.parameters(), lr=1e-3, fused=True)
        ar_ms = []

        use_graphs = os.environ.get("DN_TRAIN_GRAPHS", "1") != "0"
        gts = [dn.graphs.GraphedTrainStep(net, _net_loss, m) for m in meshes] if use_graphs else []

        def step():
            if use_graphs:                                     # one CUDA graph (forward + backward) per mesh of this rank
                dn.graphs.GraphedTrainStep.zero_grads(net)
                for g_ in gts:
                    g_.replay()
            else:
                opt.zero_grad(set_to_none=True)
                for x, y, ops_t in meshes:
                    _net_loss(net, x, y, ops_t).backward()     # gradients accumulate over this rank's meshes
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dn.dist.allreduce_gradients(net.parameters(), n_global_meshes=n_global)
            e1.record()
            ar_ms.append((e0, e1))
            opt.step()
        ms, launches = timed(step)
        torch.cuda.synchronize()
        ar = sorted(a.elapsed_time(b) for a, b in ar_ms[-steps:])
        Vtot = n_global * 20000
        nparam = sum(p_.numel() for p_ in net.parameters())
        line.update({"metric": "DiffusionNet (4 blocks) data-parallel training step, 8 meshes V=20000, Mverts/sec",
                     "value": Vtot / (ms * 1e-3) / 1e6, "ms_per_step": ms, "scaling": "strong",
                     "config": {"workload": "train 8 meshes V=20000 K=128 C=128 4 blocks, dp{}".format(world),
                                "engine": args.engine, "meshes_per_rank": len(mine), "optimizer": "Adam (fused)",
                                "fwd_bwd": "one CUDA graph per mesh (graphs.GraphedTrainStep)" if use_graphs else "eager autograd",
                                "allreduce": "one flat fp32 buffer of {} floats, NCCL".format(nparam),
                                "allreduce_ms_median": ar[len(ar) // 2], "allreduce_ms_max": ar[-1]},
                     "gpu_launches": launches})
    elif args.workload == "config3":
        # config 3: large-mesh inference, V = 200k, K = 128, C_width = 256, 4 blocks, bf16 arithmetic (DN_ENGINE_BF16:
        # one bf16 tensor-core pass, fp32 accumulate; tensors stay fp32 in HBM), one mesh per GPU
        eng = "bf16" if args.engine == "tc3x" else args.engine
        dn.set_engine(eng)
        C3 = 256
        net = _seeded_net(dn, C_in, C_out, C3, NB, dev, seed=0).eval()
        (x, y, ops_t), = _mesh_batch(dn, [(N_TORUS, M_TORUS)], K, C_in, dev, seed0=rank)
        V = x.shape[0]
        mass, _, evals, evecs, gX, gY = ops_t
        gops = dn.ops.prepare_operators(gX, gY)
        with torch.no_grad():
            fwd = lambda: net(x, mass, L=None, evals=evals, evecs=evecs, gradX=gops, gradY=None)
            ms, launches = timed(fwd)
            # one block alone, with the per-stage device times of dn_block_fwd_profile
            blk = net.blocks[1]
            xb = torch.randn(V, C3, device=dev)
            A_re, A_im = blk.gradient_features.weights()
            lins = blk.mlp.linears()
            run = lambda prof=None: dn.ops.block_forward_raw(xb, mass, evals, evecs, gops, blk.diffusion.diffusion_time, A_re,
                                                             A_im, [l.weight for l in lins], [l.bias for l in lins], True,
                                                             profile=prof)
            acc = [0.0] * len(dn.ops.PROFILE_STAGES)
            for it in range(8):
                prof = []
                run(prof)
                if it >= 2:
                    acc = [a + b for a, b in zip(acc, prof)]
            stages = {k + "_ms": a / 6 for k, a in zip(dn.ops.PROFILE_STAGES, acc)}
            blk_ms, _ = timed(run)
        pk = peaks()
        mlp_flops = 2.0 * V * (3 * C3 * C3 + 2 * C3 * C3)
        mlp_ms = stages["mlp_ms"]
        blk_flops = V * flops_per_vertex(K, C3)
        blk_bytes = V * bytes_per_vertex(K, C3)
        gpu_base = None
        if rank == 0 and world == 1:
            try:
                prev = torch.backends.cuda.matmul.allow_tf32
                torch.backends.cuda.matmul.allow_tf32 = False
                rnet = _reference_net(net.state_dict(), C_in, C_out, C3, NB, dev)
                if rnet is not None:
                    rnet.eval()
                    with torch.no_grad():
                        rf = lambda: rnet(x, mass, L=None, evals=evals, evecs=evecs, gradX=gX, gradY=gY)
                        rms, _ = timed(rf)
                        err = float((fwd() - rf()).abs().max() / rf().abs().max())
                    gpu_base = {"value": V / (rms * 1e-3) / 1e6, "unit": "Mverts/s", "ms_per_step": rms, "kind": "reference",
                                "how": "reference DiffusionNet (4 x 256), torch eager on this B200, fp32 (TF32 off)",
                                "speedup_ours": rms / ms, "max_rel_diff_vs_ours": err}
                torch.backends.cuda.matmul.allow_tf32 = prev
            except Exception as exc:
                gpu_base = {"unavailable": repr(exc)[:200]}
        line.update({"metric": "DiffusionNet (4 blocks, C_width=256) forward Mverts/sec at V=200k,K=128, bf16 arithmetic",
                     "value": world * V / (ms * 1e-3) / 1e6, "ms_per_step": ms, "scaling": "weak", "dtype": "bf16 (fp32 accumulate, fp32 tensors in HBM)",
                     "config": {"workload": "config3 net_fwd V={} K=128 C=256 4 blocks, 1 mesh per GPU".format(V), "engine": eng,
                                "block_ms": blk_ms, "block_stages_ms": stages},
                     "roofline": {"bound": "tensor", "kernel": "rows_chain16_kernel (MiniMLP 768-256-256-256 + skip)",
                                  "achieved": mlp_flops / (mlp_ms * 1e-3) / 1e12, "peak": pk["bf16_tflops_sustained"],
                                  "unit": "TFLOP/s", "frac": mlp_flops / (mlp_ms * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
                                  "hbm_frac": 4.0 * V * C3 * 4 / (mlp_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                                  "block_tflops": blk_flops / (blk_ms * 1e-3) / 1e12,
                                  "block_hbm_frac_fp32_bytes": blk_bytes / (blk_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                                  "peak_source": pk["source"], "traffic": None},
                     "gpu_launches": launches, "gpu_baseline": gpu_base})
    else:
        # config 4: 32 small meshes (V ~ 2k), 4-block net forward, meshes sharded over the ranks, CUDA-graph replay
        n_global = 32
        shapes = [(36 + i % 9, 50) for i in range(n_global)]
        shards = dn.dist.shard_meshes([dn.dist.mesh_cost(a * b, K, C) for a, b in shapes], world)
        mine = shards[rank]
        net = _seeded_net(dn, C_in, C_out, C, NB, dev, seed=0).eval()
        meshes = _mesh_batch(dn, shapes, K, C_in, dev, seed0=0)
        items = [dict(x_in=meshes[i][0], mass=meshes[i][2][0], evals=meshes[i][2][2], evecs=meshes[i][2][3],
                      gradX=meshes[i][2][4], gradY=meshes[i][2][5]) for i in mine]
        # (a) one launch sequence over the whole shard: MeshBatch (one vertex range, block-diagonal CSR, per-mesh
        #     spectral weights picked per tile) -> 5-6 launches per block whatever the number of meshes
        mb = dn.MeshBatch([dict(mass=it["mass"], evals=it["evals"], evecs=it["evecs"], gradX=it["gradX"], gradY=it["gradY"])
                           for it in items])
        x_cat = mb.pack([it["x_in"] for it in items])
        with torch.no_grad():
            ms_eager, launches = timed(lambda: net.forward_batch(mb, x_cat))
            # (a') the same launch sequence replayed as ONE CUDA graph: the route the metric is quoted on (the input is
            # copied into the graph's static buffer inside the timed call)
            gb = dn.graphs.GraphedBatch(net, mb)
            ms, _ = timed(lambda: gb.forward(x_cat))
            # (b) round 1's route for comparison: per-mesh launches replayed from CUDA graphs on 4 streams
            gn = dn.graphs.GraphedNet(net, n_streams=4)
            ms_graphs, _ = timed(lambda: gn.forward_batch(items))
            outs = net.forward_batch(mb, x_cat)
            refs = gn.forward_batch(items)
            err = max(float((o - r).abs().max() / r.abs().max()) for o, r in zip(outs, refs))
        Vtot = sum(a * b for a, b in shapes)
        line.update({"metric": "DiffusionNet (4 blocks) forward over a batch of 32 small meshes, Mverts/sec",
                     "value": Vtot / (ms * 1e-3) / 1e6, "ms_per_step": ms, "scaling": "strong",
                     "config": {"workload": "small_batch 32 meshes V~2k K=128 C=128 4 blocks, sharded x{}".format(world),
                                "engine": args.engine, "meshes_per_rank": len(mine),
                                "route": "MeshBatch: one batched launch per stage (dn_block_fwd_batched), the whole forward "
                                         "replayed as one CUDA graph (graphs.GraphedBatch)",
                                "padded_rows": mb.V, "eager_launches_ms": ms_eager, "per_mesh_cuda_graphs_ms": ms_graphs,
                                "max_rel_diff_vs_per_mesh": err},
                     "gpu_launches": launches})
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default=os.environ.get("DN_B200_ENGINE", "tc3x"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--workload", default="block_fwd", choices=["block_fwd", "fwd_bwd", "train", "small_batch", "config3"],
                    help="block_fwd = the BASELINE metric (default); the others are BASELINE configs 2 / 5 / 4 / 3")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="block_fwd: after the timed steps, write the block output of the last timed step (rank 0) as "
                         "DIR/out.npy, float32, the {} rows picked by seed {} in ascending order".format(DUMP_ROWS,
                                                                                                         DUMP_SEED))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "block_fwd"):
        ap.error("--dump-outputs is implemented for the block_fwd workload of our arm only")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.workload != "block_fwd":
        run_aux(args, rank, world, local)
        return

    import torch
    import torch.distributed as dist
    import diffusion_net_b200 as dn

    assert torch.cuda.is_available(), "bench.py (our arm) needs a GPU: there is no CPU fallback"
    # NUMA: bind this rank to its GPU's socket before any pinned buffer exists (e2e scaling over the host link)
    numa_cpus = dn.dist.bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = dn._lib.load()
    dn.set_engine(args.engine)
    steps, warm = args.steps, max(3, args.warmup)
    V = N_TORUS * M_TORUS

    host_ops, params, x_host = make_workload(dn, "cpu", rank)
    mass, L, evals, evecs, gradX, gradY = [t.to(dev) for t in host_ops]
    x = x_host.to(dev)
    blk = dn.DiffusionNetBlock(C_width=C_WIDTH, mlp_hidden_dims=[C_WIDTH, C_WIDTH], dropout=False)
    blk.load_state_dict(params, strict=True)
    blk = blk.to(dev).eval()
    xb, mb, eb, vb = x.unsqueeze(0), mass.unsqueeze(0), evals.unsqueeze(0), evecs.unsqueeze(0)

    def step():
        with torch.no_grad():
            return blk(xb, mb, None, eb, vb, [gradX], [gradY])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warm):
        out = step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = lib.dn_kernel_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.time()
    ev0.record()
    for _ in range(steps):
        out = step()
    ev1.record()
    barrier()
    launches = lib.dn_kernel_launch_count() - l0
    t_end = time.time()
    dump = None
    if args.dump_outputs and rank == 0:    # taken before the untimed steps below can touch `out`
        rows = torch.randperm(V, generator=torch.Generator().manual_seed(DUMP_SEED))[:DUMP_ROWS].sort().values
        dump = out[0].index_select(0, rows.to(dev))
    ms_total = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = float(ms_total.item()) / steps
    # the timed region may be shorter than a few nvidia-smi periods: keep the identical load
    # running (untimed) until the sampler has seen it
    while sampler.proc is not None and sampler.count_since(t_begin) < 8 and time.time() - t_begin < 3.0:
        for _ in range(10):
            out = step()
        torch.cuda.synchronize()
        t_end = time.time()
    clocks = sampler.stop(t_begin, t_end)
    value = world * V / (ms_step * 1e-3) / 1e6
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "out.npy"), dump.cpu().numpy())

    # ---- end to end through the public API from pinned host buffers ----
    pin = lambda t: t.contiguous().pin_memory()
    # the operator tuple as the framework's host-side form: fp32 arrays + the shared-pattern int32 CSR of
    # (gradX, gradY) (12 B/nnz; the reference's int64 COO pair is 40 B/nnz).  Everything goes up EVERY step.
    rp_h, ci_h, gv_h = dn.prepare_operators(gradX, gradY).to_host_csr()
    h = {"x": pin(x_host), "mass": pin(host_ops[0]), "evals": pin(host_ops[2]), "evecs": pin(host_ops[3]),
         "rowptr": rp_h, "colidx": ci_h, "gvals": gv_h}
    out_host = torch.empty(V, C_WIDTH).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in h.values())
    d2h = out_host.numel() * 4

    def e2e_fn(x, mass, evals, evecs, rowptr, colidx, gvals):
        gops = dn.ops.GradOperators.from_csr(V, rowptr, colidx, gvals)
        with torch.no_grad():
            return blk(x.unsqueeze(0), mass.unsqueeze(0), None, evals.unsqueeze(0), evecs.unsqueeze(0), [gops], None)[0]

    # public streaming helper: per step the SAME traffic as the reference's loop (features + the whole
    # operator tuple up, result down; nothing cached across steps), with upload(i+1) / kernels(i) /
    # download(i-1) on three streams
    pipe = dn.streaming.StreamedForward(e2e_fn, dev, depth=3)
    out_hosts = [out_host, torch.empty(V, C_WIDTH).pin_memory(), torch.empty(V, C_WIDTH).pin_memory()]
    for _ in range(3):                                  # warm-up: allocator, CSR prep path, host link
        pipe.result(pipe.submit(h, out_hosts[0]))
    barrier()
    main = torch.cuda.current_stream(dev)
    def timed_pipe(pp, hin):
        """median over 3 repeats of `e2e_steps` pipelined steps (host-link throughput on shared boxes is noisy)"""
        reps = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(main)
            lastt = None
            for i in range(args.e2e_steps):
                lastt = pp.submit(hin, out_hosts[i % 3])
            main.wait_event(lastt["fin"])                  # the last result has landed in host memory
            b.record(main)
            pp.drain()
            barrier()
            reps.append(a.elapsed_time(b))
        reps.sort()
        t = torch.tensor([reps[1]], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / args.e2e_steps

    e2e_val = world * V / (timed_pipe(pipe, h) * 1e-3) / 1e6

    # same pipeline with the operator tuple kept resident on the device (SURVEY.md 8f row 2): only the
    # features go up and the result comes down each step -- reported beside e2e, not as e2e
    def res_fn(x):
        with torch.no_grad():
            return blk(x.unsqueeze(0), mb, None, eb, vb, [gradX], [gradY])[0]
    pipe2 = dn.streaming.StreamedForward(res_fn, dev, depth=3)
    for _ in range(2):
        pipe2.result(pipe2.submit({"x": h["x"]}, out_hosts[0]))
    barrier()
    e2e_resident = world * V / (timed_pipe(pipe2, {"x": h["x"]}) * 1e-3) / 1e6

    # ---- per-stage device times (rank 0) from the SAME launch sequence (dn_block_fwd_profile: CUDA events on the
    # launching stream between the stages), and the roofline of every kernel of the step ----
    roof, stages, kernels = None, None, None
    if rank == 0:
        pk = peaks()
        gops = dn.prepare_operators(gradX, gradY)
        A_re, A_im = blk.gradient_features.weights()
        lins = blk.mlp.linears()
        nprof = 10
        acc = [0.0] * len(dn.ops.PROFILE_STAGES)
        import ctypes
        lib.dn_debug_gf_gather_ms.restype = ctypes.c_float
        gather_acc = 0.0
        with torch.no_grad():
            for it in range(nprof + 2):
                prof = []
                dn.ops.block_forward_raw(x, mass, evals, evecs, gops, blk.diffusion.diffusion_time, A_re, A_im,
                                         [l.weight for l in lins], [l.bias for l in lins], True, profile=prof)
                if it >= 2:
                    acc = [a + b for a, b in zip(acc, prof)]
                    gather_acc += float(lib.dn_debug_gf_gather_ms())     # the x-only gather's share of stage [4] (0: old route)
        stages = {n + "_ms": a / nprof for n, a in zip(dn.ops.PROFILE_STAGES, acc)}
        gather_x_ms = gather_acc / nprof

    # ---- the reference beside it (rank 0, N=1 only; bounded samples) ----
    cpu, gpu_base = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        host = (host_ops[0], host_ops[1], host_ops[2], host_ops[3], host_ops[4], host_ops[5], x_host)
        # (a) the same unmodified reference modules with CUDA tensors on THIS GPU: torch eager (cuBLAS fp32 with TF32
        #     off, cuSPARSE) -- the "what a user gets today by calling .cuda()" bar (BASELINE.md section 3)
        try:
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            gstep, gkind = make_baseline_step(host, params, dev)
            for _ in range(3):
                gstep()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(10):
                gstep()
            b.record()
            torch.cuda.synchronize()
            gms = a.elapsed_time(b) / 10
            torch.backends.cuda.matmul.allow_tf32 = prev
            gpu_base = {"value": V / (gms * 1e-3) / 1e6, "unit": "Mverts/s", "ms_per_step": gms, "kind": gkind,
                        "how": "reference DiffusionNetBlock, torch eager on this B200, fp32 (TF32 off), inputs resident, "
                               "10 steps after 3 warm-up",
                        "speedup_ours": gms / ms_step}
            del gstep
            torch.cuda.empty_cache()
        except Exception as exc:                      # a baseline that cannot run must not take the bench line down
            gpu_base = {"unavailable": repr(exc)[:200]}
        # (b) the reference's CPU path on the host cores
        sec, cores, kind, sweep = time_cpu_baseline(host, params, 3, 1)
        cpu = {"value": V / sec / 1e6, "unit": "Mverts/s", "cores": cores, "kind": kind,
               "sample": "same workload (1 mesh V=200000), 3 steps median, 1 warm-up; threads picked by a 1-step "
                         "sweep (seconds per step): {}".format(sweep)}

    if rank == 0:
        # the cuBLAS TF32 peak is measured LAST: a second of back-to-back GEMMs leaves the GPU power-capped for a while
        # (it inflated the stage times by 1.5x when it ran before them)
        tf32 = measure_tf32_peak(dev)
        C, K = C_WIDTH, K_EIG
        nnz = NNZ_ROW * V
        # tensor-pipe work per fp32 product in TF32-pass equivalents: the default tc3x chain issues, per 32-wide K-stage,
        # 4 kind::tf32 MMAs (hi*hi) + 4 kind::f16 bf16 MMAs (K = 16: both correction terms) = 8 MMA slots where plain
        # 3xTF32 needs 12 -> 2 equivalents (DN_TC_HYBRID=0 restores 3); bf16 engine: half a TF32 pass
        hybrid = os.environ.get("DN_TC_HYBRID", "1") != "0"
        passes = {"tc3x": 2.0 if hybrid else 3.0, "tc1x": 1.0, "bf16": 0.5}.get(args.engine, 3.0)
        # algorithmic (minimum) HBM bytes and useful fp32 flops per launch of each kernel (DESIGN.md section 4)
        work = {
            "to_basis": (4 * V * (K + C) + 4 * V, 2 * K * C * V, "to_basis_kernel (split-V tcgen05)"),
            "spectral_scale": (0, 0, "(separate launch only on the SIMT engine; part of pack_weights_kernel here)"),
            "pack_weights": (4 * 148 * K * C + 3 * 4 * (K * C + 2 * C * C + 5 * C * C), 0,
                             "pack_weights_kernel (split-V partial reduction + exp(-lambda t) scale + hi/lo weight pack)"),
            # default route at C = 128 (DN_GF_TC=1): from_basis alone, then the gradient features as an x-only gather
            # (writes [gX|gY]) + two tcgen05 GEMM launches with the inner product / tanh epilogue
            "from_basis_pq": (4 * V * (K + C), 2 * K * C * V, "rows_chain3_kernel (from_basis)"),
            "grad_features_gather": (4 * V * (C + 2 * C) + 12 * nnz + 4 * V + 4 * V * (2 * C + C), (4 * NNZ_ROW * C + 8 * C * C) * V,
                                     "spmm_gxy_blk_kernel (x-only CSR gather) + 2 x rows_chain3_kernel ([gX|gY] W_rot, "
                                     "tanh(gX*Bre+gY*Bim) epilogue)"),
            "mlp": (4 * V * (3 * C + C), 10 * C * C * V, "rows_chain3_kernel (MiniMLP + skip, 3 fused layers)"),
        }
        try:   # per-launch DRAM traffic of each kernel from the committed ncu --set full capture of this command
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as fh:
                traffic = json.load(fh)
        except Exception:
            traffic = {}
        tc_route = gather_x_ms > 0.0      # tensor-core gradient features (default at C = 128): stage [4] is three launches
        if not tc_route:                  # commuted route (DN_GF_TC=0): [P|Q] fused behind from_basis, one gather kernel
            work["from_basis_pq"] = (4 * V * (K + C + 2 * C), (2 * K * C + 4 * C * C) * V,
                                     "rows_chain3_kernel (from_basis -> [P|Q], 2 fused layers)")
            work["grad_features_gather"] = (4 * V * (3 * C + C) + 12 * nnz + 4 * V, 12 * NNZ_ROW * C * V,
                                            "spmm_features_blk_kernel (CSR gather of x, P, Q + inner product + tanh)")
        kernels = []
        names = list(dn.ops.PROFILE_STAGES)
        times = {n: stages[n + "_ms"] for n in names}
        if tc_route:
            i = names.index("grad_features_gather")
            names[i:i + 1] = ["grad_gather_x", "grad_dots_gemm"]
            times["grad_gather_x"] = gather_x_ms
            times["grad_dots_gemm"] = (stages["grad_features_gather_ms"] - gather_x_ms) / 2      # per launch (two launches)
            work["grad_gather_x"] = (4 * V * (C + 2 * C) + 12 * nnz + 4 * V, 4 * NNZ_ROW * C * V,
                                     "spmm_gxy_blk_kernel (x-only CSR gather, writes [gX|gY])")
            # (the epilogue's second read of the 64 gX / gY columns it needs comes out of L2: not counted)
            work["grad_dots_gemm"] = (4 * V * (2 * C + C // 2), 4 * C * C * V,
                                      "rows_chain3_kernel ([gX|gY] W_rot for 64 channels, tanh(gX*Bre+gY*Bim) epilogue; one of 2 launches)")
        for name in names:
            ms = times[name]
            by, fl, kname = work[name]
            ms = max(ms, 1e-6)
            gbs = by / (ms * 1e-3) / 1e9
            tfl = fl / (ms * 1e-3) / 1e12
            t_hbm = by / (pk["hbm_gbs"] * 1e9)
            t_tc = passes * fl / (tf32["tf32_tflops"] * 1e12)
            ent = {"stage": name, "kernel": kname, "ms": ms, "algorithmic_bytes": by, "useful_flops": fl,
                   "achieved_gbs": gbs, "hbm_frac": gbs / pk["hbm_gbs"],
                   "issued_tf32_tflops": passes * tfl, "tf32_frac": passes * tfl / tf32["tf32_tflops"],
                   "bound": "tensor" if t_tc > t_hbm else "hbm", "floor_ms": max(t_tc, t_hbm) * 1e3,
                   "traffic": traffic.get(name)}
            kernels.append(ent)
        dom = max(kernels, key=lambda e: e["ms"])
        if dom["bound"] == "tensor":
            roof = {"bound": "tensor", "achieved": dom["issued_tf32_tflops"], "peak": tf32["tf32_tflops"],
                    "unit": "TFLOP/s", "frac": dom["tf32_frac"],
                    "note": "tensor-pipe work issued, in TF32-pass equivalents (tc3x: TF32 hi*hi + bf16 correction MMAs = 2 "
                            "per fp32 product), over the cuBLAS TF32 GEMM rate measured in this run (burst); useful fp32 "
                            "flops are `achieved` / passes_equiv", "passes_equiv": passes}
        else:
            roof = {"bound": "hbm", "achieved": dom["achieved_gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": dom["hbm_frac"],
                    "note": "algorithmic bytes per launch / CUDA-event time over the measured copy bandwidth"}
        roof.update({"kernel": dom["kernel"], "ms": dom["ms"], "traffic": dom["traffic"],
                     "traffic_source": "profiles/r02_traffic.json (one ncu --set full launch of this command)",
                     "peak_source": pk["source"], "tf32_peak": tf32, "bf16_peak_tflops": pk["bf16_tflops"],
                     "block_hbm_frac": bytes_per_vertex(K_EIG, C) * V / (ms_step * 1e-3) / 1e9 / pk["hbm_gbs"],
                     "block_tf32_frac": passes * (4 * K * C + 14 * C * C) * V / (ms_step * 1e-3) / 1e12 / tf32["tf32_tflops"]})

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "Mverts/s", "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "engine": args.engine,
                       "parallelism": "mesh-sharded x{}".format(world), "l2": "inputs (~330 MB/step) exceed the 126 MB L2",
                       "gflop_per_step": flops_per_vertex(K_EIG, C_WIDTH) * V / 1e9,
                       "min_hbm_mb_per_step": bytes_per_vertex(K_EIG, C_WIDTH) * V / 1e6},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": "Mverts/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": args.e2e_steps, "pipeline": "StreamedForward depth 3 (upload/compute/download streams); operators uploaded every step as fp32 arrays + int32 CSR",
                    "numa_bound_cpus": (len(numa_cpus) if numa_cpus else None),
                    "operators_resident_value": e2e_resident,
                    "operators_resident_h2d_bytes_per_step": int(h["x"].numel() * 4)},
            "roofline": roof, "stages_ms": stages, "kernels": kernels, "cpu_baseline": cpu, "gpu_baseline": gpu_base,
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
