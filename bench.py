#!/usr/bin/env python
"""Benchmark: segments/s of a GraphEncoder forward+backward NT-Xent training step.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's own PyTorch code on the host CPU

Workload (BASELINE.json configs[1]): SimCLR(GraphEncoder(k=3)) on synthetic log-mel segments,
batch 512 pairs per GPU (= 1024 segments per step), fp32, Adam.  One step = zero_grad, both
views forward, NT-Xent, backward, optimizer step.  ``--dtype bf16`` runs configs[2]'s arithmetic
(torch.autocast bf16 activations, fp32 parameters).  Prints ONE JSON line (see DESIGN.md, section
"Measurement", for every key).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "segments/sec GraphEncoder fwd+bwd"
UNIT = "segments/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=512, help="pairs per GPU per step (2 segments each)")
    ap.add_argument("--cpu-batch", type=int, default=8, help="pairs per step of the CPU reference sample")
    ap.add_argument("--dtype", choices=["fp32", "bf16"], default="fp32",
                    help="fp32 = configs[1]; bf16 = torch.autocast(bfloat16) activations with fp32 parameters (configs[2])")
    ap.add_argument("--knn-algo", choices=["auto", "simt", "tc"], default="auto")
    ap.add_argument("--graph", choices=["auto", "on", "off"], default="auto",
                    help="run the step as one CUDA graph (grafp_b200.training.GraphedTrainStep); auto = on; off = eager (DistributedDataParallel at N > 1)")
    ap.add_argument("--cudnn-benchmark", choices=["on", "off"], default="on",
                    help="torch.backends.cudnn.benchmark (cuDNN picks its convolution algorithms by timing) for this arm and the "
                         "reference-eager-on-GPU arm alike; the reference's scripts leave it off: 98.8 -> 96.8 ms per step")
    ap.add_argument("--adam", choices=["foreach", "fused"], default="fused",
                    help="torch.optim.Adam implementation: PyTorch's fused kernel (default) or its foreach form: 98.8 -> 97.6 ms")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the reference-eager-on-this-GPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, run the timed step once more from the starting weights and write what "
                         "it computed to DIR/<name>.npy (float32, rank 0; see dump_outputs)")
    return ap.parse_args()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def dram_traffic():
    """Per-launch DRAM bytes of our kernels from the committed ncu --set full capture (profiles/dram_traffic.json,
    written by scripts/ncu_summary.py), keyed by op name; {} when the file is absent."""
    path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return {}


# ------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# the reference's training step (its own modules from baseline/_ref; the oracle port when that copy is absent)
# ------------------------------------------------------------------------------------------
def reference_model(cfg, device):
    """-> (kind, step_fn(spec_i, spec_j) -> loss tensor).  kind "reference": the unmodified upstream SimCLR / GraphEncoder /
    ntxent_loss; "port": the oracle's restatement of the same algorithm (CPU only)."""
    from oracle import reference_arm as RA
    if RA.available():
        ref = RA.load()
        torch.manual_seed(0)
        model = ref.SimCLR(cfg, ref.GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3)).to(device).train()
        opt = torch.optim.Adam(model.parameters(), lr=cfg["lr"])

        def step(s_i, s_j):
            opt.zero_grad(set_to_none=True)
            _, _, z_i, z_j = model(s_i, s_j)
            loss = ref.ntxent_loss(z_i, z_j, cfg)
            loss.backward()
            opt.step()
            return loss

        return "reference", step
    if device.type != "cpu":
        raise RuntimeError("no staged reference (baseline/_ref): the GPU-eager baseline needs the upstream modules")
    from grafp_b200.encoder.graph_encoder import GraphEncoder
    from grafp_b200.simclr.simclr import SimCLR
    from oracle import grafp_oracle as O
    torch.manual_seed(0)
    shapes_model = SimCLR(cfg, GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3))  # parameter container only
    params = {k: v.detach().clone() for k, v in shapes_model.state_dict().items() if not k.endswith("relative_pos")}
    trainable = [n for n, p in shapes_model.named_parameters() if p.requires_grad]
    for n in trainable:
        params[n].requires_grad_(True)
    opt = torch.optim.Adam([params[n] for n in trainable], lr=cfg["lr"])

    def step(s_i, s_j):
        opt.zero_grad(set_to_none=True)
        _, _, z_i, z_j = O.simclr_forward(params, s_i, s_j, True, k=3)
        loss = O.ntxent_loss(z_i, z_j, cfg["tau"])
        loss.backward()
        opt.step()
        return loss

    return "port", step


def cpu_reference_steps(pairs, steps, warmup, seed=1234):
    """Time `steps` SimCLR training steps of the reference on the CPU (all host threads)."""
    from grafp_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = dict(synth.DEFAULT_CFG)
    cfg["bsz_train"] = pairs
    kind, step = reference_model(cfg, torch.device("cpu"))
    s_i, s_j = synth.synth_spec(pairs, seed)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        step(s_i, s_j).item()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return {"value": 2 * pairs * steps / total, "seconds": total, "cores": cores, "pairs": pairs, "steps": steps,
            "kind": kind}


def gpu_eager_reference(dev, pairs, steps=3, warmup=1, seed=1234):
    """The unmodified reference run eager on this GPU: same step, same inputs, PyTorch-default math, at the largest
    batch <= `pairs` that fits (its (B, N, N) distance matrices and (B, C, N, k) gathers are materialised)."""
    from grafp_b200 import synth
    cfg = dict(synth.DEFAULT_CFG)
    tried = []
    B = pairs
    while B >= 8:
        cfg["bsz_train"] = B
        step = None
        try:
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats(dev)
            kind, step = reference_model(cfg, dev)
            s_i, s_j = (t.to(dev) for t in synth.synth_spec(B, seed))
            for _ in range(warmup):
                step(s_i, s_j)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(s_i, s_j).item()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            return {"value": 2 * B * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps, "pairs_per_gpu": B,
                    "segments_per_step": 2 * B, "steps": steps, "warmup": warmup,
                    "peak_memory_gb": torch.cuda.max_memory_allocated(dev) / 2**30, "kind": kind,
                    "did_not_fit": tried,
                    "what": "unmodified upstream SimCLR(GraphEncoder) + ntxent_loss + Adam from baseline/_ref, PyTorch eager "
                            "on this GPU (cuBLAS bmm, ATen topk / index / index_put_, cuDNN), fp32, PyTorch-default TF32 policy, "
                            f"cudnn.benchmark {'on' if torch.backends.cudnn.benchmark else 'off'} (this arm's setting)"}
        except torch.cuda.OutOfMemoryError:
            tried.append(B)
            del step
            B //= 2
    return {"unavailable": f"out of memory down to {B} pairs", "did_not_fit": tried}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_steps(args.cpu_batch, args.steps, args.warmup)
    what = ("the unmodified upstream modules (baseline/_ref)" if r["kind"] == "reference"
            else "oracle port of the reference (baseline/_ref not staged)")
    sample = (f"{args.steps} steps x {args.cpu_batch} pairs ({2 * args.cpu_batch} segments/step) of the same SimCLR training step, "
              f"{what} on {r['cores']} host threads")
    cfg = workload_config(args, 1)
    # this arm's step is a bounded sample: say so where the config is read, not only in the sample string
    cfg.update({"pairs_per_gpu": args.cpu_batch, "segments_per_step": 2 * args.cpu_batch,
                "sample": f"bounded CPU sample of that workload: the same training step at {args.cpu_batch} pairs per step "
                          f"instead of {args.batch} (a 512-pair step of the reference takes minutes on the host cores)"})
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    if args.dtype == "bf16":
        name = ("configs[2] arithmetic: GraphEncoder fwd+bwd NT-Xent training step, batch 512 pairs/GPU, "
                "torch.autocast(bfloat16) activations, fp32 parameters")
    else:
        name = "configs[1]: GraphEncoder fwd+bwd NT-Xent training step, batch 512 pairs/GPU, fp32"
    return {"workload": name,
            "pairs_per_gpu": args.batch, "segments_per_step": 2 * args.batch * world, "k": 3, "nodes": 1024,
            "encoder": "GraphEncoder size t (12 Grapher+FFN blocks)", "optimizer": "Adam",
            "parallelism": f"dp{world}", "cudnn_benchmark": args.cudnn_benchmark == "on", "adam": args.adam,
            "conv_math": "PyTorch default (cuDNN conv TF32 allowed, matmul fp32)"
            if args.dtype == "fp32" else "cuDNN bf16 convolutions under autocast",
            "l2": "no explicit flush: one step touches ~70 GB of activations, far above the 126 MB L2"}


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def algorithmic_work(name, m):
    """Algorithmic bytes / flops of one C-ABI call (SURVEY.md section 8d), fp32 (e = 4) or bf16 (e = 2)."""
    e = 4 if m.get("dtype", 0) == 0 else 2
    if name == "conv1x1_bn_stats_fwd":  # read the input rows and the weight, write the output rows (moments: 16 bytes / channel)
        B, N, Cin, Cout = m["B"], m["N"], m["Cin"], m["Cout"]
        G = m.get("groups", 1)
        return {"flops": 2.0 * B * N * Cin * Cout / G, "bytes": B * N * (Cin + Cout) * e + Cin * Cout * e // G}
    B, N, C = m["B"], m["N"], m["C"]
    if name == "knn_fwd":
        M, K = m["M"], m["K"]
        return {"flops": 2.0 * B * N * M * C, "bytes": B * (N * C * e + (M * C * e if M != N else 0) + N * K * 12)}
    if name == "bn_train_fwd":  # statistics pass + apply pass (+ residual read)
        return {"bytes": B * N * C * e * (3 + m.get("res", 0))}
    if name == "bn_apply_fwd":  # apply pass only: the moments came out of the convolution's epilogue
        return {"bytes": B * N * C * e * (2 + m.get("res", 0))}
    if name == "bn_train_bwd":  # reduction pass (dy, x) + apply pass (dy, x -> dx)
        return {"bytes": B * N * C * e * 5}
    if name in ("ntxent_fwd", "ntxent_bwd"):
        return {"flops": (2.0 if name == "ntxent_fwd" else 4.0) * m["N"] * m["N"] * m["C"], "bytes": 0}
    if "k" not in m:
        return {"bytes": 0}
    k = m["k"]
    idx_b = 8 if m.get("i64") else 4
    if name == "mr_aggregate_fwd":
        return {"bytes": B * (N * C * e + N * k * idx_b + 2 * N * C * e + (N * C if m.get("argmax") else 0))}
    if name == "mr_aggregate_bwd":
        return {"bytes": B * (2 * N * C * e + N * C + N * k * idx_b + N * C * e)}
    return {"bytes": 0}


_ROOFLINE_NAMES = {
    "knn_fwd": "K1 dilated k-NN graph (normalise + tcgen05 Gram / top-k)",
    "mr_aggregate_fwd": "K2 gather + max-relative + interleave",
    "mr_aggregate_bwd": "K3 argmax-routed scatter backward",
    "bn_train_fwd": "K5 train-mode BatchNorm (+ReLU / +residual) forward",
    "bn_train_bwd": "K5 backward",
    "bn_apply_fwd": "K5 forward, apply pass only (statistics from the convolution's epilogue)",
    "conv1x1_bn_stats_fwd": "1x1 convolution as tcgen05 GEMM (TF32 / bf16) with BatchNorm statistics in the epilogue",
}


def roofline_entry(name, kt, pk, ops, traffic):
    if name == "knn_fwd":
        tc = ops.knn_last_algo() == "tcgen05"
        f16 = ops.knn_last_variant() == "f16x3"
        # kind::f16 issues at the bf16 rate, kind::tf32 at half of it
        peak = pk["bf16_tflops_sustained"] / (1.0 if f16 else 2.0)
        ach = kt["tflops"]
        return {"kernel": f"{_ROOFLINE_NAMES[name]} [{ops.knn_last_algo()} {ops.knn_last_variant()}]",
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": ach / peak if ach else None, "issued_frac": 3 * ach / peak if (ach and f16) else None,
                "traffic": traffic.get(name), "ms_per_step": kt["ms_per_step"],
                "peak_source": f"{pk['source']} bf16 sustained" + ("" if f16 else " / 2 (TF32)"),
                "note": "achieved = algorithmic 2*N*M*C flops / time of the whole op (normalise launch included); the "
                        "fp16 hi/lo split issues 3 MMAs per algorithmic one (issued_frac); ncu tensor-pipe % per stage "
                        "is in profiles/" if tc else "CUDA-core fp32 path, reported against the tensor peak"}
    peak = pk["hbm_gbs"]
    return {"kernel": _ROOFLINE_NAMES.get(name, name), "bound": "hbm", "achieved": kt["gbs"], "peak": peak, "unit": "GB/s",
            "frac": kt["gbs"] / peak if kt["gbs"] else None, "traffic": traffic.get(name),
            "ms_per_step": kt["ms_per_step"], "peak_source": pk["source"]}


DUMP_ROWS = 1024          # rows of h / z kept by --dump-outputs (all of them at the default batch)
DUMP_PARAM_SAMPLE = 1 << 22


def dump_outputs(out_dir, loss, outputs, model):
    """The results of one training step as DIR/<name>.npy, float32, 25 MiB at most: ``loss``; ``h_i``, ``h_j``,
    ``z_i``, ``z_j`` (the encoder outputs and embeddings of both views, a seeded sample of DUMP_ROWS rows above that
    batch); ``grads``: a fixed seeded sample of DUMP_PARAM_SAMPLE of the 18.4 M trainable entries' gradients
    (concatenated in named_parameters order).  The updated parameters are left out: where a gradient is analytically
    zero (biases in front of a train-mode BatchNorm) Adam turns its rounding noise into a +-lr step of either sign."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": np.array(loss, dtype=np.float32)}
    for name, t in zip(("h_i", "h_j", "z_i", "z_j"), outputs):
        t = t.detach()
        if t.shape[0] > DUMP_ROWS:
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(1))[:DUMP_ROWS].sort().values
            t = t[rows.to(t.device)]
        arrays[name] = t.float().cpu().numpy()
    params = [p for p in model.parameters() if p.requires_grad]
    flat_g = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1) for p in params])
    pick = torch.randperm(flat_g.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_PARAM_SAMPLE].sort().values
    arrays["grads"] = flat_g[pick.to(flat_g.device)].float().cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    from grafp_b200 import _native, ops, synth
    from grafp_b200.encoder.graph_encoder import GraphEncoder
    from grafp_b200.simclr.simclr import SimCLR
    from grafp_b200.simclr.distributed import global_ntxent_loss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    _native.load()

    cfg = dict(synth.DEFAULT_CFG)
    cfg["bsz_train"] = args.batch
    torch.manual_seed(0)
    model = SimCLR(cfg, GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3)).to(dev).train()
    start = {k: v.clone() for k, v in model.state_dict().items()} if args.dump_outputs else None
    net = model
    # whole step incl. the gradient all-reduce as one CUDA graph per rank (GRAFP_BENCH_DP_GRAPH=0: DistributedDataParallel, eager)
    graph_dp = world > 1 and (args.graph == "on" or (args.graph == "auto" and os.environ.get("GRAFP_BENCH_DP_GRAPH", "1") != "0"))
    if world > 1 and not graph_dp:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], broadcast_buffers=True,
                                                        gradient_as_bucket_view=True)
    # auto = graph.  The step is ~6 000 launches; with the kernels at ~97 ms the host's launch rate (~94 ms of CPU per step,
    # more with 8 processes sharing the host) is the bound in eager mode: fp32 101.7 -> 99.1 ms at one GPU, 101.2 -> 97.2 ms
    # at two (profiles/r03*), bf16 75.5 -> 70.8 ms.  DistributedDataParallel's reducer cannot be captured (it touches the
    # legacy stream: cudaErrorStreamCaptureImplicit), so the multi-GPU graph replaces it by one captured all-reduce of a flat
    # gradient buffer (grafp_b200.training.FlatGradients).
    use_graph = graph_dp or (world == 1 and args.graph in ("on", "auto"))
    torch.backends.cudnn.benchmark = args.cudnn_benchmark == "on"
    opt = torch.optim.Adam(model.parameters(), lr=cfg["lr"], capturable=use_graph, fused=(args.adam == "fused") or None)
    algo = {"auto": _native.KNN_AUTO, "simt": _native.KNN_SIMT, "tc": _native.KNN_TC}[args.knn_algo]
    if algo != _native.KNN_AUTO:
        _orig = ops.knn_graph
        ops.knn_graph = lambda *a, **kw: _orig(*a, **{**kw, "algo": algo})
    bf16 = args.dtype == "bf16"

    s_i, s_j = synth.synth_spec(args.batch, 1234 + rank)
    host_i, host_j = s_i.pin_memory(), s_j.pin_memory()
    dev_i, dev_j = host_i.to(dev), host_j.to(dev)
    h2d_bytes = host_i.numel() * 4 + host_j.numel() * 4

    last_outputs = []

    def loss_of(h_i, h_j, z_i, z_j):
        if args.dump_outputs:   # under a CUDA graph these are its static outputs, refreshed by every replay
            last_outputs[:] = [h_i, h_j, z_i, z_j]
        # global-batch negatives like the reference's DataParallel gather (train.py:69-71); the loss runs in fp32
        return global_ntxent_loss(z_i.float(), z_j.float(), cfg)

    def eager_step(x_i, x_j):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            out = net(x_i, x_j)
        loss = loss_of(*out)
        loss.backward()
        opt.step()
        return loss

    step = eager_step
    if use_graph:
        # the whole step - both views forward, loss, backward, Adam - as ONE CUDA graph; new inputs are copied into
        # its static buffers (from pinned host memory in the e2e region)
        from grafp_b200.training import GraphedTrainStep
        try:
            step = GraphedTrainStep(net, opt, loss_of, [dev_i, dev_j], autocast_dtype=torch.bfloat16 if bf16 else None,
                                    data_parallel=graph_dp)
            captured = 1
        except Exception as exc:  # a capture that fails must not cost the bench line (nor hang the other ranks)
            print(f"bench.py: CUDA-graph capture failed on rank {rank} ({type(exc).__name__}: {exc}); running eagerly",
                  file=sys.stderr, flush=True)
            captured = 0
        if world > 1:   # nothing of a capture executes, so every rank gets here: agree on one form
            flag = torch.tensor([captured], device=dev, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            captured = int(flag.item())
        if not captured:
            use_graph = graph_dp = False
            step = eager_step
            if world > 1:
                net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], broadcast_buffers=True,
                                                                gradient_as_bucket_view=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(dev_i, dev_j)
    barrier()

    # ---- timed region 1: inputs resident in HBM (the `value`) ----
    timer = ops.KernelTimer(timing=not use_graph)   # (events cannot be recorded inside a replayed graph: see below)
    if not use_graph:
        ops.set_timer(timer)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step(dev_i, dev_j)
    e1.record()
    barrier()
    ms_resident = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    ops.set_timer(None)
    n_instr = args.steps

    # ---- timed region 2: end to end through the public API with host buffers (the `e2e`) ----
    losses = []
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        if use_graph:   # H2D straight into the graph's static input buffers, replay, read the loss back
            losses.append(step(host_i, host_j).item())
        else:
            x_i = host_i.to(dev, non_blocking=True)
            x_j = host_j.to(dev, non_blocking=True)
            losses.append(step(x_i, x_j).item())  # .item(): device -> host read of the step's result
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    if args.dump_outputs:
        # The state after the warmup and timed steps carries their rounding noise (unordered fp32 reductions, cuDNN's
        # timed algorithm choice), which Adam and the k-NN's near-ties amplify from step to step; so the dumped step is
        # the timed one (same graph or eager step, same inputs) run again from the starting weights and a fresh Adam state.
        with torch.no_grad():
            for k, v in model.state_dict().items():
                v.copy_(start[k])
            for state in opt.state.values():
                for t in state.values():
                    if torch.is_tensor(t):
                        t.zero_()
        loss = step(host_i, host_j) if use_graph else step(host_i.to(dev), host_j.to(dev))
        barrier()
        if rank == 0:
            dump_outputs(args.dump_outputs, loss.item(), last_outputs, model)

    ms_instr = ms_resident
    if use_graph:
        # per-kernel breakdown: the same step run eagerly (same kernels, same order) with CUDA events around every C-ABI
        # call; NOT part of `value` / `e2e`
        n_instr = min(3, args.steps)
        ops.set_timer(timer)
        timer.timing = True
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e4.record()
        for _ in range(n_instr):
            step._eager_step()
        e5.record()
        torch.cuda.synchronize()
        ops.set_timer(None)
        ms_instr = e4.elapsed_time(e5)
    ksum = timer.summary()

    t = torch.tensor([ms_resident, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_resident, ms_e2e = float(t[0]), float(t[1])
    segs = 2 * args.batch * world * args.steps
    value = segs / (ms_resident / 1e3)
    e2e_value = segs / (ms_e2e / 1e3)

    if rank == 0:
        pk = peaks()
        traffic = dram_traffic()
        kernels = {}
        for name, rec in ksum.items():
            work = {"bytes": 0.0, "flops": 0.0}
            for key, sh in rec["by_shape"].items():
                w = algorithmic_work(name, dict(key))
                work["bytes"] += w.get("bytes", 0.0) * sh["calls"]
                work["flops"] += w.get("flops", 0.0) * sh["calls"]
            sec = rec["ms_total"] / 1e3
            kernels[name] = {"calls_per_step": rec["calls"] / n_instr, "ms_total": rec["ms_total"],
                             "ms_per_step": rec["ms_total"] / n_instr,
                             "share_of_step": rec["ms_total"] / n_instr / (ms_resident / args.steps),
                             "gbs": work["bytes"] / sec / 1e9 if sec > 0 and work["bytes"] else None,
                             "tflops": work["flops"] / sec / 1e12 if sec > 0 and work["flops"] else None}
        # `roofline`: the costliest of our kernels (the contract's "dominant kernel"); `rooflines`: every hot-path kernel,
        # K1 against the tensor peak, K2 / K3 / K5 against the HBM peak
        roofline = None
        rooflines = [roofline_entry(n, kernels[n], pk, ops, traffic) for n in _ROOFLINE_NAMES if n in kernels]
        if kernels:
            top = max((n for n in kernels if n in _ROOFLINE_NAMES), key=lambda n: kernels[n]["ms_total"], default=None)
            if top is not None:
                roofline = roofline_entry(top, kernels[top], pk, ops, traffic)

        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_resident / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if not bf16 else "bf16", "data": "synthetic", "config": workload_config(args, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
            "gpu_launches": int(round(timer.launches / n_instr * args.steps)), "knn_algo": ops.knn_last_algo(),
            "cuda_graph": bool(use_graph),
            "kernel_timing": ("CUDA events around every C-ABI call of %d eagerly run steps (%.1f ms per step eager; the timed "
                              "steps replay the same kernels as one CUDA graph)" % (n_instr, ms_instr / n_instr)) if use_graph
                             else "CUDA events around every C-ABI call inside the timed region",
            "roofline": roofline, "rooflines": rooflines, "kernels": kernels, "clocks": clocks,
            "loss_last": losses[-1] if losses else None, "pairs_per_s": value / 2,
        }
        # ---- baselines (rank 0, one GPU only): the reference eager on this GPU, then on the host cores ----
        if world == 1:
            del step, opt, net, model
            torch.cuda.empty_cache()
            if not args.no_gpu_eager:
                try:
                    g = gpu_eager_reference(dev, args.batch)
                except Exception as exc:  # a missing baseline/_ref must not cost the bench line
                    g = {"unavailable": f"{type(exc).__name__}: {exc}"}
                if "value" in g:
                    g["speedup_resident"] = value / g["value"]
                    g["speedup_e2e"] = e2e_value / g["value"]
                line["gpu_eager_baseline"] = g
            if not args.no_cpu_baseline:
                r = cpu_reference_steps(args.cpu_batch, 3, 1)
                line["cpu_baseline"] = {
                    "value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                    "sample": f"3 steps x {args.cpu_batch} pairs of the same SimCLR training step ("
                              + ("the unmodified upstream modules from baseline/_ref" if r["kind"] == "reference"
                                 else "oracle port of the reference algorithm")
                              + f"), {r['seconds']:.1f} s on {r['cores']} host threads"}
        line.setdefault("cpu_baseline", None)
        print(json.dumps(line), flush=True)
    if world > 1:
        if graph_dp:
            # The CUDA graph holds captured NCCL kernels; tearing the communicator down under it hung the process at
            # exit (measured: the JSON line printed, then torchrun's children never returned).  Everything is flushed
            # and every rank is past the last collective: leave without the NCCL teardown.
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
