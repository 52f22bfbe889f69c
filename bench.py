#!/usr/bin/env python
"""Headline benchmark: Apertis SSM+MoE block forward+backward tokens/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (ApertisLayer = pre-norm + SelectiveLinearAttention + residual,
pre-norm + AdaptiveExpertSystem + residual; forward, synthetic loss of SURVEY.md 8(d), backward) over one
batch of synthetic tokens.  Workload = BASELINE.json configs[1]: the 1.5B text-only Apertis block
(hidden 704, 11 heads, d_inner 176, intermediate 2816, 8 experts top-2), seq 4096, bf16 autocast over fp32
master weights (the only low-precision mode the reference supports, SURVEY.md facts table).

N > 1 (torchrun, one rank per GPU): experts sharded E/N per rank with NCCL all-to-all dispatch/combine, every
rank keeps its own batch (weak scaling), replicated-parameter gradients all-reduced as DDP would.

--impl reference times the reference's algorithm on the host CPU: the oracle port (oracle/apertis_oracle.py,
same ATen op sequence as core.py) with all host threads, on a bounded sample of the same workload, for --steps steps
after --warmup warm-up steps.

--dump-outputs DIR writes what the last timed step of the headline workload computed (rank 0) as DIR/<name>.npy in
float32: the block output `out`, the aux losses `lb` and `rz`, `loss`, the input gradient `dx` and `grad.<parameter>`
for every parameter.  A tensor of more than DUMP_SAMPLE elements is stored as the values at DUMP_SAMPLE sorted indices
drawn with a fixed seed.  Weights, inputs, routing noise and dropout masks come from seeded generators: the same
arguments give the same inputs in every run, so two builds can be compared output for output.  With N > 1 the
gradients are rank 0's own, before the all-reduce of the replicated parameters (which the bench does into a separate
buffer, not into .grad).  The outputs of the captured graph replayed last are kept alive for the dump, so later captures
cannot reuse that memory: the work is the same, but the time of a dumping run is not strictly the time of a plain run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the source tree may be read-only: nothing is cached next to it

WORKLOADS = {
    # name: (Dm, H, I, E, K, seq)      shapes from SURVEY.md section 8 / BASELINE.md section 3
    "c1_125m": (256, 4, 1024, 8, 2, 1024),
    "c2_1p5b": (704, 11, 2816, 8, 2, 4096),
    "c4_7b": (1600, 25, 6400, 8, 2, 4096),
}
METRIC = "SSM+MoE block fwd+bwd tokens/sec"
DUMP_SAMPLE = 1 << 20               # elements kept of one dumped tensor (4 MB in float32)
DUMP_LIMIT = 64 << 20               # bytes of all dumped files together


def dump_outputs(outputs, path):
    """Writes {name: tensor} as path/<name>.npy (float32); larger tensors as a seeded sample of DUMP_SAMPLE elements."""
    arrays, total = {}, 0
    for name, t in outputs.items():
        t = torch.as_tensor(t).detach()
        flat = t.float().reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(0)
            idx = torch.randint(0, flat.numel(), (DUMP_SAMPLE,), generator=g).sort().values
            flat = flat[idx.to(flat.device)]
            a = flat.cpu().numpy()
        else:
            a = flat.cpu().numpy().reshape(tuple(t.shape))
        arrays[name] = a
        total += a.nbytes
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled WHILE the timed region runs: NVML polled from a thread every ~2 ms
    (nvidia-smi's fastest loop is too coarse for a region of tens of milliseconds); nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.mx, self.reasons = [], [], set()
        self.stop = threading.Event()
        self.thread = None
        self.p = None
        self.f = None
        self.source = None

    def _nvml_loop(self, nv, h):
        try:
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
        except Exception:
            pass
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(h))
                for bit, name in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop.wait(0.002)

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else self.idx
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            self.source = "nvml"
            return self
        except Exception:
            self.thread = None
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
            self.source = "nvidia-smi"
        except Exception:
            self.p = None
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()

    def summary(self):
        sm, mx, reasons = list(self.sm), list(self.mx), set(self.reasons)
        if self.f is not None:
            try:
                self.f.flush()
                for line in open(self.f.name):
                    c = [t.strip() for t in line.split(",")]
                    if len(c) < 8:
                        continue
                    try:
                        sm.append(float(c[1])); mx.append(float(c[2]))
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
                os.unlink(self.f.name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "source": self.source}


class _MeanSquare(torch.autograd.Function):
    """mean(out.float()^2) of SURVEY.md 8(d) with one reduction forward and one multiply backward (torch's
    pow + mean pair costs five full passes over the activations, which is harness overhead, not block work)."""

    @staticmethod
    def forward(ctx, out):
        ctx.save_for_backward(out)
        n = torch.linalg.vector_norm(out, 2, dtype=torch.float32)
        return n * n / out.numel()

    @staticmethod
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        return out * (g * (2.0 / out.numel())).to(out.dtype)


def _reference_layer(wl, dropout, device):
    """The UNMODIFIED reference ApertisLayer (baseline/_ref, installed by __graft_entry__.build()) with seeded weights of
    the reference initialiser's distributions; None when the install is absent."""
    from baseline import ref_loader
    if not ref_loader.available():
        return None
    from oracle import apertis_oracle as O
    core = ref_loader.load_core()
    Dm, H, I, E, K, seq = wl
    cfg = core.ApertisConfig(hidden_size=Dm, num_attention_heads=H, intermediate_size=I, num_hidden_layers=1,
                             attention_type="selective_ssm", use_expert_system=True, num_experts=E, experts_per_token=K,
                             vocab_size=1000, hidden_dropout_prob=dropout)
    layer = core.ApertisLayer(cfg)
    layer.load_state_dict(O.make_layer_params(Dm, H, I, E, seed=0, perturb=False), strict=True)
    return layer.to(device).train()


def reference_time(wl, Bsz, L, dropout, device, steps, warmup, autocast=None, best_of=False):
    """tokens/s of the reference block (fwd + SURVEY 8(d) loss + bwd) on `device`; falls back to the oracle port on the CPU
    when baseline/_ref is absent.  -> (tokens/s, ms per step, kind)"""
    Dm, H, I, E, K, seq = wl
    layer = _reference_layer(wl, dropout, device)
    kind = "reference"
    g = torch.Generator().manual_seed(0)
    x = torch.randn(Bsz, L, Dm, generator=g).to(device).requires_grad_(True)
    if layer is not None:
        params = list(layer.parameters())

        def step():
            for p in params:
                p.grad = None
            x.grad = None
            with torch.autocast(device.type, dtype=autocast, enabled=autocast is not None):
                out, _, _, lb, rz = layer(x)
            (out.float().pow(2).mean() + lb + rz).backward()
    else:
        from oracle import apertis_oracle as O
        assert device.type == "cpu", "the oracle port is a CPU restatement"
        kind = "port"
        sd = {k: v.requires_grad_(True) for k, v in O.make_layer_params(Dm, H, I, E, seed=0).items()}
        _, noise = O.make_inputs(Bsz, L, Dm, E, seed=0)

        def step():
            for p in sd.values():
                p.grad = None
            x.grad = None
            out, lb, rz = O.block_forward(sd, x, num_heads=H, E=E, K=K, training=True, noise=noise)
            O.block_loss(out, lb, rz).backward()

    sync = (lambda: torch.cuda.synchronize(device)) if device.type == "cuda" else (lambda: None)
    for _ in range(warmup):
        step()
    sync()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        sync()
        times.append(time.perf_counter() - t0)
    dt = min(times) if best_of else sum(times) / len(times)
    return Bsz * L / dt, dt * 1e3, kind


def cpu_reference_arm(args, wl, steps, warmup, sample_tokens):
    """The reference block on the host cores (all threads, fp32) on a bounded sample of the bench workload."""
    Dm, H, I, E, K, seq = wl
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    L = min(seq, sample_tokens)
    Bsz = max(1, sample_tokens // L)
    v, ms, kind = reference_time(wl, Bsz, L, args.dropout, torch.device("cpu"), steps, warmup)
    sample = (f"{Bsz}x{L} tokens per step of the same workload, fp32, hidden_dropout_prob {args.dropout}, {steps} steps after {warmup} warm-up, "
              f"torch {torch.__version__} CPU ops, " + ("unmodified reference ApertisLayer (baseline/_ref)" if kind == "reference" else "oracle port"))
    return v, ms, cores, sample, kind


def c1_cpu_points(steps=3):
    """BASELINE.md section 4's mandated CPU point: C1 (125M dims) at B 4 x L 1024, dropout 0.1 and 0.0, best of `steps`."""
    out = {}
    for p in (0.1, 0.0):
        v, ms, kind = reference_time(WORKLOADS["c1_125m"], 4, 1024, p, torch.device("cpu"), steps, 1, best_of=True)
        out[f"dropout_{p}"] = {"tokens_per_s": v, "ms_per_step": ms, "kind": kind}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2_1p5b", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=8, help="sequences per GPU per step")
    ap.add_argument("--dropout", type=float, default=0.1, help="hidden_dropout_prob (reference default 0.1; parity tests use 0)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--cpu-sample-tokens", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--c4-batch", type=int, default=4, help="sequences per GPU per step of the additional configs[3] measurement")
    ap.add_argument("--no-c4", action="store_true", help="skip the additional configs[3] (7B-class) measurement")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip timing the unmodified reference on the GPU")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step as a CUDA graph (auto: use it when capture and a replay check succeed)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs is not None:
        ap.error("--dump-outputs writes what the B200 path computed; it does not apply to --impl reference")
    wl = WORKLOADS[args.workload]
    Dm, H, I, E, K, seq = wl
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg_common = {"workload": f"{args.workload}: Apertis block hidden {Dm}, heads {H}, d_inner {16 * H}, intermediate {I}, "
                              f"{E} experts top-{K}, seq {seq}", "tokens_per_step_per_gpu": args.batch * seq}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = args.steps, args.warmup
        v, ms, cores, sample, kind = cpu_reference_arm(args, wl, steps, warmup, args.cpu_sample_tokens)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(cfg_common, tokens_per_step_per_gpu=None, sample=sample, hidden_dropout_prob=args.dropout),
                "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": cores, "kind": kind, "sample": sample},
                "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        try:
            line["c1_cpu_points"] = c1_cpu_points()
        except Exception as ex:
            line["c1_cpu_points"] = {"error": repr(ex)[:200]}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout to the single JSON line
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ep_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        ep_group = dist.group.WORLD
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torchrun"
    ctx = dict(dev=dev, world=world, rank=rank, local_rank=local_rank, ep_group=ep_group, args=args)

    # headline: BASELINE.json configs[1] (the configuration the metric is quoted on) at every N, so the driver's
    # scaling series compares like with like
    head = measure(args.workload, args.batch, ctx, clocks=True, dump_dir=args.dump_outputs)
    # configs[3] (7B-class, 8 experts top-2, experts sharded over the ranks) measured in the same run at every N
    extra = {}
    if not args.no_c4 and args.workload != "c4_7b":
        try:
            extra["c4_7b"] = measure("c4_7b", args.c4_batch, ctx, clocks=False)
        except Exception as ex:
            extra["c4_7b"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
    ep_check = None
    if world > 1:
        try:
            ep_check = ep_parity_check(ctx, "c4_7b")
        except Exception as ex:
            ep_check = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}

    def shutdown():
        """Multi-GPU exit without the collective teardown: the captured graphs hold NCCL work and the ranks leave at
        different times (rank 0 still runs the CPU baseline), so destroy_process_group() can block; every timed and
        reduced number is final before this point."""
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            torch.cuda.synchronize()
            os._exit(0)

    if rank != 0:
        shutdown()
        return

    pk, pk_src = peaks()
    amp = args.dtype == "bf16"
    Dm, H, I, E, K, seq = WORKLOADS[args.workload]
    tokens_per_step = args.batch * seq
    out = summarise(args.workload, args.batch, head, world, pk, pk_src, amp)
    out = dict({"metric": METRIC, "value": out.pop("value"), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": out.pop("ms_per_step"), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": dict(cfg_common, global_batch_tokens=tokens_per_step * world, hidden_dropout_prob=args.dropout,
                               parallelism=("single GPU" if world == 1 else f"ep{world} (experts sharded, all-to-all) + dp{world}"),
                               precision="bf16 autocast over fp32 master weights" if amp else "fp32 (3x bf16-split tensor-core GEMMs)",
                               l2="inputs rotate over 4 buffers (%.0f MB > 126 MB L2); per-step activations ~GBs" % (4 * tokens_per_step * Dm * 4 / 1e6)),
                "clocks": head["clocks"]}, **out)
    if world == 1:
        try:        # the long-context point of the scan sweep, next to the scan inside the block
            out["kernels"]["selective_scan_L64K"] = scan_long_context(pk["hbm_gbs"])
        except Exception as e:      # never lose the bench line over the extra measurement
            out["kernels"]["selective_scan_L64K"] = {"error": repr(e)[:200]}
    for name, m in extra.items():
        if "error" in m:
            out.setdefault("workloads", {})[name] = m
        else:
            w = summarise(name, args.c4_batch, m, world, pk, pk_src, amp)
            w["config"] = {"workload": workload_text(name), "tokens_per_step_per_gpu": args.c4_batch * WORKLOADS[name][5],
                           "hidden_dropout_prob": args.dropout}
            out.setdefault("workloads", {})[name] = w
    if ep_check is not None:
        out["ep_parity"] = ep_check
        out["ep_parity_rel_err"] = ep_check.get("max_rel_err")
    if world == 1 and not args.no_gpu_reference:
        try:
            out["gpu_reference"] = gpu_reference_leg(args, dev)
        except Exception as ex:
            out["gpu_reference"] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
    if not args.no_cpu_baseline:
        v, cms, cores, sample, kind = cpu_reference_arm(args, wl, 3, 1, args.cpu_sample_tokens)
        out["cpu_baseline"] = {"value": v, "unit": "tokens/s", "cores": cores, "kind": kind, "sample": sample, "ms_per_step": cms}
    print(json.dumps(out))
    shutdown()


def workload_text(name):
    Dm, H, I, E, K, seq = WORKLOADS[name]
    return f"{name}: Apertis block hidden {Dm}, heads {H}, d_inner {16 * H}, intermediate {I}, {E} experts top-{K}, seq {seq}"


TIMED = ["ab_grouped_gemm_nt", "ab_grouped_gemm_nn", "ab_grouped_gemm_tn", "ab_ep_grouped_gemm_nt", "ab_ep_grouped_gemm_nn",
         "ab_ssm_scan_fwd", "ab_ssm_scan_bwd",
         "ab_dense_gemm_nt", "ab_dense_gemm_nn", "ab_dense_gemm_tn"]


def build_layer(name, ctx, dropout, ep=True):
    from apertis_llm_b200 import ApertisLayerB200, BlockConfig
    from oracle import apertis_oracle as O   # only the deterministic parameter factory (reference initialiser's distributions)
    Dm, H, I, E, K, seq = WORKLOADS[name]
    cfg = BlockConfig(hidden_size=Dm, num_attention_heads=H, intermediate_size=I, num_experts=E, experts_per_token=K,
                      hidden_dropout_prob=dropout)
    layer = ApertisLayerB200(cfg, ep_group=ctx["ep_group"] if ep else None)
    layer.load_state_dict(O.make_layer_params(Dm, H, I, E, seed=0, perturb=False), strict=True)
    return layer.to(ctx["dev"]).train()


def measure(name, B, ctx, clocks, dump_dir=None):
    """One workload on this rank's GPU: device-timed steps (CUDA graph replay when it captures), per-kernel times from an
    eager pass, and the end-to-end loop with host inputs.  Times are the maximum over the ranks.  With `dump_dir`, what
    the last timed step computed is written there (dump_outputs) before anything else runs."""
    import torch.distributed as dist
    from apertis_llm_b200 import _lib
    args, dev, world, rank = ctx["args"], ctx["dev"], ctx["world"], ctx["rank"]
    Dm, H, I, E, K, seq = WORKLOADS[name]
    layer = build_layer(name, ctx, args.dropout)
    replicated = [p for n, p in layer.named_parameters() if ".expert_" not in n]
    nbuf = 4
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)
    host_x = [torch.randn(B, seq, Dm, generator=gen).pin_memory() for _ in range(nbuf)]
    dev_x = [h.to(dev, non_blocking=True).requires_grad_(True) for h in host_x]
    amp = args.dtype == "bf16"
    flat_grad = torch.zeros(sum(p.numel() for p in replicated), device=dev) if world > 1 else None
    torch.manual_seed(4321 + rank)          # routing noise and dropout masks: the same draws in every run

    def step(x, keep=None):
        """keep: a dict that receives what the step hands its caller (detached: no autograd graph is held)."""
        for p in layer.parameters():
            p.grad = None
        x.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out, _, _, lb, rz = layer(x)
        loss = _MeanSquare.apply(out) + lb + rz           # SURVEY 8(d): mean(out^2) + lb + rz
        loss.backward()
        if world > 1:                                   # DDP-equivalent: one bucket of the replicated parameters' gradients
            torch._foreach_copy_(list(flat_grad.split([p.numel() for p in replicated])), [p.grad.reshape(-1) for p in replicated])
            dist.all_reduce(flat_grad)
        if keep is not None:
            keep.update(out=out.detach(), lb=lb.detach(), rz=rz.detach(), loss=loss.detach(), dx=x.grad)
            keep.update({"grad." + n: p.grad for n, p in layer.named_parameters() if p.grad is not None})
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(max(3, args.warmup)):
        step(dev_x[i % nbuf])
    barrier()

    # ---- optional: the whole step (forward, loss, backward, gradient all-reduce) captured once per input buffer as a CUDA
    #      graph and replayed, which removes the host launch path from the step
    graphs, graph_note = None, "off"
    if args.graph != "off":
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(2):
                    step(dev_x[i % nbuf])
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            pool = None
            graphs = []
            for i in range(nbuf):
                g = torch.cuda.CUDAGraph()
                # the graph replayed last keeps what its capture returned (a replay rewrites those tensors)
                keep = {} if dump_dir is not None and i == (args.steps - 1) % nbuf else None
                with torch.cuda.graph(g, pool=pool):
                    gl = step(dev_x[i], keep)
                pool = g.pool()
                graphs.append((g, gl, keep))
            barrier()
            eager = float(step(dev_x[0]).detach())
            graphs[0][0].replay()
            replayed = float(graphs[0][1].detach())
            if not (replayed == replayed and abs(replayed - eager) <= 0.05 * abs(eager)):
                raise RuntimeError(f"graph replay loss {replayed} vs eager {eager}")
            graph_note = "on"
        except Exception as ex:            # capture is an optimisation, never a requirement
            graphs, graph_note = None, f"unavailable ({type(ex).__name__}: {str(ex)[:120]})"
            if args.graph == "on":
                raise
            barrier()

    def run_step(i, keep=None):
        if graphs is not None:
            graphs[i % nbuf][0].replay()
            return graphs[i % nbuf][1]
        return step(dev_x[i % nbuf], keep)

    # ---- timed region: device-resident inputs, CUDA events
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(2):
        run_step(i)

    class _NoClk:
        def __enter__(self): return self
        def __exit__(self, *a): pass
        def summary(self): return None

    with (ClockSampler(ctx["local_rank"]) if clocks else _NoClk()) as clk:
        barrier()
        if graphs is None:
            launches0 = _lib.launch_count
            _lib.start_timing(TIMED)
        last = {} if dump_dir is not None else None
        e0.record()
        for i in range(args.steps):
            run_step(i, last if i == args.steps - 1 else None)
        e1.record()
        barrier()
        if graphs is None:
            per_kernel = _lib.stop_timing()
            launches = _lib.launch_count - launches0
    ms = e0.elapsed_time(e1) / args.steps
    if dump_dir is not None and rank == 0:
        dump_outputs(graphs[(args.steps - 1) % nbuf][2] if graphs is not None else last, dump_dir)
    clk_summary = clk.summary()
    if graphs is not None:
        # per-kernel CUDA events cannot be read inside a replayed graph: the same steps once more, eagerly, for the
        # roofline figures and the launch count (the kernels and their inputs are identical)
        barrier()
        launches0 = _lib.launch_count
        _lib.start_timing(TIMED)
        for i in range(args.steps):
            step(dev_x[i % nbuf])
        barrier()
        per_kernel = _lib.stop_timing()
        launches = _lib.launch_count - launches0
    kept = int(layer.feed_forward.ffn.last_counts.sum().item())        # A_kept of the last step (rows through the experts)

    # ---- end to end: pinned host input -> device every step (prefetched on a copy stream), loss read back
    copy_stream = torch.cuda.Stream()
    stage = [torch.empty(B, seq, Dm, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            stage[i % 2].copy_(host_x[i % nbuf], non_blocking=True)
            ready[i % 2].record(copy_stream)

    for c in consumed:
        c.record()
    barrier()
    t0 = time.perf_counter()
    prefetch(0)
    last = 0.0
    for i in range(args.steps):
        if i + 1 < args.steps:
            prefetch(i + 1)
        torch.cuda.current_stream().wait_event(ready[i % 2])
        if graphs is not None:
            dev_x[i % nbuf].detach().copy_(stage[i % 2])           # the graph reads its own static input buffer
            consumed[i % 2].record()
            loss = run_step(i)
        else:
            x = stage[i % 2].detach().requires_grad_(True)
            loss = step(x)
            consumed[i % 2].record()
        last = loss.item()                              # device -> host read of the step's result
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps

    # ---- max over ranks
    kept_total = kept
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = t.tolist()
        k = torch.tensor([kept], device=dev, dtype=torch.int64)
        dist.all_reduce(k)
        kept_total = int(k.item())
    if graphs is not None:
        graphs.clear()
    del layer, dev_x, stage
    torch.cuda.empty_cache()
    return dict(ms=ms, e2e_ms=e2e_ms, kept_total=kept_total, per_kernel=per_kernel, launches=launches, graph_note=graph_note,
                last_loss=last, clocks=clk_summary, h2d=B * seq * Dm * 4)


def summarise(name, B, m, world, pk, pk_src, amp):
    """Headline numbers and roofline entries of one measured workload."""
    Dm, H, I, E, K, seq = WORKLOADS[name]
    steps = max(1, len(m["per_kernel"].get("ab_ssm_scan_fwd", [1])))
    tokens_per_step = B * seq
    ms, e2e_ms = m["ms"], m["e2e_ms"]
    per = lambda names: sum(sum(m["per_kernel"].get(n, [])) for n in names) / steps
    cnt = lambda names: sum(len(m["per_kernel"].get(n, [])) for n in names) / steps
    moe = ["ab_grouped_gemm_nt", "ab_grouped_gemm_nn", "ab_grouped_gemm_tn", "ab_ep_grouped_gemm_nt", "ab_ep_grouped_gemm_nn"]
    dense = ["ab_dense_gemm_nt", "ab_dense_gemm_nn", "ab_dense_gemm_tn"]
    scan = ["ab_ssm_scan_fwd", "ab_ssm_scan_bwd"]
    gemm_ms, dense_ms, scan_ms = per(moe), per(dense), per(scan)
    gemm_flops = 12.0 * Dm * I * (m["kept_total"] / world)                 # per GPU per step (SURVEY.md 8d)
    Di = 16 * H
    R = -(-Dm // 16)
    dense_flops = 6.0 * tokens_per_step * (Dm * 2 * Di + Di * (((H + 7) // 8 * 8) + 2 * Di) + Di * Dm)      # fwd + dgrad + wgrad
    es = 2 if amp else 4
    scan_bytes = tokens_per_step * (14 * Di + 3 * H) * es                  # fwd+bwd algorithmic bytes (SURVEY.md 8d)
    gemm_tflops = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    scan_gbs = scan_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    traffic, traffic_src = None, None
    try:        # mean dram__bytes_read+write per launch of this round's `ncu --set full` capture summarised under profiles/
        if name == "c2_1p5b" and B == 8 and world == 1:
            t = json.load(open(os.path.join(ROOT, "profiles", "r2_gemm_traffic.json")))
            traffic, traffic_src = t["mean_dram_bytes_per_launch"], t.get("source")
    except Exception:
        traffic = None
    roofline = {"kernel": "grouped_gemm_kernel<NT|NN|TN> (tcgen05 expert GEMM: 2 fwd + 2 dgrad + 2 wgrad launches per step)",
                "bound": "tensor", "achieved": gemm_tflops, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                "frac": gemm_tflops / pk["bf16_tflops"], "frac_of_sustained_peak": gemm_tflops / pk["bf16_tflops_sustained"],
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": pk_src + ", burst bf16 (the step is a few ms: clocks stay at their maximum, see `clocks`)",
                "ms_per_step_in_kernel": gemm_ms, "launches_per_step": cnt(moe), "share_of_step": gemm_ms / ms,
                "algorithmic_flops_per_step": gemm_flops, "kept_rows_per_step": m["kept_total"] / world}
    kernels = {"selective_scan_fwd+bwd": {"bound": "hbm", "achieved": scan_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                           "frac": scan_gbs / pk["hbm_gbs"], "ms_per_step_in_kernel": scan_ms,
                                           "algorithmic_bytes_per_step": scan_bytes, "share_of_step": scan_ms / ms},
               "ssm_projection_gemms": {"bound": "tensor", "achieved": dense_flops / (dense_ms * 1e-3) / 1e12 if dense_ms > 0 else 0.0,
                                        "unit": "TFLOP/s", "ms_per_step_in_kernel": dense_ms, "launches_per_step": cnt(dense),
                                        "share_of_step": dense_ms / ms, "note": "same tcgen05 kernel, dense entry points; small K (176..704): latency / HBM bound"}}
    return {"value": tokens_per_step * world / (ms * 1e-3), "ms_per_step": ms, "cuda_graph": m["graph_note"],
            "e2e": {"value": tokens_per_step * world / (e2e_ms * 1e-3), "unit": "tokens/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": 4,
                    "how": "pinned host x -> device each step (prefetched on a copy stream), block fwd+bwd through the module API, loss.item()"},
            "gpu_launches": m["launches"], "roofline": roofline, "kernels": kernels, "last_loss": m["last_loss"],
            "entry_point_us": {n: [round(1e3 * t, 1) for t in v[-(len(v) // steps):]] for n, v in sorted(m["per_kernel"].items()) if v}}


def ep_parity_check(ctx, name, B=1):
    """Expert parallelism against the same layer with every expert local, on this rank's own batch, before anything is
    timed: forward output, input gradient and this rank's shard of the expert weight gradients (dropout 0, the same
    routing noise on both sides).  Returns the largest relative error over the ranks."""
    import torch.distributed as dist
    dev, world, rank, group = ctx["dev"], ctx["world"], ctx["rank"], ctx["ep_group"]
    Dm, H, I, E, K, seq = WORKLOADS[name]
    ep_layer, loc_layer = build_layer(name, ctx, 0.0, ep=True), build_layer(name, ctx, 0.0, ep=False)
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    x = torch.randn(B, seq, Dm, generator=g).to(dev)
    noise = torch.randn(B * seq, E, generator=g).to(dev)
    res = {}
    for tag, layer in (("ep", ep_layer), ("local", loc_layer)):
        layer.feed_forward.ffn._draw_noise = lambda S, E_, device: noise
        xg = x.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out, _, _, lb, rz = layer(xg)
        (out.float().pow(2).mean() + lb + rz).backward()
        res[tag] = (out.detach().float(), xg.grad.float(), layer.feed_forward.ffn.expert_w1.grad.float(),
                    layer.feed_forward.ffn.last_counts.clone())
    El = E // world
    # every expert local: this rank's tokens only.  Under EP the shard holds the sum over all ranks' tokens / world
    # (what DDP's gradient averaging gives replicated experts): reduce the local-experts gradients the same way
    w1_all = res["local"][2].clone()
    dist.all_reduce(w1_all, group=group)
    w1_ref = w1_all[rank * El:(rank + 1) * El] / world
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    errs = torch.tensor([rel(res["ep"][0], res["local"][0]), rel(res["ep"][1], res["local"][1]), rel(res["ep"][2], w1_ref),
                         0.0 if torch.equal(res["ep"][3], res["local"][3]) else 1.0], device=dev, dtype=torch.float64)
    dist.all_reduce(errs, op=dist.ReduceOp.MAX, group=group)
    out, dx, dw1, cnt = errs.tolist()
    del ep_layer, loc_layer
    torch.cuda.empty_cache()
    return {"workload": workload_text(name), "tokens_per_rank": B * seq, "out_rel_err": out, "dx_rel_err": dx, "expert_w1_grad_rel_err": dw1,
            "expert_counts_equal": cnt == 0.0, "max_rel_err": max(out, dx, dw1), "precision": "bf16 autocast on both sides",
            "what": "EP layer vs the same layer with all experts local, per rank, max over ranks"}


def gpu_reference_leg(args, dev, steps=3):
    """The UNMODIFIED reference block on this B200 (CUDA fp32 and bf16 autocast), BASELINE.md section 4's 'real bar'."""
    from baseline import ref_loader
    if not ref_loader.available():
        return {"unavailable": "baseline/_ref is absent"}
    wl = WORKLOADS[args.workload]
    B, seq = args.batch, wl[5]
    out = {"workload": workload_text(args.workload), "tokens_per_step": B * seq, "hidden_dropout_prob": args.dropout,
           "how": "unmodified reference ApertisLayer on cuda, fwd + SURVEY 8(d) loss + bwd, wall clock with synchronize, mean of %d steps after 1 warm-up" % steps}
    for tag, ac in (("fp32", None), ("bf16_autocast", torch.bfloat16)):
        v, ms, _ = reference_time(wl, B, seq, args.dropout, dev, steps, 1, autocast=ac)
        out[tag] = {"tokens_per_s": v, "ms_per_step": ms}
        torch.cuda.empty_cache()
    return out


def scan_long_context(pk_hbm, L=65536, Hh=32, iters=10):
    """BASELINE.json configs[4] at its longest point (d_model 2048 -> d_inner 512, B 1, L 64K, bf16): one SSM layer's scan
    forward + backward through the C ABI against the algorithmic bytes of SURVEY.md 8(d).  The forward launch and the
    backward launches are each captured once as a CUDA graph and the replays are timed with CUDA events on the launching
    stream (device time of exactly the library's launches, no host code inside the window), L2 flushed between iterations."""
    import torch
    from apertis_llm_b200 import ops
    d = torch.device("cuda", torch.cuda.current_device())
    Di = 16 * Hh
    g = torch.Generator().manual_seed(L)
    mk = lambda *s: torch.randn(*s, generator=g).to(d, torch.bfloat16)
    xa, z, BC, dy = mk(1, L, Di), mk(1, L, Di), mk(1, L, 2 * Di), mk(1, L, Di)
    dlog = (torch.randn(1, L, Hh, generator=g) - 3.0).to(d, torch.bfloat16)
    A_log = (torch.rand(Hh, 16, generator=g) * 0.68 - 0.69).to(d)
    D = torch.ones(Di, device=d)
    leaves = [t.requires_grad_(True) for t in (xa, dlog, BC, z, A_log, D)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=d)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):                                  # warm-up (allocates the stream's workspace before the capture)
            y = ops.selective_scan(*leaves)[0]
            torch.autograd.grad(y, leaves, dy)
        torch.cuda.synchronize()
        gf, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(gf, stream=side):
            y = ops.selective_scan(*leaves)[0]
        with torch.cuda.graph(gb, stream=side, pool=gf.pool()):
            grads = torch.autograd.grad(y, leaves, dy)
        tf, tb = [], []
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        for _ in range(iters):
            flush.zero_()
            ev[0].record(side)
            gf.replay()
            ev[1].record(side)
            gb.replay()
            ev[2].record(side)
            torch.cuda.synchronize()
            tf.append(ev[0].elapsed_time(ev[1])); tb.append(ev[1].elapsed_time(ev[2]))
    torch.cuda.current_stream().wait_stream(side)
    tf.sort(); tb.sort()
    mf, mb = tf[len(tf) // 2], tb[len(tb) // 2]
    nbytes = L * (14 * Di + 3 * Hh) * 2
    gbs = nbytes / ((mf + mb) * 1e-3) / 1e9
    del grads
    return {"bound": "hbm", "achieved": gbs, "peak": pk_hbm, "unit": "GB/s", "frac": gbs / pk_hbm, "fwd_us": mf * 1e3, "bwd_us": mb * 1e3,
            "algorithmic_bytes": nbytes, "workload": "configs[4]: d_model 2048 (d_inner 512, 32 heads), B 1, L 65536, bf16, one layer's scan fwd+bwd",
            "timing": "CUDA events around graph replays of the forward launch and of the backward launches (scan + parameter reduction)",
            "schedule": "rounds (persistent, TMA-fed teams of warps walking chunks serially)"}


if __name__ == "__main__":
    main()
