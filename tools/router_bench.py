"""Times the MoE router and dispatch-plan entry points (ab_moe_router_fwd, ab_moe_plan, ab_moe_router_bwd) with CUDA
events at the C2 and C4 block shapes, with L2 overwritten before every timed launch, and reports microseconds and GB/s
over the bytes each call must move (computed from the shapes below).

    python tools/router_bench.py [--iters 50] [--json out.json]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from apertis_llm_b200 import _lib, ops  # noqa: E402
from apertis_llm_b200._lib import call, dt, ptr, query, stream_ptr  # noqa: E402

# name -> (tokens S, hidden Dm, experts E, top-K, capacity factor): 8 x 4096 tokens at C2, 4 x 4096 at C4 (bench.py)
SHAPES = {"c2": (8 * 4096, 704, 8, 2, 1.25), "c4": (4 * 4096, 1600, 8, 2, 1.25)}


def run(name, iters, flush):
    S, Dm, E, K, cf = SHAPES[name]
    d = torch.device("cuda:0")
    g = torch.Generator(device=d).manual_seed(0)
    f32 = dict(dtype=torch.float32, device=d)
    x = torch.randn(S, Dm, generator=g, **f32)
    rn_w = 1 + 0.1 * torch.randn(Dm, generator=g, **f32)
    rn_b = 0.1 * torch.randn(Dm, generator=g, **f32)
    Wr = 0.05 * torch.randn(E, Dm, generator=g, **f32)
    br = 0.01 * torch.randn(E, generator=g, **f32)
    noise = torch.randn(S, E, generator=g, **f32)
    ns = torch.full((E,), 0.07, **f32)
    cap = int(S / E * cf)
    r = ops.moe_route(x, rn_w, rn_b, 1e-12, Wr, br, noise, ns, K)
    plan = ops.moe_plan(r["idx"], r["w"], E, cap)
    max_rows = plan["max_rows"]
    dw_row = torch.randn(max_rows, generator=g, **f32)
    dxrow = torch.randn(max_rows, Dm, generator=g, **f32)
    fvec = (r["aux"][E:2 * E] / S).contiguous()
    scal = torch.tensor([0.3, 0.02], **f32)
    dx = torch.empty_like(x)
    dWr, dbr, dnw, dnb, dns = (torch.empty(E, Dm, **f32), torch.empty(E, **f32), torch.empty(Dm, **f32),
                               torch.empty(Dm, **f32), torch.empty(E, **f32))
    ws_b = torch.empty(query("ab_moe_router_bwd_workspace_bytes", S, Dm, E), dtype=torch.uint8, device=d)
    kept = int(plan["n_rows"][1])

    def bwd():
        call("ab_moe_router_bwd", ptr(x), ptr(r["stats"]), ptr(rn_w), ptr(rn_b), ptr(Wr), ptr(br), ptr(r["gates"]), ptr(r["idx"]),
             ptr(r["probs"]), ptr(r["lse"]), ptr(r["lclean"]), ptr(noise), ptr(fvec), ptr(scal), ptr(dw_row), ptr(dxrow),
             ptr(plan["row_of"]), ptr(dx), ptr(dWr), ptr(dbr), ptr(dnw), ptr(dnb), ptr(dns), ptr(ws_b), ws_b.numel(),
             S, Dm, E, K, dt(x), stream_ptr())

    es = x.element_size()
    cases = {
        # x read once; the per-token outputs (lclean, logits, gates [S,E], idx, probs, w [S,K], lse, stats) written once
        "ab_moe_router_fwd": (lambda: ops.moe_route(x, rn_w, rn_b, 1e-12, Wr, br, noise, ns, K), S * Dm * es + S * (4 * E + 3 * K + 3) * 4),
        # idx and w read, row_of written, the row maps written
        "ab_moe_plan": (lambda: ops.moe_plan(r["idx"], r["w"], E, cap), S * K * 12 + max_rows * 8),
        # x and the kept rows of dxrow read, dx written
        "ab_moe_router_bwd": (bwd, 2 * S * Dm * es + kept * Dm * 4),
    }
    scratch = torch.empty(512 * 2 ** 20, dtype=torch.uint8, device=d)      # 512 MB > 126 MB of L2
    out = {}
    for case, (fn, nbytes) in cases.items():
        for _ in range(5):
            fn()
        # no synchronisation inside the loop: the L2-overwriting fill keeps the GPU busy while the host enqueues the next
        # call, so the events time the GPU work and not the Python launch overhead
        ev = []
        for _ in range(iters):
            if flush:
                scratch.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            ev.append((a, b))
        torch.cuda.synchronize()
        times = [a.elapsed_time(b) * 1e3 for a, b in ev]
        times.sort()
        med = times[len(times) // 2]
        out[case] = {"us_median": round(med, 2), "us_min": round(times[0], 2), "bytes": nbytes,
                     "GBps": round(nbytes / med / 1e3, 1), "floor_us_at_7.7TBps": round(nbytes / 7.7e6, 2)}
    out["total_us_median"] = round(sum(v["us_median"] for v in out.values() if isinstance(v, dict)), 2)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--no-flush", action="store_true", help="do not overwrite L2 between launches")
    ap.add_argument("--shapes", default="c2,c4")
    ap.add_argument("--json", default=None, help="also write the results here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("router_bench: needs a CUDA device")
    props = torch.cuda.get_device_properties(0)
    res = {"device": props.name, "sms": props.multi_processor_count}
    try:
        import subprocess
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        res["power_limit"] = "unknown"
    for name in args.shapes.split(","):
        res[name] = run(name, args.iters, not args.no_flush)
    print(json.dumps(res, indent=1))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    _lib.load()
    main()
