#!/usr/bin/env python
"""Long-context selective-scan sweep (BASELINE.json configs[4]): d_model 2048 -> Di 512, H 32, one SSM layer's scan
kernels forward + backward, seq 2K..64K, HBM GB/s against the algorithmic bytes of SURVEY.md section 8(d).

    python tools/scan_bench.py [--dtype bf16|f32] [--mode rounds|pipe|single|two_pass] [--seqs 2048,...] [--batch 1] [--iters 20]
                               [--heads 32] [--d-state 16]     (Di = d_state * heads; the older modes take d_state 16 only)
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from apertis_llm_b200 import _lib, ops  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dtype", default="bf16")
    ap.add_argument("--mode", default="rounds")
    ap.add_argument("--tc-fwd", type=int, default=0, help="rounds schedule: forward chunk length (0 = library default)")
    ap.add_argument("--tc-bwd", type=int, default=0)
    ap.add_argument("--wps", type=int, default=0, help="rounds schedule: cap on resident warps per SM")
    ap.add_argument("--nst-fwd", type=int, default=0, help="rounds schedule: ring stages of the forward (2 | 3, 0 = default)")
    ap.add_argument("--nst-bwd", type=int, default=0)
    ap.add_argument("--seqs", default="2048,4096,8192,16384,32768,65536")
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--heads", type=int, default=32)
    ap.add_argument("--d-state", type=int, default=16, help="ssm_d_state N: 16, 32 or 64 (Di = N * heads)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--json", default="")
    ap.add_argument("--graph", action="store_true", help="time CUDA-graph replays of the launches (no host code inside the event windows)")
    args = ap.parse_args()
    d = torch.device("cuda:0")
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    es = 2 if dtype == torch.bfloat16 else 4
    mode = {"single": _lib.SCAN_SINGLE_PASS, "two_pass": _lib.SCAN_TWO_PASS, "pipe": _lib.SCAN_PIPELINED, "rounds": _lib.SCAN_ROUNDS}[args.mode]
    _lib.load().ab_ssm_scan_tune(args.tc_fwd, args.tc_bwd, args.wps, args.nst_fwd, args.nst_bwd)
    H, N = args.heads, args.d_state
    Di = N * H
    B = args.batch
    peak = 6539.2
    try:
        peak = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=d)
    out = []
    for L in [int(s) for s in args.seqs.split(",")]:
        g = torch.Generator(device="cpu").manual_seed(L)
        mk = lambda *s: torch.randn(*s, generator=g).to(d, dtype)
        xa, z, BC = mk(B, L, Di), mk(B, L, Di), mk(B, L, 2 * Di)
        dlog = (torch.randn(B, L, H, generator=g) - 3.0).to(d, dtype)
        A_log = (torch.rand(H, N, generator=g) * 0.68 - 0.69).to(d)
        D = torch.ones(Di, device=d)
        dy = mk(B, L, Di)
        leaves = [t.requires_grad_(True) for t in (xa, dlog, BC, z)]
        A_log.requires_grad_(True); D.requires_grad_(True)
        names = ["ab_ssm_scan_fwd", "ab_ssm_scan_bwd"] if mode == _lib.SCAN_ROUNDS else ["ab_selective_scan_fwd", "ab_selective_scan_bwd"]

        def run():
            y, _, _ = ops.selective_scan(xa, dlog, BC, z, A_log, D, mode=mode)
            y.backward(dy)
            for t in leaves + [A_log, D]:
                t.grad = None

        for _ in range(3):
            run()
        torch.cuda.synchronize()
        tf, tb = [], []
        if args.graph:
            lv = leaves + [A_log, D]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                yy = ops.selective_scan(xa, dlog, BC, z, A_log, D, mode=mode)[0]
                torch.autograd.grad(yy, lv, dy)
                torch.cuda.synchronize()
                gf, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with torch.cuda.graph(gf, stream=side):
                    yy = ops.selective_scan(xa, dlog, BC, z, A_log, D, mode=mode)[0]
                with torch.cuda.graph(gb, stream=side, pool=gf.pool()):
                    gg = torch.autograd.grad(yy, lv, dy)
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                for _ in range(args.iters):
                    flush.zero_()
                    ev[0].record(side); gf.replay(); ev[1].record(side); gb.replay(); ev[2].record(side)
                    torch.cuda.synchronize()
                    tf.append(ev[0].elapsed_time(ev[1])); tb.append(ev[1].elapsed_time(ev[2]))
            torch.cuda.current_stream().wait_stream(side)
            del gg
        else:
            for _ in range(args.iters):
                flush.zero_()                       # evict L2 between iterations (inputs of short sequences fit in L2)
                _lib.start_timing(names)
                run()
                t = _lib.stop_timing()
                tf.append(sum(t[names[0]])); tb.append(sum(t[names[1]]))
        tf.sort(); tb.sort()
        mf, mb = tf[len(tf) // 2], tb[len(tb) // 2]
        tok = B * L
        bf, bb = tok * (5 * Di + H) * es, tok * (9 * Di + 2 * H) * es
        rec = dict(L=L, B=B, H=H, d_state=N, Di=Di, dtype=args.dtype, mode=args.mode, fwd_us=mf * 1e3, bwd_us=mb * 1e3,
                   fwd_gbs=bf / mf / 1e6, bwd_gbs=bb / mb / 1e6, fwdbwd_gbs=(bf + bb) / (mf + mb) / 1e6,
                   frac_of_measured_peak=(bf + bb) / (mf + mb) / 1e6 / peak, tokens_per_s=tok / ((mf + mb) * 1e-3))
        out.append(rec)
        print(f"L={L:6d} N={N:2d} fwd {mf * 1e3:8.1f} us {rec['fwd_gbs']:7.0f} GB/s | bwd {mb * 1e3:8.1f} us {rec['bwd_gbs']:7.0f} GB/s | "
              f"fwd+bwd {rec['fwdbwd_gbs']:7.0f} GB/s = {100 * rec['frac_of_measured_peak']:5.1f}% of {peak:.0f}")
    if args.json:
        json.dump(out, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
