"""Per-layer convolution timing at the bench geometry (B=256 CREMA-D shape): fwd / dgrad / wgrad of every
distinct conv of both encoders, CUDA-event timed, L2 flushed between repetitions.
    python tools/conv_bench.py [--out gpurun_out/conv_bench.json] [--tag name] [--ops fwd,dgrad,wgrad]
GDL_FLAT=0 / GDL_WFLAT=0 select the generic gather kernels instead of the flat-window ones; the library reads them
once per process: run it once per setting and compare the JSON files."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))
from gdl_b200 import ops  # noqa: E402


def cases(B):
    out = []
    for tag, N, (h, w) in (("v", 3 * B, (56, 56)), ("a", B, (65, 47))):
        c = 64
        for li in range(1, 5):
            co = 64 << (li - 1)
            if li > 1:
                out.append(("%s.l%d.s2" % (tag, li), N, h, w, c, co, 3, 2, 1))
                out.append(("%s.l%d.ds" % (tag, li), N, h, w, c, co, 1, 2, 0))
                h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
            out.append(("%s.l%d.s1" % (tag, li), N, h, w, co, co, 3, 1, 1))
            c = co
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="gpurun_out/conv_bench.json")
    ap.add_argument("--tag", default="default")
    ap.add_argument("--ops", default="fwd,dgrad,wgrad")
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    ops.init()
    want = a.ops.split(",")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = {}
    for (name, N, H, W, Ci, Co, R, stride, pad) in cases(a.B):
        if a.only and a.only not in name:
            continue
        d = ops.conv_desc(N, H, W, Ci, Co, R, R, stride, pad)
        x = torch.randn(N, H, W, Ci, device="cuda").to(torch.bfloat16)
        dy = torch.randn(N, d.Ho, d.Wo, Co, device="cuda").to(torch.bfloat16)
        w = torch.randn(Co, Ci, R, R, device="cuda") * 0.05
        wp = torch.empty(Co, ops.conv_packed_k(d), device="cuda", dtype=torch.bfloat16)
        wT = torch.zeros(Ci, R * R * Co, device="cuda", dtype=torch.bfloat16)
        ops.conv_pack_weights(d, Ci, w, wp, wT)
        y = torch.empty(N, d.Ho, d.Wo, Co, device="cuda", dtype=torch.bfloat16)
        dx = torch.empty(N, H, W, Ci, device="cuda", dtype=torch.bfloat16)
        dw = torch.empty_like(w)
        ws = torch.empty(max(ops.conv_wgrad_workspace_bytes(d), 16) // 4, device="cuda")
        fl = ops.conv_flops(d)
        fns = {"fwd": lambda: ops.conv_fwd(d, x, wp, y),
               "dgrad": lambda: ops.conv_dgrad(d, dy, wT, dx),
               "wgrad": lambda: ops.conv_wgrad(d, Ci, x, dy, dw, ws)}
        for op in want:
            fn = fns[op]
            fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(a.reps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = sorted(ts)[len(ts) // 2]
            res["%s.%s" % (name, op)] = {"ms": round(ms, 4), "tflops": round(fl / ms / 1e9, 1)}
            print("%-14s %-6s N%d %dx%d C%d->%d k%d s%d  %.3f ms  %.0f TF" % (name, op, N, H, W, Ci, Co, R, stride, ms,
                                                                       fl / ms / 1e9), flush=True)
    tot = sum(v["ms"] for v in res.values())
    print("total %.3f ms" % tot)
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    allres = {}
    if os.path.exists(a.out):
        allres = json.load(open(a.out))
    allres[a.tag] = res
    json.dump(allres, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
