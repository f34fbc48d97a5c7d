#!/usr/bin/env python
# coding=utf-8
"""Times the dense projections of the bench step (2,449,029 x 100 -> 128 columns per projection) on one GPU:
round-1 kernel (one launch per projection) against tfgk_gemm_proj_f32 with 1..4 column blocks per launch."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tf_geometric_b200 import ops  # noqa: E402


def timed(fn, reps=10, warm=3, flush=None):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.add_(1.0)                      # 512 MB write: evicts the 126 MB L2
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def main():
    m, k = int(os.environ.get("M", 2449029)), int(os.environ.get("K", 100))
    dev = torch.device("cuda")
    gen = torch.Generator(device="cpu"); gen.manual_seed(0)
    x = torch.randn((m, k), generator=gen).to(dev)
    ws = [(torch.randn((k, 128), generator=gen) / 10).to(dev) for _ in range(4)]
    bias = torch.zeros(128, device=dev)
    outs = [torch.empty((m, 128), device=dev) for _ in range(4)]
    flush = torch.zeros(128 * 1024 * 1024, device=dev)
    res = {"M": m, "K": k, "peak_gbs": None}
    med, best = timed(lambda: ops.gemm(x, ws[0], bias=bias, act=ops.ACT_RELU, out=outs[0]), flush=flush)
    res["round1_single_projection_ms"] = {"median": med, "min": best}
    for nb in (1, 2, 3, 4):
        blocks = [(ws[i], bias, ops.ACT_RELU if i % 2 == 0 else ops.ACT_NONE, outs[i]) for i in range(nb)]
        med, best = timed(lambda: ops.gemm_proj(x, blocks), flush=flush)
        gb = (m * k * 4 + nb * m * 128 * 4) / 1e9
        res["proj_nb{}".format(nb)] = {"median_ms": med, "min_ms": best, "algorithmic_gb": gb,
                                      "gbs_at_median": gb / (med * 1e-3), "tf32x3_tflops": 6.0 * m * 104 * 128 * nb / (med * 1e-3) / 1e12}
    for ctas in (96,):
        blocks = [(ws[i], bias, ops.ACT_NONE, outs[i]) for i in range(3)]
        med, best = timed(lambda: ops.gemm_proj(x, blocks, max_ctas=ctas), flush=flush)
        res["proj_nb3_ctas{}".format(ctas)] = {"median_ms": med, "min_ms": best}
    print(json.dumps(res, indent=1))
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    json.dump(res, open(os.path.join(out, "bench_gemm.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
