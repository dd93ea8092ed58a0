"""Executed work of the pruned fused selection (DESIGN.md 4.1) on bench.py's workloads, against the DMMA roof.

bench.py's roofline block counts the algorithmic work of the unpruned product (N^2 + N(3d+18) per candidate), so with
pruning its `frac` reads above 1.  This tool reports what the kernels actually execute per step: every candidate
goes through the screen (phase A + the first kScreenBlocks row blocks of L^-1), the pilot and the survivors through
the full triangular product.  DMMA work per candidate (2 flops per multiply-add, structurally zero k-tiles skipped):
screen 2 * 128^2 * R(R+1)/2, full 2 * 128^2 * nb(nb+1)/2 with nb = N/128 row blocks.

  python tools/prune_stats.py [--config c3|c5] [--steps K] [--m M]      (one JSON line; needs the B200)
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCREEN_BLOCKS = 2  # kScreenBlocks, csrc/predict16.cuh
DMMA_PEAK_TFLOPS = 37.15  # profiles/r01_fp64_microbench.json, B200


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3", choices=["c3", "c5"])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--m", type=int, default=0, help="candidates per call (default: the config's)")
    args = ap.parse_args()

    import torch
    from sklearn.gaussian_process.kernels import Matern

    import bayesianoptimization_b200 as bo
    from bayesianoptimization_b200 import _lib as B
    from bench import ALPHA, CONFIGS, KAPPA, KSEEDS, XI, make_problem

    cfg = CONFIGS[args.config]
    X, y = make_problem(cfg)
    gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=cfg["ls"]), alpha=ALPHA,
                                         normalize_y=True, optimizer=None).fit(X, y)
    if cfg["acq"] == "ei":
        acq = bo.FusedAcquisition(B.ACQ_EI, gp, xi=XI, y_max=float(y.max()))
    else:
        acq = bo.FusedAcquisition(B.ACQ_UCB, gp, kappa=KAPPA)
    d, n = cfg["d"], cfg["n"]
    m = args.m or cfg["m_per_gpu"] or cfg["m_total"]
    dev = torch.device("cuda", 0)
    if cfg["scaling"] == "weak":  # candidate buffer 0 of rank 0, as bench.py builds it
        xt = torch.from_numpy(np.random.RandomState(1000).uniform(size=(m, d))).to(dev)
    else:
        parts = []
        for blk_i in range((m + (1 << 16) - 1) >> 16):
            g = torch.Generator(device=dev)
            g.manual_seed(blk_i)
            parts.append(torch.rand((1 << 16, d), generator=g, device=dev, dtype=torch.float64))
        xt = torch.cat(parts)[:m].contiguous()
    sel = torch.zeros((KSEEDS + 1, 2), dtype=torch.int64, device=dev)
    L = B.lib()
    stream = torch.cuda.current_stream()
    nb = (n + 127) // 128
    screen_fl = 2 * 128 * 128 * SCREEN_BLOCKS * (SCREEN_BLOCKS + 1) / 2
    full_fl = 2 * 128 * 128 * nb * (nb + 1) / 2
    legs = []
    for step in range(args.steps + 1):
        B.check(L.b200bo_acq_eval_dev(C.byref(acq.spec), xt.data_ptr(), m, None, None, None, KSEEDS, sel.data_ptr(),
                                      0, stream.cuda_stream))
        ms = C.c_float()
        B.check(L.b200bo_last_kernel_ms(C.byref(ms)))
        s, e = C.c_int64(), C.c_int64()
        B.check(L.b200bo_last_select_stats(C.byref(s), C.byref(e)))
        if step == 0:
            continue  # warm-up
        executed = (s.value * screen_fl + e.value * full_fl) / (ms.value * 1e-3) / 1e12
        legs.append({"kernel_ms": ms.value, "screened": s.value, "evaluated": e.value,
                     "evaluated_frac": e.value / m, "executed_tflops": executed,
                     "executed_frac_of_dmma_peak": executed / DMMA_PEAK_TFLOPS})
    print(json.dumps({"config": args.config, "m": m, "n": n, "d": d, "screen_blocks": SCREEN_BLOCKS,
                      "gpu": torch.cuda.get_device_name(0), "steps": legs}))


if __name__ == "__main__":
    main()
