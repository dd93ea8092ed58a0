#!/usr/bin/env python
"""bench.py - candidate-points/s through fused GP posterior-predict + acquisition (BASELINE.json metric).

Default workload (BASELINE configs[2], "c3"): d=16, N_train=4096, Matern-2.5 (l=0.7, alpha=1e-6,
normalize_y), EI xi=0.01, M = 2^20 uniform candidates per GPU per step, fp64, weak scaling.  One "step" =
one pass of the hot path over one candidate batch: K* build -> V = L^-1 K*^T -> (mu, sigma) -> EI ->
argmin + top-10 (selection fused into the kernel's epilogue, no acq[M] materialised).
`--config c5` = BASELINE configs[4]: d=32, N_train=8192, UCB, 2^22 candidates in TOTAL sharded over the
ranks (strong scaling), NCCL all-gather of the per-rank records for the final argmax.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3|c5] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes, as float64 .npy, the merged selection records of the LAST timed device step
(device_argmin_index, device_argmin_value, device_top_indices) and, on one rank, what the last timed
FusedAcquisition.argmin_topk call returned (e2e_*).  The inputs depend only on the arguments (fixed seeds), so two
builds can be compared output for output.

Keys beyond the base contract:
  value         candidates already resident in HBM (device entry point of the C ABI), whole job
  e2e           same metric through the package's public call with HOST ndarrays (pageable, as
                TargetSpace.random_sample returns them): H2D of the batch and D2H of the records inside
  roofline      dominant kernel vs the roof that binds it (traffic read from this round's committed ncu summary)
  cpu_baseline  the UNMODIFIED reference (vendored bayes_opt: ExpectedImprovement._get_acq on a wrap_kernel GP)
                timed on the host cores on a bounded sample, rank 0, N=1 only
  fp32_mode / throughput_mode / c5_strong / fit / suggest   secondary legs (see each entry's "what")
"""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
_REFERENCE_ARM = "--impl" in sys.argv and sys.argv[sys.argv.index("--impl") + 1:][:1] == ["reference"]
if _REFERENCE_ARM:
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is entitled to every host thread.  The BLAS /
    # OpenMP pools read these at load time, so they are set BEFORE numpy / scipy are imported.
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse  # noqa: E402
import ctypes as C  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

# the reference package: vendored unmodified by build() (oracle/vendor_ref.py, git-ignored oracle/_ref); only read here
from oracle.vendor_ref import ref_dir  # noqa: E402

_REF_DIR = ref_dir()
if _REF_DIR and _REF_DIR not in sys.path:
    sys.path.insert(0, _REF_DIR)

KSEEDS = 10
N_CAND_BUFFERS = 3  # rotated so that no step re-reads candidates from L2
CONFIGS = {
    # name: d, N_train, length_scale, acquisition, candidates, scaling
    "c3": dict(d=16, n=4096, ls=0.7, acq="ei", m_per_gpu=1 << 20, m_total=None, scaling="weak",
               label="BASELINE configs[2]: d=16, N_train=4096, Matern-2.5 l=0.7, EI xi=0.01, M=2^20 candidates "
                     f"per GPU per step, argmin+top-{KSEEDS}"),
    "c5": dict(d=32, n=8192, ls=1.0, acq="ucb", m_per_gpu=None, m_total=1 << 22, scaling="strong",
               label="BASELINE configs[4]: d=32, N_train=8192, Matern-2.5 l=1.0, UCB kappa=2.576, 2^22 candidates "
                     f"in total sharded over the ranks per step, NCCL exchange, argmin+top-{KSEEDS}"),
}
ALPHA, XI, KAPPA = 1e-6, 0.01, 2.576


def flops_per_candidate(n, d, n_gps=1):
    """SURVEY.md 8(d): F = N^2 + N(3d + 18) per GP."""
    return n_gps * (n * n + n * (3 * d + 18))


def hbm_model_bytes_per_candidate(n, d, tile, s=8):
    """SURVEY.md 8(d) 'TRSM-bound HBM' model: L^-1 re-streamed once per tile of T candidates."""
    return s * n * (n + 1) / (2 * tile) + s * n * (d + 1) / tile + s * d + s


def make_problem(cfg, seed=0):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(cfg["n"], cfg["d"]))
    y = np.sin(X.sum(1)) + 0.1 * rs.randn(cfg["n"])
    return X, y


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the reference arm: the unmodified bayes_opt closure on the host cores
# ------------------------------------------------------------------------------------------------
def reference_closure(cfg, X, y):
    """acq = ExpectedImprovement(xi)._get_acq(gp) (R/bayes_opt/acquisition.py:171-219) on the GP the
    reference builds (bayesian_optimization.py:124-130: wrap_kernel(Matern(2.5), space.kernel_transform),
    alpha=1e-6, normalize_y) at the bench's fixed length scale (optimizer=None), BASELINE.md 3.2."""
    import warnings

    from bayes_opt import acquisition
    from bayes_opt.parameter import wrap_kernel
    from bayes_opt.target_space import TargetSpace
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import Matern

    d = cfg["d"]
    space = TargetSpace(None, {f"x{i:02d}": (0.0, 1.0) for i in range(d)})
    gp = GaussianProcessRegressor(kernel=wrap_kernel(Matern(nu=2.5, length_scale=cfg["ls"]), space.kernel_transform),
                                  alpha=ALPHA, normalize_y=True, optimizer=None)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gp.fit(X, y)
    if cfg["acq"] == "ei":
        a = acquisition.ExpectedImprovement(xi=XI)
        a.y_max = float(y.max())
    else:
        a = acquisition.UpperConfidenceBound(kappa=KAPPA)
    return a._get_acq(gp=gp), space


def cpu_reference_rate(cfg, X, y, m_sample, reps=1):
    """candidates/s of the reference closure + its selection (ys.argmin(), np.argsort(ys)[:n],
    R/bayes_opt/acquisition.py:312-317), chunked at 2^14 rows (BASELINE.md 3.4)."""
    acq, space = reference_closure(cfg, X, y)
    xt = space.random_sample(m_sample, random_state=np.random.RandomState(1))

    def run(x):
        ys = np.concatenate([acq(x[i:i + (1 << 14)]) for i in range(0, len(x), 1 << 14)])
        return int(ys.argmin()), np.argsort(ys)[:KSEEDS]

    run(xt[:1024])  # warm-up
    best = np.inf
    for _ in range(reps):
        t0 = time.perf_counter()
        run(xt)
        best = min(best, time.perf_counter() - t0)
    return m_sample / best, best


def blas_pools():
    import threadpoolctl

    return [f'{i.get("internal_api")}:{i.get("num_threads")}' for i in threadpoolctl.threadpool_info()]


def base_line(args, world, cfg):
    m_desc = (f"{cfg['m_per_gpu']} per GPU" if cfg["scaling"] == "weak" else f"{cfg['m_total']} total / {world} ranks")
    return {
        "metric": f"candidate-pts/s GP-predict+{cfg['acq'].upper()} @ N_train={cfg['n']},d={cfg['d']}",
        "unit": "candidates/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": cfg["label"], "n_train": cfg["n"], "d": cfg["d"], "candidates_per_step": m_desc,
                   "l2": f"{N_CAND_BUFFERS} candidate buffers rotated + 8*N^2/2 B factor + 148 x 8*N*128 B K* scratch per "
                         "step: working set > 126 MB L2",
                   "parallelism": f"candidates sharded x{world}, model replicated"},
    }


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    if _REF_DIR is None:
        emit({"impl": "reference", "unavailable": "oracle/_ref (vendored bayes_opt) is missing: build() runs "
                                                  "oracle/vendor_ref.py where the reference source tree is present"})
        return
    import threadpoolctl

    cores = os.cpu_count()
    threadpoolctl.threadpool_limits(limits=cores)
    pools = blas_pools()
    X, y = make_problem(cfg)
    m_sample = 1 << 13 if cfg["n"] <= 4096 else 1 << 12
    for _ in range(max(args.warmup, 1) - 1):
        cpu_reference_rate(cfg, X, y, 1024)
    t0 = time.perf_counter()
    rates = [cpu_reference_rate(cfg, X, y, m_sample)[0] for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    v = float(np.median(rates))
    line = base_line(args, world, cfg)
    line.update({
        "impl": "reference", "value": v, "ms_per_step": 1e3 * m_sample / v,
        "cpu_baseline": {"value": v, "unit": "candidates/s", "cores": cores, "kind": "reference",
                         "sample": f"{m_sample} candidates/step x {args.steps} steps through the vendored bayes_opt "
                                   f"closure ({cfg['acq'].upper()}._get_acq on a wrap_kernel GP) + argmin/argsort, chunks of 2^14",
                         "blas": pools, "omp_env": os.environ.get("OMP_NUM_THREADS")},
        "e2e": {"value": v, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": wall,
    })
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, torchrun's OMP notice) write to fd 1; the contract is ONE
    JSON line on stdout.  Point fd 1 at stderr for the whole run and keep the real stdout aside."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def dump_outputs(path, arrays):
    """Each array as path/<name>.npy in float64 (row indices are exact in float64 below 2^53)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def ncu_traffic(kernel):
    """dram bytes per launch of `kernel` from this round's committed ncu capture (profiles/r02_ncu_traffic.json,
    written by tools/ncu_summary.py from the .ncu-rep), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))[kernel]
        return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"]), t.get("source")
    except Exception:
        return None, None


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary legs (fp32, throughput, c5, fit, suggest)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import bayesianoptimization_b200 as bo
    from bayesianoptimization_b200 import _lib as B
    from bayesianoptimization_b200.sharding import merge_selection, shard_range
    from sklearn.gaussian_process.kernels import Matern

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = B.lib()
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_acq(cfg, X, y, precision="fp64"):
        gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=cfg["ls"]), alpha=ALPHA,
                                             normalize_y=True, optimizer=None, device=local_rank, precision=precision)
        t0 = time.perf_counter()
        gp.fit(X, y)
        fit_s = time.perf_counter() - t0
        if cfg["acq"] == "ei":
            acq = bo.FusedAcquisition(B.ACQ_EI, gp, xi=XI, y_max=float(y.max()))
        else:
            acq = bo.FusedAcquisition(B.ACQ_UCB, gp, kappa=KAPPA)
        return gp, acq, fit_s

    def timed(fn, steps, warmup, sample_clocks=True, kernel_times=True):
        """W untimed + K timed steps, barrier + synchronize on both sides, CUDA events on the launching
        stream, max over ranks."""
        for i in range(warmup):
            fn(i)
        barrier()
        kernel_ms = []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = L.b200bo_launch_count()
        sampler = ClockSampler(local_rank)
        if rank == 0 and sample_clocks:
            sampler.start()
        ev0.record()
        for i in range(steps):
            fn(warmup + i)
            if kernel_times:
                ms = C.c_float()
                B.check(L.b200bo_last_kernel_ms(C.byref(ms)))  # CUDA events on the launching stream
                kernel_ms.append(ms.value)
        ev1.record()
        barrier()
        clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
        total_ms = ev0.elapsed_time(ev1)
        launches = L.b200bo_launch_count() - launches0
        if world > 1:
            t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms, kernel_ms, launches, clocks

    def merged_result(sel, gathered):
        stream.synchronize()
        if world > 1:
            allr = gathered.cpu().numpy()
            bi, bv, top = merge_selection(allr.view(np.float64)[:, :, 0], allr[:, :, 1], KSEEDS)
            return int(bi), float(bv), [int(t) for t in top]
        s = sel.cpu().numpy()
        return int(s[0, 1]), float(s.view(np.float64)[0, 0]), [int(t) for t in s[1:, 1]]

    def run_config(cfg, steps, warmup, with_e2e=True, precision="fp64", sample_clocks=True):
        """The hot path at one configuration: HBM-resident leg (+ exchange), then the e2e leg."""
        X, y = make_problem(cfg)
        gp, acq, fit_s = make_acq(cfg, X, y, precision)
        d = cfg["d"]
        if cfg["scaling"] == "weak":
            m_local, index_base = cfg["m_per_gpu"], rank * cfg["m_per_gpu"]
            host_bufs = [torch.from_numpy(np.random.RandomState(1000 + 17 * rank + b).uniform(size=(m_local, d)))
                         for b in range(N_CAND_BUFFERS)]
            dev_bufs = [t.to(dev) for t in host_bufs]
        else:
            # strong scaling: ONE global candidate set per buffer, defined by blocks of 2^16 rows that any rank
            # can regenerate (device generator seeded by (buffer, block)), so the union is the same for every
            # world size and the merged argmin of N ranks must equal the N=1 result.
            s0, s1 = shard_range(cfg["m_total"], rank, world)
            m_local, index_base = s1 - s0, s0
            blk = 1 << 16
            dev_bufs = []
            for b in range(N_CAND_BUFFERS):
                parts = []
                for blk_i in range(s0 // blk, (s1 + blk - 1) // blk):
                    g = torch.Generator(device=dev)
                    g.manual_seed(7919 * b + blk_i)
                    t = torch.rand((blk, d), generator=g, device=dev, dtype=torch.float64)
                    lo, hi = max(s0, blk_i * blk) - blk_i * blk, min(s1, (blk_i + 1) * blk) - blk_i * blk
                    parts.append(t[lo:hi])
                dev_bufs.append(torch.cat(parts).contiguous())
            host_bufs = [t.cpu() for t in dev_bufs] if with_e2e else []
        sel = torch.zeros((KSEEDS + 1, 2), dtype=torch.int64, device=dev)
        gathered = torch.zeros((world, KSEEDS + 1, 2), dtype=torch.int64, device=dev) if world > 1 else None
        spec = acq.spec
        exch_ms = []

        def step_device(i):
            B.check(L.b200bo_acq_eval_dev(C.byref(spec), dev_bufs[i % N_CAND_BUFFERS].data_ptr(), m_local, None,
                                          None, None, KSEEDS, sel.data_ptr(), index_base, stream.cuda_stream))
            if world > 1:  # the path's ONE exchange step: all_gather of the (argmin, top-k) records, 176 B per rank
                dist.all_gather_into_tensor(gathered, sel)

        total_ms, kernel_ms, launches, clocks = timed(step_device, steps, warmup, sample_clocks)
        m_step = world * m_local if cfg["scaling"] == "weak" else cfg["m_total"]
        last = merged_result(sel, gathered)  # what the last timed step computed
        outputs = {"device_argmin_index": last[0], "device_argmin_value": last[1], "device_top_indices": last[2]}
        step_device(0)  # untimed: the reported result is always that of candidate buffer 0 (comparable across legs / N)
        res = merged_result(sel, gathered)
        out = {"value": m_step * steps / (total_ms * 1e-3), "ms_per_step": total_ms / steps, "kernel_ms": float(np.mean(kernel_ms)),
               "launches": int(launches), "clocks": clocks, "result": {"argmin_index": res[0], "argmin_value": res[1],
                                                                      "top_indices": res[2]},
               "m_local": int(m_local), "m_step": int(m_step), "fit_s": fit_s}
        if world > 1:  # every rank's own mean kernel time (the step time is the max over ranks: GPUs of a box differ by a few %)
            t = torch.tensor([out["kernel_ms"]], dtype=torch.float64, device=dev)
            allk = torch.zeros(world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(allk, t)
            out["kernel_ms_per_rank"] = [round(float(v), 2) for v in allk.cpu()]
        if world > 1:  # the exchange alone, device-timed
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for _ in range(20):
                dist.all_gather_into_tensor(gathered, sel)
            e1.record()
            torch.cuda.synchronize()
            out["exchange_ms"] = e0.elapsed_time(e1) / 20
        if with_e2e:
            host_np = [t.numpy() for t in host_bufs]  # pageable ndarrays, as TargetSpace.random_sample returns them

            def step_e2e(i):
                # the call a user of the package makes (DeviceHooks._random_sample_minimize does exactly this): host
                # candidates in, (argmin, value, seed indices) out.  Inside: finite check, chunked H2D overlapped with
                # the fused kernel + selection, D2H of the records.
                idx, val, top = acq.argmin_topk(host_np[i % N_CAND_BUFFERS], KSEEDS)
                if world == 1:  # with more ranks this is one shard's result, not the job's
                    outputs.update(e2e_argmin_index=idx, e2e_argmin_value=val, e2e_top_indices=top)
                if world > 1:  # the exchange step, from host-side records
                    rec = torch.full((KSEEDS + 1, 2), -1, dtype=torch.int64)
                    rec[0, 0] = int(np.float64(val).view(np.int64))
                    rec[0, 1] = index_base + idx
                    rec[1:1 + len(top), 1] = torch.from_numpy(index_base + np.asarray(top, dtype=np.int64))
                    dist.all_gather_into_tensor(gathered, rec.to(dev))

            e2e_ms, _, _, _ = timed(step_e2e, steps, 1, sample_clocks=False, kernel_times=False)
            out["e2e"] = {"value": m_step * steps / (e2e_ms * 1e-3), "unit": "candidates/s",
                          "h2d_bytes_per_step": int(m_local * d * 8), "d2h_bytes_per_step": (KSEEDS + 1) * 16,
                          "ms_per_step": e2e_ms / steps,
                          "api": "FusedAcquisition.argmin_topk(host ndarray (pageable), k) - the package's public call: finite "
                                 "check, H2D of the batch in chunks overlapped with the fused kernel + selection, D2H of the records"}
        out["_keep"] = (gp, acq, dev_bufs, host_bufs, X, y)
        out["_outputs"] = outputs
        return out

    cfg = CONFIGS[args.config]
    main_leg = run_config(cfg, args.steps, args.warmup)
    gp, acq, dev_bufs, host_bufs, X, y = main_leg.pop("_keep")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main_leg.pop("_outputs"))
    extra = {}

    if not args.no_extra and args.config == "c3":
        nx = min(args.steps, 3)
        # ---- fp32 mode (N^2 term as 3xTF32 on tcgen05), same workload, device leg + its own e2e ----------
        f32 = run_config(cfg, nx, 3, with_e2e=True, precision="fp32", sample_clocks=True)
        gp32, acq32, _, _, _, _ = f32.pop("_keep")
        extra["fp32"] = f32
        # ---- throughput mode: candidates generated in the kernel (Philox), fp32 + fp64 ----------------
        lo, hi = np.zeros(cfg["d"]), np.ones(cfg["d"])
        sel_p = torch.zeros((KSEEDS + 1, 2), dtype=torch.int64, device=dev)
        m_local = cfg["m_per_gpu"]
        thr = {}
        for name, a in (("fp32", acq32), ("fp64", acq)):
            sp = a.spec

            def step_philox(i, sp=sp):
                B.check(L.b200bo_acq_select_philox_dev(C.byref(sp), 12345 + i, B.as_dp(lo), B.as_dp(hi), m_local,
                                                       rank * m_local, KSEEDS, sel_p.data_ptr(), stream.cuda_stream))

            t_ms, k_ms, _, _ = timed(step_philox, nx, 2, sample_clocks=False)
            thr[name] = {"value": world * m_local * nx / (t_ms * 1e-3), "kernel_ms": float(np.mean(k_ms))}
        extra["throughput"] = thr
        # ---- host RNG cost of the parity mode (what makes a real suggest() RNG-bound in fp32 mode) -------
        if rank == 0:
            t0 = time.perf_counter()
            rs = np.random.RandomState(5)
            np.column_stack([rs.uniform(0.0, 1.0, 1 << 18) for _ in range(cfg["d"])])
            extra["host_rng_s_per_2pow20"] = 4 * (time.perf_counter() - t0)
        del gp32, acq32

    if not args.no_extra and args.config == "c3":
        # ---- BASELINE configs[4], strong scaling: 2^22 candidates in total over the ranks -----------------
        del dev_bufs, host_bufs
        torch.cuda.empty_cache()
        c5 = run_config(CONFIGS["c5"], 2, 1, with_e2e=False, sample_clocks=False)
        c5.pop("_keep")
        extra["c5"] = c5

    if not args.no_extra and args.config == "c3" and rank == 0:
        extra["other_configs"] = other_config_legs(bo, B, local_rank)
        try:
            extra["other_configs"]["c1_readme_n25_ucb_live"] = c1_live_leg(bo, local_rank)
        except Exception as e:  # a secondary leg never takes the headline line down (e.g. bayes_opt not importable)
            extra["other_configs"]["c1_readme_n25_ucb_live"] = {"error": repr(e)}

    fitleg = None
    if not args.no_extra and args.config == "c3" and rank == 0:
        try:
            fitleg = fit_and_suggest_legs(bo, cfg, X, y, local_rank)
        except Exception as e:  # e.g. bayes_opt not importable: the acquisition-seam legs cannot run
            fitleg = {"error": repr(e)}

    if rank == 0:
        emit(report(args, world, cfg, main_leg, extra, fitleg, X, y))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def other_config_legs(bo, B, device):
    """BASELINE configs[1] (C2: d=8, N=1024, EI, 2^20 candidates) and configs[3] (C4: d=16, N=2048, PoI x 2 constraint
    GPs, 2^19 candidates) through the public host call (pageable ndarray in, records out), 1 warm-up + 2 timed calls."""
    from sklearn.gaussian_process.kernels import Matern

    out = {}

    def gp_for(X, y, ls):
        return bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=ls), alpha=ALPHA, normalize_y=True,
                                               optimizer=None, device=device).fit(X, y)

    class Constraint:  # what FusedAcquisition reads of bayes_opt's ConstraintModel
        pass

    for tag, n, d, m, kind in (("c2_d8_n1024_ei", 1024, 8, 1 << 20, "ei"), ("c4_d16_n2048_poi_2constraints", 2048, 16, 1 << 19, "poi")):
        rs = np.random.RandomState(0)
        X = rs.uniform(size=(n, d))
        y = np.sin(X.sum(1)) + 0.1 * rs.randn(n)
        gp = gp_for(X, y, 0.7)
        if kind == "ei":
            acq = bo.FusedAcquisition(B.ACQ_EI, gp, xi=XI, y_max=float(y.max()))
            n_gps = 1
        else:
            c = np.column_stack([np.cos(X.sum(1)), np.sin(2 * X.sum(1))])
            con = Constraint()
            con.model = [gp_for(X, c[:, 0], 0.9), gp_for(X, c[:, 1], 0.5)]
            con.lb, con.ub = np.array([-np.inf, -0.5]), np.array([0.6, 0.5])
            ok = np.all((c >= con.lb) & (c <= con.ub), axis=1)
            acq = bo.FusedAcquisition(B.ACQ_POI, gp, con, xi=XI, y_max=float(y[ok].max()))
            n_gps = 3
        xt = np.random.RandomState(1).uniform(size=(m, d))
        acq.argmin_topk(xt[: m // 8], KSEEDS)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            idx, val, top = acq.argmin_topk(xt, KSEEDS)
            ts.append(time.perf_counter() - t0)
        dt = float(np.min(ts))
        out[tag] = {"candidates": m, "gps_per_candidate": n_gps, "seconds": dt, "value": m / dt, "unit": "candidates/s",
                    "roofline_frac_fp64": flops_per_candidate(n, d, n_gps) * m / dt / 1e12 / 37.13,
                    "argmin_index": int(idx), "api": "FusedAcquisition.argmin_topk(host ndarray, 10), wall clock incl. H2D"}
    return out


def c1_live_leg(bo, device):
    """BASELINE configs[0]: the README's 2-D black_box_function, Matern nu=2.5, UCB, maximize(init_points=5, n_iter=20)
    (N_train reaches 25) through the reference's own BayesianOptimization driver - stock (sklearn / SciPy on the host
    cores) and with enable() (every fit / suggest on the device).  Wall seconds of the whole loop; the enabled loop is
    run twice and the second run reported (the first pays the one-off allocations)."""
    import warnings

    from bayes_opt import BayesianOptimization

    def black_box(x, y):
        return -(x**2) - (y - 1) ** 2 + 1

    def run(enabled):
        opt = BayesianOptimization(f=black_box, pbounds={"x": (2, 4), "y": (-3, 3)}, random_state=1, verbose=0)
        if enabled:
            bo.enable(opt, device=device)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            t0 = time.perf_counter()
            opt.maximize(init_points=5, n_iter=20)
            dt = time.perf_counter() - t0
        return dt, opt

    run(True)
    t_dev, o_dev = run(True)
    t_ref, o_ref = run(False)
    p_dev, p_ref = o_dev.space.params, o_ref.space.params
    return {"what": "maximize(init_points=5, n_iter=20) of the README example through bayes_opt.BayesianOptimization, wall "
                    "seconds: enable()d (device) vs stock (host cores)",
            "seconds": t_dev, "seconds_reference_cpu": t_ref, "iterations": 20,
            "max_target": float(o_dev.max["target"]), "max_target_reference": float(o_ref.max["target"]),
            "max_abs_diff_of_probed_points": float(np.max(np.abs(p_dev - p_ref))) if p_dev.shape == p_ref.shape else None,
            "same_rng_state_after": bool(all(np.array_equal(a, b) for a, b in zip(
                o_dev._random_state.get_state()[1:3], o_ref._random_state.get_state()[1:3])))}


def fit_and_suggest_legs(bo, cfg, X, y, device):
    """Driver-visible numbers for the rest of suggest(): the hyper-parameter fit (1 + 5 L-BFGS-B runs on
    -LML, SK/_gpr.py:302-340) and a complete acquisition.suggest() without refit (10 000 candidates + 10
    lockstep L-BFGS-B refinements), both at N_train=4096 through the real bayes_opt classes."""
    import warnings

    from bayes_opt.target_space import TargetSpace
    from sklearn.gaussian_process.kernels import Matern

    out = {}
    d = cfg["d"]
    gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5), alpha=ALPHA, normalize_y=True, n_restarts_optimizer=5,
                                         random_state=np.random.RandomState(3), device=device)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gp.fit(X, y)  # warm-up (allocations)
        t0 = time.perf_counter()
        gp.fit(X, y)
        out["fit_s"] = time.perf_counter() - t0
    out["fit_theta"] = [float(t) for t in gp.kernel_.theta]
    k = gp.kernel_
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        gp.log_marginal_likelihood(k.theta, eval_gradient=True)
        ts.append(time.perf_counter() - t0)
    out["lml_grad_ms"] = 1e3 * float(np.median(ts))
    space = TargetSpace(None, {f"x{i:02d}": (0.0, 1.0) for i in range(d)})
    for xi_, yi_ in zip(X[:4], y[:4]):  # suggest() only needs a non-empty space; the GP keeps the full fit
        space.register(xi_, yi_)
    ei = bo.ExpectedImprovement(xi=XI)
    rs = np.random.RandomState(11)
    gp._ensure_device_fit()
    ts = []
    for _ in range(3):
        ei.y_max = float(y.max())
        t0 = time.perf_counter()
        acq = ei._get_acq(gp=gp)
        ei._acq_min(acq, space, random_state=rs, n_random=10_000, n_smart=10)
        ts.append(time.perf_counter() - t0)
    out["suggest_nofit_s"] = float(np.median(ts))
    return out


def report(args, world, cfg, leg, extra, fitleg, X, y):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    n, d = cfg["n"], cfg["d"]
    k_ms = leg["kernel_ms"]
    flops = flops_per_candidate(n, d) * leg["m_local"]
    fp64_nominal = 64 * 2 * 148 * (peaks.get("sm_max_mhz", 1965.0) * 1e6) / 1e12  # DFMA/clk/SM nominal
    fp64_peak, peak_src = fp64_nominal, ("nominal 64 FMA/clk/SM x 148 SM x sm_max_mhz (fp64 has no tcgen05 path; "
                                         "MEASURED_PEAKS.json has no fp64 entry)")
    try:
        mb = json.load(open(os.path.join(ROOT, "profiles", "r01_fp64_microbench.json")))
        fp64_peak = max(v for k, v in mb.items() if k.startswith("dmma"))
        peak_src = ("measured on this pool: best mma.sync f64 (DMMA) rate of tools/microbench.cu, "
                    "profiles/r01_fp64_microbench.json (nominal 37.2; MEASURED_PEAKS.json has no fp64 entry)")
    except Exception:
        pass
    ach_tf = flops / (k_ms * 1e-3) / 1e12
    hbm_bytes = hbm_model_bytes_per_candidate(n, d, 128) * leg["m_local"]
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic, traffic_src = ncu_traffic("predict_acq_kernel")
    line = base_line(args, world, cfg)
    line.update({
        "value": leg["value"], "ms_per_step": leg["ms_per_step"],
        "e2e": leg.get("e2e"),
        "gpu_launches": leg["launches"],
        "clocks": leg["clocks"],
        "roofline": {
            "bound": "tensor", "pipe": "fp64 tensor path: mma.sync m8n8k4 f64 (SASS DMMA; ncu "
            "sm__pipe_tensor_subpipe_dmma) - tcgen05.mma has no f64 kind",
            "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach_tf / fp64_peak,
            "frac_of_40tf_fallback": ach_tf / 40.0,
            "traffic": traffic, "traffic_source": traffic_src,
            "kernel": "predict_acq16_kernel (16-warp variant of predict_acq_kernel, the default)", "kernel_ms": k_ms,
            "peak_source": peak_src,
            "algorithmic_flops_per_candidate": flops_per_candidate(n, d),
            "hbm_model": {"achieved": hbm_bytes / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                          "frac": hbm_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak, "tile_T": 128,
                          "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6.65 TB/s"},
        },
        "fit_seconds_fixed_theta": leg["fit_s"],
        "result": leg["result"],
    })
    if "exchange_ms" in leg:
        line["exchange_ms"] = leg["exchange_ms"]
        line["kernel_ms_per_rank"] = leg.get("kernel_ms_per_rank")
    if "fp32" in extra:
        f = extra["fp32"]
        tf32_peak = peaks.get("bf16_tflops", 1590.0) / 2.0
        executed = 3.0 * n * n * f["m_local"] / (f["kernel_ms"] * 1e-3) / 1e12  # 3 TF32 products per multiply-add
        t32, t32_src = ncu_traffic("predict_acq_tc4_kernel")
        line["fp32_mode"] = {
            "what": "same workload, N^2 term as 3xTF32 on tcgen05 (fp32 accumulate in TMEM); K*, mean, epilogue fp64",
            "value": f["value"], "unit": "candidates/s", "e2e": f.get("e2e"), "kernel_ms": f["kernel_ms"],
            "tolerance": "1e-3 rel on the predictive variance (+1e-4 s_y^2 atol), tests/test_gpu_parity.py",
            "kernel": "predict_acq_tc4_kernel (N = 256 per tcgen05.mma, row-block pairs; B200BO_TC_VARIANT=2|3 select the earlier variants)", "clocks": f["clocks"],
            "roofline": {"bound": "tensor", "achieved": executed, "peak": tf32_peak, "unit": "TFLOP/s",
                         "frac": executed / tf32_peak, "traffic": t32, "traffic_source": t32_src,
                         "note": "executed TF32 tensor flops (3 products per useful multiply-add); dense TF32 peak "
                                 "taken as half the measured bf16 peak of MEASURED_PEAKS.json",
                         "useful_tflops": flops / (f["kernel_ms"] * 1e-3) / 1e12},
            "argmin_matches_fp64": f["result"]["argmin_index"] == leg["result"]["argmin_index"],
            "argmin_value": f["result"]["argmin_value"],
        }
    if "throughput" in extra:
        line["throughput_mode"] = {
            "what": "candidate_source=device_philox: the M candidates are generated inside the fused kernel (Philox4x32-10 "
                    "keyed by seed and global row index) - no host RNG, no H2D, nothing materialised; opt-in, does not "
                    "reproduce the reference's MT19937 stream",
            "unit": "candidates/s", "fp32": extra["throughput"]["fp32"], "fp64": extra["throughput"]["fp64"],
            "host_mt19937_seconds_per_2pow20x16": extra.get("host_rng_s_per_2pow20"),
        }
    if "c5" in extra:
        c = extra["c5"]
        c5cfg = CONFIGS["c5"]
        fl = flops_per_candidate(c5cfg["n"], c5cfg["d"]) * c["m_local"]
        line["c5_strong"] = {
            "what": c5cfg["label"], "scaling": "strong", "value": c["value"], "unit": "candidates/s",
            "ms_per_step": c["ms_per_step"], "kernel_ms": c["kernel_ms"], "candidates_per_rank": c["m_local"],
            "exchange_ms": c.get("exchange_ms"), "kernel_ms_per_rank": c.get("kernel_ms_per_rank"), "result": c["result"],
            "roofline_frac_fp64": fl / (c["kernel_ms"] * 1e-3) / 1e12 / fp64_peak,
            "note": "the candidate set is defined globally (blocks of 2^16 rows regenerated from (buffer, block) seeds), so "
                    "result.argmin_index must be identical for every --gpus N",
        }
    if "other_configs" in extra:
        line["other_configs"] = extra["other_configs"]
    if fitleg and "error" in fitleg:
        line["fit"] = fitleg
    elif fitleg:
        line["fit"] = {"what": "B200GaussianProcessRegressor.fit with 1+5 L-BFGS-B runs on -LML at N_train=4096, d=16 "
                               "(SK/_gpr.py:302-340), wall seconds", "seconds": fitleg["fit_s"],
                       "lml_plus_gradient_ms": fitleg["lml_grad_ms"], "theta": fitleg["fit_theta"]}
        line["suggest"] = {"what": "acquisition hooks of one suggest() without refit at N_train=4096: 10 000 candidates "
                                   "(device argmin+top-10) + 10 L-BFGS-B refinements in lockstep, wall seconds",
                           "seconds": fitleg["suggest_nofit_s"]}
    if world == 1 and not args.no_cpu_baseline and _REF_DIR is not None:
        v, secs = cpu_reference_rate(cfg, X, y, 1 << 14)
        line["cpu_baseline"] = {
            "value": v, "unit": "candidates/s", "cores": os.cpu_count(), "kind": "reference", "blas": blas_pools(),
            "sample": f"16384 candidates ({secs:.1f} s) through the vendored bayes_opt closure "
                      f"({cfg['acq'].upper()}._get_acq on a wrap_kernel GP) + argmin/argsort, chunks of 2^14"}
    return line


if __name__ == "__main__":
    main()
