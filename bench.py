#!/usr/bin/env python
"""Headline benchmark: block least-squares fit throughput (samples/s) on BASELINE.json config 3
(CosineRandomFeatures 440 -> D = 16 x 4096 = 65536, BlockLeastSquaresEstimator(4096, numIter=1, lambda=1), k = 1000,
N = 1M rows sharded over the GPUs of one node; strong scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one complete fit over the whole batch, ending with the fitted model (all W_j, feature means, intercept) in
host memory.  The top-level `value` / `e2e` are measured in the PARITY mode (split operands: rel-Frobenius(W) <= 5e-5 against the
fp64 oracle, the tolerance the tests state); `fast_mode` carries the same two numbers for the fp16-operand mode (10-bit
mantissa, rel-Fro ~ 7e-4), and `parity` the accuracy of both modes measured in this very process on a row subsample.
`value` = N_total / (time per step) with the inputs resident in HBM; `e2e` = the same fit through the public API starting
from pinned HOST buffers (H2D of X and the class labels inside the timed region; the model lands in pinned host memory through
async copies while the fit runs) -- DESIGN.md section 7.
`--impl reference` times the CPU stand-in for the reference (the numpy/OpenBLAS fp64 oracle: the reference's own
Spark/Breeze path needs a JVM that this image does not have) on a bounded row sample of the same workload.
"""
from __future__ import annotations

import os
import sys

# BLAS threads must be chosen before numpy loads OpenBLAS; torchrun exports OMP_NUM_THREADS=1 to every rank.  Rank 0 runs
# the CPU legs (reference arm, cpu_baseline, the oracle of the parity check) on all host cores.
if int(os.environ.get("RANK", "0")) == 0:
    _cores = str(os.cpu_count() or 1)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = _cores

import argparse
import json
import subprocess
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "block-LS fit samples/sec (N=1M, D=64K, k=1K)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-rows", type=int, default=1_000_000)
    ap.add_argument("--d-in", type=int, default=440)
    ap.add_argument("--num-rf", type=int, default=16)
    ap.add_argument("--block", type=int, default=4096)
    ap.add_argument("--classes", type=int, default=1000)
    ap.add_argument("--lam", type=float, default=1.0)
    ap.add_argument("--num-iter", type=int, default=1)
    ap.add_argument("--gamma", type=float, default=0.0555)
    ap.add_argument("--cpu-rows", type=int, default=32768, help="largest row sample of the CPU baseline (SURVEY 8d: N_cpu = 32768)")
    ap.add_argument("--cpu-seconds", type=float, default=60.0, help="time budget of one CPU sample; the row count is cut to fit")
    ap.add_argument("--parity-rows", type=int, default=8192, help="rows of the in-process parity check (0: skip)")
    ap.add_argument("--parity-blocks", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fast-mode", action="store_true")
    ap.add_argument("--precision", default=os.environ.get("KS_BENCH_PRECISION", "f16x2"), choices=["tf32", "f16", "f16x2"],
                    help="operand mode of the top-level numbers (fp32 accumulate, fp64 solve in every mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the model fitted by the last timed step of the top-level mode to DIR/*.npy "
                         "(fp64; the weights as a fixed, seeded row sample, at most 64 MB in all), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ----------------------------------------------------------------------------------------- workload
def make_params(args, seed: int = 2):
    prm = np.random.default_rng(seed)
    params = [(prm.standard_normal((args.block, args.d_in)) * args.gamma, prm.random(args.block) * 2 * np.pi)
              for _ in range(args.num_rf)]
    wstar = prm.standard_normal((16, args.classes)).astype(np.float32)
    return params, wstar


def make_workload(args, lo: int, hi: int, seed: int = 2):
    """Synthetic config-3 inputs for global rows [lo, hi): X ~ N(0,1) fp32, labels planted through a fixed
    16-dim linear map + noise (SURVEY.md 8d), CosineRandomFeatures parameters shared by all ranks."""
    params, wstar = make_params(args, seed)
    rng = np.random.default_rng([seed, lo])
    X = rng.standard_normal((hi - lo, args.d_in), dtype=np.float32)
    scores = X[:, :16] @ wstar + 0.1 * rng.standard_normal((hi - lo, args.classes), dtype=np.float32)
    cls = np.argmax(scores, axis=1).astype(np.int32)
    return X, cls, params


def alg_flops(n, d_in, D, b, k, nb, num_iter=1):
    """SURVEY.md 8d: Gram 2NDb (full-GEMM convention) + A^T R 2NDk + update 2NDk + projection 2 N d_in D + solves."""
    first = 2.0 * n * D * b + 4.0 * n * D * k + 2.0 * n * d_in * D + nb * (b ** 3 / 3.0 + 2.0 * b * b * k)
    more = (num_iter - 1) * (4.0 * n * D * k + 2.0 * n * d_in * D + nb * 2.0 * b * b * k)
    return first + more


DUMP_BYTES = 64_000_000


def dump_model(model, out_dir: str, seed: int = 0) -> dict:
    """Writes what a caller of the fit receives: the feature means (D) and the intercept (k) whole, and the weights W (D x k,
    524 MB at config 3) as the rows at a fixed, seeded, sorted sample of row indices, as many as fit the 64 MB budget.
    Returns {file name: shape}."""
    xs = model.xs
    d, k = sum(w.shape[0] for w in xs), xs[0].shape[1]
    means = np.concatenate(model.feature_means)
    header = 4 * 128                                                    # one .npy header per file, the index file included
    n_rows = min(d, (DUMP_BYTES - header - means.nbytes - 8 * k) // (8 * (k + 1)))
    rows = np.sort(np.random.default_rng(seed).choice(d, size=n_rows, replace=False))
    offs = np.cumsum([0] + [w.shape[0] for w in xs])
    blk = np.searchsorted(offs, rows, side="right") - 1
    arrays = {"W_sample": np.stack([xs[j][r - offs[j]] for j, r in zip(blk, rows)]),
              "W_sample_rows": rows.astype(np.float64),
              "feature_means": means,
              "intercept": np.array(model.b_opt)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
    return {name: list(a.shape) for name, a in arrays.items()}


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, gpu_index: int):
        self.gpu_index, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index),
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------- CPU stand-in
def cpu_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return os.cpu_count() or 1, model


def _oracle_block_pass(ko, Xs, Y, params, args, n_blocks, with_solve):
    """The oracle's per-block arithmetic on `n_blocks` blocks: features, centring, Gram, A^T R, [solve,] residual update.
    Returns (seconds without the solves, seconds of the solves)."""
    t_solve = 0.0
    t0 = time.perf_counter()
    resid = Y - Y.mean(axis=0)
    for W, b in params[:n_blocks]:
        A = ko.cosine_random_features(Xs, W, b)         # block i == feature map i (b_out == blockSize)
        A -= A.mean(axis=0)
        G = A.T @ A
        C = A.T @ resid
        if with_solve:
            ts = time.perf_counter()
            dW = ko._solve_spd(G + args.lam * np.eye(G.shape[0]), C)
            t_solve += time.perf_counter() - ts
        else:
            dW = C * (1.0 / (np.trace(G) / G.shape[0] + args.lam))   # same shapes downstream, no factorisation
        resid -= A @ dW
    return time.perf_counter() - t0 - t_solve, t_solve


def cpu_baseline_record(args, nb, D, budget_s=None):
    """numpy/OpenBLAS fp64 oracle arithmetic on the host cores.  The b x b solves do not depend on N: they are timed once (two
    blocks, scaled to all nb -- identical shapes); the per-row cost is timed on all nb blocks of a row sample that is as
    large as the time budget allows (<= --cpu-rows = 32768, SURVEY 8d).  value = N / (per_row * N + solves)."""
    from oracle import keystone_oracle as ko
    budget_s = args.cpu_seconds if budget_s is None else budget_s
    cores, cpu_model = cpu_info()
    Xall, cls_all, params = make_workload(args, 0, args.cpu_rows)
    Xd = Xall.astype(np.float64)
    Yall = ko.class_label_indicators(cls_all, args.classes)
    _oracle_block_pass(ko, Xd[:1024], Yall[:1024], params, args, 1, True)            # warm the BLAS threads
    # pilot: 2 blocks on 4096 rows -> rows per second of the GEMM part, and the solve time
    pilot_rows = min(4096, args.cpu_rows)
    t_rows, t_solve2 = _oracle_block_pass(ko, Xd[:pilot_rows], Yall[:pilot_rows], params, args, 2, True)
    t_solve = t_solve2 / 2.0 * nb
    est_per_row = t_rows / 2.0 * nb / pilot_rows
    rows = args.cpu_rows
    while rows > 2048 and est_per_row * rows > budget_s:
        rows //= 2
    t_gemm, _ = _oracle_block_pass(ko, Xd[:rows], Yall[:rows], params, args, nb, False)
    per_row = t_gemm / rows
    full = args.n_rows / (per_row * args.n_rows + t_solve)
    gemm_flops = rows * (2.0 * D * args.block + 4.0 * D * args.classes + 2.0 * args.d_in * D)
    return {"value": full, "unit": "samples/s", "cores": cores, "cpu": cpu_model, "kind": "port",
            "blas_threads": os.environ.get("OPENBLAS_NUM_THREADS"),
            "sample": f"first {rows} rows x all {nb} blocks (D={D}, k={args.classes}) for the per-row cost ({t_gemm:.1f} s, "
                      f"{gemm_flops / t_gemm / 1e12:.2f} TFLOP/s fp64); the N-independent {args.block}^2 LU solves timed on 2 blocks and "
                      f"scaled to {nb} ({t_solve:.1f} s); numpy/OpenBLAS fp64 oracle -- the Spark/Breeze reference itself needs a JVM (absent)",
            "sample_rows": rows, "seconds": t_gemm + t_solve2, "per_row_seconds": per_row, "solve_seconds": t_solve,
            "gemm_tflops_fp64": gemm_flops / t_gemm / 1e12,
            "how": "value = N / (per_row_seconds * N + solve_seconds) at the benchmark's N"}


# ----------------------------------------------------------------------------------------- main
def main():
    # keep stdout to the one JSON line: NCCL prints a version banner there when NCCL_DEBUG is VERSION (or unset on some builds)
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    D = args.num_rf * args.block
    nb = args.num_rf
    mode_names = {"f16x2": "split fp16 operands hi+lo (parity mode)", "f16": "fp16 operands (fast mode)", "tf32": "tf32 operands"}
    config = {"workload": f"C3 CosineRandomFeatures({args.d_in}->{args.block})x{args.num_rf} + BlockLeastSquaresEstimator",
              "n_rows": args.n_rows, "d_in": args.d_in, "d": D, "k": args.classes, "block_size": args.block,
              "num_iter": args.num_iter, "lambda": args.lam, "parallelism": f"rows x{world}",
              "l2": "inputs larger than L2 (X 1.76 GB, slab 8-16 GB per block)",
              "precision": f"{mode_names[args.precision]}, fp32 accumulate, fp64 solve"}

    if args.impl == "reference":
        if rank != 0:
            return
        t_all = time.perf_counter()
        n_meas = max(1, args.steps)
        budget = max(10.0, min(args.cpu_seconds, 150.0 / n_meas))     # the whole run stays within a few minutes
        recs = [cpu_baseline_record(args, nb, D, budget) for _ in range(n_meas)]
        sps = float(np.mean([r["value"] for r in recs]))
        rec = dict(recs[-1]); rec["value"] = sps
        rec["values_per_step"] = [r["value"] for r in recs]
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": sps,
                          "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * args.n_rows / sps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                          "dtype": "f64", "data": "synthetic", "config": dict(config, precision="fp64 (numpy/OpenBLAS)"),
                          "cpu_baseline": rec, "wall_seconds": time.perf_counter() - t_all,
                          "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    import keystone_b200 as ks

    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        ctx = ks.Context.from_torch_distributed(local_rank)
    else:
        ctx = ks.Context(local_rank)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(local_rank)
        ctx.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lo, hi = ks.shard_range(args.n_rows, rank, world)
    X, cls, params = make_workload(args, lo, hi)
    Xp = torch.from_numpy(X).pin_memory()          # pinned host buffers for the e2e leg
    cp = torch.from_numpy(cls).pin_memory()
    rfs = [ks.CosineRandomFeatures(ctx, W, b) for W, b in params]

    def feats_of(x, maps=None):
        return ks.Pipeline.gather(rfs if maps is None else rfs[:maps]).andThen(ks.VectorCombiner())(x)

    def touch(model):
        """The fitted model as host arrays (views of the pinned mirror the fit filled while it ran); returns their bytes."""
        xs, mus, b = model.xs, model.feature_means, model.b_opt
        _ = float(xs[-1][-1, -1]) + float(b[-1])
        return sum(w.nbytes for w in xs) + sum(m.nbytes for m in mus) + b.nbytes

    # ---- kernel-only leg: inputs resident in HBM, model on the host at the end of every step
    x_dev = ctx.matrix(Xp.numpy())
    y_dev = ctx.labels_from_classes(cp.numpy(), args.classes)
    feats = feats_of(x_dev)

    def resident_leg(precision, steps, warmup, sample_clocks, keep_last=False):
        est = ks.BlockLeastSquaresEstimator(args.block, args.num_iter, args.lam, precision=precision)
        for _ in range(warmup):
            touch(est.fit(feats, y_dev))
        sampler = ClockSampler(local_rank) if sample_clocks else None
        barrier()
        if sampler:
            sampler.start()
        l0 = ctx.launch_count()
        stats, step_wall, last = [], [], None
        t0 = time.perf_counter()
        for i in range(steps):
            ts = time.perf_counter()
            if keep_last and i == steps - 1:
                last = est.fit(feats, y_dev)
                touch(last)
            else:
                touch(est.fit(feats, y_dev))
            step_wall.append(1e3 * (time.perf_counter() - ts))
            stats.append(ctx.last_fit_stats())
        barrier()
        t = max_over_ranks((time.perf_counter() - t0) / steps)
        return {"t": t, "launches": (ctx.launch_count() - l0) // max(steps, 1), "clocks": sampler.stop() if sampler else None,
                "dev_ms": max_over_ranks(float(np.mean([s["total_ms"] for s in stats]))), "step_wall": step_wall, "stats": stats[-1],
                "model": last}

    main_leg = resident_leg(args.precision, args.steps, args.warmup, True, keep_last=args.dump_outputs is not None)
    last_model, dumped = main_leg.pop("model"), None
    if last_model is not None and rank == 0:                 # every rank holds the same model
        dumped = dump_model(last_model, args.dump_outputs)
    del last_model
    fast_leg = None
    if args.precision != "f16" and not args.no_fast_mode:
        fast_leg = resident_leg("f16", args.steps, args.warmup, False)

    # ---- dominant kernel alone (same launch shape as inside the fit: S^T [S | R], N_loc x 4096 slab, k columns),
    #      CUDA events on the launching stream, 3 warm-up + 5 timed launches (inside the fit other streams' small kernels
    #      interleave with it, so an in-fit span would not isolate the kernel)
    import ctypes as C
    from keystone_b200._capi import check, lib
    sa = ctx.synthetic_normal(hi - lo, args.block, 11, lo)
    sb = ctx.synthetic_normal(hi - lo, args.classes, 12, lo)
    ms = C.c_double(0)
    ctx.set_option("precision", 0 if args.precision == "tf32" else 1)   # the debug entry converts the operands to fp16 first
    check(ctx.handle, lib().ks_debug_time_gram(ctx.handle, sa.handle, sb.handle, 3, C.byref(ms)))
    check(ctx.handle, lib().ks_debug_time_gram(ctx.handle, sa.handle, sb.handle, 5, C.byref(ms)))
    ctx.set_option("precision", 2)
    gram_ms = max_over_ranks(ms.value)
    del sa, sb

    # ---- parity of both modes vs the fp64 oracle, in this process: a row subsample (sharded over the ranks like the real
    #      fit, so the collectives are exercised at every N), the first `parity_blocks` feature maps, all k classes
    parity = None
    if args.parity_rows > 0:
        pb = min(args.parity_blocks, args.num_rf)
        plo, phi = ks.shard_range(args.parity_rows, rank, world)
        Xs, cls_s, _ = make_workload(args, 0, args.parity_rows, seed=7)
        xs_dev = ctx.matrix(Xs[plo:phi])
        ys_dev = ctx.labels_from_classes(cls_s[plo:phi], args.classes)
        fs = feats_of(xs_dev, pb)
        got = {}
        for prec in dict.fromkeys([args.precision, "f16"]):
            m = ks.BlockLeastSquaresEstimator(args.block, args.num_iter, args.lam, precision=prec).fit(fs, ys_dev)
            got[prec] = (np.concatenate(m.xs, 0).copy(), m.b_opt.copy(), m(fs).to_numpy() if world == 1 else None)
        if rank == 0:
            from oracle import keystone_oracle as ko
            t0 = time.perf_counter()
            Xd = Xs.astype(np.float64)
            blocks = [ko.cosine_random_features(Xd, W, b) for W, b in params[:pb]]
            Yd = ko.class_label_indicators(cls_s, args.classes)
            xs_o, b_o, mus_o = ko.block_ls_fit(None, Yd, args.block, args.num_iter, args.lam, feature_blocks=blocks)
            Wr = np.concatenate(xs_o, 0)
            ref = sum((blk - mu) @ w for blk, mu, w in zip(blocks, mus_o, xs_o)) + b_o
            parity = {"n_rows": args.parity_rows, "blocks": pb, "d": pb * args.block, "k": args.classes, "world": world,
                      "oracle": "numpy fp64 restatement (oracle/keystone_oracle.py), same arrays", "oracle_seconds": None, "modes": {}}
            for prec, (Wg, bg, pred) in got.items():
                rec = {"rel_fro_W": float(np.linalg.norm(Wg - Wr) / np.linalg.norm(Wr)), "max_abs_W": float(np.abs(Wg - Wr).max()),
                       "max_abs_intercept": float(np.abs(bg - b_o).max())}
                if pred is not None:
                    rec["max_abs_pred"] = float(np.abs(pred - ref).max())
                    rec["argmax_agree"] = float((pred.argmax(1) == ref.argmax(1)).mean())
                parity["modes"][prec] = rec
            parity["oracle_seconds"] = time.perf_counter() - t0
        del xs_dev, ys_dev, fs
        barrier()

    # ---- end-to-end leg: pinned host buffers -> public API -> fitted model on the host
    def e2e_leg(precision, steps):
        est = ks.BlockLeastSquaresEstimator(args.block, args.num_iter, args.lam, precision=precision)

        def step():
            xd = ctx.matrix(Xp.numpy())                                   # H2D of this rank's rows
            yd = ctx.labels_from_classes(cp.numpy(), args.classes)        # H2D of the int32 class ids
            return touch(est.fit(feats_of(xd), yd))                       # model: async D2H into pinned memory during the fit
        step()
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(steps):
            d2h = step()
        barrier()
        t = max_over_ranks((time.perf_counter() - t0) / steps)
        return {"value": args.n_rows / t, "unit": "samples/s", "ms_per_step": 1e3 * t,
                "h2d_bytes_per_step": int(X.nbytes + cls.nbytes), "d2h_bytes_per_step": int(d2h)}

    e2e = e2e_fast = None
    if not args.no_e2e:
        del feats, x_dev, y_dev
        e2e = e2e_leg(args.precision, args.steps)
        if fast_leg is not None:
            e2e_fast = e2e_leg("f16", args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (gram2_tn_kernel), timed alone with CUDA events (above)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = peaks.get("bf16_tflops") or 1700.0
    peak_src = ("MEASURED_PEAKS.json bf16_tflops (burst: the kernel is timed alone)" if peaks else
                "fallback 1.7 PFLOP/s dense bf16 burst (B200_PROFILING.md)")
    n_loc = hi - lo
    gram_launch_flops = 2.0 * n_loc * args.block * (args.block + args.classes)          # full-GEMM convention, per launch
    achieved = gram_launch_flops / (gram_ms * 1e-3) / 1e12
    executed = None
    if args.block == 4096 and args.classes == 1000:
        executed = achieved * (104 * 256 * 512) / (args.block * (args.block + args.classes))   # 72 G + 32 C pair tiles of 256 x 512
    traffic, traffic_ref = None, None
    try:
        traffic_ref = json.load(open(os.path.join(ROOT, "profiles", "gram_ncu_summary.json")))
        if traffic_ref.get("n_rows") == n_loc:
            traffic = traffic_ref.get("dram_bytes_per_launch")
    except (OSError, ValueError):
        pass
    kind = "kind::tf32" if args.precision == "tf32" else "kind::f16"
    roofline = {"kernel": f"gram2_tn_kernel (tcgen05 cta_group::2 {kind}, S^T [S | R])", "bound": "tensor", "achieved": achieved,
                "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "executed_tflops": executed, "executed_frac": executed / peak if executed else None,
                "note": "achieved = ALGORITHMIC flops 2*N_loc*b*(b+k) per launch (full-GEMM convention of the reference cost model, "
                        "SURVEY 8d) / mean launch duration; the kernel skips the lower triangle of G, so executed MMA flops are "
                        "0.65x of that: executed_tflops / executed_frac are the figures to hold against the tensor peak (the tf32 "
                        "MMA rate is half the bf16 / fp16 rate)",
                "ms_per_launch": gram_ms, "traffic_reference_capture": traffic_ref}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_record(args, nb, D)

    flops = alg_flops(args.n_rows, args.d_in, D, args.block, args.classes, nb, args.num_iter)
    st = main_leg["stats"]
    t = main_leg["t"]
    out = {"metric": METRIC, "value": args.n_rows / t, "unit": "samples/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t,
           "device_ms_per_step": main_leg["dev_ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": args.precision, "data": "synthetic", "config": config, "clocks": main_leg["clocks"],
           "gpu_launches": int(main_leg["launches"]), "step_wall_ms": main_leg["step_wall"],
           "alg_tflops": flops / t / 1e12, "executed_tflops_step": st.get("local_flops", 0) * world / t / 1e12,
           "phase_ms": {k: st[k] for k in st if k.endswith("_ms")}, "fit": {k: st[k] for k in ("mma", "pipeline", "solve", "host_mirror") if k in st},
           "model_on_host": "every step ends with all W_j, feature means and the intercept in pinned host memory (SURVEY 8d)",
           "roofline": roofline}
    if e2e:
        out["e2e"] = e2e
    if fast_leg is not None:
        tf = fast_leg["t"]
        out["fast_mode"] = {"dtype": "f16", "precision": mode_names["f16"], "value": args.n_rows / tf, "unit": "samples/s",
                            "ms_per_step": 1e3 * tf, "device_ms_per_step": fast_leg["dev_ms"], "steps": args.steps, "warmup": args.warmup,
                            "alg_tflops": flops / tf / 1e12, "gpu_launches": int(fast_leg["launches"]),
                            "phase_ms": {k: fast_leg["stats"][k] for k in fast_leg["stats"] if k.endswith("_ms")}}
        if e2e_fast:
            out["fast_mode"]["e2e"] = e2e_fast
    if parity:
        out["parity"] = parity
    if dumped:
        out["dumped_outputs"] = {"dir": args.dump_outputs, "arrays": dumped}
    if cpu_baseline:
        out["cpu_baseline"] = cpu_baseline
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
