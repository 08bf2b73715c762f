#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json: AGD iters/sec & examples/sec on logistic
10M x 1024 dense fp32 (configs[1]), 1/2/4/8 B200, next to the reference's path on the host cores.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  ... --dump-outputs DIR     also writes the weights and loss history of the timed run as DIR/<name>.npy

A "step" is one outer AGD iteration (AGD.scala:237-332) = the reference's 3 + 2b applySmooth evaluations
(flags = 0: every evaluation is executed; the history evaluation of :304 shares one sweep over X with the next
iteration's applySmooth(y), see `fused_passes` / `sweeps` / `unfused` in the output).  `value` = examples/sec =
total rows x evaluations executed / time, shards resident in HBM when the timed region starts.  `e2e` is the same metric through
the public call with HOST buffers: the shard upload from pinned host memory (what `.cache()` pays),
the run, and the results coming back are all inside its timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "AGD examples/sec (rows x applySmooth passes / s), logistic 10M x 1024 dense fp32"
SEED = 42


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--workload", default="logistic_f32", choices=["logistic_f32", "ls_bf16", "hinge_csr"],
                    help="logistic_f32 = BASELINE configs[1] (the metric; also configs[4] with --rows 100000000 --dim 512); "
                         "ls_bf16 = configs[3] shape (--rows 50000000 --dim 4096); hinge_csr = configs[2] shape "
                         "(--rows 100000000 --dim 1000000 --nnz 64)")
    ap.add_argument("--nnz", type=int, default=64, help="stored entries per row for hinge_csr")
    ap.add_argument("--collective", default="auto", choices=["auto", "nccl", "p2p"],
                    help="all-reduce of the d+4 doubles: NVLink peer-memory exchange (default when mappable) or NCCL")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the bounded CPU sample (0 = 4M, the same at every N)")
    ap.add_argument("--store", default="f32", choices=["f32", "bf16", "f64"],
                    help="HBM storage of the logistic_f32 workload; bf16 is the stated substitute that lets the 100M x 512 "
                         "shape of configs[4] fit ONE GPU (204.8 GB as fp32); f64 is what the Scala facade stores by default "
                         "(arbitrary Double features kept exact)")
    ap.add_argument("--parity-iters", type=int, default=10,
                    help="iterations of the full-size oracle comparison reported as `parity` (0 = off; on by default for "
                         "fp32 logistic workloads whose host copy is <= 64 GB)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed run returned (weights, loss history) as "
                         "DIR/<name>.npy in float64, so that two builds can be compared output for output")
    return ap.parse_args()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy in float64.  An array larger than its share of DUMP_BYTES is replaced by the
    same seeded sample of its entries on every run, so that dumps of two builds stay comparable entry for entry."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        if a.nbytes > share:
            a = a[np.sort(np.random.default_rng(SEED).choice(a.size, share // a.itemsize, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(rows_local: int, d: int):
    """dram bytes per K1 launch from the committed ncu capture, scaled to this launch's rows."""
    try:
        with open(os.path.join(ROOT, "profiles", "k1_traffic.json")) as f:
            t = json.load(f)
        if t["d"] != d:
            return None
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["rows"] * rows_local
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(gpu_index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [ln.split(", ") for ts, ln in self.lines if t0 - 0.05 <= ts <= t1 + 0.15] or \
               [ln.split(", ") for _, ln in self.lines]
        rows = [r for r in rows if len(r) >= 9]
        if not rows:
            return None
        sm = sorted(float(r[1]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[5 + k].strip().lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": reasons,
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}


# ------------------------------------------------------------------------------------ reference arm
CPU_KEYS = ("value", "unit", "cores", "kind", "sample", "runs_seconds", "host_threads", "cgroup_cpu_quota",
            "thread_calibration_examples_per_sec")
CPU_SAMPLE_ROWS = 4_000_000     # the bounded sample is the same at every N (VERDICT r1: the arm must be reproducible)


def cpu_sample_rows(args) -> int:
    return max(1000, min(args.cpu_rows or CPU_SAMPLE_ROWS, args.rows))


def cgroup_cpu_quota():
    """CPUs the container's cgroup lets it use (cpu.max quota / period), or None when unlimited / unknown."""
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] == "max":
                    return None
                return float(txt[0]) / float(txt[1])
            q = float(txt[0])
            if q <= 0:
                return None
            return q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().split()[0])
        except (OSError, ValueError, IndexError):
            continue
    return None


_CALIB = {}


def calibrate_threads(d: int, rows: int):
    """(fastest thread count, {threads: examples/s}, candidates) for the oracle's fold on this host; cached per d."""
    from oracle import oracle as O
    if d in _CALIB:
        return _CALIB[d]
    ncpu = O.host_threads()
    quota = cgroup_cpu_quota()
    cands = sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4)} | ({max(1, min(ncpu, int(quota + 0.999)))} if quota else set()),
                   reverse=True)
    w0 = np.zeros(d)
    calib = {}
    cal_rows = max(1000, min(rows, 1_000_000))
    best_t, best_v = cands[0], -1.0
    if len(cands) > 1 and rows >= 100_000:
        for T in cands:
            O.bind_threads(T)
            try:
                X = O.synth_dense_f32_placed(SEED, 0, cal_rows, d, T, T)
                y = O.synth_labels(SEED, "logistic", 0, X, O.synth_wtrue(SEED, d))
                D = O.Data(y, X=X)
                O.agd_run(D, "logistic", "simple", w0, convergence_tol=0.0, num_iterations=1, partitions=T, threads=T)
                t0 = time.perf_counter()
                r = O.agd_run(D, "logistic", "simple", w0, convergence_tol=0.0, num_iterations=1, partitions=T, threads=T)
                v = cal_rows * r.passes / (time.perf_counter() - t0)
            finally:
                O.unbind_threads()
            calib[str(T)] = v
            if v > best_v:
                best_t, best_v = T, v
            del X, D
    _CALIB[d] = (best_t, calib, cands)
    return _CALIB[d]


def cpu_reference(rows: int, d: int, steps: int, warmup: int, repeats: int = 3):
    """Times the reference's CPU path (the oracle port: treeAggregate-shaped fp64 fold, one partition per host thread)
    on a bounded sample of the same workload.  Reproducibility: thread count from the affinity mask (torchrun exports
    OMP_NUM_THREADS=1), every OpenMP thread pinned to one CPU, the sample generated by the thread that folds it (first
    touch => NUMA-local), and the median of `repeats` timed runs.  "All the host threads it can use": on these boxes the
    fold stops scaling well before the 128 hardware threads (shared host: memory bandwidth / cgroup CPU share), so a short
    calibration times the thread counts {all, one per physical core, quarter, cgroup quota} on a slice of the sample and
    the measurement uses the FASTEST -- the strongest CPU baseline this host gives, with the all-threads figure beside it."""
    from oracle import oracle as O
    ncpu = O.host_threads()
    quota = cgroup_cpu_quota()
    w0 = np.zeros(d)
    best_t, calib, cands = calibrate_threads(d, rows)
    cores = best_t
    O.bind_threads(cores)
    try:
        X = O.synth_dense_f32_placed(SEED, 0, rows, d, cores, cores)     # first `rows` rows of the workload
        y = O.synth_labels(SEED, "logistic", 0, X, O.synth_wtrue(SEED, d))
        D = O.Data(y, X=X)
        kw = dict(convergence_tol=0.0, partitions=cores, threads=cores)
        if warmup > 0:
            O.agd_run(D, "logistic", "simple", w0, num_iterations=warmup, **kw)
        runs = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            r = O.agd_run(D, "logistic", "simple", w0, num_iterations=steps, **kw)
            runs.append(time.perf_counter() - t0)
    finally:
        O.unbind_threads()
    dt = sorted(runs)[len(runs) // 2]
    return {"value": rows * r.passes / dt, "unit": "examples/s", "cores": cores, "kind": "port",
            "sample": f"first {rows} rows of the workload x {steps} AGD iterations ({r.passes} passes), median of "
                      f"{repeats} timed runs, {cores} partitions on {cores} pinned threads (fastest of the calibrated thread "
                      f"counts {cands} on this {ncpu}-thread host), first-touch placement, fp32 rows upcast to fp64",
            "host_threads": ncpu, "cgroup_cpu_quota": quota, "thread_calibration_examples_per_sec": calib,
            "seconds": dt, "runs_seconds": runs, "iters_per_sec": r.iterations / dt, "passes": r.passes, "rows": rows,
            "weights": r.weights, "loss_history": r.loss_history}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = cpu_sample_rows(args)
    steps = args.steps
    warm = 1 if args.warmup > 0 else 0
    res = cpu_reference(rows, args.dim, steps, warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"weights": res["weights"], "loss_history": res["loss_history"]})
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "examples/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": res["seconds"] / steps * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"logistic-loss AGD, {args.rows} x {args.dim} dense fp32 (BASELINE configs[1])",
                   "sample_rows": rows, "note": "staple/spark-agd needs a JVM + Spark 1.3.0 (absent): this arm times the "
                   "repo's C restatement of its treeAggregate path (oracle/), an optimistic stand-in"},
        "iters_per_sec": res["iters_per_sec"],
        "cpu_baseline": {k: res[k] for k in CPU_KEYS},
        "e2e": {"value": res["value"], "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    import spark_agd_b200 as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ctx = S.Context.from_torch_distributed(local)
    else:
        ctx = S.Context(devices=[local])
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node = --gpus"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    d = args.dim
    total_rows = args.rows * (world if args.scaling == "weak" else 1)
    wl = args.workload
    reg = 0.0
    if wl == "logistic_f32":
        store = args.store
        grad, upd, eb = S.LogisticGradient(), S.SimpleUpdater(), {"f32": 4, "bf16": 2, "f64": 8}[store]
        data = ctx.synthetic(total_rows, d, grad, seed=SEED, store=store)     # K0: never timed
    elif wl == "ls_bf16":
        grad, upd, store, eb = S.LeastSquaresGradient(), S.SimpleUpdater(), "bf16", 2
        data = ctx.synthetic(total_rows, d, grad, seed=SEED, store=store)
    else:
        grad, upd, store, eb, reg = S.HingeGradient(), S.SquaredL2Updater(), "f32", 4, 0.1
        data = ctx.synthetic_csr(total_rows, d, args.nnz, grad, seed=SEED, store=store)
    rows_local = data.local_rows(0)
    w0 = np.zeros(d)
    if args.collective != "auto":
        data.set_option("collective", args.collective)
    headline = wl == "logistic_f32" and store == "f32"
    if not headline:
        args.no_e2e = True
        args.no_cpu_baseline = True
    parity_iters = args.parity_iters if (headline and total_rows * d * 4 <= (64 << 30)) else 0

    def run(ds, iters, memoize=False, fuse=True):
        return S.run_with_stats(ds, grad, upd, 0.0, iters, reg, w0, memoize=memoize, fuse=fuse)

    # ---- warm-up, then EXACTLY K timed steps, barrier + synchronize on both sides
    barrier()
    if args.warmup > 0:
        run(data, args.warmup)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    t0 = time.time()
    w, hist, st = run(data, args.steps)
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1) if sampler else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"weights": w, "loss_history": hist})
    dev_s = max_over_ranks(st.device_ms_total / 1e3)
    value = total_rows * st.passes / dev_s
    # the bit-identical memoised pass structure (AGD_FLAG_MEMOIZE_FX), reported beside the headline; like the headline it gets
    # its own warm-up (it runs other kernel instantiations: the two-gradient sweep)
    barrier()
    if args.warmup > 0:
        run(data, args.warmup, memoize=True)
    barrier()
    w_m, hist_m, st_m = run(data, args.steps, memoize=True)
    memo_same = bool(np.array_equal(w_m, w) and np.array_equal(hist_m, hist))
    dev_s_m = max_over_ranks(st_m.device_ms_total / 1e3)
    # every evaluation as a sweep of its own (AGD_FLAG_NO_FUSE): the same results bit for bit, one more read of X per iteration
    barrier()
    if args.warmup > 0:
        run(data, args.warmup, fuse=False)
    barrier()
    _, hist_u, st_u = run(data, args.steps, fuse=False)
    dev_s_u = max_over_ranks(st_u.device_ms_total / 1e3)
    same_bits = bool(np.array_equal(hist_u, hist))   # expected on dense shards (CSR sums are atomics: equal to rounding only)

    # ---- roofline of the dominant kernel (K1), CUDA events on its own stream inside the timed region
    peak, peak_src = peaks()
    k1_ms = st.k1_ms_total / max(st.k1_launches, 1)
    k1_ms_single = st_u.k1_ms_total / max(st_u.k1_launches, 1)          # one point per sweep
    n_two = st.fused_passes
    k1_ms_two = (st.k1_ms_total - (st.k1_launches - n_two) * k1_ms_single) / n_two if n_two else None
    if wl == "hinge_csr":
        alg_bytes = rows_local * (args.nnz * (4 + eb) + 16)   # idx + value per entry, rowptr + label per row
    else:
        alg_bytes = rows_local * (d * eb + 8)     # stored row + fp64 label, per launch (DESIGN.md)
    achieved = alg_bytes / (k1_ms * 1e-3) / 1e9
    kname = data.kernel_name()                      # the K1 kernel this shard actually dispatches to
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(rows_local, d) if headline else None,
                "peak_source": peak_src, "bytes_per_launch": alg_bytes, "ms_per_launch": k1_ms,
                "launches": int(st.k1_launches), "two_point_launches": int(n_two),
                "ms_per_launch_one_point": k1_ms_single, "ms_per_launch_two_point": k1_ms_two,
                "frac_one_point": alg_bytes / (k1_ms_single * 1e-3) / 1e9 / peak,
                "k1_share_of_step": st.k1_ms_total / st.device_ms_total}

    # ---- e2e: public call with HOST buffers; shard upload + run + results inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(S, ctx, data, rows_local, total_rows, d, args, run, barrier, max_over_ranks, world)

    # ---- parity on the FULL workload (every N): the same loop on the GPU path and on the oracle, same rows
    parity = None
    if parity_iters > 0:
        parity = measure_parity(S, data, run, parity_iters, total_rows, rows_local, d, rank, world, barrier)

    # ---- CPU baseline: the oracle port on the host cores, bounded sample, rank 0 at N = 1 only
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        res = cpu_reference(cpu_sample_rows(args), d, 2, 1)
        cpu = {k: res[k] for k in CPU_KEYS}

    if rank == 0:
        wl_text = {"logistic_f32": f"logistic-loss AGD, {total_rows} x {d} dense {dict(f32='fp32', bf16='bf16 storage', f64='fp64 storage')[store]} "
                                   f"({'BASELINE configs[1]' if (total_rows, d) == (10_000_000, 1024) else 'BASELINE configs[4] shape'}), "
                                   f"SimpleUpdater, w0 = 0, convergenceTol 0, defaults L0=1 beta=.5 alpha=.9 restart",
                   "ls_bf16": f"least-squares AGD, {total_rows} x {d} dense bf16 storage (BASELINE configs[3] shape), kernel {kname}",
                   "hinge_csr": f"hinge-loss + L2 (reg 0.1) AGD, {total_rows} x {d} CSR, {args.nnz} stored entries per "
                                f"row (BASELINE configs[2] shape)"}[wl]
        line = {
            "metric": METRIC if (headline and total_rows == 10_000_000 and d == 1024) else
            f"AGD examples/sec (rows x applySmooth passes / s), {wl} {total_rows} x {d} store {store}", "value": value, "unit": "examples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_s / args.steps * 1e3, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl_text,
                       "rows": total_rows, "d": d, "store": store, "rows_per_gpu": rows_local,
                       "parallelism": f"row shards x{world}, one all-reduce of d+4 fp64 per sweep",
                       "accounting": "value = rows x applySmooth evaluations / s (the reference's unit of work, 3 + 2b per "
                                     "iteration, AGD.scala:250,269,304); `fused_passes` of them shared a sweep over X with the next "
                                     "iteration's first evaluation, `sweeps` is the number of reads of X, `physical_examples_per_sec` "
                                     "counts those reads instead; `unfused` runs every evaluation as its own sweep",
                       "l2": "inputs larger than L2: every pass streams the whole shard "
                             f"({alg_bytes / 1e9:.2f} GB) from HBM"},
            "iters_per_sec": st.iterations / dev_s, "passes": st.passes, "passes_per_iter": st.passes / st.iterations,
            "fused_passes": int(st.fused_passes), "sweeps": int(st.k1_launches),
            "physical_examples_per_sec": total_rows * st.k1_launches / dev_s,
            "backtracks": st.backtracks, "restarts": st.restarts, "final_loss": float(hist[-1]),
            "unfused": {"iters_per_sec": st_u.iterations / dev_s_u, "examples_per_sec": total_rows * st_u.passes / dev_s_u,
                        "sweeps": int(st_u.k1_launches), "loss_history_bit_identical_to_fused": same_bits,
                        "note": "AGD_FLAG_NO_FUSE: same weights and history bit for bit, 3 + 2b reads of X per iteration"},
            "memoized": {"iters_per_sec": st_m.iterations / dev_s_m, "passes_per_iter": st_m.passes / st_m.iterations,
                         "examples_per_sec": total_rows * st_m.passes / dev_s_m, "sweeps": int(st_m.k1_launches),
                         "fused_passes": int(st_m.fused_passes), "wasted_passes": int(st_m.wasted_passes),
                         "weights_and_history_bit_identical_to_default": memo_same,
                         "k1_ms_per_launch": st_m.k1_ms_total / max(st_m.k1_launches, 1),
                         "allreduce_ms_per_pass": st_m.allreduce_ms_total / max(st_m.collective_calls, 1),
                         "device_ms": dev_s_m * 1e3, "host_wall_ms": st_m.seconds_total * 1e3,
                         "note": "AGD_FLAG_MEMOIZE_FX: same weights and history bit for bit, fewer passes"},
            "allreduce_ms_per_pass": st.allreduce_ms_total / max(st.collective_calls, 1),
            "host_wall_s": st.seconds_total, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity,
            "gpu_launches": int(st.gpu_launches), "collective_calls": int(st.collective_calls),
            "collective": ("none" if world == 1 else ("nvlink peer-memory exchange" if st.collective_kind == 1 else "nccl all-reduce")),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    data.close()
    if world > 1:
        dist.destroy_process_group()


def measure_parity(S, data, run, iters, total_rows, rows_local, d, rank, world, barrier):
    """north_star's acceptance line on the metric's own configuration: `iters` iterations of the same loop on the GPU
    path (all ranks, the shards already resident) and on the oracle (rank 0, all host threads) over the SAME total_rows
    rows; weights (AGD.scala:337) and the whole loss history (:304-306) compared.  The oracle's rows come from the CPU
    twin of the on-device generator (bit-identical by construction, tests/test_synth_spec.py); every rank re-checks
    that claim on the head and the tail of its own shard as downloaded from HBM, and the labels are the ones the GPUs
    hold.  Partition order: the oracle folds `cores` contiguous partitions in order, the GPUs fold CTA slabs and then
    ranks in order -- both are AGD.scala:201-204 combOp orders, different roundings of the same sums."""
    import torch
    import torch.distributed as dist
    from oracle import oracle as O
    barrier()
    w_g, hist_g, st_g = run(data, iters)
    # every rank: (a) its shard's head / tail rows against the twin at the shard's global offset, (b) its labels
    row_lo = (rank * total_rows) // world
    chk = min(1024, rows_local)
    ok = 1
    if chk > 0:
        for r0 in (0, rows_local - chk):
            xs, _ = data.get_rows(0, r0, chk)
            ok &= int(np.array_equal(xs, O.synth_dense_f32(SEED, row_lo + r0, chk, d)))
    y_loc = data.get_labels(0, 0, rows_local)
    if world > 1:
        t_ok = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        ok = int(t_ok.item())
        sizes = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([rows_local], dtype=torch.int64, device="cuda"))
        sizes = [int(t.item()) for t in sizes]
        pad = torch.zeros(max(sizes), dtype=torch.float64, device="cuda")
        pad[:rows_local] = torch.from_numpy(y_loc).cuda()
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad)
        y = np.concatenate([p[:n].cpu().numpy() for p, n in zip(parts, sizes)]) if rank == 0 else None
    else:
        y = y_loc
    out = None
    if rank == 0:
        cores = calibrate_threads(d, total_rows)[0]          # the thread count this host folds fastest with
        O.bind_threads(cores)
        try:
            t0 = time.perf_counter()
            X = O.synth_dense_f32_placed(SEED, 0, total_rows, d, cores, cores)
            t_gen = time.perf_counter() - t0
            t0 = time.perf_counter()
            ref = O.agd_run(O.Data(y, X=X), "logistic", "simple", np.zeros(d), convergence_tol=0.0, num_iterations=iters,
                            partitions=cores, threads=cores)
            t_ref = time.perf_counter() - t0
        finally:
            O.unbind_threads()
        del X
        n = min(len(hist_g), len(ref.loss_history))
        loss_err = float(np.max(np.abs(hist_g[:n] - ref.loss_history[:n]) / np.abs(ref.loss_history[:n]))) if n else None
        out = {"rows": int(total_rows), "d": int(d), "iters": int(iters), "n_gpus": int(world),
               "w_rel_err": float(np.linalg.norm(w_g - ref.weights) / np.linalg.norm(ref.weights)),
               "w_max_abs_err": float(np.max(np.abs(w_g - ref.weights))),
               "max_loss_rel_err": loss_err, "history_len_equal": bool(len(hist_g) == len(ref.loss_history)),
               "passes_equal": bool(st_g.passes == ref.passes), "backtracks_equal": bool(st_g.backtracks == ref.backtracks),
               "restarts_equal": bool(st_g.restarts == ref.restarts), "passes": int(st_g.passes),
               "final_loss_gpu": float(hist_g[-1]), "final_loss_oracle": float(ref.loss_history[-1]),
               "shards_equal_cpu_twin": bool(ok), "tolerance": "north_star: weights within 1e-5 relative after equal iterations",
               "pass": bool(ok and len(hist_g) == len(ref.loss_history) and
                            np.linalg.norm(w_g - ref.weights) / np.linalg.norm(ref.weights) <= 1e-5 and (loss_err or 0) <= 1e-9),
               "oracle": {"cores": cores, "partitions": cores, "seconds": t_ref, "generate_seconds": t_gen,
                          "examples_per_sec": total_rows * ref.passes / t_ref,
                          "note": "the FULL workload on the host: every row, all threads (not the bounded sample of cpu_baseline)"}}
    barrier()
    return out


def measure_e2e(S, ctx, data, rows_local, total_rows, d, args, run, barrier, max_over_ranks, world):
    import torch
    shard_bytes = rows_local * d * 4
    pinned = True
    try:
        hostX = torch.empty((rows_local, d), dtype=torch.float32, pin_memory=True)
        hosty = torch.empty((rows_local,), dtype=torch.float64, pin_memory=True)
    except RuntimeError:
        pinned = False
        hostX = torch.empty((rows_local, d), dtype=torch.float32)
        hosty = torch.empty((rows_local,), dtype=torch.float64)
    Xn, yn = hostX.numpy(), hosty.numpy()
    chunk = max(1, (256 << 20) // (d * 4))
    for r0 in range(0, rows_local, chunk):               # stage the caller's host copy (not timed)
        rc = min(chunk, rows_local - r0)
        xs, ys = data.get_rows(0, r0, rc)
        Xn[r0:r0 + rc] = xs
        yn[r0:r0 + rc] = ys
    ds = data.unpersist()                                # same context (devices + communicator), empty shards
    barrier()
    t0 = time.perf_counter()
    ds.load_dense(yn, Xn, store="f32")                   # the call a user makes: cache host rows, optimise
    w, hist, st = run(ds, args.steps)
    barrier()
    dt = max_over_ranks(time.perf_counter() - t0)
    return {"value": total_rows * st.passes / dt, "unit": "examples/s", "seconds": dt,
            "h2d_bytes_per_step": (shard_bytes + rows_local * 8 + d * 8) / args.steps,
            "d2h_bytes_per_step": (d * 8 + len(hist) * 8) / args.steps + st.passes / args.steps * 64,
            "iters_per_sec": st.iterations / dt, "pinned_host": pinned,
            "what": f"agd_load_dense of the {shard_bytes / 1e9:.2f} GB fp32 shard from {'pinned' if pinned else 'pageable'} "
                    f"host memory + agd_run({args.steps} iterations) + weights/history back, per rank, wall clock max over ranks"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
