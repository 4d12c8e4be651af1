#!/usr/bin/env python
"""Benchmark of the hist boosting hot path.  Contract: see the task statement ("Measurement").

    python bench.py --gpus 1 --steps 10 --warmup 3                 # CUDA path (default arm)
    python bench.py --impl reference --steps 3 --warmup 1          # the reference's CPU hist path (oracle port)
    torchrun ... bench.py --gpus N ...                             # rows sharded over N GPUs, NCCL hist all-reduce

metric  : boosting rounds/sec (BASELINE.json) on synthetic 50M x 100 reg:squarederror, 256 bins, max_depth 6.
step    : one boosting round (one tree) over the whole matrix.
value   : K / device time of K rounds, inputs resident in HBM (CUDA events on the engine stream, max over ranks).
e2e     : MEASURED: a whole 200-round job through the public API from pinned HOST buffers -- xgb.DMatrix(numpy) [H2D],
          xgb.train(..., evals=[(dtrain, "train")]) [cuts + binning + 200 x (update + eval with a D2H of the metric)] --
          wall clock, max over ranks; value = 200 / wall.  The ingest breakdown is reported beside it.
roofline: histogram-build kernel, root launch (all rows): algorithmic bytes rows*(F+8) / mean launch time measured with
          CUDA events inside the timed region, against MEASURED_PEAKS.json hbm_gbs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PROFILE_ROUNDS = 3


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=50_000_000)
    ap.add_argument("--cols", type=int, default=100)
    ap.add_argument("--objective", default="reg:squarederror")
    ap.add_argument("--num-class", type=int, default=0)
    ap.add_argument("--max-depth", type=int, default=6)
    ap.add_argument("--max-bin", type=int, default=256)
    ap.add_argument("--seed", type=int, default=43)
    ap.add_argument("--cpu-sample-rows", type=int, default=10_000_000, help="rows of the cpu_baseline leg of the default arm")
    ap.add_argument("--reference-rows", type=int, default=0, help="rows of the --impl reference arm (first blocks of the same generator); 0 = all rows: "
                    "the full 50M x 100 job takes ~3.7 s per round on 128 host threads, ~3.5 min for 5 + 20 rounds incl. generation, cuts and binning")
    ap.add_argument("--job-rounds", type=int, default=200)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-predict", action="store_true")
    ap.add_argument("--watchdog-seconds", type=int, default=1500, help="hard exit if the whole run takes longer (a hung collective must not eat the box)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed boosting rounds (the rounds/sec metric), write the model "
                    "they trained (every tree array, float32 / float64) as DIR/<name>.npy, so two builds can be compared on identical "
                    "seeded inputs; the e2e and predict sections are not dumped, and --impl reference does not take it")
    return ap.parse_args()


def params_of(a):
    p = {"objective": a.objective, "tree_method": "hist", "max_depth": a.max_depth, "max_bin": a.max_bin, "eta": 0.3, "lambda": 1.0,
         "gamma": 0.0, "min_child_weight": 1.0}
    if a.num_class > 1:
        p["num_class"] = a.num_class
    return p


BLOCK = 1_000_000


def gen_block_torch(block_id, rows, F, seed, objective, K, device):
    """SURVEY.md 8(d) recipe: x = N(0,1) quantised to 256 levels; y = x.beta + 0.1 eps (regression), per 1M-row block."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed * 100003 + block_id)
    x = torch.randn(rows, F, generator=g, device=device, dtype=torch.float32)
    x = torch.round(torch.clamp(x, -4.0, 4.0 - 1.0 / 32) * 32) / 32
    gb = torch.Generator(device=device)
    gb.manual_seed(seed)
    if objective.startswith("multi"):
        beta = torch.randn(F, K, generator=gb, device=device) / (F ** 0.5)
        y = torch.argmax(x @ beta + torch.randn(rows, K, generator=g, device=device), dim=1).float()
    else:
        beta = torch.randn(F, generator=gb, device=device) / (F ** 0.5)
        if objective.startswith("binary") or objective == "reg:logistic":
            z = x @ beta + 0.5 * torch.randn(rows, generator=g, device=device)
            y = (torch.sigmoid(z) > torch.rand(rows, generator=g, device=device)).float()
        else:
            y = x @ beta + 0.1 * torch.randn(rows, generator=g, device=device)
    return x, y


def gen_shard(a, r0, r1, device):
    import torch
    F = a.cols
    X = torch.empty((r1 - r0, F), device=device, dtype=torch.float32)
    y = torch.empty((r1 - r0,), device=device, dtype=torch.float32)
    b = r0 // BLOCK
    pos = r0
    while pos < r1:
        bs, be = b * BLOCK, min((b + 1) * BLOCK, a.rows)
        xb, yb = gen_block_torch(b, be - bs, F, a.seed, a.objective, max(a.num_class, 1), device)
        lo, hi = max(pos, bs), min(r1, be)
        X[lo - r0:hi - r0] = xb[lo - bs:hi - bs]
        y[lo - r0:hi - r0] = yb[lo - bs:hi - bs]
        pos = hi
        b += 1
    return X, y


class ClockSampler:
    """SM clock and throttle reasons sampled with NVML every ~5 ms during the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception as e:       # pragma: no cover
            self.err = str(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, reasons))
            except Exception as e:   # pragma: no cover
                self.err = str(e)
                return
            time.sleep(0.005)

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        self.stop_flag.set()
        self.thread.join(timeout=2)
        nv = self.nv
        mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80}
        seen = set()
        for _, r in self.samples:
            for k, bit in names.items():
                if r & bit:
                    seen.add(k)
        sm = [x for x, _ in self.samples]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(mx), "samples": len(sm), "reasons": sorted(seen)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_threads():
    """Threads the CPU arm uses: every core this process may run on (never inherited from OMP_NUM_THREADS: torchrun sets it to 1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def gen_host_sample(a, S):
    """First S rows of the workload, from the SAME generator and seed as the GPU arm (gen_block_torch, block by block)."""
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    xs, ys = [], []
    for b in range((S + BLOCK - 1) // BLOCK):
        rows = min(BLOCK, a.rows - b * BLOCK, S - b * BLOCK)
        xb, yb = gen_block_torch(b, min(BLOCK, a.rows - b * BLOCK), a.cols, a.seed, a.objective, max(a.num_class, 1), dev)
        xs.append(xb[:rows].cpu().numpy()); ys.append(yb[:rows].cpu().numpy())
    return np.ascontiguousarray(np.concatenate(xs)), np.ascontiguousarray(np.concatenate(ys)), str(dev.type)


def oracle_rounds_per_sec(a, Xs, ys, steps, warmup, threads):
    """Time the CPU restatement of the reference's hist path on a bounded sample with an explicit thread count."""
    from oracle import gbt_oracle as O
    O.set_num_threads(threads)
    t0 = time.time()
    cuts = O.make_cuts(Xs, a.max_bin)
    bins = O.bin_matrix(Xs, cuts[0], cuts[1])
    ingest = time.time() - t0
    tr = O.Trainer(dict(params_of(a), nthread=threads), bins=bins, cuts=cuts, y=ys)
    for _ in range(warmup):
        tr.update()
    t0 = time.time()
    for _ in range(steps):
        tr.update()
    dt = time.time() - t0
    return steps / dt, ingest, O.num_threads()


def run_reference(a):
    """--impl reference: the reference's own CPU hist implementation.  xgboost==3.0.5 is not installable in this image
    (no network, no wheel), so this arm times the oracle port of that path on the host cores: same generator and seed
    as the GPU arm, a stated row sample, an explicit thread count."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")
    threads = host_threads()
    S = a.rows if a.reference_rows <= 0 else min(a.rows, a.reference_rows)
    X, y, gen_dev = gen_host_sample(a, S)
    rps_sample, ingest_s, cores = oracle_rounds_per_sec(a, X, y, a.steps, a.warmup, threads)
    scale = S / a.rows
    value = rps_sample * scale
    sample = ("%s %d of %d rows of the GPU arm's workload (same generator and seed, generated on %s), %d timed rounds after %d warm-up, "
              "oracle port of the xgboost CPU hist path with %d OpenMP threads%s"
              % ("all" if S == a.rows else "first", S, a.rows, gen_dev, a.steps, a.warmup, cores,
                 "" if S == a.rows else "; rounds/s scaled linearly in rows (x %d/%d)" % (S, a.rows)))
    ingest_full = ingest_s / scale
    e2e = a.job_rounds / (ingest_full + a.job_rounds / value)
    print(json.dumps({
        "impl": "reference", "metric": "boosting rounds/sec", "value": value, "unit": "rounds/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "synthetic %dx%d %s hist max_bin=%d max_depth=%d" % (a.rows, a.cols, a.objective, a.max_bin, a.max_depth),
                   "params": params_of(a), "sample_rows": S, "sample_ms_per_step": 1000.0 / rps_sample},
        "cpu_baseline": {"value": value, "unit": "rounds/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": e2e, "unit": "rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def model_hash(be, bst):
    """sha256 over the trained trees (structure, thresholds, leaf values): identical at every GPU count by construction."""
    import hashlib
    m = be.booster_export_model(bst.handle)
    h = hashlib.sha256()
    for k in ("tree_offset", "tree_info", "left", "right", "split_index", "split_bin", "default_left", "split_cond"):
        h.update(np.ascontiguousarray(m[k]).tobytes())
    return h.hexdigest()[:16], int(len(m["tree_info"]))


def dump_outputs(be, bst, out_dir):
    """The booster as the timed rounds left it: tree arrays (ints as float64, exact) and the float32 node values."""
    os.makedirs(out_dir, exist_ok=True)
    m = be.booster_export_model(bst.handle)
    for k in ("tree_offset", "tree_info", "left", "right", "parent", "split_index", "split_bin", "default_left", "split_cond",
              "base_weight", "loss_chg", "sum_hess"):
        a = np.asarray(m[k])
        np.save(os.path.join(out_dir, k + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))
    np.save(os.path.join(out_dir, "base_score.npy"), np.array([m["base_score"]], np.float64))


def predict_section(xgb, be, device, peak):
    """BASELINE config 5 (second half of the metric: predict rows/sec): a 1M-row x 28 `text/csv` request body through the
    serving path the container's default handler takes -- csv_to_dmatrix (encoder.py:35-52, here parsed on the device) then
    serve_utils.predict -> Booster.predict (serve_utils.py:200-262) -- parse and predict reported separately; plus the predictor
    kernel alone against the HBM roofline and the container's own host parse timed on a row sample."""
    import io
    import torch
    from sagemaker_xgboost_container_b200 import serving
    n, F, rounds, reps = 1_000_000, 28, 50, 5
    X, y = gen_block_torch(7, n, F, 45, "binary:logistic", 1, device)
    bst = xgb.train({"objective": "binary:logistic", "tree_method": "hist", "max_depth": 6, "max_bin": 256, "eta": 0.3},
                    xgb.DMatrix(X, label=y.cpu().numpy()), num_boost_round=rounds, verbose_eval=False)
    Xn = X.cpu().numpy()
    import pandas as pd
    buf = io.StringIO()
    pd.DataFrame(Xn).to_csv(buf, header=False, index=False, float_format="%.6g")       # SURVEY.md 8(d) config 5: '%.6g', comma
    payload = buf.getvalue().strip().encode("utf-8")
    del buf
    # warm-up, then the request: parse (H2D of the text + device parse) and predict (kernel + transform + D2H) timed separately
    d = serving.csv_to_dmatrix(payload, dtype=float)
    p0 = serving.predict(bst, "xgb_format", d, "text/csv", objective="binary:logistic")
    t_parse, t_pred = [], []
    for _ in range(reps):
        be.synchronize(); t0 = time.perf_counter()
        d = serving.csv_to_dmatrix(payload, dtype=float)
        be.synchronize(); t1 = time.perf_counter()
        p = serving.predict(bst, "xgb_format", d, "text/csv", objective="binary:logistic")
        t2 = time.perf_counter()
        t_parse.append(t1 - t0); t_pred.append(t2 - t1)
    parse_s, pred_s = float(np.median(t_parse)), float(np.median(t_pred))
    kernel_ms = be.booster_predict_kernel_ms(bst.handle, d.handle, 10)
    # the container's own host route (str.split + np.array(...).astype(float)) on a 50k-row sample of the same payload
    sample = b"\n".join(payload.split(b"\n", 50_000)[:50_000]).decode("utf-8")
    t0 = time.perf_counter()
    ref = serving._host_csv_to_array(sample, ",", float)
    host_parse_s = time.perf_counter() - t0
    same = bool(np.array_equal(be.dmatrix_get_raw(d.handle).reshape(n, F)[:50_000], ref.astype(np.float32)))
    direct = bst.predict(xgb.DMatrix(X))
    leaves = bst.predict(d, pred_leaf=True)
    alg = n * F * 4 + n * 4
    return {"workload": "default-handler path on a %d x %d text/csv body (%.0f MB, '%%.6g'), binary:logistic, %d trees depth 6" % (n, F, len(payload) / 1e6, rounds),
            "value": n / (parse_s + pred_s), "unit": "rows/s", "parse_s": parse_s, "predict_s": pred_s,
            "parse_rows_per_s": n / parse_s, "parse_text_gbs": len(payload) / parse_s / 1e9, "predict_rows_per_s": n / pred_s,
            "host_parse_reference": {"rows": 50_000, "seconds": host_parse_s, "rows_per_s": 50_000 / host_parse_s,
                                     "what": "encoder.csv_to_dmatrix's own str.split + np.array(...).astype(float) on the first 50k rows of the same body"},
            "roofline": {"bound": "hbm", "kernel": "predict_tiled_kernel", "achieved": alg / (kernel_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (kernel_ms * 1e-3) / 1e9 / peak, "ms_per_launch": kernel_ms,
                         "note": "kernel alone (CUDA events, 10 launches); 50 trees x depth 6 = 300 node visits per 112 B row make it issue-bound, not HBM-bound"},
            "e2e": {"value": n / (parse_s + pred_s), "unit": "rows/s", "h2d_bytes_per_step": int(len(payload)), "d2h_bytes_per_step": int(p.nbytes)},
            "consistent": bool(np.array_equal(p, p0) and same and np.allclose(p, direct, rtol=0, atol=1e-6)), "pred_leaf_shape": list(leaves.shape)}


def main():
    a = parse_args()
    if a.watchdog_seconds > 0:
        def _bail():
            sys.stderr.write("bench.py: watchdog fired after %d s, exiting\n" % a.watchdog_seconds)
            sys.stderr.flush()
            os._exit(3)
        wd = threading.Timer(a.watchdog_seconds, _bail)
        wd.daemon = True
        wd.start()
    if a.impl == "reference":
        if a.dump_outputs:
            sys.exit("bench.py: --dump-outputs applies to the CUDA path (--impl b200) only")
        run_reference(a)
        return
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import collective
    be = xgb.get_backend()
    dist = None
    if world > 1:
        import torch.distributed as dist
        collective.init_from_env(backend="gloo")

    def barrier():
        torch.cuda.synchronize()
        be.synchronize()
        if dist is not None:
            dist.barrier()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    r0, r1 = rank * a.rows // world, (rank + 1) * a.rows // world
    X, y = gen_shard(a, r0, r1, device)
    y_host = y.cpu().numpy()
    dtrain = xgb.DMatrix(X, label=y_host)
    params = params_of(a)
    bst = xgb.Booster(params, [dtrain])
    it = 0
    for _ in range(a.warmup):
        bst.update(dtrain, it); it += 1
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = be.launch_count()
    barrier()
    be.timer_start()
    t_host0 = time.perf_counter()
    for _ in range(a.steps):
        bst.update(dtrain, it); it += 1
    host_ms = (time.perf_counter() - t_host0) * 1e3 / a.steps       # CPU time to ENQUEUE a round (graph launches + collectives)
    ms = be.timer_stop()
    barrier()
    launches = be.launch_count() - l0
    clk = clocks.stop() if rank == 0 else None
    ms = max_over_ranks(ms)
    mhash, mtrees = model_hash(be, bst)           # after warm-up + timed rounds: the same trees at every N
    if a.dump_outputs and rank == 0:
        dump_outputs(be, bst, a.dump_outputs)
    # per-kernel CUDA-event timing of the histogram launches: the timed region above replays a CUDA graph per tree, so the
    # events bracket the same launches issued directly for PROFILE_ROUNDS further rounds right after it (same state, same data)
    be.booster_set_profile(bst.handle, True)
    t_prof0 = time.perf_counter()
    for _ in range(PROFILE_ROUNDS):
        bst.update(dtrain, it); it += 1
    prof = be.booster_get_profile(bst.handle)
    prof_ms = (time.perf_counter() - t_prof0) * 1e3 / PROFILE_ROUNDS
    be.booster_set_profile(bst.handle, False)
    value = a.steps / (ms / 1000.0)

    # ---- roofline of the histogram kernel (root launch = one full pass over this rank's rows)
    peak, peak_src = hbm_peak()
    F = a.cols
    root_ms = prof["root_hist_ms"] / max(1, prof["root_hist_launches"])
    root_rows = prof["root_hist_rows"] / max(1, prof["root_hist_launches"])
    root_bytes = root_rows * (F + 8)
    achieved = root_bytes / (root_ms * 1e-3) / 1e9 if root_ms > 0 else 0.0
    deep_bytes = prof["deep_hist_rows"] * (F + 8 + 4)          # deeper levels also read a 4 B row id per row
    all_gbs = (prof["root_hist_rows"] * (F + 8) + deep_bytes) / ((prof["root_hist_ms"] + prof["deep_hist_ms"]) * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_hist_root_traffic.json")
    if os.path.exists(tp) and world == 1:
        tj = json.load(open(tp))
        if tj.get("workload") == "synthetic %dx%d" % (a.rows, a.cols):
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]      # per launch, from the committed ncu capture
    roofline = {"bound": "hbm", "kernel": "hist_root_kernel<G-only> (root launch, all rows of the rank; constant-hessian objective: H plane cached)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "bytes_per_launch": root_bytes, "ms_per_launch": root_ms,
                "all_hist_launches_gbs": all_gbs, "all_hist_launches_frac": all_gbs / peak,
                "hist_share_of_step": (prof["root_hist_ms"] + prof["deep_hist_ms"]) / PROFILE_ROUNDS / (ms / a.steps),
                "timing": "CUDA events around each hist launch over %d rounds run right after the timed region (direct launches; the timed region replays CUDA graphs)" % PROFILE_ROUNDS}

    # ---- end to end through the public API with host buffers: a whole job, measured
    e2e = None
    if not a.no_e2e:
        del dtrain, bst
        Xh = torch.empty(X.shape, dtype=torch.float32, pin_memory=True)
        Xh.copy_(X)
        del X
        torch.cuda.empty_cache()
        Xn = Xh.numpy()
        barrier()
        t0 = time.perf_counter()
        d2 = xgb.DMatrix(Xn, label=y_host)                       # H2D of the feature matrix happens here
        be.synchronize()
        t_h2d = time.perf_counter() - t0
        res = {}
        b2 = xgb.train(params, d2, num_boost_round=a.job_rounds, evals=[(d2, "train")], evals_result=res, verbose_eval=False)
        be.synchronize()
        t_job = time.perf_counter() - t0
        barrier()
        t_job = max_over_ranks(t_job); t_h2d = max_over_ranks(t_h2d)
        last = list(res["train"].items())[0]
        e2e = {"value": a.job_rounds / t_job, "unit": "rounds/s", "h2d_bytes_per_step": int(Xn.nbytes + y_host.nbytes) // a.job_rounds,
               "d2h_bytes_per_step": 16, "job_rounds": a.job_rounds, "job_wall_s": t_job,
               "ingest": {"h2d_s": t_h2d, "cuts_bin_and_rounds_s": t_job - t_h2d, "est_rounds_s": a.job_rounds * (ms / a.steps) / 1000.0},
               "last_eval": "[%d]\ttrain-%s:%.17g" % (a.job_rounds - 1, last[0], last[1][-1]),
               "note": "measured wall clock of xgb.DMatrix(pinned host numpy) + xgb.train(%d rounds, evals=[train]) incl. H2D, cuts, binning and the per-round metric D2H" % a.job_rounds}
        del d2, b2

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        # the CPU leg runs as its own process (the reference arm on a smaller sample): OpenMP thread binding must be in the
        # environment before libgomp starts, and must NOT be in the environment of the GPU ranks (it would pin every
        # rank's launching thread onto the same core)
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1", "--rows", str(a.rows), "--cols", str(a.cols),
               "--objective", a.objective, "--num-class", str(a.num_class), "--max-depth", str(a.max_depth), "--max-bin", str(a.max_bin), "--seed", str(a.seed),
               "--reference-rows", str(min(a.rows, a.cpu_sample_rows)), "--watchdog-seconds", "600"]
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS")}
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
        try:
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception:
            cpu = {"value": None, "unit": "rounds/s", "cores": 0, "kind": "port", "sample": "cpu leg failed: %s" % (r.stderr[-300:] or r.stdout[-300:])}

    predict = None
    if rank == 0 and world == 1 and not a.no_predict:
        predict = predict_section(xgb, be, device, peak)

    if rank == 0:
        out = {
            "metric": "boosting rounds/sec", "value": value, "unit": "rounds/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": "synthetic %dx%d %s hist max_bin=%d max_depth=%d" % (a.rows, a.cols, a.objective, a.max_bin, a.max_depth),
                       "rows_per_gpu": (a.rows + world - 1) // world, "parallelism": "rows sharded x%d, per-level int64 histogram NCCL all-reduce" % world,
                       "l2": "inputs (%.1f GB of bins per GPU) exceed the 126 MB L2" % ((r1 - r0) * 32 * ((a.cols + 31) // 32) / 1e9),
                       "arithmetic": "f32 gradients rounded to a 2^-k fixed-point grid, int32 shared-memory partial sums, int64 histograms (exact), f64/f32 split gains",
                       "rounds_timed": "rounds %d..%d of a fresh booster (the rows of the built children shrink from ~50 %% to ~23 %% of N per level over the first rounds)" % (a.warmup, a.warmup + a.steps - 1),
                       "params": params},
            "gpu_launches": launches, "clocks": clk, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu, "predict": predict,
            "model_hash": mhash, "model_trees": mtrees, "host_enqueue_ms_per_step": host_ms,
        }
        print(json.dumps(out))
    if dist is not None:
        collective.finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
