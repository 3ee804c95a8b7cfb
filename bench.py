#!/usr/bin/env python
"""Headline benchmark: training ratings/s of the autoencoder hot path on synthetic data.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload ml10m] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of `batch_size` rows (train.py:30: 128):
K1 gather -> K2 encoder -> K3 decoder + masked loss + gradient -> K4 fused backward/optimizer.
A "rating" is one stored rating of the batch's rows (each is read, split into input/target by its
keep flag and consumed by the step).

  value  device-timed (CUDA events) over K steps whose row ids and keep flags are already
         resident in HBM; the working set (weights + optimizer state + store) is far larger than
         L2 for the default workload, so no explicit flush is needed (config.l2 says which)
  e2e    the same K steps through the public API (`data_reader.data_gen` -> `model.train_on_batch`):
         host RNG replay + pinned staging + H2D of row ids/flags + kernels + D2H of the metrics,
         every step, wall-clock between device synchronisations
  roofline       per-kernel CUDA-event times of a third, instrumented pass; the dominant kernel's
                 algorithmic bytes / time against MEASURED_PEAKS.json
  cpu_baseline   the oracle port of the reference (per-rating Python batch loop + dense NumPy
                 model step) on the host cores, bounded sample
`--impl reference` times that CPU port alone as the reference arm.
"""
from __future__ import annotations

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

WORKLOADS = {
    # BASELINE.json configs / SURVEY.md section 8(d). reverse=True: rows are items, columns users.
    "ml1m": dict(shape="ml1m", reverse=True, layers=1, hidden=500, act="sigmoid", aux=None, sparsity=[1.0, 1.0],
                 pass_through=True, opt=("adagrad", 0.005), dropout=0.2, aux_value=-1),
    "jester": dict(shape="jester", reverse=False, layers=2, hidden=256, act="tanh", aux="causal", sparsity=[0.5, 0.5],
                   pass_through=False, opt=("rmsprop", 0.001), dropout=None, aux_value=1),
    "ml10m": dict(shape="ml10m", reverse=True, layers=1, hidden=512, act="sigmoid", aux="dropout", sparsity=[0.5, 0.5],
                  pass_through=False, opt=("adagrad", 0.005), dropout=0.2, aux_value=-1),
    "ml10m_users": dict(shape="ml10m", reverse=False, layers=1, hidden=512, act="sigmoid", aux="dropout",
                        sparsity=[0.5, 0.5], pass_through=False, opt=("adagrad", 0.005), dropout=0.2, aux_value=-1),
    "ml20m": dict(shape="ml20m", reverse=False, layers=2, hidden=[1000, 500], act="sigmoid", aux=None,
                  sparsity=[0.5, 0.5], pass_through=False, opt=("adagrad", 0.005), dropout=0.2, aux_value=-1),
    "netflix": dict(shape="netflix", reverse=True, layers=1, hidden=1000, act="sigmoid", aux=None, sparsity=[1.0, 1.0],
                    pass_through=True, opt=("adagrad", 0.005), dropout=0.2, aux_value=-1),
    "small": dict(shape="small", reverse=True, layers=1, hidden=64, act="sigmoid", aux=None, sparsity=[1.0, 1.0],
                  pass_through=True, opt=("adagrad", 0.005), dropout=0.2, aux_value=-1),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak_tf32():
    """Dense tf32 peak in TFLOP/s: kind::tf32 runs at half the bf16 rate (K = 8 instead of 16 per
    tcgen05.mma of the same duration), so it is derived from the measured cuBLAS bf16 burst figure."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["bf16_tflops"]) / 2.0, "measured bf16 burst / 2 (MEASURED_PEAKS.json)"
    return 1590.0 / 2.0, "fallback bf16 / 2 (B200_PROFILING.md)"


def scoring_run(lib, m, rd, w, aux, rows, reps, warm, dump_dir=None):
    """Full-catalogue scoring (train.py:239 `predict` without the mask multiply) of `rows`
    validation rows per call: device-timed with the scores left in HBM, then end to end through
    `model.score` (host row ids in, [rows, N] float32 out). `dump_dir`: the last timed call's scores
    go there (write_outputs)."""
    import ctypes as C
    import torch
    from omnidirectional_collaborative_filtering_b200 import _lib
    rows = min(rows, rd.val_set_size)
    gen = rd.data_gen(rows, None, "valid", True, aux, w["aux_value"])
    batches = []
    while len(batches) < 4:
        b = next(gen)
        if b is None:
            if not batches:
                raise RuntimeError("validation set smaller than one scoring batch")
            break
        batches.append(b)
    h = m._ensure(rows, max(b.n_entries for b in batches), aux, rd)
    from omnidirectional_collaborative_filtering_b200.store import DeviceBatch
    devs = []
    for b in batches:
        d = DeviceBatch(b.n_rows, b.n_entries)
        d.fill_fixed(b.source, b.rows, b.aux_value, None)
        devs.append(d)
    N = m.owner.local_cols
    out = torch.empty((rows, N), dtype=torch.float32, device="cuda")
    optr = C.c_void_p(out.data_ptr())

    def run(n, first=0):
        for k in range(n):
            d = devs[(first + k) % len(devs)]
            _lib.check(lib.ocf_batch_regather(d.handle, None))
            _lib.check(lib.ocf_score(h, d.handle, optr, 1, None))

    run(warm)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.ocf_kernel_launches()
    e0.record()
    run(reps)
    e1.record()
    torch.cuda.synchronize()
    launches = lib.ocf_kernel_launches() - l0
    ms = e0.elapsed_time(e1) / reps
    if dump_dir is not None:
        write_outputs(dump_dir, {"scores": out.cpu().numpy()})
    lib.ocf_profile_reset()
    lib.ocf_profile_enable(1)
    run(reps)
    torch.cuda.synchronize()
    lib.ocf_profile_enable(0)
    tot, cnt = C.c_double(), C.c_int64()
    _lib.check(lib.ocf_profile_read(4, C.byref(tot), C.byref(cnt)))
    gemm_ms = tot.value / max(cnt.value, 1)
    H = w["hidden"] if isinstance(w["hidden"], int) else w["hidden"][-1]
    hp = (H + 127) // 128 * 128
    flops = 2.0 * rows * hp * N                        # the padded contraction the tensor cores run
    peak, src = tensor_peak_tf32()
    # end to end: host batch -> scores in a host array, every call
    m.score(batches[0], reuse_output=True)            # allocates the page-locked destination (untimed)
    t0 = time.perf_counter()
    n_e2e = max(2, min(reps, 5))
    for k in range(n_e2e):
        res = m.score(batches[k % len(batches)], reuse_output=True)     # page-locked destination
    e2e_s = (time.perf_counter() - t0) / n_e2e
    # top-k serving (k = 100, seen items excluded): selection on the device, k pairs per row back
    m.recommend(batches[0], k=100)
    t0 = time.perf_counter()
    for k in range(n_e2e):
        top_cols, top_scores = m.recommend(batches[k % len(batches)], k=100, exclude_seen=True)
    topk_s = (time.perf_counter() - t0) / n_e2e
    return {"rows_per_call": rows, "n_cols": int(N), "value": rows / (ms * 1e-3), "unit": "rows/s", "ms_per_call": ms,
            "topk": {"k": 100, "e2e_value": rows / topk_s, "unit": "rows/s", "ms_per_call": 1e3 * topk_s,
                     "d2h_bytes_per_step": int(top_cols.nbytes + top_scores.nbytes),
                     "note": "ocf_score_topk through model.recommend: host row ids in, 100 (column, score) pairs per row out"},
            "gpu_launches": int(launches),
            "e2e": {"value": rows / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": int(devs[0].info()["h2d_bytes"]),
                    "d2h_bytes_per_step": int(res.nbytes), "ms_per_call": 1e3 * e2e_s,
                    "note": "bounded by the PCIe read-back of the [rows, N] float32 score matrix"},
            "roofline": {"kernel": "k_score_tc2 (tcgen05 cta_group::2 kind::tf32)", "bound": "tensor", "achieved": flops / (gemm_ms * 1e-3) / 1e12,
                         "peak": peak, "unit": "TFLOP/s", "frac": flops / (gemm_ms * 1e-3) / 1e12 / peak,
                         # DRAM bytes per launch from the committed ncu --set full capture (profiles/traffic.json)
                         "traffic": ncu_traffic("score_%dx%dx%d" % (rows, N, hp), "k_score_tc2")[0],
                         "peak_source": src, "kernel_ms": gemm_ms, "share_of_step": gemm_ms / ms,
                         "out_GBs": 4.0 * rows * N / (gemm_ms * 1e-3) / 1e9}}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 2 + k and r[2 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_dataset(w, seed=0):
    """The workload's synthetic FixedSplit; cached under /tmp so the N=1,2,4,8 runs of one box
    (and the reference arm) do not each spend ~20 s regenerating it."""
    import pickle
    from omnidirectional_collaborative_filtering_b200 import synthetic
    path = "/tmp/ocf_b200_%s_%d_%d.pkl" % (w["shape"], int(w["reverse"]), seed)
    if os.path.exists(path):
        try:
            with open(path, "rb") as f:
                return pickle.load(f)
        except Exception:
            pass
    fs = synthetic.make_fixed_split(w["shape"], reverse_user_item_data=w["reverse"], seed=seed)
    try:
        tmp = path + ".%d.tmp" % os.getpid()
        with open(tmp, "wb") as f:
            pickle.dump(fs, f, protocol=4)
        os.replace(tmp, path)
    except Exception:
        pass
    return fs


def n_unique(a):
    """Number of distinct values (sort + compare; NumPy 2.3's hash-based np.unique is ~50x slower on these sizes)."""
    a = np.sort(np.asarray(a).ravel())
    return int(np.count_nonzero(a[1:] != a[:-1]) + 1) if a.size else 0


DUMP_BYTES = 60 * 10 ** 6


def write_outputs(out_dir, arrays):
    """`arrays` (name -> float32 array) as out_dir/<name>.npy, at most DUMP_BYTES in all. Smaller arrays are written
    whole; each array that would overrun its equal share of what is left keeps a sorted sample of its slices along
    its longest axis, drawn with RandomState(0), so two runs at the same shapes sample the same indices."""
    os.makedirs(out_dir, exist_ok=True)
    left, items = DUMP_BYTES, sorted(arrays.items(), key=lambda kv: kv[1].nbytes)
    for k, (name, a) in enumerate(items):
        share = left // (len(items) - k)
        if a.nbytes > share:
            axis = int(np.argmax(a.shape))
            n = a.shape[axis]
            keep = max(1, share // (a.nbytes // n))
            a = np.take(a, np.sort(np.random.RandomState(0).choice(n, keep, replace=False)), axis=axis)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
        left -= a.nbytes


def touched(batch, k_mask_blocks):
    """Unique catalogue columns the batch touches as inputs / as targets (for algorithmic bytes)."""
    csr = batch.source.csr
    cols = np.concatenate([csr.col[csr.rowptr[r]:csr.rowptr[r + 1]] for r in batch.rows])
    f = batch.flags.astype(bool)
    u_in = n_unique(cols[f])
    u_tg = n_unique(cols if batch.pass_through else cols[~f])
    return u_in, u_tg, int(f.sum()), int(cols.size if batch.pass_through else (~f).sum())


def state_words_of(w):
    return {"sgd": 2, "adagrad": 4, "rmsprop": 4, "adam": 6}[w["opt"][0]]


def ncu_traffic(workload, kernel_key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel from the committed
    `ncu --set full` summary of the CURRENT round for this workload, or None: profiles/traffic.json is written by
    scripts/ncu_summary.py from the raw capture, so the number is never a literal in this file."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        e = t.get(workload, {}).get(kernel_key)
        return (float(e["dram_bytes"]), e["source"]) if e else (None, None)
    except Exception:
        return None, None


def step_bytes(plans, w, nnz_store, n_obs_sample=8):
    """Algorithmic bytes of one train step's kernels, mean over `plans` (SURVEY.md section 8d):
    [K1, K2, K3, K4a, K4b]. K4b = S * 4 * (h_dec * U_target + h_enc * (k_in * U_input + k_obs * U_observed)) with
    S = 2 * (1 + optimizer state arrays) words per parameter and U_* the distinct columns the batch touches."""
    aux = w["aux"]
    H = w["hidden"]
    h_enc = H if isinstance(H, int) else H[0]
    h_dec = H if isinstance(H, int) else H[-1]
    k_in = 1 + (1 if aux in ("dropout", "both") else 0)          # encoder blocks selected by the input bit
    k_obs = (1 if aux in ("causal", "both") else 0)
    st = np.array([touched(p, 0) for p in plans], dtype=np.float64).mean(axis=0)   # u_in, u_tg, n_in, n_tg
    u_obs = np.mean([n_unique(np.concatenate([p.source.csr.col[p.source.csr.rowptr[r]:p.source.csr.rowptr[r + 1]]
                                              for r in p.rows])) for p in plans[:n_obs_sample]])
    n_all = float(np.mean([p.n_entries for p in plans]))
    state_words = {"sgd": 2, "adagrad": 4, "rmsprop": 4, "adam": 6}[w["opt"][0]]
    return [
        9.0 * n_all * 2,                                                       # K1: read col,val,flag + write col,val,code
        4.0 * h_enc * (st[2] * k_in + n_all * k_obs),                          # K2: one Wenc row per contributing entry
        4.0 * h_dec * st[3],                                                   # K3: one WdecT row per target entry
        40.0 * n_all,                                                          # K4a: counting sort over the batch's entries
        4.0 * state_words * (h_dec * st[1] + h_enc * (st[0] * k_in + u_obs * k_obs)),   # K4b: W + state, read + write, touched rows
    ]


# ------------------------------------------------------------------------------------------------
# CPU reference arm: the oracle port (reference algorithm, per-rating Python loop + dense NumPy)
# ------------------------------------------------------------------------------------------------
def cpu_reference(w, fs, batch_size, steps, warmup, budget_s=None, seed=0):
    from oracle import ref_batches, ref_model
    # every host core for the dense NumPy step, whatever OMP_NUM_THREADS says (torchrun sets it to 1 for N > 1)
    threads = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        cpu_reference._limit = threadpool_limits(limits=threads)          # kept alive for the whole run
        threads = max([p.get("num_threads", 1) for p in threadpool_info()] or [threads])
    except Exception:
        threads = int(os.environ.get("OMP_NUM_THREADS", threads))
    rs = np.random.RandomState(seed)
    n_batches = steps + warmup
    rows = rs.permutation(fs.train.n_rows)[:n_batches * batch_size]
    n_batches = min(n_batches, len(rows) // batch_size)
    rows = rows[:n_batches * batch_size]
    train = {}

    def add_rows(batch_rows):                             # dict-of-lists form, built lazily per batch (untimed)
        for r in batch_rows:
            c, v = fs.train.row(int(r))
            train[str(int(r))] = [[int(ci), float(vi)] for ci, vi in zip(c, v)]

    data = ref_batches.RefData(fs.n_cols, fs.train.n_rows, list(range(fs.n_cols)), eval_mode="fixed_split",
                               train=train, valid=({}, {}), test=({}, {}))
    order = [str(int(r)) for r in rows]
    aux = w["aux"]
    model = ref_model.RefModel(w["layers"], w["hidden"], fs.n_cols, batch_size, dense_activation=w["act"],
                               use_causal_info=aux is not None, use_both_masks=aux == "both",
                               dropout_probability=w["dropout"], dtype=np.float32, rng=np.random.RandomState(1))
    model.compile(ref_model.RefOptimizer(w["opt"][0], lr=w["opt"][1]), "mean_squared_error", rating_range=fs.rating_range)
    rng = np.random.RandomState(seed + 1)
    t_batch = t_model = 0.0
    ratings = 0
    done = 0
    t_start = time.perf_counter()
    for i in range(n_batches):
        add_rows(rows[i * batch_size:(i + 1) * batch_size])
        t0 = time.perf_counter()
        arrays = ref_batches.split_batch_loop(data, order, batch_size, i * batch_size, w["sparsity"], w["aux_value"],
                                              w["pass_through"], rng)
        feed = ref_batches.feed_list(arrays, aux)
        t1 = time.perf_counter()
        model.train_on_batch(feed, arrays[3])
        t2 = time.perf_counter()
        if i >= warmup:
            t_batch += t1 - t0
            t_model += t2 - t1
            ratings += sum(len(train[k]) for k in order[i * batch_size:(i + 1) * batch_size])
            done += 1
            if budget_s is not None and done >= 2 and time.perf_counter() - t_start > budget_s:
                break
    total = t_batch + t_model
    return {"value": ratings / total if total > 0 else 0.0, "unit": "ratings/s", "cores": int(threads), "kind": "port",
            "sample": "%d steps of %d rows (%d ratings) of the same workload; batch build %.1f%% / model step %.1f%% of the time"
                      % (done, batch_size, ratings, 100 * t_batch / max(total, 1e-9), 100 * t_model / max(total, 1e-9)),
            "ms_per_step": 1e3 * total / max(done, 1), "steps": done,
            "overlapped_value": ratings / max(t_batch, t_model, 1e-9)}


def other_workloads(names, args, gpus=1):
    """The remaining BASELINE configs, each in its own process (own CUDA context, a failure cannot take the headline
    line down): value / e2e / ms_per_step / roofline / per-kernel times of `bench.py --workload X`."""
    out = {}
    for name in names:
        cmd = [sys.executable, os.path.abspath(__file__), "--workload", name, "--steps", str(max(10, min(args.steps, 30))),
               "--warmup", str(args.warmup), "--no-cpu-baseline", "--no-scoring", "--others", "none", "--batch-size", str(args.batch_size)]
        t0 = time.perf_counter()
        try:
            res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
            d = json.loads(res.stdout.strip().splitlines()[-1])
            out[name] = {k: d.get(k) for k in ("value", "unit", "ms_per_step", "steps", "e2e", "roofline", "kernels", "gpu_launches", "config",
                                               "l2", "ratings_per_step", "target_ratings_per_s", "clocks")}
            out[name]["wall_s"] = time.perf_counter() - t0
        except Exception as e:
            out[name] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ml10m", choices=sorted(WORKLOADS))
    ap.add_argument("--batch-size", type=int, default=128)
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="train", choices=["train", "score"],
                    help="score: full-catalogue scoring rows/s as the line's metric (the train line carries it under 'scoring')")
    ap.add_argument("--score-rows", type=int, default=1024)
    ap.add_argument("--parallel", default="columns", choices=["columns", "rows"],
                    help="N > 1: item-dimension sharding (default) or data parallelism with a gradient all-reduce")
    ap.add_argument("--others", default=None,
                    help="comma-separated workloads whose value / e2e / roofline ride along under 'other_workloads' "
                         "(default: the other four BASELINE configs when the workload is the default one; 'none' to skip)")
    ap.add_argument("--no-scoring", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, at most "
                         "60 MB: the step's metrics and the updated weights, or the scores in --mode score); inputs are "
                         "seeded, so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs is not None and (args.impl == "reference" or world > 1):
        ap.error("--dump-outputs covers the single-GPU path of --impl ours")
    B = args.batch_size
    cfg = {"workload": "%s-shaped synthetic (%s), rows=%s, L=%d, H=%s, %s, aux=%s, train_sparsity=%s, pass_through=%s, %s lr=%g, dropout=%s, batch_size=%d"
           % (args.workload, w["shape"], "items" if w["reverse"] else "users", w["layers"], w["hidden"], w["act"], w["aux"],
              w["sparsity"], w["pass_through"], w["opt"][0], w["opt"][1], w["dropout"], B)}

    if args.impl == "reference":
        if rank != 0:
            return 0
        fs = make_dataset(w)
        warm = max(args.warmup, 0)
        res = cpu_reference(w, fs, B, args.steps, warm, budget_s=150.0)
        line = {"impl": "reference", "metric": "train ratings/sec", "value": res["value"], "unit": "ratings/s",
                "n_gpus": args.gpus, "steps": res["steps"], "warmup": warm, "ms_per_step": res["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg, "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": res["value"], "unit": "ratings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    from omnidirectional_collaborative_filtering_b200 import _lib, optimizers
    from omnidirectional_collaborative_filtering_b200.data_reader import data_reader
    from omnidirectional_collaborative_filtering_b200.model import omni_model
    from omnidirectional_collaborative_filtering_b200.store import DeviceBatch

    if world > 1:
        from omnidirectional_collaborative_filtering_b200 import dist as ocf_dist
        return ocf_dist.bench_main(args, w, cfg, rank, world)

    torch.cuda.set_device(0)
    lib = _lib.lib()
    fs = make_dataset(w)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):     # the reader prints the reference's "Finished loading data"
        rd = data_reader(fs.n_cols, fs.train.n_rows, "", eval_mode="fixed_split", data=fs)
    aux = w["aux"]
    np.random.seed(0)
    om = omni_model(w["layers"], w["hidden"], fs.n_cols, B, dense_activation=w["act"], use_causal_info=aux is not None,
                    use_both_masks=aux == "both", dropout_probability=w["dropout"], auxilliary_mask_type=aux)
    m = om.model
    opt = {"adagrad": optimizers.Adagrad, "rmsprop": optimizers.RMSprop, "adam": optimizers.Adam}[w["opt"][0]](lr=w["opt"][1])
    m.compile(opt, "mean_squared_error", rating_range=fs.rating_range)
    K, W = args.steps, max(args.warmup, 3)

    if args.mode == "score":
        sampler = ClockSampler(0)
        sc = scoring_run(lib, m, rd, w, aux, args.score_rows, K, W, args.dump_outputs)
        line = {"metric": "full-catalogue scoring rows/sec", "value": sc["value"], "unit": "rows/s", "n_gpus": 1, "steps": K,
                "warmup": W, "ms_per_step": sc["ms_per_call"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "tf32 operands, f32 accumulate", "data": "synthetic",
                "config": dict(cfg, rows_per_call=sc["rows_per_call"], n_cols=sc["n_cols"],
                               l2="outputs (%.0f MB per call) exceed the 126 MB L2" % (4e-6 * sc["rows_per_call"] * sc["n_cols"])),
                "clocks": sampler.stop(), "e2e": sc["e2e"], "gpu_launches": sc["gpu_launches"], "roofline": sc["roofline"]}
        print(json.dumps(line))
        return 0

    def gen():
        return rd.data_gen(B, w["sparsity"], "train", True, aux, w["aux_value"], pass_through_input_training=w["pass_through"])

    # ---- value: K steps on batches whose row ids / flags are resident in HBM --------------------
    g = gen()
    plans = []
    while len(plans) < K + W:
        b = next(g)
        if b is None:
            g = gen()
            continue
        b.flags                             # spend the batch's draws now (device RNG: upload + read back)
        plans.append(b)
    m._ensure(B, max(p.n_entries for p in plans), aux, rd)      # workspaces sized once for any batch of the set
    resident = []
    for p in plans:
        dev = DeviceBatch(p.n_rows, p.n_entries)
        dev.fill_split(p.source, p.rows, p.flags, p.pass_through, p.aux_value, None)
        resident.append(dev)
    import ctypes as C
    sargs = _lib.StepArgs()
    sargs.dropout_seed = om.dropout_seed

    def device_steps(devs, first_step):
        for k, dev in enumerate(devs):
            sargs.step = first_step + k
            _lib.check(lib.ocf_batch_regather(dev.handle, None))
            _lib.check(lib.ocf_train_step(m._handle, dev.handle, C.byref(sargs), None, None))

    # every resident batch object is stepped twice before the clock starts: the first pass runs as plain launches,
    # the second captures the step of that batch object into a CUDA graph, the timed pass replays the graphs
    device_steps(resident, 0)
    device_steps(resident, K + W)
    device_steps(resident[:W], 2 * (K + W))
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.ocf_kernel_launches()
    torch.cuda.synchronize()
    e0.record()
    device_steps(resident[W:], 2 * (K + W) + W)
    e1.record()
    torch.cuda.synchronize()
    launches = lib.ocf_kernel_launches() - launches0
    ms = e0.elapsed_time(e1)
    if args.dump_outputs is not None:         # before the steps below move the weights on
        outs = {"metrics": np.array(m.wait_metrics(m.steps_logged() - 1), dtype=np.float32)}
        for i, a in enumerate(m.get_weights()):
            outs["%s_%d" % ("kernel" if i % 2 == 0 else "bias", i // 2)] = a
        write_outputs(args.dump_outputs, outs)
    # the timed region lasts a few ms, nvidia-smi samples every 100 ms: keep the same steps running
    # for ~0.6 s so the clock / throttle record is taken under this load
    t_hold = time.perf_counter()
    while time.perf_counter() - t_hold < 0.6:
        device_steps(resident[W:], W)
        torch.cuda.synchronize()
    ratings = sum(p.n_entries for p in plans[W:])
    value = ratings / (ms * 1e-3)
    # SURVEY 8(d) counts a rating as one observed TARGET entry of a step; `value` counts every stored rating of the
    # batch rows (each is gathered, split and consumed). Both are reported.
    targets = sum(p.n_entries if p.pass_through else int((np.asarray(p.flags) == 0).sum()) for p in plans[W:])
    working_set = (sum(np.prod(sh) for sh in om.weight_shapes()) * 4 * state_words_of(w) / 2 + fs.train.nnz * 9) / 1e6
    if working_set > 2 * 126:
        l2_note = "no flush: weights + optimizer state + store (%.0f MB) exceed the 126 MB L2 several times over" % working_set
    else:
        l2_note = ("no flush, and weights + optimizer state + store (%.0f MB) fit or nearly fit the 126 MB L2: the kernels of this "
                   "workload run from L2, an HBM fraction is not meaningful for it (roofline.bound says 'l2')" % working_set)

    # ---- roofline: instrumented pass over the same resident batches ------------------------------
    lib.ocf_profile_reset()
    lib.ocf_profile_enable(1)
    device_steps(resident[W:], W + K)
    torch.cuda.synchronize()
    lib.ocf_profile_enable(0)
    tag_names = ["k_gather_split (K1)", "k_enc_fwd (K2)", "k_dec_fwd (K3)", "k_sort_count+alloc+place (K4a, on the batch stream)", "k_row_update (K4b)"]
    tag_ms = []
    n_prof_steps = 1
    for t in (0, 1, 2, 3, 5):
        tot, cnt = C.c_double(), C.c_int64()
        _lib.check(lib.ocf_profile_read(t, C.byref(tot), C.byref(cnt)))
        if t == 1:
            n_prof_steps = max(cnt.value, 1)
        # per step: a width list launches the row update twice (decoder rows, encoder rows)
        tag_ms.append(tot.value / max(cnt.value, 1) if t != 5 else tot.value / n_prof_steps)
    state_words = state_words_of(w)
    alg = step_bytes(plans[W:], w, fs.train.nnz)
    if w["layers"] > 1:
        # hidden [H1, H2] layers: three tcgen05 contractions each per step (forward, backward, gradient + update)
        tot, cnt = C.c_double(), C.c_int64()
        _lib.check(lib.ocf_profile_read(8, C.byref(tot), C.byref(cnt)))
        widths = w["hidden"] if isinstance(w["hidden"], (list, tuple)) else [w["hidden"]] * w["layers"]
        hid_bytes = sum(4.0 * a * b * (2 + state_words) for a, b in zip(widths[:-1], widths[1:]))   # W read twice + W/state read+write
        tag_names.append("k_gemm_tc x%d (hidden layers, tcgen05 3xTF32)" % (cnt.value // n_prof_steps))
        tag_ms.append(tot.value / n_prof_steps)
        alg = list(alg) + [hid_bytes]
    peak, peak_src = peaks()
    dom = int(np.argmax(tag_ms))
    kernels = {tag_names[t]: {"ms": tag_ms[t], "algorithmic_bytes": alg[t], "GB/s": alg[t] / (tag_ms[t] * 1e-3) / 1e9 if tag_ms[t] > 0 else None}
               for t in range(len(tag_names))}
    achieved = alg[dom] / (tag_ms[dom] * 1e-3) / 1e9
    # DRAM bytes per launch from the committed `ncu --set full` capture of this kernel on this workload
    traffic, traffic_src = ncu_traffic(args.workload, tag_names[dom].split(" ")[0]) if B == 128 else (None, None)
    roofline = {"kernel": tag_names[dom], "bound": "hbm" if working_set > 2 * 126 else "l2", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes": alg[dom], "peak_source": peak_src,
                "share_of_step": tag_ms[dom] / (ms / K),
                # the whole step against the same roofline: every kernel's algorithmic bytes / the step's device time
                "step_frac": sum(alg) / (ms / K * 1e-3) / 1e9 / peak, "step_algorithmic_bytes": sum(alg)}

    # ---- e2e: the public API, host buffers in, metrics out, every step ---------------------------
    from omnidirectional_collaborative_filtering_b200.data_reader import Prefetcher
    per_epoch = rd.train_set_size // B

    def epochs(total):
        """`total` batches, epoch by epoch like train.py:150-158: a fresh generator per epoch, drawn
        on a generator thread (the reference's GeneratorEnqueuer), consumed in order."""
        done = 0
        while done < total:
            n = min(total - done, per_epoch)
            for b in Prefetcher(gen(), n):
                yield b
            done += n

    ring_depth = max(2, int(os.environ.get("OCF_RING_DEPTH", "3")))
    for b in epochs(max(W, 3 * ring_depth)):   # three rounds of the reader's ring of batch buffers: plain, capture, replay
        m.train_on_batch(b, sync=True)
    torch.cuda.synchronize()
    h2d = 0
    e_ratings = 0
    from collections import deque
    in_flight = deque()
    lag = max(1, int(os.environ.get("OCF_BENCH_LAG", "2")))      # steps enqueued ahead of the metrics read-back (the reader holds 3 batch buffers)
    t0 = time.perf_counter()
    # generator thread: set order, row ids, the batch's place in the NumPy stream; main thread:
    # pinned staging + H2D of the row ids + kernels (the random split is drawn on the device from
    # the replayed MT19937 stream) + the D2H read of EVERY step's metrics, `lag` steps behind the enqueue
    for b in epochs(K):
        m.train_on_batch(b, sync=False)
        in_flight.append(m.steps_logged() - 1)
        if len(in_flight) > lag:
            m.wait_metrics(in_flight.popleft())   # read step i-lag's result while the later steps run
        e_ratings += b.n_entries
        h2d += b._device.info()["h2d_bytes"]
    while in_flight:
        m.wait_metrics(in_flight.popleft())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()

    line = {"metric": "train ratings/sec", "value": value, "unit": "ratings/s", "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": cfg, "l2": l2_note, "ratings_per_step": ratings / K,
            "target_ratings_per_step": targets / K, "target_ratings_per_s": targets / (ms * 1e-3),
            "clocks": clocks,
            "e2e": {"value": e_ratings / e2e_s, "unit": "ratings/s", "h2d_bytes_per_step": h2d / K,
                    "d2h_bytes_per_step": 4 * _lib.N_METRICS, "ms_per_step": 1e3 * e2e_s / K},
            "gpu_launches": int(launches), "roofline": roofline, "kernels": kernels}
    if not args.no_scoring:
        try:
            line["scoring"] = scoring_run(lib, m, rd, w, aux, args.score_rows, 10, 3)
        except Exception as e:                                  # the train line must not depend on it
            line["scoring"] = {"error": str(e)}
    others = args.others
    if others is None:
        others = "ml1m,jester,ml20m,netflix" if args.workload == "ml10m" else "none"
    if others != "none":
        # release this workload's device memory before the others run in their own processes
        m.close(); rd.close(); del resident
        line["other_workloads"] = other_workloads([x for x in others.split(",") if x], args)
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = {k: v for k, v in cpu_reference(w, fs, B, 1000, 1, budget_s=args.cpu_seconds).items()
                                if k in ("value", "unit", "cores", "kind", "sample", "overlapped_value")}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
