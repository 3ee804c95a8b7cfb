"""Ranking evaluation throughput on one GPU (DESIGN.md section 4, row `k_rank_*`).

    python scripts/rank_bench.py [--shapes ml10m,netflix] [--rows 1024] [--reps 20] [--warmup 3] [--out FILE]

For each shape (synthetic fixed split in item orientation: ML-10M, 71 567 columns; Netflix, 480 189 columns),
`rows` test rows per call with trained-looking random weights, timed with CUDA events after warm-up:
  * ocf_score with the scores left in HBM;
  * ocf_score_topk, k = 100, seen items excluded (host outputs);
  * ocf_rank_targets, seen items excluded (host outputs): evaluated rows/s for the whole call;
  * the three rank kernels alone (profiler tag 9).
The rank pass's algorithmic bytes: the score rows once per shared-memory chunk of relevant targets
(4 * N * sum over rows of max(1, ceil(n_rel / 2048))) plus the entry tiles (col, value, code read; the
workspace's key / column / entry / counter written and read back; the rank written). The score matrix is the
one ocf_score has just written, as in use, so its last part may still sit in the 126 MB L2.
Writes one JSON document (stdout, and FILE with --out); the card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"ml10m": 512, "netflix": 1000}            # hidden width of bench.py's workload of that shape
RANK_CHUNK = 2048


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6538.6, "SURVEY.md section 2 (measured on a B200)"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as exc:          # the numbers stay valid; the card is then unnamed
        return {"name": "unknown (%s)" % exc}


def run_shape(shape, hidden, rows, reps, warm):
    import torch
    from omnidirectional_collaborative_filtering_b200 import _lib, synthetic
    from omnidirectional_collaborative_filtering_b200.data_reader import data_reader
    from omnidirectional_collaborative_filtering_b200.model import omni_model
    from omnidirectional_collaborative_filtering_b200.store import DeviceBatch
    t0 = time.perf_counter()
    fs = synthetic.make_fixed_split(shape, reverse_user_item_data=True, seed=0)
    build_s = time.perf_counter() - t0
    rd = data_reader(fs.n_cols, fs.train.n_rows, "", eval_mode="fixed_split", data=fs)
    N = fs.n_cols
    rows = min(rows, rd.test_set_size)
    np.random.seed(1)
    om = omni_model(1, hidden, N, rows, dense_activation="sigmoid", use_causal_info=False)
    w = om.model.get_weights()
    rs = np.random.RandomState(2)
    w[-2] = (rs.normal(size=w[-2].shape) * 0.3).astype(np.float32)
    w[-1] = rs.normal(size=w[-1].shape).astype(np.float32)
    om.model.set_weights(w)
    m = om.model
    np.random.seed(3)
    gen = rd.data_gen(rows, None, "test", True, None, -1)
    batches = [next(gen) for _ in range(4)]
    h = m._ensure(rows, max(b.n_entries for b in batches), None, rd)
    devs = []
    for b in batches:
        d = DeviceBatch(b.n_rows, b.n_entries)
        d.fill_fixed(b.source, b.rows, b.aux_value, None)
        devs.append(d)
    lib = _lib.lib()
    out = torch.empty((rows, N), dtype=torch.float32, device="cuda")
    optr = C.c_void_p(out.data_ptr())
    E = max(b.n_entries for b in batches)
    tk_c = np.empty((rows, 100), np.int32)
    tk_s = np.empty((rows, 100), np.float32)
    r_col, r_rank = np.empty(E, np.int32), np.empty(E, np.int32)
    r_ptr, r_cand = np.empty(rows + 1, np.int32), np.empty(rows, np.int64)

    def score(d):
        _lib.check(lib.ocf_score(h, d.handle, optr, 1, None))

    def topk(d):
        _lib.check(lib.ocf_score_topk(h, d.handle, 100, 1, _lib.ptr(tk_c), _lib.ptr(tk_s), None))

    def rank(d):
        _lib.check(lib.ocf_rank_targets(h, d.handle, 1, float("-inf"), _lib.ptr(r_col), _lib.ptr(r_rank),
                                        _lib.ptr(r_ptr), _lib.ptr(r_cand), None))

    def timed(fn):
        for k in range(warm):
            fn(devs[k % len(devs)])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(reps):
            fn(devs[k % len(devs)])
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms = {"score": timed(score), "score_topk": timed(topk), "rank_targets": timed(rank)}
    lib.ocf_profile_reset()
    lib.ocf_profile_enable(1)
    for k in range(reps):
        rank(devs[k % len(devs)])
    torch.cuda.synchronize()
    lib.ocf_profile_enable(0)
    tot, cnt = C.c_double(), C.c_int64()
    _lib.check(lib.ocf_profile_read(9, C.byref(tot), C.byref(cnt)))
    kernel_ms = tot.value / max(cnt.value, 1)
    # algorithmic bytes of the rank pass, averaged over the batches the timed calls cycled through
    per = []
    for d in devs:
        rank(d)
        n_ent = int(r_ptr[-1])
        row_of = np.repeat(np.arange(rows), np.diff(r_ptr))
        n_rel = np.bincount(row_of, weights=(r_rank[:n_ent] > 0), minlength=rows).astype(np.int64)
        chunks = np.maximum(1, -(-n_rel // RANK_CHUNK))
        score_b = 4.0 * N * float(chunks.sum())
        tiles_b = 9.0 * n_ent + 32.0 * float(n_rel.sum()) + 4.0 * n_ent
        per.append((score_b, tiles_b, int(n_rel.sum()), int(chunks.max())))
    score_b = float(np.mean([p[0] for p in per]))
    tiles_b = float(np.mean([p[1] for p in per]))
    peak, peak_src = hbm_peak()
    achieved = (score_b + tiles_b) / (kernel_ms * 1e-3) / 1e9
    rd.close()
    return {
        "shape": shape, "n_cols": int(N), "rows_per_call": int(rows), "hidden": hidden, "dataset_build_s": build_s,
        "relevant_targets_per_call": float(np.mean([p[2] for p in per])), "max_chunks_per_row": max(p[3] for p in per),
        "ms_per_call": ms,
        "rows_per_s": {k: rows / (v * 1e-3) for k, v in ms.items()},
        "rank_kernels": {"ms": kernel_ms, "launch_groups": int(cnt.value), "score_bytes": score_b, "tile_bytes": tiles_b,
                         "achieved_GBs": achieved, "hbm_peak_GBs": peak, "hbm_peak_source": peak_src,
                         "frac_of_hbm_peak": achieved / peak,
                         "bound_us": (score_b + tiles_b) / (peak * 1e9) * 1e6},
        "notes": "score: device output, no sync; score_topk / rank_targets: host outputs, each call synchronises",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="ml10m,netflix")
    ap.add_argument("--rows", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from omnidirectional_collaborative_filtering_b200 import _lib
    _lib.require_gpu()
    doc = {"card": card(), "results": []}
    for s in args.shapes.split(","):
        doc["results"].append(run_shape(s, SHAPES[s], args.rows, args.reps, args.warmup))
        print(json.dumps(doc["results"][-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
