"""bench.py's host-side bookkeeping (no GPU): the algorithmic-bytes formula of SURVEY.md section 8d
on batches drawn with the host stream, for a full store and for a column shard."""
import numpy as np

import bench
from omnidirectional_collaborative_filtering_b200 import synthetic
from omnidirectional_collaborative_filtering_b200.data_reader import data_reader


def _plans(shard=None, n=3):
    fs = synthetic.make_fixed_split("small", reverse_user_item_data=True, seed=1)
    rd = data_reader(fs.n_cols, fs.train.n_rows, "", eval_mode="fixed_split", data=fs, rng_on_device=False, shard=shard)
    np.random.seed(0)
    g = rd.data_gen(32, [0.5, 0.5], "train", True, "dropout", -1)
    return fs, [next(g) for _ in range(n)]


def test_step_bytes_formula_matches_a_direct_count():
    w = dict(bench.WORKLOADS["small"], aux="dropout", hidden=64, opt=("adagrad", 0.005))
    fs, plans = _plans()
    alg = bench.step_bytes(plans, w, fs.train.nnz)
    u_in, u_tg, n_in, n_tg = [], [], [], []
    for p in plans:
        csr = p.source.csr
        cols = np.concatenate([csr.col[csr.rowptr[r]:csr.rowptr[r + 1]] for r in p.rows])
        f = p.flags.astype(bool)
        u_in.append(len(set(cols[f].tolist()))); u_tg.append(len(set(cols[~f].tolist())))
        n_in.append(int(f.sum())); n_tg.append(int((~f).sum()))
    n_all = np.mean([p.n_entries for p in plans])
    assert alg[0] == 18.0 * n_all
    assert np.isclose(alg[1], 4 * 64 * np.mean(n_in) * 2)            # data block + dropout-mask block
    assert np.isclose(alg[2], 4 * 64 * np.mean(n_tg))
    assert np.isclose(alg[4], 16 * 64 * (np.mean(u_tg) + 2 * np.mean(u_in)))


def test_step_bytes_of_shards_add_up_to_less_than_twice_the_whole():
    w = dict(bench.WORKLOADS["small"], aux="dropout", hidden=64, opt=("adagrad", 0.005))
    fs, whole = _plans()
    _, s0 = _plans(shard=(0, 2))
    _, s1 = _plans(shard=(1, 2))
    a, a0, a1 = (bench.step_bytes(p, w, 0) for p in (whole, s0, s1))
    for k in (1, 2, 4):                                               # columns are disjoint over the shards
        assert np.isclose(a0[k] + a1[k], a[k])


def test_write_outputs_caps_the_dump_with_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    rs = np.random.RandomState(3)
    arrays = {"metrics": rs.rand(6).astype(np.float32), "kernel_0": rs.rand(4000, 64).astype(np.float32),
              "bias_0": rs.rand(64).astype(np.float32), "kernel_1": rs.rand(64, 3000).astype(np.float32)}
    for run in ("a", "b"):
        bench.write_outputs(str(tmp_path / run), arrays)
    got = {n: np.load(str(tmp_path / "a" / (n + ".npy"))) for n in arrays}
    assert sum(a.nbytes for a in got.values()) <= 1 << 20
    assert np.array_equal(got["metrics"], arrays["metrics"]) and np.array_equal(got["bias_0"], arrays["bias_0"])
    assert got["kernel_0"].shape[1] == 64 and 0 < got["kernel_0"].shape[0] < 4000
    assert got["kernel_1"].shape[0] == 64 and 0 < got["kernel_1"].shape[1] < 3000
    idx = [int(np.flatnonzero((arrays["kernel_0"] == r).all(axis=1))[0]) for r in got["kernel_0"]]
    assert idx == sorted(set(idx))                                 # whole rows of the original, in order
    for n in arrays:
        assert got[n].dtype == np.float32 and np.array_equal(got[n], np.load(str(tmp_path / "b" / (n + ".npy"))))


def test_bench_rejects_runs_without_timed_steps():
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr and out.stdout == ""


def test_reference_arm_runs_on_rank_0_only():
    """Under torchrun the reference arm is rank 0's job: the other ranks exit 0 without work or output."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_line_has_the_contract_keys():
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "small", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["vs_baseline"] is None and "workload" in line["config"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
