"""Ranking evaluation host logic (no GPU): `ranking.metrics_from_ranks` on the oracle's brute-force ranks
equals the oracle's metrics read directly off the sorted candidate lists; the oracle's ranks agree with the
top-k oracle; `train.run` calls the ranking evaluation only when asked, and after every test procedure."""
import numpy as np
import pytest

from oracle import ref_rank, ref_topk
from omnidirectional_collaborative_filtering_b200 import ranking
from omnidirectional_collaborative_filtering_b200 import train as ocf_train


def _case(seed, B, N, distinct, n_tgt, n_seen, dup=True):
    """Scores with exact ties (`distinct` values), per-row targets (with a repeated column) and seen columns."""
    rs = np.random.RandomState(seed)
    scores = rs.randint(0, distinct, size=(B, N)).astype(np.float32) * np.float32(0.25)
    targets, seen = [], []
    for b in range(B):
        nt = int(rs.randint(0, n_tgt + 1)) if b else 0            # row 0: no relevant item
        cols = rs.choice(N, size=min(nt, N), replace=False)
        vals = rs.randint(1, 6, size=cols.size).astype(np.float32)
        if dup and cols.size > 1:                                   # a repeated column: the last value counts
            cols = np.append(cols, cols[0])
            vals = np.append(vals, np.float32(5.0 if vals[0] < 3 else 1.0))
        targets.append((cols, vals))
        rest = np.setdiff1d(np.arange(N), cols)
        seen.append(rs.choice(rest, size=min(n_seen, rest.size), replace=False))
    return scores, targets, seen


def _via_ranks(scores, targets, seen, ks, min_value):
    row_ptr, _, r, n_cand = ref_rank.ranks(scores, targets, seen, min_value)
    return ranking.finalize(ranking.metrics_from_ranks(row_ptr, r, n_cand, ks))


def _assert_same(got, want):
    assert got.keys() == want.keys()
    for name in want:
        if isinstance(want[name], float) and np.isnan(want[name]):
            assert np.isnan(got[name]), name
        else:
            assert got[name] == pytest.approx(want[name], rel=1e-12, abs=1e-12), name


@pytest.mark.parametrize("seed,B,N,distinct,n_tgt,n_seen", [
    (0, 12, 60, 4, 10, 5),          # heavy ties
    (1, 9, 200, 1000, 30, 20),      # few ties
    (2, 6, 7, 3, 7, 0),             # k > n_cand
    (3, 20, 500, 2, 60, 100),       # two score values only
])
@pytest.mark.parametrize("min_value", [None, 3.0])
@pytest.mark.parametrize("exclude", [False, True])
def test_metrics_from_ranks_equal_the_direct_oracle(seed, B, N, distinct, n_tgt, n_seen, min_value, exclude):
    scores, targets, seen = _case(seed, B, N, distinct, n_tgt, n_seen)
    ks = (1, 3, 10, 1000)
    seen = seen if exclude else None
    _assert_same(_via_ranks(scores, targets, seen, ks, min_value), ref_rank.metrics(scores, targets, seen, ks, min_value))


def test_rows_where_every_candidate_is_relevant_skip_auc():
    N = 8
    scores = np.arange(2 * N, dtype=np.float32).reshape(2, N)
    targets = [(np.arange(N), np.ones(N, np.float32)),                 # every column relevant: no negative
               (np.array([1, 5]), np.ones(2, np.float32))]
    want = ref_rank.metrics(scores, targets, None, (1, 4, 20), None)
    assert want["rows"] == 2 and want["AUC_rows"] == 1
    got = _via_ranks(scores, targets, None, (1, 4, 20), None)
    _assert_same(got, want)
    # the full row ranks 1..N, so its own AUC would be undefined; the other row's is the whole mean
    row_ptr, cols, r, n_cand = ref_rank.ranks(scores, targets)
    assert sorted(r[:N].tolist()) == list(range(1, N + 1))
    assert n_cand.tolist() == [N, N]


def test_no_relevant_rows_give_nan_means_and_zero_counts():
    scores = np.zeros((3, 5), dtype=np.float32)
    targets = [(np.array([], dtype=np.int64), np.array([], dtype=np.float32))] * 3
    got = _via_ranks(scores, targets, None, (5,), None)
    assert got["rows"] == 0 and got["AUC_rows"] == 0 and np.isnan(got["MRR"]) and np.isnan(got["NDCG@5"])


def test_hand_computed_row():
    # candidates in order: c3 (0.9), c0 (0.5), c2 (0.5), c1 (0.1); targets c2 and c1 -> ranks 3 and 4
    scores = np.array([[0.5, 0.1, 0.5, 0.9]], dtype=np.float32)
    targets = [(np.array([2, 1]), np.array([4.0, 2.0], np.float32))]
    row_ptr, cols, r, n_cand = ref_rank.ranks(scores, targets)
    assert cols.tolist() == [1, 2] and r.tolist() == [4, 3] and n_cand.tolist() == [4]
    got = _via_ranks(scores, targets, None, (3,), None)
    assert got["HR@3"] == 1.0 and got["precision@3"] == pytest.approx(1 / 3) and got["recall@3"] == 0.5
    assert got["NDCG@3"] == pytest.approx((1 / np.log2(4)) / (1 + 1 / np.log2(3)))
    assert got["MRR"] == pytest.approx(1 / 3)
    assert got["AUC"] == pytest.approx(0.0)          # both negatives outrank both targets
    # min_value drops c1 (value 2): one target at rank 3 among 4 candidates
    got = _via_ranks(scores, targets, None, (3,), 3.0)
    assert got["recall@3"] == 1.0 and got["AUC"] == pytest.approx(1 - 2 / 3)


def test_batches_accumulate():
    scores, targets, seen = _case(5, 16, 80, 6, 12, 4)
    ks = (2, 9)
    total = ranking.empty_sums(ks)
    for lo in range(0, 16, 5):
        part = slice(lo, lo + 5)
        row_ptr, _, r, n_cand = ref_rank.ranks(scores[part], targets[part], seen[part])
        ranking.accumulate(total, ranking.metrics_from_ranks(row_ptr, r, n_cand, ks))
    _assert_same(ranking.finalize(total), ref_rank.metrics(scores, targets, seen, ks))


@pytest.mark.parametrize("k", [1, 5, 40])
def test_ranks_agree_with_topk_membership(k):
    scores, targets, seen = _case(7, 10, 40, 5, 15, 6)
    row_ptr, cols, r, _ = ref_rank.ranks(scores, targets, seen)
    top_c, _ = ref_topk.topk(scores, k, seen)
    for b in range(scores.shape[0]):
        lo, hi = row_ptr[b], row_ptr[b + 1]
        for c, rk in zip(cols[lo:hi], r[lo:hi]):
            if rk <= k:
                assert top_c[b, rk - 1] == c
            else:
                assert c not in top_c[b]


# ---- train.run ------------------------------------------------------------------------------------------

class _Hist(object):
    def __init__(self, v):
        self.history = {"loss": [1.0], "val_accurate_MSE": [v]}


class _Net(object):
    metrics_names = ["loss", "mean_absolute_error", "accurate_MAE", "nMAE", "accurate_RMSE", "accurate_MSE"]

    def __init__(self, trace):
        self.trace, self.logged, self.epoch = trace, 0, 0

    def compile(self, **kw):
        pass

    def fit_generator(self, gen, steps, validation_data=None, validation_steps=None, verbose=0):
        self.epoch += 1
        self.trace.append(("fit",))
        return _Hist(5.0 - self.epoch)

    def get_weights(self):
        return [np.zeros(1, np.float32)]

    def set_weights(self, w):
        pass

    def save(self, path):
        pass

    def evaluate_generator(self, gen, steps):
        self.trace.append(("evaluate_generator", int(steps)))
        return [0.1, 0.2, 0.3, 0.4, 0.5, 0.6]

    def test_on_batch(self, batch, sync=True):
        self.trace.append(("test_on_batch",))
        self.logged += 1

    def steps_logged(self):
        return self.logged

    def read_metrics(self, first, count):
        return np.ones((1, 8), dtype=np.float32)

    def evaluate_ranking(self, gen, steps, ks=(10,), exclude_seen=True, min_value=None, workers=1):
        self.trace.append(("evaluate_ranking", int(steps), tuple(ks), min_value))
        return {"rows": 1, "AUC_rows": 1, "MRR": 0.5}


class _Batch(object):
    target_count = 3


class _Reader(object):
    num_items, train_set_size, val_set_size, test_set_size = 5, 40, 20, 20

    def __init__(self, trace):
        self.trace = trace

    def data_gen(self, batch_size, data_sparsity, train_val_test="train", **kw):
        self.trace.append(("data_gen", train_val_test, data_sparsity))
        return iter([_Batch()] * 100)

    def split_for_validation(self, val_split):
        pass


def _run(monkeypatch, tmp_path, eval_mode, **kw):
    trace = []
    net = _Net(trace)

    class _Owner(object):
        model = net

    monkeypatch.setattr(ocf_train, "omni_model", lambda *a, **k: _Owner())
    cfg = ocf_train.TrainConfig(max_epochs=2, batch_size=4, eval_mode=eval_mode, test_sparsities=[0.1, 0.5],
                                model_save_path=str(tmp_path) + "/", num_hidden_units=8)
    res = ocf_train.run(cfg, reader=_Reader(trace), rating_range=4.0, verbose=0, save_models=False, **kw)
    return res, trace


@pytest.mark.parametrize("eval_mode", ["fixed_split", "ablation"])
def test_train_run_ranks_only_when_asked_and_last(monkeypatch, tmp_path, eval_mode):
    base, base_trace = _run(monkeypatch, tmp_path, eval_mode)
    assert "test_ranking" not in base
    assert not [e for e in base_trace if e[0] == "evaluate_ranking"]
    res, trace = _run(monkeypatch, tmp_path, eval_mode, ranking_ks=[10, 100], ranking_min_value=4.0)
    n = len(base_trace)
    assert trace[:n] == base_trace                      # every existing call first, unchanged
    tail = trace[n:]
    steps = 20 // 4 - 1
    if eval_mode == "ablation":
        assert tail == [("data_gen", "test", 0.1), ("evaluate_ranking", steps, (10, 100), 4.0),
                        ("data_gen", "test", 0.5), ("evaluate_ranking", steps, (10, 100), 4.0)]
        assert set(res["test_ranking"]) == {0.1, 0.5}
    else:
        assert tail == [("data_gen", "test", None), ("evaluate_ranking", steps, (10, 100), 4.0)]
        assert res["test_ranking"]["MRR"] == 0.5
    for key in base:
        if key not in ("model", "save_name"):
            assert res[key] == base[key], key
