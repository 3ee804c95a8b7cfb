"""GPU parity of the ranking evaluation (`ocf_rank_targets`: prep / count / finish kernels of ocf_rank.cuh)
against the NumPy oracle applied to the scores the device itself produced (`model.score`): the same ranks as
integers, the same candidate counts; agreement with `recommend`; metrics over several batches; no side effects
on training; column shards refused; `train.run(ranking_ks=...)` end to end."""
import numpy as np
import pytest

from oracle import ref_rank
from omnidirectional_collaborative_filtering_b200 import _lib, dist as ocf_dist, optimizers, synthetic
from omnidirectional_collaborative_filtering_b200 import train as ocf_train
from omnidirectional_collaborative_filtering_b200.data_reader import Batch, data_reader
from omnidirectional_collaborative_filtering_b200.model import omni_model
from tests.helpers import cached_split, product_reader
from tests.test_shard_host import _shard_reader

pytestmark = pytest.mark.gpu

RANK_CHUNK = 2048                                   # ocf_rank.cuh: relevant targets per shared-memory chunk


def _truth(batch):
    """(seen, targets) of every batch row from the host stores: the columns K1 marks CODE_IN, and the target
    ratings (column, value) in entry order (the oracle keeps the last of a repeated column, as K1 does)."""
    seen, targets = [], []
    if batch.kind == "fixed":
        ci, ct = batch.source.in_store.csr, batch.source.tgt_store.csr
        for r in batch.rows:
            seen.append(ci.col[ci.rowptr[r]:ci.rowptr[r + 1]])
            lo, hi = ct.rowptr[r], ct.rowptr[r + 1]
            targets.append((ct.col[lo:hi], ct.val[lo:hi]))
        return seen, targets
    assert not batch.pass_through
    c, flags, o = batch.source.csr, batch.flags, 0
    for r in batch.rows:
        lo, hi = c.rowptr[r], c.rowptr[r + 1]
        f = flags[o:o + hi - lo]
        o += hi - lo
        cols, vals = c.col[lo:hi], c.val[lo:hi]
        seen.append(cols[f == 1])
        targets.append((cols[f == 0], vals[f == 0]))
    return seen, targets


def _by_col(row_ptr, cols, ranks):
    out = []
    for b in range(len(row_ptr) - 1):
        c = np.asarray(cols[row_ptr[b]:row_ptr[b + 1]], dtype=np.int64)
        r = np.asarray(ranks[row_ptr[b]:row_ptr[b + 1]], dtype=np.int64)
        o = np.argsort(c, kind="stable")
        out.append((c[o], r[o]))
    return out


def _check_batch(m, batch, exclude, min_value):
    """Device ranks == oracle ranks on the device's own scores. Returns the device result."""
    seen, targets = _truth(batch)
    scores = m.score(batch)
    got = m.rank_targets(batch, exclude_seen=exclude, min_value=min_value)
    want = ref_rank.ranks(scores, targets, seen if exclude else None, min_value)
    assert np.array_equal(got[3], want[3])                                      # candidates per row
    assert np.array_equal(np.diff(got[0]), np.diff(want[0]))                    # relevant targets per row
    for (gc, gr), (wc, wr) in zip(_by_col(got[0], got[1], got[2]), _by_col(want[0], want[1], want[2])):
        assert np.array_equal(gc, wc) and np.array_equal(gr, wr)
    return got, scores, seen, targets


def _model(n_cols, B, width, seed, flat=False):
    np.random.seed(seed)
    om = omni_model(1, width, n_cols, B, dense_activation="sigmoid", use_causal_info=False)
    w = om.model.get_weights()
    rs = np.random.RandomState(seed + 1)
    if flat:                                        # scores = bias only: a handful of distinct values, thousands of exact ties
        w[-2][:] = 0.0
        w[-1] = rs.randint(0, 5, size=w[-1].shape).astype(np.float32)
    else:
        w[-2] = (rs.normal(size=w[-2].shape) * 0.3).astype(np.float32)
        w[-1] = rs.normal(size=w[-1].shape).astype(np.float32)
    om.model.set_weights(w)
    return om


def _synthetic(shape, B, width, seed=3, flat=False):
    fs = synthetic.make_fixed_split(shape, reverse_user_item_data=True, seed=seed)
    rd = data_reader(fs.n_cols, fs.train.n_rows, "", eval_mode="fixed_split", data=fs)
    return rd, _model(fs.n_cols, B, width, seed, flat)


def _batch(rd, which, B, seed=5):
    np.random.seed(seed)
    if which == "split":                            # the ablation protocol: inputs / targets split, no pass-through
        return next(rd.data_gen(B, [0.3, 0.8], "train", True, None, -1, pass_through_input_training=False))
    return next(rd.data_gen(min(B, rd.val_set_size if which == "valid" else rd.test_set_size), None, which, True, None, -1))


@pytest.mark.parametrize("shape,B,width", [("tiny", 8, 12), ("small", 64, 48), ("ml1m", 96, 64)])
@pytest.mark.parametrize("which", ["valid", "test", "split"])
@pytest.mark.parametrize("exclude,min_value", [(True, None), (False, None), (True, 4.0), (False, 4.0)])
def test_ranks_match_oracle(shape, B, width, which, exclude, min_value):
    rd, om = _synthetic(shape, B, width)
    got, *_ = _check_batch(om.model, _batch(rd, which, B), exclude, min_value)
    if min_value is None:
        assert got[0][-1] > 0
    rd.close()


@pytest.mark.parametrize("which", ["valid", "split"])
@pytest.mark.parametrize("exclude", [True, False])
def test_ranks_on_rows_that_repeat_columns(golden_datasets, which, exclude):
    ds = golden_datasets["rev"]
    rd = product_reader(ds, "fixed_split")
    assert rd.store("train").info()["has_dups"] == 1
    om = _model(ds["n_cols"], 8, 16, 7)
    for seed in range(3):
        _check_batch(om.model, _batch(rd, which, 8, seed=seed), exclude, None)
    rd.close()


@pytest.mark.parametrize("which", ["valid", "split"])
def test_ranks_with_massive_ties(which):
    """Bias-only scores: 5 distinct values over 6040 columns; ties are broken by column."""
    rd, om = _synthetic("ml1m", 32, 32, flat=True)
    got, scores, *_ = _check_batch(om.model, _batch(rd, which, 32), True, None)
    assert len(np.unique(scores)) <= 5
    rd.close()


def test_ranks_agree_with_recommend():
    rd, om = _synthetic("ml1m", 64, 64)
    batch = _batch(rd, "test", 64)
    row_ptr, cols, ranks, _ = om.model.rank_targets(batch, exclude_seen=True)
    top, _ = om.model.recommend(batch, k=512, exclude_seen=True)
    inside = 0
    for b in range(batch.n_rows):
        c, r = cols[row_ptr[b]:row_ptr[b + 1]], ranks[row_ptr[b]:row_ptr[b + 1]]
        for cc, rr in zip(c, r):
            if rr <= 512:
                assert top[b, rr - 1] == cc
                inside += 1
        listed = set(top[b].tolist())
        assert len(listed & set(c.tolist())) == int(np.sum(r <= 512))     # no other relevant target is listed
    assert inside > 0
    rd.close()


# ---- the ML-10M catalogue width (71 567 columns in item orientation) --------------------------------------

@pytest.fixture(scope="module")
def ml10m():
    fs = cached_split("ml10m", True)
    rd = data_reader(fs.n_cols, fs.train.n_rows, "", eval_mode="fixed_split", data=fs)
    om = _model(fs.n_cols, 1024, 64, 11)
    yield fs, rd, om
    rd.close()


@pytest.mark.parametrize("B", [1, 1024])
def test_ml10m_width_batches(ml10m, B):
    fs, rd, om = ml10m
    batch = _batch(rd, "test", B, seed=B)
    got, *_ = _check_batch(om.model, batch, True, None)
    again = om.model.rank_targets(batch, exclude_seen=True)
    for x, y in zip(got, again):
        assert np.array_equal(x, y)                 # repeated calls: bit-identical


def test_ml10m_rows_spanning_several_chunks(ml10m):
    """The test set's longest target rows hold more than two shared-memory chunks of relevant targets, so every
    count CTA sweeps its slice once per chunk; a short row rides along."""
    fs, rd, om = ml10m
    src = rd.store("test")
    n_tg = np.diff(src.tgt_store.csr.rowptr)
    long_rows = np.argsort(n_tg, kind="stable")[-3:]
    assert n_tg[long_rows[-1]] > 2 * RANK_CHUNK
    rows = np.concatenate([long_rows, np.argsort(n_tg, kind="stable")[:1]]).astype(np.int32)
    tcount = int(n_tg[rows].sum())
    batch = Batch(rd, "fixed", src, rows, None, False, None, -1.0, tcount, False,
                  tcount + int(src.in_store.full_lengths[rows].sum()))
    for exclude in (True, False):
        got, *_ = _check_batch(om.model, batch, exclude, None)
        assert np.diff(got[0]).max() > 2 * RANK_CHUNK
        again = om.model.rank_targets(batch, exclude_seen=exclude)
        for x, y in zip(got, again):
            assert np.array_equal(x, y)
    _check_batch(om.model, batch, True, 4.0)


# ---- evaluate_ranking -------------------------------------------------------------------------------------

def test_evaluate_ranking_equals_oracle_metrics():
    rd, om = _synthetic("ml1m", 48, 64)
    np.random.seed(21)
    gen = rd.data_gen(48, None, "test", True, None, -1)
    batches = [next(gen) for _ in range(4)]
    ks = (1, 10, 100)
    for exclude, min_value in ((True, None), (False, 4.0)):
        got = om.model.evaluate_ranking(iter(batches), len(batches), ks=ks, exclude_seen=exclude, min_value=min_value,
                                        workers=0)
        scores, seen, targets = [], [], []
        for b in batches:
            scores.append(om.model.score(b))
            s, t = _truth(b)
            seen += s
            targets += t
        want = ref_rank.metrics(np.concatenate(scores), targets, seen if exclude else None, ks, min_value)
        assert got["rows"] == want["rows"] > 0 and got["AUC_rows"] == want["AUC_rows"]
        for name in want:
            assert got[name] == pytest.approx(want[name], rel=1e-12, abs=1e-15), name
    # through the Prefetcher (workers=1), straight from a generator
    np.random.seed(21)
    again = om.model.evaluate_ranking(rd.data_gen(48, None, "test", True, None, -1), 4, ks=ks)
    np.random.seed(21)
    assert again == om.model.evaluate_ranking(iter(batches), 4, ks=ks, workers=0)
    rd.close()


def test_evaluate_ranking_has_no_side_effects():
    rd, _ = _synthetic("small", 32, 40)
    twins = []
    for _ in range(2):
        np.random.seed(4)
        om = omni_model(1, 40, rd.num_items, 32, dense_activation="sigmoid", use_causal_info=False)
        om.model.compile(optimizers.Adagrad(lr=0.01), "mean_squared_error", rating_range=4.0)
        twins.append(om)
    a, b = twins[0].model, twins[1].model
    np.random.seed(9)
    train = next(rd.data_gen(32, [0.3, 0.8], "train", True, None, -1, pass_through_input_training=True))
    train.flags
    ma, mb = a.train_on_batch(train), b.train_on_batch(train)          # both models have state and a log
    assert ma == mb
    logged, w0 = a.steps_logged(), a.get_weights()
    np.random.seed(10)
    a.evaluate_ranking(rd.data_gen(32, None, "valid", True, None, -1), 3, ks=(5, 50))
    assert a.steps_logged() == logged
    for x, y in zip(a.get_weights(), w0):
        assert np.array_equal(x, y)
    ma, mb = a.train_on_batch(train), b.train_on_batch(train)
    assert ma == mb
    for x, y in zip(a.get_weights(), b.get_weights()):
        assert np.array_equal(x, y)
    rd.close()


def test_column_shard_refuses(golden_datasets):
    ds = golden_datasets["rev"]
    rd = _shard_reader(ds, "fixed_split", 0, 2)
    np.random.seed(11)
    om = ocf_dist.sharded_model(0, 2, 1, 16, ds["n_cols"], 8, dense_activation="sigmoid", use_causal_info=False)
    batch = _batch(rd, "valid", 8)
    with pytest.raises(ValueError, match="column shard"):
        om.model.rank_targets(batch)
    with pytest.raises(ValueError, match="column shard"):
        om.model.evaluate_ranking(iter([batch]), 1, workers=0)
    # the C entry point refuses a sharded model on its own
    h = om.model._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
    dev = batch.upload(None)
    col = np.empty(max(batch.n_entries, 1), np.int32)
    rank = np.empty_like(col)
    ptr = np.empty(batch.n_rows + 1, np.int32)
    cand = np.empty(batch.n_rows, np.int64)
    rc = _lib.lib().ocf_rank_targets(h, dev.handle, 1, float("-inf"), _lib.ptr(col), _lib.ptr(rank), _lib.ptr(ptr),
                                     _lib.ptr(cand), None)
    assert rc != 0 and b"column shard" in _lib.lib().ocf_last_error()
    rd.close()


# ---- train.run --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("eval_mode", ["fixed_split", "ablation"])
def test_train_run_reports_ranking_and_changes_nothing_else(golden_datasets, tmp_path, eval_mode):
    ds = golden_datasets["rev"]
    out = []
    for ks in (None, [10, 100]):
        rd = product_reader(ds, eval_mode)
        cfg = ocf_train.TrainConfig(max_epochs=2, batch_size=4 if eval_mode == "fixed_split" else 2, eval_mode=eval_mode, test_sparsities=[0.1, 0.5],
                                    num_hidden_units=16, model_save_path=str(tmp_path) + "/", dropout_probability=None)
        np.random.seed(2)
        res = ocf_train.run(cfg, reader=rd, rating_range=4.0, save_models=False, verbose=0, ranking_ks=ks)
        out.append(res)
        rd.close()
    base, ranked = out
    assert "test_ranking" not in base
    tr = ranked["test_ranking"]
    per = tr.values() if eval_mode == "ablation" else [tr]
    if eval_mode == "ablation":
        assert set(tr) == {0.1, 0.5}
    for r in per:
        assert set(r) >= {"rows", "AUC_rows", "MRR", "AUC", "HR@10", "NDCG@100", "recall@100", "precision@10"}
        assert r["rows"] > 0 or eval_mode == "ablation"           # ablation: one test batch of two rows
        if r["rows"]:
            assert 0.0 < r["MRR"] <= 1.0 and r["HR@10"] <= r["HR@100"]
    for key in base:
        if key not in ("model", "save_name"):
            np.testing.assert_equal(ranked[key], base[key], err_msg=key)       # NaN == NaN (tiny validation sets)
    for x, y in zip(base["model"].model.get_weights(), ranked["model"].model.get_weights()):
        assert np.array_equal(x, y)
