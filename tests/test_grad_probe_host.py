"""Host checks of tests/grad_probe.py: its sparse float64 reference is `RefModel`'s gradient, its bounds accept a
float32 step of the oracle, and they reject the faults a broken update kernel would make."""
import numpy as np
import pytest

from oracle import ref_batches, ref_model
from tests import grad_probe as gp
from tests.helpers import oracle_data, product_reader

A = 0.5          # a non-unit aux_var_value


def _batch(B, N, aux, seed, pass_through=False, heavy_cols=()):
    """Dense feed of a random split batch; every column of `heavy_cols` is held by the first 32 rows."""
    rs = np.random.RandomState(seed)
    held = rs.random_sample((B, N)) < 0.15
    for c in heavy_cols:
        held[:, c] = False
        held[:min(B, 32), c] = True
    vals = rs.randint(1, 6, size=(B, N)).astype(np.float64)
    inp = held & (rs.random_sample((B, N)) < 0.6)
    tgt = held & (~inp | pass_through)
    arrays = (np.where(inp, A, 0.0), np.where(tgt, A, 0.0), np.where(inp, vals, 0.0), np.where(tgt, vals, 0.0),
              np.where(held, A, 0.0))
    return ref_batches.feed_list(arrays, aux), arrays[3]


def _models(aux, widths, act, loss, l2, pdrop, N, B, seed=0):
    kw = dict(dense_activation=act, use_causal_info=aux is not None, use_both_masks=aux == "both",
              l2_weight_regulatization=l2, dropout_probability=pdrop)
    r64 = ref_model.RefModel(len(widths), widths, N, B, dtype=np.float64, rng=np.random.RandomState(seed), **kw)
    rs = np.random.RandomState(seed + 1)
    w = r64.get_weights()
    for i in range(1, len(w), 2):
        w[i] = rs.normal(size=w[i].shape) * 0.05
    w = [x.astype(np.float32) for x in w]
    r64.set_weights(w)
    r32 = ref_model.RefModel(len(widths), widths, N, B, dtype=np.float32, rng=np.random.RandomState(seed), **kw)
    r32.set_weights(w)
    for r in (r64, r32):
        r.compile(ref_model.RefOptimizer("sgd", lr=1.0), loss)
    net = gp.Net(widths=list(widths), activation=act, loss=loss, l2=l2, p_drop=pdrop, dropout_seed=12345)
    return r64, r32, net, w


CASES = [
    # aux, widths, act, loss, l2, pdrop, pass_through
    (None, [24], "sigmoid", "mean_squared_error", None, None, False),
    ("dropout", [40], "tanh", "mean_absolute_error", 0.01, 0.3, False),
    ("causal", [16, 20], "elu", "mean_squared_error", None, None, True),
    ("both", [30, 12, 18], "softplus", "mean_absolute_error", 0.001, 0.2, True),
    ("zeros", [33], "linear", "mean_squared_error", 0.01, None, False),
    ("dropout", [136, 24], "sigmoid", "mean_squared_error", None, 0.5, False),
]


def _keeps(net, B):
    return gp.keep_masks(net, 3, B)


@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_sparse_reference_equals_refmodel(case):
    aux, widths, act, loss, l2, pdrop, pt = case
    B, N = 12, 50
    feed, t = _batch(B, N, aux, 1, pt)
    r64, _, net, _ = _models(aux, widths, act, loss, l2, pdrop, N, B)
    keeps = _keeps(net, B)
    _, want = r64.gradients(feed, t, dropout_masks=keeps if pdrop else None)
    got, S = gp.reference(net, gp.from_dense(feed, t, aux), r64.get_weights(), keeps, 2e-5)
    for k, (g, w, s) in enumerate(zip(got, want, S)):
        assert g.shape == w.shape
        np.testing.assert_allclose(g, w, rtol=1e-12, atol=1e-12 * max(1e-30, float(np.abs(w).max())), err_msg="array %d" % k)
        assert np.all(s >= np.abs(g) - 1e-15 * np.abs(g).max())        # S bounds the gradient itself


def _sgd_device(r32, feed, t, keeps, L, pdrop, fault=None):
    """The float32 oracle standing in for the device: one SGD(lr=L) step, optionally with a fault."""
    W0 = r32.get_weights()
    _, g = r32.gradients(feed, t, dropout_masks=keeps if pdrop else None)
    g = [x.copy() for x in g]
    if fault is not None:
        g = fault(g)
    return W0, [w - np.float32(L) * x for w, x in zip(W0, g)]


def _probe(case, fault=None, B=64, N=60, heavy=()):
    aux, widths, act, loss, l2, pdrop, pt = case
    feed, t = _batch(B, N, aux, 2, pt, heavy)
    r64, r32, net, w = _models(aux, widths, act, loss, l2, pdrop, N, B)
    keeps = _keeps(net, B)
    sb = gp.from_dense(feed, t, aux)
    rho = gp.rho_for(B, [gp.pad(x) for x in widths])
    g64, S = gp.reference(net, sb, w, keeps, rho)
    L = gp.probe_lr(g64)
    W0, W1 = _sgd_device(r32, feed, t, keeps, L, pdrop, fault)
    return gp.check_sgd(W0, W1, L, g64, S, rho), (feed, t, r32, keeps, g64, L, w, net, sb, rho)


@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_sgd_probe_accepts_float32_oracle(case):
    fails, _ = _probe(case)
    assert fails == []


def test_sgd_probe_rejects_lost_heavy_matches():
    """Columns matched by more than 24 rows lose one eighth of their matches (one warp segment of the heavy walk)."""
    case = CASES[1]
    aux, widths, act, loss, l2, pdrop, pt = case
    heavy = (3, 17, 41)
    B, N = 64, 60
    feed, t = _batch(B, N, aux, 2, pt, heavy)
    # the same batch without rows 28..31 of the heavy columns (the last eighth of their 32 matches)
    feed2, t2 = [np.array(f, dtype=np.float64) for f in feed], np.array(t, dtype=np.float64)
    for f in feed2 + [t2]:
        for c in heavy:
            f[28:32, c] = 0.0
    r64, r32, net, w = _models(aux, widths, act, loss, l2, pdrop, N, B)
    keeps = _keeps(net, B)
    _, gfull = r32.gradients(feed, t, dropout_masks=keeps)
    _, gdrop = r32.gradients(feed2, t2, dropout_masks=keeps)
    rows = [c + k * N for k in range(gp.blocks_of(aux)) for c in heavy]

    def fault(g):
        g[0][rows] = gdrop[0][rows]                 # encoder rows of the heavy columns
        g[-2][:, list(heavy)] = gdrop[-2][:, list(heavy)]
        g[-1][list(heavy)] = gdrop[-1][list(heavy)]
        return g
    rho = gp.rho_for(B, [gp.pad(x) for x in widths])
    g64, S = gp.reference(net, gp.from_dense(feed, t, aux), w, keeps, rho)
    L = gp.probe_lr(g64)
    W0, W1 = _sgd_device(r32, feed, t, keeps, L, pdrop, fault)
    fails = gp.check_sgd(W0, W1, L, g64, S, rho)
    assert len(fails) >= 2, fails                  # encoder and decoder both caught
    assert not np.allclose(gfull[-2], gdrop[-2])


@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_sgd_probe_rejects_doubled_array(k):
    def fault(g):
        g[k] = g[k] * np.float32(2.0)
        return g
    fails, _ = _probe(CASES[2], fault)
    assert len(fails) == 1 and fails[0].startswith("array %d" % k), fails


def test_sgd_probe_rejects_row_written_to_neighbour():
    case = CASES[0]
    fails, ctx = _probe(case)
    assert fails == []
    feed, t, r32, keeps, g64, L, w, net, sb, rho = ctx
    W0, W1 = _sgd_device(r32, feed, t, keeps, L, None)
    c = int(sb.t_col[0])
    n = (c + 1) % sb.N
    W1[-2][:, n] = W1[-2][:, c]                    # decoder row of column c lands on column c+1
    W1[-2][:, c] = W0[-2][:, c]
    fails = gp.check_sgd(W0, W1, L, g64, gp.reference(net, sb, w, keeps, rho)[1], rho)
    assert len(fails) == 1 and fails[0].startswith("array %d" % (len(W0) - 2)), fails


def _rule_run(kind, fault_state=False, decay=0.0):
    aux, widths, act, loss, l2, pdrop, pt = CASES[1]
    B, N = 64, 60
    feed, t = _batch(B, N, aux, 2, pt, (5,))
    r64, r32, net, w = _models(aux, widths, act, loss, l2, pdrop, N, B)
    keeps = _keeps(net, B)
    sb = gp.from_dense(feed, t, aux)
    rho = gp.rho_for(B, [gp.pad(x) for x in widths])
    g64, S = gp.reference(net, sb, w, keeps, rho)
    E, lr = gp.rule_params(kind, g64)
    kw = gp.RULE_DEFAULTS[kind]
    r32.compile(ref_model.RefOptimizer(kind, lr=lr, epsilon=E, decay=decay, **kw), loss)
    probe = gp.RuleProbe(kind, E, lr, decay=decay, **kw)
    W0 = r32.get_weights()
    r32.train_on_batch(feed, t, dropout_masks=keeps)
    W1 = r32.get_weights()
    fails = probe.check(W0, W1, g64, S, rho, label="step 1 ")
    states, errs = probe.rebuild(W0, W1)
    if fault_state:
        r32.optimizer.state = {}                  # the state read as zero on step 2
    r32.train_on_batch(feed, t, dropout_masks=keeps)
    W2 = r32.get_weights()
    g64b, Sb = gp.reference(net, sb, W1, keeps, rho)
    fails += probe.check(W1, W2, g64b, Sb, rho, states=states, g1_err=errs, label="step 2 ")
    return fails


@pytest.mark.parametrize("kind,decay", [("adagrad", 0.0), ("rmsprop", 0.0), ("adam", 0.0), ("adam", 0.25)])
def test_rule_probe_accepts_float32_oracle(kind, decay):
    assert _rule_run(kind, decay=decay) == []


def test_rule_probe_rejects_rmsprop_state_read_as_zero():
    fails = _rule_run("rmsprop", fault_state=True)
    assert fails and all(f.startswith("step 2") for f in fails), fails


@pytest.mark.parametrize("pt", [False, True], ids=["split", "pass-through"])
@pytest.mark.parametrize("aux", [None, "causal", "dropout", "zeros", "both"])
def test_from_batch_keeps_last_write_of_repeated_columns(golden_datasets, aux, pt):
    """`from_batch` of the product's batches equals `from_dense` of the oracle's dense batches on a store whose rows
    repeat columns: one value per (row, column, array), the last write's (data_reader.py:158-169)."""
    ds = golden_datasets["rev"]
    rd = product_reader(ds, "fixed_split")
    rd.rng_on_device = False          # host stream where a GPU exists too: the oracle replays it
    np.random.seed(3)
    gen = rd.data_gen(8, [0.2, 0.9], "train", True, aux, -1, pass_through_input_training=pt)
    rgen = ref_batches.batch_stream(oracle_data(ds, "fixed_split"), 8, [0.2, 0.9], "train", True, aux, -1,
                                    pass_through_input_training=pt, rng=np.random.RandomState(3))
    repeats = 0
    while True:
        batch = next(gen)
        if batch is None:
            break
        csr = batch.source.csr
        for r in batch.rows:
            cols, _ = csr.row(int(r))
            repeats += len(cols) - np.unique(cols).size
        feed, targets = next(rgen)
        got, want = gp.from_batch(batch), gp.from_dense(feed, targets, aux)
        assert (got.B, got.N, got.nblk) == (want.B, want.N, want.nblk)
        assert np.array_equal(got.x0.toarray(), want.x0.toarray())
        og, ow = np.lexsort((got.t_col, got.t_row)), np.lexsort((want.t_col, want.t_row))
        for name in ("t_row", "t_col", "t_val", "t_mask"):
            assert np.array_equal(getattr(got, name)[og], getattr(want, name)[ow]), name
    assert repeats > 0                 # the batches did hold rows that repeat a column
    rd.close()


def test_variant_classifier_thresholds():
    M = 1 << 20
    # one width: WIDE up to n_cols * hp = 8 Mi, then HEAVY up to 32 Mi, then lean
    assert gp.row_launches(65536, [100], "adagrad") == [(1, 1, True, True)]
    assert gp.row_launches(65537, [100], "adagrad") == [(1, 1, False, True)]
    assert gp.row_launches(262144, [128], "sgd") == [(1, 0, False, True)]
    assert gp.row_launches(262145, [128], "sgd") == [(1, 0, False, False)]
    assert gp.row_launches(8 * M // 1024, [1000], "adam") == [(8, 3, True, True)]
    assert gp.row_launches(32 * M // 1024 + 1, [1024], "rmsprop") == [(8, 2, False, False)]
    assert gp.row_launches(32769, [1024], "adam") == [(8, 3, False, False)]
    assert gp.row_launches(8192, [1024], "adam") == [(8, 3, True, True)]
    # two ends of a width list: one launch per padded width, HEAVY decided by the wider end
    assert gp.row_launches(40000, [1024, 100], "sgd") == [(1, 0, True, True), (8, 0, False, False)]
    assert gp.row_launches(20000, [1024, 130], "sgd") == [(2, 0, True, True), (8, 0, False, True)]
    assert gp.row_launches(20000, [1024, 130], "sgd", row_parallel=True) == [(2, 4, False, False), (8, 4, False, False)]
    assert len(gp.all_instantiations()) == 8 * 4 * 3 + 8
