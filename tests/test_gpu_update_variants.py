"""Every k_row_update instantiation, element by element against a float64 reference (tests/grad_probe.py).

The host picks `k_row_update<NV, KIND, WIDE, HEAVY>` from the padded hidden width (NV = hp / 128) and the catalogue
size: WIDE up to n_cols * hp = 8 Mi floats, HEAVY (CTA-cooperative walk of columns matched by more than 24 rows) up
to n_cols * max(hp[0], hp[L-1]) = 32 Mi, the lean kernel beyond. Each cell below sits just on its variant's side of
the threshold, with a ragged width, and its stepped batch holds columns matched by exactly 24 and 25 rows (and, from
257 rows on, one matched by every row, so that each of the eight warp segments of the heavy walk spans more than
one 32-record round). Per cell: the SGD gradient probe without and with L2, and two-step Adagrad / RMSprop / Adam
rule probes; all from the same initial weights.
"""
import os

import numpy as np
import pytest

from omnidirectional_collaborative_filtering_b200 import _lib, optimizers, synthetic
from omnidirectional_collaborative_filtering_b200.data_reader import data_reader
from omnidirectional_collaborative_filtering_b200.model import omni_model
from tests import grad_probe as gp

MI = 1 << 20
A = 0.5                      # aux_var_value
SPARSITY = [0.3, 0.8]


def n_cols_for(variant, hp):
    """The catalogue just on `variant`'s side of its threshold."""
    return {"wide": (8 * MI) // hp, "heavy": (8 * MI) // hp + 1, "lean": (32 * MI) // hp + 1}[variant]


# nv, variant, B, aux, activation, loss, dropout, pass_through
CELLS = [
    (1, "wide", 4096, "dropout", "sigmoid", "mean_squared_error", None, False),
    (1, "heavy", 257, "causal", "tanh", "mean_absolute_error", 0.2, False),
    (1, "lean", 128, None, "elu", "mean_squared_error", None, True),
    (2, "wide", 100, "both", "softplus", "mean_squared_error", 0.3, False),
    (2, "heavy", 1024, "zeros", "linear", "mean_squared_error", None, False),
    (2, "lean", 257, "dropout", "sigmoid", "mean_absolute_error", None, False),
    (3, "wide", 257, None, "tanh", "mean_absolute_error", None, False),
    (3, "heavy", 8, "dropout", "elu", "mean_squared_error", 0.2, False),
    (3, "lean", 1024, None, "softplus", "mean_squared_error", None, False),
    (4, "wide", 128, "causal", "sigmoid", "mean_squared_error", None, True),
    (4, "heavy", 4096, None, "tanh", "mean_squared_error", 0.2, False),
    (4, "lean", 100, "causal", "linear", "mean_squared_error", None, False),
    (5, "wide", 1024, "zeros", "elu", "mean_absolute_error", None, False),
    (5, "heavy", 100, "both", "sigmoid", "mean_squared_error", None, False),
    (5, "lean", 8, None, "tanh", "mean_squared_error", 0.3, False),
    (6, "wide", 8, "dropout", "softplus", "mean_squared_error", 0.5, False),
    (6, "heavy", 128, None, "linear", "mean_absolute_error", None, False),
    (6, "lean", 4096, None, "sigmoid", "mean_squared_error", None, False),
    (7, "wide", 257, "both", "tanh", "mean_squared_error", None, False),
    (7, "heavy", 1024, "causal", "softplus", "mean_squared_error", 0.2, False),
    (7, "lean", 128, "dropout", "elu", "mean_squared_error", None, False),
    (8, "wide", 100, None, "sigmoid", "mean_squared_error", None, False),
    (8, "heavy", 257, "dropout", "tanh", "mean_squared_error", None, False),
    (8, "lean", 257, None, "elu", "mean_absolute_error", None, False),
]


def cell_width(nv, variant):
    return 1024 if (nv, variant) == (8, "wide") else 128 * nv - 37


# two-layer width lists mixing NV: (widths, n_cols, B, aux, activation, loss, dropout)
WIDTH_LISTS = [
    ([896, 640], 12000, 257, "dropout", "tanh", "mean_squared_error", 0.2),     # WIDE decoder, HEAVY encoder
    ([1024, 130], 20000, 128, None, "sigmoid", "mean_absolute_error", None),    # WIDE 2-wide decoder, 8-wide encoder
]

RULES = [("adagrad", 0.0), ("rmsprop", 0.0), ("adam", 0.0)]


def _store(n_cols, B, seed):
    """B rows of 8..32 random columns, plus column n_cols//3 in exactly 24 rows, n_cols//2 in exactly 25 and, when
    B >= 257, the last column in every row."""
    rs = np.random.RandomState(seed)
    special = [n_cols // 3, n_cols // 2, n_cols - 1]
    rows, cols = [], []
    for b in range(B):
        c = np.unique(rs.randint(0, n_cols - 1, size=int(rs.randint(8, 33))))
        c = c[(c != special[0]) & (c != special[1])]
        rows.append(np.full(c.size, b)); cols.append(c)
    if B >= 25:
        for c, k in ((special[0], 24), (special[1], 25)):
            r = np.sort(rs.choice(B, k, replace=False))
            rows.append(r); cols.append(np.full(k, c))
    if B >= 257:
        rows.append(np.arange(B)); cols.append(np.full(B, special[2]))
    r, c = np.concatenate(rows), np.concatenate(cols)
    v = rs.randint(1, 6, size=r.size).astype(np.float32)
    csr, keys = synthetic.csr_from_coo(r, c, v, n_cols, row_keys=np.arange(B))
    none = np.zeros(B, dtype=bool)
    fs = synthetic.FixedSplit(n_cols, csr, keys, csr, csr, keys, none, csr, csr, keys, none, 4.0)
    return fs, special


class Cell(object):
    """A store, its one stepped batch and a model over it."""

    def __init__(self, widths, n_cols, B, aux, act, loss, pdrop, pt=False, seed=0, store=_store):
        self.widths, self.n_cols, self.B, self.aux, self.act, self.loss, self.pdrop = widths, n_cols, B, aux, act, loss, pdrop
        fs, self.special = store(n_cols, B, seed)
        self.rd = data_reader(n_cols, B, "", eval_mode="fixed_split", data=fs, rng_on_device=False)
        np.random.seed(seed + 1)
        self.batch = next(self.rd.data_gen(B, SPARSITY, "train", False, aux, A, pass_through_input_training=pt))
        self.sb = gp.from_batch(self.batch)
        self.rho = gp.rho_for(B, [gp.pad(w) for w in widths])
        self._ref = {}

    def counts(self):
        csr = self.batch.source.csr
        rp = csr.rowptr
        rows = self.batch.rows.astype(np.int64)
        cols = np.concatenate([csr.col[rp[r]:rp[r + 1]] for r in rows])
        return np.bincount(cols, minlength=self.n_cols)

    def model(self, l2=None, seed=7):
        np.random.seed(seed)
        om = omni_model(len(self.widths), self.widths, self.n_cols, self.B, dense_activation=self.act,
                        use_causal_info=self.aux is not None, use_both_masks=self.aux == "both",
                        l2_weight_regulatization=l2, dropout_probability=self.pdrop, auxilliary_mask_type=self.aux)
        w = om.model.get_weights()
        rs = np.random.RandomState(seed + 1)
        for i in range(1, len(w), 2):
            w[i] = (rs.normal(size=w[i].shape) * 0.05).astype(np.float32)
        om.model.set_weights(w)
        net = gp.Net(widths=list(self.widths), activation=self.act, loss=self.loss, l2=l2, p_drop=self.pdrop,
                     dropout_seed=om.dropout_seed)
        return om, net, w

    def reference(self, om, net, W):
        """(g64, S) of the model's next step from weights W (cached per weights / dropout step)."""
        step = om.model._step if net.p_drop is not None else -1
        key = (id(W), step, net.l2)
        if key not in self._ref:           # the entry holds W, so its id is not reused while cached
            self._ref[key] = (W, gp.reference(net, self.sb, W, gp.keep_masks(net, max(step, 0), self.B), self.rho))
        return self._ref[key][1]

    def sgd_probe(self, om, net, W0, label):
        g64, S = self.reference(om, net, W0)
        L = gp.probe_lr(g64)
        om.model.set_weights(W0)
        om.model.compile(optimizers.SGD(lr=L), self.loss, rating_range=4.0)
        om.model.train_on_batch(self.batch)
        return gp.check_sgd(W0, om.model.get_weights(), L, g64, S, self.rho, label=label)

    def rule_probe(self, om, net, W0, kind, decay, label):
        g64, S = self.reference(om, net, W0)
        E, lr = gp.rule_params(kind, g64)
        opt = {"adagrad": lambda: optimizers.Adagrad(lr=lr, epsilon=E, decay=decay),
               "rmsprop": lambda: optimizers.RMSprop(lr=lr, rho=0.9, epsilon=E, decay=decay),
               "adam": lambda: optimizers.Adam(lr=lr, beta_1=0.9, beta_2=0.999, epsilon=E, decay=decay)}[kind]()
        probe = gp.RuleProbe(kind, E, lr, decay=decay, **gp.RULE_DEFAULTS[kind])
        om.model.set_weights(W0)
        om.model.compile(opt, self.loss, rating_range=4.0)
        if om.model._handle is not None:
            _lib.check(_lib.lib().ocf_model_reset_optimizer(om.model._handle))
        om.model.train_on_batch(self.batch)
        W1 = om.model.get_weights()
        fails = probe.check(W0, W1, g64, S, self.rho, label=label + " step 1 ")
        states, errs = probe.rebuild(W0, W1)
        g64b, Sb = self.reference(om, net, W1)
        om.model.train_on_batch(self.batch)
        fails += probe.check(W1, om.model.get_weights(), g64b, Sb, self.rho, states=states, g1_err=errs,
                             label=label + " step 2 ")
        self._ref.pop((id(W1), om.model._step - 1 if net.p_drop is not None else -1, net.l2), None)
        return fails

    def close(self):
        self.rd.close()


def _run_cell(cell, rules, label):
    fails = []
    om, net, W0 = cell.model()
    fails += cell.sgd_probe(om, net, W0, label + " sgd ")
    for kind, decay in rules:
        fails += cell.rule_probe(om, net, W0, kind, decay, "%s %s" % (label, kind))
    om.model.close()
    om, net, W0 = cell.model(l2=0.01)
    fails += cell.sgd_probe(om, net, W0, label + " sgd+l2 ")
    om.model.close()
    return fails


@pytest.mark.gpu
@pytest.mark.parametrize("cell", CELLS, ids=["nv%d-%s-B%d" % c[:3] for c in CELLS])
def test_update_variant_cell(cell):
    nv, variant, B, aux, act, loss, pdrop, pt = cell
    width = cell_width(nv, variant)
    n_cols = n_cols_for(variant, gp.pad(width))
    launches = gp.row_launches(n_cols, [width], "sgd")
    assert [(v, w, h) for v, _, w, h in launches] == [(nv, variant == "wide", variant != "lean")]
    c = Cell([width], n_cols, B, aux, act, loss, pdrop, pt, seed=nv)
    try:
        counts = c.counts()
        if B >= 25:
            assert counts[c.special[0]] == 24 and counts[c.special[1]] == 25
        if B >= 257:
            assert counts.max() == B and counts[c.special[2]] == B
        rules = RULES[:2] + [("adam", 0.01 if nv % 2 else 0.0)]      # half the Adam cells run a decaying lr
        fails = _run_cell(c, rules, "nv%d %s" % (nv, variant))
        assert fails == [], "\n".join(fails)
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", WIDTH_LISTS, ids=["%dx%d" % tuple(w[0]) for w in WIDTH_LISTS])
def test_width_list_mixing_nv(case):
    widths, n_cols, B, aux, act, loss, pdrop = case
    launches = gp.row_launches(n_cols, widths, "sgd")
    assert len(launches) == 2 and launches[0][2] and not launches[1][2]     # a WIDE decoder in a non-WIDE model
    c = Cell(widths, n_cols, B, aux, act, loss, pdrop, seed=11)
    try:
        fails = _run_cell(c, RULES, "%s" % widths)
        assert fails == [], "\n".join(fails)
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nv", range(1, 9))
def test_row_parallel_gradient_rows(nv):
    """World-1 row-parallel step: k_row_update<NV, KIND_GRAD> stores gradient rows, k_dense_update applies them."""
    width = 128 * nv - 37
    c = Cell([width], 3000, 100, "dropout" if nv % 2 else None, "tanh", "mean_squared_error", None, seed=20 + nv)
    try:
        om, net, W0 = c.model()
        om.model.native = (None, _lib.PAR_ROWS)
        fails = c.sgd_probe(om, net, W0, "row-parallel nv%d " % nv)
        assert fails == [], "\n".join(fails)
        om.model.close()
    finally:
        c.close()


@pytest.mark.gpu
def test_eager_captured_and_replayed_steps_agree(capfd):
    """The same SGD step from the same weights on one device batch: plain launches, then captured into a CUDA
    graph, then replayed. The weights it leaves are bit-identical, and each is inside the probe's bound."""
    c = Cell([300], n_cols_for("heavy", 384), 257, "causal", "sigmoid", "mean_squared_error", None, seed=5)
    try:
        check_graph_steps(c, capfd)
    finally:
        c.close()


def check_graph_steps(c, capfd):
    """Runs one SGD step of cell `c` three times from the same weights on one device batch (eager, captured,
    replayed) and checks the weights each leaves against the probe and against each other, bit for bit. The cell has
    no dropout: run k is step k, and the probe's reference is the step-0 one."""
    old = os.environ.get("OCF_DEBUG_GRAPH")
    os.environ["OCF_DEBUG_GRAPH"] = "1"
    try:
        om, net, W0 = c.model()
        g64, S = c.reference(om, net, W0)
        L = gp.probe_lr(g64)
        om.model.compile(optimizers.SGD(lr=L), c.loss, rating_range=4.0)
        om.model._ensure(c.batch.n_rows, c.batch.n_entries, c.batch.aux_type, c.batch.reader)
        dev = c.batch.upload(om.model.stream)
        outs, msgs = [], []
        for k in range(3):
            om.model.set_weights(W0)                   # keeps the captured graphs (weights are written in place)
            capfd.readouterr()
            om.model.step_on_device_batch(dev, c.B, k)
            W1 = om.model.get_weights()
            msgs.append(capfd.readouterr().err)
            outs.append(W1)
            assert gp.check_sgd(W0, W1, L, g64, S, c.rho, label="run %d " % k) == []
        assert "graph" not in msgs[0]
        assert "step graph captured" in msgs[1] and "failed" not in msgs[1]
        assert "graph" not in msgs[2]                  # the third step ran the captured graph
        for k in (1, 2):
            for a, b in zip(outs[0], outs[k]):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        om.model.close()
    finally:
        if old is None:
            os.environ.pop("OCF_DEBUG_GRAPH", None)
        else:
            os.environ["OCF_DEBUG_GRAPH"] = old


def test_cells_reach_every_instantiation():
    """The union of the launches of every probe above is every instantiation the dispatch can reach."""
    seen = set()
    kinds = ["sgd", "adagrad", "rmsprop", "adam"]
    for nv, variant, *_ in CELLS:
        width = cell_width(nv, variant)
        for k in kinds:
            seen.update(gp.row_launches(n_cols_for(variant, gp.pad(width)), [width], k))
    for widths, n_cols, *_ in WIDTH_LISTS:
        for k in kinds:
            seen.update(gp.row_launches(n_cols, widths, k))
    for nv in range(1, 9):
        seen.update(gp.row_launches(3000, [128 * nv - 37], "sgd", row_parallel=True))
    assert seen == gp.all_instantiations()
