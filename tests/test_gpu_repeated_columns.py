"""Training on a store whose rows repeat a column, element by element against a float64 reference (tests/grad_probe.py).

The dense arrays of the reference are last-write-wins (data_reader.py:158-169), so a row that repeats a column feeds
one value per array: the input of its last input rating, the target of its last target rating. The update's work list
(K4a) holds one match record per (column, batch row) that merges the row's ratings of the column. The stores below
repeat columns inside rows so that a cell's input and target come from different ratings, and hold one such column
in every row: matched by more than 24 batch rows, it takes the heavy (CTA-cooperative) walk of the update.
"""
import numpy as np
import pytest

from omnidirectional_collaborative_filtering_b200 import synthetic
from tests import grad_probe as gp
from tests.test_gpu_update_variants import Cell, _run_cell, check_graph_steps, n_cols_for

pytestmark = pytest.mark.gpu


def _repeating_store(n_cols, B, seed):
    """B rows of 8..32 random columns, about a third of them rated again later in the row, plus column n_cols // 2
    rated two to four times in every row."""
    rs = np.random.RandomState(seed)
    hot = n_cols // 2
    rows, cols = [], []
    for b in range(B):
        c = np.unique(rs.randint(0, n_cols - 1, size=int(rs.randint(8, 33))))
        c = c[c != hot]
        again = c[rs.random_sample(c.size) < 0.35]
        c = np.concatenate([c, np.full(int(rs.randint(2, 5)), hot), again])
        c = c[rs.permutation(c.size)]
        rows.append(np.full(c.size, b)); cols.append(c)
    r, c = np.concatenate(rows), np.concatenate(cols)
    v = rs.randint(1, 6, size=r.size).astype(np.float32)
    csr, keys = synthetic.csr_from_coo(r, c, v, n_cols, row_keys=np.arange(B))
    none = np.zeros(B, dtype=bool)
    fs = synthetic.FixedSplit(n_cols, csr, keys, csr, csr, keys, none, csr, csr, keys, none, 4.0)
    return fs, [hot]


def _split_cells(cell):
    """Cells (batch row, column) whose live input and live target are different ratings of the row."""
    batch = cell.batch
    csr = batch.source.csr
    f = np.asarray(batch.flags, dtype=bool)
    out, pos = 0, 0
    for b, r in enumerate(batch.rows):
        cols, _ = csr.row(int(r))
        fr = f[pos:pos + len(cols)]
        pos += len(cols)
        last_in, last_tg = {}, {}
        for j, c in enumerate(cols):
            if fr[j]:
                last_in[c] = j
            if not fr[j] or batch.pass_through:
                last_tg[c] = j
        out += sum(1 for c in last_in if c in last_tg and last_in[c] != last_tg[c])
    return out


# width, n_cols, B, aux, activation, loss, dropout, pass_through
CELLS = [
    (300, 3000, 64, "both", "sigmoid", "mean_squared_error", 0.2, False),
    (200, n_cols_for("heavy", 256), 128, "zeros", "tanh", "mean_absolute_error", None, True),
]


def _cell(case, seed):
    width, n_cols, B, aux, act, loss, pdrop, pt = case
    c = Cell([width], n_cols, B, aux, act, loss, pdrop, pt, seed=seed, store=_repeating_store)
    assert c.rd.store("train").info()["has_dups"] == 1
    assert _split_cells(c) > 0
    csr = c.batch.source.csr
    assert sum(c.special[0] in csr.row(int(r))[0] for r in c.batch.rows) > 24
    return c


@pytest.mark.parametrize("case", CELLS, ids=[c[3] for c in CELLS])
def test_repeated_columns_probes(case):
    """SGD, SGD + L2 (every row updated) and two-step RMSprop / Adam probes."""
    c = _cell(case, seed=31)
    try:
        fails = _run_cell(c, [("rmsprop", 0.0), ("adam", 0.0)], "repeated %s" % case[3])
        assert fails == [], "\n".join(fails)
    finally:
        c.close()


def test_repeated_columns_eager_captured_and_replayed_steps_agree(capfd):
    # no dropout: the three runs pass their own step numbers, which seed the dropout masks
    c = _cell((300, 3000, 64, "both", "sigmoid", "mean_squared_error", None, False), seed=32)
    try:
        check_graph_steps(c, capfd)
    finally:
        c.close()
