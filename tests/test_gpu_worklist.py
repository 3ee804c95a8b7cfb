"""GPU parity of the batch-side work list (K4a run ahead of the step on the batch's own stream, ocf_api.cu
`prepare_worklist`) and of the hidden-layer overlap, in the cases where the list outlives one step or is rebuilt:

* the same fill stepped several times (the list is reused, only K4b's cursors start over), then re-gathered;
* trainable flags changed between steps on the same ring of batch objects (the list's signature changes: decoder /
  encoder rows leave and re-enter it);
* the same steps with the grouping inside the step (a step driven phase by phase keeps it there) and ahead of it:
  bit-identical weights.
Against the NumPy oracle on the same batches (reference: model.py:34-99, train.py:50-51). The golden "rev" train store
repeats columns inside rows (asserted in `_streams`), so these steps also cover the list's merged match records."""
import ctypes as C

import numpy as np
import pytest

from oracle import ref_batches
from omnidirectional_collaborative_filtering_b200 import _lib
from tests.helpers import oracle_data, product_reader
from tests.test_gpu_model import _close, _close_weights, _pair

pytestmark = pytest.mark.gpu


def _streams(ds, aux, pt, seed=3, B=8):
    rd = product_reader(ds, "fixed_split")
    assert rd.store("train").info()["has_dups"] == 1
    data = oracle_data(ds, "fixed_split")
    np.random.seed(seed)
    gen = rd.data_gen(B, [0.2, 0.9], "train", True, aux, -1, pass_through_input_training=pt)
    rgen = ref_batches.batch_stream(data, B, [0.2, 0.9], "train", True, aux, -1, pass_through_input_training=pt,
                                    rng=np.random.RandomState(seed))
    return rd, gen, rgen


def _step_resident(m, dev, n_rows, step):
    """One train step on an already-filled DeviceBatch through the C ABI, metrics back."""
    args = _lib.StepArgs()
    args.dropout_seed = m.owner.dropout_seed
    args.step = step
    rec = np.empty(_lib.N_METRICS, dtype=np.float32)
    _lib.check(_lib.lib().ocf_train_step(m._handle, dev.handle, C.byref(args), _lib.ptr(rec), None))
    return [float(x) for x in rec[:6]]


@pytest.mark.parametrize("case", [(None, 1, 24, "sigmoid", None, None, "adagrad"), ("dropout", 2, 40, "tanh", None, None, "rmsprop"),
                                  ("both", 2, [36, 20], "elu", 0.01, None, "adam")], ids=["adagrad", "rmsprop-hidden", "adam-widths"])
def test_same_fill_stepped_repeatedly(golden_datasets, case):
    aux, layers, width, act, l2, pdrop, opt = case
    ds = golden_datasets["rev"]
    om, ref = _pair(ds, aux, layers, width, act, l2, pdrop, opt, "mean_squared_error")
    rd, gen, rgen = _streams(ds, aux, False)
    b = next(gen)
    feed, targets = next(rgen)
    m = om.model
    m._ensure(b.n_rows, b.n_entries, b.aux_type, b.reader)
    dev = b.upload(None)
    for step in range(4):                       # plain, captured, replayed, replayed: all on ONE fill
        got = _step_resident(m, dev, b.n_rows, step)
        want = ref.train_on_batch(feed, targets)
        _close(got, want)
    # a re-gather of the same rows and flags is a new fill: the list is built again
    _lib.check(_lib.lib().ocf_batch_regather(dev.handle, None))
    _close(_step_resident(m, dev, b.n_rows, 4), ref.train_on_batch(feed, targets))
    for g, w in zip(m.get_weights(), ref.get_weights()):
        _close_weights(g, w, m.optimizer.lr)
    rd.close()


def test_signature_changes_between_steps(golden_datasets):
    """Decoder frozen, thawed, encoder frozen, thawed on the same ring of batch objects: every change rebuilds the lists."""
    ds = golden_datasets["rev"]
    aux = "causal"
    om, ref = _pair(ds, aux, 2, 40, "sigmoid", None, None, "adagrad", "mean_squared_error")
    m = om.model
    rd = product_reader(ds, "fixed_split")
    data = oracle_data(ds, "fixed_split")

    def steps(n, seed):
        # an epoch of the golden set is 5 batches: a fresh generator per segment, the reader's ring of batch objects stays
        np.random.seed(seed)
        gen = rd.data_gen(8, [0.2, 0.9], "train", True, aux, -1, pass_through_input_training=True)
        rgen = ref_batches.batch_stream(data, 8, [0.2, 0.9], "train", True, aux, -1, pass_through_input_training=True,
                                        rng=np.random.RandomState(seed))
        for _ in range(n):
            got = m.train_on_batch(next(gen))
            feed, targets = next(rgen)
            _close(got, ref.train_on_batch(feed, targets))

    steps(4, 3)
    om._set_trainable(2, False)                  # freeze the decoder: its rows leave the work list
    ref.trainable[2] = False
    steps(4, 4)
    om._set_trainable(2, True)
    ref.trainable[2] = True
    om._set_trainable(0, False)                  # ... then the encoder's
    ref.trainable[0] = False
    steps(4, 5)
    om._set_trainable(0, True)
    ref.trainable[0] = True
    steps(3, 6)
    for g, w in zip(m.get_weights(), ref.get_weights()):
        _close_weights(g, w, m.optimizer.lr)
    rd.close()


def test_ahead_and_in_step_lists_agree(golden_datasets):
    """The same steps with the grouping inside the step (phase calls keep it there) and ahead of it give the same
    weights bit for bit: both build the same match order."""
    ds = golden_datasets["rev"]
    aux = "dropout"
    res = []
    for phased in (False, True):
        om, _ = _pair(ds, aux, 1, 64, "sigmoid", None, None, "adagrad", "mean_squared_error")
        rd, gen, _ = _streams(ds, aux, False)
        m = om.model
        for step in range(5):
            b = next(gen)
            h = m._ensure(b.n_rows, b.n_entries, b.aux_type, b.reader)
            dev = b.upload(None)
            args = m._args(b)
            args.step = step
            if not phased:
                _lib.check(_lib.lib().ocf_train_step(h, dev.handle, C.byref(args), None, None))
            else:
                for ph in (1, 2, 3):
                    args.phase = ph
                    _lib.check(_lib.lib().ocf_train_step(h, dev.handle, C.byref(args), None, None))
        res.append([w.copy() for w in m.get_weights()])
        rd.close()
    for a, b2 in zip(*res):
        np.testing.assert_array_equal(a, b2)
