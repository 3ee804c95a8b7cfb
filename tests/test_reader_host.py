"""Host logic of the product's data_reader mirror (no GPU): set handling, RNG replay, batch
order and flags, checked against the reference's golden batches by densifying the (row ids,
flags) plan on the host."""
import numpy as np
import pytest

from tests.helpers import golden_batch, host_densify, product_reader


def test_reader_plans_match_reference(golden_cases, golden_datasets, golden_batches):
    for case in golden_cases:
        ds = golden_datasets[case["dataset"]]
        rd = product_reader(ds, case["eval_mode"])
        rd.rng_on_device = False      # host stream where a GPU exists too: rng_after is read from np.random itself
        np.random.seed(case["seed"])
        if case["eval_mode"] == "ablation":
            rd.split_for_validation(case["val_split"], seed=case["split_seed"])
            assert np.array_equal(rd.train_set, golden_batches[case["id"] + "/train_set"])
            assert np.array_equal(rd.test_set, golden_batches[case["id"] + "/test_set"])
        else:
            assert rd.train_set == list(ds["train"].keys())
            assert (rd.train_set_size, rd.val_set_size, rd.test_set_size) == \
                (len(ds["train"]), len(ds["valid"][1]), len(ds["test"][1]))
        gen = rd.data_gen(case["B"], case["sparsity"], train_val_test=case["which"], shuffle=case["shuffle"],
                          auxilliary_mask_type=case["aux"], aux_var_value=case["aux_value"],
                          return_target_count=case["rtc"], pass_through_input_training=case["pass_through"])
        for n in range(case["n_batches"]):
            batch = next(gen)
            feed, targets, tc = golden_batch(golden_batches, case, n)
            got_feed, got_t = host_densify(batch)
            assert len(got_feed) == len(feed), case["id"]
            for g, w in zip(got_feed, feed):
                assert np.array_equal(g, w), (case["id"], n)
            assert np.array_equal(got_t, targets)
            assert len(batch) == (3 if tc is not None else 2)
            if tc is not None:
                assert batch.target_count == int(tc)
        assert next(gen) is None and next(gen) is None
        assert np.random.random_sample() == float(golden_batches[case["id"] + "/rng_after"]), case["id"]


def test_scalar_sparsity_is_accepted(golden_datasets):
    rd = product_reader(golden_datasets["rev"], "ablation")
    rd.rng_on_device = False          # host stream where a GPU exists too: a's flags are drawn before the reseed
    rd.split_for_validation([0.5, 0.25, 0.25], seed=1)
    np.random.seed(4)
    a = next(rd.data_gen(4, 0.4, "test"))
    np.random.seed(4)
    b = next(rd.data_gen(4, [0.4, 0.4], "test"))
    assert np.array_equal(a.flags, b.flags) and np.array_equal(a.rows, b.rows)


def test_max_batch_entries_bounds_every_batch(golden_datasets):
    rd = product_reader(golden_datasets["fwd"], "fixed_split")
    cap = rd.max_batch_entries(8)
    for which in ("train", "valid", "test"):
        gen = rd.data_gen(8, [0.5, 0.5], which)
        while True:
            b = next(gen)
            if b is None:
                break
            assert b.n_entries <= cap


# ---- the generator thread (the role of Keras' GeneratorEnqueuer under fit_generator) ---------------------------

def test_prefetcher_draws_exactly_count_items_in_order():
    from omnidirectional_collaborative_filtering_b200.data_reader import Prefetcher
    drawn = []

    def gen():
        k = 0
        while True:
            drawn.append(k)
            yield k
            k += 1

    for count, chunk in ((0, 8), (1, 8), (7, 8), (8, 8), (9, 8), (100, 8), (23, 1), (23, 5), (200, 64)):
        del drawn[:]
        assert list(Prefetcher(gen(), count, depth=3, chunk=chunk)) == list(range(count))
        # not one item more: np.random must end where synchronous consumption would leave it
        assert drawn == list(range(count))


def test_prefetcher_surfaces_generator_errors_and_exhaustion():
    from omnidirectional_collaborative_filtering_b200.data_reader import Prefetcher

    def broken():
        yield 1
        yield 2
        raise KeyError("row 7")

    got = []
    with pytest.raises(KeyError, match="row 7"):
        for item in Prefetcher(broken(), 5):
            got.append(item)
    assert got[:1] == [1]                       # what was handed over before the failure is delivered

    def short():
        yield 1

    with pytest.raises((StopIteration, RuntimeError)):
        list(Prefetcher(short(), 3))


def test_prefetched_batches_equal_inline_batches(golden_datasets):
    """The NumPy stream position and every batch are the same whether the generator runs on the prefetch thread
    (chunked hand-over) or inline."""
    from omnidirectional_collaborative_filtering_b200.data_reader import Prefetcher
    ds = golden_datasets["rev"]
    rd = product_reader(ds, "fixed_split")
    rd.rng_on_device = False
    runs = []
    for threaded in (False, True):
        np.random.seed(77)
        g = rd.data_gen(4, [0.2, 0.9], "train", True, "dropout", -1)
        n = rd.train_set_size // 4 - 1
        src = Prefetcher(g, n, chunk=3) if threaded else (next(g) for _ in range(n))
        runs.append(([(b.rows.copy(), b.flags.copy()) for b in src], np.random.random_sample()))
    (a, ta), (b, tb) = runs
    assert ta == tb and len(a) == len(b) > 3
    for (r0, f0), (r1, f1) in zip(a, b):
        assert np.array_equal(r0, r1) and np.array_equal(f0, f1)
    rd.close()
