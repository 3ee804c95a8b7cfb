"""Column sharding, host side (no GPU): shard stores, per-shard keep flags, weight slicing, and the
collective plumbing over gloo with world_size 2."""
import os

import numpy as np
import pytest

from omnidirectional_collaborative_filtering_b200 import dist as ocf_dist
from tests.helpers import golden_batch, host_densify, product_reader


def _shard_reader(ds, eval_mode, rank, world):
    from omnidirectional_collaborative_filtering_b200.data_reader import data_reader
    files = {"unique_items_list": ds["unique_cols"], "unique_users_list": ds["unique_rows"],
             "ratingsByUser_dict": ds["ablation"], "ratingsByUser_dicts_train": ds["train"],
             "ratingsByUser_dicts_valid": ds["valid"], "ratingsByUser_dicts_test": ds["test"]}
    n_rows = len(ds["unique_rows"]) if eval_mode == "ablation" else ds["n_rows"]
    return data_reader(ds["n_cols"], n_rows, "", nonsequentialusers=True, eval_mode=eval_mode, data=files,
                       shard=(rank, world))


@pytest.mark.parametrize("world", [2, 3])
def test_shard_batches_are_column_slices_of_the_reference(golden_cases, golden_datasets, golden_batches, world):
    for case in golden_cases[::3]:
        ds = golden_datasets[case["dataset"]]
        for rank in range(world):
            rd = _shard_reader(ds, case["eval_mode"], rank, world)
            rd.rng_on_device = False  # host stream where a GPU exists too: rng_after is read from np.random itself
            lo, hi = rd.col_range
            np.random.seed(case["seed"])
            if case["eval_mode"] == "ablation":
                rd.split_for_validation(case["val_split"], seed=case["split_seed"])
            gen = rd.data_gen(case["B"], case["sparsity"], train_val_test=case["which"], shuffle=case["shuffle"],
                              auxilliary_mask_type=case["aux"], aux_var_value=case["aux_value"],
                              return_target_count=case["rtc"], pass_through_input_training=case["pass_through"])
            for n in range(case["n_batches"]):
                batch = next(gen)
                feed, targets, tc = golden_batch(golden_batches, case, n)
                got_feed, got_t = host_densify(batch)
                for g, w in zip(got_feed, feed):
                    assert np.array_equal(g, w[:, lo:hi]), (case["id"], rank, n)
                assert np.array_equal(got_t, targets[:, lo:hi])
                if tc is not None:
                    assert batch.target_count == int(tc)      # counts are those of the full rows
            # every rank consumes the global stream exactly like the unsharded reader
            assert np.random.random_sample() == float(golden_batches[case["id"] + "/rng_after"])


def test_weight_slices_round_trip():
    rs = np.random.RandomState(0)
    N, H, k = 23, 5, 3
    full = [rs.normal(size=(k * N, H)), rs.normal(size=H), rs.normal(size=(H, H)), rs.normal(size=H),
            rs.normal(size=(H, N)), rs.normal(size=N)]
    full = [w.astype(np.float32) for w in full]
    for world in (1, 2, 4):
        parts = []
        for r in range(world):
            lo, hi = ocf_dist.col_range(N, r, world)
            part = ocf_dist.slice_weights(full, k, N, lo, hi)
            assert part[0].shape == (k * (hi - lo), H) and part[-2].shape == (H, hi - lo)
            parts.append(part)
        merged = ocf_dist.merge_weights(parts, k, N)
        for a, b in zip(merged, full):
            assert np.array_equal(a, b)


def _gloo_worker(rank, world, port, ds, out):
    """Each rank: slice of a dense encoder product + all-reduce == the full product; weight gather."""
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rs = np.random.RandomState(1)
        N, H, B = ds["n_cols"], 6, 8
        W = rs.normal(size=(N, H)).astype(np.float32)
        rd = _shard_reader(ds, "fixed_split", rank, world)
        lo, hi = rd.col_range
        np.random.seed(5)
        batch = next(rd.data_gen(B, [0.5, 0.5], "train", True, None, -1))
        (x, _), _ = host_densify(batch)
        z = torch.tensor(x.astype(np.float32) @ W[lo:hi])          # this shard's partial pre-activation
        dist.all_reduce(z)
        full_rd = product_reader(ds, "fixed_split")
        np.random.seed(5)
        (xf, _), _ = host_densify(next(full_rd.data_gen(B, [0.5, 0.5], "train", True, None, -1)))
        np.testing.assert_allclose(z.numpy(), xf.astype(np.float32) @ W, rtol=1e-5, atol=1e-5)
        full = [W, np.zeros(H, np.float32), rs.normal(size=(H, N)).astype(np.float32), np.zeros(N, np.float32)]
        parts = [None] * world
        dist.all_gather_object(parts, ocf_dist.slice_weights(full, 1, N, lo, hi))
        merged = ocf_dist.merge_weights(parts, 1, N)
        assert all(np.array_equal(a, b) for a, b in zip(merged, full))
        # catalogue-wide top-k from the shards' own lists (what follows model.recommend on a column shard)
        from oracle import ref_topk
        scores = np.round(np.random.RandomState(9).normal(size=(B, N)), 1).astype(np.float32)
        c, v = ref_topk.topk(scores[:, lo:hi], 5)
        got_c, got_v = ocf_dist.all_gather_topk(np.where(c >= 0, c + lo, -1).astype(np.int32), v, 5)
        want_c, want_v = ref_topk.topk(scores, 5)
        assert np.array_equal(got_c, want_c) and np.array_equal(got_v, want_v)
        out.put((rank, "ok"))
    except Exception as exc:                                   # pragma: no cover
        out.put((rank, repr(exc)))
    finally:
        dist.destroy_process_group()


def test_collectives_over_gloo_world2(golden_datasets):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29000 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, golden_datasets["rev"], out)) for r in range(2)]
    for p in procs:
        p.start()
    results = [out.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(results) == [(0, "ok"), (1, "ok")], results


def test_merge_topk_equals_topk_of_the_whole_catalogue():
    """Shard-local top-k lists merged on the host = the oracle's top-k over all columns (score descending, ties by the
    lower column, -1 / -inf padding last), including rows with fewer than k candidates."""
    from oracle import ref_topk
    from omnidirectional_collaborative_filtering_b200.dist import merge_topk
    rs = np.random.RandomState(3)
    B, N, k, world = 6, 50, 8, 4
    scores = np.round(rs.normal(size=(B, N)), 1).astype(np.float32)          # rounded: plenty of ties
    seen = rs.random_sample((B, N)) < 0.3
    seen[5, 3:] = True                                                       # a row with 3 candidates only
    bounds = [N * r // world for r in range(world + 1)]
    parts = []
    for r in range(world):
        lo, hi = bounds[r], bounds[r + 1]
        c, v = ref_topk.topk(scores[:, lo:hi], k, seen=[np.flatnonzero(row) for row in seen[:, lo:hi]])
        c = np.where(c >= 0, c + lo, -1).astype(np.int32)
        parts.append((c, v))
    got_c, got_v = merge_topk(parts, k)
    want_c, want_v = ref_topk.topk(scores, k, seen=[np.flatnonzero(row) for row in seen])
    assert np.array_equal(got_c, want_c) and np.array_equal(got_v, want_v)
    assert got_c[5, 3:].tolist() == [-1] * (k - 3)
