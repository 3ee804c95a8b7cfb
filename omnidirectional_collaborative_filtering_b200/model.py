"""Host-side mirror of the reference's `omni_model` (`model.py:33-170`) and of the Keras `Model`
methods `train.py` calls on it, over the CUDA library.

    omni_m = omni_model(numlayers, num_hidden_units, num_items, batch_size, dense_activation=..., ...)
    m = omni_m.model
    m.compile(optimizer=Adagrad(lr=0.005, epsilon=1e-08, decay=0.0), loss='mean_squared_error')
    history = m.fit_generator(train_gen, steps, validation_data=valid_gen, validation_steps=vsteps)

Arithmetic (SURVEY.md Appendix A.4-A.6) runs in `csrc/` kernels; nothing here computes.
Differences from Keras that a caller can see:
  * generators yield `data_reader.Batch` objects, not dense arrays
  * `num_hidden_units` may be a list of widths (superset; the reference uses one width)
  * `save` / `load_model` keep the reference's file names and write Keras-layout HDF5 when h5py is importable,
    `.npz` bytes otherwise (`checkpoint.py`); optimizer state is not saved, matching what `train.py:183-189`
    strips before testing
  * dropout masks come from Philox (oracle/philox.py defines the spec), not TensorFlow's RNG
"""
from __future__ import annotations

import ctypes as C
from typing import List

import numpy as np

from . import _lib
from .optimizers import Optimizer, get as get_optimizer

METRIC_NAMES = ["loss", "mean_absolute_error", "accurate_MAE", "nMAE", "accurate_RMSE", "accurate_MSE"]


class History(object):
    def __init__(self):
        self.history = {}
        self.epoch = []


class OmniNet(object):
    """The object `omni_model.model` exposes (stands in for the Keras `Model`)."""

    def __init__(self, owner):
        self.owner = owner
        self._handle = None
        self._capacity = (0, 0)
        self.optimizer: Optimizer = get_optimizer("adagrad")
        self.loss = "mean_squared_error"
        self.rating_range = 1.0
        self.metrics_names = list(METRIC_NAMES)
        self.stream = None
        self.comm = None                # dist.ShardComm when this model is a column shard
        self.native = None              # (dist.NativeComm or None, _lib.PAR_*): collectives inside the C library
        self._pinned = {}               # page-locked output buffers of predict / score, by shape
        self._step = 0
        self._compiled = False

    # -- C handle -----------------------------------------------------------------------------
    def _ensure(self, n_rows=None, n_entries=None, aux_type="keep", reader=None):
        o = self.owner
        if aux_type != "keep" and aux_type != o.aux_kind:
            o.set_aux_kind(aux_type)       # the reader decides what the aux block holds
        rows = max(int(n_rows or o.batch_size), self._capacity[0])
        entries = max(int(n_entries or 1), self._capacity[1])
        if reader is not None and (self._handle is None or entries > self._capacity[1]):
            entries = max(entries, reader.max_batch_entries(rows))     # size the workspaces once
        if self._handle is None:
            _lib.require_gpu()
            cfg = _lib.ModelConfig()
            cfg.n_cols = o.local_cols
            cfg.n_cols_total = o.input_shape
            cfg.n_layers = o.numlayers
            for i, w in enumerate(o.widths):
                cfg.widths[i] = w
            cfg.aux = _lib.AUX_TYPES[o.aux_kind]
            cfg.activation = _lib.ACTIVATIONS[o.dense_activation]
            cfg.loss = _lib.LOSSES[self.loss]
            cfg.l2 = -1.0 if o.l2 is None else float(o.l2)
            cfg.dropout_p = -1.0 if o.dropout_probability is None else float(o.dropout_probability)
            cfg.aux_var_value = -1.0
            cfg.rating_range = float(self.rating_range)
            cfg.max_rows = rows
            cfg.max_entries = entries
            cfg.sharded = int(o.sharded)
            out = C.c_void_p()
            _lib.check(_lib.lib().ocf_model_create(C.byref(cfg), C.byref(out)))
            self._handle = out
            self._capacity = (rows, entries)
            self._push_weights(o._host_weights)
            o._host_weights = None
            self._push_optimizer()
            for l, t in enumerate(o._compiled_trainable):
                _lib.check(_lib.lib().ocf_model_set_trainable(self._handle, l, int(t)))
            if self.native is not None:
                comm, mode = self.native
                _lib.check(_lib.lib().ocf_model_set_comm(self._handle, None if comm is None else comm.handle, int(mode)))
        elif rows > self._capacity[0] or entries > self._capacity[1]:
            _lib.check(_lib.lib().ocf_model_reserve(self._handle, rows, entries))
            self._capacity = (rows, entries)
        return self._handle

    def _push_weights(self, weights):
        for i, w in enumerate(weights):
            w = np.ascontiguousarray(w, dtype=np.float32)
            _lib.check(_lib.lib().ocf_model_set_weight(self._handle, i, _lib.ptr(w), w.size))

    def _push_optimizer(self):
        opt = self.optimizer
        _lib.check(_lib.lib().ocf_model_set_optimizer(self._handle, _lib.OPTIMIZERS[opt.kind], opt.lr, opt.p1,
                                                      opt.p2, opt.epsilon, opt.decay))
        _lib.check(_lib.lib().ocf_model_set_loss(self._handle, _lib.LOSSES[self.loss], float(self.rating_range)))

    # -- Keras surface --------------------------------------------------------------------------
    def compile(self, optimizer="adagrad", loss="mean_squared_error", metrics=None, rating_range=None):
        """`m.compile(...)`, train.py:131-133. The metric set is fixed to train.py's five
        (`metrics` is accepted and ignored); `rating_range` feeds nMAE (train.py:118-121)."""
        if loss not in _lib.LOSSES:
            raise ValueError("loss must be mean_squared_error or mean_absolute_error")
        self.optimizer = get_optimizer(optimizer)
        self.loss = loss
        if rating_range is not None:
            self.rating_range = float(rating_range)
        self._compiled = True
        for l in range(len(self.owner.trainable)):        # compile collects the trainable weights (both modes)
            self.owner._apply_trainable(l)
        if self._handle is not None:
            self._push_optimizer()

    def get_weights(self) -> List[np.ndarray]:
        o = self.owner
        if self._handle is None:
            return [w.copy() for w in o._host_weights]
        out = []
        shape = (C.c_int64 * 2)()
        for i in range(2 * (o.numlayers + 1)):
            _lib.check(_lib.lib().ocf_model_weight_shape(self._handle, i, shape))
            arr = np.empty((shape[0], shape[1]) if i % 2 == 0 else (shape[0],), dtype=np.float32)
            _lib.check(_lib.lib().ocf_model_get_weight(self._handle, i, _lib.ptr(arr), arr.size))
            out.append(arr)
        return out

    def set_weights(self, weights):
        o = self.owner
        shapes = o.weight_shapes()
        if len(weights) != len(shapes):
            raise ValueError("expected %d weight arrays, got %d" % (len(shapes), len(weights)))
        ws = []
        for w, s in zip(weights, shapes):
            w = np.asarray(w, dtype=np.float32)
            if tuple(w.shape) != tuple(s):
                raise ValueError("weight shape %s does not match %s" % (w.shape, s))
            ws.append(np.ascontiguousarray(w))
        if self._handle is None:
            o._host_weights = ws
        else:
            self._push_weights(ws)

    def _args(self, batch, phase=0, training=True):
        a = _lib.StepArgs()
        a.dropout_seed = self.owner.dropout_seed
        a.step = self._step & 0xFFFFFFFF
        a.row0 = int(getattr(batch, "row0", 0) or 0)
        a.rows_total = int(getattr(batch, "rows_total", 0) or 0)
        a.phase = phase
        return a

    def _metrics_from(self, rec):
        return [float(rec[0]), float(rec[1]), float(rec[2]), float(rec[3]), float(rec[4]), float(rec[5])]

    def _run_step(self, h, dev_handle, n_rows, args, rec, train):
        """One step through the C ABI; a column shard runs it as three phases with the two
        activation all-reduces between them (dist.py)."""
        fn = _lib.lib().ocf_train_step if train else _lib.lib().ocf_eval_step
        if self.comm is None or self.native is not None:
            args.phase = 0
            _lib.check(fn(h, dev_handle, C.byref(args), _lib.ptr(rec), self.stream))
            return
        args.phase = 1
        _lib.check(fn(h, dev_handle, C.byref(args), None, self.stream))
        self.comm.reduce_z(n_rows)
        args.phase = 2
        _lib.check(fn(h, dev_handle, C.byref(args), None, self.stream))
        self.comm.reduce_stats_dh(n_rows, with_dh=train)
        args.phase = 3
        _lib.check(fn(h, dev_handle, C.byref(args), _lib.ptr(rec), self.stream))

    def step_on_device_batch(self, dev, n_rows, step, train=True, row0=0, rows_total=0):
        """A step on an already-filled DeviceBatch, no host sync (bench.py's device-timed loop)."""
        args = _lib.StepArgs()
        args.dropout_seed = self.owner.dropout_seed
        args.step = int(step) & 0xFFFFFFFF
        args.row0, args.rows_total = int(row0), int(rows_total)
        self._run_step(self._handle, dev.handle, n_rows, args, None, train)

    def train_on_batch(self, batch, sync=True):
        """One optimisation step. Returns the six metric values when `sync`, else None (the
        values stay in the device log; see `read_metrics` / `wait_metrics`)."""
        h = self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
        dev = batch.upload(self.stream)
        args = self._args(batch)
        rec = np.empty(_lib.N_METRICS, dtype=np.float32) if sync else None
        self._run_step(h, dev.handle, batch.n_rows, args, rec, True)
        self._step += 1
        return self._metrics_from(rec) if sync else None

    def test_on_batch(self, batch, sync=True):
        h = self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
        dev = batch.upload(self.stream)
        args = self._args(batch, training=False)
        rec = np.empty(_lib.N_METRICS, dtype=np.float32) if sync else None
        self._run_step(h, dev.handle, batch.n_rows, args, rec, False)
        return self._metrics_from(rec) if sync else None

    def steps_logged(self):
        return int(_lib.lib().ocf_model_steps_logged(self._handle)) if self._handle is not None else 0

    def wait_metrics(self, step):
        """The six metric values of logged step `step` (one of the last 64); waits for that step
        only, later steps keep running."""
        rec = np.empty(_lib.N_METRICS, dtype=np.float32)
        _lib.check(_lib.lib().ocf_model_wait_metrics(self._handle, int(step), _lib.ptr(rec)))
        return self._metrics_from(rec)

    def read_metrics(self, first, count):
        """[count, 8] records of steps first..first+count-1 from the device log."""
        out = np.empty((count, _lib.N_METRICS), dtype=np.float32)
        if count:
            _lib.check(_lib.lib().ocf_model_read_metrics(self._handle, first, count, _lib.ptr(out), self.stream))
        return out

    def _run(self, generator, steps, train, workers=1):
        """`steps` batches through train/eval steps. Steps are enqueued without a host sync and
        the metric records, copied to pinned memory behind every step, are read back in chunks.
        workers=1 (Keras' default) draws the batches on a prefetch thread, workers=0 inline."""
        from .data_reader import Prefetcher
        steps = max(int(steps), 0)              # train.py passes floor(n/B) - 1: -1 for sets smaller than a batch; Keras runs none
        rows = []
        first = None
        pending = 0
        source = Prefetcher(generator, steps) if workers else (next(generator) for _ in range(steps))
        for batch in source:
            if batch is None:
                raise RuntimeError("generator ran out of batches (it yields None after floor(n/B) batches)")
            if first is None:
                self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
                first = _lib.lib().ocf_model_steps_logged(self._handle)
            (self.train_on_batch if train else self.test_on_batch)(batch, sync=False)
            pending += 1
            if pending == 2048:
                rows.append(self.read_metrics(first, pending))
                first += pending
                pending = 0
        if pending:
            rows.append(self.read_metrics(first, pending))
        return np.concatenate(rows, axis=0) if rows else np.zeros((0, _lib.N_METRICS), dtype=np.float32)

    def fit_generator(self, generator, steps_per_epoch, epochs=1, verbose=1, callbacks=None,
                      validation_data=None, validation_steps=None, workers=1, **_ignored):
        """`m.fit_generator(train_gen, steps, validation_data=valid_gen, validation_steps=...)`,
        train.py:157-158. Per-epoch value = mean of the per-batch values; training values are
        pre-update with dropout on, validation has dropout off (Keras semantics)."""
        hist = History()
        for epoch in range(int(epochs)):
            recs = self._run(generator, steps_per_epoch, train=True, workers=workers)
            mean = recs[:, :6].astype(np.float64).mean(axis=0) if len(recs) else np.full(6, np.nan)
            for name, v in zip(METRIC_NAMES, mean):
                hist.history.setdefault(name, []).append(float(v))
            if validation_data is not None:
                vals = self.evaluate_generator(validation_data, validation_steps, workers=workers)
                for name, v in zip(METRIC_NAMES, vals):
                    hist.history.setdefault("val_" + name, []).append(float(v))
            hist.epoch.append(epoch)
            if verbose:
                print(" - ".join("%s: %.4f" % (k, v[-1]) for k, v in hist.history.items()))
        return hist

    def evaluate_generator(self, generator, steps, workers=1, **_ignored):
        """train.py:208,218. Returns [loss, mae, accurate_MAE, nMAE, accurate_RMSE, accurate_MSE]."""
        recs = self._run(generator, steps, train=False, workers=workers)
        return [float(v) for v in recs[:, :6].astype(np.float64).mean(axis=0)]

    def _out_buffer(self, rows, reuse):
        """[rows, local_cols] float32 destination of predict / score. `reuse`: a page-locked buffer
        owned by the model (the device->host copy then runs at PCIe speed; the returned array is
        overwritten by the next call of the same shape), else a fresh pageable array."""
        shape = (int(rows), int(self.owner.local_cols))
        if not reuse:
            return np.empty(shape, dtype=np.float32)
        held = self._pinned.get(shape)
        if held is None:
            if len(self._pinned) >= 2:
                self._pinned.clear()
            held = self._pinned[shape] = _lib.PinnedArray(shape)
        return held.array

    def predict(self, batch, batch_size=None, verbose=0, reuse_output=False):
        """`best_m.predict(input_list)`, train.py:239: output_mask * full_predictions, [B, N] float32."""
        h = self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
        dev = batch.upload(self.stream)
        self._shard_encode(h, dev, batch)
        out = self._out_buffer(batch.n_rows, reuse_output)
        _lib.check(_lib.lib().ocf_predict(h, dev.handle, _lib.ptr(out), self.stream))
        return out

    def score(self, batch, reuse_output=False):
        """Full-catalogue scores `full_predictions` (model.py:82-84), [B, N] float32."""
        h = self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
        dev = batch.upload(self.stream)
        self._shard_encode(h, dev, batch)
        out = self._out_buffer(batch.n_rows, reuse_output)
        _lib.check(_lib.lib().ocf_score(h, dev.handle, _lib.ptr(out), 0, self.stream))
        return out

    def recommend(self, batch, k=10, exclude_seen=True):
        """The k best catalogue columns of every batch row by full-catalogue score, best first
        (ties: lower column first), selected on the device: (columns int32 [B, k], scores float32
        [B, k]). `exclude_seen` drops the columns a row holds as inputs. Slots beyond the available
        columns hold column -1 / score -inf. A column shard returns the top k of its own columns
        (global column ids); `dist.all_gather_topk` merges the shards' lists into the catalogue-wide top k."""
        h = self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
        dev = batch.upload(self.stream)
        self._shard_encode(h, dev, batch)
        cols = np.empty((batch.n_rows, int(k)), dtype=np.int32)
        scores = np.empty((batch.n_rows, int(k)), dtype=np.float32)
        _lib.check(_lib.lib().ocf_score_topk(h, dev.handle, int(k), int(bool(exclude_seen)), _lib.ptr(cols),
                                             _lib.ptr(scores), self.stream))
        if self.owner.col_lo:
            cols[cols >= 0] += self.owner.col_lo
        return cols, scores

    def rank_targets(self, batch, exclude_seen=True, min_value=None):
        """Exact rank of every relevant target of every batch row among the row's candidate columns, on
        the device (`ocf_rank_targets`): 1-based, in the order `recommend` uses (score descending, ties by
        lower column), so rank(t) <= k exactly when t is in `recommend(batch, k)` at position rank(t) - 1.
        Relevant targets: the row's target columns (a repeated column once), with a stored value
        >= `min_value` when given, minus the columns `exclude_seen` removes from the candidates (the row's
        inputs). With pass-through split batches every target is also an input, so with `exclude_seen`
        no row has a relevant target.
        Returns (row_ptr int64 [rows + 1], cols int32, ranks int32, n_cand int64 [rows]): row r's relevant
        targets are cols[row_ptr[r]:row_ptr[r + 1]] in entry order; n_cand[r] counts its candidates."""
        if self.owner.sharded or self.comm is not None or (self.native is not None and self.native[1] == _lib.PAR_COLUMNS):
            raise ValueError("rank_targets needs the whole catalogue; a column shard holds only part of it")
        h = self._ensure(batch.n_rows, batch.n_entries, batch.aux_type, batch.reader)
        dev = batch.upload(self.stream)
        info = (C.c_int64 * 5)()
        _lib.check(_lib.lib().ocf_batch_info(dev.handle, info))
        rows, entries = int(info[0]), int(info[1])
        col = np.empty(entries, dtype=np.int32)
        rank = np.empty(entries, dtype=np.int32)
        ent_ptr = np.empty(rows + 1, dtype=np.int32)
        n_cand = np.empty(rows, dtype=np.int64)
        mv = -np.inf if min_value is None else float(min_value)
        _lib.check(_lib.lib().ocf_rank_targets(h, dev.handle, int(bool(exclude_seen)), mv, _lib.ptr(col),
                                               _lib.ptr(rank), _lib.ptr(ent_ptr), _lib.ptr(n_cand), self.stream))
        keep = rank > 0
        before = np.concatenate(([0], np.cumsum(keep, dtype=np.int64)))
        row_ptr = before[ent_ptr.astype(np.int64)]
        return row_ptr, col[keep], rank[keep], n_cand

    def evaluate_ranking(self, generator, steps, ks=(10,), exclude_seen=True, min_value=None, workers=1):
        """Ranking quality of `recommend` over `steps` batches of `generator` (drawn as `evaluate_generator`
        draws them, through the Prefetcher when `workers`): for every relevant target its exact rank
        (`rank_targets`), then HR@k, precision@k, recall@k, NDCG@k for every k in `ks`, MRR and AUC, each the
        float64 mean over the rows that have a relevant target (AUC: and at least one other candidate).
        See `ranking` for the definitions. Returns a dict with those means and "rows" / "AUC_rows", the
        number of rows behind them. Draws nothing from np.random beyond what the generator draws; leaves
        the weights, the optimizer state and the metric log as they were."""
        from . import ranking
        from .data_reader import Prefetcher
        if self.owner.sharded or self.comm is not None or (self.native is not None and self.native[1] == _lib.PAR_COLUMNS):
            raise ValueError("evaluate_ranking needs the whole catalogue; a column shard holds only part of it")
        ks = [int(k) for k in ks]
        steps = max(int(steps), 0)
        sums = ranking.empty_sums(ks)
        source = Prefetcher(generator, steps) if workers else (next(generator) for _ in range(steps))
        for batch in source:
            if batch is None:
                raise RuntimeError("generator ran out of batches (it yields None after floor(n/B) batches)")
            row_ptr, _, ranks, n_cand = self.rank_targets(batch, exclude_seen=exclude_seen, min_value=min_value)
            ranking.accumulate(sums, ranking.metrics_from_ranks(row_ptr, ranks, n_cand, ks))
        return ranking.finalize(sums)

    def _shard_encode(self, h, dev, batch):
        """Column shards: encoder partial sums + their all-reduce before predict/score (this
        rank's output then holds its own columns)."""
        if self.comm is None or self.native is not None:
            return
        args = self._args(batch, phase=1, training=False)
        _lib.check(_lib.lib().ocf_eval_step(h, dev.handle, C.byref(args), None, self.stream))
        self.comm.reduce_z(batch.n_rows)

    def save(self, path):
        """`m.save(...)`, train.py:169: weights + architecture under exactly `path` (the reference's names carry no
        extension), as Keras-layout HDF5 when h5py is importable, else as .npz bytes; no optimizer state, which
        train.py:183-189 strips anyway. See `checkpoint.py`."""
        from . import checkpoint
        checkpoint.save(path, self.get_weights(), self.owner.config())

    def save_weights(self, path):
        from . import checkpoint
        checkpoint.save(path, self.get_weights(), None)

    def load_weights(self, path):
        from . import checkpoint
        self.set_weights(checkpoint.load(path)[1])

    def close(self):
        if self._handle is not None:
            _lib.lib().ocf_model_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class omni_model(object):
    """Drop-in for `model.omni_model` (`model.py:33-99`)."""

    def __init__(self, numlayers, num_hidden_units, input_shape, batch_size, dense_activation="tanh",
                 use_causal_info=True, use_timestamps=False, use_both_masks=False,
                 l2_weight_regulatization=None, sparse_representation=False, dropout_probability=None,
                 use_sparse_masking_layer=False, auxilliary_mask_type="default", local_cols=None, col_lo=0):
        if use_timestamps:
            raise NotImplementedError("use_timestamps: the reference's timestamp path is broken and out of scope")
        if sparse_representation:
            raise NotImplementedError("sparse_representation: inputs are never dense here; leave it False")
        if use_sparse_masking_layer:
            raise NotImplementedError("Dynamic_Masking_Layer cannot be constructed in the reference "
                                      "(model.py:186); the decoder kernel already evaluates observed entries only")
        if dense_activation not in _lib.ACTIVATIONS:
            raise ValueError("unsupported dense_activation %r" % (dense_activation,))
        self.numlayers = int(numlayers)
        if isinstance(num_hidden_units, (list, tuple)):
            self.widths = [int(w) for w in num_hidden_units]
            if len(self.widths) != self.numlayers:
                raise ValueError("need one width per hidden layer")
        else:
            self.widths = [int(num_hidden_units)] * self.numlayers
        if not 1 <= self.numlayers <= 8:
            raise ValueError("numlayers must be 1..8")
        self.num_hidden_units = self.widths[0]
        self.input_shape = int(input_shape)
        self.batch_size = int(batch_size)
        self.dense_activation = dense_activation
        self.use_causal_info = bool(use_causal_info)
        self.use_both_masks = bool(use_both_masks)
        self.l2 = l2_weight_regulatization
        self.dropout_probability = dropout_probability
        self.k_blocks = 1 + int(self.use_causal_info) + int(self.use_both_masks)
        # Which mask the aux block holds is the reader's choice (auxilliary_mask_type); the
        # model only fixes how many blocks are concatenated (model.py:47-56).
        if auxilliary_mask_type == "default":
            auxilliary_mask_type = ("both" if self.use_both_masks else "dropout") if self.use_causal_info else None
        self.set_aux_kind(auxilliary_mask_type)
        self.local_cols = self.input_shape if local_cols is None else int(local_cols)
        self.sharded = self.local_cols != self.input_shape
        self.trainable = [True] * (self.numlayers + 1)         # layer.trainable, as the caller set it
        # What the optimizer honours. "at_once" (default): a flag set after compile() takes effect immediately - what
        # the reference's transfer flows intend (model.py:109-170 called after m.compile, train.py:131-145).
        # "on_compile": the Keras 2.0.4 the reference pins collects the trainable weights at compile time, so a flag
        # set afterwards is ignored until the next compile() (the reference's own comment, model.py:137).
        self.trainable_applies = "at_once"
        self._compiled_trainable = list(self.trainable)
        # Keras draws one seed per kernel initializer and per Dropout layer from the global NumPy
        # RNG while the graph is built (SURVEY.md Appendix A.6); keep that stream position.
        self.col_lo = int(col_lo)
        dims = [self.k_blocks * self.input_shape] + self.widths + [self.input_shape]
        full = []
        seeds = []
        from .data_reader import sync_host_rng
        sync_host_rng()                     # np.random may be on loan to the GPU (data_reader.DeviceRng)
        for l in range(self.numlayers + 1):
            seed = int(np.random.randint(10e6))
            lim = np.sqrt(6.0 / (dims[l] + dims[l + 1]))                # glorot_uniform
            rs = np.random.RandomState(seed)
            full.append(rs.uniform(-lim, lim, size=(dims[l], dims[l + 1])).astype(np.float32))
            full.append(np.zeros(dims[l + 1], dtype=np.float32))
            if l < self.numlayers and dropout_probability is not None:
                seeds.append(int(np.random.randint(10e6)))
        if self.sharded:        # a column shard keeps its slice of the full initialisation
            from .dist import slice_weights
            full = slice_weights(full, self.k_blocks, self.input_shape, self.col_lo, self.col_lo + self.local_cols)
        self._host_weights = full
        self.dropout_seed = (seeds[0] if seeds else 0) | (0x0CF << 32)
        self.model = OmniNet(self)

    def set_aux_kind(self, aux_type):
        k = {None: 1, "causal": 2, "dropout": 2, "zeros": 2, "both": 3}[aux_type]
        if k != self.k_blocks:
            raise ValueError("auxilliary_mask_type %r feeds %d input blocks but the model was built for %d "
                             "(use_causal_info / use_both_masks, model.py:47-56)" % (aux_type, k, self.k_blocks))
        self.aux_kind = aux_type
        net = getattr(self, "model", None)
        if net is not None and net._handle is not None:
            _lib.check(_lib.lib().ocf_model_set_aux(net._handle, _lib.AUX_TYPES[aux_type]))

    def config(self):
        return dict(numlayers=self.numlayers, num_hidden_units=self.widths, input_shape=self.input_shape,
                    batch_size=self.batch_size, dense_activation=self.dense_activation,
                    use_causal_info=self.use_causal_info, use_both_masks=self.use_both_masks,
                    l2_weight_regulatization=self.l2, dropout_probability=self.dropout_probability,
                    auxilliary_mask_type=self.aux_kind)

    def weight_shapes(self):
        dims = [self.k_blocks * self.local_cols] + self.widths + [self.local_cols]
        out = []
        for l in range(self.numlayers + 1):
            out += [(dims[l], dims[l + 1]), (dims[l + 1],)]
        return out

    # -- model.py:102-107 ---------------------------------------------------------------------
    def save_weights(self, filename):
        self.model.save_weights(filename)

    def load_weights(self, weights):
        self.model.set_weights(weights)

    # -- weight transfer, model.py:109-170 -------------------------------------------------------
    # Every Dense layer of this architecture touches a width-H tensor, so the reference's
    # "dense layers with input or output width == num_hidden_units" filter selects all L+1.
    def _dense_pairs(self):
        w = self.model.get_weights()
        return [[w[2 * l], w[2 * l + 1]] for l in range(self.numlayers + 1)]

    def _set_dense(self, l, pair):
        """Kernel + bias of dense layer l (only these two arrays move; no round trip of the other layers)."""
        shapes = self.weight_shapes()
        arrs = []
        for k in (0, 1):
            a = np.ascontiguousarray(pair[k], dtype=np.float32)
            if tuple(a.shape) != tuple(shapes[2 * l + k]):
                raise ValueError("weight shape %s does not match %s" % (a.shape, shapes[2 * l + k]))
            arrs.append(a)
        net = self.model
        if getattr(net, "_handle", None) is None:
            if self._host_weights is not None and type(net).__name__ == "OmniNet":
                self._host_weights[2 * l], self._host_weights[2 * l + 1] = arrs[0].copy(), arrs[1].copy()
            else:                                   # a stand-in model (tests): go through its own setter
                w = net.get_weights()
                w[2 * l], w[2 * l + 1] = arrs[0], arrs[1]
                net.set_weights(w)
            return
        for k in (0, 1):
            _lib.check(_lib.lib().ocf_model_set_weight(net._handle, 2 * l + k, _lib.ptr(arrs[k]), arrs[k].size))

    def _set_trainable(self, l, flag):
        self.trainable[l] = bool(flag)
        if self.trainable_applies != "on_compile":
            self._apply_trainable(l)

    def _apply_trainable(self, l):
        self._compiled_trainable[l] = self.trainable[l]
        if getattr(self.model, "_handle", None) is not None:
            _lib.check(_lib.lib().ocf_model_set_trainable(self.model._handle, l, int(self.trainable[l])))

    def replace_dense_layer_weights(self, donor_model, layers_to_replace, make_layers_trainable=False):
        donor = _donor_pairs(donor_model)
        if layers_to_replace == "all":
            layers_to_replace = [True] * len(donor)
        for l in range(self.numlayers + 1):
            if layers_to_replace[l]:
                self._set_dense(l, donor[l])
                self._set_trainable(l, make_layers_trainable)
                print("Loaded weights for dense layer ", l)

    def manually_load_all_weights(self, donor_model):
        self.model.set_weights(_donor_weights(donor_model))

    def make_trainable(self):
        for l in range(self.numlayers):
            self._set_trainable(l, True)
        if self.input_shape == self.num_hidden_units:
            self._set_trainable(self.numlayers, True)

    def load_and_fix_for_denoising_autoencoders(self, donor_model):
        donor = _donor_pairs(donor_model)
        print("Number of weight layers to donate", len(donor))
        n_side = int(len(donor) / 2)
        n_new = self.numlayers + 1
        for l in range(n_new):
            if l < n_side:
                self._set_dense(l, donor[l])
                self._set_trainable(l, False)
                print("Loaded and fixed weights for dense layer ", l, " from donor dense layer ", l)
            elif l >= n_new - n_side:
                src = len(donor) - (n_new - l)
                self._set_dense(l, donor[src])
                self._set_trainable(l, False)
                print("Loaded and fixed weights for dense layer ", l, " from donor dense layer ", src)


def _donor_weights(donor):
    if isinstance(donor, omni_model):
        donor = donor.model
    if isinstance(donor, OmniNet):
        return donor.get_weights()
    return [np.asarray(w) for w in donor]          # a plain weight list


def _donor_pairs(donor):
    w = _donor_weights(donor)
    return [[w[2 * l], w[2 * l + 1]] for l in range(len(w) // 2)]


def load_model(path):
    """`keras.models.load_model(...)` (train.py:139,191): a model file written by `OmniNet.save` or, with h5py
    installed, by Keras itself (the reference's donors); format told by the file's first bytes (`checkpoint.py`)."""
    from . import checkpoint
    cfg, weights = checkpoint.load(path)
    if cfg is None:
        raise ValueError("%s holds weights only (save_weights); build the model and call load_weights" % path)
    from .data_reader import sync_host_rng
    sync_host_rng()
    state = np.random.get_state()                   # loading must not disturb the caller's stream
    om = omni_model(cfg["numlayers"], cfg["num_hidden_units"], cfg["input_shape"], cfg["batch_size"],
                    dense_activation=cfg["dense_activation"], use_causal_info=cfg["use_causal_info"],
                    use_both_masks=cfg["use_both_masks"], l2_weight_regulatization=cfg["l2_weight_regulatization"],
                    dropout_probability=cfg["dropout_probability"], auxilliary_mask_type=cfg["auxilliary_mask_type"])
    np.random.set_state(state)
    om.model.set_weights(weights)
    return om.model
