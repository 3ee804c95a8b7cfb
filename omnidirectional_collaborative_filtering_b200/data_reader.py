"""Host-side mirror of the reference's `data_reader` (same constructor, attributes, generator
protocol and NumPy global-RNG consumption), minus the per-rating Python loop.

What stays on the host (cheap, O(B) per batch + one vectorised RNG draw):
  * set selection, lazy permutation, floor(n/B) batches, the infinite None tail
    (`data_reader.py:314-419`)
  * the RNG replay: `uniform(lo, hi, B)` then one `random_sample(sum n)` compared against the
    per-row cdf - bit-identical to the B calls of `np.random.choice([0,1], n, p=[1-s, s])` at
    `data_reader.py:120,130` (SURVEY.md section 0, fact 9)
What moves to the GPU (`ocf_batch_fill_*`, kernel K1): everything that touches a rating.

A generator yields `Batch` objects. `omni_model.model.fit_generator/evaluate_generator/predict`
consume them directly (no dense arrays anywhere); unpacking one like the reference's tuples,
`input_list, targets = batch`, materialises the reference's dense float64 arrays through the
CUDA scatter kernel, so reference-style callers keep working.
"""
from __future__ import annotations

import ctypes as C
import os
import json
import pickle
import threading
from collections import OrderedDict

import numpy as np

from . import _lib
from .store import BatchRing, RatingStore, StorePair
from .synthetic import Csr, FixedSplit


def _csr_from_lists(lists, col_of, n_cols) -> Csr:
    """Per-row [(item, rating), ...] lists (None = no list) -> CSR, stored order kept."""
    lens = np.fromiter((0 if l is None else len(l) for l in lists), dtype=np.int64, count=len(lists))
    rowptr = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum(lens, out=rowptr[1:])
    col = np.empty(int(rowptr[-1]), dtype=np.int32)
    val64 = np.empty(int(rowptr[-1]), dtype=np.float64)
    k = 0
    for l in lists:
        if not l:
            continue
        for pair in l:
            col[k] = col_of[pair[0]]           # data_reader.py:135 (KeyError like the reference)
            val64[k] = pair[1]
            k += 1
    # The store is float32 (the model's dtype; the reference's float64 batch arrays are cast to float32 at the
    # feed). Dyadic ratings (k/2, integers) are exact; others round to the nearest float32 (~6e-8 relative) and the
    # dense view `Batch.to_dense` returns those rounded values. A finite rating beyond float32's range becomes inf,
    # as in the native parser (csrc/ocf_etl.cpp) and in the reference's own float32 feed - said out loud here.
    with np.errstate(over="ignore"):
        val = val64.astype(np.float32)
    overflow = np.isfinite(val64) & ~np.isfinite(val)
    if overflow.any():
        import warnings
        warnings.warn("%d rating(s) exceed float32's range and are stored as inf (first: %r)"
                      % (int(overflow.sum()), float(val64[np.flatnonzero(overflow)[0]])), RuntimeWarning, stacklevel=2)
    return Csr(len(lists), n_cols, rowptr, col, val)


class DeviceRng(object):
    """`np.random`'s global MT19937 stream, lent to the GPU while split batches are drawn.

    The reference draws `uniform(lo, hi, B)` + one `choice` per row from the global NumPy stream
    for every training batch (`data_reader.py:120,130`). Replaying those ~10^5 doubles per batch on
    the host bounds the whole step, so the stream itself moves: the generator hands out *tickets*
    (how many doubles a batch consumes, in drawing order), the first upload pushes the host state
    to the device (`ocf_rng_set_state`), every upload advances the device stream by exactly its
    ticket (`ocf_batch_fill_split_rng`; tickets that were drawn but never uploaded are skipped in
    order), and `release()` brings the state back into `np.random` before anything on the host
    draws again. The result is bit-identical to host-side consumption at the generator's `next()`.
    One instance per process, like the stream it stands in for."""

    _instance = None

    def __init__(self):
        self.lock = threading.RLock()
        self.handle = None
        self.active = False                 # the device holds the current state
        self.host_state = None              # np.random state at the first ticket since the last release
        self.issued = 0
        self.pending = OrderedDict()        # ticket -> draws, in drawing order
        self.layout = None                  # (workers, regenerations per block) this object asked for last

    @classmethod
    def get(cls):
        if cls._instance is None:
            cls._instance = DeviceRng()
        return cls._instance

    def ticket(self, draws):
        with self.lock:
            if self.host_state is None:
                self.host_state = np.random.get_state()
            t = self.issued
            self.issued += 1
            self.pending[t] = int(draws)
            return t

    def _activate(self):
        if self.active:
            return
        lib = _lib.lib()
        if self.handle is None:
            _lib.require_gpu()
            out = C.c_void_p()
            _lib.check(lib.ocf_rng_create(C.byref(out)))
            self.handle = out
        key = np.ascontiguousarray(self.host_state[1], dtype=np.uint32)
        _lib.check(lib.ocf_rng_set_state(self.handle, _lib.ptr(key), int(self.host_state[2])))
        self.active = True

    def configure(self, workers=0, block_regens=0, ring_words_min=0, pin=True):
        """Generator layout of the device stream (`ocf_rng_configure`): worker CTAs, regenerations per block, minimum
        ring size in words; 0 keeps a value. The stream's state and position are kept. A layout set here stays
        (`pin`); without a pinned layout the object sizes the blocks to the batches it sees (`_tune`)."""
        with self.lock:
            lib = _lib.lib()
            if self.handle is None:
                _lib.require_gpu()
                out = C.c_void_p()
                _lib.check(lib.ocf_rng_create(C.byref(out)))
                self.handle = out
            _lib.check(lib.ocf_rng_configure(self.handle, int(workers), int(block_regens), int(ring_words_min)))
            self.pinned = bool(pin)
            self.layout = None              # re-read on the next _tune

    def _tune(self, draws):
        """Generator layout for batches of `draws` doubles. One chain (CTA) makes ~0.8 G draws/s, and every block
        costs the host four launches (block, event, the jump's two kernels). A rank of a multi-GPU run replays the
        whole global batch's draws, so it gets 8 workers (16 for multi-million-draw batches), and blocks grow with
        the batch so that a batch stays a handful of blocks (8 ranks x 10 blocks of 256 regenerations per step was
        0.29 ms of API calls per 0.24 ms step, profiles/r02). Only ever grows; $OCF_RNG_WORKERS pins the workers."""
        if getattr(self, "pinned", False):
            return
        import os
        if self.layout is None:
            inf = self.info()
            self.layout = (int(inf["workers"]), int(inf["block_regens"]))
        fixed = os.environ.get("OCF_RNG_WORKERS")
        world = int(os.environ.get("WORLD_SIZE", "1"))
        workers = int(fixed) if fixed else (2 if world == 1 else (8 if draws <= 3000000 else 16))
        regens = 256
        while regens < 4096 and regens * 624 * workers < 2 * draws:
            regens *= 2
        want = (max(workers, self.layout[0]), max(regens, self.layout[1]))
        if want != self.layout:
            _lib.check(_lib.lib().ocf_rng_configure(self.handle, want[0], want[1], 0))
            self.layout = want

    def info(self):
        buf = (C.c_int64 * 6)()
        _lib.check(_lib.lib().ocf_rng_info(self.handle, buf))
        return dict(zip(("workers", "block_regens", "ring_blocks", "ring_words", "position_words", "blocks_enqueued"), list(buf)))

    def consume(self, ticket):
        """Called by the upload of a batch: positions the device stream at the batch's first draw
        and returns the rng handle; the fill then advances it by the batch's draws."""
        with self.lock:
            if ticket not in self.pending:
                raise RuntimeError("this batch's random draws were dropped: np.random was used on the host (a new "
                                   "generator, a model initialisation) before the batch was uploaded")
            self._activate()
            lib = _lib.lib()
            for t in list(self.pending):
                if t >= ticket:
                    break
                _lib.check(lib.ocf_rng_skip(self.handle, self.pending.pop(t)))   # drawn, never uploaded
            mine = self.pending.pop(ticket)
            self._tune(mine)
            # the tickets already drawn tell how far the workers MAY run ahead of this batch; two more batches is all
            # they need to (one chain makes a batch's draws in a fifth of a step), and whatever is in flight when the
            # stream goes back to the host (every epoch start: np.random.permutation) has to drain first
            ahead = int(os.environ.get("OCF_RNG_AHEAD", "3"))
            _lib.check(lib.ocf_rng_prefetch(self.handle, min(mine + sum(self.pending.values()), ahead * mine)))
            return self.handle

    def release(self):
        """Hand the stream back to `np.random` (no-op when the host already owns it)."""
        with self.lock:
            if self.host_state is None:
                return
            cur, lent = np.random.get_state(), self.host_state
            if not (cur[2] == lent[2] and cur[3] == lent[3] and cur[4] == lent[4] and np.array_equal(cur[1], lent[1])):
                # np.random was reseeded (or drawn from) on the host while the stream was on loan:
                # the host's stream is the current one, the device's copy and its open tickets lapse.
                # Draws the device already made are then NOT reflected in np.random: say so unless the host
                # clearly reseeded (a fresh seed puts the position at 624 with a new key).
                if self.active and cur[2] != 624:
                    import warnings
                    warnings.warn("np.random was drawn from on the host while its stream was lent to the GPU "
                                  "(data_reader.DeviceRng): the draws the GPU made for uploaded batches are dropped from "
                                  "the host stream. Call data_reader.sync_rng() before drawing from np.random between "
                                  "batches, or construct the reader with rng_on_device=False.", RuntimeWarning, stacklevel=3)
                self.pending.clear()
                self.active = False
                self.host_state = None
                return
            self._activate()
            lib = _lib.lib()
            for t in list(self.pending):
                _lib.check(lib.ocf_rng_skip(self.handle, self.pending.pop(t)))
            key = np.empty(624, dtype=np.uint32)
            pos = C.c_int32()
            _lib.check(lib.ocf_rng_get_state(self.handle, _lib.ptr(key), C.byref(pos)))
            st = self.host_state
            np.random.set_state((st[0], key, int(pos.value), st[3], st[4]))
            self.active = False
            self.host_state = None


def sync_host_rng():
    """Make `np.random` current again if the device holds its stream. Everything in this package
    that draws from `np.random` calls this first; call it yourself before drawing from
    `np.random` in between batches of a running generator."""
    if DeviceRng._instance is not None:
        DeviceRng._instance.release()


def device_rng_available() -> bool:
    try:
        return _lib.lib().ocf_device_count() > 0
    except _lib.OcfError:
        return False


class Batch(object):
    """One batch as (row ids, keep flags) + the stores they index. Host-only until uploaded."""

    def __init__(self, reader, kind, source, rows, flags, pass_through, aux_type, aux_value,
                 target_count, return_target_count, n_ratings=None):
        self.reader = reader
        self.kind = kind                       # "split" | "fixed"
        self.source = source                   # RatingStore | StorePair
        self.rows = np.ascontiguousarray(rows, dtype=np.int32)
        self._flags = flags                    # uint8 keep flags, or None while only (u, cdf0) are held
        self.u = self.cdf0 = self.full_len = None
        self.ticket = None                     # device-RNG mode: the batch's place in the NumPy stream
        self.sparsity = None                   #   (lo, hi) of its np.random.uniform draw
        self.rng_slice = None                  #   row-parallel slice of a global batch (see row_slice)
        self.row0 = 0                          # index of the first row inside the global batch
        self.rows_total = 0                    # rows of the global batch (0: this batch is the whole of it)
        self._dev_generation = -1
        self.pass_through = bool(pass_through)
        self.aux_type = aux_type
        self.aux_value = float(aux_value)
        self.target_count = int(target_count)
        self.return_target_count = bool(return_target_count)
        self.n_rows = int(self.rows.size)
        self.n_cols = int(source.n_cols)
        self.n_entries = int(source.lengths[self.rows].sum())      # ratings this (shard of the) batch holds
        self.n_ratings = int(n_ratings) if n_ratings is not None else self.n_entries   # of the full rows
        self._device = None

    @property
    def flags(self):
        """uint8 keep flag per rating this batch holds (1 = input). Derived on demand from the
        uniform draws; `upload` hands the draws to the library instead."""
        if self._flags is None and self.kind == "split" and self.ticket is not None:
            if self._device is None:
                self.upload(self.reader.stream)
            if self._device.generation != self._dev_generation:
                raise RuntimeError("the batch's device tiles were recycled before its keep flags were read; "
                                   "read batch.flags before uploading later batches")
            self._flags = self._device.read_flags(self.n_entries, self.reader.stream)
        elif self._flags is None and self.kind == "split":
            src = self.source
            n_full = src.full_lengths[self.rows]
            full = self.u >= np.repeat(self.cdf0, n_full)
            if src.orig_pos is not None:        # a column shard keeps the flags of its own ratings
                rp = src.csr.rowptr
                loc = rp[self.rows + 1] - rp[self.rows]
                full_off = np.cumsum(n_full) - n_full
                loc_off = np.cumsum(loc) - loc
                ent = np.repeat(rp[self.rows] - loc_off, loc) + np.arange(int(loc.sum()), dtype=np.int64)
                full = full[np.repeat(full_off, loc) + src.orig_pos[ent]]
            self._flags = full.astype(np.uint8)
        return self._flags

    def upload(self, stream=None):
        """Stage + copy + gather (K1) into one of the reader's device batch buffers."""
        if self.kind == "split" and self.ticket is not None and self._flags is None and self._device is not None:
            self.flags                          # second upload: the draws are spent, take the flags from the first
        ring = self.reader._ring_for(self.n_rows, self.n_entries)
        dev = ring.next()
        if self.kind == "split" and self.ticket is not None and self._flags is None:
            handle = DeviceRng.get().consume(self.ticket)
            dev.fill_split_rng(self.source, self.rows, handle, self.sparsity[0], self.sparsity[1], self.full_len,
                               self.pass_through, self.aux_value, stream, self.rng_slice)
            self._dev_generation = dev.generation
        elif self.kind == "split" and self._flags is None:
            dev.fill_split_uniform(self.source, self.rows, self.u, self.cdf0, self.full_len, self.pass_through,
                                   self.aux_value, stream)
        elif self.kind == "split":
            dev.fill_split(self.source, self.rows, self.flags, self.pass_through, self.aux_value, stream)
        else:
            dev.fill_fixed(self.source, self.rows, self.aux_value, stream)
        self._device = dev
        return dev

    def row_slice(self, rank, world):
        """Rows [rank*B/world, (rank+1)*B/world) of this (global) batch as a batch of their own: what a
        data-parallel rank steps on. The random split stays the global batch's: every rank replays the
        whole batch's draws and reads its own rows' (on the device, or from the host draws)."""
        if self.n_rows % world:
            raise ValueError("a global batch of %d rows does not split over %d ranks" % (self.n_rows, world))
        if self.source.orig_pos is not None if self.kind == "split" else False:
            raise ValueError("row slices are taken from an unsharded reader")
        per = self.n_rows // world
        lo = rank * per
        rows = self.rows[lo:lo + per]
        if self.kind == "fixed":
            tcount = int(self.source.tgt_store.full_lengths[rows].sum())
            sub = Batch(self.reader, "fixed", self.source, rows, None, False, self.aux_type, self.aux_value, tcount,
                        self.return_target_count, tcount + int(self.source.in_store.full_lengths[rows].sum()))
        else:
            lens = self.source.lengths[self.rows]
            before, mine = int(lens[:lo].sum()), int(lens[lo:lo + per].sum())
            sub = Batch(self.reader, "split", self.source, rows, None, self.pass_through, self.aux_type, self.aux_value,
                        mine if self.pass_through else -1, False, mine)
            if self.ticket is not None and self._flags is None:
                sub.ticket, sub.sparsity = self.ticket, self.sparsity
                sub.rng_slice = (self.n_rows, lo, before, self.n_rows + int(lens.sum()))
            elif self._flags is None:
                sub.u, sub.cdf0 = self.u[before:before + mine], self.cdf0[lo:lo + per]
            else:
                sub._flags = self._flags[before:before + mine]
        sub.row0, sub.rows_total = lo, self.n_rows
        return sub

    # -- reference-shaped view ---------------------------------------------------------------
    def to_dense(self, stream=None):
        """(input_list, targets) exactly as `data_reader.py:354-363` builds them (float64)."""
        dev = self.upload(stream)
        get = lambda which: dev.densify(which, self.n_rows, self.n_cols, stream)
        x, mask_in, mask_out, t, observed = 0, 1, 2, 3, 4
        if self.aux_type is None:
            feed = [get(x), get(mask_out)]
        else:
            if self.aux_type == "causal":
                aux = get(observed)
            elif self.aux_type in ("dropout", "both"):
                aux = get(mask_in)
            elif self.aux_type == "zeros":
                aux = np.zeros((self.n_rows, self.n_cols))
            else:
                raise ValueError("Auxilliary mask type %r doesn't exist" % (self.aux_type,))
            feed = [get(x), aux, get(mask_out)]
            if self.aux_type == "both":
                feed.append(get(observed))
        return feed, get(t)

    def _as_tuple(self):
        feed, targets = self.to_dense()
        if self.return_target_count:
            return (feed, targets, self.target_count)
        return (feed, targets)

    def __iter__(self):
        return iter(self._as_tuple())

    def __len__(self):
        return 3 if self.return_target_count else 2

    def __getitem__(self, k):
        if k == 2 and self.return_target_count:
            return self.target_count
        return self._as_tuple()[k]


class Prefetcher(object):
    """Pulls exactly `count` items from a generator on a background thread (bounded queue): the
    role Keras' GeneratorEnqueuer (workers=1, max_q_size=10) plays for `fit_generator` in the
    reference (SURVEY.md section 3.1). NumPy releases the GIL inside `random_sample` and ctypes
    releases it inside the library, so drawing batch i+1 overlaps the staging and kernel launches of
    batch i. Items cross the queue in chunks (a queue hand-off costs about as much as building a
    device-drawn batch). Exactly `count` items are drawn, so the NumPy global stream ends where
    synchronous consumption would leave it; nothing else may draw from `np.random` while the
    thread runs."""

    def __init__(self, generator, count, depth=10, chunk=8):
        import queue
        self.count = max(int(count), 0)          # Keras runs zero steps for steps <= 0 (sets smaller than one batch)
        self.queue = queue.Queue(maxsize=depth)
        self.error = None
        chunk = max(1, int(chunk))

        def work():
            try:
                left = self.count
                first = True
                while left:
                    n = 1 if first else min(chunk, left)      # the first batch goes out at once
                    first = False
                    self.queue.put([next(generator) for _ in range(n)])
                    left -= n
            except BaseException as exc:          # surfaced on the consumer side
                self.error = exc
                self.queue.put(None)

        self.thread = threading.Thread(target=work, daemon=True)
        self.thread.start()

    def __iter__(self):
        left = self.count
        while left:
            items = self.queue.get()
            if items is None:
                raise self.error
            for item in items:
                yield item
            left -= len(items)
        self.thread.join()


class data_reader(object):
    """Drop-in for `data_reader.data_reader` (`data_reader.py:11-83`).

    Extra keyword `data`: instead of reading `filepath + name + ".json"` files, take
      * a dict {file base name: object} with the same names the reference loads
        (`unique_items_list`, `ratingsByUser_dicts_train`, ...), or
      * a `synthetic.FixedSplit` (CSR arrays; `eval_mode="fixed_split"` only).
    """

    def __init__(self, num_items, num_users, filepath, nonsequentialusers=False, use_json=True,
                 eval_mode="ablation", useTimestamps=False, reverse_user_item_data=False, data=None,
                 stream=None, shard=None, rng_on_device=None):
        if useTimestamps:
            raise NotImplementedError("useTimestamps is broken in the reference (data_reader.py:132,359,409) "
                                      "and out of scope here")
        if eval_mode not in ("ablation", "fixed_split"):
            raise ValueError("eval_mode must be 'ablation' or 'fixed_split'")
        self.num_items = int(num_items)
        self.num_users = int(num_users)
        self.filepath = filepath
        self.nonsequentialusers = nonsequentialusers
        self.eval_mode = eval_mode
        self.useTimestamps = useTimestamps
        self.stream = stream
        # None: draw the random split on the GPU whenever one is present (DeviceRng); False keeps
        # the NumPy stream on the host (one random_sample per batch)
        self.rng_on_device = rng_on_device
        self._files = data if isinstance(data, dict) else None
        self._rings = {}
        self._stores = {}
        from .ingest import LoadedSplit
        if isinstance(data, FixedSplit):
            self._init_from_split(data)
        elif isinstance(data, LoadedSplit):
            self._init_from_loaded(data)
        else:
            self._init_from_files(use_json, reverse_user_item_data)
        # column shard (rank, world): this process keeps catalogue columns [lo, hi) of every set;
        # rows, set orders and the RNG replay stay those of the full data (dist.py)
        self.shard = shard
        self.col_range = (0, self.num_items)
        if shard is not None:
            rank, world = shard
            lo, hi = rank * self.num_items // world, (rank + 1) * self.num_items // world
            self.col_range = (lo, hi)
            self._stores = {k: v.column_shard(lo, hi) for k, v in self._stores.items()}
        self.local_cols = self.col_range[1] - self.col_range[0]
        print("Finished loading data")

    # -- loading -----------------------------------------------------------------------------
    def load_data(self, filepath, filename, use_json):
        if self._files is not None:
            return self._files[filename]
        if use_json:
            with open(filepath + filename + ".json", "r") as f:
                return json.load(f)
        with open(filepath + filename + ".p", "rb") as f:
            return pickle.load(f)

    def _init_from_files(self, use_json, reverse):
        N = self.num_items
        cols_name = "unique_users_list" if reverse else "unique_items_list"
        self.unique_items = self.load_data(self.filepath, cols_name, use_json)
        self.items_to_densevec = {item: i for i, item in enumerate(self.unique_items)}       # :24-28
        self.densevec_to_items = {i: item for i, item in enumerate(self.unique_items)}
        if self.nonsequentialusers:                                                           # :30-44
            self.unique_users = self.load_data(self.filepath, "unique_items_list" if reverse else "unique_users_list", use_json)
            self.users_to_densevec = {u: i for i, u in enumerate(self.unique_users)}
            self.densevec_to_users = {i: u for i, u in enumerate(self.unique_users)}
        else:
            self.densevec_to_users = {i: i for i in range(self.num_users)}
        base = "ratingsByItem" if reverse else "ratingsByUser"                                # :46-49
        if reverse and self._files is None:
            # the reference's splitter writes `ratingsByUser*` even for reversed data (TrainValidTestSplit.py:153-157)
            # while its reader asks for `ratingsByItem*`: take whichever is on disk (SURVEY Appendix B)
            import os
            probe = "_dict" if self.eval_mode == "ablation" else "_dicts_train"
            ext = ".json" if use_json else ".p"
            if not os.path.exists(self.filepath + base + probe + ext) and os.path.exists(self.filepath + "ratingsByUser" + probe + ext):
                base = "ratingsByUser"
        # JSON files on disk go through the native parser (csrc/ocf_etl.cpp): no Python object per rating.
        # In-memory `data=` dicts and pickles keep the per-rating Python loop (small / test inputs).
        native = self._files is None and use_json
        if native:
            from . import ingest
            vocab = ingest.Vocab(self.filepath + cols_name + ".json")
            load = lambda name, paired: ingest.load_ratings(self.filepath + name + ".json", vocab, paired, N)
        if self.eval_mode == "ablation":
            if native:
                keys, csr = load(base + "_dict", False)                                       # :55
                row_of = {k: i for i, k in enumerate(keys)}
                want = []
                for i in range(self.num_users):
                    raw = self.densevec_to_users[i]
                    want.append(row_of[raw] if raw in row_of else row_of[str(raw)])
                csr = csr.take_rows(np.asarray(want, dtype=np.int64))
            else:
                user_dict = self.load_data(self.filepath, base + "_dict", use_json)
                lists = []
                for i in range(self.num_users):
                    raw = self.densevec_to_users[i]
                    lists.append(user_dict[raw] if raw in user_dict else user_dict[str(raw)])
                csr = _csr_from_lists(lists, self.items_to_densevec, N)
            self._stores["train"] = RatingStore(csr)
        elif native:
            # the three files parse concurrently (ctypes releases the GIL inside the library)
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=3) as pool:
                jobs = [pool.submit(load, base + "_dicts_train", False), pool.submit(load, base + "_dicts_valid", True),
                        pool.submit(load, base + "_dicts_test", True)]
                self.train_set, train = jobs[0].result()                                      # :67-70, :78-80
                self.val_set, va_in, _, va_tg = jobs[1].result()
                self.test_set, te_in, _, te_tg = jobs[2].result()
            self._set_sizes()
            self._stores["train"] = RatingStore(train)
            self._stores["valid"] = StorePair(RatingStore(va_in), RatingStore(va_tg))
            self._stores["test"] = StorePair(RatingStore(te_in), RatingStore(te_tg))
        else:
            train = self.load_data(self.filepath, base + "_dicts_train", use_json)            # :67-70
            valid = self.load_data(self.filepath, base + "_dicts_valid", use_json)
            test = self.load_data(self.filepath, base + "_dicts_test", use_json)
            self.train_set = list(train.keys())                                               # :78-80
            self.val_set = list(valid[1].keys())
            self.test_set = list(test[1].keys())
            self._set_sizes()
            col_of = self.items_to_densevec
            self._stores["train"] = RatingStore(_csr_from_lists(list(train.values()), col_of, N))
            for name, (ins, tgs), keys in (("valid", valid, self.val_set), ("test", test, self.test_set)):
                pair = StorePair(RatingStore(_csr_from_lists([ins[k] for k in keys], col_of, N)),
                                 RatingStore(_csr_from_lists([tgs[k] for k in keys], col_of, N)))
                self._stores[name] = pair

    def _init_from_loaded(self, ls):
        """Keys + CSR stores (ingest.LoadedSplit: parsed files, or splitter.split_in_memory)."""
        if self.eval_mode != "fixed_split":
            raise ValueError("a LoadedSplit only serves eval_mode='fixed_split'")
        if ls.n_cols > self.num_items:
            raise ValueError("num_items (%d) is smaller than the split's column count (%d)" % (self.num_items, ls.n_cols))
        self.unique_items = list(range(ls.n_cols)) if ls.unique_items is None else list(ls.unique_items)
        self.items_to_densevec = {item: i for i, item in enumerate(self.unique_items)}
        self.densevec_to_items = {i: item for i, item in enumerate(self.unique_items)}
        self.densevec_to_users = {i: i for i in range(self.num_users)}
        N = self.num_items

        def widen(csr):                    # the reader's arrays are num_items wide whatever the data uses (:13,109-118)
            return Csr(csr.n_rows, N, csr.rowptr, csr.col, csr.val)

        self.train_set, train = ls.train
        self.val_set, va_in, _, va_tg = ls.valid
        self.test_set, te_in, _, te_tg = ls.test
        self._set_sizes()
        self._stores["train"] = RatingStore(widen(train))
        self._stores["valid"] = StorePair(RatingStore(widen(va_in)), RatingStore(widen(va_tg)))
        self._stores["test"] = StorePair(RatingStore(widen(te_in)), RatingStore(widen(te_tg)))

    def _set_sizes(self):
        self.train_set_size = len(self.train_set)                                             # :73-75
        self.val_set_size = len(self.val_set)
        self.test_set_size = len(self.test_set)

    def _init_from_split(self, fs: FixedSplit):
        if self.eval_mode != "fixed_split":
            raise ValueError("a FixedSplit only serves eval_mode='fixed_split'")
        if fs.n_cols != self.num_items:
            raise ValueError("num_items (%d) must equal the split's column count (%d)" % (self.num_items, fs.n_cols))
        self.unique_items = list(range(fs.n_cols))
        self.train_set = [str(int(k)) for k in fs.train_keys]
        self.val_set = [str(int(k)) for k in fs.valid_keys]
        self.test_set = [str(int(k)) for k in fs.test_keys]
        self.train_set_size, self.val_set_size, self.test_set_size = len(self.train_set), len(self.val_set), len(self.test_set)
        self._stores["train"] = RatingStore(fs.train)
        self._stores["valid"] = StorePair(RatingStore(fs.valid_in), RatingStore(fs.valid_tg))
        self._stores["test"] = StorePair(RatingStore(fs.test_in), RatingStore(fs.test_tg))

    # -- ablation row split --------------------------------------------------------------------
    def split_for_validation(self, val_split, seed=None):
        """`data_reader.py:300-312`."""
        self.val_split = val_split
        sync_host_rng()
        if seed is not None:
            np.random.seed(seed)
        order = np.random.permutation(self.num_users)
        self.train_set_size = int(self.num_users * val_split[0])
        self.val_set_size = int(self.num_users * val_split[1])
        self.test_set_size = int(self.num_users * val_split[2])
        self.train_set = order[0:self.train_set_size]
        self.val_set = order[self.train_set_size:self.train_set_size + self.val_set_size]
        self.test_set = order[self.train_set_size + self.val_set_size:]

    # -- device buffers ------------------------------------------------------------------------
    def max_batch_entries(self, batch_size) -> int:
        """Upper bound of the ratings in any batch of `batch_size` rows of any set."""
        best = 1
        for src in self._stores.values():
            lens = np.sort(np.asarray(src.lengths))
            best = max(best, int(lens[-int(batch_size):].sum()))
        return best

    def _ring_for(self, rows, entries):
        ring = self._rings.get(rows)
        if ring is None or not ring.fits(rows, entries):
            if ring is not None:
                ring.close()
            ring = BatchRing(rows, max(self.max_batch_entries(rows), entries))
            self._rings[rows] = ring
        return ring

    def store(self, which):
        return self._stores[which]

    # -- the generator ---------------------------------------------------------------------------
    def data_gen(self, batch_size, data_sparsity, train_val_test="train", shuffle=True,
                 auxilliary_mask_type="dropout", aux_var_value=-1, return_target_count=False,
                 sparse_representation=False, pass_through_input_training=False):
        """`data_reader.py:314-419`. Yields `Batch` objects, then None for ever."""
        if sparse_representation:
            raise NotImplementedError("sparse_representation needs a patched Keras backend in the reference "
                                      "(train.py:53); batches here are never dense in the first place")
        if auxilliary_mask_type not in _lib.AUX_TYPES:
            print("Auxilliary mask type ", auxilliary_mask_type, " doesn't exist")
            raise ValueError(auxilliary_mask_type)
        if train_val_test == "train":
            order, n = self.train_set, self.train_set_size
        elif train_val_test == "valid":
            order, n = self.val_set, self.val_set_size
        elif train_val_test == "test":
            order, n = self.test_set, self.test_set_size
        else:
            raise ValueError(train_val_test)
        split_mode = self.eval_mode == "ablation" or train_val_test == "train"      # :331
        if self.eval_mode == "ablation":
            rows = np.asarray(order, dtype=np.int64)       # dense row ids == store rows (:124-125)
            source = self._stores["train"]
        else:
            rows = np.arange(len(order), dtype=np.int64)   # k-th key == k-th store row
            source = self._stores[train_val_test]
        sync_host_rng()                     # np.random must be current before anything draws on the host
        if shuffle:
            rows = rows[np.random.permutation(len(order))]                          # :326-327
        on_device = split_mode and (device_rng_available() if self.rng_on_device is None else bool(self.rng_on_device))
        batch_size = int(batch_size)
        num_batches = int(np.floor(n / batch_size))                                  # :329
        if split_mode and np.isscalar(data_sparsity):
            data_sparsity = [data_sparsity, data_sparsity]      # the reference crashes here (Appendix B)
        src_split = source if split_mode else None
        lengths = source.full_lengths if split_mode else None      # the RNG replay runs on full rows
        sharded = split_mode and source.orig_pos is not None
        for i in range(num_batches):
            brow = rows[i * batch_size:(i + 1) * batch_size]
            if split_mode and on_device:
                n_b = lengths[brow]
                draws = int(n_b.sum())
                tcount = draws if pass_through_input_training else -1
                batch = Batch(self, "split", source, brow, None, pass_through_input_training,
                              auxilliary_mask_type, aux_var_value, tcount, False, draws)
                batch.ticket = DeviceRng.get().ticket(batch_size + draws)       # uniform(B) then one draw per rating
                batch.sparsity = (float(data_sparsity[0]), float(data_sparsity[1]))
                batch.full_len = n_b if sharded else None
                yield batch
            elif split_mode:
                n_b = lengths[brow]
                sync_host_rng()
                keep = np.random.uniform(low=data_sparsity[0], high=data_sparsity[1], size=batch_size)   # :120
                u = np.random.random_sample(int(n_b.sum()))                                               # :130
                p0 = 1 - keep
                cdf0 = p0 / (p0 + keep)            # np.random.choice: cdf = cumsum(p) / cumsum(p)[-1]
                tcount = int(u.size) if pass_through_input_training else -1   # split batches do not report it
                batch = Batch(self, "split", source, brow, None, pass_through_input_training,
                              auxilliary_mask_type, aux_var_value, tcount, False, int(u.size))
                batch.u, batch.cdf0 = u, cdf0
                batch.full_len = n_b if sharded else None
                yield batch
            else:
                tcount = int(source.tgt_store.full_lengths[brow].sum())                                   # :268
                n_ratings = tcount + int(source.in_store.full_lengths[brow].sum())
                yield Batch(self, "fixed", source, brow, None, False, auxilliary_mask_type,
                            aux_var_value, tcount, return_target_count, n_ratings)
        while True:                                                                                        # :418-419
            yield None

    @staticmethod
    def sync_rng():
        """Bring `np.random` up to date with the draws the GPU made for this process's batches."""
        sync_host_rng()

    def close(self):
        for ring in self._rings.values():
            ring.close()
        self._rings = {}
        for s in self._stores.values():
            if isinstance(s, StorePair):
                s.close(); s.in_store.close(); s.tgt_store.close()
            else:
                s.close()
