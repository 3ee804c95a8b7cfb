"""Device-resident rating stores and batch buffers (thin owners of the C handles)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from .synthetic import Csr


class RatingStore(object):
    """One set of per-row rating lists (what `data_reader.py:46-70` keeps as dicts) as CSR on
    the host, uploaded to HBM on first use."""

    def __init__(self, csr: Csr, orig_pos=None, full_lengths=None):
        self.csr = csr
        self._handle = None
        # column shards (dist.py): position of each kept rating inside its full row, and the full
        # row lengths (the RNG replay and target counts are defined on full rows)
        self.orig_pos = orig_pos
        self._full_lengths = full_lengths
        self._lengths = None                # the store is immutable: row lengths are computed once

    @property
    def n_rows(self):
        return self.csr.n_rows

    @property
    def n_cols(self):
        return self.csr.n_cols

    @property
    def lengths(self):
        if self._lengths is None:
            self._lengths = np.diff(self.csr.rowptr)
        return self._lengths

    @property
    def full_lengths(self):
        return self.lengths if self._full_lengths is None else self._full_lengths

    def column_shard(self, lo: int, hi: int) -> "RatingStore":
        """The ratings of catalogue columns [lo, hi), relabelled to 0..hi-lo-1 (rows unchanged)."""
        c = self.csr
        keep = (c.col >= lo) & (c.col < hi)
        rows = np.repeat(np.arange(c.n_rows, dtype=np.int64), np.diff(c.rowptr))
        pos = np.arange(c.nnz, dtype=np.int64) - c.rowptr[rows]
        rowptr = np.zeros(c.n_rows + 1, dtype=np.int64)
        np.cumsum(np.bincount(rows[keep], minlength=c.n_rows), out=rowptr[1:])
        local = Csr(c.n_rows, hi - lo, rowptr, (c.col[keep] - lo).astype(np.int32), c.val[keep].copy())
        return RatingStore(local, orig_pos=pos[keep].astype(np.int32), full_lengths=self.lengths)

    @property
    def handle(self):
        if self._handle is None:
            _lib.require_gpu()
            rowptr = np.ascontiguousarray(self.csr.rowptr, dtype=np.int64)
            col = np.ascontiguousarray(self.csr.col, dtype=np.int32)
            val = np.ascontiguousarray(self.csr.val, dtype=np.float32)
            out = C.c_void_p()
            _lib.check(_lib.lib().ocf_store_create(self.csr.n_rows, self.csr.n_cols, _lib.ptr(rowptr),
                                                   _lib.ptr(col), _lib.ptr(val), C.byref(out)))
            self._handle = out
            if self.orig_pos is not None:
                op = np.ascontiguousarray(self.orig_pos, dtype=np.int32)
                _lib.check(_lib.lib().ocf_store_set_orig_pos(out, _lib.ptr(op)))
        return self._handle

    def info(self):
        buf = (C.c_int64 * 5)()
        _lib.check(_lib.lib().ocf_store_info(self.handle, buf))
        return dict(zip(("n_rows", "n_cols", "nnz", "has_dups", "device_bytes"), list(buf)))

    def close(self):
        if self._handle is not None:
            _lib.lib().ocf_store_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class StorePair(object):
    """Fixed-split valid/test set: inputs and targets with aligned rows (`data_reader.py:372-380`)."""

    def __init__(self, in_store: RatingStore, tgt_store: RatingStore):
        assert in_store.n_rows == tgt_store.n_rows and in_store.n_cols == tgt_store.n_cols
        self.in_store, self.tgt_store = in_store, tgt_store
        self._handle = None
        self._lengths = None

    @property
    def n_rows(self):
        return self.tgt_store.n_rows

    @property
    def n_cols(self):
        return self.tgt_store.n_cols

    @property
    def lengths(self):
        if self._lengths is None:
            self._lengths = self.in_store.lengths + self.tgt_store.lengths
        return self._lengths

    def column_shard(self, lo: int, hi: int) -> "StorePair":
        return StorePair(self.in_store.column_shard(lo, hi), self.tgt_store.column_shard(lo, hi))

    @property
    def handle(self):
        if self._handle is None:
            out = C.c_void_p()
            _lib.check(_lib.lib().ocf_pair_create(self.in_store.handle, self.tgt_store.handle, C.byref(out)))
            self._handle = out
        return self._handle

    def close(self):
        if self._handle is not None:
            _lib.lib().ocf_pair_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceBatch(object):
    """One `ocf_batch`: pinned staging + device tiles."""

    def __init__(self, max_rows: int, max_entries: int):
        _lib.require_gpu()
        self.max_rows, self.max_entries = int(max_rows), int(max(max_entries, 1))
        out = C.c_void_p()
        _lib.check(_lib.lib().ocf_batch_create(self.max_rows, self.max_entries, C.byref(out)))
        self.handle = out
        self.generation = 0         # bumped by every fill: tells whether a Batch's tiles are still here

    def fill_split(self, store: RatingStore, rows: np.ndarray, flags: np.ndarray, pass_through: bool,
                   aux_value: float, stream=None):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        flags = np.ascontiguousarray(flags, dtype=np.uint8)
        _lib.check(_lib.lib().ocf_batch_fill_split(self.handle, store.handle, _lib.ptr(rows), rows.size,
                                                   _lib.ptr(flags), flags.size, int(bool(pass_through)),
                                                   float(aux_value), stream))
        self.generation += 1

    def fill_split_uniform(self, store: RatingStore, rows: np.ndarray, u: np.ndarray, cdf0: np.ndarray,
                           full_len, pass_through: bool, aux_value: float, stream=None):
        """Like fill_split, from the raw uniform draws: the library derives the keep flags
        (u >= cdf0 of the row) while it stages the batch."""
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        u = np.ascontiguousarray(u, dtype=np.float64)
        cdf0 = np.ascontiguousarray(cdf0, dtype=np.float64)
        orig = None if store.orig_pos is None else np.ascontiguousarray(store.orig_pos, dtype=np.int32)
        fl = None if full_len is None else np.ascontiguousarray(full_len, dtype=np.int64)
        _lib.check(_lib.lib().ocf_batch_fill_split_uniform(self.handle, store.handle, _lib.ptr(rows), rows.size,
                                                           _lib.ptr(u), u.size, _lib.ptr(cdf0), _lib.ptr(orig),
                                                           _lib.ptr(fl), int(bool(pass_through)), float(aux_value), stream))
        self.generation += 1

    def fill_split_rng(self, store: RatingStore, rows: np.ndarray, rng_handle, lo: float, hi: float, full_len,
                       pass_through: bool, aux_value: float, stream=None, rng_slice=None):
        """Like fill_split, with the random split drawn on the device from the NumPy stream the
        `DeviceRng` holds (only the row ids cross PCIe)."""
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        fl = None if full_len is None else np.ascontiguousarray(full_len, dtype=np.int64)
        sl = None
        if rng_slice is not None:           # (rows of the drawing unit, first row, ratings before it, all draws)
            sl = C.byref(_lib.RngSlice(int(rng_slice[0]), int(rng_slice[1]), int(rng_slice[2]), int(rng_slice[3])))
        _lib.check(_lib.lib().ocf_batch_fill_split_rng(self.handle, store.handle, _lib.ptr(rows), rows.size, rng_handle,
                                                       float(lo), float(hi), _lib.ptr(fl), int(bool(pass_through)),
                                                       float(aux_value), sl, stream))
        self.generation += 1

    def read_flags(self, n_entries: int, stream=None) -> np.ndarray:
        out = np.empty(int(n_entries), dtype=np.uint8)
        _lib.check(_lib.lib().ocf_batch_read_flags(self.handle, _lib.ptr(out), out.size, stream))
        return out

    def fill_fixed(self, pair: StorePair, rows: np.ndarray, aux_value: float, stream=None):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        _lib.check(_lib.lib().ocf_batch_fill_fixed(self.handle, pair.handle, _lib.ptr(rows), rows.size,
                                                   float(aux_value), stream))
        self.generation += 1

    def info(self):
        buf = (C.c_int64 * 5)()
        _lib.check(_lib.lib().ocf_batch_info(self.handle, buf))
        return dict(zip(("rows", "entries", "items", "target_count", "h2d_bytes"), list(buf)))

    def densify(self, which: int, n_rows: int, n_cols: int, stream=None) -> np.ndarray:
        out = np.empty((n_rows, n_cols), dtype=np.float64)
        _lib.check(_lib.lib().ocf_batch_densify(self.handle, int(which), _lib.ptr(out), stream))
        return out

    def close(self):
        if self.handle is not None:
            _lib.lib().ocf_batch_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchRing(object):
    """A few DeviceBatch objects used round-robin, so staging batch i+1 on the host overlaps
    the device work of batch i."""

    def __init__(self, max_rows: int, max_entries: int, depth: int = 0):
        self.max_rows, self.max_entries = int(max_rows), int(max_entries)
        depth = depth or max(2, int(os.environ.get("OCF_RING_DEPTH", "3")))
        self.slots = [DeviceBatch(max_rows, max_entries) for _ in range(depth)]
        self.cursor = 0

    def fits(self, rows: int, entries: int) -> bool:
        return rows <= self.max_rows and entries <= self.max_entries

    def next(self) -> DeviceBatch:
        slot = self.slots[self.cursor]
        self.cursor = (self.cursor + 1) % len(self.slots)
        return slot

    def close(self):
        for s in self.slots:
            s.close()
        self.slots = []
