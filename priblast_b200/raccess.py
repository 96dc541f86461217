"""Host-side mirror of the reference's `class Raccess` (raccess.hpp:37-62) on top of the C ABI.

    Raccess(w, delta)                      <->  Raccess(int w, int delta)                  raccess.hpp:54
    Raccess(db_name, w, delta, path)       <->  Raccess(db_name, w, delta, path)           raccess.hpp:39
    .run(seq) -> (acc, cond)               <->  Run(seq, accessibility, conditional_accessibility)  :61
    .run_to_file(seq, idx)                 <->  Run(seq, idx)  (writes priblast_tmp_acc<rank>_<idx>.acc) :60
    .run_batch(seqs)                       <->  the OpenMP loop of db_construction.cpp:182-223

`delta` may also be a sequence of increasing minimum accessible lengths (at most 32): one context then computes all of
them, sharing the inside and outside passes, and run / run_batch / fetch return a dict {delta: what an int-delta
context returns}, bit-identical to it.

Differences, on purpose: invalid arguments raise ValueError instead of `exit(1)` (raccess.hpp:42-50),
and everything runs on one B200 through libpriblast_acc.so — there is no CPU path.
"""
from __future__ import annotations

import ctypes
import os
from collections.abc import Sequence
from typing import Iterable

import numpy as np

from . import _capi


def _probe_bytes_offset():
    """Byte offset of the character data inside a CPython `bytes` object, or None if the layout is not the expected
    one (then Raccess._marshal copies instead of pointing)."""
    off = bytes.__basicsize__ - 1
    for probe in (b"pRIblast", bytes(range(1, 200))):
        if ctypes.string_at(id(probe) + off, len(probe)) != probe:
            return None
    return off


_BYTES_OFFSET = _probe_bytes_offset()


def _as_bytes(seq) -> bytes:
    if isinstance(seq, bytes):
        return seq
    if isinstance(seq, str):
        return seq.encode("ascii", errors="replace")
    return bytes(seq)


def packed_layout(lens: Sequence[int]):
    """Float offsets (acc_off, cond_off, total) of the packed [acc L | cond L] per-sequence image."""
    lens = np.asarray(lens, dtype=np.int64)
    base = np.zeros(len(lens), dtype=np.int64)
    if len(lens):
        base[1:] = np.cumsum(2 * lens)[:-1]
    return base, base + lens, int((2 * lens).sum())


class AccResults(Sequence):
    """[(acc, cond), ...] as views into the one packed output buffer, made on demand (building thousands of numpy
    views eagerly costs more than the device-to-host copy of their data)."""

    def __init__(self, out, acc_off, cond_off, lens):
        self.out, self._a, self._c, self._l = out, acc_off, cond_off, lens

    def __len__(self):
        return len(self._l)

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self[i] for i in range(*k.indices(len(self)))]
        if k < 0:
            k += len(self)
        if not 0 <= k < len(self):
            raise IndexError(k)
        a, c, l = int(self._a[k]), int(self._c[k]), int(self._l[k])
        return self.out[a:a + l], self.out[c:c + l]


class Raccess:
    def __init__(self, *args, device: int = 0, max_batch_bytes: int = 0, mode: int = 0):
        """delta: an int, or a sequence of increasing ints (see the module docstring); `.lengths` is the tuple."""
        if len(args) == 2:
            w, delta = args
            db_name, path = "db", ""
        elif len(args) == 4:
            db_name, w, delta, path = args
            if len(db_name) == 0:
                raise ValueError("Error: -o option is required")  # raccess.hpp:42-45
        else:
            raise TypeError("Raccess(w, delta) or Raccess(db_name, w, delta, path)")
        self._multi = isinstance(delta, Iterable)
        self.lengths = tuple(int(d) for d in delta) if self._multi else (int(delta),)
        if any(d <= 1 for d in self.lengths):
            raise ValueError("Error: -d option must be greater than 1")  # raccess.hpp:47-50
        self.maximal_span = int(w)
        # the one length of an int-delta context (None with a list: record_bytes / run_to_file then need a delta)
        self.min_accessible_length = None if self._multi else self.lengths[0]
        self.path = path
        self.rank = 0
        self._lib = _capi.load()
        self._ctx = ctypes.c_void_p()
        prm = _capi.AccParams(self.maximal_span, self.lengths[0] if self.lengths else 0, int(device), int(mode),
                              int(max_batch_bytes))
        if self._multi:
            lengths = np.asarray(self.lengths, dtype=np.int32)
            _capi.check(self._lib.prib_acc_create_lengths(ctypes.byref(self._ctx), ctypes.byref(prm), len(lengths),
                                                          lengths.ctypes.data_as(_capi.c_i32p)))
        else:
            _capi.check(self._lib.prib_acc_create(ctypes.byref(self._ctx), ctypes.byref(prm)))
        self._staged_lens = None

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.prib_acc_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- the reference's two Run overloads ----------------------------------------------------------
    def run(self, sequence):
        """Run(seq, acc, cond): two float32 vectors of length L (raccess.cpp:484-528); {delta: (acc, cond)} for a
        list of lengths."""
        res = self.run_batch([sequence])
        if self._multi:
            return {d: r[0] for d, r in res.items()}
        return res[0]

    def _delta_to_write(self, delta):
        if delta is None:
            if self._multi:
                raise ValueError("this context computes several minimum accessible lengths: give the one to write")
            return self.min_accessible_length
        if int(delta) not in self.lengths:
            raise ValueError(f"minimum accessible length {delta} is not one of this context's {self.lengths}")
        return int(delta)

    def run_to_file(self, sequence, idx: int, delta: int | None = None) -> str:
        """Run(seq, idx): writes the per-sequence temp .acc file (raccess.cpp:447-481, utils.cpp:62-72) for `delta`
        (default: the context's one length)."""
        delta = self._delta_to_write(delta)
        res = self.run(sequence)
        acc, cond = res[delta] if self._multi else res
        name = f"priblast_tmp_acc{self.rank}_{idx}.acc"
        fn = os.path.join(self.path, name) if self.path else name
        with open(fn, "wb") as f:
            f.write(self.record_bytes(acc, cond, delta))
        return fn

    def record_bytes(self, acc: np.ndarray, cond: np.ndarray, delta: int | None = None) -> bytes:
        """The `.acc` record of one sequence at `delta` (default: the context's one length)."""
        delta = self._delta_to_write(delta)
        L = len(acc)
        n = self._lib.prib_acc_record_bytes(L, delta)
        if n < 0:
            raise ValueError("sequence shorter than the minimum accessible length")
        buf = ctypes.create_string_buffer(int(n))
        a = np.ascontiguousarray(acc, dtype=np.float32)
        c = np.ascontiguousarray(cond, dtype=np.float32)
        w = self._lib.prib_acc_write_record(a.ctypes.data_as(_capi.c_f32p), c.ctypes.data_as(_capi.c_f32p), L,
                                            delta, buf)
        assert w == n
        return buf.raw

    # -- batched form (what the db step uses) -------------------------------------------------------
    def _marshal(self, seqs: Iterable):
        """(keep-alive, n, lens, char**) for the C ABI.  No copy of the bases on this side: the pointer array holds
        the addresses of the `bytes` objects' own buffers (the library makes the one host copy, into its page-locked
        arena, batch by batch under the kernels of the previous batch).  Building a ctypes array of n `c_char_p`
        costs ~0.6 us per sequence and joining the sequences into one buffer ~0.4 ns per base -- either is more
        than the host-to-device copy of the bases -- so the addresses are computed with numpy from `id()` and the
        data offset of a CPython bytes object, checked once at import (`_BYTES_OFFSET`); if that check ever fails the
        sequences are joined into one buffer instead."""
        bs = [s if type(s) is bytes else _as_bytes(s) for s in seqs]
        n = len(bs)
        lens = np.fromiter(map(len, bs), dtype=np.int32, count=n)
        if _BYTES_OFFSET is not None:
            ptrs = np.fromiter(map(id, bs), dtype=np.uint64, count=n) if n else np.zeros(1, dtype=np.uint64)
            ptrs += np.uint64(_BYTES_OFFSET)
            keep = bs
        else:
            blob = np.frombuffer(b"".join(bs) or b"\0", dtype=np.uint8)
            ptrs = np.empty(max(n, 1), dtype=np.uint64)
            ptrs[0] = blob.ctypes.data
            if n > 1:
                np.cumsum(lens[:-1], dtype=np.uint64, out=ptrs[1:n])
                ptrs[1:n] += np.uint64(blob.ctypes.data)
            keep = blob
        arr = ptrs.ctypes.data_as(ctypes.POINTER(ctypes.c_char_p))
        return (keep, ptrs), n, lens, arr

    def _layout(self, lens):
        """Offsets of the packed image of every length, back to back (the layout prib_acc_fetch copies straight)."""
        acc_off, cond_off, total = packed_layout(lens)
        k = len(self.lengths)
        shift = np.repeat(np.arange(k, dtype=np.int64) * total, len(lens))
        return np.tile(acc_off, k) + shift, np.tile(cond_off, k) + shift, total * k

    def _results(self, out, acc_off, cond_off, lens):
        n = len(lens)
        res = {d: AccResults(out, acc_off[l * n:(l + 1) * n], cond_off[l * n:(l + 1) * n], lens)
               for l, d in enumerate(self.lengths)}
        return res if self._multi else res[self.lengths[0]]

    def run_batch(self, seqs: Iterable, out: np.ndarray | None = None):
        """All sequences in one C-ABI call; returns [(acc, cond), ...] as views into one buffer ({delta: [...]} for a
        list of lengths)."""
        bs, n, lens, arr = self._marshal(seqs)
        acc_off, cond_off, total = self._layout(lens)
        if out is None:
            out = np.empty(max(total, 1), dtype=np.float32)
        assert out.dtype == np.float32 and out.size >= total
        _capi.check(self._lib.prib_acc_run(self._ctx, n, arr, lens.ctypes.data_as(_capi.c_i32p),
                                           out.ctypes.data_as(ctypes.c_void_p),
                                           acc_off.ctypes.data_as(_capi.c_i64p),
                                           cond_off.ctypes.data_as(_capi.c_i64p)))
        return self._results(out, acc_off, cond_off, lens)

    # -- split form: inputs resident on the device ---------------------------------------------------
    def stage(self, seqs: Iterable) -> int:
        bs, n, lens, arr = self._marshal(seqs)
        _capi.check(self._lib.prib_acc_stage(self._ctx, n, arr, lens.ctypes.data_as(_capi.c_i32p)))
        self._staged_lens = lens
        return int(lens.sum())

    def compute(self) -> None:
        _capi.check(self._lib.prib_acc_compute(self._ctx))

    def sync(self) -> None:
        _capi.check(self._lib.prib_acc_sync(self._ctx))

    def fetch(self, out: np.ndarray | None = None):
        lens = self._staged_lens
        acc_off, cond_off, total = self._layout(lens)
        if out is None:
            out = np.empty(max(total, 1), dtype=np.float32)
        _capi.check(self._lib.prib_acc_fetch(self._ctx, out.ctypes.data_as(ctypes.c_void_p),
                                             acc_off.ctypes.data_as(_capi.c_i64p),
                                             cond_off.ctypes.data_as(_capi.c_i64p)))
        return self._results(out, acc_off, cond_off, lens)

    def set_stream(self, cuda_stream_handle: int | None) -> None:
        _capi.check(self._lib.prib_acc_set_stream(self._ctx, ctypes.c_void_p(cuda_stream_handle or 0)))

    def counters(self) -> dict:
        c = _capi.AccCounters()
        _capi.check(self._lib.prib_acc_get_counters(self._ctx, ctypes.byref(c)))
        d = {k: getattr(c, k) for k, _ in c._fields_}
        d["phase_ms"] = dict(zip(_capi.PHASE_NAMES, list(c.phase_ms)))
        d["fp32_flagged"] = list(c.fp32_flagged)
        return d


def suffix_array(text, device: int = 0) -> np.ndarray:
    """Suffix array (int32) of an encoded database page on the GPU: the drop-in for the reference's
    `sais(T, SA, n)` (sais.cpp:656, called at db_construction.cpp:334).  `text`: bytes / uint8 array of
    symbols 0..9 (encoder.hpp:36-78)."""
    t = np.ascontiguousarray(np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else text,
                             dtype=np.uint8)
    sa = np.empty(len(t), dtype=np.int32)
    lib = _capi.load()
    _capi.check(lib.prib_suffix_array(t.ctypes.data_as(ctypes.c_void_p), len(t), sa.ctypes.data_as(_capi.c_i32p),
                                      int(device)))
    return sa
