"""Host pipeline over the C ABI: pack -> K1 count -> (K1x/K2) -> K3 -> K4/K5.

PyTorch is used only as plumbing: device/pinned allocations, streams, and
``torch.distributed`` (NCCL) for the one exchange step of the kNN (all-gather
of the operand shards).  All arithmetic happens inside libkarma_b200.so.

Column dictionary (kmer.py:146-179).  kmer.py's columns are the k-mer strings
that occur anywhere in the input, in ``sorted()`` order.  The GPU counts into
the full ACGT code space (already in sorted order) and reports which columns
are present; this module turns presence bits (+ the keys of non-ACGT windows
from K1x) into the column list and a compaction map.  That is dictionary
bookkeeping over <= a few thousand strings, not a compute fallback.
"""
import ctypes
from ctypes import byref, c_float, c_int64, c_void_p

import numpy as np
import torch

from . import _lib
from ._lib import (KB_COUNT_NO_COLUMNS, KB_KNN_AUTO, KB_MODE_5P6, KB_MODE_DENSE_4_5, KB_MODE_DENSE_5_6, KB_MODE_K,
                   check, ptr)

_BASES = "ACGT"
SORTED_K_MIN, SORTED_K_MAX = 8, 16          # integer k of the sorted counting path (kb_kmer_sorted_collect)


def is_sorted_mode(mode):
    return mode >= KB_MODE_K(SORTED_K_MIN)


def mode_of(kmer_size):
    """kmer.py's kmer_size ("5p6" or int) or a dense-mode name -> KB_MODE_*."""
    if kmer_size == "5p6":
        return KB_MODE_5P6
    if kmer_size == "5+6":
        return KB_MODE_DENSE_5_6
    if kmer_size == "4+5":
        return KB_MODE_DENSE_4_5
    if isinstance(kmer_size, (int, np.integer)) and not isinstance(kmer_size, bool):
        # k <= 7: dense shared-memory histograms over the ACGT code space; 8 <= k <= 16: sorted k-mer keys
        # (columns = the observed k-mers, as in kmer.py).  Beyond 16 a k-mer no longer fits the 128-bit sort key.
        if not 1 <= int(kmer_size) <= SORTED_K_MAX:
            raise _lib.KarmaB200Error(-4, "integer k-mer sizes 1..%d are built (got %r)" % (SORTED_K_MAX, kmer_size))
        return KB_MODE_K(int(kmer_size))
    # same failure kmer.py produces for e.g. "4p5": len(seq) - "4p5" -> TypeError (kmer.py:84)
    raise TypeError("unsupported operand type(s) for -: 'int' and %r" % type(kmer_size).__name__)


def _kmer(code, k):
    return "".join(_BASES[(code >> (2 * (k - 1 - t))) & 3] for t in range(k))


_names_cache = {}


def mode_column_names(mode):
    """Names of the fixed ACGT columns of a mode, in column order."""
    if mode in _names_cache:
        return _names_cache[mode]
    if mode == KB_MODE_5P6:
        # sorted(5-mers U string-palindromic 6-mers), kmer.py:172: x1x2x3x3x2x1 follows x1x2x3x3x2
        names = []
        for c in range(1024):
            s = _kmer(c, 5)
            names.append(s)
            if s[3] == s[2] and s[4] == s[1]:
                names.append(s + s[0])
    elif mode == KB_MODE_DENSE_5_6:
        names = [_kmer(c, 5) for c in range(1024)] + [_kmer(c, 6) for c in range(4096)]
    elif mode == KB_MODE_DENSE_4_5:
        names = [_kmer(c, 4) for c in range(256)] + [_kmer(c, 5) for c in range(1024)]
    else:
        k = mode - 16
        names = [_kmer(c, k) for c in range(4 ** k)]
    _names_cache[mode] = names
    return names


def decode_exotic_key(key):
    """63-bit key of kb_exotic_collect -> the k-mer string (latin-1 bytes)."""
    out = []
    for t in range(7):
        v = (int(key) >> (9 * (6 - t))) & 511
        if v == 0:
            break
        out.append(chr(v - 1))
    return "".join(out)


def shard_bounds(n_total, world, rank):
    """Contiguous row shard of ``rank``: blocks of per=ceil(n/world) rows, so that the
    index of a row in the zero-padded all-gathered key set equals its global index."""
    per = -(-n_total // world) if n_total else 0
    lo = min(rank * per, n_total)
    hi = min(lo + per, n_total)
    return lo, hi, per


def merge_columns(names, present, exotic_names):
    """kmer.py:172-177: the column list is sorted(observed k-mer strings).
    names/present describe the fixed ACGT columns (already in sorted order);
    exotic_names are the k-mers with non-ACGT characters (any order, unique).
    Returns (columns, colmap int32[len(names)], keycol int32[len(exotic_names)])."""
    present = np.asarray(present, dtype=bool)
    merged = sorted([(names[i], 0, int(i)) for i in np.flatnonzero(present)] +
                    [(s, 1, j) for j, s in enumerate(exotic_names)])
    columns = [m[0] for m in merged]
    colmap = np.full(len(names), -1, dtype=np.int32)
    keycol = np.full(len(exotic_names), -1, dtype=np.int32)
    for dst, (_, kind, src) in enumerate(merged):
        if kind == 0:
            colmap[src] = dst
        else:
            keycol[src] = dst
    return columns, colmap, keycol


def all_gather_padded(t, n, per, group, fill=0):
    """All-gather row shards of unequal length: rows [0,n) of ``t`` are padded to
    ``per`` rows with ``fill`` and gathered into (per*world, ...).  Works for any
    backend/device (NCCL on GPU, gloo on CPU)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    pad = torch.full((per,) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=t.device)
    pad[:n] = t[:n]
    out = torch.empty((per * world,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    return out


class ZeroRowError(Exception):
    """A contig shorter than k: kmer.py logs an error and exit(1)s (kmer.py:250-258)."""

    def __init__(self, row):
        super().__init__("Values of row %d are all zero, which should not be the case." % row)
        self.row = row


class Engine:
    """One GPU, one context.  Not thread-safe."""

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise _lib.KarmaB200Error(_lib.KB_ENOGPU, "no CUDA device visible: karma_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        torch.cuda.set_device(self.device)
        h = c_void_p()
        check(self.lib.kb_create(byref(h), self.device_index))
        self.ctx = h
        self._ws = None          # kNN workspace (grown on demand)
        self._side = None        # D2H stream of the profile download
        self._up = None          # H2D stream of the chunked upload
        self._host = {}          # reusable pinned result buffers
        self._hold_stream = False
        self.timing_enabled = False
        self.last_uncertified = 0
        self._bind_stream()

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.kb_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _bind_stream(self):
        """Point the library at torch's current stream (skipped while a pass holds the binding)."""
        if self._hold_stream:
            return
        check(self.lib.kb_set_stream(self.ctx, c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    # ---- timing / accounting -------------------------------------------------
    def enable_timing(self, on=True):
        check(self.lib.kb_enable_timing(self.ctx, 1 if on else 0))
        self.timing_enabled = bool(on)

    def stage_ms(self, stage):
        """(mean ms, launches) of a stage since the last read; synchronises."""
        ms, n = c_float(), ctypes.c_int()
        check(self.lib.kb_stage_ms(self.ctx, _lib.STAGES[stage], byref(ms), byref(n)))
        return ms.value, n.value

    def launches(self):
        return int(self.lib.kb_launch_count(self.ctx))

    # ---- host-side plumbing -------------------------------------------------------
    def side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(self.device)
        return self._side

    def host_buffer(self, name, shape, dtype, reuse):
        """Pinned host tensor for a result.  ``reuse``: one buffer per name, kept by the
        engine and overwritten by the next call."""
        if not reuse:
            return torch.empty(shape, dtype=dtype, pin_memory=True)
        cache = self._host
        t = cache.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = torch.empty(shape, dtype=dtype, pin_memory=True)
            cache[name] = t
        return t

    # ---- uploads ---------------------------------------------------------------
    def upload(self, bases, offsets, key_len, pinned=False):
        """Host arrays -> device tensors.  ``bases`` is padded so that the kernel's
        aligned 128-bit loads stay inside the allocation."""
        total = int(offsets[-1])
        cap = (total + 15) // 16 * 16 + 32
        d_bases = torch.empty(cap, dtype=torch.uint8, device=self.device)
        hb = bases if isinstance(bases, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(bases))
        ho = offsets if isinstance(offsets, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64))
        hk = key_len if isinstance(key_len, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(key_len, dtype=np.int32))
        d_bases[:total].copy_(hb[:total], non_blocking=True)
        d_offsets = ho.to(self.device, non_blocking=True)
        d_key_len = hk.to(self.device, non_blocking=True)
        return d_bases, d_offsets, d_key_len

    def upload_chunked(self, bases, offsets, key_len, n_chunks):
        """Like upload(), but the bases go up in ``n_chunks`` row chunks on a copy stream, each
        followed by an event, so that counting (and the profile download, which uses the other
        DMA direction) can start while the rest of the assembly is still in flight.
        Returns (d_bases, d_offsets, d_key_len, [(row_lo, row_hi, event), ...])."""
        n = len(offsets) - 1
        total = int(offsets[-1])
        cap = (total + 15) // 16 * 16 + 32
        d_bases = torch.empty(cap, dtype=torch.uint8, device=self.device)
        hb = bases if isinstance(bases, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(bases))
        ho = offsets if isinstance(offsets, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64))
        hk = key_len if isinstance(key_len, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(key_len, dtype=np.int32))
        main = torch.cuda.current_stream(self.device)
        if self._up is None:
            self._up = torch.cuda.Stream(self.device)
        up = self._up
        up.wait_stream(main)
        chunks = []
        with torch.cuda.stream(up):
            d_offsets = ho.to(self.device, non_blocking=True)
            d_key_len = hk.to(self.device, non_blocking=True)
            for c in range(n_chunks):
                lo, hi = n * c // n_chunks, n * (c + 1) // n_chunks
                b0, b1 = int(ho[lo]), int(ho[hi])
                if b1 > b0:
                    d_bases[b0:b1].copy_(hb[b0:b1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(up)
                chunks.append((lo, hi, ev))
        d_bases.record_stream(up)                      # allocated for the main stream, filled on the copy stream
        d_offsets.record_stream(main)                  # allocated on the copy stream, consumed on the main stream
        d_key_len.record_stream(main)
        return d_bases, d_offsets, d_key_len, chunks

    # ---- K1 ----------------------------------------------------------------------
    def count(self, d_bases, d_offsets, n, mode, counts=None, exotic=None, presence=None, zero_presence=True,
              columns=True):
        """u32 counts (n, D) [torch.int32 storage], exotic tallies (n,), presence (D+1,):
        presence[c] != 0 iff column c occurs, presence[D] bit0 iff a window holds a non-ACGT byte.
        ``columns=False``: only presence[D] is written (K3 can derive the column words)."""
        self._bind_stream()
        cols = check(self.lib.kb_mode_columns(mode))
        if not columns:
            mode = mode | KB_COUNT_NO_COLUMNS
        if counts is None:
            counts = torch.empty((n, cols), dtype=torch.int32, device=self.device)
        if exotic is None:
            exotic = torch.empty(n, dtype=torch.int32, device=self.device)
        if presence is None:
            presence = torch.empty(cols + 1, dtype=torch.int32, device=self.device)
        if zero_presence:
            presence.zero_()
        check(self.lib.kb_count(self.ctx, mode, ptr(d_bases), ptr(d_offsets), n, ptr(counts), counts.stride(0),
                                ptr(exotic), ptr(presence)))
        return counts, exotic, presence

    def count_profile(self, d_bases, d_offsets, d_key_len, lo, hi, mode, profile, operand, rowmeta, exotic, presence,
                      flags_or, rows_alloc=None):
        """K1+K3 fused (kb_count_profile) on rows [lo, hi) of preallocated outputs; the call that reaches the last
        real row also writes the gather padding rows up to ``rows_alloc``."""
        self._bind_stream()
        n = d_offsets.numel() - 1
        n_alloc = hi - lo
        if rows_alloc is not None and hi == n:
            n_alloc = int(rows_alloc) - lo
        if n_alloc <= 0:
            return
        check(self.lib.kb_count_profile(self.ctx, mode, ptr(d_bases), ptr(d_offsets[lo:]), ptr(d_key_len[lo:]) if hi > lo else None,
                                        hi - lo, n_alloc, ptr(profile[lo:]) if profile is not None and hi > lo else None,
                                        profile.stride(0) if profile is not None else 0,
                                        ptr(operand[lo:]) if operand is not None else None,
                                        operand.stride(0) if operand is not None else 0,
                                        ptr(rowmeta[lo:]), ptr(exotic[lo:]) if exotic is not None and hi > lo else None,
                                        ptr(presence), ptr(flags_or)))

    def count_stats(self):
        nl, ex = c_int64(), c_int64()
        check(self.lib.kb_count_stats(self.ctx, byref(nl), byref(ex)))
        return nl.value, ex.value

    # ---- K1x / K2: column dictionary ---------------------------------------------
    def build_columns(self, mode, d_bases, d_offsets, n, counts, exotic, presence, group=None, reduced=False):
        """kmer.py:146-179.  Returns (columns, counts') where columns is the sorted
        list of observed k-mer strings and counts' the (n, D') matrix in that order.
        One collective (MAX over the presence vector, which also carries the
        "non-ACGT window seen" flag) and one D2H copy."""
        self._bind_stream()
        names = mode_column_names(mode)
        if group is not None and not reduced:
            import torch.distributed as dist
            dist.all_reduce(presence, op=dist.ReduceOp.MAX, group=group)
        pres_h = presence.cpu().numpy()
        present = pres_h[:len(names)] != 0
        any_exotic = bool(pres_h[len(names)])
        keys = np.zeros(0, dtype=np.uint64)
        if any_exotic:
            nk, ne = c_int64(), c_int64()
            check(self.lib.kb_exotic_collect(self.ctx, mode, ptr(d_bases), ptr(d_offsets), n, ptr(exotic),
                                             byref(nk), byref(ne)))
            keys = np.empty(nk.value, dtype=np.uint64)
            if nk.value:
                check(self.lib.kb_exotic_fetch(self.ctx, keys.ctypes.data_as(c_void_p), None, None, None))
            if group is not None:
                import torch.distributed as dist
                gathered = [None] * dist.get_world_size(group)
                dist.all_gather_object(gathered, keys, group=group)
                all_keys = np.unique(np.concatenate(gathered)) if gathered else keys
            else:
                all_keys = keys
        else:
            all_keys = keys
        if present.all() and len(all_keys) == 0:
            return list(names), counts
        exo_names = [decode_exotic_key(k) for k in all_keys]
        columns, colmap, keycol_all = merge_columns(names, present, exo_names)
        d_out = len(columns)
        ld_out = max(4, (d_out + 3) // 4 * 4)
        out = torch.empty((n, ld_out), dtype=torch.int32, device=self.device)
        d_colmap = torch.from_numpy(colmap).to(self.device)
        check(self.lib.kb_compact(self.ctx, ptr(counts), counts.stride(0), counts.shape[1], ptr(d_colmap), n,
                                  ptr(out), ld_out, d_out))
        if len(keys):
            # local unique keys -> destination columns
            pos = np.searchsorted(all_keys, keys)
            d_keycol = torch.from_numpy(keycol_all[pos]).to(self.device)
            check(self.lib.kb_exotic_scatter(self.ctx, ptr(d_keycol), ptr(out), ld_out))
        return columns, out[:, :d_out]

    def build_columns_sorted(self, k, d_bases, d_offsets, n, group=None):
        """Integer k >= 8 (kmer.py:83-85, :146-179): every k-window becomes a 128-bit key on the GPU, sorted and
        reduced to the observed k-mers (= kmer.py's sorted() columns) and the (row, column, count) entries, which are
        scattered into a zeroed count matrix.  Returns (columns, counts (n, D'))."""
        self._bind_stream()
        nk, ne = c_int64(), c_int64()
        check(self.lib.kb_kmer_sorted_collect(self.ctx, int(k), ptr(d_bases), ptr(d_offsets), n, byref(nk), byref(ne)))
        hi = np.zeros(nk.value, dtype=np.uint64)
        lo = np.zeros(nk.value, dtype=np.uint64)
        if nk.value:
            check(self.lib.kb_kmer_sorted_fetch(self.ctx, hi.ctypes.data_as(c_void_p), lo.ctypes.data_as(c_void_p)))

        def as_bytes(h, l):          # (m, 16) big-endian bytes: lexicographic order == key order == Python string order
            return np.concatenate([h.astype(">u8").view(np.uint8).reshape(-1, 8), l.astype(">u8").view(np.uint8).reshape(-1, 8)], axis=1)
        mine = np.ascontiguousarray(as_bytes(hi, lo)).view("S16").reshape(-1)
        if group is not None:
            import torch.distributed as dist
            gathered = [None] * dist.get_world_size(group)
            dist.all_gather_object(gathered, mine, group=group)
            all_keys = np.unique(np.concatenate(gathered))
        else:
            all_keys = mine
        raw = np.frombuffer(np.ascontiguousarray(all_keys).tobytes().ljust(16 * len(all_keys), b"\0"), dtype=np.uint8).reshape(-1, 16)[:, :k]
        columns = [bytes(r).decode("latin-1") for r in raw]
        d_cols = len(columns)
        ld = max(4, (d_cols + 3) // 4 * 4)
        counts = torch.zeros((n, ld), dtype=torch.int32, device=self.device)
        if nk.value:
            key_col = np.searchsorted(all_keys, mine).astype(np.int32) if group is not None else np.arange(nk.value, dtype=np.int32)
            d_keycol = torch.from_numpy(key_col).to(self.device)
            check(self.lib.kb_exotic_scatter(self.ctx, ptr(d_keycol), ptr(counts), ld))
        return columns, counts[:, :d_cols]

    # ---- K3 ------------------------------------------------------------------------
    def normalise(self, counts, d_cols, d_key_len, want_profile=True, want_operand=True, profile=None,
                  rows_alloc=None, launch=True, presence=None, flags_or=None):
        """K3.  With ``rows_alloc`` > n the kNN inputs are allocated with that many rows
        (the equal-size shard a rank contributes to the exchange); K3 writes the padding rows
        (zero counts, flagged so that they can never be neighbours).  ``presence`` (D+1 words,
        accumulating) / ``flags_or`` (1 word, accumulating) as in kb_normalise."""
        self._bind_stream()
        n = counts.shape[0]
        rows = n if rows_alloc is None else max(n, int(rows_alloc))
        ldp = d_cols
        if want_profile and profile is None:
            profile = torch.empty((n, ldp), dtype=torch.float64, device=self.device)
        dp = (d_cols + 63) // 64 * 64
        operand = torch.empty((rows, dp), dtype=torch.float16, device=self.device) if want_operand else None
        # kb_rowmeta records (32 B): [sqnorm f64 | key_len i32 | flags i32 | cm_x f32 | cm_y f32 | 2 x reserved]
        rowmeta = torch.empty((rows, 8), dtype=torch.int32, device=self.device)
        if launch:
            self.normalise_rows(counts, d_cols, d_key_len, 0, n, profile, operand, rowmeta, rows, presence, flags_or)
        return profile, operand, rowmeta

    def normalise_rows(self, counts, d_cols, d_key_len, lo, hi, profile, operand, rowmeta, rows_alloc=None,
                       presence=None, flags_or=None):
        """K3 on rows [lo, hi) of preallocated outputs (the chunked upload path runs it per chunk);
        ``rows_alloc``: total rows of operand/rowmeta -- the call that reaches the last real row also writes
        the padding rows behind it."""
        self._bind_stream()
        n = counts.shape[0]
        n_alloc = hi - lo
        if rows_alloc is not None and hi == n:
            n_alloc = int(rows_alloc) - lo
        if n_alloc <= 0:
            return
        c = counts[lo:hi] if hi > lo else counts[0:0]
        check(self.lib.kb_normalise(self.ctx, ptr(c) if hi > lo else None, counts.stride(0), d_cols,
                                    ptr(d_key_len[lo:hi]) if hi > lo else None, hi - lo, n_alloc,
                                    ptr(profile[lo:hi]) if profile is not None and hi > lo else None,
                                    profile.stride(0) if profile is not None else 0,
                                    ptr(operand[lo:]) if operand is not None else None,
                                    operand.stride(0) if operand is not None else 0, ptr(rowmeta[lo:]),
                                    ptr(presence), ptr(flags_or)))

    # ---- K4 + K5 ---------------------------------------------------------------------
    def knn_enqueue(self, operand, rowmeta, k, q_row0=0, nq=None, impl=KB_KNN_AUTO, want_d2=False,
                    flag_rows=None, flag_counts=None, out=None, xchg=None):
        """Enqueue K4 (+K4x) + K5.  Returns (idx, dist, d2, fixup): ``fixup()`` synchronises, redoes the rows
        K5 could not certify with exact distances to all keys (kb_knn_fixup) and returns how many there were.
        flag_rows (int32, ascending key rows) / flag_counts (u32 rows, same order) describe the rows the
        tensor path cannot score exactly (kb_rowmeta flags 1|2).  ``out``: preallocated (idx, dist)."""
        self._bind_stream()
        nk, dp = operand.shape
        nq = nk - q_row0 if nq is None else nq
        n_flag = 0 if flag_rows is None else int(flag_rows.numel())
        need = check(self.lib.kb_knn_workspace_bytes(self.ctx, nq, nk, q_row0, dp, k, impl, n_flag))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        ws = self._ws
        if out is None:
            idx = torch.empty((nq, k), dtype=torch.int32, device=self.device)
            dist = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        else:
            idx, dist = out
        d2 = torch.empty((nq, k), dtype=torch.float64, device=self.device) if want_d2 else None
        args = (self.ctx, impl, k, ptr(operand), operand.stride(0), dp, ptr(rowmeta), nk, q_row0, nq,
                ptr(flag_rows) if n_flag else None, ptr(flag_counts) if n_flag else None,
                flag_counts.stride(0) if n_flag else 0, flag_counts.shape[1] if n_flag else 0, n_flag,
                ptr(idx), ptr(dist), ptr(d2), ptr(ws), ws.numel())
        check(self.lib.kb_knn(*args, xchg))

        def fixup():
            self._bind_stream()
            return check(self.lib.kb_knn_fixup(*args))
        return idx, dist, d2, fixup

    def knn(self, operand, rowmeta, k, **kw):
        """K4 (+K4x) + K5 + the exact pass over rows that could not be certified.  Synchronises."""
        idx, dist, d2, fixup = self.knn_enqueue(operand, rowmeta, k, **kw)
        self.last_uncertified = fixup()
        return idx, dist, d2

    def word_view(self, addr):
        """1-element int32 tensor aliasing a device word inside the kNN workspace."""
        off = addr - self._ws.data_ptr()
        assert 0 <= off < self._ws.numel() and off % 4 == 0
        return self._ws[off:off + 4].view(torch.int32)

    def uncertified_word(self, nq, nk, q_row0, dp, k, impl, n_flag=0):
        """Device address (int) of the word in which the last knn_enqueue of this shape counts its uncertified rows."""
        out = c_void_p()
        check(self.lib.kb_knn_uncertified_ptr(self.ctx, nq, nk, q_row0, dp, k, impl, n_flag, ptr(self._ws), byref(out)))
        return out.value


# ---------------------------------------------------------------------------------------
# whole path
# ---------------------------------------------------------------------------------------

def all_gather_rows(t, group):
    """All-gather equal row shards into one (rows*world, ...) tensor."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    out = torch.empty((t.shape[0] * world,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t, group=group)
    return out


def device_pass(engine, *args, **kwargs):
    """See _device_pass.  The stream binding of the library is taken once for the whole pass."""
    engine._bind_stream()
    held = engine._hold_stream
    engine._hold_stream = True
    try:
        return _device_pass(engine, *args, **kwargs)
    finally:
        engine._hold_stream = held


def _presence_summary(pres, faithful):
    """(exotic_seen, all_columns_present) from a presence vector: [D] bit0 = a non-ACGT byte was seen,
    bit1 = some CTA of K3 saw every column (then the per-column words were not written)."""
    last = int(pres[-1])
    return bool(last & 1), bool(last & 2) or bool(np.asarray(pres[:-1]).all())


def _device_pass(engine, d_bases, d_offsets, d_key_len, n, kmer_size="5p6", n_neighbors=None, impl=KB_KNN_AUTO,
                 want_profile=True, group=None, rank=0, world=1, n_total=None, gather_lists=False, bufs=None,
                 on_profile=None, optimistic=True, row0=0, chunks=None):
    """The hot path on device-resident inputs: K1 -> column dictionary (-> K1x/K2) -> K3
    [-> all-gather of the operand shards -> K4 (-> K4x) -> K5 (-> K6)].  Returns device tensors plus
    the column list.  This is the eager, general form (any input); `PassPlan` is the pre-planned,
    graph-captured form of its optimistic branch for repeated passes.

    ``optimistic``: real assemblies contain every ACGT k-mer column, no non-ACGT bytes and no
    row beyond the exact range of the tensor path, so the whole pass is enqueued without a
    host round trip on that assumption; a few validation words are copied back asynchronously and
    checked at the end (one synchronisation per pass).  If the assumption fails the pass is redone on
    the general path (compaction, exotic keys, exact side path).  ``bufs``: optional preallocated
    counts/exotic/presence tensors.  ``on_profile(profile, lo, hi)`` is called as soon as K3 of rows
    [lo, hi) has been enqueued (to start their D2H).  ``chunks`` = [(row_lo, row_hi, event)] from
    upload_chunked: the optimistic pass then counts/normalises chunk by chunk as the uploads land."""
    mode = mode_of(kmer_size)
    b = bufs or {}
    faithful = mode == KB_MODE_5P6 or mode >= 16
    sorted_k = is_sorted_mode(mode)
    if sorted_k:
        optimistic = False                              # the columns are the observed k-mers: nothing to assume
    names = [] if sorted_k else mode_column_names(mode)
    main = torch.cuda.current_stream(engine.device)
    multi = group is not None and world > 1
    cols_full = len(names)
    per = shard_bounds(n_total, world, rank)[2] if multi else None
    want_knn = n_neighbors is not None
    if chunks and not optimistic:
        for _, _, ev in chunks:
            main.wait_event(ev)
        chunks = None
    counts = None                                       # the optimistic pass never materialises the u32 count rows
    if not optimistic:
        counts = None if sorted_k else (b.get("counts") if b.get("counts") is not None else
                                        torch.empty((n, cols_full), dtype=torch.int32, device=engine.device))
    exotic = b.get("exotic") if b.get("exotic") is not None else torch.empty(n, dtype=torch.int32, device=engine.device)
    presence = b.get("presence") if b.get("presence") is not None else torch.empty(cols_full + 1, dtype=torch.int32, device=engine.device)
    presence.zero_()
    d_or = torch.zeros(1, dtype=torch.int32, device=engine.device)
    profile = operand = rowmeta = None
    if optimistic:
        # K1+K3 fused: every contig's histogram goes straight to its profile / operand / record rows
        rows = n if per is None else max(n, int(per))
        profile = torch.empty((n, cols_full), dtype=torch.float64, device=engine.device) if want_profile else None
        operand = torch.empty((rows, (cols_full + 63) // 64 * 64), dtype=torch.float16, device=engine.device) if want_knn else None
        rowmeta = torch.empty((rows, 8), dtype=torch.int32, device=engine.device)
        for lo, hi, ev in (chunks or [(0, n, None)]):
            if ev is not None:
                main.wait_event(ev)
            if hi > lo or hi == n:
                engine.count_profile(d_bases, d_offsets[:n + 1], d_key_len, lo, hi, mode, profile, operand, rowmeta, exotic,
                                     presence, d_or, rows_alloc=rowmeta.shape[0])
            if hi > lo and on_profile is not None and profile is not None:
                on_profile(profile, lo, hi)
        columns = names
    elif sorted_k:
        columns, counts = engine.build_columns_sorted(mode - 16, d_bases, d_offsets, n, group=group if multi else None)
    else:
        engine.count(d_bases, d_offsets, n, mode, counts, exotic, presence, zero_presence=False)
        if multi:
            import torch.distributed as dist
            dist.all_reduce(presence, op=dist.ReduceOp.MAX, group=group)     # one D+1 word collective
        if faithful:
            columns, counts = engine.build_columns(mode, d_bases, d_offsets, n, counts, exotic, presence,
                                                   group=group if multi else None, reduced=True)
        else:
            if int(presence[-1].item()) & 1:
                raise _lib.KarmaB200Error(-4, "dense column modes accept A/C/G/T only (some windows contain other bytes)")
            columns = names
    d_cols = len(columns)
    if d_cols == 0:
        raise ZeroRowError(row0)
    if not optimistic:
        if counts.stride(0) % 4 != 0 or counts.data_ptr() % 16 != 0:
            counts = counts.contiguous()
        profile, operand, rowmeta = engine.normalise(counts, d_cols, d_key_len, want_profile=want_profile,
                                                     want_operand=want_knn, rows_alloc=per, flags_or=d_or)
        if on_profile is not None and profile is not None:
            on_profile(profile, 0, n)
    out = {"columns": columns, "d_cols": d_cols, "counts": counts, "profile": profile, "operand": operand,
           "rowmeta": rowmeta, "idx": None, "dist": None}
    all_op, all_meta = operand, rowmeta
    if multi and not want_knn:
        # every rank must reach the same verdict on the row flags (a contig shorter than k anywhere stops them all)
        import torch.distributed as dist
        dist.all_reduce(d_or, op=dist.ReduceOp.BOR, group=group)
    if want_knn and multi:
        # the one exchange step: every rank needs all keys -- the fp16 operand shards and the 32-byte row records
        all_op = all_gather_rows(operand, group)
        all_meta = all_gather_rows(rowmeta, group)
        check(engine.lib.kb_rowmeta_flags_or(engine.ctx, ptr(all_meta), all_meta.shape[0], ptr(d_or)))   # every rank's flags
    n_real = n_total if multi else n                    # padded index == global row: real rows are [0, n_real)
    h_val = engine.host_buffer("validation", (cols_full + 4,), torch.int32, True)   # [0] flags OR, [1] uncertified rows, [3..] presence
    d_unc = None

    def fetch_validation_words():
        # Small D2H copies are issued only where the stream has nothing left to launch behind
        # them: a copy queued between K3 and K4 would sit behind the 0.4 GB profile transfer on
        # the D2H copy engine and stall the kNN kernels of this stream.
        h_val[0:1].copy_(d_or, non_blocking=True)
        if d_unc is not None:
            h_val[1:2].copy_(d_unc, non_blocking=True)
        h_val[3:].copy_(presence, non_blocking=True)
        torch.cuda.current_stream(engine.device).synchronize()

    def flags_host():
        """Per-row flags (general path only: the optimistic path reads just the OR word)."""
        return all_meta[:n_real, 3].cpu().numpy()

    if want_knn:
        flag_rows = flag_counts = None
        ids = []
        if not optimistic:
            fetch_validation_words()
            if int(h_val.numpy()[0]) & 3:                 # some row is beyond the exact range of the tensor path
                ids = np.flatnonzero((flags_host() & 3) != 0).astype(np.int32)
            if len(ids):
                # true u32 count rows of the flagged contigs, in ascending global order
                lo = rank * per if multi else 0
                mine = ids[(ids >= lo) & (ids < lo + n)] - lo
                local = counts[torch.from_numpy(mine.astype(np.int64)).to(engine.device)][:, :d_cols].contiguous() \
                    if len(mine) else torch.zeros((0, d_cols), dtype=torch.int32, device=engine.device)
                if multi:
                    fmax = max(int(((ids >= r * per) & (ids < (r + 1) * per)).sum()) for r in range(world))
                    pad = torch.zeros((fmax, d_cols), dtype=torch.int32, device=engine.device)
                    pad[:len(mine)] = local
                    allc = all_gather_rows(pad, group)
                    keep = np.concatenate([r * fmax + np.arange(int(((ids >= r * per) & (ids < (r + 1) * per)).sum()))
                                           for r in range(world)]).astype(np.int64)
                    flag_counts = allc[torch.from_numpy(keep).to(engine.device)].contiguous()
                else:
                    flag_counts = local
                flag_rows = torch.from_numpy(ids).to(engine.device)
        q_row0 = rank * per if multi else 0
        if n > 0:
            idx, dst, _, fixup = engine.knn_enqueue(all_op, all_meta, n_neighbors, q_row0=q_row0, nq=n, impl=impl,
                                                    flag_rows=flag_rows, flag_counts=flag_counts)
            impl_used = impl if impl != KB_KNN_AUTO else (_lib.KB_KNN_TC if all_op.shape[0] >= 512 else _lib.KB_KNN_SIMT)
            unc_addr = engine.uncertified_word(n, all_op.shape[0], q_row0, all_op.shape[1], n_neighbors, impl_used,
                                               0 if flag_rows is None else int(flag_rows.numel()))
            d_unc = engine.word_view(unc_addr)
        else:
            # a rank without rows (fewer contigs than ranks) still takes part in every collective
            idx = torch.empty((0, n_neighbors), dtype=torch.int32, device=engine.device)
            dst = torch.empty((0, n_neighbors), dtype=torch.float32, device=engine.device)
            d_unc = torch.zeros(1, dtype=torch.int32, device=engine.device)

            def fixup():
                return 0

        def gather_all_lists():
            # k-lists back to every rank: [idx | dist bits] packed per row, plus one row-block that carries
            # the validation words (presence, flags, uncertified rows) -- one collective
            w2 = 2 * n_neighbors
            nwords = cols_full + 3
            extra = -(-nwords // w2)
            packed = torch.empty((per + extra, w2), dtype=torch.int32, device=engine.device)
            if per > n:
                packed[n:per] = -1
            packed[:n, :n_neighbors] = idx
            packed[:n, n_neighbors:] = dst.view(torch.int32)
            tail = packed[per:].view(-1)
            tail[:cols_full + 1] = presence
            tail[cols_full + 1:cols_full + 2] = d_or
            tail[cols_full + 2:cols_full + 3] = d_unc
            g = all_gather_rows(packed, group).view(world, per + extra, w2)
            lists = g[:, :per].reshape(world * per, w2)
            out.update(all_idx=lists[:, :n_neighbors], all_dist=lists[:, n_neighbors:].view(torch.float32))
            return g[:, per:].reshape(world, -1)[:, :nwords]

        if multi and gather_lists:
            words = gather_all_lists()                               # (world, D+3)
            presence = words[:, :cols_full + 1].max(dim=0).values.contiguous()
            d_or = words[:, cols_full + 1].max().reshape(1).contiguous() | d_or
            d_unc = words[:, cols_full + 2].max().reshape(1).contiguous()
        out.update(idx=idx, dist=dst)

    # ---- validation (the only host synchronisation of an optimistic pass)
    fetch_validation_words()
    hv = h_val.numpy()
    flags_or = int(hv[0])
    if want_knn and int(hv[1]) > 0 and not (optimistic and (flags_or & 3)):
        # some row could not be certified from its candidate list: exact pass over all keys for those rows
        # (every rank takes part when the lists are shared, so that the re-gather below stays collective)
        out["uncertified"] = int(fixup())
        if multi and gather_lists:
            gather_all_lists()
    if optimistic:
        exo, complete = _presence_summary(hv[3:], faithful)
        redo = False
        if exo:
            if not faithful:
                raise _lib.KarmaB200Error(-4, "dense column modes accept A/C/G/T only (some windows contain other bytes)")
            redo = True
        if faithful and not complete:
            redo = True
        if want_knn and (flags_or & 3):
            redo = True
        if redo:
            return _device_pass(engine, d_bases, d_offsets, d_key_len, n, kmer_size, n_neighbors, impl, want_profile,
                                group, rank, world, n_total, gather_lists, bufs, on_profile, optimistic=False, row0=row0,
                                chunks=None)
    if flags_or & 4:
        # a contig shorter than k (kmer.py:250-258): report the first such row of this rank
        own = rowmeta[:n, 3].cpu().numpy()
        zero = np.flatnonzero(own & 4)
        if len(zero):
            raise ZeroRowError(int(zero[0]) + row0)
        if multi:
            raise ZeroRowError(-1)                       # the all-zero row lives on another rank
    return out


def profile_and_knn(engine, bases, offsets, key_len, kmer_size="5p6", n_neighbors=None,
                    impl=KB_KNN_AUTO, want_profile=True, group=None, rank=0, world=1, row0=0, n_total=None,
                    reuse_host=False, on_knn=None, host_profile=True):
    """Run the hot path on host buffers (what KmerClustering and bench.py's e2e leg call).

    bases/offsets/key_len describe THIS rank's contigs (all of them when world==1).
    Returns dict(columns, profile (n,D') float64 ndarray or None, knn_idx, knn_dist)
    where the kNN rows are this rank's contigs against ALL contigs (global indices).
    Raises ZeroRowError when a contig is shorter than k (kmer.py:250-258).

    The float64 profile (the largest transfer of the path: 8*D' bytes per contig) goes
    back to pinned host memory on a side stream while the kNN kernels run.  With
    ``reuse_host`` the pinned result buffers are owned by the engine and overwritten
    by the next call (a serving loop); otherwise every call returns fresh arrays.
    ``on_knn(idx, dist)`` is called as soon as the k-lists are on the host, before the profile download has
    finished (50k contigs, 5p6: about 4 ms against 8 ms for the whole call).

    ``host_profile=False`` keeps the profile on the device for device consumers (``cluster.cluster_from_lists``):
    the download is skipped, ``profile`` is None, and ``d_profile`` (float64 [n, D']) with ``d_idx`` (int32 [n, k])
    and ``d_dist`` (float32 [n, k]) are device tensors.  The k-lists are still copied to ``knn_idx`` / ``knn_dist``.
    """
    n = len(offsets) - 1
    main = torch.cuda.current_stream(engine.device)
    side = engine.side_stream()
    chunks = None
    if n >= 4096:
        # H2D in row chunks: counting and the (opposite-direction) profile download start early
        d_bases, d_offsets, d_key_len, chunks = engine.upload_chunked(bases, offsets, key_len, 4)
    else:
        d_bases, d_offsets, d_key_len = engine.upload(bases, offsets, key_len)
    hold = {}

    def start_download(profile, lo, hi):
        # D2H of profile rows [lo, hi) on the side stream, ordered after their K3, overlapping
        # the remaining uploads and the kNN
        h = hold.get("profile")
        if h is None or tuple(h.shape) != tuple(profile.shape):
            h = engine.host_buffer("profile", tuple(profile.shape), torch.float64, reuse_host)
            hold["profile"] = h
        ready = torch.cuda.Event()
        ready.record(main)
        side.wait_event(ready)
        with torch.cuda.stream(side):
            h[lo:hi].copy_(profile[lo:hi], non_blocking=True)
        profile.record_stream(side)

    r = device_pass(engine, d_bases, d_offsets, d_key_len, n, kmer_size, n_neighbors=n_neighbors, impl=impl,
                    want_profile=want_profile, group=group, rank=rank, world=world, n_total=n_total,
                    on_profile=start_download if want_profile and host_profile else None, row0=row0, chunks=chunks)
    out = {"columns": r["columns"], "profile": None, "knn_idx": None, "knn_dist": None,
           "d_profile": r["profile"], "d_operand": r["operand"], "uncertified": r.get("uncertified", 0)}
    if not host_profile:
        out.update(d_idx=r["idx"], d_dist=r["dist"])
    if n_neighbors is not None:
        h_idx = engine.host_buffer("knn_idx", tuple(r["idx"].shape), torch.int32, reuse_host)
        h_dst = engine.host_buffer("knn_dist", tuple(r["dist"].shape), torch.float32, reuse_host)
        h_idx.copy_(r["idx"], non_blocking=True)
        h_dst.copy_(r["dist"], non_blocking=True)
        main.synchronize()
        out["knn_idx"] = h_idx.numpy()
        out["knn_dist"] = h_dst.numpy()
        if on_knn is not None:
            # the k-lists are on the host now; the float64 profile (8*D' bytes per contig over PCIe) is still in flight
            on_knn(out["knn_idx"], out["knn_dist"])
    if want_profile and host_profile:
        side.synchronize()
        out["profile"] = hold["profile"].numpy()
    return out


# ---------------------------------------------------------------------------------------
# the pre-planned pass: static buffers, one enqueue, CUDA graph, peer-memory exchange
# ---------------------------------------------------------------------------------------

class _KnnXchg(ctypes.Structure):
    """kb_knn_xchg of include/karma_b200.h"""
    _fields_ = [("d_arrive", c_void_p), ("d_epoch", c_void_p), ("rows_per_src", c_int64), ("n_peers", ctypes.c_int32),
                ("self_rank", ctypes.c_int32), ("d_peer_idx", c_void_p), ("d_peer_dist", c_void_p)]


class _RawDevice:
    """__cuda_array_interface__ view of raw device memory (the exchange arena is allocated by the library)."""

    def __init__(self, addr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(addr), False), "version": 2}


def _round_up(x, m):
    return (x + m - 1) // m * m


def host_chunks(offsets, chunks):
    """Row chunks of about equal bases for the host-to-host pass: [(row_lo, row_hi, byte_lo, byte_hi)], covering every
    row once, in order; at most ``chunks`` of them and none for fewer than ~1024 rows each."""
    on = np.asarray(offsets, dtype=np.int64)
    n = len(on) - 1
    total = int(on[-1])
    c = max(1, min(int(chunks), n // 1024 if n >= 2048 else 1))
    cuts = [0] + [int(np.searchsorted(on, total * i / c)) for i in range(1, c)] + [n]
    cuts = sorted(set(min(max(x, 0), n) for x in cuts))
    if len(cuts) == 1:
        cuts = [0, n]
    return [(lo, hi, int(on[lo]), int(on[hi])) for lo, hi in zip(cuts[:-1], cuts[1:])]


class PassPlan:
    """The optimistic hot path (K1 -> K3 -> exchange -> K4 -> K5) of `_device_pass`, planned once for a shape and
    then re-run with ONE enqueue: every buffer is static, nothing is allocated and nothing synchronises inside
    a pass, so the pass can be (and by default is) captured in a CUDA graph.

    Multi-GPU (one process per GPU): the exchange runs over peer memory (kb_xchg_*, NVLink): after K3 the operand
    and row-record shards are pushed into every peer's arena on a side stream while K4 already sweeps the local
    shard (its TMA producer waits for the arrival flag of a shard before its first key tile); K5 stores the
    k-lists into every peer's gathered result arrays.  No NCCL call is on the path; `group` is used once, to
    hand the IPC handles round.

    A pass is validated afterwards from a few words per rank (flags OR, uncertified rows, presence summary):
    `run()` enqueues pass i and returns a token; `check(token)` waits for that pass only -- call it after the
    next `run()` to keep the GPU busy.  If the optimistic assumptions fail (non-ACGT bytes, a missing column, a
    row beyond the exact range of the tensor path) `check` returns False and the caller redoes the input with
    `device_pass(..., optimistic=False)`; rows K5 could not certify are redone in place (exact pass)."""

    def __init__(self, engine, n, total_bases, kmer_size="5p6", n_neighbors=None, impl=_lib.KB_KNN_TC,
                 want_profile=True, group=None, rank=0, world=1, n_total=None, graph=True):
        self.engine = engine
        self.lib = engine.lib
        dev = engine.device
        self.n, self.k, self.world, self.rank, self.group = int(n), n_neighbors, int(world), int(rank), group
        self.multi = group is not None and world > 1
        self.n_total = int(n_total) if self.multi else self.n
        self.mode = mode_of(kmer_size)
        if is_sorted_mode(self.mode):
            raise _lib.KarmaB200Error(-4, "PassPlan serves the fixed-column modes (k <= 7, 5p6, 5+6, 4+5); integer k >= 8 has "
                                      "data-dependent columns: use device_pass / profile_and_knn")
        self.kmer_size = kmer_size
        self.faithful = self.mode == KB_MODE_5P6 or self.mode >= 16
        self.cols = check(self.lib.kb_mode_columns(self.mode))
        self.dp = _round_up(self.cols, 64)
        self.per = shard_bounds(self.n_total, self.world, self.rank)[2] if self.multi else self.n
        self.q_row0 = self.rank * self.per if self.multi else 0
        self.nk = self.per * self.world if self.multi else self.n
        self.impl = impl if impl != KB_KNN_AUTO else (_lib.KB_KNN_TC if self.nk >= 512 else _lib.KB_KNN_SIMT)
        self.want_knn = n_neighbors is not None
        k = self.k or 1
        # inputs
        cap = _round_up(int(total_bases), 16) + 32
        self.d_bases = torch.zeros(cap, dtype=torch.uint8, device=dev)
        self.d_offsets = torch.zeros(self.n + 1, dtype=torch.int64, device=dev)
        self.d_key_len = torch.ones(max(self.n, 1), dtype=torch.int32, device=dev)
        # K1 / K3 products (the u32 count rows are never materialised: kb_count_profile)
        self.exotic = torch.empty(max(self.n, 1), dtype=torch.int32, device=dev)
        self.rec_words = self.cols + 1 + 4                      # per-rank record: [flags OR, uncertified rows, 0, 0, presence[0..D]]
        self.profile = torch.empty((self.n, self.cols), dtype=torch.float64, device=dev) if want_profile else None
        self.x = None
        self.side = None
        if self.multi and self.want_knn:
            self._setup_exchange(k)
        else:
            self.operand_all = torch.empty((self.nk, self.dp), dtype=torch.float16, device=dev) if self.want_knn else None
            self.rowmeta_all = torch.empty((self.nk, 8), dtype=torch.int32, device=dev)
            self.all_idx = torch.empty((self.nk, k), dtype=torch.int32, device=dev) if self.want_knn else None
            self.all_dist = torch.empty((self.nk, k), dtype=torch.float32, device=dev) if self.want_knn else None
            self.rec_all = torch.zeros((1, self.rec_words), dtype=torch.int32, device=dev)
        self.idx = self.all_idx[self.q_row0:self.q_row0 + self.n] if self.want_knn else None
        self.dist = self.all_dist[self.q_row0:self.q_row0 + self.n] if self.want_knn else None
        self.rec = self.rec_all[self.rank if self.x is not None else 0]
        self.presence = self.rec[4:]                             # K1/K3 write the presence vector straight into the record
        self.ws = None
        self._unc = None
        if self.want_knn:
            need = check(self.lib.kb_knn_workspace_bytes(engine.ctx, self.n, self.nk, self.q_row0, self.dp, self.k, self.impl, 0))
            self.ws = torch.empty(need, dtype=torch.uint8, device=dev)
            out = c_void_p()
            check(self.lib.kb_knn_uncertified_ptr(engine.ctx, self.n, self.nk, self.q_row0, self.dp, self.k, self.impl, 0,
                                                  ptr(self.ws), byref(out)))
            off = out.value - self.ws.data_ptr()
            self._unc = self.ws[off:off + 4].view(torch.int32)
        self.h_val = [torch.zeros(tuple(self.rec_all.shape), dtype=torch.int32).pin_memory() for _ in range(2)]
        self._events = [torch.cuda.Event(), torch.cuda.Event()]
        self._step = 0
        self.graph = None
        self._want_graph = bool(graph)
        self._io = None                                         # host-to-host pass (bind_host / run_host)
        self._marks = None                                      # diagnostics: [(name, event)] filled by an eager enqueue
        self.host = None

    # ---- exchange set-up (once) -----------------------------------------------------------
    def _setup_exchange(self, k):
        import torch.distributed as dist
        dev = self.engine.device
        W, per, dp = self.world, self.per, self.dp
        off = 1024
        lay = {}
        for name, nbytes in (("operand", W * per * dp * 2), ("rowmeta", W * per * 32), ("idx", W * per * k * 4),
                             ("dist", W * per * k * 4), ("rec", W * self.rec_words * 4)):
            lay[name] = off
            off = _round_up(off + nbytes, 256)
        self._lay, total = lay, off
        x, local = c_void_p(), c_void_p()
        handle = (ctypes.c_uint8 * 64)()
        rc = self.lib.kb_xchg_create(self.engine.ctx, W, self.rank, total, byref(x), byref(local), handle)
        mine = bytes(handle) if rc == 0 else None
        err = None if rc == 0 else self.lib.kb_last_error().decode("utf-8", "replace")
        got = [None] * W
        dist.all_gather_object(got, (mine, err), group=self.group)
        if any(h is None for h, _ in got):
            raise _lib.KarmaB200Error(-2, "peer-memory arena could not be created on every rank: %r" % ([e for _, e in got],))
        rc = self.lib.kb_xchg_attach(x, b"".join(h for h, _ in got))
        err = None if rc == 0 else self.lib.kb_last_error().decode("utf-8", "replace")
        got = [None] * W
        dist.all_gather_object(got, err, group=self.group)
        if any(e is not None for e in got):
            raise _lib.KarmaB200Error(-2, "peer-memory arenas could not be mapped on every rank: %r" % (got,))
        self.x = x
        base = local.value
        arena = torch.as_tensor(_RawDevice(base, total), device=dev)
        self._arena = arena

        def view(name, nbytes, dtype, shape):
            return arena[lay[name]:lay[name] + nbytes].view(dtype).view(shape)
        self.operand_all = view("operand", W * per * dp * 2, torch.float16, (W * per, dp))
        self.rowmeta_all = view("rowmeta", W * per * 32, torch.int32, (W * per, 8))
        self.all_idx = view("idx", W * per * k * 4, torch.int32, (W * per, k))
        self.all_dist = view("dist", W * per * k * 4, torch.float32, (W * per, k))
        self.rec_all = view("rec", W * self.rec_words * 4, torch.int32, (W, self.rec_words))
        self.rec_all.zero_()
        # peers' gathered result arrays as seen from here (K5 stores its rows there)
        pi, pd = [], []
        for p in range(W):
            if p == self.rank:
                continue
            pp = c_void_p()
            check(self.lib.kb_xchg_peer_ptr(x, p, byref(pp)))
            pi.append(pp.value + lay["idx"])
            pd.append(pp.value + lay["dist"])
        self._peer_idx = torch.tensor(pi, dtype=torch.int64, device=dev)
        self._peer_dist = torch.tensor(pd, dtype=torch.int64, device=dev)
        arrive, epoch = c_void_p(), c_void_p()
        check(self.lib.kb_xchg_flags(x, byref(arrive), byref(epoch)))
        self._xchg = _KnnXchg(arrive.value, epoch.value, per, W - 1, self.rank, self._peer_idx.data_ptr(), self._peer_dist.data_ptr())
        self._regions = ((ctypes.c_int64 * 2)(lay["operand"], lay["rowmeta"]), (ctypes.c_int64 * 2)(per * dp * 2, per * 32))
        self.side = torch.cuda.Stream(dev)
        # first touch of the peers' arenas (sets up the peer mappings) before any pass waits for data
        self.engine._bind_stream()
        lists = (ctypes.c_int64 * 4)(lay["operand"], lay["rowmeta"], lay["idx"], lay["dist"])
        sizes = (ctypes.c_int64 * 4)(per * dp * 2, per * 32, per * k * 4, per * k * 4)
        check(self.lib.kb_xchg_warm(x, 4, lists, sizes))
        torch.cuda.synchronize(dev)
        dist.barrier(group=self.group)

    def close(self):
        if self.x is not None:
            torch.cuda.synchronize(self.engine.device)
            self.graph = None
            if self._io is not None:
                self._io["graph"] = None
            self.lib.kb_xchg_destroy(self.x)
            self.x = None

    # ---- inputs ---------------------------------------------------------------------------
    def load(self, bases, offsets, key_len):
        """Copy this rank's contigs (host or device tensors / arrays) into the plan's input buffers."""
        def t(a, dtype):
            return a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=dtype))
        o = t(offsets, np.int64)
        total = int(o[-1])
        if o.numel() != self.n + 1 or _round_up(total, 16) + 32 > self.d_bases.numel():
            raise ValueError("PassPlan was planned for %d contigs / %d bases" % (self.n, self.d_bases.numel() - 32))
        self.d_bases[:total].copy_(t(bases, np.uint8)[:total], non_blocking=True)
        self.d_offsets.copy_(o, non_blocking=True)
        if self.n:
            self.d_key_len.copy_(t(key_len, np.int32), non_blocking=True)

    # ---- one pass ---------------------------------------------------------------------------
    def enqueue(self, host_io=False):
        """K1 -> K3 -> [push] -> K4 -> K5 -> [finish] on the current stream.  No allocation, no synchronisation.
        ``host_io`` (after `bind_host`): the pass starts from the pinned host inputs and ends with the float64
        profile rows, this rank's k-lists and the validation words in pinned host memory -- the bases go up in row
        chunks on a copy stream, every chunk is counted as it lands and its profile rows start their download on a
        second copy stream (the other DMA direction) while the remaining uploads, the exchange and the kNN run."""
        e, lib = self.engine, self.lib
        e._bind_stream()
        main = torch.cuda.current_stream(e.device)
        io = self._io if host_io else None
        marks = self._marks

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(main)
                marks.append((name, ev))
        mark("start")
        if io is not None:
            fork = torch.cuda.Event()
            fork.record(main)
            io["up"].wait_event(fork)
            io["down"].wait_event(fork)
            landed = []
            with torch.cuda.stream(io["up"]):
                self.d_offsets.copy_(io["h_offsets"], non_blocking=True)
                if self.n:
                    self.d_key_len.copy_(io["h_key_len"], non_blocking=True)
                for (lo, hi, b0, b1) in io["chunks"]:
                    if b1 > b0:
                        self.d_bases[b0:b1].copy_(io["h_bases"][b0:b1], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(io["up"])
                    landed.append(ev)
        if self.x is not None:
            check(lib.kb_xchg_begin(self.x))
        self.rec.zero_()                                        # flags, uncertified rows and the presence vector
        mark("begin")
        n_alloc = self.per if self.x is not None else self.n
        q0 = self.q_row0
        # K1+K3 fused: the histogram of every contig goes straight to its profile / operand / record rows
        for c, (lo, hi, _, _) in enumerate(io["chunks"] if io is not None else [(0, self.n, 0, 0)]):
            if io is not None:
                main.wait_event(landed[c])
            rows_out = (n_alloc if hi == self.n else hi) - lo   # the last chunk also writes the gather padding rows
            if rows_out > 0:
                check(lib.kb_count_profile(e.ctx, self.mode, ptr(self.d_bases), ptr(self.d_offsets[lo:]),
                                           ptr(self.d_key_len[lo:]) if hi > lo else None, hi - lo, rows_out,
                                           ptr(self.profile[lo:]) if self.profile is not None and hi > lo else None, self.cols,
                                           ptr(self.operand_all[q0 + lo:]) if self.want_knn else None, self.dp,
                                           ptr(self.rowmeta_all[q0 + lo:]), ptr(self.exotic[lo:]) if hi > lo else None,
                                           ptr(self.presence), ptr(self.rec)))
            if io is not None and self.profile is not None and hi > lo:
                ev = torch.cuda.Event()
                ev.record(main)
                io["down"].wait_event(ev)
                with torch.cuda.stream(io["down"]):
                    io["h_profile"][lo:hi].copy_(self.profile[lo:hi], non_blocking=True)
        mark("count")
        if self.x is not None:
            ev = torch.cuda.Event()
            ev.record(main)
            self.side.wait_event(ev)
            check(lib.kb_xchg_push(self.x, c_void_p(self.side.cuda_stream), 2, self._regions[0], self._regions[1]))
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(self.side)
                marks.append(("push_done(side)", ev))
        if self.want_knn and self.n:
            check(lib.kb_knn(e.ctx, self.impl, self.k, ptr(self.operand_all), self.dp, self.dp, ptr(self.rowmeta_all),
                             self.nk, self.q_row0, self.n, None, None, 0, 0, 0, ptr(self.idx), ptr(self.dist), None,
                             ptr(self.ws), self.ws.numel(), byref(self._xchg) if self.x is not None else None))
            self.rec[1:2].copy_(self._unc, non_blocking=True)
        mark("knn")
        if self.x is not None:
            check(lib.kb_xchg_finish(self.x, self._lay["rec"], self.rec_words))
            mark("finish")
            main.wait_stream(self.side)
        mark("end")
        if io is not None:
            # small results last: they queue behind the profile rows on the D2H copy engine and must not hold back K4
            if self.want_knn and self.n:
                io["h_idx"].copy_(self.idx, non_blocking=True)
                io["h_dist"].copy_(self.dist, non_blocking=True)
            io["h_rec"].copy_(self.rec_all, non_blocking=True)
            main.wait_stream(io["up"])
            main.wait_stream(io["down"])

    # ---- host-to-host passes ----------------------------------------------------------------
    def bind_host(self, bases, offsets, key_len, chunks=4):
        """Stage this rank's contigs (host arrays / tensors) in the plan's pinned input buffers and plan the
        host-to-host pass for them: row chunks of about equal bases.  The pinned buffers (``plan.host["h_bases"]``,
        ``["h_offsets"]``, ``["h_key_len"]``) may afterwards be rewritten in place with other contigs of the SAME
        offsets; a different set of contig lengths needs another `bind_host` (the chunk bounds are part of the
        captured graph).  Results of `run_host` land in ``plan.host["h_profile" | "h_idx" | "h_dist"]``."""
        dev = self.engine.device

        def t(a, dtype):
            return a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=dtype))
        o = t(offsets, np.int64)
        total = int(o[-1])
        if o.numel() != self.n + 1 or _round_up(total, 16) + 32 > self.d_bases.numel():
            raise ValueError("PassPlan was planned for %d contigs / %d bases" % (self.n, self.d_bases.numel() - 32))
        io = self._io
        if io is None:
            k = self.k or 1
            io = {"up": torch.cuda.Stream(dev), "down": torch.cuda.Stream(dev),
                  "h_bases": torch.zeros(self.d_bases.numel(), dtype=torch.uint8, pin_memory=True),
                  "h_offsets": torch.zeros(self.n + 1, dtype=torch.int64, pin_memory=True),
                  "h_key_len": torch.ones(max(self.n, 1), dtype=torch.int32, pin_memory=True),
                  "h_profile": torch.empty((self.n, self.cols), dtype=torch.float64, pin_memory=True) if self.profile is not None else None,
                  "h_idx": torch.empty((self.n, k), dtype=torch.int32, pin_memory=True) if self.want_knn else None,
                  "h_dist": torch.empty((self.n, k), dtype=torch.float32, pin_memory=True) if self.want_knn else None,
                  "h_rec": torch.zeros(tuple(self.rec_all.shape), dtype=torch.int32, pin_memory=True),
                  "done": torch.cuda.Event(), "chunks": None, "graph": None}
            self._io = io
            self.host = io
        hb = t(bases, np.uint8)
        if hb.data_ptr() != io["h_bases"].data_ptr():
            io["h_bases"][:total].copy_(hb[:total])
        if o.data_ptr() != io["h_offsets"].data_ptr():
            io["h_offsets"].copy_(o)
        if self.n and t(key_len, np.int32).data_ptr() != io["h_key_len"].data_ptr():
            io["h_key_len"].copy_(t(key_len, np.int32))
        plan = host_chunks(io["h_offsets"].numpy(), chunks)
        if plan != io["chunks"]:
            io["chunks"] = plan
            io["graph"] = None

    def run_host(self):
        """One host-to-host pass over the bound inputs (one graph replay when the plan is graph-captured), waited
        for and validated.  Returns dict(ok, flags_or, uncertified, exotic, complete, profile, knn_idx, knn_dist):
        numpy views of the plan's pinned result buffers, overwritten by the next call.  Every rank calls it at
        the same point."""
        io = self._io
        e = self.engine
        if self._want_graph and io["graph"] is None:
            timing = e.timing_enabled
            e.enable_timing(False)
            self.enqueue(host_io=True)
            torch.cuda.synchronize(e.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.enqueue(host_io=True)
            io["graph"] = g
            e._bind_stream()
            torch.cuda.synchronize(e.device)
            e.enable_timing(timing)
            if self.multi:
                import torch.distributed as dist
                dist.barrier(group=self.group)
        if io["graph"] is not None:
            io["graph"].replay()
        else:
            self.enqueue(host_io=True)
        io["done"].record(torch.cuda.current_stream(e.device))
        io["done"].synchronize()
        out = self._verdict(io["h_rec"].numpy())
        out["profile"] = io["h_profile"].numpy() if io["h_profile"] is not None else None
        out["knn_idx"] = io["h_idx"].numpy() if io["h_idx"] is not None else None
        out["knn_dist"] = io["h_dist"].numpy() if io["h_dist"] is not None else None
        return out

    def capture(self, warmup=2):
        """Warm up eagerly (uploads the K4 piece table, sizes scratch buffers), then capture the pass in a CUDA
        graph.  Every rank must call this at the same point."""
        e = self.engine
        timing = e.timing_enabled
        e.enable_timing(False)
        for _ in range(warmup):
            self.enqueue()
        torch.cuda.synchronize(e.device)
        if self._want_graph:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.enqueue()
            self.graph = g
            e._bind_stream()
        torch.cuda.synchronize(e.device)
        e.enable_timing(timing)

    def run(self):
        """Enqueue one pass (graph replay when captured) plus the copy of the validation words; returns a token."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self.enqueue()
        slot = self._step & 1
        self.h_val[slot].copy_(self.rec_all, non_blocking=True)
        self._events[slot].record(torch.cuda.current_stream(self.engine.device))
        self._step += 1
        return self._step - 1

    def check(self, token):
        """Wait for pass `token` (the latest or the one before) and read its validation words.
        Returns dict(ok, flags_or, uncertified, exotic, complete)."""
        if token < self._step - 2:
            raise ValueError("the validation words of that pass have been overwritten")
        slot = token & 1
        self._events[slot].synchronize()
        return self._verdict(self.h_val[slot].numpy())

    def _verdict(self, v):
        flags_or = int(np.bitwise_or.reduce(v[:, 0]))
        unc = int(v[:, 1].sum())
        pres = np.bitwise_or.reduce(v[:, 4:], axis=0)            # OR over the ranks: column words, [D] = exotic | complete bits
        exo, complete = _presence_summary(pres, self.faithful)
        ok = not exo and (complete or not self.faithful) and not (self.want_knn and (flags_or & 3)) and not (flags_or & 4)
        return {"ok": ok, "flags_or": flags_or, "uncertified": unc, "exotic": exo, "complete": complete}

    def fixup(self):
        """Exact pass over the rows K5 could not certify (all ranks call it when any rank has such rows);
        the patched rows are shared again.  Synchronises."""
        e = self.engine
        e._bind_stream()
        n = check(self.lib.kb_knn_fixup(e.ctx, self.impl, self.k, ptr(self.operand_all), self.dp, self.dp, ptr(self.rowmeta_all),
                                        self.nk, self.q_row0, self.n, None, None, 0, 0, 0, ptr(self.idx), ptr(self.dist), None,
                                        ptr(self.ws), self.ws.numel()))
        if self.multi:
            import torch.distributed as dist
            for t in (self.all_idx, self.all_dist):
                shard = t[self.q_row0:self.q_row0 + self.per].clone()
                dist.all_gather_into_tensor(t, shard, group=self.group)
        return int(n)

    def columns(self):
        return mode_column_names(self.mode)
