"""ctypes binding of the C ABI (include/ugrep_b200.h) — the call a Python user makes.

The host-side mirror of the reference interface: ``Pattern`` stands for a compiled
``reflex::Pattern`` (opcode words + prefilter fields), ``Scanner`` for one
``reflex::Matcher`` bound to a device stream; ``count_lines`` / ``count_matches`` /
``find_all`` are the three ``Grep::search`` loops of the configs
(/root/reference/src/ugrep.cpp:10567-10586, :10536-10566, :10857-11047).

There is no CPU fallback: if ``libugrep_b200.so`` is missing or no CUDA device is
usable, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UGX_LIB") or os.path.join(HERE, "libugrep_b200.so")  # UGX_LIB: A/B builds (tools/variants.py)

MATCH_DTYPE = np.dtype([("line", "<u8"), ("offset", "<u8"), ("len", "<u4"), ("cap", "<u4")])
# ugx_line: one record per line (find_lines): line number, the line's [bol, eol), its first match (offset, len, cap)
LINE_DTYPE = np.dtype([("line", "<u8"), ("bol", "<u8"), ("eol", "<u8"), ("offset", "<u8"), ("len", "<u4"), ("cap", "<u4")])
LINES_INVERT = 1

ADVANCE_NAMES = ["none", "pin1_one", "pin1_pma", "pin1_pmh", "pin_one", "pin_pma", "pin_pmh", "min1", "min2", "min3",
                 "min4", "pma", "char", "char_pma", "char_pmh", "string", "string_pma", "string_pmh"]

EXPORTS = ["ugx_last_error", "ugx_kernel_name", "ugx_plan_describe", "ugx_abi_version", "ugx_pattern_create", "ugx_pattern_load", "ugx_pattern_info_get",
           "ugx_pattern_destroy", "ugx_scanner_create", "ugx_scanner_destroy", "ugx_count_lines", "ugx_count_matches",
           "ugx_viability_describe", "ugx_search_describe", "ugx_check_text", "ugx_compile_literal", "ugx_compile_words", "ugx_compile_words_ex", "ugx_compile_plain_regex", "ugx_count_batch", "ugx_sharded_create", "ugx_sharded_destroy", "ugx_sharded_set_option", "ugx_sharded_scan", "ugx_sharded_last_error", "ugx_find_all", "ugx_find_all_device", "ugx_scanner_fetch", "ugx_scanner_set_option", "ugx_count_newlines",
           "ugx_find_lines", "ugx_find_lines_device", "ugx_scanner_fetch_lines", "ugx_sharded_find_lines",
           "ugx_find_all_batch", "ugx_find_lines_batch", "ugx_find_context", "ugx_find_context_device",
           "ugx_find_context_batch", "ugx_count_lines_bool", "ugx_find_lines_bool", "ugx_find_lines_bool_device",
           "ugx_count_lines_bool_batch", "ugx_find_lines_bool_batch"]


class UgxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("ugx error %d: %s" % (code, msg))
        self.code = code


class _Totals(C.Structure):
    _fields_ = [("matches", C.c_uint64), ("newlines", C.c_uint64), ("flags", C.c_uint64),
                ("kernel_ms", C.c_float), ("launches", C.c_uint32), ("kernel", C.c_uint32)]


class BoolClause(C.Structure):
    """ugx_bool_clause: the clause holds on a line on which a pattern of `pos` has a match or one of `neg` has none"""
    _fields_ = [("pos", C.c_uint32), ("neg", C.c_uint32)]


BOOL_MAX_PATTERNS = 32


def bool_clauses(cnf):
    """The ugx_bool_clause array of a CNF written as a list of clauses, each a list of ints: j = pattern j has a match
    on the line, ~j = pattern j has none.  `-e A --and -e B` is [[0], [1]], `A --andnot B` is [[0], [~1]], `--bool
    'A|B -C'` is [[0, 1], [~2]].  Malformed input (not a list of non-empty lists of ints in [-32, 31]) raises
    ValueError; whether a pattern index exists is checked by the library against its pattern count."""
    if not isinstance(cnf, (list, tuple)):
        raise ValueError("a CNF is a list of clauses")
    out = (BoolClause * len(cnf))()
    for c, clause in enumerate(cnf):
        if not isinstance(clause, (list, tuple)) or len(clause) == 0:
            raise ValueError("clause %d: a clause is a non-empty list of ints" % c)
        for t in clause:
            if isinstance(t, bool) or not isinstance(t, (int, np.integer)):
                raise ValueError("clause %d: %r is not an int" % (c, t))
            t = int(t)
            if not -BOOL_MAX_PATTERNS <= t < BOOL_MAX_PATTERNS:
                raise ValueError("clause %d: %d names no pattern (0..31, or ~0..~31)" % (c, t))
            if t >= 0:
                out[c].pos |= 1 << t
            else:
                out[c].neg |= 1 << ~t
    return out


class _TextInfo(C.Structure):
    _fields_ = [("is_utf8", C.c_uint32), ("has_nul", C.c_uint32), ("kernel_ms", C.c_float), ("launches", C.c_uint32)]


class _Info(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("nop", "states", "classes", "table_bytes", "table_in_smem", "advance",
                                          "has_meta", "lookback")]


@dataclass
class Totals:
    matches: int
    newlines: int
    flags: int
    kernel_ms: float
    launches: int
    kernel: str = "none"


_lib = None


def lib():
    """Load the CUDA library; raises if it has not been built (python -m ugrep_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise UgxError(-1, "%s is missing: build it with `python -m ugrep_b200.build` (CUDA only, no CPU fallback)"
                           % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.ugx_last_error.restype = C.c_char_p
        L.ugx_kernel_name.restype = C.c_char_p
        L.ugx_kernel_name.argtypes = [C.c_uint32]
        L.ugx_pattern_create.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.ugx_pattern_load.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
        L.ugx_pattern_info_get.argtypes = [C.c_void_p, C.POINTER(_Info)]
        L.ugx_pattern_destroy.argtypes = [C.c_void_p]
        L.ugx_pattern_destroy.restype = None
        L.ugx_scanner_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.ugx_scanner_destroy.argtypes = [C.c_void_p]
        L.ugx_scanner_destroy.restype = None
        L.ugx_count_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(_Totals)]
        L.ugx_count_matches.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(_Totals)]
        L.ugx_count_newlines.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(_Totals)]
        L.ugx_find_all.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                   C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_find_all_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_scanner_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.ugx_scanner_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]
        L.ugx_find_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32,
                                     C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_find_lines_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                            C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_scanner_fetch_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]
        L.ugx_find_all_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                         C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64),
                                         C.POINTER(_Totals)]
        L.ugx_find_lines_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                           C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                           C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_find_context.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                       C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64,
                                       C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_find_context_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64,
                                              C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_find_context_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                             C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                             C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        bool_args = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]
        L.ugx_count_lines_bool.argtypes = bool_args + [C.c_uint32, C.POINTER(_Totals)]
        L.ugx_find_lines_bool_device.argtypes = bool_args + [C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(C.c_void_p),
                                                             C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        L.ugx_find_lines_bool.argtypes = bool_args + [C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64,
                                                      C.POINTER(C.c_uint64), C.POINTER(_Totals)]
        bool_batch = bool_args + [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]
        L.ugx_count_lines_bool_batch.argtypes = bool_batch + [C.c_void_p, C.POINTER(_Totals)]
        L.ugx_find_lines_bool_batch.argtypes = bool_batch + [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64),
                                                             C.POINTER(_Totals)]
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise UgxError(rc, lib().ugx_last_error().decode("utf-8", "replace"))


def _buffer(data):
    """(pointer, nbytes, keepalive) for a CUDA tensor, numpy array or bytes-like."""
    if hasattr(data, "data_ptr") and hasattr(data, "is_cuda"):
        if data.dtype.itemsize != 1:
            raise TypeError("expected a uint8/int8 tensor")
        if not data.is_contiguous():
            data = data.contiguous()
        return data.data_ptr(), data.numel(), data
    if isinstance(data, (bytes, bytearray, memoryview)):
        a = np.frombuffer(data, dtype=np.uint8)
    else:
        a = np.ascontiguousarray(data, dtype=np.uint8)
    return a.ctypes.data, a.size, a


def _pack_files(files):
    """(buffer, begins, lens) of the batch entry points: the files (bytes-like) back to back on 16-byte boundaries in
    one host buffer, as a batching feeder would pack them; the padding between files is 'X'."""
    begins = np.zeros(len(files), dtype=np.uint64)
    lens = np.array([len(f) for f in files], dtype=np.uint64)
    at = 0
    for i, f in enumerate(files):
        begins[i] = at
        at = (at + len(f) + 15) & ~15
    pack = np.full(max(at, 16), 0x58, dtype=np.uint8)
    for i, f in enumerate(files):
        pack[int(begins[i]):int(begins[i]) + len(f)] = np.frombuffer(bytes(f), dtype=np.uint8)
    return pack, begins, lens


def _batch_input(files):
    """(pointer, nbytes, keepalive, begins, lens) of a batch: a list of bytes-like packed by _pack_files, or an already
    packed (buffer, begins, lens) with the buffer as _buffer takes it"""
    if isinstance(files, tuple):
        data, begins, lens = files
        begins = np.ascontiguousarray(begins, dtype=np.uint64)
        lens = np.ascontiguousarray(lens, dtype=np.uint64)
    else:
        data, begins, lens = _pack_files(files)
    ptr, n, keep = _buffer(data)
    return C.c_void_p(ptr), n, keep, begins, lens


PREFILTER_BYTES = 12 * 4 + 256 + 256 + 2048 + 4096 + 4096 + 32 + 32 + 256


def compile_literal(text: bytes):
    """(opcode words, ugx_prefilter bytes) of one fixed string, as the reference's compiler would produce them"""
    L = lib()
    L.ugx_compile_literal.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p]
    opc = np.zeros(2 * (len(text) + 1) + 2, dtype=np.uint32)
    nop = C.c_uint32()
    pf = C.create_string_buffer(PREFILTER_BYTES)
    rc = L.ugx_compile_literal(bytes(text), len(text), opc.ctypes.data, len(opc), C.byref(nop), pf)
    if rc != 0:
        raise UgxError(rc, "ugx_compile_literal: literal outside its scope" if rc == 2 else "ugx_compile_literal failed")
    return opc[:nop.value].copy(), pf.raw


def compile_words(words, icase: bool = False):
    """(opcode words, ugx_prefilter bytes) of a list of fixed strings (`ugrep -F [-i] -f FILE`), as the reference's
    compiler would produce them; UgxError code 2 when the list is outside the restated part of the compiler"""
    L = lib()
    L.ugx_compile_words_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32,
                                       C.POINTER(C.c_uint32), C.c_void_p]
    ws = [bytes(w) for w in words]
    ptrs = (C.c_char_p * len(ws))(*ws)
    lens = (C.c_uint32 * len(ws))(*[len(w) for w in ws])
    cap = 4 * sum(len(w) + 2 for w in ws) + 16
    opc = np.zeros(cap, dtype=np.uint32)
    nop = C.c_uint32()
    pf = C.create_string_buffer(PREFILTER_BYTES)
    rc = L.ugx_compile_words_ex(ptrs, lens, len(ws), 1 if icase else 0, opc.ctypes.data, cap, C.byref(nop), pf)
    if rc != 0:
        raise UgxError(rc, "ugx_compile_words: list outside its scope" if rc == 2 else "ugx_compile_words failed")
    return opc[:nop.value].copy(), pf.raw


class Pattern:
    """A compiled pattern uploaded to one device (immutable, shareable)."""

    def __init__(self, handle, device: int):
        self._h = handle
        self.device = device

    @classmethod
    def load(cls, path: str, device: int = 0) -> "Pattern":
        h = C.c_void_p()
        _check(lib().ugx_pattern_load(os.fsencode(path), device, C.byref(h)))
        return cls(h, device)

    @classmethod
    def literal(cls, text: bytes, device: int = 0, icase: bool = False) -> "Pattern":
        """`ugrep -F [-i] TEXT`: compiled by the library itself (ugx_compile_literal; with -i the word-list compiler on a
        list of one), no reference binary needed"""
        opc, pf = compile_words([text], True) if icase else compile_literal(text)
        h = C.c_void_p()
        _check(lib().ugx_pattern_create(opc.ctypes.data, len(opc), pf, 0, device, C.byref(h)))
        return cls(h, device)

    @classmethod
    def words(cls, words, device: int = 0, icase: bool = False) -> "Pattern":
        """`ugrep -F [-i] -f FILE`: compiled by the library itself (ugx_compile_words_ex)"""
        opc, pf = compile_words(words, icase)
        h = C.c_void_p()
        _check(lib().ugx_pattern_create(opc.ctypes.data, len(opc), pf, 0, device, C.byref(h)))
        return cls(h, device)

    @property
    def info(self) -> dict:
        i = _Info()
        _check(lib().ugx_pattern_info_get(self._h, C.byref(i)))
        d = {n: getattr(i, n) for n, _ in _Info._fields_}
        d["advance_name"] = ADVANCE_NAMES[d["advance"]] if d["advance"] < len(ADVANCE_NAMES) else "?"
        return d

    def close(self):
        if self._h:
            lib().ugx_pattern_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Scanner:
    """Per-thread / per-stream scan context (the Matcher side of the boundary)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._h = C.c_void_p()
        self.device = device
        _check(lib().ugx_scanner_create(device, C.c_void_p(stream or 0), C.byref(self._h)))

    def set_option(self, name: str, value: int) -> None:
        _check(lib().ugx_scanner_set_option(self._h, name.encode(), int(value)))

    def _totals(self, t: _Totals) -> Totals:
        return Totals(t.matches, t.newlines, t.flags, t.kernel_ms, t.launches,
                      lib().ugx_kernel_name(t.kernel).decode())

    def count_lines(self, pattern: Pattern, data) -> Totals:
        ptr, n, keep = _buffer(data)
        t = _Totals()
        _check(lib().ugx_count_lines(self._h, pattern._h, C.c_void_p(ptr), n, C.byref(t)))
        return self._totals(t)

    def count_matches(self, pattern: Pattern, data) -> Totals:
        ptr, n, keep = _buffer(data)
        t = _Totals()
        _check(lib().ugx_count_matches(self._h, pattern._h, C.c_void_p(ptr), n, C.byref(t)))
        return self._totals(t)

    def count_newlines(self, data) -> Totals:
        """reflex::nlcount over the buffer (totals.newlines)"""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        _check(lib().ugx_count_newlines(self._h, C.c_void_p(ptr), n, C.byref(t)))
        return self._totals(t)

    def count_batch(self, pattern: Pattern, files, mode: str = "lines"):
        """`ugrep -c` / `ugrep -c -o` of many files in ONE launch: (per-file counts, totals).  The files (bytes-like)
        are packed back to back on 16-byte boundaries into one host buffer, as a batching feeder would; or `files` is
        an already packed (buffer, begins, lens) with a host or device buffer."""
        ptr, n, keep, begins, lens = _batch_input(files)
        counts = np.zeros(max(1, len(lens)), dtype=np.uint64)
        t = _Totals()
        lib().ugx_count_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                          C.c_uint64, C.c_int, C.c_void_p, C.POINTER(_Totals)]
        _check(lib().ugx_count_batch(self._h, pattern._h, ptr, n, begins.ctypes.data, lens.ctypes.data,
                                     len(lens), 0 if mode == "lines" else 1, counts.ctypes.data, C.byref(t)))
        return counts[:len(lens)], self._totals(t)

    def batch_records_device(self, pattern: Pattern, files, lines: bool, invert: bool = False):
        """ugx_find_lines_batch (lines) or ugx_find_all_batch with the records left on the device: (first, totals);
        fetch_lines() / fetch() page through them.  `files` is a list of bytes-like, packed as for count_batch, or an
        already packed (buffer, begins, lens) with a host or device buffer and begins on 16-byte boundaries."""
        ptr, n, keep, begins, lens = _batch_input(files)
        first = np.zeros(len(lens) + 1, dtype=np.uint64)
        cnt = C.c_uint64()
        t = _Totals()
        args = (self._h, pattern._h, ptr, n, begins.ctypes.data, lens.ctypes.data, len(lens))
        if lines:
            _check(lib().ugx_find_lines_batch(*args, LINES_INVERT if invert else 0, first.ctypes.data, None, 0,
                                              C.byref(cnt), C.byref(t)))
        else:
            _check(lib().ugx_find_all_batch(*args, first.ctypes.data, None, 0, C.byref(cnt), C.byref(t)))
        return first, self._totals(t)

    def find_all_batch(self, pattern: Pattern, files):
        """`ugrep -o -n -b` of many files in one launch sequence: (match records, first, totals).  File i's records are
        rec[first[i]:first[i + 1]], exactly find_all(file i) with offsets and line numbers relative to the file.
        `files` as for batch_records_device."""
        first, t = self.batch_records_device(pattern, files, False)
        return self.fetch(0, t.matches), first, t

    def find_lines_batch(self, pattern: Pattern, files, invert: bool = False):
        """`ugrep -n` / `ugrep -v -n` of many files in one launch sequence: (line records, first, totals).  File i's
        records are rec[first[i]:first[i + 1]], exactly find_lines(file i, invert).  `files` as for
        batch_records_device."""
        first, t = self.batch_records_device(pattern, files, True, invert)
        return self.fetch_lines(0, t.matches), first, t

    def check_text(self, data) -> dict:
        """reflex::isutf8 / NUL test over the buffer (ugrep's binary-file detection)"""
        ptr, n, keep = _buffer(data)
        t = _TextInfo()
        lib().ugx_check_text.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(_TextInfo)]
        _check(lib().ugx_check_text(self._h, C.c_void_p(ptr), n, C.byref(t)))
        return {"is_utf8": bool(t.is_utf8), "has_nul": bool(t.has_nul), "kernel_ms": t.kernel_ms}

    def find_all_device(self, pattern: Pattern, data, base_offset: int = 0, base_line: int = 0) -> Totals:
        """Like find_all but the records stay on the device (fetch() copies a range to the host)."""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        dev = C.c_void_p()
        cnt = C.c_uint64()
        _check(lib().ugx_find_all_device(self._h, pattern._h, C.c_void_p(ptr), n, base_offset, base_line,
                                         C.byref(dev), C.byref(cnt), C.byref(t)))
        self.last_records = (dev.value, cnt.value)
        return self._totals(t)

    def fetch(self, first: int, count: int) -> np.ndarray:
        out = np.zeros(count, dtype=MATCH_DTYPE)
        if count:
            _check(lib().ugx_scanner_fetch(self._h, out.ctypes.data, first, count))
        return out

    def find_all(self, pattern: Pattern, data, base_offset: int = 0, base_line: int = 0):
        """All matches in input order as a structured array (line, offset, len, cap) + totals."""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        dev = C.c_void_p()
        cnt = C.c_uint64()
        _check(lib().ugx_find_all_device(self._h, pattern._h, C.c_void_p(ptr), n, base_offset, base_line,
                                         C.byref(dev), C.byref(cnt), C.byref(t)))
        out = np.zeros(cnt.value, dtype=MATCH_DTYPE)
        if cnt.value:
            _check(lib().ugx_scanner_fetch(self._h, out.ctypes.data, 0, cnt.value))
        return out, self._totals(t)

    def find_lines_device(self, pattern: Pattern, data, invert: bool = False, base_offset: int = 0,
                          base_line: int = 0) -> Totals:
        """Like find_lines but the records stay on the device (fetch_lines() copies a range to the host); the match
        records of find_all_device stay valid alongside."""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        dev = C.c_void_p()
        cnt = C.c_uint64()
        _check(lib().ugx_find_lines_device(self._h, pattern._h, C.c_void_p(ptr), n, base_offset, base_line,
                                           LINES_INVERT if invert else 0, C.byref(dev), C.byref(cnt), C.byref(t)))
        self.last_lines = (dev.value, cnt.value)
        return self._totals(t)

    def fetch_lines(self, first: int, count: int) -> np.ndarray:
        out = np.zeros(count, dtype=LINE_DTYPE)
        if count:
            _check(lib().ugx_scanner_fetch_lines(self._h, out.ctypes.data, first, count))
        return out

    def find_lines(self, pattern: Pattern, data, invert: bool = False, base_offset: int = 0, base_line: int = 0):
        """The lines the `ugrep -c` loop counts, each with its first match, in input order as a structured array
        (line, bol, eol, offset, len, cap) + totals; with invert the lines without a match (`ugrep -v`)."""
        t = self.find_lines_device(pattern, data, invert, base_offset, base_line)
        return self.fetch_lines(0, self.last_lines[1]), t

    def find_context_device(self, pattern: Pattern, data, before: int = 0, after: int = 0, invert: bool = False,
                            base_offset: int = 0, base_line: int = 0) -> Totals:
        """Like find_context but the records stay on the device: self.last_lines = (device pointer, printed lines),
        and fetch_lines() copies a range to the host.  totals.matches counts the selected lines."""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        dev = C.c_void_p()
        cnt = C.c_uint64()
        _check(lib().ugx_find_context_device(self._h, pattern._h, C.c_void_p(ptr), n, base_offset, base_line,
                                             LINES_INVERT if invert else 0, before, after, C.byref(dev), C.byref(cnt),
                                             C.byref(t)))
        self.last_lines = (dev.value, cnt.value)
        return self._totals(t)

    def find_context(self, pattern: Pattern, data, before: int = 0, after: int = 0, invert: bool = False,
                     base_offset: int = 0, base_line: int = 0):
        """`ugrep -n -B before -A after` (with invert `ugrep -v -n ...`): one record per printed line, in input order,
        each exactly as find_lines gives that line in its own polarity, + totals.  A record is a selected line iff
        (cap != 0) != invert, otherwise a context line; a gap in the line numbers is a group separator."""
        t = self.find_context_device(pattern, data, before, after, invert, base_offset, base_line)
        return self.fetch_lines(0, self.last_lines[1]), t

    def find_context_batch(self, pattern: Pattern, files, before: int = 0, after: int = 0, invert: bool = False):
        """`ugrep -rn -B before -A after` of many files in one launch sequence: (line records, first, totals).  File
        i's records are rec[first[i]:first[i + 1]], exactly find_context(file i); context never crosses files.
        `files` as for batch_records_device."""
        ptr, n, keep, begins, lens = _batch_input(files)
        first = np.zeros(len(lens) + 1, dtype=np.uint64)
        cnt = C.c_uint64()
        t = _Totals()
        _check(lib().ugx_find_context_batch(self._h, pattern._h, ptr, n, begins.ctypes.data, lens.ctypes.data,
                                            len(lens), LINES_INVERT if invert else 0, before, after, first.ctypes.data,
                                            None, 0, C.byref(cnt), C.byref(t)))
        return self.fetch_lines(0, cnt.value), first, self._totals(t)

    @staticmethod
    def _bool_query(patterns, cnf):
        """(pattern handle array, count, clause array, count) for the ugx_*_lines_bool calls; `cnf` is a CNF as
        bool_clauses takes it, or an already built BoolClause array"""
        pats = (C.c_void_p * len(patterns))(*[p._h for p in patterns])
        clauses = cnf if isinstance(cnf, C.Array) else bool_clauses(cnf)
        return pats, len(patterns), clauses, len(clauses)

    def count_lines_bool(self, patterns, cnf, data, invert: bool = False) -> Totals:
        """The number of lines that satisfy the CNF over the patterns' matching lines (`ugrep -c -e A --and -e B`,
        `--andnot`, `--bool`; with invert `-v`) in totals.matches.  See bool_clauses for the CNF."""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        _check(lib().ugx_count_lines_bool(self._h, *self._bool_query(patterns, cnf), C.c_void_p(ptr), n,
                                          LINES_INVERT if invert else 0, C.byref(t)))
        return self._totals(t)

    def find_lines_bool_device(self, patterns, cnf, data, invert: bool = False, base_offset: int = 0,
                               base_line: int = 0) -> Totals:
        """Like find_lines_bool but the records stay on the device: self.last_lines = (device pointer, records), and
        fetch_lines() copies a range to the host."""
        ptr, n, keep = _buffer(data)
        t = _Totals()
        dev = C.c_void_p()
        cnt = C.c_uint64()
        _check(lib().ugx_find_lines_bool_device(self._h, *self._bool_query(patterns, cnf), C.c_void_p(ptr), n,
                                                base_offset, base_line, LINES_INVERT if invert else 0, C.byref(dev),
                                                C.byref(cnt), C.byref(t)))
        self.last_lines = (dev.value, cnt.value)
        return self._totals(t)

    def find_lines_bool(self, patterns, cnf, data, invert: bool = False, base_offset: int = 0, base_line: int = 0):
        """The lines that satisfy the CNF (with invert: that do not), in input order as LINE_DTYPE records + totals.
        offset = bol, len = 0, and cap is the line's term mask: bit j set iff patterns[j] matches on the line."""
        t = self.find_lines_bool_device(patterns, cnf, data, invert, base_offset, base_line)
        return self.fetch_lines(0, self.last_lines[1]), t

    def count_lines_bool_batch(self, patterns, cnf, files, invert: bool = False):
        """`ugrep -rc -e A --and -e B` of many files in one launch sequence: (per-file counts, totals).  counts[i] is
        count_lines_bool(file i).matches; `-l` is counts != 0.  `files` as for batch_records_device."""
        ptr, n, keep, begins, lens = _batch_input(files)
        counts = np.zeros(max(1, len(lens)), dtype=np.uint64)
        t = _Totals()
        _check(lib().ugx_count_lines_bool_batch(self._h, *self._bool_query(patterns, cnf), ptr, n, begins.ctypes.data,
                                                lens.ctypes.data, len(lens), LINES_INVERT if invert else 0,
                                                counts.ctypes.data, C.byref(t)))
        return counts[:len(lens)], self._totals(t)

    def find_lines_bool_batch_device(self, patterns, cnf, files, invert: bool = False):
        """ugx_find_lines_bool_batch with the records left on the device: (first, totals); fetch_lines() pages through
        them.  `files` as for batch_records_device."""
        ptr, n, keep, begins, lens = _batch_input(files)
        first = np.zeros(len(lens) + 1, dtype=np.uint64)
        cnt = C.c_uint64()
        t = _Totals()
        _check(lib().ugx_find_lines_bool_batch(self._h, *self._bool_query(patterns, cnf), ptr, n, begins.ctypes.data,
                                               lens.ctypes.data, len(lens), LINES_INVERT if invert else 0,
                                               first.ctypes.data, None, 0, C.byref(cnt), C.byref(t)))
        return first, self._totals(t)

    def find_lines_bool_batch(self, patterns, cnf, files, invert: bool = False):
        """`ugrep -rn -e A --and -e B` of many files in one launch sequence: (line records, first, totals).  File i's
        records are rec[first[i]:first[i + 1]], exactly find_lines_bool(file i, invert).  `files` as for
        batch_records_device."""
        first, t = self.find_lines_bool_batch_device(patterns, cnf, files, invert)
        return self.fetch_lines(0, t.matches), first, t

    def close(self):
        if self._h:
            lib().ugx_scanner_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Shard(C.Structure):
    _fields_ = [("device", C.c_int32), ("reserved", C.c_uint32), ("begin", C.c_uint64), ("end", C.c_uint64),
                ("matches", C.c_uint64), ("newlines", C.c_uint64), ("line_base", C.c_uint64), ("record_base", C.c_uint64),
                ("kernel_ms", C.c_float), ("reserved2", C.c_uint32)]


def read_ugxp(path: str):
    """(opcode words, prefilter bytes, matcher flags) of a UGXP pattern file (include/ugrep_b200.h ugx_file_header)"""
    raw = open(path, "rb").read()
    if raw[:8] != b"UGXP\x01\x00\x00\x00":
        raise UgxError(6, "not a UGXP pattern file: %s" % path)
    nop, _, pfsize, flags = np.frombuffer(raw, dtype="<u4", count=4, offset=8)
    pf = raw[24:24 + int(pfsize)]
    opc = np.frombuffer(raw, dtype="<u4", count=int(nop), offset=24 + int(pfsize)).copy()
    return opc, pf, int(flags)


def compile_plain(patterns, icase: bool = False):
    """`ugrep [-i] -e A -e B ...` WITHOUT -F, for patterns that are alternations of plain strings (escaped operators,
    \\t, \\Q..\\E and top-level | allowed): ugx_compile_plain_regex on the patterns joined with |, as ugrep joins
    them.  UgxError code 2 for anything else: the regex compiler proper is not part of this library."""
    L = lib()
    L.ugx_compile_plain_regex.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                                          C.c_void_p]
    regex = b"|".join(bytes(p) for p in patterns)
    cap = 4 * (len(regex) + 2 * (regex.count(b"|") + 1)) + 16
    opc = np.zeros(cap, dtype=np.uint32)
    nop = C.c_uint32()
    pf = C.create_string_buffer(PREFILTER_BYTES)
    rc = L.ugx_compile_plain_regex(regex, len(regex), 1 if icase else 0, opc.ctypes.data, cap, C.byref(nop), pf)
    if rc != 0:
        raise UgxError(rc, "ugx_compile_plain_regex: not an alternation of plain strings" if rc == 2 else
                       "ugx_compile_plain_regex failed")
    return opc[:nop.value].copy(), pf.raw


def write_ugxp(path: str, opc, pf: bytes, flags: int = 0) -> None:
    """the inverse of read_ugxp: a UGXP pattern file from compiled words (no regex text is stored)"""
    import struct
    with open(path, "wb") as f:
        f.write(b"UGXP\x01\x00\x00\x00" + struct.pack("<4I", len(opc), 0, len(pf), int(flags)) + bytes(pf)
                + np.asarray(opc, dtype="<u4").tobytes())


class Sharded:
    """One process, several GPUs: ugx_sharded_* (line-aligned shards of one host buffer, one device each)."""

    MODES = {"lines": 0, "matches": 1, "records": 2}

    def __init__(self, pattern_path: str, devices):
        L = lib()
        L.ugx_sharded_create.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_void_p)]
        L.ugx_sharded_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                       C.POINTER(C.c_uint64), C.POINTER(_Totals), C.c_void_p]
        L.ugx_sharded_find_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64,
                                             C.POINTER(C.c_uint64), C.POINTER(_Totals), C.c_void_p]
        L.ugx_sharded_destroy.argtypes = [C.c_void_p]
        L.ugx_sharded_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.ugx_sharded_last_error.restype = C.c_char_p
        opc, pf, flags = read_ugxp(pattern_path)
        self.devices = list(devices)
        devs = (C.c_int * len(self.devices))(*self.devices)
        self._h = C.c_void_p()
        rc = L.ugx_sharded_create(opc.ctypes.data, len(opc), pf, flags, devs, len(self.devices), C.byref(self._h))
        if rc != 0:
            raise UgxError(rc, L.ugx_sharded_last_error().decode("utf-8", "replace"))

    def set_option(self, name: str, value: int) -> None:
        rc = lib().ugx_sharded_set_option(self._h, name.encode(), int(value))
        if rc != 0:
            raise UgxError(rc, lib().ugx_sharded_last_error().decode("utf-8", "replace"))

    def scan(self, data, mode: str = "lines", cap: int | None = None):
        """-> (totals, records or None, per-shard info)"""
        ptr, n, keep = _buffer(data)
        if hasattr(keep, "is_cuda"):
            raise TypeError("ugx_sharded_scan takes host memory")
        t = _Totals()
        shards = (_Shard * len(self.devices))()
        cnt = C.c_uint64()
        out = None
        m = self.MODES[mode]
        if m == 2:
            out = np.zeros(cap if cap is not None else max(1024, n // 8), dtype=MATCH_DTYPE)
        rc = lib().ugx_sharded_scan(self._h, C.c_void_p(ptr), n, m, out.ctypes.data if out is not None else None,
                                    len(out) if out is not None else 0, C.byref(cnt), C.byref(t), shards)
        if rc != 0:
            raise UgxError(rc, lib().ugx_sharded_last_error().decode("utf-8", "replace"))
        info = [{f: getattr(sh, f) for f, _ in _Shard._fields_ if not f.startswith("reserved")} for sh in shards]
        tot = Totals(t.matches, t.newlines, t.flags, t.kernel_ms, t.launches, lib().ugx_kernel_name(t.kernel).decode())
        return tot, (out[:cnt.value] if out is not None else None), info

    def find_lines(self, data, invert: bool = False, cap: int | None = None):
        """-> (line records of all shards in input order, totals, per-shard info); shard record_base = line records
        before the shard"""
        ptr, n, keep = _buffer(data)
        if hasattr(keep, "is_cuda"):
            raise TypeError("ugx_sharded_find_lines takes host memory")
        t = _Totals()
        shards = (_Shard * len(self.devices))()
        cnt = C.c_uint64()
        if cap is None:
            cap = n // 2 + 16 if invert else max(1024, n // 16)
        out = np.zeros(cap, dtype=LINE_DTYPE)
        args = (self._h, C.c_void_p(ptr), n, LINES_INVERT if invert else 0)
        rc = lib().ugx_sharded_find_lines(*args, out.ctypes.data, cap, C.byref(cnt), C.byref(t), shards)
        if rc == 5:  # UGX_E_OVERFLOW: *n_out holds the count
            cap = cnt.value
            out = np.zeros(max(cap, 1), dtype=LINE_DTYPE)
            rc = lib().ugx_sharded_find_lines(*args, out.ctypes.data, cap, C.byref(cnt), C.byref(t), shards)
        if rc != 0:
            raise UgxError(rc, lib().ugx_sharded_last_error().decode("utf-8", "replace"))
        info = [{f: getattr(sh, f) for f, _ in _Shard._fields_ if not f.startswith("reserved")} for sh in shards]
        tot = Totals(t.matches, t.newlines, t.flags, t.kernel_ms, t.launches, lib().ugx_kernel_name(t.kernel).decode())
        return out[:cnt.value], tot, info

    def close(self):
        if self._h:
            lib().ugx_sharded_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
