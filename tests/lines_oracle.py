"""ctypes access to the oracle's line records (tests/oracle_lines.c: the `ugrep -c` loop of oracle/oracle.c recording
the match it finds on each line, plus the complement for `-v`).

TEST INFRASTRUCTURE: the library is compiled on first use into a temporary directory (keyed by the sources' hash), so
the repository tree stays as it is.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "oracle_lines.c"), os.path.join(ROOT, "oracle", "oracle.c"),
           os.path.join(ROOT, "oracle", "oracle.h"), os.path.join(ROOT, "include", "ugrep_b200.h")]
LINE_DTYPE = np.dtype([("line", "<u8"), ("bol", "<u8"), ("eol", "<u8"), ("offset", "<u8"), ("len", "<u4"), ("cap", "<u4")])

_lib = None


def _build() -> str:
    h = hashlib.sha256()
    for p in SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), "ugx_oracle_lines_%s_%d" % (h.hexdigest()[:16], os.getuid()))
    so = os.path.join(d, "liboracle_lines.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        if cc is None:
            raise RuntimeError("no C compiler for the oracle's line records")
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.run([cc, "-O2", "-Wall", "-fPIC", "-shared", "-o", tmp, SOURCES[0]], check=True)
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(_build())
        L.ora_pattern_load.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.ora_pattern_destroy.argtypes = [C.c_void_p]
        L.ora_find_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int,
                                     C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        _lib = L
    return _lib


class LinesOracle:
    """one compiled pattern of the oracle, for its line records"""

    def __init__(self, path: str):
        self.handle = C.c_void_p()
        rc = lib().ora_pattern_load(os.fsencode(path), C.byref(self.handle))
        if rc != 0:
            raise RuntimeError("ora_pattern_load(%s) -> %d" % (path, rc))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().ora_pattern_destroy(self.handle)
                self.handle = None
        except Exception:  # interpreter shutdown
            pass

    def find_lines(self, data, invert: bool = False, base_offset: int = 0, base_line: int = 0) -> np.ndarray:
        """the `ugrep -c` loop's lines with their first match (ugx_line records), or with invert the other lines"""
        a = np.frombuffer(bytes(data), dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else \
            np.ascontiguousarray(data, dtype=np.uint8)
        n = C.c_uint64()
        cap = a.size + 16
        out = np.zeros(cap, dtype=LINE_DTYPE)
        rc = lib().ora_find_lines(self.handle, a.ctypes.data, a.size, base_offset, base_line, 1 if invert else 0,
                                  out.ctypes.data, cap, C.byref(n))
        if rc != 0:
            raise RuntimeError("ora_find_lines -> %d" % rc)
        return out[: n.value].copy()


def oracle(path: str):
    """the oracle's pattern (oracle_lib.OraclePattern: counts, match records, ...) with find_lines added"""
    import oracle_lib as O

    class _Oracle(O.OraclePattern):
        def __init__(self, p):
            super().__init__(p)
            self._lines = LinesOracle(p)

        def find_lines(self, data, invert: bool = False, base_offset: int = 0, base_line: int = 0) -> np.ndarray:
            return self._lines.find_lines(data, invert, base_offset, base_line)

    return _Oracle(path)
