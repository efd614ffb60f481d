"""ctypes binding of the truncated-encode emulator harness (tests/simt/sim_truncate.cpp; test infrastructure)."""
import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(os.path.dirname(_DIR)), "cyberfabric-core_b200", "csrc")
SO = os.path.join(_DIR, "_build", "libcfbpe_sim_truncate.so")

_lib = None


def build():
    """g++ with the flags of tests/simt/build.py; rebuilt when a source is newer than the library"""
    srcs = [os.path.join(_DIR, "sim_truncate.cpp"), os.path.join(_CSRC, "vocab.cpp")]
    deps = srcs + [os.path.join(_DIR, f) for f in ("sim_harness.cpp", "cusim.h")] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in deps):
        return SO
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-fno-omit-frame-pointer",
                           "-Wall", "-Wno-unused-function", "-Wno-unknown-pragmas", "-Wno-sign-compare", "-DCFBPE_SIM=1", "-o", SO] + srcs)
    return SO


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.sim_vocab_build.restype = C.c_void_p
        L.sim_vocab_build.argtypes = [C.c_char_p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p, C.c_size_t]
        L.sim_vocab_free.argtypes = [C.c_void_p]
        L.sim_encode_truncated.restype = C.c_int
        L.sim_encode_truncated.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                           C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class Vocab:
    """a vocabulary's packed tables, built by this harness (csrc/vocab.cpp)"""

    def __init__(self, file_bytes, fmt, pattern, max_ranks=0):
        err = C.create_string_buffer(256)
        self._h = lib().sim_vocab_build(file_bytes, len(file_bytes), fmt, pattern, max_ranks, err, 256)
        if not self._h:
            raise ValueError(err.value.decode())

    def __del__(self):
        if getattr(self, "_h", None):
            lib().sim_vocab_free(self._h)
            self._h = None


def pack(prompts):
    offs = np.zeros(len(prompts) + 1, dtype=np.uint64)
    if prompts:
        offs[1:] = np.cumsum([len(p) for p in prompts], dtype=np.uint64)
    data = np.frombuffer(b"".join(prompts), dtype=np.uint8).copy() if prompts else np.zeros(0, np.uint8)
    return data, offs


def encode_truncated(vocabs, prompts, max_tokens, keep=0, pad_id=0, budgets=None, vocab_ids=None, want_rows=True, want_cut=True):
    """K1..K3, then the window stage: (rc, rows [n, L] | None, kept, counts, cut | None, pieces taken by the long-piece kernels)"""
    data, offs = pack(prompts)
    n = len(prompts)
    rows = np.full((max(n, 1), max_tokens), 0xDEADBEEF, dtype=np.uint32) if want_rows else None
    kept = np.full(max(n, 1), 0xDEADBEEF, dtype=np.uint32)
    counts = np.full(max(n, 1), 0xDEADBEEF, dtype=np.uint32)
    cut = np.full(max(n, 1), 0xDEADBEEF, dtype=np.uint64) if want_cut else None
    bud = None if budgets is None else np.ascontiguousarray(budgets, dtype=np.uint32)
    vh = (C.c_void_p * len(vocabs))(*[v._h for v in vocabs])
    vid = None if vocab_ids is None else np.ascontiguousarray(vocab_ids, dtype=np.uint8)
    dbuf = np.concatenate([data, np.zeros(64, np.uint8)])
    nlong = C.c_uint64(0)

    def ptr(a):
        return None if a is None else a.ctypes.data
    rc = lib().sim_encode_truncated(vh, len(vocabs), n, dbuf.ctypes.data, offs.ctypes.data, ptr(vid), max_tokens, keep, pad_id,
                                    ptr(bud), ptr(rows), kept.ctypes.data, counts.ctypes.data, ptr(cut), C.byref(nlong))
    return rc, None if rows is None else rows[:n], kept[:n], counts[:n], None if cut is None else cut[:n], nlong.value
