"""ctypes binding of libcfbpe.so (include/cfbpe.h).  No fallback: if the CUDA library is not
built or no sm_100 device is present, loading / creating a context raises."""
import ctypes as C
import os

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # effective if CUDA is not initialised yet; see csrc/cfbpe.cu:cfbpe_create
_DIR = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("CFBPE_SO_VARIANT") or os.path.join(_DIR, "libcfbpe.so")   # CFBPE_SO_VARIANT: A/B builds (tools only)

OK, ENOENT, EIO, ENOMEM, ENODEV, EINVAL, ENOSPC, EILSEQ = 0, -2, -5, -12, -19, -22, -28, -84
FORMAT_TIKTOKEN, FORMAT_TEKKEN_JSON = 0, 1
PATTERN_CL100K, PATTERN_O200K, PATTERN_LLAMA3, PATTERN_TEKKEN = 0, 1, 2, 3
PATTERN_IDS = {"cl100k": 0, "o200k": 1, "llama3": 2, "tekken": 3}
MAX_VOCABS = 8
NUM_KERNELS = 10
KERNEL_NAMES = ["pretok_split", "bpe_encode", "bpe_long", "flag_count", "tile_scan", "emit_compact", "bpe_list", "long_scan", "bpe_merge", "window"]
KEEP_HEAD, KEEP_TAIL = 0, 1
KEEP = {"head": KEEP_HEAD, "tail": KEEP_TAIL}

# every symbol include/cfbpe.h declares (checked by tests/test_abi.py without a GPU)
EXPORTS = [
    "cfbpe_abi_version", "cfbpe_build_id", "cfbpe_create", "cfbpe_destroy", "cfbpe_last_error", "cfbpe_vocab_load",
    "cfbpe_vocab_get_info", "cfbpe_vocab_export", "cfbpe_vocab_import", "cfbpe_encode_batch", "cfbpe_count_batch",
    "cfbpe_encode_batch_device", "cfbpe_device_status", "cfbpe_host_alloc", "cfbpe_host_free",
    "cfbpe_profile_enable", "cfbpe_profile_read", "cfbpe_decode_batch", "cfbpe_encode_truncated", "cfbpe_encode_truncated_device",
]


MAX_DEVICES = 8


class Config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("max_batch_bytes", C.c_uint64),
                ("max_prompts", C.c_uint32), ("flags", C.c_uint32),
                ("devices", C.c_int32 * MAX_DEVICES), ("n_devices", C.c_uint32), ("n_workspaces", C.c_uint32)]


class VocabInfo(C.Structure):
    _fields_ = [("n_ranks", C.c_uint32), ("pattern_id", C.c_uint32), ("max_token_len", C.c_uint32),
                ("n_pair_entries", C.c_uint32), ("table_bytes", C.c_uint64)]


class Profile(C.Structure):
    _fields_ = [("kernel_ms", C.c_float * NUM_KERNELS), ("kernel_launches", C.c_uint32 * NUM_KERNELS),
                ("h2d_ms", C.c_float), ("d2h_ms", C.c_float), ("total_ms", C.c_float),
                ("n_tokens", C.c_uint64), ("n_bytes", C.c_uint64), ("n_long_pieces", C.c_uint64),
                ("n_long_bytes", C.c_uint64), ("n_long_tokens", C.c_uint64),
                ("n_miss_pieces", C.c_uint64), ("n_list_pieces", C.c_uint64), ("n_list_parts", C.c_uint64), ("n_extra_tokens", C.c_uint64)]


_lib = None


def load():
    """dlopen libcfbpe.so; raises if the extension has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError("libcfbpe.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'`. "
                           "There is no CPU fallback." % SO_PATH)
    L = C.CDLL(SO_PATH)
    vp, u8p = C.c_void_p, C.c_void_p
    L.cfbpe_abi_version.restype = C.c_int
    L.cfbpe_build_id.restype = C.c_char_p
    # refuse a binary that was not built from the sources next to it (a failed rebuild must not go unnoticed)
    bpy = os.path.join(os.path.dirname(_DIR), "build.py")
    if os.path.exists(bpy) and os.path.isdir(os.path.join(os.path.dirname(_DIR), "csrc")):
        import importlib.util
        spec = importlib.util.spec_from_file_location("cfbpe_build", bpy)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        want, got = mod.source_hash(), L.cfbpe_build_id().decode()
        if want != got and not os.environ.get("CFBPE_SO_VARIANT"):
            raise RuntimeError("libcfbpe.so is stale (built from %s, sources are %s): rebuild with "
                               "`python -c 'import __graft_entry__ as g; g.build()'`" % (got, want))
    L.cfbpe_create.restype = C.c_int
    L.cfbpe_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.cfbpe_destroy.argtypes = [vp]
    L.cfbpe_destroy.restype = None
    L.cfbpe_last_error.restype = C.c_char_p
    L.cfbpe_last_error.argtypes = [vp]
    L.cfbpe_vocab_load.restype = C.c_int
    L.cfbpe_vocab_load.argtypes = [vp, C.c_uint32, C.c_char_p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32]
    L.cfbpe_vocab_get_info.restype = C.c_int
    L.cfbpe_vocab_get_info.argtypes = [vp, C.c_uint32, C.POINTER(VocabInfo)]
    L.cfbpe_vocab_export.restype = C.c_int
    L.cfbpe_vocab_export.argtypes = [vp, C.c_uint32, u8p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.cfbpe_vocab_import.restype = C.c_int
    L.cfbpe_vocab_import.argtypes = [vp, C.c_uint32, u8p, C.c_uint64]
    L.cfbpe_encode_batch.restype = C.c_int
    L.cfbpe_encode_batch.argtypes = [vp, C.c_uint32, u8p, vp, u8p, vp, C.c_uint64, vp, vp]
    L.cfbpe_count_batch.restype = C.c_int
    L.cfbpe_count_batch.argtypes = [vp, C.c_uint32, u8p, vp, u8p, vp]
    L.cfbpe_decode_batch.restype = C.c_int
    L.cfbpe_decode_batch.argtypes = [vp, C.c_uint32, vp, vp, u8p, vp, C.c_uint64, vp]
    L.cfbpe_encode_batch_device.restype = C.c_int
    L.cfbpe_encode_batch_device.argtypes = [vp, C.c_uint32, vp, C.c_uint64, vp, vp, vp, C.c_uint64, vp, vp,
                                            C.POINTER(C.c_uint64), vp]
    L.cfbpe_encode_truncated.restype = C.c_int
    L.cfbpe_encode_truncated.argtypes = [vp, C.c_uint32, u8p, vp, u8p, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp, vp, vp]
    L.cfbpe_encode_truncated_device.restype = C.c_int
    L.cfbpe_encode_truncated_device.argtypes = [vp, C.c_uint32, vp, C.c_uint64, vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp,
                                                vp, vp, vp]
    L.cfbpe_device_status.restype = C.c_int
    L.cfbpe_device_status.argtypes = [vp, vp]
    L.cfbpe_host_alloc.restype = vp
    L.cfbpe_host_alloc.argtypes = [vp, C.c_size_t]
    L.cfbpe_host_free.restype = None
    L.cfbpe_host_free.argtypes = [vp, vp]
    L.cfbpe_profile_enable.restype = C.c_int
    L.cfbpe_profile_enable.argtypes = [vp, C.c_int]
    L.cfbpe_profile_read.restype = C.c_int
    L.cfbpe_profile_read.argtypes = [vp, C.POINTER(Profile)]
    _lib = L
    return L


class NativeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("cfbpe error %d: %s" % (code, msg))
        self.code = code


class PinnedArray:
    """numpy view over page-locked host memory owned by the library (cfbpe_host_alloc)."""

    def __init__(self, ctx, shape, dtype):
        self._ctx = ctx
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) if not isinstance(shape, int) else shape
        self.nbytes = max(n * dtype.itemsize, 1)
        self.ptr = load().cfbpe_host_alloc(ctx._h, self.nbytes)
        if not self.ptr:
            raise NativeError(ENOMEM, "cfbpe_host_alloc failed")
        buf = (C.c_uint8 * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)

    def free(self):
        if self.ptr and self._ctx._h:
            self.array = None
            load().cfbpe_host_free(self._ctx._h, self.ptr)
        self.ptr = None


class Context:
    """One context: one device (`device`) or several (`devices`: a host batch is sharded over them, NCCL inside the library),
    `n_workspaces` independent workspaces per device (that many calls run concurrently).  max_batch_bytes is per device."""

    def __init__(self, device=0, max_batch_bytes=0, max_prompts=0, devices=None, n_workspaces=1):
        self._h = None
        L = load()
        cfg = Config(C.sizeof(Config), device, max_batch_bytes, max_prompts, 0)
        if devices:
            if len(devices) > MAX_DEVICES:
                raise NativeError(EINVAL, "at most %d devices" % MAX_DEVICES)
            for i, d in enumerate(devices):
                cfg.devices[i] = int(d)
            cfg.n_devices = len(devices)
            device = int(devices[0])
        cfg.n_workspaces = int(n_workspaces)
        self.devices = list(devices) if devices else [device]
        self.n_workspaces = int(n_workspaces)
        h = C.c_void_p()
        rc = L.cfbpe_create(C.byref(cfg), C.byref(h))
        if rc != OK:
            raise NativeError(rc, "cfbpe_create failed (no sm_100 device visible?)" if rc == ENODEV else
                              ("cfbpe_create failed: " + L.cfbpe_last_error(None).decode("utf-8", "replace")))
        self._h = h
        self.device = device

    def close(self):
        if self._h:
            load().cfbpe_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise NativeError(rc, load().cfbpe_last_error(self._h).decode("utf-8", "replace"))

    # ---- vocab
    def vocab_load(self, vocab_id, file_bytes, fmt, pattern_id, max_ranks=0):
        self._check(load().cfbpe_vocab_load(self._h, vocab_id, file_bytes, len(file_bytes), fmt, pattern_id, max_ranks))

    def vocab_info(self, vocab_id):
        vi = VocabInfo()
        self._check(load().cfbpe_vocab_get_info(self._h, vocab_id, C.byref(vi)))
        return {"n_ranks": vi.n_ranks, "pattern_id": vi.pattern_id, "max_token_len": vi.max_token_len,
                "n_pair_entries": vi.n_pair_entries, "table_bytes": vi.table_bytes}

    def vocab_export(self, vocab_id) -> np.ndarray:
        size = C.c_uint64(0)
        self._check(load().cfbpe_vocab_export(self._h, vocab_id, None, 0, C.byref(size)))
        buf = np.empty(size.value, dtype=np.uint8)
        self._check(load().cfbpe_vocab_export(self._h, vocab_id, buf.ctypes.data, size.value, C.byref(size)))
        return buf

    def vocab_import(self, vocab_id, blob: np.ndarray):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self._check(load().cfbpe_vocab_import(self._h, vocab_id, blob.ctypes.data, blob.size))

    # ---- host-buffer API
    @staticmethod
    def _check_inputs(data, offsets, vocab_ids, what="bytes", dtype=np.uint8):
        """The C ABI takes pointers without lengths: what it cannot check is checked here (the Rust binding does the same on
        its slices) -- dtypes, contiguity, offsets[n] inside the buffer, one vocab id per prompt."""
        def bad(msg):
            return NativeError(EINVAL, msg)
        if not isinstance(offsets, np.ndarray) or offsets.dtype != np.uint64 or offsets.ndim != 1 or len(offsets) < 1 or not offsets.flags.c_contiguous:
            raise bad("offsets must be a C-contiguous uint64 array of n+1 entries")
        if not isinstance(data, np.ndarray) or data.dtype != dtype or data.ndim != 1 or not data.flags.c_contiguous:
            raise bad("%s must be a C-contiguous 1-D %s array" % (what, np.dtype(dtype).name))
        n = len(offsets) - 1
        if int(offsets[n]) > data.size:
            raise bad("offsets[n] = %d exceeds len(%s) = %d" % (int(offsets[n]), what, data.size))
        if vocab_ids is not None:
            if not isinstance(vocab_ids, np.ndarray) or vocab_ids.dtype != np.uint8 or vocab_ids.ndim != 1 or len(vocab_ids) < n or not vocab_ids.flags.c_contiguous:
                raise bad("vocab_ids must be a C-contiguous uint8 array with one entry per prompt")
        return n

    def encode_batch(self, data: np.ndarray, offsets: np.ndarray, vocab_ids=None, out_ids=None, out_offsets=None,
                     out_counts=None):
        n = self._check_inputs(data, offsets, vocab_ids)
        total = int(offsets[n])
        if out_ids is None:
            out_ids = np.empty(max(total, 1), dtype=np.uint32)
        if out_offsets is None:
            out_offsets = np.empty(n + 1, dtype=np.uint64)
        if out_counts is None:
            out_counts = np.empty(max(n, 1), dtype=np.uint32)
        vid = None if vocab_ids is None else vocab_ids.ctypes.data
        rc = load().cfbpe_encode_batch(self._h, n, data.ctypes.data if data.size else None, offsets.ctypes.data, vid,
                                       out_ids.ctypes.data, out_ids.size, out_offsets.ctypes.data,
                                       out_counts.ctypes.data)
        self._check(rc)
        return out_ids[:int(out_offsets[n])], out_offsets, out_counts[:n]

    def count_batch(self, data: np.ndarray, offsets: np.ndarray, vocab_ids=None, out_counts=None):
        n = self._check_inputs(data, offsets, vocab_ids)
        if out_counts is None:
            out_counts = np.empty(max(n, 1), dtype=np.uint32)
        vid = None if vocab_ids is None else vocab_ids.ctypes.data
        self._check(load().cfbpe_count_batch(self._h, n, data.ctypes.data if data.size else None, offsets.ctypes.data,
                                             vid, out_counts.ctypes.data))
        return out_counts[:n]

    def encode_truncated(self, data: np.ndarray, offsets: np.ndarray, vocab_ids=None, *, max_tokens, keep=KEEP_HEAD, pad_id=0,
                         budgets=None, want_ids=True):
        """Every prompt cut to k_i = min(count_i, budgets[i], max_tokens) tokens (include/cfbpe.h: cfbpe_encode_truncated).
        keep: KEEP_HEAD | KEEP_TAIL (or "head" | "tail").  Returns (rows uint32 [n, max_tokens] | None without want_ids, kept uint32 n,
        counts uint32 n (untruncated), cut uint64 n (byte offset of the cut inside each prompt))."""
        n = self._check_inputs(data, offsets, vocab_ids)
        keep = KEEP.get(keep, keep) if isinstance(keep, str) else int(keep)
        if budgets is not None:
            if not isinstance(budgets, np.ndarray) or budgets.dtype != np.uint32 or budgets.ndim != 1 or len(budgets) != n or not budgets.flags.c_contiguous:
                raise NativeError(EINVAL, "budgets must be a C-contiguous uint32 array with one entry per prompt")
        rows = np.empty((n, int(max_tokens)), dtype=np.uint32) if want_ids and max_tokens > 0 else None
        kept = np.empty(max(n, 1), dtype=np.uint32)
        counts = np.empty(max(n, 1), dtype=np.uint32)
        cut = np.empty(max(n, 1), dtype=np.uint64)
        vid = None if vocab_ids is None else vocab_ids.ctypes.data
        rc = load().cfbpe_encode_truncated(self._h, n, data.ctypes.data if data.size else None, offsets.ctypes.data, vid, int(max_tokens),
                                           keep, int(pad_id), None if budgets is None else budgets.ctypes.data,
                                           None if rows is None or not rows.size else rows.ctypes.data, kept.ctypes.data,
                                           counts.ctypes.data, cut.ctypes.data)
        self._check(rc)
        return rows, kept[:n], counts[:n], cut[:n]

    def decode_batch(self, ids: np.ndarray, id_offsets: np.ndarray, vocab_ids=None, out_cap=None, out_bytes=None, out_offsets=None):
        """ids (uint32, packed) + id_offsets (uint64, n+1) -> (bytes uint8, byte offsets uint64 n+1).
        out_bytes / out_offsets: caller's buffers (pinned ones make the download several times faster)"""
        n = self._check_inputs(ids, id_offsets, vocab_ids, "ids", np.uint32)
        if out_offsets is None:
            out_offsets = np.zeros(n + 1, dtype=np.uint64)
        vid = None if vocab_ids is None else vocab_ids.ctypes.data
        if out_bytes is not None:
            self._check(load().cfbpe_decode_batch(self._h, n, ids.ctypes.data if ids.size else None, id_offsets.ctypes.data, vid,
                                                  out_bytes.ctypes.data, out_bytes.size, out_offsets.ctypes.data))
            return out_bytes[:int(out_offsets[n])], out_offsets
        cap = int(out_cap) if out_cap is not None else max(int(len(ids)) * 8 + 64, 64)
        while True:
            out = np.empty(max(cap, 1), dtype=np.uint8)
            rc = load().cfbpe_decode_batch(self._h, n, ids.ctypes.data if ids.size else None, id_offsets.ctypes.data, vid,
                                           out.ctypes.data, cap, out_offsets.ctypes.data)
            if rc == ENOSPC and out_cap is None:
                cap = int(out_offsets[n])
                continue
            self._check(rc)
            return out[:int(out_offsets[n])], out_offsets

    # ---- device-buffer API (raw pointers; torch tensors pass .data_ptr())
    def encode_batch_device(self, n_prompts, d_bytes, total_bytes, d_offsets, d_vocab_ids, d_out_ids, out_cap,
                            d_out_offsets, d_out_counts, stream=0, sync=True):
        nt = C.c_uint64(0)
        rc = load().cfbpe_encode_batch_device(self._h, n_prompts, d_bytes, total_bytes, d_offsets, d_vocab_ids,
                                              d_out_ids, out_cap, d_out_offsets, d_out_counts,
                                              C.byref(nt) if sync else None, stream)
        self._check(rc)
        return nt.value if sync else None

    def encode_truncated_device(self, n_prompts, d_bytes, total_bytes, d_offsets, d_vocab_ids, max_tokens, keep, pad_id, d_budgets,
                                d_out_rows, d_out_kept, d_out_counts, d_out_cut, stream=0):
        """asynchronous, as encode_batch_device(sync=False): errors come from device_status"""
        self._check(load().cfbpe_encode_truncated_device(self._h, n_prompts, d_bytes, total_bytes, d_offsets, d_vocab_ids, int(max_tokens),
                                                         int(keep), int(pad_id), d_budgets, d_out_rows, d_out_kept, d_out_counts,
                                                         d_out_cut, stream))

    def device_status(self, stream=0):
        self._check(load().cfbpe_device_status(self._h, stream))

    def pinned(self, shape, dtype):
        return PinnedArray(self, shape, dtype)

    def profile_enable(self, on=True):
        self._check(load().cfbpe_profile_enable(self._h, 1 if on else 0))

    def profile_read(self):
        p = Profile()
        self._check(load().cfbpe_profile_read(self._h, C.byref(p)))
        return {"kernel_ms": {KERNEL_NAMES[i]: p.kernel_ms[i] for i in range(NUM_KERNELS)},
                "kernel_launches": {KERNEL_NAMES[i]: p.kernel_launches[i] for i in range(NUM_KERNELS)},
                "h2d_ms": p.h2d_ms, "d2h_ms": p.d2h_ms, "total_ms": p.total_ms, "n_tokens": p.n_tokens,
                "n_bytes": p.n_bytes, "n_long_pieces": p.n_long_pieces, "n_long_bytes": p.n_long_bytes,
                "n_long_tokens": p.n_long_tokens, "n_miss_pieces": p.n_miss_pieces, "n_list_pieces": p.n_list_pieces,
                "n_list_parts": p.n_list_parts, "n_extra_tokens": p.n_extra_tokens}
