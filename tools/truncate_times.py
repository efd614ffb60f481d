#!/usr/bin/env python3
"""Cost of the truncated encode (cfbpe_encode_truncated) on BASELINE.json config 3 (65 536 prompts of 8..4096 B), host path:
  count_batch                     the token counts alone
  count-only truncation           kept counts and byte cuts, no id leaves the device (HEAD and TAIL, L = 512)
  rows                            n x L id rows, kept counts, cuts (L = 128, 512, 2048; HEAD)
  encode + host slicing           what a caller does without it: the whole id stream down, rows and cuts built in numpy
Host wall time of one call, median of REPS calls after WARM warm-up calls, pinned host buffers throughout; then the window kernels'
event time (cfbpe_profile kernel_ms[9], a one-shot call with profiling on) for each truncation case.  The card's name and power
limit are read in the same run.  Writes profiles/truncate_times_<tag>.jsonl (or OUTDIR/truncate_times_<tag>.jsonl).
usage: truncate_times.py TAG [OUTDIR]"""
import os; os.environ.setdefault("CFBPE_ALLOW_STAND_IN", "1")
import base64, json, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "cyberfabric-core_b200")):
    sys.path.insert(0, p)
import numpy as np
from cfbpe import _native as N, plugin as P, workload as W

WARM, REPS = 3, 11
tag = sys.argv[1] if len(sys.argv) > 1 else "dev"
outdir = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles")
os.makedirs(outdir, exist_ok=True)
out_path = os.path.join(outdir, "truncate_times_%s.jsonl" % tag)

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
card = q.stdout.strip()

data, offs, vid, meta = W.make_config(3, 1.0)
n, total = len(offs) - 1, int(offs[-1])
plug = P.GpuBpeTokenizerPlugin(0, tuple(meta["vocabs"]), 256 << 20, 1 << 17)
ctx, lib = plug.ctx, N.load()
rv = plug.resolved[meta["vocabs"][0]]
tok_len = np.array([len(base64.b64decode(l.split()[0])) for l in rv.file_bytes.splitlines()[:rv.max_ranks or None]], dtype=np.uint64)

hb = ctx.pinned(total, np.uint8); hb.array[:] = data
h_ids, h_off, h_cnt = ctx.pinned(total + 1, np.uint32), ctx.pinned(n + 1, np.uint64), ctx.pinned(n, np.uint32)
h_rows = ctx.pinned(n * 2048, np.uint32)
h_kept, h_cut = ctx.pinned(n, np.uint32), ctx.pinned(n, np.uint64)


def truncated(L, keep, rows):
    rc = lib.cfbpe_encode_truncated(ctx._h, n, hb.ptr, offs.ctypes.data, None, L, keep, 0, None, h_rows.ptr if rows else None,
                                    h_kept.ptr, h_cnt.ptr, h_cut.ptr)
    assert rc == 0, rc


def encode_and_slice(L):
    ids, off, cnt = ctx.encode_batch(hb.array, offs, None, h_ids.array, h_off.array, h_cnt.array)
    k = np.minimum(cnt, L).astype(np.int64)
    j = np.arange(L, dtype=np.int64)
    idx = np.minimum(off[:-1, None].astype(np.int64) + j[None, :], max(len(ids) - 1, 0))
    rows = np.where(j[None, :] < k[:, None], ids[idx], 0).astype(np.uint32)
    cum = np.zeros(len(ids) + 1, dtype=np.uint64)
    np.cumsum(tok_len[ids], out=cum[1:])
    cut = cum[off[:-1].astype(np.int64) + k] - cum[off[:-1].astype(np.int64)]
    return rows, cut


def timed(fn):
    for _ in range(WARM):
        fn()
    t = []
    for _ in range(REPS):
        t0 = time.perf_counter(); fn(); t.append(time.perf_counter() - t0)
    return float(np.median(t)) * 1e3, float(min(t)) * 1e3


def window_ms(L, keep, rows):
    ctx.profile_enable(True)
    ms = []
    for _ in range(WARM + REPS):
        truncated(L, keep, rows)
        ms.append(ctx.profile_read()["kernel_ms"]["window"])
    ctx.profile_enable(False)
    return float(np.median(ms[WARM:]))


# the rows equal the host-side slices of the full encoding (the comparison is of equal results)
truncated(512, 0, True)
ref_rows, ref_cut = encode_and_slice(512)
assert np.array_equal(h_rows.array[:n * 512].reshape(n, 512), ref_rows) and np.array_equal(h_cut.array, ref_cut)

cases = [("count_batch", None, None, lambda: ctx.count_batch(hb.array, offs, None, h_cnt.array), None)]
cases += [("count-only truncation", 512, k, (lambda k=k: truncated(512, k, False)), (512, k, False)) for k in (0, 1)]
cases += [("rows", L, 0, (lambda L=L: truncated(L, 0, True)), (L, 0, True)) for L in (128, 512, 2048)]
cases += [("encode + host slicing", L, 0, (lambda L=L: encode_and_slice(L)), None) for L in (128, 512, 2048)]
with open(out_path, "w") as f:
    for name, L, keep, fn, prof in cases:
        med, best = timed(fn)
        rec = {"case": name, "max_tokens": L, "keep": None if keep is None else ("head", "tail")[keep], "median_ms": round(med, 3),
               "min_ms": round(best, 3), "calls": REPS, "prompts": n, "bytes": total,
               "rows_bytes": n * L * 4 if L and "count-only" not in name else 0,
               "window_kernels_ms": round(window_ms(*prof), 4) if prof else None, "card": card}
        print(json.dumps(rec), flush=True)
        f.write(json.dumps(rec) + "\n")
plug.close()
